"""python -m mapper_b200 on 1, 2, 4 and 8 GPUs, and xm_rank_names against the host ranking it replaced.

Generates from a seed, in a temporary directory:
  - 20 M Illumina-style read names (fixed width, random lane / tile / x / y), ranked by xm_rank_names (wall time; device time of its
    kernels and copies from torch.profiler) and by np.unique(np.array(names, dtype=object), return_inverse=True) on this host;
  - configs[4] shape: a 50 Mbp reference in 8 contigs and 100 k x 10 kbp FASTA reads, mapped with --split-queries-past-size 1000 --out-sam;
  - configs[3] shape: a 250 Mbp reference in 50 contigs with 5 % repeats and 5 M x 150 bp FASTQ reads, mapped with --out-sam --out-vcf
    --out-mutations.
For every device count that exists (1, 2, 4, 8) it runs the command once per input and reports the wall time per phase (the command's
"wall s" line on stderr), the align kernel time per device, and the SHA-256 of every output, which must agree across device counts.
Usage: python tools/time_multi_gpu.py --out profiles/NAME.json [--names N] [--long-reads N] [--short-reads N]"""
import argparse
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mapper_b200 import capi, synth  # noqa: E402


def illumina_names(n, seed):
    """n names "A00123:8:H2FJ3DSXX:<lane>:<tile>:<x>:<y>" of one width: a (blob, offsets) pair."""
    rng = np.random.default_rng(seed)
    fields = [(rng.integers(1, 5, n), 1), (rng.integers(1101, 2679, n), 4), (rng.integers(10000, 32768, n), 5), (rng.integers(1000, 99999, n), 5)]
    cols = [np.frombuffer(b"A00123:8:H2FJ3DSXX", np.uint8)[None, :].repeat(n, 0)]
    for v, w in fields:
        digits = (v[:, None] // 10 ** np.arange(w - 1, -1, -1)[None, :]) % 10 + ord("0")
        cols += [np.full((n, 1), ord(":"), np.uint8), digits.astype(np.uint8)]
    m = np.concatenate(cols, axis=1)
    return m.tobytes(), np.arange(n + 1, dtype=np.int64) * m.shape[1]


def time_ranking(n):
    import torch
    from torch.profiler import ProfilerActivity, profile
    blob, off = illumina_names(n, seed=7)
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.rank_names(blob[:off[1000]], off[:1001])   # warm-up: module load
    t0 = time.perf_counter()
    got = g.rank_names(blob, off)
    wall = time.perf_counter() - t0
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g.rank_names(blob, off)
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kern_us = sum(e.device_time for e in ev if "emcpy" not in e.name and "emset" not in e.name)
    copy_us = sum(e.device_time for e in ev if "emcpy" in e.name)
    g.close()
    w = int(off[1])
    t0 = time.perf_counter()
    names = [blob[i * w:(i + 1) * w] for i in range(n)]
    t_list = time.perf_counter() - t0
    t0 = time.perf_counter()
    want = np.unique(np.array(names, dtype=object), return_inverse=True)[1].astype(np.int64).reshape(-1)
    t_unique = time.perf_counter() - t0
    return dict(names=n, name_bytes=w, distinct=int(want.max()) + 1, xm_rank_names=dict(wall_s=wall, device_kernel_s=kern_us / 1e6, device_copy_s=copy_us / 1e6),
                host_np_unique=dict(build_bytes_list_s=t_list, np_unique_s=t_unique), identical=bool(np.array_equal(got, want)))


def write_fasta(path, records):
    with open(path, "wb") as f:
        for name, codes in records:
            t = synth.LETTERS[codes]
            pad = (-len(t)) % 80
            rows = np.concatenate([t, np.zeros(pad, np.uint8)]).reshape(-1, 80)
            lines = np.concatenate([rows, np.full((len(rows), 1), ord("\n"), np.uint8)], axis=1)
            body = lines.tobytes()
            if pad:
                body = body[:-(pad + 1)] + b"\n"
            f.write(b">" + name.encode() + b"\n" + body)


def write_reads(path, ref, n, read_len, fastq, seed, indel_rate):
    with open(path, "wb") as f:
        step = max(1, min(n, (250000 * 150) // read_len))
        for lo in range(0, n, step):
            k = min(step, n - lo)
            b = synth.simulate_reads_fast(ref, k, read_len, seed=seed + lo, indel_rate=indel_rate)
            w = b["packed"].reshape(k, -1)
            codes = np.stack([w & 15, (w >> 4) & 15, (w >> 8) & 15, (w >> 12) & 15], axis=2).reshape(k, -1)[:, :read_len]
            seq = synth.LETTERS[codes]
            nl = np.full((k, 1), ord("\n"), np.uint8)
            names = np.frombuffer(b"".join((b"@" if fastq else b">") + b"r%09d\n" % (lo + i) for i in range(k)), np.uint8).reshape(k, -1)
            parts = [names, seq, nl]
            if fastq:
                parts += [np.frombuffer(b"+\n", np.uint8)[None, :].repeat(k, 0), np.full((k, read_len), ord("I"), np.uint8), nl]
            f.write(np.concatenate(parts, axis=1).tobytes())


def sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def run_command(d, args, outs, devices):
    paths = {k: os.path.join(d, "out." + k) for k in outs}
    flags = sum([["--out-" + {"sam": "sam", "vcf": "vcf", "mut": "mutations"}[k], p] for k, p in paths.items()], [])
    argv = [sys.executable, "-m", "mapper_b200", *args, *flags, "--device", ",".join(map(str, devices))]
    t0 = time.perf_counter()
    r = subprocess.run(argv, cwd=ROOT, capture_output=True, text=True)
    wall = time.perf_counter() - t0
    if r.returncode:
        return dict(devices=len(devices), error=r.stderr[-2000:])
    lines = [ln for ln in r.stderr.splitlines() if ln.startswith("mapper_b200:")]
    phases = {k: float(v) for k, v in re.findall(r"([a-z-]+) ([0-9.]+)", lines[-1].split("wall s:")[1])}
    per_dev = [float(x) for x in lines[-2].split("per device ")[1].rstrip(")").split()]
    out = dict(devices=len(devices), wall_s=wall, phases_s=phases, align_kernel_s_per_device=per_dev, stderr=lines,
               sha256={k: sha(p) for k, p in paths.items()}, bytes={k: os.path.getsize(p) for k, p in paths.items()})
    for p in paths.values():
        os.remove(p)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--names", type=int, default=20000000)
    ap.add_argument("--long-reads", type=int, default=100000)
    ap.add_argument("--short-reads", type=int, default=5000000)
    a = ap.parse_args()
    import torch
    n_gpu = torch.cuda.device_count()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    report = dict(gpu=smi[0] if smi else None, gpus_visible=n_gpu, gpus=smi)
    report["rank_names"] = time_ranking(a.names)
    print(json.dumps(report["rank_names"]), flush=True)
    counts = [c for c in (1, 2, 4, 8) if c <= n_gpu]
    d = tempfile.mkdtemp(prefix="time_multi_gpu_")
    try:
        inputs = {}
        ref = synth.random_reference(50000000, seed=41, n_contigs=8)
        write_fasta(os.path.join(d, "ref50.fa"), ref)
        write_reads(os.path.join(d, "long.fa"), ref, a.long_reads, 10000, False, seed=42, indel_rate=0.0001)
        inputs["c4_long_split"] = dict(args=["--reference", os.path.join(d, "ref50.fa"), "--queries", os.path.join(d, "long.fa"),
                                             "--split-queries-past-size", "1000"], outs=["sam"],
                                       shape="50 Mbp reference in 8 contigs, %d x 10 kbp FASTA reads (1%% substitutions, 0.01%%/base indels) split past 1000" % a.long_reads)
        ref = synth.random_reference(250000000, seed=43, n_contigs=50, repeat_fraction=0.05)
        write_fasta(os.path.join(d, "ref250.fa"), ref)
        write_reads(os.path.join(d, "short.fq"), ref, a.short_reads, 150, True, seed=44, indel_rate=0.001)
        del ref
        inputs["c3_short_vcf"] = dict(args=["--reference", os.path.join(d, "ref250.fa"), "--queries", os.path.join(d, "short.fq")], outs=["sam", "vcf", "mut"],
                                      shape="250 Mbp reference in 50 contigs with 5%% repeats, %d x 150 bp FASTQ reads (1%% substitutions, 0.1%%/base indels)" % a.short_reads)
        report["commands"] = {}
        for key, inp in inputs.items():
            runs = []
            for c in counts:
                runs.append(run_command(d, inp["args"], inp["outs"], list(range(c))))
                print(json.dumps({key: runs[-1]}), flush=True)
            ok = [r for r in runs if "sha256" in r]
            report["commands"][key] = dict(shape=inp["shape"], argv="python -m mapper_b200 " + " ".join(os.path.basename(x) if os.sep in x else x for x in inp["args"]),
                                           input_bytes=sum(os.path.getsize(x) for x in inp["args"] if os.sep in x), runs=runs,
                                           outputs_identical_across_device_counts=bool(ok) and all(r["sha256"] == ok[0]["sha256"] for r in ok))
    finally:
        shutil.rmtree(d)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
