"""Device read parsing (xm_parse_reads) at configs[1] size, next to the alignment it feeds.

Generates from a seed, in the output directory: a 5 Mbp reference and 1 M x 150 bp single-end FASTQ reads (about 320 MB).  Reports in
one JSON document:
  - the parser's device time over the whole file (torch.profiler, CUDA kernels of the parse calls: the xm_parse_* kernels and their cub
    scans) and GB/s of text, plus its host<->device copy time;
  - the wall time of every xm_parse_reads call (64 MiB chunks, as python -m mapper_b200 hands them over);
  - the whole `python -m mapper_b200 --out-sam` run's wall time next to the summed XM_STAT_KERNEL_NS of its batches;
  - the GPU's name and power limit.
Usage: python tools/time_parse.py --out DIR/time_parse.json (the inputs are generated in DIR and removed at the end)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mapper_b200 import __main__ as cli  # noqa: E402
from mapper_b200 import capi, synth  # noqa: E402


def write_inputs(d, n_reads, read_len, seed):
    ref = synth.random_reference(5000000, seed=seed)
    cli_ref = os.path.join(d, "ref.fa")
    with open(cli_ref, "w") as f:
        for name, codes in ref:
            f.write(">%s\n" % name)
            t = synth.codes_to_text(codes)
            f.write("\n".join(t[k:k + 80] for k in range(0, len(t), 80)) + "\n")
    fq = os.path.join(d, "reads.fq")
    with open(fq, "wb") as f:
        for lo in range(0, n_reads, 250000):
            n = min(250000, n_reads - lo)
            b = synth.simulate_reads_fast(ref, n, read_len, seed=seed + 1 + lo)
            w = b["packed"].reshape(n, -1)
            codes = np.stack([w & 15, (w >> 4) & 15, (w >> 8) & 15, (w >> 12) & 15], axis=2).reshape(n, -1)[:, :read_len]
            seq = synth.LETTERS[codes]
            names = np.frombuffer(b"".join(b"@r%09d\n" % (lo + i) for i in range(n)), np.uint8).reshape(n, -1)
            nl = np.full((n, 1), ord("\n"), np.uint8)
            rec = np.concatenate([names, seq, nl, np.frombuffer(b"+\n", np.uint8)[None, :].repeat(n, 0), np.full((n, read_len), ord("I"), np.uint8), nl], axis=1)
            f.write(rec.tobytes())
    return cli_ref, fq


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON report; the inputs are generated in its directory")
    ap.add_argument("--reads", type=int, default=1000000)
    a = ap.parse_args()
    d = os.path.dirname(os.path.abspath(a.out))
    os.makedirs(d, exist_ok=True)
    ref, fq = write_inputs(d, a.reads, 150, seed=1)
    size = os.path.getsize(fq)
    import torch
    from torch.profiler import ProfilerActivity, profile
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)

    def parse_file():
        src, calls, n = cli.Source(fq, 0), [], 0
        while not src.done():
            t0 = time.perf_counter()
            arrays, k = src.take(g)
            calls.append(time.perf_counter() - t0)
            n += k
        return calls, n
    parse_file()   # warm-up: buffers, pinned staging, module load
    calls, n_records = parse_file()
    assert n_records == a.reads
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        parse_file()
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernel_us = sum(e.device_time for e in kern if "emcpy" not in e.name and "emset" not in e.name)
    copy_us = sum(e.device_time for e in kern if "emcpy" in e.name)
    names = sorted({e.name for e in kern if e.name.startswith("_Z") or "xm_parse" in e.name or "Device" in e.name})
    g.close()
    t0 = time.perf_counter()
    r = subprocess.run([sys.executable, "-m", "mapper_b200", "--reference", ref, "--queries", fq, "--out-sam", os.path.join(d, "reads.sam")],
                       cwd=ROOT, capture_output=True, text=True)
    wall = time.perf_counter() - t0
    assert r.returncode == 0, r.stderr
    summary = [ln for ln in r.stderr.splitlines() if ln.startswith("mapper_b200:")][-1]
    batches = int(summary.split(" in ")[1].split()[0])
    align_s = float(summary.split("align kernels ")[1].split()[0])
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()[0]
    out = dict(gpu=gpu, input=dict(reads=a.reads, read_len=150, fastq_bytes=size, reference_bp=5000000, chunk_bytes=cli.CHUNK_BYTES),
               parse=dict(device_kernel_s=kernel_us / 1e6, gb_per_s_of_text=size / (kernel_us / 1e6) / 1e9, copy_s=copy_us / 1e6,
                          calls=len(calls), wall_s_per_call=[round(c, 4) for c in calls], wall_s_total=sum(calls),
                          wall_gb_per_s=size / sum(calls) / 1e9, kernels_seen=names[:40]),
               command=dict(argv="python -m mapper_b200 --reference ref.fa --queries reads.fq --out-sam reads.sam", wall_s=wall, batches=batches,
                            align_kernel_s=align_s, parse_device_s_per_batch=kernel_us / 1e6 / batches, align_kernel_s_per_batch=align_s / batches,
                            parse_share_of_align=(kernel_us / 1e6) / align_s, stderr_summary=summary))
    for f in ("reads.fq", "reads.sam", "ref.fa"):
        os.remove(os.path.join(d, f))
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
