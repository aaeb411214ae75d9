"""Times the VCF and mutations bodies formatted by the library (xm_format_vcf / xm_format_mutations) on a whole reference, in ranges
of 2^22 positions, contigs in name order as VcfWriter / MutationsWriter visit them:
  - configs[2] shape: 5 Mbp reference, 2 M paired reads (1 M pairs of 150 bp);
  - configs[3] shape, one GPU's share: 250 Mbp in 50 contigs, 2.5 M reads of 150 bp.
Per body (VCF with support, VCF without support, mutations with the default filter): wall time of the calls (host clock; each call
ends with the text in host memory), kernel time of the same pass in a second, profiled pass (torch.profiler, CUDA activities: the
library's kernels and the cub scans it launches), bytes of text and text GB/s over the wall time.
At the configs[3] shape it also checks that ranged output concatenates to whole-contig output (VCF and mutations, three contigs)
and that the VCF has exactly one position line per position of nonzero depth (counted with numpy from counts_fetch / variants_fetch).
For scale it times the Python test oracle (tests/variants_oracle.py, a pure-Python restatement, not QuickVariants' Java writer) on a
100 kbp slice and checks that its body equals the library's.  Prints one JSON line with the GPU's name and power limit.

    python tools/time_format_variants.py [--shapes c2,c3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from mapper_b200 import capi, synth  # noqa: E402

RANGE = 1 << 22
JOB = 8192


def gpu_identity():
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_format_variants: no CUDA device (the library has no CPU path)")
    name = torch.cuda.get_device_name(0)
    power = None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True, timeout=60)
        power = float(out.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return name, power


def setup(ref, batch, chunk=500000):
    """A handle with the reference, the device index, duplications and counts of the batch (aligned in chunks of queries)."""
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.set_reference_from_codes([c for _, c in ref])
    g.build_index(150)
    g.build_duplications(-1, -1, 2, 1000)
    g.counts_enable(0.1)
    nq = len(batch["n_seqs"])
    seq_first = np.concatenate([[0], np.cumsum(batch["n_seqs"].astype(np.int64))])
    for q0 in range(0, nq, chunk):
        q1 = min(nq, q0 + chunk)
        s0, s1 = int(seq_first[q0]), int(seq_first[q1])
        w0, w1 = int(batch["seq_word_off"][s0]), int(batch["seq_word_off"][s1])
        sub = dict(packed=batch["packed"][w0:w1], seq_word_off=(batch["seq_word_off"][s0:s1 + 1] - w0).astype(np.int64),
                   seq_len=batch["seq_len"][s0:s1], n_seqs=batch["n_seqs"][q0:q1], expected_inner=batch["expected_inner"][q0:q1],
                   per_penalty=batch["per_penalty"][q0:q1])
        g.counts_batch_info(s0)
        g.align_batch(sub)
    return g


def upload_examples(g, batch):
    """xm_variants_set_examples straight from the packed batch (sequence gid = its index in the batch)."""
    gids = g.variants_examples()
    off, lens = batch["seq_word_off"], batch["seq_len"]
    nw = (lens[gids].astype(np.int64) + 3) // 4
    new_off = np.concatenate([[0], np.cumsum(nw)]).astype(np.int64)
    idx = np.repeat(off[gids] - new_off[:-1], nw) + np.arange(int(new_off[-1]))
    words = np.concatenate([batch["packed"][idx], np.zeros(1, np.uint16)])
    l32 = np.ascontiguousarray(lens[gids], dtype=np.int32)
    g._ok(g.L.xm_variants_set_examples(g.h, C.c_int64(len(gids)), capi._ptr(np.ascontiguousarray(gids)), capi._ptr(words), capi._ptr(new_off), capi._ptr(l32)))
    return len(gids)


def ranges(n):
    return [(a, min(n, a + RANGE)) for a in range(0, n, RANGE)]


def raw_call(g, kind, c, name, a, b, flt):
    """One format call; returns (pointer, bytes) of the text in the handle's pinned buffer."""
    text, nb = C.c_char_p(), C.c_int64()
    f = capi.to_xm_filter(flt)
    if kind == "mutations":
        g._ok(g.L.xm_format_mutations(g.h, c, name.encode(), C.c_int64(a), C.c_int64(b), C.byref(f), C.byref(text), C.byref(nb)))
    else:
        g._ok(g.L.xm_format_vcf(g.h, c, name.encode(), C.c_int64(a), C.c_int64(b), C.byref(f), 1, int(kind == "vcf_support"), C.byref(text), C.byref(nb)))
    return text, nb.value


DEFAULT = dict(minSNPTotalDepth=5, minSNPDepthFraction=0.9, minIndelTotalStartDepth=1, minIndelStartDepthFraction=0.8,
               minIndelContinuationTotalDepth=1, minIndelContinuationDepthFraction=0.7)   # MutationDetectionParameters.defaultFilter()


def whole_pass(g, ref, kind, on_text=None):
    flt = DEFAULT if kind == "mutations" else None
    total, t = 0, 0.0
    for name, c in sorted((n, i) for i, (n, _) in enumerate(ref)):
        for a, b in ranges(len(ref[c][1])):
            t0 = time.perf_counter()
            p, nb = raw_call(g, kind, c, name, a, b, flt)
            t += time.perf_counter() - t0
            total += nb
            if on_text:
                on_text(name, c, a, b, C.string_at(p, nb))
    return total, t


def kernel_seconds(g, ref, kind):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        whole_pass(g, ref, kind)
        torch.cuda.synchronize()
    us = 0.0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and ("fmt" in e.name or "Scan" in e.name or "scan" in e.name):
            us += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    return us / 1e6


def time_shape(g, ref, label):
    out = {}
    for kind in ("vcf_support", "vcf", "mutations"):
        whole_pass(g, ref, kind)   # warm-up: module load, buffer sizes
        nbytes, wall = whole_pass(g, ref, kind)
        ks = kernel_seconds(g, ref, kind)
        out[kind] = dict(bytes=nbytes, wall_s=round(wall, 4), kernel_s=round(ks, 4), text_gb_per_s_wall=round(nbytes / wall / 1e9, 3))
        print(label, kind, out[kind], flush=True)
    return out


def checks_c3(g, ref):
    # chunked == whole for three contigs
    names = sorted((n, i) for i, (n, _) in enumerate(ref))[:3]
    for name, c in names:
        n = len(ref[c][1])
        for kind in ("vcf", "mutations"):
            flt = DEFAULT if kind == "mutations" else None
            p, nb = raw_call(g, kind, c, name, 0, n, flt)
            whole = C.string_at(p, nb)
            parts = []
            for a, b in ranges(n):
                p, nb = raw_call(g, kind, c, name, a, b, flt)
                parts.append(C.string_at(p, nb))
            if b"".join(parts) != whole:
                raise SystemExit("time_format_variants: ranged %s text of %s differs from the whole-contig text" % (kind, name))
    # one VCF position line per position of nonzero depth
    t = g.variants_fetch()
    off = np.concatenate([[0], np.cumsum([len(s) for _, s in ref])])
    at = t["gpos"][(t["ins"] < 0) & (t["count"] > 0)]
    lines = {}

    def count_lines(name, c, a, b, text):
        rows = text.count(b"\n" + name.encode() + b"\t-") + int(text.startswith(name.encode() + b"\t-"))
        lines[c] = lines.get(c, 0) + text.count(b"\n") - rows
    whole_pass(g, ref, "vcf", count_lines)
    for c in range(len(ref)):
        depth = (g.counts_fetch(c).reshape(4, -1) > 0).any(axis=0)
        sel = at[(at >= off[c]) & (at < off[c + 1])] - off[c]
        depth[sel] = True
        if int(depth.sum()) != lines.get(c, 0):
            raise SystemExit("time_format_variants: contig %d has %d positions with depth but %d VCF position lines" % (c, int(depth.sum()), lines.get(c, 0)))
    return dict(chunks_equal_whole=True, vcf_lines_equal_depth_positions=True, positions_with_depth=int(sum(lines.values())))


def oracle_slice():
    """The Python oracle on a 100 kbp reference at configs[2]'s depth (60x of 150 bp reads), from the device's tables."""
    import variants_oracle as vo
    ref = synth.random_reference(100000, seed=11)
    batch = synth.simulate_reads_fast(ref, 40000, 150, seed=12, paired=False)
    g = setup(ref, batch)
    upload_examples(g, batch)
    name = ref[0][0]
    lib = g.format_vcf(0, name, 0, len(ref[0][1]))
    t = g.variants_fetch()
    t["contig"] = np.zeros(len(t["gpos"]), dtype=np.int64)
    t["pos"] = t["gpos"]
    from mapper_b200.synth import unpack_reads
    reads = [m for q in unpack_reads(batch) for m in q]
    store = vo.Store.from_device(ref, 0.1, [g.counts_fetch(0)], t,
                                 lambda gid, rev: vo.Seq("q%d" % gid + ("-rev" if rev else ""), gid, vo.COMP[reads[gid][::-1]] if rev else reads[gid]))
    t0 = time.perf_counter()
    body = vo.vcf_body(store)
    dt = time.perf_counter() - t0
    g.close()
    return dict(positions=len(ref[0][1]), python_oracle_vcf_s=round(dt, 3), bytes=len(body), equal_to_library=body == lib)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="c2,c3")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu, power = gpu_identity()
    line = dict(what="xm_format_vcf / xm_format_mutations over whole references in ranges of 2^22 positions", gpu=gpu, power_limit_w=power)
    for shape in a.shapes.split(","):
        t0 = time.perf_counter()
        if shape == "c2":
            ref = synth.random_reference(5000000, seed=1)
            batch = synth.simulate_reads_fast(ref, 2000000, 150, seed=2, paired=True, inner_mean=300.0, inner_sd=30.0, per_penalty=50.0)
        else:
            ref = synth.random_reference(250000000, seed=4, n_contigs=50, repeat_fraction=0.05, repeat_copies=(2, 4), repeat_len=(1000, 5000))
            ref = sorted(ref, key=lambda c: -len(c[1]))
            parts = [synth.simulate_reads_fast(ref, 500000, 150, seed=5 + 17 * k) for k in range(5)]
            batch = dict(seq_word_off=np.concatenate([p["seq_word_off"][:-1] + sum(int(q["seq_word_off"][-1]) for q in parts[:i]) for i, p in enumerate(parts)]
                                                     + [np.array([sum(int(q["seq_word_off"][-1]) for q in parts)], dtype=np.int64)]))
            for k in ("packed", "seq_len", "n_seqs", "expected_inner", "per_penalty"):
                batch[k] = np.concatenate([p[k] for p in parts])
        g = setup(ref, batch)
        n_ex = upload_examples(g, batch)
        res = dict(bases=sum(len(c) for _, c in ref), contigs=len(ref), sequences=int(batch["n_seqs"].astype(np.int64).sum()),
                   table_entries=g.variants_count(), examples=n_ex, setup_s=round(time.perf_counter() - t0, 1))
        res.update(time_shape(g, ref, shape))
        if shape == "c3":
            res["checks"] = checks_c3(g, ref)
        g.close()
        line[shape] = res
    line["oracle_100kbp"] = oracle_slice()
    text = json.dumps(line)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    if not line["oracle_100kbp"]["equal_to_library"]:
        raise SystemExit("time_format_variants: the oracle's VCF body of the 100 kbp slice differs from the library's")


if __name__ == "__main__":
    main()
