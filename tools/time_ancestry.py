"""Times --infer-ancestors on the configs[4] reference (BASELINE.json: "-anc" reference, 50 Mbp, 3-6-copy families): xm_infer_ancestors
end to end (host clock around the blocking call, after one warm-up call) and per stage (its XM_TRACE_SETUP line), next to the oracle's
three CPU steps on the same host (index build through 2 * minDuplicationLength, duplication detection, ancestry analysis).  Checks that
the "-anc" codes and the number of changed positions are equal, and prints one JSON line with the GPU's name and power limit.

    python tools/time_ancestry.py [--bases 50000000] [--seed 6] [--contigs 10] [--out FILE]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import xm_oracle as xo  # noqa: E402
from mapper_b200 import capi, synth  # noqa: E402


def gpu_identity():
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_ancestry: no CUDA device (the library has no CPU path)")
    name = torch.cuda.get_device_name(0)
    power = None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True, timeout=60)
        power = float(out.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return name, power


def traced_call(fn):
    """Runs fn() with the process's stderr captured (the library's XM_TRACE_SETUP lines go there); returns (result, seconds, text)."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as f:
        os.dup2(f.fileno(), 2)
        try:
            t0 = time.perf_counter()
            r = fn()
            dt = time.perf_counter() - t0
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read().decode(errors="replace")
    sys.stderr.write(text)
    return r, dt, text


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=50000000)
    ap.add_argument("--seed", type=int, default=6)
    ap.add_argument("--contigs", type=int, default=10)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = gpu_identity()
    params = synth.DEFAULT_PARAMS
    thr = params["max_error_rate"] / params["mutation"]
    ref = synth.random_reference(a.bases, seed=a.seed, n_contigs=a.contigs, repeat_fraction=0.08, repeat_copies=(3, 6))
    total = sum(len(s) for _, s in ref)
    min_dup = 1
    while (1 << min_dup) < total:
        min_dup += 1

    # the oracle, as M/Mapper.java:666-692 sets it up (tests/parity.py: inferred_ancestor_oracle), one step at a time
    t0 = time.perf_counter()
    db0 = xo.Oracle([(n, synth.codes_to_text(s)) for n, s in ref], sort_by_length=True, min_interesting=min_dup, max_short=8, threads=a.threads,
                    dup=dict(min_len=min_dup, max_len=2 * min_dup, min_copies=3, window=1))
    db0.build_through(2 * min_dup)
    t1 = time.perf_counter()
    db0.detect_duplications()
    t2 = time.perf_counter()
    anc = db0.infer_ancestors(thr)
    t3 = time.perf_counter()
    originals = [db0.contig(i)[1] for i in range(db0.num_contigs())]
    changed_oracle = sum(int((c != o).sum()) for (_, c), o in zip(anc, originals))

    g = capi.XMapper(params, device=0)
    os.environ["XM_TRACE_SETUP"] = "1"
    g.set_reference_from_codes(originals)
    g.infer_ancestors(thr, min_interesting=min_dup, max_short=8)          # warm-up: module load, first allocations
    g.set_reference_from_codes(originals)
    n_changed, seconds, trace = traced_call(lambda: g.infer_ancestors(thr, min_interesting=min_dup, max_short=8))
    m = re.search(r"infer ancestors: index ([0-9.]+) s, scan ([0-9.]+) s .*merge ([0-9.]+) s .*analysis ([0-9.]+) s .*apply ([0-9.]+) s", trace)
    stages = dict(zip(["index", "scan", "merge", "analysis", "apply"], [float(x) for x in m.groups()])) if m else None
    equal = all(np.array_equal(g.get_reference(i), c) for i, (_, c) in enumerate(anc)) and n_changed == changed_oracle
    g.close()
    line = dict(what="xm_infer_ancestors on configs[4]'s reference", bases=total, contigs=a.contigs, seed=a.seed, min_dup=min_dup,
                threshold=thr, gpu=name, power_limit_w=power, library_s=round(seconds, 4), library_stages_s=stages,
                oracle_s=dict(index=round(t1 - t0, 3), detection=round(t2 - t1, 3), analysis=round(t3 - t2, 3)), oracle_threads=a.threads,
                positions_changed=n_changed, oracle_positions_changed=changed_oracle, anc_codes_equal=bool(equal))
    text = json.dumps(line)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    if not equal:
        raise SystemExit("time_ancestry: the library's -anc reference differs from the oracle's")


if __name__ == "__main__":
    main()
