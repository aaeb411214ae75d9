#!/usr/bin/env python3
"""Benchmark of the X-Mapper aligner stage on B200 (BASELINE.json: aligned reads/sec + DP GCUPS; CPU path beside it).

A step = one pass of the hot path (seed lookup -> candidate windows -> scoring/traceback -> result arrays) over one batch of synthetic reads.
  N = 1  : BASELINE.json configs[1] - 5 Mbp random reference, 1 M simulated 150 bp single-end reads with 1 % substitutions + small indels.
  N > 1  : BASELINE.json configs[3] - 250 Mbp reference in 50 contigs with 2-4-copy repeat families, 20 M / 8 = 2.5 M reads per GPU per step
           (reads sharded, index replicated: weak scaling), the per-position count planes (4 GB per GPU) and the sparse variant table that feed
           --out-vcf / --out-mutations reset at the start of every step and reduced over all ranks INSIDE the timed step by the library's
           own NCCL communicator (xm_counts_reduce: ncclAllReduce of the planes, all-gather + reduce-by-key of the variant entries).
  --workload c1|c3 forces either at any N (c3 at N=1 runs the same step with a one-rank "reduce" = the local table reduce only).

  python bench.py --gpus 1 --steps 3 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
  python bench.py --impl reference ...        # the reference algorithm's CPU restatement on the host cores
  python bench.py ... --dump-outputs DIR      # also write the last timed step's results (seeded sample, float64 .npy) to compare builds

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "aligned reads/sec"
UNIT = "reads/s"
DUMP_LIMIT = 64 << 20   # bytes of .npy data --dump-outputs writes at most
DUMP_SEED = 12345


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "c1", "c3"])
    ap.add_argument("--reads", type=int, default=0, help="reads per step per GPU (default: 1,000,000 for c1; 2,500,000 for c3)")
    ap.add_argument("--ref-bases", type=int, default=0)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--paired", action="store_true")
    ap.add_argument("--counts", action="store_true", help="accumulate the count planes / variant table (always on for c3)")
    ap.add_argument("--cpu-sample", type=int, default=1000000, help="reads in the cpu_baseline sample (about 30 core-seconds of the oracle)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (float64, a fixed seeded sample, at most 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.workload == "auto":
        a.workload = "c1" if world == 1 else "c3"
    if a.workload == "c3":
        a.counts = True
        a.reads = a.reads or 2500000
        a.ref_bases = a.ref_bases or 250000000
    else:
        a.reads = a.reads or 1000000
        a.ref_bases = a.ref_bases or 5000000
    return a


def workload_name(a):
    if a.workload == "c3":
        return ("synthetic %.3g Mbp reference in 50 contigs with 5%% of sequence in 2-4-copy repeat families, %s simulated %d bp %s reads/step/GPU, 1%% substitutions "
                "+ 0.1%%/base indels, count planes + variant table reduced over the ranks every step (BASELINE.json configs[3])") % (
            a.ref_bases / 1e6, "{:,}".format(a.reads), a.read_len, "paired-end 2x" if a.paired else "single-end")
    return "synthetic %.3g Mbp reference, %s simulated %d bp %s reads/step/GPU, 1%% substitutions + 0.1%%/base indels (BASELINE.json configs[%d])" % (
        a.ref_bases / 1e6, "{:,}".format(a.reads), a.read_len, "paired-end 2x" if a.paired else "single-end", 2 if a.paired else 1)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.5)

    def summary(self):
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max(int(s[1]) for s in self.samples if s[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) > 2 + i and s[2 + i].lower().startswith("active")})
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx, reasons=reasons, samples=len(self.samples))


def make_inputs(a, seed_offset):
    from mapper_b200 import synth
    if a.workload == "c3":
        ref = synth.random_reference(a.ref_bases, seed=4, n_contigs=50, repeat_fraction=0.05, repeat_copies=(2, 4), repeat_len=(1000, 5000))
        ref = sorted(ref, key=lambda c: -len(c[1]))   # Mapper.sortAndComplementReference: longest contig first (stable)
    else:
        ref = synth.random_reference(a.ref_bases, seed=1)
    parts, chunk = [], 500000
    for k, lo in enumerate(range(0, a.reads, chunk)):   # in chunks: the vectorised simulator holds n x (L + 16) int64 indices
        n = min(chunk, a.reads - lo)
        parts.append(synth.simulate_reads_fast(ref, n, a.read_len, seed=(5 if a.workload == "c3" else 2) + 1000 * seed_offset + 17 * k, paired=a.paired,
                                               inner_mean=300.0, inner_sd=30.0, per_penalty=50.0))
    if len(parts) == 1:
        return ref, parts[0]
    batch = {}
    words = 0
    offs = []
    for p in parts:
        offs.append(p["seq_word_off"][:-1] + words)
        words += int(p["seq_word_off"][-1])
    batch["seq_word_off"] = np.concatenate(offs + [np.array([words], dtype=np.int64)])
    for k in ("packed", "seq_len", "n_seqs", "expected_inner", "per_penalty"):
        batch[k] = np.concatenate([p[k] for p in parts])
    return ref, batch


def cpu_arm(a, ref, batch, n_reads, threads):
    """The reference's algorithm on the host cores: the oracle port (oracle/, C++ restatement of the Java aligner).
    bench.py is allowed to execute oracle/ here and only here (cpu_baseline / --impl reference)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import xm_oracle as xo
    from mapper_b200 import synth
    t0 = time.time()
    db = xo.Oracle([(n, synth.codes_to_text(s)) for n, s in ref], sort_by_length=True, threads=threads, dup=dict(min_copies=2, window=1000))
    db.build_through(a.read_len)
    db.detect_duplications()
    t_index = time.time() - t0
    n_mates = 2 if a.paired else 1
    ns = n_reads * n_mates
    sub = dict(packed=batch["packed"][:batch["seq_word_off"][ns]], seq_word_off=batch["seq_word_off"][:ns + 1], seq_len=batch["seq_len"][:ns],
               n_seqs=batch["n_seqs"][:n_reads], expected_inner=batch["expected_inner"][:n_reads], per_penalty=batch["per_penalty"][:n_reads])
    sub = {k: np.ascontiguousarray(v) for k, v in sub.items()}

    def run():
        t = time.time()
        r = db.align_batch(synth.DEFAULT_PARAMS, sub, threads=threads)
        return time.time() - t, r
    return run, t_index


class DevArray:
    """A raw device pointer as a __cuda_array_interface__ object (torch.as_tensor wraps it without a copy)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1

    if a.impl == "reference":
        # the reference arm: rank 0 alone runs and prints; other ranks exit 0 without work
        if rank != 0:
            return 0
        ref, batch = make_inputs(a, 0)
        n_sample = min(a.reads, a.cpu_sample)
        run, t_index = cpu_arm(a, ref, batch, n_sample, cores)
        for _ in range(max(0, min(a.warmup, 1))):
            run()
        times = []
        for _ in range(a.steps):
            dt, r = run()
            times.append(dt)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, r)
        total = sum(times)
        value = n_sample * a.steps / total
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=a.warmup, ms_per_step=1000.0 * total / a.steps,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic", impl="reference",
                    config=dict(workload=workload_name(a), sample="%d reads per step (bounded sample of the workload)" % n_sample),
                    cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="port",
                                      sample="%d reads/step x %d steps; C++ restatement of mathjeff/Mapper @ ae7f346a (the Java reference cannot be built here: no JVM), %d threads" % (n_sample, a.steps, cores)),
                    e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), index_build_s=t_index)
        _emit(line)
        return 0

    import torch
    import torch.distributed as dist
    from mapper_b200 import capi, synth
    if not torch.cuda.is_available():
        print("bench.py: no CUDA device; the product has no CPU path", file=sys.stderr)
        return 2
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ref, batch = make_inputs(a, rank)
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=local_rank)
    t0 = time.time()
    g.set_reference([synth.pack_contig(s) for _, s in ref], [len(s) for _, s in ref])
    g.build_index(a.read_len)  # on the device
    t_index_only = time.time() - t0
    g.build_duplications(-1, -1, 2, 1000)
    t_index = time.time() - t0
    comm_nranks = 0
    if a.counts:
        g.counts_enable(0.1)
        if world > 1:
            # xm_comm_init / xm_counts_reduce: torch.distributed only carries the 128-byte NCCL id from rank 0 to the others.
            # The first reduce runs here, on planes that are still all zero, so that NCCL's channel setup is not in the timed one.
            uid = torch.tensor(list(g.comm_unique_id() if rank == 0 else bytes(128)), dtype=torch.uint8, device="cuda")
            dist.broadcast(uid, 0)
            g.comm_init(world, rank, bytes(uid.cpu().tolist()))
            g.counts_reduce()
            comm_nranks = world
    peaks_issue = g.measure_peaks()
    mi, mb = g.index_info()
    index_bytes = 0
    for n in range(mb + 1):
        cap, npos = g.index_length_size(n)
        index_bytes += 8 * cap + 4 * npos

    # pinned host copies (e2e leg) and device-resident copies (kernel leg)
    keys = ["packed", "seq_word_off", "seq_len", "n_seqs", "expected_inner", "per_penalty"]
    pinned, dev = {}, {}
    for k in keys:
        arr = batch[k]
        view = arr.view(np.int16) if arr.dtype == np.uint16 else arr
        t = torch.from_numpy(view.copy()).pin_memory()
        pinned[k] = t.numpy().view(arr.dtype)
        dev[k] = t.cuda(non_blocking=False)
    host_batch = {k: pinned[k] for k in keys}
    nq = len(batch["n_seqs"])
    n_words = int(batch["seq_word_off"][-1])
    reduce_every_step = a.counts and a.workload == "c3"
    nccl_ms = [0.0, 0.0, 0]   # sums over the steps: device ms of the plane all-reduce, ms of the variant-table exchange, calls
    plane_ptr, plane_ints = g.counts_device_ptr() if a.counts else (0, 0)

    def planes_tensor():
        return torch.as_tensor(DevArray(plane_ptr, plane_ints, "<i4"), device="cuda")

    def begin_step():
        """A step is a whole run: planes and variant table start from zero (device memset of the planes); returns its time in s."""
        if not reduce_every_step:
            return 0.0
        torch.cuda.synchronize()
        t = time.time()
        g.counts_enable(0.1)
        torch.cuda.synchronize()
        return time.time() - t

    def end_step():
        """The exchange step of the path: returns its wall time in s (xm_counts_reduce blocks until the collective has finished)."""
        if not reduce_every_step:
            return 0.0
        torch.cuda.synchronize()
        t = time.time()
        if world > 1:
            g.counts_reduce()
            pm, vm = g.counts_reduce_times()
            nccl_ms[0] += pm; nccl_ms[1] += vm; nccl_ms[2] += 1
        else:
            g.variants_count()     # one rank: the local sort + reduce-by-key of the variant records is all that is left of the exchange
        return time.time() - t

    def step_device():
        tb = begin_step()
        r = g.align_batch_device(nq, dev["packed"].data_ptr(), n_words, dev["seq_word_off"].data_ptr(), dev["seq_len"].data_ptr(), dev["n_seqs"].data_ptr(),
                                 dev["expected_inner"].data_ptr(), dev["per_penalty"].data_ptr(), a.read_len)
        return r, tb + end_step()

    def step_host():
        tb = begin_step()
        r = g.align_batch(host_batch, copy=False)  # results stay in the library's pinned slab (zero-copy views)
        return r, tb + end_step()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        r, _ = step_device()
    bad = int((r["q_status"] != 0).sum())
    # the same step on ONE GPU of this box while the others idle (rank 0 alone, no collective): what the N-GPU number is to be held against,
    # since the driver's N=1 run measures configs[1] and this run configs[3]
    solo = None
    if world > 1 and reduce_every_step:
        barrier()
        if rank == 0:
            ns = 0
            ex = 0.0
            k = min(a.steps, 3)
            for _ in range(k):
                tb = begin_step()
                rs = g.align_batch_device(nq, dev["packed"].data_ptr(), n_words, dev["seq_word_off"].data_ptr(), dev["seq_len"].data_ptr(), dev["n_seqs"].data_ptr(),
                                          dev["expected_inner"].data_ptr(), dev["per_penalty"].data_ptr(), a.read_len)
                torch.cuda.synchronize()
                t = time.time()
                g.variants_count()
                ex += tb + time.time() - t
                ns += int(rs["stats"][capi.STAT["kernel_ns"]])
            solo = dict(value=nq * k / (ns / 1e9 + ex), unit=UNIT, ms_per_step=1000.0 * (ns / 1e9 + ex) / k, steps=k,
                        note="rank 0 alone on the same workload, the other GPUs idle, no collective (local reduce of the variant records only)")
        barrier()
    # ---- timed: kernel leg (inputs resident in HBM), device time from CUDA events inside the library + the exchange step ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    t0 = time.time()
    dev_ns = 0
    easy_ns_sum = full_ns_sum = 0
    launches = 0
    reduce_s = 0.0
    stats = None
    for _ in range(a.steps):
        r, tr = step_device()
        reduce_s += tr
        dev_ns += int(r["stats"][capi.STAT["kernel_ns"]])
        easy_ns_sum += int(r["stats"][capi.STAT["easy_ns"]])
        full_ns_sum += int(r["stats"][capi.STAT["tier0_ns"]])
        launches += int(r["stats"][capi.STAT["launches"]])
        stats = r["stats"]
    barrier()
    wall_dev = time.time() - t0
    if a.dump_outputs and rank == 0:
        # before any other step runs: the count planes and the variant table are still those of the last timed step
        extra = {}
        if a.counts:
            rng = np.random.default_rng(DUMP_SEED)
            pidx = np.unique(rng.integers(0, plane_ints, size=min(plane_ints, 1 << 20)))
            extra["count_planes_index"] = pidx
            extra["count_planes"] = planes_tensor()[torch.from_numpy(pidx).cuda()].cpu().numpy()
            var = g.variants_fetch()
            vidx = np.sort(rng.choice(len(var["count"]), size=min(len(var["count"]), 1 << 16), replace=False))
            extra["variants_index"] = vidx
            for k in ("gpos", "region", "dir", "ins", "allele", "count", "ex_gid", "ex_rev", "ex_index"):
                extra["variants_" + k] = var[k][vidx]
        dump_outputs(a.dump_outputs, r, extra)
    # reduced planes against the one-GPU planes, size-independent: the all-reduced checksum equals the sum of the ranks' local checksums
    # of the same step, and every rank holds the same reduced variant table
    reduce_check = None
    if reduce_every_step and world > 1:
        begin_step()
        g.align_batch_device(nq, dev["packed"].data_ptr(), n_words, dev["seq_word_off"].data_ptr(), dev["seq_len"].data_ptr(), dev["n_seqs"].data_ptr(),
                             dev["expected_inner"].data_ptr(), dev["per_penalty"].data_ptr(), a.read_len)
        local = planes_tensor().sum(dtype=torch.int64)
        n_local = torch.tensor([g.variants_count()], dtype=torch.int64, device="cuda")
        g.counts_reduce()
        total = planes_tensor().sum(dtype=torch.int64)
        n_total = torch.tensor([g.variants_count()], dtype=torch.int64, device="cuda")
        want = local.clone()
        dist.all_reduce(want)
        lo, hi = n_total.clone(), n_total.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_local, op=dist.ReduceOp.MAX)
        reduce_check = dict(plane_checksum_matches=bool(int(want) == int(total)), plane_checksum=int(total), variant_entries=int(hi),
                            same_table_size_on_every_rank=bool(int(lo) == int(hi)), merged_not_smaller_than_any_shard=bool(int(hi) >= int(n_local)))
    # ---- timed: end to end through the C ABI with host buffers (H2D + kernels + D2H + result assembly + the exchange step) ----
    keep = [step_host() for _ in range(3)]  # untimed warm-up of the host path: the staging buffers of all three batch slots and the pinned result slabs
    del keep
    barrier()
    t0 = time.time()
    h2d = d2h = 0
    for _ in range(a.steps):
        r2, _ = step_host()
        bad_e2e = int(np.count_nonzero(r2["q_status"]))  # read the step's result on the host
        h2d = int(r2["stats"][capi.STAT["h2d_bytes"]])
        d2h = int(r2["stats"][capi.STAT["d2h_bytes"]])
    barrier()
    wall_e2e = time.time() - t0
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # max over ranks
    tvals = torch.tensor([dev_ns / 1e9 + reduce_s, wall_dev, wall_e2e, reduce_s, dev_ns / 1e9], dtype=torch.float64, device="cuda")
    tmin = tvals.clone()
    if world > 1:
        dist.all_reduce(tvals, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
    t_dev, t_wall_dev, t_e2e, t_reduce, t_align = [float(x) for x in tvals.tolist()]
    total_reads = nq * a.steps * world
    value = total_reads / t_dev
    e2e_value = total_reads / t_e2e

    if rank == 0:
        aligned = int((np.diff(r["comp_choice_off"])[r["q_comp_off"][:-1]] > 0).sum())
        S = capi.STAT
        clocks = sampler.summary()
        # Two align kernels per step: the first pass over every read (xm_align_kernel<true>) and the full aligner over the reads
        # it handed on (xm_align_kernel<false>).  Algorithmic bytes per launch (SURVEY.md §8d): 8 B per bucket probe, 4 B position +
        # 19 B flank window per hit, ceil(L/2) B of packed read per query, ceil(L/2) B of reference per ungapped score.
        half = (a.read_len + 1) // 2
        n_mates = 2 if a.paired else 1
        probes, hits, straight = int(stats[S["probes"]]), int(stats[S["hits"]]), int(stats[S["straight"]])
        e_probes, e_hits, e_straight = int(stats[S["easy_probes"]]), int(stats[S["easy_hits"]]), int(stats[S["easy_straight"]])
        n_easy_in, n_easy_done = int(stats[S["easy"]]), int(stats[S["easy_done"]])
        n_full_in = int(stats[S["tier0"]])
        bytes_easy = 8 * e_probes + 23 * e_hits + half * n_mates * n_easy_in + half * e_straight
        bytes_full = 8 * (probes - e_probes) + 23 * (hits - e_hits) + half * n_mates * n_full_in + half * (straight - e_straight)
        ms_easy = easy_ns_sum / 1e6 / a.steps  # average launch duration over the timed steps (CUDA events on the library stream)
        ms_full = full_ns_sum / 1e6 / a.steps
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        # ncu counters of the two kernels (one capture of this command, summarised under profiles/): only quoted for the workload they were taken on
        prof = {}
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", "r2_kernel_counters.json")))
            if t["workload"] == dict(reads=a.reads, read_len=a.read_len, paired=bool(a.paired), ref_bases=a.ref_bases):
                prof = t
        except Exception:
            pass
        dom_full = ms_full >= ms_easy
        dom_key = "full" if dom_full else "first_pass"
        dom_bytes, dom_ms = (bytes_full, ms_full) if dom_full else (bytes_easy, ms_easy)
        dom_name = "xm_align_kernel<false> (full aligner over the reads the first pass handed on)" if dom_full else "xm_align_kernel<true> (first pass over every read)"
        hbm_achieved = dom_bytes / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else None
        pk = prof.get(dom_key) or {}
        # The bound that binds is instruction issue (SURVEY.md §8d: pyramid build and gapped search are issue-bound; the index gathers move
        # < 0.1 % of the HBM roofline).  achieved = warp-instructions of one launch (ncu smsp__inst_executed.sum of the same command) / the
        # launch duration measured live; peak = the dispatch ceiling measured live by xm_measure_peaks (FFMA chains on every SM).
        issue_peak = peaks_issue["alu"]
        warp_inst = pk.get("warp_instructions")
        issue_achieved = (warp_inst / (dom_ms / 1e3)) if (warp_inst and dom_ms > 0) else None
        lanes = pk.get("active_lanes_per_instruction")
        roof = dict(bound="issue", kernel=dom_name, achieved=(issue_achieved / 1e9 if issue_achieved else None), peak=issue_peak / 1e9, unit="G warp-instructions/s",
                    frac=(issue_achieved / issue_peak if issue_achieved else None),
                    peak_source="measured live: xm_measure_peaks (independent FFMA chains on every SM = one warp-instruction per scheduler per clock, CUDA events); INT32 IMAD %.0f G/s, FP64 DADD %.0f G/s" % (peaks_issue["int32"] / 1e9, peaks_issue["fp64"] / 1e9),
                    achieved_source=(prof.get("source") if warp_inst else "no ncu capture for this workload: issue rate not quoted"),
                    kernel_ms_per_launch=dom_ms,
                    useful_thread_instruction_fraction=((issue_achieved / issue_peak) * (pk["useful_lanes_per_instruction"] / 32.0) if (issue_achieved and pk.get("useful_lanes_per_instruction")) else None),
                    lanes_note=("%.1f of 32 lanes active per instruction; the per-query control code is warp-uniform (every lane repeats the same scalar), only the inner loops (pyramid rows, hit verification, ungapped scores, table fills) give the lanes distinct work" % lanes if lanes else None),
                    traffic=((pk["dram_bytes_read"] + pk["dram_bytes_write"]) if pk.get("dram_bytes_read") is not None else None),
                    hbm=dict(bound="hbm", achieved=hbm_achieved, peak=peak, unit="GB/s", frac=(hbm_achieved / peak) if hbm_achieved else None,
                             algorithmic_bytes_per_launch=dom_bytes, peak_source=peak_src,
                             note="seed-lookup gathers + flank windows + packed reads + reference per ungapped score (SURVEY.md §8d); reported for completeness, it does not bind"),
                    other_kernel=dict(name="xm_align_kernel<true> (first pass)" if dom_full else "xm_align_kernel<false>",
                                      algorithmic_bytes_per_launch=bytes_easy if dom_full else bytes_full, kernel_ms_per_launch=ms_easy if dom_full else ms_full,
                                      issue_frac=((prof.get("first_pass" if dom_full else "full") or {}).get("warp_instructions", 0) / ((ms_easy if dom_full else ms_full) / 1e3) / issue_peak
                                                  if (prof.get("first_pass" if dom_full else "full") and (ms_easy if dom_full else ms_full) > 0) else None)))
        # DP: GCUPS over PathAligner TIME (SM clock ticks spent inside path_align summed over warps / resident warps / SM clock), against the
        # FP64 pipe: one lattice cell = ~12 FP64 min/add instructions (SURVEY.md §8d) -> peak cell rate = measured DADD rate x 32 lanes / 12
        cells, explored = int(stats[S["path_cells"]]), int(stats[S["path_steps"]])
        sm_hz = (clocks["sm_mhz"] or 1965) * 1e6
        resident_warps = peaks_issue["sm_count"] * 64
        t_path = float(stats[S["cyc_path"]]) / resident_warps / sm_hz if resident_warps else 0.0
        cell_peak = peaks_issue["fp64"] * 32 / 12.0
        gcups = dict(value=(cells / t_path / 1e9) if t_path > 0 else None, unit="GCUPS", cells_per_step=cells, cells_explored_per_step=explored,
                     explored_gcups=(explored / t_path / 1e9) if t_path > 0 else None, path_aligner_calls=int(stats[S["path_calls"]]),
                     path_aligner_ms_per_step=1000.0 * t_path, whole_step_gcups=cells / (t_dev / a.steps) / 1e9,
                     peak_gcups=cell_peak / 1e9, frac_of_fp64_peak=((explored / t_path) / cell_peak) if t_path > 0 else None,
                     note="cells = A x B of every PathAligner lattice (SURVEY.md §8d); explored = nodes popped by the best-first search; time = SM ticks inside path_align "
                          "summed over warps / %d resident warps / %.0f MHz; peak = measured FP64 DADD rate x 32 lanes / 12 FP64 ops per cell; frac uses the EXPLORED cells" % (resident_warps, sm_hz / 1e6))
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup, ms_per_step=1000.0 * t_dev / a.steps,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                    config=dict(workload=workload_name(a), reads_per_step_per_gpu=nq, parallelism="reads sharded x%d, index replicated" % world,
                                l2="inputs larger than L2: index %.0f MB + packed reads %.0f MB + per-warp workspaces (GBs) per step vs 126 MB L2" % (index_bytes / 1e6, batch["packed"].nbytes / 1e6),
                                timing="value: CUDA-event device time of all kernels of a step (library stream)%s, max over ranks; e2e: wall clock around xm_align_batch with pinned host buffers%s" % (
                                    (" + the exchange step (xm_counts_reduce, wall clock around the blocking call)", " + the exchange step") if reduce_every_step else ("", ""))),
                    e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, ms_per_step=1000.0 * t_e2e / a.steps),
                    gpu_launches=launches, roofline=roof, gcups=gcups, clocks=clocks,
                    aligned_fraction=aligned / nq, failed_queries=bad, index_build_s=t_index, index_build_device_s=t_index_only,
                    first_pass=dict(queries=n_easy_in, completed=n_easy_done, ms=ms_easy),
                    full_pass=dict(tiers=[int(stats[S["tier0"]]), int(stats[S["tier1"]]), int(stats[S["tier2"]])],
                                   ms=[float(stats[S["tier%d_ns" % t]]) / 1e6 for t in range(3)]),
                    wall_ms_per_step_device_api=1000.0 * t_wall_dev / a.steps,
                    exchange=(dict(collective="xm_counts_reduce: ncclAllReduce(int32 sum) of the count planes + all-gather / reduce-by-key of the variant table, in the library (libnccl loaded at run time)",
                                   comm_nranks=comm_nranks, plane_bytes_per_gpu=plane_ints * 4, exchange_ms_per_step=1000.0 * t_reduce / a.steps,
                                   plane_allreduce_ms=(nccl_ms[0] / nccl_ms[2]) if nccl_ms[2] else None, variant_exchange_ms=(nccl_ms[1] / nccl_ms[2]) if nccl_ms[2] else None,
                                   plane_allreduce_bus_gbs=((plane_ints * 4) * 2.0 * (world - 1) / world / (nccl_ms[0] / nccl_ms[2] / 1e3) / 1e9) if (nccl_ms[2] and nccl_ms[0] > 0) else None,
                                   note="exchange_ms_per_step = reset of the planes + ncclAllReduce of the planes (device time: plane_allreduce_ms, rank 0) + exchange and merge of the variant table (variant_exchange_ms), wall clock, max over ranks",
                                   align_ms_per_step_max_rank=1000.0 * t_align / a.steps, align_ms_per_step_min_rank=1000.0 * float(tmin[4]) / a.steps, check=reduce_check)
                              if reduce_every_step else None),
                    single_gpu_same_workload=solo,
                    allreduce_ms=(1000.0 * t_reduce / a.steps) if reduce_every_step else None)
        if not a.no_cpu_baseline and world == 1:
            n_sample = min(a.reads, a.cpu_sample)
            run, _ = cpu_arm(a, ref, batch, n_sample, cores)
            dt, rc = run()
            # the oracle's results for the sample double as a parity check of this run's device results (bit for bit, doubles included)
            line["parity"] = dict(reads=n_sample, identical_to_oracle=bool(same_prefix(rc, r, n_sample)),
                                  note="all eleven result arrays of the first `reads` queries of rank 0 compared with the CPU oracle")
            line["cpu_baseline"] = dict(value=n_sample / dt, unit=UNIT, cores=cores, kind="port",
                                        sample="%d reads of the same workload, %.1f s on %d threads; C++ restatement of mathjeff/Mapper @ ae7f346a (no JVM available)" % (n_sample, dt, cores))
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    g.close()
    return 0


def same_prefix(want, got, n):
    """True if the result arrays of the first n queries of `got` equal `want` (a result for exactly those n queries) bit for bit."""
    c = int(got["q_comp_off"][n]); ch = int(got["comp_choice_off"][c]); sa = int(got["choice_sa_off"][ch]); bl = int(got["sa_block_off"][sa])
    sizes = dict(q_comp_off=n + 1, comp_choice_off=c + 1, choice_sa_off=ch + 1, sa_block_off=sa + 1, choice_f64=4 * ch, sa_f64=2 * sa,
                 choice_inner=ch, sa_contig=sa, blocks=4 * bl, q_status=n, sa_reversed=sa)
    for k, m in sizes.items():
        x, y = np.ascontiguousarray(want[k]), np.ascontiguousarray(got[k][:m])
        if x.dtype != y.dtype:
            x = x.astype(y.dtype)
        if len(x) != m or x.tobytes() != y.tobytes():
            return False
    return True


def _children(off, rows):
    """Rows `rows` (ascending) of the CSR offsets `off`: (indices of their children, the children's offsets rebased to the selection)."""
    lens = off[rows + 1] - off[rows]
    new_off = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum(lens, out=new_off[1:])
    return np.repeat(off[rows] - new_off[:-1], lens) + np.arange(new_off[-1]), new_off


def select_queries(r, qs):
    """The result arrays of the queries qs (ascending indices), laid out as the library returns them for a batch of those queries alone."""
    comps, q_off = _children(r["q_comp_off"], qs)
    choices, c_off = _children(r["comp_choice_off"], comps)
    sas, ch_off = _children(r["choice_sa_off"], choices)
    blocks, sa_off = _children(r["sa_block_off"], sas)
    return dict(q_comp_off=q_off, comp_choice_off=c_off, choice_sa_off=ch_off, sa_block_off=sa_off,
                choice_f64=np.asarray(r["choice_f64"]).reshape(-1, 4)[choices].ravel(), sa_f64=np.asarray(r["sa_f64"]).reshape(-1, 2)[sas].ravel(),
                choice_inner=r["choice_inner"][choices], sa_contig=r["sa_contig"][sas], blocks=np.asarray(r["blocks"]).reshape(-1, 4)[blocks].ravel(),
                q_status=r["q_status"][qs], sa_reversed=r["sa_reversed"][sas])


def dump_outputs(path, r, extra=None):
    """Writes what a caller of the timed path received in the last step as path/<name>.npy, every array as float64 (the integers
    involved are below 2^53, so exact): the result arrays of a fixed, seeded sample of the queries (query_index.npy lists them) and
    `extra`, arrays already sampled by the caller.  The sample is drawn with a fixed seed: 2^17 queries (all of a smaller batch),
    halved while the files would exceed DUMP_LIMIT."""
    out = {k: np.asarray(v, dtype=np.float64) for k, v in (extra or {}).items()}
    size = lambda arrays: sum(128 + v.nbytes for v in arrays.values())   # a .npy file of a 1-D array = 128-byte header + data
    room = DUMP_LIMIT - size(out)
    nq = len(r["q_status"])
    k = min(nq, 1 << 17)
    while True:
        qs = np.sort(np.random.default_rng(DUMP_SEED).choice(nq, size=k, replace=False))
        sel = {n: np.asarray(v, dtype=np.float64) for n, v in select_queries(r, qs).items()}
        sel["query_index"] = qs.astype(np.float64)
        if size(sel) <= room:
            break
        k //= 2
    out.update(sel)
    os.makedirs(path, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(path, name + ".npy"), v)


def _emit(line):
    """The contract is ONE JSON line on stdout: libraries (NCCL's version banner, torchrun) write to fd 1 as well, so fd 1 is
    pointed at stderr for the whole run and the line goes to the saved descriptor."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)

if __name__ == "__main__":
    sys.exit(main())
