"""Device memory of a handle: everything a handle allocated is returned when it is closed, across index rebuilds that replace a bigger
set of tables by a smaller one (host builder, then the device builder), the duplication scan, the count planes and the variant table; and
a result arena that overflows is grown with what the first pass wrote kept."""
import gc
import os

import pytest

import parity
from mapper_b200 import capi, synth

pytestmark = pytest.mark.gpu
THREADS = os.cpu_count() or 4
# cudaMalloc hands out whole 2 MiB pages, and small buffers share pages the driver may keep mapped: four pages of slack.  The index
# tables the second build drops come to about 30 MB.
TOLERANCE = 4 * (2 << 20)


def free_bytes():
    import torch
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info(0)[0]


def run_sequence(ref_bases, n_reads, seed):
    ref = synth.random_reference(ref_bases, seed=seed, n_contigs=2, repeat_fraction=0.05, repeat_len=(200, 1000))
    batch = synth.simulate_reads(ref, n_reads, 150, seed=seed + 1)
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.set_reference_from_codes(ref)
    g.build_index(150, threads=THREADS)   # host-built tables of lengths up to 150, uploaded by the first align
    g.align_batch(batch)
    g.build_index(40, threads=THREADS)    # fewer tables: the upload drops those of lengths 41..150
    g.align_batch(batch)
    g.build_index(150)                    # the device builder replaces the uploaded tables
    g.build_duplications(-1, -1, 2, 1000)
    g.counts_enable(0.1)                  # count planes and the variant table
    g.align_batch(batch)
    g.close()


def test_handle_returns_its_device_memory():
    gc.collect()
    free_bytes()   # the process's own CUDA context first
    # Kernels are loaded on their first launch (lazy module loading), and the first handle raises the stack limit: a small run of the
    # same sequence first, so that the reading below already counts both.
    run_sequence(200000, 200, seed=41)
    before = free_bytes()
    run_sequence(3000000, 2000, seed=43)
    after = free_bytes()
    assert before - after <= TOLERANCE, "the handle kept %.1f MB of device memory after close()" % ((before - after) / 1e6)


def test_result_arena_overflow_rerun():
    """1 kbp reads with 1.5 % indels: about 30 alignment blocks per read against the 6 per sequence (+ 16384) a fresh handle reserves,
    so the first batch outgrows the block arena; it is grown (keeping what was written) and the affected queries run again.  The same
    batch on the grown handle fits at once: both give the same results, and the first needed more kernel launches."""
    ref = synth.random_reference(1000000, seed=51, n_contigs=2)
    batch = synth.simulate_reads(ref, 1500, 1000, seed=52, sub_rate=0.005, indel_rate=0.015)
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.set_reference_from_codes(ref)
    g.build_index(1000)
    grown = g.align_batch(batch, strict=True)
    fits = g.align_batch(batch, strict=True)
    parity.assert_same_results(fits, grown, "result arena grown during the batch")
    assert len(grown["blocks"]) // 4 > 6 * len(batch["n_seqs"]) + 16384
    launches = capi.STAT["launches"]
    assert grown["stats"][launches] > fits["stats"][launches]
    g.close()
