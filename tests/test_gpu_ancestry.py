"""--infer-ancestors through the library alone: xm_infer_ancestors replaces the handle's reference by its "-anc" reference (IUPAC unions
where AncestryDetector inferred a recent common ancestor, M/AncestryDetector.java:89-439); every comparison is exact, code for code,
against the oracle's AncestryDetector (oracle/xo_ancestry.h)."""
import json
import os
import re

import numpy as np
import pytest

import parity
from mapper_b200 import capi, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V = json.load(open(os.path.join(ROOT, "tests", "golden", "junit_vectors.json")))
THREADS = os.cpu_count() or 4
XM_ERR_STATE = -3


def codes_of(text):
    return np.array([synth.LETTERS.tobytes().index(c.encode()) for c in text], dtype=np.uint8)


def min_dup_len(contigs):
    total, n = sum(len(c) for c in contigs), 1
    while (1 << n) < total:   # SequenceDatabase.log2RoundUp(totalForwardSize)
        n += 1
    return n


def threshold():
    return synth.DEFAULT_PARAMS["max_error_rate"] / synth.DEFAULT_PARAMS["mutation"]


def pasted_copies(ref, seed, families, copies, unit_len=(300, 1500), divergence=0.01, inverted=False):
    """ref with extra repeat families pasted over it; inverted: every other copy is the reverse complement of the unit."""
    rng = np.random.default_rng(seed)
    contigs = [(n, s.copy()) for n, s in ref]
    for _ in range(families):
        rl = int(rng.integers(unit_len[0], unit_len[1] + 1))
        unit = synth.CODES[rng.integers(0, 4, size=rl)]
        for k in range(int(rng.integers(copies[0], copies[1] + 1))):
            seq = contigs[int(rng.integers(0, len(contigs)))][1]
            pos = int(rng.integers(0, len(seq) - rl))
            copy = unit.copy()
            nmut = rng.binomial(rl, divergence)
            if nmut:
                copy[rng.integers(0, rl, size=nmut)] = synth.CODES[rng.integers(0, 4, size=nmut)]
            if inverted and k % 2:
                copy = synth.COMP[copy[::-1]]
            seq[pos:pos + rl] = copy
    return contigs


def oracle_and_originals(ref):
    """(oracle over the "-anc" reference, changed positions, original contigs in the oracle's database order)."""
    db, changed = parity.inferred_ancestor_oracle(ref, synth.DEFAULT_PARAMS, threads=THREADS)
    by_name = dict(ref)
    originals = [by_name[db.contig(i)[0][:-len("-anc")]] for i in range(db.num_contigs())]
    return db, changed, originals


def infer_like_mapper(g, originals):
    """M/Mapper.java:675-681: minInterestingSize = minDuplicationLength, 8 short matches, MaxErrorRate / MutationPenalty."""
    return g.infer_ancestors(threshold(), min_interesting=min_dup_len(originals), max_short=8)


def assert_same_anc(g, db, changed, n_changed, what):
    for i in range(db.num_contigs()):
        want = db.contig(i)[1]
        got = g.get_reference(i)
        if not np.array_equal(want, got):
            bad = np.flatnonzero(want != got)
            raise AssertionError("%s: contig %d differs at %d positions, first %d: oracle %s, library %s" % (
                what, i, len(bad), bad[0], synth.codes_to_text(want[bad[0]:bad[0] + 1]), synth.codes_to_text(got[bad[0]:bad[0] + 1])))
    assert n_changed == changed, what


def run_parity(ref, what, monkeypatch=None, env=None):
    db, changed, originals = oracle_and_originals(ref)
    if env:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.set_reference_from_codes(originals)
    n_changed = infer_like_mapper(g, originals)
    assert_same_anc(g, db, changed, n_changed, what)
    g.close()
    return changed


@pytest.mark.parametrize("case", V["ancestry_cases"], ids=[c["name"] for c in V["ancestry_cases"]])
def test_junit_ancestry_strings(case):
    """The eight strings of T/AncestryDetector_Test.java:10-91: default index parameters, verifyNoDuplicateAnalyses on."""
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.set_reference_from_codes([codes_of(case["reference"])])
    n = g.infer_ancestors(case["threshold"], verify=True)
    got = synth.codes_to_text(g.get_reference(0))
    assert got == case["expected"]
    assert n == sum(a != b for a, b in zip(case["reference"], case["expected"]))
    g.close()


@pytest.mark.parametrize("n_bases,n_contigs,seed", [(500000, 4, 21), (1000000, 7, 22), (2000000, 10, 23)])
def test_random_references_with_repeat_families(n_bases, n_contigs, seed):
    ref = synth.random_reference(n_bases, seed=seed, n_contigs=n_contigs, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 5000))
    assert run_parity(ref, "%d bp, %d contigs, seed %d" % (n_bases, n_contigs, seed)) > 100


def test_inverted_copies():
    base = synth.random_reference(1000000, seed=31, n_contigs=5, repeat_fraction=0.03, repeat_copies=(3, 6), repeat_len=(1000, 3000))
    ref = pasted_copies(base, seed=32, families=8, copies=(3, 6), inverted=True)
    assert run_parity(ref, "inverted copies") > 100


def test_family_larger_than_a_warp():
    """45 copies of one unit: groups of 90 members (both strands), analysed by lanes striding over their members."""
    base = synth.random_reference(1000000, seed=41, n_contigs=4)
    ref = pasted_copies(base, seed=42, families=1, copies=(45, 45), unit_len=(300, 300), divergence=0.02)
    assert run_parity(ref, "45-copy family") > 10


def test_scratch_overflow_second_attempt(monkeypatch, capfd):
    """XM_ANC_SCRATCH=64: analyses longer than 64 steps run out of the first attempt's scratch and are re-run with their own."""
    ref = synth.random_reference(1000000, seed=51, n_contigs=6, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 5000))
    assert run_parity(ref, "XM_ANC_SCRATCH=64", monkeypatch, {"XM_ANC_SCRATCH": "64", "XM_TRACE_SETUP": "1"}) > 100
    m = re.search(r"infer ancestors: .*\((\d+) analyses re-run\)", capfd.readouterr().err)
    assert m and int(m.group(1)) > 0


def test_positions_past_2_to_the_32(monkeypatch):
    """XM_POSITION_BIAS moves the reference past 2^32 (40-bit global positions): the same "-anc" codes."""
    ref = synth.random_reference(1000000, seed=61, n_contigs=5, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 5000))
    assert run_parity(ref, "XM_POSITION_BIAS=2^33+12345", monkeypatch, {"XM_POSITION_BIAS": str(2 ** 33 + 12345)}) > 100


def test_reference_without_duplications():
    ref = synth.random_reference(300000, seed=71, n_contigs=3)
    db, changed, originals = oracle_and_originals(ref)
    assert changed == 0
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.set_reference_from_codes(originals)
    assert infer_like_mapper(g, originals) == 0
    for i, c in enumerate(originals):
        assert np.array_equal(g.get_reference(i), c)
    g.close()


def test_state_handling():
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    n = capi.C.c_int64()
    assert g.L.xm_infer_ancestors(g.h, capi.C.c_double(0.1), -1, -1, 0, capi.C.byref(n)) == XM_ERR_STATE   # no reference yet
    ref = synth.random_reference(300000, seed=81, n_contigs=3, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 3000))
    originals = [c for _, c in ref]
    g.set_reference_from_codes(originals)
    g.build_index(150)
    g.build_duplications(-1, -1, 2, 1000)
    assert g.index_info()[1] >= 150
    infer_like_mapper(g, originals)
    assert g.index_info()[1] == 0                     # the old index is gone
    batch = synth.simulate_reads([(n, g.get_reference(i)) for i, (n, _) in enumerate(ref)], 50, 150, seed=82)
    with pytest.raises(capi.XmError, match="status %d" % XM_ERR_STATE):
        g.align_batch(batch)                          # until an index is built
    g.build_index(150)
    g.build_duplications(-1, -1, 2, 1000)
    got = g.align_batch(batch, strict=True)
    assert len(got["q_status"]) == 50
    g.close()


def test_config4_infer_ancestors_through_the_library():
    """configs[4] with --infer-ancestors and no oracle on the product side: infer on the device, device index builder, duplication
    table, 10 kbp reads split past 1000 - bit for bit the oracle's pipeline on the same reference."""
    ref = synth.random_reference(2000000, seed=6, n_contigs=10, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 5000))
    db, changed, originals = oracle_and_originals(ref)
    assert changed > 500
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    g.set_reference_from_codes(originals)
    n_changed = infer_like_mapper(g, originals)
    assert_same_anc(g, db, changed, n_changed, "configs[4] reference")
    g.build_index(1000)                               # the device builder, over the "-anc" reference
    g.build_duplications(-1, -1, 2, 1000)
    long_batch = synth.simulate_reads(ref, 40, 10000, seed=8, sub_rate=0.01, indel_rate=0.005)
    pieces, _ = synth.split_queries([q[0] for q in synth.unpack_reads(long_batch)], 1000)
    batch = synth.batch_from_reads(pieces)
    got = g.align_batch(batch, strict=True)
    want = db.align_batch(synth.DEFAULT_PARAMS, batch, threads=THREADS)
    parity.assert_same_results(want, got, "configs[4] --infer-ancestors through the library")
    g.close()
