"""VCF and mutations bodies formatted on the device (xm_format_vcf / xm_format_mutations) against tests/variants_oracle.py, byte for
byte: the reference's MutationsWriter KATs, BASELINE.json configs[0], random references (single and paired reads, ambiguous reads,
indels, an IUPAC reference) under three filters, range splits, the carry-in of _could_be_deletion, states and arguments, two GPUs."""
import json
import os
import threading

import numpy as np
import pytest

import parity
import variants_oracle as vo
import xm_oracle as xo
from mapper_b200 import capi, synth
from test_gpu_variants import flat, name_ranks

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
V = json.load(open(os.path.join(HERE, "golden", "junit_vectors.json")))
JOB = 8192
TIGHT = vo.Filter(minIndelTotalStartDepth=1, minIndelStartDepthFraction=0.2, minIndelContinuationTotalDepth=1,
                  minIndelContinuationDepthFraction=0.1)


def fdict(flt):
    return None if flt is None else {k: getattr(flt, k) for k in capi.FILTER_FIELDS}


def by_name(contigs):
    return sorted((n, c) for c, (n, _) in enumerate(contigs))


def device_vcf(g, contigs, flt=None, inm=True, support=True, cuts=None):
    """Contigs in name order (the host's TreeMap), each over the ranges cuts(length) gives (default: the whole contig)."""
    out = []
    for name, c in by_name(contigs):
        n = len(contigs[c][1])
        cc = cuts(n) if cuts else [0, n]
        out += [g.format_vcf(c, name, a, b, fdict(flt), inm, support) for a, b in zip(cc, cc[1:])]
    return "".join(out)


def device_mutations(g, contigs, flt=None, cuts=None):
    out = []
    for name, c in by_name(contigs):
        n = len(contigs[c][1])
        cc = cuts(n) if cuts else [0, n]
        out += [g.format_mutations(c, name, a, b, fdict(flt)) for a, b in zip(cc, cc[1:])]
    return "".join(out)


def random_cuts(rng, grid):
    def cuts(n):
        k = rng.integers(1, 6)
        inner = sorted(set((rng.integers(0, n + 1, size=k) // grid * grid).tolist()) - {0, n})
        return [0] + inner + [n]
    return cuts


def upload_examples(g, all_reads):
    g.set_variant_examples({gid: all_reads[gid] for gid in g.variants_examples().tolist()})


@pytest.mark.parametrize("case", V["mutations_cases"], ids=[c["name"] for c in V["mutations_cases"]])
def test_mutations_writer_tables_on_device(case):
    """T/MutationsWriter_Test: the 9 tables, aligned on the device with the case's parameters and formatted there."""
    db = xo.Oracle([("ref", case["reference"])], sort_by_length=False, dup=case["dup"])
    batch = parity.batch_from_texts([[case["query"]]])
    g = capi.XMapper(case["params"], device=0)
    parity.feed_from_oracle(g, db, len(case["query"]) + 2, case["dup"]["window"])
    g.counts_enable(case["end_fraction"])
    got = g.align_batch(batch, strict=True)
    parity.assert_same_results(db.align_batch(case["params"], batch), got, case["name"])
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    assert device_mutations(g, contigs, vo.Filter(**case["filter"])) == case["expected"]
    g.close()


def test_vcf_writer_cases_do_not_align():
    """QVT/VcfWriter_Test builds its alignments by hand.  None of its five cases (simpleTest, mutationTest,
    mutationWithoutSupportReads, oneReadWithMultipleAlignments, readWithThreeAlignments) can run through the library: their reads
    are 4 and 5 bases long, shorter than any seed, so neither the oracle aligner nor the device finds an alignment, and the counts
    stay empty.  This test pins that, and that the device bodies are then empty.  The five bodies stay covered on the CPU by
    tests/test_variants_oracle.py::test_vcf_bodies."""
    params = V["examples"]["params"]
    for case in V["vcf_cases"]:
        db = xo.Oracle([("contig1", case["reference"])], dup=dict(min_copies=2, window=1))
        batch = parity.batch_from_texts([[case["seq"]]])
        want = db.align_batch(params, batch)
        assert int(want["comp_choice_off"][-1]) == 0, case["name"]
        g = capi.XMapper(params, device=0)
        parity.feed_from_oracle(g, db, len(case["seq"]) + 2, 1)
        g.counts_enable(0.0)
        got = g.align_batch(batch, strict=True)
        parity.assert_same_results(want, got, case["name"])
        contigs = [db.contig(0)]
        upload_examples(g, [])
        assert device_vcf(g, contigs, support=case["support"]) == "" and device_mutations(g, contigs) == ""
        g.close()


def test_examples_config0_bodies():
    """BASELINE.json configs[0] as test_gpu_variants.test_examples_config0 sets it up: the device's VCF body (with support) and
    mutations body (default filter) equal the committed fixture."""
    ex = V["examples"]
    db = xo.Oracle([(n, t) for n, t in ex["reference"]], sort_by_length=True, dup=dict(min_copies=2, window=1000))
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    names = [n for n, _ in ex["queries"]]
    batch = parity.batch_from_texts([[t] for _, t in ex["queries"]])
    g = capi.XMapper(ex["params"], device=0)
    parity.feed_reference(g, db)
    g.build_index(max(len(t) for _, t in ex["queries"]) + 2)
    g.build_duplications(-1, -1, 2, 1000)
    g.counts_enable(0.1)
    g.counts_batch_info(0, name_ranks(names))
    g.align_batch(batch, strict=True)
    upload_examples(g, flat(synth.unpack_reads(batch)))
    golden = json.load(open(os.path.join(HERE, "golden", "examples_expected.json")))
    assert device_vcf(g, contigs) == golden["vcf_body"]
    assert device_mutations(g, contigs, vo.Filter.default()) == golden["mutations_body"]
    g.close()


def iupac_reference(seed, n_bases):
    """Two contigs of n_bases each; the second carries N and two-base IUPAC codes."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(2):
        _, codes = synth.random_reference(n_bases, seed=seed + 17 * k, n_contigs=1, repeat_fraction=0.1, repeat_len=(150, 600), repeat_divergence=0.0)[0]
        name = "chr%d" % (k + 1)
        codes = codes.copy()
        if k == 0:
            out.append((name, codes))
            continue
        at = rng.choice(len(codes), size=len(codes) // 2000, replace=False)
        codes[at] = rng.choice(np.array([15, 5, 10, 3, 12], dtype=np.uint8), size=len(at))   # N and two-base codes
        out.append((name, codes))
    return out


def run_reads(g, contigs, store, batches, seed):
    """Aligns the batches on the device and accumulates the device's results into the oracle's Store; returns the reads by gid."""
    rng = np.random.default_rng(seed)
    universe = sorted("r%d" % i for i in range(40))
    all_reads, all_names = [], []
    for batch in batches:
        reads = synth.unpack_reads(batch)
        n_seq = sum(len(q) for q in reads)
        names = ["r%d" % rng.integers(0, 40) for _ in range(n_seq)]
        first = len(all_names)
        all_reads += flat(reads); all_names += names
        g.counts_batch_info(first, np.array([universe.index(n) for n in names], dtype=np.int64))
        got = g.align_batch(batch, strict=False)
        vo.accumulate(store, got, reads, names, first_seq_id=first)
    return all_reads


@pytest.mark.parametrize("paired", [False, True], ids=["single", "paired"])
def test_bodies_vs_oracle(paired):
    """Two 31 kbp contigs (four mutations jobs each), one with IUPAC letters in the reference; ambiguous reads with indels.  The
    device bodies equal vo.vcf_body / vo.mutations_body over the Store accumulated from the same device alignments, under the empty,
    the default and a tight-indel filter; the two parameter sets share the include_non_mutations / show_support combinations out."""
    from test_emu_parity import ambiguate
    ref = iupac_reference(401 + paired, 31000)
    db = xo.Oracle([(n, synth.codes_to_text(s)) for n, s in ref], sort_by_length=True, dup=dict(min_copies=2, window=1000))
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    assert any(vo.is_ambiguous_code(int(x)) and x != 15 for _, c in contigs for x in c) and any((c == 15).any() for _, c in contigs)
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    parity.feed_reference(g, db)
    g.build_index(100)
    g.build_duplications(-1, -1, 2, 1000)
    g.counts_enable(0.1)
    store = vo.Store(contigs, 0.1)
    batches = [ambiguate(synth.simulate_reads(contigs, 3000, 100, seed=410 + 3 * it + paired, sub_rate=0.02, indel_rate=0.008, paired=paired,
                                              inner_mean=60.0, inner_sd=40.0), 420 + it, 0.004) for it in range(2)]
    all_reads = run_reads(g, contigs, store, batches, 430 + paired)
    upload_examples(g, all_reads)
    # _could_be_deletion decides both ways under TIGHT
    decided = [store._could_be_deletion(c, i, TIGHT) for c in range(len(contigs)) for i in range(0, len(contigs[c][1]))
               if store.position(c, i).alt_count("-") > 0]
    assert True in decided and False in decided
    combos = [(True, True), (False, False), (True, False)] if not paired else [(False, True), (True, True), (False, False)]
    for flt, (inm, support) in zip((vo.Filter(), vo.Filter.default(), TIGHT), combos):
        assert device_vcf(g, contigs, flt, inm, support) == vo.vcf_body(store, flt, inm, support), (flt.__dict__, inm, support)
        assert device_mutations(g, contigs, flt) == vo.mutations_body(store, flt), flt.__dict__
    # any split of the VCF, any 8192-aligned split of the mutations, concatenates to the whole
    rng = np.random.default_rng(440 + paired)
    for flt in (vo.Filter(), TIGHT):
        whole_v, whole_m = device_vcf(g, contigs, flt), device_mutations(g, contigs, flt)
        for _ in range(3):
            assert device_vcf(g, contigs, flt, cuts=random_cuts(rng, 1)) == whole_v
            assert device_mutations(g, contigs, flt, cuts=random_cuts(rng, JOB)) == whole_m
    g.close()


def test_deletion_runs_across_boundaries():
    """Crafted deletions: a 7-base run over the 8192 boundary (two mutations records, as MutationsWriter's jobs give), a chain of
    continuation-only positions behind a start-supported one (true), and one behind a position without deletions (false); ranges
    that start inside both chains need the carry-in walk."""
    ref = synth.random_reference(20000, seed=501, n_contigs=1)
    db = xo.Oracle([(n, synth.codes_to_text(s)) for n, s in ref], sort_by_length=True, dup=dict(min_copies=2, window=1000))
    name, codes = db.contig(0)
    text = synth.codes_to_text(codes)
    reads = []
    for k in range(16):
        for (a, b), n_del in (((8189, 8196), 4), ((8189, 8191), 4), ((12001, 12005), 2)):
            lo = a - 60 - k
            if k < n_del:
                reads.append(text[lo:a] + text[b:b + 75 + k])
            else:
                reads.append(text[lo:lo + 135 + (b - a) + k])
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    parity.feed_reference(g, db)
    g.build_index(150)
    g.build_duplications(-1, -1, 2, 1000)
    g.counts_enable(0.1)
    contigs = [(name, codes)]
    store = vo.Store(contigs, 0.1)
    batch = parity.batch_from_texts([[r] for r in reads])
    got = g.align_batch(batch, strict=True)
    vo.accumulate(store, got, synth.unpack_reads(batch), ["q%d" % i for i in range(len(reads))])
    upload_examples(g, flat(synth.unpack_reads(batch)))
    # the aligner places the runs at 8187..8191 + 8192..8193 and 11999..12002; 12001 is continuation-only, behind 11998 without deletions
    p = store.position(0, 12001)
    assert p.alt_count("-") > 0 and not TIGHT.supports_indel_start(p) and TIGHT.supports_indel_continuation(p)
    assert store._could_be_deletion(0, 8193, TIGHT) and not store._could_be_deletion(0, 12001, TIGHT)
    mut = vo.mutations_body(store)
    runs = [ln.split("\t") for ln in mut.splitlines() if set(ln.split("\t")[3]) == {"-"}]
    assert [(r[1], len(r[3])) for r in runs if 8180 < int(r[1]) < 8200] == [("8188", 5), ("8193", 2)]   # 8187..8191 | 8192..8193
    assert device_mutations(g, contigs) == mut
    for flt in (vo.Filter(), TIGHT):
        want = vo.vcf_body(store, flt)
        assert device_vcf(g, contigs, flt) == want
        for cut in (8188, 8192, 8193, 8195, 12000, 12001, 12002):
            assert device_vcf(g, contigs, flt, cuts=lambda n: [0, cut, n]) == want, (flt.__dict__, cut)
        assert device_mutations(g, contigs, flt, cuts=lambda n: [0, JOB, 2 * JOB, n]) == vo.mutations_body(store, flt)
    g.close()


def test_states_and_arguments():
    ref = synth.random_reference(30000, seed=601, n_contigs=2)
    db = xo.Oracle([(n, synth.codes_to_text(s)) for n, s in ref], sort_by_length=True, dup=dict(min_copies=2, window=1000))
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    g = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    parity.feed_reference(g, db)
    g.build_index(100)
    g.build_duplications(-1, -1, 2, 1000)
    n0 = len(contigs[0][1])

    def status(f):
        try:
            f()
            return 0
        except capi.XmError as e:
            return int(str(e).split()[1].rstrip(":"))
    # counts off
    assert status(lambda: g.format_vcf(0, "a", 0, n0, None, True, False)) == -3
    assert status(lambda: g.format_mutations(0, "a", 0, n0)) == -3
    assert status(lambda: g.variants_examples()) == -3
    g.counts_enable(0.1)
    batches = [synth.simulate_reads(contigs, 800, 100, seed=602 + i, sub_rate=0.02, indel_rate=0.004) for i in range(2)]
    all_reads = flat(synth.unpack_reads(batches[0]))
    g.align_batch(batches[0])
    # support without examples; show_support=0 and mutations need none
    assert status(lambda: g.format_vcf(0, "a", 0, n0)) == -3
    no_support = g.format_vcf(0, "a", 0, n0, None, True, False)
    assert no_support.count("\n") > 1000 and g.format_mutations(0, "a", 0, n0).count("\n") > 10
    # wrong example arrays
    gids = g.variants_examples()
    assert len(gids) > 10 and np.all(np.diff(gids) > 0)
    L = g.L
    packed = [synth.pack_contig(all_reads[i]) for i in gids]
    off = np.concatenate([[0], np.cumsum([len(p) for p in packed])]).astype(np.int64)
    words = np.concatenate(packed + [np.zeros(1, np.uint16)])
    lens = np.array([len(all_reads[i]) for i in gids], dtype=np.int32)
    ptr = capi._ptr
    assert L.xm_variants_set_examples(g.h, len(gids) - 1, ptr(gids), ptr(words), ptr(off), ptr(lens)) == -1
    swapped = gids.copy(); swapped[[0, 1]] = swapped[[1, 0]]
    assert L.xm_variants_set_examples(g.h, len(gids), ptr(swapped), ptr(words), ptr(off), ptr(lens)) == -1
    short = lens.copy(); short[3] -= 1
    assert L.xm_variants_set_examples(g.h, len(gids), ptr(gids), ptr(words), ptr(off), ptr(short)) == -1
    assert status(lambda: g.format_vcf(0, "a", 0, n0)) == -3
    assert L.xm_variants_set_examples(g.h, len(gids), ptr(gids), ptr(words), ptr(off), ptr(lens)) == 0
    with_support = g.format_vcf(0, "a", 0, n0)
    assert with_support.count("\n") == no_support.count("\n") and "[" in with_support
    # stale after another batch
    g.align_batch(batches[1])
    assert status(lambda: g.format_vcf(0, "a", 0, n0)) == -3
    assert g.format_vcf(0, "a", 0, n0, None, True, False).count("\n") >= no_support.count("\n")
    # bad contig / range / grid
    for f in (lambda: g.format_vcf(2, "a", 0, 10, None, True, False), lambda: g.format_vcf(-1, "a", 0, 10, None, True, False),
              lambda: g.format_vcf(0, "a", 5, 4, None, True, False), lambda: g.format_vcf(0, "a", -1, 4, None, True, False),
              lambda: g.format_vcf(0, "a", 0, n0 + 1, None, True, False), lambda: g.format_mutations(0, "a", 100, n0),
              lambda: g.format_mutations(0, "a", 0, JOB + 1)):
        assert status(f) == -1
    assert g.format_vcf(0, "a", 7, 7, None, True, False) == ""
    assert g.format_mutations(0, "a", 0, n0) == g.format_mutations(0, "a", 0, JOB) + g.format_mutations(0, "a", JOB, n0)
    g.close()


def test_two_gpus_after_reduce():
    """After xm_counts_reduce over two handles, rank 0's bodies equal those of one handle that aligned all the reads."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ref = synth.random_reference(70000, seed=701, n_contigs=2)
    db = xo.Oracle([(n, synth.codes_to_text(s)) for n, s in ref], sort_by_length=True, dup=dict(min_copies=2, window=1000))
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    batches = [synth.simulate_reads(contigs, 2000, 120, seed=710 + r, sub_rate=0.01, indel_rate=0.004) for r in range(2)]
    firsts = [0, int(batches[0]["n_seqs"].astype(np.int64).sum())]
    all_reads = flat(synth.unpack_reads(batches[0])) + flat(synth.unpack_reads(batches[1]))

    def make(dev):
        g = capi.XMapper(synth.DEFAULT_PARAMS, device=dev)
        parity.feed_reference(g, db)
        g.build_index(120)
        g.build_duplications(-1, -1, 2, 1000)
        g.counts_enable(0.1)
        return g

    def bodies(g):
        upload_examples(g, all_reads)
        return device_vcf(g, contigs), device_mutations(g, contigs, vo.Filter.default())

    g = make(0)
    for b, f in zip(batches, firsts):
        g.counts_batch_info(f)
        g.align_batch(b, strict=True)
    want = bodies(g)
    assert want[0].count("\n") > 10000
    g.close()
    hs = [make(0), make(1)]
    uid = hs[0].comm_unique_id()
    errs = []

    def run(rank):
        try:
            hs[rank].comm_init(2, rank, uid)
            hs[rank].counts_batch_info(firsts[rank])
            hs[rank].align_batch(batches[rank], strict=True)
            hs[rank].counts_reduce()
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [t.start() for t in th]
    [t.join(timeout=120) for t in th]
    assert not errs, errs
    assert bodies(hs[0]) == want
    [h.close() for h in hs]
