"""python -m mapper_b200 --device 0,1[,2,3]: the four inputs of test_gpu_cli.py (single-end with duplicate reads under other names, paired
with --spacing, split 10 kbp reads, --infer-ancestors), with batches small enough that every device gets at least three.  The SAM, VCF and
mutations files must be byte for byte those of --device 0, and their bodies the oracle's.  Plus a SAM-only run.  These need >= 2 GPUs.
On one GPU, the several-handle set-up and dispatch run with two handles on that GPU (SAM only: a communicator needs distinct GPUs)."""
import subprocess
import sys
import time

import numpy as np
import pytest

import parity
from mapper_b200 import __main__ as cli
from mapper_b200 import capi, synth
from test_gpu_cli import PARAMS, THREADS, ROOT, assert_bodies, expected, oracle_db, run_cli, write_fasta, write_fastq

pytestmark = pytest.mark.gpu


def device_lists():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two GPUs")
    return ["0,1"] + (["0,1,2,3"] if n >= 4 else [])


def check_devices(tmp_path, args, want):
    one = run_cli(str(tmp_path), *args, "--device", "0")
    assert_bodies(one, want)
    for devs in device_lists():
        assert run_cli(str(tmp_path), *args, "--device", devs) == one, devs


def test_single_end_duplicate_names(tmp_path):
    device_lists()
    ref = synth.random_reference(80000, seed=901, n_contigs=3)
    db = oracle_db(ref)
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    reads = [q[0] for q in synth.unpack_reads(synth.simulate_reads(contigs, 1200, 100, seed=902, sub_rate=0.02, indel_rate=0.005))]
    rng = np.random.default_rng(903)
    reads += [reads[i] for i in rng.choice(len(reads), size=200, replace=False)]
    names = ["q%05d" % x for x in rng.permutation(100000)[:len(reads)]]
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    write_fastq(tmp_path / "reads.fq", [(n, synth.codes_to_text(r)) for n, r in zip(names, reads)])
    check_devices(tmp_path, ["--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fq"), "--batch-reads", "100"],
                  expected(db, synth.batch_from_reads(reads), names))


def test_paired_spacing(tmp_path):
    device_lists()
    ref = synth.random_reference(80000, seed=911, n_contigs=2)
    db = oracle_db(ref)
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    batch = synth.simulate_reads(contigs, 600, 100, seed=912, sub_rate=0.02, indel_rate=0.004, paired=True, inner_mean=300.0)
    mates = synth.unpack_reads(batch)
    names = ["p%d/%d" % (i, m + 1) for i in range(len(mates)) for m in range(2)]
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    for m in range(2):
        write_fastq(tmp_path / ("r%d.fq" % (m + 1)), [("p%d/%d" % (i, m + 1), synth.codes_to_text(q[m])) for i, q in enumerate(mates)])
    check_devices(tmp_path, ["--reference", str(tmp_path / "ref.fa"), "--paired-queries", str(tmp_path / "r1.fq"), str(tmp_path / "r2.fq"),
                             "--spacing", "300", "50", "--batch-reads", "50"], expected(db, batch, names))


def test_long_reads_split(tmp_path):
    device_lists()
    ref = synth.random_reference(300000, seed=921, n_contigs=2)
    db = oracle_db(ref)
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    reads = [q[0] for q in synth.unpack_reads(synth.simulate_reads(contigs, 24, 10000, seed=922, sub_rate=0.01, indel_rate=0.002))]
    pieces, parent = synth.split_queries(reads, 1000)
    names = []
    for i, p in enumerate(parent):
        first = int(np.nonzero(parent == p)[0][0])
        n, L, k = int((parent == p).sum()), len(reads[p]), i - first
        names.append("long%d[%d:%d]" % (p, L * k // n, L * (k + 1) // n))
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    write_fasta(tmp_path / "reads.fa", [("long%d" % i, synth.codes_to_text(r)) for i, r in enumerate(reads)], width=80)
    check_devices(tmp_path, ["--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fa"), "--split-queries-past-size", "1000",
                             "--batch-reads", "2"], expected(db, synth.batch_from_reads(pieces), names))


def test_infer_ancestors(tmp_path):
    device_lists()
    ref = synth.random_reference(300000, seed=931, n_contigs=3, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 3000))
    db, changed = parity.inferred_ancestor_oracle(ref, PARAMS, threads=THREADS)
    assert changed > 0
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    batch = synth.simulate_reads(contigs, 800, 150, seed=932, sub_rate=0.01, indel_rate=0.002)
    names = ["r%d" % i for i in range(len(batch["n_seqs"]))]
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    write_fasta(tmp_path / "reads.fa", [(n, synth.codes_to_text(q[0])) for n, q in zip(names, synth.unpack_reads(batch))])
    check_devices(tmp_path, ["--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fa"), "--infer-ancestors", "--batch-reads", "60"],
                  expected(db, batch, names))


def test_sam_only(tmp_path):
    devs = device_lists()
    ref = synth.random_reference(80000, seed=941, n_contigs=2)
    db = oracle_db(ref)
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    batch = synth.simulate_reads(contigs, 900, 120, seed=942, sub_rate=0.02, indel_rate=0.004)
    names = ["s%d" % i for i in range(len(batch["n_seqs"]))]
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    write_fastq(tmp_path / "reads.fq", [(n, synth.codes_to_text(q[0])) for n, q in zip(names, synth.unpack_reads(batch))])
    out = {}
    for d in ["0"] + devs:
        sam = str(tmp_path / ("out%s.sam" % d.replace(",", "")))
        r = subprocess.run([sys.executable, "-m", "mapper_b200", "--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fq"),
                            "--batch-reads", "70", "--device", d, "--out-sam", sam], cwd=ROOT, capture_output=True, text=True, timeout=1800)
        assert r.returncode == 0, r.stderr
        assert "on %d device" % len(d.split(",")) in r.stderr
        out[d] = open(sam).read()
    assert all(v == out["0"] for v in out.values())
    assert "".join(ln for ln in out["0"].splitlines(keepends=True) if not ln.startswith("@")) == expected(db, batch, names)["sam"]


def test_two_handles_one_gpu(tmp_path):
    """The "-anc" reference copied from the first handle to the second, the index built on both at once, batches alternating between
    them: the SAM of --device 0."""
    ref = synth.random_reference(300000, seed=951, n_contigs=3, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 3000))
    reads = synth.simulate_reads(ref, 700, 150, seed=952, sub_rate=0.01, indel_rate=0.002)
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    write_fasta(tmp_path / "reads.fa", [("r%d" % i, synth.codes_to_text(q[0])) for i, q in enumerate(synth.unpack_reads(reads))])
    args = ["--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fa"), "--infer-ancestors", "--batch-reads", "60"]
    r = subprocess.run([sys.executable, "-m", "mapper_b200", *args, "--out-sam", str(tmp_path / "one.sam")], cwd=ROOT, capture_output=True, text=True,
                       timeout=1800)
    assert r.returncode == 0, r.stderr
    hs = [capi.XMapper(PARAMS, device=0) for _ in range(2)]
    try:
        cli.map_files(cli.parse_args(args + ["--out-sam", str(tmp_path / "two.sam")]), PARAMS, (0.0, 1.0), hs, time.perf_counter())
        assert [hs[1].get_reference(c).tolist() for c in range(3)] == [hs[0].get_reference(c).tolist() for c in range(3)]
    finally:
        [h.close() for h in hs]
    one = open(tmp_path / "one.sam").read()
    assert open(tmp_path / "two.sam").read() == one and one.count("\n") > 700
