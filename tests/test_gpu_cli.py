"""python -m mapper_b200 as a subprocess on the GPU: BASELINE.json configs[0] against the committed bodies, and random inputs against the
oracle (tests/sam_oracle.py over Oracle.align_batch, tests/variants_oracle.py accumulated with the reads' names): single-end FASTQ over
several batches with duplicate reads under other names, paired FASTQ with --spacing, 10 kbp FASTA reads split past 1000, an inferred-
ancestor reference; and the same output whatever --batch-reads is."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import parity
import sam_oracle
import variants_oracle as vo
import xm_oracle as xo
from mapper_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.join(ROOT, "tests")
THREADS = os.cpu_count() or 4
PARAMS = synth.DEFAULT_PARAMS


def write_fasta(path, records, width=70):
    with open(path, "w") as f:
        for name, text in records:
            f.write(">%s\n" % name)
            for k in range(0, len(text), width):
                f.write(text[k:k + width] + "\n")


def write_fastq(path, records):
    with open(path, "w") as f:
        for name, text in records:
            f.write("@%s\n%s\n+\n%s\n" % (name, text, "I" * len(text)))


def run_cli(tmp, *args):
    out = {k: os.path.join(tmp, "out." + k) for k in ("sam", "vcf", "mut")}
    r = subprocess.run([sys.executable, "-m", "mapper_b200", *args, "--out-sam", out["sam"], "--out-vcf", out["vcf"], "--out-mutations", out["mut"]],
                       cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr
    return {k: open(v).read() for k, v in out.items()}


def body(text, marker):
    return "".join(ln for ln in text.splitlines(keepends=True) if not ln.startswith(marker))


def expected(db, batch, names, end_fraction=0.1):
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    res = db.align_batch(PARAMS, batch, threads=THREADS)
    store = vo.Store(contigs, end_fraction)
    vo.accumulate(store, res, synth.unpack_reads(batch), names)
    return dict(sam=sam_oracle.format_sam(res, batch, names, [n for n, _ in contigs]), vcf=vo.vcf_body(store),
                mut=vo.mutations_body(store, vo.Filter.default()))


def assert_bodies(got, want):
    assert body(got["sam"], "@") == want["sam"]
    assert body(got["vcf"], "#") == want["vcf"]
    assert got["mut"] == want["mut"]


def oracle_db(ref):
    return xo.Oracle([(n, synth.codes_to_text(s)) for n, s in ref], sort_by_length=True, threads=THREADS, dup=dict(min_copies=2, window=1000))


def test_examples_config0(tmp_path):
    ex = json.load(open(os.path.join(HERE, "golden", "junit_vectors.json")))["examples"]
    write_fasta(tmp_path / "reference.fasta", ex["reference"])
    write_fasta(tmp_path / "queries.fasta", ex["queries"])
    got = run_cli(str(tmp_path), "--reference", str(tmp_path / "reference.fasta"), "--queries", str(tmp_path / "queries.fasta"))
    golden = json.load(open(os.path.join(HERE, "golden", "examples_expected.json")))
    assert body(got["sam"], "@") == golden["sam_body"]
    assert body(got["vcf"], "#") == golden["vcf_body"]
    assert got["mut"] == golden["mutations_body"]
    assert got["sam"].startswith("@SQ\tSN:%s\tLN:" % golden["contig_order"][0])


def test_single_end_fastq_batches_and_duplicate_names(tmp_path):
    ref = synth.random_reference(80000, seed=901, n_contigs=3)
    db = oracle_db(ref)
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    reads = [q[0] for q in synth.unpack_reads(synth.simulate_reads(contigs, 1200, 100, seed=902, sub_rate=0.02, indel_rate=0.005))]
    rng = np.random.default_rng(903)
    dup = rng.choice(len(reads), size=200, replace=False)
    reads += [reads[i] for i in dup]   # the same read under another name: example ties fall to the name order
    names = ["q%05d" % x for x in rng.permutation(100000)[:len(reads)]]
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    write_fastq(tmp_path / "reads.fq", [(n, synth.codes_to_text(r)) for n, r in zip(names, reads)])
    args = ["--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fq")]
    many = run_cli(str(tmp_path), *args, "--batch-reads", "300")
    assert_bodies(many, expected(db, synth.batch_from_reads(reads), names))
    assert run_cli(str(tmp_path), *args, "--batch-reads", "100000") == many


def test_paired_fastq_spacing(tmp_path):
    ref = synth.random_reference(80000, seed=911, n_contigs=2)
    db = oracle_db(ref)
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    batch = synth.simulate_reads(contigs, 600, 100, seed=912, sub_rate=0.02, indel_rate=0.004, paired=True, inner_mean=300.0)
    mates = synth.unpack_reads(batch)
    names = ["p%d/%d" % (i, m + 1) for i in range(len(mates)) for m in range(2)]
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    for m in range(2):
        write_fastq(tmp_path / ("r%d.fq" % (m + 1)), [("p%d/%d" % (i, m + 1), synth.codes_to_text(q[m])) for i, q in enumerate(mates)])
    got = run_cli(str(tmp_path), "--reference", str(tmp_path / "ref.fa"), "--paired-queries", str(tmp_path / "r1.fq"), str(tmp_path / "r2.fq"),
                  "--spacing", "300", "50", "--batch-reads", "250")
    assert_bodies(got, expected(db, batch, names))


def test_long_fasta_reads_split(tmp_path):
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
    got = run_cli(str(tmp_path), "--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fa"), "--split-queries-past-size", "1000",
                  "--batch-reads", "10")
    assert_bodies(got, expected(db, synth.batch_from_reads(pieces), names))


def test_infer_ancestors(tmp_path):
    ref = synth.random_reference(300000, seed=931, n_contigs=3, repeat_fraction=0.08, repeat_copies=(3, 6), repeat_len=(1000, 3000))
    db, changed = parity.inferred_ancestor_oracle(ref, PARAMS, threads=THREADS)
    assert changed > 0
    contigs = [db.contig(i) for i in range(db.num_contigs())]
    batch = synth.simulate_reads(contigs, 800, 150, seed=932, sub_rate=0.01, indel_rate=0.002)
    names = ["r%d" % i for i in range(len(batch["n_seqs"]))]
    write_fasta(tmp_path / "ref.fa", [(n, synth.codes_to_text(s)) for n, s in ref])
    write_fasta(tmp_path / "reads.fa", [(n, synth.codes_to_text(q[0])) for n, q in zip(names, synth.unpack_reads(batch))])
    got = run_cli(str(tmp_path), "--reference", str(tmp_path / "ref.fa"), "--queries", str(tmp_path / "reads.fa"), "--infer-ancestors")
    assert_bodies(got, expected(db, batch, names))
