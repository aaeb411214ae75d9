"""python -m mapper_b200 without a device: --help, and every reference flag the command does not implement exits with status 2 naming it."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args):
    return subprocess.run([sys.executable, "-m", "mapper_b200", *args], cwd=ROOT, capture_output=True, text=True, timeout=120)


def test_help():
    r = run("--help")
    assert r.returncode == 0
    for flag in ("--reference", "--queries", "--paired-queries", "--spacing", "--split-queries-past-size", "--infer-ancestors", "--no-gapmers",
                 "--out-sam", "--out-vcf", "--out-mutations", "--distinguish-query-ends", "--device", "--batch-reads"):
        assert flag in r.stdout, flag


@pytest.mark.parametrize("flag", [["--out-refs-map-count", "x"], ["--out-unaligned", "x"], ["--cache-dir", "d"], ["--num-threads", "4"],
                                  ["--verify-consistent-db"], ["--snp-threshold", "5"], ["--indel-start-threshold=1"], ["--max-penalty", "0.2"]])
def test_unsupported_flag(flag):
    r = run("--reference", "ref.fa", "--queries", "q.fq", "--out-vcf", "out.vcf", *flag)
    assert r.returncode == 2
    assert "unsupported flag: " + flag[0].split("=")[0] in r.stderr


def test_abbreviations_are_not_accepted():
    r = run("--reference", "ref.fa", "--queries", "q.fq", "--out-v", "out.vcf")
    assert r.returncode == 2 and "--out-v" in r.stderr


def test_queries_required():
    assert run("--reference", "ref.fa").returncode == 2
