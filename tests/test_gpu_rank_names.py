"""xm_rank_names on the device against np.unique(names, dtype=object)'s inverse, the host ranking it replaces: empty and single inputs,
Illumina-style names, duplicates, empty names, NUL and high bytes, lengths around the 7-byte chunks, a 300-byte common prefix, the names
xm_parse_reads gives split reads, and bad offsets."""
import numpy as np
import pytest

from mapper_b200 import capi, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    h = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    yield h
    h.close()


def blob(names):
    off = np.zeros(len(names) + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in names])
    return b"".join(names), off


def check(g, names):
    want = np.unique(np.array(names, dtype=object), return_inverse=True)[1].astype(np.int64).reshape(-1) if names else np.zeros(0, np.int64)
    got = g.rank_names(*blob(names))
    assert got.dtype == np.int64 and np.array_equal(got, want)


def test_zero_and_one(g):
    check(g, [])
    check(g, [b"read1"])
    check(g, [b""])


def test_illumina_names(g):
    rng = np.random.default_rng(1)
    n = 1 << 20
    lane, tile, x, y = rng.integers(1, 5, n), rng.integers(1101, 1199, n), rng.integers(1000, 32000, n), rng.integers(1000, 32000, n)
    names = [b"A00123:8:H2FJ3DSXX:%d:%d:%d:%d 1:N:0:ATCACG" % t for t in zip(lane, tile, x, y)]
    check(g, names)


def test_duplicates_and_empty_names(g):
    rng = np.random.default_rng(2)
    base = [b"q%05d" % i for i in rng.permutation(3000)] + [b""] * 5
    check(g, [base[i] for i in rng.integers(0, len(base), 20000)])


def test_nul_and_high_bytes(g):
    rng = np.random.default_rng(3)
    alphabet = np.array([0, 1, 0x41, 0x7f, 0x80, 0xc3, 0xff], np.uint8)
    names = [bytes(alphabet[rng.integers(0, len(alphabet), rng.integers(0, 12))].tolist()) for _ in range(50000)]
    names += [b"a", b"a\0", b"a\0\0", b"a\x01", b"a\xff", b"\xff", b"\0", b"", b"\0" * 7, b"\0" * 8, b"\0" * 9]
    check(g, names)


def test_chunk_boundaries(g):
    rng = np.random.default_rng(4)
    names = []
    for k in range(1, 8):
        for L in (7 * k - 1, 7 * k, 7 * k + 1):
            for _ in range(300):
                s = bytearray(b"x" * L)
                if rng.random() < 0.7 and L:
                    s[rng.integers(0, L)] = int(rng.choice([0, 0x77, 0x79, 0xff]))
                names.append(bytes(s))
    check(g, names)


def test_300_byte_common_prefix(g):
    rng = np.random.default_rng(5)
    prefix = bytes(rng.integers(0, 256, 300).tolist())
    names = [prefix + b"%d" % i for i in rng.permutation(200000)] + [prefix, prefix[:299], prefix + b"\0"]
    check(g, names)


def test_split_read_names(g):
    rng = np.random.default_rng(6)
    recs = []
    for i in range(400):
        L = int(rng.integers(1, 5000))
        recs.append(">long%d\n%s\n" % (i % 150, "".join(rng.choice(list("ACGT"), L))))   # repeated record names: equal piece names
    a, _ = g.parse_reads_raw("".join(recs).encode(), capi.FASTA, split_size=1000)
    names = [a["names"][a["name_off"][i]:a["name_off"][i + 1]] for i in range(len(a["seq_len"]))]
    assert any(b"[" in x for x in names)
    check(g, names)
    assert np.array_equal(g.rank_names(a["names"], a["name_off"]), g.rank_names(*blob(names)))


def test_bad_offsets(g):
    with pytest.raises(capi.XmError, match="non-decreasing"):
        g.rank_names(b"abcd", np.array([0, 3, 2, 4], np.int64))
    with pytest.raises(capi.XmError, match=r"name_off\[0\]"):
        g.rank_names(b"abcd", np.array([1, 4], np.int64))
