"""xm_parse_reads against a restatement in numpy: FASTA wrapped at any width with CRLF, lowercase and every IUPAC letter; FASTQ; chunked
input carrying n_consumed; --split-queries-past-size pieces; max_records; malformed input; incomplete last records."""
import numpy as np
import pytest

from mapper_b200 import capi, synth

pytestmark = pytest.mark.gpu
IUPAC = b"ACMGRSVTWYHKDBN"
CODE = {c: int(np.nonzero(synth.LETTERS == c)[0][0]) for c in IUPAC}
CODE.update({c + 32: v for c, v in CODE.items()})   # lowercase


def codes(seq):
    return np.array([CODE[c] for c in seq], dtype=np.uint8)


def restate(text, fastq):
    """(names, code arrays) of the records of text, parsed by the rules of include/xmapper_b200.h."""
    lines = [ln[:-1] if ln.endswith(b"\r") else ln for ln in text.split(b"\n")]
    if lines and lines[-1] == b"":
        lines.pop()
    names, seqs = [], []
    if fastq:
        for i in range(0, len(lines), 4):
            names.append(lines[i][1:])
            seqs.append(codes(lines[i + 1]))
    else:
        for ln in lines:
            if ln.startswith(b">"):
                names.append(ln[1:])
                seqs.append([])
            elif ln:
                seqs[-1].append(ln)
        seqs = [codes(b"".join(s)) for s in seqs]
    return names, seqs


def random_records(rng, n, lo, hi, letters=b"ACGT", p_iupac=0.02):
    out = []
    for i in range(n):
        L = int(rng.integers(lo, hi + 1))
        s = bytearray(rng.choice(np.frombuffer(letters, np.uint8), size=L).tobytes())
        for k in np.nonzero(rng.random(L) < p_iupac)[0]:
            s[k] = IUPAC[rng.integers(0, len(IUPAC))]
        low = rng.random(L) < 0.1
        s = bytes(c + 32 if lw else c for c, lw in zip(s, low))
        out.append((b"read_%d some description %d" % (i, rng.integers(0, 1000)), s))
    return out


def fasta(records, width, crlf=False, blank=False):
    nl = b"\r\n" if crlf else b"\n"
    out = []
    for name, s in records:
        out.append(b">" + name + nl)
        out += [s[k:k + width] + nl for k in range(0, len(s), width)]
        if blank:
            out.append(nl)
    return b"".join(out)


def fastq(records, crlf=False):
    nl = b"\r\n" if crlf else b"\n"
    return b"".join(b"@" + n + nl + s + nl + b"+" + nl + b"I" * len(s) + nl for n, s in records)


@pytest.fixture(scope="module")
def g():
    h = capi.XMapper(synth.DEFAULT_PARAMS, device=0)
    yield h
    h.close()


def check(got, names, seqs, records=None):
    batch, got_names, rec, _ = got
    packed, off, lens = synth.pack_reads(seqs)
    assert np.array_equal(batch["seq_len"], lens)
    assert np.array_equal(batch["seq_word_off"], off)
    assert np.array_equal(batch["packed"][:len(packed)], packed)
    assert got_names == [n.decode() for n in names]
    assert np.array_equal(rec, np.arange(len(seqs)) if records is None else records)


@pytest.mark.parametrize("width,crlf,blank", [(60, False, False), (80, True, True), (7, False, True)])
def test_fasta(g, width, crlf, blank):
    rng = np.random.default_rng(width)
    recs = random_records(rng, 300, 0, 700, p_iupac=0.05)
    recs[0] = (b"all", IUPAC + IUPAC.lower())
    text = fasta(recs, width, crlf, blank)
    names, seqs = restate(text, False)
    got = g.parse_reads(text, capi.FASTA)
    check(got, names, seqs)
    assert got[3] == len(text)


@pytest.mark.parametrize("crlf", [False, True])
def test_fastq(g, crlf):
    rng = np.random.default_rng(7 + crlf)
    text = fastq(random_records(rng, 2000, 1, 300), crlf)
    names, seqs = restate(text, True)
    got = g.parse_reads(text, capi.FASTQ)
    check(got, names, seqs)
    assert got[3] == len(text)
    # the last line needs no '\n' at the end of the input
    check(g.parse_reads(text.rstrip(b"\r\n"), capi.FASTQ), names, seqs)


@pytest.mark.parametrize("fmt", [capi.FASTA, capi.FASTQ])
def test_chunks_concatenate_to_one_call(g, fmt):
    rng = np.random.default_rng(11 + fmt)
    recs = random_records(rng, 1500, 50, 400)
    text = fastq(recs) if fmt == capi.FASTQ else fasta(recs, 61, crlf=True)
    whole, _ = g.parse_reads_raw(text, fmt)
    cuts = sorted(set(rng.integers(1, len(text), size=25).tolist()))
    names, seqs, buf, pos = [], [], b"", 0
    for end in cuts + [len(text)]:
        buf += text[pos:end]
        pos = end
        batch, nm, rec, used = g.parse_reads(buf, fmt, at_eof=end == len(text))
        names += nm
        seqs += [q[0] for q in synth.unpack_reads(batch)]
        buf = buf[used:]
    assert buf == b""
    wb, wn, _, _ = g.parse_reads(text, fmt)
    assert names == wn
    packed, off, lens = synth.pack_reads(seqs)
    assert np.array_equal(packed, whole["packed"]) and np.array_equal(off, whole["seq_word_off"]) and np.array_equal(lens, whole["seq_len"])


def test_split(g):
    rng = np.random.default_rng(21)
    recs = random_records(rng, 40, 1, 4000) + [(b"r2500", b"ACGT" * 625)]
    text = fasta(recs, 80)
    names, seqs = restate(text, False)
    pieces, parent = synth.split_queries(seqs, 1000)
    batch, got_names, rec, _ = g.parse_reads(text, capi.FASTA, split_size=1000)
    want_names = []
    for i, p in enumerate(parent):
        L, n = len(seqs[p]), int((parent == p).sum())
        k = i - int(np.nonzero(parent == p)[0][0])
        want_names.append(names[p] + (b"[%d:%d]" % (L * k // n, L * (k + 1) // n) if n > 1 else b""))
    check((batch, got_names, rec, 0), want_names, pieces, parent)
    last = [int(x) for x in batch["seq_len"][rec == len(recs) - 1]]
    assert last == [833, 833, 834] and got_names[-3:] == ["r2500[0:833]", "r2500[833:1666]", "r2500[1666:2500]"]


@pytest.mark.parametrize("fmt", [capi.FASTA, capi.FASTQ])
def test_max_records(g, fmt):
    rng = np.random.default_rng(31)
    recs = random_records(rng, 100, 10, 200)
    text = fastq(recs) if fmt == capi.FASTQ else fasta(recs, 60)
    names, seqs = restate(text, fmt == capi.FASTQ)
    batch, nm, rec, used = g.parse_reads(text, fmt, max_records=37)
    check((batch, nm, rec, used), names[:37], seqs[:37])
    rest = g.parse_reads(text[used:], fmt)
    check(rest, names[37:], seqs[37:])
    assert g.parse_reads(text, fmt, max_records=0)[3] == 0


def test_incomplete_last_record_is_not_consumed(g):
    rng = np.random.default_rng(41)
    recs = random_records(rng, 10, 20, 100)
    fq = fastq(recs)
    cut = fq[:-5]   # inside the last quality line
    batch, nm, rec, used = g.parse_reads(cut, capi.FASTQ, at_eof=False)
    assert len(nm) == 9 and used == len(fastq(recs[:9]))
    fa = fasta(recs, 50)
    batch, nm, rec, used = g.parse_reads(fa, capi.FASTA, at_eof=False)   # the last record may go on in the next chunk
    assert len(nm) == 9 and used == len(fasta(recs[:9], 50))
    assert g.parse_reads(fa, capi.FASTA, at_eof=True)[3] == len(fa)


@pytest.mark.parametrize("fmt,text,record", [
    (capi.FASTQ, b"@a\nACGT\n+\nIIII\n@b\nACXT\n+\nIIII\n", 1),
    (capi.FASTQ, b"@a\nACGT\n+\nIIII\n@b\nACGT\n+\nIII\n", 1),
    (capi.FASTQ, b"@a\nACGT\n+\nIIII\n@b\nACGT\nIIII\n@c\nA\n+\nI\n", 1),
    (capi.FASTQ, b"@a\nACGT\n+\nIIII\n@b\nAC", 1),
    (capi.FASTA, b">a\nACGT\n>b\nAC GT\n>c\nA\n", 1),
    (capi.FASTA, b">a\nACGT\n>b\nACGT\n>c\nAC-A\n", 2),
])
def test_malformed(g, fmt, text, record):
    with pytest.raises(capi.XmError) as e:
        g.parse_reads(text, fmt)
    assert "status -1" in str(e.value) and ("record %d," % record) in str(e.value)
