"""python -m mapper_b200: map FASTA/FASTQ reads against a FASTA reference on one GPU and write SAM, VCF and mutations files.

The front end of X-Mapper's Mapper.run (SURVEY.md §3.1), driving the C ABI; it holds no algorithm.
  1. Reference: parsed on the device (xm_parse_reads), contigs sorted as Mapper.sortAndComplementReference sorts them (descending
     length, ties in input order), xm_set_reference, optionally xm_infer_ancestors (--infer-ancestors, set up as M/Mapper.java:666-692),
     xm_build_index(longest query or split piece) and xm_build_duplications(-1, -1, 2, 1000).
  2. A pre-pass over the queries: the longest sequence for the index and, when counts are written, the rank of every sequence name in
     byte order (String.compareTo for ASCII names), the name order DirectionalAlignments.betterExample breaks example ties with.
  3. Batches: parsed on the device while the previous batch aligns (a second thread), xm_counts_batch_info, xm_align_batch and
     xm_format_sam right after it in the same thread (the slot rule of INTEGRATION.md §1).  A query the device could not align is an
     error naming the read, never a silent drop.
  4. After the last batch: the example reads of the VCF support column are read again from the inputs and uploaded, and the VCF and
     mutations bodies are formatted on the device per contig, in name order (VcfWriter.java:111-114).

Headers are this command's own: the reference's header texts are not in this repository and embed the command line (BASELINE.md §5),
so SAM gets @SQ lines in database order, the VCF a #CHROM column line, and the mutations file none.  Parity with the reference is for the
bodies.  Files ending in .gz are read through gzip on the host.  Every reference flag this command does not implement exits with
status 2 and names the flag.
"""
import argparse
import gzip
import queue
import sys
import threading

import numpy as np

from mapper_b200 import capi, synth

CHUNK_BYTES = 64 << 20              # text handed to one xm_parse_reads call (grown when a record does not fit)
VCF_RANGE = 1 << 20                 # positions per xm_format_vcf call
MUTATIONS_RANGE = 128 * 8192        # positions per xm_format_mutations call (a multiple of the writer's 8192-position jobs)
# MutationDetectionParameters defaults: no thresholds for the VCF, MutationDetectionParameters.defaultFilter() for the mutations file
MUTATIONS_FILTER = dict(minSNPTotalDepth=5, minSNPDepthFraction=0.9, minIndelTotalStartDepth=1, minIndelStartDepthFraction=0.8,
                        minIndelContinuationTotalDepth=1, minIndelContinuationDepthFraction=0.7)
KNOWN_UNSUPPORTED = ["--out-refs-map-count", "--out-unaligned", "--cache-dir", "--num-threads", "--verify-consistent-db",
                     "--snp-threshold", "--indel-start-threshold", "--indel-continue-threshold"]


def parse_args(argv):
    p = argparse.ArgumentParser(prog="python -m mapper_b200", allow_abbrev=False, description=__doc__.split("\n")[0],
                                epilog="Not supported (exit status 2): " + ", ".join(KNOWN_UNSUPPORTED) +
                                ", penalty and threshold options, and any other flag of the reference not listed above.")
    p.add_argument("--reference", nargs="+", required=True, metavar="FILE", help="reference FASTA files")
    p.add_argument("--queries", nargs="+", default=[], metavar="FILE", help="query FASTA or FASTQ files")
    p.add_argument("--paired-queries", nargs=2, action="append", default=[], metavar=("R1", "R2"), help="paired query files (FASTA or FASTQ)")
    p.add_argument("--spacing", nargs=2, type=float, metavar=("EXPECTED", "PER_PENALTY"),
                   help="expected inner distance of pairs and its deviation per unit of penalty (QV/Query.java:17-30)")
    p.add_argument("--split-queries-past-size", type=int, default=0, metavar="N", help="split reads longer than N into equal pieces")
    p.add_argument("--infer-ancestors", action="store_true", help="infer ancestral references before mapping")
    p.add_argument("--no-gapmers", action="store_true", help="index without gapmers")
    p.add_argument("--out-sam", metavar="F")
    p.add_argument("--out-vcf", metavar="F")
    p.add_argument("--out-mutations", metavar="F")
    p.add_argument("--distinguish-query-ends", type=float, default=0.1, metavar="F", help="query_end_fraction of the counts (default 0.1)")
    p.add_argument("--device", type=int, default=0, metavar="N", help="CUDA device")
    p.add_argument("--batch-reads", type=int, default=262144, metavar="N", help="queries per alignment batch")
    args, extra = p.parse_known_args(argv)
    for a in extra:
        if a.startswith("-"):
            p.exit(2, "%s: error: unsupported flag: %s\n" % (p.prog, a.split("=")[0]))
    if extra:
        p.error("unexpected argument: %s" % extra[0])
    if not args.queries and not args.paired_queries:
        p.error("no queries (--queries or --paired-queries)")
    if args.batch_reads < 1 or args.split_queries_past_size < 0:
        p.error("--batch-reads must be positive and --split-queries-past-size non-negative")
    return args


def fmt_of(path):
    """FASTQ when the first non-blank byte is '@', else FASTA."""
    with open_text(path) as f:
        head = f.read(4096).lstrip()
    return capi.FASTQ if head[:1] == b"@" else capi.FASTA


def open_text(path):
    return gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb")


def gather(data, starts, lens):
    """data[starts[i] : starts[i] + lens[i]] for all i, back to back, and the offsets of the pieces."""
    lens = np.asarray(lens, dtype=np.int64)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    idx = np.repeat(np.asarray(starts, dtype=np.int64) - off[:-1], lens) + np.arange(off[-1], dtype=np.int64)
    return data[idx], off


def select(a, which):
    """The sequences `which` of a parsed array dict, in that order."""
    wo, no = a["seq_word_off"], a["name_off"]
    packed, word_off = gather(a["packed"], wo[which], wo[np.asarray(which) + 1] - wo[which])
    names, name_off = gather(np.frombuffer(a["names"], dtype=np.uint8), no[which], no[np.asarray(which) + 1] - no[which])
    return dict(packed=packed, seq_word_off=word_off, seq_len=a["seq_len"][which], names=names.tobytes(), name_off=name_off)


def concat(parts):
    """Sequences of several parsed array dicts, back to back."""
    def offsets(key, size):
        shift = np.cumsum([0] + [size(p) for p in parts])
        return np.concatenate([p[key][:-1] + shift[i] for i, p in enumerate(parts)] + [shift[-1:]]).astype(np.int64)
    return dict(packed=np.concatenate([p["packed"] for p in parts]), seq_word_off=offsets("seq_word_off", lambda p: len(p["packed"])),
                seq_len=np.concatenate([p["seq_len"] for p in parts]), names=b"".join(p["names"] for p in parts),
                name_off=offsets("name_off", lambda p: len(p["names"])))


class Source:
    """One FASTA/FASTQ file read in chunks; the bytes a parse leaves (an incomplete last record) are passed again with the next chunk."""

    def __init__(self, path, split):
        self.path, self.split, self.fmt = path, split, fmt_of(path)
        self.f = open_text(path)
        self.buf, self.eof, self.chunk = b"", False, CHUNK_BYTES

    def done(self):
        return self.eof and not self.buf

    def take(self, g, want=-1, exact=False):
        """Parses up to `want` records (< 0: all complete ones in the buffer); exact: exactly `want` unless the file ends first.
        Returns (array dict, number of records)."""
        while True:
            if not self.eof and len(self.buf) < self.chunk:
                more = self.f.read(self.chunk - len(self.buf))
                self.eof = not more
                self.buf += more
            try:
                a, used = g.parse_reads_raw(self.buf, self.fmt, self.split, self.eof, want)
            except capi.XmError as e:
                raise SystemExit("%s: %s" % (self.path, e))
            n = int(a["record"][-1]) + 1 if len(a["record"]) else 0
            if n == want or self.eof or (n > 0 and not exact):
                self.buf = self.buf[used:]
                return a, n
            self.chunk *= 2   # a record longer than the buffer, or fewer records than the mate file has in this batch


def query_batches(g, args, batch_reads):
    """Yields (array dict of the batch's sequences in query order, mates adjacent; sequences per query) over all query files."""
    split = args.split_queries_past_size
    for path in args.queries:
        src = Source(path, split)
        while not src.done():
            a, _ = src.take(g, batch_reads)
            if len(a["seq_len"]):
                yield a, 1
    for r1, r2 in args.paired_queries:
        s1, s2 = Source(r1, 0), Source(r2, 0)
        while not s1.done():
            a1, n = s1.take(g, batch_reads)
            if n == 0:
                continue
            a2, n2 = s2.take(g, n, exact=True)
            if n2 != n:
                raise SystemExit("%s has fewer records than %s" % (r2, r1))
            order = np.stack([np.arange(n), np.arange(n) + n], axis=1).reshape(-1)   # mate 1, mate 2 of each query
            yield select(concat([a1, a2]), order), 2
        if s2.take(g, 1)[1]:
            raise SystemExit("%s has more records than %s" % (r2, r1))


def prefetch(gen):
    """Runs the generator one item ahead in a second thread: the next chunk is parsed while the current batch aligns."""
    q = queue.Queue(maxsize=1)
    end = object()

    def run():
        try:
            for item in gen:
                q.put(item)
            q.put(end)
        except BaseException as e:  # noqa: BLE001 - handed to the consumer
            q.put(e)
    threading.Thread(target=run, daemon=True).start()
    while True:
        item = q.get()
        if item is end:
            return
        if isinstance(item, BaseException):
            raise item
        yield item


def load_reference(g, paths):
    """Contigs of all reference files, sorted by descending length (stable), uploaded; returns [(name bytes, length)]."""
    parts = []
    for path in paths:
        src = Source(path, 0)
        if src.fmt != capi.FASTA:
            raise SystemExit("%s: the reference must be FASTA" % path)
        while not src.done():
            a, n = src.take(g)
            if n:
                parts.append(a)
    if not parts:
        raise SystemExit("the reference has no contigs")
    a = concat(parts)
    lens = a["seq_len"].astype(np.int64)
    order = sorted(range(len(lens)), key=lambda i: -lens[i])
    wo, no = a["seq_word_off"], a["name_off"]
    g.set_reference([a["packed"][wo[i]:wo[i + 1]] for i in order], [int(lens[i]) for i in order])
    return [(a["names"][no[i]:no[i + 1]], int(lens[i])) for i in order]


def main(argv=None):
    args = parse_args(sys.argv[1:] if argv is None else argv)
    params = dict(synth.DEFAULT_PARAMS, enable_gapmers=0 if args.no_gapmers else 1)
    paired_model = args.spacing or (0.0, 1.0)   # without --spacing: the library's Query.java defaults
    g = capi.XMapper(params, device=args.device)
    contigs = load_reference(g, args.reference)
    if args.infer_ancestors:
        total, min_dup = sum(n for _, n in contigs), 1
        while (1 << min_dup) < total:   # minDuplicationLength = SequenceDatabase.log2RoundUp(totalForwardSize)
            min_dup += 1
        g.infer_ancestors(params["max_error_rate"] / params["mutation"], min_interesting=min_dup, max_short=8)
        contigs = [(name + b"-anc", n) for name, n in contigs]   # the inferred sequences are named "<name>-anc" (M/Mapper.java:675-681)
    counts = bool(args.out_vcf or args.out_mutations)
    # pre-pass: longest sequence, and the name rank of every sequence
    max_len, names = 1, []
    for a, _ in query_batches(g, args, 1 << 22):
        if len(a["seq_len"]):
            max_len = max(max_len, int(a["seq_len"].max()))
        if counts:
            no, blob = a["name_off"], a["names"]
            names += [blob[no[i]:no[i + 1]] for i in range(len(no) - 1)]
    g.build_index(max_len)
    g.build_duplications(-1, -1, 2, 1000)
    ranks = None
    if counts:
        ranks = np.unique(np.array(names, dtype=object), return_inverse=True)[1].astype(np.int64).reshape(-1)
        g.counts_enable(args.distinguish_query_ends)
    contig_names = (b"".join(n for n, _ in contigs), np.concatenate([[0], np.cumsum([len(n) for n, _ in contigs])]).astype(np.int64))
    sam = open(args.out_sam, "wb") if args.out_sam else None
    if sam:
        sam.write(b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (n, ln) for n, ln in contigs))
    first, n_batches, kernel_ns = 0, 0, 0
    for a, per_query in prefetch(query_batches(g, args, args.batch_reads)):
        n_seq = len(a["seq_len"])
        nq = n_seq // per_query
        batch = dict(packed=a["packed"] if len(a["packed"]) else np.zeros(1, np.uint16), seq_word_off=a["seq_word_off"], seq_len=a["seq_len"],
                     n_seqs=np.full(nq, per_query, dtype=np.uint8),
                     expected_inner=np.full(nq, paired_model[0] if per_query == 2 else 0.0), per_penalty=np.full(nq, paired_model[1] if per_query == 2 else 1.0))
        if counts:
            g.counts_batch_info(first, ranks[first:first + n_seq])
        res, text = g.align_batch_sam(batch, (a["names"], a["name_off"]), contig_names, strict=False)
        bad = np.nonzero(res["q_status"])[0]
        if len(bad):
            s = int(bad[0]) * per_query
            raise SystemExit("query %r could not be aligned on the device (status %d); %d queries of this batch failed" %
                             (a["names"][a["name_off"][s]:a["name_off"][s + 1]].decode(errors="replace"), int(res["q_status"][bad[0]]), len(bad)))
        if sam:
            sam.write(text.encode())
        first += n_seq
        n_batches += 1
        kernel_ns += int(res["stats"][capi.STAT["kernel_ns"]])
    if sam:
        sam.close()
    print("mapper_b200: %d sequences in %d batches, align kernels %.3f s (device time)" % (first, n_batches, kernel_ns / 1e9), file=sys.stderr)
    by_name = sorted(range(len(contigs)), key=lambda c: contigs[c][0])   # TreeMap<String> order of the contig names
    if args.out_vcf:
        upload_examples(g, args)
        with open(args.out_vcf, "wb") as f:
            f.write(b"#CHROM\tPOS\tREF\tALT\tDEPTH\tMIDDLE_COUNTS\tEND_COUNTS\tSUPPORT\n")
            for c in by_name:
                name, ln = contigs[c]
                for s in range(0, ln, VCF_RANGE):
                    f.write(g.format_vcf(c, name, s, min(ln, s + VCF_RANGE)).encode())
    if args.out_mutations:
        with open(args.out_mutations, "wb") as f:
            for c in by_name:
                name, ln = contigs[c]
                for s in range(0, ln, MUTATIONS_RANGE):
                    f.write(g.format_mutations(c, name, s, min(ln, s + MUTATIONS_RANGE), MUTATIONS_FILTER).encode())
    g.close()


def upload_examples(g, args):
    """The reads the VCF support column names, read once more from the inputs (sequence ids are the order of the reads)."""
    gids = g.variants_examples()
    parts, first = [], 0
    for a, _ in query_batches(g, args, 1 << 22):
        n = len(a["seq_len"])
        lo, hi = np.searchsorted(gids, [first, first + n])
        if hi > lo:
            parts.append(select(a, gids[lo:hi] - first))
        first += n
    ex = concat(parts) if parts else dict(packed=np.zeros(0, np.uint16), seq_word_off=np.zeros(1, np.int64), seq_len=np.zeros(0, np.int32))
    g.upload_variant_examples(gids, ex["packed"], ex["seq_word_off"], ex["seq_len"])


if __name__ == "__main__":
    main()
