"""python -m mapper_b200: map FASTA/FASTQ reads against a FASTA reference on one or more GPUs and write SAM, VCF and mutations files.

The front end of X-Mapper's Mapper.run (SURVEY.md §3.1), driving the C ABI; it holds no algorithm.  --device takes one CUDA ordinal or a
comma list of them: one handle per device, every handle holding the same reference, index and duplication table.
  1. Reference: parsed on the first device (xm_parse_reads), contigs sorted as Mapper.sortAndComplementReference sorts them (descending
     length, ties in input order) and given to every handle (xm_set_reference).  --infer-ancestors (set up as M/Mapper.java:666-692) runs
     on the first device, whose "-anc" contigs go to the others (xm_get_reference -> xm_set_reference).  xm_build_index(longest query or
     split piece) and xm_build_duplications(-1, -1, 2, 1000) run on all devices at once.
  2. A pre-pass over the queries: the longest sequence for the index and, when counts are written, the rank of every sequence name in
     byte order (String.compareTo for ASCII names), the name order DirectionalAlignments.betterExample breaks example ties with.  The
     names are ranked on the first device (xm_rank_names).
  3. Batches, in file order: parsed on the first device while earlier batches align (a second thread), then batch k goes to device
     k mod N.  Each device's worker thread runs xm_counts_batch_info, xm_align_batch and xm_format_sam (the slot rule of INTEGRATION.md
     §1); the SAM text is written in batch order.  A query the device could not align is an error naming the read, never a silent drop.
  4. After the last batch, with several devices: the count planes and variant tables are reduced over all of them (xm_comm_init,
     xm_counts_reduce over NCCL), so the first handle holds the whole table.  Then the example reads of the VCF support column are read
     again from the inputs and uploaded, and the VCF and mutations bodies are formatted on the first device per contig, in name order
     (VcfWriter.java:111-114).

Headers are this command's own: the reference's header texts are not in this repository and embed the command line (BASELINE.md §5),
so SAM gets @SQ lines in database order, the VCF a #CHROM column line, and the mutations file none.  Parity with the reference is for the
bodies.  The output does not depend on the number of devices.  Files ending in .gz are read through gzip on the host.  Every reference
flag this command does not implement exits with status 2 and names the flag.
"""
import argparse
import gzip
import queue
import sys
import threading
import time

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
    p.add_argument("--device", type=device_list, default=[0], metavar="N[,M...]", help="CUDA device, or a comma list of distinct devices")
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


def device_list(text):
    """--device: "N" or "N,M,...", distinct non-negative ordinals."""
    try:
        devs = [int(x) for x in text.split(",")]
    except ValueError:
        raise argparse.ArgumentTypeError("expected N or a comma list N,M,... of CUDA devices, got %r" % text) from None
    if any(d < 0 for d in devs) or len(set(devs)) != len(devs):
        raise argparse.ArgumentTypeError("devices must be distinct and non-negative, got %r" % text)
    return devs


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
    """Runs the generator one item ahead in a second thread: the next chunk is parsed while the current batches align.  Closing the
    returned generator early stops that thread and joins it."""
    q = queue.Queue(maxsize=1)
    end, stop = object(), threading.Event()

    def run():
        try:
            for item in gen:
                if stop.is_set():
                    return
                q.put(item)
            q.put(end)
        except BaseException as e:  # noqa: BLE001 - handed to the consumer
            q.put(e)
    t = threading.Thread(target=run, daemon=True)
    t.start()
    try:
        while True:
            item = q.get()
            if item is end:
                return
            if isinstance(item, BaseException):
                raise item
            yield item
    finally:
        stop.set()
        while t.is_alive():   # a put the producer may be blocked in
            try:
                q.get(timeout=0.05)
            except queue.Empty:
                pass
        t.join()


def on_all(handles, fn):
    """fn(rank, handle) for every handle at once, one thread each; all threads are joined, then the first error is raised."""
    errors = [None] * len(handles)

    def run(d):
        try:
            fn(d, handles[d])
        except BaseException as e:  # noqa: BLE001 - raised below, after the join
            errors[d] = e
    threads = [threading.Thread(target=run, args=(d,)) for d in range(len(handles))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in errors:
        if e is not None:
            raise e


def read_reference(g, paths):
    """Contigs of all reference files parsed on g, sorted by descending length (stable): (packed contigs, lengths, names)."""
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
    return ([a["packed"][wo[i]:wo[i + 1]] for i in order], [int(lens[i]) for i in order], [a["names"][no[i]:no[i + 1]] for i in order])


def align_one(g, first, a, per_query, ranks, paired_model, contig_names):
    """One batch on handle g: returns (SAM text, align kernel ns).  first: global id of the batch's first sequence."""
    n_seq = len(a["seq_len"])
    nq = n_seq // per_query
    batch = dict(packed=a["packed"] if len(a["packed"]) else np.zeros(1, np.uint16), seq_word_off=a["seq_word_off"], seq_len=a["seq_len"],
                 n_seqs=np.full(nq, per_query, dtype=np.uint8),
                 expected_inner=np.full(nq, paired_model[0] if per_query == 2 else 0.0), per_penalty=np.full(nq, paired_model[1] if per_query == 2 else 1.0))
    if ranks is not None:
        g.counts_batch_info(first, ranks[first:first + n_seq])
    res, text = g.align_batch_sam(batch, (a["names"], a["name_off"]), contig_names, strict=False)
    bad = np.nonzero(res["q_status"])[0]
    if len(bad):
        s = int(bad[0]) * per_query
        raise SystemExit("query %r could not be aligned on the device (status %d); %d queries of this batch failed" %
                         (a["names"][a["name_off"][s]:a["name_off"][s + 1]].decode(errors="replace"), int(res["q_status"][bad[0]]), len(bad)))
    return text, int(res["stats"][capi.STAT["kernel_ns"]])


def map_batches(handles, batches, ranks, paired_model, contig_names, write, reduce=False):
    """Aligns `batches` ((array dict, sequences per query) in file order): batch k on handles[k % N], in one worker thread per handle,
    with the global id of its first sequence and, when ranks is given, its sequences' name ranks (xm_counts_batch_info).  write() gets
    the SAM text of every batch, in batch order.  reduce: after the last batch, once every worker has finished without error, the
    counts of all handles are reduced (xm_comm_init + xm_counts_reduce, collectives entered by one thread per handle).
    An error in `batches` or in a worker stops the dispatch; every thread is joined before the error of the earliest batch is raised.
    Returns (sequences, batches, align kernel ns per handle, reduce wall seconds)."""
    n_dev = len(handles)
    inbox = [queue.Queue(maxsize=2) for _ in handles]
    done = queue.Queue()
    failed = threading.Event()
    kernel_ns = [0] * n_dev

    def worker(d):
        while True:
            job = inbox[d].get()
            if job is None:
                return
            if failed.is_set():
                continue   # drained, so that the dispatcher never blocks on a stopped worker
            k, first, a, per_query = job
            try:
                text, ns = align_one(handles[d], first, a, per_query, ranks, paired_model, contig_names)
                kernel_ns[d] += ns
                done.put((k, text, None))
            except BaseException as e:  # noqa: BLE001 - raised by the dispatcher
                failed.set()
                done.put((k, None, e))

    threads = [threading.Thread(target=worker, args=(d,)) for d in range(n_dev)]
    for t in threads:
        t.start()
    ready, errors = {}, []
    n_out = n_batches = first = 0

    def flush():   # results that have arrived, written in batch order up to the first error
        nonlocal n_out
        while True:
            try:
                k, text, e = done.get_nowait()
            except queue.Empty:
                return
            if e is not None:
                errors.append((k, e))
            ready[k] = text
            while n_out in ready and not errors:
                write(ready.pop(n_out))
                n_out += 1

    try:
        for a, per_query in batches:
            if failed.is_set():
                break
            inbox[n_batches % n_dev].put((n_batches, first, a, per_query))
            first += len(a["seq_len"])
            n_batches += 1
            flush()
    except BaseException as e:  # noqa: BLE001 - raised below, after every thread has been joined
        errors.append((n_batches, e))
    finally:
        close = getattr(batches, "close", None)
        if close:
            close()
        for q in inbox:
            q.put(None)
        for t in threads:
            t.join()
    flush()
    if errors:
        raise min(errors, key=lambda x: x[0])[1]
    reduce_s = 0.0
    if reduce:
        t0 = time.perf_counter()
        uid = handles[0].comm_unique_id()
        on_all(handles, lambda d, g: (g.comm_init(n_dev, d, uid), g.counts_reduce()))
        reduce_s = time.perf_counter() - t0
    return first, n_batches, kernel_ns, reduce_s


def main(argv=None):
    args = parse_args(sys.argv[1:] if argv is None else argv)
    params = dict(synth.DEFAULT_PARAMS, enable_gapmers=0 if args.no_gapmers else 1)
    paired_model = args.spacing or (0.0, 1.0)   # without --spacing: the library's Query.java defaults
    t0 = time.perf_counter()
    handles = []
    try:
        for dev in args.device:
            handles.append(capi.XMapper(params, device=dev))
        map_files(args, params, paired_model, handles, t0)
    finally:
        for g in handles:
            g.close()


def map_files(args, params, paired_model, handles, t0):
    g = handles[0]
    packed, lens, names = read_reference(g, args.reference)
    on_all(handles, lambda d, h: h.set_reference(packed, lens))
    if args.infer_ancestors:
        total, min_dup = sum(lens), 1
        while (1 << min_dup) < total:   # minDuplicationLength = SequenceDatabase.log2RoundUp(totalForwardSize)
            min_dup += 1
        g.infer_ancestors(params["max_error_rate"] / params["mutation"], min_interesting=min_dup, max_short=8)
        names = [name + b"-anc" for name in names]   # the inferred sequences are named "<name>-anc" (M/Mapper.java:675-681)
        if len(handles) > 1:
            anc = [synth.pack_contig(g.get_reference(c)) for c in range(len(lens))]
            on_all(handles[1:], lambda d, h: h.set_reference(anc, lens))
    contigs = list(zip(names, lens))
    counts = bool(args.out_vcf or args.out_mutations)
    t_setup = time.perf_counter()
    # pre-pass: longest sequence, and the name rank of every sequence
    max_len, blobs, offs, n_name_bytes = 1, [], [], 0
    for a, _ in query_batches(g, args, 1 << 22):
        if len(a["seq_len"]):
            max_len = max(max_len, int(a["seq_len"].max()))
        if counts:
            blobs.append(a["names"])
            offs.append(a["name_off"][1:] + n_name_bytes)
            n_name_bytes += len(a["names"])
    ranks = g.rank_names(b"".join(blobs), np.concatenate([np.zeros(1, np.int64)] + offs)) if counts else None
    del blobs, offs
    t_prepass = time.perf_counter()

    def build(d, h):
        h.build_index(max_len)
        h.build_duplications(-1, -1, 2, 1000)
        if counts:
            h.counts_enable(args.distinguish_query_ends)
    on_all(handles, build)
    t_index = time.perf_counter()
    contig_names = (b"".join(n for n, _ in contigs), np.concatenate([[0], np.cumsum([len(n) for n, _ in contigs])]).astype(np.int64))
    sam = open(args.out_sam, "wb") if args.out_sam else None
    try:
        if sam:
            sam.write(b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (n, ln) for n, ln in contigs))
        write = (lambda text: sam.write(text.encode())) if sam else (lambda text: None)
        n_seq, n_batches, kernel_ns, reduce_s = map_batches(handles, prefetch(query_batches(g, args, args.batch_reads)), ranks, paired_model,
                                                            contig_names, write, reduce=counts and len(handles) > 1)
    finally:
        if sam:
            sam.close()
    t_map = time.perf_counter()
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
    t_end = time.perf_counter()
    print("mapper_b200: %d sequences in %d batches on %d device%s, align kernels %.3f s (device time; per device %s)" %
          (n_seq, n_batches, len(handles), "s" if len(handles) > 1 else "", sum(kernel_ns) / 1e9, " ".join("%.3f" % (k / 1e9) for k in kernel_ns)),
          file=sys.stderr)
    print("mapper_b200: wall s: set-up %.3f, pre-pass %.3f, index %.3f, mapping %.3f, reduce %.3f, formatting %.3f" %
          (t_setup - t0, t_prepass - t_setup, t_index - t_prepass, t_map - t_index - reduce_s, reduce_s, t_end - t_map), file=sys.stderr)


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
