"""ctypes binding of libxmapper_b200.so (include/xmapper_b200.h).

This is the thin layer a host uses to drive the CUDA aligner stage; it holds no algorithm.  Loading fails loudly
if the shared library has not been built (`python -c "import __graft_entry__ as g; g.build()"`), and xm_create
fails when no CUDA device is visible: there is no CPU fallback anywhere in this package.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("XM_LIB_PATH") or os.path.join(HERE, "libxmapper_b200.so")  # XM_LIB_PATH: build-variant experiments

EXPORTS = ["xm_create", "xm_destroy", "xm_last_error", "xm_set_reference", "xm_set_index_length", "xm_finish_index",
           "xm_set_index_length_wide", "xm_build_index", "xm_get_index_length", "xm_get_index_length_wide", "xm_index_info", "xm_set_duplications", "xm_build_duplications", "xm_build_duplications_host",
           "xm_get_duplications", "xm_infer_ancestors", "xm_get_reference", "xm_align_batch", "xm_align_batch_device", "xm_results_array", "xm_release_results",
           "xm_counts_enable", "xm_counts_device_ptr", "xm_counts_fetch", "xm_format_sam",
           "xm_comm_unique_id", "xm_comm_init", "xm_counts_reduce", "xm_counts_batch_info", "xm_variants_fetch", "xm_measure_peaks", "xm_counts_reduce_times",
           "xm_variants_examples", "xm_variants_set_examples", "xm_format_vcf", "xm_format_mutations",
           "xm_parse_reads", "xm_reads_array", "xm_release_reads", "xm_rank_names"]

RESULT_ARRAYS = [("q_comp_off", np.int64), ("comp_choice_off", np.int64), ("choice_sa_off", np.int64), ("sa_block_off", np.int64),
                 ("choice_f64", np.float64), ("sa_f64", np.float64), ("choice_inner", np.int32), ("sa_contig", np.int32),
                 ("blocks", np.int32), ("q_status", np.int32), ("sa_reversed", np.uint8), ("stats", np.int64), ("q_cycles", np.int64)]
READS_ARRAYS = [("packed", np.uint16), ("seq_word_off", np.int64), ("seq_len", np.int32), ("name_off", np.int64), ("names", np.uint8),
                ("record", np.int64)]
FASTA, FASTQ = 0, 1
STAT = dict(kernel_ns=0, launches=1, tier0=2, tier1=3, tier2=4, probes=5, seeds=6, hits=7, straight=8, path_calls=9,
            path_steps=10, path_cells=11, h2d_bytes=12, d2h_bytes=13, align_kernel_ns=14, tier0_ns=15, tier1_ns=16, tier2_ns=17,
            cyc_seed=18, cyc_straight=19, cyc_hba=20, cyc_path=21, cyc_tables=22, cyc_spare=23, cyc_total=24, easy=25, easy_ns=26, easy_done=27, easy_probes=28, easy_hits=29, easy_straight=30)


class XmParams(C.Structure):
    _fields_ = [("mutation_penalty", C.c_double), ("insertion_start_penalty", C.c_double), ("insertion_extension_penalty", C.c_double),
                ("deletion_start_penalty", C.c_double), ("deletion_extension_penalty", C.c_double), ("max_error_rate", C.c_double),
                ("unaligned_penalty", C.c_double), ("ambiguity_penalty", C.c_double), ("max_penalty_span", C.c_double),
                ("max_num_matches", C.c_int32), ("enable_gapmers", C.c_int32)]


class XmVariantFilter(C.Structure):
    _fields_ = [("min_snp_total_depth", C.c_float), ("min_snp_depth_fraction", C.c_float),
                ("min_indel_start_total_depth", C.c_float), ("min_indel_start_depth_fraction", C.c_float),
                ("min_indel_continuation_total_depth", C.c_float), ("min_indel_continuation_depth_fraction", C.c_float)]


# MutationDetectionParameters field names -> xm_variant_filter fields
FILTER_FIELDS = dict(minSNPTotalDepth="min_snp_total_depth", minSNPDepthFraction="min_snp_depth_fraction",
                     minIndelTotalStartDepth="min_indel_start_total_depth", minIndelStartDepthFraction="min_indel_start_depth_fraction",
                     minIndelContinuationTotalDepth="min_indel_continuation_total_depth",
                     minIndelContinuationDepthFraction="min_indel_continuation_depth_fraction")


def to_xm_filter(flt):
    """flt: None (the empty filter) or a dict keyed by FILTER_FIELDS' names (missing thresholds are 0)."""
    f = XmVariantFilter()
    for k, v in (flt or {}).items():
        if k not in FILTER_FIELDS:
            raise ValueError("unknown filter threshold %r (expected one of %s)" % (k, ", ".join(FILTER_FIELDS)))
        setattr(f, FILTER_FIELDS[k], float(v))
    return f


_LIB = None


def load_library():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libxmapper_b200.so is not built (%s missing). Build it with __graft_entry__.build(); "
                               "there is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.xm_last_error.restype = C.c_char_p
        L.xm_results_array.restype = C.c_int64
        L.xm_reads_array.restype = C.c_int64
        _LIB = L
    return _LIB


def to_xm_params(d):
    p = XmParams()
    p.mutation_penalty = d["mutation"]
    p.insertion_start_penalty = d["ins_start"]
    p.insertion_extension_penalty = d["ins_ext"]
    p.deletion_start_penalty = d["del_start"]
    p.deletion_extension_penalty = d["del_ext"]
    p.max_error_rate = d["max_error_rate"]
    p.unaligned_penalty = d["unaligned"]
    p.ambiguity_penalty = d["ambiguity"]
    p.max_penalty_span = d["max_penalty_span"]
    p.max_num_matches = int(d.get("max_num_matches", 2147483647))
    p.enable_gapmers = int(d.get("enable_gapmers", 1))
    return p


class XmError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _bytes(s):
    return s if isinstance(s, bytes) else s.encode()


class _ResultOwner:
    """Keeps an xm_results alive while zero-copy views of its arrays are in use."""

    def __init__(self, lib, r):
        self.lib, self.r = lib, r

    def __del__(self):
        if self.r is not None:
            self.lib.xm_release_results(self.r)
            self.r = None


class XMapper:
    """One xm_handle: the aligner stage of one GPU."""

    def __init__(self, params, device=0):
        self.L = load_library()
        self.h = C.c_void_p()
        p = to_xm_params(params)
        rc = self.L.xm_create(C.byref(p), int(device), C.byref(self.h))
        if rc != 0:
            self.h = None
            raise XmError("xm_create failed with status %d (no CUDA device? this library has no CPU path)" % rc)
        self._keep = []

    def _ok(self, rc, allow=()):
        if rc != 0 and rc not in allow:
            raise XmError("status %d: %s" % (rc, self.L.xm_last_error(self.h).decode()))
        return rc

    def close(self):
        if self.h:
            self.L.xm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- reference / index / duplications ----
    def set_reference(self, packed_contigs, lengths):
        n = len(packed_contigs)
        packed_contigs = [np.ascontiguousarray(p, dtype=np.uint16) for p in packed_contigs]
        arr = (C.c_void_p * n)(*[p.ctypes.data for p in packed_contigs])
        lens = np.asarray(lengths, dtype=np.int32)
        self._keep = [packed_contigs, lens]
        self._ok(self.L.xm_set_reference(self.h, n, arr, _ptr(lens)))
        self.contig_lengths = [int(x) for x in lens]

    def set_reference_from_codes(self, contigs):
        """contigs: list of uint8 code arrays (or of (name, codes) pairs), in database order."""
        codes = [c[1] if isinstance(c, tuple) else c for c in contigs]
        from mapper_b200 import synth
        self.set_reference([synth.pack_contig(c) for c in codes], [len(c) for c in codes])

    def infer_ancestors(self, threshold, min_interesting=-1, max_short=-1, verify=False):
        """xm_infer_ancestors: replaces the reference by its "-anc" reference (the index and duplication table are discarded);
        returns the number of forward positions whose code changed."""
        n = C.c_int64()
        self._ok(self.L.xm_infer_ancestors(self.h, C.c_double(threshold), int(min_interesting), int(max_short), int(bool(verify)), C.byref(n)))
        return n.value

    def get_reference(self, contig):
        """Codes (uint8, one per base) of forward contig `contig` as the handle holds it now."""
        n = self.contig_lengths[contig]
        out = np.zeros(max((n + 3) // 4, 1), dtype=np.uint16)
        self._ok(self.L.xm_get_reference(self.h, int(contig), _ptr(out)))
        return np.stack([out & 15, (out >> 4) & 15, (out >> 8) & 15, (out >> 12) & 15], axis=1).reshape(-1)[:n].astype(np.uint8)

    def set_index_length(self, t, wide=False):
        """wide: positions are uint64 (xm_set_index_length_wide; required when 2 x the reference size exceeds 2^32)."""
        off = np.ascontiguousarray(t["offsets"], dtype=np.int64)
        over = np.ascontiguousarray(t["overfull"], dtype=np.uint8)
        pos = np.ascontiguousarray(t["positions"], dtype=np.uint64 if wide else np.uint32)
        if len(pos) == 0:
            pos = np.zeros(1, dtype=pos.dtype)
        f = self.L.xm_set_index_length_wide if wide else self.L.xm_set_index_length
        self._ok(f(self.h, int(t["used"]), int(t["capacity"]), int(t["max_count"]), _ptr(off), _ptr(over), _ptr(pos)))

    def finish_index(self, min_interesting, max_built):
        self._ok(self.L.xm_finish_index(self.h, int(min_interesting), int(max_built)))

    def build_index(self, max_used, threads=0):
        """threads == 0: the device builder; threads > 0: the library's host builder (kept as its cross-check)."""
        self._ok(self.L.xm_build_index(self.h, int(max_used), int(threads)))

    def index_info(self):
        a, b = C.c_int32(), C.c_int32()
        self._ok(self.L.xm_index_info(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def get_index_length(self, n, wide=False):
        cap, mx, npos = C.c_int32(), C.c_int32(), C.c_int64()
        self._ok(self.L.xm_get_index_length(self.h, n, C.byref(cap), C.byref(mx), C.byref(npos), None, None, None))
        off = np.zeros(cap.value + 1, dtype=np.int64)
        over = np.zeros(cap.value, dtype=np.uint8)
        pos = np.zeros(max(npos.value, 1), dtype=np.uint64 if wide else np.uint32)
        f = self.L.xm_get_index_length_wide if wide else self.L.xm_get_index_length
        self._ok(f(self.h, n, C.byref(cap), C.byref(mx), C.byref(npos), _ptr(off), _ptr(over), _ptr(pos)))
        return dict(used=n, capacity=cap.value, max_count=mx.value, offsets=off, overfull=over, positions=pos[:npos.value])

    def index_length_size(self, n):
        """(capacity, number of positions) of the table for numBasepairsUsed == n, without copying it."""
        cap, mx, npos = C.c_int32(), C.c_int32(), C.c_int64()
        self._ok(self.L.xm_get_index_length(self.h, n, C.byref(cap), C.byref(mx), C.byref(npos), None, None, None))
        return cap.value, npos.value

    def set_duplications(self, window, granularity, contig, starts):
        s = np.ascontiguousarray(starts, dtype=np.int32)
        n = len(s)
        if n == 0:
            s = np.zeros(1, dtype=np.int32)
        self._ok(self.L.xm_set_duplications(self.h, int(window), C.c_double(granularity), int(contig), n, _ptr(s)))

    def build_duplications(self, min_len=-1, max_len=-1, min_copies=2, window=1000, host=False):
        """host=False: bucket scan on the device; host=True: the library's host-thread detector (its cross-check)."""
        f = self.L.xm_build_duplications_host if host else self.L.xm_build_duplications
        self._ok(f(self.h, min_len, max_len, min_copies, window))

    def get_duplications(self, contig):
        n = C.c_int32()
        self._ok(self.L.xm_get_duplications(self.h, contig, C.byref(n), None))
        out = np.zeros(max(n.value, 1), dtype=np.int32)
        self._ok(self.L.xm_get_duplications(self.h, contig, C.byref(n), _ptr(out)))
        return out[:n.value]

    # ---- alignment ----
    def _take(self, r, copy=True):
        """copy=False: the arrays are views into the library's pinned result slab (what a JNI/FFM host maps as direct
        buffers); they stay valid while the returned dict's "_owner" is alive."""
        out = {}
        for i, (name, dt) in enumerate(RESULT_ARRAYS):
            ptr = C.c_void_p()
            n = self.L.xm_results_array(r, i, C.byref(ptr))
            if n > 0:
                v = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(n * np.dtype(dt).itemsize,)).view(dt)
                out[name] = v.copy() if copy else v
            else:
                out[name] = np.zeros(0, dtype=dt)
        if copy:
            self.L.xm_release_results(r)
        else:
            out["_owner"] = _ResultOwner(self.L, r)
        return out

    def align_batch(self, batch, strict=False, copy=True, **_):
        """batch: dict(packed uint16, seq_word_off int64, seq_len int32, n_seqs uint8, expected_inner f64, per_penalty f64) in HOST memory."""
        nq = len(batch["n_seqs"])
        r = C.c_void_p()
        rc = self.L.xm_align_batch(self.h, nq, _ptr(batch["packed"]), _ptr(batch["seq_word_off"]), _ptr(batch["seq_len"]), _ptr(batch["n_seqs"]),
                                   _ptr(batch["expected_inner"]), _ptr(batch["per_penalty"]), C.byref(r))
        self._ok(rc, allow=() if strict else (-4,))
        return self._take(r, copy)

    def align_batch_sam(self, batch, seq_names, contig_names, strict=False):
        """Aligns a host batch and returns (results, SAM text): the text is formatted on the device (xm_format_sam) from the result
        arrays while they are still resident.  seq_names: one name per sequence (mate) of the batch; contig_names: xm_set_reference order."""
        nq = len(batch["n_seqs"])
        r = C.c_void_p()
        rc = self.L.xm_align_batch(self.h, nq, _ptr(batch["packed"]), _ptr(batch["seq_word_off"]), _ptr(batch["seq_len"]), _ptr(batch["n_seqs"]),
                                   _ptr(batch["expected_inner"]), _ptr(batch["per_penalty"]), C.byref(r))
        self._ok(rc, allow=() if strict else (-4,))
        try:
            sam = self.format_sam(r, seq_names, contig_names)
        finally:
            out = self._take(r, True)
        return out, sam

    def format_sam(self, r, seq_names, contig_names):
        """seq_names / contig_names: lists of str, or (bytes, int64 offsets) pairs as parse_reads_raw returns them."""
        def blob(names):
            if isinstance(names, tuple):
                return bytes(names[0]) + b"\0", np.ascontiguousarray(names[1], dtype=np.int64)
            enc = [n.encode() for n in names]
            off = np.zeros(len(enc) + 1, dtype=np.int64)
            if enc:
                off[1:] = np.cumsum([len(e) for e in enc])
            return b"".join(enc) + b"\0", off
        sb, so = blob(seq_names)
        cb, co = blob(contig_names)
        text, n = C.c_char_p(), C.c_int64()
        self._ok(self.L.xm_format_sam(self.h, r, sb, _ptr(so), cb, _ptr(co), C.byref(text), C.byref(n)))
        return C.string_at(text, n.value).decode()

    def align_batch_device(self, nq, d_packed, n_words, d_seq_word_off, d_seq_len, d_n_seqs, d_expected, d_per, max_seq_len, strict=False, copy=True):
        """All arguments are device pointers (ints) on this handle's GPU."""
        r = C.c_void_p()
        rc = self.L.xm_align_batch_device(self.h, int(nq), C.c_void_p(d_packed), C.c_int64(n_words), C.c_void_p(d_seq_word_off), C.c_void_p(d_seq_len),
                                          C.c_void_p(d_n_seqs), C.c_void_p(d_expected), C.c_void_p(d_per), int(max_seq_len), C.byref(r))
        self._ok(rc, allow=() if strict else (-4,))
        return self._take(r, copy)

    # ---- read ingestion ----
    def parse_reads_raw(self, text, fmt, split_size=0, at_eof=True, max_records=-1):
        """xm_parse_reads over bytes `text` (fmt: FASTA or FASTQ): (dict of the arrays of enum xm_reads_array, copied; "names" is
        bytes), n_consumed."""
        r, n_consumed = C.c_void_p(), C.c_int64()
        self._ok(self.L.xm_parse_reads(self.h, int(fmt), text, C.c_int64(len(text)), int(bool(at_eof)), C.c_int64(max_records), int(split_size),
                                       C.byref(r), C.byref(n_consumed)))
        out = {}
        try:
            for i, (name, dt) in enumerate(READS_ARRAYS):
                ptr = C.c_void_p()
                n = self.L.xm_reads_array(r, i, C.byref(ptr))
                nb = n * np.dtype(dt).itemsize
                out[name] = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(nb,)).view(dt).copy() if nb else np.zeros(0, dtype=dt)
        finally:
            self.L.xm_release_reads(r)
        out["names"] = out["names"].tobytes()
        return out, n_consumed.value

    def parse_reads(self, text, fmt, split_size=0, at_eof=True, max_records=-1):
        """FASTA / FASTQ text parsed on the device.  Returns (batch of single-sequence queries in the shape align_batch takes, names as a
        list of str, record index per sequence, n_consumed)."""
        a, n_consumed = self.parse_reads_raw(text, fmt, split_size, at_eof, max_records)
        n = len(a["seq_len"])
        packed = a["packed"] if len(a["packed"]) else np.zeros(1, dtype=np.uint16)
        batch = dict(packed=packed, seq_word_off=a["seq_word_off"], seq_len=a["seq_len"], n_seqs=np.ones(n, dtype=np.uint8),
                     expected_inner=np.zeros(n, dtype=np.float64), per_penalty=np.ones(n, dtype=np.float64))
        off, blob = a["name_off"], a["names"]
        names = [blob[off[i]:off[i + 1]].decode("utf-8", "surrogateescape") for i in range(n)]
        return batch, names, a["record"], n_consumed

    def rank_names(self, names, name_off):
        """xm_rank_names: int64 ranks of the names names[name_off[i]:name_off[i + 1]] (bytes, or a uint8 array) in unsigned byte order,
        equal names ranked equal: np.unique(names, return_inverse=True)[1], computed on the device."""
        off = np.ascontiguousarray(name_off, dtype=np.int64)
        if off.ndim != 1 or len(off) < 1:
            raise ValueError("name_off needs n + 1 entries")
        blob = np.frombuffer(names, dtype=np.uint8) if isinstance(names, (bytes, bytearray)) else np.ascontiguousarray(names, dtype=np.uint8)
        out = np.zeros(len(off) - 1, dtype=np.int64)
        self._ok(self.L.xm_rank_names(self.h, C.c_int64(len(off) - 1), _ptr(blob), _ptr(off), _ptr(out)))
        return out

    # ---- per-position counts ----
    def counts_enable(self, query_end_fraction=0.1):
        self._ok(self.L.xm_counts_enable(self.h, C.c_double(query_end_fraction)))

    def counts_batch_info(self, first_sequence_id, order_keys=None):
        """Before align_batch: global id of the batch's first sequence and (optionally) a name-order key per sequence."""
        if order_keys is None:
            self._ok(self.L.xm_counts_batch_info(self.h, C.c_int64(first_sequence_id), None, C.c_int64(0)))
        else:
            k = np.ascontiguousarray(order_keys, dtype=np.int64)
            self._ok(self.L.xm_counts_batch_info(self.h, C.c_int64(first_sequence_id), _ptr(k), C.c_int64(len(k))))

    def variants_count(self):
        """Reduces the variant records accumulated so far (device sort + reduce-by-key) and returns the number of table entries."""
        n = C.c_int64()
        self._ok(self.L.xm_variants_fetch(self.h, C.byref(n), None, None, None, None))
        return n.value

    def variants_fetch(self):
        """The sparse variant table, decoded: dict of arrays gpos, region, dir, ins (-1: at the position), allele, count, ex_gid, ex_rev, ex_index."""
        n = C.c_int64()
        self._ok(self.L.xm_variants_fetch(self.h, C.byref(n), None, None, None, None))
        m = max(n.value, 1)
        keys, counts, gid, idx = np.zeros(m, np.uint64), np.zeros(m, np.int32), np.zeros(m, np.int64), np.zeros(m, np.int32)
        self._ok(self.L.xm_variants_fetch(self.h, C.byref(n), _ptr(keys), _ptr(counts), _ptr(gid), _ptr(idx)))
        keys, counts, gid, idx = keys[:n.value], counts[:n.value], gid[:n.value], idx[:n.value]
        return dict(key=keys, gpos=(keys >> np.uint64(21)).astype(np.int64), region=((keys >> np.uint64(20)) & np.uint64(1)).astype(np.int32),
                    dir=((keys >> np.uint64(19)) & np.uint64(1)).astype(np.int32), ins=((keys >> np.uint64(3)) & np.uint64(0xFFFF)).astype(np.int32) - 1,
                    allele=(keys & np.uint64(7)).astype(np.int32), count=counts, ex_gid=gid >> 1, ex_rev=(gid & 1).astype(np.int32), ex_index=idx)

    def measure_peaks(self):
        """Issue-rate micro-benchmarks (warp-instructions/s over the chip): dict(int32, fp64, alu, sm_count, sm_clock_hz)."""
        out = (C.c_double * 5)()
        self._ok(self.L.xm_measure_peaks(self.h, out))
        return dict(int32=out[0], fp64=out[1], alu=out[2], sm_count=int(out[3]), sm_clock_hz=out[4])

    def counts_device_ptr(self):
        p, n = C.c_void_p(), C.c_int64()
        self._ok(self.L.xm_counts_device_ptr(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def comm_unique_id(self):
        buf = (C.c_uint8 * 128)()
        rc = self.L.xm_comm_unique_id(buf)
        if rc != 0:
            raise XmError("xm_comm_unique_id: status %d (libnccl not loadable?)" % rc)
        return bytes(buf)

    def comm_init(self, n_ranks, rank, unique_id):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._ok(self.L.xm_comm_init(self.h, int(n_ranks), int(rank), buf))

    def counts_reduce(self):
        self._ok(self.L.xm_counts_reduce(self.h))

    def counts_reduce_times(self):
        a, b = C.c_double(), C.c_double()
        self._ok(self.L.xm_counts_reduce_times(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def counts_fetch(self, contig):
        out = np.zeros(4 * self.contig_lengths[contig], dtype=np.int32)
        self._ok(self.L.xm_counts_fetch(self.h, contig, _ptr(out)))
        return out.reshape(2, 2, -1)

    # ---- VCF / mutations bodies ----
    def variants_examples(self):
        """The global sequence ids (ascending) whose reads the VCF support column of the current variant table can show."""
        n = C.c_int64()
        self._ok(self.L.xm_variants_examples(self.h, C.byref(n), None))
        out = np.zeros(max(n.value, 1), dtype=np.int64)
        self._ok(self.L.xm_variants_examples(self.h, C.byref(n), _ptr(out)))
        return out[:n.value]

    def set_variant_examples(self, codes_by_gid):
        """Uploads the forward reads of variants_examples(): codes_by_gid maps a global sequence id to its uint8 codes."""
        from mapper_b200 import synth
        gids = self.variants_examples()
        packed = [synth.pack_contig(np.asarray(codes_by_gid[int(g)], dtype=np.uint8)) for g in gids]
        lens = np.array([len(codes_by_gid[int(g)]) for g in gids], dtype=np.int32)
        off = np.zeros(len(gids) + 1, dtype=np.int64)
        if len(gids):
            off[1:] = np.cumsum([len(p) for p in packed])
        self.upload_variant_examples(gids, np.concatenate(packed + [np.zeros(0, dtype=np.uint16)]), off, lens)

    def upload_variant_examples(self, gids, packed, seq_word_off, seq_len):
        """xm_variants_set_examples with the reads already packed (gids as variants_examples() lists them)."""
        words = np.concatenate([np.asarray(packed, dtype=np.uint16), np.zeros(1, dtype=np.uint16)])
        self._ok(self.L.xm_variants_set_examples(self.h, C.c_int64(len(gids)), _ptr(np.ascontiguousarray(gids, dtype=np.int64)), _ptr(words),
                                                 _ptr(np.ascontiguousarray(seq_word_off, dtype=np.int64)), _ptr(np.ascontiguousarray(seq_len, dtype=np.int32))))

    def format_vcf(self, contig, name, start, end, flt=None, include_non_mutations=True, show_support=True):
        """VCF body lines of positions [start, end) of contig `contig` named `name` (str or bytes); flt: dict of MutationDetectionParameters
        thresholds or None."""
        f = to_xm_filter(flt)
        text, n = C.c_char_p(), C.c_int64()
        self._ok(self.L.xm_format_vcf(self.h, int(contig), _bytes(name), C.c_int64(start), C.c_int64(end), C.byref(f), int(bool(include_non_mutations)),
                                      int(bool(show_support)), C.byref(text), C.byref(n)))
        return C.string_at(text, n.value).decode()

    def format_mutations(self, contig, name, start, end, flt=None):
        """Mutations body lines of [start, end) of contig `contig` (start and end on the 8192 grid, or end = the contig length)."""
        f = to_xm_filter(flt)
        text, n = C.c_char_p(), C.c_int64()
        self._ok(self.L.xm_format_mutations(self.h, int(contig), _bytes(name), C.c_int64(start), C.c_int64(end), C.byref(f), C.byref(text), C.byref(n)))
        return C.string_at(text, n.value).decode()
