// xmapper_b200 — VCF and mutations bodies on the device (SURVEY.md §8 row f1, from the count tables to the text).
// Included by xm_capi.cu after xm_counts.cuh.
//
// The specification is tests/variants_oracle.py, followed statement by statement: Store.position / Store.insertion (QV/Alignments,
// AlignmentsSection, RegionAlignments, DirectionalAlignments :98-160), FilteredAlignments (f_position, _could_be_deletion, f_insertion),
// QV/MutationsFormatterWorker.java:25-147 and QV/VcfFormatterWorker.java:27-159.  Every count is a Java float built from the int32
// units of 1/100 in the oracle's addition order (the library builds with -fmad=false; no comparison leaves float).
//
// One call formats positions [start, end) of one forward contig:
//   xm_fmt_carry_kernel   one block: the table entries of the range (two binary searches) and the carry-in of _could_be_deletion, a
//                         left walk from start - 1 to the first decisive position (or the contig start) in steps of one block;
//   xm_fmt_decide_kernel  per position: supports_indel_start -> true, else !supports_indel_continuation -> false, else "undecided";
//   cub inclusive scan    "last decisive value wins" gives _could_be_deletion of every position of the range;
//   xm_fmt_kernel<MODE, false>  per position: bytes of its text; exclusive scan; xm_fmt_kernel<MODE, true> writes them.
// A thread finds its position's entries by a binary search inside the range's entries: no per-position index array and no extra
// pass, and the threads of a warp follow nearly the same search path, so the loads hit in cache.
#pragma once
#include "xm_text.cuh"

struct VarFilter { float snp_total, snp_frac, start_total, start_frac, cont_total, cont_frac; };   // xm_variant_filter
enum { XM_FMT_VCF = 0, XM_FMT_MUT = 1 };
static const int XM_FMT_JOB = 8192;   // MutationsWriter's job length: deletion runs are flushed at its boundaries

struct FmtD {
  RefD ref;
  const int32_t* planes; const int64_t* contig_off;
  const VarRec* recs; unsigned long long n_recs;
  unsigned long long* range;          // [2]: entries [lo, hi) of the positions [start, end) (xm_fmt_carry_kernel)
  int contig; long long start, end;
  VarFilter f;
  const char* name; int name_len;
  int include_non_mutations, show_support;
  uint8_t* dec;                       // [n + 1]: dec[0] carry-in, dec[1 + t] position start + t (0 undecided, 1 false, 2 true)
  const uint8_t* could_delete;        // [n + 1]: the inclusive scan of dec
  long long* len;                     // [n + 1]: bytes per position, then exclusive offsets
  char* text;
  const int32_t* ex_slot;             // per table entry: its example in the uploaded list
  const uint16_t* ex_words; const int64_t* ex_word_off; const int32_t* ex_len;
};

__device__ __constant__ const char XM_KEYS[7] = "ACGTN-";   // AlignmentPosition_DirectionCounts.makeKeys
__device__ __constant__ const char XM_LETTERS[17] = "-ACMGRSVTWYHKDBN";

__device__ __forceinline__ float fmt_units(int32_t s) { return (float)s / 100.0f; }

// AlignmentPosition: containers [direction: 0 forward, 1 reverse][region: 0 middle, 1 end] of scaled counts; sample[k] = the table
// entry whose example is shown for KEYS[k], -1: none
struct FmtPos {
  char ref_char;
  int32_t ref[2][2], ign[2][2], cnt[2][2][6];
  long long sample[6];
  __device__ void init(char rc) {
    ref_char = rc;
    for (int d = 0; d < 2; d++) for (int e = 0; e < 2; e++) { ref[d][e] = 0; ign[d][e] = 0; for (int k = 0; k < 6; k++) cnt[d][e][k] = 0; }
    for (int k = 0; k < 6; k++) sample[k] = -1;
  }
  __device__ void put_scaled(int allele, int32_t scaled, int dir, int end) {
    if (XM_KEYS[allele] == ref_char) ref[dir][end] = scaled; else cnt[dir][end][allele] = scaled;
  }
  // forwardMiddle + forwardEnd + reverseMiddle + reverseEnd
  __device__ float refc() const { return ((fmt_units(ref[0][0]) + fmt_units(ref[0][1])) + fmt_units(ref[1][0])) + fmt_units(ref[1][1]); }
  __device__ float ignc() const { return ((fmt_units(ign[0][0]) + fmt_units(ign[0][1])) + fmt_units(ign[1][0])) + fmt_units(ign[1][1]); }
  __device__ float alt_count(int k) const { return ((fmt_units(cnt[0][0][k]) + fmt_units(cnt[0][1][k])) + fmt_units(cnt[1][0][k])) + fmt_units(cnt[1][1][k]); }
  __device__ bool has_alts() const {
    for (int d = 0; d < 2; d++) for (int e = 0; e < 2; e++) for (int k = 0; k < 6; k++) if (cnt[d][e][k] != 0) return true;
    return false;
  }
  __device__ bool has_alt(int k) const {
    for (int d = 0; d < 2; d++) for (int e = 0; e < 2; e++) if (fmt_units(cnt[d][e][k]) > 0) return true;
    return false;
  }
  __device__ unsigned alts() const {   // nonzero_alternates as a bit set over KEYS
    unsigned m = 0;
    if (has_alts()) for (int k = 0; k < 6; k++) if (has_alt(k)) m |= 1u << k;
    return m;
  }
  __device__ float count() const {     // getCount :169-178
    float t = refc() + ignc();
    if (has_alts()) for (int k = 0; k < 6; k++) t = t + alt_count(k);
    return t;
  }
  __device__ float middle_ref() const { return fmt_units(ref[0][0]) + fmt_units(ref[1][0]); }
  __device__ float end_ref() const { return fmt_units(ref[0][1]) + fmt_units(ref[1][1]); }
  __device__ float middle_alt(int k) const { return fmt_units(cnt[0][0][k]) + fmt_units(cnt[1][0][k]); }
  __device__ float end_alt(int k) const { return fmt_units(cnt[0][1][k]) + fmt_units(cnt[1][1][k]); }
  __device__ float middle_count() const {   // :192-201
    float t = middle_ref() + (fmt_units(ign[0][0]) + fmt_units(ign[1][0]));
    if (has_alts()) for (int k = 0; k < 6; k++) t = t + middle_alt(k);
    return t;
  }
  __device__ float end_count() const {      // :207-215 (no ignored term)
    float t = end_ref();
    if (has_alts()) for (int k = 0; k < 6; k++) t = t + end_alt(k);
    return t;
  }
  __device__ void ignore_alternate(int k) {   // :15-27
    if (XM_KEYS[k] == ref_char) return;
    for (int d = 0; d < 2; d++) for (int e = 0; e < 2; e++) { ign[d][e] += cnt[d][e][k]; cnt[d][e][k] = 0; }
  }
  __device__ char most_popular_alternate() const {   // :107-120
    float mx = 0.0f; char best = ' ';
    if (has_alts()) for (int k = 0; k < 6; k++) { const float c = alt_count(k); if (c > mx || k == 0) { mx = c; best = XM_KEYS[k]; } }
    return best;
  }
};

// MutationDetectionParameters
__device__ __forceinline__ bool fmt_supports_snp(const VarFilter& f, float depth, float total) {
  if (total < f.snp_total || depth <= 0) return false;
  return !(depth / total < f.snp_frac);
}
__device__ bool fmt_supports_indel(const FmtPos& p, float min_total, float min_frac) {
  const float mid = p.middle_count();
  if (mid < min_total) return false;
  float mi, ei;
  if (p.ref_char == '-') { mi = mid - p.middle_ref(); ei = p.end_count() - p.end_ref(); }
  else { mi = p.middle_alt(5); ei = p.end_alt(5); }
  if (mi <= 0 && ei <= 0) return false;
  return !(mi / mid < min_frac);
}

__device__ __forceinline__ unsigned long long fmt_gkey(const FmtD& D, long long pos) { return (unsigned long long)(D.contig_off[D.contig] + pos) << 21; }
__device__ unsigned long long fmt_lower_bound(const VarRec* r, unsigned long long lo, unsigned long long hi, unsigned long long key) {
  while (lo < hi) { const unsigned long long mid = lo + (hi - lo) / 2; if (r[mid].key < key) lo = mid + 1; else hi = mid; }
  return lo;
}
// the entries of position i: [*e0, *e1) inside [lo, hi)
__device__ void fmt_entries(const FmtD& D, long long i, unsigned long long lo, unsigned long long hi, unsigned long long* e0, unsigned long long* e1) {
  const unsigned long long k = fmt_gkey(D, i);
  unsigned long long a = fmt_lower_bound(D.recs, lo, hi, k), b = a;
  while (b < hi && (D.recs[b].key >> 21) == (k >> 21)) b++;
  *e0 = a; *e1 = b;
}
__device__ __forceinline__ SeqView fmt_example(const FmtD& D, unsigned long long e) {
  const int s = D.ex_slot[e];
  SeqView v; v.w = D.ex_words + D.ex_word_off[s]; v.len = D.ex_len[s]; v.rc = (int)(D.recs[e].ex_gid & 1); v.bytes = nullptr; v.b0 = 0; v.bn = 0;
  return v;
}
// putSampleAlternateSequence :69-92: the shown index is always the entry's ex_index; the letter it is filed under comes from the read
__device__ void fmt_put_sample(const FmtD& D, FmtPos& p, unsigned long long e, bool at_position) {
  const int idx = D.recs[e].ex_index;
  int k;
  if (at_position && idx < 0) k = 5;
  else {
    const uint8_t c = fmt_example(D, e).at(idx);
    if (bp_is_ambiguous(c)) return;
    k = c == 1 ? 0 : c == 2 ? 1 : c == 4 ? 2 : c == 8 ? 3 : 5;
  }
  p.sample[k] = (long long)e;
}
__device__ __forceinline__ int32_t fmt_plane(const FmtD& D, long long i, int region, int dir) {
  return D.planes[D.contig_off[D.contig] * 4 + (long long)(region * 2 + dir) * D.ref.len[D.contig] + i];
}
// Store.position: regions end -> middle, directions reverse -> forward (the last example put wins)
__device__ void fmt_position(const FmtD& D, long long i, unsigned long long e0, unsigned long long e1, bool samples, FmtPos& p) {
  p.init(XM_LETTERS[D.ref.contig(D.contig, 0).at((int)i)]);
  for (int q = 0; q < 4; q++) {
    const int region = 1 - (q >> 1), dir = 1 - (q & 1);
    for (unsigned long long e = e0; e < e1; e++) {
      const unsigned long long key = D.recs[e].key;
      if ((int)((key >> 19) & 3) != region * 2 + dir || ((key >> 3) & 0xFFFF) != 0) continue;
      p.put_scaled((int)(key & 7), D.recs[e].count, dir, region);
      if (samples) fmt_put_sample(D, p, e, true);
    }
    p.ref[dir][region] = fmt_plane(D, i, region, dir);
  }
}
// Store.insertion: column k of the insertion after position i; regions end -> middle, directions forward -> reverse
__device__ void fmt_insertion(const FmtD& D, long long i, int k, unsigned long long e0, unsigned long long e1, bool samples, FmtPos& p) {
  p.init('-');
  for (int q = 0; q < 4; q++) {
    const int region = 1 - (q >> 1), dir = q & 1;
    int32_t scaled_ins = 0, at_pos[6] = {0, 0, 0, 0, 0, 0};
    for (unsigned long long e = e0; e < e1; e++) {
      const unsigned long long key = D.recs[e].key;
      if ((int)((key >> 19) & 3) != region * 2 + dir) continue;
      const int col = (int)((key >> 3) & 0xFFFF), allele = (int)(key & 7);
      if (col == 0) { at_pos[allele] = D.recs[e].count; continue; }
      if (col != k + 1) continue;
      p.put_scaled(allele, D.recs[e].count, dir, region);
      scaled_ins += D.recs[e].count;
      if (samples) fmt_put_sample(D, p, e, false);
    }
    // the "non-insertion" term: getCount of a Position holding only this (region, direction), times 100
    float base = fmt_units(fmt_plane(D, i, region, dir));
    bool any = false;
    for (int a = 0; a < 6; a++) any |= at_pos[a] != 0;
    if (any) for (int a = 0; a < 6; a++) base = base + fmt_units(at_pos[a]);
    const int non = (int)(base * 100.0f) - scaled_ins;
    if (non > 0) p.put_scaled(5, non, dir, region);
  }
}
__device__ uint8_t fmt_decisive(const FmtD& D, long long i, unsigned long long lo, unsigned long long hi) {
  unsigned long long e0, e1;
  fmt_entries(D, i, lo, hi, &e0, &e1);
  FmtPos p;
  fmt_position(D, i, e0, e1, false, p);
  if (fmt_supports_indel(p, D.f.start_total, D.f.start_frac)) return 2;
  if (!fmt_supports_indel(p, D.f.cont_total, D.f.cont_frac)) return 1;
  return 0;
}
// FilteredAlignments.getPosition
__device__ void fmt_f_position(const FmtD& D, long long i, unsigned long long e0, unsigned long long e1, bool samples, FmtPos& p) {
  fmt_position(D, i, e0, e1, samples, p);
  const float total = p.count();
  const unsigned m = p.alts();
  for (int k = 0; k < 5; k++) if ((m >> k) & 1) if (!fmt_supports_snp(D.f, p.alt_count(k), total)) p.ignore_alternate(k);
  if (p.has_alts() && D.could_delete[i - D.start + 1] != 2) p.ignore_alternate(5);
}
// FilteredAlignments.getInsertion
__device__ void fmt_f_insertion(const FmtD& D, long long i, int k, unsigned long long e0, unsigned long long e1, bool samples, FmtPos& p) {
  fmt_insertion(D, i, k, e0, e1, samples, p);
  if (!p.has_alts()) return;
  const bool keep = k == 0 ? fmt_supports_indel(p, D.f.start_total, D.f.start_frac) : fmt_supports_indel(p, D.f.cont_total, D.f.cont_frac);
  if (!keep) { const unsigned m = p.alts(); for (int a = 0; a < 6; a++) if ((m >> a) & 1) p.ignore_alternate(a); }
}

__device__ void fmt_number(SamOut& o, float x) {   // AlignmentPosition.formatNumber :161-167
  if (x == truncf(x) && fabsf(x) < 9.0e18f) o.num((long long)x); else o.jfloat(x);
}
__device__ void fmt_counts_text(SamOut& o, const FmtPos& p, int k, int is_end) {   // getCounts :122-149; k < 0: the reference
  if (k < 0 || XM_KEYS[k] == p.ref_char) { fmt_number(o, fmt_units(p.ref[0][is_end])); o.ch(','); fmt_number(o, fmt_units(p.ref[1][is_end])); }
  else { fmt_number(o, fmt_units(p.cnt[0][is_end][k])); o.ch(','); fmt_number(o, fmt_units(p.cnt[1][is_end][k])); }
}
// VcfFormatterWorker.format :27-110, one line
__device__ void fmt_vcf_line(SamOut& o, const FmtD& D, long long row, const FmtPos& p) {
  const unsigned m = p.alts();
  o.str(D.name, D.name_len); o.ch('\t'); o.num(row); o.ch('\t'); o.ch(p.ref_char); o.ch('\t');
  if (!m) o.ch('.');
  { bool first = true; for (int k = 0; k < 6; k++) if ((m >> k) & 1) { if (!first) o.ch(','); o.ch(XM_KEYS[k]); first = false; } }
  o.ch('\t'); fmt_number(o, p.count());
  for (int is_end = 0; is_end < 2; is_end++) {
    o.ch('\t'); fmt_counts_text(o, p, -1, is_end);
    for (int k = 0; k < 6; k++) if ((m >> k) & 1) { o.ch(';'); fmt_counts_text(o, p, k, is_end); }
  }
  if (D.show_support) {
    o.ch('\t');
    const int n_alts = __popc(m);
    if (n_alts == 0 || (n_alts == 1 && p.sample[__ffs(m) - 1] < 0)) o.ch('.');
    else {
      bool first = true;
      for (int k = 0; k < 6; k++) if ((m >> k) & 1) {
        if (!first) o.ch(',');
        first = false;
        const long long e = p.sample[k];
        if (e < 0) continue;
        const SeqView v = fmt_example(D, (unsigned long long)e);
        int idx = D.recs[e].ex_index;
        if (idx < 0) {
          idx = -idx;
          for (int t = 0; t < idx; t++) o.ch(XM_LETTERS[v.at(t)]);
          o.lit("[-]");
          for (int t = idx; t < v.len; t++) o.ch(XM_LETTERS[v.at(t)]);
        } else {
          for (int t = 0; t < idx; t++) o.ch(XM_LETTERS[v.at(t)]);
          o.ch('['); o.ch(XM_LETTERS[v.at(idx)]); o.ch(']');
          for (int t = idx + 1; t < v.len; t++) o.ch(XM_LETTERS[v.at(t)]);
        }
      }
    }
  }
  o.ch('\n');
}
__device__ void fmt_mut_tail(SamOut& o, float depth, float total) { o.ch('\t'); fmt_number(o, depth); o.ch('\t'); fmt_number(o, total); o.ch('\n'); }
__device__ __forceinline__ void fmt_mut_head(SamOut& o, const FmtD& D, long long row) { o.str(D.name, D.name_len); o.ch('\t'); o.num(row); o.ch('\t'); }
__device__ bool fmt_is_deletion(const FmtD& D, long long j, unsigned long long lo, unsigned long long hi, FmtPos& p) {
  unsigned long long e0, e1;
  fmt_entries(D, j, lo, hi, &e0, &e1);
  fmt_f_position(D, j, e0, e1, false, p);
  return p.alt_count(5) > 0;
}
// write_deletions: the run of deletion positions ending at `last` (inside one job)
__device__ void fmt_deletion_run(SamOut& o, const FmtD& D, long long last, long long job0, unsigned long long lo, unsigned long long hi) {
  float depth = -1.0f, total = -1.0f;
  long long first = last;
  FmtPos p;
  for (long long j = last; j >= job0 && fmt_is_deletion(D, j, lo, hi, p); j--) {
    const float t = p.middle_count(), d = p.middle_alt(5);
    if (depth < 0 || depth > d) depth = d;
    if (total < 0 || total > t) total = t;
    first = j;
  }
  const SeqView rv = D.ref.contig(D.contig, 0);
  fmt_mut_head(o, D, first + 1);
  for (long long j = first; j <= last; j++) o.ch(XM_LETTERS[rv.at((int)j)]);
  o.ch('\t');
  for (long long j = first; j <= last; j++) o.ch('-');
  fmt_mut_tail(o, depth, total);
}

__global__ void __launch_bounds__(256) xm_fmt_carry_kernel(FmtD D) {
  __shared__ int first;
  if (threadIdx.x == 0) {
    D.range[0] = fmt_lower_bound(D.recs, 0, D.n_recs, fmt_gkey(D, D.start));
    D.range[1] = fmt_lower_bound(D.recs, 0, D.n_recs, fmt_gkey(D, D.end));
    D.dec[0] = 2;   // _could_be_deletion is true when the walk reaches the contig start
  }
  for (long long top = D.start - 1; top >= 0; top -= blockDim.x) {
    if (threadIdx.x == 0) first = 0x7fffffff;
    __syncthreads();
    const long long j = top - (long long)threadIdx.x;
    const uint8_t d = j >= 0 ? fmt_decisive(D, j, 0, D.n_recs) : 0;
    if (d) atomicMin(&first, (int)threadIdx.x);
    __syncthreads();
    if (d && first == (int)threadIdx.x) D.dec[0] = d;
    const bool done = first != 0x7fffffff;
    __syncthreads();
    if (done) break;
  }
}
__global__ void __launch_bounds__(128) xm_fmt_decide_kernel(FmtD D) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= D.end - D.start) return;
  D.dec[t + 1] = fmt_decisive(D, D.start + t, D.range[0], D.range[1]);
}
struct FmtLastDecisive { __device__ __forceinline__ uint8_t operator()(uint8_t a, uint8_t b) const { return b ? b : a; } };

template <int MODE, bool WRITE>
__global__ void __launch_bounds__(128) xm_fmt_kernel(FmtD D) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= D.end - D.start) return;
  const long long i = D.start + t;
  const unsigned long long lo = D.range[0], hi = D.range[1];
  SamOut o; o.n = 0; o.p = WRITE ? D.text + D.len[t] : nullptr;
  unsigned long long e0, e1;
  fmt_entries(D, i, lo, hi, &e0, &e1);
  FmtPos p, q;
  if (MODE == XM_FMT_VCF) {
    fmt_f_position(D, i, e0, e1, D.show_support != 0, p);
    if (p.count() > 0 && (D.include_non_mutations || p.has_alts())) fmt_vcf_line(o, D, i + 1, p);
    for (int k = 0;; k++) {
      fmt_f_insertion(D, i, k, e0, e1, D.show_support != 0, q);
      if (!q.has_alts()) break;
      fmt_vcf_line(o, D, -(i + 1), q);
    }
  } else {
    fmt_f_position(D, i, e0, e1, false, p);
    const float total = p.count();
    if (total > 0) {
      const unsigned m = p.alts();
      if (m && p.ref_char != 'N')
        for (int k = 0; k < 5; k++) if ((m >> k) & 1) { fmt_mut_head(o, D, i + 1); o.ch(p.ref_char); o.ch('\t'); o.ch(XM_KEYS[k]); fmt_mut_tail(o, p.alt_count(k), total); }
      int n_cand = 0; float depth = 0.0f;
      for (;; n_cand++) {
        fmt_f_insertion(D, i, n_cand, e0, e1, false, q);
        if (!q.has_alts()) break;
        depth = q.middle_count() - q.middle_ref();
      }
      if (n_cand) {
        fmt_mut_head(o, D, i + 1);
        for (int k = 0; k < n_cand; k++) o.ch('-');
        o.ch('\t');
        for (int k = 0; k < n_cand; k++) { fmt_f_insertion(D, i, k, e0, e1, false, q); o.ch(q.most_popular_alternate()); }
        fmt_mut_tail(o, depth, p.middle_count());
      }
    }
    // a deletion run is written after the records of the position that ends it, or after the last position of its job
    const long long job0 = i / XM_FMT_JOB * XM_FMT_JOB;
    const long long job1 = min((long long)D.ref.len[D.contig], job0 + XM_FMT_JOB);
    const bool del = p.alt_count(5) > 0;
    if (!del && i > job0 && fmt_is_deletion(D, i - 1, lo, hi, q)) fmt_deletion_run(o, D, i - 1, job0, lo, hi);
    if (del && i == job1 - 1) fmt_deletion_run(o, D, i, job0, lo, hi);
  }
  if (!WRITE) D.len[t] = o.n;
}

// the support column's reads: the distinct sequence ids the table's examples name, and per entry its slot in the uploaded list
__global__ void xm_ex_ids_kernel(const VarRec* recs, unsigned long long n, unsigned long long* ids) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) ids[i] = (unsigned long long)(recs[i].ex_gid >> 1);
}
__global__ void xm_ex_slot_kernel(const VarRec* recs, unsigned long long n, const int64_t* gids, int n_ex, const int32_t* len, int32_t* slot, unsigned int* bad) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long g = recs[i].ex_gid >> 1;
  int lo = 0, hi = n_ex;
  while (lo < hi) { const int mid = (lo + hi) / 2; if (gids[mid] < g) lo = mid + 1; else hi = mid; }
  const bool ok = lo < n_ex && gids[lo] == g && len[lo] == recs[i].ex_len;   // the read the counts kernel saw has that length
  slot[i] = ok ? lo : 0;
  if (!ok) atomicAdd(bad, 1u);
}
