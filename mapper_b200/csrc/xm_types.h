// xmapper_b200 device core — shared types.
// This header is compiled by nvcc for sm_100a (the product) and by g++ for the test-only host emulation
// harness (tests/emu/), which exists so the device logic can be checked against the oracle on a box without a
// GPU.  The shipped library never runs this code on the CPU.
// One source serves both builds, lane-split loops included: see "the warp" below.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define XM_HD __host__ __device__
#define XM_INLINE __host__ __device__ __forceinline__
// XM_FN: a function that must exist ONCE in the kernel image.  The per-query code is large and every warp is in a
// different phase of a different query, so code size is paid for in instruction-cache misses (ncu: stall_no_instruction).
#define XM_FN __host__ __device__ __noinline__
#define XM_NOUNROLL _Pragma("unroll 1")
#else
#define XM_HD
#define XM_INLINE inline
#define XM_FN inline
#define XM_NOUNROLL
// CUDA's 16-byte vector for the lane-strided clears; may_alias: it writes over int16_t / uint32_t arrays
struct __attribute__((may_alias)) uint4 { uint32_t x, y, z, w; };
inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { uint4 v; v.x = x; v.y = y; v.z = z; v.w = w; return v; }
#endif

#if defined(XM_TRACE) && !defined(__CUDA_ARCH__)
#include <stdio.h>
#define XM_T(...) fprintf(stderr, __VA_ARGS__)
#else
#define XM_T(...)
#endif

namespace xm {

// ---- per-query status ----
enum : int {
  Q_OK = 0,
  Q_NEED_MORE = 1,        // workspace tier exhausted: the host re-runs the query in the next tier
  Q_OUT_FULL = 2,         // result arena exhausted: the host grows it and re-runs the query
  Q_HARD = 3,             // first-pass kernel only: the cascade must go past the outer StraightAligner; re-run by the full kernel
  Q_AMBIGUOUS_QUERY = -2,
  Q_INDEX_TOO_SHORT = -3,
  Q_WORKSPACE = -5,
  Q_INTERNAL = -6
};

static const int JMAX = 2147483647;
#define XM_DISALLOWED 1000000.0

// ---- Java numeric semantics (JLS 5.1.3, 15.17-18) ----
XM_INLINE int j2i(double v) {
  if (v != v) return 0;
  if (v >= 2147483647.0) return 2147483647;
  if (v <= -2147483648.0) return (-2147483647 - 1);
  return (int)v;
}
XM_INLINE int32_t wadd(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }
XM_INLINE int32_t wmul(int32_t a, int32_t b) { return (int32_t)((uint32_t)a * (uint32_t)b); }
XM_INLINE int32_t jabs(int32_t v) { return v < 0 ? (int32_t)(0u - (uint32_t)v) : v; }
XM_INLINE double dmin(double a, double b) { return a < b ? a : b; }  // operands are never NaN / -0.0 on this path
XM_INLINE double dmax(double a, double b) { return a > b ? a : b; }
XM_INLINE int imin(int a, int b) { return a < b ? a : b; }
XM_INLINE int imax(int a, int b) { return a > b ? a : b; }
XM_INLINE int iabs(int a) { return a < 0 ? -a : a; }
XM_INLINE double next_up(double v) {  // Math.nextUp for finite v
  if (v == 0.0) return 4.9406564584124654e-324;
  union { double d; int64_t i; } u;
  u.d = v;
  if (v > 0) u.i += 1; else u.i -= 1;
  return u.d;
}
XM_INLINE double divide_round_up(double a, double b) {  // QueryMatch_Aligner.java:56-61
  double r = a / b;
  if (r * b < a) r = next_up(r);
  return r;
}

// ---- QV/Basepairs.java ----
XM_INLINE uint8_t bp_complement(uint8_t e) { return (uint8_t)(((e & 8) >> 3) | ((e & 4) >> 1) | ((e & 2) << 1) | ((e & 1) << 3)); }
XM_INLINE bool bp_can_match(uint8_t a, uint8_t b) { return (a & b) != 0; }
XM_INLINE int bp_num_choices(uint8_t e) { return ((e >> 3) & 1) + ((e >> 2) & 1) + ((e >> 1) & 1) + (e & 1); }
XM_INLINE bool bp_is_ambiguous(uint8_t e) { return e != 0 && e != 1 && e != 2 && e != 4 && e != 8; }
XM_INLINE bool bp_is_fully_ambiguous(uint8_t e) { return bp_num_choices(e) > 3; }

// ---- M/AlignmentParameters.java ----
struct Params {
  double mutation, ins_start, ins_ext, del_start, del_ext, max_error_rate, unaligned, ambiguity, span;
  int max_num_matches;
  int start_free;  // StartingInsertionStartFree
  const double* pen_tab;  // 256 entries [q << 4 | r] of the formula below, filled once per kernel launch (device: shared memory)
  // 1024 entries [q << 5 | r] over 5-bit codes: bit 0 canMatch, bit 1 penalty == 0, bit 2 either base fully ambiguous; code 16 is the
  // sentinel the PathAligner pads its two sections with ("off the section": canMatch, nothing else), so the search needs no bounds checks
  const uint8_t* cls_tab;
  XM_INLINE double starting_ins_start() const { return start_free ? 0.0 : ins_start; }
  XM_INLINE double min_possible_nonzero() const {
    double r = mutation;
    r = dmin(r, starting_ins_start() + ins_start);
    r = dmin(r, del_start + del_ext);
    return r;
  }
  XM_INLINE double base_penalty_formula(uint8_t q, uint8_t r) const {  // :156-180
    if (!bp_can_match(r, q)) return mutation;
    return ambiguity * ((bp_num_choices((uint8_t)(q | r)) - 1.0) / 3.0);
  }
  XM_INLINE double base_penalty(uint8_t q, uint8_t r) const { return pen_tab[((int)q << 4) | (int)r]; }
};

// A sequence seen through QV's packed layout; rc != 0 is a ReverseComplementSequence view (QV/ReverseComplementSequence.java:14-17)
struct SeqView {
  const uint16_t* w;
  int len;
  int rc;
  const uint8_t* bytes;  // optional: positions [b0, b0 + bn) of the same view unpacked to one code per byte (whole queries: ws_init; reference windows: qma_align_match)
  int b0, bn;
  XM_INLINE uint8_t at(int i) const {
    if (bytes) { unsigned k = (unsigned)(i - b0); if (k < (unsigned)bn) return bytes[k]; }
    int j = rc ? len - 1 - i : i;
    uint8_t c = (uint8_t)((w[j >> 2] >> ((j & 3) << 2)) & 15);
    return rc ? bp_complement(c) : c;
  }
};

// ---- reference, index, duplication table (device-resident, read-only) ----
struct RefD {
  int n_contigs;
  const uint16_t* words;     // all forward strands, each contig starting at a 16-byte aligned word offset
  const int64_t* word_off;   // n_contigs
  const int32_t* len;        // n_contigs
  const int64_t* gstart;     // 2*n_contigs+1: global start of sequence id s (even: forward, odd: reverse complement)
  int64_t total_fr;
  XM_INLINE SeqView contig(int c, int rc) const { SeqView v; v.w = words + word_off[c]; v.len = len[c]; v.rc = rc; v.bytes = nullptr; return v; }
  // QV/SequenceDatabase.decodePosition :170-209 — last sequence whose start <= encoded
  XM_INLINE void decode(int64_t g, int& seq_id, int& off) const {
    int lo = 0, hi = 2 * n_contigs;  // invariant: gstart[lo] <= g < gstart[hi]
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (gstart[mid] <= g) lo = mid; else hi = mid; }
    seq_id = lo; off = (int)(g - gstart[lo]);
  }
};

// bucket word: start (40 bits) << 24 | overfull << 16 | count (16 bits)
struct TableD {
  int capacity;
  int max_count;
  const uint64_t* buckets;   // capacity entries; nullptr for the empty PackedMap(1,1)
  const uint32_t* positions;     // low 32 bits of the global positions
  const uint8_t* positions_hi;   // bits 32-39, nullptr while the reference's forward + reverse size fits 32 bits (QV/SequenceDatabase.java:69-74 sizes positions the same way)
  XM_INLINE int64_t position(int64_t i) const { return (int64_t)positions[i] | (positions_hi ? ((int64_t)positions_hi[i] << 32) : 0); }
};
struct IndexD {
  int min_interesting;
  int max_built;
  int gapmers;
  const TableD* tables;      // max_built+1
};
struct DupD {
  int window;
  double granularity;
  const int64_t* off;        // n_contigs+1
  const int32_t* starts;     // sorted per contig
};

struct QueryIn {             // one query of the batch
  SeqView seq[2];            // as read
  int n_seqs;
  double expected_inner, per_penalty;
  XM_INLINE int length() const { return seq[0].len + (n_seqs > 1 ? seq[1].len : 0); }
};

// ---- result arena (device global memory, bump-allocated with atomics) ----
struct OutChoice { double spacing, multiplier, bonus, total; int inner; int n_sa; int64_t sa_first; };
struct OutSA { double penalty, aligned; int contig; int reversed; int n_blocks; int pad; int64_t block_first; };
struct OutQuery { int status; int n_comp; int n_choice[2]; int64_t choice_first[2]; };
struct OutArena {
  OutQuery* q;                 // n_queries
  OutChoice* choices; long long cap_choices;
  OutSA* sas; long long cap_sas;
  int32_t* blocks; long long cap_blocks;  // 4 ints per block
  unsigned long long* used;    // [0] choices, [1] sas, [2] blocks
  unsigned long long* stats;   // [0] probes [1] seeds [2] hits [3] straight [4] path calls [5] path steps [6] path cells
};

// ---- the warp ----
// On the device one WARP owns a query and all 32 lanes execute the per-query code in lock step on identical
// values (warp-uniform control flow; data-parallel inner loops are split across lanes where marked).  Side effects
// that must happen once per query are issued by lane 0 and their result is broadcast.
// Lane-split loops are written once, through the helpers below (on the device: the intrinsic with the full mask).  The host
// emulation is a warp of one lane - a ballot is the predicate, a shuffle or a sum returns its argument, warp_sync() does
// nothing - so such a loop runs serially in base order; compaction across lanes, the replay of lanes j > 0 and the xor tree
// run only on the GPU.  nvcc's host pass sees XM_LANES == 1 too: no type or host-side size may depend on it.
#if defined(__CUDA_ARCH__)
static constexpr int XM_LANES = 32;
__device__ __forceinline__ int lane_id() { return (int)(threadIdx.x & 31); }
__device__ __forceinline__ unsigned warp_ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
__device__ __forceinline__ bool warp_any(bool p) { return __any_sync(0xffffffffu, p); }
template <class T> __device__ __forceinline__ T warp_shfl(T v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }
__device__ __forceinline__ uint32_t warp_xor_sum(uint32_t v) {  // every lane gets the (wrapping) sum of all 32
  v += __shfl_xor_sync(0xffffffffu, v, 16);
  v += __shfl_xor_sync(0xffffffffu, v, 8);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v;
}
__device__ __forceinline__ void warp_sync() { __syncwarp(); }
__device__ __forceinline__ int first_bit(unsigned m) { return __ffs(m); }   // 1 + index of the lowest set bit, 0 for none
__device__ __forceinline__ int bit_count(unsigned m) { return __popc(m); }
#else
static constexpr int XM_LANES = 1;
inline int lane_id() { return 0; }
inline unsigned warp_ballot(bool p) { return p ? 1u : 0u; }
inline bool warp_any(bool p) { return p; }
template <class T> inline T warp_shfl(T v, int) { return v; }
inline int warp_sum(int v) { return v; }
inline uint32_t warp_xor_sum(uint32_t v) { return v; }
inline void warp_sync() {}
inline int first_bit(unsigned m) { return __builtin_ffs((int)m); }
inline int bit_count(unsigned m) { return __builtin_popcount(m); }
#endif

XM_INLINE unsigned long long xm_atomic_add(unsigned long long* p, unsigned long long v) {
#if defined(__CUDA_ARCH__)
  unsigned long long o = 0;
  if ((threadIdx.x & 31) == 0) o = atomicAdd(p, v);
  return __shfl_sync(0xffffffffu, o, 0);
#else
  unsigned long long o = *p; *p = o + v; return o;
#endif
}

}  // namespace xm
