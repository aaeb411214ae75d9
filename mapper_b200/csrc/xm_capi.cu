// xmapper_b200 — CUDA kernels + the C ABI (include/xmapper_b200.h).
// One query per WARP (warp-uniform control flow, lane-parallel inner loops); queries are handed out dynamically
// (atomic ticket) to a persistent grid sized from the SM count.  Every warp owns a private workspace arena in HBM;
// queries that exhaust the arena of one tier are collected and re-run from scratch in the next tier (bigger arenas,
// fewer warps).  The alignment path has no CPU implementation: the host only stages inputs and launches; the result
// arrays, the SAM text and the count records are assembled by kernels.
#include "../../include/xmapper_b200.h"
#include "xm_align.h"
#include "xm_host_model.h"
#include "xm_results.h"
#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/transform_input_iterator.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_run_length_encode.cuh>
#include <memory>
#include <chrono>
#include <dlfcn.h>
#include <nccl.h>
#include <mutex>
#include <condition_variable>
#include <string>
#include <vector>
#include <cstdio>
#include <cstdlib>

using namespace xm;

// ---------------------------------------------------------------- kernels
// first pass: blocks of 4 warps, 16 per SM (64 warps per SM at 32 registers).  full kernel: blocks of 32 warps, XM_FULL_MIN_BLOCKS
// per SM - the kernel is bound by instruction delivery (SM instruction-cache hit rate 55 %, the GPC instruction cache at 50-80 % of
// its request rate), so its run time is the same at 24, 32 or 64 warps per SM (profiles/r2_*).
#ifndef XM_BLOCK
#define XM_BLOCK 128
#endif
#ifndef XM_MIN_BLOCKS
#define XM_MIN_BLOCKS 16
#endif
#ifndef XM_FULL_BLOCK
#define XM_FULL_BLOCK 1024
#endif
#ifndef XM_FULL_MIN_BLOCKS
#define XM_FULL_MIN_BLOCKS 2
#endif
struct BatchD {
  int n_queries;
  const uint16_t* packed; const int64_t* seq_word_off; const int32_t* seq_len; const int64_t* first_seq;  // first_seq: n_queries+1
  const double* expected_inner; const double* per_penalty;
};
struct LaunchD {
  RefD ref; IndexD ix; DupD dup; Params prm;
  BatchD batch;
  OutArena out;
  const int32_t* ids; int n_ids;          // queries of this tier (nullptr = identity)
  const int* n_ids_ptr;                   // non-null: the number of queries is read from the device (left there by the previous launch), n_ids is only its bound
  int* ticket;                            // dynamic work counter
  int32_t* need_more; int* n_need_more;   // queries to re-run in the next tier
  int32_t* need_more_key;                 // first pass: cost estimate per entry of need_more (nullptr otherwise)
  int32_t* out_full; int* n_out_full;     // queries to re-run after growing the result arena
  char* arenas; long long arena_bytes;
  char* big_arenas; long long big_arena_bytes; int n_big; int* big_busy;  // pool of next-tier-sized arenas: a query that outgrows its warp's arena is re-run at once in a free one
  int last_tier;
  int dyn_stride;                         // bytes of dynamic shared memory per warp: the TMA staging area (XM_STAGE_BYTES) with use_tma, else 0
  int use_tma;                            // full kernel: reference windows are fetched with cp.async.bulk into the warp's staging area in shared memory
  long long* q_cycles;                    // optional per-query cost probe (XM_QCYCLES=1): clock64 ticks of the tier that finished it
};

// EASY = true: first pass over every query (small arenas, no cascade code in the image); false: the full aligner
// over the queries the first pass handed on.
template <bool EASY>
__global__ void __launch_bounds__(EASY ? XM_BLOCK : XM_FULL_BLOCK, EASY ? XM_MIN_BLOCKS : XM_FULL_MIN_BLOCKS) xm_align_kernel(LaunchD L) {
  const int lane = threadIdx.x & 31;
  const int warp_in_block = (int)(threadIdx.x >> 5), warps_per_block = (int)(blockDim.x >> 5);
  const long long warp = (long long)blockIdx.x * warps_per_block + warp_in_block;   // arena slot
  char* arena = L.arenas + warp * L.arena_bytes;
  __shared__ double s_pen[256];
  __shared__ uint8_t s_cls[1024];
  // the per-query state lives in shared memory, one slot per warp: in local memory every lane would keep (and
  // write through to L2/HBM) its own copy of the same bytes
  __shared__ WS s_ws[(EASY ? XM_BLOCK : XM_FULL_BLOCK) / 32];
  WS& w = s_ws[threadIdx.x >> 5];
  fill_pen_tab(L.prm, s_pen, s_cls, threadIdx.x, blockDim.x);
  __syncthreads();
  L.prm.pen_tab = s_pen; L.prm.cls_tab = s_cls;
  if (!EASY) {
    extern __shared__ __align__(16) unsigned char xm_dyn_smem[];
    unsigned char* stage = L.use_tma ? xm_dyn_smem + (size_t)warp_in_block * L.dyn_stride : nullptr;
#if defined(__CUDA_ARCH__)
    if (lane == 0) { w.stage = stage; w.stage_phase = 0; if (stage) stage_init(stage); }
#endif
    __syncwarp();
  }
  unsigned long long st[14] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  if (L.n_ids_ptr) L.n_ids = *L.n_ids_ptr;
  while (true) {
    int t = 0;
    if (lane == 0) t = atomicAdd(L.ticket, 1);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= L.n_ids) break;
    __syncwarp();   // every query starts with the warp converged: the per-query code runs on warp-shared state with all 32 lanes
#if defined(XM_DBG_UNIFORM)
    const bool split_at_start = __activemask() != 0xffffffffu;
    int dbg_split = 0;
#endif
    int qi = L.ids ? L.ids[t] : t;
    QueryIn q;
    long long c0 = L.q_cycles ? clock64() : 0;
    long long s0 = L.batch.first_seq[qi];
    q.n_seqs = (int)(L.batch.first_seq[qi + 1] - s0);
    for (int s = 0; s < q.n_seqs; s++) { q.seq[s].w = L.batch.packed + L.batch.seq_word_off[s0 + s]; q.seq[s].len = L.batch.seq_len[s0 + s]; q.seq[s].rc = 0; q.seq[s].bytes = nullptr; }
    if (q.n_seqs < 2) { q.seq[1] = q.seq[0]; q.seq[1].len = 0; }
    q.expected_inner = q.n_seqs > 1 ? L.batch.expected_inner[qi] : 0.0;
    q.per_penalty = q.n_seqs > 1 ? L.batch.per_penalty[qi] : 1.0;
    OutQuery rec; rec.status = 0; rec.n_comp = 1; rec.n_choice[0] = 0; rec.n_choice[1] = 0; rec.choice_first[0] = 0; rec.choice_first[1] = 0;
    w.hard_hint = 1 << 20;  // anything but Q_HARD (workspace exhausted in the first pass): assume long
    if (EASY) w.stage = nullptr;
    if (!ws_init(w, arena, L.arena_bytes, &L.ref, &L.ix, &L.dup, L.prm, q, !EASY)) w.status = Q_NEED_MORE;
    else align_query<EASY>(w, L.out, rec);
    __syncwarp();
#if defined(XM_DBG_UNIFORM)
    if (__activemask() != 0xffffffffu) dbg_split = 8000;
#endif
    int status = w.status;
    if (status == Q_HARD) status = Q_NEED_MORE;
    if (!EASY && status == Q_NEED_MORE && L.n_big > 0) {
      // escalate in place: grab a free big arena (no waiting - if none is free the query goes to the next tier as before)
      int slot = -1;
#if defined(XM_DBG_UNIFORM)
      if (__activemask() != 0xffffffffu) dbg_split = 8001;
#endif
      // every lane walks the slots (uniform control flow); only the claim itself is lane 0's
      for (int i = 0; i < L.n_big && slot < 0; i++) {
        const int j = (int)((warp + i) % L.n_big);
        int got = 0;
        if (lane == 0) got = (atomicCAS(&L.big_busy[j], 0, 1) == 0) ? 1 : 0;
        got = __shfl_sync(0xffffffffu, got, 0);
        if (got) slot = j;
      }
      __syncwarp();
#if defined(XM_DBG_UNIFORM)
      if (__activemask() != 0xffffffffu && dbg_split == 0) dbg_split = 8002;
#endif
      if (slot >= 0) {
        rec.status = 0; rec.n_comp = 1; rec.n_choice[0] = 0; rec.n_choice[1] = 0; rec.choice_first[0] = 0; rec.choice_first[1] = 0;
        if (!ws_init(w, L.big_arenas + (long long)slot * L.big_arena_bytes, L.big_arena_bytes, &L.ref, &L.ix, &L.dup, L.prm, q, true)) w.status = Q_NEED_MORE;
        else align_query<EASY>(w, L.out, rec);
        __syncwarp();
        status = w.status;
        __threadfence();
        if (lane == 0) atomicExch(&L.big_busy[slot], 0);
        __syncwarp();
      }
    }
    if (status == Q_NEED_MORE) {
      if (L.last_tier) status = Q_WORKSPACE;
      else if (lane == 0) { int k = atomicAdd(L.n_need_more, 1); L.need_more[k] = qi; if (L.need_more_key) L.need_more_key[k] = w.hard_hint; }
    } else if (status == Q_OUT_FULL) { if (lane == 0) { int k = atomicAdd(L.n_out_full, 1); L.out_full[k] = qi; } }
    rec.status = status;
#if defined(XM_DBG_UNIFORM)
    if (split_at_start) rec.status = -7777; else if (dbg_split) rec.status = -dbg_split; else if (w.st_cyc[5] != 0) rec.status = -(int)(100000 + w.st_cyc[5]);
#endif
    if (lane == 0) {
      L.out.q[qi] = rec;
      if (L.q_cycles) L.q_cycles[qi] = clock64() - c0;
    }
    __syncwarp();
    if (status != Q_NEED_MORE && status != Q_OUT_FULL) {
      st[0] += w.st_probes; st[1] += w.st_seeds; st[2] += w.st_hits; st[3] += w.st_straight; st[4] += w.st_path_calls; st[5] += w.st_path_steps; st[6] += w.st_path_cells;
      for (int i = 0; i < 6; i++) st[7 + i] += w.st_cyc[i];
      if (L.q_cycles) st[13] += (unsigned long long)(clock64() - c0);
    }
  }
  if (lane == 0) for (int i = 0; i < 14; i++) if (st[i]) atomicAdd(&L.out.stats[i], st[i]);
}


// ---- issue-rate micro-benchmarks (BASELINE.md §2 / SURVEY.md §8d: the roofline denominators of this path are instruction issue
// and the FP64 pipe, measured on the box, not taken from a datasheet).  Each thread runs `iters` rounds of 8 independent dependent
// chains; the kernels are launched over every SM at full occupancy and timed with CUDA events by xm_measure_peaks.
template <int KIND>
__global__ void __launch_bounds__(256) xm_peak_kernel(int iters, unsigned long long* sink, double seed) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (KIND == 0) {          // INT32 pipe: IMAD chains (the hash mixing / index arithmetic class of instructions)
    int a0 = tid, a1 = tid + 1, a2 = tid + 2, a3 = tid + 3, a4 = tid + 4, a5 = tid + 5, a6 = tid + 6, a7 = tid + 7;
    const int m = (int)seed | 1;
    #pragma unroll 1
    for (int i = 0; i < iters; i++) {
      #pragma unroll
      for (int k = 0; k < 16; k++) { a0 = a0 * m + a1; a1 = a1 * m + a2; a2 = a2 * m + a3; a3 = a3 * m + a4; a4 = a4 * m + a5; a5 = a5 * m + a6; a6 = a6 * m + a7; a7 = a7 * m + a0; }
    }
    if ((a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7) == 0x7fffffff) sink[0] = (unsigned long long)a0;
  } else if (KIND == 1) {   // FP64 pipe: DADD chains (penalty sums / min-add groups of the lattice search)
    double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
    #pragma unroll 1
    for (int i = 0; i < iters; i++) {
      #pragma unroll
      for (int k = 0; k < 16; k++) { a0 += a1; a1 += a2; a2 += a3; a3 += a4; a4 += a5; a5 += a6; a6 += a7; a7 += a0; }
    }
    if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 0.123) sink[0] = 1;
  } else {                  // the issue-slot ceiling: 8 independent FP32 FFMA chains (full-rate pipe: one warp-instruction per scheduler per clock)
    float f0 = (float)seed, f1 = f0 + 1.0f, f2 = f0 + 2.0f, f3 = f0 + 3.0f, f4 = f0 + 4.0f, f5 = f0 + 5.0f, f6 = f0 + 6.0f, f7 = f0 + 7.0f;
    const float c = (float)seed * 1e-9f;
    #pragma unroll 1
    for (int i = 0; i < iters; i++) {
      #pragma unroll
      for (int k = 0; k < 16; k++) {
        f0 = __fmaf_rn(f0, c, f1); f1 = __fmaf_rn(f1, c, f2); f2 = __fmaf_rn(f2, c, f3); f3 = __fmaf_rn(f3, c, f4);
        f4 = __fmaf_rn(f4, c, f5); f5 = __fmaf_rn(f5, c, f6); f6 = __fmaf_rn(f6, c, f7); f7 = __fmaf_rn(f7, c, f0);
      }
    }
    if (f0 + f1 + f2 + f3 + f4 + f5 + f6 + f7 == 0.123f) sink[0] = 1;
  }
}

// ---- result CSR assembly on the device (include/xmapper_b200.h: xm_results_array) ----
// The align kernels bump-allocate choices / sequence alignments / blocks in completion order.  These two kernels put
// them into query order as the eleven CSR arrays of the C ABI, laid out back to back in one slab that goes to the
// host in a single transfer (the host used to walk 1 M records with push_back: 160 ms per 1 M reads).
struct CsrD {
  int64_t* q_comp_off; int64_t* comp_choice_off; int64_t* choice_sa_off; int64_t* sa_block_off;
  double* choice_f64; double* sa_f64; int32_t* choice_inner; int32_t* sa_contig; int32_t* blocks; int32_t* q_status; uint8_t* sa_reversed;
};
// cnt: 4 arrays of nq + 1 int64 (components, choices, sequence alignments, blocks per query; the extra element is 0)
__global__ void xm_csr_count_kernel(OutArena out, int nq, long long* cnt) {
  int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q > nq) return;
  long long n_comp = 0, n_ch = 0, n_sa = 0, n_blk = 0;
  if (q < nq) {
    const OutQuery oq = out.q[q];
    n_comp = oq.status == 0 ? oq.n_comp : 1;
    if (oq.status == 0) {
      for (int c = 0; c < oq.n_comp; c++) {
        n_ch += oq.n_choice[c];
        for (int k = 0; k < oq.n_choice[c]; k++) {
          const OutChoice& ch = out.choices[oq.choice_first[c] + k];
          n_sa += ch.n_sa;
          for (int s = 0; s < ch.n_sa; s++) n_blk += out.sas[ch.sa_first + s].n_blocks;
        }
      }
    }
  }
  const long long stride = (long long)nq + 1;
  cnt[q] = n_comp; cnt[stride + q] = n_ch; cnt[2 * stride + q] = n_sa; cnt[3 * stride + q] = n_blk;
}
// base: exclusive sums of cnt (same layout); base[k * stride + nq] is the total of array k
__global__ void xm_csr_fill_kernel(OutArena out, int nq, const long long* base, CsrD c) {
  int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const long long stride = (long long)nq + 1;
  long long i_comp = base[q], i_ch = base[stride + q], i_sa = base[2 * stride + q], i_blk = base[3 * stride + q];
  if (q == 0) { c.q_comp_off[0] = 0; c.comp_choice_off[0] = 0; c.choice_sa_off[0] = 0; c.sa_block_off[0] = 0; }
  const OutQuery oq = out.q[q];
  c.q_status[q] = oq.status;
  const int n_comp = oq.status == 0 ? oq.n_comp : 1;
  for (int cc = 0; cc < n_comp; cc++) {
    const int n_ch = oq.status == 0 ? oq.n_choice[cc] : 0;
    for (int k = 0; k < n_ch; k++) {
      const OutChoice ch = out.choices[oq.choice_first[cc] + k];
      c.choice_f64[4 * i_ch] = ch.spacing; c.choice_f64[4 * i_ch + 1] = ch.multiplier; c.choice_f64[4 * i_ch + 2] = ch.bonus; c.choice_f64[4 * i_ch + 3] = ch.total;
      c.choice_inner[i_ch] = ch.inner;
      for (int s = 0; s < ch.n_sa; s++) {
        const OutSA sa = out.sas[ch.sa_first + s];
        c.sa_contig[i_sa] = sa.contig; c.sa_reversed[i_sa] = (uint8_t)sa.reversed;
        c.sa_f64[2 * i_sa] = sa.penalty; c.sa_f64[2 * i_sa + 1] = sa.aligned;
        const int4* src = (const int4*)out.blocks + sa.block_first;
        int4* dst = (int4*)c.blocks + i_blk;
        for (int b = 0; b < sa.n_blocks; b++) dst[b] = src[b];
        i_blk += sa.n_blocks;
        i_sa++;
        c.sa_block_off[i_sa] = i_blk;
      }
      i_ch++;
      c.choice_sa_off[i_ch] = i_sa;
    }
    i_comp++;
    c.comp_choice_off[i_comp] = i_ch;
  }
  c.q_comp_off[q + 1] = i_comp;
}

// ---- hash-block index built on the device (M/HashBlock_Database.java:490-665 + M/PackedMap.java:99-153 semantics) ----
// xm_index_emit_kernel: one warp per reference slice builds the slice's hash-block pyramid level by level (lanes take 32
//   block pairs per round, ballot compaction - the query pyramid's scheme) and, per level, emits (numBasepairsUsed, bucket,
//   global position) for every block's gapmer in its primary and/or secondary polarity.
// Two radix sorts order the entries by (used, bucket, position); a run-length pass yields the bucket counts; xm_index_runs /
// xm_index_fill write the PackedMap words (offset | overfull | count, empty buckets carry the running offset) and compact
// the positions of the buckets that are not overfull.  The tables are bit-identical to the host builder's.
struct IndexBuildD {
  RefD ref;
  const int* slice_contig; const int* slice_start; int n_slices, slice_len;
  int hi, min_interesting, gapmers;
  const int* cap;                      // hi + 1 capacities
  char* arenas; long long arena_bytes; // per warp: two level buffers
  unsigned long long* keys; void* vals; int wide; unsigned long long cap_entries;   // vals: uint32 global positions, uint64 when the reference needs more than 32 bits (wide)
  __device__ __forceinline__ void store_pos(unsigned long long o, long long g) const { if (wide) ((unsigned long long*)vals)[o] = (unsigned long long)g; else ((uint32_t*)vals)[o] = (uint32_t)g; }
  unsigned long long* n_entries; int* ticket; int* fail;
  int used_lo, used_hi;             // only blocks with used_lo <= numBasepairsUsed <= used_hi are emitted (a build chunked by block length)
  unsigned long long* hist;         // counting pass: entries per numBasepairsUsed (hi + 1 counters), nullptr = not wanted
  // counting pass: adds this lane's entries to hist[used]; lanes with the same length share one atomic
  __device__ __forceinline__ void count_used(int used, int n) const {
    const unsigned active = __activemask();
    const unsigned peers = __match_any_sync(active, used);
    const int total = __reduce_add_sync(peers, n);
    if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[used], (unsigned long long)total);
  }
};
static const unsigned long long XM_IX_MULTI = 1ull << 63;   // key bit of a MultiHashBlock possibility: above the sorted bits, dropped by the de-duplication
__device__ __forceinline__ int32_t ext_hash_lane(const SeqView& seq, int from, int n, int dir, bool complement) {  // one block per LANE
  int32_t h = 0;
  for (int k = 0; k < n; k++) {
    uint8_t c = seq.at(from + dir * k);
    if (complement) c = bp_complement(c);
    h = wadd(wmul(h, 7654337), ext_char_to_int(c));
  }
  return h;
}
__device__ __forceinline__ bool gapmer_lane(const HB& b, const SeqView& seq, HB& out) {  // HashBlock.withGapAndExtension :67-150
  if (b.gap_dir == 0) { out = b; return true; }
  int target = b.len + (jabs(b.fwd > b.rev ? b.fwd : b.rev) % 3) + b.extra;
  int gap = b.len / 2;
  int ext = target - gap;
  int32_t h;
  HB r;
  if (b.gap_dir < 0) {
    int ext_end = b.start - gap, ext_start = ext_end - ext;
    if (ext_start < 0) return false;
    h = ext_hash_lane(seq, ext_end - 1, ext, -1, false);
    r.start = ext_start; r.len = ext + gap + b.len;
  } else {
    int ext_start = b.end() + gap, ext_end = ext_start + ext;
    if (ext_end > seq.len) return false;
    h = ext_hash_lane(seq, ext_start, ext, 1, true);
    r.start = b.start; r.len = b.len + gap + ext;
  }
  r.fwd = wadd(b.fwd, h); r.rev = wadd(b.rev, h);
  r.used = b.len + ext;
  r.gap_dir = 0; r.flags = 0; r.extra = 0; r.ident = 0;
  out = r;
  return true;
}
__global__ void __launch_bounds__(128) xm_index_emit_kernel(IndexBuildD B) {
  const int lane = threadIdx.x & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int cap_lvl = B.slice_len + B.hi + 2 + 32;
  HB16* buf0 = (HB16*)(B.arenas + warp * B.arena_bytes);
  HB16* buf1 = buf0 + cap_lvl;
  while (true) {
    int t = 0;
    if (lane == 0) t = atomicAdd(B.ticket, 1);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= B.n_slices) break;
    const int contig = B.slice_contig[t], s = B.slice_start[t];
    const SeqView seq = B.ref.contig(contig, 0);
    const int e = min(seq.len, s + B.slice_len);
    const int ext_end = min(seq.len, e + B.hi + 2);
    const long long g_fwd = B.ref.gstart[2 * contig], g_rev = B.ref.gstart[2 * contig + 1];
    HB16* cur = buf0; HB16* nxt = buf1;
    int n_cur = ext_end - s;
    for (int k = lane; k < n_cur; k += 32) cur[k] = base_block16(seq.at(s + k), k);
    __syncwarp();
    while (n_cur > 0) {
      bool any_short = false;
      for (int base = 0; base < n_cur; base += 32) {
        const int idx = base + lane;
        HB16 c16; bool valid = false;
        if (idx < n_cur) { c16 = cur[idx]; valid = (s + (int)c16.start) < e; }
        if (__ballot_sync(0xffffffffu, valid) == 0) break;   // starts ascend: nothing further lies in the slice
        bool prim = false, sec = false; HB g;
        if (valid) {
          if ((int)c16.len <= B.hi) {
            any_short = true;
            HB b; b.start = s + c16.start; b.len = c16.len; b.used = c16.len; b.fwd = c16.fwd; b.rev = c16.rev; b.gap_dir = c16.gap_dir; b.flags = c16.flags; b.extra = c16.extra; b.ident = 0;
            bool ok = true;
            if (B.gapmers) ok = gapmer_lane(b, seq, g); else g = b;
            if (ok && g.used >= B.min_interesting && g.used <= B.hi && g.used >= B.used_lo && g.used <= B.used_hi) {
              const bool rml = g.rml(), rmr = g.rmr();
              prim = (rml != rmr) ? rml : (g.fwd >= g.rev);
              sec = (rml != rmr) ? rmr : (g.fwd <= g.rev);   // HashBlock.isSecondaryPolarity :339-343
            }
          }
        }
        if (B.hist != nullptr && (prim || sec)) B.count_used(g.used, (prim ? 1 : 0) + (sec ? 1 : 0));
        const unsigned pm = __ballot_sync(0xffffffffu, prim), sm = __ballot_sync(0xffffffffu, sec);
        const int total = __popc(pm) + __popc(sm);
        if (total) {
          unsigned long long at = 0;
          if (lane == 0) at = atomicAdd(B.n_entries, (unsigned long long)total);
          at = __shfl_sync(0xffffffffu, at, 0);
          if (B.keys != nullptr && at + total <= B.cap_entries) {
            const int c = B.cap[(prim || sec) ? g.used : 0];
            if (prim) { int r = g.fwd % c; if (r < 0) r += c; const unsigned long long o = at + __popc(pm & lt_mask); B.keys[o] = ((unsigned long long)g.used << 32) | (unsigned)r; B.store_pos(o, g_fwd + g.start); }
            if (sec) { int r = g.rev % c; if (r < 0) r += c; const unsigned long long o = at + __popc(pm) + __popc(sm & lt_mask); B.keys[o] = ((unsigned long long)g.used << 32) | (unsigned)r; B.store_pos(o, g_rev + (seq.len - g.end())); }
          }
        }
      }
      if (!__any_sync(0xffffffffu, any_short)) break;
      int n_new = 0;
      __syncwarp();
      for (int base = 0; base < n_cur - 1; base += 32) {
        const int i = base + lane;
        bool keep = false; HB16 L, R;
        if (i < n_cur - 1) { L = cur[i]; R = cur[i + 1]; keep = ((int)L.start + (int)L.len >= (int)R.start) && ((L.flags & 2) || (R.flags & 1)); }
        const unsigned mask = __ballot_sync(0xffffffffu, keep);
        if (keep) nxt[n_new + __popc(mask & lt_mask)] = merge_blocks16(L, R);
        n_new += __popc(mask);
      }
      __syncwarp();
      HB16* tmp = cur; cur = nxt; nxt = tmp; n_cur = n_new;
    }
  }
}

// Slices of an IUPAC-ambiguous reference (an "-anc" reference, M/AncestryDetector.java:323-327): one warp per slice builds the
// MultiHashBlock pyramid of the slice's window with the query path's own builder (pyr_build -> pyr_build_ambiguous,
// M/HashBlock_ParentRow.java:69-191) in a per-warp arena, then lanes take a row's entries and walk their possibilities; an entry
// of a multi-block carries XM_IX_MULTI so that xm_index_dedupe_kernel can apply PackedMap.add(preventDuplicates) :117-131.
__global__ void __launch_bounds__(32) xm_index_emit_amb_kernel(IndexBuildD B) {
  __shared__ WS w;
  const int lane = threadIdx.x & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  char* arena = B.arenas + (long long)blockIdx.x * B.arena_bytes;
  while (true) {
    int t = 0;
    if (lane == 0) t = atomicAdd(B.ticket, 1);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= B.n_slices) break;
    const int contig = B.slice_contig[t], s = B.slice_start[t];
    const SeqView full = B.ref.contig(contig, 0);
    const int e = min(full.len, s + B.slice_len);
    const int wlen = min(full.len, e + 4 * B.hi + 256) - s;   // the host builder's halo (xm_host_model.h: ambiguous_window_blocks)
    const long long g_fwd = B.ref.gstart[2 * contig], g_rev = B.ref.gstart[2 * contig + 1];
    __syncwarp();
    for (int k = lane; k < (int)(sizeof(WS) / 4); k += 32) ((uint32_t*)&w)[k] = 0;
    __syncwarp();
    MatePath& m = w.mp[0];
    Pyr& P = m.pyr;
    {
      SeqView v; v.w = full.w + (s >> 2); v.len = wlen; v.rc = 0; v.bytes = nullptr; v.b0 = 0; v.bn = 0;   // s is a multiple of 4
      m.q = v;
      const long long cap = 10LL * wlen + 256;
      const long long lev_bytes = ((long long)(wlen + 3) * 4 + 15) & ~15LL;
      char* p = arena;
      P.cap_levels = wlen + 2; P.cap_blocks = (int)cap;
      P.level_off = (int32_t*)p; p += lev_bytes;
      P.blk = (HB16*)p; p += cap * 16; P.child = (int16_t*)p; p += cap * 2; P.up = (int16_t*)p; p += cap * 2;
      p += (16 - ((uintptr_t)p & 15)) & 15;
      w.scratch = p; w.scratch_size = (long long)(arena + B.arena_bytes - p) & ~15LL; w.scratch_top = 0;
    }
    __syncwarp();
    const bool built = pyr_build(w, m) && w.status == 0;
    __syncwarp();
    if (!built) { if (lane == 0) atomicExch(B.fail, w.status ? w.status : Q_NEED_MORE); continue; }
    for (int level = 0; level < P.n_levels; level++) {
      const int n = pyr_level_size(P, level);
      const HB16* row = P.blk + P.level_off[level];
      bool any_short = false;
      for (int base = 0; base < n; base += 32) {
        const int idx = base + lane;
        HB16 c; bool valid = false; int k_n = 0;
        if (idx < n) { c = row[idx]; valid = (s + (int)c.start) < e; if (valid) k_n = pyr_num_opts(c); }
        if (__ballot_sync(0xffffffffu, valid) == 0) break;   // starts ascend within a row
        const int k_max = __reduce_max_sync(0xffffffffu, k_n);
        const unsigned long long multi = (valid && (c.flags & HB_MULTI)) ? XM_IX_MULTI : 0ull;
        for (int k = 0; k < k_max; k++) {
          bool prim = false, sec = false; HB g;
          if (k < k_n) {
            HB16 o16; bool has = true;
            if (c.flags & HB_MULTI) { const POpt* o = P.opt + c.fwd + k; has = o->has != 0; o16 = o->hb; } else o16 = c;
            if (has) {
              if ((int)o16.len <= B.hi) any_short = true;
              HB b; b.start = s + o16.start; b.len = o16.len; b.used = o16.len; b.fwd = o16.fwd; b.rev = o16.rev; b.gap_dir = o16.gap_dir; b.flags = o16.flags; b.extra = o16.extra; b.ident = 0;
              bool ok = true;
              if (B.gapmers) ok = gapmer_lane(b, full, g); else g = b;
              if (ok && g.used >= B.min_interesting && g.used <= B.hi && g.used >= B.used_lo && g.used <= B.used_hi) {
                const bool rml = g.rml(), rmr = g.rmr();
                prim = (rml != rmr) ? rml : (g.fwd >= g.rev);
                sec = (rml != rmr) ? rmr : (g.fwd <= g.rev);
              }
            }
          }
          if (B.hist != nullptr && (prim || sec)) B.count_used(g.used, (prim ? 1 : 0) + (sec ? 1 : 0));
          const unsigned pm = __ballot_sync(0xffffffffu, prim), sm = __ballot_sync(0xffffffffu, sec);
          const int total = __popc(pm) + __popc(sm);
          if (total) {
            unsigned long long at = 0;
            if (lane == 0) at = atomicAdd(B.n_entries, (unsigned long long)total);
            at = __shfl_sync(0xffffffffu, at, 0);
            if (B.keys != nullptr && at + total <= B.cap_entries) {
              const int cp = B.cap[(prim || sec) ? g.used : 0];
              if (prim) { int r = g.fwd % cp; if (r < 0) r += cp; const unsigned long long o = at + __popc(pm & lt_mask); B.keys[o] = multi | ((unsigned long long)g.used << 32) | (unsigned)r; B.store_pos(o, g_fwd + g.start); }
              if (sec) { int r = g.rev % cp; if (r < 0) r += cp; const unsigned long long o = at + __popc(pm) + __popc(sm & lt_mask); B.keys[o] = multi | ((unsigned long long)g.used << 32) | (unsigned)r; B.store_pos(o, g_rev + (full.len - g.end())); }
            }
          }
        }
      }
      if (!__any_sync(0xffffffffu, any_short)) break;
    }
  }
}
// PackedMap.add(preventDuplicates) on the sorted entries: a multi-block possibility is dropped when the same (length, bucket,
// position) was already added - by a plain block (which are never de-duplicated among themselves) or by another possibility.
template <typename PosT>
__global__ void xm_index_dedupe_kernel(const unsigned long long* keys, const PosT* vals, int n, unsigned char* keep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long k = keys[i];
  if (!(k & XM_IX_MULTI)) { keep[i] = 1; return; }
  const unsigned long long km = k & ~XM_IX_MULTI; const PosT p = vals[i];
  bool drop = i > 0 && (keys[i - 1] & ~XM_IX_MULTI) == km && vals[i - 1] == p;
  for (int j = i + 1; !drop && j < n && (keys[j] & ~XM_IX_MULTI) == km && vals[j] == p; j++) drop = !(keys[j] & XM_IX_MULTI);
  keep[i] = drop ? 0 : 1;
}
struct IxUnmulti { __host__ __device__ unsigned long long operator()(unsigned long long k) const { return k & ~XM_IX_MULTI; } };
// per run r of equal (used, bucket): kept[r] = count unless the bucket is overfull
__global__ void xm_index_runs_kernel(const unsigned long long* run_key, const int* run_cnt, int n_runs, long long* kept, int max_short) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_runs) return;
  if (r == n_runs) { kept[r] = 0; return; }
  const int n = (int)(run_key[r] >> 32);
  int mx = n * n; if (mx < max_short) mx = max_short; if (mx > 32766) mx = 32766; if (mx < 1) mx = 1;   // HostModel::max_count_for
  kept[r] = run_cnt[r] > mx ? 0 : run_cnt[r];
}
// first_run[n] = first run whose used >= n (n = 0 .. hi + 1)
__global__ void xm_index_first_run_kernel(const unsigned long long* run_key, int n_runs, int hi, int* first_run) {
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n > hi + 1) return;
  int lo = 0, h = n_runs;
  while (lo < h) { int mid = (lo + h) >> 1; if ((int)(run_key[mid] >> 32) < n) lo = mid + 1; else h = mid; }
  first_run[n] = lo;
}
template <typename PosT>
struct IndexFillD {
  const unsigned long long* run_key; const int* run_cnt; const long long* run_start; const long long* kept_off; int n_runs;
  const int* first_run; const int* cap; const long long* bucket_base;   // per used: offset of its bucket words in `buckets`
  const PosT* sorted_pos; unsigned long long* buckets; uint32_t* positions; uint8_t* positions_hi;  // positions: all lengths back to back, in kept_off order (low 32 bits; bits 32-39 in positions_hi when PosT is 64 bits wide)
};
template <typename PosT>
__global__ void xm_index_fill_kernel(IndexFillD<PosT> F) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= F.n_runs) return;
  const int n = (int)(F.run_key[r] >> 32); const unsigned bucket = (unsigned)F.run_key[r];
  const long long base_n = F.kept_off[F.first_run[n]];
  const long long off = F.kept_off[r] - base_n;
  const int cnt = F.run_cnt[r];
  const bool over = (F.kept_off[r + 1] - F.kept_off[r]) == 0 && cnt > 0;
  unsigned long long* bw = F.buckets + F.bucket_base[n];
  // empty buckets between the previous run of this length and this one carry the running offset (= this run's offset)
  unsigned first_empty = 0;
  if (r > F.first_run[n]) first_empty = (unsigned)F.run_key[r - 1] + 1;
  for (unsigned b = first_empty; b < bucket; b++) bw[b] = ((unsigned long long)off << 24);
  bw[bucket] = ((unsigned long long)off << 24) | ((unsigned long long)(over ? 1 : 0) << 16) | (unsigned long long)(over ? 0 : (cnt & 0xFFFF));
  if (r + 1 == F.first_run[n + 1]) {  // last run of this length: the tail of the table
    const long long end_off = F.kept_off[r + 1] - base_n;
    for (unsigned b = bucket + 1; b < (unsigned)F.cap[n]; b++) bw[b] = ((unsigned long long)end_off << 24);
  }
  if (!over) { const long long src = F.run_start[r], dst = F.kept_off[r]; for (int k = 0; k < cnt; k++) { const PosT v = F.sorted_pos[src + k]; F.positions[dst + k] = (uint32_t)v; if (sizeof(PosT) > 4) F.positions_hi[dst + k] = (uint8_t)((unsigned long long)v >> 32); } }
}

// ---- SAM bodies on the device (QV/SamWriter.java:118-352) ----
// One thread per query walks its records in the reference's order (components, choices, sequence alignments) twice:
// xm_sam_kernel<false> measures the text, an exclusive scan places the queries, xm_sam_kernel<true> writes it.
struct SamD {
  CsrD c;                                   // the result CSR of the batch, still resident from xm_align_batch
  const char* seq_names; const int64_t* seq_name_off;        // one name per SEQUENCE (mate)
  const char* contig_names; const int64_t* contig_name_off;
  long long* q_len;                         // per query: bytes of text (count pass), then exclusive offsets
  char* text;
};
#include "xm_text.cuh"
template <bool WRITE>
__global__ void xm_sam_kernel(SamD S, BatchD batch, int nq) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  SamOut o; o.n = 0; o.p = WRITE ? S.text + S.q_len[q] : nullptr;
  const CsrD& c = S.c;
  const long long s0 = batch.first_seq[q];
  const long long comp0 = c.q_comp_off[q], comp1 = c.q_comp_off[q + 1];
  const int n_comp = (int)(comp1 - comp0);
  int having = 0;                                  // getNumQueriesHavingAlignments :85-93
  for (long long cc = comp0; cc < comp1; cc++) if (c.comp_choice_off[cc + 1] > c.comp_choice_off[cc]) having++;
  for (long long cc = comp0; cc < comp1; cc++) {   // formatQueryAlignments :118-137
    const int sub = (int)(cc - comp0);
    const long long k0 = c.comp_choice_off[cc], k1 = c.comp_choice_off[cc + 1];
    double min_pen = 2147483647.0;
    for (long long k = k0; k < k1; k++) { const double pen = c.choice_f64[4 * k + 3]; if (pen < min_pen) min_pen = pen; }
    for (long long k = k0; k < k1; k++) {
      const double pen = c.choice_f64[4 * k + 3];
      const bool has_min = (pen - min_pen) <= fabs(min_pen) / 100000;
      const long long a0 = c.choice_sa_off[k], a1 = c.choice_sa_off[k + 1];
      const int n_sa = (int)(a1 - a0);
      const bool multi = n_sa > 1 || n_comp > 1;   // queryHadMultipleSequences :279-285
      for (long long a = a0; a < a1; a++) {        // formatQueryAlignment :139-223
        const int i = (int)(a - a0);
        const int mate = (n_comp == 2) ? sub : i;
        const long long sid = s0 + mate;
        const int qlen = batch.seq_len[sid];
        const bool rev = c.sa_reversed[a] != 0;
        const long long other = (n_sa == 2) ? (a == a0 ? a0 + 1 : a0) : -1;  // getPaired :334-342
        o.str(S.seq_names + S.seq_name_off[sid], S.seq_name_off[sid + 1] - S.seq_name_off[sid]); o.ch('\t');
        int flags = 0;                             // getSamFlags :288-331
        if (rev) flags += 16;
        if (multi) {
          flags += 1;
          if (n_sa > 1) { flags += 2; if (other >= 0 && c.sa_reversed[other] != 0) flags += 32; }
          if (!(n_sa > 1 || having > 1)) flags += 8;
          const int seq_index = sub + i;
          flags += (seq_index == 0) ? 64 : 128;
        }
        if (!has_min) flags += 256;
        o.num(flags); o.ch('\t');
        const int contig = c.sa_contig[a];
        o.str(S.contig_names + S.contig_name_off[contig], S.contig_name_off[contig + 1] - S.contig_name_off[contig]); o.ch('\t');
        const int32_t* blk = c.blocks + 4 * c.sa_block_off[a];
        const int n_blk = (int)(c.sa_block_off[a + 1] - c.sa_block_off[a]);
        o.num((long long)blk[1] + 1); o.ch('\t');  // POS :344-346
        o.num(has_min ? 255 : 0); o.ch('\t');      // MAPQ :242-261
        int consumed = 0;                          // CIGAR :166-190
        for (int b = 0; b < n_blk; b++) {
          const int as = blk[4 * b], al = blk[4 * b + 2], bl = blk[4 * b + 3];
          if (as != consumed) { o.num(as); o.ch('S'); consumed = as; }  // (the reference throws if this happens after the first block)
          if (al == bl) { o.num(al); o.ch('M'); } else if (al > bl) { o.num(al); o.ch('I'); } else { o.num(bl); o.ch('D'); }
          consumed += al;
        }
        if (consumed < qlen) { o.num(qlen - consumed); o.ch('S'); }
        o.ch('\t');
        if (other >= 0) {
          const int oc = c.sa_contig[other];
          o.str(S.contig_names + S.contig_name_off[oc], S.contig_name_off[oc + 1] - S.contig_name_off[oc]); o.ch('\t');
          o.num((long long)c.blocks[4 * c.sa_block_off[other] + 1] + 1); o.ch('\t');
        } else o.lit("*\t0\t");
        o.num(qlen); o.ch('\t');                   // TLEN (sic: the query length)
        SeqView qv; qv.w = batch.packed + batch.seq_word_off[sid]; qv.len = qlen; qv.rc = rev ? 1 : 0; qv.bytes = nullptr; qv.b0 = 0; qv.bn = 0;
        for (int t = 0; t < qlen; t++) o.ch("-ACMGRSVTWYHKDBN"[qv.at(t)]);  // SEQ: text of sequenceA (the reverse complement for reversed alignments)
        o.lit("\t*\t");
        if (multi) { o.score("cs:", pen); o.ch('\t'); }
        o.score("AS:", c.sa_f64[2 * a]);
        o.ch('\n');
      }
    }
  }
  if (!WRITE) S.q_len[q] = o.n;
}

// ---------------------------------------------------------------- handle
// The one owner of device memory in this file: every cudaMalloc / cudaFree is here, and a buffer is freed when its owner goes away.
struct DevBuf {
  void* p = nullptr; size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept { if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; } return *this; }
  ~DevBuf() { release(); }
  bool ensure(size_t bytes) {
    if (bytes <= cap) return true;
    release();
    size_t want = bytes + bytes / 8 + 256;
    if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); if (cudaMalloc(&p, bytes) != cudaSuccess) { p = nullptr; return false; } want = bytes; }
    cap = want;
    return true;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  // ensure (at least 16 bytes) + a synchronous host->device copy
  bool upload(const void* src, size_t bytes) { return ensure(bytes ? bytes : 16) && (!bytes || cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess); }
  // exactly `bytes`, keeping the first keep_bytes (copied on st, which is synchronised); on failure the old buffer stays as it was
  bool grow(size_t bytes, size_t keep_bytes, cudaStream_t st) {
    void* np = nullptr;
    if (cudaMalloc(&np, bytes) != cudaSuccess) { cudaGetLastError(); return false; }
    if ((keep_bytes && cudaMemcpyAsync(np, p, keep_bytes, cudaMemcpyDeviceToDevice, st) != cudaSuccess) || cudaStreamSynchronize(st) != cudaSuccess) { cudaFree(np); return false; }
    release(); p = np; cap = bytes;
    return true;
  }
};

#include "xm_counts.cuh"
#include "xm_variants_fmt.cuh"
#include "xm_parse.cuh"
#include "xm_names.cuh"

// pinned host slabs for results, recycled between batches (cudaHostAlloc of 100 MB costs tens of ms)
struct PinnedPool {
  std::mutex mu;
  std::vector<std::pair<void*, size_t>> free_list;
  void* take(size_t bytes, size_t& cap) {
    {
      std::lock_guard<std::mutex> g(mu);
      for (size_t i = 0; i < free_list.size(); i++) if (free_list[i].second >= bytes) { void* p = free_list[i].first; cap = free_list[i].second; free_list.erase(free_list.begin() + (long)i); return p; }
    }
    void* p = nullptr;
    size_t want = bytes + bytes / 4 + 4096;
    if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    cap = want;
    return p;
  }
  void give(void* p, size_t cap) {
    std::lock_guard<std::mutex> g(mu);
    if (free_list.size() >= 4) { size_t smallest = 0; for (size_t i = 1; i < free_list.size(); i++) if (free_list[i].second < free_list[smallest].second) smallest = i;
      if (free_list[smallest].second < cap) { cudaFreeHost(free_list[smallest].first); free_list[smallest] = {p, cap}; } else cudaFreeHost(p);
      return; }
    free_list.push_back({p, cap});
  }
  ~PinnedPool() { for (auto& f : free_list) cudaFreeHost(f.first); }
};
struct xm_results {
  ResultsHost r;
  uint64_t serial = 0; int nq = 0, slot = -1;   // which batch slot of the handle holds its device copy, and that slot's use counter at the time
  void* sam = nullptr; size_t sam_cap = 0;   // pinned text of the latest xm_format_sam (from the same pool as the slab)
  std::shared_ptr<PinnedPool> pool; void* slab = nullptr; size_t slab_cap = 0;
  ~xm_results() { if (slab && pool) pool->give(slab, slab_cap); if (sam && pool) pool->give(sam, sam_cap); }
};
// the arrays of one xm_parse_reads call (enum xm_reads_array), views into one pinned slab
struct xm_reads {
  std::shared_ptr<PinnedPool> pool; void* slab = nullptr; size_t slab_cap = 0;
  int64_t off[6] = {0, 0, 0, 0, 0, 0}, n[6] = {0, 0, 0, 0, 0, 0};
  ~xm_reads() { if (slab && pool) pool->give(slab, slab_cap); }
};

// ---- NCCL, loaded at run time (the host process may already carry its own libnccl; no link-time dependency) ----
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};
static NcclApi& nccl_api() {
  static NcclApi a;
  static std::once_flag once;
  std::call_once(once, [] {
    a.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // the copy the process already loaded (e.g. torch's), else the system one
    if (!a.lib) a.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!a.lib) a.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!a.lib) return;
    a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(a.lib, "ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))dlsym(a.lib, "ncclCommInitRank");
    a.AllReduce = (decltype(a.AllReduce))dlsym(a.lib, "ncclAllReduce");
    a.Broadcast = (decltype(a.Broadcast))dlsym(a.lib, "ncclBroadcast");
    a.AllGather = (decltype(a.AllGather))dlsym(a.lib, "ncclAllGather");
    a.GroupStart = (decltype(a.GroupStart))dlsym(a.lib, "ncclGroupStart");
    a.GroupEnd = (decltype(a.GroupEnd))dlsym(a.lib, "ncclGroupEnd");
    a.CommDestroy = (decltype(a.CommDestroy))dlsym(a.lib, "ncclCommDestroy");
    a.GetErrorString = (decltype(a.GetErrorString))dlsym(a.lib, "ncclGetErrorString");
    a.ok = a.GetUniqueId && a.CommInitRank && a.AllReduce && a.Broadcast && a.AllGather && a.GroupStart && a.GroupEnd && a.CommDestroy && a.GetErrorString;
  });
  return a;
}

struct xm_handle {
  HostModel m;
  int device = 0, sm_count = 148, blocks_per_sm = 4;
  std::string err;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev2 = nullptr, ev3 = nullptr, ev4 = nullptr, ev5 = nullptr;
  // device mirror of the model
  uint64_t mirrored_generation = ~0ull, mirrored_dup_generation = ~0ull;
  DevBuf d_words, d_word_off, d_len, d_gstart, d_tables, d_dup_off, d_dup_starts;
  std::vector<DevBuf> d_buckets, d_positions, d_positions_hi;
  std::vector<TableD> tables_host;   // host copy of the device table descriptors
  std::vector<DevBuf> d_ix_chunks;   // tables the device index builder left in place: per chunk of block lengths, {bucket words, positions, positions bits 32-39}
  RefD ref{}; IndexD ix{}; DupD dup{};
  // Batches in flight.  A call of xm_align_batch owns one slot from its first host->device copy to its last device->host copy: the
  // slot's staging buffers, its copy stream and its device copy of the result arrays.  The kernels of different calls run one after
  // the other on `stream` (compute_mu + the order of the events), so the copies of one call overlap the kernels of another:
  // concurrent callers on one handle (M/Api.java:78, M/Mapper.java:1026-1040: N AlignerWorkers) keep the GPU busy back to back.
  struct BatchSlot {
    DevBuf d_packed, d_seq_word_off, d_seq_len, d_n_seqs, d_expected, d_per, d_first_seq, d_csr_slab;
    cudaStream_t copy = nullptr; cudaEvent_t h2d_done = nullptr, kernels_done = nullptr, ev0 = nullptr, ev1 = nullptr;
    BatchD batch{}; uint64_t serial = 0, last_use = 0; bool busy = false;
  };
  uint64_t use_counter = 0;
  static const int N_SLOTS = 3;
  BatchSlot slots[N_SLOTS];
  std::mutex slot_mu; std::condition_variable slot_cv;
  std::mutex compute_mu;     // everything that launches kernels on `stream` or touches the shared work buffers below
  DevBuf d_chunk;
  DevBuf d_q, d_choices, d_sas, d_blocks, d_misc, d_ids_a, d_ids_b, d_ids_full, d_ws, d_qcycles;
  DevBuf d_csr_cnt, d_csr_base, d_csr_tmp, d_keys_a, d_keys_b, d_sort_tmp, d_big, d_big_busy;
  DevBuf d_sam_len, d_sam_text, d_sam_names, d_sam_name_off, d_sam_cnames, d_sam_cname_off;
  std::shared_ptr<PinnedPool> pinned = std::make_shared<PinnedPool>();
  bool probe_cycles = false;
  bool use_tma = true;    // false when the full kernel cannot get its dynamic shared memory: reference windows are then unpacked from global memory
  long long cap_choices = 0, cap_sas = 0, cap_blocks = 0;
  size_t ws_budget = (size_t)128 << 30;  // clamped to 60 % of the free device memory in xm_create
  // counts
  bool counts_enabled = false; double end_fraction = 0.1;
  DevBuf d_planes, d_contig_off; long long n_plane_ints = 0;
  // sparse variant table (xm_counts.cuh): recs[0, var_n) = reduced entries followed by raw records of the batches since the last reduce
  DevBuf d_var, d_var_n, d_order, d_var_sizes; VarScratch var_scratch;
  unsigned long long var_n = 0, var_cap = 0, var_reduced_n = 0;
  long long next_gid = 0;                       // global id of the first sequence of the next batch (xm_counts_batch_info overrides it)
  bool have_batch_info = false; long long info_first_gid = 0; std::vector<int64_t> info_order;
  // VCF / mutations bodies (xm_variants_fmt.cuh).  var_gen changes whenever the planes or the table do (a batch accumulates, a reduce
  // runs, counts are enabled); the example list and the uploaded example texts belong to the generation they were made for.
  unsigned long long var_gen = 0, ex_list_gen = ~0ull, ex_gen = ~0ull;
  std::vector<int64_t> ex_list;
  DevBuf d_ex_words, d_ex_word_off, d_ex_len, d_ex_gids, d_ex_slot, d_ex_bad;
  DevBuf d_fmt_dec, d_fmt_state, d_fmt_len, d_fmt_range, d_fmt_name, d_fmt_text, d_fmt_tmp, d_fmt_ids;
  void* fmt_text = nullptr; size_t fmt_cap = 0;   // pinned text of the latest xm_format_vcf / xm_format_mutations
  // read parsing (xm_parse.cuh): its own lock, stream and buffers, so that parsing the next chunk overlaps the batch being aligned
  std::mutex parse_mu; cudaStream_t parse_stream = nullptr;
  DevBuf d_pz_text, d_pz_tiles, d_pz_line_end, d_pz_flag, d_pz_line_rec, d_pz_rec_line, d_pz_bases, d_pz_lbase, d_pz_pieces, d_pz_piece_off;
  DevBuf d_pz_start, d_pz_len, d_pz_rec, d_pz_words, d_pz_name_len, d_pz_word_off, d_pz_name_off, d_pz_slab, d_pz_tmp, d_pz_misc;
  void* pz_stage = nullptr; size_t pz_stage_cap = 0;   // pinned staging of the text
  ncclComm_t comm = nullptr; int comm_ranks = 0, comm_rank = 0;
  double last_planes_ms = 0, last_variants_ms = 0;   // xm_counts_reduce: device time of the plane all-reduce, wall time of the variant-table exchange   // xm_comm_init: the communicator xm_counts_reduce uses
};

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(e_); return XM_ERR_CUDA; } } while (0)
// RAII lease of a batch slot: the least recently used free one, so that the device copies of recent results live as long as possible
struct SlotLease {
  xm_handle* h; int i;
  explicit SlotLease(xm_handle* hh) : h(hh), i(-1) {
    std::unique_lock<std::mutex> g(h->slot_mu);
    while (true) {
      for (int k = 0; k < xm_handle::N_SLOTS; k++) if (!h->slots[k].busy && (i < 0 || h->slots[k].last_use < h->slots[i].last_use)) i = k;
      if (i >= 0) break;
      h->slot_cv.wait(g);
    }
    h->slots[i].busy = true; h->slots[i].last_use = ++h->use_counter; h->slots[i].serial++;
  }
  ~SlotLease() { { std::lock_guard<std::mutex> g(h->slot_mu); h->slots[i].busy = false; } h->slot_cv.notify_one(); }
  xm_handle::BatchSlot& slot() { return h->slots[i]; }
};

// the reference codes and their layout, and the device view of them (h->ref)
static int upload_reference(xm_handle* h) {
  const HostModel& M = h->m;
  if (!h->d_words.upload(M.words.data(), M.words.size() * 2) || !h->d_word_off.upload(M.word_off.data(), M.word_off.size() * 8) ||
      !h->d_len.upload(M.len.data(), M.len.size() * 4) || !h->d_gstart.upload(M.gstart.data(), M.gstart.size() * 8)) { h->err = "device upload failed (reference)"; return XM_ERR_CUDA; }
  h->ref.n_contigs = M.n_contigs; h->ref.words = (const uint16_t*)h->d_words.p; h->ref.word_off = (const int64_t*)h->d_word_off.p;
  h->ref.len = (const int32_t*)h->d_len.p; h->ref.gstart = (const int64_t*)h->d_gstart.p; h->ref.total_fr = M.total_fr;
  return XM_OK;
}

static int mirror_model(xm_handle* h) {
  HostModel& M = h->m;
  if (h->mirrored_generation == M.generation && h->mirrored_dup_generation == M.dup_generation) return XM_OK;
  if (M.n_contigs < 1) { h->err = "reference not set"; return XM_ERR_STATE; }
  if (!M.index_finished) { h->err = "index not set (xm_set_index_length + xm_finish_index, or xm_build_index)"; return XM_ERR_STATE; }
  bool ok = true;
  if (h->mirrored_generation != M.generation) {   // reference + index tables
    if (int rc = upload_reference(h)) return rc;
    size_t nt = (size_t)M.max_built + 1;
    if (M.tables.size() < nt) M.tables.resize(nt);
    h->d_ix_chunks.clear();
    h->d_buckets.resize(nt); h->d_positions.resize(nt); h->d_positions_hi.resize(nt);
    std::vector<TableD> tabs(nt);
    for (size_t i = 0; ok && i < nt; i++) {
      const HostTable& T = M.tables[i];
      tabs[i].capacity = T.capacity; tabs[i].max_count = T.max_count; tabs[i].buckets = nullptr; tabs[i].positions = nullptr; tabs[i].positions_hi = nullptr;
      if (!T.buckets.empty()) {
        ok = h->d_buckets[i].upload(T.buckets.data(), T.buckets.size() * 8) && h->d_positions[i].upload(T.positions.data(), T.positions.size() * 4);
        tabs[i].buckets = (const uint64_t*)h->d_buckets[i].p; tabs[i].positions = (const uint32_t*)h->d_positions[i].p;
        if (ok && !T.positions_hi.empty()) { ok = h->d_positions_hi[i].upload(T.positions_hi.data(), T.positions_hi.size()); tabs[i].positions_hi = (const uint8_t*)h->d_positions_hi[i].p; }
      }
    }
    ok = ok && h->d_tables.upload(tabs.data(), nt * sizeof(TableD));
    h->tables_host = tabs;
  }
  if (ok) {   // the duplication table (small; re-uploaded on its own when only it changed)
    std::vector<int64_t> doff; std::vector<int32_t> dst;
    M.dup_csr(doff, dst);
    ok = h->d_dup_off.upload(doff.data(), doff.size() * 8) && h->d_dup_starts.upload(dst.data(), dst.size() * 4);
  }
  if (!ok) { h->err = std::string("device upload failed: ") + cudaGetErrorString(cudaGetLastError()); return XM_ERR_CUDA; }
  h->ix.min_interesting = M.min_interesting; h->ix.max_built = M.max_built; h->ix.gapmers = M.gapmers; h->ix.tables = (const TableD*)h->d_tables.p;
  h->dup.window = M.dup_window; h->dup.granularity = M.dup_granularity; h->dup.off = (const int64_t*)h->d_dup_off.p; h->dup.starts = (const int32_t*)h->d_dup_starts.p;
  h->mirrored_generation = M.generation; h->mirrored_dup_generation = M.dup_generation;
  return XM_OK;
}

// ---- duplication detector, first half on the device (M/DuplicationDetector.java:129-214) ----
// xm_dup_scan_kernel walks the buckets of one table: lanes test 32 bucket words at a time, and every bucket that holds at least
// min_copies positions (and is not overfull) is then grouped by the whole warp - lookupByForwardHash :41-52 lists every stored
// position plus its reverse complement, the blocks are grouped by their text (first and last ceil(length / 4) bases, blocks with an
// ambiguous base dropped), and every block of a group of >= min_copies distinct (sequence, start) pairs is a duplication.  The
// forward-strand ones are appended to `recs`; HostModel::merge_duplications applies saveDuplications' order-dependent containment
// rule to them (a std::map walk per block, the part that stays on the host).
struct DupItem { unsigned long long klo, khi; int32_t sid, st; };   // sid < 0: not a member (ambiguous text, or an image that repeats a stored position)
struct DupScanD {
  RefD ref; TableD t; int bl, min_copies, prefix;
  char* scratch; long long scratch_stride;   // per warp: 2 * max_count items (GROUPS: followed by 3 int32 per item)
  HostModel::DupRecH* recs; unsigned long long cap; unsigned long long* n_recs;
  HostModel::DupGrpRec* grecs; int* n_groups; int max_items;   // GROUPS only
};
// GROUPS = false: the duplication table's scan (forward-strand blocks, one record each).  GROUPS = true: the ancestry detector's scan
// (M/AncestryDetector.java:89-147 reads M/Duplication.java objects): every text group of a bucket with >= min_copies distinct members
// gets an id, and every member - on both strands, reverse-strand images included - becomes one record (sequence, start, length,
// count, hashcode, group id) in `grecs`.
template <bool GROUPS>
__global__ void __launch_bounds__(128) xm_dup_scan_kernel(DupScanD D) {
  const int lane = threadIdx.x & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  DupItem* items = (DupItem*)(D.scratch + warp * D.scratch_stride);
  int* g_count = GROUPS ? (int*)(items + D.max_items) : nullptr;   // per item: members of its text group, first item of the group, group id
  int* g_first = GROUPS ? g_count + D.max_items : nullptr;
  int* g_id = GROUPS ? g_first + D.max_items : nullptr;
  for (long long base = warp * 32; base < D.t.capacity; base += n_warps * 32) {
    const long long my = base + lane;
    unsigned long long word = 0;
    if (my < D.t.capacity) word = D.t.buckets[my];
    const bool want = !((word >> 16) & 1) && (int)(word & 0xFFFF) >= D.min_copies;
    unsigned todo = __ballot_sync(0xffffffffu, want);
    while (todo) {
      const int src = __ffs(todo) - 1; todo &= todo - 1;
      const unsigned long long wd = __shfl_sync(0xffffffffu, word, src);
      const int c = (int)(wd & 0xFFFF), n = 2 * c;
      const long long pos0 = (long long)(wd >> 24);
      for (int k = lane; k < n; k += 32) {
        const long long g = D.t.position(pos0 + k % c);
        int sid, st; D.ref.decode(g, sid, st);
        bool out = false;
        if (k >= c) {   // the reverse complement of a stored block; a set: dropped when that block is itself stored in this bucket
          sid ^= 1; st = D.ref.len[sid >> 1] - st - D.bl;
          const long long gi = D.ref.gstart[sid] + st;
          for (int x = 0; x < c && !out; x++) out = D.t.position(pos0 + x) == gi;
        }
        const SeqView v = D.ref.contig(sid >> 1, sid & 1);
        unsigned long long klo = 0, khi = 0;
        for (int i = 0; i < D.prefix; i++) {
          const unsigned a = v.at(st + i), b = v.at(st + D.bl - D.prefix + i);
          out |= bp_is_ambiguous((uint8_t)a) || bp_is_ambiguous((uint8_t)b);
          klo = (klo << 4) | a; khi = (khi << 4) | b;
        }
        DupItem it; it.klo = klo; it.khi = khi; it.sid = out ? -1 : sid; it.st = st;
        items[k] = it;
      }
      __syncwarp();
      if constexpr (!GROUPS) {
        for (int ib = 0; ib < n; ib += 32) {
          const int i = ib + lane;
          DupItem me; me.sid = -1; me.klo = 0; me.khi = 0; me.st = 0;
          if (i < n) me = items[i];
          int count = 0;
          for (int j = 0; j < n; j++) { const DupItem o = items[j]; count += (o.sid >= 0 && o.klo == me.klo && o.khi == me.khi) ? 1 : 0; }
          const bool emit = me.sid >= 0 && !(me.sid & 1) && count >= D.min_copies;
          const unsigned em = __ballot_sync(0xffffffffu, emit);
          if (em) {
            unsigned long long at = 0;
            if (lane == 0) at = atomicAdd(D.n_recs, (unsigned long long)__popc(em));
            at = __shfl_sync(0xffffffffu, at, 0) + __popc(em & lt_mask);
            if (emit && at < D.cap) { HostModel::DupRecH r; r.contig = me.sid >> 1; r.st = me.st; r.count_len = count | (D.bl << 24); r.hc = (int32_t)(base + src); D.recs[at] = r; }
          }
        }
      } else {
        // pass 1: group sizes, and an id for every group of >= min_copies members (allocated by its first item)
        for (int i = lane; i < n; i += 32) {
          const DupItem me = items[i];
          int count = 0, first = -1;
          if (me.sid >= 0)
            for (int j = 0; j < n; j++) { const DupItem o = items[j]; if (o.sid >= 0 && o.klo == me.klo && o.khi == me.khi) { count++; if (first < 0) first = j; } }
          g_count[i] = count; g_first[i] = first;
          if (me.sid >= 0 && first == i && count >= D.min_copies) g_id[i] = atomicAdd(D.n_groups, 1);
        }
        __syncwarp();
        // pass 2: one record per member
        for (int ib = 0; ib < n; ib += 32) {
          const int i = ib + lane;
          bool emit = false; int sid = -1, stv = 0, count = 0, gid = -1;
          if (i < n) { sid = items[i].sid; stv = items[i].st; count = g_count[i]; emit = sid >= 0 && count >= D.min_copies; if (emit) gid = g_id[g_first[i]]; }
          const unsigned em = __ballot_sync(0xffffffffu, emit);
          if (em) {
            unsigned long long at = 0;
            if (lane == 0) at = atomicAdd(D.n_recs, (unsigned long long)__popc(em));
            at = __shfl_sync(0xffffffffu, at, 0) + __popc(em & lt_mask);
            if (emit && at < D.cap) { HostModel::DupGrpRec r; r.sid = sid; r.st = stv; r.count_len = count | (D.bl << 24); r.hc = (int32_t)(base + src); r.gid = gid; D.grecs[at] = r; }
          }
        }
      }
      __syncwarp();
    }
  }
}
// xm_dup_scan_kernel<GROUPS> over the tables of lengths min_len..max_len.  The records come back in `recs` and stay in `d_recs`:
// the ancestry code goes on reading them on the device.
template <class Rec> struct DupScan { std::vector<Rec> recs; DevBuf d_recs; int n_groups = 0; };
template <bool GROUPS, class Rec>
static int dup_scan(xm_handle* h, int min_len, int max_len, int min_copies, DupScan<Rec>& out) {
  const char* what = GROUPS ? "ancestry group" : "duplication";
  cudaStream_t st = h->stream;
  const int blocks = h->sm_count * 8, warps = blocks * 4;
  int max_items = 2;
  for (int bl = std::max(1, min_len); bl <= max_len; bl++) max_items = std::max(max_items, 2 * h->tables_host[(size_t)bl].max_count);
  DevBuf d_scratch, d_n;
  DupScanD D; D.ref = h->ref; D.min_copies = min_copies; D.max_items = max_items; D.recs = nullptr; D.grecs = nullptr;
  D.scratch_stride = (((long long)max_items * (long long)(sizeof(DupItem) + (GROUPS ? 12 : 0))) + 255) & ~255LL;
  if (!d_scratch.ensure((size_t)warps * (size_t)D.scratch_stride) || !d_n.ensure(16)) { h->err = std::string("out of device memory (") + what + " scan)"; return XM_ERR_CUDA; }
  D.scratch = (char*)d_scratch.p; D.n_recs = (unsigned long long*)d_n.p; D.n_groups = (int*)((char*)d_n.p + 8);
  unsigned long long cap = 1ull << 20, found = 0;
  for (int attempt = 0; attempt < 2; attempt++) {   // second attempt: the buffer sized by the first one's count
    if (!out.d_recs.ensure((size_t)cap * sizeof(Rec))) { h->err = std::string("out of device memory (") + what + " records)"; return XM_ERR_CUDA; }
    if constexpr (GROUPS) D.grecs = (Rec*)out.d_recs.p; else D.recs = (Rec*)out.d_recs.p;
    D.cap = cap;
    CK(cudaMemsetAsync(d_n.p, 0, 16, st));
    for (int bl = std::max(1, min_len); bl <= max_len; bl++) {
      const TableD& T = h->tables_host[(size_t)bl];
      if (T.buckets == nullptr) continue;
      D.t = T; D.bl = bl; D.prefix = (bl + 3) / 4;
      xm_dup_scan_kernel<GROUPS><<<blocks, 128, 0, st>>>(D);
    }
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&found, d_n.p, 8, cudaMemcpyDeviceToHost, st));
    if (GROUPS) CK(cudaMemcpyAsync(&out.n_groups, (char*)d_n.p + 8, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (found <= cap) break;
    cap = found;
  }
  out.recs.resize((size_t)found);
  if (found) CK(cudaMemcpy(out.recs.data(), out.d_recs.p, (size_t)found * sizeof(Rec), cudaMemcpyDeviceToHost));
  return XM_OK;
}
static int build_duplications_device(xm_handle* h, int min_len, int max_len, int min_copies, int window) {
  HostModel& M = h->m;
  if (min_len < 0) min_len = M.choose_min_dup_len();
  if (max_len < 0) max_len = 2 * M.choose_min_dup_len();
  if (max_len > M.max_built) max_len = M.max_built;
  if (max_len > 64) { h->err = "xm_build_duplications: block lengths above 64 are not supported by the device scan (128-bit text keys); xm_build_duplications_host takes any length"; return XM_ERR_ARG; }
  if (min_copies < 1) min_copies = 1;
  const bool trace = getenv("XM_TRACE_SETUP") != nullptr;
  const double t_begin = now_s();
  if (int rc = mirror_model(h)) return rc;
  const double t_mirror = now_s();
  DupScan<HostModel::DupRecH> S;
  if (int rc = dup_scan<false>(h, min_len, max_len, min_copies, S)) return rc;
  const double t_scan = now_s();
  const size_t found = S.recs.size();
  M.merge_duplications(S.recs, min_len, window);
  if (trace) fprintf(stderr, "[xm] duplications: mirror %.3f s, device scan of lengths %d..%d %.3f s (%zu blocks found), merge %.3f s\n", t_mirror - t_begin, min_len, max_len, t_scan - t_mirror, found, now_s() - t_scan);
  return XM_OK;
}

// ---- ancestor inference on the device (--infer-ancestors: M/AncestryDetector.java:89-439, as M/Mapper.java:666-692 sets it up) ----
// infer_ancestors_device: a temporary index of the original reference (build_index_device with the caller's minInterestingSize and
// maxNumShortMatches), the group scan (xm_dup_scan_kernel<true>), saveDuplications on the host over all 2 * n_contigs sequences with the
// groups kept (HostModel::merge_duplication_groups), then xm_ancestry_kernel - one warp per (group, polarity) analysis,
// AncestryDetector.analyze :157-337 - and xm_anc_apply_kernel, which writes the inferred unions into the packed reference.
// Every analysis reads the original codes only, and a position can be written once (M/OverriddenSequence.java:19-27), so the order in
// which the analyses run does not change the result.  Writes are kept per global position: one bit per position of both strands detects
// a second write; only forward-strand writes reach the code plane (the reverse sequences are regenerated from the forward ones).
struct AncMember { int32_t sid, start, bound, cur, best_idx; uint32_t flags; double cum, best; };   // one SimilarityAnalysis
enum : uint32_t { ANC_AV = 1, ANC_IN = 2, ANC_NLI = 4, ANC_NLA = 8 };   // available, interested; this step: no longer interested / available
struct AncD {
  RefD ref;
  const HostModel::DupGrpRec* recs; const uint32_t* member; const int* goff;   // members of group g: recs[member[goff[g] .. goff[g + 1])]
  const int64_t* moff; const int32_t* mst; const int32_t* mlen; const int32_t* mgid;   // merged map of sequence s: [moff[s], moff[s + 1]), starts ascending
  const int32_t* groups; int n_work;   // the analysed groups; work item w: group groups[w >> 1], polarity (w & 1) ? +1 : -1
  const int32_t* retry_item; const int32_t* retry_resume; const long long* retry_off;   // second attempt: items, the step their writes resume at, scratch offsets
  AncMember* state; long long n_members;   // per polarity, one AncMember per group member
  uint8_t* popular; long long pop_cap;     // first attempt: pop_cap steps of `popular` per warp
  int* ticket;
  unsigned int* written; uint8_t* plane; const int64_t* fwd_off;   // written: bit per position of both strands; plane: forward codes (0xFF: untouched)
  int* ovf_n; int32_t* ovf_item; int32_t* ovf_resume; long long* ovf_need;
  int* err;   // [0] != 0: a position was written twice, [1] its sequence id, [2] its index
  double threshold, match1, mismatch1, leave_bonus; int verify;   // matchScore(1), mismatchScore(1), mismatchScore(3) * -1 (:423-431)
};
__device__ __forceinline__ uint8_t anc_code(const RefD& ref, int sid, int i) { return ref.contig(sid >> 1, sid & 1).at(i); }
__device__ __forceinline__ void anc_add(AncMember& s, double v) {   // SimilarityAnalysis.addScore
  s.cum += v;
  if (s.cum > s.best) { s.best = s.cum; s.best_idx = s.cur; }
}
__device__ __forceinline__ void anc_write(const AncD& A, int sid, int index, uint8_t code) {   // :339-351 + OverriddenSequence.putEncoded
  const long long bit = A.ref.gstart[sid] - A.ref.gstart[0] + index;
  const unsigned m = 1u << (unsigned)(bit & 31);
  if (atomicOr(&A.written[bit >> 5], m) & m) {
    if (atomicCAS(&A.err[0], 0, 1) == 0) { A.err[1] = sid; A.err[2] = index; }
    return;
  }
  if (!(sid & 1)) A.plane[A.fwd_off[sid >> 1] + index] = code;
}
__global__ void __launch_bounds__(128) xm_ancestry_kernel(AncD A) {
  __shared__ int hist_s[4][16];
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  int* hist = hist_s[threadIdx.x >> 5];
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  while (true) {
    int t = 0;
    if (lane == 0) t = atomicAdd(A.ticket, 1);
    t = __shfl_sync(full, t, 0);
    if (t >= A.n_work) break;
    int item = t, resume = 0;
    uint8_t* popular = A.popular + warp * A.pop_cap; long long cap = A.pop_cap;
    if (A.retry_item) { item = A.retry_item[t]; resume = A.retry_resume[t]; popular = A.popular + A.retry_off[t]; cap = A.retry_off[t + 1] - A.retry_off[t]; }
    const int gid = A.groups[item >> 1], pol = (item & 1) ? 1 : -1;
    const int m0 = A.goff[gid], nm = A.goff[gid + 1] - m0;
    const int L = A.recs[A.member[m0]].count_len >> 24;
    const bool small = nm <= 32;   // one member per lane: its analysis stays in registers
    AncMember* S = A.state + (item & 1) * A.n_members + m0;
    AncMember reg; reg.sid = 0; reg.start = reg.bound = reg.cur = reg.best_idx = 0; reg.flags = 0; reg.cum = reg.best = 0;
    // set-up: analysisBounds :384-421 (every merged entry has >= 3 instances, so interestingBefore / After are the neighbouring
    // entries) and interest :88-90 (the entry saved at this (sequence, start) still belongs to this group)
    int n_av = 0, n_in = 0; long long need = 0;
    for (int j = lane; j < nm; j += 32) {
      const HostModel::DupGrpRec r = A.recs[A.member[m0 + j]];
      const int slen = A.ref.len[r.sid >> 1];
      const long long lo = A.moff[r.sid], hi = A.moff[r.sid + 1];
      long long a = lo, b = hi;   // first entry with start >= r.st
      while (a < b) { const long long mid = (a + b) >> 1; if (A.mst[mid] < r.st) a = mid + 1; else b = mid; }
      const bool exact = a < hi && A.mst[a] == r.st;
      const int middle = r.st + L / 2;
      int initial, bound;
      if (pol > 0) {
        initial = middle + 1; bound = slen;
        const long long nx = exact ? a + 1 : a;
        if (nx < hi) bound = (middle + (A.mst[nx] + A.mlen[nx] / 2)) / 2 + 1;
      } else {
        initial = middle; bound = -1;
        if (a > lo) bound = ((A.mst[a - 1] + A.mlen[a - 1] / 2) + middle) / 2;
      }
      const bool valid = (bound - initial) * pol >= 0;
      const bool in = valid && exact && A.mgid[a] == gid;
      AncMember s;
      s.sid = r.sid; s.start = initial; s.bound = bound; s.cur = initial; s.best_idx = initial;
      s.flags = (valid ? ANC_AV : 0u) | (in ? ANC_IN : 0u);
      s.cum = s.best = A.threshold * (double)L;   // matchScore(length)
      n_av += valid ? 1 : 0; n_in += in ? 1 : 0;
      if (in) need = max(need, (long long)(bound - initial) * pol + 1);   // an interested analysis leaves at its bound at the latest
      if (small) reg = s; else S[j] = s;
    }
    n_av = __reduce_add_sync(full, n_av); n_in = __reduce_add_sync(full, n_in);
    for (int o = 16; o > 0; o >>= 1) need = max(need, __shfl_xor_sync(full, need, o));
    __syncwarp();
    long long step = 0;
    while (n_in >= 1 && n_av >= 3) {   // :94-137
      if (step >= cap) {   // out of scratch: the second attempt re-runs the analysis and writes from this step on
        if (lane == 0) { const int o = atomicAdd(A.ovf_n, 1); A.ovf_item[o] = item; A.ovf_resume[o] = (int32_t)step; A.ovf_need[o] = need; }
        break;
      }
      if (lane < 16) hist[lane] = 0;
      __syncwarp();
      for (int j = lane; j < nm; j += 32) {   // :96-102
        AncMember s;
        if (small) s = reg; else s = S[j];
        uint32_t f = s.flags & (ANC_AV | ANC_IN);
        if ((f & ANC_IN) && s.cur == s.bound) f |= ANC_NLI;
        if (f & ANC_AV) {
          if (s.cur < 0 || s.cur >= A.ref.len[s.sid >> 1]) { f |= ANC_NLA; if (f & ANC_IN) f |= ANC_NLI; }
          else atomicAdd(&hist[anc_code(A.ref, s.sid, s.cur)], 1);
        }
        if (small) reg.flags = f; else S[j].flags = f;
      }
      __syncwarp();
      // :103-111 the most frequent code, scanned in ascending code order; a tie gives 0 ('-')
      const int cnt = lane < 16 ? hist[lane] : 0;
      const int mx = __reduce_max_sync(full, cnt);
      const unsigned at_max = __ballot_sync(full, cnt == mx && cnt > 0);
      const uint8_t best = (mx == 0 || __popc(at_max) > 1) ? (uint8_t)0 : (uint8_t)(__ffs(at_max) - 1);
      if (lane == 0) popular[step] = best;
      __syncwarp();
      int av = 0, in = 0;
      for (int base = 0; base < nm; base += 32) {
        const int j = base + lane;
        bool leaves = false;
        AncMember s = reg;
        if (j < nm) {
          if (!small) s = S[j];
          const uint32_t f = s.flags;
          bool nli = (f & ANC_NLI) != 0, inn = (f & ANC_IN) != 0, ava = (f & ANC_AV) != 0;
          if (nli) {   // :112-117 a leaver with a neighbour and a non-negative score earns mismatchScore(3) * -1
            if (s.cur >= 0 && s.cur < A.ref.len[s.sid >> 1] && s.cum >= 0) anc_add(s, A.leave_bonus);
            inn = false;
          }
          if (f & ANC_NLA) ava = false;
          if (ava) {   // :119-123
            anc_add(s, anc_code(A.ref, s.sid, s.cur) == best ? A.match1 : A.mismatch1);
            if (s.cum < 0) { ava = false; if (inn) { nli = true; inn = false; } }
          }
          if (ava) s.cur += pol;   // :126
          s.flags = (ava ? ANC_AV : 0u) | (inn ? ANC_IN : 0u);
          if (small) reg = s; else S[j] = s;
          av += ava ? 1 : 0; in += inn ? 1 : 0;
          leaves = nli && step >= resume;
        }
        // :127-136 an analysis that stops being interested writes the popular codes over its own sequence, from its start up to its
        // best index (never reaching its bound); the whole warp writes one leaver's stretch at a time
        unsigned lm = __ballot_sync(full, leaves);
        while (lm) {
          const int src = __ffs(lm) - 1; lm &= lm - 1;
          const int sid = __shfl_sync(full, s.sid, src), start = __shfl_sync(full, s.start, src);
          const int bound = __shfl_sync(full, s.bound, src), best_idx = __shfl_sync(full, s.best_idx, src);
          const long long end = min(min((long long)(bound - start) * pol, (long long)(best_idx - start) * pol + 1), step + 1);
          for (long long off = lane; off < end; off += 32) {
            const int index = start + (int)off * pol;
            const uint8_t anc = popular[off], here = anc_code(A.ref, sid, index);
            if ((anc != here && anc != 0) || A.verify) anc_write(A, sid, index, (uint8_t)(anc | here));
          }
        }
      }
      n_av = __reduce_add_sync(full, av); n_in = __reduce_add_sync(full, in);
      step++;
    }
    __syncwarp();
  }
}
// The forward code plane into the packed reference (one thread per 16-bit word); counts the positions whose code changed.
__global__ void __launch_bounds__(256) xm_anc_apply_kernel(uint16_t* words, long long n_words, const int64_t* word_off, const int32_t* len, int n_contigs,
                                                           const int64_t* fwd_off, const uint8_t* plane, unsigned long long* n_changed) {
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned changed = 0;
  if (w < n_words) {
    int lo = 0, hi = n_contigs;   // the last contig whose first word is <= w
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (word_off[mid] <= w) lo = mid; else hi = mid; }
    const long long i0 = (w - word_off[lo]) * 4;
    if (w >= word_off[lo] && i0 < len[lo]) {
      unsigned v = words[w];
      const unsigned v0 = v;
      for (int k = 0; k < 4 && i0 + k < len[lo]; k++) {
        const unsigned c = plane[fwd_off[lo] + i0 + k];
        if (c == 0xFF) continue;
        if (((v >> (4 * k)) & 15u) != c) { changed++; v = (v & ~(15u << (4 * k))) | (c << (4 * k)); }
      }
      if (v != v0) words[w] = (uint16_t)v;
    }
  }
  const unsigned total = __reduce_add_sync(0xffffffffu, changed);
  if ((threadIdx.x & 31) == 0 && total) atomicAdd(n_changed, (unsigned long long)total);
}
__global__ void xm_anc_keys_kernel(const HostModel::DupGrpRec* recs, int n, uint32_t* keys, uint32_t* vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { keys[i] = (uint32_t)recs[i].gid; vals[i] = (uint32_t)i; }
}
// goff[g] = first member of group g in the sorted order, goff[n_groups] = n
__global__ void xm_anc_goff_kernel(const uint32_t* keys, int n, int n_groups, int* goff) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int k = (int)keys[i];
  for (int g = (i == 0 ? 0 : (int)keys[i - 1] + 1); g <= k; g++) goff[g] = i;
  if (i == n - 1) for (int g = k + 1; g <= n_groups; g++) goff[g] = n;
}
// xm_parse_reads: scans on the parser's stream, with its own scratch
template <class In, class Out>
static cudaError_t pz_scan(xm_handle* h, const In* in, Out* out, int n, bool inclusive) {
  cudaStream_t st = h->parse_stream;
  size_t tb = 0;
  if (inclusive) cub::DeviceScan::InclusiveSum(nullptr, tb, in, out, n, st); else cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, n, st);
  if (!h->d_pz_tmp.ensure(tb + 16)) return cudaErrorMemoryAllocation;
  return inclusive ? cub::DeviceScan::InclusiveSum(h->d_pz_tmp.p, tb, in, out, n, st) : cub::DeviceScan::ExclusiveSum(h->d_pz_tmp.p, tb, in, out, n, st);
}
static unsigned pz_blocks(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

extern "C" {

int xm_create(const xm_params* p, int device, xm_handle** out) {
  if (!p || !out) return XM_ERR_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n < 1 || device < 0 || device >= n) {
    fprintf(stderr, "xmapper_b200: no CUDA device %d (this library has no CPU path)\n", device);
    return XM_ERR_CUDA;
  }
  xm_handle* h = new xm_handle();
  h->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete h; return XM_ERR_CUDA; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  h->sm_count = prop.multiProcessorCount;
  { int nb = 0; if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, xm_align_kernel<true>, XM_BLOCK, 0) == cudaSuccess && nb > 0) h->blocks_per_sm = nb; }
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&h->parse_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&h->ev2) != cudaSuccess || cudaEventCreate(&h->ev3) != cudaSuccess || cudaEventCreate(&h->ev4) != cudaSuccess || cudaEventCreate(&h->ev5) != cudaSuccess) {
    fprintf(stderr, "xmapper_b200: stream/event creation failed: %s\n", cudaGetErrorString(cudaGetLastError()));
    xm_destroy(h); return XM_ERR_CUDA;
  }
  if (cudaFuncSetAttribute(xm_align_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (XM_FULL_BLOCK / 32) * XM_STAGE_BYTES) != cudaSuccess) { cudaGetLastError(); h->use_tma = false; }
  for (auto& sl : h->slots) {
    if (cudaStreamCreateWithFlags(&sl.copy, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&sl.h2d_done, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&sl.kernels_done, cudaEventDisableTiming) != cudaSuccess || cudaEventCreate(&sl.ev0) != cudaSuccess || cudaEventCreate(&sl.ev1) != cudaSuccess) {
      fprintf(stderr, "xmapper_b200: stream/event creation failed: %s\n", cudaGetErrorString(cudaGetLastError()));
      xm_destroy(h); return XM_ERR_CUDA;
    }
  }
  size_t stack = 8 * 1024;  // the call graph has no cycle any more: ptxas reports 3.5 KB for the deepest chain; 8 KB leaves margin without reserving 10 GB of local memory
  if (const char* e = getenv("XM_STACK_BYTES")) stack = (size_t)atoll(e);
  {  // the limit belongs to the whole primary context (the JVM, torch, other handles): only ever raise it
    size_t cur = 0;
    if (cudaDeviceGetLimit(&cur, cudaLimitStackSize) != cudaSuccess) cur = 0;
    if (cur < stack && cudaDeviceSetLimit(cudaLimitStackSize, stack) != cudaSuccess) {
      fprintf(stderr, "xmapper_b200: cannot raise the device stack limit to %zu bytes: %s\n", stack, cudaGetErrorString(cudaGetLastError()));
      xm_destroy(h); return XM_ERR_CUDA;
    }
  }
  if (const char* e = getenv("XM_WS_BYTES")) h->ws_budget = (size_t)atoll(e);
  if (const char* e = getenv("XM_QCYCLES")) h->probe_cycles = atoi(e) != 0;
  size_t free_b = 0, total_b = 0;
  // long reads need big per-warp arenas; the kernels are latency bound, so the budget decides how many warps stay resident:
  // up to 60 % of the free HBM (1 kbp reads: 24 GB -> 10 warps per SM, 3.7 s per 100 k reads; 59 GB -> 1.8 s)
  if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && h->ws_budget > free_b * 6 / 10) h->ws_budget = free_b * 6 / 10;
  Params& q = h->m.prm;
  q.mutation = p->mutation_penalty; q.ins_start = p->insertion_start_penalty; q.ins_ext = p->insertion_extension_penalty;
  q.del_start = p->deletion_start_penalty; q.del_ext = p->deletion_extension_penalty; q.max_error_rate = p->max_error_rate;
  q.unaligned = p->unaligned_penalty; q.ambiguity = p->ambiguity_penalty; q.span = p->max_penalty_span;
  q.max_num_matches = p->max_num_matches; q.start_free = 0; q.pen_tab = nullptr; q.cls_tab = nullptr;
  h->m.gapmers = p->enable_gapmers ? 1 : 0;
  *out = h;
  return XM_OK;
}

void xm_destroy(xm_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->comm && nccl_api().ok) { nccl_api().CommDestroy(h->comm); h->comm = nullptr; }
  for (auto& sl : h->slots) {
    if (sl.copy) cudaStreamDestroy(sl.copy);
    for (cudaEvent_t e : {sl.h2d_done, sl.kernels_done, sl.ev0, sl.ev1}) if (e) cudaEventDestroy(e);
  }
  if (h->fmt_text) h->pinned->give(h->fmt_text, h->fmt_cap);
  if (h->pz_stage) h->pinned->give(h->pz_stage, h->pz_stage_cap);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->parse_stream) cudaStreamDestroy(h->parse_stream);
  for (cudaEvent_t e : {h->ev2, h->ev3, h->ev4, h->ev5}) if (e) cudaEventDestroy(e);
  delete h;
}
const char* xm_last_error(const xm_handle* h) { return h ? h->err.c_str() : "null handle"; }

int xm_set_reference(xm_handle* h, int32_t n, const uint16_t* const* packed4, const int32_t* lengths) {
  if (!h || n < 1 || !packed4 || !lengths) return XM_ERR_ARG;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  long long total = 0;
  for (int i = 0; i < n; i++) { if (lengths[i] < 1) { h->err = "contig of length < 1"; return XM_ERR_ARG; } total += lengths[i]; }
  // XM_POSITION_BIAS (tests): global position of the first contig, as if a reference of that many bases preceded it - moves every
  // index position past 2^32 without a multi-gigabase reference in memory
  long long bias = 0; if (const char* e = getenv("XM_POSITION_BIAS")) bias = atoll(e);
  if (bias < 0 || bias + 2 * total >= (1LL << 40)) { h->err = "reference too large for 40-bit global positions"; return XM_ERR_ARG; }
  h->m.position_bias = bias;
  h->m.set_reference(n, packed4, lengths);
  h->counts_enabled = false;
  return XM_OK;
}
int xm_set_index_length(xm_handle* h, int32_t n_used, int32_t capacity, int32_t max_count, const int64_t* offsets, const uint8_t* overfull, const uint32_t* positions) {
  if (!h || n_used < 0 || capacity < 1 || !offsets) return XM_ERR_ARG;
  if (max_count > 32766) { h->err = "max_count > 32766"; return XM_ERR_ARG; }
  if (offsets[0] != 0) { h->err = "xm_set_index_length: offsets[0] != 0"; return XM_ERR_ARG; }
  for (int32_t b = 0; b < capacity; b++) {
    const int64_t cnt = offsets[b + 1] - offsets[b];
    if (cnt < 0) { h->err = "xm_set_index_length: offsets are not non-decreasing"; return XM_ERR_ARG; }
    if (cnt > 65535 || (cnt > max_count && !(overfull && overfull[b]))) { h->err = "xm_set_index_length: a bucket that is not overfull holds more than max_count positions"; return XM_ERR_ARG; }
  }
  if (offsets[capacity] >= (1LL << 40)) { h->err = "xm_set_index_length: more than 2^40 positions"; return XM_ERR_ARG; }
  if (offsets[capacity] > 0 && !positions) return XM_ERR_ARG;
  if (h->m.wide_positions()) { h->err = "xm_set_index_length: the reference needs more than 32 bits per position - use xm_set_index_length_wide"; return XM_ERR_ARG; }
  h->m.set_index_length(n_used, capacity, max_count, offsets, overfull, positions);
  return XM_OK;
}
int xm_set_index_length_wide(xm_handle* h, int32_t n_used, int32_t capacity, int32_t max_count, const int64_t* offsets, const uint8_t* overfull, const uint64_t* positions) {
  if (!h || n_used < 0 || capacity < 1 || !offsets) return XM_ERR_ARG;
  if (max_count > 32766) { h->err = "max_count > 32766"; return XM_ERR_ARG; }
  if (offsets[0] != 0) { h->err = "xm_set_index_length_wide: offsets[0] != 0"; return XM_ERR_ARG; }
  for (int32_t b = 0; b < capacity; b++) {
    const int64_t cnt = offsets[b + 1] - offsets[b];
    if (cnt < 0) { h->err = "xm_set_index_length_wide: offsets are not non-decreasing"; return XM_ERR_ARG; }
    if (cnt > 65535 || (cnt > max_count && !(overfull && overfull[b]))) { h->err = "xm_set_index_length_wide: a bucket that is not overfull holds more than max_count positions"; return XM_ERR_ARG; }
  }
  if (offsets[capacity] >= (1LL << 40)) { h->err = "xm_set_index_length_wide: more than 2^40 positions"; return XM_ERR_ARG; }
  if (offsets[capacity] > 0 && !positions) return XM_ERR_ARG;
  for (int64_t i = 0; i < offsets[capacity]; i++) if (positions[i] >= (uint64_t)h->m.position_end) { h->err = "xm_set_index_length_wide: a position lies past the end of the reference"; return XM_ERR_ARG; }
  h->m.set_index_length(n_used, capacity, max_count, offsets, overfull, positions, true);
  return XM_OK;
}
int xm_finish_index(xm_handle* h, int32_t min_interesting, int32_t max_built) {
  if (!h || min_interesting < 1 || max_built < 0) return XM_ERR_ARG;
  h->m.finish_index(min_interesting, max_built);
  return XM_OK;
}
// xm_build_index(h, max_used, 0): the tables of M/HashBlock_Database.java built by the kernels above.  min_interesting > 0 / max_short:
// the database's minInterestingSize and maxNumShortMatches when a caller chooses them (:68-89; xm_infer_ancestors), else the defaults.
static int build_index_device(xm_handle* h, int max_used, int min_interesting = -1, int max_short = 5) {
  HostModel& M = h->m;
  int hi = 0; std::vector<int> cap;
  if (!M.index_plan(max_used, hi, cap, h->err, min_interesting)) return XM_ERR_ARG;
  if (hi > 16000) { h->err = "xm_build_index: lengths above 16000 are not supported by the device builder (16-bit block coordinates within a slice)"; return XM_ERR_ARG; }
  int key_bits = 33; while ((1 << (key_bits - 32)) <= hi) key_bits++;   // sort key = used << 32 | bucket
  cudaStream_t st = h->stream;
  if (int rc = upload_reference(h)) return rc;
  IndexBuildD B;
  B.ref = h->ref;
  const int slice_len = 8192;
  std::vector<int> sc, ss, amb_sc, amb_ss;   // plain slices; slices whose window holds an IUPAC-ambiguous base (the host builder's test)
  for (int c = 0; c < M.n_contigs; c++) for (int s0 = 0; s0 < M.len[(size_t)c]; s0 += slice_len) {
    bool amb = false;
    if (M.ref_ambiguous) {
      SeqView seq = M.contig_view(c, 0);
      const int scan_end = std::min(seq.len, std::min(seq.len, s0 + slice_len) + 4 * hi + 256);
      for (int i = s0; i < scan_end && !amb; i++) amb = bp_is_ambiguous(seq.at(i));
    }
    if (amb) { amb_sc.push_back(c); amb_ss.push_back(s0); } else { sc.push_back(c); ss.push_back(s0); }
  }
  const int n_amb = (int)amb_sc.size();
  if (n_amb && slice_len + 4 * hi + 256 > 32000) { h->err = "xm_build_index: hash lengths this long are not supported on IUPAC-ambiguous references (16-bit window coordinates)"; return XM_ERR_ARG; }
  DevBuf d_amb_sc, d_amb_ss, d_amb_arena, d_keep, d_pos_hi;
  DevBuf d_sc, d_ss, d_cap, d_cnt, d_keys_a, d_keys_b, d_vals_a, d_vals_b, d_tmp, d_run_key, d_run_cnt, d_nruns, d_cnt64, d_kept, d_first, d_bbase, d_buckets, d_pos;
  if (!d_sc.upload(sc.data(), sc.size() * 4) || !d_ss.upload(ss.data(), ss.size() * 4) || !d_cap.upload(cap.data(), cap.size() * 4) || !d_cnt.ensure(64)) { h->err = "out of device memory (index build)"; return XM_ERR_CUDA; }
  B.slice_contig = (const int*)d_sc.p; B.slice_start = (const int*)d_ss.p; B.n_slices = (int)sc.size(); B.slice_len = slice_len;
  B.hi = hi; B.min_interesting = M.min_interesting; B.gapmers = M.gapmers; B.cap = (const int*)d_cap.p;
  const int blocks = h->sm_count * 8, warps = blocks * 4;
  B.arena_bytes = (((long long)(slice_len + hi + 2 + 32) * 2 * (long long)sizeof(HB16)) + 255) & ~255LL;
  if (!h->d_ws.ensure((size_t)warps * (size_t)B.arena_bytes)) { h->err = "out of device memory (index build workspace)"; return XM_ERR_CUDA; }
  B.arenas = (char*)h->d_ws.p;
  B.n_entries = (unsigned long long*)d_cnt.p; B.ticket = (int*)((char*)d_cnt.p + 16); B.fail = (int*)((char*)d_cnt.p + 32);
  // ambiguous slices: one warp (one block) each, with an arena for the window's MultiHashBlock pyramid and its possibilities
  IndexBuildD A = B;
  int amb_blocks = 0;
  if (n_amb) {
    if (!d_amb_sc.upload(amb_sc.data(), amb_sc.size() * 4) || !d_amb_ss.upload(amb_ss.data(), amb_ss.size() * 4)) { h->err = "out of device memory (index build)"; return XM_ERR_CUDA; }
    const long long wlen = slice_len + 4LL * hi + 256;
    long long amb_mb = 64; if (const char* e = getenv("XM_INDEX_AMB_ARENA_MB")) amb_mb = std::max(8, atoi(e));
    A.arena_bytes = ((((wlen + 3) * 4 + 15) & ~15LL) + (10 * wlen + 256) * 20 + 64 + (amb_mb << 20) + 255) & ~255LL;
    amb_blocks = std::min(n_amb, h->sm_count * 2);
    while (amb_blocks > 1 && !d_amb_arena.ensure((size_t)amb_blocks * (size_t)A.arena_bytes)) { cudaGetLastError(); amb_blocks /= 2; }
    if (!d_amb_arena.ensure((size_t)amb_blocks * (size_t)A.arena_bytes)) { h->err = "out of device memory (ambiguous index workspace)"; return XM_ERR_CUDA; }
    A.arenas = (char*)d_amb_arena.p;
    A.slice_contig = (const int*)d_amb_sc.p; A.slice_start = (const int*)d_amb_ss.p; A.n_slices = n_amb;
  }
  DevBuf d_hist;
  if (!d_hist.ensure(((size_t)hi + 2) * 8)) { h->err = "out of device memory (index build)"; return XM_ERR_CUDA; }
  int used_lo = 0, used_hi = 0x7fffffff;   // the block lengths of the current chunk
  auto emit = [&](unsigned long long* keys, void* vals, unsigned long long cap_entries) -> int {
    B.keys = A.keys = keys; B.vals = A.vals = vals; B.wide = A.wide = M.wide_positions() ? 1 : 0; B.cap_entries = A.cap_entries = cap_entries;
    B.used_lo = A.used_lo = used_lo; B.used_hi = A.used_hi = used_hi;
    B.hist = A.hist = (keys == nullptr) ? (unsigned long long*)d_hist.p : nullptr;
    if (keys == nullptr) CK(cudaMemsetAsync(d_hist.p, 0, ((size_t)hi + 2) * 8, st));
    CK(cudaMemsetAsync(d_cnt.p, 0, 64, st));
    if (B.n_slices) xm_index_emit_kernel<<<blocks, 128, 0, st>>>(B);
    if (n_amb) { CK(cudaMemsetAsync(B.ticket, 0, 4, st)); xm_index_emit_amb_kernel<<<amb_blocks, 32, 0, st>>>(A); }
    CK(cudaGetLastError());
    return XM_OK;
  };
  // pass 1 counts the entries, pass 2 writes them
  if (int rc = emit(nullptr, nullptr, 0)) return rc;
  unsigned long long cnt_host[8] = {0};
  CK(cudaMemcpyAsync(cnt_host, d_cnt.p, 64, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  unsigned long long E = cnt_host[0];
  if (const int fs = (int)(cnt_host[4] & 0xffffffffu)) { h->err = "xm_build_index: MultiHashBlock expansion of the reference ran out of workspace (status " + std::to_string(fs) + "); raise XM_INDEX_AMB_ARENA_MB or use the host builder (n_threads > 0)"; return XM_ERR_ARG; }
  M.tables.assign((size_t)hi + 1, HostTable());
  std::vector<long long> tab_bbase((size_t)hi + 2, 0), tab_koff((size_t)hi + 2, 0);
  const bool wide = M.wide_positions();
  const int pos_bits = wide ? 40 : 32;
  // One sort handles < 2^31 entries and has to fit the device next to the finished tables: the build is chunked by block length.
  // Every chunk runs the emit kernels again with a length filter (the pyramids are cheap next to the sorts).
  std::vector<unsigned long long> hist((size_t)hi + 2, 0);
  CK(cudaMemcpy(hist.data(), d_hist.p, ((size_t)hi + 2) * 8, cudaMemcpyDeviceToHost));
  unsigned long long max_entries = (1ull << 31) - 1;
  {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
      // per entry: key / value double buffers, run keys + counts, sort scratch, keep flag, the four 64-bit scan arrays over the runs (a
      // random reference has almost one run per entry), and the finished tables (bucket word + position)
      const unsigned long long per_entry = 2 * (8 + (wide ? 8 : 4)) + 12 + 8 + 1 + 32 + 13;
      max_entries = std::min<unsigned long long>(max_entries, (unsigned long long)((double)free_b * 0.75) / per_entry);
    }
    if (const char* e = getenv("XM_INDEX_MAX_ENTRIES")) max_entries = std::min<unsigned long long>(max_entries, std::max(1LL, atoll(e)));
  }
  std::vector<std::pair<int, int>> chunks;
  {
    int lo = 0; unsigned long long acc = 0;
    for (int k = 0; k <= hi; k++) {
      if (hist[(size_t)k] > max_entries) { h->err = "xm_build_index: the blocks of length " + std::to_string(k) + " alone (" + std::to_string(hist[(size_t)k]) + " entries) exceed what one sort can hold on this device; use the host builder (n_threads > 0) or upload the tables"; return XM_ERR_ARG; }
      if (acc + hist[(size_t)k] > max_entries) { chunks.push_back({lo, k - 1}); lo = k; acc = 0; }
      acc += hist[(size_t)k];
    }
    chunks.push_back({lo, hi});
  }
  if (getenv("XM_TRACE_SETUP")) fprintf(stderr, "[xm] index build: %llu entries for block lengths <= %d, at most %llu per sort: %zu chunk(s) of lengths\n", E, hi, max_entries, chunks.size());
  h->d_buckets.clear(); h->d_positions.clear(); h->d_positions_hi.clear(); h->d_ix_chunks.clear();   // the old tables go before the new ones are allocated
  std::vector<TableD> tabs((size_t)hi + 1);
  for (int k = 0; k <= hi; k++) { tabs[(size_t)k].capacity = 1; tabs[(size_t)k].max_count = 1; tabs[(size_t)k].buckets = nullptr; tabs[(size_t)k].positions = nullptr; tabs[(size_t)k].positions_hi = nullptr; }
  auto sort_fill = [&](auto pos_tag) -> int {
    using PosT = decltype(pos_tag);
    if (!d_keys_a.ensure(E * 8) || !d_keys_b.ensure(E * 8) || !d_vals_a.ensure(E * sizeof(PosT)) || !d_vals_b.ensure(E * sizeof(PosT))) { h->err = "out of device memory (index entries)"; return XM_ERR_CUDA; }
    if (int rc = emit((unsigned long long*)d_keys_a.p, d_vals_a.p, E)) return rc;
    int n = (int)E;
    // (used, bucket, position) order: sort by position, then a stable sort by (used << 32 | bucket)
    size_t t1 = 0, t2 = 0, t3 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, (const PosT*)d_vals_a.p, (PosT*)d_vals_b.p, (const unsigned long long*)d_keys_a.p, (unsigned long long*)d_keys_b.p, n, 0, pos_bits, st);
    cub::DeviceRadixSort::SortPairs(nullptr, t2, (const unsigned long long*)d_keys_b.p, (unsigned long long*)d_keys_a.p, (const PosT*)d_vals_b.p, (PosT*)d_vals_a.p, n, 0, key_bits, st);
    if (!d_run_key.ensure(E * 8) || !d_run_cnt.ensure(E * 4) || !d_nruns.ensure(16)) { h->err = "out of device memory (index runs)"; return XM_ERR_CUDA; }
    cub::DeviceRunLengthEncode::Encode(nullptr, t3, (const unsigned long long*)d_keys_a.p, (unsigned long long*)d_run_key.p, (int*)d_run_cnt.p, (int*)d_nruns.p, n, st);
    size_t t4 = 0, t5 = 0;
    cub::TransformInputIterator<unsigned long long, IxUnmulti, const unsigned long long*> unmulti((const unsigned long long*)d_keys_a.p, IxUnmulti());
    if (n_amb) {
      cub::DeviceSelect::Flagged(nullptr, t4, unmulti, (const unsigned char*)nullptr, (unsigned long long*)d_keys_b.p, (int*)d_nruns.p, n, st);
      cub::DeviceSelect::Flagged(nullptr, t5, (const PosT*)d_vals_a.p, (const unsigned char*)nullptr, (PosT*)d_vals_b.p, (int*)d_nruns.p, n, st);
    }
    size_t tb = t1 > t2 ? t1 : t2; if (t3 > tb) tb = t3; if (t4 > tb) tb = t4; if (t5 > tb) tb = t5;
    if (!d_tmp.ensure(tb + (size_t)E * 8 + 4096)) { h->err = "out of device memory (index sort)"; return XM_ERR_CUDA; }
    size_t q = tb;
    CK(cub::DeviceRadixSort::SortPairs(d_tmp.p, q, (const PosT*)d_vals_a.p, (PosT*)d_vals_b.p, (const unsigned long long*)d_keys_a.p, (unsigned long long*)d_keys_b.p, n, 0, pos_bits, st));
    q = tb;
    CK(cub::DeviceRadixSort::SortPairs(d_tmp.p, q, (const unsigned long long*)d_keys_b.p, (unsigned long long*)d_keys_a.p, (const PosT*)d_vals_b.p, (PosT*)d_vals_a.p, n, 0, key_bits, st));
    const unsigned long long* skeys = (const unsigned long long*)d_keys_a.p; const PosT* svals = (const PosT*)d_vals_a.p;
    if (n_amb) {   // PackedMap.add(preventDuplicates): drop the repeated possibilities of multi-blocks, clear the flag bit
      if (!d_keep.ensure((size_t)n + 16)) { h->err = "out of device memory (index de-duplication)"; return XM_ERR_CUDA; }
      xm_index_dedupe_kernel<<<(n + 255) / 256, 256, 0, st>>>(skeys, svals, n, (unsigned char*)d_keep.p);
      q = tb; CK(cub::DeviceSelect::Flagged(d_tmp.p, q, unmulti, (const unsigned char*)d_keep.p, (unsigned long long*)d_keys_b.p, (int*)d_nruns.p, n, st));
      q = tb; CK(cub::DeviceSelect::Flagged(d_tmp.p, q, svals, (const unsigned char*)d_keep.p, (PosT*)d_vals_b.p, (int*)d_nruns.p, n, st));
      int kept_n = 0;
      CK(cudaMemcpyAsync(&kept_n, d_nruns.p, 4, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      n = kept_n; skeys = (const unsigned long long*)d_keys_b.p; svals = (const PosT*)d_vals_b.p;
    }
    q = tb;
    CK(cub::DeviceRunLengthEncode::Encode(d_tmp.p, q, skeys, (unsigned long long*)d_run_key.p, (int*)d_run_cnt.p, (int*)d_nruns.p, n, st));
    int n_runs = 0;
    CK(cudaMemcpyAsync(&n_runs, d_nruns.p, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    // offsets: run_start = scan of counts, kept_off = scan of the counts of the buckets that are not overfull
    if (!d_cnt64.ensure(((size_t)n_runs + 1) * 16) || !d_kept.ensure(((size_t)n_runs + 1) * 16) || !d_first.ensure(((size_t)hi + 2) * 4)) { h->err = "out of device memory (index offsets)"; return XM_ERR_CUDA; }
    long long* kept = (long long*)d_kept.p; long long* kept_off = kept + (n_runs + 1);
    long long* cnt64 = (long long*)d_cnt64.p; long long* run_start = cnt64 + (n_runs + 1);
    xm_index_runs_kernel<<<(n_runs + 256) / 256, 256, 0, st>>>((const unsigned long long*)d_run_key.p, (const int*)d_run_cnt.p, n_runs, kept, max_short);
    CK(cudaMemsetAsync(cnt64, 0, ((size_t)n_runs + 1) * 8, st));  // widen the int32 counts to int64 for the scan
    CK(cudaMemcpy2DAsync(cnt64, 8, d_run_cnt.p, 4, 4, (size_t)n_runs, cudaMemcpyDeviceToDevice, st));
    q = tb; CK(cub::DeviceScan::ExclusiveSum(d_tmp.p, q, (const long long*)kept, kept_off, n_runs + 1, st));
    q = tb; CK(cub::DeviceScan::ExclusiveSum(d_tmp.p, q, (const long long*)cnt64, run_start, n_runs + 1, st));
    xm_index_first_run_kernel<<<(hi + 2 + 255) / 256, 256, 0, st>>>((const unsigned long long*)d_run_key.p, n_runs, hi, (int*)d_first.p);
    std::vector<int> first((size_t)hi + 2);
    CK(cudaMemcpyAsync(first.data(), d_first.p, first.size() * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    std::vector<long long> koff((size_t)hi + 2);
    for (int k = 0; k <= hi + 1; k++) CK(cudaMemcpy(&koff[(size_t)k], kept_off + first[(size_t)k], 8, cudaMemcpyDeviceToHost));
    std::vector<long long> bbase((size_t)hi + 2, 0);
    long long words = 0;
    for (int k = 0; k <= hi; k++) { bbase[(size_t)k] = words; if (first[(size_t)k + 1] > first[(size_t)k]) words += cap[(size_t)k]; }
    const long long n_pos = koff[(size_t)hi + 1];
    tab_bbase = bbase; tab_koff = koff;
    if (!d_bbase.upload(bbase.data(), bbase.size() * 8) || !d_buckets.ensure((size_t)words * 8 + 16) || !d_pos.ensure((size_t)n_pos * 4 + 16) || (wide && !d_pos_hi.ensure((size_t)n_pos + 16))) { h->err = "out of device memory (index tables)"; return XM_ERR_CUDA; }
    IndexFillD<PosT> F;
    F.run_key = (const unsigned long long*)d_run_key.p; F.run_cnt = (const int*)d_run_cnt.p; F.run_start = run_start; F.kept_off = kept_off; F.n_runs = n_runs;
    F.first_run = (const int*)d_first.p; F.cap = (const int*)d_cap.p; F.bucket_base = (const long long*)d_bbase.p;
    F.sorted_pos = svals; F.buckets = (unsigned long long*)d_buckets.p; F.positions = (uint32_t*)d_pos.p; F.positions_hi = wide ? (uint8_t*)d_pos_hi.p : nullptr;
    xm_index_fill_kernel<<<(n_runs + 255) / 256, 256, 0, st>>>(F);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    for (int k = 1; k <= hi; k++) {
      if (first[(size_t)k + 1] <= first[(size_t)k]) continue;   // no block of this length: PackedMap(1, 1)
      HostTable& T = M.tables[(size_t)k];
      T.capacity = cap[(size_t)k]; T.max_count = HostModel::max_count_for(k, max_short);
      T.buckets.resize((size_t)T.capacity);
      CK(cudaMemcpy(T.buckets.data(), (const unsigned long long*)d_buckets.p + bbase[(size_t)k], (size_t)T.capacity * 8, cudaMemcpyDeviceToHost));
      const long long np = koff[(size_t)k + 1] - koff[(size_t)k];
      T.positions.resize((size_t)np);
      if (np) CK(cudaMemcpy(T.positions.data(), (const uint32_t*)d_pos.p + koff[(size_t)k], (size_t)np * 4, cudaMemcpyDeviceToHost));
      if (wide) { T.positions_hi.resize((size_t)np); if (np) CK(cudaMemcpy(T.positions_hi.data(), (const uint8_t*)d_pos_hi.p + koff[(size_t)k], (size_t)np, cudaMemcpyDeviceToHost)); }
    }
    return XM_OK;
  };
  for (const auto& ch : chunks) {
    used_lo = ch.first; used_hi = ch.second;
    E = 0; for (int k = used_lo; k <= used_hi; k++) E += hist[(size_t)k];
    if (E == 0) continue;
    if (int rc = wide ? sort_fill((unsigned long long)0) : sort_fill((uint32_t)0)) return rc;
    // the chunk's tables stay where the fill kernel wrote them
    const size_t at = h->d_ix_chunks.size();
    h->d_ix_chunks.resize(at + 3);
    std::swap(h->d_ix_chunks[at], d_buckets); std::swap(h->d_ix_chunks[at + 1], d_pos); std::swap(h->d_ix_chunks[at + 2], d_pos_hi);
    for (int k = std::max(1, used_lo); k <= used_hi; k++) {
      const HostTable& T = M.tables[(size_t)k];
      tabs[(size_t)k].capacity = T.capacity; tabs[(size_t)k].max_count = T.max_count;
      if (T.buckets.empty()) continue;
      tabs[(size_t)k].buckets = (const uint64_t*)h->d_ix_chunks[at].p + tab_bbase[(size_t)k]; tabs[(size_t)k].positions = (const uint32_t*)h->d_ix_chunks[at + 1].p + tab_koff[(size_t)k];
      if (wide) tabs[(size_t)k].positions_hi = (const uint8_t*)h->d_ix_chunks[at + 2].p + tab_koff[(size_t)k];
    }
  }
  M.max_built = hi; M.index_finished = true; M.generation++;
  // the tables stay where the fill kernels wrote them: the device view is current, nothing is uploaded again
  if (!h->d_tables.upload(tabs.data(), tabs.size() * sizeof(TableD))) { h->err = "device upload failed (index tables)"; return XM_ERR_CUDA; }
  h->tables_host = tabs;
  h->mirrored_generation = M.generation; h->mirrored_dup_generation = ~0ull;   // mirror_model still uploads the duplication table and sets the views
  return XM_OK;
}

static int infer_ancestors_device(xm_handle* h, double threshold, int min_interesting, int max_short, bool verify, int64_t* n_changed) {
  HostModel& M = h->m;
  const bool trace = getenv("XM_TRACE_SETUP") != nullptr;
  const double t_begin = now_s();
  *n_changed = 0;
  // a) the temporary index: lengths up to 2 * minDuplicationLength (M/DuplicationDetector.java:17-31)
  const int min_len = M.choose_min_dup_len(), max_len = 2 * min_len;
  if (max_len > 64) { h->err = "xm_infer_ancestors: duplication lengths above 64 (a reference over 2^32 bases) are not supported by the device scan"; return XM_ERR_ARG; }
  if (int rc = build_index_device(h, max_len, min_interesting, max_short)) return rc;
  if (int rc = mirror_model(h)) return rc;
  const double t_index = now_s();
  // b) the group scan: DuplicationDetector(3 copies, window 1) :129-214, every member of every group
  cudaStream_t st = h->stream;
  const int blocks = h->sm_count * 8, warps = blocks * 4;
  DupScan<HostModel::DupGrpRec> S;
  if (int rc = dup_scan<true>(h, min_len, max_len, 3, S)) return rc;
  if (S.recs.size() >= (1ull << 31)) { h->err = "xm_infer_ancestors: more than 2^31 duplication group members"; return XM_ERR_ARG; }
  const int n_rec = (int)S.recs.size(), n_groups = S.n_groups;
  const double t_scan = now_s();
  // c) saveDuplications with the groups kept, every sequence; the groups some merged entry still references (DuplicationDetector.getAll)
  std::vector<std::vector<std::pair<int32_t, HostModel::Dup>>> by_seq;
  M.merge_duplication_groups(S.recs, 1, by_seq);
  const size_t n_seqs = 2 * (size_t)M.n_contigs;
  std::vector<int64_t> moff(n_seqs + 1, 0);
  std::vector<int32_t> mst, mlen, mgid;
  std::vector<char> referenced((size_t)n_groups, 0);
  for (size_t s = 0; s < n_seqs; s++) {
    for (const auto& e : by_seq[s]) { mst.push_back(e.first); mlen.push_back(e.second.length); mgid.push_back(e.second.group); referenced[(size_t)e.second.group] = 1; }
    moff[s + 1] = (int64_t)mst.size();
  }
  std::vector<int32_t> groups;
  for (int g = 0; g < n_groups; g++) if (referenced[(size_t)g]) groups.push_back(g);
  const double t_merge = now_s();
  double t_analysis = t_merge;
  int n_retried = 0;
  DevBuf d_ctr, d_keys, d_vals, d_keys2, d_vals2, d_tmp, d_goff, d_moff, d_mst, d_mlen, d_mgid, d_groups, d_state, d_pop, d_bits, d_plane, d_fwd_off, d_ovf, d_retry, d_retry_off;
  if (!groups.empty()) {
    if (!d_moff.upload(moff.data(), moff.size() * 8) || !d_mst.upload(mst.data(), mst.size() * 4) || !d_mlen.upload(mlen.data(), mlen.size() * 4) ||
        !d_mgid.upload(mgid.data(), mgid.size() * 4) || !d_groups.upload(groups.data(), groups.size() * 4)) { h->err = "device upload failed (merged duplications)"; return XM_ERR_CUDA; }
    // the member CSR: records sorted by group id
    int key_bits = 1; while (key_bits < 32 && (1ll << key_bits) < (long long)n_groups) key_bits++;
    if (!d_keys.ensure((size_t)n_rec * 4) || !d_vals.ensure((size_t)n_rec * 4) || !d_keys2.ensure((size_t)n_rec * 4) || !d_vals2.ensure((size_t)n_rec * 4) ||
        !d_goff.ensure(((size_t)n_groups + 1) * 4)) { h->err = "out of device memory (ancestry groups)"; return XM_ERR_CUDA; }
    xm_anc_keys_kernel<<<(n_rec + 255) / 256, 256, 0, st>>>((const HostModel::DupGrpRec*)S.d_recs.p, n_rec, (uint32_t*)d_keys.p, (uint32_t*)d_vals.p);
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, (const uint32_t*)d_keys.p, (uint32_t*)d_keys2.p, (const uint32_t*)d_vals.p, (uint32_t*)d_vals2.p, n_rec, 0, key_bits, st);
    if (!d_tmp.ensure(tb + 16)) { h->err = "out of device memory (ancestry group sort)"; return XM_ERR_CUDA; }
    CK(cub::DeviceRadixSort::SortPairs(d_tmp.p, tb, (const uint32_t*)d_keys.p, (uint32_t*)d_keys2.p, (const uint32_t*)d_vals.p, (uint32_t*)d_vals2.p, n_rec, 0, key_bits, st));
    xm_anc_goff_kernel<<<(n_rec + 255) / 256, 256, 0, st>>>((const uint32_t*)d_keys2.p, n_rec, n_groups, (int*)d_goff.p);
    // d) the analyses
    long long pop_cap = 32768;   // steps of one analysis the first attempt holds (XM_ANC_SCRATCH: forces the second attempt in tests)
    if (const char* e = getenv("XM_ANC_SCRATCH")) pop_cap = std::max(1LL, atoll(e));
    std::vector<int64_t> fwd_off((size_t)M.n_contigs + 1, 0);
    for (int c = 0; c < M.n_contigs; c++) fwd_off[(size_t)c + 1] = fwd_off[(size_t)c] + M.len[(size_t)c];
    const int n_work = 2 * (int)groups.size();
    const size_t bit_words = (size_t)((M.total_fr + 31) / 32);
    if (!d_state.ensure(2 * (size_t)n_rec * sizeof(AncMember)) || !d_pop.ensure((size_t)warps * (size_t)pop_cap) || !d_bits.ensure(bit_words * 4) ||
        !d_plane.ensure((size_t)M.total_forward) || !d_fwd_off.upload(fwd_off.data(), fwd_off.size() * 8) || !d_ovf.ensure((size_t)n_work * 16 + 64) || !d_ctr.ensure(64)) {
      h->err = "out of device memory (ancestry analyses)"; return XM_ERR_CUDA;
    }
    CK(cudaMemsetAsync(d_bits.p, 0, bit_words * 4, st));
    CK(cudaMemsetAsync(d_plane.p, 0xFF, (size_t)M.total_forward, st));
    AncD A;
    A.ref = h->ref; A.recs = (const HostModel::DupGrpRec*)S.d_recs.p; A.member = (const uint32_t*)d_vals2.p; A.goff = (const int*)d_goff.p;
    A.moff = (const int64_t*)d_moff.p; A.mst = (const int32_t*)d_mst.p; A.mlen = (const int32_t*)d_mlen.p; A.mgid = (const int32_t*)d_mgid.p;
    A.groups = (const int32_t*)d_groups.p; A.n_work = n_work;
    A.retry_item = nullptr; A.retry_resume = nullptr; A.retry_off = nullptr;
    A.state = (AncMember*)d_state.p; A.n_members = n_rec;
    A.popular = (uint8_t*)d_pop.p; A.pop_cap = pop_cap;
    int* counters = (int*)d_ctr.p;   // [0] ticket, [1] overflow count, [2..4] error record
    A.ticket = counters; A.ovf_n = counters + 1; A.err = counters + 2;
    A.written = (unsigned int*)d_bits.p; A.plane = (uint8_t*)d_plane.p; A.fwd_off = (const int64_t*)d_fwd_off.p;
    A.ovf_need = (long long*)d_ovf.p; A.ovf_item = (int32_t*)((char*)d_ovf.p + (size_t)n_work * 8); A.ovf_resume = A.ovf_item + n_work;
    A.threshold = threshold;
    A.match1 = threshold * 1;                   // matchScore(1)
    A.mismatch1 = -1 + threshold * 1;           // mismatchScore(1)
    A.leave_bonus = (-3 + threshold * 3) * -1;  // mismatchScore(3) * -1
    A.verify = verify ? 1 : 0;
    CK(cudaMemsetAsync(d_ctr.p, 0, 64, st));
    xm_ancestry_kernel<<<blocks, 128, 0, st>>>(A);
    CK(cudaGetLastError());
    int ctr[8] = {0};
    CK(cudaMemcpyAsync(ctr, d_ctr.p, 32, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (ctr[1] > 0) {   // second attempt: the analyses that ran out of scratch, each with the scratch its bounds can need
      const int n_ovf = ctr[1];
      n_retried = n_ovf;
      std::vector<long long> need((size_t)n_ovf);
      std::vector<int32_t> ovf_item((size_t)n_ovf), ovf_resume((size_t)n_ovf);
      CK(cudaMemcpy(need.data(), A.ovf_need, (size_t)n_ovf * 8, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(ovf_item.data(), A.ovf_item, (size_t)n_ovf * 4, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(ovf_resume.data(), A.ovf_resume, (size_t)n_ovf * 4, cudaMemcpyDeviceToHost));
      size_t free_b = 0, total_b = 0;
      long long budget = 1LL << 30;
      if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) budget = std::max(budget, (long long)(free_b / 2));
      for (int i0 = 0; i0 < n_ovf;) {   // batches of analyses whose scratch fits the budget
        std::vector<int32_t> retry;   // items, then resume steps
        std::vector<long long> off(1, 0);
        int i1 = i0;
        while (i1 < n_ovf && (i1 == i0 || off.back() + need[(size_t)i1] <= budget)) { off.push_back(off.back() + ((need[(size_t)i1] + 15) & ~15LL)); i1++; }
        const int nb = i1 - i0;
        retry.insert(retry.end(), ovf_item.begin() + i0, ovf_item.begin() + i1);
        retry.insert(retry.end(), ovf_resume.begin() + i0, ovf_resume.begin() + i1);
        if (!d_retry.upload(retry.data(), retry.size() * 4) || !d_retry_off.upload(off.data(), off.size() * 8) || !d_pop.ensure((size_t)off.back() + 16)) {
          h->err = "out of device memory (ancestry analyses, second attempt)"; return XM_ERR_CUDA;
        }
        A.retry_item = (const int32_t*)d_retry.p; A.retry_resume = A.retry_item + nb; A.retry_off = (const long long*)d_retry_off.p;
        A.popular = (uint8_t*)d_pop.p; A.n_work = nb;
        CK(cudaMemsetAsync(d_ctr.p, 0, 8, st));   // ticket and overflow count; the error record stays
        xm_ancestry_kernel<<<blocks, 128, 0, st>>>(A);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(ctr, d_ctr.p, 32, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (ctr[1] != 0) { h->err = "xm_infer_ancestors: an analysis outran the scratch its bounds allow (internal error)"; return XM_ERR_STATE; }
        i0 = i1;
      }
    }
    t_analysis = now_s();
    if (ctr[2]) {   // OverriddenSequence.putEncoded :19-27
      const int sid = ctr[3];
      h->err = "Cannot override contig " + std::to_string(sid >> 1) + ((sid & 1) ? "-rev" : "") + "[" + std::to_string(ctr[4]) + "]: already overridden";
      return XM_ERR_STATE;
    }
    // e) the forward plane into the packed reference, and back into the handle's reference
    const long long n_words = (long long)M.words.size();
    xm_anc_apply_kernel<<<(unsigned)((n_words + 255) / 256), 256, 0, st>>>((uint16_t*)h->d_words.p, n_words, (const int64_t*)h->d_word_off.p, (const int32_t*)h->d_len.p, M.n_contigs,
                                                                          (const int64_t*)d_fwd_off.p, (const uint8_t*)d_plane.p, (unsigned long long*)((char*)d_ctr.p + 32));
    CK(cudaGetLastError());
    unsigned long long changed = 0;
    CK(cudaMemcpyAsync(&changed, (char*)d_ctr.p + 32, 8, cudaMemcpyDeviceToHost, st));
    std::vector<uint16_t> words((size_t)n_words);
    CK(cudaMemcpyAsync(words.data(), h->d_words.p, (size_t)n_words * 2, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    M.words.swap(words);
    *n_changed = (int64_t)changed;
  }
  if (trace) fprintf(stderr, "[xm] infer ancestors: index %.3f s, scan %.3f s (%d members of %d groups), merge %.3f s (%zu groups analysed), analysis %.3f s (%d analyses re-run), apply %.3f s (%lld positions changed)\n",
                     t_index - t_begin, t_scan - t_index, n_rec, n_groups, t_merge - t_scan, groups.size(), t_analysis - t_merge, n_retried, now_s() - t_analysis, (long long)*n_changed);
  return XM_OK;
}

int xm_build_index(xm_handle* h, int32_t max_used, int32_t n_threads) {
  if (!h) return XM_ERR_ARG;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  if (h->m.n_contigs < 1) { h->err = "reference not set"; return XM_ERR_STATE; }
  if (n_threads <= 0) { CK(cudaSetDevice(h->device)); return build_index_device(h, max_used); }  // the device builder; n_threads > 0: the host builder it is checked against
  if (!h->m.build_index(max_used, n_threads, h->err)) return XM_ERR_ARG;
  return XM_OK;
}
int xm_get_index_length(xm_handle* h, int32_t n, int32_t* capacity, int32_t* max_count, int64_t* n_positions, int64_t* offsets, uint8_t* overfull, uint32_t* positions) {
  if (!h || n < 0 || n > h->m.max_built || (size_t)n >= h->m.tables.size()) return XM_ERR_ARG;
  int c, m; int64_t np;
  if (positions && h->m.wide_positions()) { h->err = "xm_get_index_length: the reference needs more than 32 bits per position - use xm_get_index_length_wide"; return XM_ERR_ARG; }
  h->m.get_index_length(n, c, m, np, offsets, overfull, positions);
  if (capacity) *capacity = c;
  if (max_count) *max_count = m;
  if (n_positions) *n_positions = np;
  return XM_OK;
}
int xm_get_index_length_wide(xm_handle* h, int32_t n, int32_t* capacity, int32_t* max_count, int64_t* n_positions, int64_t* offsets, uint8_t* overfull, uint64_t* positions) {
  if (!h || n < 0 || n > h->m.max_built || (size_t)n >= h->m.tables.size()) return XM_ERR_ARG;
  int c, m; int64_t np;
  h->m.get_index_length(n, c, m, np, offsets, overfull, nullptr, positions);
  if (capacity) *capacity = c;
  if (max_count) *max_count = m;
  if (n_positions) *n_positions = np;
  return XM_OK;
}
int xm_index_info(xm_handle* h, int32_t* mi, int32_t* mb) { if (!h) return XM_ERR_ARG; if (mi) *mi = h->m.min_interesting; if (mb) *mb = h->m.max_built; return XM_OK; }
int xm_set_duplications(xm_handle* h, int32_t window, double granularity, int32_t contig, int32_t n, const int32_t* starts) {
  if (!h || window < 1 || contig < 0 || contig >= h->m.n_contigs || n < 0) return XM_ERR_ARG;
  h->m.set_duplications(window, granularity, contig, n, starts);
  return XM_OK;
}
int xm_build_duplications(xm_handle* h, int32_t min_len, int32_t max_len, int32_t min_copies, int32_t window) {
  if (!h || window < 1) return XM_ERR_ARG;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  if (!h->m.index_finished) { h->err = "index not set"; return XM_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  return build_duplications_device(h, min_len, max_len, min_copies, window);
}
int xm_build_duplications_host(xm_handle* h, int32_t min_len, int32_t max_len, int32_t min_copies, int32_t window) {
  if (!h || window < 1) return XM_ERR_ARG;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  if (!h->m.index_finished) { h->err = "index not set"; return XM_ERR_STATE; }
  h->m.build_duplications(min_len, max_len, min_copies, window);
  return XM_OK;
}
int xm_infer_ancestors(xm_handle* h, double dissimilarity_threshold, int32_t min_interesting_size, int32_t max_short_matches, int32_t verify_no_duplicate_analyses,
                       int64_t* n_changed) {
  if (!h || !n_changed) return XM_ERR_ARG;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  if (h->m.n_contigs < 1) { h->err = "reference not set"; return XM_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  const int rc = infer_ancestors_device(h, dissimilarity_threshold, min_interesting_size > 0 ? min_interesting_size : -1, max_short_matches < 0 ? 5 : max_short_matches,
                                        verify_no_duplicate_analyses != 0, n_changed);
  // The temporary index replaced the handle's tables: in every case the index and the duplication table are gone, as after
  // xm_set_reference; the codes changed only on success (infer_ancestors_device touches HostModel::words last).
  if (rc != XM_OK) *n_changed = 0;
  h->m.reference_codes_changed();
  h->d_ix_chunks.clear(); h->d_buckets.clear(); h->d_positions.clear(); h->d_positions_hi.clear();
  return rc;
}
int xm_get_reference(xm_handle* h, int32_t contig, uint16_t* packed4) {
  if (!h || !packed4) return XM_ERR_ARG;
  if (h->m.n_contigs < 1) { h->err = "reference not set"; return XM_ERR_STATE; }
  if (contig < 0 || contig >= h->m.n_contigs) return XM_ERR_ARG;
  const size_t nw = ((size_t)h->m.len[(size_t)contig] + 3) / 4;
  memcpy(packed4, h->m.words.data() + h->m.word_off[(size_t)contig], nw * 2);
  return XM_OK;
}
int xm_get_duplications(xm_handle* h, int32_t contig, int32_t* n, int32_t* starts) {
  if (!h || contig < 0 || contig >= h->m.n_contigs) return XM_ERR_ARG;
  auto& v = h->m.dup_starts[(size_t)contig];
  if (n) *n = (int)v.size();
  if (starts) for (size_t i = 0; i < v.size(); i++) starts[i] = v[i];
  return XM_OK;
}


// MatchDatabase.addAlignments for the batch whose results sit in L.out: reference-base planes + raw variant records.
static int var_reduce_now(xm_handle* h) {
  if (h->var_n == h->var_reduced_n) return XM_OK;
  unsigned long long n_out = 0;
  if (!var_sort_reduce((VarRec*)h->d_var.p, h->var_n, h->var_scratch, h->stream, &n_out, h->err)) return XM_ERR_CUDA;
  h->var_n = n_out; h->var_reduced_n = n_out;
  return XM_OK;
}
static int var_reserve(xm_handle* h, unsigned long long want) {   // keeps recs[0, var_n)
  if (want <= h->var_cap) return XM_OK;
  const unsigned long long ncap = want + want / 2 + 65536;
  if (!h->d_var.grow((size_t)ncap * sizeof(VarRec), (size_t)h->var_n * sizeof(VarRec), h->stream)) { h->err = "out of device memory (variant table)"; return XM_ERR_CUDA; }
  h->var_cap = ncap;
  return XM_OK;
}
// enqueue: one launch of xm_counts_kernel behind the align kernels; the number of records it wanted to write comes back in *n_after
// with the caller's next synchronisation.  finish: grows the record buffer and emits the batch's records again if they did not fit.
struct CountsPending { CountsD C; VarOut V; };
static int counts_enqueue(xm_handle* h, const LaunchD& L, int nq, long long n_seqs_total, int& launches, CountsPending& P, unsigned long long* n_after) {
  cudaStream_t st = h->stream;
  CountsD& C = P.C; VarOut& V = P.V;
  h->var_gen++;
  C.planes = (int32_t*)h->d_planes.p; C.contig_off = (const int64_t*)h->d_contig_off.p; C.end_fraction = h->end_fraction;
  V.order = nullptr;
  V.first_gid = h->have_batch_info ? h->info_first_gid : h->next_gid;
  if (h->have_batch_info && !h->info_order.empty()) {
    if ((long long)h->info_order.size() != n_seqs_total) { h->err = "xm_counts_batch_info: order keys do not match the number of sequences of the batch"; return XM_ERR_ARG; }
    if (!h->d_order.ensure((size_t)n_seqs_total * 8)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
    CK(cudaMemcpyAsync(h->d_order.p, h->info_order.data(), (size_t)n_seqs_total * 8, cudaMemcpyHostToDevice, st));
    V.order = (const int64_t*)h->d_order.p;
  }
  h->next_gid = V.first_gid + n_seqs_total; h->have_batch_info = false;
  int rc = var_reserve(h, h->var_n + (unsigned long long)n_seqs_total * 4 + 4096);   // ~1.6 records per 150 bp read at 1 % differences
  if (rc != XM_OK) return rc;
  if (!h->d_var_n.ensure(16)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
  V.recs = (VarRec*)h->d_var.p; V.n = (unsigned long long*)h->d_var_n.p; V.cap = h->var_cap;
  CK(cudaMemcpyAsync(h->d_var_n.p, &h->var_n, 8, cudaMemcpyHostToDevice, st));
  xm_counts_kernel<true><<<(nq + 127) / 128, 128, 0, st>>>(h->ref, L.batch, L.out, C, V, nq);
  launches++;
  CK(cudaMemcpyAsync(n_after, h->d_var_n.p, 8, cudaMemcpyDeviceToHost, st));
  return XM_OK;
}
static int counts_finish(xm_handle* h, const LaunchD& L, int nq, int& launches, CountsPending& P, unsigned long long n_after) {
  cudaStream_t st = h->stream;
  while (n_after > h->var_cap) {
    // more records than room: grow and emit the batch's records again (the planes were already updated)
    int rc = var_reserve(h, n_after);
    if (rc != XM_OK) return rc;
    P.V.recs = (VarRec*)h->d_var.p; P.V.cap = h->var_cap;
    CK(cudaMemcpyAsync(h->d_var_n.p, &h->var_n, 8, cudaMemcpyHostToDevice, st));
    xm_counts_kernel<false><<<(nq + 127) / 128, 128, 0, st>>>(h->ref, L.batch, L.out, P.C, P.V, nq);
    launches++;
    CK(cudaMemcpyAsync(&n_after, h->d_var_n.p, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
  }
  h->var_n = n_after;
  if (h->var_n - h->var_reduced_n > (1ull << 24) && h->var_n - h->var_reduced_n > h->var_reduced_n / 2) return var_reduce_now(h);
  return XM_OK;
}

struct NSeqsAt {   // n_seqs_per_query[i] as int64, 0 past the end
  const uint8_t* p; int n;
  __host__ __device__ long long operator()(int i) const { return i < n ? (long long)p[i] : 0LL; }
};
static int align_batch_impl(xm_handle* h, SlotLease& lease, bool wait_h2d, int32_t nq, const uint16_t* d_packed, int64_t n_words, const int64_t* d_seq_word_off, const int32_t* d_seq_len,
                            const uint8_t* d_n_seqs, const double* d_expected, const double* d_per, int32_t max_seq_len, long long n_seqs_total_hint, xm_results** out) {
  xm_handle::BatchSlot& slot = lease.slot();
  if (out) *out = nullptr;
  if (!h || nq < 0 || !out) return XM_ERR_ARG;
  CK(cudaSetDevice(h->device));
  // from here to the CSR fill this call owns the handle's stream and work buffers; the copies before and after run on the slot's stream
  std::unique_lock<std::mutex> compute(h->compute_mu);
  int rc = mirror_model(h);
  if (rc != XM_OK) return rc;
  (void)n_words;
  cudaStream_t st = h->stream;
  if (wait_h2d) CK(cudaStreamWaitEvent(st, slot.h2d_done, 0));
  // owned here until the call succeeds (or ends with XM_ERR_QUERY, where the results are still delivered): every early
  // error return frees the results and gives the pinned slab back to the pool
  std::unique_ptr<xm_results> R_owner(new xm_results());
  xm_results* R = R_owner.get();
  R->r.stats.assign(XM_STAT_COUNT, 0);
  if (nq == 0) { R->r.assemble(0, nullptr, nullptr, nullptr, nullptr); R->serial = slot.serial; R->slot = lease.i; R->nq = 0; *out = R_owner.release(); return XM_OK; }
  // first_seq = exclusive scan of n_seqs (cub, on the device: nq + 1 items, the last one reads as 0 so that first_seq[nq] is the total)
  size_t scan0_tmp = 0;
  {
    cub::TransformInputIterator<long long, NSeqsAt, cub::CountingInputIterator<int>> it(cub::CountingInputIterator<int>(0), NSeqsAt{d_n_seqs, nq});
    cub::DeviceScan::ExclusiveSum(nullptr, scan0_tmp, it, (long long*)nullptr, nq + 1, st);
  }
  if (!slot.d_first_seq.ensure(((size_t)nq + 1) * 8) || !h->d_chunk.ensure(scan0_tmp + 16)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
  CK(cudaEventRecord(slot.ev0, st));
  {
    cub::TransformInputIterator<long long, NSeqsAt, cub::CountingInputIterator<int>> it(cub::CountingInputIterator<int>(0), NSeqsAt{d_n_seqs, nq});
    size_t tb = scan0_tmp;
    CK(cub::DeviceScan::ExclusiveSum(h->d_chunk.p, tb, it, (long long*)slot.d_first_seq.p, nq + 1, st));
  }
  // sizes the result arena: exact when the caller counted the sequences (xm_align_batch), else the bound of two per query
  const long long n_seqs_total = n_seqs_total_hint >= 0 ? n_seqs_total_hint : 2LL * nq;
  int launches = 0;

  // result arena
  long long want_c = (long long)nq * 2 + 4096, want_s = n_seqs_total * 2 + 4096, want_b = n_seqs_total * 6 + 16384;
  if (h->cap_choices < want_c) { if (!h->d_choices.ensure((size_t)want_c * sizeof(OutChoice))) { h->err = "out of device memory"; return XM_ERR_CUDA; } h->cap_choices = want_c; }
  if (h->cap_sas < want_s) { if (!h->d_sas.ensure((size_t)want_s * sizeof(OutSA))) { h->err = "out of device memory"; return XM_ERR_CUDA; } h->cap_sas = want_s; }
  if (h->cap_blocks < want_b) { if (!h->d_blocks.ensure((size_t)want_b * 16)) { h->err = "out of device memory"; return XM_ERR_CUDA; } h->cap_blocks = want_b; }
  if (!h->d_q.ensure((size_t)nq * sizeof(OutQuery)) || !h->d_misc.ensure(512) || !h->d_ids_a.ensure((size_t)nq * 4) || !h->d_ids_b.ensure((size_t)nq * 4) || !h->d_ids_full.ensure((size_t)nq * 4)) {
    h->err = "out of device memory"; return XM_ERR_CUDA;
  }
  // misc: [0..2] used (u64) [3..16] stats (u64) [20..27] ints: 0 ticket, 1 n_need_more, 2 n_out_full, 4 ticket of tier 0, 5 n_need_more of tier 0;
  // [32..38] the stats as they stood after the first pass
  CK(cudaMemsetAsync(h->d_misc.p, 0, 512, st));
  unsigned long long* d_used = (unsigned long long*)h->d_misc.p;
  unsigned long long* d_stats = d_used + 3;
  int* d_ints = (int*)(d_used + 20);
  unsigned long long* d_easy_stats = d_used + 32;

  LaunchD L;
  L.ref = h->ref; L.ix = h->ix; L.dup = h->dup; L.prm = h->m.prm;
  L.batch.n_queries = nq; L.batch.packed = d_packed; L.batch.seq_word_off = d_seq_word_off; L.batch.seq_len = d_seq_len;
  L.batch.first_seq = (const int64_t*)slot.d_first_seq.p; L.batch.expected_inner = d_expected; L.batch.per_penalty = d_per;
  L.out.q = (OutQuery*)h->d_q.p; L.out.choices = (OutChoice*)h->d_choices.p; L.out.cap_choices = h->cap_choices;
  L.out.sas = (OutSA*)h->d_sas.p; L.out.cap_sas = h->cap_sas; L.out.blocks = (int32_t*)h->d_blocks.p; L.out.cap_blocks = h->cap_blocks;
  L.out.used = d_used; L.out.stats = d_stats;
  L.ticket = d_ints; L.n_need_more = d_ints + 1; L.n_out_full = d_ints + 2;
  L.out_full = (int32_t*)h->d_ids_full.p;
  L.q_cycles = nullptr; L.n_ids_ptr = nullptr;
  if (h->probe_cycles) { if (!h->d_qcycles.ensure((size_t)nq * 8)) { h->err = "out of device memory"; return XM_ERR_CUDA; } L.q_cycles = (long long*)h->d_qcycles.p; }

  const int block = XM_BLOCK, warps_per_block = XM_BLOCK / 32;
  float align_ms_tier0 = 0, easy_ms = 0, tier_ms[XM_NUM_TIERS] = {0};
  unsigned long long easy_stats[7] = {0, 0, 0, 0, 0, 0, 0};
  // One launch of the align kernel.  tier < 0: the first pass (blocks of 4 warps); tier >= 0: the full aligner (one resident wave of
  // blocks of `cpb` warps).  n_ids_dev != nullptr: the query count is on the device (n_ids is its bound) - nothing comes back to the host.
  auto launch_tier = [&](int tier, const int32_t* ids, int n_ids, const int* n_ids_dev, int32_t* need_more_out, int* ticket, int* n_need_more,
                         cudaEvent_t e0, cudaEvent_t e1) -> int {
    int cpb = warps_per_block, blocks = 1;
    long long arena = 0;
    if (tier < 0) {
      arena = easy_arena_bytes(max_seq_len, 2);
      long long max_warps = (long long)(h->ws_budget / (size_t)arena);
      long long warps = (long long)h->sm_count * h->blocks_per_sm * warps_per_block;  // one resident wave: the kernel is persistent (ticket loop)
      if (warps > max_warps) warps = max_warps;
      if (warps > n_ids) warps = n_ids;
      blocks = (int)((warps + warps_per_block - 1) / warps_per_block);
      if (blocks < 1) blocks = 1;
      if ((long long)blocks * warps_per_block * arena > (long long)h->ws_budget && blocks > 1) blocks = (int)(h->ws_budget / (size_t)(arena * warps_per_block));
    } else {
      cpb = XM_FULL_BLOCK / 32;
      const int slots = h->sm_count * XM_FULL_MIN_BLOCKS;   // resident blocks of the full kernel
      long long resident = (long long)slots * cpb;
      arena = tier_arena_bytes(tier, max_seq_len, 2, (long long)h->ws_budget, resident);
      long long clients = resident, max_warps = (long long)(h->ws_budget / (size_t)arena);
      if (clients > max_warps) clients = max_warps;
      if (clients > n_ids) clients = n_ids;
      if (clients < 1) { h->err = "workspace budget too small for one query"; return XM_ERR_CUDA; }
      if (clients < (long long)slots * cpb) cpb = (int)(clients / slots);
      if (cpb < 1) cpb = 1;
      blocks = (int)(clients / cpb);
      if (blocks > slots) blocks = slots;
    }
    if (blocks < 1) { h->err = "workspace budget too small for one block"; return XM_ERR_CUDA; }
    L.use_tma = (tier >= 0 && h->use_tma) ? 1 : 0;
    if (!h->d_ws.ensure((size_t)blocks * cpb * (size_t)arena)) { h->err = "out of device memory (workspace)"; return XM_ERR_CUDA; }
    CK(cudaMemsetAsync(ticket, 0, 4, st));
    CK(cudaMemsetAsync(n_need_more, 0, 4, st));
    // generation word of every arena's lattice map: 0 = not used since this launch began (whatever the buffer held before)
    if (tier >= 0) CK(cudaMemset2DAsync(h->d_ws.p, (size_t)arena, 0, 16, (size_t)blocks * cpb, st));
    L.ticket = ticket; L.n_need_more = n_need_more;
    L.ids = ids; L.n_ids = n_ids; L.n_ids_ptr = n_ids_dev; L.need_more = need_more_out; L.arenas = (char*)h->d_ws.p; L.arena_bytes = arena; L.last_tier = (tier == XM_NUM_TIERS - 1);
    L.need_more_key = nullptr;
    L.big_arenas = nullptr; L.big_arena_bytes = 0; L.n_big = 0; L.big_busy = nullptr;
    if (tier >= 0 && tier + 1 < XM_NUM_TIERS) {
      // a small pool of next-tier arenas inside this launch: the rare queries that outgrow their arena do not wait for a launch of their own
      const long long big = tier_arena_bytes(tier + 1, max_seq_len, 2, (long long)h->ws_budget, (long long)h->sm_count * XM_FULL_MIN_BLOCKS * (XM_FULL_BLOCK / 32));
      int n_big = 64;
      while (n_big > 0 && (long long)n_big * big > (long long)h->ws_budget / 4) n_big /= 2;
      if (n_big > 0 && big > arena && h->d_big.ensure((size_t)n_big * (size_t)big) && h->d_big_busy.ensure((size_t)n_big * 4)) {
        CK(cudaMemsetAsync(h->d_big_busy.p, 0, (size_t)n_big * 4, st));
        CK(cudaMemset2DAsync(h->d_big.p, (size_t)big, 0, 16, (size_t)n_big, st));
        L.big_arenas = (char*)h->d_big.p; L.big_arena_bytes = big; L.n_big = n_big; L.big_busy = (int*)h->d_big_busy.p;
      }
    }
    if (tier < 0) {
      if (!h->d_keys_a.ensure((size_t)n_ids * 4) || !h->d_keys_b.ensure((size_t)n_ids * 4)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
      CK(cudaMemsetAsync(h->d_keys_a.p, 0x80, (size_t)n_ids * 4, st));   // slots the kernel leaves unused sort last (key 0x80808080 < 0)
      L.need_more_key = (int32_t*)h->d_keys_a.p;
    }
    CK(cudaEventRecord(e0, st));
    L.dyn_stride = L.use_tma ? XM_STAGE_BYTES : 0;
    if (tier < 0) xm_align_kernel<true><<<blocks, block, 0, st>>>(L);
    else xm_align_kernel<false><<<blocks, 32 * cpb, (size_t)cpb * (size_t)L.dyn_stride, st>>>(L);
    CK(cudaEventRecord(e1, st));
    launches++;
    CK(cudaGetLastError());
    return XM_OK;
  };
  // The synchronous tier loop: every launch is followed by a read-back of its counters.  Used for what the fast path below leaves
  // over - queries that outgrew the tier-0 arenas (rare) and re-runs after growing the result arena (rarer).
  auto run_tiers_sync = [&](int first_tier, const int32_t* ids, int n_ids, int32_t* next_ids) -> int {
    for (int tier = first_tier; tier < XM_NUM_TIERS && n_ids > 0; tier++) {
      int rc3 = launch_tier(tier, ids, n_ids, nullptr, next_ids, d_ints, d_ints + 1, h->ev2, h->ev3);
      if (rc3 != XM_OK) return rc3;
      R->r.stats[XM_STAT_TIER0_QUERIES + tier] += n_ids;
      int counts[3];
      CK(cudaMemcpyAsync(counts, d_ints, 12, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      { float t = 0; cudaEventElapsedTime(&t, h->ev2, h->ev3); tier_ms[tier] += t; }
      int32_t* other = (next_ids == (int32_t*)h->d_ids_a.p) ? (int32_t*)h->d_ids_b.p : (int32_t*)h->d_ids_a.p;
      ids = next_ids; n_ids = counts[1]; next_ids = other;
    }
    return XM_OK;
  };
  // ---- fast path: first pass over every query, class sort of the queries it hands on, tier 0 of the full aligner - three launches
  // back to back, the count of handed-on queries stays on the device ----
  int32_t* ids_a = (int32_t*)h->d_ids_a.p; int32_t* ids_b = (int32_t*)h->d_ids_b.p;
  rc = launch_tier(-1, nullptr, nq, nullptr, ids_a, d_ints, d_ints + 1, h->ev2, h->ev3);
  if (rc != XM_OK) return rc;
  R->r.stats[XM_STAT_EASY_QUERIES] += nq;
  CK(cudaMemcpyAsync(d_easy_stats, d_stats, 7 * 8, cudaMemcpyDeviceToDevice, st));
  const int32_t* hard_ids = ids_a;
  if (nq > 1) {
    // longest first: the persistent full kernel ends when its slowest query does, so the queries the first pass scored worst (most
    // likely gapped) start first and the cheap ones fill the tail; co-resident warps also run the same kind of query, which the
    // instruction caches reward.  All nq slots are sorted (the unused ones carry the smallest key), so no count is needed here.
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairsDescending(nullptr, tb, (const int32_t*)h->d_keys_a.p, (int32_t*)h->d_keys_b.p, (const int32_t*)ids_a, ids_b, nq, 0, 32, st);
    if (!h->d_sort_tmp.ensure(tb + 16)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
    CK(cub::DeviceRadixSort::SortPairsDescending(h->d_sort_tmp.p, tb, (const int32_t*)h->d_keys_a.p, (int32_t*)h->d_keys_b.p, (const int32_t*)ids_a, ids_b, nq, 0, 32, st));
    hard_ids = ids_b;
  }
  int32_t* t0_need_more = (hard_ids == ids_a) ? ids_b : ids_a;
  rc = launch_tier(0, hard_ids, nq, d_ints + 1, t0_need_more, d_ints + 4, d_ints + 5, h->ev4, h->ev5);
  if (rc != XM_OK) return rc;
  int fast_counts[8];
  long long real_seqs_total = 0;
  CK(cudaMemcpyAsync(&real_seqs_total, (const long long*)slot.d_first_seq.p + nq, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(fast_counts, d_ints, 32, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(easy_stats, d_easy_stats, sizeof(easy_stats), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));   // sync 1 of 3 per batch
  { float t = 0; cudaEventElapsedTime(&t, h->ev2, h->ev3); easy_ms = t; align_ms_tier0 = t; cudaEventElapsedTime(&t, h->ev4, h->ev5); tier_ms[0] += t; }
  R->r.stats[XM_STAT_EASY_DONE] += nq - fast_counts[1];
  R->r.stats[XM_STAT_TIER0_QUERIES] += fast_counts[1];
  if (fast_counts[5] > 0) {   // queries that outgrew the tier-0 arenas (and found no pooled big arena)
    rc = run_tiers_sync(1, t0_need_more, fast_counts[5], (t0_need_more == ids_a) ? ids_b : ids_a);
    if (rc != XM_OK) return rc;
  }
  for (int round = 0; round < 4; round++) {   // result arena overflow: grow (keeping what was written) and re-run the affected queries
    int n_full = 0;
    CK(cudaMemcpy(&n_full, d_ints + 2, 4, cudaMemcpyDeviceToHost));
    if (n_full == 0) break;
    unsigned long long used[3];
    CK(cudaMemcpy(used, d_used, 24, cudaMemcpyDeviceToHost));
    auto grow = [&](DevBuf& b, long long& cap, unsigned long long& u, size_t elem) -> bool {
      const unsigned long long keep = std::min(u, (unsigned long long)cap);
      const long long ncap = (long long)(2 * std::max(u, (unsigned long long)cap)) + 4096;
      if (!b.grow((size_t)ncap * elem, (size_t)keep * elem, st)) return false;
      cap = ncap; u = keep;
      return true;
    };
    if (!grow(h->d_choices, h->cap_choices, used[0], sizeof(OutChoice)) || !grow(h->d_sas, h->cap_sas, used[1], sizeof(OutSA)) || !grow(h->d_blocks, h->cap_blocks, used[2], 16)) {
      h->err = "out of device memory (results)"; return XM_ERR_CUDA;
    }
    CK(cudaMemcpy(d_used, used, 24, cudaMemcpyHostToDevice));
    L.out.choices = (OutChoice*)h->d_choices.p; L.out.cap_choices = h->cap_choices; L.out.sas = (OutSA*)h->d_sas.p; L.out.cap_sas = h->cap_sas;
    L.out.blocks = (int32_t*)h->d_blocks.p; L.out.cap_blocks = h->cap_blocks;
    // the out_full list becomes the id list of the next round (copy it, the kernel will append to it again)
    CK(cudaMemcpy(ids_a, h->d_ids_full.p, (size_t)n_full * 4, cudaMemcpyDeviceToDevice));
    CK(cudaMemset(d_ints + 2, 0, 4));
    rc = run_tiers_sync(0, ids_a, n_full, ids_b);
    if (rc != XM_OK) return rc;
  }
  CountsPending counts_pending; unsigned long long var_n_after = 0;
  if (h->counts_enabled) {
    int rc2 = counts_enqueue(h, L, nq, real_seqs_total, launches, counts_pending, &var_n_after);
    if (rc2 != XM_OK) return rc2;
  }
  // D2H
  unsigned long long misc[20];
  CK(cudaMemcpyAsync(misc, h->d_misc.p, sizeof(misc), cudaMemcpyDeviceToHost, st));   // complete at sync 2
  // CSR assembly on the device, then one transfer into a pinned slab
  const bool host_times = getenv("XM_HOST_TIMES") != nullptr;
  const double t_csr0 = now_ms();
  const long long stride = (long long)nq + 1;
  size_t scan_tmp = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (const long long*)nullptr, (long long*)nullptr, (int)stride, st);
  if (!h->d_csr_cnt.ensure((size_t)stride * 32) || !h->d_csr_base.ensure((size_t)stride * 32) || !h->d_csr_tmp.ensure(scan_tmp + 16)) { h->err = "out of device memory (csr)"; return XM_ERR_CUDA; }
  long long* d_cnt = (long long*)h->d_csr_cnt.p; long long* d_base = (long long*)h->d_csr_base.p;
  xm_csr_count_kernel<<<(int)((stride + 255) / 256), 256, 0, st>>>(L.out, nq, d_cnt);
  for (int k = 0; k < 4; k++) { size_t tb = scan_tmp; CK(cub::DeviceScan::ExclusiveSum(h->d_csr_tmp.p, tb, d_cnt + k * stride, d_base + k * stride, (int)stride, st)); }
  long long totals[4];
  for (int k = 0; k < 4; k++) CK(cudaMemcpyAsync(&totals[k], d_base + k * stride + nq, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));   // sync 2 of 3 per batch
  CK(cudaGetLastError());
  if (h->counts_enabled) {
    int rc2 = counts_finish(h, L, nq, launches, counts_pending, var_n_after);
    if (rc2 != XM_OK) return rc2;
  }
  const long long n_comp = totals[0], n_ch = totals[1], n_sa = totals[2], n_blk = totals[3];
  {
    int64_t n[11] = {(int64_t)nq + 1, n_comp + 1, n_ch + 1, n_sa + 1, 4 * n_ch, 2 * n_sa, n_ch, n_sa, 4 * n_blk, (int64_t)nq, n_sa};
    const int elem[11] = {8, 8, 8, 8, 8, 8, 4, 4, 4, 4, 1};
    int64_t off = 0;
    for (int i = 0; i < 11; i++) { R->r.slab_off[i] = off; R->r.slab_n[i] = n[i]; off += (n[i] * elem[i] + 15) & ~(int64_t)15; }
    size_t slab_bytes = (size_t)off + 16;
    if (!slot.d_csr_slab.ensure(slab_bytes)) { h->err = "out of device memory (csr slab)"; return XM_ERR_CUDA; }
    R->pool = h->pinned;
    R->slab = h->pinned->take(slab_bytes, R->slab_cap);
    if (!R->slab) { h->err = "out of pinned host memory (results)"; return XM_ERR_CUDA; }
    char* d = (char*)slot.d_csr_slab.p;
    CsrD c;
    c.q_comp_off = (int64_t*)(d + R->r.slab_off[0]); c.comp_choice_off = (int64_t*)(d + R->r.slab_off[1]); c.choice_sa_off = (int64_t*)(d + R->r.slab_off[2]);
    c.sa_block_off = (int64_t*)(d + R->r.slab_off[3]); c.choice_f64 = (double*)(d + R->r.slab_off[4]); c.sa_f64 = (double*)(d + R->r.slab_off[5]);
    c.choice_inner = (int32_t*)(d + R->r.slab_off[6]); c.sa_contig = (int32_t*)(d + R->r.slab_off[7]); c.blocks = (int32_t*)(d + R->r.slab_off[8]);
    c.q_status = (int32_t*)(d + R->r.slab_off[9]); c.sa_reversed = (uint8_t*)(d + R->r.slab_off[10]);
    xm_csr_fill_kernel<<<(nq + 255) / 256, 256, 0, st>>>(L.out, nq, d_base, c);
    launches += 2;  // xm_csr_count + xm_csr_fill (the cub scans in between are library kernels)
    CK(cudaGetLastError());
    CK(cudaEventRecord(slot.ev1, st));  // device time of a step = every kernel from the scan of n_seqs to the CSR fill
    CK(cudaEventRecord(slot.kernels_done, st));
    if (h->probe_cycles) { R->r.q_cycles.resize((size_t)nq); CK(cudaMemcpyAsync(R->r.q_cycles.data(), h->d_qcycles.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st)); }
    slot.batch = L.batch; R->serial = slot.serial; R->slot = lease.i; R->nq = nq;
    compute.unlock();   // the next caller's kernels may follow; this call's results leave on the slot's own stream
    CK(cudaStreamWaitEvent(slot.copy, slot.kernels_done, 0));
    CK(cudaMemcpyAsync(R->slab, d, slab_bytes, cudaMemcpyDeviceToHost, slot.copy));
    CK(cudaStreamSynchronize(slot.copy));   // sync 3 of 3 per batch
    R->r.slab = (const char*)R->slab;
    if (host_times) fprintf(stderr, "[xm]   csr assembly + slab D2H (%.0f MB): %.1f ms\n", (double)slab_bytes / 1e6, now_ms() - t_csr0);
    R->r.stats[XM_STAT_D2H_BYTES] = (int64_t)(slab_bytes + sizeof(misc) + 32);
  }
  float ms = 0;
  cudaEventElapsedTime(&ms, slot.ev0, slot.ev1);
  R->r.stats[XM_STAT_KERNEL_NS] = (int64_t)((double)ms * 1e6);
  R->r.stats[XM_STAT_ALIGN_KERNEL_NS] = (int64_t)((double)align_ms_tier0 * 1e6);
  R->r.stats[XM_STAT_LAUNCHES] = launches;
  for (int t = 0; t < XM_NUM_TIERS && t < 3; t++) R->r.stats[XM_STAT_TIER0_NS + t] = (int64_t)((double)tier_ms[t] * 1e6);
  R->r.stats[XM_STAT_EASY_NS] = (int64_t)((double)easy_ms * 1e6);
  R->r.stats[XM_STAT_EASY_PROBES] = (int64_t)easy_stats[0]; R->r.stats[XM_STAT_EASY_HITS] = (int64_t)easy_stats[2]; R->r.stats[XM_STAT_EASY_STRAIGHT] = (int64_t)easy_stats[3];
  R->r.stats[XM_STAT_PROBES] = (int64_t)misc[3]; R->r.stats[XM_STAT_SEEDS] = (int64_t)misc[4]; R->r.stats[XM_STAT_HITS] = (int64_t)misc[5];
  R->r.stats[XM_STAT_STRAIGHT] = (int64_t)misc[6]; R->r.stats[XM_STAT_PATH_CALLS] = (int64_t)misc[7]; R->r.stats[XM_STAT_PATH_STEPS] = (int64_t)misc[8];
  R->r.stats[XM_STAT_PATH_CELLS] = (int64_t)misc[9];
  for (int i = 0; i < 7; i++) R->r.stats[XM_STAT_CYC_SEED + i] = (int64_t)misc[10 + i];
  *out = R_owner.release();
  const int32_t* q_status = (const int32_t*)(R->r.slab + R->r.slab_off[9]);
  for (int i = 0; i < nq; i++) if (q_status[i] != 0) { h->err = "at least one query could not be aligned on the device (see q_status)"; return XM_ERR_QUERY; }
  return XM_OK;
}

int xm_align_batch_device(xm_handle* h, int32_t nq, const uint16_t* d_packed, int64_t n_words, const int64_t* d_seq_word_off, const int32_t* d_seq_len,
                          const uint8_t* d_n_seqs, const double* d_expected, const double* d_per, int32_t max_seq_len, xm_results** out) {
  if (out) *out = nullptr;
  if (!h || nq < 0 || !out) return XM_ERR_ARG;
  SlotLease lease(h);
  return align_batch_impl(h, lease, false, nq, d_packed, n_words, d_seq_word_off, d_seq_len, d_n_seqs, d_expected, d_per, max_seq_len, -1, out);
}

int xm_align_batch(xm_handle* h, int32_t nq, const uint16_t* packed4, const int64_t* seq_word_off, const int32_t* seq_len, const uint8_t* n_seqs,
                   const double* expected_inner, const double* per_penalty, xm_results** out) {
  if (out) *out = nullptr;
  if (!h || nq < 0 || !out || (nq > 0 && (!packed4 || !seq_word_off || !seq_len || !n_seqs))) return XM_ERR_ARG;
  const bool host_times = getenv("XM_HOST_TIMES") != nullptr;
  const double t_in = now_ms();
  CK(cudaSetDevice(h->device));
  long long n_seqs_total = 0;
  for (int i = 0; i < nq; i++) { if (n_seqs[i] < 1 || n_seqs[i] > 2) { h->err = "n_seqs_per_query must be 1 or 2"; return XM_ERR_ARG; } n_seqs_total += n_seqs[i]; }
  int max_len = 1;
  for (long long s = 0; s < n_seqs_total; s++) if (seq_len[s] > max_len) max_len = seq_len[s];
  int64_t n_words = nq > 0 ? seq_word_off[n_seqs_total] : 0;
  // Query.java:17-30 defaults for hosts that pass no spacing model: expected inner distance 0, one base of deviation per unit penalty
  std::vector<double> zeros, ones;
  if (!expected_inner) zeros.assign((size_t)nq + 1, 0.0);
  if (!per_penalty) ones.assign((size_t)nq + 1, 1.0);
  SlotLease lease(h);   // waits while every slot is in flight (N_SLOTS concurrent callers)
  xm_handle::BatchSlot& sl = lease.slot();
  if (!sl.d_packed.ensure((size_t)n_words * 2 + 16) || !sl.d_seq_word_off.ensure(((size_t)n_seqs_total + 1) * 8) || !sl.d_seq_len.ensure((size_t)n_seqs_total * 4 + 16) ||
      !sl.d_n_seqs.ensure((size_t)nq + 16) || !sl.d_expected.ensure((size_t)nq * 8 + 16) || !sl.d_per.ensure((size_t)nq * 8 + 16)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
  if (nq > 0) {   // on the slot's copy stream: overlaps the kernels of whichever batch holds the compute section right now
    CK(cudaMemcpyAsync(sl.d_packed.p, packed4, (size_t)n_words * 2, cudaMemcpyHostToDevice, sl.copy));
    CK(cudaMemcpyAsync(sl.d_seq_word_off.p, seq_word_off, ((size_t)n_seqs_total + 1) * 8, cudaMemcpyHostToDevice, sl.copy));
    CK(cudaMemcpyAsync(sl.d_seq_len.p, seq_len, (size_t)n_seqs_total * 4, cudaMemcpyHostToDevice, sl.copy));
    CK(cudaMemcpyAsync(sl.d_n_seqs.p, n_seqs, (size_t)nq, cudaMemcpyHostToDevice, sl.copy));
    CK(cudaMemcpyAsync(sl.d_expected.p, expected_inner ? expected_inner : zeros.data(), (size_t)nq * 8, cudaMemcpyHostToDevice, sl.copy));
    CK(cudaMemcpyAsync(sl.d_per.p, per_penalty ? per_penalty : ones.data(), (size_t)nq * 8, cudaMemcpyHostToDevice, sl.copy));
    CK(cudaEventRecord(sl.h2d_done, sl.copy));
  }   // no host synchronisation: the kernels wait for h2d_done on the device (zeros / ones live until this function returns)
  const double t_h2d = now_ms();
  int rc = align_batch_impl(h, lease, nq > 0, nq, (const uint16_t*)sl.d_packed.p, n_words, (const int64_t*)sl.d_seq_word_off.p, (const int32_t*)sl.d_seq_len.p,
                            (const uint8_t*)sl.d_n_seqs.p, (const double*)sl.d_expected.p, (const double*)sl.d_per.p, max_len, n_seqs_total, out);
  if (*out) (*out)->r.stats[XM_STAT_H2D_BYTES] = (int64_t)((size_t)n_words * 2 + ((size_t)n_seqs_total + 1) * 8 + (size_t)n_seqs_total * 4 + (size_t)nq * 17);
  if (host_times && *out) fprintf(stderr, "[xm] xm_align_batch: validate+H2D %.1f ms, device call %.1f ms (kernels %.1f ms)\n", t_h2d - t_in, now_ms() - t_h2d, (double)(*out)->r.stats[XM_STAT_KERNEL_NS] / 1e6);
  return rc;
}

int xm_format_sam(xm_handle* h, xm_results* r, const char* seq_names, const int64_t* seq_name_off, const char* contig_names, const int64_t* contig_name_off,
                  const char** text, int64_t* n_bytes) {
  if (!h || !r || !seq_names || !seq_name_off || !contig_names || !contig_name_off || !text || !n_bytes) return XM_ERR_ARG;
  CK(cudaSetDevice(h->device));
  const int nq = r->nq;
  *text = ""; *n_bytes = 0;
  if (nq == 0) return XM_OK;
  // the device copy of the results lives in the batch slot that produced them until that slot serves another batch
  struct Hold {
    xm_handle* h; int i; bool ok;
    Hold(xm_handle* hh, int slot, uint64_t serial) : h(hh), i(slot), ok(false) {
      if (i < 0 || i >= xm_handle::N_SLOTS) return;
      std::unique_lock<std::mutex> g(h->slot_mu);
      while (h->slots[i].busy && h->slots[i].serial == serial) h->slot_cv.wait(g);
      if (h->slots[i].serial == serial) { h->slots[i].busy = true; ok = true; }
    }
    ~Hold() { if (ok) { { std::lock_guard<std::mutex> g(h->slot_mu); h->slots[i].busy = false; } h->slot_cv.notify_one(); } }
  } hold(h, r->slot, r->serial);
  if (!hold.ok || r->r.slab == nullptr) { h->err = "xm_format_sam: the device copy of these results is gone (their batch slot has served a later xm_align_batch)"; return XM_ERR_STATE; }
  xm_handle::BatchSlot& slot = h->slots[r->slot];
  std::lock_guard<std::mutex> compute(h->compute_mu);
  cudaStream_t st = h->stream;
  // number of sequences = first_seq[nq] on the device; the host passes name offsets for all of them
  long long n_seq_total = 0;
  CK(cudaMemcpy(&n_seq_total, slot.batch.first_seq + nq, 8, cudaMemcpyDeviceToHost));
  const int n_contigs = h->m.n_contigs;
  const size_t names_bytes = (size_t)seq_name_off[n_seq_total], cnames_bytes = (size_t)contig_name_off[n_contigs];
  if (!h->d_sam_names.ensure(names_bytes + 16) || !h->d_sam_name_off.ensure(((size_t)n_seq_total + 1) * 8) || !h->d_sam_cnames.ensure(cnames_bytes + 16) ||
      !h->d_sam_cname_off.ensure(((size_t)n_contigs + 1) * 8) || !h->d_sam_len.ensure(((size_t)nq + 1) * 8)) { h->err = "out of device memory (sam)"; return XM_ERR_CUDA; }
  CK(cudaMemcpyAsync(h->d_sam_names.p, seq_names, names_bytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->d_sam_name_off.p, seq_name_off, ((size_t)n_seq_total + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->d_sam_cnames.p, contig_names, cnames_bytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->d_sam_cname_off.p, contig_name_off, ((size_t)n_contigs + 1) * 8, cudaMemcpyHostToDevice, st));
  SamD S;
  char* d = (char*)slot.d_csr_slab.p;
  const int64_t* off = r->r.slab_off;
  S.c.q_comp_off = (int64_t*)(d + off[0]); S.c.comp_choice_off = (int64_t*)(d + off[1]); S.c.choice_sa_off = (int64_t*)(d + off[2]); S.c.sa_block_off = (int64_t*)(d + off[3]);
  S.c.choice_f64 = (double*)(d + off[4]); S.c.sa_f64 = (double*)(d + off[5]); S.c.choice_inner = (int32_t*)(d + off[6]); S.c.sa_contig = (int32_t*)(d + off[7]);
  S.c.blocks = (int32_t*)(d + off[8]); S.c.q_status = (int32_t*)(d + off[9]); S.c.sa_reversed = (uint8_t*)(d + off[10]);
  S.seq_names = (const char*)h->d_sam_names.p; S.seq_name_off = (const int64_t*)h->d_sam_name_off.p;
  S.contig_names = (const char*)h->d_sam_cnames.p; S.contig_name_off = (const int64_t*)h->d_sam_cname_off.p;
  S.q_len = (long long*)h->d_sam_len.p; S.text = nullptr;
  CK(cudaMemsetAsync((char*)h->d_sam_len.p + (size_t)nq * 8, 0, 8, st));
  xm_sam_kernel<false><<<(nq + 127) / 128, 128, 0, st>>>(S, slot.batch, nq);
  size_t tb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tb, (const long long*)nullptr, (long long*)nullptr, nq + 1, st);
  if (!h->d_csr_tmp.ensure(tb + 16)) { h->err = "out of device memory (sam)"; return XM_ERR_CUDA; }
  CK(cub::DeviceScan::ExclusiveSum(h->d_csr_tmp.p, tb, (const long long*)S.q_len, S.q_len, nq + 1, st));
  long long total = 0;
  CK(cudaMemcpyAsync(&total, S.q_len + nq, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (!h->d_sam_text.ensure((size_t)total + 16)) { h->err = "out of device memory (sam text)"; return XM_ERR_CUDA; }
  S.text = (char*)h->d_sam_text.p;
  xm_sam_kernel<true><<<(nq + 127) / 128, 128, 0, st>>>(S, slot.batch, nq);
  CK(cudaGetLastError());
  if (!r->pool) r->pool = h->pinned;
  if (r->sam && r->sam_cap < (size_t)total + 1) { r->pool->give(r->sam, r->sam_cap); r->sam = nullptr; }
  if (!r->sam) r->sam = r->pool->take((size_t)total + 1, r->sam_cap);
  if (!r->sam) { h->err = "out of pinned host memory (sam text)"; return XM_ERR_CUDA; }
  CK(cudaMemcpyAsync(r->sam, S.text, (size_t)total, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  ((char*)r->sam)[(size_t)total] = 0;
  *text = (const char*)r->sam; *n_bytes = total;
  return XM_OK;
}

int64_t xm_results_array(const xm_results* r, int which, const void** ptr) { if (!r || !ptr) return -1; return r->r.array(which, ptr); }
void xm_release_results(xm_results* r) { delete r; }

int xm_counts_enable(xm_handle* h, double query_end_fraction) {
  if (!h || h->m.n_contigs < 1) return XM_ERR_STATE;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  std::vector<int64_t> off((size_t)h->m.n_contigs + 1, 0);
  for (int c = 0; c < h->m.n_contigs; c++) off[(size_t)c + 1] = off[(size_t)c] + h->m.len[(size_t)c];
  h->n_plane_ints = off[(size_t)h->m.n_contigs] * 4;
  if (!h->d_planes.ensure((size_t)h->n_plane_ints * 4) || !h->d_contig_off.ensure(off.size() * 8)) { h->err = "out of device memory (count planes)"; return XM_ERR_CUDA; }
  CK(cudaMemsetAsync(h->d_planes.p, 0, (size_t)h->n_plane_ints * 4, h->stream));   // ordered before the next batch's kernels on the handle's stream
  CK(cudaMemcpyAsync(h->d_contig_off.p, off.data(), off.size() * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->end_fraction = query_end_fraction; h->counts_enabled = true;
  h->var_n = 0; h->var_reduced_n = 0; h->next_gid = 0; h->have_batch_info = false;
  h->var_gen++;
  return XM_OK;
}
int xm_comm_unique_id(uint8_t* id128) {
  if (!id128) return XM_ERR_ARG;
  NcclApi& N = nccl_api();
  if (!N.ok) return XM_ERR_STATE;
  ncclUniqueId id;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  if (N.GetUniqueId(&id) != ncclSuccess) return XM_ERR_CUDA;
  memcpy(id128, &id, 128);
  return XM_OK;
}
int xm_comm_init(xm_handle* h, int32_t n_ranks, int32_t rank, const uint8_t* id128) {
  if (!h || !id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return XM_ERR_ARG;
  NcclApi& N = nccl_api();
  if (!N.ok) { h->err = "libnccl.so.2 could not be loaded"; return XM_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  if (h->comm) { N.CommDestroy(h->comm); h->comm = nullptr; }
  ncclUniqueId id; memcpy(&id, id128, 128);
  ncclResult_t r = N.CommInitRank(&h->comm, n_ranks, id, rank);
  if (r != ncclSuccess) { h->err = std::string("ncclCommInitRank: ") + N.GetErrorString(r); h->comm = nullptr; return XM_ERR_CUDA; }
  h->comm_ranks = n_ranks; h->comm_rank = rank;
  return XM_OK;
}
int xm_counts_reduce(xm_handle* h) {
  if (!h || !h->counts_enabled) return XM_ERR_STATE;
  if (!h->comm) { h->err = "xm_counts_reduce: xm_comm_init was not called"; return XM_ERR_STATE; }
  std::lock_guard<std::mutex> compute(h->compute_mu);
  NcclApi& N = nccl_api();
  CK(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  // int32 sums are exact and order-free: every rank ends with the planes of the whole run (QV/DirectionalAlignments.java:20-28)
  h->var_gen++;
  CK(cudaEventRecord(h->ev2, st));
  ncclResult_t r = N.AllReduce(h->d_planes.p, h->d_planes.p, (size_t)h->n_plane_ints, ncclInt32, ncclSum, h->comm, st);
  if (r != ncclSuccess) { h->err = std::string("ncclAllReduce: ") + N.GetErrorString(r); return XM_ERR_CUDA; }
  CK(cudaEventRecord(h->ev3, st));
  const double t_var0 = now_ms();
  // the sparse variant tables: every rank reduces its own, all-gathers the sizes, receives every other rank's entries behind its own
  // (one broadcast per rank, grouped) and reduces the concatenation - (sum, best example) is associative and commutative, so every
  // rank ends with the table of the whole run
  int rc = var_reduce_now(h);
  if (rc != XM_OK) return rc;
  const int nr = h->comm_ranks;
  if (!h->d_var_sizes.ensure((size_t)(nr + 1) * 8)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
  unsigned long long mine = h->var_n;
  unsigned long long* d_sizes = (unsigned long long*)h->d_var_sizes.p;
  CK(cudaMemcpyAsync(d_sizes + nr, &mine, 8, cudaMemcpyHostToDevice, st));
  r = N.AllGather(d_sizes + nr, d_sizes, 1, ncclUint64, h->comm, st);
  if (r != ncclSuccess) { h->err = std::string("ncclAllGather: ") + N.GetErrorString(r); return XM_ERR_CUDA; }
  std::vector<unsigned long long> sizes((size_t)nr);
  CK(cudaMemcpyAsync(sizes.data(), d_sizes, (size_t)nr * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  unsigned long long total = 0; int me = -1;
  for (int i = 0; i < nr; i++) total += sizes[(size_t)i];
  { int rk = 0; /* my rank = the slot that holds my size first; ncclCommUserRank is not loaded, so xm_comm_init recorded it */ rk = h->comm_rank; me = rk; }
  rc = var_reserve(h, total);
  if (rc != XM_OK) return rc;
  if (total > mine) {
    // layout after the exchange: [mine][rank 0's][rank 1's]... without my own slot
    VarRec* base = (VarRec*)h->d_var.p;
    unsigned long long at = mine;
    N.GroupStart();
    for (int i = 0; i < nr; i++) {
      const size_t bytes = (size_t)sizes[(size_t)i] * sizeof(VarRec);
      if (bytes == 0) continue;
      if (i == me) r = N.Broadcast(base, base, bytes, ncclUint8, i, h->comm, st);
      else { r = N.Broadcast(base + at, base + at, bytes, ncclUint8, i, h->comm, st); at += sizes[(size_t)i]; }
      if (r != ncclSuccess) { N.GroupEnd(); h->err = std::string("ncclBroadcast: ") + N.GetErrorString(r); return XM_ERR_CUDA; }
    }
    r = N.GroupEnd();
    if (r != ncclSuccess) { h->err = std::string("ncclGroupEnd: ") + N.GetErrorString(r); return XM_ERR_CUDA; }
    h->var_n = total; h->var_reduced_n = 0;
    rc = var_reduce_now(h);
    if (rc != XM_OK) return rc;
  }
  CK(cudaStreamSynchronize(st));
  { float ms = 0; cudaEventElapsedTime(&ms, h->ev2, h->ev3); h->last_planes_ms = ms; h->last_variants_ms = now_ms() - t_var0 - ms; if (h->last_variants_ms < 0) h->last_variants_ms = 0; }
  return XM_OK;
}
int xm_counts_reduce_times(xm_handle* h, double* planes_ms, double* variants_ms) {
  if (!h) return XM_ERR_ARG;
  if (planes_ms) *planes_ms = h->last_planes_ms;
  if (variants_ms) *variants_ms = h->last_variants_ms;
  return XM_OK;
}
int xm_counts_batch_info(xm_handle* h, int64_t first_sequence_id, const int64_t* seq_order_key, int64_t n_sequences) {
  if (!h || first_sequence_id < 0 || n_sequences < 0) return XM_ERR_ARG;
  h->have_batch_info = true; h->info_first_gid = first_sequence_id;
  h->info_order.clear();
  if (seq_order_key) h->info_order.assign(seq_order_key, seq_order_key + n_sequences);
  return XM_OK;
}
int xm_variants_fetch(xm_handle* h, int64_t* n, uint64_t* keys, int32_t* counts, int64_t* ex_gid, int32_t* ex_index) {
  if (!h || !h->counts_enabled) return XM_ERR_STATE;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  int rc = var_reduce_now(h);
  if (rc != XM_OK) return rc;
  if (n) *n = (int64_t)h->var_n;
  if (!keys && !counts && !ex_gid && !ex_index) return XM_OK;
  std::vector<VarRec> host((size_t)h->var_n);
  if (h->var_n) CK(cudaMemcpy(host.data(), h->d_var.p, (size_t)h->var_n * sizeof(VarRec), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < host.size(); i++) {
    if (keys) keys[i] = host[i].key;
    if (counts) counts[i] = host[i].count;
    if (ex_gid) ex_gid[i] = host[i].ex_gid;
    if (ex_index) ex_index[i] = host[i].ex_index;
  }
  return XM_OK;
}

// ---- VCF / mutations bodies (xm_variants_fmt.cuh) ----
// the sorted distinct example ids of the current table, cached for its generation
static int ex_list_refresh(xm_handle* h) {
  int rc = var_reduce_now(h);
  if (rc != XM_OK) return rc;
  if (h->ex_list_gen == h->var_gen) return XM_OK;
  cudaStream_t st = h->stream;
  const unsigned long long n = h->var_n;
  h->ex_list.clear();
  if (n) {
    const int ni = (int)n;
    size_t t1 = 0, t2 = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, t1, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, ni, 0, 64, st);
    cub::DeviceSelect::Unique(nullptr, t2, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (int*)nullptr, ni, st);
    const size_t tb = (t1 > t2 ? t1 : t2) + 256;
    if (!h->d_fmt_ids.ensure((size_t)n * 16 + 16) || !h->d_fmt_tmp.ensure(tb)) { h->err = "out of device memory (variant examples)"; return XM_ERR_CUDA; }
    unsigned long long* a = (unsigned long long*)h->d_fmt_ids.p;
    unsigned long long* b = a + n;
    int* d_count = (int*)(b + n);
    xm_ex_ids_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const VarRec*)h->d_var.p, n, a);
    size_t q = tb;
    CK(cub::DeviceRadixSort::SortKeys(h->d_fmt_tmp.p, q, a, b, ni, 0, 64, st));
    q = tb;
    CK(cub::DeviceSelect::Unique(h->d_fmt_tmp.p, q, b, a, d_count, ni, st));
    int count = 0;
    CK(cudaMemcpyAsync(&count, d_count, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    h->ex_list.resize((size_t)count);
    CK(cudaMemcpyAsync(h->ex_list.data(), a, (size_t)count * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  h->ex_list_gen = h->var_gen;
  return XM_OK;
}
int xm_variants_examples(xm_handle* h, int64_t* n, int64_t* gids) {
  if (!h || !n) return XM_ERR_ARG;
  if (!h->counts_enabled) { h->err = "xm_variants_examples: counts are not enabled"; return XM_ERR_STATE; }
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  int rc = ex_list_refresh(h);
  if (rc != XM_OK) return rc;
  *n = (int64_t)h->ex_list.size();
  if (gids) for (size_t i = 0; i < h->ex_list.size(); i++) gids[i] = h->ex_list[i];
  return XM_OK;
}
int xm_variants_set_examples(xm_handle* h, int64_t n, const int64_t* gids, const uint16_t* packed4, const int64_t* seq_word_off, const int32_t* seq_len) {
  if (!h || n < 0 || (n > 0 && (!gids || !packed4 || !seq_word_off || !seq_len))) return XM_ERR_ARG;
  if (!h->counts_enabled) { h->err = "xm_variants_set_examples: counts are not enabled"; return XM_ERR_STATE; }
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  int rc = ex_list_refresh(h);
  if (rc != XM_OK) return rc;
  h->ex_gen = ~0ull;
  if ((size_t)n != h->ex_list.size()) { h->err = "xm_variants_set_examples: " + std::to_string(n) + " sequences given, the variant table names " + std::to_string(h->ex_list.size()); return XM_ERR_ARG; }
  for (int64_t i = 0; i < n; i++) {
    if (gids[i] != h->ex_list[(size_t)i]) { h->err = "xm_variants_set_examples: sequence " + std::to_string(i) + " is not the one xm_variants_examples lists there"; return XM_ERR_ARG; }
    if (seq_len[i] < 0 || seq_word_off[i] < 0 || seq_word_off[i] + (seq_len[i] + 3) / 4 > seq_word_off[n]) { h->err = "xm_variants_set_examples: sequence " + std::to_string(i) + " lies outside packed4"; return XM_ERR_ARG; }
  }
  cudaStream_t st = h->stream;
  const size_t n_words = n ? (size_t)seq_word_off[n] : 0;
  if (!h->d_ex_words.ensure(n_words * 2 + 16) || !h->d_ex_word_off.ensure((size_t)n * 8 + 16) || !h->d_ex_len.ensure((size_t)n * 4 + 16) ||
      !h->d_ex_gids.ensure((size_t)n * 8 + 16) || !h->d_ex_slot.ensure((size_t)h->var_n * 4 + 16) || !h->d_ex_bad.ensure(16)) { h->err = "out of device memory (variant examples)"; return XM_ERR_CUDA; }
  if (n) {
    CK(cudaMemcpyAsync(h->d_ex_words.p, packed4, n_words * 2, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_ex_word_off.p, seq_word_off, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_ex_len.p, seq_len, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_ex_gids.p, gids, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  }
  CK(cudaMemsetAsync(h->d_ex_bad.p, 0, 4, st));
  if (h->var_n)
    xm_ex_slot_kernel<<<(unsigned)((h->var_n + 255) / 256), 256, 0, st>>>((const VarRec*)h->d_var.p, h->var_n, (const int64_t*)h->d_ex_gids.p, (int)n,
                                                                          (const int32_t*)h->d_ex_len.p, (int32_t*)h->d_ex_slot.p, (unsigned int*)h->d_ex_bad.p);
  unsigned int bad = 0;
  CK(cudaMemcpyAsync(&bad, h->d_ex_bad.p, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (bad) { h->err = "xm_variants_set_examples: " + std::to_string(bad) + " table entries name a read whose given length differs from the read they counted"; return XM_ERR_ARG; }
  h->ex_gen = h->var_gen;
  return XM_OK;
}
static int format_variants(xm_handle* h, int mode, int32_t contig, const char* contig_name, int64_t start, int64_t end, const xm_variant_filter* f,
                           int32_t include_non_mutations, int32_t show_support, const char** text, int64_t* n_bytes) {
  const char* fn = mode == XM_FMT_VCF ? "xm_format_vcf" : "xm_format_mutations";
  if (!h || !contig_name || !text || !n_bytes) return XM_ERR_ARG;
  *text = ""; *n_bytes = 0;
  if (!h->counts_enabled) { h->err = std::string(fn) + ": counts are not enabled"; return XM_ERR_STATE; }
  if (contig < 0 || contig >= h->m.n_contigs) { h->err = std::string(fn) + ": no contig " + std::to_string(contig); return XM_ERR_ARG; }
  const long long len = h->m.len[(size_t)contig];
  if (start < 0 || start > end || end > len) { h->err = std::string(fn) + ": range [" + std::to_string(start) + ", " + std::to_string(end) + ") is not inside [0, " + std::to_string(len) + ")"; return XM_ERR_ARG; }
  if (mode == XM_FMT_MUT && (start % XM_FMT_JOB != 0 || (end % XM_FMT_JOB != 0 && end != len))) { h->err = "xm_format_mutations: start and end must be multiples of 8192 (end may be the contig length)"; return XM_ERR_ARG; }
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  int rc = mirror_model(h);
  if (rc != XM_OK) return rc;
  rc = var_reduce_now(h);
  if (rc != XM_OK) return rc;
  if (show_support && h->ex_gen != h->var_gen) { h->err = "xm_format_vcf: the support column needs the example reads of the current variant table (xm_variants_examples, xm_variants_set_examples)"; return XM_ERR_STATE; }
  const long long n = end - start;
  if (n == 0) return XM_OK;
  if (n + 1 >= (1ll << 31)) { h->err = std::string(fn) + ": ranges hold fewer than 2^31 - 1 positions"; return XM_ERR_ARG; }
  cudaStream_t st = h->stream;
  const size_t name_len = strlen(contig_name);
  if (!h->d_fmt_dec.ensure((size_t)n + 16) || !h->d_fmt_state.ensure((size_t)n + 16) || !h->d_fmt_len.ensure(((size_t)n + 1) * 8) || !h->d_fmt_range.ensure(16) ||
      !h->d_fmt_name.ensure(name_len + 16) || !h->d_ex_slot.ensure(16)) { h->err = std::string("out of device memory (") + fn + ")"; return XM_ERR_CUDA; }
  CK(cudaMemcpyAsync(h->d_fmt_name.p, contig_name, name_len, cudaMemcpyHostToDevice, st));
  FmtD D;
  D.ref = h->ref; D.planes = (const int32_t*)h->d_planes.p; D.contig_off = (const int64_t*)h->d_contig_off.p;
  D.recs = (const VarRec*)h->d_var.p; D.n_recs = h->var_n; D.range = (unsigned long long*)h->d_fmt_range.p;
  D.contig = contig; D.start = start; D.end = end;
  D.f = VarFilter{0, 0, 0, 0, 0, 0};
  if (f) D.f = VarFilter{f->min_snp_total_depth, f->min_snp_depth_fraction, f->min_indel_start_total_depth, f->min_indel_start_depth_fraction,
                         f->min_indel_continuation_total_depth, f->min_indel_continuation_depth_fraction};
  D.name = (const char*)h->d_fmt_name.p; D.name_len = (int)name_len;
  D.include_non_mutations = include_non_mutations ? 1 : 0; D.show_support = (mode == XM_FMT_VCF && show_support) ? 1 : 0;
  D.dec = (uint8_t*)h->d_fmt_dec.p; D.could_delete = (const uint8_t*)h->d_fmt_state.p; D.len = (long long*)h->d_fmt_len.p; D.text = nullptr;
  D.ex_slot = (const int32_t*)h->d_ex_slot.p; D.ex_words = (const uint16_t*)h->d_ex_words.p; D.ex_word_off = (const int64_t*)h->d_ex_word_off.p; D.ex_len = (const int32_t*)h->d_ex_len.p;
  const unsigned blocks = (unsigned)((n + 127) / 128);
  xm_fmt_carry_kernel<<<1, 256, 0, st>>>(D);
  xm_fmt_decide_kernel<<<blocks, 128, 0, st>>>(D);
  size_t t1 = 0, t2 = 0;
  cub::DeviceScan::InclusiveScan(nullptr, t1, (const uint8_t*)nullptr, (uint8_t*)nullptr, FmtLastDecisive(), (int)(n + 1), st);
  cub::DeviceScan::ExclusiveSum(nullptr, t2, (const long long*)nullptr, (long long*)nullptr, (int)(n + 1), st);
  const size_t tb = (t1 > t2 ? t1 : t2) + 256;
  if (!h->d_fmt_tmp.ensure(tb)) { h->err = std::string("out of device memory (") + fn + ")"; return XM_ERR_CUDA; }
  size_t q = tb;
  CK(cub::DeviceScan::InclusiveScan(h->d_fmt_tmp.p, q, D.dec, (uint8_t*)h->d_fmt_state.p, FmtLastDecisive(), (int)(n + 1), st));
  CK(cudaMemsetAsync(D.len + n, 0, 8, st));
  if (mode == XM_FMT_VCF) xm_fmt_kernel<XM_FMT_VCF, false><<<blocks, 128, 0, st>>>(D); else xm_fmt_kernel<XM_FMT_MUT, false><<<blocks, 128, 0, st>>>(D);
  q = tb;
  CK(cub::DeviceScan::ExclusiveSum(h->d_fmt_tmp.p, q, (const long long*)D.len, D.len, (int)(n + 1), st));
  long long total = 0;
  CK(cudaMemcpyAsync(&total, D.len + n, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (!h->d_fmt_text.ensure((size_t)total + 16)) { h->err = std::string("out of device memory (") + fn + " text)"; return XM_ERR_CUDA; }
  D.text = (char*)h->d_fmt_text.p;
  if (mode == XM_FMT_VCF) xm_fmt_kernel<XM_FMT_VCF, true><<<blocks, 128, 0, st>>>(D); else xm_fmt_kernel<XM_FMT_MUT, true><<<blocks, 128, 0, st>>>(D);
  CK(cudaGetLastError());
  if (h->fmt_text && h->fmt_cap < (size_t)total + 1) { h->pinned->give(h->fmt_text, h->fmt_cap); h->fmt_text = nullptr; }
  if (!h->fmt_text) h->fmt_text = h->pinned->take((size_t)total + 1, h->fmt_cap);
  if (!h->fmt_text) { h->err = std::string("out of pinned host memory (") + fn + " text)"; return XM_ERR_CUDA; }
  CK(cudaMemcpyAsync(h->fmt_text, D.text, (size_t)total, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  ((char*)h->fmt_text)[(size_t)total] = 0;
  *text = (const char*)h->fmt_text; *n_bytes = total;
  return XM_OK;
}
int xm_format_vcf(xm_handle* h, int32_t contig, const char* contig_name, int64_t start, int64_t end, const xm_variant_filter* f,
                  int32_t include_non_mutations, int32_t show_support, const char** text, int64_t* n_bytes) {
  return format_variants(h, XM_FMT_VCF, contig, contig_name, start, end, f, include_non_mutations, show_support, text, n_bytes);
}
int xm_format_mutations(xm_handle* h, int32_t contig, const char* contig_name, int64_t start, int64_t end, const xm_variant_filter* f,
                        const char** text, int64_t* n_bytes) {
  return format_variants(h, XM_FMT_MUT, contig, contig_name, start, end, f, 0, 0, text, n_bytes);
}

int xm_parse_reads(xm_handle* h, int32_t format, const char* text, int64_t n_bytes, int32_t at_eof, int64_t max_records, int32_t split_size,
                   xm_reads** out, int64_t* n_consumed) {
  if (out) *out = nullptr;
  if (n_consumed) *n_consumed = 0;
  if (!h || !out || !n_consumed || (format != XM_FASTA && format != XM_FASTQ) || n_bytes < 0 || (n_bytes > 0 && !text) || split_size < 0) return XM_ERR_ARG;
  if (n_bytes >= (1ll << 31)) { h->err = "xm_parse_reads: pass fewer than 2^31 bytes per call"; return XM_ERR_ARG; }
  std::lock_guard<std::mutex> parse(h->parse_mu);
  CK(cudaSetDevice(h->device));
  cudaStream_t st = h->parse_stream;
  const bool fastq = format == XM_FASTQ;
  const long long n = n_bytes;
  const char* fmt_name = fastq ? "FASTQ" : "FASTA";
  // the text goes up through the pinned staging buffer
  if (h->pz_stage && h->pz_stage_cap < (size_t)n + 1) { h->pinned->give(h->pz_stage, h->pz_stage_cap); h->pz_stage = nullptr; }
  if (!h->pz_stage) h->pz_stage = h->pinned->take((size_t)n + 1, h->pz_stage_cap);
  if (!h->pz_stage) { h->err = "out of pinned host memory (xm_parse_reads)"; return XM_ERR_CUDA; }
  if (n) memcpy(h->pz_stage, text, (size_t)n);
  const int n_tiles = (int)std::max<long long>(1, (n + PZ_TILE - 1) / PZ_TILE);
  if (!h->d_pz_text.ensure((size_t)n + 16) || !h->d_pz_tiles.ensure(((size_t)n_tiles + 1) * 8) || !h->d_pz_misc.ensure(64)) { h->err = "out of device memory (xm_parse_reads)"; return XM_ERR_CUDA; }
  const char* d_text = (const char*)h->d_pz_text.p;
  unsigned int* tile_cnt = (unsigned int*)h->d_pz_tiles.p;
  unsigned int* tile_off = tile_cnt + n_tiles + 1;
  PzErr* d_err = (PzErr*)h->d_pz_misc.p;
  int* d_count = (int*)((char*)h->d_pz_misc.p + 32);
  if (n) CK(cudaMemcpyAsync(h->d_pz_text.p, h->pz_stage, (size_t)n, cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(d_err, 0xff, sizeof(PzErr), st));
  // line ends
  xm_parse_nl_kernel<false><<<n_tiles, PZ_THREADS, 0, st>>>(d_text, n, tile_cnt, nullptr, nullptr);
  CK(cudaMemsetAsync(tile_cnt + n_tiles, 0, 4, st));
  CK(pz_scan(h, tile_cnt, tile_off, n_tiles + 1, false));
  unsigned int n_nl = 0;
  CK(cudaMemcpyAsync(&n_nl, tile_off + n_tiles, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const bool tail = at_eof && n > 0 && text[n - 1] != '\n';   // the last line of the input needs no '\n'
  const int n_lines = (int)n_nl + (tail ? 1 : 0);
  const long long text_end = n;
  if (!h->d_pz_line_end.ensure(((size_t)n_lines + 1) * 8)) { h->err = "out of device memory (xm_parse_reads)"; return XM_ERR_CUDA; }
  long long* line_end = (long long*)h->d_pz_line_end.p;
  xm_parse_nl_kernel<true><<<n_tiles, PZ_THREADS, 0, st>>>(d_text, n, tile_cnt, tile_off, line_end);
  if (tail) CK(cudaMemcpyAsync(line_end + n_nl, &text_end, 8, cudaMemcpyHostToDevice, st));
  ParseD P;
  P.text = d_text; P.n = n; P.fastq = fastq ? 1 : 0; P.split = split_size; P.line_end = line_end; P.n_lines = n_lines;
  P.rec_line = nullptr; P.line_rec = nullptr; P.lbase = nullptr; P.err = d_err;
  // records: complete ones only, at most max_records
  long long n_rec = 0, n_avail = 0;
  int lines_end = 0;
  if (fastq) {
    n_avail = n_lines / 4;
    n_rec = max_records >= 0 ? std::min<long long>(n_avail, max_records) : n_avail;
    lines_end = (int)(4 * n_rec);
  } else {
    if (!h->d_pz_flag.ensure(((size_t)n_lines + 1) * 4) || !h->d_pz_line_rec.ensure(((size_t)n_lines + 1) * 4) || !h->d_pz_rec_line.ensure(((size_t)n_lines + 2) * 4)) {
      h->err = "out of device memory (xm_parse_reads)"; return XM_ERR_CUDA;
    }
    int* flag = (int*)h->d_pz_flag.p;
    int* rec_line = (int*)h->d_pz_rec_line.p;
    int n_hdr = 0;
    if (n_lines) {
      xm_parse_class_kernel<<<pz_blocks(n_lines, 256), 256, 0, st>>>(P, flag);
      CK(pz_scan(h, flag, (int*)h->d_pz_line_rec.p, n_lines, true));
      size_t tb = 0;
      cub::DeviceSelect::Flagged(nullptr, tb, cub::CountingInputIterator<int>(0), flag, rec_line, d_count, n_lines, st);
      if (!h->d_pz_tmp.ensure(tb + 16)) { h->err = "out of device memory (xm_parse_reads)"; return XM_ERR_CUDA; }
      CK(cub::DeviceSelect::Flagged(h->d_pz_tmp.p, tb, cub::CountingInputIterator<int>(0), flag, rec_line, d_count, n_lines, st));
      CK(cudaMemcpyAsync(&n_hdr, d_count, 4, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
    n_avail = at_eof ? n_hdr : std::max(n_hdr - 1, 0);   // without the end of the input, a record is complete when the next header is seen
    n_rec = max_records >= 0 ? std::min<long long>(n_avail, max_records) : n_avail;
    lines_end = n_lines;
    if (n_rec < n_hdr) { CK(cudaMemcpyAsync(&lines_end, rec_line + n_rec, 4, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st)); }
    else CK(cudaMemcpyAsync(rec_line + n_rec, &lines_end, 4, cudaMemcpyHostToDevice, st));
    P.rec_line = rec_line; P.line_rec = (const int*)h->d_pz_line_rec.p;
  }
  P.n_rec = (int)n_rec; P.lines_end = lines_end;
  // bytes taken: through the end of the last parsed record, or all of it when the input ends after it
  const bool all = at_eof && (fastq ? n_rec == n_avail : lines_end == n_lines);
  long long consumed = 0, tail_start = 0;
  if (lines_end > 0) { CK(cudaMemcpyAsync(&tail_start, line_end + lines_end - 1, 8, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st)); tail_start++; }
  consumed = all ? n : tail_start;
  // per line bases and checks, per record pieces
  if (!h->d_pz_bases.ensure(((size_t)lines_end + 1) * 8) || !h->d_pz_lbase.ensure(((size_t)lines_end + 1) * 8) ||
      !h->d_pz_pieces.ensure(((size_t)n_rec + 1) * 8) || !h->d_pz_piece_off.ensure(((size_t)n_rec + 1) * 8)) { h->err = "out of device memory (xm_parse_reads)"; return XM_ERR_CUDA; }
  xm_parse_lines_kernel<<<pz_blocks(lines_end + 1, 256), 256, 0, st>>>(P, (long long*)h->d_pz_bases.p);
  CK(pz_scan(h, (const long long*)h->d_pz_bases.p, (long long*)h->d_pz_lbase.p, lines_end + 1, false));
  P.lbase = (const long long*)h->d_pz_lbase.p;
  xm_parse_rec_kernel<<<pz_blocks(n_rec + 1, 256), 256, 0, st>>>(P, (long long*)h->d_pz_pieces.p);
  CK(pz_scan(h, (const long long*)h->d_pz_pieces.p, (long long*)h->d_pz_piece_off.p, (int)n_rec + 1, false));
  long long n_seq = 0;
  PzErr e;
  CK(cudaMemcpyAsync(&n_seq, (const long long*)h->d_pz_piece_off.p + n_rec, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&e, d_err, sizeof(PzErr), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  auto fail = [&](const PzErr& x) {
    const long long off = (long long)(x.key >> 3), line = (long long)x.line;
    const int kind = (int)(x.key & 7);
    long long rec = line / 4;
    if (!fastq) { int lr = 0; if (cudaMemcpy(&lr, P.line_rec + line, 4, cudaMemcpyDeviceToHost) != cudaSuccess) cudaGetLastError(); rec = lr - 1; }
    std::string what;
    switch (kind) {
      case PZ_BAD_BASE: { char b[64]; snprintf(b, sizeof b, "byte 0x%02x ('%c') is not an IUPAC base letter", (unsigned char)text[off], text[off] >= 32 && text[off] < 127 ? text[off] : '?'); what = b; break; }
      case PZ_BAD_MARKER: what = "a FASTQ record must start with a '@' line"; break;
      case PZ_NO_PLUS: what = "missing '+' line (multi-line FASTQ is not supported)"; break;
      case PZ_QUAL_LEN: what = "the quality line is not as long as the sequence line"; break;
      case PZ_BEFORE_HEADER: what = "text before the first '>' header"; break;
    }
    h->err = std::string("xm_parse_reads: ") + fmt_name + " record " + std::to_string(rec) + ", byte offset " + std::to_string(off) + ": " + what;
    return XM_ERR_ARG;
  };
  if (e.key != ~0ull) return fail(e);
  if (fastq && all) {   // only blank lines may follow the last complete record
    for (long long i = tail_start; i < n; i++) if (text[i] != '\n' && text[i] != '\r') {
      h->err = "xm_parse_reads: FASTQ record " + std::to_string(n_rec) + ", byte offset " + std::to_string(tail_start) + ": the input ends inside the record (a record is four lines)";
      return XM_ERR_ARG;
    }
  }
  if (n_seq >= (1ll << 31)) { h->err = "xm_parse_reads: more than 2^31 - 1 sequences in one call"; return XM_ERR_ARG; }
  // pieces, word and name offsets
  const size_t ns1 = (size_t)n_seq + 1;
  if (!h->d_pz_start.ensure(ns1 * 8) || !h->d_pz_len.ensure(ns1 * 4) || !h->d_pz_rec.ensure(ns1 * 8) || !h->d_pz_words.ensure(ns1 * 8) ||
      !h->d_pz_name_len.ensure(ns1 * 8) || !h->d_pz_word_off.ensure(ns1 * 8) || !h->d_pz_name_off.ensure(ns1 * 8)) { h->err = "out of device memory (xm_parse_reads)"; return XM_ERR_CUDA; }
  PieceD Q;
  Q.piece_off = (const long long*)h->d_pz_piece_off.p; Q.start = (long long*)h->d_pz_start.p; Q.len = (int32_t*)h->d_pz_len.p; Q.rec = (int64_t*)h->d_pz_rec.p;
  Q.words = (long long*)h->d_pz_words.p; Q.name_len = (long long*)h->d_pz_name_len.p;
  if (n_rec) xm_parse_piece_kernel<<<pz_blocks(n_rec, 128), 128, 0, st>>>(P, Q);
  CK(cudaMemsetAsync(Q.words + n_seq, 0, 8, st));
  CK(cudaMemsetAsync(Q.name_len + n_seq, 0, 8, st));
  CK(pz_scan(h, (const long long*)Q.words, (long long*)h->d_pz_word_off.p, (int)ns1, false));
  CK(pz_scan(h, (const long long*)Q.name_len, (long long*)h->d_pz_name_off.p, (int)ns1, false));
  long long tot[2] = {0, 0};
  CK(cudaMemcpyAsync(&tot[0], (const long long*)h->d_pz_word_off.p + n_seq, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&tot[1], (const long long*)h->d_pz_name_off.p + n_seq, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  // one device slab in the layout of the host slab: packed, seq_word_off, seq_len, name_off, names, record
  std::unique_ptr<xm_reads> R(new xm_reads());
  const int64_t counts[6] = {tot[0], (int64_t)ns1, n_seq, (int64_t)ns1, tot[1], n_seq};
  const int64_t widths[6] = {2, 8, 4, 8, 1, 8};
  size_t bytes = 0;
  for (int k = 0; k < 6; k++) { R->off[k] = (int64_t)bytes; R->n[k] = counts[k]; bytes += ((size_t)(counts[k] * widths[k]) + 15) & ~(size_t)15; }
  if (!h->d_pz_slab.ensure(bytes + 16)) { h->err = "out of device memory (xm_parse_reads)"; return XM_ERR_CUDA; }
  char* ds = (char*)h->d_pz_slab.p;
  CK(cudaMemcpyAsync(ds + R->off[1], h->d_pz_word_off.p, ns1 * 8, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(ds + R->off[2], h->d_pz_len.p, (size_t)n_seq * 4, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(ds + R->off[3], h->d_pz_name_off.p, ns1 * 8, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(ds + R->off[5], h->d_pz_rec.p, (size_t)n_seq * 8, cudaMemcpyDeviceToDevice, st));
  PackD K;
  K.start = Q.start; K.len = Q.len; K.rec = Q.rec; K.word_off = (const int64_t*)h->d_pz_word_off.p; K.name_off = (const int64_t*)h->d_pz_name_off.p;
  K.packed = (uint16_t*)(ds + R->off[0]); K.names = ds + R->off[4]; K.n_seq = n_seq;
  if (n_seq) {
    xm_parse_pack_kernel<<<pz_blocks(n_seq * 32, 256), 256, 0, st>>>(P, K);
    xm_parse_names_kernel<<<pz_blocks(n_seq * 32, 256), 256, 0, st>>>(P, K);
  }
  CK(cudaGetLastError());
  R->pool = h->pinned;
  R->slab = h->pinned->take(bytes + 16, R->slab_cap);
  if (!R->slab) { h->err = "out of pinned host memory (xm_parse_reads)"; return XM_ERR_CUDA; }
  CK(cudaMemcpyAsync(R->slab, ds, bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&e, d_err, sizeof(PzErr), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (e.key != ~0ull) return fail(e);
  *n_consumed = consumed;
  *out = R.release();
  return XM_OK;
}
int64_t xm_reads_array(const xm_reads* r, int which, const void** ptr) {
  if (!r || !ptr || which < 0 || which > XM_R_RECORD) return -1;
  *ptr = (const char*)r->slab + r->off[which];
  return r->n[which];
}
void xm_release_reads(xm_reads* r) { delete r; }

int xm_rank_names(xm_handle* h, int64_t n, const char* names, const int64_t* name_off, int64_t* ranks) {
  if (!h) return XM_ERR_ARG;
  if (n < 0 || n >= (1ll << 31) || !name_off || (n > 0 && !ranks)) { h->err = "xm_rank_names: 0 <= n < 2^31 names, name_off[n + 1] and ranks[n] are required"; return XM_ERR_ARG; }
  if (name_off[0] != 0) { h->err = "xm_rank_names: name_off[0] != 0"; return XM_ERR_ARG; }
  for (int64_t i = 0; i < n; i++) if (name_off[i + 1] < name_off[i]) { h->err = "xm_rank_names: name_off is not non-decreasing at " + std::to_string(i); return XM_ERR_ARG; }
  const int64_t n_bytes = name_off[n];
  if (n_bytes > 0 && !names) { h->err = "xm_rank_names: names is NULL"; return XM_ERR_ARG; }
  if (n == 0) return XM_OK;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  const int ni = (int)n;
  int label_bits = 1;
  while ((1ll << label_bits) < n) label_bits++;
  // scratch for this call only: it is freed on return, so ranking a large run leaves no device memory behind for the batches
  DevBuf d_names, d_off, d_act, d_act2, d_key, d_key2, d_iota, d_p1, d_lab1, d_p2, d_sin, d_sout, d_keep, d_final, d_tmp, d_misc;
  const size_t N = (size_t)n;
  if (!d_names.ensure((size_t)n_bytes + 16) || !d_off.ensure((N + 1) * 8) || !d_act.ensure(N * 8) || !d_act2.ensure(N * 8) || !d_key.ensure(N * 8) ||
      !d_key2.ensure(N * 8) || !d_iota.ensure(N * 4) || !d_p1.ensure(N * 4) || !d_lab1.ensure(N * 4) || !d_p2.ensure(N * 4) ||
      !d_sin.ensure((N + 1) * 8) || !d_sout.ensure((N + 1) * 8) || !d_keep.ensure(N) || !d_final.ensure(N * 4) || !d_misc.ensure(16)) {
    h->err = "out of device memory (xm_rank_names)"; return XM_ERR_CUDA;
  }
  uint64_t *act = (uint64_t*)d_act.p, *act2 = (uint64_t*)d_act2.p, *key = (uint64_t*)d_key.p, *key2 = (uint64_t*)d_key2.p;
  uint32_t *iota = (uint32_t*)d_iota.p, *p1 = (uint32_t*)d_p1.p, *lab1 = (uint32_t*)d_lab1.p, *p2 = (uint32_t*)d_p2.p, *fin = (uint32_t*)d_final.p;
  int2 *sin = (int2*)d_sin.p, *sout = (int2*)d_sout.p;
  uint8_t* keep = (uint8_t*)d_keep.p;
  int* d_count = (int*)d_misc.p;
  size_t t1 = 0, t2 = 0, t3 = 0, t4 = 0, t5 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, t1, key, key2, iota, p1, ni, 0, 64, st);
  cub::DeviceRadixSort::SortPairs(nullptr, t2, lab1, iota, p1, p2, ni, 0, label_bits, st);
  cub::DeviceScan::InclusiveScan(nullptr, t3, sin, sout, RnMax2(), ni, st);
  cub::DeviceSelect::Flagged(nullptr, t4, key, keep, act, d_count, ni, st);
  cub::DeviceScan::ExclusiveSum(nullptr, t5, (const int*)nullptr, (int*)nullptr, ni + 1, st);
  const size_t tb = std::max(std::max(std::max(t1, t2), std::max(t3, t4)), t5) + 256;
  if (!d_tmp.ensure(tb)) { h->err = "out of device memory (xm_rank_names)"; return XM_ERR_CUDA; }
  if (n_bytes) CK(cudaMemcpyAsync(d_names.p, names, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_off.p, name_off, (N + 1) * 8, cudaMemcpyHostToDevice, st));
  // every name starts in the one class of label 0, as item (0 << 32 | i)
  xm_rank_init_kernel<<<pz_blocks(n, RN_THREADS), RN_THREADS, 0, st>>>(ni, act);
  int m = ni;
  for (int d = 0; m > 0; d++) {
    const unsigned blocks = pz_blocks(m, RN_THREADS);
    size_t q;
    xm_rank_key_kernel<<<blocks, RN_THREADS, 0, st>>>((const uint8_t*)d_names.p, (const int64_t*)d_off.p, act, m, d, key, iota);
    q = tb; CK(cub::DeviceRadixSort::SortPairs(d_tmp.p, q, key, key2, iota, p1, m, 0, 64, st));
    xm_rank_label_kernel<<<blocks, RN_THREADS, 0, st>>>(act, p1, m, lab1);
    q = tb; CK(cub::DeviceRadixSort::SortPairs(d_tmp.p, q, lab1, iota, p1, p2, m, 0, label_bits, st));
    xm_rank_gather_kernel<<<blocks, RN_THREADS, 0, st>>>(act, key, p2, m, act2, key2);
    xm_rank_flags_kernel<<<blocks, RN_THREADS, 0, st>>>(act2, key2, m, sin);
    q = tb; CK(cub::DeviceScan::InclusiveScan(d_tmp.p, q, sin, sout, RnMax2(), m, st));
    xm_rank_split_kernel<<<blocks, RN_THREADS, 0, st>>>(act2, key2, sout, m, fin, keep, key);
    q = tb; CK(cub::DeviceSelect::Flagged(d_tmp.p, q, key, keep, act, d_count, m, st));
    CK(cudaMemcpyAsync(&m, d_count, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  // dense ranks: the number of labels in use below a name's label
  int* mark = (int*)d_sin.p;
  int* below = (int*)d_sout.p;
  CK(cudaMemsetAsync(mark, 0, (N + 1) * 4, st));
  xm_rank_mark_kernel<<<pz_blocks(n, RN_THREADS), RN_THREADS, 0, st>>>(fin, ni, mark);
  size_t q = tb;
  CK(cub::DeviceScan::ExclusiveSum(d_tmp.p, q, mark, below, ni + 1, st));
  xm_rank_dense_kernel<<<pz_blocks(n, RN_THREADS), RN_THREADS, 0, st>>>(fin, below, ni, (int64_t*)d_act2.p);
  CK(cudaMemcpyAsync(ranks, d_act2.p, N * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  return XM_OK;
}

// out[0] INT32 IMAD, out[1] FP64 DADD, out[2] FP32 FFMA (full-rate pipe = the dispatch ceiling): sustained warp-instructions per second over the whole chip (the loop
// bodies are 128 arithmetic instructions per iteration per warp; loop overhead is below 2 %); out[3] = SM count, out[4] = SM clock in Hz
// (cudaDevAttrClockRate: the maximum; the achieved clock under load is sampled by the caller).
int xm_measure_peaks(xm_handle* h, double* out) {
  if (!h || !out) return XM_ERR_ARG;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  if (!h->d_misc.ensure(256)) { h->err = "out of device memory"; return XM_ERR_CUDA; }
  const int blocks = h->sm_count * 8, threads = 256, iters = 2000;
  const double warp_inst = (double)blocks * (threads / 32) * (double)iters * 128.0;
  for (int kind = 0; kind < 3; kind++) {
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
      CK(cudaEventRecord(h->ev2, st));
      if (kind == 0) xm_peak_kernel<0><<<blocks, threads, 0, st>>>(iters, (unsigned long long*)h->d_misc.p, 3.0);
      else if (kind == 1) xm_peak_kernel<1><<<blocks, threads, 0, st>>>(iters, (unsigned long long*)h->d_misc.p, 1e-9);
      else xm_peak_kernel<2><<<blocks, threads, 0, st>>>(iters, (unsigned long long*)h->d_misc.p, 12345.0);
      CK(cudaEventRecord(h->ev3, st));
      CK(cudaStreamSynchronize(st));
      CK(cudaGetLastError());
      float ms = 0; cudaEventElapsedTime(&ms, h->ev2, h->ev3);
      if (rep > 0 && ms < best) best = ms;
    }
    out[kind] = warp_inst / ((double)best * 1e-3);
  }
  int clk_khz = 0;
  cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, h->device);
  out[3] = (double)h->sm_count; out[4] = (double)clk_khz * 1e3;
  return XM_OK;
}
int xm_counts_device_ptr(xm_handle* h, void** d_ptr, int64_t* n_int32) {
  if (!h || !h->counts_enabled) return XM_ERR_STATE;
  if (d_ptr) *d_ptr = h->d_planes.p;
  if (n_int32) *n_int32 = h->n_plane_ints;
  return XM_OK;
}
int xm_counts_fetch(xm_handle* h, int32_t contig, int32_t* out) {
  if (!h || !h->counts_enabled || contig < 0 || contig >= h->m.n_contigs || !out) return XM_ERR_ARG;
  std::lock_guard<std::mutex> compute(h->compute_mu);
  CK(cudaSetDevice(h->device));
  long long off = 0;
  for (int c = 0; c < contig; c++) off += h->m.len[(size_t)c];
  CK(cudaMemcpy(out, (int32_t*)h->d_planes.p + off * 4, (size_t)h->m.len[(size_t)contig] * 16, cudaMemcpyDeviceToHost));
  return XM_OK;
}

}  // extern "C"
