// xmapper_b200 — read names ranked on the device (xm_rank_names).  Included by xm_capi.cu after xm_parse.cuh.
//
// The rank of a name is the number of distinct names smaller than it in unsigned byte order, a proper prefix first: the name order
// DirectionalAlignments.betterExample breaks example ties with.  The names are split into classes of names that are equal so far,
// refined most significant chunk first.  Round d looks at bytes [7d, 7d + 7) of every name still in an unresolved class:
//   xm_rank_key_kernel     per item: a 64-bit key, those 7 bytes big-endian (zeros past the end) in bits 63..8 and
//                          min(max(len - 7d, 0), 8) in bits 7..0, so NUL bytes inside a name and proper prefixes keep their order;
//   cub radix sorts         by key, then (stable) by class label: the items in (label, key) order;
//   xm_rank_gather_kernel  the items and keys in that order;
//   xm_rank_flags_kernel   per position t: t where a class starts, t where a (class, key) run starts (0 elsewhere);
//   cub scan (max)          the start of each position's class and run;
//   xm_rank_split_kernel   new label = class label + (run start - class start).  A run is final once it has one member or its key's
//                          low byte is < 8 (all its names end in this chunk and are equal); final items write their label.
//   cub select              the items of runs that are not final, for the next round.
// A label is the position in the sorted order of all n names at which its class starts, so resolved items drop out of later rounds
// without renumbering the others.  Round d + 1 only holds names longer than 7d + 7 bytes: at most ceil(longest / 7) + 1 rounds.  At the
// end xm_rank_mark_kernel marks the labels in use, an exclusive sum counts the marks below each label, and xm_rank_dense_kernel gives
// every name the count at its label.
#pragma once

static const int RN_THREADS = 256;

__global__ void __launch_bounds__(RN_THREADS) xm_rank_init_kernel(int n, uint64_t* act) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) act[i] = (uint64_t)i;
}

// key of item j (act[j]: label << 32 | name index) in round d
__global__ void __launch_bounds__(RN_THREADS) xm_rank_key_kernel(const uint8_t* names, const int64_t* name_off, const uint64_t* act, int m, int d,
                                                                 uint64_t* key, uint32_t* iota) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const uint32_t i = (uint32_t)act[j];
  const int64_t s = name_off[i], len = name_off[i + 1] - s, p = 7LL * d;
  uint64_t k = 0;
  for (int b = 0; b < 7; b++) k = (k << 8) | (p + b < len ? (uint64_t)names[s + p + b] : 0ull);
  const int64_t rest = len - p;
  key[j] = (k << 8) | (uint64_t)(rest < 0 ? 0 : rest > 8 ? 8 : rest);
  iota[j] = (uint32_t)j;
}

__global__ void __launch_bounds__(RN_THREADS) xm_rank_label_kernel(const uint64_t* act, const uint32_t* perm, int m, uint32_t* label) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < m) label[t] = (uint32_t)(act[perm[t]] >> 32);
}

__global__ void __launch_bounds__(RN_THREADS) xm_rank_gather_kernel(const uint64_t* act, const uint64_t* key, const uint32_t* perm, int m,
                                                                    uint64_t* act2, uint64_t* key2) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  act2[t] = act[perm[t]]; key2[t] = key[perm[t]];
}

__device__ __forceinline__ bool rn_class_start(const uint64_t* act, int t) { return t == 0 || (act[t] >> 32) != (act[t - 1] >> 32); }
__device__ __forceinline__ bool rn_run_start(const uint64_t* act, const uint64_t* key, int t) { return rn_class_start(act, t) || key[t] != key[t - 1]; }

__global__ void __launch_bounds__(RN_THREADS) xm_rank_flags_kernel(const uint64_t* act, const uint64_t* key, int m, int2* starts) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < m) starts[t] = make_int2(rn_class_start(act, t) ? t : 0, rn_run_start(act, key, t) ? t : 0);
}

struct RnMax2 {
  __device__ __forceinline__ int2 operator()(const int2& a, const int2& b) const { return make_int2(max(a.x, b.x), max(a.y, b.y)); }
};

// next[t]: the item with its new label; keep[t] = 1 when it stays for the next round
__global__ void __launch_bounds__(RN_THREADS) xm_rank_split_kernel(const uint64_t* act, const uint64_t* key, const int2* starts, int m,
                                                                   uint32_t* final_label, uint8_t* keep, uint64_t* next) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  const uint64_t a = act[t];
  const uint32_t label = (uint32_t)(a >> 32) + (uint32_t)(starts[t].y - starts[t].x);
  const bool single = starts[t].y == t && (t + 1 == m || rn_run_start(act, key, t + 1));
  const bool done = single || (key[t] & 0xffu) < 8u;
  if (done) final_label[(uint32_t)a] = label;
  keep[t] = done ? 0 : 1;
  next[t] = ((uint64_t)label << 32) | (a & 0xffffffffull);
}

__global__ void __launch_bounds__(RN_THREADS) xm_rank_mark_kernel(const uint32_t* final_label, int n, int* mark) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) mark[final_label[i]] = 1;
}

__global__ void __launch_bounds__(RN_THREADS) xm_rank_dense_kernel(const uint32_t* final_label, const int* below, int n, int64_t* ranks) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) ranks[i] = below[final_label[i]];
}
