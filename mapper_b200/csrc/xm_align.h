// xmapper_b200 device core — scoring + traceback cascade, pair model, per-query driver.
// Reproduces M/StraightAligner.java, M/SkipHighAmbiguity_Aligner.java, M/HashBlock_Aligner.java,
// M/HashBlock_Matcher.java (direct-address tables replaced by an on-the-fly scan of the same sections with the
// same recurrence, including its quirks), M/CountMap.java, M/BlockAligner.java, M/PathAligner.java (literal
// best-first search: dense node grid + binary heap keyed (priority, insertion order)), M/QueryMatch_Aligner.java,
// M/AlignerWorker.java:306-644.  All penalties are IEEE doubles added in the reference's order (compile with
// -fmad=false).
#pragma once
#include "xm_seed.h"

namespace xm {

struct Blk { int a_start, b_start, a_len, b_len; };
struct DAln {  // SequenceAlignment; valid == 0 is null
  int valid, n;
  Blk* b;
  double penalty, aligned;
  int ref_reversed;
};
struct ACtx {  // the two sequences an alignMatch works on
  SeqView a; int a_reversed_obj;  // query.getComplementedFrom() != null
  SeqView b;
};
struct Sec { int start, end; XM_INLINE int length() const { return end - start; } };

struct MatcherD {  // M/HashBlock_Matcher.java state
  int ref_start, ref_len, block_len, section_len, max_section_index;
  int loc_size;           // locations.size()
  uint32_t* materialized; // bit i: locations[i] != null
  int mat_words;
  // direct-address tables of the materialised sections (HashBlock_Matcher.indexSection :40-77): entry = position
  // relative to the section start, T_NO or T_MULTI.  A few slots per matcher; sections beyond them are scanned.
  int16_t* tables; int table_entries, n_slots, slots_used;
  int slot_section[8];
};
static const int16_t T_NO = -1, T_MULTI = -2;
struct Analysis {  // M/AlignmentAnalysis.java
  MatcherD* matcher;
  int predicted, last_checked, confident;
  double max_ins, max_del;
};

XM_INLINE DAln aln_null() { DAln a; a.valid = 0; a.n = 0; a.b = nullptr; a.penalty = 0; a.aligned = 0; a.ref_reversed = 0; return a; }

XM_FN double block_penalty(const Params& p, const ACtx& c, const Blk& k) {  // AlignmentParameters.getPenalty(AlignedBlock) :106-126
  double pen = 0;
  if (k.a_len == k.b_len) {
    // lanes classify 32 base pairs at a time; the non-zero penalties are then added in base order (x + 0.0 == x, so
    // skipping the zero terms keeps the reference's left-to-right double sum bit for bit)
    const int lane = lane_id();
    XM_NOUNROLL
    for (int base = 0; base < k.a_len; base += XM_LANES) {
      const int i = base + lane;
      double v = 0;
      if (i < k.a_len) v = p.base_penalty(c.a.at(k.a_start + i), c.b.at(k.b_start + i));
      unsigned m = warp_ballot(v != 0);
      XM_NOUNROLL
      while (m) { const int src = first_bit(m) - 1; m &= m - 1; pen += warp_shfl(v, src); }
    }
    warp_sync();
  } else if (k.a_len > 0) { pen += p.ins_start; pen += p.ins_ext * k.a_len; }
  else { pen += p.del_start; pen += p.del_ext * k.b_len; }
  return pen;
}
XM_FN double block_penalty_range(const Params& p, const SeqView& a, const SeqView& b, const Blk& k, int start_b, int end_b) {  // :128-154
  double pen = 0;
  if (k.a_len == k.b_len) {
    const int lane = lane_id();
    XM_NOUNROLL
    for (int base = 0; base < k.a_len; base += XM_LANES) {
      const int i = base + lane, bi = k.b_start + i;
      double v = 0;
      if (i < k.a_len && bi >= start_b && bi < end_b) v = p.base_penalty(a.at(k.a_start + i), b.at(bi));
      unsigned m = warp_ballot(v != 0);
      XM_NOUNROLL
      while (m) { const int src = first_bit(m) - 1; m &= m - 1; pen += warp_shfl(v, src); }
    }
    warp_sync();
  } else if (k.b_start < end_b && k.b_start + k.b_len > start_b) {
    if (k.a_len > 0) { pen += p.ins_start; pen += p.ins_ext * k.a_len; } else { pen += p.del_start; pen += p.del_ext * k.b_len; }
  }
  return pen;
}
// AlignmentParameters.newSequenceAlignment :73-95 — blocks must already live in scratch/store
XM_FN DAln new_aln(const Params& p, const ACtx& c, Blk* blocks, int n, int ref_reversed) {
  int aligned_len = 0;
  double total = 0;
  XM_NOUNROLL
  for (int i = 0; i < n; i++) { total += block_penalty(p, c, blocks[i]); aligned_len += blocks[i].a_len; }
  if (n > 0 && p.start_free && blocks[0].b_len == 0) total -= p.ins_start;
  double aligned = total;
  if (n > 0) { int un = c.a.len - aligned_len; total += (double)un * p.unaligned; }
  DAln r; r.valid = 1; r.n = n; r.b = blocks; r.penalty = total; r.aligned = aligned; r.ref_reversed = ref_reversed;
  return r;
}
XM_INLINE int aln_start_a(const DAln& a) { return a.b[0].a_start; }
XM_INLINE int aln_end_a(const DAln& a) { return a.b[a.n - 1].a_start + a.b[a.n - 1].a_len; }
XM_INLINE int aln_start_b(const DAln& a) { return a.b[0].b_start; }
XM_INLINE int aln_end_b(const DAln& a) { return a.b[a.n - 1].b_start + a.b[a.n - 1].b_len; }

// ---------------- HashBlock_Matcher ----------------
static const int M_NO = -1, M_MULTI = -2, M_UNKNOWN = -3;

XM_HD inline int log4_floor_plus1(int x) {  // (int)(Math.log(x) / Math.log(4) + 1) for x >= 1, x not a power of 4 boundary-sensitive: exact integers
  int k = 0; long long p = 4;
  XM_NOUNROLL
  while (p <= (long long)x) { k++; p *= 4; }
  return k + 1;
}
XM_FN MatcherD* matcher_new(WS& w, const ACtx& c, const Sec& rsec, int section_len) {  // :14-29
  MatcherD* m = (MatcherD*)w.salloc(sizeof(MatcherD));
  if (!m) return nullptr;
  if (section_len < 1) section_len = 1;
  // (int)(log(5s)/log(4) + 1): 5s is never a power of 4, so the integer form is exact
  m->block_len = log4_floor_plus1(section_len * 5);
  if (m->block_len < 3) m->block_len = 3;
  m->ref_start = rsec.start; m->ref_len = rsec.length(); m->section_len = section_len;
  m->max_section_index = (c.b.len - 1 - m->ref_start) / section_len;
  m->loc_size = 0;
  // lookups only ask for sections that intersect [ref_start, ref_start + ref_len] (matcher_lookup clamps to the
  // window), so the "materialised" bitmap needs ref_len / section_len + 2 bits; an index beyond it asks for more workspace
  int n_sec = imin(m->max_section_index + 1, (m->ref_len + 1) / section_len + 2);
  int words = (n_sec + 31) / 32;
  if (words < 1) words = 1;
  if (words > 4096) words = 4096;
  m->mat_words = words;
  m->materialized = (uint32_t*)w.salloc((long long)words * 4);
  if (!m->materialized) return nullptr;
  XM_NOUNROLL
  for (int i = 0; i < words; i++) m->materialized[i] = 0;
  m->tables = nullptr; m->table_entries = 0; m->n_slots = 0; m->slots_used = 0;
  if (section_len >= 3 && section_len < 32000 && m->block_len <= 7) {
    int entries = 1 << (2 * m->block_len);
    int slots = imin(8, m->max_section_index + 1);
    long long bytes = (long long)slots * entries * 2 + 16;
    if (slots > 0 && w.scratch_top + bytes + 4096 <= w.scratch_size / 2) {  // optional: without room the sections are scanned instead
      char* p = (char*)w.salloc(bytes);
      p += (16 - ((uintptr_t)p & 15)) & 15;
      m->tables = (int16_t*)p; m->table_entries = entries; m->n_slots = slots;
    }
  }
  return m;
}
XM_HD inline int matcher_encode(const SeqView& s, int index, int block_len) {  // encodeBlock :79-91
  if (index + block_len > s.len) return M_UNKNOWN;
  int sum = 0;
  XM_NOUNROLL
  for (int i = 0; i < block_len; i++) {
    uint8_t h = s.at(index + i);
    if (bp_is_ambiguous(h)) return M_UNKNOWN;
    sum = sum * 4 + (h == 1 ? 0 : h == 2 ? 1 : h == 4 ? 2 : 3);  // code 0 ('-') would throw in the reference; never present
  }
  return sum;
}
// indexSection(sectionIndex) :40-77, visiting every (position, encoding) the reference stores
template <class F>
XM_INLINE void matcher_scan_encodings(const MatcherD& m, const SeqView& ref, int section_index, F&& f) {
  int max_poss = (1 << (2 * m.block_len)) - 1;
  int prev = M_UNKNOWN;
  int start = m.ref_start + section_index * m.section_len;
  int end = imin(start + m.section_len, m.ref_start + m.ref_len - m.block_len);
  XM_NOUNROLL
  for (int i = start; i < end; i++) {
    int enc;
    if (prev == M_UNKNOWN) enc = matcher_encode(ref, i, m.block_len);
    else {
      uint8_t nc = ref.at(i + m.block_len - 1);
      if (bp_is_ambiguous(nc)) enc = M_UNKNOWN;
      else enc = ((prev * 4) & max_poss) + (nc == 1 ? 0 : nc == 2 ? 1 : nc == 4 ? 2 : 3);
    }
    if (enc == M_UNKNOWN) continue;
    f(i - start, enc);
    prev = enc;
  }
}
// value of section[encoded] after indexSection(sectionIndex)
XM_FN int matcher_section_value(WS& w, MatcherD& m, const SeqView& ref, int section_index, int target) {
  XM_CHECK_MASK(w);
  int start = m.ref_start + section_index * m.section_len;
  if (m.tables != nullptr) {
    int slot = -1;
    XM_NOUNROLL
    for (int i = 0; i < m.slots_used; i++) if (m.slot_section[i] == section_index) { slot = i; break; }
    if (slot < 0 && m.slots_used < m.n_slots) {
      PhaseClock pc_(&w.st_cyc[4]);
      slot = m.slots_used++;
      m.slot_section[slot] = section_index;
      int16_t* t = m.tables + (long long)slot * m.table_entries;
      {  // lanes clear the table to T_NO together (16 bytes per lane per round; table_entries is a multiple of 8)
        uint4 fill = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
        uint4* t4 = (uint4*)t;
        int n16 = m.table_entries / 8;
        XM_NOUNROLL
        for (int i = lane_id(); i < n16; i += XM_LANES) t4[i] = fill;
        warp_sync();
      }
      matcher_scan_encodings(m, ref, section_index, [&](int rel, int enc) { t[enc] = (t[enc] == T_NO) ? (int16_t)rel : T_MULTI; });
    }
    if (slot >= 0) {
      int16_t v = m.tables[(long long)slot * m.table_entries + target];
      return v == T_NO ? M_NO : v == T_MULTI ? M_MULTI : start + (int)v;
    }
  }
  int value = M_NO;
  matcher_scan_encodings(m, ref, section_index, [&](int rel, int enc) { if (enc == target) value = (value == M_NO) ? start + rel : M_MULTI; });
  return value;
}
XM_HD inline bool matcher_get_section(WS& w, MatcherD& m, int index) {  // getSection :203-215; false = null entry
  if (index >= m.mat_words * 32) { w.fail(Q_NEED_MORE); return false; }
  if (m.loc_size > index) return (m.materialized[index >> 5] >> (index & 31)) & 1;
  m.loc_size = index + 1;
  m.materialized[index >> 5] |= (1u << (index & 31));
  return true;
}
XM_FN int matcher_scan_section(const MatcherD& m, const ACtx& c, int query_index, int section_index) {  // :143-171
  int result = M_NO;
  int start = m.ref_start + section_index * m.section_len, end = start + m.section_len;
  XM_NOUNROLL
  for (int i = start; i < end; i++) {
    bool ok = !(i + m.block_len > m.ref_start + m.ref_len);
    // canPositionsMatch reads query/reference without bounds checks; out-of-range reads throw in the reference
    XM_NOUNROLL
    for (int k = 0; ok && k < m.block_len; k++) {
      if (query_index + k >= c.a.len || i + k >= c.b.len) { ok = false; break; }
      if (!bp_can_match(c.a.at(query_index + k), c.b.at(i + k))) ok = false;
    }
    if (ok) { if (result == M_NO) result = i; else return M_MULTI; }
  }
  return result;
}
XM_FN int matcher_lookup(WS& w, MatcherD& m, const ACtx& c, int query_index, int min_ref, int max_ref) {  // :98-141
  XM_CHECK_MASK(w);
  if (min_ref < 0) return M_UNKNOWN;
  if (max_ref > c.b.len) return M_UNKNOWN;
  int enc = matcher_encode(c.a, query_index, m.block_len);
  if (enc < 0) return M_UNKNOWN;
  int matched = M_NO;
  int min_sec = imax(0, (min_ref - m.ref_start) / m.section_len);
  int max_sec = imin(m.max_section_index, (max_ref - m.ref_start) / m.section_len);
  XM_NOUNROLL
  for (int si = min_sec; si <= max_sec; si++) {
    bool have = matcher_get_section(w, m, si);
    if (w.status != 0) return M_UNKNOWN;
    int looked;
    if (m.section_len < 3) looked = matcher_scan_section(m, c, query_index, si);
    else { if (have) looked = matcher_section_value(w, m, c.b, si, enc); else return M_UNKNOWN; }
    if (looked == M_UNKNOWN) return M_UNKNOWN;
    if (looked == M_MULTI) return M_MULTI;
    if (looked == M_NO) continue;
    if (looked < min_ref || looked > max_ref) continue;
    if (matched != M_NO) return M_MULTI;
    matched = looked;
  }
  return matched;
}

// ---------------- PathAligner ----------------
// One lattice node (M/AlignmentNode.java), 32 bytes = one DRAM sector.  The lattice is a dense W x H array in a region of the arena that
// is dedicated to it (WS::cell_hdr): meta carries the generation of the search that wrote the node, so a node of another generation
// is absent and nothing is cleared between searches.  stamp = value of the search's write counter when the node was last written: a
// neighbour whose stamp is newer than the stamps of all three of its predecessors would be recomputed from unchanged inputs, i.e. to
// the values it already holds, so its evaluation is skipped (39 % of all evaluations on the 150 bp workload).
struct alignas(16) PNode { double pen, ins_x, ins_y; uint32_t stamp; uint32_t meta; };
struct alignas(8) PMeta { uint32_t stamp, meta; };   // the last 8 bytes of a node, read with one 64-bit load  // meta = generation << 8 | flags (2 reachedMain, 4 reachedOther)
// One queued node: packed (x, y) and the next entry of the same priority (-1 = last).
struct PEnt { uint32_t xy; int32_t next; };
struct PathState {
  Params prm; ACtx ctx;
  int an_confident; double an_max_ins, an_max_del;   // the AlignmentAnalysis in force, by value
  int start_a, end_a, start_b, end_b, A, B, W, H;
  int diagonal, step, reverse, may_extend;
  int start_x, start_y, goal_x, goal_y;
  PNode* nodes; uint32_t gen; uint32_t clock;   // node (x, y) = nodes[x * H + y]; present iff (meta >> 8) == gen
  const uint8_t* qa; const uint8_t* rb;  // the two sections, one code per byte
  PEnt* ent; int ent_cap;
  double max_interesting;
};
XM_INLINE uint8_t pa_qa(const PathState& s, int i) { return s.qa[i]; }
XM_INLINE uint8_t pa_rb(const PathState& s, int j) { return s.rb[j]; }
XM_INLINE bool pa_can_remove(const Blk& b) {  // canRemoveSection :358-366
  if (b.a_len <= 0 && b.b_len <= 0) return true;
  if ((b.a_start <= 0 && b.a_len <= 0) || (b.b_start <= 0 && b.b_len <= 0)) return true;
  return false;
}
XM_INLINE uint32_t pa_pack_xy(int x, int y) { return ((uint32_t)(uint16_t)(int16_t)x << 16) | (uint32_t)(uint16_t)(int16_t)y; }

// The reference's queue is a TreeMap<priority, List<node>> (PathAligner.java:446-473,153-192): nodes of the lowest
// priority are processed in insertion order, including the ones appended while that list is being walked.  PaQueue
// keeps exactly that structure: one FIFO (linked through PEnt::next) per distinct priority.  On the device the
// buckets live in REGISTERS, one bucket per lane: finding the bucket of a priority is one compare + ballot, and the
// bucket being drained (the minimum) is held warp-uniformly - so a pop is two loads and a push two stores, where a
// binary heap cost a dependent chain of ~8 loads per operation.  Buckets beyond 32 go to a spill array kept SORTED by
// priority (binary search to find, lane-parallel shift to insert, the front is the minimum): long reads with large
// budgets keep hundreds of distinct priorities alive.
struct PaOverflow { double key; int head, tail; };
// The warp-uniform state of one search: its constants and the queue's scalars.  On the device it lives in shared memory, one frame
// per warp (pa_frame), and is read where it is used: at 32 registers the search cannot hold all of it, and a value that ptxas
// spills goes to local memory, where every lane keeps (and writes through to L2/HBM) its own copy of the same bytes, while a
// shared-memory read is one broadcast load.  Writes follow the warp-uniform rule (§3 of DESIGN.md): all lanes store the same
// value while the warp is converged.
struct PaFrame {
  const double* pen_tab; const uint8_t* cls_tab; PNode* nodes; const uint8_t* qa; const uint8_t* rb;
  double ins_start, ins_ext, del_start, del_ext, unaligned, max_ins, max_del, budget, min_indel;
  unsigned long long steps;
  // PaQueue: popped entries are chained for reuse once the fresh ones run out; cur_* is the bucket being drained
  // (cur_key == activePenalty); the live spill buckets are ovf[ovf_lo, ovf_hi), ascending keys
  PEnt* ent; PaOverflow* ovf;
  double cur_key;
  int n_ent, cap, free_head, cur_head, cur_tail, ovf_lo, ovf_hi, cap_ovf;
  int A, B, H, step, goal_x, goal_y, diagonal;
  uint32_t gen, clock;   // clock: the write counter (PNode::stamp)
  int16_t tx, ty, x, y;  // the node being expanded and the neighbour being evaluated (a lattice side is at most 32000)
  uint8_t may_extend, confident;
};
static_assert(sizeof(PaFrame) == 224, "32 frames keep the full kernel's static shared memory within 48 KB");
// A frame value read where it is used.  On the device this is a volatile shared-memory load: the compiler neither merges it with an
// earlier load nor keeps the value in a register across the loop body, where it would be spilled.
template <class T> XM_INLINE T pa_ld(const T& v) {
#if defined(__CUDA_ARCH__)
  return *(const volatile T*)&v;
#else
  return v;
#endif
}
#if defined(__CUDA_ARCH__)
__shared__ PaFrame pa_frame[32];   // one per warp of the block; only the full kernel's image contains the search
#endif
struct PaQueue {
#if defined(__CUDA_ARCH__)
  double bkey; int bhead, btail;           // this lane's bucket (bhead < 0: free)
#else
  double bkey[32]; int bhead[32], btail[32];
#endif
  XM_INLINE void init(PaFrame& f, PEnt* e, int capacity, PaOverflow* o, int cap_o) {
    f.ent = e; f.n_ent = 0; f.cap = capacity; f.free_head = -1; f.cur_key = 0; f.cur_head = -1; f.cur_tail = -1; f.ovf = o; f.ovf_lo = 0; f.ovf_hi = 0; f.cap_ovf = cap_o;
#if defined(__CUDA_ARCH__)
    bkey = 0; bhead = -1; btail = -1;
#else
    for (int i = 0; i < 32; i++) { bkey[i] = 0; bhead[i] = -1; btail[i] = -1; }
#endif
  }
  // 0 ok, 1 out of entry space, 2 out of overflow space.  pri >= cur_key always (estimates are clamped to activePenalty).
  XM_INLINE int push(PaFrame& f, double pri, int x, int y) {
    PEnt* const ent = f.ent;
    int id;
    if (f.n_ent < f.cap) { id = f.n_ent; f.n_ent = id + 1; }
    else { id = f.free_head; if (id < 0) return 1; f.free_head = ent[id].next; }
    PEnt e; e.xy = pa_pack_xy(x, y); e.next = -1;
    ent[id] = e;
    if (pri == f.cur_key) {
      const int t = f.cur_tail;
      if (t >= 0) ent[t].next = id; else f.cur_head = id;
      f.cur_tail = id;
      return 0;
    }
#if defined(__CUDA_ARCH__)
    const int lane = (int)(threadIdx.x & 31);
    const unsigned hit = __ballot_sync(0xffffffffu, bhead >= 0 && bkey == pri);
    if (hit != 0) {
      const int b = __ffs(hit) - 1;
      const int t = __shfl_sync(0xffffffffu, btail, b);
      ent[t].next = id;
      if (lane == b) btail = id;
      return 0;
    }
#else
    for (int b = 0; b < 32; b++) if (bhead[b] >= 0 && bkey[b] == pri) { ent[btail[b]].next = id; btail[b] = id; return 0; }
#endif
    // spill array: first position with key >= pri.  On the device the lanes probe 32 pivots per round (a 32-ary search: two
    // dependent loads for up to 1024 buckets, where a binary search chases ten)
    PaOverflow* const ovf = f.ovf;
    int lo = f.ovf_lo, hi = f.ovf_hi;
#if defined(__CUDA_ARCH__)
    XM_NOUNROLL
    while (hi - lo > 0) {
      const int n = hi - lo;
      const int stride = (n + 31) >> 5;                       // 32 pivots: the LAST element of each chunk of `stride`
      const int at = lo + imin(n, (lane + 1) * stride) - 1;
      const bool less = ovf[at].key < pri;                     // monotone over lanes (ascending keys)
      const int k = __popc(__ballot_sync(0xffffffffu, less));  // chunks entirely below pri
      const int nlo = lo + imin(n, k * stride);
      if (k >= 32 || nlo >= hi) { lo = hi; break; }
      hi = lo + imin(n, (k + 1) * stride); lo = nlo;
      if (stride == 1) { break; }                              // chunk k is one element and it is >= pri
    }
#else
    XM_NOUNROLL
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ovf[mid].key < pri) lo = mid + 1; else hi = mid; }
#endif
    if (lo < f.ovf_hi && ovf[lo].key == pri) { ent[ovf[lo].tail].next = id; ovf[lo].tail = id; return 0; }
#if defined(__CUDA_ARCH__)
    const unsigned fre = __ballot_sync(0xffffffffu, bhead < 0);
    if (fre != 0) { const int b = __ffs(fre) - 1; if (lane == b) { bkey = pri; bhead = id; btail = id; } return 0; }
#else
    for (int b = 0; b < 32; b++) if (bhead[b] < 0) { bkey[b] = pri; bhead[b] = id; btail[b] = id; return 0; }
#endif
    if (f.ovf_hi >= f.cap_ovf) {
      const int olo = f.ovf_lo;
      if (olo == 0) return 2;
      const int n = f.ovf_hi - olo;  // slide the live range back to the start of the array
#if defined(__CUDA_ARCH__)
      XM_NOUNROLL
      for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        PaOverflow t; if (i < n) t = ovf[olo + i];
        __syncwarp();
        if (i < n) ovf[i] = t;
        __syncwarp();
      }
#else
      for (int i = 0; i < n; i++) ovf[i] = ovf[olo + i];
#endif
      lo -= olo; f.ovf_lo = 0; f.ovf_hi = n;
    }
    {  // insert at lo: shift [lo, ovf_hi) up by one, highest elements first
      const int ohi = f.ovf_hi;
#if defined(__CUDA_ARCH__)
      XM_NOUNROLL
      for (int top = ohi; top > lo; top -= 32) {
        const int i = top - 1 - lane;
        PaOverflow t; if (i >= lo) t = ovf[i];
        __syncwarp();
        if (i >= lo) ovf[i + 1] = t;
        __syncwarp();
      }
#else
      for (int i = ohi - 1; i >= lo; i--) ovf[i + 1] = ovf[i];
#endif
      PaOverflow t; t.key = pri; t.head = id; t.tail = id;
      ovf[lo] = t;
      f.ovf_hi = ohi + 1;
    }
    return 0;
  }
  // false: queue empty.  Otherwise (x, y) of the next node in the reference's order; f.cur_key is its priority.
  XM_INLINE bool pop(PaFrame& f, int& x, int& y) {
    PEnt* const ent = f.ent;
    int head = f.cur_head;
    if (head < 0) {  // next bucket = the smallest remaining priority (all are > cur_key)
      bool have = false; double best = 0; int where = -1;  // where: 0..31 lane bucket, 32+i overflow entry i
#if defined(__CUDA_ARCH__)
      const int lane = (int)(threadIdx.x & 31);
      const unsigned live = __ballot_sync(0xffffffffu, bhead >= 0);
      if (live != 0) {
        // non-negative doubles order like their bit patterns: min of the high words, then of the low words among ties
        const unsigned long long bits = (unsigned long long)__double_as_longlong(bkey);
        const unsigned hi = bhead >= 0 ? (unsigned)(bits >> 32) : 0xffffffffu;
        const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
        const unsigned lo = (bhead >= 0 && hi == mhi) ? (unsigned)bits : 0xffffffffu;
        const unsigned mlo = __reduce_min_sync(0xffffffffu, lo);
        const unsigned who = __ballot_sync(0xffffffffu, bhead >= 0 && hi == mhi && (unsigned)bits == mlo);
        where = __ffs(who) - 1;
        best = __longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo));
        have = true;
      }
#else
      for (int b = 0; b < 32; b++) if (bhead[b] >= 0 && (!have || bkey[b] < best)) { have = true; best = bkey[b]; where = b; }
#endif
      const int olo = f.ovf_lo;
      if (olo < f.ovf_hi && (!have || f.ovf[olo].key < best)) { have = true; best = f.ovf[olo].key; where = 32; }
      if (!have) return false;
      f.cur_key = best;
      if (where >= 32) {
        const PaOverflow o = f.ovf[olo];
        head = o.head; f.cur_tail = o.tail;
        if (olo + 1 == f.ovf_hi) { f.ovf_lo = 0; f.ovf_hi = 0; } else f.ovf_lo = olo + 1;
      } else {
#if defined(__CUDA_ARCH__)
        head = __shfl_sync(0xffffffffu, bhead, where); f.cur_tail = __shfl_sync(0xffffffffu, btail, where);
        if (lane == where) bhead = -1;
#else
        head = bhead[where]; f.cur_tail = btail[where]; bhead[where] = -1;
#endif
      }
    }
    const PEnt e = ent[head];
    ent[head].next = f.free_head; f.free_head = head;
    f.cur_head = e.next;
    if (e.next < 0) f.cur_tail = -1;
    x = (int)(int16_t)(e.xy >> 16); y = (int)(int16_t)(e.xy & 0xffffu);
    return true;
  }
};

XM_INLINE int pa_signed_dist(const PathState& s, int x, int y) { return x - y - s.diagonal; }
XM_INLINE PNode pa_node(const PathState& s, int idx) {   // a node as the traceback reads it: past L1, it visits each node about once
#if defined(__CUDA_ARCH__)
  const double2 a = __ldcg((const double2*)&s.nodes[idx]);
  const double2 b = __ldcg((const double2*)&s.nodes[idx] + 1);
  PNode n; n.pen = a.x; n.ins_x = a.y; n.ins_y = b.x;
  const unsigned long long m = (unsigned long long)__double_as_longlong(b.y);
  n.stamp = (uint32_t)m; n.meta = (uint32_t)(m >> 32);
  return n;
#else
  return s.nodes[idx];
#endif
}
XM_INLINE bool pa_get(const PathState& s, int x, int y, int& idx) {
  if (x < 0 || x >= s.W || y < 0 || y >= s.H) return false;
  idx = x * s.H + y;
  return (pa_node(s, idx).meta >> 8) == s.gen;
}
XM_HD inline double pa_estimate(const PathState& s, int x, int y, const PNode& n, int fl) {  // estimateOverallPenalty :475-521
  if (!s.an_confident) return n.pen;
  int sd = pa_signed_dist(s, x, y);
  const Params& p = s.prm;
  if (fl & 2) {
    if (sd * s.step > 0) { double ie = fabs(sd * p.ins_ext); if (ie > s.an_max_ins) return XM_DISALLOWED; }
    else { double de = fabs(sd * p.del_ext); if (de > s.an_max_del) return XM_DISALLOWED; }
    if (fl & 4) return n.pen;
    return n.pen + dmin(p.ins_start + p.ins_ext, p.del_start + p.del_ext);
  }
  if (sd * s.step < 0) {
    double ie = fabs(sd * p.ins_ext);
    if (ie > s.an_max_ins) return XM_DISALLOWED;
    double is = dmin(p.ins_start, n.ins_x - n.pen);
    return n.pen + is + ie;
  } else {
    double de = fabs(sd * p.del_ext);
    if (de > s.an_max_del) return XM_DISALLOWED;
    double ds = dmin(p.del_start, n.ins_y - n.pen);
    return n.pen + ds + de;
  }
}
// PathAligner.align :120-192: seeds the queue (:120-150) and runs the best-first search (:153-192) with explore
// :722-729, update :555-571, computeUpdated :573-719, putNode :446-473 and estimateOverallPenalty :475-521 folded
// into ONE compact loop: every per-search constant is read from the warp's PaFrame where it is used, the three neighbours
// share one copy of the update code, and base pairs are classified through the 256-entry tables.  This loop is where gapped
// reads spend their time.  Returns 0 goal reached (last_x/last_y), 1 over budget (null), 2 failed (w.status set).
XM_FN int pa_search(WS& w, PathState& S, PaOverflow* ovf, int cap_ovf, int& last_x, int& last_y) {
  XM_CHECK_MASK(w);
#if defined(__CUDA_ARCH__)
  PaFrame& F = pa_frame[threadIdx.x >> 5];
#else
  PaFrame frame; PaFrame& F = frame;
#endif
  F.A = S.A; F.B = S.B; F.H = S.H; F.step = S.step; F.goal_x = S.goal_x; F.goal_y = S.goal_y; F.diagonal = S.diagonal;
  F.may_extend = S.may_extend != 0; F.confident = S.an_confident != 0;
  F.ins_start = S.prm.ins_start; F.ins_ext = S.prm.ins_ext; F.del_start = S.prm.del_start; F.del_ext = S.prm.del_ext; F.unaligned = S.prm.unaligned;
  F.max_ins = S.an_max_ins; F.max_del = S.an_max_del; F.budget = S.max_interesting + 0.000001;
  F.min_indel = dmin(S.prm.ins_start + S.prm.ins_ext, S.prm.del_start + S.prm.del_ext);
  F.pen_tab = S.prm.pen_tab; F.cls_tab = S.prm.cls_tab; F.nodes = S.nodes; F.qa = S.qa; F.rb = S.rb;
  F.gen = S.gen; F.clock = S.clock; F.steps = 0;
  PaQueue Q;
  Q.init(F, S.ent, S.ent_cap, ovf, cap_ovf);
  int qrc = 0;
  // seeding :120-150.  activePenalty is 0 here, estimates are never negative: no clamping needed.  One loop (one copy of
  // the queue code) walks the free-start nodes :120-139 and then the query-overhang nodes :140-150.
  {
    const int A = S.A, B = S.B, step = S.step, start_x = S.start_x, start_y = S.start_y;
    const bool along_y = B >= A, may_extend = S.may_extend != 0;
    double sisp = XM_DISALLOWED;
    if (along_y && may_extend) sisp = S.prm.starting_ins_start();
    const int cnt1 = (along_y ? imax(0, B - A) : imax(0, A - B)) + 1;
    const int cnt2 = may_extend ? imax(0, j2i(S.an_max_ins / S.prm.del_ext) - 1) : 0;
    XM_NOUNROLL
    for (int i = 0; i < cnt1 + cnt2 && qrc == 0; i++) {
      PNode n; int x, y;
      if (i < cnt1) {
        n.pen = 0; n.ins_x = along_y ? sisp : XM_DISALLOWED; n.ins_y = XM_DISALLOWED;
        x = along_y ? start_x : start_x + i * step; y = along_y ? start_y + i * step : start_y;
      } else {
        const int k = i - cnt1 + 1;
        x = start_x + k * step; y = start_y;
        n.pen = k * S.prm.unaligned; n.ins_x = XM_DISALLOWED; n.ins_y = XM_DISALLOWED;
        // outside the lattice the reference still queues the node (saveNode ignores x < 0; x > width is stored but
        // never read), and popping it can end the search when its priority exceeds the budget
        if (x < -32000 || x > 32000) { qrc = 1; break; }
      }
      const uint32_t clock = F.clock + 1;
      F.clock = clock;
      n.stamp = clock; n.meta = S.gen << 8;
      qrc = Q.push(F, pa_estimate(S, x, y, n, 0), x, y);
      if (x >= 0 && x < S.W) S.nodes[x * S.H + y] = n;
    }
  }
  int rc = 2;
  XM_NOUNROLL
  while (qrc == 0) {
    {
      int tx, ty;
      if (!Q.pop(F, tx, ty)) { w.fail(Q_INTERNAL); break; }  // priorities.poll() == null -> NullPointerException
      F.tx = (int16_t)tx; F.ty = (int16_t)ty;
      F.steps = F.steps + 1;
      if (F.cur_key > F.budget) { rc = 1; break; }
      if (tx == F.goal_x) { last_x = tx; last_y = ty; rc = 0; break; }
    }
    XM_NOUNROLL
    for (int nb = 0; nb < 3; nb++) {  // (x+step, y), (x, y+step), (x+step, y+step)
      {
        const int step = pa_ld(F.step);
        const int x = pa_ld(F.tx) + (nb != 1 ? step : 0), y = pa_ld(F.ty) + (nb != 0 ? step : 0);
        if (x <= 0 || x > pa_ld(F.A) || y <= 0 || y > pa_ld(F.B)) continue;
        F.x = (int16_t)x; F.y = (int16_t)y;
      }
      // below, the neighbour's coordinates and index and the search's constants are read from the frame where they are used
      uint32_t fpk;   // 3 flag bits (1 present | 6 reached) per predecessor: overlay, insertion, deletion
      bool he;
      {
        PNode* const nodes = pa_ld(F.nodes);
        const int step = pa_ld(F.step), ie = pa_ld(F.x) * pa_ld(F.H) + pa_ld(F.y), il = ie - step * pa_ld(F.H), iu = ie - step, id = il - step;
        // stamp (low word) and meta (high word) of the node and of its three predecessors: four independent 8-byte loads
        const PMeta me = *(const PMeta*)&nodes[ie].stamp, ml = *(const PMeta*)&nodes[il].stamp, mu = *(const PMeta*)&nodes[iu].stamp, md = *(const PMeta*)&nodes[id].stamp;
        const uint32_t gen = pa_ld(F.gen);
        he = (me.meta >> 8) == gen;
        const bool hl = (ml.meta >> 8) == gen, hu = (mu.meta >> 8) == gen, hd = (md.meta >> 8) == gen;
        if (he) {
          // every predecessor was last written before this node was: recomputing it would reproduce the values it holds (no improvement)
          uint32_t newest = 0;
          if (hl && ml.stamp > newest) newest = ml.stamp;
          if (hu && mu.stamp > newest) newest = mu.stamp;
          if (hd && md.stamp > newest) newest = md.stamp;
          if (me.stamp > newest) continue;
        }
        fpk = (hd ? (1u | (md.meta & 6u)) : 0u) | (hl ? (1u | (ml.meta & 6u)) << 3 : 0u) | (hu ? (1u | (mu.meta & 6u)) << 6 : 0u);
      }
      double ins_x = XM_DISALLOWED, ins_y = XM_DISALLOWED, overlay = XM_DISALLOWED;
      {
        PNode* const nodes = pa_ld(F.nodes);
        const uint8_t* const qa = pa_ld(F.qa); const uint8_t* const rb = pa_ld(F.rb); const uint8_t* const cls_tab = pa_ld(F.cls_tab);
        const int x = pa_ld(F.x), y = pa_ld(F.y), step = pa_ld(F.step), ie = x * pa_ld(F.H) + y;
        if (fpk & 1u) overlay = nodes[ie - step * pa_ld(F.H) - step].pen + pa_ld(F.pen_tab)[((int)qa[x - 1] << 4) | (int)rb[y - 1]];
        if (fpk & 8u) {
          const int il = ie - step * pa_ld(F.H);
          const double lp = nodes[il].pen;
          if (y == pa_ld(F.goal_y) && pa_ld(F.may_extend)) ins_x = lp + pa_ld(F.unaligned);
          else {
            // qa / rb are padded with the sentinel code on both sides: an index off the section leaves the move allowed, as in the reference
            bool allowed = (cls_tab[((int)qa[x - 1 - step] << 5) | (int)rb[y - 1]] & 1) != 0;
            if (allowed) allowed = (cls_tab[((int)qa[x - 1] << 5) | (int)rb[y - 1 + step]] & 6) == 0;
            const double nw = allowed ? lp + pa_ld(F.ins_start) + pa_ld(F.ins_ext) : XM_DISALLOWED;
            ins_x = dmin(nodes[il].ins_x + pa_ld(F.ins_ext), nw);
          }
        }
        if (fpk & 64u) {
          const int iu = ie - step;
          bool allowed = (cls_tab[((int)qa[x - 1] << 5) | (int)rb[y - 1 - step]] & 1) != 0;
          if (allowed) allowed = (cls_tab[((int)qa[x - 1 + step] << 5) | (int)rb[y - 1]] & 6) == 0;
          const double nw = allowed ? nodes[iu].pen + pa_ld(F.del_start) + pa_ld(F.del_ext) : XM_DISALLOWED;
          ins_y = dmin(nodes[iu].ins_y + pa_ld(F.del_ext), nw);
        }
      }
      const double best = dmin(dmin(overlay, ins_x), ins_y);
      if (he) {
        const PNode* const o = pa_ld(F.nodes) + (pa_ld(F.x) * pa_ld(F.H) + pa_ld(F.y));
        if (!(best < o->pen || ins_x < o->ins_x || ins_y < o->ins_y)) continue;
      }
      const int sd = pa_ld(F.x) - pa_ld(F.y) - pa_ld(F.diagonal);
      int fl = 0;
      if (best != XM_DISALLOWED) {
        const uint32_t src = (best == overlay) ? fpk : (best == ins_x) ? fpk >> 3 : fpk >> 6;
        fl = (int)(src & 6u) | (sd == 0 ? 2 : 4);
      }
      // estimateOverallPenalty :475-521
      double est = best;
      if (pa_ld(F.confident)) {
        const int sds = sd * pa_ld(F.step);
        if (fl & 2) {
          const bool over = (sds > 0) ? (fabs(sd * pa_ld(F.ins_ext)) > pa_ld(F.max_ins)) : (fabs(sd * pa_ld(F.del_ext)) > pa_ld(F.max_del));
          if (over) est = XM_DISALLOWED;
          else if (!(fl & 4)) est = best + pa_ld(F.min_indel);
        } else if (sds < 0) {
          const double ie_ = fabs(sd * pa_ld(F.ins_ext));
          if (ie_ > pa_ld(F.max_ins)) est = XM_DISALLOWED;
          else est = best + dmin(pa_ld(F.ins_start), ins_x - best) + ie_;
        } else {
          const double de = fabs(sd * pa_ld(F.del_ext));
          if (de > pa_ld(F.max_del)) est = XM_DISALLOWED;
          else est = best + dmin(pa_ld(F.del_start), ins_y - best) + de;
        }
      }
      // the node is stored before it is queued, so that none of its values has to outlive the queue code; a push that fails
      // ends the search with Q_NEED_MORE, and no later search reads a node of this generation
      const uint32_t clock = pa_ld(F.clock) + 1;
      F.clock = clock;
      PNode n; n.pen = best; n.ins_x = ins_x; n.ins_y = ins_y; n.stamp = clock; n.meta = (pa_ld(F.gen) << 8) | (uint32_t)fl;
      pa_ld(F.nodes)[(pa_ld(F.x) * pa_ld(F.H) + pa_ld(F.y))] = n;
      const double active = pa_ld(F.cur_key);
      if (est < active) est = active;
      qrc = Q.push(F, est, pa_ld(F.x), pa_ld(F.y));
      if (qrc != 0) break;
    }
  }
  S.clock = F.clock;
  if (qrc != 0) { w.fail(Q_NEED_MORE); rc = 2; }
  w.st_path_steps += F.steps;
  return rc;
}

XM_FN DAln path_align(WS& w, const ACtx& c, const Sec& q, const Sec& r, const Params& p, Analysis& an) {  // PathAligner.align :55-293
  XM_CHECK_MASK(w);
  PhaseClock pc_(&w.st_cyc[3]);
  long long mark = w.scratch_top;
  PathState* sp = (PathState*)w.salloc(sizeof(PathState));
  if (!sp) return aln_null();
  PathState& s = *sp;
  s.prm = p; s.ctx = c; s.an_confident = an.confident; s.an_max_ins = an.max_ins; s.an_max_del = an.max_del;
  s.max_interesting = q.length() * p.max_error_rate;
  s.start_a = q.start; s.end_a = q.end; s.start_b = r.start; s.end_b = r.end;
  s.A = q.length(); s.B = r.length(); s.W = s.A + 2; s.H = s.B + 2;
  s.diagonal = s.start_b - (s.start_a + an.predicted);
  {  // unpack both sections once (lanes split the bases on the device)
    uint8_t* qa = (uint8_t*)w.salloc(s.A + 5); uint8_t* rb = (uint8_t*)w.salloc(s.B + 5);
    if (w.status != 0) { w.scratch_top = mark; return aln_null(); }
    qa += 2; rb += 2;   // two sentinel codes (16) on either side: the search reads one position past both ends (xm_types.h: Params::cls_tab)
    XM_NOUNROLL
    for (int k = 0; k < 2; k++) { qa[-1 - k] = 16; qa[s.A + k] = 16; rb[-1 - k] = 16; rb[s.B + k] = 16; }
    for (int k = lane_id(); k < s.A; k += XM_LANES) qa[k] = c.a.at(s.start_a + k);
    for (int k = lane_id(); k < s.B; k += XM_LANES) rb[k] = c.b.at(s.start_b + k);
    warp_sync();
    s.qa = qa; s.rb = rb;
  }
  w.st_path_calls++; w.st_path_cells += (unsigned long long)s.A * (unsigned long long)s.B;
  {  // chooseSearchReverse :17-53
    int sum_mis = 0, num_mis = 0, sum_mat = 0, num_mat = 0;
    int si = imax(s.start_a, s.start_b - an.predicted), ei = imin(s.end_a, s.end_b - an.predicted);
    int length = ei - si;
    XM_NOUNROLL
    for (int i = lane_id(); i < length; i += XM_LANES) {  // integer sums: any order
      int j = i - s.diagonal;
      if (j >= 0 && j < s.B) {
        if (!bp_can_match(pa_qa(s, i), pa_rb(s, j))) { sum_mis += i; num_mis++; } else { sum_mat += i; num_mat++; }
      }
    }
    warp_sync();   // different trip counts above: converge before the warp-shared search state is written
    sum_mis = warp_sum(sum_mis); num_mis = warp_sum(num_mis);
    sum_mat = warp_sum(sum_mat); num_mat = warp_sum(num_mat);
    s.reverse = (num_mis > 1 && num_mat > 1) ? ((sum_mis / num_mis) > (sum_mat / num_mat) ? 1 : 0) : 1;
  }
  if (s.reverse) { s.step = -1; s.may_extend = (s.start_b == 0); } else { s.step = 1; s.may_extend = (s.end_b == c.b.len); }
  if (s.reverse) { s.start_x = s.W - 1; s.start_y = s.H - 1; s.goal_x = 1; s.goal_y = 1; }
  else { s.start_x = 0; s.start_y = 0; s.goal_x = s.W - 2; s.goal_y = s.H - 2; }
  long long cells = (long long)s.W * (long long)s.H;
  if (s.W > 32000 || s.H > 32000) { w.fail(Q_NEED_MORE); w.scratch_top = mark; return aln_null(); }
  // the lattice: W x H nodes in the arena's dedicated region; a new generation makes every node absent
  const long long map_words = cells * (long long)(sizeof(PNode) / 4);
  if (w.cell_hdr == nullptr || map_words > w.cell_words) { w.fail(Q_NEED_MORE); w.scratch_top = mark; return aln_null(); }
  {
    uint32_t gen = w.cell_hdr[0];
    if (gen == 0 || gen >= 0xFFFFFF) {   // first search in this arena since the launch began, or the 24-bit generation wrapped: clear the region
      const long long n16 = (w.cell_words + 3) >> 2;   // cell_words is a multiple of 4 (ws_init)
      uint4* c4 = (uint4*)w.cellmap;
      XM_NOUNROLL
      for (long long i = (long long)lane_id(); i < n16; i += XM_LANES) c4[i] = make_uint4(0u, 0u, 0u, 0u);
      warp_sync();
      gen = 0;
    }
    gen++;
    if (lane_id() == 0) w.cell_hdr[0] = gen;
    warp_sync();
    s.nodes = (PNode*)w.cellmap; s.gen = gen; s.clock = 0;
  }
  long long remaining = w.scratch_size - w.scratch_top;
  // one spill bucket per distinct live priority: a budget of P has at most ~P / 0.1 of them per rounding variant
  int cap_ovf = (int)(s.max_interesting * 64.0) + 256;
  if ((long long)cap_ovf * (long long)sizeof(PaOverflow) > remaining / 8) cap_ovf = (int)((remaining / 8) / (long long)sizeof(PaOverflow));
  PaOverflow* ovf = (PaOverflow*)w.salloc((long long)cap_ovf * (long long)sizeof(PaOverflow));
  long long ent_cap = (remaining / 2) / (long long)sizeof(PEnt);
  if (ent_cap > 3 * cells + 64) ent_cap = 3 * cells + 64;
  s.ent_cap = (int)ent_cap;
  s.ent = (PEnt*)w.salloc(ent_cap * (long long)sizeof(PEnt));
  if (w.status != 0 || s.ent_cap < 8) { w.fail(Q_NEED_MORE); w.scratch_top = mark; return aln_null(); }
  int last_x = -1, last_y = -1;
  {
    const int rc = pa_search(w, s, ovf, cap_ovf, last_x, last_y);
    if (rc == 1 && w.status == 0) { w.scratch_top = mark; return aln_null(); }
  }
  if (w.status != 0) { w.scratch_top = mark; return aln_null(); }
  // traceback :193-269. Blocks are collected in a temporary array placed after the heap.
  int max_blocks = s.A + s.B + 4;
  Blk* tb = (Blk*)w.salloc((long long)max_blocks * (long long)sizeof(Blk));
  if (!tb) { w.scratch_top = mark; return aln_null(); }
  int nb = 0;
  int i = last_x, j = last_y, idx;
  XM_NOUNROLL
  while (i != s.start_x && j != s.start_y) {
    if (!pa_get(s, i, j, idx)) { w.fail(Q_INTERNAL); break; }
    PNode node = pa_node(s, idx);
    Blk k;
    if (node.pen == node.ins_x) {
      int old_i = i;
      i -= s.step;
      XM_NOUNROLL
      while (i != s.start_x) {
        if (!pa_get(s, i, j, idx)) { w.fail(Q_INTERNAL); break; }
        const PNode o = pa_node(s, idx);
        if (o.pen + p.ins_start + p.ins_ext < o.ins_x + p.ins_ext) break;
        i -= s.step;
      }
      if (s.reverse) { k.a_start = s.start_a + old_i - 1; k.b_start = s.start_b + j - 1; k.a_len = i - old_i; k.b_len = 0; }
      else { k.a_start = s.start_a + i; k.b_start = s.start_b + j; k.a_len = old_i - i; k.b_len = 0; }
    } else if (node.pen == node.ins_y) {
      int old_j = j;
      j -= s.step;
      XM_NOUNROLL
      while (j != s.start_y) {
        if (!pa_get(s, i, j, idx)) { w.fail(Q_INTERNAL); break; }
        const PNode o = pa_node(s, idx);
        if (o.pen + p.del_start + p.del_ext < o.ins_y + p.del_ext) break;
        j -= s.step;
      }
      if (s.reverse) { k.a_start = s.start_a + i - 1; k.b_start = s.start_b + old_j - 1; k.a_len = 0; k.b_len = j - old_j; }
      else { k.a_start = s.start_a + i; k.b_start = s.start_b + j; k.a_len = 0; k.b_len = old_j - j; }
    } else {
      int old_i = i, old_j = j;
      i -= s.step; j -= s.step;
      XM_NOUNROLL
      while (i != s.start_x && j != s.start_y) {
        if (!pa_get(s, i, j, idx)) { w.fail(Q_INTERNAL); break; }
        const PNode o = pa_node(s, idx);
        if (o.pen == o.ins_x || o.pen == o.ins_y) break;
        i -= s.step; j -= s.step;
      }
      if (s.reverse) { k.a_start = s.start_a + old_i - 1; k.b_start = s.start_b + old_j - 1; k.a_len = i - old_i; k.b_len = j - old_j; }
      else { k.a_start = s.start_a + i; k.b_start = s.start_b + j; k.a_len = old_i - i; k.b_len = old_j - j; }
    }
    if (w.status != 0) break;
    if (nb >= max_blocks) { w.fail(Q_INTERNAL); break; }
    tb[nb++] = k;
  }
  if (w.status != 0) { w.scratch_top = mark; return aln_null(); }
  if (!s.reverse) { for (int a = 0, b = nb - 1; a < b; a++, b--) { Blk t = tb[a]; tb[a] = tb[b]; tb[b] = t; } }
  if (nb < 1) { w.scratch_top = mark; return aln_null(); }
  // justify :307-352
  XM_NOUNROLL
  for (int m = 1; m < nb - 1; m++) {
    XM_NOUNROLL
    while (true) {
      Blk left = tb[m - 1], mid = tb[m], right = tb[m + 1];
      if ((mid.a_len > 0) == (mid.b_len > 0)) break;
      if (left.a_len == 0 || left.b_len == 0) break;
      if (right.a_len == 0 || right.b_len == 0) break;
      if (mid.a_len > 0) { if (c.a.at(left.a_start + left.a_len - 1) != c.a.at(mid.a_start + mid.a_len - 1)) break; }
      else { if (c.b.at(left.b_start + left.b_len - 1) != c.b.at(mid.b_start + mid.b_len - 1)) break; }
      left.a_len -= 1; left.b_len -= 1;
      mid.a_start -= 1; mid.b_start -= 1;
      right.a_start -= 1; right.b_start -= 1; right.a_len += 1; right.b_len += 1;
      tb[m - 1] = left; tb[m] = mid; tb[m + 1] = right;
    }
  }
  int first = 0;
  XM_NOUNROLL
  while (true) {
    if (first >= nb) { w.fail(Q_INTERNAL); w.scratch_top = mark; return aln_null(); }  // sections.get(0) on an empty list
    if (!pa_can_remove(tb[first])) break;
    first++;
  }
  int n_out = nb - first;
  double max_int = s.max_interesting;  // PathState is overwritten below
  // keep the result blocks at the bottom of this call's scratch frame
  w.scratch_top = mark;
  Blk* out = (Blk*)w.salloc((long long)n_out * (long long)sizeof(Blk));
  XM_NOUNROLL
  for (int a = 0; a < n_out; a++) out[a] = tb[first + a];  // tb lies above `out` in the same frame: forward copy is safe
  DAln res = new_aln(p, c, out, n_out, c.a_reversed_obj);
  if (res.aligned > max_int) { w.scratch_top = mark; return aln_null(); }
  return res;
}

// ---------------- cascade ----------------
// stage ids follow QueryMatch_Aligner.buildAligner :18-29 from the outside in
enum { ST_STRAIGHT1 = 0, ST_SKIP = 1, ST_HBA1 = 2, ST_BLOCK = 3, ST_STRAIGHT2 = 4, ST_HBA2 = 5, ST_STRAIGHT3 = 6, ST_PATH = 7 };
// The cascade is a template over the stage so that the call graph has no cycle: with a (bounded) recursion in it ptxas
// falls back to a conservative ABI for EVERY function of the kernel (memory descriptors re-materialised with two R2UR
// before each load/store, callee-saved registers spilled at every call).
template <int STAGE>
XM_HD DAln cascade_t(WS& w, const ACtx& c, const Sec& q, const Sec& r, const Params& p, Analysis& an);

XM_HD inline DAln straight_alignment(WS& w, const ACtx& c, const Sec& q, const Sec& r, const Params& p, const Analysis& an) {  // :73-94
  int qs = q.start, qe = q.end, rs = r.start, re = r.end, off = an.predicted;
  if (qs + off > rs) rs = qs + off; else qs = rs - off;
  if (qe + off < re) re = qe + off; else qe = re - off;
  Blk* b = (Blk*)w.salloc(sizeof(Blk));
  if (!b) return aln_null();
  b->a_start = qs; b->b_start = rs; b->a_len = qe - qs; b->b_len = re - rs;
  return new_aln(p, c, b, 1, c.a_reversed_obj);
}
// EASY = the first-pass kernel: it completes a query only when every alignMatch is settled by the outermost
// StraightAligner; the first time the cascade would go deeper the query is handed to the full kernel (Q_HARD).
template <bool EASY, int STAGE>
XM_FN DAln straight_align_t(WS& w, const ACtx& c, const Sec& q, const Sec& r, const Params& p, Analysis& an) {  // StraightAligner.align :13-71
  XM_CHECK_MASK(w);
  an.last_checked = an.predicted;
  w.st_straight++;
  DAln simple;
  { PhaseClock pc_(&w.st_cyc[1]); simple = straight_alignment(w, c, q, r, p, an); }
  if (!simple.valid) return simple;
  double sp = simple.aligned;
  double max_interesting = q.length() * p.max_error_rate;
  double indel = dmin(p.starting_ins_start() + p.ins_ext, p.del_start + p.del_ext);
  if (sp <= 0) return simple;
  if (an.confident) {
    if (sp <= indel || (an.max_ins <= 0 && an.max_del <= 0)) { if (sp <= max_interesting) return simple; return aln_null(); }
    if (indel > max_interesting) return aln_null();
  }
  double rate = simple.aligned / q.length();
  Params sub = p;
  sub.max_error_rate = dmin(rate, p.max_error_rate);
  if constexpr (EASY) { w.hard_hint = (int)(sp * 16.0); w.fail(Q_HARD); return aln_null(); }
  else {
    DAln a = cascade_t<STAGE + 1>(w, c, q, r, sub, an);
    if (w.status != 0) return aln_null();
    if (!a.valid || a.aligned >= sp) { if (sp <= max_interesting) return simple; }
    return a;
  }
}

struct CountMapD {  // M/CountMap.java with a small open list instead of HashMap
  int most_key, most_count, have;
  int* keys; int* vals; int n, cap;
};
XM_HD inline void countmap_put(WS& w, CountMapD& m, int key, int val) {
  XM_NOUNROLL
  for (int i = 0; i < m.n; i++) if (m.keys[i] == key) { m.vals[i] = val; return; }
  if (m.n >= m.cap) { w.fail(Q_NEED_MORE); return; }
  m.keys[m.n] = key; m.vals[m.n] = val; m.n++;
}
XM_FN void countmap_add(WS& w, CountMapD& m, int key, int value) {
  if (key == m.most_key || m.most_count == 0) {
    m.most_count += value; m.most_key = key;
    if (m.have) countmap_put(w, m, m.most_key, m.most_count);
  } else {
    if (!m.have) { m.have = 1; countmap_put(w, m, m.most_key, m.most_count); }
    int count = value;
    XM_NOUNROLL
    for (int i = 0; i < m.n; i++) if (m.keys[i] == key) { count = m.vals[i] + value; break; }
    countmap_put(w, m, key, count);
    if (count > m.most_count) { m.most_key = key; m.most_count = count; }
  }
}

XM_HD inline double min_indel_penalty_for_block_mismatches(int n, const Params& p) {  // HashBlock_Aligner.java:286-310
  n = imax(1, n);
  double per_initial = dmin(p.starting_ins_start() + p.ins_ext, p.del_start + p.del_ext);
  double per_ext = dmin(p.ins_ext, p.del_ext);
  double per_subseq_indel = dmin(p.ins_start + p.ins_ext, p.del_start + p.del_ext);
  double per_subseq = dmin(p.mutation, per_subseq_indel);
  if (n <= 1) return per_initial;
  if (n <= 2) return per_initial + per_ext;
  return per_initial + per_ext + (n - 2) * per_subseq;
}
XM_HD inline double max_ext_long_insertion(int n, double total, const Params& p, int block_len) {  // :322-354
  double avail = total - p.starting_ins_start();
  double only_snps = n * p.mutation;
  double per_block = block_len * p.ins_ext;
  double extra_per_block = per_block - p.mutation;
  if (extra_per_block <= 0) return avail;
  if (n < 2) return avail;
  double short_ext = 2 * p.ins_ext;
  if (short_ext > avail) return avail;
  double short_snps = 2 * p.mutation;
  double past = avail - only_snps;
  double for_blocks = past + short_snps - short_ext;
  double num = for_blocks / extra_per_block;
  double r = (num * block_len + 2) * p.ins_ext;
  r = dmin(r, avail);
  if (r < short_ext) r = 0;
  return r;
}
XM_HD inline double max_ext_many_insertions(int n, double total, const Params& p) {  // :356-376
  double avail = total + (p.ins_start - p.starting_ins_start());
  double only_snps = n * p.mutation;
  double per_short = p.ins_start + 2 * p.ins_ext;
  double extra = per_short - 2 * p.mutation;
  if (extra <= 0) return avail;
  double num = (avail - only_snps) / extra;
  if (num < 1) num = 0;
  double r = num * 2 * p.ins_ext;
  return dmin(r, avail);
}
XM_HD inline double max_ext_many_deletions(int n, double total, const Params& p) {  // :378-400
  double avail = total;
  double only_snps = n * p.mutation;
  double per_short = p.del_start + 2 * p.del_ext;
  double extra = per_short - 2 * p.mutation;
  if (extra <= 0) return avail;
  double num = (avail - only_snps) / extra;
  if (num < 1) num = 0;
  double r = num * 2 * p.del_ext;
  r = dmin(r, avail);
  if (r < 0) r = 0;
  return r;
}

struct PenaltyAnalysisD { double min_possible, max_ins, max_del; int offset_most, num_best; };

XM_FN PenaltyAnalysisD hba_analyze(WS& w, const ACtx& c, const Sec& q, const Sec& r, const Params& p, Analysis& an) {  // analyzePenalty :94-283
  XM_CHECK_MASK(w);
  PenaltyAnalysisD res; res.min_possible = 0; res.max_ins = 0; res.max_del = 0; res.offset_most = 0; res.num_best = 0;
  PhaseClock pc_(&w.st_cyc[2]);
  MatcherD* matcher = an.matcher;
  double max_interesting = p.max_error_rate * q.length();
  int num_mis = 0;
  int max_nonmatch_end = q.start;
  int late_ins = 0, late_del = 0;
  int min_off = r.start - q.start, max_off = r.end - q.end;
  int uncertainty = max_off - min_off;
  if (matcher == nullptr || iabs(matcher->section_len - uncertainty) > uncertainty / 2) {
    matcher = matcher_new(w, c, r, uncertainty);
    if (!matcher) return res;
    if (an.matcher == nullptr) an.matcher = matcher;
  }
  long long mark = w.scratch_top;
  CountMapD counts; counts.most_key = 0; counts.most_count = 0; counts.have = 0; counts.n = 0;
  counts.cap = q.length() + 4;
  counts.keys = (int*)w.salloc((long long)counts.cap * 4); counts.vals = (int*)w.salloc((long long)counts.cap * 4);
  if (w.status != 0) return res;
  int bl = matcher->block_len;
  int max_block_start = q.end - bl;
  XM_NOUNROLL
  for (int bs = q.start; bs <= max_block_start; bs++) {
    if (w.status != 0) return res;
    if (bs >= max_nonmatch_end) {
      int position = matcher_lookup(w, *matcher, c, bs, bs + min_off, bs + max_off + 1);
      int offset = position - bs;
      if (position == M_UNKNOWN || position == M_MULTI) continue;
      if (position == M_NO) {
        num_mis++; max_nonmatch_end = bs + bl;
        if (min_indel_penalty_for_block_mismatches(num_mis, p) > max_interesting) break;
        continue;
      }
      int other = position;
      int reverse_count = imin(bs - max_nonmatch_end, other);
      bool found = false;
      const int lane = lane_id();
      XM_NOUNROLL
      for (int base = 1; base <= reverse_count && !found; base += XM_LANES) {  // any mismatch among the bases left of the block
        const int i = base + lane;
        const bool bad = (i <= reverse_count) && !bp_can_match(c.a.at(bs - i), c.b.at(other - i));
        if (warp_ballot(bad) != 0) found = true;
      }
      warp_sync();
      if (found) { num_mis++; max_nonmatch_end = bs + bl; }
      if (!found) {
        int fwd = q.end - bs;
        XM_NOUNROLL
        for (int base = bl; base < fwd && !found; base += XM_LANES) {  // first mismatch right of the block
          const int i = base + lane, ia = bs + i, ib = other + i;
          bool bad = false;
          if (i < fwd) { uint8_t ca = c.a.at(ia); uint8_t cb = (ib < r.end) ? c.b.at(ib) : (uint8_t)0; bad = !bp_can_match(ca, cb); }
          const unsigned m = warp_ballot(bad);
          if (m != 0) { num_mis++; found = true; max_nonmatch_end = bs + base + (first_bit(m) - 1) + 1; }
        }
        warp_sync();
        if (!found) max_nonmatch_end = q.end;
        int num_other = 0;
        int fwd2 = max_nonmatch_end - bs - bl;
        XM_NOUNROLL
        for (int i = bl; i < fwd2; i++) {
          int ia = bs + i;
          int res2 = matcher_lookup(w, *matcher, c, ia, ia + min_off, ia + max_off + 1);
          if (res2 >= 0 && (res2 - ia) == offset) { num_other++; i = i - 1 + bl; }
        }
        if (offset != counts.most_key && counts.most_count > 0) { if (offset > counts.most_key) late_del += num_other; else late_ins += num_other; }
        countmap_add(w, counts, offset, num_other);
      }
      if (found) { if (min_indel_penalty_for_block_mismatches(num_mis, p) > max_interesting) break; }
      else countmap_add(w, counts, offset, 1);
    }
  }
  int most_off = counts.most_key, most_cnt = counts.most_count;
  w.scratch_top = mark;
  res.min_possible = min_indel_penalty_for_block_mismatches(num_mis, p);
  bool could_differ = most_cnt < 1 || an.last_checked != most_off;
  if (could_differ) { double mp = num_mis * p.mutation; if (res.min_possible > mp) res.min_possible = mp; }
  double long_ins = max_ext_long_insertion(num_mis + late_del, max_interesting, p, bl);
  double many_ins = max_ext_many_insertions(num_mis + late_ins, max_interesting, p);
  res.max_ins = dmax(long_ins, many_ins);
  res.max_del = max_ext_many_deletions(num_mis + late_ins, max_interesting, p);
  if (res.max_ins > an.max_ins) res.max_ins = an.max_ins;
  if (res.max_del > an.max_del) res.max_del = an.max_del;
  if (most_cnt < 1) most_off = an.predicted;
  res.offset_most = most_off; res.num_best = most_cnt;
  return res;
}

template <int STAGE>
XM_FN DAln hba_align(WS& w, const ACtx& c, const Sec& q, const Sec& r_in, const Params& p, Analysis& an_in) {  // HashBlock_Aligner.align :21-81 (tail recursion as a loop)
  XM_CHECK_MASK(w);
  Sec r = r_in;
  Analysis cur = an_in;       // the analysis object of the current recursion level
  Analysis* anp = &an_in;     // first level mutates the caller's object (hashBlock_matcher assignment)
  XM_NOUNROLL
  while (true) {
    double max_interesting = p.max_error_rate * q.length();
    if (q.length() > r.length()) return cascade_t<STAGE + 1>(w, c, q, r, p, *anp);
    PenaltyAnalysisD pa = hba_analyze(w, c, q, r, p, *anp);
    if (w.status != 0) return aln_null();
    if (pa.min_possible > max_interesting) return aln_null();
    Analysis sub = *anp;  // child()
    sub.max_ins = pa.max_ins; sub.max_del = pa.max_del;
    double extra = pa.num_best * p.mutation + pa.min_possible;
    if (extra > max_interesting) { sub.predicted = pa.offset_most; sub.confident = 1; }
    else { if (!anp->confident) sub.predicted = pa.offset_most; }
    if (anp->confident && sub.predicted == anp->predicted) sub.confident = 1;
    Sec rsub = r;
    if (sub.confident) {
      int max_del_len = j2i((double)pa.max_del / (double)p.del_ext);
      int max_ins_len = j2i((double)pa.max_ins / (double)p.ins_ext);
      int max_indel = imax(max_del_len, max_ins_len);
      rsub.start = imax(r.start, wadd(wadd(q.start, sub.predicted), -max_indel));
      rsub.end = imin(r.end, wadd(wadd(q.end, sub.predicted), max_indel));
    }
    if (rsub.length() < r.length()) { cur = sub; anp = &cur; r = rsub; continue; }
    return cascade_t<STAGE + 1>(w, c, q, rsub, p, sub);
  }
}

XM_FN DAln block_align_piece(WS& w, const ACtx& c, const Sec& q, const Sec& r, double max_penalty, const Params& p, bool first_piece, const Analysis& parent) {  // alignPiece :215-249
  if (max_penalty < 0) return aln_null();
  Sec rsub = r;
  if (parent.confident) {
    int max_ins_len = j2i((double)parent.max_ins / (double)p.ins_ext);
    int max_del_len = j2i((double)parent.max_del / (double)p.del_ext);
    int max_indel = imax(max_ins_len, max_del_len);
    int rs = imax(r.start, wadd(wadd(q.start, parent.predicted), -max_indel));
    int re = imin(r.end, wadd(wadd(q.end, parent.predicted), max_indel));
    if (re > rs) { rsub.start = rs; rsub.end = re; }
  }
  Params sub = p;
  if (!first_piece) sub.start_free = 1;
  sub.max_error_rate = max_penalty / q.length();
  Analysis child = parent;
  child.confident = 0;
  return cascade_t<ST_BLOCK + 1>(w, c, q, rsub, sub, child);
}
XM_FN DAln block_try_merge(WS& w, const ACtx& c, const DAln& left, const DAln& right, const Params& p) {  // doTryMerge :158-212
  if (aln_end_b(left) != aln_start_b(right)) return aln_null();
  const Blk& l = left.b[left.n - 1];
  const Blk& rr = right.b[0];
  if (!(((l.a_len > 0) == (rr.a_len > 0)) && ((l.b_len > 0) == (rr.b_len > 0)))) return aln_null();
  if (l.a_start + l.a_len != rr.a_start) return aln_null();
  if (l.b_start + l.b_len != rr.b_start) return aln_null();
  int n = left.n + right.n - 1;
  Blk* b = (Blk*)w.salloc((long long)n * (long long)sizeof(Blk));
  if (!b) return aln_null();
  int k = 0;
  XM_NOUNROLL
  for (int i = 0; i < left.n - 1; i++) b[k++] = left.b[i];
  Blk mid; mid.a_start = l.a_start; mid.b_start = l.b_start; mid.a_len = l.a_len + rr.a_len; mid.b_len = l.b_len + rr.b_len;
  b[k++] = mid;
  XM_NOUNROLL
  for (int i = 1; i < right.n; i++) b[k++] = right.b[i];
  return new_aln(p, c, b, n, left.ref_reversed);
}
XM_FN DAln block_align(WS& w, const ACtx& c, const Sec& q, const Sec& r, const Params& p, Analysis& an) {  // BlockAligner.align :17-36
  XM_CHECK_MASK(w);
  double max_interesting = p.max_error_rate * q.length();
  // initialAlignments :39-96
  double max_initial = p.max_error_rate * c.a.len;
  int nbe = j2i(log((double)r.length() / log(4.0))) + 1;  // sic :48
  int num_hashblocks = q.length() / nbe + 1;
  int target_per_block = j2i(sqrt((double)num_hashblocks)) + 1;
  int target_block_size = target_per_block * nbe;
  int num_blocks = q.length() / target_block_size;
  if (num_blocks < 1) return aln_null();
  DAln* cur = (DAln*)w.salloc((long long)num_blocks * (long long)sizeof(DAln));
  DAln* nxt = (DAln*)w.salloc((long long)num_blocks * (long long)sizeof(DAln));
  if (w.status != 0) return aln_null();
  XM_NOUNROLL
  for (int i = 0; i < num_blocks; i++) cur[i] = aln_null();
  double used = 0;
  int remaining = num_blocks;
  XM_NOUNROLL
  while (true) {
    bool failed = false, failed_then_found = false;
    int start_pos = q.start;
    XM_NOUNROLL
    for (int i = 0; i < num_blocks; i++) {
      int end_pos = q.start + (int)((long long)q.length() * (i + 1) / num_blocks);
      if (!cur[i].valid) {
        Sec qs; qs.start = start_pos; qs.end = end_pos;
        double avg = (max_initial - used) / remaining;
        DAln sub = block_align_piece(w, c, qs, r, avg, p, i == 0, an);
        if (w.status != 0) return aln_null();
        if (sub.valid) { if (failed) failed_then_found = true; remaining--; cur[i] = sub; used += sub.aligned; }
        else failed = true;
      }
      start_pos = end_pos;
    }
    if (remaining < 1) break;
    if (!failed_then_found) return aln_null();
  }
  int n = num_blocks;
  bool even = false;
  XM_NOUNROLL
  while (n > 1) {  // joinAlignments :99-144
    double used_pen = 0;
    XM_NOUNROLL
    for (int i = 0; i < n; i++) used_pen += cur[i].aligned;
    int m = 0;
    XM_NOUNROLL
    for (int i = 0; i < n; i += 2) {
      DAln merge;
      DAln left = cur[i];
      if (i + 1 < n) {
        DAln right = cur[i + 1];
        merge = block_try_merge(w, c, left, right, p);
        if (w.status != 0) return aln_null();
        if (!merge.valid) {
          used_pen -= left.aligned; used_pen -= right.aligned;
          Sec qs; qs.start = aln_start_a(left); qs.end = aln_end_a(right);
          merge = block_align_piece(w, c, qs, r, max_interesting - used_pen, p, i == 0, an);
          if (w.status != 0) return aln_null();
          if (!merge.valid) return aln_null();
          used_pen += merge.aligned;
        } else if (!even) { nxt[m++] = left; i--; continue; }
      } else merge = left;
      nxt[m++] = merge;
    }
    DAln* t = cur; cur = nxt; nxt = t;
    n = m;
    even = !even;
  }
  return cur[0];
}

template <int STAGE>
XM_HD inline DAln cascade_t(WS& w, const ACtx& c, const Sec& q, const Sec& r, const Params& p, Analysis& an) {
  if (w.status != 0) return aln_null();
  if constexpr (STAGE == ST_STRAIGHT1 || STAGE == ST_STRAIGHT2 || STAGE == ST_STRAIGHT3) return straight_align_t<false, STAGE>(w, c, q, r, p, an);
  else if constexpr (STAGE == ST_SKIP) {  // SkipHighAmbiguity_Aligner.align :13-28
    int amb = 0;
    XM_NOUNROLL
    for (int base = r.start; base < r.end; base += XM_LANES) {
      const int i = base + lane_id();
      amb += bit_count(warp_ballot(i < r.end && bp_is_ambiguous(c.b.at(i))));
    }
    warp_sync();
    if (amb >= r.length() / 4) return aln_null();
    return cascade_t<STAGE + 1>(w, c, q, r, p, an);
  }
  else if constexpr (STAGE == ST_HBA1 || STAGE == ST_HBA2) return hba_align<STAGE>(w, c, q, r, p, an);
  else if constexpr (STAGE == ST_BLOCK) return block_align(w, c, q, r, p, an);
  else return path_align(w, c, q, r, p, an);
}


// ---- reference windows through TMA (cp.async.bulk) into shared memory ----
// Layout of a warp's staging area (XM_STAGE_BYTES): [0,8) mbarrier; [16, 16 + XM_STAGE_PACKED) the packed window as the bulk copy
// delivers it (16-byte aligned source, whole 16-byte units); then XM_STAGE_WINDOW bytes: the window, one code per byte.
static const int XM_STAGE_PACKED = 176, XM_STAGE_WINDOW = 320, XM_STAGE_BYTES = 16 + XM_STAGE_PACKED + XM_STAGE_WINDOW;
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ void stage_init(unsigned char* stage) {   // lane 0, once per warp
  const unsigned int mbar = (unsigned int)__cvta_generic_to_shared(stage);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(mbar) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// Fetches bases [start, end) of the forward strand `ref` into the staging area and unpacks them; returns the byte window or nullptr
// when the window does not fit (the caller then unpacks from global memory).  One elected lane issues the bulk copy; the warp waits on
// the mbarrier (phase bit in WS) and the 32 lanes unpack from shared memory.
__device__ __noinline__ const uint8_t* stage_window(WS& w, const SeqView& ref, int start, int end) {
  const int wn = end - start;
  if (w.stage == nullptr || ref.rc || wn < 1 || wn > XM_STAGE_WINDOW) return nullptr;
  const char* first = (const char*)ref.w + ((start >> 2) << 1);                 // the 16-bit word that holds base `start`
  const char* src = (const char*)((unsigned long long)first & ~15ull);
  const int lead = (int)(first - src);
  const int bytes = (lead + (((end + 3) >> 2) << 1) - ((start >> 2) << 1) + 15) & ~15;
  if (bytes > XM_STAGE_PACKED) return nullptr;
  const int lane = (int)(threadIdx.x & 31);
  unsigned char* packed = w.stage + 16;
  uint8_t* out = w.stage + 16 + XM_STAGE_PACKED;
  const unsigned int mbar = (unsigned int)__cvta_generic_to_shared(w.stage);
  const unsigned int phase = w.stage_phase;
  __syncwarp();
  if (lane == 0) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");              // earlier generic-proxy reads of the area are done
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"((unsigned int)__cvta_generic_to_shared(packed)), "l"(src), "r"(bytes), "r"(mbar) : "memory");
  }
  unsigned int done = 0;
  while (!done) {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.b32 %0, 1, 0, p; }" : "=r"(done) : "r"(mbar), "r"(phase) : "memory");
  }
  const unsigned short* words = (const unsigned short*)(packed + lead);
  const int w0 = start >> 2;
  for (int k = lane; k < wn; k += 32) { const int b = start + k; out[k] = (uint8_t)((words[(b >> 2) - w0] >> ((b & 3) << 2)) & 15); }
  __syncwarp();
  if (lane == 0) w.stage_phase = phase ^ 1u;
  __syncwarp();
  return out;
}
#endif

// ---------------- QueryMatch_Aligner ----------------
struct SAStore { int contig, ref_reversed, a_mate, a_rev, n_blk, pad; double penalty, aligned; Blk* blk; };
struct QAStore { double spacing, multiplier, bonus, total; int inner, n_sa; SAStore sa[2]; };
struct QMX { SM comp[2]; int n, priority, hint; };  // QueryMatch with explicit components
struct QMA {  // QueryMatch_Aligner instance
  Params prm; double best_penalty; int q_len;
  QAStore** good; int n_good, cap_good;
};

XM_INLINE void* store_alloc(WS& w, long long bytes) {
  bytes = (bytes + 7) & ~7LL;
  if (w.store_top + bytes > w.store_size) { w.fail(Q_NEED_MORE); return nullptr; }
  void* p = w.store + w.store_top; w.store_top += bytes; return p;
}
XM_HD inline void qma_init(WS& w, QMA& a, const Params& p, int q_len, int cap) {
  a.prm = p; a.best_penalty = (double)JMAX; a.q_len = q_len; a.n_good = 0; a.cap_good = cap;
  a.good = (QAStore**)store_alloc(w, (long long)cap * (long long)sizeof(QAStore*));
}
XM_INLINE int sa_start_b(const SAStore& s) { return s.blk[0].b_start; }
XM_INLINE int sa_end_b(const SAStore& s) { return s.blk[s.n_blk - 1].b_start + s.blk[s.n_blk - 1].b_len; }
XM_INLINE int sa_start_a(const SAStore& s) { return s.blk[0].a_start; }
XM_INLINE int sa_end_a(const SAStore& s) { return s.blk[s.n_blk - 1].a_start + s.blk[s.n_blk - 1].a_len; }

// QueryMatch_Aligner.alignMatch(SequenceMatch, parameters) :412-462. c describes a and b.
template <bool EASY>
XM_FN DAln qma_align_match(WS& w, const ACtx& c, const SM& sm, const Params& p, double per_penalty) {
  XM_CHECK_MASK(w);
  int a_len = c.a.len, b_len = c.b.len;
  int sb = imax(0, sm.offset), eb = imin(sm.offset + a_len, b_len);
  Sec q; q.start = sb - sm.offset; q.end = eb - sm.offset;
  double max_interesting = q.length() * p.max_error_rate;
  int max_indel = j2i(dmax((double)0, (double)(max_interesting - p.del_start) / p.del_ext));
  int max_shift, best_offset = sm.offset;
  if (sm.from_hash) max_shift = max_indel;
  else {
    max_shift = j2i((double)max_interesting * per_penalty);
    if (max_shift < 0) return aln_null();
    if (best_offset + a_len > b_len) best_offset = b_len - a_len;
    if (best_offset < 0) best_offset = 0;
    q.start = 0; q.end = a_len;
  }
  Sec r; r.start = imax(0, sb - max_shift); r.end = imin(eb + max_shift, b_len);
  Analysis an; an.matcher = nullptr; an.last_checked = 0;
  an.max_ins = max_interesting - p.ins_start; an.max_del = max_interesting - p.del_start;
  an.predicted = best_offset; an.confident = sm.from_hash ? 1 : 0;
  if (EASY) return straight_align_t<true, ST_STRAIGHT1>(w, c, q, r, p, an);
  {  // every stage of the cascade reads the reference through this window: fetch it once - by TMA into shared memory when it fits the
     // warp's staging area, else unpacked from global memory into the arena (lanes split the bases)
    const int wn = r.end - r.start;
#if defined(__CUDA_ARCH__)
    const uint8_t* sw = stage_window(w, c.b, r.start, r.end);
    if (sw != nullptr) {
      ACtx cw = c;
      cw.b.bytes = sw; cw.b.b0 = r.start; cw.b.bn = wn;
      return cascade_t<ST_STRAIGHT1>(w, cw, q, r, p, an);
    }
#endif
    if (wn > 0 && w.scratch_top + wn + 64 <= w.scratch_size) {
      uint8_t* wb = (uint8_t*)w.salloc(wn);
      XM_NOUNROLL
      for (int k = lane_id(); k < wn; k += XM_LANES) wb[k] = c.b.at(r.start + k);
      warp_sync();
      ACtx cw = c;
      cw.b.bytes = wb; cw.b.b0 = r.start; cw.b.bn = wn;
      return cascade_t<ST_STRAIGHT1>(w, cw, q, r, p, an);
    }
  }
  return cascade_t<ST_STRAIGHT1>(w, c, q, r, p, an);
}
XM_HD inline bool sa_store_from(WS& w, SAStore& out, const DAln& a, int contig, int a_mate, int a_rev) {
  out.contig = contig; out.ref_reversed = a.ref_reversed; out.a_mate = a_mate; out.a_rev = a_rev; out.n_blk = a.n; out.pad = 0;
  out.penalty = a.penalty; out.aligned = a.aligned;
  out.blk = (Blk*)store_alloc(w, (long long)a.n * (long long)sizeof(Blk));
  if (!out.blk) return false;
  XM_NOUNROLL
  for (int i = 0; i < a.n; i++) out.blk[i] = a.b[i];
  return true;
}
XM_HD inline int sa_len_a_before(const SAStore& s, int index_b) {  // SequenceAlignment.getLengthABefore :98-117
  int total = 0;
  XM_NOUNROLL
  for (int i = 0; i < s.n_blk; i++) {
    const Blk& b = s.blk[i];
    if (index_b <= b.b_start) break;
    if (b.a_len < 1) continue;
    if (b.a_len > b.b_len) total += b.a_len;
    else if (index_b < b.b_start + b.b_len) total += index_b - b.b_start;
    else total += b.a_len;
  }
  return total;
}
XM_HD inline int sa_len_a_after(const SAStore& s, int index_b) {  // :119-139
  int total = 0;
  XM_NOUNROLL
  for (int i = 0; i < s.n_blk; i++) {
    const Blk& b = s.blk[i];
    if (index_b >= b.b_start + b.b_len) continue;
    if (b.a_len < 1) continue;
    if (b.a_len > b.b_len) total += b.a_len;
    else if (index_b > b.b_start) total += b.b_start + b.b_len - index_b;
    else total += b.a_len;
  }
  return total;
}
XM_HD inline int sa_insert_a_or_b(const SAStore& s) { int t = 0; for (int i = 0; i < s.n_blk; i++) if (s.blk[i].a_len != s.blk[i].b_len) t += s.blk[i].a_len + s.blk[i].b_len; return t; }
XM_FN double sa_penalty_range(WS& w, const Params& p, const SAStore& s, int start_b, int end_b) {  // getPenalty(alignment, startB, endB) :97-103
  SeqView a = w.query_view(s.a_mate, s.a_rev);
  SeqView b = w.ref->contig(s.contig, 0);
  double t = 0;
  XM_NOUNROLL
  for (int i = 0; i < s.n_blk; i++) t += block_penalty_range(p, a, b, s.blk[i], start_b, end_b);
  return t;
}
// extract :365-405 — cuts [query_start, query_end) of the joined alignment for the read (mate, rev)
XM_FN bool qma_extract(WS& w, const Params& p, const DAln& joined, int query_start, int query_end, int mate, int rev, int contig, bool reverse, SAStore& out) {
  int ref_reversed = (joined.ref_reversed != 0) != reverse ? 1 : 0;
  long long mark = w.scratch_top;
  Blk* blocks = (Blk*)w.salloc((long long)joined.n * (long long)sizeof(Blk));
  if (!blocks) return false;
  int n = 0;
  XM_NOUNROLL
  for (int i = 0; i < joined.n; i++) {
    const Blk& b = joined.b[i];
    if (b.a_start >= query_end) break;
    if (b.a_start + b.a_len <= query_start) continue;
    int sel_s = imax(b.a_start, query_start), sel_e = imin(b.a_start + b.a_len, query_end);
    int ql = sel_e - sel_s, rl, rs;
    if (b.a_len == b.b_len) { rl = ql; rs = sel_s + (b.b_start - b.a_start); }
    else if (b.a_len > b.b_len) { rl = 0; rs = b.b_start; }
    else { rl = b.b_len; rs = sel_s + (b.b_start - b.a_start); }
    Blk k; k.a_start = sel_s - query_start; k.b_start = rs; k.a_len = ql; k.b_len = rl;
    blocks[n++] = k;
  }
  if (n < 1) { w.scratch_top = mark; return false; }
  ACtx c; c.a = w.query_view(mate, rev); c.a_reversed_obj = rev; c.b = w.ref->contig(contig, 0);
  DAln a = new_aln(p, c, blocks, n, ref_reversed);
  bool ok = sa_store_from(w, out, a, contig, mate, rev);
  w.scratch_top = mark;
  return ok;
}

XM_HD inline int qmx_distance(const WS& w, const QMX& m, const SM& a, const SM& b) {  // QueryMatch.getDistance :124-133
  if (a.contig != b.contig) return JMAX;
  if (m.comp[0].rev) return sm_start_b(w, a) - sm_end_b(w, b);
  return sm_start_b(w, b) - sm_end_b(w, a);
}

// doAlign :94-272; returns stored alignment or nullptr
template <bool EASY>
XM_FN QAStore* qma_do_align(WS& w, QMA& A, const QMX& match, double extra_spacing, int q_total_len_for_spacing) {
  XM_CHECK_MASK(w);
  const Params& P = A.prm;
  int spacing_i = 0;
  if (match.n >= 2) spacing_i = qmx_distance(w, match, match.comp[0], match.comp[1]);
  double inner = spacing_i + extra_spacing;
  // computeSpacingPenalty :530-546 (query = the aligner's query)
  double spacing_penalty;
  {
    double expected = w.query.expected_inner;
    int total_len = q_total_len_for_spacing;
    if (inner < 0 && inner > -1 * total_len) spacing_penalty = 0;
    else spacing_penalty = (double)j2i(fabs(inner - expected) / w.query.per_penalty);
  }
  double multiplier = 1, bonus = 0;
  int match_total_len = 0;
  XM_NOUNROLL
  for (int i = 0; i < match.n; i++) match_total_len += w.query.seq[match.comp[i].mate].len;
  double max_allowed = next_up(match_total_len * P.max_error_rate);
  if (inner > 0) { double mp = spacing_penalty + match.priority * P.mutation; if (mp > max_allowed) return nullptr; }
  long long mark = w.scratch_top;
  long long store_mark = w.store_top;
  QAStore* qa = (QAStore*)store_alloc(w, sizeof(QAStore));
  if (!qa) return nullptr;
  qa->n_sa = match.n;
  bool have = false;
  double comps_penalty = 0;
  if (match.n > 1 && inner < 0) {
    // tryJoinQuerySequences :274-319
    const SM& m1 = match.comp[0]; const SM& m2 = match.comp[1];
    int off = m2.offset - m1.offset;
    const SM& s1m = (off >= 0) ? m1 : m2; const SM& s2m = (off >= 0) ? m2 : m1;
    int offset = off >= 0 ? off : -off;
    SeqView s1 = w.query_view(s1m.mate, s1m.rev), s2 = w.query_view(s2m.mate, s2m.rev);
    int suffix_start = s1.len - offset;
    bool joinable = suffix_start >= 0;
    if (joinable) {
      int end2 = imin(s2.len, s1.len - offset);
      XM_NOUNROLL
      for (int i2 = 0; i2 < end2; i2++) if (s1.at(i2 + offset) != s2.at(i2)) { joinable = false; break; }
    }
    if (joinable) {
      if (suffix_start > s2.len) { w.fail(Q_INTERNAL); return nullptr; }  // getRange throws in the reference
      int jl = s1.len + (s2.len - suffix_start);
      uint16_t* jw = (uint16_t*)w.salloc((long long)((jl + 3) / 4 + 1) * 2);
      if (!jw) return nullptr;
      XM_NOUNROLL
      for (int i = 0; i < (jl + 3) / 4 + 1; i++) jw[i] = 0;
      XM_NOUNROLL
      for (int i = 0; i < jl; i++) {
        uint8_t code = i < s1.len ? s1.at(i) : s2.at(suffix_start + (i - s1.len));
        jw[i >> 2] = (uint16_t)(jw[i >> 2] | ((uint16_t)code << ((i & 3) << 2)));
      }
      // computeJoinedAlignment :321-331
      ACtx jc; jc.a.w = jw; jc.a.len = jl; jc.a.rc = 0; jc.a.bytes = nullptr; jc.a_reversed_obj = 0; jc.b = w.ref->contig(m1.contig, 0);
      SM jm; jm.mate = -1; jm.rev = 0; jm.contig = m1.contig; jm.offset = imin(m1.offset, m2.offset); jm.from_hash = 1;
      Params sub = P; sub.max_error_rate = next_up(sub.max_error_rate);
      DAln ja = qma_align_match<EASY>(w, jc, jm, sub, w.query.per_penalty);
      if (w.status != 0) return nullptr;
      // splitAlignment :332-363
      if (!ja.valid) { w.scratch_top = mark; w.store_top = store_mark; return nullptr; }
      int l1 = w.query.seq[m1.mate].len, l2 = w.query.seq[m2.mate].len;
      bool ok1, ok2;
      if (off >= 0) {
        ok1 = qma_extract(w, P, ja, 0, l1, m1.mate, m1.rev, m1.contig, m1.rev != 0, qa->sa[0]);
        ok2 = qma_extract(w, P, ja, off, l2 + off, m2.mate, m2.rev, m2.contig, m2.rev != 0, qa->sa[1]);
      } else {
        ok2 = qma_extract(w, P, ja, 0, l2, m2.mate, m2.rev, m2.contig, m2.rev != 0, qa->sa[1]);
        ok1 = qma_extract(w, P, ja, -off, l1 - off, m1.mate, m1.rev, m1.contig, m1.rev != 0, qa->sa[0]);
      }
      if (w.status != 0) return nullptr;
      if (!ok1 || !ok2) { w.scratch_top = mark; w.store_top = store_mark; return nullptr; }
      have = true;
      comps_penalty += qa->sa[0].penalty; comps_penalty += qa->sa[1].penalty;
    }
  }
  if (!have) {
    bool remaining[2] = {true, true};
    int num_remaining = match.n;
    int first, stepi, last;
    if (match.hint) { first = 0; stepi = 1; last = match.n; } else { first = match.n - 1; stepi = -1; last = -1; }
    double max_total;
    if (inner < 0 && match.n > 1) {
      double qtl = match_total_len;
      double est_overlap = dmin(-1 * inner, (double)imin(w.query.seq[match.comp[0].mate].len, w.query.seq[match.comp[1].mate].len));
      double est_unique = qtl - est_overlap;
      max_total = divide_round_up(max_allowed - spacing_penalty, qtl) * est_unique * 2;
    } else max_total = max_allowed - spacing_penalty;
    XM_NOUNROLL
    while (true) {
      int num_bases = 0;
      XM_NOUNROLL
      for (int i = 0; i < match.n; i++) if (remaining[i]) num_bases += w.query.seq[match.comp[i].mate].len;
      if (num_bases < 1) break;
      double avg = divide_round_up(max_total - comps_penalty, (double)num_bases);
      Params prem = P; prem.max_error_rate = avg;
      bool found = false;
      XM_NOUNROLL
      for (int i = first; i != last; i += stepi) {
        if (remaining[i]) {
          const SM& sm = match.comp[i];
          ACtx c; c.a = w.query_view(sm.mate, sm.rev); c.a_reversed_obj = sm.rev; c.b = w.ref->contig(sm.contig, 0);
          long long m2 = w.scratch_top;
          DAln sa = qma_align_match<EASY>(w, c, sm, prem, w.query.per_penalty);
          if (w.status != 0) return nullptr;
          if (sa.valid) {
            if (!sa_store_from(w, qa->sa[i], sa, sm.contig, sm.mate, sm.rev)) return nullptr;
            w.scratch_top = m2;
            found = true; remaining[i] = false; comps_penalty += sa.penalty; num_remaining--;
            break;
          }
          w.scratch_top = m2;
        }
      }
      if (num_remaining < 1) break;
      if (!found) { w.scratch_top = mark; w.store_top = store_mark; return nullptr; }
    }
  }
  w.scratch_top = mark;
  double total_used = comps_penalty;
  if (inner < 0) {
    // computeDuplicationBonus :506-520
    if (match.n >= 2) {
      const SAStore& a = qa->sa[0]; const SAStore& b = qa->sa[1];
      double ov = imin(sa_end_b(a), sa_end_b(b)) - imax(sa_start_b(a), sa_start_b(b));
      if (ov < 0) bonus = 0;
      else bonus = (sa_penalty_range(w, P, a, sa_start_b(b), sa_end_b(b)) + sa_penalty_range(w, P, b, sa_start_b(a), sa_end_b(a))) / 2;
    }
    total_used -= bonus;
    // multiplyPenaltyForOverlap :464-504
    double multiplied = total_used;
    if (match.n >= 2) {
      const SAStore& f = qa->sa[0]; const SAStore& s = qa->sa[1];
      double ovb = imin(sa_end_b(f), sa_end_b(s)) - imax(sa_start_b(f), sa_start_b(s));
      if (ovb > 0) {
        int unique_a;
        int f_len_a = sa_end_a(f) - sa_start_a(f), s_len_a = sa_end_a(s) - sa_start_a(s);
        if (sa_start_b(f) <= sa_start_b(s)) unique_a = sa_len_a_before(f, sa_start_b(s)) + s_len_a + sa_len_a_after(f, sa_end_b(s));
        else unique_a = sa_len_a_before(s, sa_start_b(f)) + f_len_a + sa_len_a_after(s, sa_end_b(f));
        double deletion = imin(sa_insert_a_or_b(f), sa_insert_a_or_b(s));
        unique_a = j2i((double)unique_a - deletion);
        if (unique_a > 0) { int total_a = f_len_a + s_len_a; multiplied = divide_round_up(total_used, (double)unique_a) * total_a; }
      }
    }
    if (total_used != 0) multiplier = multiplied / total_used; else multiplier = 1;
    total_used = multiplied;
  }
  total_used += spacing_penalty;
  if (total_used > max_allowed) { w.store_top = store_mark; return nullptr; }
  qa->spacing = spacing_penalty; qa->multiplier = multiplier; qa->bonus = bonus; qa->total = total_used;
  qa->inner = match.n > 1 ? sa_start_b(qa->sa[1]) - sa_end_b(qa->sa[0]) : 0;
  return qa;
}
template <bool EASY>
XM_FN QAStore* qma_align(WS& w, QMA& A, const QMX& match, double extra_spacing, int q_total_len) {  // align :39-54
  QAStore* a = qma_do_align<EASY>(w, A, match, extra_spacing, q_total_len);
  if (a != nullptr) {
    if (a->total < A.best_penalty) {
      A.best_penalty = a->total;
      double nt = a->total + A.prm.span;
      double nr = divide_round_up(nt, (double)A.q_len);
      if (nr < A.prm.max_error_rate) A.prm.max_error_rate = nr;
    }
    if (A.n_good >= A.cap_good) { w.fail(Q_NEED_MORE); return nullptr; }
    A.good[A.n_good++] = a;
  }
  return a;
}
XM_INLINE int32_t qa_hash(const QAStore& q) {  // QueryAlignment.hashCode :226-233
  int32_t h = 0;
  XM_NOUNROLL
  for (int i = 0; i < q.n_sa; i++) h = wadd(wmul(h, 1001), q.sa[i].blk[0].b_start - q.sa[i].blk[0].a_start);
  return h;
}
XM_HD inline bool qa_equals(const QAStore& a, const QAStore& b) {  // QueryAlignment.equals :235-256 + SequenceAlignment.equals + AlignedBlock.equals
  if (a.spacing != b.spacing || a.multiplier != b.multiplier || a.bonus != b.bonus || a.total != b.total) return false;
  if (a.inner != b.inner || a.n_sa != b.n_sa) return false;
  XM_NOUNROLL
  for (int i = 0; i < a.n_sa; i++) {
    const SAStore& x = a.sa[i]; const SAStore& y = b.sa[i];
    if (x.n_blk != y.n_blk || x.ref_reversed != y.ref_reversed) return false;
    if (x.contig != y.contig || x.a_mate != y.a_mate || x.a_rev != y.a_rev) return false;
    XM_NOUNROLL
    for (int k = 0; k < x.n_blk; k++) {
      const Blk& p = x.blk[k]; const Blk& q = y.blk[k];
      if (p.a_start != q.a_start || p.b_start != q.b_start || p.a_len != q.a_len || p.b_len != q.b_len) return false;
    }
  }
  return true;
}
// getBestAlignments :71-83 + withoutDuplicates :86-92 (java.util.HashSet iteration order). Writes indices into out (scratch), returns count.
XM_FN int qma_best(WS& w, QMA& A, QAStore**& out) {
  XM_CHECK_MASK(w);
  double max_anywhere = A.q_len * A.prm.max_error_rate;
  double cutoff = A.best_penalty + A.prm.span;
  if (cutoff > max_anywhere) cutoff = max_anywhere;
  int nb = 0;
  QAStore** best = (QAStore**)w.salloc((long long)(A.n_good > 0 ? A.n_good : 1) * (long long)sizeof(QAStore*));
  out = best;
  if (!best) return 0;
  XM_NOUNROLL
  for (int i = 0; i < A.n_good; i++) if (A.good[i]->total <= cutoff) best[nb++] = A.good[i];
  if (nb <= 1) return nb;
  int cap = imax((int)((float)nb / .75f) + 1, 16);
  int n = 1; while (n < cap) n <<= 1;
  // bucket index per element, then stable order by bucket with duplicates removed
  int* bucket = (int*)w.salloc((long long)nb * 4);
  uint8_t* drop = (uint8_t*)w.salloc(nb);
  QAStore** sorted = (QAStore**)w.salloc((long long)nb * (long long)sizeof(QAStore*));
  if (w.status != 0) return 0;
  XM_NOUNROLL
  for (int i = 0; i < nb; i++) {
    uint32_t h = (uint32_t)qa_hash(*best[i]); h ^= (h >> 16);
    bucket[i] = (int)(h & (uint32_t)(n - 1));
    drop[i] = 0;
    XM_NOUNROLL
    for (int j = 0; j < i; j++) if (!drop[j] && bucket[j] == bucket[i] && qa_hash(*best[j]) == qa_hash(*best[i]) && qa_equals(*best[j], *best[i])) { drop[i] = 1; break; }
  }
  int m = 0;
  // emit in ascending bucket order, insertion order within a bucket
  int prev_bucket = -1;
  XM_NOUNROLL
  while (true) {
    int nbk = -1;
    XM_NOUNROLL
    for (int i = 0; i < nb; i++) if (!drop[i] && bucket[i] > prev_bucket && (nbk < 0 || bucket[i] < nbk)) nbk = bucket[i];
    if (nbk < 0) break;
    XM_NOUNROLL
    for (int i = 0; i < nb; i++) if (!drop[i] && bucket[i] == nbk) sorted[m++] = best[i];
    prev_bucket = nbk;
  }
  out = sorted;
  return m;
}

// ---------------- AlignerWorker ----------------
XM_HD inline double penalty_lower_bound(const WS& w, int k) {  // getPenaltyLowerBound :487-491
  double mp = k * w.prm.mutation;
  double ip = w.ix->min_interesting * k * w.prm.del_ext;
  return dmin(mp, ip);
}
XM_HD inline bool dup_may_contain(const WS& w, int contig, int start_index, int end_index) {  // Readable_DuplicationDetector.mayContainDuplicationInRange :28-47
  const DupD& d = *w.dup;
  int ws = start_index / d.window, we = end_index / d.window;
  long long lo = d.off[contig], hi = d.off[contig + 1];
  if (lo == hi) return false;
  // floorEntry(endIndex)
  long long a = lo, b = hi;  // first index with starts > end_index
  XM_NOUNROLL
  while (a < b) { long long mid = (a + b) >> 1; if (d.starts[mid] > end_index) b = mid; else a = mid + 1; }
  if (a > lo) { int wnd = d.starts[a - 1] / d.window; if (wnd >= ws && wnd <= we) return true; }
  // ceilingEntry(startIndex)
  a = lo; b = hi;  // first index with starts >= start_index
  XM_NOUNROLL
  while (a < b) { long long mid = (a + b) >> 1; if (d.starts[mid] >= start_index) b = mid; else a = mid + 1; }
  if (a < hi) { int wnd = d.starts[a] / d.window; if (wnd >= ws && wnd <= we) return true; }
  return false;
}
XM_HD inline bool qa_has_indel(const QAStore& q) { for (int i = 0; i < q.n_sa; i++) if (q.sa[i].n_blk > 1) return true; return false; }
XM_HD inline bool qa_has_ambiguous(const WS& w, const QAStore& q) {
  XM_NOUNROLL
  for (int i = 0; i < q.n_sa; i++) {
    const SAStore& s = q.sa[i];
    SeqView a = w.query_view(s.a_mate, s.a_rev), b = w.ref->contig(s.contig, 0);
    XM_NOUNROLL
    for (int k = 0; k < s.n_blk; k++) {
      XM_NOUNROLL
      for (int t = 0; t < s.blk[k].a_len; t++) if (bp_is_ambiguous(a.at(s.blk[k].a_start + t))) return true;
      XM_NOUNROLL
      for (int t = 0; t < s.blk[k].b_len; t++) if (bp_is_ambiguous(b.at(s.blk[k].b_start + t))) return true;
    }
  }
  return false;
}
XM_FN bool quickly_confident(WS& w, const QAStore* best, const QMX& bm) {  // quicklyConfidentInBestAlignment :494-587
  XM_CHECK_MASK(w);
  if (best == nullptr) return false;
  if (qa_has_indel(*best)) return false;
  int contig = bm.comp[0].contig;
  int first_sb = sm_start_b(w, bm.comp[0]), last_sb = sm_start_b(w, bm.comp[bm.n - 1]);
  int match_start = imin(first_sb, last_sb), match_end = imax(first_sb, last_sb);  // QueryMatch.getStartIndexB/getEndIndexB (sic)
  double gran = w.dup->granularity;
  double penalty = best->total;
  double num_mut = (penalty + w.prm.span) / w.prm.mutation;
  int qtl = 0; for (int i = 0; i < bm.n; i++) qtl += w.query.seq[bm.comp[i].mate].len;
  double rate = num_mut / qtl;
  if (penalty <= 0 && w.prm.span < w.prm.min_possible_nonzero()) return true;
  double p_mut = 1 - pow(1 - rate, gran);
  double acceptable = 1.0 / (double)w.ref->total_fr;
  double n_unmatched = log(acceptable) / log(p_mut);
  double total_len = n_unmatched * gran;
  double middle = (double)((match_start + match_end) / 2);
  double half = (double)((match_end - match_start + 1) / 2);
  double window = (total_len != total_len) ? total_len : dmax(total_len, half);  // Math.max propagates NaN
  int ws = j2i(middle - window), we = j2i(middle + window);
  bool near = false;
  if (dup_may_contain(w, contig, ws, we)) near = true;
  else if (match_start <= window) near = true;
  else if (match_end >= w.ref->len[contig] - window) near = true;
  if (near) return false;
  if (qa_has_ambiguous(w, *best)) return false;
  return true;
}

XM_HD inline QMX qmx_from_qm(const WS& w, const QM& q) {
  QMX x; x.n = (q.c[1] >= 0) ? 2 : 1; x.priority = q.priority; x.hint = q.hint;
  x.comp[0] = qm_comp(w, q, 0);
  if (x.n > 1) x.comp[1] = qm_comp(w, q, 1); else x.comp[1] = x.comp[0];
  return x;
}

// emits one component's choices into the result arena
XM_FN void emit_component(WS& w, OutArena& out, OutQuery& oq, int comp_index, QAStore** list, int n) {
  XM_CHECK_MASK(w);
  oq.n_choice[comp_index] = n;
  if (n == 0) { oq.choice_first[comp_index] = 0; return; }
  long long n_sa = 0, n_blk = 0;
  XM_NOUNROLL
  for (int i = 0; i < n; i++) { n_sa += list[i]->n_sa; for (int s = 0; s < list[i]->n_sa; s++) n_blk += list[i]->sa[s].n_blk; }
  long long c0 = (long long)xm_atomic_add(&out.used[0], (unsigned long long)n);
  long long s0 = (long long)xm_atomic_add(&out.used[1], (unsigned long long)n_sa);
  long long b0 = (long long)xm_atomic_add(&out.used[2], (unsigned long long)n_blk);
  if (c0 + n > out.cap_choices || s0 + n_sa > out.cap_sas || b0 + n_blk > out.cap_blocks) { w.fail(Q_OUT_FULL); return; }
  oq.choice_first[comp_index] = c0;
  XM_NOUNROLL
  for (int i = 0; i < n; i++) {
    const QAStore& q = *list[i];
    OutChoice& oc = out.choices[c0 + i];
    oc.spacing = q.spacing; oc.multiplier = q.multiplier; oc.bonus = q.bonus; oc.total = q.total; oc.inner = q.inner; oc.n_sa = q.n_sa; oc.sa_first = s0;
    XM_NOUNROLL
    for (int s = 0; s < q.n_sa; s++) {
      const SAStore& sa = q.sa[s];
      OutSA& os = out.sas[s0++];
      os.penalty = sa.penalty; os.aligned = sa.aligned; os.contig = sa.contig; os.reversed = sa.ref_reversed; os.n_blocks = sa.n_blk; os.pad = 0; os.block_first = b0;
      XM_NOUNROLL
      for (int k = 0; k < sa.n_blk; k++) { int32_t* d = out.blocks + 4 * (b0++); d[0] = sa.blk[k].a_start; d[1] = sa.blk[k].b_start; d[2] = sa.blk[k].a_len; d[3] = sa.blk[k].b_len; }
    }
  }
}

// AlignerWorker.alignToAncestralReference :306-484 (+ getUnpairedAlignments :602-644). Results go to `out`.
template <bool EASY>
XM_HD inline void align_query(WS& w, OutArena& out, OutQuery& oq) {
  oq.n_comp = 1; oq.n_choice[0] = 0; oq.n_choice[1] = 0; oq.choice_first[0] = 0; oq.choice_first[1] = 0;
  const Params& P = w.prm;
  int nseq = w.query.n_seqs;
  XM_NOUNROLL
  for (int i = 0; i < nseq; i++) if (w.query.seq[i].len < 1) { w.fail(Q_INTERNAL); return; }
  double max_interesting = w.query.length() * P.max_error_rate;
  int max_inner = j2i(max_interesting * w.query.per_penalty + w.query.expected_inner);
  w.pc_max_offset_between = max_inner + w.mp[0].q.len;
  int cap_good = (int)(w.store_size / 512);
  if (cap_good < 16) cap_good = 16;
  if (cap_good > 65536) cap_good = 65536;
  QMA A;
  qma_init(w, A, P, w.query.length(), cap_good);
  if (w.status != 0) return;
  QAStore* optimistic = nullptr;
  bool have_opt = false; QM opt_qm; opt_qm.c[0] = -1; opt_qm.c[1] = -1; opt_qm.priority = 0; opt_qm.hint = 0;
  int opt_n = nseq;
  int num_mis = 0;
  int filt = pc_optimistic_best(w);
  if (w.status != 0) return;
  int n_best = 0, best_i = -1;
  XM_NOUNROLL
  for (int i = 0; i < w.n_assembled; i++) if (w.assembled[i].priority == filt) { n_best++; best_i = i; }
  if (n_best == 1) {
    opt_qm = w.assembled[best_i]; have_opt = true;
    QMX x = qmx_from_qm(w, opt_qm);
    optimistic = qma_align<EASY>(w, A, x, 0, w.query.length());
    if (w.status != 0) return;
    if (quickly_confident(w, optimistic, x)) { QAStore* l[1] = {optimistic}; emit_component(w, out, oq, 0, l, 1); return; }
  }
  if (optimistic != nullptr) {
    XM_NOUNROLL
    while (true) {
      double possible = penalty_lower_bound(w, num_mis);
      if (possible > optimistic->total + P.span) { QAStore* l[1] = {optimistic}; emit_component(w, out, oq, 0, l, 1); return; }
      pc_find_good_up_to(w, num_mis);
      if (w.status != 0) return;
      int k = num_mis;
      num_mis++;
      bool done = false;
      XM_NOUNROLL
      for (int i = 0; i < w.n_assembled; i++) {
        if (w.assembled[i].priority != k) continue;
        if (!qm_same_position(opt_qm, opt_n, w.assembled[i], nseq)) { done = true; break; }
      }
      if (done) break;
    }
  }
  double best_penalty = (double)JMAX;
  int cand = 0;
  XM_NOUNROLL
  while (true) {
    double est = penalty_lower_bound(w, cand);
    if (est > best_penalty + P.span) break;
    if (cand > pc_num_blocks(w)) break;
    pc_find_good_up_to(w, cand);
    if (w.status != 0) return;
    // the candidate list is a filtered view of w.assembled, which alignMatch does not modify
    XM_NOUNROLL
    for (int i = 0; i < w.n_assembled; i++) {
      if (w.assembled[i].priority != cand) continue;
      QAStore* a;
      if (have_opt && qm_same_position(w.assembled[i], nseq, opt_qm, opt_n)) a = optimistic;
      else { QMX x = qmx_from_qm(w, w.assembled[i]); a = qma_align<EASY>(w, A, x, 0, w.query.length()); }
      if (w.status != 0) return;
      if (a != nullptr) { if (best_penalty > a->total) best_penalty = a->total; }
    }
    if (est >= max_interesting) break;
    cand++;
  }
  long long mark = w.scratch_top;
  QAStore** best_list;
  int nb = qma_best(w, A, best_list);
  if (w.status != 0) return;
  if (nb < 1 && nseq > 1) {
    w.scratch_top = mark;
    if (pc_find_partially_good(w)) {
      XM_NOUNROLL
      for (int i = 0; i < w.n_assembled && w.status == 0; i++) {
        QMX x = qmx_from_qm(w, w.assembled[i]);
        QAStore* a = qma_align<EASY>(w, A, x, 0, w.query.length());
        if (a != nullptr) { if (best_penalty > a->total) best_penalty = a->total; }
      }
    }
    if (w.status != 0) return;
    mark = w.scratch_top;
    nb = qma_best(w, A, best_list);
    if (w.status != 0) return;
  }
  if (nb < 1 && nseq > 1) {
    // getUnpairedAlignments :602-644
    w.scratch_top = mark;
    oq.n_comp = 2;
    XM_NOUNROLL
    for (int si = 0; si < nseq; si++) {
      int slen = w.query.seq[si].len;
      double max_sub = slen * P.max_error_rate;
      int max_mut = j2i(max_sub / P.mutation);
      CL l = counting_find_good_up_to(w, w.mp[si], max_mut);
      if (w.status != 0) return;
      QMA S;
      qma_init(w, S, P, slen, cap_good);
      if (w.status != 0) return;
      int cur = -1, ci;
      XM_NOUNROLL
      while ((ci = list_next(w, w.mp[si], l, cur)) >= 0) {
        SM sm = counter_match(w.mp[si], w.mp[si].counters[ci]);
        int min_inner;
        if (si % 2 == 1) min_inner = sm_start_b(w, sm); else min_inner = w.ref->len[sm.contig] - sm_end_b(w, sm);
        double inner = min_inner;
        if (inner < w.query.expected_inner) inner = w.query.expected_inner;
        double sp = inner / w.query.per_penalty;
        if (sp > max_sub) continue;
        QMX x; x.n = 1; x.comp[0] = sm; x.comp[1] = sm; x.priority = -1; x.hint = 0;
        qma_align<EASY>(w, S, x, inner, slen);
        if (w.status != 0) return;
      }
      long long m2 = w.scratch_top;
      QAStore** sub_list;
      int ns = qma_best(w, S, sub_list);
      if (w.status != 0) return;
      emit_component(w, out, oq, si, sub_list, ns);
      w.scratch_top = m2;
      if (w.status != 0) return;
    }
    return;
  }
  if ((long long)nb > (long long)P.max_num_matches) { oq.n_choice[0] = 0; return; }
  emit_component(w, out, oq, 0, best_list, nb);
}

// Carves the per-thread workspace out of a flat arena and resets all per-query state.
// fills the 256-entry pair-penalty table (Params::pen_tab) with the reference's formula
XM_HD inline void fill_pen_tab(const Params& prm, double* tab, uint8_t* cls, int first, int step) {  // tab: 256 doubles, cls: 1024 bytes
  for (int i = first; i < 256; i += step) tab[i] = prm.base_penalty_formula((uint8_t)(i >> 4), (uint8_t)(i & 15));
  for (int i = first; i < 1024; i += step) {
    const int q = i >> 5, r = i & 31;
    if (q >= 16 || r >= 16) { cls[i] = 1; continue; }   // a sentinel: the reference skips both checks when an index is off the section
    const double v = prm.base_penalty_formula((uint8_t)q, (uint8_t)r);
    cls[i] = (uint8_t)((bp_can_match((uint8_t)q, (uint8_t)r) ? 1 : 0) | (v == 0 ? 2 : 0) | ((bp_is_fully_ambiguous((uint8_t)q) || bp_is_fully_ambiguous((uint8_t)r)) ? 4 : 0));
  }
}
// with_lattice: the arena begins with the PathAligner lattice (3/8 of the arena, behind a 16-byte header: [0] generation, 0 = the
// region has not been used since the launch began - the host clears this word before every launch).  The region keeps its place and
// meaning across the queries an arena serves, which is what lets a search start without clearing anything.
XM_HD inline bool ws_init(WS& w, char* arena, long long arena_bytes, const RefD* ref, const IndexD* ix, const DupD* dup, const Params& prm, const QueryIn& q, bool with_lattice = true) {
  w.cell_hdr = nullptr; w.cellmap = nullptr; w.cell_words = 0;
  if (with_lattice) {
    const long long region = (arena_bytes * 3 / 8) & ~15LL;
    w.cell_hdr = (uint32_t*)arena; w.cellmap = (uint32_t*)(arena + 16); w.cell_words = (region - 16) / 4;
    arena += region; arena_bytes -= region;
  }
  w.ref = ref; w.ix = ix; w.dup = dup; w.prm = prm; w.query = q;
  w.status = 0; w.next_list_id = 1;
  w.pc_have_prev = 0; w.pc_found_nonempty = 0; w.n_assembled = 0;
  w.st_probes = w.st_seeds = w.st_hits = w.st_straight = w.st_path_calls = w.st_path_steps = w.st_path_cells = 0;
  XM_NOUNROLL
  for (int i = 0; i < 6; i++) w.st_cyc[i] = 0;
  XM_CHECK_MASK(w);
  long long top = 0;
  auto take = [&](long long bytes) -> char* { bytes = (bytes + 15) & ~15LL; char* p = arena + top; top += bytes; return p; };
  // pyramids: a block's level never exceeds its length, so len + 2 levels always suffice; ~4 blocks per base are
  // typical, 8 are provisioned when the arena allows (pyr_build asks for the next tier when a read needs more)
  long long pyr_total = 0;
  long long pyr_bytes[2] = {0, 0};
  XM_NOUNROLL
  for (int i = 0; i < q.n_seqs; i++) { pyr_bytes[i] = pyr_arena_bytes(q.seq[i].len); pyr_total += pyr_bytes[i]; }
  if (pyr_total > arena_bytes / 2) {
    XM_NOUNROLL
    for (int i = 0; i < q.n_seqs; i++) pyr_bytes[i] = (long long)((double)pyr_bytes[i] * (double)(arena_bytes / 2) / (double)pyr_total) & ~15LL;
    pyr_total = arena_bytes / 2;
  }
  long long rest = arena_bytes - pyr_total - 512 - 2 * (long long)(q.seq[0].len + (q.n_seqs > 1 ? q.seq[1].len : 0) + 64);
  if (rest < 4096) return false;
  // split of the remainder: counters 12%, history+pending 6%, assembled 8%, store 24%, scratch 50%
  int cap_counters = (int)(rest * 12 / 100 / q.n_seqs / (long long)(sizeof(Counter) + sizeof(int)));
  int cap_hist = (int)(rest * 3 / 100 / q.n_seqs / (long long)sizeof(Hist));
  int cap_pend = (int)(rest * 3 / 100 / q.n_seqs / (long long)sizeof(HB));
  int cap_asm = (int)(rest * 8 / 100 / (long long)sizeof(QM));
  if (cap_counters < 8 || cap_hist < 8 || cap_pend < 4 || cap_asm < 8) return false;
  XM_NOUNROLL
  for (int i = 0; i < q.n_seqs; i++) {
    MatePath& m = w.mp[i];
    m.mate = i; m.path_is_rc = (i > 0) ? 1 : 0;
    {  // unpack the read in both orientations, one code per byte (lanes split the bases on the device)
      int len = q.seq[i].len;
      uint8_t* f = (uint8_t*)take(len + 1); uint8_t* r = (uint8_t*)take(len + 1);
      SeqView pv = q.seq[i]; pv.rc = 0; pv.bytes = nullptr;
      for (int k = lane_id(); k < len; k += XM_LANES) { uint8_t c = pv.at(k); f[k] = c; r[len - 1 - k] = bp_complement(c); }
      warp_sync();
      w.qbytes[i][0] = f; w.qbytes[i][1] = r;
      w.query.seq[i].bytes = nullptr;
    }
    m.q = w.query_view(i, m.path_is_rc);
    {
      int len = q.seq[i].len;
      Pyr& P = m.pyr;
      P.cap_levels = len + 2;
      long long lev_bytes = ((long long)(P.cap_levels + 1) * 4 + 15) & ~15LL;
      long long cap = (pyr_bytes[i] - lev_bytes - 64) / 20;
      if (cap < len + 8) return false;
      if (cap > 32000) cap = 32000;
      cap &= ~7LL;
      P.cap_blocks = (int)cap;
      P.level_off = (int32_t*)take(lev_bytes);
      P.blk = (HB16*)take(cap * 16); P.child = (int16_t*)take(cap * 2); P.up = (int16_t*)take(cap * 2);
      P.n_levels = 0;
    }
    XM_NOUNROLL
    m.counters = (Counter*)take((long long)cap_counters * (long long)sizeof(Counter)); m.n_counters = 0; m.cap_counters = cap_counters;
    m.good = (int*)take((long long)cap_counters * 4); m.n_good = 0;
    m.history = (Hist*)take((long long)cap_hist * (long long)sizeof(Hist)); m.n_hist = 0; m.cap_hist = cap_hist;
    m.pending = (HB*)take((long long)cap_pend * (long long)sizeof(HB)); m.pend_head = 0; m.pend_cnt = 0; m.cap_pend = cap_pend;
    m.found_good = 0; m.n_blocks_anywhere = 0; m.max_nonoverlap_visited = 0; m.n_nonoverlap_visited = 0; m.min_num_distinct = -1; m.done = 0;
    // Counting_HashBlockPath constructor :33-36
    int max_possible_indel = j2i((m.q.len * prm.max_error_rate - prm.del_start) / prm.del_ext);
    m.max_indel_consider = max_possible_indel / 2;
    m.ph_valid = 0; m.pa_valid = 0;
    path_init(w, m);
  }
  w.assembled = (QM*)take((long long)cap_asm * (long long)sizeof(QM)); w.cap_assembled = cap_asm;
  long long store_bytes = (rest * 24 / 100) & ~15LL;
  w.store = take(store_bytes); w.store_size = store_bytes; w.store_top = 0;
  long long scratch_bytes = (arena_bytes - top - 64) & ~15LL;
  if (scratch_bytes < 1024) return false;
  w.scratch = take(scratch_bytes); w.scratch_size = scratch_bytes; w.scratch_top = 0;
  XM_NOUNROLL
  XM_CHECK_MASK(w);
  for (int i = 0; i < q.n_seqs; i++) if (!pyr_build(w, w.mp[i])) break;  // sets w.status itself (next tier, or ambiguous query)
  return true;
}

}  // namespace xm
