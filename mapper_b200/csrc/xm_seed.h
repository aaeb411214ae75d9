// xmapper_b200 device core — seeding: content-defined hash blocks, gapmers, the seed walk, index lookups,
// flank verification, candidate binning and mate pairing.  One query per thread; all state lives in the
// per-thread workspace (WS).  Reproduces, result for result:
//   M/HashBlock.java, M/HashBlock_BaseRow.java, M/HashBlock_ParentRow.java (rows are kept as small sliding
//   windows: a block is a pure function of the bases at and after its start, so a row may restart its scan at
//   any requested position — same blocks as the reference's append-only lists, bounded memory),
//   M/HashBlockPath.java, M/Readable_HashBlock_Database.java, M/PackedMap.java (read side),
//   M/Counting_HashBlockPath.java, M/HashBlockMatch_Counter.java, M/HashBlockPaths_Counter.java.
#pragma once
#include "xm_types.h"

namespace xm {

struct HB {  // M/HashBlock.java:385-397
  int start, len, used;
  int32_t fwd, rev;
  int8_t gap_dir;
  uint8_t flags;  // 1 requestMergeLeft, 2 requestMergeRight, 4 nextRequestMergeLeft, 8 nextRequestMergeRight
  int16_t extra;
  long long ident;  // object identity stand-in (HashBlockMatch_Counter.update compares references)
  XM_INLINE int end() const { return start + len; }
  XM_INLINE bool rml() const { return flags & 1; }
  XM_INLINE bool rmr() const { return flags & 2; }
  XM_INLINE bool primary() const { return (rml() != rmr()) ? rml() : (fwd >= rev); }  // :332-337
  XM_INLINE int32_t lookup_key() const { return primary() ? fwd : rev; }
};

XM_INLINE int max_gapmer_used(int len) { return len + len * 9 / 8 + 1; }  // HashBlock.java:12-14

XM_INLINE int32_t merge_hash(int l_len, int32_t l_h, int r_len, int32_t r_h) {  // :261-269
  unsigned long long rl = (unsigned long long)((long long)l_h + 1) * (unsigned long long)(54323LL + 323LL * (long long)r_len);
  unsigned long long rr = (unsigned long long)(long long)wadd(r_h, 1) * (unsigned long long)(long long)l_len;
  unsigned long long top = rl + rr;
  return wadd((int32_t)(uint32_t)top, (int32_t)(uint32_t)(top >> 32));
}

XM_INLINE HB base_block(uint8_t code, int index) {  // HashBlock(char,int) + hashChar :60-65,171-188
  HB b;
  b.start = index; b.len = 1; b.used = 1; b.gap_dir = 0; b.extra = 0;
  b.fwd = (code == 1) ? 0 : (code == 2) ? 1 : (code == 4) ? 2 : 3;
  bool rml = (b.fwd / 2 == 0), nrml = (b.fwd % 2 == 0);
  b.flags = (uint8_t)((rml ? 1 : 2) | (nrml ? 4 : 8));
  b.rev = 3 - b.fwd;
  b.ident = index;
  return b;
}

XM_FN HB merge_blocks(const HB& L, const HB& R, int level) {  // HashBlock(seq,start,len,l,r) :20-44 + mergeHashes :192-259
  HB b;
  b.start = L.start; b.len = R.end() - L.start; b.used = b.len;
  b.fwd = merge_hash(L.len, L.fwd, R.len, R.fwd);
  b.rev = merge_hash(R.len, R.rev, L.len, L.rev);
  bool rml = true, rmr = true, nrml = true, nrmr = true;
  int anchor = 0;  // 0 none, 1 left, 2 right
  if (L.fwd != R.rev) anchor = (L.fwd > R.rev) ? 2 : 1;
  if (anchor != 0 && b.fwd != b.rev) {
    const HB& A = (anchor == 2) ? R : L;
    const HB& O = (anchor == 2) ? L : R;
    bool is_reverse = b.fwd < b.rev;
    bool invert = is_reverse == (anchor == 2);
    bool aL = (A.flags & 4) != 0, aR = (A.flags & 8) != 0;
    if (aL && aR) { if (anchor == 2) aR = false; else aL = false; }
    bool oL = (O.flags & 4) != 0, oR = (O.flags & 8) != 0;
    if (oL && oR) { if (anchor == 1) oL = false; else oR = false; }  // "other == rightParent" <=> anchor is left
    rml = aL != invert; rmr = aR != invert; nrml = oL != invert; nrmr = oR != invert;
  }
  if (L.len != R.len) { rml = (L.len > R.len); rmr = !rml; nrml = !rml; nrmr = !nrml; }
  if (b.fwd != b.rev) {
    if (rml && rmr) { rml = (b.fwd > b.rev); rmr = !rml; }
    if (nrml && nrmr) { nrml = rml; nrmr = !nrml; }
  }
  b.flags = (uint8_t)((rml ? 1 : 0) | (rmr ? 2 : 0) | (nrml ? 4 : 0) | (nrmr ? 8 : 0));
  b.gap_dir = 0;
  if (rml != rmr) b.gap_dir = rml ? 1 : -1;
  else if (L.fwd != R.rev) b.gap_dir = (L.fwd > R.rev) ? 1 : -1;
  b.extra = (int16_t)((L.len + R.len - b.len) / 4);
  b.ident = ((long long)level << 40) | (long long)b.start;
  return b;
}

XM_INLINE int ext_char_to_int(uint8_t c) { return c == 1 ? 1 : c == 2 ? 2 : c == 4 ? 3 : c == 8 ? 4 : 0; }

// HashBlock.withGapAndExtension :67-150. false = null
// h = fold(h * 7654337 + value(base)) over n bases starting at `from`, stepping `dir` (HashBlock.java:107-135).
// Integer wrap-around arithmetic is a ring, so on the device 32 lanes each take one base of a 32-base chunk,
// weight it with the matching power of the multiplier and add the chunk up with shuffles: same 32-bit result.
XM_HD inline int32_t ext_hash(const SeqView& seq, int from, int n, int dir, bool complement) {
  int32_t h = 0;
#if defined(__CUDA_ARCH__)
  constexpr uint32_t M1 = 7654337u, M2 = M1 * M1, M4 = M2 * M2, M8 = M4 * M4, M16 = M8 * M8, M32 = M16 * M16;
  const int lane = (int)(threadIdx.x & 31);
  XM_NOUNROLL
  for (int base = 0; base < n; base += 32) {
    const int cnt = imin(32, n - base);
    uint32_t term = 0;
    if (lane < cnt) {
      uint8_t c = seq.at(from + dir * (base + lane));
      if (complement) c = bp_complement(c);
      const int e = cnt - 1 - lane;
      uint32_t pw = 1u;
      if (e & 1) pw *= M1;
      if (e & 2) pw *= M2;
      if (e & 4) pw *= M4;
      if (e & 8) pw *= M8;
      if (e & 16) pw *= M16;
      term = (uint32_t)ext_char_to_int(c) * pw;
    }
    __syncwarp();
    term += __shfl_xor_sync(0xffffffffu, term, 16);
    term += __shfl_xor_sync(0xffffffffu, term, 8);
    term += __shfl_xor_sync(0xffffffffu, term, 4);
    term += __shfl_xor_sync(0xffffffffu, term, 2);
    term += __shfl_xor_sync(0xffffffffu, term, 1);
    uint32_t pc = (cnt == 32) ? M32 : 1u;
    if (cnt != 32) { if (cnt & 1) pc *= M1; if (cnt & 2) pc *= M2; if (cnt & 4) pc *= M4; if (cnt & 8) pc *= M8; if (cnt & 16) pc *= M16; }
    h = (int32_t)((uint32_t)h * pc + term);
  }
#else
  for (int k = 0; k < n; k++) {
    uint8_t c = seq.at(from + dir * k);
    if (complement) c = bp_complement(c);
    h = wadd(wmul(h, 7654337), ext_char_to_int(c));
  }
#endif
  return h;
}
XM_FN bool with_gap_and_extension(const HB& b, const SeqView& seq, HB& out) {
  if (b.gap_dir == 0) { out = b; return true; }
  int target = b.len + (jabs(b.fwd > b.rev ? b.fwd : b.rev) % 3) + b.extra;
  int gap = b.len / 2;
  int ext = target - gap;
  int32_t h;
  HB r;
  if (b.gap_dir < 0) {
    int ext_end = b.start - gap, ext_start = ext_end - ext;
    if (ext_start < 0) return false;
    h = ext_hash(seq, ext_end - 1, ext, -1, false);
    r.start = ext_start; r.len = ext + gap + b.len;
  } else {
    int ext_start = b.end() + gap, ext_end = ext_start + ext;
    if (ext_end > seq.len) return false;
    h = ext_hash(seq, ext_start, ext, 1, true);
    r.start = b.start; r.len = b.len + gap + ext;
  }
  r.fwd = wadd(b.fwd, h); r.rev = wadd(b.rev, h);
  r.used = b.len + ext;
  r.gap_dir = 0; r.flags = 0; r.extra = 0; r.ident = 0;
  out = r;
  return true;
}

// ---------------- workspace ----------------
// The query's hash-block pyramid (HashBlock_Pyramid / HashBlock_ParentRow), built EAGERLY and in full when the
// workspace is set up: a block is a pure function of the bases it covers, so the reference's lazily grown rows and this
// table hold the same blocks.  Level L+1 = merge(b[i], b[i+1]) of the consecutive level-L blocks that satisfy
// shouldMergeBlocks (HashBlock_ParentRow.java:69-127,200-208); on the device the 32 lanes take 32 pairs per round and
// compact the survivors with a ballot.  child/up are the links the seed walk follows instead of searching.
XM_INLINE long long pyr_arena_bytes(int len) { return (((long long)(len + 3) * 4 + 15) & ~15LL) + 64 + 20LL * (8LL * len + 64); }
struct HB16 { int16_t start, len; int32_t fwd, rev; uint8_t flags; int8_t gap_dir; int16_t extra; };
// One possibility of a MultiHashBlock (M/ConditionalHashBlock.java): the block (valid iff has) that exists when the
// IUPAC-ambiguous bases at the positions listed in kv take the listed bases - M/SequenceCondition.java as a short sorted list of
// (position << 2 | base: A0 C1 G2 T3).  A stored possibility constrains only the ambiguous positions inside its block, and a
// multi-block with more than 64 possibilities is dropped (HashBlock_ParentRow.java:10,109,165), so the lists stay short; a condition
// that would need more than POPT_MAX_KEYS entries fails the sequence loudly (Q_AMBIGUOUS_QUERY) instead of being truncated.
static const int POPT_MAX_KEYS = 31;
struct POpt { HB16 hb; int32_t n_kv; uint32_t kv[POPT_MAX_KEYS]; int has, pad; };
static const uint8_t HB_MULTI = 0x80;  // HB16::flags / HB::flags: the entry is a MultiHashBlock; fwd = first POpt, rev = number of POpts
struct Pyr {
  POpt* opt; int n_opt, cap_opt;   // possibilities of the multi-blocks (only queries with ambiguous bases)
  HB16* blk;          // all levels back to back, each level ascending by start
  int16_t* child;     // per block: index within the level below of its left parent (level 0: -1)
  int16_t* up;        // per block: index within the level above of the block it is the left parent of, or -1
  int32_t* level_off; // n_levels + 1
  int n_levels, cap_blocks, cap_levels;
};

struct Counter {  // M/HashBlockMatch_Counter.java
  int set, contig, offset;  // set 0 = reversed matches ("forwardMatchCounters"), 1 = the others
  int num_matches, num_distinct, last_mismatched_pos;
  long long last_matched_ident;
  int has_last, hist_processed, good, priority;
  int next, prev;
};
struct Hist { int start, end; long long ident; };
struct SM { int mate, rev, contig, offset, from_hash; };  // M/SequenceMatch.java: a = rev ? RC(read[mate]) : read[mate]
struct CL { int id, kind, G, k, size; };                  // lazily evaluated List<HashBlockMatch_Counter>
struct QM { int c[2]; int priority; int hint; };          // M/QueryMatch.java, components as counter indices

struct MatePath {
  SeqView q;  // sequence the path walks (mate 2: reverse complement of the read, AlignerWorker.java:317-318)
  int mate, path_is_rc;
  Pyr pyr; int cur_idx;  // cur_idx: index of cur within level batch_index (-1: cur is not a pyramid block)
  // HashBlockPath
  int batch_index, cur_valid; HB cur; int have_gapmer; HB gapmer;
  int have_prev, have_prevprev; int32_t prev_fwd, prevprev_fwd; long long gapmer_serial;
  // Counting_HashBlockPath
  Counter* counters; int n_counters, cap_counters;
  int* good; int n_good;
  Hist* history; int n_hist, cap_hist;
  HB* pending; int pend_head, pend_cnt, cap_pend;
  int found_good, n_blocks_anywhere, max_nonoverlap_visited, n_nonoverlap_visited, min_num_distinct, done, max_indel_consider;
  int ph_valid; CL ph;   // previousHighPriorityMatchCounters
  int pa_valid; CL pa;   // previousAllPositions
};

struct DAlnStore;  // xm_align.h

#if defined(__CUDA_ARCH__)
#define XM_CLK() ((unsigned long long)clock64())
#else
#define XM_CLK() 0ull
#endif
struct PhaseClock {  // adds the ticks between construction and destruction to *slot
  unsigned long long* slot; unsigned long long t0;
  XM_INLINE PhaseClock(unsigned long long* s) : slot(s), t0(XM_CLK()) {}
  XM_INLINE ~PhaseClock() { *slot += XM_CLK() - t0; }
};

struct WS {
  const RefD* ref; const IndexD* ix; const DupD* dup;
  Params prm; QueryIn query;
  int status;
  int next_list_id;
  MatePath mp[2];
  // HashBlockPaths_Counter
  int pc_max_offset_between, pc_have_prev, pc_prev_ids[2], pc_found_nonempty;
  QM* assembled; int n_assembled, cap_assembled;
  // scratch (stack discipline)
  char* scratch; long long scratch_size, scratch_top;
  // alignment store (xm_align.h)
  char* store; long long store_size, store_top;
  unsigned long long st_probes, st_seeds, st_hits, st_straight, st_path_calls, st_path_steps, st_path_cells;
  unsigned long long st_cyc[6];  // SM clock ticks per phase (device only): 0 seed step, 1 straight score, 2 HashBlock_Aligner analysis, 3 PathAligner, 4 matcher table builds, 5 spare

  XM_INLINE void fail(int s) { if (status == 0) { status = s; XM_T("FAIL status=%d\n", s); } }
  XM_INLINE void* salloc(long long bytes) {
    bytes = (bytes + 7) & ~7LL;
    if (scratch_top + bytes > scratch_size) { fail(Q_NEED_MORE); return nullptr; }
    void* p = scratch + scratch_top; scratch_top += bytes; return p;
  }
  // TMA staging area of this warp in shared memory (device, full kernel): an mbarrier, the packed reference window as cp.async.bulk
  // delivers it, and the window unpacked to one code per byte (what every stage of the cascade reads).  nullptr: windows are unpacked
  // from global memory into the arena.
  unsigned char* stage; unsigned int stage_phase;
  uint32_t* cell_hdr; uint32_t* cellmap; long long cell_words;  // PathAligner lattice map region of the arena (xm_align.h: PathState::cell)
  uint8_t* qbytes[2][2];  // [mate][reverse-complemented]: one code per byte
  int hard_hint;  // first pass: cost estimate of a query handed to the full kernel (its ungapped penalty), used to start long queries first
  XM_INLINE SeqView query_view(int mate, int rev) const { SeqView v = query.seq[mate]; v.rc = rev; v.bytes = qbytes[mate][rev]; v.b0 = 0; v.bn = v.len; return v; }
};

XM_INLINE int sm_start_b(const WS& w, const SM& m) { return imax(0, m.offset); }
XM_INLINE int sm_end_b(const WS& w, const SM& m) { return imin(m.offset + w.query.seq[m.mate].len, w.ref->len[m.contig]); }
XM_INLINE SM counter_match(const MatePath& m, const Counter& c) {
  SM s; s.mate = m.mate; s.rev = (c.set == 0) ? 1 : 0; s.contig = c.contig; s.offset = c.offset; s.from_hash = 1; return s;
}

// ---------------- pyramid ----------------
XM_INLINE HB16 base_block16(uint8_t code, int index) {  // HashBlock(char,int) + hashChar :60-65,171-188
  HB16 b;
  b.start = (int16_t)index; b.len = 1; b.gap_dir = 0; b.extra = 0;
  b.fwd = (code == 1) ? 0 : (code == 2) ? 1 : (code == 4) ? 2 : 3;
  bool rml = (b.fwd / 2 == 0), nrml = (b.fwd % 2 == 0);
  b.flags = (uint8_t)((rml ? 1 : 2) | (nrml ? 4 : 8));
  b.rev = 3 - b.fwd;
  return b;
}
XM_HD inline HB16 merge_blocks16(const HB16& L, const HB16& R) {  // HashBlock(seq,start,len,l,r) :20-44 + mergeHashes :192-259
  HB16 b;
  int blen = (R.start + R.len) - L.start;
  b.start = L.start; b.len = (int16_t)blen;
  b.fwd = merge_hash(L.len, L.fwd, R.len, R.fwd);
  b.rev = merge_hash(R.len, R.rev, L.len, L.rev);
  bool rml = true, rmr = true, nrml = true, nrmr = true;
  int anchor = 0;  // 0 none, 1 left, 2 right
  if (L.fwd != R.rev) anchor = (L.fwd > R.rev) ? 2 : 1;
  if (anchor != 0 && b.fwd != b.rev) {
    const HB16& A = (anchor == 2) ? R : L;
    const HB16& O = (anchor == 2) ? L : R;
    bool is_reverse = b.fwd < b.rev;
    bool invert = is_reverse == (anchor == 2);
    bool aL = (A.flags & 4) != 0, aR = (A.flags & 8) != 0;
    if (aL && aR) { if (anchor == 2) aR = false; else aL = false; }
    bool oL = (O.flags & 4) != 0, oR = (O.flags & 8) != 0;
    if (oL && oR) { if (anchor == 1) oL = false; else oR = false; }  // "other == rightParent" <=> anchor is left
    rml = aL != invert; rmr = aR != invert; nrml = oL != invert; nrmr = oR != invert;
  }
  if (L.len != R.len) { rml = (L.len > R.len); rmr = !rml; nrml = !rml; nrmr = !nrml; }
  if (b.fwd != b.rev) {
    if (rml && rmr) { rml = (b.fwd > b.rev); rmr = !rml; }
    if (nrml && nrmr) { nrml = rml; nrmr = !nrml; }
  }
  b.flags = (uint8_t)((rml ? 1 : 0) | (rmr ? 2 : 0) | (nrml ? 4 : 0) | (nrmr ? 8 : 0));
  b.gap_dir = 0;
  if (rml != rmr) b.gap_dir = rml ? 1 : -1;
  else if (L.fwd != R.rev) b.gap_dir = (L.fwd > R.rev) ? 1 : -1;
  b.extra = (int16_t)((L.len + R.len - blen) / 4);
  return b;
}
XM_INLINE HB pyr_block(const Pyr& P, int level, int idx) {
  const HB16 c = P.blk[P.level_off[level] + idx];
  HB b;
  b.start = c.start; b.len = c.len; b.used = c.len; b.fwd = c.fwd; b.rev = c.rev; b.gap_dir = c.gap_dir; b.flags = c.flags; b.extra = c.extra;
  b.ident = ((long long)level << 40) | (long long)c.start;
  return b;
}
XM_INLINE int pyr_level_size(const Pyr& P, int level) { return (level >= 0 && level < P.n_levels) ? P.level_off[level + 1] - P.level_off[level] : 0; }
// first block of `level` whose start > p (HashBlock_ParentRow.getAfter :44-59 / HashBlock_BaseRow.get), or -1
XM_FN int pyr_find_after(const Pyr& P, int level, int p) {
  int n = pyr_level_size(P, level);
  const HB16* b = P.blk + (n > 0 ? P.level_off[level] : 0);
  int lo = 0, hi = n;
  XM_NOUNROLL
  while (lo < hi) { int mid = (lo + hi) >> 1; if ((int)b[mid].start > p) hi = mid; else lo = mid + 1; }
  return lo < n ? lo : -1;
}
// ---- queries with IUPAC-ambiguous bases: MultiHashBlocks (M/MultiHashBlock.java, M/ConditionalHashBlock.java,
// M/SequenceCondition.java, HashBlock_BaseRow.java:27-59, HashBlock_ParentRow.java:69-191) ----
// Rare, so built by a scalar pass.  A multi-block occupies one entry of its level like any block (same start, child and
// up links); the walk only ever asks for its start and steps past it (HashBlockPath.skipMultiblocks :130-140), but its
// possibilities decide which blocks exist above it, so they are kept in full.
XM_INLINE bool popt_intersect(const POpt& a, const POpt& b, POpt& out, bool& overflow) {  // SequenceCondition.intersect :27-106; false = conflict
  int i = 0, j = 0, n = 0;
  uint32_t kv[2 * POPT_MAX_KEYS];
  XM_NOUNROLL
  while (i < a.n_kv && j < b.n_kv) {
    const uint32_t x = a.kv[i], y = b.kv[j];
    if ((x >> 2) < (y >> 2)) { kv[n++] = x; i++; }
    else if ((y >> 2) < (x >> 2)) { kv[n++] = y; j++; }
    else { if (x != y) return false; kv[n++] = x; i++; j++; }
  }
  XM_NOUNROLL
  while (i < a.n_kv) kv[n++] = a.kv[i++];
  XM_NOUNROLL
  while (j < b.n_kv) kv[n++] = b.kv[j++];
  if (n > POPT_MAX_KEYS) { overflow = true; n = POPT_MAX_KEYS; }
  out.n_kv = n;
  XM_NOUNROLL
  for (int k = 0; k < n; k++) out.kv[k] = kv[k];
  return true;
}
XM_INLINE bool hb16_should_merge(const HB16& L, const HB16& R) {  // shouldMergeBlocks :200-208
  return ((int)L.start + (int)L.len >= (int)R.start) && ((L.flags & 2) || (R.flags & 1));
}
// possibilities of entry e of a level: a single block counts as one unconditional possibility
XM_INLINE int pyr_num_opts(const HB16& e) { return (e.flags & HB_MULTI) ? (int)e.rev : 1; }
XM_INLINE POpt pyr_opt(const Pyr& P, const HB16& e, int k) {
  if (e.flags & HB_MULTI) return P.opt[e.fwd + k];
  POpt o; o.hb = e; o.n_kv = 0; o.has = 1; o.pad = 0; return o;
}
#if defined(XM_DBG_UNIFORM) && defined(__CUDA_ARCH__)
#define XM_CHECK_MASK(wref) do { if (__activemask() != 0xffffffffu && (wref).st_cyc[5] == 0) (wref).st_cyc[5] = (unsigned long long)__LINE__ + ((unsigned long long)(__FILE__[3] == 's' ? 1 : __FILE__[3] == 'a' ? 2 : 3) * 10000ull); } while (0)
#define XM_CHECK_UNIFORM(tag, val_) do { const unsigned _am = __activemask(); const int _v = (int)(val_); const int _v0 = __shfl_sync(_am, _v, __ffs(_am) - 1); \
  if (_am != 0xffffffffu) { w.status = -(3000 + __LINE__); return false; } if (__any_sync(_am, _v != _v0)) { w.status = -(2000 + __LINE__); return false; } } while (0)
#else
#define XM_CHECK_UNIFORM(tag, val_) do { } while (0)
#define XM_CHECK_MASK(wref) do { } while (0)
#endif
struct PExpandFrame { int j, k, found, pad; POpt cond; };
// HashBlock_ParentRow.expand :137-191 with its recursion unrolled onto `stack`: appends to res[0..n_res)
XM_FN bool pyr_expand(WS& w, const Pyr& P, const HB16* prev, int n_prev, const HB16& left, const POpt& start_cond, int j_from,
                      POpt* res, int& n_res, int cap_res, PExpandFrame* stack, int cap_stack) {
  const int max_combos = 64;  // maxNumCombinationsToExpand :10
  int sp = 0;
  stack[0].j = j_from + 1; stack[0].k = 0; stack[0].found = 0; stack[0].cond = start_cond; sp = 1;
  XM_NOUNROLL
  while (sp > 0) {
    PExpandFrame& f = stack[sp - 1];
    if (f.j >= n_prev) { sp--; continue; }           // getAfter(...) == null
    XM_CHECK_UNIFORM("sp", sp); XM_CHECK_UNIFORM("f.j", f.j); XM_CHECK_UNIFORM("f.k", f.k);
    const HB16 nxt = prev[f.j];
    if (f.k >= pyr_num_opts(nxt)) { sp--; continue; }
    const POpt ro = pyr_opt(P, nxt, f.k);
    f.k++;
    POpt inter;
    bool overflow = false;
    if (!popt_intersect(f.cond, ro, inter, overflow)) { if (f.found) sp--; continue; }  // :163-167 (break once an intersection was seen)
    if (overflow) { w.fail(Q_AMBIGUOUS_QUERY); return false; }
    XM_CHECK_UNIFORM("inter.n_kv", inter.n_kv); XM_CHECK_UNIFORM("ro.has", ro.has);
    f.found = 1;
    if (n_res > max_combos) { sp--; continue; }      // :170 return
    if (!ro.has) {                                   // :171-174 look further right under the narrowed condition
      if (sp >= cap_stack) { w.fail(Q_NEED_MORE); return false; }
      const int nj = f.j + 1;
      PExpandFrame& g = stack[sp++];
      g.j = nj; g.k = 0; g.found = 0; g.cond = inter; g.cond.has = 0;
      continue;
    }
    if (n_res >= cap_res) { w.fail(Q_NEED_MORE); return false; }
    POpt c = inter; c.pad = 0;
    if (hb16_should_merge(left, ro.hb)) { c.has = 1; c.hb = merge_blocks16(left, ro.hb); } else { c.has = 0; c.hb = left; }
    res[n_res++] = c;
  }
  return true;
}
XM_FN bool pyr_build_ambiguous(WS& w, MatePath& m) {
  Pyr& P = m.pyr;
  const int len = m.q.len;
  // possibilities live at the bottom of the scratch stack for the whole query (ws_init calls this before anything marks it)
  long long room = (w.scratch_size - w.scratch_top) / 4;
  P.cap_opt = (int)(room / (long long)sizeof(POpt)); P.n_opt = 0;
  if (P.cap_opt < 256) { w.fail(Q_NEED_MORE); return false; }
  P.opt = (POpt*)w.salloc((long long)P.cap_opt * (long long)sizeof(POpt));
  const int cap_res = 160, cap_stack = 96;
  POpt* res = (POpt*)w.salloc((long long)cap_res * (long long)sizeof(POpt));
  PExpandFrame* stack = (PExpandFrame*)w.salloc((long long)cap_stack * (long long)sizeof(PExpandFrame));
  if (w.status != 0) return false;
  int n_amb = 0;
  XM_CHECK_UNIFORM("entry", len);
  XM_CHECK_UNIFORM("bytes", (int)(unsigned long long)m.q.bytes);
  XM_NOUNROLL
  for (int k = 0; k < len; k++) {  // HashBlock_BaseRow.get :27-59
    const uint8_t code = m.q.at(k);
    XM_CHECK_UNIFORM("code", code);
    XM_CHECK_UNIFORM("k", k);
    XM_CHECK_UNIFORM("nopt_in", P.n_opt);
    P.child[k] = -1; P.up[k] = -1;
    if (!bp_is_ambiguous(code)) { P.blk[k] = base_block16(code, k); continue; }
    HB16 e; e.start = (int16_t)k; e.len = 1; e.fwd = P.n_opt; e.rev = 0; e.flags = HB_MULTI; e.gap_dir = 0; e.extra = 0;
    XM_NOUNROLL
    for (int o = 0; o < 4; o++) {
      const uint8_t base = (uint8_t)(1 << o);
      if (!bp_can_match(code, base)) continue;
      if (P.n_opt >= P.cap_opt) { w.fail(Q_NEED_MORE); return false; }
      POpt c; c.hb = base_block16(base, k); c.has = 1; c.pad = 0; c.n_kv = 1; c.kv[0] = ((uint32_t)k << 2) | (uint32_t)o;
      P.opt[P.n_opt++] = c; e.rev++;
    }
    XM_CHECK_UNIFORM("e.rev", e.rev);
    XM_CHECK_UNIFORM("nopt_out", P.n_opt);
    P.blk[k] = e;
    n_amb++;
  }
  XM_CHECK_UNIFORM("n_amb", n_amb);
  XM_CHECK_UNIFORM("n_opt0", P.n_opt);
  P.level_off[0] = 0; P.level_off[1] = len; P.n_levels = 1;
  int prev_off = 0, n_prev = len, level = 1;
  XM_NOUNROLL
  while (n_prev >= 2) {  // HashBlock_ParentRow.maybeMakeBlock :69-127 for every block of the row below
    if (level >= P.cap_levels) { w.fail(Q_NEED_MORE); return false; }
    const int cur_off = prev_off + n_prev;
    const HB16* prev = P.blk + prev_off;
    int n_new = 0;
    XM_NOUNROLL
    for (int i = 0; i < n_prev - 1; i++) {
      const HB16 L = prev[i], R = prev[i + 1];
      HB16 made; bool keep = false;
      if (!((L.flags | R.flags) & HB_MULTI)) { keep = hb16_should_merge(L, R); if (keep) made = merge_blocks16(L, R); }
      else {
        int n_res = 0;
        const int n_left = pyr_num_opts(L);
        XM_NOUNROLL
        for (int a = 0; a < n_left; a++) {
          const POpt lo = pyr_opt(P, L, a);
          if (lo.has) { if (!pyr_expand(w, P, prev, n_prev, lo.hb, lo, i, res, n_res, cap_res, stack, cap_stack)) return false; }
          else { if (n_res >= cap_res) { w.fail(Q_NEED_MORE); return false; } res[n_res] = lo; res[n_res].has = 0; n_res++; }
        }
        XM_CHECK_UNIFORM("n_res", n_res); XM_CHECK_UNIFORM("n_left", n_left);
        bool any = false;
        for (int a = 0; a < n_res; a++) any |= res[a].has != 0;
        if (n_res > 0 && n_res <= 64 && any) {
          if (P.n_opt + n_res > P.cap_opt) { w.fail(Q_NEED_MORE); return false; }
          made.start = L.start; made.len = 0; made.fwd = P.n_opt; made.rev = n_res; made.flags = HB_MULTI; made.gap_dir = 0; made.extra = 0;
          for (int a = 0; a < n_res; a++) P.opt[P.n_opt++] = res[a];
          keep = true;
        }
      }
      XM_CHECK_UNIFORM("keep", keep); XM_CHECK_UNIFORM("n_new", n_new); XM_CHECK_UNIFORM("i", i); XM_CHECK_UNIFORM("n_prev", n_prev);
      if (keep) {
        if (cur_off + n_new + 1 > P.cap_blocks) { w.fail(Q_NEED_MORE); return false; }
        P.blk[cur_off + n_new] = made; P.child[cur_off + n_new] = (int16_t)i; P.up[cur_off + n_new] = -1;
        P.up[prev_off + i] = (int16_t)n_new;
        n_new++;
      } else P.up[prev_off + i] = -1;
    }
    if (n_new == 0) break;
    P.level_off[level + 1] = cur_off + n_new; P.n_levels = level + 1;
    prev_off = cur_off; n_prev = n_new; level++;
  }
  return true;
}
XM_FN bool pyr_build(WS& w, MatePath& m) {
  Pyr& P = m.pyr;
  const int len = m.q.len;
  XM_CHECK_MASK(w);
  if (len > P.cap_blocks || P.cap_levels < 2 || len > 32000) { w.fail(Q_NEED_MORE); return false; }
#if defined(__CUDA_ARCH__)
  const int lane = (int)(threadIdx.x & 31);
  const unsigned lt_mask = (1u << lane) - 1u;
  bool amb = false;
  XM_NOUNROLL
  for (int k = lane; k < len; k += 32) {
    uint8_t code = m.q.at(k);
    amb |= bp_is_ambiguous(code);
    P.blk[k] = base_block16(code, k); P.child[k] = -1; P.up[k] = -1;
  }
  // The lanes leave the loop after different trip counts.  A vote synchronises them for the vote only; what follows (the scalar
  // MultiHashBlock build in particular) is executed by every lane on the same warp-shared state and needs the warp CONVERGED.
  __syncwarp();
  XM_CHECK_MASK(w);
  amb = __any_sync(0xffffffffu, amb);
  XM_CHECK_MASK(w);
#else
  bool amb = false;
  for (int k = 0; k < len; k++) {
    uint8_t code = m.q.at(k);
    amb |= bp_is_ambiguous(code);
    P.blk[k] = base_block16(code, k); P.child[k] = -1; P.up[k] = -1;
  }
#endif
  P.level_off[0] = 0; P.level_off[1] = len; P.n_levels = 1;
  P.opt = nullptr; P.n_opt = 0; P.cap_opt = 0;
  if (amb) return pyr_build_ambiguous(w, m);  // IUPAC-ambiguous query bases: MultiHashBlocks, scalar build
  int prev_off = 0, n_prev = len, level = 1;
  XM_NOUNROLL
  while (n_prev >= 2) {
    if (level >= P.cap_levels) { w.fail(Q_NEED_MORE); return false; }
    const int cur_off = prev_off + n_prev;
    int n_new = 0;
#if defined(__CUDA_ARCH__)
    __syncwarp();
    XM_NOUNROLL
    for (int base = 0; base < n_prev - 1; base += 32) {
      const int i = base + lane;
      const bool valid = i < n_prev - 1;
      bool keep = false;
      HB16 L, R;
      if (valid) {
        L = P.blk[prev_off + i]; R = P.blk[prev_off + i + 1];
        keep = ((int)L.start + (int)L.len >= (int)R.start) && ((L.flags & 2) || (R.flags & 1));  // shouldMergeBlocks :200-208
      }
      const unsigned mask = __ballot_sync(0xffffffffu, keep);
      const int total = __popc(mask);
      if (cur_off + n_new + total > P.cap_blocks) { w.fail(Q_NEED_MORE); return false; }
      const int pos = n_new + __popc(mask & lt_mask);
      if (keep) { P.blk[cur_off + pos] = merge_blocks16(L, R); P.child[cur_off + pos] = (int16_t)i; P.up[cur_off + pos] = -1; }
      if (valid) P.up[prev_off + i] = keep ? (int16_t)pos : (int16_t)-1;
      n_new += total;
    }
    __syncwarp();
#else
    for (int i = 0; i < n_prev - 1; i++) {
      const HB16 L = P.blk[prev_off + i], R = P.blk[prev_off + i + 1];
      bool keep = ((int)L.start + (int)L.len >= (int)R.start) && ((L.flags & 2) || (R.flags & 1));
      if (keep) {
        if (cur_off + n_new + 1 > P.cap_blocks) { w.fail(Q_NEED_MORE); return false; }
        P.blk[cur_off + n_new] = merge_blocks16(L, R); P.child[cur_off + n_new] = (int16_t)i; P.up[cur_off + n_new] = -1;
        P.up[prev_off + i] = (int16_t)n_new;
        n_new++;
      } else P.up[prev_off + i] = -1;
    }
#endif
    if (n_new == 0) break;
    P.level_off[level + 1] = cur_off + n_new; P.n_levels = level + 1;
    prev_off = cur_off; n_prev = n_new; level++;
  }
  return true;
}

// ---------------- index reads (Readable_HashBlock_Database / PackedMap) ----------------
XM_HD inline bool ix_table(WS& w, int used, const TableD*& t) {
  if (used > w.ix->max_built) { w.fail(Q_INDEX_TOO_SHORT); return false; }
  t = &w.ix->tables[used];
  return true;
}
XM_INLINE uint64_t ix_bucket(const TableD& t, int32_t key) {
  int r = key % t.capacity;
  if (r < 0) r += t.capacity;
  return t.buckets[r];
}
XM_HD inline int ix_num_matches_lower_bound(WS& w, const HB& b) {  // Readable_HashBlock_Database.java:72-80
  if (b.used < w.ix->min_interesting) return JMAX;
  const TableD* t;
  if (!ix_table(w, b.used, t)) return JMAX;
  w.st_probes++;
  if (t->buckets == nullptr) return 0;
  uint64_t word = ix_bucket(*t, b.lookup_key());
  if ((word >> 16) & 1) return JMAX;
  return (int)(word & 0xFFFF);
}
XM_HD inline int ix_max_num_matches_allowed(WS& w, const HB& b) {  // :82-90
  if (b.used < w.ix->min_interesting) return -1;
  const TableD* t;
  if (!ix_table(w, b.used, t)) return 0;
  return t->max_count;
}

// ---------------- HashBlockPath ----------------
XM_HD inline void path_init(WS& w, MatePath& m) {
  m.batch_index = -1; m.cur_valid = 1; m.cur_idx = -1;
  HB d; d.start = 0; d.len = 0; d.used = 0; d.fwd = 0; d.rev = 0; d.gap_dir = 0; d.flags = 0; d.extra = 0; d.ident = -1;  // new HashBlock(0, 0)
  m.cur = d; m.have_gapmer = 0; m.have_prev = 0; m.have_prevprev = 0; m.prev_fwd = 0; m.prevprev_fwd = 0; m.gapmer_serial = 0;
}
XM_HD inline bool path_with_gap(WS& w, MatePath& m, HB& out) {  // :197-203
  if (!w.ix->gapmers) { out = m.cur; return true; }
  if (!m.have_gapmer) {
    HB g;
    if (!with_gap_and_extension(m.cur, m.q, g)) return false;
    if (m.cur.gap_dir != 0) g.ident = (1LL << 60) + (m.gapmer_serial++);
    m.gapmer = g; m.have_gapmer = 1;
  }
  out = m.gapmer;
  return true;
}
XM_HD inline void path_set(MatePath& m, int level, int idx) { m.batch_index = level; m.cur_idx = idx; m.cur = pyr_block(m.pyr, level, idx); m.cur_valid = 1; }
XM_HD inline void path_move_right(WS& w, MatePath& m) {  // :125-128  row.getAfter(cur.start)
  int nxt = -1;
  if (m.batch_index >= 0) {
    if (m.cur_idx >= 0) { nxt = m.cur_idx + 1; if (nxt >= pyr_level_size(m.pyr, m.batch_index)) nxt = -1; }
    else nxt = pyr_find_after(m.pyr, m.batch_index, m.cur.start);
  }
  if (nxt >= 0) path_set(m, m.batch_index, nxt); else m.cur_valid = 0;
  m.have_gapmer = 0;
}
XM_HD inline void path_move_down(WS& w, MatePath& m) {  // :99-108  the row below, first block after cur.start
  int level = m.batch_index - 1;
  int nxt;
  if (m.cur_idx >= 0) { nxt = (int)m.pyr.child[m.pyr.level_off[m.batch_index] + m.cur_idx] + 1; if (nxt >= pyr_level_size(m.pyr, level)) nxt = -1; }
  else nxt = pyr_find_after(m.pyr, level, m.cur.start);
  m.batch_index = level;
  if (nxt >= 0) path_set(m, level, nxt); else { m.cur_valid = 0; m.cur_idx = -1; }
  m.have_gapmer = 0;
}
XM_HD inline void path_move_up_or_right(WS& w, MatePath& m) {  // :111-122  the row above, block starting exactly at cur.start
  int u = -1;
  if (m.cur_idx >= 0) u = (int)m.pyr.up[m.pyr.level_off[m.batch_index] + m.cur_idx];
  else {
    int level = m.batch_index + 1;
    int f = pyr_find_after(m.pyr, level, m.cur.start - 1);
    if (f >= 0 && (int)m.pyr.blk[m.pyr.level_off[level] + f].start == m.cur.start) u = f;
  }
  if (u >= 0) { path_set(m, m.batch_index + 1, u); m.have_gapmer = 0; }
  else path_move_right(w, m);
}
XM_HD inline int path_max_allowed(WS& w, MatePath& m, const HB& b) {  // :205-219
  if (b.len >= m.q.len / 6) return ix_max_num_matches_allowed(w, b);
  if (b.rmr()) return 5;
  return b.used + 1;
}
XM_HD inline bool path_advance(WS& w, MatePath& m) {  // advanceToNextPosition :143-195 
  const HB single = m.cur;
  if (max_gapmer_used(single.len) < w.ix->min_interesting && w.ix->gapmers) path_move_up_or_right(w, m);
  else {
    HB ext;
    if (path_with_gap(w, m, ext)) {
      int num = ix_num_matches_lower_bound(w, ext);
      if (num < 6) { if (m.batch_index > 0) path_move_down(w, m); else path_move_right(w, m); }
      else if (num > path_max_allowed(w, m, ext)) path_move_up_or_right(w, m);
      else path_move_right(w, m);
    } else {
      int typical = single.len * 3 / 2;
      if (typical <= w.ix->min_interesting && w.ix->gapmers) path_move_up_or_right(w, m);
      else { if (m.batch_index > 0) path_move_down(w, m); else path_move_right(w, m); }
    }
  }
  XM_NOUNROLL
  while (m.cur_valid && (m.cur.flags & HB_MULTI)) {  // skipMultiblocks :130-140
    if (m.batch_index > 0) path_move_down(w, m); else path_move_right(w, m);
  }
  return m.cur_valid && w.status == 0;
}
XM_HD inline bool path_next_interesting_block(WS& w, MatePath& m, HB& out) {  // getNextInterestingBlock :27-50 + :68-96
  if (!m.cur_valid) return false;
  XM_NOUNROLL
  while (true) {
    if (!path_advance(w, m)) return false;
    HB ext;
    if (!path_with_gap(w, m, ext)) continue;
    if (!(ix_num_matches_lower_bound(w, ext) <= path_max_allowed(w, m, ext))) continue;
    if (w.status != 0) return false;
    // recentlySeen :52-65
    bool seen = (m.have_prev && ext.fwd == m.prev_fwd) || (m.have_prevprev && ext.fwd == m.prevprev_fwd);
    m.have_prevprev = m.have_prev; m.prevprev_fwd = m.prev_fwd; m.have_prev = 1; m.prev_fwd = ext.fwd;
    if (seen) continue;
    out = ext;
    return true;
  }
}

// ---------------- Counting_HashBlockPath ----------------
XM_HD inline void counter_update(MatePath& m, Counter& c, const WS& w) {  // HashBlockMatch_Counter.update :50-55,83-97
  int blen = w.ref->len[c.contig];
  XM_NOUNROLL
  while (c.hist_processed < m.n_hist) {
    const Hist& h = m.history[c.hist_processed];
    if (!(c.has_last && h.ident == c.last_matched_ident)) {
      if (h.start >= c.last_mismatched_pos) {
        if (c.offset + h.end <= blen) { c.num_distinct++; c.last_mismatched_pos = h.end; }
      }
    }
    c.hist_processed++;
  }
}
XM_HD inline void counter_declare_good(MatePath& m, Counter& c, int idx, const WS& w) {  // declareGood :282-287
  if (!c.good) { m.good[m.n_good++] = idx; c.good = 1; counter_update(m, c, w); c.priority = c.num_distinct; }
}
XM_HD inline void counting_add_match(WS& w, MatePath& m, const SM& full, const HB& qb, int ci, int qb_num_matches) {  // addMatch :254-279
  Counter& c = m.counters[ci];
  c.num_matches++; c.has_last = 1; c.last_matched_ident = qb.ident;
  counter_update(m, c, w);
  if (c.num_matches <= 1) {
    if (c.num_matches == 1) { m.found_good = 1; counter_declare_good(m, c, ci, w); }
    else if (qb_num_matches <= qb.len) {
      int from_start = full.offset;
      int from_end = w.ref->len[full.contig] - (full.offset + w.query.seq[full.mate].len);
      if (imin(from_start, from_end) < 0) counter_declare_good(m, c, ci, w);
    }
  }
}
XM_FN void counting_update_matches(WS& w, MatePath& m, const SM& sm, const HB& qb, int qb_num_matches) {  // updateMatches :193-252
  XM_CHECK_MASK(w);
  int set = sm.rev ? 0 : 1;  // reversed matches live in "forwardMatchCounters" (:197-200, SURVEY §9-5)
  int cur = -1, lower = -1, higher = -1;
  XM_NOUNROLL
  for (int i = 0; i < m.n_counters; i++) {
    const Counter& c = m.counters[i];
    if (c.set != set || c.contig != sm.contig) continue;
    if (c.offset == sm.offset) { cur = i; break; }
    if (c.offset < sm.offset) { if (lower < 0 || c.offset > m.counters[lower].offset) lower = i; }
    else { if (higher < 0 || c.offset < m.counters[higher].offset) higher = i; }
  }
  if (cur < 0) {
    if (m.n_counters >= m.cap_counters) { w.fail(Q_NEED_MORE); return; }
    cur = m.n_counters++;
    Counter& c = m.counters[cur];
    c.set = set; c.contig = sm.contig; c.offset = sm.offset;
    c.num_matches = 0; c.num_distinct = m.n_nonoverlap_visited; c.last_mismatched_pos = qb.start;
    c.has_last = 0; c.last_matched_ident = 0; c.hist_processed = m.n_hist - 1; c.good = 0; c.priority = 0; c.next = -1; c.prev = -1;
    if (lower >= 0 && iabs(m.counters[lower].offset - sm.offset) <= m.max_indel_consider) { c.prev = lower; m.counters[lower].next = cur; }
    if (higher >= 0 && iabs(m.counters[higher].offset - sm.offset) <= m.max_indel_consider) { c.next = higher; m.counters[higher].prev = cur; }
  }
  int pc = m.counters[cur].prev, nc = m.counters[cur].next;
  if (pc >= 0) counting_add_match(w, m, sm, qb, pc, qb_num_matches);
  if (nc >= 0) counting_add_match(w, m, sm, qb, nc, qb_num_matches);
  bool update_this = true;
  if ((pc >= 0 && m.counters[pc].good) || (nc >= 0 && m.counters[nc].good)) { if (!m.counters[cur].good) update_this = false; }
  if (update_this) counting_add_match(w, m, sm, qb, cur, qb_num_matches);
}
// key order of tryEnsureGoodMatchCounter / getAllPositions: set 0 first, then contig, then offset (TreeMap)
XM_INLINE bool counter_key_less(const Counter& a, const Counter& b) {
  if (a.set != b.set) return a.set < b.set;
  if (a.contig != b.contig) return a.contig < b.contig;
  return a.offset < b.offset;
}
XM_HD inline int counters_next_sorted(const MatePath& m, int n, int after) {  // smallest key greater than counters[after] among [0, n)
  int best = -1;
  XM_NOUNROLL
  for (int i = 0; i < n; i++) {
    if (after >= 0 && !counter_key_less(m.counters[after], m.counters[i])) continue;
    if (best < 0 || counter_key_less(m.counters[i], m.counters[best])) best = i;
  }
  return best;
}
XM_FN void counting_try_ensure_good(WS& w, MatePath& m) {  // :292-308
  XM_CHECK_MASK(w);
  if (!m.found_good && m.n_counters <= m.q.len) {
    int after = -1;
    XM_NOUNROLL
    while (true) {
      int i = counters_next_sorted(m, m.n_counters, after);
      if (i < 0) break;
      counter_declare_good(m, m.counters[i], i, w);
      after = i;
    }
    m.found_good = 1;
  }
}
XM_HD inline bool counting_next_block(WS& w, MatePath& m, HB& out) {  // getNextInterestingBlock :344-368
  m.pa_valid = 0;
  XM_NOUNROLL
  while (true) {
    HB b;
    if (!path_next_interesting_block(w, m, b)) {
      if (w.status != 0) return false;
      if (m.pend_cnt < 1) return false;
      out = m.pending[m.pend_head]; m.pend_head = (m.pend_head + 1) % m.cap_pend; m.pend_cnt--;
      return true;
    }
    if (b.start < m.max_nonoverlap_visited) {
      if (m.pend_cnt >= m.cap_pend) { w.fail(Q_NEED_MORE); return false; }
      m.pending[(m.pend_head + m.pend_cnt) % m.cap_pend] = b; m.pend_cnt++;
      continue;
    }
    out = b;
    return true;
  }
}
// One index hit of seed qb at global position pos: decode, flank verification (Counting_HashBlockPath.step :98-153)
// and the resulting SequenceMatch (:155-166).  mate < 0 = rejected.
XM_FN SM verify_hit(const WS& w, const MatePath& m, const HB& qb, int64_t pos, bool invert) {
  SM full; full.mate = -1; full.rev = 0; full.contig = 0; full.offset = 0; full.from_hash = 1;
  int seq_id, rstart;
  w.ref->decode(pos, seq_id, rstart);
  if (invert) { seq_id ^= 1; rstart = w.ref->len[seq_id >> 1] - rstart - qb.len; }
  const int contig = seq_id >> 1, on_rc = seq_id & 1;
  const SeqView cms = w.ref->contig(contig, on_rc);
  const int qlen = m.q.len;
  int mism = 0, mat = 0;
  XM_NOUNROLL
  for (int d = 1; d < 20; d++) {
    int qi = qb.start - d;
    if (qi >= 0 && qi < qlen) {
      int ri = rstart - d;
      if (ri >= 0 && ri < cms.len) { if (!bp_can_match(m.q.at(qi), cms.at(ri))) mism++; else mat++; }
    }
    qi = qb.start + qb.len - 1 + d;
    if (qi >= 0 && qi < qlen) {
      int ri = rstart + qb.len - 1 + d;
      if (ri >= 0 && ri < cms.len) { if (!bp_can_match(m.q.at(qi), cms.at(ri))) mism++; else mat++; }
    }
    if (mat < mism) break;
    if (mat >= mism + qb.used) break;
  }
  XM_T("  hit seq=%d rstart=%d mism=%d mat=%d\n", seq_id, rstart, mism, mat);
  if (mism > mat) return full;
  full.mate = m.mate; full.contig = contig;
  if (on_rc) {  // :155-166
    int rq = qlen - qb.end();
    int rr = cms.len - (rstart + qb.len);
    full.rev = m.path_is_rc ? 0 : 1;  // a = reverseComplementQuery
    full.offset = rr - rq;
  } else { full.rev = m.path_is_rc ? 1 : 0; full.offset = rstart - qb.start; }
  return full;
}
XM_FN bool counting_step(WS& w, MatePath& m) {  // step :40-179
  XM_CHECK_MASK(w);
  if (m.done || w.status != 0) return false;
  PhaseClock pc_(&w.st_cyc[0]);
  HB qb;
  const TableD* t = nullptr;
  uint64_t word = 0;
  int count = 0;
  XM_NOUNROLL
  while (true) {  // getNextInterestingMatch :371-388 + matchBlock (Readable_HashBlock_Database.java:22-38)
    if (!counting_next_block(w, m, qb)) {
      if (w.status != 0) return false;
      m.done = 1;
      if (m.n_blocks_anywhere < 1) counting_try_ensure_good(w, m);
      return false;
    }
    if (qb.used < w.ix->min_interesting) continue;  // null
    if (!ix_table(w, qb.used, t)) return false;
    if (t->buckets == nullptr) { count = 0; break; }
    word = ix_bucket(*t, qb.lookup_key());
    if ((word >> 16) & 1) continue;  // too many matches => null
    count = (int)(word & 0xFFFF);
    if (count > t->max_count) continue;
    break;
  }
  if (m.n_hist >= m.cap_hist) { w.fail(Q_NEED_MORE); return false; }
  XM_T("seed start=%d len=%d used=%d fwd=%d rev=%d count=%d invert=%d\n", qb.start, qb.len, qb.used, qb.fwd, qb.rev, count, (int)!qb.primary());
  Hist hh; hh.start = qb.start; hh.end = qb.end(); hh.ident = qb.ident;
  m.history[m.n_hist++] = hh;
  w.st_seeds++; w.st_hits += (unsigned long long)count;
  bool invert = !qb.primary();
  const int64_t pos0 = (int64_t)(word >> 24);   // first position of the bucket
  // Each hit is verified independently (flank comparison, :98-153); the bins are then updated in bucket order.
  // On the device 32 lanes verify 32 hits at a time and lane results are replayed in order by the whole warp.
#if defined(__CUDA_ARCH__)
  const int lane = (int)(threadIdx.x & 31);
  XM_NOUNROLL
  for (int base = 0; base < count; base += 32) {
    const int n = imin(32, count - base);
    SM mine; mine.mate = -1; mine.rev = 0; mine.contig = 0; mine.offset = 0; mine.from_hash = 1;
    if (lane < n) mine = verify_hit(w, m, qb, t->position(pos0 + base + lane), invert);
    __syncwarp();   // back from the divergent call: the replay below updates warp-shared state with every lane
    XM_NOUNROLL
    for (int j = 0; j < n; j++) {
      SM full;
      full.mate = __shfl_sync(0xffffffffu, mine.mate, j);
      if (full.mate < 0) continue;
      full.rev = __shfl_sync(0xffffffffu, mine.rev, j); full.contig = __shfl_sync(0xffffffffu, mine.contig, j);
      full.offset = __shfl_sync(0xffffffffu, mine.offset, j); full.from_hash = 1;
      counting_update_matches(w, m, full, qb, count);
      if (w.status != 0) return false;
    }
  }
#else
  for (int k = 0; k < count; k++) {
    SM full = verify_hit(w, m, qb, t->position(pos0 + k), invert);
    if (full.mate < 0) continue;
    counting_update_matches(w, m, full, qb, count);
    if (w.status != 0) return false;
  }
#endif
  if (qb.start >= m.max_nonoverlap_visited) { m.max_nonoverlap_visited = qb.end(); m.n_nonoverlap_visited++; }
  m.n_blocks_anywhere++;
  m.min_num_distinct = -1;
  return true;
}

// ---- lazily evaluated counter lists ----
// kind 0: good[0..G) with priority <= k     (findGoodPositionsHavingPriorityUpTo :406-433)
// kind 2: good[0..G) with numDistinct <= k  (getBestMatches :471-493)
// kind 1: all counters [0..G) in key order  (getAllPositions :435-452)
XM_FN int list_next(WS& w, MatePath& m, const CL& l, int& cursor) {  // cursor starts at -1; returns counter index or -1
  if (l.kind == 1) { int i = counters_next_sorted(m, l.G, cursor); cursor = i; return i; }
  XM_NOUNROLL
  for (int i = cursor + 1; i < l.G; i++) {
    Counter& c = m.counters[m.good[i]];
    bool take;
    if (l.kind == 0) take = c.priority <= l.k;
    else { counter_update(m, c, w); take = c.num_distinct <= l.k; }
    if (take) { cursor = i; return m.good[i]; }
  }
  cursor = l.G;
  return -1;
}
XM_FN int list_size(WS& w, MatePath& m, const CL& l) {
  if (l.kind == 1) return l.G;
  int n = 0, cur = -1;
  XM_NOUNROLL
  while (list_next(w, m, l, cur) >= 0) n++;
  return n;
}
XM_FN CL counting_find_good_up_to(WS& w, MatePath& m, int priority) {  // :406-433
  XM_NOUNROLL
  while (true) {
    if (m.n_nonoverlap_visited >= wadd(priority, 1)) break;
    if (!counting_step(w, m)) break;
  }
  if (m.ph_valid && m.ph.size == m.n_good) return m.ph;
  CL l; l.id = w.next_list_id++; l.kind = 0; l.G = m.n_good; l.k = priority; l.size = 0;
  l.size = list_size(w, m, l);
  m.ph = l; m.ph_valid = 1;
  return l;
}
XM_HD inline CL counting_all_positions(WS& w, MatePath& m) {
  if (!m.pa_valid) { CL l; l.id = w.next_list_id++; l.kind = 1; l.G = m.n_counters; l.k = 0; l.size = m.n_counters; m.pa = l; m.pa_valid = 1; }
  return m.pa;
}
XM_FN CL counting_best_matches(WS& w, MatePath& m) {  // getBestMatches :471-493 + getNumGoodDistinctMismatches :458-470
  CL l; l.id = w.next_list_id++; l.kind = 2; l.G = 0; l.k = 0; l.size = 0;
  if (m.n_blocks_anywhere < 1) return l;
  if (m.min_num_distinct < 0) {
    int mn = m.n_nonoverlap_visited - 1;
    XM_NOUNROLL
    for (int i = 0; i < m.n_good; i++) { Counter& c = m.counters[m.good[i]]; counter_update(m, c, w); if (mn >= c.num_distinct) mn = c.num_distinct; }
    m.min_num_distinct = mn;
  }
  l.G = m.n_good; l.k = m.min_num_distinct;
  l.size = list_size(w, m, l);
  return l;
}

// ---------------- HashBlockPaths_Counter ----------------
XM_HD inline int pc_count_priority(WS& w, const QM& q) {  // countPriority :314-334
  const Counter& c1 = w.mp[0].counters[q.c[0]]; const Counter& c2 = w.mp[1].counters[q.c[1]];
  SM m1 = counter_match(w.mp[0], c1), m2 = counter_match(w.mp[1], c2);
  if (sm_start_b(w, m1) < sm_end_b(w, m2) && sm_end_b(w, m1) > sm_start_b(w, m2)) return imax(imax(0, c1.priority), c2.priority);
  return c1.priority + c2.priority;
}
// matchWithoutCache :136-246 + assembleQueryMatches :248-265
XM_FN void pc_match_without_cache(WS& w, const CL* lists, int n_lists) {
  XM_CHECK_MASK(w);
  w.n_assembled = 0;
  if (n_lists == 1) {
    int cur = -1, ci;
    XM_NOUNROLL
    while ((ci = list_next(w, w.mp[0], lists[0], cur)) >= 0) {
      if (w.n_assembled >= w.cap_assembled) { w.fail(Q_NEED_MORE); return; }
      QM q; q.c[0] = ci; q.c[1] = -1; q.priority = w.mp[0].counters[ci].priority; q.hint = 0;
      w.assembled[w.n_assembled++] = q;
    }
    return;
  }
  bool last_largest = lists[0].size <= lists[1].size;
  int first_ci = last_largest ? 0 : 1, second_ci = 1 - first_ci;
  MatePath& A = w.mp[first_ci]; MatePath& B = w.mp[second_ci];
  long long mark = w.scratch_top;
  int na = lists[first_ci].size;
  int* a_idx = (int*)w.salloc((long long)sizeof(int) * (na > 0 ? na : 1));
  int* near = (int*)w.salloc((long long)sizeof(int) * (na > 0 ? na : 1));
  if (w.status != 0) return;
  { int cur = -1, ci, k = 0; while ((ci = list_next(w, A, lists[first_ci], cur)) >= 0 && k < na) a_idx[k++] = ci; na = k; }
  int cur = -1, cb;
  XM_NOUNROLL
  while ((cb = list_next(w, B, lists[second_ci], cur)) >= 0) {
    const Counter& c = B.counters[cb];
    bool b_rev = (c.set == 0);
    bool b_qrev = (b_rev == (second_ci % 2 == 0));
    int max_reverse = B.q.len / 2;
    int s0, s1;
    bool other_earlier = (b_qrev == last_largest);
    if (other_earlier) { s0 = c.offset - max_reverse; s1 = c.offset + w.pc_max_offset_between; }
    else { s0 = c.offset - w.pc_max_offset_between; s1 = c.offset + max_reverse; }
    int nn = 0;
    XM_NOUNROLL
    for (int k = 0; k < na; k++) {
      const Counter& a = A.counters[a_idx[k]];
      bool a_qrev = ((a.set == 0) == (first_ci % 2 == 0));
      if (a_qrev != b_qrev || a.contig != c.contig) continue;
      if (a.offset < s0 || a.offset > s1) continue;
      int j = nn++;  // insertion sort by offset ascending
      XM_NOUNROLL
      while (j > 0 && A.counters[near[j - 1]].offset > a.offset) { near[j] = near[j - 1]; j--; }
      near[j] = a_idx[k];
    }
    bool desc = b_qrev && nn > 1;
    XM_NOUNROLL
    for (int t = 0; t < nn; t++) {
      int ai = near[desc ? nn - 1 - t : t];
      if (w.n_assembled >= w.cap_assembled) { w.fail(Q_NEED_MORE); w.scratch_top = mark; return; }
      QM q;
      if (last_largest) { q.c[0] = ai; q.c[1] = cb; } else { q.c[0] = cb; q.c[1] = ai; }
      Counter& g0 = w.mp[0].counters[q.c[0]]; Counter& g1 = w.mp[1].counters[q.c[1]];
      counter_update(w.mp[0], g0, w); counter_update(w.mp[1], g1, w);
      q.hint = g0.num_distinct < g1.num_distinct ? 1 : 0;
      q.priority = pc_count_priority(w, q);
      w.assembled[w.n_assembled++] = q;
    }
  }
  w.scratch_top = mark;
}
XM_HD inline void pc_match(WS& w, const CL* lists, int n_lists) {  // match :116-133 (list identity cache, SURVEY §9-18)
  bool same = w.pc_have_prev != 0;
  if (same) for (int i = 0; i < n_lists; i++) if (w.pc_prev_ids[i] != lists[i].id) { same = false; break; }
  if (!same) {
    pc_match_without_cache(w, lists, n_lists);
    XM_NOUNROLL
    for (int i = 0; i < n_lists; i++) w.pc_prev_ids[i] = lists[i].id;
    w.pc_have_prev = 1;
  }
}
XM_FN void pc_find_good_up_to(WS& w, int k) {  // findGoodPositionsWithPriorityUpTo :52-82
  XM_CHECK_MASK(w);
  CL lists[2];
  int n = w.query.n_seqs;
  XM_NOUNROLL
  for (int i = 0; i < n; i++) {
    lists[i] = counting_find_good_up_to(w, w.mp[i], k);
    if (lists[i].size >= 1) w.pc_found_nonempty = 1;
  }
  if (w.status != 0) return;
  pc_match(w, lists, n);
}
// optimisticGetBestMatches :84-98; returns the priority to filter on (filterMatchesHavingMinPriority selects the MAX, §9-5)
XM_FN int pc_optimistic_best(WS& w) {
  CL lists[2];
  int n = w.query.n_seqs;
  XM_NOUNROLL
  for (int i = 0; i < n; i++) {
    XM_NOUNROLL
    while (true) {
      CL best = counting_best_matches(w, w.mp[i]);
      if (best.size == 1 || !counting_step(w, w.mp[i])) { lists[i] = best; break; }
    }
    if (w.status != 0) return -1;
  }
  pc_match(w, lists, n);
  int mn = -1;
  XM_NOUNROLL
  for (int i = 0; i < w.n_assembled; i++) if (mn < 0 || mn < w.assembled[i].priority) mn = w.assembled[i].priority;
  return mn;
}
XM_FN bool pc_find_partially_good(WS& w) {  // findPartiallyGoodPositions :26-50; false = empty list
  XM_CHECK_MASK(w);
  if (w.query.n_seqs != 2) return false;
  if (!w.pc_found_nonempty) return false;
  CL lists[2];
  bool good = false, bad = false;
  XM_NOUNROLL
  for (int i = 0; i < 2; i++) {
    CL here = counting_find_good_up_to(w, w.mp[i], JMAX);
    if (here.size == 0) { bad = true; here = counting_all_positions(w, w.mp[i]); } else good = true;
    lists[i] = here;
  }
  if (w.status != 0) return false;
  if (good && bad) { pc_match(w, lists, 2); return true; }
  return false;
}
XM_HD inline int pc_num_blocks(const WS& w) { int t = 0; for (int i = 0; i < w.query.n_seqs; i++) t += w.mp[i].n_blocks_anywhere; return t; }

// QueryMatch helpers (M/QueryMatch.java)
XM_HD inline SM qm_comp(const WS& w, const QM& q, int i) {
  const MatePath& m = w.mp[i];
  const Counter& c = m.counters[q.c[i]];
  SM s; s.mate = i; s.rev = (c.set == 0) ? 1 : 0; s.contig = c.contig; s.offset = c.offset; s.from_hash = 1;
  return s;
}
XM_INLINE bool qm_same_position(const QM& a, int na, const QM& b, int nb) {  // samePosition :83-95 (counters are unique per position)
  if (na != nb) return false;
  XM_NOUNROLL
  for (int i = 0; i < na; i++) if (a.c[i] != b.c[i]) return false;
  return true;
}

}  // namespace xm
