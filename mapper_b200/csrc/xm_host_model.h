// xmapper_b200 — host-side model behind the C ABI: reference, per-length bucket tables in the device layout,
// duplication table; plus the library's own index builder and duplication detector (reference-time
// preprocessing, multi-threaded C++; the device-side builder is a later row of SURVEY.md §8f).
// No CUDA in this header: xm_capi.cu mirrors these arrays to the GPU.
//
// Index builder follows M/HashBlock_Database.java:490-665 (which blocks exist, gapmer extension, per-length
// capacity estimate, per-bucket cap, polarity), M/PackedMap.java:99-153 and QV/ByteKeyStore.java (sorted bucket,
// overfull bucket dropped).  Duplication detector follows M/DuplicationDetector.java:129-436.
#pragma once
#include "xm_seed.h"
#include <vector>
#include <string>
#include <map>
#include <set>
#include <thread>
#include <atomic>
#include <algorithm>
#include <cmath>
#include <cstring>

namespace xm {

struct HostTable {
  int capacity = 1, max_count = 1;
  std::vector<uint64_t> buckets;   // empty => PackedMap(1,1)
  std::vector<uint32_t> positions;     // low 32 bits
  std::vector<uint8_t> positions_hi;   // bits 32-39; empty while the reference's forward + reverse size fits 32 bits
  int64_t position(size_t i) const { return (int64_t)positions[i] | (positions_hi.empty() ? 0 : ((int64_t)positions_hi[i] << 32)); }
};

struct HostModel {
  Params prm{};
  int gapmers = 1;
  // reference
  int n_contigs = 0;
  std::vector<uint16_t> words;
  std::vector<int64_t> word_off;
  std::vector<int32_t> len;
  std::vector<int64_t> gstart;
  int64_t total_forward = 0, total_fr = 0;
  int64_t position_bias = 0;   // global position of the first contig (0 in production; tests move the reference past 2^32 with it)
  int64_t position_end = 0;    // one past the last global position (= position_bias + total_fr)
  bool wide_positions() const { return position_end > (1LL << 32); }
  bool ref_ambiguous = false;
  // index
  std::vector<HostTable> tables;
  int min_interesting = 1, max_built = 0;
  bool index_finished = false;
  // duplications
  int dup_window = 1; double dup_granularity = 1;
  std::vector<std::vector<int32_t>> dup_starts;
  bool dup_set = false;
  uint64_t dup_generation = 0;   // bumped by changes of the duplication table alone (mirror_model re-uploads only that)
  uint64_t generation = 0;  // bumped on every change so the device mirror knows to refresh

  SeqView contig_view(int c, int rc) const { SeqView v; v.w = words.data() + word_off[c]; v.len = len[c]; v.rc = rc; v.bytes = nullptr; return v; }

  void set_reference(int n, const uint16_t* const* packed4, const int32_t* lengths) {
    n_contigs = n; words.clear(); word_off.assign(n, 0); len.assign(lengths, lengths + n); gstart.assign(2 * (size_t)n + 1, 0);
    total_forward = 0; ref_ambiguous = false;
    for (int c = 0; c < n; c++) {
      size_t w0 = (words.size() + 7) & ~(size_t)7;  // 16-byte aligned contig starts
      words.resize(w0, 0);
      word_off[c] = (int64_t)w0;
      size_t nw = ((size_t)lengths[c] + 3) / 4;
      words.insert(words.end(), packed4[c], packed4[c] + nw);
      total_forward += lengths[c];
    }
    words.resize((words.size() + 15) & ~(size_t)7, 0);
    int64_t g = position_bias;
    for (int c = 0; c < n; c++) { gstart[2 * c] = g; g += lengths[c]; gstart[2 * c + 1] = g; g += lengths[c]; }
    gstart[2 * (size_t)n] = g; position_end = g; total_fr = g - position_bias;
    reference_codes_changed();
  }
  // after the codes of the reference changed (set_reference, or the "-anc" reference written over it): everything derived from them is gone
  void reference_codes_changed() {
    ref_ambiguous = false;
    for (int c = 0; c < n_contigs && !ref_ambiguous; c++) { SeqView v = contig_view(c, 0); for (int i = 0; i < v.len; i++) if (bp_is_ambiguous(v.at(i))) { ref_ambiguous = true; break; } }
    tables.clear(); max_built = 0; index_finished = false; dup_starts.assign((size_t)n_contigs, {}); dup_set = false; dup_generation++;
    generation++;
  }

  static uint64_t bucket_word(int64_t start, bool overfull, int count) { return ((uint64_t)start << 24) | ((uint64_t)(overfull ? 1 : 0) << 16) | (uint64_t)(count & 0xFFFF); }

  // positions: uint32 (wide64 false) or uint64 (wide64 true) global positions
  void set_index_length(int n_used, int capacity, int max_count, const int64_t* offsets, const uint8_t* overfull, const void* positions, bool wide64 = false) {
    if ((int)tables.size() <= n_used) tables.resize((size_t)n_used + 1);
    HostTable& T = tables[(size_t)n_used];
    T.capacity = capacity < 1 ? 1 : capacity; T.max_count = max_count;
    T.buckets.clear(); T.positions.clear(); T.positions_hi.clear();
    int64_t total = offsets ? offsets[capacity] : 0;
    if (offsets) {
      T.buckets.resize((size_t)T.capacity);
      for (int b = 0; b < capacity; b++) T.buckets[(size_t)b] = bucket_word(offsets[b], overfull && overfull[b], (int)(offsets[b + 1] - offsets[b]));
      if (!wide64) { const uint32_t* p = (const uint32_t*)positions; T.positions.assign(p, p + total); if (wide_positions()) T.positions_hi.assign((size_t)total, 0); }
      else {
        const uint64_t* p = (const uint64_t*)positions;
        T.positions.resize((size_t)total);
        if (wide_positions()) T.positions_hi.resize((size_t)total);
        for (int64_t i = 0; i < total; i++) { T.positions[(size_t)i] = (uint32_t)p[i]; if (wide_positions()) T.positions_hi[(size_t)i] = (uint8_t)(p[i] >> 32); }
      }
    }
    generation++;
  }
  void finish_index(int min_int, int built) {
    min_interesting = min_int; max_built = built;
    if ((int)tables.size() <= built) tables.resize((size_t)built + 1);
    index_finished = true; generation++;
  }

  // ---- the library's own index builder ----
  static int log2_round_up(long long value) { int nb = 1; long long e = 2; while (true) { if (e >= value) return nb; nb++; e *= 2; } }
  int choose_min_dup_len() const { return log2_round_up(total_forward); }
  int estimate_capacity(int n) const {  // HashBlock_Database.estimateRequiredCapacity :620-665
    int anchor = gapmers ? n * 2 / 3 : n;
    double size_p = std::min(1.0, 2.0 / anchor), off_p = std::min(1.0, 2.0 / anchor);
    double poss = size_p * off_p;
    long long max_seqs = (n <= 16) ? (1LL << (n * 2)) : (1LL << 32);
    long long max_stored = max_seqs / 2;
    double mh = (double)max_stored * poss;
    long long max_hashcodes = mh >= 9.2233720368547758e18 ? INT64_MAX : (long long)mh;
    long long num_blocks = (long long)((double)total_forward * poss);
    double existence = 1 - std::pow((double)((double)max_hashcodes - 1.0) / (double)max_hashcodes, (double)num_blocks);
    int unique = j2i((double)max_hashcodes * existence);
    if (unique % 2 == 0) unique++;
    return unique;
  }
  static int max_count_for(int n, int max_short) { int m = n * n; if (m < max_short) m = max_short; if (m > 32766) m = 32766; if (m < 1) m = 1; return m; }

  struct Entry { uint32_t bucket; uint64_t pos; };

  // what both index builders start from: minInterestingSize :51-55 (or the one a caller passes, :68-89), the longest length built and
  // the capacity per length
  bool index_plan(int max_used, int& hi, std::vector<int>& cap, std::string& err, int min_interesting_size = -1) {
    min_interesting = min_interesting_size > 0 ? min_interesting_size : j2i(std::max((std::log((double)(total_forward + 1)) / std::log(4.0)) - 2, 1.0));
    hi = std::max(max_used, 2 * choose_min_dup_len());
    cap.assign((size_t)hi + 1, 1);
    for (int n = 1; n <= hi; n++) { int c = estimate_capacity(n); cap[(size_t)n] = c < 1 ? 1 : c; }
    return true;
  }
  // Blocks of an IUPAC-ambiguous stretch of the reference (an "-anc" reference, M/AncestryDetector.java:323-327): the device core's
  // MultiHashBlock pyramid (pyr_build -> pyr_build_ambiguous, M/HashBlock_ParentRow.java:69-191) over a window of the contig; calls
  // emit(block in contig coordinates, is_multi) for every block / possibility whose start lies in [s, e).
  template <class F>
  bool ambiguous_window_blocks(int contig, int s, int e, int hi, std::vector<char>& arena, std::string& err, F&& emit) const {
    SeqView full = contig_view(contig, 0);
    const int halo = 4 * hi + 256;   // a multi-block's possibilities differ in length; generous so that every possibility of a block that starts before e is complete
    const int w_end = std::min(full.len, e + halo);
    const int wlen = w_end - s;
    if (wlen > 32000) { err = "xm_build_index: hash lengths this long are not supported on IUPAC-ambiguous references (16-bit window coordinates)"; return false; }
    WS w; memset((void*)&w, 0, sizeof(WS));
    MatePath m; memset((void*)&m, 0, sizeof(MatePath));
    SeqView v; v.w = full.w + (s >> 2); v.len = wlen; v.rc = 0; v.bytes = nullptr; v.b0 = 0; v.bn = 0;   // s is a multiple of 4
    m.q = v;
    const long long cap = 10LL * wlen + 256;
    const long long lev_bytes = ((long long)(wlen + 3) * 4 + 15) & ~15LL;
    const long long need = lev_bytes + cap * 20 + 64 + (192LL << 20);
    if ((long long)arena.size() < need) arena.resize((size_t)need);
    char* p = arena.data();
    Pyr& P = m.pyr;
    P.cap_levels = wlen + 2; P.cap_blocks = (int)std::min<long long>(cap, 2000000000LL);
    P.level_off = (int32_t*)p; p += lev_bytes;
    P.blk = (HB16*)p; p += cap * 16; P.child = (int16_t*)p; p += cap * 2; P.up = (int16_t*)p; p += cap * 2;
    p += (16 - ((uintptr_t)p & 15)) & 15;
    w.scratch = p; w.scratch_size = (long long)(arena.data() + arena.size() - p) & ~15LL; w.scratch_top = 0;
    if (!pyr_build(w, m) || w.status != 0) { err = "xm_build_index: MultiHashBlock expansion of the reference ran out of workspace (status " + std::to_string(w.status) + ")"; return false; }
    for (int level = 0; level < P.n_levels; level++) {
      const int n = pyr_level_size(P, level);
      const HB16* row = P.blk + P.level_off[level];
      bool any_short = false;
      for (int i = 0; i < n; i++) {
        const HB16& c = row[i];
        if (s + (int)c.start >= e) break;
        const int k_n = pyr_num_opts(c);
        for (int k = 0; k < k_n; k++) {
          const POpt o = pyr_opt(P, c, k);
          if (!o.has) continue;
          if ((int)o.hb.len <= hi) any_short = true;
          HB b; b.start = s + o.hb.start; b.len = o.hb.len; b.used = o.hb.len; b.fwd = o.hb.fwd; b.rev = o.hb.rev; b.gap_dir = o.hb.gap_dir; b.flags = o.hb.flags; b.extra = o.hb.extra; b.ident = 0;
          emit(b, (c.flags & HB_MULTI) != 0);
        }
      }
      if (!any_short) break;
    }
    return true;
  }
  bool build_index(int max_used, int n_threads, std::string& err) {
    min_interesting = j2i(std::max((std::log((double)(total_forward + 1)) / std::log(4.0)) - 2, 1.0));  // :51-55
    int hi = std::max(max_used, 2 * choose_min_dup_len());
    std::vector<int> cap((size_t)hi + 1, 1);
    for (int n = 1; n <= hi; n++) { int c = estimate_capacity(n); cap[(size_t)n] = c < 1 ? 1 : c; }
    struct Slice { int contig, s, e; };
    std::vector<Slice> slices;
    const int slice_len = ref_ambiguous ? 8192 : 65536;
    for (int c = 0; c < n_contigs; c++) for (int s = 0; s < len[c]; s += slice_len) slices.push_back({c, s, std::min(len[c], s + slice_len)});
    int nt = std::max(1, n_threads);
    std::vector<std::vector<std::vector<Entry>>> parts((size_t)nt), multi_parts((size_t)nt);
    for (auto& p : parts) p.resize((size_t)hi + 1);
    for (auto& p : multi_parts) p.resize((size_t)hi + 1);
    std::vector<std::string> errs((size_t)nt);
    std::atomic<size_t> next(0);
    auto work = [&](int t) {
      std::vector<HB> cur, nxt;
      std::vector<char> amb_arena;
      while (true) {
        size_t si = next.fetch_add(1);
        if (si >= slices.size()) break;
        const Slice& sl = slices[si];
        SeqView seq = contig_view(sl.contig, 0);
        int ext_end = std::min(seq.len, sl.e + hi + 2);
        auto add_block = [&](const HB& b, bool is_multi) {
          HB g;
          if (gapmers) { if (!with_gap_and_extension(b, seq, g)) return; } else g = b;
          int n = g.used;
          if (n < min_interesting || n > hi) return;
          int c = cap[(size_t)n];
          bool rml = g.rml(), rmr = g.rmr();
          bool primary = (rml != rmr) ? rml : (g.fwd >= g.rev);
          bool secondary = (rml != rmr) ? rmr : (g.fwd <= g.rev);  // HashBlock.isSecondaryPolarity :339-343
          auto& dst = is_multi ? multi_parts[(size_t)t][(size_t)n] : parts[(size_t)t][(size_t)n];
          if (primary) { int r = g.fwd % c; if (r < 0) r += c; dst.push_back({(uint32_t)r, (uint64_t)(gstart[2 * sl.contig] + g.start)}); }
          if (secondary) { int r = g.rev % c; if (r < 0) r += c; dst.push_back({(uint32_t)r, (uint64_t)(gstart[2 * sl.contig + 1] + (seq.len - g.end()))}); }
        };
        if (ref_ambiguous) {
          bool amb = false;
          const int scan_end = std::min(seq.len, sl.e + 4 * hi + 256);
          for (int i = sl.s; i < scan_end && !amb; i++) amb = bp_is_ambiguous(seq.at(i));
          if (amb) {
            if (!ambiguous_window_blocks(sl.contig, sl.s, sl.e, hi, amb_arena, errs[(size_t)t], add_block)) return;
            continue;
          }
        }
        cur.clear();
        for (int i = sl.s; i < ext_end; i++) cur.push_back(base_block(seq.at(i), i));
        int level = 0;
        while (!cur.empty()) {
          bool any_short = false;
          for (const HB& b : cur) {
            if (b.start >= sl.e) break;
            if (b.len <= hi) any_short = true;
            add_block(b, false);
          }
          if (!any_short) break;
          level++;
          nxt.clear();
          for (size_t i = 0; i + 1 < cur.size(); i++) {
            const HB& L = cur[i]; const HB& R = cur[i + 1];
            if (L.end() >= R.start && (L.rmr() || R.rml())) nxt.push_back(merge_blocks(L, R, level));
          }
          cur.swap(nxt);
        }
      }
    };
    if (nt == 1) work(0);
    else { std::vector<std::thread> th; for (int t = 0; t < nt; t++) th.emplace_back(work, t); for (auto& x : th) x.join(); }
    for (auto& e : errs) if (!e.empty()) { err = e; return false; }
    tables.assign((size_t)hi + 1, HostTable());
    std::atomic<int> nn(1);
    auto fin = [&]() {
      while (true) {
        int n = nn.fetch_add(1);
        if (n > hi) break;
        size_t total = 0, total_multi = 0;
        for (int t = 0; t < nt; t++) { total += parts[(size_t)t][(size_t)n].size(); total_multi += multi_parts[(size_t)t][(size_t)n].size(); }
        HostTable& T = tables[(size_t)n];
        if (total + total_multi == 0) { T.capacity = 1; T.max_count = 1; continue; }
        T.capacity = cap[(size_t)n]; T.max_count = max_count_for(n, 5);
        std::vector<Entry> all; all.reserve(total + total_multi);
        for (int t = 0; t < nt; t++) { auto& v = parts[(size_t)t][(size_t)n]; all.insert(all.end(), v.begin(), v.end()); std::vector<Entry>().swap(v); }
        std::sort(all.begin(), all.end(), [](const Entry& a, const Entry& b) { return a.bucket != b.bucket ? a.bucket < b.bucket : a.pos < b.pos; });
        if (total_multi) {
          // PackedMap.add(preventDuplicates) :117-131: a possibility of a multi-block that is already in its bucket is skipped (plain
          // blocks are never de-duplicated among themselves)
          std::vector<Entry> mm;
          for (int t = 0; t < nt; t++) { auto& v = multi_parts[(size_t)t][(size_t)n]; mm.insert(mm.end(), v.begin(), v.end()); std::vector<Entry>().swap(v); }
          auto less = [](const Entry& a, const Entry& b) { return a.bucket != b.bucket ? a.bucket < b.bucket : a.pos < b.pos; };
          std::sort(mm.begin(), mm.end(), less);
          std::vector<Entry> keep;
          for (size_t i = 0; i < mm.size(); i++) {
            if (i > 0 && mm[i].bucket == mm[i - 1].bucket && mm[i].pos == mm[i - 1].pos) continue;
            if (std::binary_search(all.begin(), all.end(), mm[i], less)) continue;
            keep.push_back(mm[i]);
          }
          std::vector<Entry> merged(all.size() + keep.size());
          std::merge(all.begin(), all.end(), keep.begin(), keep.end(), merged.begin(), less);
          all.swap(merged);
        }
        T.buckets.assign((size_t)T.capacity, 0);
        size_t i = 0; int64_t off = 0;
        for (int b = 0; b < T.capacity; b++) {
          size_t j = i;
          while (j < all.size() && all[j].bucket == (uint32_t)b) j++;
          int64_t cnt = (int64_t)(j - i);
          if (cnt > T.max_count) T.buckets[(size_t)b] = bucket_word(off, true, 0);
          else { T.buckets[(size_t)b] = bucket_word(off, false, (int)cnt); for (size_t k = i; k < j; k++) { T.positions.push_back((uint32_t)all[k].pos); if (wide_positions()) T.positions_hi.push_back((uint8_t)(all[k].pos >> 32)); } off += cnt; }
          i = j;
        }
      }
    };
    if (nt == 1) fin();
    else { std::vector<std::thread> th; for (int t = 0; t < nt; t++) th.emplace_back(fin); for (auto& x : th) x.join(); }
    max_built = hi; index_finished = true; generation++;
    return true;
  }

  // reads a table back in the xm_set_index_length layout
  void get_index_length(int n, int& capacity, int& max_count, int64_t& n_pos, int64_t* offsets, uint8_t* overfull, uint32_t* positions, uint64_t* positions64 = nullptr) const {
    const HostTable& T = tables[(size_t)n];
    capacity = T.capacity; max_count = T.max_count; n_pos = (int64_t)T.positions.size();
    if (offsets) {
      if (T.buckets.empty()) { for (int b = 0; b <= T.capacity; b++) offsets[b] = 0; if (overfull) for (int b = 0; b < T.capacity; b++) overfull[b] = 0; }
      else {
        for (int b = 0; b < T.capacity; b++) { offsets[b] = (int64_t)(T.buckets[(size_t)b] >> 24); if (overfull) overfull[b] = (uint8_t)((T.buckets[(size_t)b] >> 16) & 1); }
        offsets[T.capacity] = n_pos;
      }
    }
    if (positions && n_pos) memcpy(positions, T.positions.data(), (size_t)n_pos * 4);
    if (positions64) for (int64_t i = 0; i < n_pos; i++) positions64[i] = (uint64_t)T.position((size_t)i);
  }

  // ---- duplication detector (DuplicationDetector.process :129-214, saveDuplications :332-400) ----
  struct Dup { int length, count; int group = -1; };   // group: the duplication group (M/Duplication.java object) when the merge keeps them
  static int compare_dups(int window, int s1, const Dup& d1, int s2, const Dup& d2) {  // :406-436
    if (window > 1) { if (s1 / window != s2 / window) return 0; }
    int e1 = s1 + d1.length, e2 = s2 + d2.length;
    if (s1 <= s2 && e1 >= e2) return 1;
    if (s1 >= s2 && e1 <= e2) return -1;
    if (window > 1) { int cd = d1.count - d2.count; if (cd != 0) return cd; if (s1 != s2) return s1 - s2; }
    return 0;
  }
  // saveDuplications :332-400 for one block: the map keeps, per window, the blocks that contain no other block
  static void dup_insert(std::map<int, Dup>& m, int window, int ds, const Dup& nd) {
    bool insert = true;
    while (true) {
      auto it = m.upper_bound(ds);
      if (it != m.begin()) { --it; int c = compare_dups(window, ds, nd, it->first, it->second); if (c > 0) { insert = false; break; } if (c < 0) { m.erase(it); continue; } }
      break;
    }
    while (true) {
      auto it = m.lower_bound(ds);
      if (it != m.end()) { int c = compare_dups(window, ds, nd, it->first, it->second); if (c > 0) { insert = false; break; } if (c < 0) { m.erase(it); continue; } }
      break;
    }
    if (insert) m[ds] = nd;
  }
  // The second half of the detector for blocks found by the device scan (xm_capi.cu: xm_dup_scan_kernel): `recs` are the forward-strand
  // blocks of every length, (length, hashcode, contig, start, count); they are merged in the reference's order - lengths ascending,
  // saveDuplications once per 10000 hashcodes, sequences and starts ascending within such a chunk, the last hashcode winning when a
  // chunk names a start twice.  Only forward-strand maps are kept: the table that is handed out (dup_starts) never reads the others.
  struct DupRecH { int32_t contig, st, count_len, hc; };   // count_len = count | length << 24
  // A member of a duplication group as the group scan (xm_dup_scan_kernel<true>) finds it: every (sequence, start) of the group on both
  // strands, sid = 2 * contig + (reverse strand), gid = the group's identity
  struct DupGrpRec { int32_t sid, st, count_len, hc, gid; };
  static int rec_group(const DupRecH&) { return -1; }
  static int rec_group(const DupGrpRec& r) { return r.gid; }
  // saveDuplications over the records of one unit (a stretch that no other unit's blocks interact with): sorts them into the reference's
  // order - lengths ascending, one saveDuplications per 10000 hashcodes, starts ascending within such a chunk, the last hashcode winning
  // when a chunk names a start twice - and returns the surviving map
  template <class R>
  static void merge_unit(R* lo, R* hi, int window, std::map<int, Dup>& m) {
    const int chunk_len = 10000;
    std::sort(lo, hi, [&](const R& a, const R& b) {
      const int la = a.count_len >> 24, lb = b.count_len >> 24;
      if (la != lb) return la < lb;
      const int ca = a.hc / chunk_len, cb = b.hc / chunk_len;
      if (ca != cb) return ca < cb;
      if (a.st != b.st) return a.st < b.st;
      return a.hc < b.hc;
    });
    for (R* r = lo; r < hi; r++) {
      if (r + 1 < hi) { const R& x = r[1]; if ((x.count_len >> 24) == (r->count_len >> 24) && x.hc / chunk_len == r->hc / chunk_len && x.st == r->st) continue; }
      dup_insert(m, window, r->st, Dup{r->count_len >> 24, r->count_len & 0xFFFFFF, rec_group(*r)});
    }
  }
  void merge_duplications(std::vector<DupRecH>& recs, int min_len, int window) {
    dup_window = window; dup_granularity = gapmers ? (double)(min_len * 5 / 8) : (double)min_len;  // :67-77
    // Units that cannot interact are merged by different threads: contigs, and - when window > 1, where compareDuplications :406-436
    // only relates blocks of one window - stretches of whole windows within a contig.
    const long long seg = window > 1 ? (long long)window * ((1000000 + window - 1) / window) : (1LL << 40);
    std::vector<long long> unit_base((size_t)n_contigs + 1, 0);
    for (int c = 0; c < n_contigs; c++) unit_base[(size_t)c + 1] = unit_base[(size_t)c] + ((long long)len[(size_t)c] + seg - 1) / seg + 1;
    const size_t n_units = (size_t)unit_base[(size_t)n_contigs];
    auto unit_of = [&](const DupRecH& r) { return (size_t)(unit_base[(size_t)r.contig] + (long long)r.st / seg); };
    std::vector<size_t> first(n_units + 1, 0);
    for (const DupRecH& r : recs) first[unit_of(r) + 1]++;
    for (size_t u = 0; u < n_units; u++) first[u + 1] += first[u];
    std::vector<DupRecH> by_unit(recs.size());
    { std::vector<size_t> at(first.begin(), first.end() - 1); for (const DupRecH& r : recs) by_unit[at[unit_of(r)]++] = r; }
    std::vector<std::vector<int32_t>> unit_starts(n_units);
    std::atomic<size_t> next(0);
    auto work = [&]() {
      while (true) {
        const size_t u = next.fetch_add(1);
        if (u >= n_units) break;
        DupRecH* lo = by_unit.data() + first[u]; DupRecH* hi = by_unit.data() + first[u + 1];
        if (lo == hi) continue;
        std::map<int, Dup> m;
        merge_unit(lo, hi, window, m);
        for (auto& e : m) unit_starts[u].push_back(e.first);
      }
    };
    unsigned hw = std::thread::hardware_concurrency();
    const int n_thr = (int)std::max<size_t>(1, std::min<size_t>(std::min(hw ? hw : 1u, 32u), recs.size() / 4096 + 1));
    if (n_thr == 1) work();
    else { std::vector<std::thread> th; for (int t = 0; t < n_thr; t++) th.emplace_back(work); for (auto& x : th) x.join(); }
    dup_starts.assign((size_t)n_contigs, {});
    for (int c = 0; c < n_contigs; c++)
      for (long long u = unit_base[(size_t)c]; u < unit_base[(size_t)c + 1]; u++) dup_starts[(size_t)c].insert(dup_starts[(size_t)c].end(), unit_starts[(size_t)u].begin(), unit_starts[(size_t)u].end());
    dup_set = true; dup_generation++;
  }
  // The same merge for the ancestry detector (window 1, M/Mapper.java:675-681): the maps of all 2 * n_contigs sequences - bounds and
  // interest are looked up in the map of a member's own sequence, which may be a reverse one - with the group of every surviving entry.
  // With window 1 a unit is a sequence.  by_seq[sid]: (start, Dup) in start order.  Leaves the handle's own duplication table alone.
  void merge_duplication_groups(const std::vector<DupGrpRec>& recs, int window, std::vector<std::vector<std::pair<int32_t, Dup>>>& by_seq) const {
    const size_t n_seqs = 2 * (size_t)n_contigs;
    std::vector<size_t> first(n_seqs + 1, 0);
    for (const DupGrpRec& r : recs) first[(size_t)r.sid + 1]++;
    for (size_t s = 0; s < n_seqs; s++) first[s + 1] += first[s];
    std::vector<DupGrpRec> by_unit(recs.size());
    { std::vector<size_t> at(first.begin(), first.end() - 1); for (const DupGrpRec& r : recs) by_unit[at[(size_t)r.sid]++] = r; }
    by_seq.assign(n_seqs, {});
    std::atomic<size_t> next(0);
    auto work = [&]() {
      while (true) {
        const size_t s = next.fetch_add(1);
        if (s >= n_seqs) break;
        if (first[s] == first[s + 1]) continue;
        std::map<int, Dup> m;
        merge_unit(by_unit.data() + first[s], by_unit.data() + first[s + 1], window, m);
        by_seq[s].assign(m.begin(), m.end());
      }
    };
    unsigned hw = std::thread::hardware_concurrency();
    const int n_thr = (int)std::max<size_t>(1, std::min<size_t>(std::min<size_t>(hw ? hw : 1u, 32u), std::min(n_seqs, recs.size() / 4096 + 1)));
    if (n_thr == 1) work();
    else { std::vector<std::thread> th; for (int t = 0; t < n_thr; t++) th.emplace_back(work); for (auto& x : th) x.join(); }
  }
  // via_merge: the blocks this scan finds go through merge_duplications (the path the device scan feeds) instead of the maps below -
  // how the CPU tests check that routine against this one
  void build_duplications(int min_len, int max_len, int min_copies, int window, bool via_merge = false) {
    std::vector<DupRecH> merge_recs;
    if (min_len < 0) min_len = choose_min_dup_len();
    if (max_len < 0) max_len = 2 * choose_min_dup_len();
    dup_window = window; dup_granularity = gapmers ? (double)(min_len * 5 / 8) : (double)min_len;  // :67-77
    std::vector<std::map<int, Dup>> all((size_t)2 * n_contigs);  // per sequence id
    auto save = [&](std::map<int, std::map<int, Dup>>& blocks) {
      for (auto& e : blocks) for (auto& pos : e.second) dup_insert(all[(size_t)e.first], window, pos.first, pos.second);
      blocks.clear();
    };
    // The per-bucket grouping (the expensive part) is independent across buckets: threads build the `blocks` of chunks of
    // 10000 buckets in parallel; the chunks are then merged in the reference's order (saveDuplications every 10000 hashcodes).
    const int chunk_len = 10000;
    unsigned hw = std::thread::hardware_concurrency();
    const int n_thr = (int)std::max(1u, std::min(hw ? hw : 1u, 32u));
    for (int bl = min_len; bl <= max_len && bl <= max_built; bl++) {
      const HostTable& T = tables[(size_t)bl];
      const int n_chunks = (T.capacity + chunk_len - 1) / chunk_len;
      std::vector<std::map<int, std::map<int, Dup>>> chunk_blocks((size_t)n_chunks);
      auto scan_chunk = [&](int ci) {
        std::map<int, std::map<int, Dup>>& blocks = chunk_blocks[(size_t)ci];
        const int hc_end = std::min(T.capacity, (ci + 1) * chunk_len);
        for (int hc = ci * chunk_len; hc < hc_end; hc++) {
          if (T.buckets.empty()) continue;
          uint64_t word = T.buckets[(size_t)hc];
          int cnt = (int)(word & 0xFFFF);
          if (((word >> 16) & 1) || cnt < min_copies) continue;
          // lookupByForwardHash :41-52: every stored position plus its reverse complement (using numBasepairsUsed as the length)
          std::map<std::string, std::set<std::pair<int, int>>> by_text;
          int prefix = (bl + 3) / 4;
          for (int k = 0; k < 2 * cnt; k++) {
            int64_t g = T.position((size_t)(word >> 24) + (size_t)(k % cnt));
            int sid = (int)(std::upper_bound(gstart.begin(), gstart.end(), g) - gstart.begin()) - 1;
            int st = (int)(g - gstart[(size_t)sid]);
            if (k >= cnt) { sid ^= 1; st = len[(size_t)(sid >> 1)] - st - bl; }
            SeqView v = contig_view(sid >> 1, sid & 1);
            std::string text; bool amb = false;
            for (int i = 0; i < prefix; i++) { uint8_t c = v.at(st + i); if (bp_is_ambiguous(c)) amb = true; text.push_back((char)c); }
            for (int i = 0; i < prefix; i++) { uint8_t c = v.at(st + bl - prefix + i); if (bp_is_ambiguous(c)) amb = true; text.push_back((char)c); }
            if (!amb) by_text[text].insert({sid, st});
          }
          for (auto& g : by_text) {
            Dup d{bl, (int)g.second.size()};
            if (d.count >= min_copies) for (auto& u : g.second) blocks[u.first][u.second] = d;
          }
        }
      };
      if (n_thr == 1 || n_chunks < 2) { for (int ci = 0; ci < n_chunks; ci++) scan_chunk(ci); }
      else {
        std::atomic<int> next_chunk(0);
        std::vector<std::thread> th;
        for (int t = 0; t < std::min(n_thr, n_chunks); t++) th.emplace_back([&]() { while (true) { int ci = next_chunk.fetch_add(1); if (ci >= n_chunks) break; scan_chunk(ci); } });
        for (auto& x : th) x.join();
      }
      for (int ci = 0; ci < n_chunks; ci++) {
        if (via_merge) { for (auto& e : chunk_blocks[(size_t)ci]) if (!(e.first & 1)) for (auto& pos : e.second) merge_recs.push_back({e.first >> 1, pos.first, pos.second.count | (bl << 24), ci * chunk_len}); }
        else save(chunk_blocks[(size_t)ci]);
      }
    }
    if (via_merge) { merge_duplications(merge_recs, min_len, window); return; }
    dup_starts.assign((size_t)n_contigs, {});
    for (int c = 0; c < n_contigs; c++) for (auto& e : all[(size_t)2 * c]) dup_starts[(size_t)c].push_back(e.first);
    dup_set = true; dup_generation++;
  }
  void set_duplications(int window, double granularity, int contig, int n, const int32_t* starts) {
    dup_window = window; dup_granularity = granularity;
    if ((int)dup_starts.size() < n_contigs) dup_starts.resize((size_t)n_contigs);
    dup_starts[(size_t)contig].assign(starts, starts + n);
    dup_set = true; dup_generation++;
  }
  // the duplication table as DupD reads it: the starts of contig c are starts[off[c], off[c + 1]); one trailing 0 keeps `starts`
  // non-empty when no contig has a duplication
  void dup_csr(std::vector<int64_t>& off, std::vector<int32_t>& starts) const {
    off.assign((size_t)n_contigs + 1, 0); starts.clear();
    for (int c = 0; c < n_contigs; c++) { if ((size_t)c < dup_starts.size()) starts.insert(starts.end(), dup_starts[(size_t)c].begin(), dup_starts[(size_t)c].end()); off[(size_t)c + 1] = (int64_t)starts.size(); }
    starts.push_back(0);
  }
};

// Workspace tiers: bytes of per-query arena. Queries that exhaust a tier are re-run from scratch in the next one
// (the algorithm is deterministic), so small arenas keep the common case at full occupancy.
static const int XM_NUM_TIERS = 3;
// Workspace per warp of the first-pass ("easy") kernel: pyramid rows, counters, candidate lists and a handful of
// single-block alignments; no lattice.
inline long long easy_arena_bytes(int max_seq_len, int n_seqs_max) {
  long long rows = pyr_arena_bytes(max_seq_len) * n_seqs_max;
  long long b = std::max<long long>(64 * 1024, rows + 48 * 1024 + 8 * (long long)max_seq_len);
  return (b + 255) & ~255LL;
}
// Workspace per WARP (one warp owns one query at a time).  Tier 0 is sized to hold a PathAligner lattice over the
// whole read (so that almost nothing is re-run) whenever one resident wave of such arenas fits the budget; otherwise
// it shrinks towards "a lattice over a BlockAligner piece".  Each further tier is 4x larger (fewer warps).
inline long long tier_arena_bytes(int tier, int max_seq_len, int n_seqs_max, long long budget = 24LL << 30, long long resident_warps = 148 * 16) {
  long long rows = pyr_arena_bytes(max_seq_len) * n_seqs_max;
  long long grid = (long long)(max_seq_len + 2) * (long long)(max_seq_len * 2 + 64) * 26;  // full-read PathAligner grid + heap share
  long long small = std::max<long long>(256 * 1024, rows * 2 + grid / 4);
  long long full = rows * 2 + grid * 5 / 2;
  long long a0 = full;
  if (a0 * resident_warps > budget) a0 = std::max<long long>(small, budget / std::max<long long>(1, resident_warps));
  long long b = a0;
  for (int i = 0; i < tier; i++) b *= 4;
  if (tier == 2) b = std::max<long long>(b, rows * 4 + grid * 16);
  return (b + 255) & ~255LL;  // arenas are carved back to back: keep every one 256-byte aligned
}

}  // namespace xm
