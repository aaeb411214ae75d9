// TEST INFRASTRUCTURE ONLY — host emulation of the device core (mapper_b200/csrc/xm_*.h compiled with g++).
// It lets the kernel logic be compared with the oracle on a box without a GPU, one query per loop iteration,
// with the same workspace tiers the CUDA launcher uses.  It is NOT part of the product: libxmapper_b200.so never
// contains this file and has no CPU path.
// The emulation runs the device source itself: the per-query code's lane-split loops are written through the warp helpers of
// xm_types.h, which g++ compiles as a warp of one lane (XM_LANES = 1), so each loop runs serially in base order.  What one lane
// cannot exercise - compaction across lanes, the replay of lanes j > 0, the xor tree across lanes - and the device-only parts
// (the lattice search's 32-bucket queue and shared-memory frame, TMA staging) are covered by the GPU tests only.
#include <cstring>
#include "../../mapper_b200/csrc/xm_align.h"
#include "../../mapper_b200/csrc/xm_host_model.h"
#include "../../mapper_b200/csrc/xm_results.h"
#include <thread>
#include <mutex>

using namespace xm;

namespace {
struct CParams { double mutation, ins_start, ins_ext, del_start, del_ext, max_error_rate, unaligned, ambiguity, span; int32_t max_num_matches, enable_gapmers; };
struct Emu { HostModel m; std::string err; double pen[256]; uint8_t cls[1024]; };
}

extern "C" {

void* xe_create(const CParams* p) {
  Emu* e = new Emu();
  Params& q = e->m.prm;
  q.mutation = p->mutation; q.ins_start = p->ins_start; q.ins_ext = p->ins_ext; q.del_start = p->del_start; q.del_ext = p->del_ext;
  q.max_error_rate = p->max_error_rate; q.unaligned = p->unaligned; q.ambiguity = p->ambiguity; q.span = p->span;
  q.max_num_matches = p->max_num_matches; q.start_free = 0;
  fill_pen_tab(q, e->pen, e->cls, 0, 1);
  q.pen_tab = e->pen; q.cls_tab = e->cls;
  e->m.gapmers = p->enable_gapmers;
  return e;
}
void xe_destroy(void* h) { delete (Emu*)h; }
const char* xe_last_error(void* h) { return ((Emu*)h)->err.c_str(); }
int xe_set_reference(void* h, int n, const uint16_t* const* packed, const int32_t* lens) { ((Emu*)h)->m.set_reference(n, packed, lens); return 0; }
int xe_set_index_length(void* h, int n_used, int cap, int maxc, const int64_t* off, const uint8_t* over, const uint32_t* pos) { ((Emu*)h)->m.set_index_length(n_used, cap, maxc, off, over, pos); return 0; }
int xe_set_position_bias(void* h, long long bias) { ((Emu*)h)->m.position_bias = bias; return 0; }   // before xe_set_reference
int xe_set_index_length_wide(void* h, int n_used, int cap, int maxc, const int64_t* off, const uint8_t* over, const uint64_t* pos) { ((Emu*)h)->m.set_index_length(n_used, cap, maxc, off, over, pos, true); return 0; }
int xe_get_index_positions_wide(void* h, int n, uint64_t* pos) {
  Emu* e = (Emu*)h;
  if (n < 0 || n > e->m.max_built) return -1;
  int c, m; int64_t np;
  e->m.get_index_length(n, c, m, np, nullptr, nullptr, nullptr, pos);
  return 0;
}
int xe_finish_index(void* h, int mi, int mb) { ((Emu*)h)->m.finish_index(mi, mb); return 0; }
int xe_build_index(void* h, int max_used, int threads) { Emu* e = (Emu*)h; return e->m.build_index(max_used, threads, e->err) ? 0 : -1; }
int xe_index_info(void* h, int* mi, int* mb) { *mi = ((Emu*)h)->m.min_interesting; *mb = ((Emu*)h)->m.max_built; return 0; }
int xe_get_index_length(void* h, int n, int* cap, int* maxc, int64_t* npos, int64_t* off, uint8_t* over, uint32_t* pos) {
  Emu* e = (Emu*)h;
  if (n < 0 || n > e->m.max_built) return -1;
  int c, m; int64_t np;
  e->m.get_index_length(n, c, m, np, off, over, pos);
  *cap = c; *maxc = m; *npos = np;
  return 0;
}
int xe_set_duplications(void* h, int window, double gran, int contig, int n, const int32_t* starts) { ((Emu*)h)->m.set_duplications(window, gran, contig, n, starts); return 0; }
int xe_build_duplications(void* h, int min_len, int max_len, int min_copies, int window) { ((Emu*)h)->m.build_duplications(min_len, max_len, min_copies, window); return 0; }
int xe_build_duplications_via_merge(void* h, int min_len, int max_len, int min_copies, int window) { ((Emu*)h)->m.build_duplications(min_len, max_len, min_copies, window, true); return 0; }
int xe_get_duplications(void* h, int contig, int* n, int32_t* starts) {
  Emu* e = (Emu*)h;
  auto& v = e->m.dup_starts[(size_t)contig];
  *n = (int)v.size();
  if (starts) for (size_t i = 0; i < v.size(); i++) starts[i] = v[i];
  return 0;
}

void* xe_align_batch(void* h, int nq, const uint16_t* packed, const int64_t* seq_word_off, const int32_t* seq_len, const uint8_t* n_seqs,
                     const double* expected_inner, const double* per_penalty, int threads, int max_tier) {
  Emu* e = (Emu*)h;
  HostModel& M = e->m;
  // "device" structs over host arrays
  RefD ref; ref.n_contigs = M.n_contigs; ref.words = M.words.data(); ref.word_off = M.word_off.data(); ref.len = M.len.data(); ref.gstart = M.gstart.data(); ref.total_fr = M.total_fr;
  std::vector<TableD> tabs(M.tables.size());
  for (size_t i = 0; i < M.tables.size(); i++) { tabs[i].capacity = M.tables[i].capacity; tabs[i].max_count = M.tables[i].max_count; tabs[i].buckets = M.tables[i].buckets.empty() ? nullptr : M.tables[i].buckets.data(); tabs[i].positions = M.tables[i].positions.data(); tabs[i].positions_hi = M.tables[i].positions_hi.empty() ? nullptr : M.tables[i].positions_hi.data(); }
  IndexD ix; ix.min_interesting = M.min_interesting; ix.max_built = M.max_built; ix.gapmers = M.gapmers; ix.tables = tabs.data();
  std::vector<int64_t> doff; std::vector<int32_t> dst;
  M.dup_csr(doff, dst);
  DupD dup; dup.window = M.dup_window; dup.granularity = M.dup_granularity; dup.off = doff.data(); dup.starts = dst.data();

  std::vector<int64_t> first((size_t)nq + 1, 0);
  int max_len = 1;
  for (int i = 0; i < nq; i++) first[(size_t)i + 1] = first[(size_t)i] + n_seqs[i];
  for (int64_t s = 0; s < first[(size_t)nq]; s++) max_len = std::max(max_len, (int)seq_len[s]);
  std::vector<OutQuery> oq((size_t)nq);
  // result arena sized generously; grown on overflow
  long long capc = (long long)nq * 4 + 1024, caps = (long long)nq * 8 + 1024, capb = (long long)nq * 32 + 4096;
  std::vector<OutChoice> choices((size_t)capc); std::vector<OutSA> sas((size_t)caps); std::vector<int32_t> blocks((size_t)capb * 4);
  unsigned long long used[3] = {0, 0, 0};
  std::vector<unsigned long long> stats(8, 0);
  std::vector<int> tier_count(XM_NUM_TIERS, 0);
  int n_easy = 0;
  std::mutex mu;
  int nt = std::max(1, threads);
  auto work = [&](int t) {
    std::vector<std::vector<char>> arenas((size_t)XM_NUM_TIERS);
    std::vector<char> easy_arena;
    int leasy = 0;
    unsigned long long lstats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int ltier[XM_NUM_TIERS] = {0, 0, 0};
    for (int qi = t; qi < nq; qi += nt) {
      QueryIn q; q.n_seqs = n_seqs[qi];
      for (int s = 0; s < q.n_seqs; s++) { int64_t sid = first[(size_t)qi] + s; q.seq[s].w = packed + seq_word_off[sid]; q.seq[s].len = seq_len[sid]; q.seq[s].rc = 0; q.seq[s].bytes = nullptr; }
      if (q.n_seqs < 2) { q.seq[1] = q.seq[0]; q.seq[1].len = 0; }
      q.expected_inner = q.n_seqs > 1 ? expected_inner[qi] : 0; q.per_penalty = q.n_seqs > 1 ? per_penalty[qi] : 1;
      int status = Q_NEED_MORE;
      {  // first pass: the EASY instantiation in its small arena, exactly as the library's first kernel runs it
        long long bytes = easy_arena_bytes(max_len, 2);
        if ((long long)easy_arena.size() < bytes) easy_arena.resize((size_t)bytes);
        WS w;
        OutArena out; out.q = oq.data(); out.choices = choices.data(); out.cap_choices = capc; out.sas = sas.data(); out.cap_sas = caps;
        out.blocks = blocks.data(); out.cap_blocks = capb; out.stats = nullptr;
        OutQuery rec; rec.status = 0; rec.n_comp = 1; rec.n_choice[0] = rec.n_choice[1] = 0; rec.choice_first[0] = rec.choice_first[1] = 0;
        if (ws_init(w, easy_arena.data(), bytes, &ref, &ix, &dup, M.prm, q, false)) {
          std::lock_guard<std::mutex> lock(mu);
          out.used = used;
          align_query<true>(w, out, rec);
          if (w.status != Q_HARD && w.status != Q_NEED_MORE) {
            status = w.status; rec.status = status; oq[(size_t)qi] = rec; leasy++;
            lstats[0] += w.st_probes; lstats[1] += w.st_seeds; lstats[2] += w.st_hits; lstats[3] += w.st_straight;
          }
        }
      }
      for (int tier = 0; tier < XM_NUM_TIERS && tier <= max_tier && status == Q_NEED_MORE; tier++) {
        long long bytes = tier_arena_bytes(tier, max_len, 2);
        if ((long long)arenas[(size_t)tier].size() < bytes) { arenas[(size_t)tier].resize((size_t)bytes); memset(arenas[(size_t)tier].data(), 0, 16); }  // generation word of the lattice map: 0 = clear before use
        WS w;
        OutArena out; out.q = oq.data(); out.choices = choices.data(); out.cap_choices = capc; out.sas = sas.data(); out.cap_sas = caps;
        out.blocks = blocks.data(); out.cap_blocks = capb; out.stats = nullptr;
        OutQuery rec; rec.status = 0; rec.n_comp = 1; rec.n_choice[0] = rec.n_choice[1] = 0; rec.choice_first[0] = rec.choice_first[1] = 0;
        ltier[tier]++;
        if (!ws_init(w, arenas[(size_t)tier].data(), bytes, &ref, &ix, &dup, M.prm, q)) { status = Q_NEED_MORE; continue; }
        {
          std::lock_guard<std::mutex> lock(mu);  // the bump counters are plain integers on the host
          out.used = used;
          align_query<false>(w, out, rec);
        }
        status = w.status;
        rec.status = status;
        if (status == 0 || tier == XM_NUM_TIERS - 1 || tier == max_tier) {
          lstats[0] += w.st_probes; lstats[1] += w.st_seeds; lstats[2] += w.st_hits; lstats[3] += w.st_straight;
          lstats[4] += w.st_path_calls; lstats[5] += w.st_path_steps; lstats[6] += w.st_path_cells;
        }
        oq[(size_t)qi] = rec;
      }
      if (status == Q_NEED_MORE) oq[(size_t)qi].status = Q_WORKSPACE;
    }
    std::lock_guard<std::mutex> lock(mu);
    for (int i = 0; i < 8; i++) stats[(size_t)i] += lstats[i];
    for (int i = 0; i < XM_NUM_TIERS; i++) tier_count[(size_t)i] += ltier[i];
    n_easy += leasy;
  };
  if (nt == 1) work(0);
  else { std::vector<std::thread> th; for (int t = 0; t < nt; t++) th.emplace_back(work, t); for (auto& x : th) x.join(); }
  ResultsHost* R = new ResultsHost();
  R->assemble(nq, oq.data(), choices.data(), sas.data(), blocks.data());
  R->stats.assign(32, 0);
  R->stats[25] = n_easy;
  R->stats[2] = tier_count[0]; R->stats[3] = tier_count[1]; R->stats[4] = tier_count[2];
  R->stats[5] = (int64_t)stats[0]; R->stats[6] = (int64_t)stats[1]; R->stats[7] = (int64_t)stats[2]; R->stats[8] = (int64_t)stats[3];
  R->stats[9] = (int64_t)stats[4]; R->stats[10] = (int64_t)stats[5]; R->stats[11] = (int64_t)stats[6];
  return R;
}
int64_t xe_results_array(void* r, int which, const void** ptr) { return ((ResultsHost*)r)->array(which, ptr); }
void xe_results_free(void* r) { delete (ResultsHost*)r; }

}  // extern "C"
