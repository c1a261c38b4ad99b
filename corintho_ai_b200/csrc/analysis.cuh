// Analysis: the reference's DockerMC (corintho_ai/cpp/src/dockermc.cpp) for a batch of given
// positions. Position g is searched by one testing-mode TrainMC on the analysis' per-game storage
// (one "game" per position, engine.cu's GameStore): its tree of the side to move starts as a single node
// holding the caller's position, TrainMC::doIteration runs until the turn is complete, the root
// statistics are written out and TrainMC::chooseMove picks the move. Nothing continues into the
// opponent's turn, which is why this is its own kernel rather than a branch of run_game or
// k_match_iterate. The rounds around it (request scan / pack / network) are the self-play ones
// (k_scan_requests / k_pack_requests in training selection, every live position), so the answers
// of position g sit at the contiguous offset offs[g].
#ifndef CORINTHO_B200_ANALYSIS_CUH
#define CORINTHO_B200_ANALYSIS_CUH

#include "tree.cuh"

namespace cb200 {

struct AnalysisOut {
  int32_t *moves, *results;  // [n]
  float *values;             // [n]
  int32_t *visits;           // [n][96]
  float *evals;              // [n][96]; null = not wanted
};

// Root statistics of position g, read before the move is chosen: per move id the child's visits_
// and evaluation_ (0 for illegal or unexpanded moves), the root's evaluation_ and result code.
// One lane per slot scatters into shared memory; the rows then leave coalesced, one lane per move.
__device__ __forceinline__ void write_root_stats(Ctx &c, WarpSm &sm, int g, const AnalysisOut &out,
                                                 bool searched) {
  float *ev = sm.fval, *vis = sm.dval;  // visits travel as int bits
  for (int m = c.lane; m < CB200_NUM_MOVES; m += 32) ev[m] = 0.0f, vis[m] = __int_as_float(0);
  g_sync(c);
  if (searched) {
    const uint32_t *r = c.base + c.root_off;
    const int n = (int)(r[4] & 0xffu);
    for (int e = c.lane; e < n; e += 32) {
      const uint4 s = ld4(r + 8 + 4 * e);
      if (s3_has(s.w)) ev[s3_move(s.w)] = __uint_as_float(s.x), vis[s3_move(s.w)] = __uint_as_float(s.y);
    }
  }
  g_sync(c);
  int32_t *vo = out.visits + (size_t)g * CB200_NUM_MOVES;
  float *eo = out.evals != nullptr ? out.evals + (size_t)g * CB200_NUM_MOVES : nullptr;
  for (int m = c.lane; m < CB200_NUM_MOVES; m += 32) {
    vo[m] = __float_as_int(vis[m]);
    if (eo != nullptr) eo[m] = ev[m];
  }
  if (c.lane == 0) out.values[g] = searched ? c.root_eval : 0.0f, out.results[g] = c.root_result;
  g_sync(c);
}

// One TrainMC::doIteration per warp and live position (answers of position g at offs[g]).
// roots[g] = the caller's position; its byte 6 names the side to move and so the tree searched.
// max_searches is the searcher's budget (the trainer's own may be larger: it must cover spe).
__global__ void __launch_bounds__(kTreeWarps * 32, 4)
    k_analysis_iterate(TreeParams P, int max_searches, const ulonglong2 *__restrict__ roots,
                       const float *__restrict__ eval, const float *__restrict__ probs, long prs,
                       long pcs, const int32_t *__restrict__ offs, AnalysisOut out) {
  __shared__ WarpSm sm_all[kTreeWarps];
  const int warp = threadIdx.x >> 5;
  const int g = blockIdx.x * kTreeWarps + warp;
  if (g >= P.num_games) return;
  int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  if (ctl[CW_DONE]) return;
  WarpSm &sm = sm_all[warp];
  const ulonglong2 rv = roots[g];
  const CState root{rv.x, rv.y};
  Ctx c;
  c.to_play = (int)((root.w1 >> 48) & 0xffu), c.parity = 0, c.result = ctl[CW_RESULT];
  c.mate_turn = 0, c.n_samples = 0;
  c.n_pending = ctl[CW_N_PENDING], c.error = ctl[CW_ERROR], c.spare = ctl[CW_SPARE];
  c.mt_idx = ctl[CW_MT_IDX];
  c.d_sims = 0, c.d_evals = 0, c.d_moves = 0, c.d_searches = 0;
  CB_PROF(c.t_ingest = c.t_search = c.t_move = c.n_none = c.n_copy = 0;
          c.t_sel = c.t_exp = c.n_lvl = c.n_exp = c.n_exact = 0;)
  c.work = 0, c.yielded = 0;
  c.arenas = P.arenas + (size_t)g * 3 * P.arena_words;
  c.mt = P.mt + (size_t)g * 624;
  c.pending = P.pending + (size_t)g * P.spe * kPendWords;
  c.tree_ctl = P.tree + (size_t)g * 2 * kTreeCtlWords;
  c.leaf_state = P.leaf_state + (size_t)g * P.spe;
  c.sample_state = nullptr, c.sample_probs = nullptr;
  TreeParams Pm = P;
  Pm.testing = 1, Pm.yield_budget = 0, Pm.max_searches = max_searches;
  load_tree(c, Pm, c.to_play);
  bool done = false;
  if (!c.has_root) {  // first round of a run: the position becomes a single-node tree at depth 0
    fresh_tree(c, Pm, root, 0);
    c.searches_done = 0;  // doIteration queues the root for evaluation (trainmc.cpp:150-152)
    if (r_terminal(c.root_result)) {  // no legal move: nothing to search, report the result
      write_root_stats(c, sm, g, out, false);
      if (c.lane == 0) out.moves[g] = -1;
      done = true;
    }
  }
  if (!done) {
    const long off = offs[g];
    const bool turn_done = tree_do_iteration(c, Pm, sm, eval + off, probs + off * prs, prs, pcs);
    if (!c.error && turn_done) {
      write_root_stats(c, sm, g, out, true);
      c.d_sims += c.searches_done;
      c.d_moves += 1;
      const int choice = choose_move(c, Pm, sm, (float *)nullptr);
      if (c.lane == 0) out.moves[g] = choice;
      done = true;
    }
  }
  if (c.error) done = true;
  store_tree(c);
  if (c.lane == 0) {
    ctl[CW_TO_PLAY] = c.to_play, ctl[CW_N_PENDING] = c.n_pending, ctl[CW_ERROR] = c.error;
    ctl[CW_SPARE] = c.spare, ctl[CW_MT_IDX] = c.mt_idx;
    if (done) ctl[CW_DONE] = 1;
    long long *cnt = P.counters + (size_t)g * 4;
    cnt[0] += c.d_sims, cnt[1] += c.d_moves, cnt[2] += c.d_evals, cnt[3] += c.d_searches;
  }
}

}  // namespace cb200
#endif
