// Match / Tourney game step (SURVEY 8f-1): Match::doIteration + chooseMoveAndContinue
// (corintho_ai/cpp/src/match.cpp:66-77, 193-251) on the same per-game storage and tree kernels
// as self-play. Differences from SelfPlayer: every side has its own search budget (Player,
// match.h:13-31), a side may be a random player without a tree (match.cpp:27-33, 196-203), the
// authoritative position lives outside both trees (Match::root_, match.h:96; here in the control
// block), both trees run in testing mode, and requests are batched per model id (Tourney,
// tourney.cpp:24-72). External-evaluator API only (the reference's Tourney has no other).
#ifndef CORINTHO_B200_MATCH_CUH
#define CORINTHO_B200_MATCH_CUH

#include "tree.cuh"

namespace cb200 {

struct MatchSide {  // one Player as seen by one match
  int32_t model_id, max_searches, spe, random;
  float c_puct, epsilon;
  int32_t player_id;
  int32_t log_slot;  // side 0 only: index of the match's text-log area, -1 = not logged
};

// control-block words of a match beyond the self-play ones (CW_* in tree.cuh)
enum MatchCtlWord { MW_ROOT0 = 12, MW_ROOT1, MW_ROOT2, MW_ROOT3, MW_DEPTH };
static_assert(MW_DEPTH < kCtlWords, "control block too small");

__device__ __forceinline__ void apply_side(TreeParams &Pm, const MatchSide &s) {
  Pm.max_searches = s.max_searches, Pm.spe = s.spe;
  Pm.c_puct = s.c_puct, Pm.epsilon = s.epsilon;
}

// std::uniform_int_distribution<int32_t>(0, n - 1)(mt19937) as libstdc++ (GCC 11+) draws it:
// Lemire's nearly divisionless method on the 64-bit product (bits/uniform_int_dist.h, _S_nd)
__device__ __forceinline__ int uniform_index(Ctx &c, uint32_t n) {
  unsigned long long product = (unsigned long long)rng_one(c) * n;
  uint32_t low = (uint32_t)product;
  if (low < n) {
    const uint32_t threshold = (0u - n) % n;
    while (low < threshold) {
      product = (unsigned long long)rng_one(c) * n;
      low = (uint32_t)product;
    }
  }
  return (int)(product >> 32);
}

__device__ __forceinline__ bool match_selected(const int32_t *ctl, const MatchSide *sides,
                                               int model_id) {
  return !ctl[CW_DONE] && sides[ctl[CW_TO_PLAY]].model_id == model_id;
}
// Match::num_requests (match.cpp:44-48)
__device__ __forceinline__ int match_requests(const int32_t *ctl, const MatchSide *sides) {
  return sides[ctl[CW_TO_PLAY]].random ? 0 : ctl[CW_N_PENDING];
}

// One Match::doIteration per warp. offs[g] = first answer row of match g (computed by
// k_match_scan with the reference's own offset rule).
__global__ void __launch_bounds__(kTreeWarps * 32, 4)
    k_match_iterate(TreeParams P, const MatchSide *__restrict__ sides_all,
                    const float *__restrict__ eval, const float *__restrict__ probs,
                    const int32_t *__restrict__ offs, int model_id, long prs, long pcs) {
  __shared__ WarpSm sm_all[kTreeWarps];
  const int warp = threadIdx.x >> 5;
  const int g = blockIdx.x * kTreeWarps + warp;
  if (g >= P.num_games) return;
  int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  const MatchSide *sides = sides_all + 2 * (size_t)g;
  if (!match_selected(ctl, sides, model_id)) return;
  WarpSm &sm = sm_all[warp];
  Ctx c;
  c.to_play = ctl[CW_TO_PLAY], c.parity = 0, c.result = ctl[CW_RESULT];
  c.mate_turn = 0, c.n_samples = 0;
  c.n_pending = ctl[CW_N_PENDING], c.error = ctl[CW_ERROR], c.spare = ctl[CW_SPARE];
  c.mt_idx = ctl[CW_MT_IDX];
  c.d_sims = 0, c.d_evals = 0, c.d_moves = 0, c.d_searches = 0;
  CB_PROF(c.t_ingest = c.t_search = c.t_move = c.n_none = c.n_copy = 0;
          c.t_sel = c.t_exp = c.n_lvl = c.n_exp = c.n_exact = 0;)
  c.work = 0, c.yielded = 0;
  c.arenas = P.arenas + (size_t)g * 3 * P.arena_words;
  c.mt = P.mt + (size_t)g * 624;
  c.pending = P.pending + (size_t)g * P.spe * kPendWords;  // P.spe = largest budget (stride)
  c.tree_ctl = P.tree + (size_t)g * 2 * kTreeCtlWords;
  c.leaf_state = P.leaf_state + (size_t)g * P.spe;
  c.sample_state = nullptr, c.sample_probs = nullptr;
  CState root;
  root.w0 = (uint64_t)(uint32_t)ctl[MW_ROOT0] | ((uint64_t)(uint32_t)ctl[MW_ROOT1] << 32);
  root.w1 = (uint64_t)(uint32_t)ctl[MW_ROOT2] | ((uint64_t)(uint32_t)ctl[MW_ROOT3] << 32);
  int depth = ctl[MW_DEPTH];
  TreeParams Pm = P;
  Pm.testing = 1, Pm.vsqrt = nullptr, Pm.yield_budget = 0;
  bool is_random = sides[c.to_play].random != 0;
  apply_side(Pm, sides[c.to_play]);
  if (!is_random) load_tree(c, Pm, c.to_play);
  const long off = offs[g];
  // probs element (row k, move m) = probs[k * prs + m * pcs] (row-major from the host API and the
  // fp32 network, move-major from the tensor-core network; see receive_eval)
  const float *ev_p = eval + off, *pr_p = probs + off * prs;
  // per-match text log (Match::writePreMoveLogs / writeMoveChoice / endGame, match.cpp:79-180):
  // same records as self-play (tree.cuh, log_pre_move); [13] = 1 when a random player moved
  const int log_slot = P.log_buf != nullptr ? sides[0].log_slot : -1;
  int log_n = log_slot >= 0 ? P.log_count[log_slot] : 0;
  bool done = false;
  for (;;) {
    // Match::doIteration: a random player moves at once, a searching player iterates first
    bool turn_done = true;
    if (!is_random) turn_done = tree_do_iteration(c, Pm, sm, ev_p, pr_p, prs, pcs);
    if (c.error || !turn_done) break;
    // one pass of Match::chooseMoveAndContinue's loop
    uint32_t *lrec = nullptr;
    if (log_slot >= 0 && log_n < kLogMaxMoves)
      lrec = P.log_buf + ((size_t)log_slot * kLogMaxMoves + log_n) * kLogWords;
    if (lrec != nullptr) {
      if (c.lane == 0) {
        lrec[13] = is_random ? 1u : 0u;
        lrec[1] = (uint32_t)c.to_play, lrec[5] = 0u, lrec[6] = 0u;
        if (!is_random)
          log_pre_move(c.base, c.root_off, c.to_play, c.root_visits, c.root_eval, c.root_result, lrec);
      }
      g_sync(c);
    }
    int choice;
    if (is_random) {
      uint32_t m[3];
      legal_moves(root, m, DeviceLB());
      const int n = __popc(m[0]) + __popc(m[1]) + __popc(m[2]);
      choice = nth_move(m, uniform_index(c, (uint32_t)n)) & 127;
    } else {
      c.d_sims += c.searches_done;
      c.d_moves += 1;
      choice = choose_move(c, Pm, sm, (float *)nullptr);
      if (c.error) break;
      g_sync(c);
    }
    root = do_move(root, choice);
    depth += 1;
    uint32_t m[3];
    const bool lines = legal_moves(root, m, DeviceLB());
    if (lrec != nullptr) {
      if (c.lane == 0) {
        lrec[7] = (uint32_t)choice;
        lrec[8] = (uint32_t)root.w0, lrec[9] = (uint32_t)(root.w0 >> 32);
        lrec[10] = (uint32_t)root.w1, lrec[11] = (uint32_t)(root.w1 >> 32);
        int res = 0;
        if ((m[0] | m[1] | m[2]) == 0u)
          res = 1 + (!lines ? kResultDraw : (c.to_play == 1 ? kResultLoss : kResultWin));
        lrec[12] = (uint32_t)res;
      }
      log_n += 1;
    }
    if ((m[0] | m[1] | m[2]) == 0u) {  // endGame (match.cpp:161-190)
      c.result = !lines ? kResultDraw : (c.to_play == 1 ? kResultLoss : kResultWin);
      if (!is_random) {
        c.has_root = 0;
        store_tree(c);
      }
      if (!sides[1 - c.to_play].random) {
        load_tree(c, Pm, 1 - c.to_play);
        c.has_root = 0;
        store_tree(c);
      }
      c.n_pending = 0;
      is_random = true;  // nothing left to store below
      done = true;
      break;
    }
    if (!is_random) store_tree(c);
    c.to_play = 1 - c.to_play;
    is_random = sides[c.to_play].random != 0;
    apply_side(Pm, sides[c.to_play]);
    if (is_random) continue;
    load_tree(c, Pm, c.to_play);
    if (!c.has_root) {  // first turn of this player: createRoot + doIteration (match.cpp:232-236)
      fresh_tree(c, Pm, root, depth);
      c.searches_done = 0;
      continue;  // doIteration queues the new root for evaluation and returns false
    }
    const bool need_eval = receive_opponent_move(c, Pm, choice, root, depth);
    if (c.error || need_eval) break;
  }
  if (c.error) done = true;
  if (!is_random) store_tree(c);
  if (c.lane == 0) {
    ctl[CW_TO_PLAY] = c.to_play, ctl[CW_RESULT] = c.result;
    ctl[CW_N_PENDING] = c.n_pending, ctl[CW_ERROR] = c.error;
    ctl[CW_SPARE] = c.spare, ctl[CW_MT_IDX] = c.mt_idx;
    ctl[MW_ROOT0] = (int32_t)(uint32_t)root.w0, ctl[MW_ROOT1] = (int32_t)(uint32_t)(root.w0 >> 32);
    ctl[MW_ROOT2] = (int32_t)(uint32_t)root.w1, ctl[MW_ROOT3] = (int32_t)(uint32_t)(root.w1 >> 32);
    ctl[MW_DEPTH] = depth;
    if (log_slot >= 0) P.log_count[log_slot] = log_n;
    if (done) ctl[CW_DONE] = 1;
    long long *cnt = P.counters + (size_t)g * 4;
    cnt[0] += c.d_sims, cnt[1] += c.d_moves, cnt[2] += c.d_evals;
  }
}

// Offsets of both kinds for one model id (one CTA of 1024 threads; both are prefix sums).
// pack_offs = contiguous packing of Tourney::writeRequests (tourney.cpp:44-52);
// iter_offs = the answer offsets of Tourney::doIteration (tourney.cpp:54-62), which advance by
// the request count of match i-1 whenever match i is selected -- literally (SURVEY Q14).
// summary = {requests of the selected matches, matches not done, error code, max row read}.
__global__ void __launch_bounds__(1024)
    k_match_scan(TreeParams P, const MatchSide *__restrict__ sides_all, int model_id,
                 int32_t *__restrict__ pack_offs, int32_t *__restrict__ iter_offs,
                 int32_t *__restrict__ summary) {
  __shared__ int s_pack[1024], s_it[1024];
  __shared__ int s_live, s_err, s_max;
  const int t = threadIdx.x;
  if (t == 0) s_live = 0, s_err = 0, s_max = 0;
  __syncthreads();
  const int per = (P.num_games + 1023) / 1024;
  const int g0 = t * per, g1 = min(P.num_games, g0 + per);
  // the amount iter_offs advances at match g, and the rows match g packs
  auto step_of = [&](int g, int &n_sel) -> int {
    const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
    const bool sel = match_selected(ctl, sides_all + 2 * (size_t)g, model_id);
    n_sel = sel ? match_requests(ctl, sides_all + 2 * (size_t)g) : -1;
    return (g > 0 && sel)
               ? match_requests(P.ctl + (size_t)(g - 1) * kCtlWords, sides_all + 2 * (size_t)(g - 1))
               : 0;
  };
  int pack = 0, it = 0, live = 0, err = 0;
  for (int g = g0; g < g1; ++g) {
    int n_sel;
    it += step_of(g, n_sel);
    if (n_sel >= 0) pack += n_sel;
    const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
    if (!ctl[CW_DONE]) ++live;
    if (ctl[CW_ERROR]) err = ctl[CW_ERROR];
  }
  s_pack[t] = pack, s_it[t] = it;
  if (live) atomicAdd(&s_live, live);
  if (err) atomicMin(&s_err, err);
  __syncthreads();
  for (int d = 1; d < 1024; d <<= 1) {  // Hillis-Steele inclusive scans over the 1024 partials
    const int a = (t >= d) ? s_pack[t - d] : 0, b = (t >= d) ? s_it[t - d] : 0;
    __syncthreads();
    s_pack[t] += a, s_it[t] += b;
    __syncthreads();
  }
  int run_pack = s_pack[t] - pack, run_it = s_it[t] - it, max_row = 0;
  for (int g = g0; g < g1; ++g) {
    int n_sel;
    run_it += step_of(g, n_sel);
    iter_offs[g] = run_it;
    pack_offs[g] = run_pack;
    if (n_sel >= 0) {
      run_pack += n_sel;
      if (run_it + n_sel > max_row) max_row = run_it + n_sel;
    }
  }
  if (max_row) atomicMax(&s_max, max_row);
  __syncthreads();
  if (t == 0) summary[0] = s_pack[1023], summary[1] = s_live, summary[2] = s_err, summary[3] = s_max;
}

// Tourney::writeRequests (tourney.cpp:44-52): 70-float rows of the selected matches
__global__ void __launch_bounds__(256)
    k_match_pack(TreeParams P, const MatchSide *__restrict__ sides_all, int model_id,
                 const int32_t *__restrict__ pack_offs, float *__restrict__ rows,
                 ulonglong2 *__restrict__ packed) {
  const int g = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= P.num_games) return;
  const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  const MatchSide *sides = sides_all + 2 * (size_t)g;
  if (!match_selected(ctl, sides, model_id)) return;
  const int np = match_requests(ctl, sides);
  const ulonglong2 *ls = P.leaf_state + (size_t)g * P.spe;
  if (packed)  // fused tourney: leaf cstates in request order for the device-resident network
    for (int k = lane; k < np; k += 32) packed[(size_t)pack_offs[g] + k] = ls[k];
  if (!rows) return;
  float *out = rows + (size_t)pack_offs[g] * CB200_STATE_SIZE;
  for (int f = lane; f < np * CB200_STATE_SIZE; f += 32) {
    const int k = f / CB200_STATE_SIZE, j = f - k * CB200_STATE_SIZE;
    const ulonglong2 v = ls[k];
    out[f] = encode_elem(CState{v.x, v.y}, j);
  }
}

}  // namespace cb200
#endif
