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

#include "persistent.cuh"

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

// The structural invariants of a cstate that the engine accepts from a caller (checked over the
// reachable positions of 1 000 000 random play-outs by tests/test_oracle_analysis.py): side to move
// 0 or 1, byte 7 zero, at most 4 pieces of a kind in a hand, frozen squares occupied, and every
// piece of a kind either on the board or in a hand (8 of each kind). The one definition behind
// cb200_check_states and the per-position check of k_analysis_persistent.
__host__ __device__ inline int valid_state_popc(uint32_t x) {
#ifdef __CUDA_ARCH__
  return __popc(x);
#else
  return __builtin_popcount(x);
#endif
}
__host__ __device__ inline bool valid_state(uint64_t w0, uint64_t w1) {
  if (((w1 >> 48) & 0xff) > 1 || (w1 >> 56) != 0) return false;
  const uint32_t base = (uint32_t)(w0 & 0xffff), column = (uint32_t)((w0 >> 16) & 0xffff);
  const uint32_t capital = (uint32_t)((w0 >> 32) & 0xffff), frozen = (uint32_t)(w0 >> 48);
  if (frozen & ~(base | column | capital)) return false;
  const uint32_t plane[3] = {base, column, capital};
  for (int t = 0; t < 3; ++t) {
    const int h0 = (int)((w1 >> (8 * t)) & 0xff), h1 = (int)((w1 >> (8 * (3 + t))) & 0xff);
    if (h0 > 4 || h1 > 4 || valid_state_popc(plane[t]) != 8 - h0 - h1) return false;
  }
  return true;
}

// One TrainMC::doIteration of position g by one warp, answers of its last requests at row `off`
// (eval[off], probs[off * prs + move * pcs]). roots[g] = the caller's position; its byte 6 names the
// side to move and so the tree searched. max_searches is the searcher's budget (the store's own may
// be larger: it must cover spe). On return *n_pending = the requests now queued in
// P.leaf_state[g * spe ..] and *error = the position's error code (both uniform over the warp);
// the result is true when the position is finished (its outputs written, unless it failed).
__device__ __forceinline__ bool analysis_step(const TreeParams &P, int max_searches, int g,
                                              const ulonglong2 *__restrict__ roots, WarpSm &sm,
                                              const float *__restrict__ eval,
                                              const float *__restrict__ probs, long prs, long pcs,
                                              long off, const AnalysisOut &out, int *n_pending,
                                              int *error) {
  int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  const ulonglong2 rv = roots[g];
  const CState root{rv.x, rv.y};
  Ctx c;
  ctx_open(c, P, g, ctl, false);
  c.to_play = (int)((root.w1 >> 48) & 0xffu), c.result = kResultNone;  // a position, not a game
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
    ctx_close(c, ctl, false);
    if (done) ctl[CW_DONE] = 1;
    long long *cnt = P.counters + (size_t)g * 4;
    cnt[0] += c.d_sims, cnt[1] += c.d_moves, cnt[2] += c.d_evals, cnt[3] += c.d_searches;
  }
  *n_pending = c.n_pending, *error = c.error;
  return done;
}

// One round of every live position (answers of position g at offs[g]).
__global__ void __launch_bounds__(kTreeWarps * 32, 4)
    k_analysis_iterate(TreeParams P, int max_searches, const ulonglong2 *__restrict__ roots,
                       const float *__restrict__ eval, const float *__restrict__ probs, long prs,
                       long pcs, const int32_t *__restrict__ offs, AnalysisOut out) {
  __shared__ WarpSm sm_all[kTreeWarps];
  const int warp = threadIdx.x >> 5;
  const int g = blockIdx.x * kTreeWarps + warp;
  if (g >= P.num_games) return;
  if (P.ctl[(size_t)g * kCtlWords + CW_DONE]) return;
  int n_pending, error;
  analysis_step(P, max_searches, g, roots, sm_all[warp], eval, probs, prs, pcs, offs[g], out, &n_pending,
                &error);
}

// ---- device-resident analysis (cb200_analysis_run_device) ----------------------------------------

// The outputs of a position that was not searched to the end: move -1, result `code`, zeros.
__device__ __forceinline__ void write_failed(int lane, int g, const AnalysisOut &out, int code) {
  int32_t *vo = out.visits + (size_t)g * CB200_NUM_MOVES;
  float *eo = out.evals != nullptr ? out.evals + (size_t)g * CB200_NUM_MOVES : nullptr;
  for (int m = lane; m < CB200_NUM_MOVES; m += 32) {
    vo[m] = 0;
    if (eo != nullptr) eo[m] = 0.0f;
  }
  if (lane == 0) out.moves[g] = -1, out.results[g] = code, out.values[g] = 0.0f;
}

// Analysis in one persistent launch: one CTA per SM holds kGames positions, one warp each (16 with
// bf16 / fp16 operands, 512 threads, the network on the first 256; 8 with bf16x3, 256 threads, one
// network tile on the first 128). A round is analysis_step of every warp's position, its requests
// appended to the CTA's rows [row0, row0 + kGames * spe) with one shared atomicAdd per position,
// then tc_forward over those rows, whose answers (move-major, leading dimension ld) the next round
// reads. The first wave is dealt round-robin (slot = warp * grid + block) so that a small batch
// spreads over every SM; a warp whose position finishes takes the next one in the same round
// (ctr[0] counts the draws after the first wave), and the CTA leaves once no warp holds a live
// position. A position's first round checks its state (valid_state); rejected ones and searches that
// fail get write_failed, counted in ctr[1], the most negative code in ctr[2]; ctr starts at zero. A
// position's order of operations is k_analysis_iterate's, and a network row does not depend on the
// other rows of its batch: the outputs are cb200_analysis_run's.
template <int kMode, int kGames>
__global__ void __launch_bounds__(kGames * 32, 1)
    k_analysis_persistent(TreeParams P, int max_searches, const uint8_t *__restrict__ W,
                          const ulonglong2 *__restrict__ states, float *eval, float *probs, int ld,
                          ulonglong2 *packed, int32_t *ctr, AnalysisOut out) {
  constexpr int kNetThreads = ps_net_threads<kGames>();
  constexpr int kTileRows = kNetThreads;  // rows per tc_forward call
  const bool net_thread = threadIdx.x < kNetThreads;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ int32_t s_ctr[2];  // requests of this round, live positions
  TcState S;
  if (net_thread) tc_setup(S, smem, kNetThreads, kMode == 2 ? 2 : 1);
  WarpSm *sm_all = reinterpret_cast<WarpSm *>(smem + ps_tree_smem_off<kMode, kGames>());
  const int warp = threadIdx.x / 32, lane = threadIdx.x & 31;
  WarpSm &sm = sm_all[warp];
  const int n = P.num_games;
  const int row0 = blockIdx.x * kGames * P.spe;
  int g = warp * gridDim.x + blockIdx.x;
  if (g >= n) g = -1;
  bool fresh = true;  // g has not been stepped yet
  for (;;) {
    if (threadIdx.x == 0) s_ctr[0] = 0, s_ctr[1] = 0;
    __syncthreads();
    while (g >= 0) {
      bool done = false;
      int n_pending = 0, error = 0;
      if (fresh) {
        const ulonglong2 v = states[g];
        fresh = false;
        if (!valid_state(v.x, v.y)) error = CB200_ERR_ARG, done = true;
      }
      if (!done) {
        int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
        done = analysis_step(P, max_searches, g, states, sm, eval, probs, 1, ld, ctl[CW_REQ_BASE], out, &n_pending,
                             &error);
        if (!done) {  // queue the requests in this CTA's rows
          int base = 0;
          if (lane == 0) {
            if (n_pending > 0) base = atomicAdd(&s_ctr[0], n_pending);
            atomicAdd(&s_ctr[1], 1);
            ctl[CW_REQ_BASE] = row0 + base;
          }
          base = __shfl_sync(0xffffffffu, base, 0);
          __syncwarp();  // lane 0's leaf states of analysis_step are visible to the whole warp
          const ulonglong2 *ls = P.leaf_state + (size_t)g * P.spe;
          for (int k = lane; k < n_pending; k += 32) packed[row0 + base + k] = ls[k];
          break;
        }
      }
      if (error) {
        write_failed(lane, g, out, error);
        if (lane == 0) atomicAdd(ctr + 1, 1), atomicMin(ctr + 2, error);
      }
      int next = 0;
      if (lane == 0) next = atomicAdd(ctr, 1) + gridDim.x * kGames;  // past the first wave
      next = __shfl_sync(0xffffffffu, next, 0);
      g = next < n ? next : -1;
      fresh = true;
    }
    __syncthreads();
    const int reqs = s_ctr[0], live = s_ctr[1];
    if (net_thread)
      for (int r0 = 0; r0 < reqs; r0 += kTileRows) {
        const int rows = reqs - r0 < kTileRows ? reqs - r0 : kTileRows;
        tc_forward<kMode>(S, W, packed + row0 + r0, rows, 0, eval + row0 + r0, probs + row0 + r0, ld);
      }
    __syncthreads();  // answers visible to every warp; counters read before they are cleared
    if (live == 0) break;
  }
  if (net_thread) tc_teardown(S);
}

}  // namespace cb200
#endif
