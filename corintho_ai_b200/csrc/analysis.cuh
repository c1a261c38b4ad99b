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

// The first n outputs of std::mt19937(seed) (the per-position seeds of store_reset) by one CTA of
// kMtThreads threads. The state is seeded by one thread (the recurrence is sequential); every block
// twist runs in the phases of its in-place dependencies -- words [0, 227) read old words only,
// [227, 454) and [454, 623) read words the previous phase wrote, word 623 reads the new words 0 and
// 396 -- each phase reading into registers before a barrier and writing after it.
constexpr int kMtThreads = 256;  // >= 227, the longest phase
__global__ void __launch_bounds__(kMtThreads) k_mt_outputs(uint32_t seed, int n, uint32_t *__restrict__ out) {
  __shared__ uint32_t mt[624];
  const int t = threadIdx.x;
  if (t == 0) {
    uint32_t prev = seed;
    mt[0] = prev;
    for (int i = 1; i < 624; ++i) {
      prev = 1812433253u * (prev ^ (prev >> 30)) + (uint32_t)i;
      mt[i] = prev;
    }
  }
  __syncthreads();
  constexpr int kPhase[5] = {0, 227, 454, 623, 624};
  for (int b0 = 0; b0 < n; b0 += 624) {
#pragma unroll
    for (int ph = 0; ph < 4; ++ph) {
      const int i = kPhase[ph] + t;  // a phase has at most 227 words: one per thread
      const bool mine = i < kPhase[ph + 1];
      uint32_t v = 0;
      if (mine) {
        const uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
        v = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1) ? 0x9908b0dfu : 0u);
      }
      __syncthreads();
      if (mine) mt[i] = v;
      __syncthreads();
    }
    for (int i = t; i < 624 && b0 + i < n; i += kMtThreads) {
      uint32_t y = mt[i];
      y ^= y >> 11;
      y ^= (y << 7) & 0x9d2c5680u;
      y ^= (y << 15) & 0xefc60000u;
      y ^= y >> 18;
      out[b0 + i] = y;
    }
  }
}

// The control and tree blocks store_reset writes, for positions [0, P.num_games) (first_game 0),
// and the work counter of k_analysis_persistent: ctr = {next position, failed positions, min error}.
__global__ void k_analysis_reset(TreeParams P, int32_t *__restrict__ ctr, int next0) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g == 0) ctr[0] = next0, ctr[1] = 0, ctr[2] = 0;
  if (g >= P.num_games) return;
  int32_t *c = P.ctl + (size_t)g * kCtlWords;
  for (int w = 0; w < kCtlWords; ++w) c[w] = 0;
  c[CW_PARITY] = g & 1;
  c[CW_SPARE] = 2;
  c[CW_MT_IDX] = 624;
  for (int p = 0; p < 2; ++p) {
    int32_t *tw = P.tree + ((size_t)g * 2 + p) * kTreeCtlWords;
    for (int w = 0; w < kTreeCtlWords; ++w) tw[w] = 0;
    tw[TW_ARENA] = p;
    tw[TW_ROOT_VISITS] = 1;
    tw[TW_ROOT_ALLV] = 1;
  }
}

// Analysis in one persistent launch: one CTA per SM holds kGames positions, one warp each (16 with
// bf16 / fp16 operands, 512 threads, the network on the first 256; 8 with bf16x3, 256 threads, one
// network tile on the first 128). A round is analysis_step of every warp's position, its requests
// appended to the CTA's rows [row0, row0 + kGames * spe) with one shared atomicAdd per position,
// then tc_forward over those rows, whose answers (move-major, leading dimension ld) the next round
// reads. The first wave is dealt round-robin (slot = warp * grid + block) so that a small batch
// spreads over every SM; a warp whose position finishes takes the next one from ctr[0] in the same
// round, and the CTA leaves once no warp holds a live position. A position's first round checks its
// state (valid_state); rejected ones and searches that fail get write_failed, counted in ctr[1], the
// most negative code in ctr[2]. A position's order of operations is k_analysis_iterate's, and a
// network row does not depend on the other rows of its batch: the outputs are cb200_analysis_run's.
template <int kMode, int kGames>
__global__ void __launch_bounds__(kGames * 32, 1)
    k_analysis_persistent(TreeParams P, int max_searches, const uint8_t *__restrict__ W,
                          const ulonglong2 *__restrict__ states, float *eval, float *probs, int ld,
                          ulonglong2 *packed, int32_t *ctr, AnalysisOut out) {
  static_assert(kGames == 8 || kGames == 16, "one or two network tiles per CTA");
  static_assert(ps_smem_bytes<kMode, kGames>() <= 227 * 1024, "bf16x3 fits with 8 games per CTA only");
  constexpr int kNetThreads = kGames == 8 ? 128 : kTcThreads;  // one tile or two
  constexpr int kTileRows = kNetThreads;                        // rows per tc_forward call
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
      if (lane == 0) next = atomicAdd(ctr, 1);
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
