// K7: persistent fused self-play for the phase with few live games.
//
// While thousands of games are live the lock-step loop [k_mlp_tc -> k_iterate] keeps every SM
// busy, but each launch lasts as long as its slowest game and every iteration pays two kernel
// boundaries. Once all live games fit on the GPU at 16 games per SM, one CTA per SM takes 8 or 16
// games and loops by itself:
//     game step of its games (one warp each: run_game = SelfPlayer::doIteration)
//  -> the tensor-core network on the <= 128 / 256 leaf positions they queued (tc_forward)
// without leaving the SM, so a CTA only ever waits for its own games. Requests and answers
// travel through CTA-private rows of small global buffers (L2 resident). Per-game order of
// operations is unchanged, hence so is every result (tests compare against the lock-step run).
#ifndef CORINTHO_B200_PERSISTENT_CUH
#define CORINTHO_B200_PERSISTENT_CUH

#include "mlp_tc.cuh"
#include "tree.cuh"

namespace cb200 {

constexpr int kPsRowsPerGame = 16;           // request rows reserved per game (needs spe <= 16)
// shared memory of a persistent CTA: the network's (one tile for 8 games, two for 16; bf16x3 holds
// hi and lo copies and fits with 8 games only), then one WarpSm per game
template <int kMode, int kGames>
__host__ __device__ constexpr size_t ps_tree_smem_off() {
  return (tc_smem_bytes(kGames == 8 ? 1 : 2, kMode == 2 ? 2 : 1) + 127) / 128 * 128;
}
template <int kMode, int kGames>
__host__ __device__ constexpr size_t ps_smem_bytes() {
  constexpr size_t bytes = ps_tree_smem_off<kMode, kGames>() + kGames * sizeof(WarpSm);
  static_assert(bytes <= 227 * 1024, "bf16x3 fits with 8 games per CTA only");
  return bytes;
}
// threads of a persistent CTA that run the network: one tile for 8 games, two for 16
template <int kGames>
__host__ __device__ constexpr int ps_net_threads() {
  static_assert(kGames == 8 || kGames == 16, "one or two network tiles per CTA");
  return kGames == 8 ? 128 : kTcThreads;
}

// kGames = 8 (one network tile) or 16 (two tiles) games per CTA, one warp each (256 / 512
// threads; the network is run by the first 256 or -- a single tile -- 128 of them). Games are dealt
// round-robin over the CTAs (slot = group * gridDim.x + blockIdx.x) so that every SM gets its share
// however few games are left. All CTAs stop at their next round boundary once `exit_done` games of
// this launch have finished (the host then deals the remaining games again). out[0] += games still
// live when the CTA stopped, out[1] = min error code, out[2] = max rounds executed by a CTA,
// out[3] = games finished during the launch.
template <int kMode, int kGames>
__global__ void __launch_bounds__(kGames * 32, 1)
    k_selfplay_persistent(TreeParams P, const uint8_t *__restrict__ W,
                          const uint8_t *__restrict__ W1, const int32_t *__restrict__ game_list,
                          int n_list, const float *eval0, const float *probs0, long pcs0,
                          float *eval, float *probs, int ld, ulonglong2 *packed, int max_rounds,
                          int exit_done, int iteration0, int32_t *out) {
  constexpr int kNetThreads = ps_net_threads<kGames>();
  const bool net_thread = threadIdx.x < kNetThreads;
  constexpr int kRows = kGames * kPsRowsPerGame;
  extern __shared__ __align__(128) uint8_t smem[];
  // [0] requests of this round (model 0), [1] live games, [2] error, [3] stop, [4] requests
  // for model 1 (two-model runs: W1 != nullptr, every CTA owns two row regions of kRows)
  __shared__ int32_t s_ctr[8];
  const bool two = W1 != nullptr;
  TcState S;
  if (net_thread) tc_setup(S, smem, kNetThreads, kMode == 2 ? 2 : 1);
  WarpSm *sm_all = reinterpret_cast<WarpSm *>(smem + ps_tree_smem_off<kMode, kGames>());
  const int grp = threadIdx.x / 32;
  const int slot = grp * gridDim.x + blockIdx.x;
  const int g = slot < n_list ? game_list[slot] : -1;
  const int row0 = blockIdx.x * kRows * (two ? 2 : 1);
  if (threadIdx.x == 0) s_ctr[2] = 0, s_ctr[3] = 0;  // published by the first barrier of the loop
  // games dealt to this CTA (all live at launch)
  int prev_live = ((int)n_list - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  if (prev_live > kGames) prev_live = kGames;
  if (prev_live < 0) prev_live = 0;
  int round = 0, live = 0;
  for (; round < max_rounds; ++round) {
    if (threadIdx.x == 0) s_ctr[0] = 0, s_ctr[1] = 0, s_ctr[4] = 0;
    __syncthreads();
    if (g >= 0) {
      const bool ext = round == 0;  // answers of the requests queued before this launch
      run_game<true>(P, g, sm_all[grp], ext ? eval0 : eval, ext ? probs0 : probs, 1,
                     ext ? pcs0 : (long)ld, nullptr, -1, iteration0 + round, 0, &s_ctr[0],
                     &s_ctr[1], &s_ctr[2], row0, packed, two ? kRows : 0);
    }
    __syncthreads();
    const int n = s_ctr[0], n1 = s_ctr[4];
    live = s_ctr[1];
    if (threadIdx.x == 0) {
      if (live < prev_live) atomicAdd(out + 3, prev_live - live);
      prev_live = live;
      if (*(volatile int32_t *)(out + 3) >= exit_done) s_ctr[3] = 1;
    }
    // every round ends with the network, so the answers of all queued requests are in the
    // CTA's rows whenever the kernel stops (a later launch continues from there)
    if (net_thread && n > 0)
      tc_forward<kMode>(S, W, packed + row0, n, 0, eval + row0, probs + row0, ld);
    if (net_thread && n1 > 0)
      tc_forward<kMode>(S, W1, packed + row0 + kRows, n1, 0, eval + row0 + kRows, probs + row0 + kRows, ld);
    __syncthreads();  // answers visible to every warp; counters read before they are cleared
    if (live == 0 || s_ctr[3]) {
      ++round;
      break;
    }
  }
  if (net_thread) tc_teardown(S);
  if (threadIdx.x == 0) {
    if (live) atomicAdd(out, live);
    if (s_ctr[2]) atomicMin(out + 1, s_ctr[2]);
    atomicMax(out + 2, round);
  }
}

}  // namespace cb200
#endif
