// K1: game-logic kernel (BASELINE.json configs[1]).
// Per state: 16 B read (cstate), 16 B written (legal mask + flags), 16 B written (next state);
// the optional 70-float NN encoding is written warp-cooperatively so stores stay coalesced.
// HBM-bound by construction; see DESIGN.md "K1" for the roofline arithmetic. Two kernels:
// k_game_step_encode when the encoding is requested, k_game_step_pairw otherwise. The forms
// measured against the latter in round 2 are in profiles/r02_k1_paired_variants.txt.
#ifndef CORINTHO_B200_GAME_STEP_CUH
#define CORINTHO_B200_GAME_STEP_CUH

#include "common.cuh"

namespace cb200 {

constexpr int kStepThreads = 256;

// Encoding form (the 70-float NN encoding is requested): one thread per state.
__global__ void __launch_bounds__(kStepThreads)
    k_game_step_encode(int64_t n, const ulonglong2 *__restrict__ states, uint64_t seed,
                       uint4 *__restrict__ mask_flags, ulonglong2 *__restrict__ next,
                       float *__restrict__ enc) {
  __shared__ ulonglong2 sm_states[kStepThreads];
  // 32-bit indices: the launcher refuses more than 2^31 - 2^20 states per call; the loop counter
  // is unsigned so that the last `+= stride` cannot wrap
  const unsigned stride = gridDim.x * kStepThreads;
  // every warp runs the same number of trips so the cooperative encode stays convergent
  const unsigned n_round = (unsigned)(((n + 31) / 32) * 32);
  for (unsigned iu = blockIdx.x * kStepThreads + threadIdx.x; iu < n_round; iu += stride) {
    const int i = (int)iu;
    const bool live = i < n;
    CState s{0, 0};
    if (live) {
      const ulonglong2 v = __ldg(states + i);
      s.w0 = v.x, s.w1 = v.y;
      uint32_t m[3];
      const bool lines = legal_moves_t<true>(s, m, DeviceLB());
      const int nl = __popc(m[0]) + __popc(m[1]) + __popc(m[2]);
      const int result = terminal_result(nl, lines);
      // compute the move for every state, keep it only where one exists
      // r % nl with nl <= 96: quotient estimate from floor(2^32 / nl) (one below at most), fix-up
      const uint32_t rnd = step_rnd(seed, (uint64_t)i), dv = (uint32_t)max(nl, 1);
      uint32_t rem = rnd - __umulhi(rnd, __ldg(d_inv32 + dv)) * dv;
      rem -= rem >= dv ? dv : 0u;
      const int pick = nth_move(m, (int)rem);
      const CState moved = do_move(s, pick & 127);
      const int chosen = nl > 0 ? pick : 0x7f;
      CState o;
      o.w0 = nl > 0 ? moved.w0 : s.w0, o.w1 = nl > 0 ? moved.w1 : s.w1;
      mask_flags[i] = make_uint4(m[0], m[1], m[2],
                                 (uint32_t)result | (lines ? 4u : 0u) | ((uint32_t)nl << 8) |
                                     ((uint32_t)chosen << 16));
      next[i] = make_ulonglong2(o.w0, o.w1);
    }
    // warp-cooperative write of 32 x 70 contiguous floats (game.cpp:45-58 layout)
    const int lane = threadIdx.x & 31;
    ulonglong2 *ws = sm_states + (threadIdx.x & ~31);
    ws[lane] = make_ulonglong2(s.w0, s.w1);
    __syncwarp();
    const int64_t base = i - lane;
    const int64_t left = n - base;
    const int cnt = left >= 32 ? 32 : (left > 0 ? (int)left : 0);
    float *out = enc + base * CB200_STATE_SIZE;
    for (int f = lane; f < cnt * CB200_STATE_SIZE; f += 32) {
      const int si = f / CB200_STATE_SIZE, j = f - si * CB200_STATE_SIZE;
      const ulonglong2 v = ws[si];
      out[f] = encode_elem(CState{v.x, v.y}, j);
    }
    __syncwarp();
  }
}

// Paired form helpers. 85 % of reachable positions contain no line, and for them the legal mask
// is the basic-rule mask; the line rules (category search, four table masks, capital fix-ups) are
// ~60 % of the instruction stream of one position per thread without the encoding. The paired kernel cuts the
// integer-ALU work per position (the ALU pipe is what bounds K1, DESIGN.md section 4):
//   * a thread takes TWO positions per trip (i and i + 256: both loads and all stores stay
//     coalesced) and runs the basic-rule mask and the "any line?" test on both at once, one
//     position in each 16-bit half of every plane register (basic_moves_pair);
//   * nth_move's last three levels and do_move's move decode are shared-memory tables
//     (nth_move_lut / do_move_lut, 4.3 KB per CTA);
//   * positions with a line are queued and finished later by full warps.
struct SmemLB {
  const uint32_t *p;
  __device__ __forceinline__ const uint32_t *operator()(int idx) const { return p + 4 * idx; }
};
struct SmemNthLut {
  const uint8_t *p;
  __device__ __forceinline__ uint32_t operator()(uint32_t i) const { return p[i]; }
};

// seed_c = seed + 0x9E3779B97F4A7C15 (computed once per thread): step_rnd's first line as one
// multiply-add
__device__ __forceinline__ void game_step_finish_lut(int i, const CState &s, const uint32_t m[3], bool lines,
                                                     uint64_t seed_c, uint4 *__restrict__ mask_flags,
                                                     ulonglong2 *__restrict__ next, const uint32_t *ML, SmemNthLut NL,
                                                     const uint32_t *inv32) {
  const int nl = __popc(m[0]) + __popc(m[1]) + __popc(m[2]);
  const uint32_t rnd = step_rnd_mix(seed_c + (uint64_t)(uint32_t)i * 0x9E3779B97F4A7C15ull);
  // rnd % nl as in k_game_step_encode; inv32[0] = 0 leaves a meaningless rem that nl == 0 never uses
  const uint32_t dv = (uint32_t)nl;
  uint32_t rem = rnd - __umulhi(rnd, inv32[dv]) * dv;
  rem -= rem >= dv ? dv : 0u;
  CState o = s;
  uint32_t tail = (lines ? (uint32_t)kResultLoss | 4u : (uint32_t)kResultDraw) | (0x7fu << 16);  // no legal move
  if (nl > 0) {
    const int pick = nth_move_lut(m, (int)rem, NL);
    o = do_move_lut(s, pick, ML);
    tail = (lines ? 4u : 0u) | ((uint32_t)nl << 8) | ((uint32_t)pick << 16);
  }
  mask_flags[i] = make_uint4(m[0], m[1], m[2], tail);
  next[i] = make_ulonglong2(o.w0, o.w1);
}

// Both positions of a thread finished together, without a branch: the two dependent chains
// (popcount -> rank -> nth_move -> table -> do_move) are independent of each other, so the
// compiler can interleave them; lanes whose position is queued (or absent) compute a discarded
// result in the slots they would idle in anyway. Only the stores are predicated. A position
// without a legal move draws a meaningless but in-range move id (nth_move_lut never leaves the
// tables) and keeps its state by a select.
__device__ __forceinline__ void game_step_finish_one_sel(const CState &s, const uint32_t m[3], uint32_t idx,
                                                         uint64_t seed_c, const uint32_t *ML, SmemNthLut NL,
                                                         const uint32_t *inv32, uint32_t &tail, CState &o) {
  const int nl = __popc(m[0]) + __popc(m[1]) + __popc(m[2]);
  const uint32_t rnd = step_rnd_mix(seed_c + (uint64_t)idx * 0x9E3779B97F4A7C15ull);
  const uint32_t dv = (uint32_t)nl;
  uint32_t rem = rnd - __umulhi(rnd, inv32[dv]) * dv;
  rem -= rem >= dv ? dv : 0u;
  const int pick = nth_move_lut(m, (int)rem, NL);
  const CState moved = do_move_lut(s, pick, ML);
  const bool any = nl > 0;
  o.w0 = any ? moved.w0 : s.w0, o.w1 = any ? moved.w1 : s.w1;
  tail = any ? (((uint32_t)nl << 8) | ((uint32_t)pick << 16)) : ((uint32_t)kResultDraw | (0x7fu << 16));
}

// K1, paired form with one queue per WARP. A single queue per CTA synchronises the CTA twice per
// trip: its ncu capture showed the warps of a CTA waiting together for their loads right after the
// barrier (long-scoreboard 7.2, barrier 2.5 stall cycles per issue, issue slots 66 % busy). Here
// every warp owns a queue of 96 entries and a warp-uniform count in a register:
//   * appending is two ballots and predicated stores (no atomics, no branch: the warp is still
//     converged right after basic_moves_pair);
//   * a warp flushes 32 queued positions whenever it has them -- __syncwarp only, no __syncthreads
//     inside the loop, so the 56 warps of an SM drift apart and cover each other's load latency;
//   * the next trip's two positions are requested before the current ones are processed;
//   * the positions without a line are finished by game_step_finish_one_sel, both at once.
__global__ void __launch_bounds__(kStepThreads, 1)
    k_game_step_pairw(int64_t n, const ulonglong2 *__restrict__ states, uint64_t seed,
                      uint4 *__restrict__ mask_flags, ulonglong2 *__restrict__ next) {
  constexpr int kWarps = kStepThreads / 32;
  constexpr int kWQ = 96;  // fewer than 32 entries before a trip, at most 64 more
  __shared__ ulonglong2 q_state[kWarps * kWQ];
  __shared__ uint4 q_mask[kWarps * kWQ];  // basic-rule mask (x, y, z) and the position's index (w)
  __shared__ __align__(16) uint32_t s_move[96 * kMoveLutWords];
  __shared__ __align__(16) uint8_t s_nth[256 * 8];
  __shared__ uint32_t s_inv[128];
  __shared__ __align__(16) uint32_t s_lb[103 * 4];  // line-breaker masks (1.6 KB): the flush reads four per position
  const int tid = threadIdx.x;
  if (tid < 103) reinterpret_cast<uint4 *>(s_lb)[tid] = reinterpret_cast<const uint4 *>(d_line_breakers)[tid];
  reinterpret_cast<uint2 *>(s_nth)[tid] = reinterpret_cast<const uint2 *>(d_nth_lut)[tid];
  if (tid < 128) s_inv[tid] = d_inv32[tid];
  if (tid < 96 * kMoveLutWords / 4)
    reinterpret_cast<uint4 *>(s_move)[tid] = reinterpret_cast<const uint4 *>(d_move_lut)[tid];
  __syncthreads();
  const uint32_t *ML = s_move;
  const SmemNthLut NL{s_nth};
  const int lane = tid & 31;
  const unsigned lt = (1u << lane) - 1u;
  ulonglong2 *qs = q_state + (tid >> 5) * kWQ;
  uint4 *qm = q_mask + (tid >> 5) * kWQ;
  int qn = 0;  // entries in this warp's queue (warp-uniform)
  const uint64_t seed_c = seed + 0x9E3779B97F4A7C15ull;
  constexpr int kTrip = 2 * kStepThreads;
  const unsigned un = (unsigned)n;
  const unsigned stride = gridDim.x * kTrip;  // unsigned: the last `+= stride` cannot wrap
  const unsigned n_round = (unsigned)(((n + kTrip - 1) / kTrip) * kTrip);  // every lane of a warp runs every trip
  const ulonglong2 none = make_ulonglong2(0ull, 0ull);  // empty board, no pieces: no move, no line
  unsigned base = blockIdx.x * kTrip;
  ulonglong2 pa = none, pb = none;
  if (base < n_round) {
    if (base + tid < un) pa = __ldg(states + base + tid);
    if (base + tid + kStepThreads < un) pb = __ldg(states + base + tid + kStepThreads);
  }
  for (; base < n_round; base += stride) {
    const unsigned ua = base + tid, ub = ua + kStepThreads;
    const bool ha = ua < un, hb = ub < un;
    const ulonglong2 va = pa, vb = pb;
    const unsigned na = ua + stride, nb = ub + stride;  // past n_round means past n
    pa = na < un ? __ldg(states + na) : none;
    pb = nb < un ? __ldg(states + nb) : none;
    const CState a{va.x, va.y}, b{vb.x, vb.y};
    uint32_t ma[3], mb[3];
    bool la, lb;
    basic_moves_pair(a, b, ma, mb, la, lb);
    const bool qa = ha && la, qb = hb && lb;
    const unsigned ba = __ballot_sync(kFull, qa), bb = __ballot_sync(kFull, qb);
    if (qa) {
      const int slot = qn + __popc(ba & lt);
      qs[slot] = va, qm[slot] = make_uint4(ma[0], ma[1], ma[2], ua);
    }
    qn += __popc(ba);
    if (qb) {
      const int slot = qn + __popc(bb & lt);
      qs[slot] = vb, qm[slot] = make_uint4(mb[0], mb[1], mb[2], ub);
    }
    qn += __popc(bb);
    uint32_t ta, tb;
    CState oa, ob;
    game_step_finish_one_sel(a, ma, ua, seed_c, ML, NL, s_inv, ta, oa);
    game_step_finish_one_sel(b, mb, ub, seed_c, ML, NL, s_inv, tb, ob);
    if (ha && !la) {
      mask_flags[ua] = make_uint4(ma[0], ma[1], ma[2], ta);
      next[ua] = make_ulonglong2(oa.w0, oa.w1);
    }
    if (hb && !lb) {
      mask_flags[ub] = make_uint4(mb[0], mb[1], mb[2], tb);
      next[ub] = make_ulonglong2(ob.w0, ob.w1);
    }
    __syncwarp();  // the appended entries are visible to the whole warp
    while (qn >= 32) {  // warp-uniform
      qn -= 32;
      const ulonglong2 v = qs[qn + lane];
      const uint4 w = qm[qn + lane];
      const CState s{v.x, v.y};
      uint32_t m[3] = {w.x, w.y, w.z};
      const bool lines = line_rules_on_basic(s, m, SmemLB{s_lb});
      game_step_finish_lut((int)w.w, s, m, lines, seed_c, mask_flags, next, ML, NL, s_inv);
    }
    __syncwarp();  // flush reads done before the next trip's appends reuse the slots
  }
  // drain: every warp is left with fewer than 32 entries; pooled over the CTA (fewer than 256) so
  // that full warps process them instead of eight half-empty ones
  __shared__ int s_left[kWarps];
  if (lane == 0) s_left[tid >> 5] = qn;
  __syncthreads();
  int total = 0, src = -1;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) {
    const int c = s_left[w];
    if (src < 0 && tid < total + c) src = w * kWQ + (tid - total);
    total += c;
  }
  if (src >= 0) {
    const ulonglong2 v = q_state[src];
    const uint4 w = q_mask[src];
    const CState s{v.x, v.y};
    uint32_t m[3] = {w.x, w.y, w.z};
    const bool lines = line_rules_on_basic(s, m, SmemLB{s_lb});
    game_step_finish_lut((int)w.w, s, m, lines, seed_c, mask_flags, next, ML, NL, s_inv);
  }
}

// resident CTAs of the paired kernel per SM (register- and shared-memory-limited), asked once
inline int k1_pair_ctas_per_sm() {
  static int ctas = 0;
  if (ctas == 0) {
    int v = 0;
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_game_step_pairw, kStepThreads, 0);
    ctas = e == cudaSuccess && v >= 1 ? v : 4;
  }
  return ctas;
}

inline int launch_game_step(int64_t n, const void *d_states, uint64_t seed, void *d_mask_flags,
                            void *d_next, void *d_enc) {
  if (n <= 0) return CB200_OK;
  if (n > (int64_t)0x7FF00000) return set_error(CB200_ERR_ARG, "cb200_game_step: at most 2^31 - 2^20 states per call");
  int rc = ensure_tables();
  if (rc != CB200_OK) return rc;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (d_enc) {
    // persistent-style grid: a multiple of the SM count, 8 resident CTAs of 256 threads per SM
    const int64_t want = (n + kStepThreads - 1) / kStepThreads;
    const int64_t cap = (int64_t)sms * 8 * 4;
    const int grid = (int)(want < cap ? want : cap);
    k_game_step_encode<<<grid, kStepThreads, 0, cur_stream()>>>(
        n, (const ulonglong2 *)d_states, seed, (uint4 *)d_mask_flags, (ulonglong2 *)d_next,
        (float *)d_enc);
  } else {
    // 8 waves of CTAs, each looping over its share
    const int64_t want = (n + 2 * kStepThreads - 1) / (2 * kStepThreads);
    const int64_t cap = (int64_t)sms * k1_pair_ctas_per_sm() * 8;
    const int grid = (int)(want < cap ? want : cap);
    k_game_step_pairw<<<grid, kStepThreads, 0, cur_stream()>>>(
        n, (const ulonglong2 *)d_states, seed, (uint4 *)d_mask_flags, (ulonglong2 *)d_next);
  }
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  return CB200_OK;
}

}  // namespace cb200
#endif
