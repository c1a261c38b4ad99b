// K2-K6: the self-play game step -- one warp per game executes
// SelfPlayer::doIteration (corintho_ai/cpp/src/selfplayer.cpp:115-122) for it:
//   eval ingest + backup   TrainMC::receiveEval      trainmc.cpp:269-296 (212-267)
//   PUCT select / expand   TrainMC::search           trainmc.cpp:602-696 (chooseNext 540-600)
//   terminal deduction     TrainMC::propagateTerminal trainmc.cpp:497-538
//   move choice, re-root   TrainMC::chooseMove*      trainmc.cpp:110-137, 298-495
//   turn hand-over         SelfPlayer::chooseMoveAndContinue selfplayer.cpp:246-291
//
// Data layout (HBM, per game): three node arenas (two trees + one spare for re-rooting), each a
// bump-allocated array of 32-bit words holding node records
//     header[8]  w0..w3 cstate, w4 = n_legal | depth<<8, w5 = denominator (f32 bits)
//     slot[n][4] one 16-byte slot per legal move in ascending id order:
//                {child evaluation_ f32, child visits_ i32, child record offset,
//                 move | prior<<7 | result<<16 | all_visited<<19 | has_child<<20 |
//                 child_n_legal<<21 | child_has_children<<28}
// A node's statistics live in its parent's slot, so PUCT selection at a node is ONE coalesced
// read of header+slots (lane e loads slots e, e + 32, ... as uint4) and virtual loss is a plain store.
// Two games per warp (16 lanes each) were measured on a B200 and were slower: fewer warp
// instructions per game step, but a longer dependent chain per game, and the step is bound by
// that chain (DESIGN.md section 8).
// The root record is at word root_off (re-rooting is in place; the kept subtree is compacted
// into the spare arena only when room runs out); root statistics are in the per-tree control
// block. The per-game context (Ctx) lives in registers: every device function below is
// force-inlined into k_iterate, which has a single TrainMC::doIteration call site.
// Float expression types follow the reference literally (double intermediates, no FMA
// contraction): explicit __f*_rn / __d*_rn intrinsics are used for every rounded operation.
#ifndef CORINTHO_B200_TREE_CUH
#define CORINTHO_B200_TREE_CUH

#include "common.cuh"

namespace cb200 {

// Straggler instrumentation (tools/prof_timeline.py): build with -DCB200_PHASE_PROF=1 to record
// per-phase cycles; off by default so that the hot loops carry no clock reads.
#ifndef CB200_PHASE_PROF
#define CB200_PHASE_PROF 0
#endif
#if CB200_PHASE_PROF
#define CB_CLOCK() clock64()
#define CB_PROF(...) __VA_ARGS__
#else
#define CB_CLOCK() 0ll
#define CB_PROF(...)
#endif

constexpr int kMaxPath = 64;
constexpr int kPendWords = 2 + kMaxPath;  // leaf_off, path_len, path[kMaxPath]
constexpr int kMaxSamples = 64;
constexpr int kVsqrtCap = 2048;  // entries of the c_puct*sqrt(visits) table
constexpr int kTreeWarps = 4;    // warps (= games) per CTA of the lock-step kernels
constexpr int kCtlWords = 20;  // CW_* below; words 12-16 belong to Match (match.cuh)
constexpr int kTreeCtlWords = 12;

enum CtlWord {
  CW_TO_PLAY = 0, CW_PARITY, CW_RESULT, CW_MATE_TURN, CW_N_SAMPLES, CW_N_PENDING, CW_ERROR,
  CW_DONE, CW_SPARE, CW_MT_IDX, CW_REQ_BASE, CW_YIELD
};
enum TreeWord {
  TW_ARENA = 0, TW_HAS_ROOT, TW_USED, TW_ROOT_EVAL, TW_ROOT_VISITS, TW_ROOT_RESULT, TW_ROOT_ALLV,
  TW_SEARCHES_DONE, TW_ROOT_OFF
};

struct TreeParams {
  int num_games, first_game, total_games;
  int max_searches, spe;
  float c_puct, epsilon;
  const float *vsqrt;        // [kVsqrtCap] float(double(c_puct) * sqrt(double(i)))
  int testing;
  uint32_t arena_words;
  uint32_t *arenas;          // [G][3][arena_words]
  int32_t *ctl;              // [G][kCtlWords]
  int32_t *tree;             // [G][2][kTreeCtlWords]
  uint32_t *mt;              // [G][624]
  uint32_t *pending;         // [G][spe][kPendWords]
  ulonglong2 *leaf_state;    // [G][spe]
  ulonglong2 *sample_state;  // [G][kMaxSamples]
  float *sample_probs;       // [G][kMaxSamples][96]
  long long *counters;       // [G][4] simulations, moves, leaf evals, searches so far
  // fused (device-resident) mode: the kernel instance covers games [game_begin, game_end) of one
  // stream group; request rows are handed out with one atomicAdd per game
  int game_begin, game_end;
  int group_row0;            // first request row owned by this group
  int32_t *group_ctr;        // [0..1] request count per parity, [2..3] live games per parity, [4] error
  ulonglong2 *packed;        // [num_games*spe] leaf cstates in request-row order
  // fused lock-step mode: live_list[game_begin + i], i < *live_count, are the group's games that
  // were not finished when the list was last rebuilt (k_group_live_list), so that finished games
  // do not leave half-empty warps behind; the lock-step game step launches only these
  const int32_t *live_list;
  const int32_t *live_count;
  // fused mode: a game whose doIteration needs more than this many select levels + searches in
  // one launch parks (keeps its partial request list, asks for no evaluation) and resumes in the
  // next launch, so that one long iteration does not hold back every other game; 0 = never
  int yield_budget;
  // per-game text logs (selfplayer.cpp:124-204): the first n_logged games of this trainer write
  // one record per move (layout: kLog* below) that the host formats; null = no logged games
  int n_logged;
  uint32_t *log_buf;         // [n_logged][kLogMaxMoves][kLogWords]
  int32_t *log_count;        // [n_logged] records written
  // optional straggler instrumentation (null = off): [0..2] max cycles of one warp in ingest /
  // search / move phases, [3..5] summed cycles, [6] rolled-back searches, [7] words re-rooted
  unsigned long long *phase_prof;
};

constexpr int kFlatCap = 448;  // legal-move slots processed per flat ingest chunk
// per-game scratch in shared memory (one per warp)
struct WarpSm {
  __align__(16) float f[100];
  uint32_t node[kMaxPath + 1];
  uint32_t slot[kMaxPath + 1];
  // flat eval-ingest scratch (receive_eval): per-element and per-leaf arrays
  float fval[kFlatCap];
  float dval[kFlatCap];
  uint8_t mv[kFlatCap];
  uint8_t own[kFlatCap];  // leaf (lane) owning each flat element
  uint32_t l_off[32];
  int l_pre[33];
  float l_a[32];
  float l_b[32];
};

// ---- slot word 3 ---------------------------------------------------------------------------
__device__ __forceinline__ int s3_move(uint32_t w) { return w & 0x7f; }
__device__ __forceinline__ int s3_prior(uint32_t w) { return (w >> 7) & 0x1ff; }
__device__ __forceinline__ int s3_result(uint32_t w) { return (w >> 16) & 7; }
__device__ __forceinline__ bool s3_allv(uint32_t w) { return (w >> 19) & 1; }
__device__ __forceinline__ bool s3_has(uint32_t w) { return (w >> 20) & 1; }
__device__ __forceinline__ int s3_cnl(uint32_t w) { return (w >> 21) & 0x7f; }
__device__ __forceinline__ bool s3_gc(uint32_t w) { return (w >> 28) & 1; }
constexpr uint32_t kS3Allv = 1u << 19, kS3Has = 1u << 20, kS3Gc = 1u << 28;

__device__ __forceinline__ bool r_known(int r) { return r != kResultNone; }
__device__ __forceinline__ bool r_terminal(int r) { return r == kResultLoss || r == kResultDraw; }
__device__ __forceinline__ bool r_won(int r) { return r == kDeducedWin; }
__device__ __forceinline__ bool r_lost(int r) { return r == kResultLoss || r == kDeducedLoss; }
__device__ __forceinline__ bool r_drawn(int r) { return r == kResultDraw || r == kDeducedDraw; }

__device__ __forceinline__ void prefetch_l1(const void *p) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}
__device__ __forceinline__ uint4 ld4(const uint32_t *p) {
  return *reinterpret_cast<const uint4 *>(p);
}
__device__ __forceinline__ void st4(uint32_t *p, uint4 v) { *reinterpret_cast<uint4 *>(p) = v; }
__device__ __forceinline__ uint32_t fkey(float f) {  // order-preserving float -> uint
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
constexpr uint32_t kKeyNegInf = 0x007FFFFFu;

// 1/x for a positive normal double: rcp.approx.ftz.f64 (>= 20 good bits) refined twice
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = fma(r, fma(-x, r, 1.0), r);
  r = fma(r, fma(-x, r, 1.0), r);
  return r;
}

// Per-warp view of one game. Every member except lane is uniform over the warp.
struct Ctx {
  int lane = threadIdx.x & 31;
  // game control (selfplayer.h:88-111)
  int to_play, parity, result, mate_turn, n_samples, n_pending, error, spare, mt_idx;
  int d_sims, d_evals, d_moves, d_searches;  // work done in this launch (< 2^31 by far)
#if CB200_PHASE_PROF
  long long t_ingest, t_search, t_move, n_none, n_copy;  // instrumented build only: these would
  long long t_sel, t_exp, n_lvl, n_exp, n_exact;         // otherwise hold 20 registers for nothing
#endif
  int work, yielded;
  // current tree (trainmc.h:160-188)
  int cur_p, arena, has_root;
  uint32_t used;
  uint32_t root_off;  // word offset of the root record in its arena (re-rooting is in place)
  float root_eval;
  int root_visits, root_result, root_allv, searches_done;
  uint32_t *base;
  // per-game storage
  uint32_t *arenas, *mt, *pending;
  int32_t *tree_ctl;
  ulonglong2 *leaf_state, *sample_state;
  float *sample_probs;
};

// ---- collectives over the warp of one game ---------------------------------------------------
__device__ __forceinline__ void g_sync(const Ctx &) { __syncwarp(kFull); }
__device__ __forceinline__ unsigned g_ballot(const Ctx &, bool p) { return __ballot_sync(kFull, p); }
__device__ __forceinline__ bool g_all(const Ctx &, bool p) { return __all_sync(kFull, p); }
template <class T> __device__ __forceinline__ T g_shfl(const Ctx &, T v, int src) {
  return __shfl_sync(kFull, v, src);
}
template <class T> __device__ __forceinline__ T g_shfl_up(const Ctx &, T v, int d) {
  return __shfl_up_sync(kFull, v, d);
}
__device__ __forceinline__ int g_max(const Ctx &, int v) { return __reduce_max_sync(kFull, v); }
__device__ __forceinline__ uint32_t g_max(const Ctx &, uint32_t v) { return __reduce_max_sync(kFull, v); }
__device__ __forceinline__ int g_min(const Ctx &, int v) { return __reduce_min_sync(kFull, v); }
__device__ __forceinline__ int g_add(const Ctx &, int v) { return __reduce_add_sync(kFull, v); }
__device__ __forceinline__ unsigned g_match(const Ctx &, uint32_t v) { return __match_any_sync(kFull, v); }

__device__ __forceinline__ uint32_t g_incl_scan(const Ctx &c, uint32_t v) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = g_shfl_up(c, v, d);
    if (c.lane >= d) v += o;
  }
  return v;
}

__device__ __forceinline__ void load_tree(Ctx &c, const TreeParams &P, int p) {
  const int32_t *t = c.tree_ctl + p * kTreeCtlWords;
  const int4 a = *reinterpret_cast<const int4 *>(t);
  const int4 b = *reinterpret_cast<const int4 *>(t + 4);
  c.cur_p = p;
  c.arena = a.x, c.has_root = a.y, c.used = (uint32_t)a.z, c.root_eval = __int_as_float(a.w);
  c.root_visits = b.x, c.root_result = b.y, c.root_allv = b.z, c.searches_done = b.w;
  c.root_off = (uint32_t)t[TW_ROOT_OFF];
  c.base = c.arenas + (size_t)c.arena * P.arena_words;
}
__device__ __forceinline__ void store_tree(Ctx &c) {
  if (c.lane == 0) {
    int32_t *t = c.tree_ctl + c.cur_p * kTreeCtlWords;
    *reinterpret_cast<int4 *>(t) =
        make_int4(c.arena, c.has_root, (int)c.used, __float_as_int(c.root_eval));
    *reinterpret_cast<int4 *>(t + 4) =
        make_int4(c.root_visits, c.root_result, c.root_allv, c.searches_done);
    t[TW_ROOT_OFF] = (int)c.root_off;
  }
  g_sync(c);
}

// ---- per-game MT19937 (std::mt19937 stream shared by both trees, selfplayer.h:88) -----------
// The 624-word state is a ring that is regenerated lazily: word p of the next generation is
//   new[p] = old[p + 397] ^ twist(old[p], old[p + 1])        (indices mod 624),
// computed right before it is drawn. Going through the ring in order this is exactly
// std::mt19937's block twist (positions below p already hold the new generation, which is what
// new[p] needs for p >= 227 and for p = 623), but the work is spread evenly over the draws
// instead of arriving as one 624-word twist at a data-dependent time (1 670 -> 570 warp
// instructions per game iteration, DESIGN.md section 8). mt_idx = position of the next word
// (624 = wrap to 0 first).
__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= y >> 18;
  return y;
}
__device__ __forceinline__ uint32_t mt_next_word(const uint32_t *mt, int p) {
  const uint32_t a = mt[p], b = mt[p + 1 == 624 ? 0 : p + 1];
  const uint32_t m = mt[p + 397 >= 624 ? p + 397 - 624 : p + 397];
  const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
  return m ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}
__device__ __forceinline__ uint32_t rng_one(Ctx &c) {
  if (c.mt_idx >= 624) c.mt_idx = 0;
  const uint32_t w = mt_next_word(c.mt, c.mt_idx);  // every lane reads the same three words
  g_sync(c);
  if (c.lane == 0) c.mt[c.mt_idx] = w;
  g_sync(c);
  c.mt_idx += 1;
  return mt_temper(w);
}

__device__ __forceinline__ void copy_words(uint32_t *dst, const uint32_t *src, uint32_t nwords,
                                           int lane) {
  const uint4 *s = reinterpret_cast<const uint4 *>(src);
  uint4 *d = reinterpret_cast<uint4 *>(dst);
  for (uint32_t i = lane; i < (nwords >> 2); i += 32) d[i] = s[i];
}

// ---- node construction (Node ctor + initializeEdges, node.cpp:31-39, 256-283) ---------------
__device__ __forceinline__ int make_record(Ctx &c, const TreeParams &P, const CState &st,
                                           int depth, int &result) {
  uint32_t m[3];
  const bool lines = legal_moves(st, m, DeviceLB());
  const int n0 = __popc(m[0]), n1 = __popc(m[1]), n2 = __popc(m[2]);
  const int n = n0 + n1 + n2;
  const uint32_t off = c.used;
  result = kResultNone;
  if (off + 8u + 4u * (uint32_t)n > P.arena_words) {
    c.error = CB200_ERR_OVERFLOW;
    return -1;
  }
  uint32_t *r = c.base + off;
  if (c.lane == 0) {
    st4(r, make_uint4((uint32_t)st.w0, (uint32_t)(st.w0 >> 32), (uint32_t)st.w1,
                      (uint32_t)(st.w1 >> 32)));
    st4(r + 4, make_uint4((uint32_t)n | ((uint32_t)depth << 8), 0u, 0u, 0u));
  }
  // slot of move id b = rank of bit b among the legal moves; lane l writes ids l, l + 32, l + 64
#pragma unroll
  for (int w = 0; w < 3; ++w) {
    const int pre = w == 0 ? 0 : (w == 1 ? n0 : n0 + n1);
    const int b = c.lane;
    if ((m[w] >> b) & 1u)
      st4(r + 8 + 4 * (pre + __popc(m[w] & ((1u << b) - 1u))),
          make_uint4(0u, 0u, 0u, (uint32_t)(32 * w + b)));
  }
  c.used = off + 8u + 4u * (uint32_t)n;
  result = terminal_result(n, lines);
  g_sync(c);
  return n;
}

__device__ __forceinline__ CState rec_state(const uint32_t *r) {
  const uint4 h = ld4(r);
  CState s;
  s.w0 = (uint64_t)h.x | ((uint64_t)h.y << 32);
  s.w1 = (uint64_t)h.z | ((uint64_t)h.w << 32);
  return s;
}

// Single-node tree (Node(game, depth) node.cpp:25-29; reset paths trainmc.cpp:397-404,461-468)
__device__ __forceinline__ void fresh_tree(Ctx &c, const TreeParams &P, const CState &st,
                                           int depth) {
  c.used = 0;
  c.root_off = 0;
  int result;
  make_record(c, P, st, depth, result);
  c.has_root = 1;
  c.root_eval = 0.0f;
  c.root_visits = 1;
  c.root_result = result;
  c.root_allv = 1;
}

// queue the root for evaluation (trainmc.cpp:150-152, 160-162, 198-200)
__device__ __forceinline__ void request_root(Ctx &c) {
  if (c.lane == 0) {
    uint32_t *pd = c.pending + c.n_pending * kPendWords;
    const uint4 h = ld4(c.base + c.root_off);
    pd[0] = c.root_off, pd[1] = (c.base[c.root_off + 4] & 0xffu) << 8;  // path length 0 | n_legal << 8
    c.leaf_state[c.n_pending] = make_ulonglong2((uint64_t)h.x | ((uint64_t)h.y << 32),
                                                (uint64_t)h.z | ((uint64_t)h.w << 32));
  }
  c.n_pending += 1;
  g_sync(c);
}

// ---- TrainMC::moveDown (trainmc.cpp:475-495): child behind root slot e becomes the root -----
// Breadth-first copy of the kept subtree into the spare arena; only records that have
// children are queued for scanning (queue grows down from the top of the target arena).
__device__ __forceinline__ void move_down(Ctx &c, const TreeParams &P, int e) {
  const uint32_t *src = c.base;
  uint32_t *dst = c.arenas + (size_t)c.spare * P.arena_words;
  const uint4 s = ld4(src + c.root_off + 8 + 4 * e);
  c.root_eval = __uint_as_float(s.x);
  c.root_visits = (int)s.y;
  c.root_result = s3_result(s.w);
  c.root_allv = s3_allv(s.w) ? 1 : 0;
  // Re-root in place while the arena still has room for a full move's worth of new nodes
  // (max_searches nodes of up to 48 slots); the discarded siblings stay behind as garbage.
  // Only when the room runs out is the kept subtree compacted into the spare arena.
  const uint32_t reserve = (uint32_t)(P.max_searches + 64) * (8u + 4u * 48u);
  if (c.used + reserve <= P.arena_words) {
    c.root_off = s.z;
    c.searches_done = 0;
    return;
  }
  const uint32_t sz = 8u + 4u * (uint32_t)s3_cnl(s.w);
  copy_words(dst, src + s.z, sz, c.lane);
  uint32_t alloc = sz;
  int q_head = 0, q_tail = 0;
  uint32_t *q = dst + (P.arena_words - 1);
  if (s3_gc(s.w)) {
    if (c.lane == 0) q[0] = 0;
    q_tail = 1;
  }
  g_sync(c);
  const uint32_t lt = (1u << c.lane) - 1u;
  while (q_head < q_tail) {
    const uint32_t roff = *(volatile uint32_t *)(q - q_head);
    ++q_head;
    uint32_t *r = dst + roff;
    const int rn = (int)(r[4] & 0xffu);
    for (int e0 = 0; e0 < rn; e0 += 32) {
      const int ee = e0 + c.lane;
      bool has = false, gc = false;
      uint32_t coff = 0, csz = 0;
      if (ee < rn) {
        const uint4 cs = ld4(r + 8 + 4 * ee);
        has = s3_has(cs.w);
        if (has) csz = 8u + 4u * (uint32_t)s3_cnl(cs.w), coff = cs.z, gc = s3_gc(cs.w);
      }
      const uint32_t incl = g_incl_scan(c, csz);
      const uint32_t excl = incl - csz;
      const uint32_t total = g_shfl(c, incl, 31);
      const unsigned gm = g_ballot(c, gc);
      const int ngc = __popc(gm);
      if (alloc + total + (uint32_t)(q_tail + ngc) > P.arena_words) {
        c.error = CB200_ERR_OVERFLOW;
        return;
      }
      if (has) r[8 + 4 * ee + 2] = alloc + excl;
      if (gc) *(q - (q_tail + __popc(gm & lt))) = alloc + excl;
      q_tail += ngc;
      unsigned hm = g_ballot(c, has);
      while (hm) {
        const int sl = __ffs((int)hm) - 1;
        hm &= hm - 1;
        const uint32_t so = g_shfl(c, coff, sl);
        const uint32_t sw = g_shfl(c, csz, sl);
        const uint32_t dof = alloc + g_shfl(c, excl, sl);
        copy_words(dst + dof, src + so, sw, c.lane);
      }
      alloc += total;
    }
    g_sync(c);
  }
  const int old = c.arena;
  c.arena = c.spare;
  c.spare = old;
  c.base = dst;
  c.used = alloc;
  c.root_off = 0;
  c.searches_done = 0;
  CB_PROF(c.n_copy += alloc;)
}

// ---- TrainMC::receiveEval (trainmc.cpp:269-296), latency-oriented restatement ----------------
// probs element (answer row k, move m) = probs[k * prs + m * pcs]: row-major [n][96] from the
// host API (prs 96, pcs 1), move-major [96][ld] from the tensor-core network (prs 1, pcs ld).
// Same arithmetic, in the same order per leaf, as the reference loop, but organised so that the
// loads of all pending leaves (processed 32 at a time) are in flight together:
//   "flat" phases  : one lane per legal-move slot over the concatenation of all leaves
//                    (the MT19937 draw of flat element i is simply draw number i); the leaf an
//                    element belongs to comes from a byte array filled once per chunk;
//   "leaf" phases  : one lane per leaf for the order-dependent float sums / max / integer sum;
//   backup         : per tree level, the lanes whose paths meet in the same slot are grouped with
//                    __match_any_sync and the lowest lane applies the adds in leaf order.
__device__ __forceinline__ void receive_eval(Ctx &c, const TreeParams &P, WarpSm &sm,
                                             const float *eval, const float *probs, long prs,
                                             long pcs) {
  constexpr int kE = 4;       // flat elements per lane per trip
  constexpr int kTrip = 128;  // flat elements per trip
  const int np_all = c.n_pending;
  const int lane = c.lane;
  const int prs32 = (int)prs, pcs32 = (int)pcs;  // element offsets fit 31 bits (<= 96 * rows)
  for (int b0 = 0; b0 < np_all; b0 += 32) {
  const int np = min(32, np_all - b0);
  const float *eval_b = eval + b0;
  const float *probs_b = probs + (long)b0 * prs;
  // ---- leaf phase 0: pending records (leaf offset, path length | n_legal << 8)
  uint32_t my_off = 0;
  int my_n = 0, my_plen = 0;
  float my_ev = 0.0f;
  const uint32_t *my_pd = c.pending + (b0 + lane) * kPendWords;
  if (lane < np) {
    const uint2 h = *reinterpret_cast<const uint2 *>(my_pd);
    my_off = h.x;
    my_plen = (int)(h.y & 0xffu);
    my_n = (int)(h.y >> 8);
    my_ev = eval_b[lane];
  }
  // path slots of the first four levels: in flight while the priors are processed
  uint32_t path4[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) path4[u] = (lane < np && my_plen > u) ? my_pd[2 + u] : 0u;
  const int incl = (int)g_incl_scan(c, (uint32_t)my_n);
  sm.l_pre[lane] = incl - my_n;
  if (lane == 31) sm.l_pre[32] = incl;
  sm.l_off[lane] = my_off;
  g_sync(c);
  for (int k0 = 0; k0 < np;) {
    // chunk [k0, k1): as many leaves as fit in the scratch arrays
    const int base_i = sm.l_pre[k0];
    // first leaf k >= k0 whose end no longer fits (prefix sums are monotone): one ballot
    const bool fits = lane >= k0 && lane < np && sm.l_pre[lane + 1] - base_i <= kFlatCap;
    const unsigned fm = g_ballot(c, fits) >> k0;
    int k1 = k0 + (fm == 0xffffffffu ? 32 : __ffs((int)~fm) - 1);
    if (k1 == k0) k1 = k0 + 1;  // a single leaf always goes through (checked below)
    const int T = sm.l_pre[k1] - base_i;
    if (T > kFlatCap) {  // a single leaf with more than kFlatCap moves cannot exist (<= 96)
      c.error = CB200_ERR_STATE;
      return;
    }
    const bool mine = lane >= k0 && lane < k1;
    const int my_i0 = sm.l_pre[lane] - base_i;
    const int my_cnt = mine ? my_n : 0;
    const int nmax = g_max(c, my_cnt);
#pragma unroll 4
    for (int j = 0; j < nmax; ++j)
      if (j < my_cnt) sm.own[my_i0 + j] = (uint8_t)lane;
    g_sync(c);
    // ---- flat phase 1: move ids and network priors of every legal move (getFilteredProbs).
    // kE elements per lane per trip; the slot words of the next trip are requested before the
    // priors of this one are consumed.
    uint32_t w3n[kE];
#pragma unroll
    for (int u = 0; u < kE; ++u) {
      const int i = lane + 32 * u;
      w3n[u] = 0;
      if (i < T) {
        const int k = sm.own[i];
        w3n[u] = c.base[sm.l_off[k] + 8 + 4 * (i + base_i - sm.l_pre[k]) + 3];
      }
    }
    for (int i0 = 0; i0 < T; i0 += kTrip) {
      uint32_t w3[kE];
      float pv4[kE];
#pragma unroll
      for (int u = 0; u < kE; ++u) {
        const int i = i0 + lane + 32 * u;
        w3[u] = w3n[u];
        pv4[u] = 0.0f;
        if (i < T) pv4[u] = probs_b[(int)sm.own[i] * prs32 + s3_move(w3[u]) * pcs32];
      }
      if (i0 + kTrip < T) {
#pragma unroll
        for (int u = 0; u < kE; ++u) {
          const int i = i0 + kTrip + lane + 32 * u;
          w3n[u] = 0;
          if (i < T) {
            const int k = sm.own[i];
            w3n[u] = c.base[sm.l_off[k] + 8 + 4 * (i + base_i - sm.l_pre[k]) + 3];
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kE; ++u) {
        const int i = i0 + lane + 32 * u;
        if (i < T) sm.mv[i] = (uint8_t)s3_move(w3[u]), sm.fval[i] = pv4[u];
      }
    }
    // ---- flat phase 2: one MT19937 draw per slot, in order (generateDirichlet). The state words
    // are regenerated where they are drawn (see mt_next_word): per trip every lane computes its
    // new words from the old ring contents, then the ring is updated. A trip spans at most
    // kTrip <= 128 consecutive positions, fewer than the 227 that separate a word from the
    // newest word it depends on.
    for (int done = 0; done < T;) {
      if (c.mt_idx >= 624) c.mt_idx = 0;
      const int seg = min(624 - c.mt_idx, T - done);
      for (int i0 = 0; i0 < seg; i0 += kTrip) {
        uint32_t y[kE];
#pragma unroll
        for (int u = 0; u < kE; ++u) {
          const int i = i0 + lane + 32 * u;
          y[u] = i < seg ? mt_next_word(c.mt, c.mt_idx + i) : 0u;
        }
        g_sync(c);
        float g[kE];
#pragma unroll
        for (int u = 0; u < kE; ++u) g[u] = d_gamma[mt_temper(y[u]) & 1023u];
#pragma unroll
        for (int u = 0; u < kE; ++u) {
          const int i = i0 + lane + 32 * u;
          if (i < seg) c.mt[c.mt_idx + i] = y[u], sm.dval[done + i] = g[u];
        }
        g_sync(c);
      }
      c.mt_idx += seg;
      done += seg;
    }
    g_sync(c);
    // ---- leaf phase 3: both float sums in edge order;
    // scalar = 1/sum * (1 - eps), dscalar = 1/noise sum * eps
    {
      float sum = 0.0f, dsum = 0.0f;
#pragma unroll 4
      for (int j = 0; j < nmax; ++j)
        if (j < my_cnt) {
          sum = __fadd_rn(sum, sm.fval[my_i0 + j]);
          dsum = __fadd_rn(dsum, sm.dval[my_i0 + j]);
        }
      if (mine) {
        sm.l_a[lane] = __double2float_rn(
            __dmul_rn(__drcp_rn((double)sum), (double)__fsub_rn(1.0f, P.epsilon)));
        sm.l_b[lane] =
            __double2float_rn(__dmul_rn(__drcp_rn((double)dsum), (double)P.epsilon));
      }
    }
    g_sync(c);
    // ---- flat phase 4: weighted = filtered*scalar + dirichlet*dscalar (setProbs)
#pragma unroll 2
    for (int i = lane; i < T; i += 32) {
      const int k = sm.own[i];
      sm.fval[i] = __fadd_rn(__fmul_rn(sm.fval[i], sm.l_a[k]), __fmul_rn(sm.dval[i], sm.l_b[k]));
    }
    g_sync(c);
    // ---- leaf phase 5: max (from 0.0f), denom = 511 / max. std::max(w, max) keeps a NaN w and
    // drops a NaN max, where fmaxf would drop the NaN w (an infinite probability makes one).
    {
      float mx = 0.0f;
#pragma unroll 4
      for (int j = 0; j < nmax; ++j)
        if (j < my_cnt) {
          const float w = sm.fval[my_i0 + j];
          mx = w < mx ? mx : w;
        }
      if (mine) sm.l_a[lane] = __fdiv_rn(511.0f, mx);
    }
    g_sync(c);
    // ---- flat phase 6: 9-bit integer priors. A leaf is evaluated before it can get children,
    // so its slot words are still {0, 0, 0, move}: the new word is move | prior << 7.
#pragma unroll 2
    for (int i = lane; i < T; i += 32) {
      const int k = sm.own[i];
      const int j = i + base_i - sm.l_pre[k];
      const double x = (double)__fmul_rn(sm.fval[i], sm.l_a[k]);
      const long long q = (long long)floor(x + 0.5);  // lround for x >= 0
      const int prob = q < 1 ? 1 : (int)q;
      c.base[sm.l_off[k] + 8 + 4 * j + 3] = (uint32_t)sm.mv[i] | (((uint32_t)prob & 0x1ffu) << 7);
      sm.dval[i] = __int_as_float(prob);
    }
    g_sync(c);
    // ---- leaf phase 7: denominator = 1 / float(sum of integer priors)
    {
      int qsum = 0;
#pragma unroll 4
      for (int j = 0; j < nmax; ++j)
        if (j < my_cnt) qsum += __float_as_int(sm.dval[my_i0 + j]);
      if (mine) c.base[my_off + 5] = __float_as_uint(__double2float_rn(__drcp_rn((double)(float)qsum)));
    }
    g_sync(c);
    k0 = k1;
  }
  // ---- backup (trainmc.cpp:281-292). Level L slot of leaf k = path[L-1]; the leaf itself
  // (L == plen) takes e-1, its parent -e-1, ... Adds to one slot are applied in leaf order.
  // Four levels per trip so that their slot reads overlap.
  const int maxlen = g_max(c, my_plen);
  const float d_even = __double2float_rn(__dsub_rn((double)my_ev, 1.0));
  const float d_odd = __double2float_rn(__dsub_rn((double)-my_ev, 1.0));
  for (int L0 = 1; L0 <= maxlen; L0 += 4) {
    uint32_t addr[4];
    bool owner[4];
    unsigned grp[4];
    float v[4];
    uint32_t w3[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int L = L0 + u;
      const bool act = lane < np && my_plen >= L;
      uint32_t a = 0xFFFFFF00u + (uint32_t)lane;
      if (act) a = L0 == 1 ? path4[u] : my_pd[2 + L - 1];
      addr[u] = a;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      owner[u] = false, grp[u] = 0, v[u] = 0.0f, w3[u] = 0;
      if (L0 + u <= maxlen) {
        const bool act = lane < np && my_plen >= L0 + u;
        grp[u] = g_match(c, addr[u]);
        owner[u] = act && (__ffs((int)grp[u]) - 1 == lane);
        if (owner[u]) {
          const uint32_t *sp = c.base + addr[u];
          v[u] = __uint_as_float(sp[0]), w3[u] = sp[3];
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (L0 + u <= maxlen) {
        const float d = ((my_plen - (L0 + u)) & 1) ? d_odd : d_even;
        for (int m = 0; m < np; ++m) {
          const float dm = g_shfl(c, d, m);
          if (owner[u] && ((grp[u] >> m) & 1u)) v[u] = __fadd_rn(v[u], dm);
        }
        if (owner[u]) {
          uint32_t *sp = c.base + addr[u];
          sp[0] = __float_as_uint(v[u]), sp[3] = w3[u] & ~kS3Allv;
        }
      }
    }
  }
  for (int m = 0; m < np; ++m) {
    const float de = g_shfl(c, d_even, m);
    const float dd = g_shfl(c, d_odd, m);
    const int pl = g_shfl(c, my_plen, m);
    c.root_eval = __fadd_rn(c.root_eval, (pl & 1) ? dd : de);
  }
  g_sync(c);
  }  // batch of <= 32 leaves
  c.root_allv = 0;
  c.d_evals += np_all;
  c.n_pending = 0;
}

// PUCT value of one slot (chooseNext, trainmc.cpp:540-600); -inf = not selectable. divided =
// the fast path could not decide the rounding and the value came from the two IEEE divisions.
__device__ __forceinline__ float puct_u(const uint4 s, float denominator, float v_sqrt, bool &divided) {
  divided = false;
  const float prob = __fmul_rn((float)s3_prior(s.w), denominator);
  const float pvf = __fmul_rn(prob, v_sqrt);
  float u = pvf;  // no child yet, or a drawn child
  if (s3_has(s.w)) {
    const int cr = s3_result(s.w);
    if ((r_known(cr) && !r_drawn(cr)) || s3_allv(s.w)) {
      u = -INFINITY;
    } else if (!r_drawn(cr)) {
      // reference: u = float(-E/N + (P*v)/(N+1)) with both quotients and the sum rounded in
      // double. Fast path: multiply by approximate reciprocals (20-bit hardware seed + 2 Newton
      // steps, relative error < 2^-50, so each product is within 2^-49 of the true quotient) and
      // accept the result only if every double within 2^-46*(|a|+|b|) rounds to the same float;
      // otherwise do it exactly.
      const int cvi = (int)s.y;
      const double ne = -(double)__uint_as_float(s.x);
      const double pv = (double)pvf;
      // the reference divides by float(N) and float(N) + 1.0, which differ from N and N + 1 above 2^24
      const double dn = (double)(float)cvi, dn1 = __dadd_rn(dn, 1.0);
      const double ra = fast_rcp(dn), rb = fast_rcp(dn1);
      const double a = __dmul_rn(ne, ra);
      const double b = __dmul_rn(pv, rb);
      const double sf = __dadd_rn(a, b);
      const double tol = __dmul_rn(__dadd_rn(fabs(a), fabs(b)), 0x1p-46);
      const float ulo = __double2float_rn(__dsub_rn(sf, tol));
      const float uhi = __double2float_rn(__dadd_rn(sf, tol));
      u = ulo;
      if (!(ulo == uhi)) {
        divided = true;
        const double a = __ddiv_rn(ne, dn);
        const double b = __ddiv_rn(pv, dn1);
        u = __double2float_rn(__dadd_rn(a, b));
      }
    }
  }
  return __fadd_rn(u, 0.0f);  // -0.0 -> +0.0 so the integer key orders like operator>
}
__device__ __forceinline__ float puct_u(const uint4 s, float denominator, float v_sqrt) {
  bool divided;
  return puct_u(s, denominator, v_sqrt, divided);
}

// Cheap screening of the same value: an interval [lo, hi] that provably contains puct_u().
// Slots without a (non-drawn) child are exact (lo == hi == the reference's float product). For
// visited children the float expression -E*rcp(N) + pv*rcp(N+1) is within 2^-22*(|a|+|b|) of the
// real-number value (rcp.approx: 1 ulp; three roundings) and the reference's double-rounded
// float within 2^-24 of it, so a half-width of 2^-20*(|a|+|b|) leaves a 3x margin. The argmax
// is decided from the intervals whenever they separate; otherwise search() redoes the level
// with puct_u().
__device__ __forceinline__ bool puct_bounds(const uint4 s, float denominator, float v_sqrt,
                                            float &lo, float &hi) {
  // straight-line (select-only) code: result codes are classified with bit tables
  const uint32_t w = s.w;
  // classify by the 5 bits {has_child, all_visited, result[3]} = w[20:16] with two bit tables.
  // With a child: not selectable if pending/exhausted (all_visited) or decided and not drawn
  // (results {1, 3, 4, 6}); the value is inexact unless the child is drawn {2, 5}.
  const uint32_t cls = (w >> 16) & 31u;
  constexpr uint32_t kUnsel = 0xFF5A0000u;    // has=1: allv=1 -> all; allv=0 -> results 1,3,4,6
  constexpr uint32_t kInexact = 0x00810000u;  // has=1, allv=0, results 0 and 7 (7 is unused)
  const bool unsel = (kUnsel >> cls) & 1u;
  const bool inexact = (kInexact >> cls) & 1u;
  const float prob = __fmul_rn((float)s3_prior(w), denominator);
  const float pvf = __fadd_rn(__fmul_rn(prob, v_sqrt), 0.0f);
  const float fn = (float)(int)s.y;
  float ra, rb;
  asm("rcp.approx.f32 %0, %1;" : "=f"(ra) : "f"(fn));
  asm("rcp.approx.f32 %0, %1;" : "=f"(rb) : "f"(__fadd_rn(fn, 1.0f)));
  const float a = __fmul_rn(-__uint_as_float(s.x), ra);
  const float b = __fmul_rn(pvf, rb);
  const float u = __fadd_rn(a, b);
  const float d = __fmul_rn(__fadd_rn(fabsf(a), fabsf(b)), 0x1p-20f);
  // centre and half-width by selection, then one subtraction and one addition. Neither bound can
  // be -0.0: b >= +0 makes u = a + b a +0.0 when it is zero, x - x is +0.0, and pvf was normalised.
  const float centre = unsel ? -INFINITY : (inexact ? u : pvf);
  const float half = inexact ? d : 0.0f;
  lo = __fsub_rn(centre, half), hi = __fadd_rn(centre, half);
  return inexact;
}
// order-preserving float <-> signed int (for redux.sync.max.s32); no -0.0 inputs
__device__ __forceinline__ int skey(float f) {
  const int b = __float_as_int(f);
  return b ^ ((b >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float skey_inv(int k) {
  return __int_as_float(k ^ ((k >> 31) & 0x7fffffff));
}

// ---- TrainMC::chooseNext (trainmc.cpp:540-600) at one node, for the whole warp ---------------
// s[j] = slot lane + 32 * j of the record at r (lanes past the last slot hold a word that
// classifies as "not selectable"); slots from kS * 32 on are read from r. Returns the chosen slot
// (the first maximum); no_slot = no slot is selectable; exact = the level went to the exact pass.
template <int kS>
__device__ __forceinline__ int select_slot(const Ctx &c, const TreeParams &P, const uint32_t *r,
                                           const uint4 (&s)[kS], int n, float denominator,
                                           int cur_visits, bool &no_slot, bool &exact) {
  // sqrt(float) binds to double sqrt(double) (SURVEY Q9); small arguments come from a table
  // filled by the host with the same expression
  float v_sqrt;
  if (P.vsqrt != nullptr && (unsigned)cur_visits < (unsigned)kVsqrtCap)
    v_sqrt = __ldg(P.vsqrt + cur_visits);
  else
    v_sqrt = __double2float_rn(__dmul_rn((double)P.c_puct, sqrt((double)(float)cur_visits)));
  int emin = -1;
  bool none = false;
  exact = false;
  if (n <= kS * 32) {
    // screening pass: interval per slot, decide when a single slot (or only exact ones) can
    // hold the maximum
    float lo[kS], hi[kS];
    bool in[kS];
    float lmx = -INFINITY;
#pragma unroll
    for (int j = 0; j < kS; ++j) {
      lo[j] = hi[j] = -INFINITY, in[j] = false;
      if (j == 0 || n > 32 * j) in[j] = puct_bounds(s[j], denominator, v_sqrt, lo[j], hi[j]);  // warp-uniform
      lmx = fmaxf(lmx, lo[j]);
    }
    const float lmax = skey_inv(g_max(c, skey(lmx)));
    if (lmax == -INFINITY) {
      none = true;
    } else {
      // candidates = slots whose interval reaches lmax; per lane: how many, the first one, and
      // whether any of them is inexact -- then three warp collectives whatever kS is
      int cnt_l = 0, first_l = 0x7fffffff;
      bool cin = false;
#pragma unroll
      for (int j = kS - 1; j >= 0; --j) {
        const bool cj = hi[j] >= lmax;
        cin = cin || (cj && in[j]);
        cnt_l += cj ? 1 : 0;
        first_l = cj ? c.lane + 32 * j : first_l;
      }
      const int cnt = g_add(c, cnt_l);
      const bool any_in = g_ballot(c, cin) != 0u;
      if (!any_in || cnt == 1) emin = g_min(c, first_l);  // ties: the lowest slot wins (operator>)
    }
  }
  if (emin < 0 && !none) {
    // exact pass (rare): the reference's expression for every slot
    exact = true;
    float best_u = -INFINITY;
    int best_e = 0x7fffffff;
    for (int e = c.lane, j = 0; e < n; e += 32, ++j) {
      uint4 sx;
      if (j < kS) {
        sx = s[0];
#pragma unroll
        for (int q = 1; q < kS; ++q)
          if (j == q) sx = s[q];
      } else {
        sx = ld4(r + 8 + 4 * e);
      }
      const float u = puct_u(sx, denominator, v_sqrt);
      if (u > best_u) best_u = u, best_e = e;
    }
    const uint32_t key = fkey(best_u);
    const uint32_t kmax = g_max(c, key);
    none = (kmax == kKeyNegInf);
    if (!none) emin = g_min(c, key == kmax ? best_e : 0x7fffffff);
  }
  no_slot = none;  // a copy of the local flag, not emin < 0: search() compiles as it did inline
  return emin;
}

// ---- TrainMC::search (trainmc.cpp:602-696) --------------------------------------------------
// The select loop only walks down existing children; a new edge ends it and the expansion
// (do_move + legal moves + record write, the long scalar part) runs after the loop.
__device__ __forceinline__ void search(Ctx &c, const TreeParams &P, WarpSm &sm) {
  constexpr int kS = 2;  // slot registers per lane: 64 slots screened
  ++c.searches_done;
  c.work += 1;
  int level = 0;
  uint32_t node = c.root_off;
  int cur_result = c.root_result;
  int cur_visits = c.root_visits;
  float cur_eval = c.root_eval;
  uint32_t cur_w3 = 0;
  if (c.lane == 0) sm.node[0] = c.root_off;
  CState leaf_state{0, 0};
  int leaf_n = 0;
  // number of legal moves of the node we stand on: known from the parent's slot below the
  // root, so the slot loads do not wait for the header load (one memory round trip per level)
  int cur_n = (int)(c.base[node + 4] & 0xffu);
  // the path (slot of every node below the root) goes straight into the pending record this
  // search will queue if it ends in an evaluation request
  uint32_t *pd_path = c.pending + c.n_pending * kPendWords + 2;
  bool expand = false;  // the loop ended on an edge without a child: {ex_so, ex_w3, ex_depth}
  uint32_t ex_so = 0, ex_w3 = 0;
  int ex_depth = 0;
  while (!r_terminal(cur_result)) {
    CB_PROF(const long long tl0 = CB_CLOCK();)
    CB_PROF(c.n_lvl += 1;)
    c.work += 1;
    const uint32_t *r = c.base + node;
    const int n = cur_n;
    // lanes past the last slot hold a word that classifies as "not selectable"
    const uint4 zero4 = make_uint4(0, 0, 0, kS3Has | kS3Allv);
    uint4 s[kS];
#pragma unroll
    for (int j = 0; j < kS; ++j)
      s[j] = c.lane + 32 * j < n ? ld4(r + 8 + 4 * (c.lane + 32 * j)) : zero4;
    const uint4 h1 = ld4(r + 4);
    const int depth = (int)((h1.x >> 8) & 0xffu);
    const float denominator = __uint_as_float(h1.y);
    bool none, exact;
    const int emin = select_slot(c, P, r, s, n, denominator, cur_visits, none, exact);
    CB_PROF(c.n_exact += exact ? 1 : 0;)
    // virtual loss on the node we stand on (trainmc.cpp:611,625)
    if (level == 0) {
      c.root_visits += 1;
      c.root_eval = __fadd_rn(c.root_eval, 1.0f);
    } else if (c.lane == 0) {
      uint32_t *sl = c.base + sm.slot[level];
      sl[0] = __float_as_uint(__fadd_rn(cur_eval, 1.0f));
      sl[1] = (uint32_t)(cur_visits + 1);
    }
    if (none) {  // kNone (trainmc.cpp:629-643): flag, roll the whole path back, uncount
      if (level == 0) {
        c.root_allv = 1;
      } else if (c.lane == 0) {
        c.base[sm.slot[level] + 3] = cur_w3 | kS3Allv;
      }
      if (c.lane == 0) {
        for (int l = level; l >= 1; --l) {
          uint32_t *sl = c.base + sm.slot[l];
          sl[0] = __float_as_uint(__fsub_rn(__uint_as_float(sl[0]), 1.0f));
          sl[1] = sl[1] - 1u;
        }
      }
      c.root_visits -= 1;
      c.root_eval = __fsub_rn(c.root_eval, 1.0f);
      --c.searches_done;
      CB_PROF(c.n_none += 1;)
      g_sync(c);
      return;
    }
    const int owner = emin & 31, oj = emin / 32;
    const uint32_t so = node + 8u + 4u * (uint32_t)emin;
    uint4 best_s = s[0];
#pragma unroll
    for (int q = 1; q < kS; ++q)
      if (oj == q) best_s = s[q];
    if (oj >= kS && c.lane == owner) best_s = ld4(r + 8 + 4 * emin);
    const uint32_t ch_w3 = g_shfl(c, best_s.w, owner);
    CB_PROF(c.t_sel += CB_CLOCK() - tl0;)
    if (!s3_has(ch_w3)) {  // kNew (trainmc.cpp:645-660): expand below, after the loop
      if (level + 1 >= kMaxPath) {
        c.error = CB200_ERR_OVERFLOW;
        return;
      }
      expand = true, ex_so = so, ex_w3 = ch_w3, ex_depth = depth;
      break;
    }
    // existing child: descend
    const uint32_t ch_off = g_shfl(c, best_s.z, owner);
    cur_eval = __uint_as_float(g_shfl(c, best_s.x, owner));
    cur_visits = (int)g_shfl(c, best_s.y, owner);
    cur_w3 = ch_w3;
    cur_result = s3_result(ch_w3);
    cur_n = s3_cnl(ch_w3);
    ++level;
    if (c.lane == 0) {
      sm.node[level] = ch_off;
      sm.slot[level] = so;
      pd_path[level - 1] = so;
    }
    node = ch_off;
    g_sync(c);
  }
  if (expand) {
    CB_PROF(const long long te0 = CB_CLOCK(); c.n_exp += 1;)
    const CState ps = rec_state(c.base + node);
    leaf_state = do_move(ps, s3_move(ex_w3));
    const uint32_t coff = c.used;
    int result;
    const int cn = make_record(c, P, leaf_state, ex_depth + 1, result);
    if (cn < 0) return;
    leaf_n = cn;
    if (c.lane == 0) {
      const float e0 = r_terminal(result) ? (result == kResultDraw ? 0.0f : -1.0f) : 1.0f;
      st4(c.base + ex_so, make_uint4(__float_as_uint(e0), 1u, coff,
                                     (ex_w3 & 0xffffu) | ((uint32_t)result << 16) | kS3Allv |
                                         kS3Has | ((uint32_t)cn << 21)));
      if (level > 0 && !s3_gc(cur_w3)) c.base[sm.slot[level] + 3] = cur_w3 | kS3Gc;
      sm.node[level + 1] = coff;
      sm.slot[level + 1] = ex_so;
      pd_path[level] = ex_so;
    }
    ++level;
    node = coff;
    cur_result = result;
    g_sync(c);
    CB_PROF(c.t_exp += CB_CLOCK() - te0;)
  }
  if (r_terminal(cur_result)) {
    // propagateTerminal (trainmc.cpp:497-538) along the explicit path
    int l = level;
    int res_l = cur_result;
    while (l != 0) {
      if (r_lost(res_l)) {
        --l;
        if (l == 0) {
          c.root_result = kDeducedWin;
        } else if (c.lane == 0) {
          uint32_t *w = c.base + sm.slot[l] + 3;
          *w = (*w & ~(7u << 16)) | ((uint32_t)kDeducedWin << 16);
        }
      } else {
        --l;
        const uint32_t *pr = c.base + sm.node[l];
        const int pn = (int)(pr[4] & 0xffu);
        bool ok = true;
        for (int e = c.lane; e < pn; e += 32) {
          const uint32_t w = pr[8 + 4 * e + 3];
          if (!s3_has(w) || !r_known(s3_result(w))) ok = false;
        }
        if (!g_all(c, ok)) break;
        // Q4: the drawn() test is on the parent itself
        const int pres = (l == 0) ? c.root_result : s3_result(c.base[sm.slot[l] + 3]);
        const int nr = r_drawn(pres) ? kDeducedDraw : kDeducedLoss;
        if (l == 0) {
          c.root_result = nr;
        } else if (c.lane == 0) {
          uint32_t *w = c.base + sm.slot[l] + 3;
          *w = (*w & ~(7u << 16)) | ((uint32_t)nr << 16);
        }
      }
      g_sync(c);
      res_l = (l == 0) ? c.root_result : s3_result(c.base[sm.slot[l] + 3]);
    }
    // terminal backup (trainmc.cpp:666-682): leaf value was stored at creation
    float ce = (cur_result == kResultDraw) ? 0.0f : -1.0f;
    for (int lv = level - 1; lv >= 1; --lv) {
      if (c.lane == 0) {
        uint32_t *sl = c.base + sm.slot[lv];
        sl[0] = __float_as_uint(
            __fadd_rn(__uint_as_float(sl[0]), __double2float_rn(__dsub_rn((double)ce, 1.0))));
      }
      ce = -ce;
    }
    c.root_eval = __fadd_rn(c.root_eval, __double2float_rn(__dsub_rn((double)ce, 1.0)));
    g_sync(c);
  } else {
    // request an evaluation (trainmc.cpp:684-691): remember the leaf and the path to it
    uint32_t *pd = c.pending + c.n_pending * kPendWords;
    if (c.lane == 0) {
      pd[0] = node, pd[1] = (uint32_t)level | ((uint32_t)leaf_n << 8);
      c.leaf_state[c.n_pending] = make_ulonglong2(leaf_state.w0, leaf_state.w1);
    }
    c.n_pending += 1;
    g_sync(c);
  }
}

// ---- TrainMC::doIteration (trainmc.cpp:139-178) ---------------------------------------------
__device__ __forceinline__ bool tree_do_iteration(Ctx &c, const TreeParams &P, WarpSm &sm,
                                                  const float *eval, const float *probs,
                                                  long prs = 0, long pcs = 0,
                                                  bool resume = false) {
  if (!c.has_root) {
    fresh_tree(c, P, start_state(), 0);
    c.searches_done = 1;
    c.d_searches += 1;
    request_root(c);
    return false;
  }
  if (c.searches_done == 0 && c.root_visits == 1 && c.root_allv) {
    c.searches_done = 1;
    c.d_searches += 1;
    request_root(c);
    return false;
  }
  CB_PROF(long long t0 = CB_CLOCK();)
  if (c.n_pending > 0 && !resume) receive_eval(c, P, sm, eval, probs, prs, pcs);
  CB_PROF(long long t1 = CB_CLOCK(); c.t_ingest += t1 - t0;)
  const int sd0 = c.searches_done;
  while (c.n_pending < P.spe && c.searches_done < P.max_searches && !r_known(c.root_result) &&
         !c.root_allv && !c.error) {
    if (P.yield_budget > 0 && c.work >= P.yield_budget) {
      c.yielded = 1;  // parked: continue this doIteration in the next launch
      break;
    }
    search(c, P, sm);
  }
  CB_PROF(c.t_search += CB_CLOCK() - t1;)
  c.d_searches += c.searches_done - sd0;
  if (c.yielded) return false;
  return (c.searches_done == P.max_searches || r_known(c.root_result)) && c.n_pending == 0;
}

// TrainMC::chooseHighProbMove (trainmc.cpp:298-308) incl. the int32 max_prob quirk (Q3)
__device__ __forceinline__ int choose_high_prob(Ctx &c, WarpSm &sm) {
  const uint32_t *r = c.base + c.root_off;
  const int n = (int)(r[4] & 0xffu);
  const float denominator = __uint_as_float(r[5]);
  for (int e = c.lane; e < n; e += 32)
    sm.f[e] = __fmul_rn((float)s3_prior(r[8 + 4 * e + 3]), denominator);
  g_sync(c);
  int max_prob = 0, idx = -1;
  for (int i = 0; i < n; ++i) {
    const float pr = sm.f[i];
    if (pr > (float)max_prob) max_prob = (int)pr, idx = i;
  }
  g_sync(c);
  return idx < 0 ? 0 : s3_move(r[8 + 4 * idx + 3]);
}

// "Reset tree" (trainmc.cpp:397-404, 461-468): single node reached by `move` from the root
__device__ __forceinline__ void reset_tree_after(Ctx &c, const TreeParams &P, int move) {
  const CState st = do_move(rec_state(c.base + c.root_off), move);
  const int depth = (int)((c.base[c.root_off + 4] >> 8) & 0xffu) + 1;
  g_sync(c);
  fresh_tree(c, P, st, depth);
  c.searches_done = 0;
}

// ---- TrainMC::chooseMove (trainmc.cpp:110-137, 310-473) -------------------------------------
// Lane l looks at root slots l, l + 32, ... (ascending); per-lane bests are merged with the
// reference's tie-breaks (first slot wins).
__device__ __forceinline__ int choose_move(Ctx &c, const TreeParams &P, WarpSm &sm,
                                           float *prob_sample) {
  const uint32_t *r = c.base + c.root_off;
  const int n = (int)(r[4] & 0xffu);
  const int depth = (int)((r[4] >> 8) & 0xffu);
  const bool root_lost = r_lost(c.root_result);
  if (r_won(c.root_result) || root_lost || r_drawn(c.root_result)) {
    // chooseMoveWon: first lost child. chooseMoveLostDrawn: most visited (first on ties),
    // skipping won children unless the root is lost.
    const bool won = r_won(c.root_result);
    int best_key = -1, best_e = 0x7fffffff;
    for (int e = c.lane; e < n; e += 32) {
      const uint4 sl = ld4(r + 8 + 4 * e);
      if (s3_has(sl.w)) {
        const int cr = s3_result(sl.w);
        int key = -1;
        if (won) {
          if (r_lost(cr)) key = 1;
        } else if ((int)sl.y > 0 && (root_lost || !r_won(cr))) {
          key = (int)sl.y;
        }
        if (key > best_key) best_key = key, best_e = e;
      }
    }
    const int kmax = g_max(c, best_key);
    if (kmax < 0) {  // unreachable in the reference (null dereference there); fail loudly
      c.error = CB200_ERR_STATE;
      return 0;
    }
    const int emin = g_min(c, best_key == kmax ? best_e : 0x7fffffff);
    const int choice = s3_move(r[8 + 4 * emin + 3]);
    if (prob_sample && c.lane == 0) prob_sample[choice] = 1.0f;
    move_down(c, P, emin);
    return choice;
  }
  if (depth < 6 && !P.testing) {  // chooseMoveOpening (trainmc.cpp:375-436)
    int choice = choose_high_prob(c, sm);
    int vis = 0;
    for (int e = c.lane; e < n; e += 32) {
      const uint4 sl = ld4(r + 8 + 4 * e);
      if (s3_has(sl.w) && !r_won(s3_result(sl.w))) vis += (int)sl.y;
    }
    const int visits = g_add(c, vis);
    const float denominator = __double2float_rn(__ddiv_rn(1.0, (double)(float)visits));
    for (int e = c.lane; e < n; e += 32) {
      const uint4 sl = ld4(r + 8 + 4 * e);
      if (s3_has(sl.w) && !r_won(s3_result(sl.w)))
        prob_sample[s3_move(sl.w)] = __fmul_rn((float)(int)sl.y, denominator);
    }
    if (visits == 0) {
      if (c.lane == 0) prob_sample[choice] = 1.0f;
      reset_tree_after(c, P, choice);
      return choice;
    }
    const int target = (int)(rng_one(c) % (uint32_t)visits);
    int carry = 0, found = -1;
    for (int e0 = 0; e0 < n && found < 0; e0 += 32) {
      const int e = e0 + c.lane;
      bool elig = false;
      uint32_t v = 0u;
      if (e < n) {
        const uint4 sl = ld4(r + 8 + 4 * e);
        elig = s3_has(sl.w) && !r_won(s3_result(sl.w));
        if (elig) v = sl.y;
      }
      const uint32_t incl = g_incl_scan(c, v) + (uint32_t)carry;
      const unsigned hit = g_ballot(c, elig && (int)incl > target);
      if (hit) found = e0 + (__ffs((int)hit) - 1);
      carry = (int)g_shfl(c, incl, 31);
    }
    choice = s3_move(r[8 + 4 * found + 3]);
    move_down(c, P, found);
    return choice;
  }
  // chooseMoveNormal (trainmc.cpp:438-473): most visited non-won child, ties by evaluation
  // (draws count 0), first wins; start values (0, 0.0)
  int choice = choose_high_prob(c, sm);
  int bv = 0, be = 0x7fffffff;
  float bf = 0.0f;
  for (int e = c.lane; e < n; e += 32) {
    const uint4 sl = ld4(r + 8 + 4 * e);
    if (s3_has(sl.w) && !r_won(s3_result(sl.w))) {
      const int cr = s3_result(sl.w);
      float ev = __uint_as_float(sl.x);
      if (cr == kResultDraw || cr == kDeducedDraw) ev = 0.0f;
      ev = __fadd_rn(ev, 0.0f);
      const int cv = (int)sl.y;
      if (cv > bv || (cv == bv && ev > bf)) bv = cv, bf = ev, be = e;
    }
  }
  const int vmax = g_max(c, bv);
  const uint32_t fk = (bv == vmax && be != 0x7fffffff) ? fkey(bf) : 0u;
  const uint32_t fmax = g_max(c, fk);
  const int emin = g_min(c, (bv == vmax && be != 0x7fffffff && fk == fmax) ? be : 0x7fffffff);
  if (emin != 0x7fffffff) choice = s3_move(r[8 + 4 * emin + 3]);
  if (prob_sample && c.lane == 0) prob_sample[choice] = 1.0f;
  if (vmax == 0 || emin == 0x7fffffff) {
    reset_tree_after(c, P, choice);
    return choice;
  }
  move_down(c, P, emin);
  return choice;
}

// ---- TrainMC::receiveOpponentMove (trainmc.cpp:180-204) -------------------------------------
__device__ __forceinline__ bool receive_opponent_move(Ctx &c, const TreeParams &P, int move,
                                                      const CState &st, int depth) {
  const uint32_t *r = c.base + c.root_off;
  const int n = (int)(r[4] & 0xffu);
  int found = 0x7fffffff;
  for (int e = c.lane; e < n; e += 32) {
    const uint32_t w = r[8 + 4 * e + 3];
    if (s3_has(w) && s3_move(w) == move) found = e;
  }
  found = g_min(c, found);
  if (found != 0x7fffffff) {
    move_down(c, P, found);
    return false;
  }
  fresh_tree(c, P, st, depth);
  request_root(c);
  c.searches_done = 1;
  c.d_searches += 1;
  return true;
}

// ---- per-move log records (SelfPlayer::writePreMoveLogs / writeMoves / writeMoveChoice,
// selfplayer.cpp:124-204; Node::printMainLine, node.cpp:197-239). The device stores the numbers,
// the host prints them with the reference's stream formatting (engine.cu, format_log_record).
// Record: [0] root depth, [1] to_play, [2] root visits, [3] root evaluation bits, [4] root
// result, [5] main-line entries, [6] visited root children, [7] chosen move, [8..11] position
// after the move, [12] 0 or 1 + game result when the move ended the game, [13] 1 = a Match's
// random player moved (no pre-move section);
// main line at kLogMain: {depth, move, visits, evaluation bits, result, probability bits};
// children at kLogKids: {move, visits, evaluation bits, probability bits, result}.
constexpr int kLogWords = 1024, kLogMain = 16, kLogMainMax = 64, kLogKids = kLogMain + 6 * kLogMainMax;
constexpr int kLogMaxMoves = 130;
static_assert(kLogKids + 5 * CB200_NUM_MOVES <= kLogWords, "log record too small");

__device__ __forceinline__ uint32_t *log_record(const Ctx &c, const TreeParams &P) {
  if (P.log_buf == nullptr) return nullptr;
  const int g = (int)((c.tree_ctl - P.tree) / (2 * kTreeCtlWords));
  if (g >= P.n_logged) return nullptr;
  const int k = P.log_count[g];
  if (k >= kLogMaxMoves) return nullptr;
  return P.log_buf + ((size_t)g * kLogMaxMoves + k) * kLogWords;
}

__device__ __noinline__ void log_pre_move(const uint32_t *base, uint32_t root_off, int to_play,
                                          int root_visits, float root_eval, int root_result,
                                          uint32_t *rec) {
  const uint32_t *r = base + root_off;
  rec[0] = (r[4] >> 8) & 0xffu, rec[1] = (uint32_t)to_play, rec[2] = (uint32_t)root_visits;
  rec[3] = __float_as_uint(root_eval), rec[4] = (uint32_t)root_result;
  {  // visited children of the root, in edge order
    const int n = (int)(r[4] & 0xffu);
    const float denom = __uint_as_float(r[5]);
    int nk = 0;
    for (int e = 0; e < n; ++e) {
      const uint4 s = ld4(r + 8 + 4 * e);
      if (!s3_has(s.w)) continue;
      uint32_t *k = rec + kLogKids + 5 * nk++;
      k[0] = (uint32_t)s3_move(s.w), k[1] = s.y, k[2] = s.x;
      k[3] = __float_as_uint(__fmul_rn((float)s3_prior(s.w), denom)), k[4] = (uint32_t)s3_result(s.w);
    }
    rec[6] = (uint32_t)nk;
  }
  int nm = 0;
  uint32_t node = root_off;
  while (nm < kLogMainMax) {  // Node::printMainLine
    const uint32_t *rn = base + node;
    const int n = (int)(rn[4] & 0xffu);
    const float denom = __uint_as_float(rn[5]);
    int best = -1, max_visits = 0;
    float max_eval = 0.0f, prob = 0.0f;
    uint4 bs = make_uint4(0, 0, 0, 0);
    for (int e = 0; e < n; ++e) {
      const uint4 s = ld4(rn + 8 + 4 * e);
      if (!s3_has(s.w)) continue;
      const int cr = s3_result(s.w), vis = (int)s.y;
      const float ev = __uint_as_float(s.x);
      if (cr == kDeducedLoss || cr == kResultLoss) {
        best = e, max_visits = vis, prob = __fmul_rn((float)s3_prior(s.w), denom), bs = s;
        break;
      }
      if (vis > max_visits || (vis == max_visits && ev > max_eval)) {
        best = e, max_visits = vis, max_eval = ev, bs = s;
        prob = __fmul_rn((float)s3_prior(s.w), denom);
      }
    }
    if (best < 0) break;
    uint32_t *m = rec + kLogMain + 6 * nm++;
    m[0] = ((rn[4] >> 8) & 0xffu) + 1u, m[1] = (uint32_t)s3_move(bs.w), m[2] = (uint32_t)max_visits;
    m[3] = __float_as_uint(max_eval), m[4] = (uint32_t)s3_result(bs.w), m[5] = __float_as_uint(prob);
    node = bs.z;
  }
  rec[5] = (uint32_t)nm;
}

// ---- SelfPlayer::chooseMoveAndContinue (selfplayer.cpp:246-291) -----------------------------
// defer_search (fused mode only): after handing the move to the opponent, do not run the
// opponent's searches inside this call; the next game step finds no pending answers and
// performs exactly the same TrainMC::doIteration then. The order of operations within the game
// is unchanged (so are its results); only the launch in which they happen moves, which keeps
// the mover's lanes from doing two search phases in one launch.
// Returns kTurnWait (an evaluation is pending, or the next search was deferred), kTurnOver (game
// finished) or kTurnIterate (the caller must run TrainMC::doIteration for the side now to move,
// without answers, and come back here if that completes the turn as well).
enum : int { kTurnWait = 0, kTurnOver = 1, kTurnIterate = 2 };
__device__ __forceinline__ int choose_move_and_continue(Ctx &c, const TreeParams &P, WarpSm &sm,
                                                        bool defer_search) {
  {
    if (r_known(c.root_result) && c.mate_turn == 0) c.mate_turn = c.n_samples + 1;
    c.d_sims += c.searches_done;
    c.d_moves += 1;
    if (c.d_moves > 128) {  // no Corintho game has this many plies: refuse to spin
      c.error = CB200_ERR_STATE;
      return kTurnOver;
    }
    uint32_t *log_rec = log_record(c, P);
    if (log_rec != nullptr) {
      if (c.lane == 0)
        log_pre_move(c.base, c.root_off, c.to_play, c.root_visits, c.root_eval, c.root_result, log_rec);
      g_sync(c);
    }
    int choice;
    if (!P.testing) {  // SelfPlayer::chooseMove (selfplayer.cpp:234-244)
      if (c.n_samples >= kMaxSamples) {
        c.error = CB200_ERR_OVERFLOW;
        return kTurnOver;
      }
      float *ps = c.sample_probs + (size_t)c.n_samples * CB200_NUM_MOVES;
      for (int j = c.lane; j < CB200_NUM_MOVES; j += 32) ps[j] = 0.0f;
      if (c.lane == 0) {
        const uint4 h = ld4(c.base + c.root_off);
        c.sample_state[c.n_samples] = make_ulonglong2((uint64_t)h.x | ((uint64_t)h.y << 32),
                                                      (uint64_t)h.z | ((uint64_t)h.w << 32));
      }
      g_sync(c);
      choice = choose_move(c, P, sm, ps);
      c.n_samples += 1;
    } else {
      choice = choose_move(c, P, sm, (float *)nullptr);
    }
    if (c.error) return kTurnOver;
    g_sync(c);
    if (log_rec != nullptr && c.lane == 0) {  // writeMoveChoice + endGame's result line
      const uint4 h = ld4(c.base + c.root_off);
      log_rec[7] = (uint32_t)choice, log_rec[8] = h.x, log_rec[9] = h.y, log_rec[10] = h.z, log_rec[11] = h.w;
      int res = 0;
      if (r_terminal(c.root_result))
        res = 1 + (c.root_result == kResultDraw ? kResultDraw : (c.to_play == 1 ? kResultLoss : kResultWin));
      log_rec[12] = (uint32_t)res, log_rec[13] = 0u;
      __threadfence();
      P.log_count[(c.tree_ctl - P.tree) / (2 * kTreeCtlWords)] += 1;
    }
    if (r_terminal(c.root_result)) {  // endGame (selfplayer.cpp:206-232)
      if (c.root_result == kResultDraw)
        c.result = kResultDraw;
      else if (c.to_play == 1)
        c.result = kResultLoss;
      else
        c.result = kResultWin;
      c.has_root = 0;
      store_tree(c);
      load_tree(c, P, 1 - c.cur_p);
      c.has_root = 0;
      return kTurnOver;
    }
    const CState st = rec_state(c.base + c.root_off);
    const int depth = (int)((c.base[c.root_off + 4] >> 8) & 0xffu);
    c.to_play = 1 - c.to_play;
    store_tree(c);
    load_tree(c, P, c.to_play);
    if (!c.has_root) {
      fresh_tree(c, P, st, depth);
      c.searches_done = 0;
      return kTurnIterate;  // doIteration will just queue the fresh root for evaluation
    }
    const bool need_eval = receive_opponent_move(c, P, choice, st, depth);
    if (c.error) return kTurnOver;
    if (need_eval || defer_search) return kTurnWait;
    return kTurnIterate;
  }
}

// Which games take part in this call (trainer.cpp:39-49, 79-101, 164-236)
__device__ __forceinline__ bool game_selected(const int32_t *ctl, int to_play) {
  if (ctl[CW_DONE]) return false;
  if (to_play != 0 && to_play != 1) return true;
  return ctl[CW_TO_PLAY] == ((to_play + ctl[CW_PARITY]) & 1);
}

// ---- the per-game frame of every driver (run_game, k_match_iterate, analysis_step) ------------
// Game g's Ctx from its control block ctl: the control words, no work done yet, the game's storage.
// Self-play games keep their parity, mate turn and samples; matches and analyses search in testing
// mode from parity 0 and keep no samples.
__device__ __forceinline__ void ctx_open(Ctx &c, const TreeParams &P, int g, const int32_t *ctl,
                                         bool self_play) {
  c.to_play = ctl[CW_TO_PLAY], c.parity = self_play ? ctl[CW_PARITY] : 0, c.result = ctl[CW_RESULT];
  c.mate_turn = self_play ? ctl[CW_MATE_TURN] : 0, c.n_samples = self_play ? ctl[CW_N_SAMPLES] : 0;
  c.n_pending = ctl[CW_N_PENDING], c.error = ctl[CW_ERROR], c.spare = ctl[CW_SPARE];
  c.mt_idx = ctl[CW_MT_IDX];
  c.d_sims = 0, c.d_evals = 0, c.d_moves = 0, c.d_searches = 0;
  CB_PROF(c.t_ingest = c.t_search = c.t_move = c.n_none = c.n_copy = 0;
          c.t_sel = c.t_exp = c.n_lvl = c.n_exp = c.n_exact = 0;)
  c.work = 0, c.yielded = 0;
  c.arenas = P.arenas + (size_t)g * 3 * P.arena_words;
  c.mt = P.mt + (size_t)g * 624;
  c.pending = P.pending + (size_t)g * P.spe * kPendWords;  // P.spe = the largest budget (stride)
  c.tree_ctl = P.tree + (size_t)g * 2 * kTreeCtlWords;
  c.leaf_state = P.leaf_state + (size_t)g * P.spe;
  c.sample_state = self_play ? P.sample_state + (size_t)g * kMaxSamples : nullptr;
  c.sample_probs = self_play ? P.sample_probs + (size_t)g * kMaxSamples * CB200_NUM_MOVES : nullptr;
}
// The control words back (lane 0); CW_DONE and the counters are the caller's.
__device__ __forceinline__ void ctx_close(const Ctx &c, int32_t *ctl, bool self_play) {
  ctl[CW_TO_PLAY] = c.to_play, ctl[CW_RESULT] = c.result;
  if (self_play) ctl[CW_MATE_TURN] = c.mate_turn, ctl[CW_N_SAMPLES] = c.n_samples;
  ctl[CW_N_PENDING] = c.n_pending, ctl[CW_ERROR] = c.error;
  ctl[CW_SPARE] = c.spare, ctl[CW_MT_IDX] = c.mt_idx;
}

// One SelfPlayer::doIteration for game g, executed by one warp. offs[g] = index of
// game g's first answer row in eval/probs (exclusive prefix sum of the request counts the answers
// were produced for). kFused: answers are read at the row the game was handed last time
// (ctl[CW_REQ_BASE]); the new leaf states are appended to `packed` at row0 + (rows handed out
// by one atomicAdd on *req_ctr per game); *live_ctr counts the games that are not finished and
// *err_ctr keeps the most negative error code.
template <bool kFused>
__device__ __forceinline__ void run_game(const TreeParams &P, int g, WarpSm &sm,
                                         const float *__restrict__ eval,
                                         const float *__restrict__ probs, long prs, long pcs,
                                         const int32_t *__restrict__ offs, int to_play,
                                         int iteration, int stagger_div, int32_t *req_ctr,
                                         int32_t *live_ctr, int32_t *err_ctr, int row0,
                                         ulonglong2 *packed, int rows_per_model = 0) {
  int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  if (!game_selected(ctl, to_play)) return;
  const bool training = (to_play != 0 && to_play != 1);
  Ctx c;
  // staggered start (trainer.cpp:184-186), on the global game index
  if (training && stagger_div > 0 && (P.first_game + g) / stagger_div > iteration) {
    if (kFused && c.lane == 0) atomicAdd(live_ctr, 1);
    return;  // not started yet, but alive
  }
  ctx_open(c, P, g, ctl, true);
  bool resume = kFused && ctl[CW_YIELD] != 0;
  const int off = kFused ? ctl[CW_REQ_BASE] : offs[g];
  if (kFused && c.n_pending > 0 && !resume) {
    // This launch will ingest evaluations: request everything whose address is already known
    // (MT19937 state, pending records, this game's rows of the move-major probability matrix)
    // so that the DRAM/L2 round trips overlap the control-block loads and each other.
    for (int i = c.lane * 32; i < 624; i += 1024) prefetch_l1(c.mt + i);
    const int pw = c.n_pending * kPendWords;
    for (int i = c.lane * 32; i < pw; i += 1024) prefetch_l1(c.pending + i);
    if (pcs > 1)
      for (int m = c.lane; m < CB200_NUM_MOVES; m += 32) prefetch_l1(probs + (long)m * pcs + off);
  }
  load_tree(c, P, c.to_play);
  // SelfPlayer::doIteration (selfplayer.cpp:115-122) with chooseMoveAndContinue's loop
  // (selfplayer.cpp:246-291) unrolled here so that doIteration has a single call site
  bool done = false;
  const float *ev_p = eval + off, *pr_p = probs + (long)off * prs;
  for (;;) {
    const bool turn_done = tree_do_iteration(c, P, sm, ev_p, pr_p, prs, pcs, resume);
    resume = false;
    if (c.error || !turn_done) break;
    CB_PROF(const long long tm = CB_CLOCK();)
    const int r = choose_move_and_continue(c, P, sm, kFused);
    CB_PROF(c.t_move += CB_CLOCK() - tm;)
    if (r == kTurnOver) {
      done = true;
      break;
    }
    if (r == kTurnWait) break;
  }
  if (c.error) done = true;
  store_tree(c);
  if (kFused) {
    // two-model runs (rows_per_model > 0): the requests of the side now to move are answered by
    // model (to_play + parity) & 1 (trainer.cpp:166, main.pyx:74-81); each model has its own row
    // region and request counter (req_ctr[0], req_ctr[4])
    if (rows_per_model > 0 && ((c.to_play + c.parity) & 1)) row0 += rows_per_model, req_ctr += 4;
    int base = 0;
    if (c.lane == 0) {
      if (c.n_pending > 0 && !c.yielded) base = atomicAdd(req_ctr, c.n_pending);
      if (!done) atomicAdd(live_ctr, 1);
      if (c.error) atomicMin(err_ctr, c.error);
      ctl[CW_REQ_BASE] = row0 + base;
    }
    base = g_shfl(c, base, 0);
    if (!c.yielded)
      for (int k = c.lane; k < c.n_pending; k += 32) packed[row0 + base + k] = c.leaf_state[k];
    if (c.lane == 0) ctl[CW_YIELD] = c.yielded;
  }
  if (c.lane == 0) {
    ctx_close(c, ctl, true);
    if (done) {
      // a finished game's samples may be picked up by the streaming emit kernel on another
      // stream: everything the game wrote must be visible before the flag is
      __threadfence();
      ctl[CW_DONE] = 1;
    }
    long long *cnt = P.counters + (size_t)g * 4;
    // reductions without a return value: nothing waits for the old counter values
    if (c.d_sims) atomicAdd((unsigned long long *)cnt, (unsigned long long)c.d_sims);
    if (c.d_moves) atomicAdd((unsigned long long *)cnt + 1, (unsigned long long)c.d_moves);
    if (c.d_evals) atomicAdd((unsigned long long *)cnt + 2, (unsigned long long)c.d_evals);
    // searches performed in this launch: the running form of the simulation count (equal to
    // cnt[0] once every game is over), which lets the host attribute simulations to launches
    if (c.d_searches) atomicAdd((unsigned long long *)cnt + 3, (unsigned long long)c.d_searches);
#if CB200_PHASE_PROF
    if (P.phase_prof) {
      atomicMax(P.phase_prof + 0, (unsigned long long)c.t_ingest);
      atomicMax(P.phase_prof + 1, (unsigned long long)c.t_search);
      atomicMax(P.phase_prof + 2, (unsigned long long)c.t_move);
      atomicAdd(P.phase_prof + 3, (unsigned long long)c.t_ingest);
      atomicAdd(P.phase_prof + 4, (unsigned long long)c.t_search);
      atomicAdd(P.phase_prof + 5, (unsigned long long)c.t_move);
      atomicAdd(P.phase_prof + 6, (unsigned long long)c.n_none);
      atomicAdd(P.phase_prof + 7, (unsigned long long)c.n_copy);
      atomicAdd(P.phase_prof + 8, (unsigned long long)c.t_sel);
      atomicAdd(P.phase_prof + 9, (unsigned long long)c.t_exp);
      atomicAdd(P.phase_prof + 10, (unsigned long long)c.n_lvl);
      atomicAdd(P.phase_prof + 11, (unsigned long long)c.n_exp);
      atomicAdd(P.phase_prof + 12, (unsigned long long)c.n_exact);
    }
#endif
  }
}

// Lock-step game step: one warp per game, all games of the trainer (or the live games of one
// stream group, through the group's live list).
template <bool kFused, int kMinBlocks>
__global__ void __launch_bounds__(kTreeWarps * 32, kMinBlocks)
    k_iterate(TreeParams P, const float *__restrict__ eval, const float *__restrict__ probs,
              long prs, long pcs, const int32_t *__restrict__ offs, int to_play, int iteration,
              int stagger_div) {
  __shared__ WarpSm sm_all[kTreeWarps];
  const int grp = threadIdx.x / 32;
  const int idx = blockIdx.x * kTreeWarps + grp;
  int g;
  if (kFused) {
    if (idx >= *P.live_count) return;
    g = __ldg(P.live_list + P.game_begin + idx);  // read-only while the game step runs
  } else {
    g = idx;
    if (g >= P.num_games) return;
  }
  const int par = (iteration + 1) & 1;
  run_game<kFused>(P, g, sm_all[grp], eval, probs, prs, pcs, offs, to_play, iteration,
                   stagger_div, kFused ? P.group_ctr + par : nullptr,
                   kFused ? P.group_ctr + 2 + par : nullptr, kFused ? P.group_ctr + 4 : nullptr,
                   P.group_row0, P.packed);
}

// Live games of one stream group, ascending (one warp per group): list[game_begin + i], i < n.
__global__ void k_group_live_list(TreeParams P, int32_t *__restrict__ list, int32_t *__restrict__ count) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  int n = 0;
  for (int g0 = P.game_begin; g0 < P.game_end; g0 += 32) {
    const int g = g0 + lane;
    const bool live = g < P.game_end && !P.ctl[(size_t)g * kCtlWords + CW_DONE];
    const unsigned m = __ballot_sync(0xffffffffu, live);
    if (live) list[P.game_begin + n + __popc(m & ((1u << lane) - 1u))] = g;
    n += __popc(m);
  }
  if (lane == 0) *count = n;
}

// Exclusive prefix sum of the request counts of the selected games (single CTA).
// summary = {total requests, games not done, error code of any game}
__global__ void __launch_bounds__(1024)
    k_scan_requests(TreeParams P, int to_play, int32_t *__restrict__ offs,
                    int32_t *__restrict__ summary) {
  __shared__ int s_part[1024];
  __shared__ int s_live, s_err;
  const int t = threadIdx.x;
  if (t == 0) s_live = 0, s_err = 0;
  __syncthreads();
  const int per = (P.num_games + 1023) / 1024;
  const int g0 = t * per, g1 = min(P.num_games, g0 + per);
  int sum = 0, live = 0, err = 0;
  for (int g = g0; g < g1; ++g) {
    const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
    if (game_selected(ctl, to_play)) sum += ctl[CW_N_PENDING];
    if (!ctl[CW_DONE]) ++live;
    if (ctl[CW_ERROR]) err = ctl[CW_ERROR];
  }
  s_part[t] = sum;
  if (live) atomicAdd(&s_live, live);
  if (err) atomicMin(&s_err, err);
  __syncthreads();
  // Hillis-Steele inclusive scan over the 1024 partials
  for (int d = 1; d < 1024; d <<= 1) {
    const int v = (t >= d) ? s_part[t - d] : 0;
    __syncthreads();
    s_part[t] += v;
    __syncthreads();
  }
  int run = s_part[t] - sum;
  for (int g = g0; g < g1; ++g) {
    const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
    offs[g] = run;
    if (game_selected(ctl, to_play)) run += ctl[CW_N_PENDING];
  }
  if (t == 1023) summary[0] = s_part[1023];
  if (t == 0) summary[1] = s_live, summary[2] = s_err;
}

// The first np queued leaf states of game g as request rows off, off + 1, ... (one warp): the
// packed cstates for a device-resident network (packed != null) and the 70-float rows
// (rows != null).
__device__ __forceinline__ void pack_game_requests(const TreeParams &P, int g, int np, size_t off, int lane,
                                                   float *__restrict__ rows, ulonglong2 *__restrict__ packed) {
  const ulonglong2 *ls = P.leaf_state + (size_t)g * P.spe;
  if (packed)
    for (int k = lane; k < np; k += 32) packed[off + k] = ls[k];
  if (rows) {
    float *out = rows + off * CB200_STATE_SIZE;
    for (int f = lane; f < np * CB200_STATE_SIZE; f += 32) {
      const int k = f / CB200_STATE_SIZE, j = f - k * CB200_STATE_SIZE;
      const ulonglong2 v = ls[k];
      out[f] = encode_elem(CState{v.x, v.y}, j);
    }
  }
}

// Trainer::writeRequests (trainer.cpp:79-101): expand the queued leaf states of the selected
// games to 70-float rows, game-index-major; also emits the packed cstates for the fused net.
__global__ void __launch_bounds__(256)
    k_pack_requests(TreeParams P, int to_play, const int32_t *__restrict__ offs,
                    float *__restrict__ rows, ulonglong2 *__restrict__ packed) {
  const int g = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (g >= P.num_games) return;
  const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  if (!game_selected(ctl, to_play)) return;
  pack_game_requests(P, g, ctl[CW_N_PENDING], (size_t)offs[g], threadIdx.x & 31, rows, packed);
}

}  // namespace cb200
#endif
