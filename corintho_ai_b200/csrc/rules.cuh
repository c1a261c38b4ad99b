// Corintho game rules on a bit-plane packed state -- branch-light SWAR code shared by the
// game-logic kernel (one thread per state) and the tree kernels (warp-uniform expand).
//
// Packed state ("cstate", 16 bytes; include/corintho_b200.h):
//   w0: four 16-bit planes, bit s = row*4+col of plane t at bit 16*t+s,
//       t = 0 base, 1 column, 2 capital, 3 frozen
//       (reference: Game::board_ bit row*16+col*4+t, cpp/include/game.h:124-126)
//   w1: byte i<6 = pieces_[i] (P0{B,C,A},P1{B,C,A}, game.h:127-131), byte 6 = to_play_
//
// Behaviour restated from the reference (never its code):
//   legal moves   cpp/src/game.cpp:28-43 (getLegalMoves), 193-242 (canPlace/canMove),
//                 249-405 (line rules, first-found line per category, capital fix-ups)
//   move codec    cpp/src/move.cpp:11-42
//   do_move       cpp/src/game.cpp:60-96
//   NN encoding   cpp/src/game.cpp:45-58
//   terminal test cpp/src/node.cpp:256-271
#ifndef CORINTHO_B200_RULES_CUH
#define CORINTHO_B200_RULES_CUH

#include <stdint.h>

#if defined(__CUDACC__)
#define CB_HD __host__ __device__ __forceinline__
#else
#define CB_HD inline
#endif

namespace cb200 {

struct CState {
  uint64_t w0, w1;
};

enum : int {
  kResultNone = 0,
  kResultLoss = 1,
  kResultDraw = 2,
  kResultWin = 3,
  kDeducedLoss = 4,
  kDeducedDraw = 5,
  kDeducedWin = 6
};

CB_HD int cb_popc(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __popc(x);
#else
  return __builtin_popcount(x);
#endif
}
CB_HD int cb_ffs(uint32_t x) {  // 1-based index of lowest set bit, 0 if none
#if defined(__CUDA_ARCH__)
  return __ffs((int)x);
#else
  return __builtin_ffs((int)x);
#endif
}

CB_HD CState start_state() {
  CState s;
  s.w0 = 0;
  s.w1 = 0x0000040404040404ull;
  return s;
}

// 3-in-4 row index compression: bits {4r+c, c<3} -> {3r+c}
CB_HD uint32_t compress3(uint32_t v) {
  return (v & 0x7u) | ((v >> 1) & 0x38u) | ((v >> 2) & 0x1C0u) | ((v >> 3) & 0xE00u);
}

// AND the 96-bit line-breaker mask `idx` into (m0, m1, m2). Device tables are padded to four
// 16-byte-aligned words, so one 128-bit load fetches a mask.
template <class LBFn>
CB_HD void lb_and(LBFn LB, int idx, uint32_t &m0, uint32_t &m1, uint32_t &m2) {
  const uint32_t *lb = LB(idx);
#ifdef __CUDA_ARCH__
  const uint4 v = *reinterpret_cast<const uint4 *>(lb);
  m0 &= v.x, m1 &= v.y, m2 &= v.z;
#else
  m0 &= lb[0], m1 &= lb[1], m2 &= lb[2];
#endif
}

// Legal-move mask (96 bits in m[0..2], bit id&31 of word id>>5) and the "lines present" flag.
// LB(idx) must return a pointer to the 3 words of line-breaker mask idx (util.h:85-290 data);
// idx 102 must return an all-ones mask ("no line in this category").
// kBranchless: thread-per-state callers (K1) get select-only code (every category ANDs a table
// entry, 102 when there is no line); warp-uniform callers keep early-outs that skip work.
template <bool kBranchless, class LBFn>
CB_HD bool legal_moves_t(const CState &st, uint32_t m[3], LBFn LB) {
  const uint32_t lo = (uint32_t)st.w0, hi = (uint32_t)(st.w0 >> 32);
  const uint32_t B = lo & 0xFFFFu, C = lo >> 16, A = hi & 0xFFFFu, F = hi >> 16;
  const uint32_t O = B | C | A;
  const uint32_t E = ~O & 0xFFFFu;
  // squares by top piece (game.cpp:158-168) and by bottom piece (170-180)
  const uint32_t T2 = A, T1 = C & ~A, T0 = B & ~(C | A);
  const uint32_t bot1 = C & ~B, bot2 = A & ~(B | C);
  const uint32_t nF = ~F;
  // canMove (game.cpp:222-232): both non-empty, neither frozen, bottom(from)-top(to)==1
  const uint32_t X1 = bot1 & nF, X2 = bot2 & nF, Y0 = T0 & nF, Y1 = T1 & nF;
  const uint32_t mr = ((X1 & (Y0 >> 1)) | (X2 & (Y1 >> 1))) & 0x7777u;
  const uint32_t md = ((X1 & (Y0 >> 4)) | (X2 & (Y1 >> 4))) & 0x0FFFu;
  const uint32_t ml = ((X1 & (Y0 << 1)) | (X2 & (Y1 << 1))) & 0xEEEEu;
  const uint32_t mu = ((X1 & (Y0 << 4)) | (X2 & (Y1 << 4))) & 0xFFF0u;
  const uint32_t R12 = compress3(mr), L12 = compress3(ml >> 1), D12 = md, U12 = mu >> 4;
  // canPlace (game.cpp:193-220)
  const uint32_t tp = (uint32_t)(st.w1 >> 48) & 1u;
  const uint32_t pcs = (uint32_t)(st.w1 >> (24 * tp)) & 0xFFFFFFu;
  const uint32_t pb = (pcs & 0xFFu) ? E : 0u;
  const uint32_t pc = (pcs & 0xFF00u) ? (E | Y0) : 0u;
  const uint32_t pa = (pcs & 0xFF0000u) ? (E | Y1) : 0u;
  uint32_t m0 = R12 | (D12 << 12) | (L12 << 24);
  uint32_t m1 = (L12 >> 8) | (U12 << 4) | (pb << 16);
  uint32_t m2 = pc | (pa << 16);
  bool lines = false;

#include "rules_lines.inc"
  m[0] = m0, m[1] = m1, m[2] = m2;
  return lines;
}
// legal_moves_t for a position whose basic-rule mask is known already (K1 queues it with the
// position): only the line rules are left
template <class LBFn>
CB_HD bool line_rules_on_basic(const CState &st, uint32_t m[3], LBFn LB) {
  const uint32_t lo = (uint32_t)st.w0, hi = (uint32_t)(st.w0 >> 32);
  const uint32_t B = lo & 0xFFFFu, C = lo >> 16, A = hi & 0xFFFFu;
  const uint32_t T2 = A, T1 = C & ~A, T0 = B & ~(C | A);
  constexpr bool kBranchless = false;
  uint32_t m0 = m[0], m1 = m[1], m2 = m[2];
  bool lines = false;
#include "rules_lines.inc"
  m[0] = m0, m[1] = m1, m[2] = m2;
  return lines;
}
// First half of legal_moves_t for callers that treat positions with a line separately (K1): the
// basic-rule mask (canPlace / canMove only) and whether ANY line exists on the board -- the
// union of the four `has` conditions above. Without a line the basic mask IS the legal mask.
CB_HD bool basic_moves(const CState &st, uint32_t m[3]) {
  const uint32_t lo = (uint32_t)st.w0, hi = (uint32_t)(st.w0 >> 32);
  const uint32_t B = lo & 0xFFFFu, C = lo >> 16, A = hi & 0xFFFFu, F = hi >> 16;
  const uint32_t O = B | C | A;
  const uint32_t E = ~O & 0xFFFFu;
  const uint32_t T2 = A, T1 = C & ~A, T0 = B & ~(C | A);
  const uint32_t bot1 = C & ~B, bot2 = A & ~(B | C);
  const uint32_t nF = ~F;
  const uint32_t X1 = bot1 & nF, X2 = bot2 & nF, Y0 = T0 & nF, Y1 = T1 & nF;
  const uint32_t mr = ((X1 & (Y0 >> 1)) | (X2 & (Y1 >> 1))) & 0x7777u;
  const uint32_t md = ((X1 & (Y0 >> 4)) | (X2 & (Y1 >> 4))) & 0x0FFFu;
  const uint32_t ml = ((X1 & (Y0 << 1)) | (X2 & (Y1 << 1))) & 0xEEEEu;
  const uint32_t mu = ((X1 & (Y0 << 4)) | (X2 & (Y1 << 4))) & 0xFFF0u;
  const uint32_t R12 = compress3(mr), L12 = compress3(ml >> 1), D12 = md, U12 = mu >> 4;
  const uint32_t tp = (uint32_t)(st.w1 >> 48) & 1u;
  const uint32_t pcs = (uint32_t)(st.w1 >> (24 * tp)) & 0xFFFFFFu;
  const uint32_t pb = (pcs & 0xFFu) ? E : 0u;
  const uint32_t pc = (pcs & 0xFF00u) ? (E | Y0) : 0u;
  const uint32_t pa = (pcs & 0xFF0000u) ? (E | Y1) : 0u;
  m[0] = R12 | (D12 << 12) | (L12 << 24);
  m[1] = (L12 >> 8) | (U12 << 4) | (pb << 16);
  m[2] = pc | (pa << 16);
  // three equal tops in a row (step 1, starts in columns 0-1), in a column (step 4, rows 0-1), on
  // a diagonal (step 5 from squares 0, 1, 4, 5; step 3 from squares 2, 3, 6, 7): the three planes
  // are disjoint, so each step needs one AND chain per plane
  uint32_t row = 0, col = 0, d5 = 0, d3 = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int p = 0; p < 3; ++p) {
    const uint32_t T = p == 0 ? T0 : (p == 1 ? T1 : T2);
    row |= T & (T >> 1) & (T >> 2);
    col |= T & (T >> 4) & (T >> 8);
    d5 |= T & (T >> 5) & (T >> 10);
    d3 |= T & (T >> 3) & (T >> 6);
  }
  return ((row & 0x3333u) | (col & 0x00FFu) | (d5 & 0x33u) | (d3 & 0xCCu)) != 0u;
}

template <class LBFn>
CB_HD bool legal_moves(const CState &st, uint32_t m[3], LBFn LB) {
  return legal_moves_t<false>(st, m, LB);
}

// game.cpp:60-96 (no legality check, like the reference); select-only code
CB_HD CState do_move(const CState &st, int move) {
  CState o;
  uint64_t w0 = st.w0 & 0x0000FFFFFFFFFFFFull;  // clear every frozen bit
  uint64_t w1 = st.w1;
  const uint32_t tp = (uint32_t)(w1 >> 48) & 1u;
  const bool is_place = move >= 48;
  // place: 48 + piece*16 + square
  const int piece = (move - 48) >> 4;
  // move: dir = id/12 (0 right, 1 down, 2 left, 3 up), r = id%12 (move.cpp:11-42)
  // (small unsigned multiply-shift divisions: exact for ids 0..47 / r 0..11)
  const uint32_t um = (uint32_t)move & 63u;
  const int dir = (int)((um * 43u) >> 9), r = (int)um - dir * 12;
  const int rq = (int)(((uint32_t)r * 11u) >> 5);  // r / 3
  const int r3 = rq * 4 + (r - rq * 3);            // (row, col<3) of a horizontal move
  const int from = dir == 0 ? r3 : (dir == 1 ? r : (dir == 2 ? r3 + 1 : r + 4));
  const int to_m = dir == 0 ? r3 + 1 : (dir == 1 ? r + 4 : (dir == 2 ? r3 : r));
  const int to = is_place ? (move & 15) : to_m;
  const int fsh = is_place ? 0 : from;
  const uint64_t planes = is_place ? 0ull : 0x0000000100010001ull;
  const uint64_t stack = (w0 >> fsh) & planes;
  w0 &= ~(planes << fsh);
  w0 |= stack << to;
  w0 |= is_place ? (1ull << (16 * (piece & 3) + to)) : 0ull;
  w0 |= 1ull << (48 + to);
  w1 -= is_place ? (1ull << (8 * (tp * 3 + (uint32_t)(piece & 3)))) : 0ull;
  w1 ^= 1ull << 48;
  o.w0 = w0, o.w1 = w1;
  return o;
}

// One element of the 70-float NN input (game.cpp:45-58)
CB_HD float encode_elem(const CState &st, int j) {
  if (j < 64) return (float)((st.w0 >> (16 * (j & 3) + (j >> 2))) & 1ull);
  const uint32_t tp = (uint32_t)(st.w1 >> 48) & 1u;
  int i = (int)tp * 3 + (j - 64);
  if (i >= 6) i -= 6;
  return (float)((st.w1 >> (8 * i)) & 0xFFull) * 0.25f;
}

// node.cpp:256-271: no legal move -> the mover lost if a line exists, else draw
CB_HD int terminal_result(int n_legal, bool lines) {
  return n_legal == 0 ? (lines ? kResultLoss : kResultDraw) : kResultNone;
}

// id of the k-th (0-based) set bit of the 96-bit mask (popcount binary search, no loops)
CB_HD int nth_move(const uint32_t m[3], int k) {
  const int c0 = cb_popc(m[0]), c1 = cb_popc(m[1]);
  const bool in0 = k < c0, in1 = k < c0 + c1;
  uint32_t w = in0 ? m[0] : (in1 ? m[1] : m[2]);
  int base = in0 ? 0 : (in1 ? 32 : 64);
  k -= in0 ? 0 : (in1 ? c0 : c0 + c1);
#pragma unroll
  for (int sh = 16; sh >= 1; sh >>= 1) {
    const int c = cb_popc(w & ((1u << sh) - 1u));
    const bool up = k >= c;
    k -= up ? c : 0;
    w = up ? (w >> sh) : w;
    base += up ? sh : 0;
  }
  return base;
}

// ---- K1 fast-path forms (game_step.cuh, k_game_step_pairw). Same results as basic_moves /
// nth_move / do_move above (tests/host_shim checks them against each other on the host and the
// GPU tests against the oracle); written for the integer-ALU pipe, which bounds K1:
//   * two positions per thread share every plane operation (16-bit planes of position a in the
//     low half of a register, of position b in the high half);
//   * the move decode of do_move and the last three levels of nth_move are table look-ups
//     (shared memory on the device: the load/store pipe has room, the ALU pipe has none).

// shift by (n & 31) / (n & 63): what SHF.*.W does; lets a table word be used as a shift count
// without extracting the field first
CB_HD uint32_t shr_w(uint32_t x, uint32_t n) {
#if defined(__CUDA_ARCH__)
  return __funnelshift_r(x, 0u, n);
#else
  return x >> (n & 31u);
#endif
}
// low word of the 64-bit value hi:lo shifted right by (n & 31)
CB_HD uint32_t shr_w64(uint32_t lo, uint32_t hi, uint32_t n) {
#if defined(__CUDA_ARCH__)
  return __funnelshift_r(lo, hi, n);
#else
  return (uint32_t)((((uint64_t)hi << 32) | lo) >> (n & 31u));
#endif
}
CB_HD uint32_t shl_w(uint32_t x, uint32_t n) {
#if defined(__CUDA_ARCH__)
  return __funnelshift_l(0u, x, n);
#else
  return x << (n & 31u);
#endif
}

// Move table (move.cpp:11-42 decode and every constant of do_move, done once on the host): four
// words per move id, then two more per move id behind them (two arrays, so that the 16-byte and
// the 8-byte load of a warp spread over the shared-memory banks):
//   [4 id + 0] from | to << 8   stack moves: the squares; placements: from = to (moving a stack
//                               onto itself changes nothing)
//   [4 id + 1] piece-count decrement of the side to move, as seen by player 0: 1 << 8 * piece for
//              a placement, 0 for a stack move
//   [4 id + 2], [4 id + 3] AND mask of w0 (low, high word): clears the frozen plane and, for a
//              stack move, the three piece bits of `from`
//   [384 + 2 id], [385 + 2 id] OR mask of w0: the frozen bit of `to` and, for a placement, the
//              piece's plane bit
constexpr int kMoveLutWords = 6;  // per move id
constexpr int kMoveLutOr = 96 * 4;  // first word of the OR masks
inline void build_move_lut(uint32_t out[96 * kMoveLutWords]) {
  for (int id = 0; id < 96; ++id) {
    uint32_t from, to, dec;
    uint64_t andm = 0x0000FFFFFFFFFFFFull, orm;
    if (id < 48) {
      const int dir = id / 12, r = id % 12, r3 = (r / 3) * 4 + r % 3;
      from = (uint32_t)(dir == 0 ? r3 : (dir == 1 ? r : (dir == 2 ? r3 + 1 : r + 4)));
      to = (uint32_t)(dir == 0 ? r3 + 1 : (dir == 1 ? r + 4 : (dir == 2 ? r3 : r)));
      dec = 0;
      andm &= ~(0x0000000100010001ull << from);
      orm = 1ull << (48 + to);
    } else {
      to = (uint32_t)(id & 15), from = to, dec = 1u << (8 * ((id - 48) >> 4));
      orm = (1ull << (48 + to)) | (1ull << (id - 48));  // id - 48 = 16 * piece + to
    }
    uint32_t *e = out + 4 * id, *f = out + kMoveLutOr + 2 * id;
    e[0] = from | (to << 8), e[1] = dec, e[2] = (uint32_t)andm, e[3] = (uint32_t)(andm >> 32);
    f[0] = (uint32_t)orm, f[1] = (uint32_t)(orm >> 32);
  }
}
// Byte table of nth_move_lut: entry v * 8 + k = index of the k-th (0-based) set bit of byte v
inline void build_nth_lut(uint8_t out[256 * 8]) {
  for (int v = 0; v < 256; ++v) {
    int k = 0;
    for (int b = 0; b < 8; ++b)
      if ((v >> b) & 1) out[v * 8 + k++] = (uint8_t)b;
    for (; k < 8; ++k) out[v * 8 + k] = 0;
  }
}

// do_move by table: `lut` is the table of build_move_lut (16-byte aligned). Legal moves only (a
// placement's piece count is positive, so the decrement never borrows).
CB_HD CState do_move_lut(const CState &st, int move, const uint32_t *lut) {
  const uint32_t *e = lut + 4 * move, *f = lut + kMoveLutOr + 2 * move;
#if defined(__CUDA_ARCH__)
  const uint4 q = *reinterpret_cast<const uint4 *>(e);
  const uint2 r = *reinterpret_cast<const uint2 *>(f);
  const uint32_t ex = q.x, ey = q.y, and_lo = q.z, and_hi = q.w, or_lo = r.x, or_hi = r.y;
#else
  const uint32_t ex = e[0], ey = e[1], and_lo = e[2], and_hi = e[3], or_lo = f[0], or_hi = f[1];
#endif
  const uint32_t lo = (uint32_t)st.w0, hi = (uint32_t)(st.w0 >> 32);
  const uint32_t tsh = ex >> 8;  // `to`; the shifts below use the low five bits of their count
  // the stack of `from` (base and column bits s, 16 + s of lo; capital bit s of hi) lands on `to`
  const uint32_t lo2 = (lo & and_lo) | or_lo | shl_w(shr_w(lo, ex) & 0x00010001u, tsh);
  const uint32_t hi2 = (hi & and_hi) | or_hi | shl_w(shr_w(hi, ex) & 1u, tsh);
  CState o;
  o.w0 = (uint64_t)lo2 | ((uint64_t)hi2 << 32);
  // the mover's counts sit 24 bits up for player 1; one signed multiply-add, then flip to_play
  const uint32_t tp = (uint32_t)(st.w1 >> 48) & 1u;
  const int32_t scale = tp ? -(1 << 24) : -1;
  o.w1 = (uint64_t)((int64_t)st.w1 + (int64_t)(int32_t)ey * (int64_t)scale) ^ (1ull << 48);
  return o;
}

// nth_move with the levels below a byte from the table NL(v * 8 + k)
template <class NLFn>
CB_HD int nth_move_lut(const uint32_t m[3], int k, NLFn NL) {
  const int c0 = cb_popc(m[0]), c1 = cb_popc(m[1]);
  const bool in0 = k < c0, in1 = k < c0 + c1;
  uint32_t w = in0 ? m[0] : (in1 ? m[1] : m[2]);
  int base = in0 ? 0 : (in1 ? 32 : 64);
  k -= in0 ? 0 : (in1 ? c0 : c0 + c1);
  {
    const int c = cb_popc(w & 0xFFFFu);
    const bool up = k >= c;
    k -= up ? c : 0, w = up ? (w >> 16) : w, base += up ? 16 : 0;
  }
  {
    const int c = cb_popc(w & 0xFFu);
    const bool up = k >= c;
    k -= up ? c : 0, w = up ? (w >> 8) : w, base += up ? 8 : 0;
  }
  return base + (int)NL((w & 0xFFu) * 8u + (uint32_t)(k & 7));
}

// basic_moves for two positions at once. Every shifted plane is masked so that no bit crosses
// from one half into the other: right shifts by 1 / 4 are followed by 0x7777 / 0x0FFF, left
// shifts by 0xEEEE / 0xFFF0, and the line tests keep only start squares whose three squares lie
// inside one half (the masks of basic_moves, doubled).
CB_HD void basic_moves_pair(const CState &a, const CState &b, uint32_t ma[3], uint32_t mb[3], bool &line_a,
                            bool &line_b) {
  const uint32_t alo = (uint32_t)a.w0, ahi = (uint32_t)(a.w0 >> 32);
  const uint32_t blo = (uint32_t)b.w0, bhi = (uint32_t)(b.w0 >> 32);
#if defined(__CUDA_ARCH__)
  const uint32_t B = __byte_perm(alo, blo, 0x5410), C = __byte_perm(alo, blo, 0x7632);
  const uint32_t A = __byte_perm(ahi, bhi, 0x5410), F = __byte_perm(ahi, bhi, 0x7632);
#else
  const uint32_t B = (alo & 0xFFFFu) | (blo << 16), C = (alo >> 16) | (blo & 0xFFFF0000u);
  const uint32_t A = (ahi & 0xFFFFu) | (bhi << 16), F = (ahi >> 16) | (bhi & 0xFFFF0000u);
#endif
  const uint32_t E = ~(B | C | A);
  const uint32_t T2 = A, T1 = C & ~A, T0 = B & ~(C | A);
  const uint32_t nF = ~F;
  const uint32_t X1 = C & ~B & nF, X2 = A & ~(B | C) & nF, Y0 = T0 & nF, Y1 = T1 & nF;
  const uint32_t mr = ((X1 & (Y0 >> 1)) | (X2 & (Y1 >> 1))) & 0x77777777u;
  const uint32_t md = ((X1 & (Y0 >> 4)) | (X2 & (Y1 >> 4))) & 0x0FFF0FFFu;
  const uint32_t ml = ((X1 & (Y0 << 1)) | (X2 & (Y1 << 1))) & 0xEEEEEEEEu;
  const uint32_t mu = ((X1 & (Y0 << 4)) | (X2 & (Y1 << 4))) & 0xFFF0FFF0u;
  // compress3 with LEFT shifts only (they run on the FMA pipe as multiplications, right shifts
  // on the ALU pipe): row r moves up by 3 - r, so R3 = compress3(mr) << 3 and, because ml holds
  // columns 1-3, L4 = compress3(ml >> 1) << 4. The masks drop whatever a shift carries from the
  // low half into the high half.
  const uint32_t R3 = ((mr << 3) & 0x00380038u) | ((mr << 2) & 0x01C001C0u) | ((mr << 1) & 0x0E000E00u) |
                      (mr & 0x70007000u);
  const uint32_t L4 = ((ml << 3) & 0x00700070u) | ((ml << 2) & 0x03800380u) | ((ml << 1) & 0x1C001C00u) |
                      (ml & 0xE000E000u);
  const uint32_t EY0 = E | Y0, EY1 = E | Y1;
  {
    const uint32_t alo1 = (uint32_t)a.w1, ahi1 = (uint32_t)(a.w1 >> 32);
    const uint32_t pcs = shr_w64(alo1, ahi1, ((ahi1 >> 16) & 1u) * 24u);
    const uint32_t pb = (pcs & 0xFFu) ? (E << 16) : 0u;
    const uint32_t pc = (pcs & 0xFF00u) ? (EY0 & 0xFFFFu) : 0u;
    const uint32_t pa = (pcs & 0xFF0000u) ? (EY1 << 16) : 0u;
    ma[0] = ((R3 >> 3) & 0xFFFu) | ((md << 12) & 0x00FFF000u) | (L4 << 20);
    ma[1] = ((L4 >> 12) & 0xFu) | (mu & 0xFFF0u) | pb;
    ma[2] = pc | pa;
  }
  {
    const uint32_t blo1 = (uint32_t)b.w1, bhi1 = (uint32_t)(b.w1 >> 32);
    const uint32_t pcs = shr_w64(blo1, bhi1, ((bhi1 >> 16) & 1u) * 24u);
    const uint32_t pb = (pcs & 0xFFu) ? (E & 0xFFFF0000u) : 0u;
    const uint32_t pc = (pcs & 0xFF00u) ? (EY0 >> 16) : 0u;
    const uint32_t pa = (pcs & 0xFF0000u) ? (EY1 & 0xFFFF0000u) : 0u;
    mb[0] = (R3 >> 19) | ((md >> 4) & 0x00FFF000u) | ((L4 << 4) & 0xFF000000u);
    mb[1] = (L4 >> 28) | ((mu >> 16) & 0xFFF0u) | pb;
    mb[2] = pc | pa;
  }
  // Lines, again with left shifts: P_k marks the squares whose top equals the top k squares
  // before them (the three top planes are disjoint), P_k & (P_k << k) the END square of three
  // equal tops with step k. Valid end squares: step 1 columns 2-3, step 4 rows 2-3, step 5
  // squares 10, 11, 14, 15, step 3 squares 8, 9, 12, 13 -- none of them can be reached by a bit
  // shifted in from the low half.
  const uint32_t P1 = (T0 & (T0 << 1)) | (T1 & (T1 << 1)) | (T2 & (T2 << 1));
  const uint32_t P4 = (T0 & (T0 << 4)) | (T1 & (T1 << 4)) | (T2 & (T2 << 4));
  const uint32_t P5 = (T0 & (T0 << 5)) | (T1 & (T1 << 5)) | (T2 & (T2 << 5));
  const uint32_t P3 = (T0 & (T0 << 3)) | (T1 & (T1 << 3)) | (T2 & (T2 << 3));
  const uint32_t any = (P1 & (P1 << 1) & 0xCCCCCCCCu) | (P4 & (P4 << 4) & 0xFF00FF00u) |
                       (P5 & (P5 << 5) & 0xCC00CC00u) | (P3 & (P3 << 3) & 0x33003300u);
  line_a = (any & 0xFFFFu) != 0u;
  line_b = (any >> 16) != 0u;
}

// deterministic per-state random word of the game-logic workload (splitmix64 finaliser)
CB_HD uint32_t step_rnd_mix(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return (uint32_t)((z ^ (z >> 31)) >> 32);
}
CB_HD uint32_t step_rnd(uint64_t seed, uint64_t i) { return step_rnd_mix(seed + (i + 1) * 0x9E3779B97F4A7C15ull); }

}  // namespace cb200
#endif
