// TEST INFRASTRUCTURE: compiles the product's SWAR rules header (corintho_ai_b200/csrc/rules.cuh)
// for the HOST so its logic can be checked against the oracle on machines without a GPU.
// This is not a CPU fallback: nothing in the product links it.
#include <stdint.h>
#include "../../corintho_ai_b200/csrc/corintho_tables.h"
#include "../../corintho_ai_b200/csrc/rules.cuh"

extern "C" void shim_step_batch(int64_t n, const uint64_t *states, uint64_t seed, uint32_t *maskflags,
                                uint64_t *next, float *enc) {
  using namespace cb200;
  static const uint32_t ones[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
  auto LB = [](int idx) { return idx < 102 ? kCLineBreakers[idx] : ones; };
  for (int64_t i = 0; i < n; ++i) {
    CState s{states[2 * i], states[2 * i + 1]};
    uint32_t m[3];
    bool lines = (i & 1) ? legal_moves_t<true>(s, m, LB) : legal_moves_t<false>(s, m, LB);
    int nl = cb_popc(m[0]) + cb_popc(m[1]) + cb_popc(m[2]);
    int result = terminal_result(nl, lines);
    int chosen = 0x7f;
    CState o = s;
    if (nl > 0) {
      chosen = nth_move(m, (int)(step_rnd(seed, (uint64_t)i) % (uint32_t)nl));
      o = do_move(s, chosen);
    }
    maskflags[4 * i] = m[0], maskflags[4 * i + 1] = m[1], maskflags[4 * i + 2] = m[2];
    maskflags[4 * i + 3] = (uint32_t)result | (lines ? 4u : 0u) | ((uint32_t)nl << 8) | ((uint32_t)chosen << 16);
    next[2 * i] = o.w0, next[2 * i + 1] = o.w1;
    if (enc) for (int j = 0; j < 70; ++j) enc[70 * i + j] = encode_elem(s, j);
  }
}
extern "C" uint32_t shim_step_rnd(uint64_t seed, uint64_t i) { return cb200::step_rnd(seed, i); }

// basic_moves() (the first half of legal_moves_t; the paired K1 kernel runs its paired form,
// basic_moves_pair, on every position):
// its "any line" flag must equal legal_moves_t's, and without a line its mask IS the legal mask.
// Returns the number of positions where that fails.
extern "C" int64_t shim_basic_moves_check(int64_t n, const uint64_t *states) {
  using namespace cb200;
  static const uint32_t ones[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
  auto LB = [](int idx) { return idx < 102 ? kCLineBreakers[idx] : ones; };
  int64_t bad = 0;
  for (int64_t i = 0; i < n; ++i) {
    CState s{states[2 * i], states[2 * i + 1]};
    uint32_t m[3], b[3];
    const bool lines = legal_moves_t<false>(s, m, LB);
    const bool any = basic_moves(s, b);
    if (any != lines) ++bad;
    else if (!any && (b[0] != m[0] || b[1] != m[1] || b[2] != m[2])) ++bad;
    else if (any && ((m[0] & ~b[0]) | (m[1] & ~b[1]) | (m[2] & ~b[2]))) ++bad;  // line rules only remove moves
  }
  return bad;
}

// The paired K1 kernel's forms (basic_moves_pair, nth_move_lut, do_move_lut) against the ones
// they replace, on the host. Positions i and n-1-i are paired (so both halves see every
// position); for every position every legal move goes through do_move_lut and every rank k
// through nth_move_lut. Returns the number of disagreements.
extern "C" int64_t shim_fast_path_check(int64_t n, const uint64_t *states) {
  using namespace cb200;
  static const uint32_t ones[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
  auto LB = [](int idx) { return idx < 102 ? kCLineBreakers[idx] : ones; };
  static uint32_t mv[96 * kMoveLutWords];
  static uint8_t nth[256 * 8];
  build_move_lut(mv), build_nth_lut(nth);
  const uint32_t *ML = mv;
  auto NL = [](uint32_t i) { return (uint32_t)nth[i]; };
  int64_t bad = 0;
  for (int64_t i = 0; i < n; ++i) {
    const CState a{states[2 * i], states[2 * i + 1]};
    const int64_t j = n - 1 - i;
    const CState b{states[2 * j], states[2 * j + 1]};
    uint32_t ra[3], rb[3], pa[3], pb[3];
    const bool la = basic_moves(a, ra), lb = basic_moves(b, rb);
    bool qa, qb;
    basic_moves_pair(a, b, pa, pb, qa, qb);
    if (qa != la || qb != lb) ++bad;
    for (int w = 0; w < 3; ++w)
      if (pa[w] != ra[w] || pb[w] != rb[w]) ++bad;
    uint32_t m[3];
    legal_moves_t<false>(a, m, LB);
    const int nl = cb_popc(m[0]) + cb_popc(m[1]) + cb_popc(m[2]);
    for (int k = 0; k < nl; ++k) {
      const int id = nth_move(m, k);
      if (nth_move_lut(m, k, NL) != id) ++bad;
      const CState x = do_move(a, id), y = do_move_lut(a, id, ML);
      if (x.w0 != y.w0 || x.w1 != y.w1) ++bad;
    }
    // the basic-rule mask is what the fast path draws from when no line exists; its moves are a
    // superset of the legal ones, so run them through both do_move forms as well
    for (int id = 0; id < 96; ++id)
      if ((ra[id >> 5] >> (id & 31)) & 1u) {
        const CState x = do_move(a, id), y = do_move_lut(a, id, ML);
        if (x.w0 != y.w0 || x.w1 != y.w1) ++bad;
      }
  }
  return bad;
}
