// TEST INFRASTRUCTURE ONLY -- CPU oracle for the Corintho self-play path (see corintho_oracle.h).
//
// A sequential restatement of the reference algorithm on flat arenas (no pointers): every tree
// is a bump-allocated array of 32-bit words holding node records
//     header[8]  : w0..w3 = packed game state, w4 = n_legal | depth<<8, w5 = denominator bits
//     slot[n][4] : one per legal move, ascending move id (the reference's edges_ array,
//                  node.cpp:273-282) and, once the move has been tried, the statistics of the
//                  child reached through it (the reference keeps those in the child Node,
//                  node.h:150-186):
//                  s0 = child evaluation_ (f32 bits), s1 = child visits_,
//                  s2 = child record offset, s3 = move | prior<<7 | result<<16 | all_visited<<19 |
//                       has_child<<20 | child_n_legal<<21
// The root record sits at offset 0; the root's own statistics live in the Tree struct.
// Re-rooting (TrainMC::moveDown, trainmc.cpp:475-495) copies the kept subtree breadth-first
// into the game's spare arena. Float expression types follow the reference literally
// (SURVEY.md Q9): this file is compiled with -ffp-contract=off.

#include "corintho_oracle.h"

#include <math.h>
#include <omp.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <map>
#include <vector>

#include "oracle_tables.inc"

namespace {

constexpr int kNumMoves = 96;
constexpr int kStateSize = 70;
constexpr int kMaxPath = 64;
constexpr int kMaxSamples = 64;

enum : int {
  kResultNone = 0,
  kResultLoss = 1,
  kResultDraw = 2,
  kResultWin = 3,
  kDeducedLoss = 4,
  kDeducedDraw = 5,
  kDeducedWin = 6
};

inline float bits_f(uint32_t b) {
  float f;
  memcpy(&f, &b, 4);
  return f;
}
inline uint32_t f_bits(float f) {
  uint32_t b;
  memcpy(&b, &f, 4);
  return b;
}

// ------------------------------------------------------------------------------------------
// Move codec (move.cpp:11-42): ids 0-11 right, 12-23 down, 24-35 left, 36-47 up, 48-95 place.
struct MoveInfo {
  int is_place, piece, r0, c0, r1, c1;
};
MoveInfo decode_move(int id) {
  MoveInfo m{0, -1, -1, -1, -1, -1};
  if (id >= 48) {
    m.is_place = 1;
    m.piece = (id - 48) / 16;
    m.r1 = (id % 16) / 4;
    m.c1 = id % 4;
  } else if (id < 12) {
    m.r0 = id / 3, m.c0 = id % 3, m.r1 = m.r0, m.c1 = m.c0 + 1;
  } else if (id < 24) {
    m.r0 = (id - 12) / 4, m.c0 = id % 4, m.r1 = m.r0 + 1, m.c1 = m.c0;
  } else if (id < 36) {
    m.r0 = (id - 24) / 3, m.c0 = id % 3 + 1, m.r1 = m.r0, m.c1 = m.c0 - 1;
  } else {
    m.r0 = (id - 36) / 4 + 1, m.c0 = id % 4, m.r1 = m.r0 - 1, m.c1 = m.c0;
  }
  return m;
}
// move.cpp:80-108
int encode_place(int row, int col, int piece) { return 48 + piece * 16 + row * 4 + col; }
int encode_move(int r0, int c0, int r1, int c1) {
  if (c0 < c1) return r0 * 3 + c0;
  if (r0 < r1) return 12 + r0 * 4 + c0;
  if (c0 > c1) return 24 + r0 * 3 + (c0 - 1);
  return 36 + (r0 - 1) * 4 + c0;
}

// ------------------------------------------------------------------------------------------
// Game rules on the packed state.
struct State {
  uint64_t w0, w1;
};
inline int sq(const State &s, int row, int col) { return (s.w0 >> (row * 16 + col * 4)) & 0xF; }
inline int pieces(const State &s, int i) { return (s.w1 >> (8 * i)) & 0xff; }
inline int to_play(const State &s) { return (s.w1 >> 48) & 0xff; }
// game.cpp:158-180
inline int top_of(int b) { return (b & 4) ? 2 : (b & 2) ? 1 : (b & 1) ? 0 : -1; }
inline int bottom_of(int b) { return (b & 1) ? 0 : (b & 2) ? 1 : (b & 4) ? 2 : 3; }

struct Mask {
  uint32_t w[3];
  void and_line(int idx) {
    for (int k = 0; k < 3; ++k) w[k] &= kOLineBreakers[idx][k];
  }
  void clear(int id) { w[id >> 5] &= ~(1u << (id & 31)); }
  bool get(int id) const { return (w[id >> 5] >> (id & 31)) & 1; }
  int count() const {
    return __builtin_popcount(w[0]) + __builtin_popcount(w[1]) + __builtin_popcount(w[2]);
  }
};

// game.cpp:249-315. Space{a,b,flip}: flip swaps the coordinates (util.h:18-35).
bool apply_rowcol(const State &s, Mask &m, bool is_col) {
  auto at = [&](int a, int b) { return is_col ? sq(s, b, a) : sq(s, a, b); };
  for (int i = 0; i < 4; ++i) {
    int t0 = top_of(at(i, 0)), t1 = top_of(at(i, 1)), t2 = top_of(at(i, 2)), t3 = top_of(at(i, 3));
    if (t1 == -1 || t2 == -1) continue;
    if (t0 == t1 && t1 == t2 && t2 == t3) {
      m.and_line((is_col ? 5 : 2) * 12 + i * 3 + t0);
      return true;
    }
    for (int ext : {3, 0}) {
      if (t1 == t2 && ((ext == 3 && t0 == t1) || (ext == 0 && t2 == t3))) {
        int cat = is_col ? (ext == 0 ? 4 : 3) : (ext == 0 ? 1 : 0);
        m.and_line(cat * 12 + i * 3 + t1);
        if (t1 == 2) {
          // capital fix-ups along the perpendicular line through `ext` (game.cpp:280-309)
          auto cap = [&](int k) { return (at(k, ext) & 4) != 0; };
          auto mv = [&](int ka, int kb) {
            return is_col ? encode_move(ext, ka, ext, kb) : encode_move(ka, ext, kb, ext);
          };
          if (!cap(0)) m.clear(mv(0, 1));
          if (!cap(1)) m.clear(mv(1, 0)), m.clear(mv(1, 2));
          if (!cap(2)) m.clear(mv(2, 1)), m.clear(mv(2, 3));
          if (!cap(3)) m.clear(mv(3, 2));
        }
        return true;
      }
    }
  }
  return false;
}
// game.cpp:317-360
bool apply_long_diag(const State &s, Mask &m) {
  for (int flip = 0; flip < 2; ++flip) {
    int t0 = top_of(sq(s, 0, flip ? 3 : 0)), t1 = top_of(sq(s, 1, flip ? 2 : 1));
    int t2 = top_of(sq(s, 2, flip ? 1 : 2)), t3 = top_of(sq(s, 3, flip ? 0 : 3));
    if (t1 == -1 || t2 == -1) continue;
    if (t0 == t1 && t1 == t2 && t2 == t3) {
      m.and_line(72 + (flip ? 5 : 2) * 3 + t1);
      return true;
    }
    if (t0 == t1 && t1 == t2) {
      m.and_line(72 + (flip ? 3 : 0) * 3 + t1);
      return true;
    }
    if (t1 == t2 && t2 == t3) {
      m.and_line(72 + (flip ? 4 : 1) * 3 + t1);
      return true;
    }
  }
  return false;
}
// game.cpp:362-391
bool apply_short_diag(const State &s, Mask &m) {
  static const int sqs[4][3][2] = {{{1, 1}, {0, 2}, {2, 0}},
                                   {{1, 2}, {0, 1}, {2, 3}},
                                   {{2, 2}, {1, 3}, {3, 1}},
                                   {{2, 1}, {1, 0}, {3, 2}}};
  for (int d = 0; d < 4; ++d) {
    int t = top_of(sq(s, sqs[d][0][0], sqs[d][0][1]));
    if (t != -1 && t == top_of(sq(s, sqs[d][1][0], sqs[d][1][1])) &&
        t == top_of(sq(s, sqs[d][2][0], sqs[d][2][1]))) {
      m.and_line(72 + (6 + d) * 3 + t);
      return true;
    }
  }
  return false;
}
// game.cpp:193-242
bool basic_legal(const State &s, int id) {
  MoveInfo mv = decode_move(id);
  if (mv.is_place) {
    if (pieces(s, to_play(s) * 3 + mv.piece) == 0) return false;
    int b = sq(s, mv.r1, mv.c1);
    if ((b & 7) == 0) return true;
    if (b & 8) return false;
    if (mv.piece == 0) return false;
    if (mv.piece == 1) return !(b & 6);
    return !((b & 4) || ((b & 1) && !(b & 2)));
  }
  int a = sq(s, mv.r0, mv.c0), b = sq(s, mv.r1, mv.c1);
  if ((a & 7) == 0 || (b & 7) == 0) return false;
  if ((a & 8) || (b & 8)) return false;
  return bottom_of(a & 7) - top_of(b & 7) == 1;
}
// game.cpp:28-43, 393-405
bool legal_moves(const State &s, Mask &m) {
  m.w[0] = m.w[1] = m.w[2] = 0xFFFFFFFFu;
  bool lines = false;
  lines |= apply_rowcol(s, m, false);
  lines |= apply_rowcol(s, m, true);
  lines |= apply_long_diag(s, m);
  lines |= apply_short_diag(s, m);
  for (int i = 0; i < kNumMoves; ++i)
    if (m.get(i) && !basic_legal(s, i)) m.clear(i);
  return lines;
}
// game.cpp:60-96
State do_move(const State &s, int id) {
  MoveInfo mv = decode_move(id);
  State o = s;
  o.w0 &= ~0x8888888888888888ull;
  int tp = to_play(s);
  int dst = mv.r1 * 16 + mv.c1 * 4;
  if (mv.is_place) {
    int pi = tp * 3 + mv.piece;
    uint64_t cnt = (uint64_t)(pieces(s, pi) - 1) & 0xff;
    o.w1 = (o.w1 & ~(0xffull << (8 * pi))) | (cnt << (8 * pi));
    o.w0 |= 1ull << (dst + mv.piece);
  } else {
    int src = mv.r0 * 16 + mv.c0 * 4;
    uint64_t stack = (o.w0 >> src) & 7;
    o.w0 |= stack << dst;
    o.w0 &= ~(7ull << src);
  }
  o.w0 |= 8ull << dst;
  o.w1 = (o.w1 & ~(0xffull << 48)) | ((uint64_t)(1 - tp) << 48);
  return o;
}
// game.cpp:45-58
void encode_state(const State &s, float out[kStateSize]) {
  for (int i = 0; i < 64; ++i) out[i] = ((s.w0 >> i) & 1) ? 1.0 : 0.0;
  int tp = to_play(s);
  for (int i = 0; i < 6; ++i) out[64 + i] = static_cast<float>(pieces(s, (tp * 3 + i) % 6)) * 0.25;
}
State start_state() {
  State s{0, 0};
  for (int i = 0; i < 6; ++i) s.w1 |= 4ull << (8 * i);
  return s;
}

// ------------------------------------------------------------------------------------------
// MT19937 (std::mt19937 semantics: 32-bit outputs, seed via the 1812433253 recurrence).
struct MT {
  uint32_t mt[624];
  int idx;
  void seed(uint32_t s) {
    mt[0] = s;
    for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + i;
    idx = 624;
  }
  void twist() {
    for (int i = 0; i < 624; ++i) {
      uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
      mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1) ? 0x9908b0dfu : 0u);
    }
    idx = 0;
  }
  uint32_t next() {
    if (idx >= 624) twist();
    uint32_t y = mt[idx++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
  }
};

// ------------------------------------------------------------------------------------------
// Slot word order (same as the CUDA engine, corintho_ai_b200/csrc/tree.cuh)
constexpr int kSEval = 0, kSVis = 1, kSOff = 2;
// Slot word s3 bit fields
inline int s3_move(uint32_t w) { return w & 0x7f; }
inline int s3_prior(uint32_t w) { return (w >> 7) & 0x1ff; }
inline int s3_result(uint32_t w) { return (w >> 16) & 7; }
inline bool s3_allv(uint32_t w) { return (w >> 19) & 1; }
inline bool s3_has(uint32_t w) { return (w >> 20) & 1; }
inline int s3_cnl(uint32_t w) { return (w >> 21) & 0x7f; }
inline uint32_t s3_set_result(uint32_t w, int r) { return (w & ~(7u << 16)) | ((uint32_t)r << 16); }
inline uint32_t s3_set_allv(uint32_t w, bool v) { return (w & ~(1u << 19)) | ((uint32_t)v << 19); }

inline bool r_known(int r) { return r != kResultNone; }
inline bool r_terminal(int r) { return r == kResultLoss || r == kResultDraw; }
inline bool r_won(int r) { return r == kDeducedWin; }
inline bool r_lost(int r) { return r == kResultLoss || r == kDeducedLoss; }
inline bool r_drawn(int r) { return r == kResultDraw || r == kDeducedDraw; }

struct Tree {
  int arena = -1;  // which of the game's three arenas
  bool has_root = false;
  uint32_t used = 0;  // words
  float root_eval = 0.0f;
  int root_visits = 1;
  int root_result = kResultNone;
  bool root_allv = true;
  int searches_done = 0;
};

struct Pending {
  uint32_t leaf_off;
  int path_len;
  uint32_t path[kMaxPath];  // slot offsets, level 1 (child of root) .. leaf
};

struct Sample {
  State state;
  float probs[kNumMoves];
};

struct Params {
  int max_searches, spe;
  float c_puct, epsilon;
  bool testing;
  uint32_t arena_words;
};

struct GameRec {
  MT rng;
  std::vector<uint32_t> arena[3];
  int spare = 2;
  Tree tree[2];
  int to_play = 0;
  int parity = 0;
  std::vector<Pending> pending;  // belongs to tree[to_play]
  std::vector<Sample> samples;
  int result = kResultNone;
  int mate_turn = 0;
  bool error = false;
  int64_t sims = 0, moves = 0, evals = 0;
};

struct Engine {
  Params p;
  std::vector<GameRec> games;
  std::vector<char> done;
  int iterations_done = 0;
  int num_threads = 1;
};

inline uint32_t *rec(GameRec &g, Tree &t, uint32_t off) { return g.arena[t.arena].data() + off; }

// Build a node record at `off` for `st` (Node ctor + initializeEdges, node.cpp:31-39,256-283).
// Returns n_legal and the terminal result through *result; advances t.used.
int make_record(GameRec &g, Tree &t, const Params &p, const State &st, int depth, int *result) {
  Mask m;
  bool lines = legal_moves(st, m);
  int n = m.count();
  uint32_t off = t.used;
  if (off + 8 + 4 * (uint32_t)n > p.arena_words) {
    g.error = true;
    *result = kResultNone;
    return -1;
  }
  uint32_t *r = rec(g, t, off);
  r[0] = (uint32_t)st.w0, r[1] = (uint32_t)(st.w0 >> 32);
  r[2] = (uint32_t)st.w1, r[3] = (uint32_t)(st.w1 >> 32);
  r[4] = (uint32_t)n | ((uint32_t)depth << 8);
  r[5] = f_bits(0.0f);
  r[6] = r[7] = 0;
  int e = 0;
  for (int i = 0; i < kNumMoves; ++i)
    if (m.get(i)) {
      uint32_t *s = r + 8 + 4 * e++;
      s[kSOff] = 0, s[kSEval] = 0, s[kSVis] = 0, s[3] = (uint32_t)i;
    }
  t.used = off + 8 + 4 * n;
  *result = n == 0 ? (lines ? kResultLoss : kResultDraw) : kResultNone;
  return n;
}

inline State rec_state(const uint32_t *r) {
  return State{(uint64_t)r[0] | ((uint64_t)r[1] << 32), (uint64_t)r[2] | ((uint64_t)r[3] << 32)};
}
inline int rec_nlegal(const uint32_t *r) { return r[4] & 0xff; }
inline int rec_depth(const uint32_t *r) { return (r[4] >> 8) & 0xff; }

// Fresh single-node tree (Node(game, depth), node.cpp:25-29; also the "reset tree" paths
// trainmc.cpp:397-404, 461-468 after the move has been applied by the caller).
void fresh_tree(GameRec &g, Tree &t, const Params &p, const State &st, int depth) {
  if (t.arena < 0) {  // first use: take the spare, hand back nothing
    t.arena = g.spare;
    g.spare = -1;
  }
  t.used = 0;
  int result;
  make_record(g, t, p, st, depth, &result);
  t.has_root = true;
  t.root_eval = 0.0f;
  t.root_visits = 1;
  t.root_result = result;
  t.root_allv = true;
}

void request_root(GameRec &g) {
  Pending pd;
  pd.leaf_off = 0;
  pd.path_len = 0;
  g.pending.push_back(pd);
}

// TrainMC::moveDown (trainmc.cpp:475-495): the child behind root slot `e` becomes the root.
// Breadth-first copy of its subtree into the spare arena.
void move_down(GameRec &g, Tree &t, int e) {
  uint32_t *src = g.arena[t.arena].data();
  uint32_t *slot = src + 8 + 4 * e;
  int dst_id = g.spare;
  uint32_t *dst = g.arena[dst_id].data();
  t.root_eval = bits_f(slot[kSEval]);
  t.root_visits = (int)slot[kSVis];
  t.root_result = s3_result(slot[3]);
  t.root_allv = s3_allv(slot[3]);
  uint32_t sz = 8 + 4 * (uint32_t)s3_cnl(slot[3]);
  memcpy(dst, src + slot[kSOff], sz * 4);
  uint32_t scan = 0, alloc = sz;
  while (scan < alloc) {
    uint32_t *r = dst + scan;
    int n = rec_nlegal(r);
    for (int k = 0; k < n; ++k) {
      uint32_t *s = r + 8 + 4 * k;
      if (s3_has(s[3])) {
        uint32_t csz = 8 + 4 * (uint32_t)s3_cnl(s[3]);
        memcpy(dst + alloc, src + s[kSOff], csz * 4);
        s[kSOff] = alloc;
        alloc += csz;
      }
    }
    scan += 8 + 4 * n;
  }
  g.spare = t.arena;
  t.arena = dst_id;
  t.used = alloc;
  t.searches_done = 0;
}

// TrainMC::receiveEval (trainmc.cpp:269-296) with getFilteredProbs (212-234),
// generateDirichlet (236-246), setProbs (248-267).
void receive_eval(GameRec &g, Tree &t, const Params &p, const float *eval, const float *probs) {
  for (size_t i = 0; i < g.pending.size(); ++i) {
    Pending &pd = g.pending[i];
    uint32_t *r = rec(g, t, pd.leaf_off);
    int n = rec_nlegal(r);
    float filtered[kNumMoves], dirichlet[kNumMoves];
    float sum = 0.0;
    for (int j = 0; j < n; ++j) {
      filtered[j] = probs[kNumMoves * i + s3_move(r[8 + 4 * j + 3])];
      sum += filtered[j];
    }
    float scalar = 1.0 / sum * (1 - p.epsilon);
    for (int j = 0; j < n; ++j) filtered[j] *= scalar;
    sum = 0.0;
    for (int j = 0; j < n; ++j) {
      dirichlet[j] = bits_f(kOGammaBits[g.rng.next() % 1024]);
      sum += dirichlet[j];
    }
    scalar = 1.0 / sum * p.epsilon;
    for (int j = 0; j < n; ++j) dirichlet[j] *= scalar;
    float weighted[kNumMoves];
    float max_prob = 0.0;
    for (int j = 0; j < n; ++j) {
      weighted[j] = filtered[j] + dirichlet[j];
      max_prob = (weighted[j] < max_prob) ? max_prob : weighted[j];  // std::max(w, max_prob)
    }
    float denom = 511.0f / max_prob;
    int final_sum = 0;
    for (int j = 0; j < n; ++j) {
      long q = lround(weighted[j] * denom);
      int prob = (int)q < 1 ? 1 : (int)q;
      uint32_t &w = r[8 + 4 * j + 3];
      w = (w & ~(0x1ffu << 7)) | ((uint32_t)(prob & 0x1ff) << 7);  // 9-bit field, node.h:116
      final_sum += prob;
    }
    r[5] = f_bits((float)(1.0 / static_cast<float>(final_sum)));
    // backup (trainmc.cpp:281-292)
    float cur_eval = eval[i];
    uint32_t *base = g.arena[t.arena].data();
    for (int lvl = pd.path_len - 1; lvl >= 0; --lvl) {
      uint32_t *s = base + pd.path[lvl];
      float d = cur_eval - 1.0;
      s[kSEval] = f_bits(bits_f(s[kSEval]) + d);
      s[3] = s3_set_allv(s[3], false);
      cur_eval *= -1.0;
    }
    float d = cur_eval - 1.0;
    t.root_eval += d;
  }
  t.root_allv = false;
  g.evals += (int64_t)g.pending.size();
  g.pending.clear();
}

// TrainMC::search (trainmc.cpp:602-696) with chooseNext (540-600) and propagateTerminal
// (497-538) inlined on the explicit path.
void search(GameRec &g, Tree &t, const Params &p) {
  uint32_t *base = g.arena[t.arena].data();
  ++t.searches_done;
  uint32_t node_off[kMaxPath + 1];  // record offset per level (0 = root)
  uint32_t slot_off[kMaxPath + 1];  // slot through which level L was reached (L>=1)
  int level = 0;
  node_off[0] = 0;
  int cur_result = t.root_result;
  int cur_visits = t.root_visits;
  while (!r_terminal(cur_result)) {
    uint32_t *r = base + node_off[level];
    int n = rec_nlegal(r);
    float denominator = bits_f(r[5]);
    // ---- chooseNext
    float max_eval = -INFINITY;
    int choice = -1;
    // unqualified sqrt(float) binds to double sqrt(double) in the reference TU (SURVEY Q9)
    float v_sqrt = (float)((double)p.c_puct * sqrt((double)static_cast<float>(cur_visits)));
    for (int e = 0; e < n; ++e) {
      const uint32_t *s = r + 8 + 4 * e;
      float u = -INFINITY;
      float prob = static_cast<float>(s3_prior(s[3])) * denominator;
      if (s3_has(s[3])) {
        int cr = s3_result(s[3]);
        if ((!r_known(cr) || r_drawn(cr)) && !s3_allv(s[3])) {
          if (r_drawn(cr)) {
            u = prob * v_sqrt;
          } else {
            int cv = (int)s[kSVis];
            u = -1.0 * bits_f(s[kSEval]) / static_cast<float>(cv) +
                prob * v_sqrt / (static_cast<float>(cv) + 1.0);
          }
        }
      } else {
        u = prob * v_sqrt;
      }
      if (u > max_eval) {
        max_eval = u;
        choice = e;
      }
    }
    // ---- virtual loss on the node we stand on (trainmc.cpp:611,625)
    auto bump = [&](int lvl, int dv, float de) {
      if (lvl == 0) {
        t.root_visits += dv;
        t.root_eval += de;
      } else {
        uint32_t *s = base + slot_off[lvl];
        s[kSVis] = (uint32_t)((int)s[kSVis] + dv);
        s[kSEval] = f_bits(bits_f(s[kSEval]) + de);
      }
    };
    bump(level, +1, 1.0f);
    if (choice < 0) {  // kNone (trainmc.cpp:629-643)
      if (level == 0)
        t.root_allv = true;
      else
        base[slot_off[level] + 3] = s3_set_allv(base[slot_off[level] + 3], true);
      for (int l = level; l >= 0; --l) bump(l, -1, -1.0f);
      --t.searches_done;
      return;
    }
    uint32_t *s = r + 8 + 4 * choice;
    uint32_t so = node_off[level] + 8 + 4 * choice;
    if (!s3_has(s[3])) {  // kNew: expand
      if (level + 1 >= kMaxPath) {
        g.error = true;
        return;
      }
      State child = do_move(rec_state(r), s3_move(s[3]));
      uint32_t coff = t.used;
      int result;
      int cn = make_record(g, t, p, child, rec_depth(r) + 1, &result);
      if (cn < 0) return;
      base = g.arena[t.arena].data();
      s = base + so;
      s[kSOff] = coff;
      s[kSEval] = f_bits(0.0f);
      s[kSVis] = 1;
      s[3] = (s[3] & 0xffffu) | ((uint32_t)result << 16) | (1u << 19) | (1u << 20) |
             ((uint32_t)cn << 21);
      ++level;
      node_off[level] = coff;
      slot_off[level] = so;
      cur_result = result;
      cur_visits = 1;
      break;
    }
    ++level;
    node_off[level] = s[kSOff];
    slot_off[level] = so;
    cur_result = s3_result(s[3]);
    cur_visits = (int)s[kSVis];
  }
  if (r_terminal(cur_result)) {
    // ---- propagateTerminal (trainmc.cpp:497-538)
    {
      int l = level;
      int res_l = cur_result;  // result of the node at level l
      while (l != 0) {
        auto get_res = [&](int lvl) {
          return lvl == 0 ? t.root_result : s3_result(base[slot_off[lvl] + 3]);
        };
        auto set_res = [&](int lvl, int rr) {
          if (lvl == 0)
            t.root_result = rr;
          else
            base[slot_off[lvl] + 3] = s3_set_result(base[slot_off[lvl] + 3], rr);
        };
        if (r_lost(res_l)) {
          --l;
          set_res(l, kDeducedWin);
        } else {
          --l;
          uint32_t *pr = base + node_off[l];
          int pn = rec_nlegal(pr);
          bool all_known = true;
          for (int k = 0; k < pn; ++k) {
            uint32_t w3 = pr[8 + 4 * k + 3];
            if (!s3_has(w3) || !r_known(s3_result(w3))) {
              all_known = false;
              break;
            }
          }
          if (!all_known) break;
          bool has_draw = r_drawn(get_res(l));  // Q4: tests the parent itself
          set_res(l, has_draw ? kDeducedDraw : kDeducedLoss);
        }
        res_l = get_res(l);
      }
    }
    // ---- terminal backup (trainmc.cpp:666-682)
    float cur_eval = -1.0;
    if (r_drawn(cur_result)) cur_eval = 0.0;
    base[slot_off[level] + kSEval] = f_bits(cur_eval);
    for (int l = level - 1; l >= 0; --l) {
      float d = cur_eval - 1.0;
      if (l == 0)
        t.root_eval += d;
      else
        base[slot_off[l] + kSEval] = f_bits(bits_f(base[slot_off[l] + kSEval]) + d);
      cur_eval *= -1.0;
    }
  } else {
    base[slot_off[level] + kSEval] = f_bits(1.0f);
    Pending pd;
    pd.leaf_off = node_off[level];
    pd.path_len = level;
    for (int l = 1; l <= level; ++l) pd.path[l - 1] = slot_off[l];
    g.pending.push_back(pd);
  }
}

// TrainMC::doIteration (trainmc.cpp:139-178)
bool tree_do_iteration(GameRec &g, Tree &t, const Params &p, const float *eval,
                       const float *probs) {
  if (!t.has_root) {
    fresh_tree(g, t, p, start_state(), 0);
    t.searches_done = 1;
    request_root(g);
    return false;
  }
  if (t.searches_done == 0 && t.root_visits == 1 && t.root_allv) {
    t.searches_done = 1;
    request_root(g);
    return false;
  }
  if (!g.pending.empty()) receive_eval(g, t, p, eval, probs);
  while ((int)g.pending.size() < p.spe && t.searches_done < p.max_searches &&
         !r_known(t.root_result) && !t.root_allv && !g.error) {
    search(g, t, p);
  }
  return (t.searches_done == p.max_searches || r_known(t.root_result)) && g.pending.empty();
}

// TrainMC::chooseHighProbMove (trainmc.cpp:298-308), int32 max_prob quirk (Q3)
int choose_high_prob(GameRec &g, Tree &t) {
  uint32_t *r = rec(g, t, 0);
  int n = rec_nlegal(r);
  float denominator = bits_f(r[5]);
  int32_t max_prob = 0;
  int choice = 0;
  for (int i = 0; i < n; ++i) {
    float pr = static_cast<float>(s3_prior(r[8 + 4 * i + 3])) * denominator;
    if (pr > max_prob) {
      max_prob = pr;
      choice = s3_move(r[8 + 4 * i + 3]);
    }
  }
  return choice;
}

// Replace the tree by the single node reached by `move` from the root (trainmc.cpp:397-404)
void reset_tree_after(GameRec &g, Tree &t, const Params &p, int move) {
  uint32_t *r = rec(g, t, 0);
  State st = do_move(rec_state(r), move);
  int depth = rec_depth(r) + 1;
  fresh_tree(g, t, p, st, depth);
  t.searches_done = 0;
}

// TrainMC::chooseMove (trainmc.cpp:110-137) and the four strategies (310-473).
// Returns the move id; prob_sample may be null (testing).
int choose_move(GameRec &g, Tree &t, const Params &p, float *prob_sample) {
  uint32_t *r = rec(g, t, 0);
  int n = rec_nlegal(r);
  auto slot = [&](int e) { return r + 8 + 4 * e; };
  if (r_won(t.root_result)) {  // chooseMoveWon
    int choice = 0, best = -1;
    for (int e = 0; e < n; ++e)
      if (s3_has(slot(e)[3]) && r_lost(s3_result(slot(e)[3]))) {
        choice = s3_move(slot(e)[3]);
        best = e;
        break;
      }
    if (prob_sample) prob_sample[choice] = 1.0;
    if (best < 0) {  // unreachable in the reference (would dereference null); fail loudly
      g.error = true;
      return choice;
    }
    move_down(g, t, best);
    return choice;
  }
  if (r_lost(t.root_result) || r_drawn(t.root_result)) {  // chooseMoveLostDrawn
    int max_visits = 0, choice = 0, best = -1;
    for (int e = 0; e < n; ++e) {
      if (!s3_has(slot(e)[3])) continue;
      int cv = (int)slot(e)[kSVis];
      if (cv > max_visits && (r_lost(t.root_result) || !r_won(s3_result(slot(e)[3])))) {
        choice = s3_move(slot(e)[3]);
        best = e;
        max_visits = cv;
      }
    }
    if (prob_sample) prob_sample[choice] = 1.0;
    if (best < 0) {
      g.error = true;
      return choice;
    }
    move_down(g, t, best);
    return choice;
  }
  if (rec_depth(r) < 6 && !p.testing) {  // chooseMoveOpening
    int choice = choose_high_prob(g, t);
    int visits = 0;
    for (int e = 0; e < n; ++e)
      if (s3_has(slot(e)[3]) && !r_won(s3_result(slot(e)[3]))) visits += (int)slot(e)[kSVis];
    float denominator = 1.0 / static_cast<float>(visits);
    if (prob_sample)
      for (int e = 0; e < n; ++e)
        if (s3_has(slot(e)[3]) && !r_won(s3_result(slot(e)[3])))
          prob_sample[s3_move(slot(e)[3])] = static_cast<float>((int)slot(e)[kSVis]) * denominator;
    if (visits == 0) {
      prob_sample[choice] = 1.0;
      reset_tree_after(g, t, p, choice);
      return choice;
    }
    int target = g.rng.next() % visits;
    int total = 0, best = -1;
    for (int e = 0; e < n; ++e)
      if (s3_has(slot(e)[3]) && !r_won(s3_result(slot(e)[3]))) {
        total += (int)slot(e)[kSVis];
        if (total > target) {
          choice = s3_move(slot(e)[3]);
          best = e;
          break;
        }
      }
    move_down(g, t, best);
    return choice;
  }
  // chooseMoveNormal
  int max_visits = 0;
  float max_eval = 0.0;
  int choice = choose_high_prob(g, t);
  int best = -1;
  for (int e = 0; e < n; ++e) {
    if (!s3_has(slot(e)[3])) continue;
    int cr = s3_result(slot(e)[3]);
    if (r_won(cr)) continue;
    float ev = bits_f(slot(e)[kSEval]);
    if (cr == kResultDraw || cr == kDeducedDraw) ev = 0.0;
    int cv = (int)slot(e)[kSVis];
    if (cv > max_visits || (cv == max_visits && ev > max_eval)) {
      choice = s3_move(slot(e)[3]);
      best = e;
      max_visits = cv;
      max_eval = ev;
    }
  }
  if (prob_sample) prob_sample[choice] = 1.0;
  if (max_visits == 0) {
    reset_tree_after(g, t, p, choice);
    return choice;
  }
  move_down(g, t, best);
  return choice;
}

// TrainMC::receiveOpponentMove (trainmc.cpp:180-204)
bool receive_opponent_move(GameRec &g, Tree &t, const Params &p, int move, const State &st,
                           int depth) {
  uint32_t *r = rec(g, t, 0);
  int n = rec_nlegal(r);
  for (int e = 0; e < n; ++e) {
    uint32_t w3 = r[8 + 4 * e + 3];
    if (s3_has(w3) && s3_move(w3) == move) {
      move_down(g, t, e);
      return false;
    }
  }
  fresh_tree(g, t, p, st, depth);
  request_root(g);
  t.searches_done = 1;
  return true;
}

void drop_tree(GameRec &g, Tree &t) {
  t.has_root = false;
  (void)g;
}

// SelfPlayer::chooseMoveAndContinue (selfplayer.cpp:246-291) incl. chooseMove (234-244) and
// endGame (206-232). Returns true when the game is over.
bool choose_move_and_continue(GameRec &g, const Params &p) {
  bool need_eval = false;
  while (!need_eval) {
    Tree &t = g.tree[g.to_play];
    if (r_known(t.root_result) && g.mate_turn == 0) g.mate_turn = (int)g.samples.size() + 1;
    g.sims += t.searches_done;
    g.moves += 1;
    int choice;
    if (!p.testing) {
      Sample smp;
      smp.state = rec_state(rec(g, t, 0));
      memset(smp.probs, 0, sizeof(smp.probs));
      choice = choose_move(g, t, p, smp.probs);
      g.samples.push_back(smp);
      if ((int)g.samples.size() > kMaxSamples) g.error = true;
    } else {
      choice = choose_move(g, t, p, nullptr);
    }
    if (g.error) return true;
    if (r_terminal(t.root_result)) {  // endGame
      if (t.root_result == kResultDraw)
        g.result = kResultDraw;
      else if (g.to_play == 1)
        g.result = kResultLoss;
      else
        g.result = kResultWin;
      drop_tree(g, g.tree[0]);
      drop_tree(g, g.tree[1]);
      return true;
    }
    g.to_play = 1 - g.to_play;
    Tree &o = g.tree[g.to_play];
    const uint32_t *mr = rec(g, t, 0);  // mover's new root
    State st = rec_state(mr);
    int depth = rec_depth(mr);
    if (!o.has_root) {
      fresh_tree(g, o, p, st, depth);
      o.searches_done = 0;
      return tree_do_iteration(g, o, p, nullptr, nullptr);  // always false: root needs an eval
    }
    need_eval = receive_opponent_move(g, o, p, choice, st, depth);
    if (!need_eval) need_eval = !tree_do_iteration(g, o, p, nullptr, nullptr);
  }
  return false;
}

// SelfPlayer::doIteration (selfplayer.cpp:115-122)
bool game_do_iteration(GameRec &g, const Params &p, const float *eval, const float *probs) {
  bool done = tree_do_iteration(g, g.tree[g.to_play], p, eval, probs);
  if (g.error) return true;
  if (done) return choose_move_and_continue(g, p);
  return false;
}

int game_num_requests(const GameRec &g) { return (int)g.pending.size(); }

float game_score(const GameRec &g) {  // selfplayer.cpp:57-64
  if (g.result == kResultLoss) return 0.0;
  if (g.result == kResultWin) return 1.0;
  return 0.5;
}


// ---- Match (match.h:33-101, match.cpp) ---------------------------------------------------------
// One game between two players with their own search budgets (Player, match.h:13-31). A random
// player has no tree (match.cpp:27-33). The authoritative position lives outside both trees
// (Match::root_, match.h:96).
struct MatchRec {
  GameRec g;
  Params p[2];
  bool random[2] = {false, false};
  int ids[2] = {0, 0};
  int model_ids[2] = {0, 0};
  State root;
  int root_depth = 0;
};

// std::uniform_int_distribution<int32_t>(0, n - 1)(mt19937) as libstdc++ (GCC 11+) implements it:
// Lemire's nearly divisionless method on a 64-bit product (bits/uniform_int_dist.h, _S_nd)
int uniform_index(MT &rng, uint32_t n) {
  uint64_t product = (uint64_t)rng.next() * (uint64_t)n;
  uint32_t low = (uint32_t)product;
  if (low < n) {
    const uint32_t threshold = (0u - n) % n;
    while (low < threshold) {
      product = (uint64_t)rng.next() * (uint64_t)n;
      low = (uint32_t)product;
    }
  }
  return (int)(product >> 32);
}

// Match::chooseMoveAndContinue (match.cpp:208-251) incl. chooseMove (193-206), endGame (161-190)
bool match_choose_move_and_continue(MatchRec &m) {
  GameRec &g = m.g;
  bool need_eval = false;
  while (!need_eval) {
    int choice;
    if (m.random[g.to_play]) {
      Mask lm;
      legal_moves(m.root, lm);
      int moves[kNumMoves], n = 0;
      for (int id = 0; id < kNumMoves; ++id)
        if (lm.get(id)) moves[n++] = id;
      choice = moves[uniform_index(g.rng, (uint32_t)n)];
    } else {
      Tree &t = g.tree[g.to_play];
      g.sims += t.searches_done;
      g.moves += 1;
      choice = choose_move(g, t, m.p[g.to_play], nullptr);
      if (g.error) return true;
    }
    m.root = do_move(m.root, choice);
    m.root_depth += 1;
    Mask lm;
    const bool lines = legal_moves(m.root, lm);
    if (lm.count() == 0) {  // endGame
      if (!lines)
        g.result = kResultDraw;
      else if (g.to_play == 1)
        g.result = kResultLoss;
      else
        g.result = kResultWin;
      drop_tree(g, g.tree[0]);
      drop_tree(g, g.tree[1]);
      g.pending.clear();
      return true;
    }
    g.to_play = 1 - g.to_play;
    if (m.random[g.to_play]) continue;
    Tree &o = g.tree[g.to_play];
    const Params &po = m.p[g.to_play];
    if (!o.has_root) {
      fresh_tree(g, o, po, m.root, m.root_depth);
      o.searches_done = 0;
      return tree_do_iteration(g, o, po, nullptr, nullptr);  // always false: root needs an eval
    }
    need_eval = receive_opponent_move(g, o, po, choice, m.root, m.root_depth);
    if (!need_eval) need_eval = !tree_do_iteration(g, o, po, nullptr, nullptr);
  }
  return false;
}

// Match::doIteration (match.cpp:66-77)
bool match_do_iteration(MatchRec &m, const float *eval, const float *probs) {
  GameRec &g = m.g;
  if (m.random[g.to_play]) return match_choose_move_and_continue(m);
  bool done = tree_do_iteration(g, g.tree[g.to_play], m.p[g.to_play], eval, probs);
  if (g.error) return true;
  if (done) return match_choose_move_and_continue(m);
  return false;
}

// Match::num_requests (match.cpp:44-48): the side to move's queue; a random player has none
int match_num_requests(const MatchRec &m) {
  if (m.random[m.g.to_play]) return 0;
  return (int)m.g.pending.size();
}

struct PlayerCfg {
  int model_id, max_searches, spe;
  float c_puct, epsilon;
  bool random;
};

struct TourneyRec {
  std::vector<MatchRec *> matches;
  std::vector<char> done;
  std::map<int, PlayerCfg> players;
  MT generator;  // std::mt19937 default seed (tourney.h:42)
  int num_threads = 1;
  TourneyRec() { generator.seed(5489u); }
  ~TourneyRec() {
    for (MatchRec *m : matches) delete m;
  }
};

}  // namespace

// ==========================================================================================
extern "C" {

void orc_line_breaker(int idx, uint32_t out[3]) {
  for (int k = 0; k < 3; ++k) out[k] = kOLineBreakers[idx][k];
}
float orc_gamma_sample(int i) { return bits_f(kOGammaBits[i]); }

void orc_move_decode(int id, int out[6]) {
  MoveInfo m = decode_move(id);
  out[0] = m.is_place, out[1] = m.piece, out[2] = m.r0, out[3] = m.c0, out[4] = m.r1,
  out[5] = m.c1;
}
int orc_encode_place(int row, int col, int piece) { return encode_place(row, col, piece); }
int orc_encode_move(int r0, int c0, int r1, int c1) { return encode_move(r0, c0, r1, c1); }

void orc_game_start(uint64_t st[2]) {
  State s = start_state();
  st[0] = s.w0, st[1] = s.w1;
}
int orc_game_legal(const uint64_t st[2], uint32_t mask[3]) {
  Mask m;
  bool lines = legal_moves(State{st[0], st[1]}, m);
  mask[0] = m.w[0], mask[1] = m.w[1], mask[2] = m.w[2];
  return lines ? 1 : 0;
}
void orc_game_do_move(const uint64_t st[2], int move, uint64_t out[2]) {
  State o = do_move(State{st[0], st[1]}, move);
  out[0] = o.w0, out[1] = o.w1;
}
void orc_game_encode(const uint64_t st[2], float out[70]) {
  encode_state(State{st[0], st[1]}, out);
}
void orc_game_step_batch(int64_t n, const uint64_t *states, const uint32_t *rnd, uint32_t *masks,
                         uint32_t *flags, uint64_t *next, float *enc, int num_threads) {
  omp_set_num_threads(num_threads > 0 ? num_threads : 1);
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; ++i) {
    State s{states[2 * i], states[2 * i + 1]};
    Mask m;
    bool lines = legal_moves(s, m);
    masks[3 * i] = m.w[0], masks[3 * i + 1] = m.w[1], masks[3 * i + 2] = m.w[2];
    int nl = m.count();
    int result = nl == 0 ? (lines ? kResultLoss : kResultDraw) : kResultNone;
    if (enc) encode_state(s, enc + kStateSize * i);
    int chosen = 0x7f;
    State o = s;
    if (nl > 0) {
      int k = rnd[i] % nl;
      for (int mv = 0; mv < kNumMoves; ++mv)
        if (m.get(mv) && k-- == 0) {
          chosen = mv;
          break;
        }
      o = do_move(s, chosen);
    }
    next[2 * i] = o.w0, next[2 * i + 1] = o.w1;
    flags[i] = (uint32_t)result | (lines ? 4u : 0u) | ((uint32_t)nl << 8) | ((uint32_t)chosen << 16);
  }
}

// Reachable states from uniformly random legal play-outs, the generator of ref_gen_states
// (ref_harness.cpp) restated on the oracle's rules: every position of every play-out (start and
// terminal positions included) is emitted until n states exist. Returns the number of play-outs.
int64_t orc_gen_states(uint64_t seed, int64_t n, uint64_t *out) {
  uint64_t s = seed;
  int64_t count = 0, games = 0;
  while (count < n) {
    State g = start_state();
    ++games;
    for (;;) {
      out[2 * count] = g.w0, out[2 * count + 1] = g.w1;
      if (++count >= n) break;
      Mask m;
      legal_moves(g, m);
      int nl = m.count();
      if (nl == 0) break;
      uint64_t z = (s += 0x9E3779B97F4A7C15ull);  // splitmix64
      z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
      z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
      int k = (int)((z ^ (z >> 31)) % (uint64_t)nl);
      int chosen = 0;
      for (int mv = 0; mv < kNumMoves; ++mv)
        if (m.get(mv) && k-- == 0) {
          chosen = mv;
          break;
        }
      g = do_move(g, chosen);
    }
  }
  return games;
}

// ---- Trainer (trainer.cpp:18-256) --------------------------------------------------------
// Shard of a larger run (the engine's multi-GPU partitioning, not in the reference): global games
// [first_game, first_game + num_games) of the seed stream of mt19937(seed), parity = global index
// % 2 (trainer.cpp:238-256 applied to the global index). The staggered start uses local indices;
// it only moves games between iterations and does not change any per-game result.
void *orc_trainer_create_shard(int first_game, int num_games, const char *log_folder, int seed,
                               int max_searches, int searches_per_eval, float c_puct, float epsilon,
                               int num_logged, int num_threads, int testing);
void *orc_trainer_create(int num_games, const char *log_folder, int seed, int max_searches,
                         int searches_per_eval, float c_puct, float epsilon, int num_logged,
                         int num_threads, int testing) {
  return orc_trainer_create_shard(0, num_games, log_folder, seed, max_searches, searches_per_eval,
                                  c_puct, epsilon, num_logged, num_threads, testing);
}
void *orc_trainer_create_shard(int first_game, int num_games, const char *log_folder, int seed,
                               int max_searches, int searches_per_eval, float c_puct, float epsilon,
                               int num_logged, int num_threads, int testing) {
  (void)log_folder;
  (void)num_logged;
  Engine *E = new Engine();
  E->p = Params{max_searches, searches_per_eval, c_puct, epsilon, testing != 0, 0};
  // arena budget: kept subtree + max_searches new nodes, with head-room (fails loudly if hit)
  uint64_t nodes = (uint64_t)max_searches * 3 + 64;
  E->p.arena_words = (uint32_t)(nodes * (8 + 4 * 40));
  E->num_threads = num_threads > 0 ? num_threads : 1;
  E->games.resize(num_games);
  E->done.assign(num_games, 0);
  MT gen;
  gen.seed((uint32_t)seed);
  for (int i = 0; i < first_game; ++i) gen.next();
  for (int i = 0; i < num_games; ++i) {
    GameRec &g = E->games[i];
    g.rng.seed(gen.next());
    g.parity = (first_game + i) % 2;
    for (int a = 0; a < 3; ++a) g.arena[a].assign(E->p.arena_words, 0);
    g.tree[0].arena = 0;
    g.tree[1].arena = 1;
    g.spare = 2;
    g.pending.reserve(searches_per_eval);
  }
  return E;
}
void orc_trainer_destroy(void *h) { delete static_cast<Engine *>(h); }

static bool game_selected(const Engine *E, size_t i, int to_play) {
  if (E->done[i]) return false;
  if (to_play != 0 && to_play != 1) return true;
  return E->games[i].to_play == (to_play + E->games[i].parity) % 2;
}

int orc_trainer_num_requests(void *h, int to_play) {
  Engine *E = static_cast<Engine *>(h);
  int n = 0;
  for (size_t i = 0; i < E->games.size(); ++i)
    if (game_selected(E, i, to_play)) n += game_num_requests(E->games[i]);
  return n;
}

void orc_trainer_write_requests(void *h, float *game_states, int to_play) {
  Engine *E = static_cast<Engine *>(h);
  int64_t off = 0;
  for (size_t i = 0; i < E->games.size(); ++i) {
    if (!game_selected(E, i, to_play)) continue;
    GameRec &g = E->games[i];
    Tree &t = g.tree[g.to_play];
    for (size_t k = 0; k < g.pending.size(); ++k) {
      encode_state(rec_state(rec(g, t, g.pending[k].leaf_off)), game_states + kStateSize * off);
      ++off;
    }
  }
}

int orc_trainer_do_iteration(void *h, const float *eval, const float *probs, int to_play) {
  Engine *E = static_cast<Engine *>(h);
  size_t G = E->games.size();
  bool training = (to_play != 0 && to_play != 1);
  std::vector<int64_t> offsets(G, 0);
  int64_t off = 0;
  for (size_t i = 0; i < G; ++i) {
    offsets[i] = off;
    if (training ? !E->done[i] : game_selected(E, i, to_play)) off += game_num_requests(E->games[i]);
  }
  size_t stagger = G / (size_t)E->p.max_searches;
  if (stagger < 1) stagger = 1;
  omp_set_num_threads(E->num_threads);
#pragma omp parallel for schedule(dynamic, 1)
  for (size_t i = 0; i < G; ++i) {
    if (training) {
      if (E->done[i]) continue;
      if (i / stagger > (size_t)E->iterations_done) continue;  // trainer.cpp:184-186
    } else if (!game_selected(E, i, to_play)) {
      continue;
    }
    bool d = game_do_iteration(E->games[i], E->p, eval ? eval + offsets[i] : nullptr,
                               probs ? probs + kNumMoves * offsets[i] : nullptr);
    if (d) E->done[i] = 1;
  }
  if (training) ++E->iterations_done;
  for (size_t i = 0; i < G; ++i) {
    if (E->games[i].error) return -1;
  }
  for (size_t i = 0; i < G; ++i)
    if (!E->done[i]) return 0;
  return 1;
}

int orc_trainer_num_samples(void *h) {
  Engine *E = static_cast<Engine *>(h);
  int n = 0;
  for (auto &g : E->games) n += (int)g.samples.size();
  return n;
}

// SelfPlayer::writeSamples (selfplayer.cpp:79-113) / Trainer::writeSamples (trainer.cpp:103-113)
void orc_trainer_write_samples(void *h, float *game_states, float *eval_samples,
                               float *prob_samples) {
  Engine *E = static_cast<Engine *>(h);
  int64_t off = 0;
  for (auto &g : E->games) {
    float evaluation = 1.0;
    if (g.result == kResultDraw) evaluation = 0.0;
    for (int i = (int)g.samples.size() - 1; i >= 0; --i) {
      float gs[kStateSize];
      encode_state(g.samples[i].state, gs);
      for (int k = 0; k < 8; ++k) {
        float *o = game_states + ((off + i) * 8 + k) * kStateSize;
        for (int j = 0; j < 64; ++j) o[j] = gs[kOSpaceSym[k][j / 4] * 4 + j % 4];
        for (int j = 64; j < kStateSize; ++j) o[j] = gs[j];
        eval_samples[(off + i) * 8 + k] = evaluation;
        float *po = prob_samples + ((off + i) * 8 + k) * kNumMoves;
        for (int j = 0; j < kNumMoves; ++j) po[j] = g.samples[i].probs[kOMoveSym[k][j]];
      }
      evaluation *= -1.0;
    }
    off += (int64_t)g.samples.size();
  }
}

float orc_trainer_score(void *h) {  // trainer.cpp:59-68
  Engine *E = static_cast<Engine *>(h);
  float score = 0;
  // even (global) indices first, then odd ones; g.parity == i % 2 unless this is a shard
  for (size_t i = 0; i < E->games.size(); ++i)
    if (E->games[i].parity == 0) score += game_score(E->games[i]);
  for (size_t i = 0; i < E->games.size(); ++i)
    if (E->games[i].parity == 1) score += 1.0 - game_score(E->games[i]);
  return score / E->games.size();
}

float orc_trainer_avg_mate_length(void *h) {  // trainer.cpp:70-77, selfplayer.cpp:66-71
  Engine *E = static_cast<Engine *>(h);
  int total = 0;
  for (auto &g : E->games)
    total += g.mate_turn == 0 ? 0 : (int)g.samples.size() - g.mate_turn + 1;
  return static_cast<float>(total) / E->games.size();
}

void orc_trainer_game_results(void *h, int32_t *results) {  // per game: util.h:58-61 result code
  Engine *E = static_cast<Engine *>(h);
  for (size_t i = 0; i < E->games.size(); ++i) results[i] = E->games[i].result;
}

void orc_trainer_counters(void *h, int64_t out[3]) {
  Engine *E = static_cast<Engine *>(h);
  out[0] = out[1] = out[2] = 0;
  for (auto &g : E->games) out[0] += g.sims, out[1] += g.moves, out[2] += g.evals;
}

int orc_trainer_dump_tree(void *h, int game, int player, int64_t out[8], uint32_t *words,
                          int cap) {
  Engine *E = static_cast<Engine *>(h);
  GameRec &g = E->games[game];
  Tree &t = g.tree[player];
  out[0] = t.has_root, out[1] = t.used, out[2] = t.root_visits, out[3] = t.root_result;
  out[4] = t.root_allv, out[5] = t.searches_done, out[6] = f_bits(t.root_eval), out[7] = g.to_play;
  if (t.has_root && words) {
    int n = (int)t.used < cap ? (int)t.used : cap;
    memcpy(words, g.arena[t.arena].data(), (size_t)n * 4);
  }
  return (int)t.used;
}


// ---- Tourney (tourney.h:12-46, tourney.cpp) ----------------------------------------------------
void *orc_tourney_create(int num_threads, const char *log_folder) {
  (void)log_folder;
  TourneyRec *T = new TourneyRec();
  T->num_threads = num_threads > 0 ? num_threads : 1;
  return T;
}
void orc_tourney_destroy(void *h) { delete static_cast<TourneyRec *>(h); }

void orc_tourney_add_player(void *h, int player_id, int model_id, int max_searches,
                            int searches_per_eval, float c_puct, float epsilon, int random) {
  static_cast<TourneyRec *>(h)->players[player_id] =
      PlayerCfg{model_id, max_searches, searches_per_eval, c_puct, epsilon, random != 0};
}

// Tourney::addMatch (tourney.cpp:80-96): the match seed is the next draw of the tourney generator
void orc_tourney_add_match(void *h, int player1, int player2, int logging) {
  (void)logging;
  TourneyRec *T = static_cast<TourneyRec *>(h);
  MatchRec *m = new MatchRec();
  const int pid[2] = {player1, player2};
  int max_ms = 1, max_spe = 1;
  for (int s = 0; s < 2; ++s) {
    const PlayerCfg &c = T->players[pid[s]];
    m->p[s] = Params{c.max_searches, c.spe, c.c_puct, c.epsilon, true, 0};
    m->random[s] = c.random;
    m->ids[s] = pid[s];
    m->model_ids[s] = c.model_id;
    if (c.max_searches > max_ms) max_ms = c.max_searches;
    if (c.spe > max_spe) max_spe = c.spe;
  }
  const uint32_t words = (uint32_t)(((uint64_t)max_ms * 3 + 64) * (8 + 4 * 40));
  m->p[0].arena_words = m->p[1].arena_words = words;
  GameRec &g = m->g;
  g.rng.seed(T->generator.next());
  for (int a = 0; a < 3; ++a) g.arena[a].assign(words, 0);
  g.tree[0].arena = 0;
  g.tree[1].arena = 1;
  g.spare = 2;
  g.pending.reserve(max_spe);
  m->root = start_state();
  m->root_depth = 0;
  T->matches.push_back(m);
  T->done.push_back(0);
}

int orc_tourney_all_done(void *h) {
  TourneyRec *T = static_cast<TourneyRec *>(h);
  for (char d : T->done)
    if (!d) return 0;
  return 1;
}

static bool match_selected(const TourneyRec *T, size_t i, int id) {
  return !T->done[i] && T->matches[i]->model_ids[T->matches[i]->g.to_play] == id;
}

int orc_tourney_num_requests(void *h, int id) {
  TourneyRec *T = static_cast<TourneyRec *>(h);
  int n = 0;
  for (size_t i = 0; i < T->matches.size(); ++i)
    if (match_selected(T, i, id)) n += match_num_requests(*T->matches[i]);
  return n;
}

void orc_tourney_write_requests(void *h, float *game_states, int id) {
  TourneyRec *T = static_cast<TourneyRec *>(h);
  int64_t off = 0;
  for (size_t i = 0; i < T->matches.size(); ++i) {
    if (!match_selected(T, i, id)) continue;
    MatchRec &m = *T->matches[i];
    if (m.random[m.g.to_play]) continue;
    GameRec &g = m.g;
    Tree &t = g.tree[g.to_play];
    for (size_t k = 0; k < g.pending.size(); ++k) {
      encode_state(rec_state(rec(g, t, g.pending[k].leaf_off)), game_states + kStateSize * off);
      ++off;
    }
  }
}

// Tourney::doIteration (tourney.cpp:54-72). The answer offset of match i is advanced by the
// request count of match i-1 whenever match i itself is selected -- literally as written there
// (SURVEY Q14); it equals the packing of writeRequests when the selected matches are adjacent.
int orc_tourney_do_iteration(void *h, const float *eval, const float *probs, int id) {
  TourneyRec *T = static_cast<TourneyRec *>(h);
  const size_t n = T->matches.size();
  std::vector<int64_t> offsets(n, 0);
  int64_t off = 0;
  for (size_t i = 1; i < n; ++i) {
    if (match_selected(T, i, id)) off += match_num_requests(*T->matches[i - 1]);
    offsets[i] = off;
  }
  omp_set_num_threads(T->num_threads);
#pragma omp parallel for schedule(dynamic, 1)
  for (size_t i = 0; i < n; ++i) {
    if (!match_selected(T, i, id)) continue;
    if (match_do_iteration(*T->matches[i], eval + offsets[i], probs + kNumMoves * offsets[i]))
      T->done[i] = 1;
  }
  for (size_t i = 0; i < n; ++i)
    if (T->matches[i]->g.error) return -1;
  return 0;
}

// Tourney::writeScores (tourney.cpp:34-42): "<player1> <player2> <score>" per finished match
void orc_tourney_write_scores(void *h, const char *file) {
  TourneyRec *T = static_cast<TourneyRec *>(h);
  FILE *f = fopen(file, "w");
  if (!f) return;
  for (size_t i = 0; i < T->matches.size(); ++i) {
    if (!T->done[i]) continue;
    const MatchRec &m = *T->matches[i];
    const float sc = game_score(m.g);
    fprintf(f, "%d %d %s\n", m.ids[0], m.ids[1], sc == 0.5f ? "0.5" : (sc == 1.0f ? "1" : "0"));
  }
  fclose(f);
}

}  // extern "C"
