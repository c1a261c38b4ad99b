// TEST INFRASTRUCTURE ONLY -- the analysis restatement (the batched DockerMC, dockermc.cpp) on top of
// the CPU oracle. It includes oracle/corintho_oracle.cpp as it stands, so the search it runs is the
// oracle's own Tree / tree_do_iteration / choose_move (pinned to the reference), and adds the
// analysis object and a white-box arena dump of the oracle Trainer. Built into a library of its own
// by tests/analysis_oracle.py (which also binds it); the oracle's entry points in that library are
// the oracle's. Compile with the oracle's flags (-ffp-contract=off).
#include "../oracle/corintho_oracle.cpp"

namespace {

// ---- Analysis: one testing-mode TrainMC per given position, stopped after its move choice ------
// (the batched form of the reference's DockerMC, dockermc.cpp). Position i is a GameRec whose
// generator is seeded with the i-th output of mt19937(seed) (trainer.cpp:238-256) and whose tree
// of the side to move starts as a single node at depth 0 holding the position.
struct AnalysisRec {
  Params p;
  std::vector<GameRec> games;
  std::vector<char> done;
  std::vector<int32_t> moves, results, visits;  // visits [n][96]
  std::vector<float> values, evals;             // evals [n][96]
};

// The structural invariants of a position the engine accepts from a caller (reference bit order):
// side to move 0 or 1, byte 7 zero, at most 4 pieces of a kind in a hand, frozen squares occupied,
// and every piece of a kind either on the board or in a hand (8 of each kind).
bool valid_state(const State &s) {
  const int to_play = (int)((s.w1 >> 48) & 0xff);
  if (to_play > 1 || (s.w1 >> 56) != 0) return false;
  uint32_t plane[4] = {0, 0, 0, 0};
  for (int sq = 0; sq < 16; ++sq)
    for (int t = 0; t < 4; ++t)
      if ((s.w0 >> (4 * sq + t)) & 1) plane[t] |= 1u << sq;
  if (plane[3] & ~(plane[0] | plane[1] | plane[2])) return false;
  for (int t = 0; t < 3; ++t) {
    const int h0 = (int)((s.w1 >> (8 * t)) & 0xff), h1 = (int)((s.w1 >> (8 * (3 + t))) & 0xff);
    if (h0 > 4 || h1 > 4 || __builtin_popcount(plane[t]) != 8 - h0 - h1) return false;
  }
  return true;
}

}  // namespace

// Analysis: position i (reference bit order) searched by one testing-mode TrainMC whose generator
// is seeded with the i-th output of mt19937(seed), stopped after its move choice. External-evaluator
// protocol: num_requests, write_requests, evaluate, do_iteration (answers packed contiguously) until
// do_iteration returns 1. create returns NULL for bad parameters or a state orc_state_valid rejects.
// A position without a legal move is not searched (move -1, its terminal result). results():
// moves[n], results[n] (root result code, util.h:58-61 / kDeduced*), values[n] (root evaluation_),
// visits[n][96] and evals[n][96] (child visits_ / evaluation_ per move id, 0 when not expanded).
// orc_trainer_dump_arena: raw words of one of a Trainer game's three arenas; out = {tree 0 arena,
// tree 1 arena, spare arena}. Re-rooting copies the kept subtree out of the mover's arena, so right
// after a move the spare arena still holds the mover's tree as it stood when the move was chosen.
extern "C" {

// ---- Analysis (the batched DockerMC, dockermc.cpp) ---------------------------------------------
int orc_state_valid(const uint64_t st[2]) { return valid_state(State{st[0], st[1]}) ? 1 : 0; }

void *orc_analysis_create(int n, const uint64_t *states, int seed, int max_searches,
                          int searches_per_eval, float c_puct, float epsilon) {
  if (n <= 0 || !states || max_searches <= 0 || searches_per_eval <= 0) return nullptr;
  for (int i = 0; i < n; ++i)
    if (!valid_state(State{states[2 * i], states[2 * i + 1]})) return nullptr;
  AnalysisRec *A = new AnalysisRec();
  A->p = Params{max_searches, searches_per_eval, c_puct, epsilon, true, 0};
  A->p.arena_words = (uint32_t)(((uint64_t)max_searches * 3 + 64) * (8 + 4 * 40));
  A->games.resize(n);
  A->done.assign(n, 0);
  A->moves.assign(n, -1);
  A->results.assign(n, kResultNone);
  A->values.assign(n, 0.0f);
  A->visits.assign((size_t)n * kNumMoves, 0);
  A->evals.assign((size_t)n * kNumMoves, 0.0f);
  MT gen;
  gen.seed((uint32_t)seed);
  for (int i = 0; i < n; ++i) {
    GameRec &g = A->games[i];
    g.rng.seed(gen.next());
    for (int a = 0; a < 3; ++a) g.arena[a].assign(A->p.arena_words, 0);
    g.tree[0].arena = 0;
    g.tree[1].arena = 1;
    g.spare = 2;
    const State root{states[2 * i], states[2 * i + 1]};
    g.to_play = (int)((root.w1 >> 48) & 0xff);
    Mask m;
    const bool lines = legal_moves(root, m);
    if (m.count() == 0) {  // nothing to search: report the terminal result
      A->results[i] = lines ? kResultLoss : kResultDraw;
      A->done[i] = 1;
      continue;
    }
    Tree &t = g.tree[g.to_play];
    fresh_tree(g, t, A->p, root, 0);
    t.searches_done = 0;  // the first doIteration queues the root for evaluation
  }
  return A;
}

void orc_analysis_destroy(void *h) { delete static_cast<AnalysisRec *>(h); }

int orc_analysis_num_requests(void *h) {
  AnalysisRec *A = static_cast<AnalysisRec *>(h);
  int n = 0;
  for (size_t i = 0; i < A->games.size(); ++i)
    if (!A->done[i]) n += game_num_requests(A->games[i]);
  return n;
}

void orc_analysis_write_requests(void *h, float *game_states) {
  AnalysisRec *A = static_cast<AnalysisRec *>(h);
  int64_t off = 0;
  for (size_t i = 0; i < A->games.size(); ++i) {
    if (A->done[i]) continue;
    GameRec &g = A->games[i];
    Tree &t = g.tree[g.to_play];
    for (size_t k = 0; k < g.pending.size(); ++k)
      encode_state(rec_state(rec(g, t, g.pending[k].leaf_off)), game_states + kStateSize * off++);
  }
}

// TrainMC::doIteration for every position not done yet (answers packed contiguously in the order
// of write_requests); a position whose search is complete reports its root and chooses its move.
// Returns 1 when every position is done, 0 otherwise, -1 on an arena / path overflow.
int orc_analysis_do_iteration(void *h, const float *eval, const float *probs) {
  AnalysisRec *A = static_cast<AnalysisRec *>(h);
  int64_t off = 0;
  for (size_t i = 0; i < A->games.size(); ++i) {
    if (A->done[i]) continue;
    GameRec &g = A->games[i];
    Tree &t = g.tree[g.to_play];
    const int64_t np = game_num_requests(g);
    const bool turn_done = tree_do_iteration(g, t, A->p, eval ? eval + off : nullptr,
                                             probs ? probs + kNumMoves * off : nullptr);
    off += np;
    if (g.error) return -1;
    if (!turn_done) continue;
    const uint32_t *r = rec(g, t, 0);
    for (int e = 0; e < rec_nlegal(r); ++e) {
      const uint32_t *s = r + 8 + 4 * e;
      if (!s3_has(s[3])) continue;
      A->visits[i * kNumMoves + s3_move(s[3])] = (int32_t)s[kSVis];
      A->evals[i * kNumMoves + s3_move(s[3])] = bits_f(s[kSEval]);
    }
    A->values[i] = t.root_eval;
    A->results[i] = t.root_result;
    g.sims += t.searches_done;
    g.moves += 1;
    A->moves[i] = choose_move(g, t, A->p, nullptr);
    if (g.error) return -1;
    A->done[i] = 1;
  }
  for (char d : A->done)
    if (!d) return 0;
  return 1;
}

void orc_analysis_results(void *h, int32_t *moves, int32_t *results, float *values, int32_t *visits,
                          float *evals) {
  AnalysisRec *A = static_cast<AnalysisRec *>(h);
  const size_t n = A->games.size();
  memcpy(moves, A->moves.data(), n * 4);
  memcpy(results, A->results.data(), n * 4);
  memcpy(values, A->values.data(), n * 4);
  memcpy(visits, A->visits.data(), n * kNumMoves * 4);
  memcpy(evals, A->evals.data(), n * kNumMoves * 4);
}

// {simulations, leaf evaluations} summed over the positions
void orc_analysis_counters(void *h, int64_t out[2]) {
  AnalysisRec *A = static_cast<AnalysisRec *>(h);
  out[0] = out[1] = 0;
  for (auto &g : A->games) out[0] += g.sims, out[1] += g.evals;
}

int orc_trainer_dump_arena(void *h, int game, int arena, uint32_t *words, int cap, int32_t out[3]) {
  Engine *E = static_cast<Engine *>(h);
  GameRec &g = E->games[game];
  out[0] = g.tree[0].arena, out[1] = g.tree[1].arena, out[2] = g.spare;
  const int n = (int)g.arena[arena].size() < cap ? (int)g.arena[arena].size() : cap;
  memcpy(words, g.arena[arena].data(), (size_t)n * 4);
  return n;
}

}  // extern "C"
