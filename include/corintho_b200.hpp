/* corintho_b200.hpp -- the reference's C++ classes, header-only, on the C ABI of corintho_b200.h.
 *
 * `Trainer` has the public members of corintho_ai/cpp/include/trainer.h:17-53 and `Tourney` those
 * of corintho_ai/cpp/include/tourney.h:12-46, with the same argument order, types and meaning, so
 * that the reference's Cython bindings keep their `cdef cppclass` blocks unchanged and only name
 * another file:
 *
 *     cdef extern from "../cpp/src/trainer.cpp":   ->   cdef extern from "corintho_b200.hpp":
 *     (corintho_ai/python/main.pyx:17)
 *     cdef extern from "../cpp/src/tourney.cpp":   ->   cdef extern from "corintho_b200.hpp":
 *     (corintho_ai/rating/tourney.pyx:15)
 *
 * The reference reports failures by C++ exception through Cython's `except +`; so do these classes
 * (std::runtime_error carrying cb200_last_error(), a Python RuntimeError after `except +`). bindings/cython/ holds
 * a binding written that way; tests build it and drive the engine through it.
 * No state lives here besides the opaque handle: the work happens in libcorintho_b200.so. */
#ifndef CORINTHO_B200_HPP
#define CORINTHO_B200_HPP

#include <algorithm>
#include <map>
#include <stdexcept>
#include <string>

#include "corintho_b200.h"

namespace cb200_host {

inline int check(int rc) {
  if (rc >= 0) return rc;
  throw std::runtime_error(cb200_last_error());
}

/* trainer.h:17-53. */
class Trainer {
 public:
  Trainer(int num_games, const std::string &log_folder, int seed, int max_searches = 1600,
          int searches_per_eval = 16, float c_puct = 1.0f, float epsilon = 0.25f, int num_logged = 10,
          int num_threads = 1, bool testing = false)
      : h_{cb200_trainer_create(num_games, log_folder.c_str(), seed, max_searches, searches_per_eval,
                                c_puct, epsilon, num_logged, num_threads, testing ? 1 : 0)} {
    if (!h_) throw std::runtime_error(cb200_last_error());
  }
  ~Trainer() { cb200_trainer_destroy(h_); }
  Trainer(const Trainer &) = delete;
  Trainer &operator=(const Trainer &) = delete;

  int num_requests(int to_play = -1) { return check(cb200_trainer_num_requests(h_, to_play)); }
  int num_samples() { return check(cb200_trainer_num_samples(h_)); }
  float score() { return cb200_trainer_score(h_); }
  float avg_mate_length() { return cb200_trainer_avg_mate_length(h_); }
  void writeRequests(float *game_states, int to_play = -1) {
    check(cb200_trainer_write_requests(h_, game_states, to_play));
  }
  void writeSamples(float *game_states, float *eval_samples, float *prob_samples) {
    check(cb200_trainer_write_samples(h_, game_states, eval_samples, prob_samples));
  }
  void writeScores(const std::string &file) { check(cb200_trainer_write_scores(h_, file.c_str())); }
  bool doIteration(float *evaluations, float *probabilities, int to_play = -1) {
    return check(cb200_trainer_do_iteration(h_, evaluations, probabilities, to_play)) == 1;
  }

  /* Beyond the reference: the fused path (network on the device, no host round trip per
   * iteration); INTEGRATION.md section 3. */
  void setWeights(int model, const float *weights, size_t n_floats, int precision) {
    check(cb200_trainer_set_weights(h_, model, weights, n_floats, precision));
  }
  bool runSelfplay(int max_iterations = 0, int stagger = 0) {
    return check(cb200_trainer_run_selfplay(h_, max_iterations, stagger)) == 1;
  }
  cb200_trainer *handle() { return h_; }

 private:
  cb200_trainer *h_;
};

/* tourney.h:12-46. The reference's doIteration takes no buffer length, and its answer offsets
 * (tourney.cpp:54-62) advance by the pending requests of the PREVIOUS match whatever model that
 * match waits for, so a call can read rows past the requests of its own model: up to the summed
 * searches_per_eval of every seat of every match. max_rows() is that bound -- size eval / probs
 * with it (rating/tourney.pyx:95-110 sizes them per model, which the reference itself can
 * overrun); doIteration hands it to the engine, which reads exactly the rows the offsets name. */
class Tourney {
 public:
  Tourney(int num_threads, const std::string &log_folder)
      : h_{cb200_tourney_create(num_threads, log_folder.c_str())} {
    if (!h_) throw std::runtime_error(cb200_last_error());
  }
  ~Tourney() { cb200_tourney_destroy(h_); }
  Tourney(const Tourney &) = delete;
  Tourney &operator=(const Tourney &) = delete;

  bool all_done() { return check(cb200_tourney_all_done(h_)) == 1; }
  int num_requests(int id) { return check(cb200_tourney_num_requests(h_, id)); }
  void writeScores(const std::string &filename) { check(cb200_tourney_write_scores(h_, filename.c_str())); }
  void writeRequests(float *game_states, int id) { check(cb200_tourney_write_requests(h_, game_states, id)); }
  void doIteration(float *eval, float *probs, int id) {
    check(cb200_tourney_do_iteration(h_, eval, probs, max_rows(), id));
  }
  void addPlayer(int player_id, int model_id, int max_searches = 1600, int searches_per_eval = 16,
                 float c_puct = 1.0f, float epsilon = 0.25f, bool random = false) {
    check(cb200_tourney_add_player(h_, player_id, model_id, max_searches, searches_per_eval, c_puct, epsilon,
                                   random ? 1 : 0));
    spe_[player_id] = searches_per_eval;
  }
  void addMatch(int player1, int player2, bool logging = false) {
    check(cb200_tourney_add_match(h_, player1, player2, logging ? 1 : 0));
    rows_ += spe_.at(player1) + spe_.at(player2);
  }
  /* rows the caller's eval / probs buffers must hold (see above) */
  int max_rows() const { return std::max(rows_, 1); }

  /* Beyond the reference: networks resident on the device, whole rounds per call (INTEGRATION.md 6). */
  void setWeights(int model_id, const float *weights, size_t n_floats, int precision) {
    check(cb200_tourney_set_weights(h_, model_id, weights, n_floats, precision));
  }
  bool run(int max_rounds = 0) { return check(cb200_tourney_run(h_, max_rounds)) == 1; }
  cb200_tourney *handle() { return h_; }

 private:
  cb200_tourney *h_;
  std::map<int, int> spe_;
  int rows_ = 0;
};

/* Beyond the reference: the batched DockerMC (dockermc.cpp) -- a searched move choice and the root
 * statistics for every given position (cb200_analysis_run in corintho_b200.h; INTEGRATION.md 7). */
class Analysis {
 public:
  Analysis(int max_positions, int max_searches = 1600, int searches_per_eval = 16, float c_puct = 1.0f,
           float epsilon = 0.25f)
      : h_{cb200_analysis_create(max_positions, max_searches, searches_per_eval, c_puct, epsilon)} {
    if (!h_) throw std::runtime_error(cb200_last_error());
  }
  ~Analysis() { cb200_analysis_destroy(h_); }
  Analysis(const Analysis &) = delete;
  Analysis &operator=(const Analysis &) = delete;

  void setWeights(const float *weights, size_t n_floats, int precision) {
    check(cb200_analysis_set_weights(h_, weights, n_floats, precision));
  }
  void run(int n, const uint64_t *states, int seed, int32_t *moves, int32_t *results, float *values,
           int32_t *visits, float *evals = nullptr) {
    check(cb200_analysis_run(h_, n, states, seed, moves, results, values, visits, evals));
  }
  /* run() on device buffers in one persistent kernel, enqueued on the library's current stream
   * without waiting (cb200_analysis_run_device: per-position error results, graph capture). */
  void runDevice(int n, const void *states_device, int seed, void *moves_device, void *results_device,
                 void *values_device, void *visits_device, void *evals_device = nullptr,
                 void *status_device = nullptr) {
    check(cb200_analysis_run_device(h_, n, states_device, seed, moves_device, results_device, values_device,
                                    visits_device, evals_device, status_device));
  }

  /* External-evaluator protocol (cb200_analysis_begin .. _results): the caller's network answers
   * the requests between rounds, as docker/choose_move.pyx does for DockerMC. */
  void begin(int n, const uint64_t *states, int seed) { check(cb200_analysis_begin(h_, n, states, seed)); }
  int num_requests() { return check(cb200_analysis_num_requests(h_)); }
  void writeRequests(float *game_states) { check(cb200_analysis_write_requests(h_, game_states)); }
  bool doIteration(const float *eval, const float *probs, int rows) {
    return check(cb200_analysis_do_iteration(h_, eval, probs, rows)) == 1;
  }
  void results(int32_t *moves, int32_t *results, float *values, int32_t *visits, float *evals = nullptr) {
    check(cb200_analysis_results(h_, moves, results, values, visits, evals));
  }
  /* device buffers, on the library's current stream (see corintho_b200.h) */
  void writeRequestsDevice(void *rows_device) { check(cb200_analysis_write_requests_device(h_, rows_device)); }
  bool doIterationDevice(const void *eval_device, const void *probs_device, int rows) {
    return check(cb200_analysis_do_iteration_device(h_, eval_device, probs_device, rows)) == 1;
  }
  cb200_analysis *handle() { return h_; }

 private:
  cb200_analysis *h_;
};

}  // namespace cb200_host

#ifndef CB200_HPP_NO_GLOBAL_NAMES
using cb200_host::Analysis;
using cb200_host::Tourney;
using cb200_host::Trainer;
#endif

#endif
