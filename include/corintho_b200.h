/* corintho_b200 -- C ABI of the B200-native Corintho self-play engine (libcorintho_b200.so).
 *
 * Drop-in boundary for ONE path of maxjiang216/corintho-ai: self-play position / move-
 * probability generation behind the reference's `Trainer` class
 * (corintho_ai/cpp/include/trainer.h:17-53), which the reference binds from Cython with
 * `cdef extern from "../cpp/src/trainer.cpp"` (corintho_ai/python/main.pyx:17-38).
 * Every cb200_trainer_* entry point below names the Trainer member it replaces; argument
 * meaning, buffer layout and call protocol are the reference's (SURVEY.md 8b). The reference
 * throws C++ exceptions across Cython (`except +`); this ABI returns codes instead and keeps
 * the message in cb200_last_error(). INTEGRATION.md shows the Cython stub a maintainer adds.
 *
 * All pointers are plain host pointers unless a name says `_device`. No CPU fallback exists:
 * every entry point fails with CB200_ERR_CUDA when no sm_100-class device can be used.
 *
 * Packed game state ("cstate", 16 bytes):
 *   w0: four 16-bit planes; plane t (0 base, 1 column, 2 capital, 3 frozen) holds square
 *       s = row*4+col at bit 16*t+s   (reference Game::board_ bit row*16+col*4+t, game.h:124-126)
 *   w1: byte i<6 = pieces_[i] (P0{B,C,A}, P1{B,C,A}, game.h:127-131), byte 6 = to_play_, byte 7 = 0
 */
#ifndef CORINTHO_B200_H
#define CORINTHO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CB200_NUM_MOVES 96       /* util.h:43 kNumMoves */
#define CB200_STATE_SIZE 70      /* util.h:41 kGameStateSize */
#define CB200_NUM_SYMMETRIES 8   /* util.h:47 kNumSymmetries */

enum {
  CB200_OK = 0,
  CB200_ERR_ARG = -1,      /* invalid argument (the reference only assert()s, trainer.cpp:25-34) */
  CB200_ERR_CUDA = -2,     /* CUDA failure or no usable device */
  CB200_ERR_OVERFLOW = -3, /* a per-game node arena, path or sample buffer overflowed */
  CB200_ERR_STATE = -4     /* call out of protocol (e.g. fused run without weights) */
};

/* Message of the last error on the calling thread ("" if none). */
const char *cb200_last_error(void);
/* Number of visible CUDA devices (<=0: none usable). */
int cb200_device_count(void);
/* Bind the calling thread / subsequently created objects to a device (default 0). */
int cb200_set_device(int device);
/* Launch on this cudaStream_t from now on (NULL = the legacy default stream). */
int cb200_set_stream(void *cuda_stream);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t cb200_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Game logic (BASELINE.json configs[1]); replaces, per state:
 *   Game::getLegalMoves  (cpp/src/game.cpp:28-43)   -> mask words 0..2
 *   Node::initializeEdges terminal test (cpp/src/node.cpp:256-271) -> flags
 *   Game::doMove         (cpp/src/game.cpp:60-96)   -> next
 *   Game::writeGameState (cpp/src/game.cpp:45-58)   -> enc (optional)
 * For state i the move applied is the (rnd_i % n_legal)-th legal move in ascending id order,
 * rnd_i = high 32 bits of splitmix64(seed, i) (rules.cuh step_rnd); `next` = state if terminal.
 *   mask_flags[i] = {mask[0], mask[1], mask[2],
 *                    result | lines<<2 | n_legal<<8 | chosen_move<<16}   (chosen 0x7f if none)
 *   result: 0 none, 1 mover lost (no move, line present), 2 draw (util.h:58-60)
 */
int cb200_game_step(int64_t n, const uint64_t *states /* [n][2] */, uint64_t seed,
                    uint32_t *mask_flags /* [n][4] */, uint64_t *next /* [n][2] */,
                    float *enc /* [n][70] or NULL */);
/* Same on device-resident buffers, asynchronous on the current stream. */
int cb200_game_step_device(int64_t n, const void *states_device, uint64_t seed,
                           void *mask_flags_device, void *next_device, void *enc_device);

/* ------------------------------------------------------------------------------------------
 * Trainer (cpp/include/trainer.h:17-53).
 */
typedef struct cb200_trainer cb200_trainer;

/* Trainer::Trainer(num_games, log_folder, seed, max_searches, searches_per_eval, c_puct,
 *                  epsilon, num_logged, num_threads, testing)        trainer.cpp:18-37
 * Game i is seeded with the i-th output of mt19937(seed) and has parity i%2 (trainer.cpp:238-256).
 * num_threads is accepted for signature compatibility (the GPU engine has no host threads).
 * The first num_logged games write log_folder/game_<i>.txt like the reference
 * (selfplayer.cpp:124-204; a folder that does not exist silently yields no log).
 * Returns NULL on error. */
cb200_trainer *cb200_trainer_create(int num_games, const char *log_folder, int seed,
                                    int max_searches, int searches_per_eval, float c_puct,
                                    float epsilon, int num_logged, int num_threads, int testing);
/* Multi-GPU sharding: the trainer owns global games [first_game, first_game+num_games) of a
 * run of total_games games (seeds = outputs first_game.. of the same mt19937(seed) stream,
 * parity = global index & 1), so the union over ranks equals a single-GPU run. */
cb200_trainer *cb200_trainer_create_shard(int total_games, int first_game, int num_games,
                                          const char *log_folder, int seed, int max_searches,
                                          int searches_per_eval, float c_puct, float epsilon,
                                          int num_logged, int testing);
void cb200_trainer_destroy(cb200_trainer *t);

/* bool Trainer::doIteration(float eval[], float probs[], int to_play)   trainer.cpp:164-236
 * eval[n], probs[n][96]: answers to the previous write_requests, same order. First call ignores
 * them. to_play = -1 training; 0/1 two-model testing mode. Returns 1 when every game is done,
 * 0 otherwise, <0 on error. */
int cb200_trainer_do_iteration(cb200_trainer *t, const float *eval, const float *probs,
                               int to_play);
/* int Trainer::num_requests(int to_play)                                trainer.cpp:39-49 */
int cb200_trainer_num_requests(cb200_trainer *t, int to_play);
/* void Trainer::writeRequests(float *game_states, int to_play)          trainer.cpp:79-101
 * game_states[num_requests][70], game-index-major, request-order-minor. */
int cb200_trainer_write_requests(cb200_trainer *t, float *game_states, int to_play);
/* int Trainer::num_samples()                                            trainer.cpp:51-57 */
int cb200_trainer_num_samples(cb200_trainer *t);
/* void Trainer::writeSamples(game_states, eval_samples, prob_samples)   trainer.cpp:103-113
 * [num_samples*8][70], [num_samples*8], [num_samples*8][96] incl. the 8 symmetries
 * (selfplayer.cpp:79-113). */
int cb200_trainer_write_samples(cb200_trainer *t, float *game_states, float *eval_samples,
                                float *prob_samples);
/* float Trainer::score()                                                trainer.cpp:59-68 */
float cb200_trainer_score(cb200_trainer *t);
/* float Trainer::avg_mate_length()                                      trainer.cpp:70-77 */
float cb200_trainer_avg_mate_length(cb200_trainer *t);
/* void Trainer::writeScores(const std::string &file)                    trainer.cpp:115-162 */
int cb200_trainer_write_scores(cb200_trainer *t, const char *file);

/* ---- engine-only additions (no reference counterpart) ---------------------------------- */

/* Exact counters of the metric (SURVEY.md 8d): out = {simulations, moves, leaf_evals,
 * iterations}. simulations = sum over moves of the mover's searches_done_ when it moved. */
int cb200_trainer_counters(cb200_trainer *t, int64_t out[4]);

/* Un-augmented samples (one row per move, identity symmetry only) and per-game results, for
 * the NCCL gather: states[num_samples][2] cstate words, probs[num_samples][96],
 * labels[num_samples], game_of[num_samples] (local game index). Any pointer may be NULL. */
int cb200_trainer_write_raw_samples(cb200_trainer *t, uint64_t *states, float *probs,
                                    float *labels, int32_t *game_of);
/* Same rows on the device for the NCCL gather: *rows_device -> float [n_rows][102] =
 * {cstate as 4 bit-cast words, probs[96], label, global game index bit-cast}; the buffer is owned
 * by the trainer and valid until the next call. */
int cb200_trainer_raw_samples_device(cb200_trainer *t, void **rows_device, int *n_rows);
/* Streaming sample output for fused runs. Once enabled, cb200_trainer_run_selfplay expands the
 * samples of every FINISHED game (all 8 symmetries: exactly the rows Trainer::writeSamples
 * produces for that game, selfplayer.cpp:79-113) on the device and copies them to pinned host
 * memory owned by the trainer while the remaining games keep playing, so that the device->host
 * transfer overlaps the run instead of following it. Rows arrive in game COMPLETION order:
 * game_of[i] is the global game index of sample i, whose rows are 8*i .. 8*i+7 (a stable sort by
 * game_of restores writeSamples' order; a trainer that shuffles its samples need not bother).
 * max_samples: capacity in un-augmented samples (< 0: num_games * 32; 0: switch streaming off).
 * cb200_trainer_streamed_samples waits for the outstanding copies and returns host pointers that
 * stay valid until the next reset / run; CB200_ERR_OVERFLOW if the capacity was too small (the
 * run itself is unaffected and cb200_trainer_write_samples still works). */
int cb200_trainer_stream_samples(cb200_trainer *t, int64_t max_samples);
int cb200_trainer_streamed_samples(cb200_trainer *t, const float **game_states /* [n*8][70] */,
                                   const float **eval_samples /* [n*8] */,
                                   const float **prob_samples /* [n*8][96] */,
                                   const int32_t **game_of /* [n] */, int *n_samples);
/* Multi-GPU (one trainer per GPU, contiguous game shards: cb200_trainer_create_shard): the one
 * collective of the path -- an all-gather of the finished un-augmented samples over NCCL, straight
 * from and to device memory. `nccl_comm` is an ncclComm_t of the caller's (any NCCL 2.x loaded in
 * the process; the library resolves the NCCL entry points at run time and links nothing), or one
 * made by cb200_nccl_comm_create from an ncclUniqueId (128 bytes) that rank 0 obtained with
 * cb200_nccl_unique_id and distributed by any means. On return *rows_device -> float
 * [*n_rows][102] rows of ALL ranks in rank (= global game) order, layout as in
 * cb200_trainer_raw_samples_device, owned by the trainer and valid until its next call;
 * rows_per_rank[world] (may be NULL) receives the per-rank counts. Collective: every rank of
 * the communicator must call it. */
int cb200_nccl_unique_id(void *id_out /* 128 bytes */);
void *cb200_nccl_comm_create(int rank, int world, const void *unique_id /* 128 bytes */);
void cb200_nccl_comm_destroy(void *nccl_comm);
int cb200_trainer_allgather_samples(cb200_trainer *t, void *nccl_comm, void **rows_device, int *n_rows,
                                    int32_t *rows_per_rank);
/* per game: result (util.h:58-61: 1 first player lost, 2 draw, 3 first player won) */
int cb200_trainer_game_results(cb200_trainer *t, int32_t *results /* [num_games] */);

/* Network weights for the fused (device-resident) evaluator; model 0 is the only model in
 * training mode, models 0/1 are "new"/"best" in testing mode (main.pyx:74-81).
 * Architecture corintho_ai/python/wrapper.py:256-271 with BatchNorm already folded:
 *   weights = W1[70][100], b1[100], (W_l[100][100], b_l[100]) l=2..12, Wh[100][97], bh[97]
 * row-major [in][out] like Keras Dense kernels; head column 0 = value (tanh), 1..96 = policy
 * logits (softmax). n_floats must be 127997. precision: 0 = fp32 SIMT kernel (parity mode,
 * 1e-5), 1 = bf16 tcgen05 tensor-core kernel with fp32 accumulation (2e-2 on random-init
 * networks), 2 = the same kernel with fp16 operands (activations must stay below 65504),
 * 3 = "bf16x3": the same kernel with every operand carried as a bf16 hi + lo pair and three MMAs
 * per k-step (16 significant bits; < 1e-3 on the reference's trained checkpoints, whose folded
 * BatchNorm scales make single bf16 / fp16 operands miss the 2e-2 bar; ~2x the network time). */
int cb200_trainer_set_weights(cb200_trainer *t, int model, const float *weights, size_t n_floats,
                              int precision);
/* Evaluate positions with the resident network (the engine's replacement for the Keras
 * predict call main.pyx:70-83): game_states[n][70] -> eval[n], probs[n][96]. */
int cb200_trainer_evaluate(cb200_trainer *t, int model, int n, const float *game_states,
                           float *eval, float *probs);
/* Fused self-play: runs Trainer::doIteration + writeRequests + network evaluation entirely on
 * the device until every game is done or max_iterations (<=0: unlimited) iterations ran.
 * stagger != 0 reproduces the reference's staggered game start (trainer.cpp:184-186).
 * Returns 1 when all games are done, 0 if stopped by max_iterations, <0 on error. */
int cb200_trainer_run_selfplay(cb200_trainer *t, int max_iterations, int stagger);

/* Re-initialise every game for a new run with `seed` (same shape, allocations reused). */
int cb200_trainer_reset(cb200_trainer *t, int seed);
/* Per-kernel-class device timing with CUDA events on the launch stream (bench.py roofline):
 * classes 0 request scan, 1 request pack, 2 network, 3 game step (tree), 4 persistent fused
 * tail with 8 games per CTA (network + game step in one kernel), 5 the same with 16 games per
 * CTA; 6-7 unused. */
int cb200_trainer_set_profiling(cb200_trainer *t, int enable);
/* Work attribution of fused training-mode runs made while profiling was enabled: out =
 * {simulations done by lock-step game-step launches, simulations in total, leaf evaluations
 * ingested by lock-step launches, leaf evaluations in total}; the remainder belongs to the
 * persistent kernels (classes 4 and 5). Reset by cb200_trainer_set_profiling. */
int cb200_trainer_phase_split(cb200_trainer *t, int64_t out[4]);
/* Host-clock duration (ms) of the two phases of the fused training runs made since the last
 * cb200_trainer_set_profiling call: out = {lock-step phase (stream groups), persistent kernels}.
 * The phases are separated by host synchronisation points; measured with or without profiling. */
int cb200_trainer_phase_times(cb200_trainer *t, double out_ms[2]);
int cb200_trainer_kernel_times(cb200_trainer *t, double out_ms[8], int64_t out_launches[8]);

/* Debug: per-warp phase cycle maxima/sums of the game-step kernel since the last call:
 * out = {max ingest, max search, max move, sum ingest, sum search, sum move, rolled-back
 * searches, words copied by re-rooting, sum select cycles, sum expand cycles, tree levels
 * visited, expansions}. enable != 0 switches the instrumentation on. */
int cb200_trainer_phase_profile(cb200_trainer *t, int enable, uint64_t out[16]);

/* White-box dump of one search tree for engine-vs-oracle debugging (same layout as
 * oracle/corintho_oracle.h orc_trainer_dump_tree). */
int cb200_trainer_dump_tree(cb200_trainer *t, int game, int player, int64_t out[8],
                            uint32_t *words, int cap);

/* ---- Tourney: matches between players with their own search budgets (rating runs) ----------
 * Replaces class Tourney (corintho_ai/cpp/include/tourney.h:12-46, bound by Cython in
 * corintho_ai/rating/tourney.pyx:13-25) with class Match behind it (cpp/include/match.h:33-101):
 * per-player max_searches / searches_per_eval / c_puct / epsilon, random players (no search, one
 * uniform draw per move), requests batched per MODEL id. External-evaluator protocol exactly as
 * rating/tourney.pyx:112-173 drives it: for every model id (negative ids = random players) ->
 * num_requests, write_requests, evaluate, do_iteration; until all_done. The answer offsets follow
 * tourney.cpp:54-62 literally. All players and matches must be added before the first call that
 * needs the device (add_* return CB200_ERR_STATE afterwards). Matches added with logging != 0
 * write log_folder/match_<p1>_<p2>_<index>.txt like the reference (match.cpp:79-180).
 * `rows` = number of rows the caller's eval / probs buffers hold. */
typedef struct cb200_tourney cb200_tourney;
cb200_tourney *cb200_tourney_create(int num_threads, const char *log_folder);
void cb200_tourney_destroy(cb200_tourney *t);
int cb200_tourney_add_player(cb200_tourney *t, int player_id, int model_id, int max_searches,
                             int searches_per_eval, float c_puct, float epsilon, int random);
int cb200_tourney_add_match(cb200_tourney *t, int player1, int player2, int logging);
int cb200_tourney_all_done(cb200_tourney *t);                 /* 1 / 0, negative = error */
int cb200_tourney_num_requests(cb200_tourney *t, int model_id);
int cb200_tourney_write_requests(cb200_tourney *t, float *game_states, int model_id);
int cb200_tourney_do_iteration(cb200_tourney *t, const float *eval, const float *probs, int rows,
                               int model_id);
int cb200_tourney_write_scores(cb200_tourney *t, const char *file);
/* Fused tourney: the loop of rating/tourney.pyx:112-173 entirely on the device. Every model id
 * >= 0 that a player uses gets a device-resident network (same weight layout and precision codes
 * as cb200_trainer_set_weights); cb200_tourney_run then plays rounds -- for every model id in
 * first-seen order: request offsets, request packing, that model's network, Match::doIteration
 * with the reference's answer-offset rule (tourney.cpp:54-62) -- until every match is over or
 * max_rounds (<= 0: unlimited) rounds were played. Returns 1 when all matches are done, 0 when
 * stopped by max_rounds, < 0 on error. Note: a model whose tensor-core answers are read with
 * row-major evaluators cannot share answer rows across models within one round; like the
 * reference loop, the answer buffers persist between calls. */
int cb200_tourney_set_weights(cb200_tourney *t, int model_id, const float *weights, size_t n_floats,
                              int precision);
int cb200_tourney_run(cb200_tourney *t, int max_rounds);
/* out = {simulations, moves, leaf evaluations, do_iteration calls} over all matches */
int cb200_tourney_counters(cb200_tourney *t, int64_t out[4]);

/* ---- Analysis: the engine's move and search statistics for given positions ------------------
 * The batched form of the reference's DockerMC (corintho_ai/cpp/src/dockermc.cpp, served by
 * docker/choose_move.pyx): every position is searched by one testing-mode TrainMC with the
 * resident network, which then chooses its move exactly as TrainMC::chooseMove does in testing
 * mode (trainmc.cpp:110-137, 438-473; no opening randomisation). Parameters max_searches,
 * searches_per_eval, c_puct, epsilon: meaning and validation as in cb200_tourney_add_player
 * (searches_per_eval <= 64). The object holds device storage for max_positions positions, sized
 * once and reused by every run. */
typedef struct cb200_analysis cb200_analysis;
cb200_analysis *cb200_analysis_create(int max_positions, int max_searches, int searches_per_eval,
                                      float c_puct, float epsilon);  /* NULL on error */
void cb200_analysis_destroy(cb200_analysis *a);
/* Same weight layout and precision codes as cb200_trainer_set_weights. */
int cb200_analysis_set_weights(cb200_analysis *a, const float *weights, size_t n_floats, int precision);
/* Search every position of states[n][2] (cstates, layout at the top of this file).
 *   Random stream: position i's mt19937 is seeded with the i-th output of mt19937(seed), the rule of
 *     the Trainer's game seeds (trainer.cpp:238-256), so a position's outputs depend only on its
 *     index, the seed, the parameters and the network -- not on n or the rest of the batch.
 *   Side to move: byte 6 of the cstate; that side's tree is searched. Depth is not an input (in
 *     testing mode only the logs read it).
 *   Outputs, read from the root before the move is applied:
 *     moves[i]     the move id chosen (-1 for a position without a legal move);
 *     results[i]   the root's result code, from the view of the side to move:
 *                  0 unknown, 1 lost (no legal move, a line on the board), 2 drawn (no legal move,
 *                  no line), 4 proven lost, 5 proven drawn, 6 proven won (util.h:58-61 kResult*,
 *                  kDeduced*); 3 never occurs;
 *     values[i]    the root's evaluation_: the running sum the search keeps over the root's
 *                  visits, from the view of the side to move (higher is better for it);
 *     visits[i][m] the visits_ of the child reached by move id m (0 for an illegal or unexpanded
 *                  move);
 *     evals[i][m]  that child's evaluation_, from the view of the side to move in the child (the
 *                  opponent): -evals / visits is the move's mean value for the side to move, the
 *                  exploitation term of PUCT selection (trainmc.cpp:540-600). May be NULL.
 *   A position without a legal move is not searched: move -1, result 1 or 2, visits and value 0.
 * Errors: CB200_ERR_ARG for n <= 0, n > max_positions, a null required pointer or a state that
 * cb200_check_states rejects; CB200_ERR_STATE without weights; CB200_ERR_OVERFLOW when a search
 * overflowed its node arena; CB200_ERR_CUDA without a usable device. The object stays usable after
 * an error. */
int cb200_analysis_run(cb200_analysis *a, int n, const uint64_t *states, int seed,
                       int32_t *moves /* [n] */, int32_t *results /* [n] */, float *values /* [n] */,
                       int32_t *visits /* [n][96] */, float *evals /* [n][96] or NULL */);
/* External-evaluator protocol: the same searches with the caller's network instead of the resident
 * one (no weights needed), driven like docker/choose_move.pyx drives DockerMC and like the Trainer's
 * doIteration / writeRequests:
 *     begin; while (!do_iteration(eval, probs, rows)) { n = num_requests; write_requests(rows[n][70]);
 *                                                       evaluate rows -> eval[n], probs[n][96]; }
 *     results
 * The first do_iteration takes no answers (num_requests is 0 after begin) and queues the roots.
 * Given the same answers, every output equals what cb200_analysis_run computes with a network that
 * gives those answers.
 *   begin         opens a session on states[n][2]: validation, seeds and errors of cb200_analysis_run
 *                 (except that no weights are needed). A begin during an open session restarts it;
 *                 a begin that fails leaves no session open.
 *   num_requests  rows the next do_iteration reads (no device work).
 *   write_requests  game_states[num_requests][70], position-major, then in the order the position
 *                 queued its leaves (Trainer::writeRequests' order).
 *   do_iteration  one round with row-major answers to the last write_requests: eval[rows],
 *                 probs[rows][96] (probabilities need not be normalised: the search renormalises over
 *                 the legal moves). rows = what the buffers hold; fewer than num_requests is
 *                 CB200_ERR_ARG. Returns 1 when every position is done (and does no work once it is),
 *                 0 if not, < 0 on error.
 *   results       the outputs of cb200_analysis_run (evals may be NULL); CB200_ERR_STATE before
 *                 do_iteration has returned 1. May be called again until the next begin / run.
 * Calls other than begin without an open session are CB200_ERR_STATE; cb200_analysis_run discards
 * an open session. Null and negative-size arguments are CB200_ERR_ARG before anything else is looked
 * at; argument errors leave the session as it was. An error while a round runs -- CB200_ERR_OVERFLOW
 * when a node arena overflowed, CB200_ERR_CUDA -- ends the session. Either way the object stays
 * usable for a new begin or run. */
int cb200_analysis_begin(cb200_analysis *a, int n, const uint64_t *states /* [n][2] */, int seed);
int cb200_analysis_num_requests(cb200_analysis *a);
int cb200_analysis_write_requests(cb200_analysis *a, float *game_states /* [num_requests][70] */);
int cb200_analysis_do_iteration(cb200_analysis *a, const float *eval /* [rows] */,
                                const float *probs /* [rows][96] */, int rows);
int cb200_analysis_results(cb200_analysis *a, int32_t *moves /* [n] */, int32_t *results /* [n] */,
                           float *values /* [n] */, int32_t *visits /* [n][96] */,
                           float *evals /* [n][96] or NULL */);
/* Device forms, for an evaluator that lives on the GPU: the same calls on device memory, ordered on
 * the library's current stream (cb200_set_stream) and never staged through the host.
 *   write_requests_device  packs the rows (float [num_requests][70]) into rows_device and returns
 *                 without waiting: the rows are complete in the order of the current stream, so work
 *                 queued on that stream may read them directly; another stream must wait for it first
 *                 (an event recorded on the current stream after the call, or a synchronisation).
 *   do_iteration_device  the kernel reads eval_device[rows] and probs_device[rows][96] (float,
 *                 row-major) in place. The caller's writes to them must be complete in the order of
 *                 the current stream when the call is made: issued on that stream, or on a stream the
 *                 current stream has been made to wait for. The call returns after the round
 *                 (it reads back the summary), so the buffers may be reused as soon as it returns.
 * A buffer that is not device (or managed) memory of the device the analysis was created on is
 * CB200_ERR_ARG. */
int cb200_analysis_write_requests_device(cb200_analysis *a, void *rows_device);
int cb200_analysis_do_iteration_device(cb200_analysis *a, const void *eval_device, const void *probs_device,
                                       int rows);
/* cb200_analysis_run for positions and outputs in device memory, with the resident tensor-core
 * network, in one persistent kernel: stream-ordered, no host round trip.
 *   Outputs: for every valid position, bit for bit those of cb200_analysis_run on the same states,
 *     seed, parameters and weights (moves, results, values, visits, evals; same seed rule).
 *   Stream order: everything is enqueued on the library's current stream (cb200_set_stream) and the
 *     call returns without waiting for the device. It makes no synchronisation, host copy,
 *     allocation or read-back, so it may be captured in a CUDA graph -- except the first call after
 *     create / set_weights, which uploads the weights and allocates its buffers (make one warm-up
 *     call before capturing). The outputs are complete in the order of that stream. states_device is
 *     read while the kernel runs: do not change it before then. Two calls on different streams must
 *     be ordered by the caller. The host-synchronous calls on the object (run, begin, results,
 *     counters, set_weights, destroy) first wait for the last uncaptured call; replays of a captured
 *     one are ordered by the caller like any other work on their stream.
 *   Per-position errors (the call cannot return them): a state cb200_check_states rejects gets
 *     results[i] = CB200_ERR_ARG, moves[i] = -1 and zero value, visits and evals; a search that
 *     overflows its node arena gets results[i] = CB200_ERR_OVERFLOW, moves[i] = -1 and the same zeros.
 *     The other positions are searched as usual. status_device (may be NULL) receives
 *     {positions with an error result, most negative error result or 0}.
 *   Call errors, checked before anything is enqueued (the object stays usable): CB200_ERR_ARG for n
 *     outside [1, max_positions], a null required pointer, a buffer that is not device (or managed)
 *     memory of the analysis' device, or states_device not 16-byte aligned; CB200_ERR_STATE without
 *     weights or with fp32 weights (precision 0: use cb200_analysis_run); CB200_ERR_CUDA without a
 *     usable device. Like cb200_analysis_run, the call discards an open protocol session.
 *   cb200_analysis_counters afterwards returns this call's totals (equal to cb200_analysis_run's). */
int cb200_analysis_run_device(cb200_analysis *a, int n, const void *states_device /* u64 [n][2] */, int seed,
                              void *moves_device /* i32 [n] */, void *results_device /* i32 [n] */,
                              void *values_device /* f32 [n] */, void *visits_device /* i32 [n][96] */,
                              void *evals_device /* f32 [n][96] or NULL */,
                              void *status_device /* i32 [2] or NULL */);
/* out = {simulations, leaf evaluations} of the last run, device run or session; while a session is
 * open, its running totals so far (like the oracle's counters). */
int cb200_analysis_counters(cb200_analysis *a, int64_t out[2]);
/* Structural check of cstates given by a caller (no device needed): byte 6 (side to move) 0 or 1,
 * byte 7 zero, at most 4 pieces of a kind in either hand, frozen squares occupied, and for every
 * kind, pieces on the board = 8 - both hands' count. valid[i] (may be NULL) = 1 / 0. Returns the
 * number of rejected states, < 0 on bad arguments. */
int64_t cb200_check_states(int64_t n, const uint64_t *states /* [n][2] */, uint8_t *valid);

#ifdef __cplusplus
}
#endif
#endif /* CORINTHO_B200_H */
