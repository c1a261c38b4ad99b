// libcorintho_b200.so -- host side of the B200 self-play engine and its C ABI
// (include/corintho_b200.h). Mirrors the reference Trainer (corintho_ai/cpp/src/trainer.cpp)
// call for call; all game state lives in HBM and every step of the path is a CUDA kernel.
// There is deliberately no CPU implementation of the path in this library.

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <fstream>
#include <iomanip>
#include <memory>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "game_step.cuh"
#include "mlp.cuh"
#include "mlp_tc.cuh"
#include "tree.cuh"
#include "persistent.cuh"
#include "match.cuh"
#include "analysis.cuh"
#include "gather.cuh"

using namespace cb200;

namespace cb200 {

__device__ uint8_t d_space_sym[8 * 16];
__device__ uint8_t d_move_sym[8 * 96];

// SelfPlayer::writeSamples (selfplayer.cpp:79-113): 8 symmetries per stored sample.
// One warp per (game, sample); soff[g] = index of game g's first sample row. Streaming form
// (emitted != nullptr): only the games stamped `stamp` by k_emit_assign take part, and game_of
// receives the global game index of every (un-augmented) sample.
__global__ void __launch_bounds__(256)
    k_write_samples(TreeParams P, const int32_t *__restrict__ soff, float *__restrict__ gs_out,
                    float *__restrict__ ev_out, float *__restrict__ pr_out,
                    const int32_t *__restrict__ emitted, int stamp, int32_t *__restrict__ game_of) {
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int g = w / kMaxSamples, i = w - g * kMaxSamples;
  if (g >= P.num_games) return;
  if (emitted != nullptr && emitted[g] != stamp) return;
  const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  const int ns = ctl[CW_N_SAMPLES];
  if (i >= ns) return;
  if (game_of != nullptr && lane == 0) game_of[soff[g] + i] = P.first_game + g;
  const ulonglong2 sv = P.sample_state[(size_t)g * kMaxSamples + i];
  const CState st{sv.x, sv.y};
  const float *pr = P.sample_probs + ((size_t)g * kMaxSamples + i) * CB200_NUM_MOVES;
  float ev = ctl[CW_RESULT] == kResultDraw ? 0.0f : 1.0f;
  if ((ns - 1 - i) & 1) ev = -ev;  // evaluation *= -1.0 per step back from the last move
  const size_t row = ((size_t)soff[g] + i) * 8;
  for (int k = 0; k < 8; ++k) {
    float *go = gs_out + (row + k) * CB200_STATE_SIZE;
    for (int j = lane; j < CB200_STATE_SIZE; j += 32) {
      const int src = j < 64 ? d_space_sym[k * 16 + (j >> 2)] * 4 + (j & 3) : j;
      go[j] = encode_elem(st, src);
    }
    if (lane == 0) ev_out[row + k] = ev;
    float *po = pr_out + (row + k) * CB200_NUM_MOVES;
    for (int j = lane; j < CB200_NUM_MOVES; j += 32) po[j] = pr[d_move_sym[k * 96 + j]];
  }
}

// Streaming sample output: finished games that have not been emitted yet get their block of
// sample rows (one atomicAdd per game: completion order, not game order) and the stamp of this
// emission round. ctr[0] = samples handed out so far, ctr[1] = 1 if a game did not fit.
__global__ void k_emit_assign(TreeParams P, int32_t *__restrict__ emitted, int32_t *__restrict__ ctr,
                              int cap_samples, int32_t *__restrict__ soff, int stamp) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.num_games) return;
  const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  if (!*(volatile const int32_t *)(ctl + CW_DONE) || emitted[g] != 0) return;
  __threadfence();  // pairs with the fence before the game's CW_DONE store
  const int ns = *(volatile const int32_t *)(ctl + CW_N_SAMPLES);
  const int base = atomicAdd(ctr, ns);
  if (base + ns > cap_samples) {
    atomicSub(ctr, ns);
    ctr[1] = 1;
    return;
  }
  soff[g] = base;
  emitted[g] = stamp;
}

// move-major network output [96][ld] -> row-major [rows][96] (cb200_trainer_evaluate)
__global__ void k_probs_row_major(const float *__restrict__ mm, int ld, int rows, float *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * CB200_NUM_MOVES) return;
  const int r = i / CB200_NUM_MOVES, m = i - r * CB200_NUM_MOVES;
  out[i] = mm[(size_t)m * ld + r];
}

// Un-augmented samples as 102-float rows for the NCCL gather: 4 words of cstate (bit-cast),
// 96 move probabilities, the value label, the global game index (bit-cast).
__global__ void __launch_bounds__(256)
    k_pack_raw_samples(TreeParams P, const int32_t *__restrict__ soff, float *__restrict__ rows) {
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int g = w / kMaxSamples, i = w - g * kMaxSamples;
  if (g >= P.num_games) return;
  const int32_t *ctl = P.ctl + (size_t)g * kCtlWords;
  const int ns = ctl[CW_N_SAMPLES];
  if (i >= ns) return;
  float *out = rows + ((size_t)soff[g] + i) * 102;
  const float *pr = P.sample_probs + ((size_t)g * kMaxSamples + i) * CB200_NUM_MOVES;
  for (int j = lane; j < CB200_NUM_MOVES; j += 32) out[4 + j] = pr[j];
  if (lane == 0) {
    const ulonglong2 sv = P.sample_state[(size_t)g * kMaxSamples + i];
    out[0] = __uint_as_float((uint32_t)sv.x), out[1] = __uint_as_float((uint32_t)(sv.x >> 32));
    out[2] = __uint_as_float((uint32_t)sv.y), out[3] = __uint_as_float((uint32_t)(sv.y >> 32));
    float ev = ctl[CW_RESULT] == kResultDraw ? 0.0f : 1.0f;
    if ((ns - 1 - i) & 1) ev = -ev;
    out[100] = ev;
    out[101] = __int_as_float(P.first_game + g);
  }
}

}  // namespace cb200

// ==============================================================================================
struct cb200_trainer {
  int device = 0;
  TreeParams P{};
  int iterations_done = 0;
  int stagger_div = 1;
  std::string log_folder;
  size_t cap = 0;  // num_games * spe request rows
  float *d_eval = nullptr, *d_probs = nullptr, *d_rows = nullptr;
  ulonglong2 *d_packed = nullptr;
  int32_t *d_offs = nullptr, *d_summary = nullptr, *d_soff = nullptr;
  float *d_samp = nullptr;  // cached output buffer of write_samples
  size_t samp_rows = 0;
  float *d_raw = nullptr;   // cached [rows][102] buffer of raw_samples_device
  size_t raw_rows = 0;
  float *d_gath = nullptr;  // all-gather: [world][max rows][102] padded blocks, then the result
  size_t gath_floats = 0;
  int32_t *d_gcounts = nullptr, *h_gcounts = nullptr;  // [world + 1] rows per rank (+ own count)
  int gcounts_world = 0;    // communicator size the count buffers were allocated for
  int32_t *h_summary = nullptr;  // pinned
  NetF32 net32[2];
  NetTC nettc[2];
  int precision[2] = {-1, -1};
  std::vector<int32_t> h_ctl;
  int seed = 0;
  // fused mode: games are split into independent stream groups (no lock-step across groups)
  int n_groups = 1;
  int32_t *d_live_list = nullptr;   // [num_games] live games per stream group (TreeParams::live_list)
  int32_t *d_live_count = nullptr;  // [n_groups]
  std::vector<cudaStream_t> g_stream;
  std::vector<int> g_begin, g_end;
  int32_t *d_gctr = nullptr;  // [n_groups][8] device counters (TreeParams::group_ctr)
  int32_t *h_gctr = nullptr;  // pinned mirror
  // per-game text logs of the first num_logged games (trainer.cpp:243-250)
  std::vector<std::unique_ptr<std::ofstream>> log_files;  // [P.n_logged]; null = could not open
  std::vector<int> log_written;                           // records already formatted
  std::vector<int32_t> h_log_count;
  std::vector<uint32_t> h_log_rec;
  // persistent fused tail (persistent.cuh): CTA-private request/answer rows and the live list
  int ps_ctas = 0;                 // CTAs the device holds (one per SM)
  int32_t *d_ps_list = nullptr;    // [num_games]
  int32_t *d_ps_out = nullptr;     // [8] live, error, rounds, finished | list length
  int32_t *h_ps_out = nullptr;     // pinned
  float *d_ps_eval[2] = {nullptr, nullptr};   // [ps_ld] answers, ping-pong between launches
  float *d_ps_probs[2] = {nullptr, nullptr};  // [96][ps_ld] move-major
  ulonglong2 *d_ps_packed = nullptr;          // [ps_ld] request rows (live within one round)
  int ps_ld = 0;                   // rows = ps_ctas * 16 games * 16 requests * 2 models
  int ps_n = 0;                    // games in the live list
  int ps_cur = 0;                  // buffer holding the answers of the queued requests
  bool ps_active = false;          // the games now live in the persistent loop's rows
  bool ps_from_lockstep = false;   // ... except that the next launch reads d_eval/d_probs first
  // streaming sample output (cb200_trainer_stream_samples): finished games' samples, all 8
  // symmetries, go to pinned host memory while the run continues
  bool stream_on = false;
  size_t st_cap = 0;               // allocated capacity in (un-augmented) samples
  size_t st_limit = 0;             // capacity requested by the caller (<= st_cap)
  float *d_st = nullptr;           // device staging [cap*8][70] | [cap*8] | [cap*8][96]
  float *h_st = nullptr;           // pinned host mirror, same layout
  int32_t *d_st_game = nullptr, *h_st_game = nullptr;  // [cap] global game index per sample
  int32_t *d_st_ctr = nullptr, *h_st_ctr = nullptr;    // [2] samples handed out, overflow flag
  int32_t *d_emitted = nullptr;    // [num_games] emission round of a game's samples (0 = not yet)
  int32_t *d_st_soff = nullptr;    // [num_games] first sample row of an emitted game
  cudaStream_t st_stream = nullptr;
  cudaEvent_t st_ev = nullptr;
  bool st_pending = false;         // st_ev marks a counter read-back that has not been consumed
  size_t st_copied = 0;            // samples whose device->host copy has been queued
  int st_round = 0;
  // per-kernel-class CUDA-event timing (bench.py roofline): 0 scan, 1 pack, 2 network, 3 iterate
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<int> ev_class;  // class of the pair starting at ev_pool[2*i]
  size_t ev_used = 0;
  // profiling: running search / leaf-evaluation counts attributed to the lock-step launches
  // (the rest of a run belongs to the persistent kernels); marks = values at the last snapshot
  long long searches_now = 0, searches_mark = 0, evals_mark = 0;
  long long lockstep_searches = 0, lockstep_evals = 0, total_searches = 0, total_evals = 0;
  // host-clock duration of the two phases of fused training runs (always on; the switch between
  // them is a host synchronisation point anyway); cleared by cb200_trainer_set_profiling
  double lockstep_wall_ms = 0, tail_wall_ms = 0;
  double class_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long class_launches[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

extern "C" int cb200_trainer_counters(cb200_trainer *t, int64_t out[4]);

namespace {

constexpr size_t kAnswerSlack = 128;  // spare rows behind the answer buffers

uint32_t mt_seed_word(uint32_t prev, int i) { return 1812433253u * (prev ^ (prev >> 30)) + i; }

struct HostMT {
  uint32_t mt[624];
  int idx = 624;
  void seed(uint32_t s) {
    mt[0] = s;
    for (int i = 1; i < 624; ++i) mt[i] = mt_seed_word(mt[i - 1], i);
    idx = 624;
  }
  uint32_t next() {
    if (idx >= 624) {
      for (int i = 0; i < 624; ++i) {
        uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
        mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1) ? 0x9908b0dfu : 0u);
      }
      idx = 0;
    }
    uint32_t y = mt[idx++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
  }
};

int upload_tables_once() {
  int rc = ensure_tables();
  if (rc != CB200_OK) return rc;
  static bool sym_ready[16] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && sym_ready[dev]) return CB200_OK;
  CB_CUDA(cudaMemcpyToSymbol(d_space_sym, kCSpaceSym, sizeof(kCSpaceSym)));
  CB_CUDA(cudaMemcpyToSymbol(d_move_sym, kCMoveSym, sizeof(kCMoveSym)));

  if (dev < 16) sym_ready[dev] = true;
  return CB200_OK;
}

template <class T>
int dmalloc(T **p, size_t count) {
  CB_CUDA(cudaMalloc((void **)p, count * sizeof(T)));
  return CB200_OK;
}

// ---- optional per-launch timing ---------------------------------------------------------------
int prof_drain(cb200_trainer *t) {  // caller has synchronised the stream
  for (size_t i = 0; i < t->ev_used; ++i) {
    float ms = 0.f;
    CB_CUDA(cudaEventElapsedTime(&ms, t->ev_pool[2 * i], t->ev_pool[2 * i + 1]));
    t->class_ms[t->ev_class[i]] += ms;
    t->class_launches[t->ev_class[i]] += 1;
  }
  t->ev_used = 0;
  return CB200_OK;
}
struct ProfScope {
  cb200_trainer *t;
  bool on;
  size_t idx = 0;
  cudaStream_t st;
  ProfScope(cb200_trainer *t_, int cls, cudaStream_t stream = cur_stream())
      : t(t_), on(t_->profiling), st(stream) {
    if (!on) return;
    if (2 * (t->ev_used + 1) > t->ev_pool.size()) {
      for (int k = 0; k < 2; ++k) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        t->ev_pool.push_back(e);
      }
      t->ev_class.push_back(cls);
    }
    idx = t->ev_used++;
    t->ev_class[idx] = cls;
    cudaEventRecord(t->ev_pool[2 * idx], st);
  }
  ~ProfScope() {
    if (on) cudaEventRecord(t->ev_pool[2 * idx + 1], st);
  }
};

// profiling only: attribute the searches / leaf evaluations since the last mark to the lock-step
// launches (to_lockstep) or to the persistent kernels
int prof_mark(cb200_trainer *t, bool to_lockstep) {
  int64_t c4[4];
  int rc = cb200_trainer_counters(t, c4);
  if (rc != CB200_OK) return rc;
  if (to_lockstep) {
    t->lockstep_searches += t->searches_now - t->searches_mark;
    t->lockstep_evals += c4[2] - t->evals_mark;
  }
  t->total_searches += t->searches_now - t->searches_mark;
  t->total_evals += c4[2] - t->evals_mark;
  t->searches_mark = t->searches_now, t->evals_mark = c4[2];
  return CB200_OK;
}

int scan(cb200_trainer *t, int to_play) {
  ProfScope ps(t, 0);
  k_scan_requests<<<1, 1024, 0, cur_stream()>>>(t->P, to_play, t->d_offs, t->d_summary);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  return CB200_OK;
}

int fetch_summary(cb200_trainer *t) {
  CB_CUDA(cudaMemcpyAsync(t->h_summary, t->d_summary, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost,
                          cur_stream()));
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  if (t->profiling) {
    int rc = prof_drain(t);
    if (rc != CB200_OK) return rc;
  }
  if (t->h_summary[2] != 0)
    return set_error(t->h_summary[2],
                     "a game overflowed its node arena / path / sample buffer (raise "
                     "CB200_ARENA_NODES) or reached an impossible state");
  return CB200_OK;
}

// probs_move_major: answers were written by the tensor-core network as [96][cap]
int iterate(cb200_trainer *t, const float *d_eval, const float *d_probs, int to_play,
            bool probs_move_major = false) {
  const long prs = probs_move_major ? 1 : CB200_NUM_MOVES;
  const long pcs = probs_move_major ? (long)t->cap : 1;
  ProfScope ps(t, 3);
  k_iterate<false, 4><<<(t->P.num_games + kTreeWarps - 1) / kTreeWarps, kTreeWarps * 32, 0, cur_stream()>>>(
      t->P, d_eval, d_probs, prs, pcs, t->d_offs, to_play, t->iterations_done, t->stagger_div);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  if (to_play != 0 && to_play != 1) ++t->iterations_done;
  return CB200_OK;
}

int pack(cb200_trainer *t, int to_play, float *d_rows, ulonglong2 *d_packed) {
  const int grid = (t->P.num_games + 7) / 8;
  ProfScope ps(t, 1);
  k_pack_requests<<<grid, 256, 0, cur_stream()>>>(t->P, to_play, t->d_offs, d_rows, d_packed);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  return CB200_OK;
}

int run_net(cb200_trainer *t, int model, const ulonglong2 *d_states, const int32_t *d_n,
            int n_static, int n_max) {
  ProfScope ps(t, 2);
  if (t->precision[model] == 0)
    return launch_mlp_f32(t->net32[model], d_states, d_n, n_static, n_max, t->d_eval, t->d_probs);
  if (t->precision[model] == 1)
    return launch_mlp_tc(t->nettc[model], d_states, d_n, n_static, n_max, t->d_eval, t->d_probs,
                         (int)t->cap);
  return set_error(CB200_ERR_STATE, "no weights set for this model (cb200_trainer_set_weights)");
}

int guard(cb200_trainer *t) {
  last_error_ref().clear();  // a message always belongs to the call that failed last
  if (!t) return set_error(CB200_ERR_ARG, "null trainer");
  CB_CUDA(cudaSetDevice(t->device));
  return CB200_OK;
}

}  // namespace


// ---- per-game text logs ------------------------------------------------------------------------
// The statements below follow the reference's stream output one by one (same libstdc++
// formatting, including the sticky std::fixed << setprecision(6) that SelfPlayer::writeEval
// leaves on the stream), fed from the device's per-move records (tree.cuh, log_pre_move).
static const char *str_result(int r) {  // strResult, util.cpp:5-25
  switch (r) {
    case kResultLoss: return "L";
    case kResultDraw: return "D";
    case kResultWin: return "W";
    case kDeducedLoss: return "DL";
    case kDeducedDraw: return "DD";
    case kDeducedWin: return "DW";
    default: return "N";
  }
}
static void put_move(std::ostream &os, int id) {  // operator<<(Move), move.cpp:56-78
  static const char cols[] = "abcd";  // getColName, util.cpp
  if (id >= 48) {
    const int piece = (id - 48) / 16, row = ((id - 48) % 16) / 4, col = (id - 48) % 4;
    os << "BCA"[piece] << cols[col] << 4 - row;
    return;
  }
  int r0, c0;
  char dir;
  if (id < 12) r0 = id / 3, c0 = id % 3, dir = 'R';            // right: (r, c) -> (r, c + 1)
  else if (id < 24) r0 = (id - 12) / 4, c0 = (id - 12) % 4, dir = 'D';   // down
  else if (id < 36) r0 = (id - 24) / 3, c0 = (id - 24) % 3 + 1, dir = 'L';  // left
  else r0 = (id - 36) / 4 + 1, c0 = (id - 36) % 4, dir = 'U';  // up
  os << cols[c0] << 4 - r0 << dir;
}
static void put_eval(std::ostream &os, int result, float evaluation, int visits) {  // writeEval
  if (result != kResultNone) {
    os << str_result(result);
    return;
  }
  os << std::fixed << std::setprecision(6) << evaluation / visits;
}
static void put_game(std::ostream &os, const uint32_t w[4]) {  // operator<<(Game), game.cpp:98-139
  const uint64_t w0 = (uint64_t)w[0] | ((uint64_t)w[1] << 32), w1 = (uint64_t)w[2] | ((uint64_t)w[3] << 32);
  for (int row = 0; row < 4; ++row) {
    for (int col = 0; col < 4; ++col) {
      const int b = row * 4 + col;  // cstate planes: base, column, capital, frozen (16 bits each)
      os << (((w0 >> b) & 1) ? 'B' : ' ') << (((w0 >> (16 + b)) & 1) ? 'C' : ' ')
         << (((w0 >> (32 + b)) & 1) ? 'A' : ' ') << (((w0 >> (48 + b)) & 1) ? '#' : ' ');
      if (col < 3) os << '|';
    }
    if (row < 3) os << "\n-------------------\n";
  }
  os << '\n';
  for (int player = 0; player < 2; ++player) {
    os << "Player " << player + 1 << ": ";
    os << "B: " << (int)((w1 >> (8 * (player * 3 + 0))) & 0xff) << ' ';
    os << "C: " << (int)((w1 >> (8 * (player * 3 + 1))) & 0xff) << ' ';
    os << "A: " << (int)((w1 >> (8 * (player * 3 + 2))) & 0xff) << '\n';
  }
  os << "Player " << (int)((w1 >> 48) & 0xff) + 1 << " to play";
}
static float bits_to_float(uint32_t b) {
  float f;
  memcpy(&f, &b, 4);
  return f;
}
static void format_move_choice(std::ostream &os, const uint32_t *rec);
static void format_log_record(std::ostream &os, const uint32_t *rec) {
  if (rec[13] != 0) {  // a Match's random player: no pre-move section (match.cpp:213-215)
    format_move_choice(os, rec);
    return;
  }
  // writePreMoveLogs (selfplayer.cpp:177-188)
  os << "TURN " << (int32_t)rec[0] << "\nPLAYER " << (int32_t)(rec[1] + 1) << " TO PLAY\nVISITS: "
     << (int32_t)rec[2] << '\n';
  os << "POSITION EVALUATION: ";
  put_eval(os, (int)rec[4], bits_to_float(rec[3]), (int)rec[2]);
  os << '\n';
  // writeMoves (selfplayer.cpp:137-175): main line (node.cpp:197-239), then the other moves
  os << "LEGAL MOVES:\n";
  for (uint32_t i = 0; i < rec[5]; ++i) {
    const uint32_t *m = rec + kLogMain + 6 * i;
    os << (int32_t)m[0] << ". ";
    put_move(os, (int)m[1]);
    os << " V: " << (int32_t)m[2] << " E: ";
    if ((int)m[4] != kResultNone)
      os << str_result((int)m[4]);
    else
      os << bits_to_float(m[3]) / (float)(int32_t)m[2];
    os << " p: " << bits_to_float(m[5]) << '\t';
  }
  os << '\n';
  struct MoveData {
    int32_t visits;
    float evaluation, probability;
    int32_t move, result;
    float eval_sum;
  };
  std::vector<MoveData> moves;
  for (uint32_t j = 0; j < rec[6]; ++j) {
    const uint32_t *k = rec + kLogKids + 5 * j;
    const int32_t vis = (int32_t)k[1];
    moves.push_back(MoveData{vis, bits_to_float(k[2]) / static_cast<float>(vis), bits_to_float(k[3]),
                             (int32_t)k[0], (int32_t)k[4], bits_to_float(k[2])});
  }
  std::sort(moves.begin(), moves.end(), [](const MoveData &a, const MoveData &b) -> bool {
    if (a.visits != b.visits) return a.visits > b.visits;
    if (a.evaluation != b.evaluation) return a.evaluation > b.evaluation;
    if (a.probability != b.probability) return a.probability > b.probability;
    return a.move < b.move;
  });
  for (size_t i = 1; i < moves.size(); ++i) {
    put_move(os, moves[i].move);
    os << " V: " << moves[i].visits << " E: ";
    put_eval(os, moves[i].result, moves[i].eval_sum, moves[i].visits);
    os << " P: " << moves[i].probability << '\t';
  }
  os << '\n';
  format_move_choice(os, rec);
}
static void format_move_choice(std::ostream &os, const uint32_t *rec) {
  // writeMoveChoice (selfplayer.cpp:190-194)
  os << "CHOSE MOVE ";
  put_move(os, (int)rec[7]);
  os << "\nNEW POSITION:\n";
  put_game(os, rec + 8);
  os << "\n\n";
  if (rec[12] != 0) {  // endGame (selfplayer.cpp:217-224)
    if ((int)rec[12] - 1 == kResultDraw)
      os << "GAME IS DRAWN.\n";
    else
      os << "PLAYER " << (int32_t)rec[1] + 1 << " WON!\n";
  }
}

// append the records written since the last call to the log files
static int drain_logs(cb200_trainer *t) {
  TreeParams &P = t->P;
  if (P.n_logged <= 0) return CB200_OK;
  t->h_log_count.resize(P.n_logged);
  CB_CUDA(cudaMemcpy(t->h_log_count.data(), P.log_count, (size_t)P.n_logged * sizeof(int32_t),
                     cudaMemcpyDeviceToHost));
  for (int g = 0; g < P.n_logged; ++g) {
    const int have = t->h_log_count[g], done = t->log_written[g];
    if (have <= done) continue;
    t->log_written[g] = have;
    if (!t->log_files[g]) continue;
    t->h_log_rec.resize((size_t)(have - done) * kLogWords);
    CB_CUDA(cudaMemcpy(t->h_log_rec.data(), P.log_buf + ((size_t)g * kLogMaxMoves + done) * kLogWords,
                       t->h_log_rec.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (int k = 0; k < have - done; ++k)
      format_log_record(*t->log_files[g], t->h_log_rec.data() + (size_t)k * kLogWords);
    t->log_files[g]->flush();
  }
  return CB200_OK;
}

// std::mt19937(seed) state expansion (one thread per game; the recurrence is sequential)
__global__ void k_seed_mt(int n, const uint32_t *__restrict__ seeds, uint32_t *__restrict__ mt) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  uint32_t *m = mt + (size_t)g * 624;
  uint32_t prev = seeds[g];
  m[0] = prev;
  for (int i = 1; i < 624; ++i) {
    prev = 1812433253u * (prev ^ (prev >> 30)) + (uint32_t)i;
    m[i] = prev;
  }
}

// (Re)open log_folder/game_<i>.txt for the logged games of this shard, truncating like the
// reference's ofstream(..., out) does for every new Trainer (trainer.cpp:243-250); a missing
// folder silently produces no log.
static void open_log_files(cb200_trainer *t) {
  t->log_files.clear();
  for (int i = 0; i < t->P.n_logged; ++i) {
    auto f = std::make_unique<std::ofstream>(
        t->log_folder + "/game_" + std::to_string(t->P.first_game + i) + ".txt", std::ofstream::out);
    if (!f->is_open()) f.reset();
    t->log_files.push_back(std::move(f));
  }
}

// initialisation: per-game seeds (trainer.cpp:238-256) from the host generator, MT19937 states
// expanded on the device, control blocks
static int init_state(cb200_trainer *t) {
  TreeParams &P = t->P;
  const size_t Gn = (size_t)P.num_games;
  std::vector<int32_t> ctl(Gn * kCtlWords, 0), tree(Gn * 2 * kTreeCtlWords, 0);
  std::vector<uint32_t> seeds(Gn);
  HostMT gen;
  gen.seed((uint32_t)t->seed);
  for (int i = 0; i < P.first_game; ++i) gen.next();
  for (size_t g = 0; g < Gn; ++g) {
    seeds[g] = gen.next();
    int32_t *c = ctl.data() + g * kCtlWords;
    c[CW_PARITY] = (int)((P.first_game + g) & 1);
    c[CW_SPARE] = 2;
    c[CW_MT_IDX] = 624;
    for (int p = 0; p < 2; ++p) {
      int32_t *tw = tree.data() + (g * 2 + p) * kTreeCtlWords;
      tw[TW_ARENA] = p;
      tw[TW_ROOT_VISITS] = 1;
      tw[TW_ROOT_ALLV] = 1;
    }
  }
  cudaStream_t s = cur_stream();
  CB_CUDA(cudaMemcpyAsync(P.ctl, ctl.data(), ctl.size() * 4, cudaMemcpyHostToDevice, s));
  CB_CUDA(cudaMemcpyAsync(P.tree, tree.data(), tree.size() * 4, cudaMemcpyHostToDevice, s));
  // the seeds travel through the (still unused) request-offset buffer
  CB_CUDA(cudaMemcpyAsync(t->d_offs, seeds.data(), Gn * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  k_seed_mt<<<(int)((Gn + 127) / 128), 128, 0, s>>>((int)Gn, (const uint32_t *)t->d_offs, P.mt);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  CB_CUDA(cudaMemsetAsync(P.counters, 0, Gn * 4 * sizeof(long long), s));
  CB_CUDA(cudaMemsetAsync(t->d_offs, 0, Gn * sizeof(int32_t), s));
  CB_CUDA(cudaMemsetAsync(t->d_summary, 0, 4 * sizeof(int32_t), s));
  CB_CUDA(cudaMemsetAsync(t->d_eval, 0, t->cap * sizeof(float), s));
  CB_CUDA(cudaMemsetAsync(t->d_probs, 0, t->cap * CB200_NUM_MOVES * sizeof(float), s));
  CB_CUDA(cudaMemsetAsync(t->d_gctr, 0, (size_t)t->n_groups * 8 * sizeof(int32_t), s));
  CB_CUDA(cudaStreamSynchronize(s));
  if (P.n_logged > 0) {
    CB_CUDA(cudaMemset(P.log_count, 0, (size_t)P.n_logged * sizeof(int32_t)));
    std::fill(t->log_written.begin(), t->log_written.end(), 0);
    open_log_files(t);  // a run after reset() starts its transcripts afresh
  }
  t->iterations_done = 0;
  t->ps_active = false, t->ps_from_lockstep = false, t->ps_n = 0, t->ps_cur = 0;
  if (t->stream_on) {
    CB_CUDA(cudaStreamSynchronize(t->st_stream));
    CB_CUDA(cudaMemset(t->d_emitted, 0, Gn * sizeof(int32_t)));
    CB_CUDA(cudaMemset(t->d_st_ctr, 0, 2 * sizeof(int32_t)));
    t->st_pending = false, t->st_copied = 0, t->st_round = 0;
    t->h_st_ctr[0] = t->h_st_ctr[1] = 0;
  }
  return CB200_OK;
}

// ==============================================================================================
extern "C" {

const char *cb200_last_error(void) { return last_error_ref().c_str(); }

int cb200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int cb200_set_device(int device) {
  CB_CUDA(cudaSetDevice(device));
  return CB200_OK;
}

int cb200_set_stream(void *cuda_stream) {
  set_cur_stream((cudaStream_t)cuda_stream);
  return CB200_OK;
}

int64_t cb200_launch_count(void) { return G().launches.load(); }

int cb200_game_step_device(int64_t n, const void *states_device, uint64_t seed,
                           void *mask_flags_device, void *next_device, void *enc_device) {
  if (n < 0 || (n > 0 && (!states_device || !mask_flags_device || !next_device)))
    return set_error(CB200_ERR_ARG, "cb200_game_step_device: bad arguments");
  return launch_game_step(n, states_device, seed, mask_flags_device, next_device, enc_device);
}

int cb200_game_step(int64_t n, const uint64_t *states, uint64_t seed, uint32_t *mask_flags,
                    uint64_t *next, float *enc) {
  if (n < 0 || (n > 0 && (!states || !mask_flags || !next)))
    return set_error(CB200_ERR_ARG, "cb200_game_step: bad arguments");
  if (n == 0) return CB200_OK;
  void *d_s = nullptr, *d_m = nullptr, *d_n = nullptr, *d_e = nullptr;
  int rc = CB200_OK;
  cudaError_t e;
  if ((e = cudaMalloc(&d_s, n * 16)) != cudaSuccess || (e = cudaMalloc(&d_m, n * 16)) != cudaSuccess ||
      (e = cudaMalloc(&d_n, n * 16)) != cudaSuccess ||
      (enc && (e = cudaMalloc(&d_e, n * CB200_STATE_SIZE * sizeof(float))) != cudaSuccess)) {
    rc = set_error(CB200_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  }
  cudaStream_t s = cur_stream();
  if (rc == CB200_OK && (e = cudaMemcpyAsync(d_s, states, n * 16, cudaMemcpyHostToDevice, s)) != cudaSuccess)
    rc = set_error(CB200_ERR_CUDA, cudaGetErrorString(e));
  if (rc == CB200_OK) rc = launch_game_step(n, d_s, seed, d_m, d_n, d_e);
  if (rc == CB200_OK) {
    e = cudaMemcpyAsync(mask_flags, d_m, n * 16, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(next, d_n, n * 16, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && enc)
      e = cudaMemcpyAsync(enc, d_e, n * CB200_STATE_SIZE * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) rc = set_error(CB200_ERR_CUDA, cudaGetErrorString(e));
  }
  cudaFree(d_s), cudaFree(d_m), cudaFree(d_n), cudaFree(d_e);
  return rc;
}

// ---- Trainer --------------------------------------------------------------------------------
cb200_trainer *cb200_trainer_create_shard(int total_games, int first_game, int num_games,
                                          const char *log_folder, int seed, int max_searches,
                                          int searches_per_eval, float c_puct, float epsilon,
                                          int num_logged, int testing) {
  last_error_ref().clear();
  // the reference only assert()s these (trainer.cpp:25-34); here they are hard errors
  if (num_games <= 0 || total_games < num_games || first_game < 0 ||
      first_game + num_games > total_games || max_searches <= 0 || searches_per_eval <= 0 ||
      max_searches < searches_per_eval || !(c_puct > 0.0f) || !(epsilon >= 0.0f) ||
      !(epsilon <= 1.0f)) {
    set_error(CB200_ERR_ARG, "cb200_trainer_create: invalid argument");
    return nullptr;
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || upload_tables_once() != CB200_OK) {
    if (last_error_ref().empty()) set_error(CB200_ERR_CUDA, "no usable CUDA device");
    return nullptr;
  }
  cb200_trainer *t = new cb200_trainer();
  t->device = dev;
  t->log_folder = log_folder ? log_folder : "";
  TreeParams &P = t->P;
  P.num_games = num_games, P.first_game = first_game, P.total_games = total_games;
  P.max_searches = max_searches, P.spe = searches_per_eval;
  P.c_puct = c_puct, P.epsilon = epsilon, P.testing = testing ? 1 : 0;
  // arena budget: kept subtree + max_searches new nodes per move with head-room; a game that
  // still overflows fails loudly (CB200_ERR_OVERFLOW). ~28 slots/node on average.
  long long nodes = (long long)max_searches * 5 / 2 + 96;
  long long words = nodes * (8 + 4 * 28);
  if (const char *env = getenv("CB200_ARENA_NODES")) {
    words = atoll(env) * (8 + 4 * 28);
  } else {
    // Larger arenas make in-place re-rooting the common case (compaction only when room runs
    // out). The node arenas of one trainer take at most an explicit budget -- 48 GiB by default,
    // CB200_ARENA_BUDGET_MB overrides -- capped at 16 moves' worth of nodes per arena and never
    // below the minimum above; a co-resident trainer keeps the rest of the HBM.
    long long budget_bytes = 48ll << 30;
    if (const char *env = getenv("CB200_ARENA_BUDGET_MB")) budget_bytes = atoll(env) << 20;
    long long budget = budget_bytes / ((long long)num_games * 3 * 4);
    const long long cap = (long long)max_searches * 16 * (8 + 4 * 28);
    if (budget > cap) budget = cap;
    if (budget > words) words = budget;
  }
  words = (words + 3) & ~3ll;
  if (words < 1024) words = 1024;
  if (words > 0x7fffff00ll) words = 0x7fffff00ll;
  P.arena_words = (uint32_t)words;
  t->stagger_div = total_games / max_searches;
  if (t->stagger_div < 1) t->stagger_div = 1;
  const size_t Gn = (size_t)num_games;
  t->cap = Gn * searches_per_eval;
  if (t->cap * CB200_NUM_MOVES >= (size_t)1 << 31) {  // the kernels index answers with 31 bits
    set_error(CB200_ERR_ARG, "cb200_trainer_create: num_games * searches_per_eval too large for one trainer");
    delete t;
    return nullptr;
  }
  bool ok = dmalloc(&P.arenas, Gn * 3 * P.arena_words) == CB200_OK &&
            dmalloc(&P.ctl, Gn * kCtlWords) == CB200_OK &&
            dmalloc(&P.tree, Gn * 2 * kTreeCtlWords) == CB200_OK &&
            dmalloc(&P.mt, Gn * 624) == CB200_OK &&
            dmalloc(&P.pending, t->cap * kPendWords) == CB200_OK &&
            dmalloc(&P.leaf_state, t->cap) == CB200_OK &&
            dmalloc(&P.sample_state, Gn * kMaxSamples) == CB200_OK &&
            dmalloc(&P.sample_probs, Gn * kMaxSamples * CB200_NUM_MOVES) == CB200_OK &&
            dmalloc(&P.counters, Gn * 4) == CB200_OK &&
            // (+ kAnswerSlack rows: a fused tourney reads its answers at the reference's own offsets,
            // tourney.cpp:54-62, which may run a few rows past the requests of the call)
            dmalloc(&t->d_eval, t->cap + kAnswerSlack) == CB200_OK &&
            dmalloc(&t->d_probs, (t->cap + kAnswerSlack) * CB200_NUM_MOVES) == CB200_OK &&
            dmalloc(&t->d_rows, t->cap * CB200_STATE_SIZE) == CB200_OK &&
            dmalloc(&t->d_packed, t->cap) == CB200_OK && dmalloc(&t->d_offs, Gn) == CB200_OK &&
            dmalloc(&t->d_soff, Gn) == CB200_OK && dmalloc(&t->d_summary, 4) == CB200_OK &&
            cudaMallocHost((void **)&t->h_summary, 4 * sizeof(int32_t)) == cudaSuccess;
  if (ok) {
    // c_puct * sqrt(visits) exactly as trainmc.cpp:568 evaluates it (double sqrt, double product,
    // one rounding to float); IEEE sqrt is correctly rounded on host and device alike
    float *d_vsqrt = nullptr;
    std::vector<float> vs(kVsqrtCap);
    for (int i = 0; i < kVsqrtCap; ++i)
      vs[i] = (float)((double)c_puct * sqrt((double)(float)i));
    ok = dmalloc(&d_vsqrt, (size_t)kVsqrtCap) == CB200_OK &&
         cudaMemcpy(d_vsqrt, vs.data(), sizeof(float) * kVsqrtCap, cudaMemcpyHostToDevice) ==
             cudaSuccess;
    P.vsqrt = d_vsqrt;
  }
  if (ok) {
    // logged games = global indices [0, num_logged) (trainer.cpp:243-250) that fall in this shard
    long long nl = (long long)num_logged - first_game;
    if (nl < 0) nl = 0;
    if (nl > num_games) nl = num_games;
    P.n_logged = (int)nl;
    if (P.n_logged > 0) {
      ok = dmalloc(&P.log_buf, (size_t)P.n_logged * kLogMaxMoves * kLogWords) == CB200_OK &&
           dmalloc(&P.log_count, (size_t)P.n_logged) == CB200_OK;
      if (ok) ok = cudaMemset(P.log_count, 0, (size_t)P.n_logged * sizeof(int32_t)) == cudaSuccess;
      t->log_written.assign(P.n_logged, 0);
    }
  }
  if (!ok) {
    if (last_error_ref().empty()) set_error(CB200_ERR_CUDA, "allocation failed");
    cb200_trainer_destroy(t);
    return nullptr;
  }
  // stream groups for the fused loop
  // A launch ends when its slowest game does, so large batches are split over a few independent
  // streams (a group only waits for its own stragglers); CB200_GROUPS overrides.
  int ng = num_games >= 16384 ? 8 : (num_games >= 2048 ? 6 : (num_games >= 512 ? 2 : 1));
  if (const char *env = getenv("CB200_GROUPS")) ng = atoi(env);
  if (ng < 1) ng = 1;
  while (ng > 1 && num_games / ng < 64) ng /= 2;
  t->n_groups = ng;
  // group boundaries fall on whole CTAs of the lock-step kernel (kTreeWarps games)
  int per = ((num_games + ng - 1) / ng + kTreeWarps - 1) / kTreeWarps * kTreeWarps;
  for (int g = 0; g < ng; ++g) {
    int b = g * per, e = b + per < num_games ? b + per : num_games;
    if (b >= num_games) {
      t->n_groups = g;
      break;
    }
    cudaStream_t st;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
      set_error(CB200_ERR_CUDA, "cudaStreamCreate failed");
      cb200_trainer_destroy(t);
      return nullptr;
    }
    t->g_stream.push_back(st), t->g_begin.push_back(b), t->g_end.push_back(e);
  }
  {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    t->ps_ctas = sms;
  }
  t->ps_ld = t->ps_ctas * 16 * kPsRowsPerGame * 2;  // x2: two row regions in two-model runs
  const size_t ps_rows = (size_t)t->ps_ld;
  if (dmalloc(&t->d_gctr, (size_t)t->n_groups * 8) != CB200_OK ||
      dmalloc(&t->d_live_list, Gn) != CB200_OK || dmalloc(&t->d_live_count, (size_t)t->n_groups) != CB200_OK ||
      dmalloc(&t->d_ps_list, Gn) != CB200_OK || dmalloc(&t->d_ps_out, 8) != CB200_OK ||
      dmalloc(&t->d_ps_eval[0], ps_rows) != CB200_OK ||
      dmalloc(&t->d_ps_eval[1], ps_rows) != CB200_OK ||
      dmalloc(&t->d_ps_probs[0], ps_rows * CB200_NUM_MOVES) != CB200_OK ||
      dmalloc(&t->d_ps_probs[1], ps_rows * CB200_NUM_MOVES) != CB200_OK ||
      dmalloc(&t->d_ps_packed, ps_rows) != CB200_OK ||
      cudaMallocHost((void **)&t->h_ps_out, 8 * sizeof(int32_t)) != cudaSuccess ||
      cudaMallocHost((void **)&t->h_gctr, (size_t)t->n_groups * 8 * sizeof(int32_t)) != cudaSuccess) {
    if (last_error_ref().empty()) set_error(CB200_ERR_CUDA, "allocation failed");
    cb200_trainer_destroy(t);
    return nullptr;
  }
  P.game_begin = 0, P.game_end = num_games, P.group_row0 = 0, P.group_ctr = nullptr;
  P.live_list = nullptr, P.live_count = nullptr;
  P.packed = t->d_packed;
  P.phase_prof = nullptr;
  t->seed = seed;
  if (init_state(t) != CB200_OK) {
    cb200_trainer_destroy(t);
    return nullptr;
  }
  return t;
}

cb200_trainer *cb200_trainer_create(int num_games, const char *log_folder, int seed,
                                    int max_searches, int searches_per_eval, float c_puct,
                                    float epsilon, int num_logged, int num_threads, int testing) {
  (void)num_threads;
  return cb200_trainer_create_shard(num_games, 0, num_games, log_folder, seed, max_searches,
                                    searches_per_eval, c_puct, epsilon, num_logged, testing);
}

// debug: straggler instrumentation of the game-step kernel (see TreeParams::phase_prof)
int cb200_trainer_phase_profile(cb200_trainer *t, int enable, uint64_t out[16]) {
  int rc = guard(t);
  if (rc) return rc;
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  if (t->P.phase_prof && out) {
    CB_CUDA(cudaMemcpy(out, t->P.phase_prof, 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    CB_CUDA(cudaMemset(t->P.phase_prof, 0, 16 * sizeof(uint64_t)));
  }
  if (enable && !t->P.phase_prof) {
    CB_CUDA(cudaMalloc((void **)&t->P.phase_prof, 16 * sizeof(uint64_t)));
    CB_CUDA(cudaMemset(t->P.phase_prof, 0, 16 * sizeof(uint64_t)));
  } else if (!enable && t->P.phase_prof) {
    cudaFree(t->P.phase_prof);
    t->P.phase_prof = nullptr;
  }
  return CB200_OK;
}

int cb200_trainer_reset(cb200_trainer *t, int seed) {
  int rc = guard(t);
  if (rc) return rc;
  t->seed = seed;
  return init_state(t);
}

int cb200_trainer_set_profiling(cb200_trainer *t, int enable) {
  int rc = guard(t);
  if (rc) return rc;
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  if ((rc = prof_drain(t)) != CB200_OK) return rc;
  t->profiling = enable != 0;
  for (int i = 0; i < 8; ++i) t->class_ms[i] = 0, t->class_launches[i] = 0;
  t->lockstep_searches = t->lockstep_evals = t->total_searches = t->total_evals = 0;
  t->lockstep_wall_ms = t->tail_wall_ms = 0;
  return CB200_OK;
}

int cb200_trainer_phase_times(cb200_trainer *t, double out_ms[2]) {
  int rc = guard(t);
  if (rc) return rc;
  out_ms[0] = t->lockstep_wall_ms, out_ms[1] = t->tail_wall_ms;
  return CB200_OK;
}

int cb200_trainer_phase_split(cb200_trainer *t, int64_t out[4]) {
  int rc = guard(t);
  if (rc) return rc;
  out[0] = t->lockstep_searches, out[1] = t->total_searches;
  out[2] = t->lockstep_evals, out[3] = t->total_evals;
  return CB200_OK;
}

int cb200_trainer_kernel_times(cb200_trainer *t, double out_ms[8], int64_t out_launches[8]) {
  int rc = guard(t);
  if (rc) return rc;
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  if ((rc = prof_drain(t)) != CB200_OK) return rc;
  for (int i = 0; i < 8; ++i) out_ms[i] = t->class_ms[i], out_launches[i] = t->class_launches[i];
  return CB200_OK;
}

void cb200_trainer_destroy(cb200_trainer *t) {
  if (!t) return;
  cudaSetDevice(t->device);
  for (cudaEvent_t e : t->ev_pool) cudaEventDestroy(e);
  TreeParams &P = t->P;
  cudaFree(P.log_buf), cudaFree(P.log_count);
  cudaFree(t->d_ps_list), cudaFree(t->d_ps_out), cudaFree(t->d_ps_eval[0]), cudaFree(t->d_ps_eval[1]);
  cudaFree(t->d_ps_probs[0]), cudaFree(t->d_ps_probs[1]);
  cudaFree(t->d_ps_packed), cudaFreeHost(t->h_ps_out);
  cudaFree((void *)P.vsqrt), cudaFree(P.arenas), cudaFree(P.ctl), cudaFree(P.tree), cudaFree(P.mt), cudaFree(P.pending);
  cudaFree(P.leaf_state), cudaFree(P.sample_state), cudaFree(P.sample_probs), cudaFree(P.counters);
  cudaFree(t->d_eval), cudaFree(t->d_probs), cudaFree(t->d_rows), cudaFree(t->d_packed);
  cudaFree(t->d_offs), cudaFree(t->d_soff), cudaFree(t->d_summary), cudaFree(P.phase_prof);
  cudaFree(t->d_samp);
  cudaFree(t->d_raw);
  cudaFree(t->d_gath), cudaFree(t->d_gcounts);
  if (t->h_gcounts) cudaFreeHost(t->h_gcounts);
  cudaFree(t->d_st), cudaFree(t->d_st_game), cudaFree(t->d_st_ctr), cudaFree(t->d_emitted), cudaFree(t->d_st_soff);
  if (t->h_st) cudaFreeHost(t->h_st);
  if (t->h_st_game) cudaFreeHost(t->h_st_game);
  if (t->h_st_ctr) cudaFreeHost(t->h_st_ctr);
  if (t->st_ev) cudaEventDestroy(t->st_ev);
  if (t->st_stream) cudaStreamDestroy(t->st_stream);
  if (t->h_summary) cudaFreeHost(t->h_summary);
  if (t->h_gctr) cudaFreeHost(t->h_gctr);
  cudaFree(t->d_gctr), cudaFree(t->d_live_list), cudaFree(t->d_live_count);
  for (cudaStream_t st : t->g_stream) cudaStreamDestroy(st);
  for (int m = 0; m < 2; ++m) {
    cudaFree(t->net32[m].w);
    net_tc_free(t->nettc[m]);
  }
  delete t;
}

int cb200_trainer_num_requests(cb200_trainer *t, int to_play) {
  int rc = guard(t);
  if (rc) return rc;
  if ((rc = scan(t, to_play)) != CB200_OK) return rc;
  if ((rc = fetch_summary(t)) != CB200_OK) return rc;
  return t->h_summary[0];
}

int cb200_trainer_write_requests(cb200_trainer *t, float *game_states, int to_play) {
  int rc = guard(t);
  if (rc) return rc;
  if (!game_states) return set_error(CB200_ERR_ARG, "null game_states");
  if ((rc = scan(t, to_play)) != CB200_OK) return rc;
  if ((rc = pack(t, to_play, t->d_rows, nullptr)) != CB200_OK) return rc;
  if ((rc = fetch_summary(t)) != CB200_OK) return rc;
  const int n = t->h_summary[0];
  if (n > 0) {
    CB_CUDA(cudaMemcpyAsync(game_states, t->d_rows, (size_t)n * CB200_STATE_SIZE * sizeof(float),
                            cudaMemcpyDeviceToHost, cur_stream()));
    CB_CUDA(cudaStreamSynchronize(cur_stream()));
  }
  return CB200_OK;
}

int cb200_trainer_do_iteration(cb200_trainer *t, const float *eval, const float *probs,
                               int to_play) {
  int rc = guard(t);
  if (rc) return rc;
  if (t->ps_active)
    return set_error(CB200_ERR_STATE, "cb200_trainer_do_iteration: this trainer is in the middle of a "
                                      "fused run (persistent kernel); call cb200_trainer_reset first");
  // offsets of the answers = prefix sums of the request counts they were written for
  if ((rc = scan(t, to_play)) != CB200_OK) return rc;
  if ((rc = fetch_summary(t)) != CB200_OK) return rc;
  const int n = t->h_summary[0];
  if (n > 0) {
    if (!eval || !probs) return set_error(CB200_ERR_ARG, "requests pending but eval/probs null");
    CB_CUDA(cudaMemcpyAsync(t->d_eval, eval, (size_t)n * sizeof(float), cudaMemcpyHostToDevice,
                            cur_stream()));
    CB_CUDA(cudaMemcpyAsync(t->d_probs, probs, (size_t)n * CB200_NUM_MOVES * sizeof(float),
                            cudaMemcpyHostToDevice, cur_stream()));
  }
  if ((rc = iterate(t, t->d_eval, t->d_probs, to_play)) != CB200_OK) return rc;
  if ((rc = scan(t, to_play)) != CB200_OK) return rc;
  if ((rc = fetch_summary(t)) != CB200_OK) return rc;
  if ((rc = drain_logs(t)) != CB200_OK) return rc;
  return t->h_summary[1] == 0 ? 1 : 0;
}

static int fetch_ctl(cb200_trainer *t) {
  t->h_ctl.resize((size_t)t->P.num_games * kCtlWords);
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  CB_CUDA(cudaMemcpy(t->h_ctl.data(), t->P.ctl, t->h_ctl.size() * 4, cudaMemcpyDeviceToHost));
  return CB200_OK;
}

int cb200_trainer_num_samples(cb200_trainer *t) {
  int rc = guard(t);
  if (rc) return rc;
  if ((rc = fetch_ctl(t)) != CB200_OK) return rc;
  long long n = 0;
  for (int g = 0; g < t->P.num_games; ++g) n += t->h_ctl[(size_t)g * kCtlWords + CW_N_SAMPLES];
  return (int)n;
}

int cb200_trainer_write_samples(cb200_trainer *t, float *game_states, float *eval_samples,
                                float *prob_samples) {
  int rc = guard(t);
  if (rc) return rc;
  if (!game_states || !eval_samples || !prob_samples) return set_error(CB200_ERR_ARG, "null buffer");
  if ((rc = fetch_ctl(t)) != CB200_OK) return rc;
  const int Gn = t->P.num_games;
  std::vector<int32_t> soff(Gn);
  long long ns = 0;
  for (int g = 0; g < Gn; ++g) {
    soff[g] = (int32_t)ns;
    ns += t->h_ctl[(size_t)g * kCtlWords + CW_N_SAMPLES];
  }
  if (ns == 0) return CB200_OK;
  const size_t rows = (size_t)ns * 8;
  if (rows > t->samp_rows) {  // one cached device buffer: [rows][70] + [rows] + [rows][96]
    cudaFree(t->d_samp);
    t->d_samp = nullptr, t->samp_rows = 0;
    const size_t want = rows + rows / 4 + 1024;
    rc = dmalloc(&t->d_samp, want * (CB200_STATE_SIZE + 1 + CB200_NUM_MOVES));
    if (rc != CB200_OK) return rc;
    t->samp_rows = want;
  }
  float *d_gs = t->d_samp, *d_ev = d_gs + t->samp_rows * CB200_STATE_SIZE, *d_pr = d_ev + t->samp_rows;
  {
    cudaStream_t s = cur_stream();
    cudaError_t e = cudaMemcpyAsync(t->d_soff, soff.data(), Gn * sizeof(int32_t),
                                    cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
      const long long warps = (long long)Gn * kMaxSamples;
      k_write_samples<<<(unsigned)((warps + 7) / 8), 256, 0, s>>>(t->P, t->d_soff, d_gs, d_ev, d_pr, nullptr, 0, nullptr);
      CB_LAUNCHED();
      e = cudaGetLastError();
    }
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(game_states, d_gs, rows * CB200_STATE_SIZE * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(eval_samples, d_ev, rows * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(prob_samples, d_pr, rows * CB200_NUM_MOVES * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) rc = set_error(CB200_ERR_CUDA, cudaGetErrorString(e));
  }
  return rc;
}

static float game_score(int result) {  // SelfPlayer::score selfplayer.cpp:57-64
  if (result == kResultLoss) return 0.0f;
  if (result == kResultWin) return 1.0f;
  return 0.5f;
}

float cb200_trainer_score(cb200_trainer *t) {  // trainer.cpp:59-68
  if (guard(t) || fetch_ctl(t)) return NAN;
  const int Gn = t->P.num_games;
  float score = 0;
  for (int g = 0; g < Gn; ++g)
    if (((t->P.first_game + g) & 1) == 0) score += game_score(t->h_ctl[(size_t)g * kCtlWords + CW_RESULT]);
  for (int g = 0; g < Gn; ++g)
    if ((t->P.first_game + g) & 1)
      score = (float)(score + (1.0 - game_score(t->h_ctl[(size_t)g * kCtlWords + CW_RESULT])));
  return score / (float)(size_t)Gn;
}

float cb200_trainer_avg_mate_length(cb200_trainer *t) {  // trainer.cpp:70-77
  if (guard(t) || fetch_ctl(t)) return NAN;
  const int Gn = t->P.num_games;
  int total = 0;
  for (int g = 0; g < Gn; ++g) {
    const int32_t *c = t->h_ctl.data() + (size_t)g * kCtlWords;
    total += c[CW_MATE_TURN] == 0 ? 0 : c[CW_N_SAMPLES] - c[CW_MATE_TURN] + 1;  // selfplayer.cpp:66-71
  }
  return (float)total / (float)(size_t)Gn;
}

int cb200_trainer_write_scores(cb200_trainer *t, const char *file) {  // trainer.cpp:115-162
  int rc = guard(t);
  if (rc) return rc;
  if (!file) return set_error(CB200_ERR_ARG, "null file");
  if ((rc = fetch_ctl(t)) != CB200_OK) return rc;
  const int Gn = t->P.num_games;
  std::vector<float> scores(Gn);
  for (int g = 0; g < Gn; ++g) {
    float s = game_score(t->h_ctl[(size_t)g * kCtlWords + CW_RESULT]);
    scores[g] = ((t->P.first_game + g) & 1) ? (float)(1.0 - s) : s;
  }
  std::ofstream f(file, std::ofstream::out);
  if (!f) return set_error(CB200_ERR_ARG, std::string("cannot open ") + file);
  const char *names[2] = {"First", "Second"};
  const int half = Gn / 2;
  for (int side = 0; side < 2; ++side) {
    int wins = 0, draws = 0;
    for (int g = side; g < Gn; g += 2) {
      if (scores[g] == 1.0f) ++wins;
      else if (scores[g] == 0.5f) ++draws;
    }
    f << names[side] << " player wins: " << wins << " / " << half << " = "
      << static_cast<float>(wins) / half << "\n" << names[side] << " player draws: " << draws
      << " / " << half << " = " << static_cast<float>(draws) / half << "\n" << names[side]
      << " player losses: " << half - wins - draws << " / " << half << " = "
      << static_cast<float>(half - wins - draws) / half << '\n';
  }
  return CB200_OK;
}

int cb200_trainer_counters(cb200_trainer *t, int64_t out[4]) {
  int rc = guard(t);
  if (rc) return rc;
  std::vector<long long> h((size_t)t->P.num_games * 4);
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  CB_CUDA(cudaMemcpy(h.data(), t->P.counters, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
  out[0] = out[1] = out[2] = 0;
  long long searches = 0;
  for (int g = 0; g < t->P.num_games; ++g)
    out[0] += h[4 * g], out[1] += h[4 * g + 1], out[2] += h[4 * g + 2], searches += h[4 * g + 3];
  t->searches_now = searches;
  out[3] = t->iterations_done;
  return CB200_OK;
}

int cb200_trainer_game_results(cb200_trainer *t, int32_t *results) {
  int rc = guard(t);
  if (rc) return rc;
  if ((rc = fetch_ctl(t)) != CB200_OK) return rc;
  for (int g = 0; g < t->P.num_games; ++g) results[g] = t->h_ctl[(size_t)g * kCtlWords + CW_RESULT];
  return CB200_OK;
}

int cb200_trainer_write_raw_samples(cb200_trainer *t, uint64_t *states, float *probs, float *labels,
                                    int32_t *game_of) {
  int rc = guard(t);
  if (rc) return rc;
  if ((rc = fetch_ctl(t)) != CB200_OK) return rc;
  const int Gn = t->P.num_games;
  std::vector<ulonglong2> hs;
  std::vector<float> hp;
  if (states) {
    hs.resize((size_t)Gn * kMaxSamples);
    CB_CUDA(cudaMemcpy(hs.data(), t->P.sample_state, hs.size() * sizeof(ulonglong2), cudaMemcpyDeviceToHost));
  }
  if (probs) {
    hp.resize((size_t)Gn * kMaxSamples * CB200_NUM_MOVES);
    CB_CUDA(cudaMemcpy(hp.data(), t->P.sample_probs, hp.size() * sizeof(float), cudaMemcpyDeviceToHost));
  }
  size_t row = 0;
  for (int g = 0; g < Gn; ++g) {
    const int32_t *c = t->h_ctl.data() + (size_t)g * kCtlWords;
    const int ns = c[CW_N_SAMPLES];
    for (int i = 0; i < ns; ++i, ++row) {
      if (states) states[2 * row] = hs[(size_t)g * kMaxSamples + i].x, states[2 * row + 1] = hs[(size_t)g * kMaxSamples + i].y;
      if (probs) memcpy(probs + row * CB200_NUM_MOVES, hp.data() + ((size_t)g * kMaxSamples + i) * CB200_NUM_MOVES, CB200_NUM_MOVES * sizeof(float));
      if (labels) {
        float ev = c[CW_RESULT] == kResultDraw ? 0.0f : 1.0f;
        labels[row] = ((ns - 1 - i) & 1) ? -ev : ev;
      }
      if (game_of) game_of[row] = g;
    }
  }
  return CB200_OK;
}

int cb200_trainer_raw_samples_device(cb200_trainer *t, void **rows_device, int *n_rows) {
  int rc = guard(t);
  if (rc) return rc;
  if (!rows_device || !n_rows) return set_error(CB200_ERR_ARG, "null output");
  if ((rc = fetch_ctl(t)) != CB200_OK) return rc;
  const int Gn = t->P.num_games;
  std::vector<int32_t> soff(Gn);
  long long ns = 0;
  for (int g = 0; g < Gn; ++g) {
    soff[g] = (int32_t)ns;
    ns += t->h_ctl[(size_t)g * kCtlWords + CW_N_SAMPLES];
  }
  if ((size_t)ns > t->raw_rows) {
    cudaFree(t->d_raw);
    t->d_raw = nullptr, t->raw_rows = 0;
    const size_t want = (size_t)ns + (size_t)ns / 4 + 1024;
    if ((rc = dmalloc(&t->d_raw, want * 102)) != CB200_OK) return rc;
    t->raw_rows = want;
  }
  cudaStream_t s = cur_stream();
  CB_CUDA(cudaMemcpyAsync(t->d_soff, soff.data(), Gn * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  if (ns > 0) {
    const long long warps = (long long)Gn * kMaxSamples;
    k_pack_raw_samples<<<(unsigned)((warps + 7) / 8), 256, 0, s>>>(t->P, t->d_soff, t->d_raw);
    CB_LAUNCHED();
    CB_CUDA(cudaGetLastError());
  }
  CB_CUDA(cudaStreamSynchronize(s));
  *rows_device = t->d_raw;
  *n_rows = (int)ns;
  return CB200_OK;
}

static int emit_finished(cb200_trainer *t, bool final);

// ---- NCCL all-gather of the finished samples (SURVEY 8e) ---------------------------------------
int cb200_nccl_unique_id(void *id_out) {
  last_error_ref().clear();
  NcclApi &N = nccl_api();
  if (!N.ok) return set_error(CB200_ERR_STATE, "libnccl.so.2 is not available in this process");
  if (!id_out) return set_error(CB200_ERR_ARG, "null id");
  CB_NCCL(N.GetUniqueId((NcclUniqueId *)id_out));
  return CB200_OK;
}

void *cb200_nccl_comm_create(int rank, int world, const void *unique_id) {
  last_error_ref().clear();
  NcclApi &N = nccl_api();
  if (!N.ok || !unique_id || world <= 0 || rank < 0 || rank >= world) {
    set_error(CB200_ERR_ARG, "cb200_nccl_comm_create: NCCL unavailable or bad arguments");
    return nullptr;
  }
  NcclUniqueId id;
  memcpy(&id, unique_id, sizeof(id));
  void *comm = nullptr;
  const int r = N.CommInitRank(&comm, world, id, rank);
  if (r != 0) {
    set_error(CB200_ERR_CUDA, std::string("ncclCommInitRank: ") + N.GetErrorString(r));
    return nullptr;
  }
  return comm;
}

void cb200_nccl_comm_destroy(void *nccl_comm) {
  NcclApi &N = nccl_api();
  if (N.ok && nccl_comm) N.CommDestroy(nccl_comm);
}

int cb200_trainer_allgather_samples(cb200_trainer *t, void *nccl_comm, void **rows_device, int *n_rows,
                                    int32_t *rows_per_rank) {
  int rc = guard(t);
  if (rc) return rc;
  NcclApi &N = nccl_api();
  if (!N.ok) return set_error(CB200_ERR_STATE, "libnccl.so.2 is not available in this process");
  if (!nccl_comm || !rows_device || !n_rows) return set_error(CB200_ERR_ARG, "null argument");
  int world = 0, rank = 0;
  CB_NCCL(N.CommCount(nccl_comm, &world));
  CB_NCCL(N.CommUserRank(nccl_comm, &rank));
  void *mine = nullptr;
  int n_mine = 0;
  if ((rc = cb200_trainer_raw_samples_device(t, &mine, &n_mine)) != CB200_OK) return rc;
  cudaStream_t st = cur_stream();
  if (world > t->gcounts_world) {  // first call, or a larger communicator than before
    cudaFree(t->d_gcounts);
    if (t->h_gcounts) cudaFreeHost(t->h_gcounts);
    t->d_gcounts = nullptr, t->h_gcounts = nullptr, t->gcounts_world = 0;
    if ((rc = dmalloc(&t->d_gcounts, (size_t)world + 1)) != CB200_OK) return rc;
    CB_CUDA(cudaMallocHost((void **)&t->h_gcounts, ((size_t)world + 1) * sizeof(int32_t)));
    t->gcounts_world = world;
  }
  // 1. row counts of every rank
  t->h_gcounts[world] = n_mine;
  CB_CUDA(cudaMemcpyAsync(t->d_gcounts + world, t->h_gcounts + world, sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CB_NCCL(N.AllGather(t->d_gcounts + world, t->d_gcounts, 1, kNcclInt32, nccl_comm, st));
  CB_CUDA(cudaMemcpyAsync(t->h_gcounts, t->d_gcounts, (size_t)world * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CB_CUDA(cudaStreamSynchronize(st));
  long long total = 0;
  int max_rows = 1;
  for (int r = 0; r < world; ++r) {
    total += t->h_gcounts[r];
    if (t->h_gcounts[r] > max_rows) max_rows = t->h_gcounts[r];
    if (rows_per_rank) rows_per_rank[r] = t->h_gcounts[r];
  }
  // 2. padded all-gather straight from / to device memory, then compaction in rank order
  const size_t padded = (size_t)world * max_rows * 102, need = padded + (size_t)max_rows * 102 + (size_t)total * 102;
  if (need > t->gath_floats) {
    cudaFree(t->d_gath);
    t->d_gath = nullptr, t->gath_floats = 0;
    if ((rc = dmalloc(&t->d_gath, need + need / 4)) != CB200_OK) return rc;
    t->gath_floats = need + need / 4;
  }
  float *d_pad = t->d_gath, *d_send = d_pad + padded, *d_out = d_send + (size_t)max_rows * 102;
  if (n_mine > 0)
    CB_CUDA(cudaMemcpyAsync(d_send, mine, (size_t)n_mine * 102 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  CB_NCCL(N.AllGather(d_send, d_pad, (size_t)max_rows * 102, kNcclFloat32, nccl_comm, st));
  if (total > 0) {
    k_compact_gathered<<<dim3(64, world), 256, 0, st>>>(d_pad, d_out, t->d_gcounts, world, max_rows, 102);
    CB_LAUNCHED();
    CB_CUDA(cudaGetLastError());
  }
  CB_CUDA(cudaStreamSynchronize(st));
  *rows_device = d_out;
  *n_rows = (int)total;
  return CB200_OK;
}

int cb200_trainer_stream_samples(cb200_trainer *t, int64_t max_samples) {
  int rc = guard(t);
  if (rc) return rc;
  if (t->P.testing) return set_error(CB200_ERR_STATE, "testing-mode trainers produce no samples");
  if (max_samples == 0) {
    t->stream_on = false;
    return CB200_OK;
  }
  if (max_samples < 0) max_samples = (int64_t)t->P.num_games * 32;  // ~20 moves per game on average
  if (max_samples > (int64_t)t->P.num_games * kMaxSamples) max_samples = (int64_t)t->P.num_games * kMaxSamples;
  if (max_samples * 8 >= (1ll << 31)) return set_error(CB200_ERR_ARG, "max_samples too large");
  if ((size_t)max_samples > t->st_cap) {
    cudaFree(t->d_st), cudaFree(t->d_st_game);
    if (t->h_st) cudaFreeHost(t->h_st);
    if (t->h_st_game) cudaFreeHost(t->h_st_game);
    t->d_st = nullptr, t->d_st_game = nullptr, t->h_st = nullptr, t->h_st_game = nullptr, t->st_cap = 0;
    const size_t floats = (size_t)max_samples * 8 * (CB200_STATE_SIZE + 1 + CB200_NUM_MOVES);
    if ((rc = dmalloc(&t->d_st, floats)) != CB200_OK || (rc = dmalloc(&t->d_st_game, (size_t)max_samples)) != CB200_OK)
      return rc;
    CB_CUDA(cudaMallocHost((void **)&t->h_st, floats * sizeof(float)));
    CB_CUDA(cudaMallocHost((void **)&t->h_st_game, (size_t)max_samples * sizeof(int32_t)));
    t->st_cap = (size_t)max_samples;
  }
  if (!t->d_emitted) {
    const size_t Gn = (size_t)t->P.num_games;
    if ((rc = dmalloc(&t->d_emitted, Gn)) != CB200_OK || (rc = dmalloc(&t->d_st_soff, Gn)) != CB200_OK ||
        (rc = dmalloc(&t->d_st_ctr, 2)) != CB200_OK)
      return rc;
    CB_CUDA(cudaMallocHost((void **)&t->h_st_ctr, 2 * sizeof(int32_t)));
    CB_CUDA(cudaStreamCreateWithFlags(&t->st_stream, cudaStreamNonBlocking));
    CB_CUDA(cudaEventCreateWithFlags(&t->st_ev, cudaEventDisableTiming));
  }
  CB_CUDA(cudaStreamSynchronize(t->st_stream));
  CB_CUDA(cudaMemset(t->d_emitted, 0, (size_t)t->P.num_games * sizeof(int32_t)));
  CB_CUDA(cudaMemset(t->d_st_ctr, 0, 2 * sizeof(int32_t)));
  t->st_pending = false, t->st_copied = 0, t->st_round = 0;
  t->h_st_ctr[0] = t->h_st_ctr[1] = 0;
  t->st_limit = (size_t)max_samples;
  t->stream_on = true;
  return CB200_OK;
}

int cb200_trainer_streamed_samples(cb200_trainer *t, const float **game_states, const float **eval_samples,
                                   const float **prob_samples, const int32_t **game_of, int *n_samples) {
  int rc = guard(t);
  if (rc) return rc;
  if (!t->stream_on) return set_error(CB200_ERR_STATE, "cb200_trainer_stream_samples was not enabled");
  if (!game_states || !eval_samples || !prob_samples || !game_of || !n_samples)
    return set_error(CB200_ERR_ARG, "null output");
  // work queued on the self-play streams is complete when run_selfplay has returned
  if ((rc = emit_finished(t, true)) != CB200_OK) return rc;
  if (t->h_st_ctr[1] != 0)
    return set_error(CB200_ERR_OVERFLOW, "the sample staging buffer is too small for this run: enable streaming "
                                         "with a larger max_samples (or use cb200_trainer_write_samples)");
  const size_t R = t->st_cap * 8;
  *game_states = t->h_st, *eval_samples = t->h_st + R * CB200_STATE_SIZE;
  *prob_samples = t->h_st + R * CB200_STATE_SIZE + R;
  *game_of = t->h_st_game;
  *n_samples = (int)t->st_copied;
  return CB200_OK;
}

int cb200_trainer_set_weights(cb200_trainer *t, int model, const float *weights, size_t n_floats,
                              int precision) {
  int rc = guard(t);
  if (rc) return rc;
  if (model < 0 || model > 1 || !weights || n_floats != kNetWeightFloats ||
      (precision < 0 || precision > 3))
    return set_error(CB200_ERR_ARG, "cb200_trainer_set_weights: bad arguments (127997 floats, precision 0|1|2|3)");
  // tensor-core operand modes: precision 1 -> bf16, 2 -> fp16, 3 -> bf16x3 (hi + lo operands)
  rc = precision == 0 ? net_f32_upload(t->net32[model], weights)
                      : net_tc_upload(t->nettc[model], weights, precision == 1 ? 0 : (precision == 2 ? 1 : 2));
  // precisions 1-3 share the tensor-core kernel and the move-major output
  if (rc == CB200_OK) t->precision[model] = precision == 0 ? 0 : 1;
  return rc;
}

int cb200_trainer_evaluate(cb200_trainer *t, int model, int n, const float *game_states,
                           float *eval, float *probs) {
  int rc = guard(t);
  if (rc) return rc;
  if (model < 0 || model > 1 || n < 0 || (size_t)n > t->cap || !game_states || !eval || !probs)
    return set_error(CB200_ERR_ARG, "cb200_trainer_evaluate: bad arguments (n <= num_games*searches_per_eval)");
  if (n == 0) return CB200_OK;
  // pack the 70-float rows back into cstates on the host (rows hold only 0/1 and k/4 values)
  std::vector<ulonglong2> hs(n);
  for (int i = 0; i < n; ++i) {
    const float *r = game_states + (size_t)i * CB200_STATE_SIZE;
    uint64_t w0 = 0, w1 = 0;
    for (int j = 0; j < 64; ++j)
      if (r[j] != 0.0f) w0 |= 1ull << (16 * (j & 3) + (j >> 2));
    // the encoding holds the mover's pieces first; keep that order with to_play = 0
    for (int j = 0; j < 6; ++j) w1 |= (uint64_t)(int)(r[64 + j] * 4.0f + 0.5f) << (8 * j);
    hs[i] = make_ulonglong2(w0, w1);
  }
  cudaStream_t s = cur_stream();
  CB_CUDA(cudaMemcpyAsync(t->d_packed, hs.data(), (size_t)n * sizeof(ulonglong2), cudaMemcpyHostToDevice, s));
  if ((rc = run_net(t, model, t->d_packed, nullptr, n, n)) != CB200_OK) return rc;
  CB_CUDA(cudaMemcpyAsync(eval, t->d_eval, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (t->precision[model] == 1) {  // move-major [96][cap] on the device -> row-major for the caller
    // transposed on the device into the (idle) request-row buffer: cap * 70 floats >= n * 96 is not
    // guaranteed, so rows go through it in slices
    const size_t slice = t->cap * CB200_STATE_SIZE / CB200_NUM_MOVES;
    for (size_t r0 = 0; r0 < (size_t)n; r0 += slice) {
      const int rows = (int)std::min(slice, (size_t)n - r0);
      k_probs_row_major<<<(rows * CB200_NUM_MOVES + 255) / 256, 256, 0, s>>>(t->d_probs + r0, (int)t->cap, rows,
                                                                             t->d_rows);
      CB_LAUNCHED();
      CB_CUDA(cudaGetLastError());
      CB_CUDA(cudaMemcpyAsync(probs + r0 * CB200_NUM_MOVES, t->d_rows, (size_t)rows * CB200_NUM_MOVES * sizeof(float),
                              cudaMemcpyDeviceToHost, s));
    }
    CB_CUDA(cudaStreamSynchronize(s));
    return CB200_OK;
  }
  CB_CUDA(cudaMemcpyAsync(probs, t->d_probs, (size_t)n * CB200_NUM_MOVES * sizeof(float), cudaMemcpyDeviceToHost, s));
  CB_CUDA(cudaStreamSynchronize(s));
  return CB200_OK;
}

// Persistent fused tail (persistent.cuh). Called with every stream idle. Runs the remaining games
// (or `max_rounds` iterations of them) as a sequence of persistent launches; between launches
// the live games are listed again so that they spread evenly over the SMs (8 games per CTA
// once they fit, else 16). A launch reads the answers of the requests queued before it from the
// buffer the previous launch (or the lock-step loop) wrote, and writes its own into the other.
static int ps_list_games(cb200_trainer *t) {
  cudaStream_t st = t->g_stream[0];
  k_live_list<<<1, 32, 0, st>>>(t->P, t->d_ps_list, t->d_ps_out + 4);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  CB_CUDA(cudaMemcpyAsync(t->h_ps_out + 4, t->d_ps_out + 4, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CB_CUDA(cudaStreamSynchronize(st));
  t->ps_n = t->h_ps_out[4];
  return CB200_OK;
}

extern "C++" {
template <int kMode, int kGames>
static int ps_launch(cb200_trainer *t, const TreeParams &P, int rounds, int exit_done) {
  static bool attr_set[16] = {false};
  if (t->device < 16 && !attr_set[t->device]) {
    CB_CUDA(cudaFuncSetAttribute(k_selfplay_persistent<kMode, kGames>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)ps_smem_bytes<kMode, kGames>()));
    attr_set[t->device] = true;
  }
  const float *ev0 = t->ps_from_lockstep ? t->d_eval : t->d_ps_eval[t->ps_cur];
  const float *pr0 = t->ps_from_lockstep ? t->d_probs : t->d_ps_probs[t->ps_cur];
  const long pcs0 = t->ps_from_lockstep ? (long)t->cap : (long)t->ps_ld;
  const int nxt = 1 - t->ps_cur;
  // one CTA per SM, games dealt round-robin (every CTA gets ceil or floor of ps_n / grid)
  const int grid = t->ps_n < t->ps_ctas ? t->ps_n : t->ps_ctas;
  // two-model (gating match) runs: model 1 answers the other side's requests
  const uint8_t *w1 = P.testing ? (const uint8_t *)t->nettc[1].w : nullptr;
  k_selfplay_persistent<kMode, kGames><<<grid, kGames * 32, ps_smem_bytes<kMode, kGames>(), t->g_stream[0]>>>(
      P, (const uint8_t *)t->nettc[0].w, w1, t->d_ps_list, t->ps_n, ev0, pr0, pcs0, t->d_ps_eval[nxt],
      t->d_ps_probs[nxt], t->ps_ld, t->d_ps_packed, rounds, exit_done, t->iterations_done,
      t->d_ps_out);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  return CB200_OK;
}
}  // extern "C++"

// Streaming sample output. Called whenever the host has control during a fused run (every batch
// of lock-step iterations, between persistent launches) and once at the end (final): queues the
// device->host copy of the rows the PREVIOUS round produced (their count has reached the host by
// now), then stamps the games that finished since and expands their samples into the staging
// buffer. Everything runs on its own stream, beside the self-play kernels.
static int emit_finished(cb200_trainer *t, bool final) {
  if (!t->stream_on) return CB200_OK;
  cudaStream_t st = t->st_stream;
  const size_t R = t->st_cap * 8;
  float *d_gs = t->d_st, *d_ev = d_gs + R * CB200_STATE_SIZE, *d_pr = d_ev + R;
  float *h_gs = t->h_st, *h_ev = h_gs + R * CB200_STATE_SIZE, *h_pr = h_ev + R;
  for (int pass = 0; pass < (final ? 2 : 1); ++pass) {
    if (t->st_pending) {
      CB_CUDA(cudaEventSynchronize(t->st_ev));
      t->st_pending = false;
      const size_t total = (size_t)t->h_st_ctr[0], a = t->st_copied;
      if (total > a) {
        const size_t n = total - a;
        CB_CUDA(cudaMemcpyAsync(h_gs + a * 8 * CB200_STATE_SIZE, d_gs + a * 8 * CB200_STATE_SIZE,
                                n * 8 * CB200_STATE_SIZE * sizeof(float), cudaMemcpyDeviceToHost, st));
        CB_CUDA(cudaMemcpyAsync(h_ev + a * 8, d_ev + a * 8, n * 8 * sizeof(float), cudaMemcpyDeviceToHost, st));
        CB_CUDA(cudaMemcpyAsync(h_pr + a * 8 * CB200_NUM_MOVES, d_pr + a * 8 * CB200_NUM_MOVES,
                                n * 8 * CB200_NUM_MOVES * sizeof(float), cudaMemcpyDeviceToHost, st));
        CB_CUDA(cudaMemcpyAsync(t->h_st_game + a, t->d_st_game + a, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        t->st_copied = total;
      }
    }
    if (pass == 1) break;
    const int Gn = t->P.num_games;
    ++t->st_round;
    k_emit_assign<<<(Gn + 255) / 256, 256, 0, st>>>(t->P, t->d_emitted, t->d_st_ctr, (int)t->st_limit, t->d_st_soff,
                                                     t->st_round);
    CB_LAUNCHED();
    const long long warps = (long long)Gn * kMaxSamples;
    k_write_samples<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(t->P, t->d_st_soff, d_gs, d_ev, d_pr, t->d_emitted,
                                                                 t->st_round, t->d_st_game);
    CB_LAUNCHED();
    CB_CUDA(cudaGetLastError());
    CB_CUDA(cudaMemcpyAsync(t->h_st_ctr, t->d_st_ctr, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaEventRecord(t->st_ev, st));
    t->st_pending = true;
  }
  if (final) CB_CUDA(cudaStreamSynchronize(st));
  return CB200_OK;
}

static int run_persistent(cb200_trainer *t, int max_rounds, int *rounds_done, bool *all_done) {
  cudaStream_t st = t->g_stream[0];
  *rounds_done = 0, *all_done = false;
  TreeParams P = t->P;
  // parking inside the persistent kernels (CB200_PS_YIELD = work budget per round, 0 = off; only
  // while at least CB200_PS_YIELD_MIN_LIVE games are live)
  int ps_yield = 0, ps_yield_min = 512;
  if (const char *e = getenv("CB200_PS_YIELD")) ps_yield = atoi(e);
  if (const char *e = getenv("CB200_PS_YIELD_MIN_LIVE")) ps_yield_min = atoi(e);
  while (*rounds_done < max_rounds) {
    P.yield_budget = t->ps_n >= ps_yield_min ? ps_yield : 0;
    if (t->ps_n == 0) {
      *all_done = true;
      break;
    }
    const int rounds = max_rounds - *rounds_done;
    // deal the games again once half of them have finished (not worth it for the last few)
    int redeal_pct = 50, redeal_min = 64;
    if (const char *e = getenv("CB200_PS_REDEAL_PCT")) redeal_pct = atoi(e);
    if (const char *e = getenv("CB200_PS_REDEAL_MIN")) redeal_min = atoi(e);
    int exit_done = t->ps_n > redeal_min ? (int)((long long)t->ps_n * redeal_pct / 100) : 0x7fffffff;
    if (exit_done < 1) exit_done = 1;
    if (getenv("CB200_PS_NO_REDEAL")) exit_done = 0x7fffffff;
    const int mode = t->nettc[0].mode;  // 0 bf16, 1 fp16, 2 bf16x3 (8 games per CTA only: shared memory)
    const bool wide = t->ps_n > t->ps_ctas * 8;
    if (wide && mode == 2)
      return set_error(CB200_ERR_STATE, "persistent kernel: bf16x3 networks run at most 8 games per SM");
    CB_CUDA(cudaMemsetAsync(t->d_ps_out, 0, 4 * sizeof(int32_t), st));
    int rc;
    {
      ProfScope ps(t, wide ? 5 : 4, st);
      if (mode == 2)
        rc = ps_launch<2, 8>(t, P, rounds, exit_done);
      else if (mode == 1)
        rc = wide ? ps_launch<1, 16>(t, P, rounds, exit_done) : ps_launch<1, 8>(t, P, rounds, exit_done);
      else
        rc = wide ? ps_launch<0, 16>(t, P, rounds, exit_done) : ps_launch<0, 8>(t, P, rounds, exit_done);
    }
    if (rc != CB200_OK) return rc;
    CB_CUDA(cudaMemcpyAsync(t->h_ps_out, t->d_ps_out, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaStreamSynchronize(st));
    if (t->profiling && (rc = prof_drain(t)) != CB200_OK) return rc;
    t->ps_from_lockstep = false;
    t->ps_cur = 1 - t->ps_cur;
    if (t->h_ps_out[1] != 0)
      return set_error(t->h_ps_out[1], "a game overflowed its node arena / path / sample buffer (raise "
                                       "CB200_ARENA_NODES) or reached an impossible state");
    // CTAs stop at different rounds (all games finished / the re-deal trigger): the launch
    // advanced the run by at most out[2] iterations
    const int ran = t->h_ps_out[2];
    *rounds_done += ran;
    t->iterations_done += ran;
    if (t->h_ps_out[0] == 0) {
      t->ps_n = 0;
      *all_done = true;
      break;
    }
    if ((rc = ps_list_games(t)) != CB200_OK) return rc;
    if ((rc = emit_finished(t, false)) != CB200_OK) return rc;
  }
  return CB200_OK;
}

// Fused training-mode loop: every stream group runs [network -> game step] per iteration on its
// own stream; groups never wait for each other, so one slow game (a long re-rooting) only delays
// its own group while the other groups keep the SMs and the tensor cores busy.
static int run_selfplay_groups(cb200_trainer *t, int max_iterations) {
  const int model = 0;
  const bool tc = t->precision[model] == 1;
  const long prs = tc ? 1 : CB200_NUM_MOVES, pcs = tc ? (long)t->cap : 1;
  const int ng = t->n_groups;
  std::vector<char> active(ng, 1);
  // work queued on the default stream (weights, reset) must be visible to the group streams
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  int done_iters = 0, result = 0;
  long long live_games = t->P.num_games;
  auto wall0 = std::chrono::steady_clock::now();
  auto lap_ms = [&wall0]() {
    const auto now = std::chrono::steady_clock::now();
    const double ms = std::chrono::duration<double, std::milli>(now - wall0).count();
    wall0 = now;
    return ms;
  };
  // parking budget (TreeParams::yield_budget): a typical doIteration is ~16 searches x ~3 levels
  // = ~60 units; while many games are live, longer ones (end-game searches that keep hitting
  // terminal nodes) are cut into several launches. Once few games are left nobody gains from
  // parking, and it would only stretch the last games.
  int yield_budget = 96, yield_min_live = 128;
  if (const char *e = getenv("CB200_YIELD")) yield_budget = atoi(e);
  if (const char *e = getenv("CB200_YIELD_MIN_LIVE")) yield_min_live = atoi(e);
  // Persistent tail: once every live game fits on the device at 16 games per SM (and all games
  // have started), the rest of the run happens inside persistent kernels (persistent.cuh).
  // (bf16x3 networks hold hi and lo operand copies in shared memory: 8 games per SM, not 16)
  const bool ps_ok = tc && t->P.spe <= kPsRowsPerGame && !getenv("CB200_NO_PERSISTENT");
  const long long ps_max = (long long)t->ps_ctas * (t->nettc[model].mode == 2 ? 8 : 16);
  long long ps_capacity = ps_max;
  if (const char *e = getenv("CB200_PS_CAPACITY")) ps_capacity = atoll(e);
  if (ps_capacity > ps_max) ps_capacity = ps_max;
  const int stagger_span =
      t->stagger_div > 0 ? (t->P.first_game + t->P.num_games - 1) / t->stagger_div : 0;
  // With several stream groups the network runs in single-tile CTAs of 128 threads (13 K
  // registers) that fit beside five 80-register game-step CTAs, so that one group's network
  // overlaps the other groups' tree work (2-3 % per run).
  const bool overlap = tc && ng > 1 && getenv("CB200_NO_OVERLAP") == nullptr;
  const bool use_lists = getenv("CB200_NO_LIVE_LIST") == nullptr;
  std::vector<int> group_live(ng, -1);  // live games per group at the last host sync (-1 = unknown)
  while (max_iterations <= 0 || done_iters < max_iterations) {
    if (!t->ps_active && ps_ok && live_games <= ps_capacity && t->iterations_done > stagger_span) {
      // evaluate the requests queued by the last lock-step game step, then list the live games
      const int it = t->iterations_done;
      for (int g = 0; g < ng; ++g) {
        if (!active[g]) continue;
        const int gb = t->g_begin[g], ge = t->g_end[g];
        const int row0 = gb * t->P.spe, rows = (ge - gb) * t->P.spe;
        int32_t *ctr = t->d_gctr + g * 8;
        ProfScope ps(t, 2, t->g_stream[g]);
        int rc = launch_mlp_tc(t->nettc[model], t->d_packed + row0, ctr + (it & 1), 0, rows,
                               t->d_eval + row0, t->d_probs + row0, (int)t->cap,
                               ctr + ((it + 1) & 1), t->g_stream[g], true);
        if (rc != CB200_OK) return rc;
      }
      for (int g = 0; g < ng; ++g)
        if (active[g]) CB_CUDA(cudaStreamSynchronize(t->g_stream[g]));
      int rc = ps_list_games(t);
      if (rc != CB200_OK) return rc;
      t->ps_active = true, t->ps_from_lockstep = true;
      t->lockstep_wall_ms += lap_ms();
      if (t->profiling && (rc = prof_mark(t, true)) != CB200_OK) return rc;
    }
    if (t->ps_active) {
      int rounds = 0;
      bool all_done = false;
      const int cap = max_iterations > 0 ? max_iterations - done_iters : (1 << 30);
      lap_ms();
      int rc = run_persistent(t, cap, &rounds, &all_done);
      if (rc != CB200_OK) return rc;
      t->tail_wall_ms += lap_ms();
      done_iters += rounds;
      if (all_done) result = 1;
      break;
    }
    const int yb = live_games >= yield_min_live ? yield_budget : 0;
    int batch = 32;
    if (max_iterations > 0 && max_iterations - done_iters < batch) batch = max_iterations - done_iters;
    // the games of each group that are still live (finished games would leave idle warps
    // behind): rebuilt once per batch on the group's own stream
    for (int g = 0; g < ng && use_lists; ++g) {
      if (!active[g]) continue;
      TreeParams P = t->P;
      P.game_begin = t->g_begin[g], P.game_end = t->g_end[g];
      k_group_live_list<<<1, 32, 0, t->g_stream[g]>>>(P, t->d_live_list, t->d_live_count + g);
      CB_LAUNCHED();
      CB_CUDA(cudaGetLastError());
    }
    for (int i = 0; i < batch; ++i) {
      const int it = t->iterations_done;
      for (int g = 0; g < ng; ++g) {
        if (!active[g]) continue;
        cudaStream_t st = t->g_stream[g];
        const int gb = t->g_begin[g], ge = t->g_end[g];
        const int row0 = gb * t->P.spe, rows = (ge - gb) * t->P.spe;
        int32_t *ctr = t->d_gctr + g * 8;
        int rc;
        {
          ProfScope ps(t, 2, st);
          if (tc)
            rc = launch_mlp_tc(t->nettc[model], t->d_packed + row0, ctr + (it & 1), 0, rows, t->d_eval + row0,
                               t->d_probs + row0, (int)t->cap, ctr + ((it + 1) & 1), st, true, overlap);
          else
            rc = launch_mlp_f32(t->net32[model], t->d_packed + row0, ctr + (it & 1), 0, rows, t->d_eval + row0,
                                t->d_probs + (size_t)row0 * CB200_NUM_MOVES, ctr + ((it + 1) & 1), st, true);
        }
        if (rc != CB200_OK) return rc;
        TreeParams P = t->P;
        P.game_begin = gb, P.game_end = ge, P.group_row0 = row0, P.group_ctr = ctr;
        P.yield_budget = yb;
        int width = ge - gb;  // warps to launch: the group's games, or its live games
        if (use_lists) {
          P.live_list = t->d_live_list, P.live_count = t->d_live_count + g;
          if (group_live[g] >= 0 && group_live[g] < width) width = group_live[g];
        }
        {
          ProfScope ps(t, 3, st);
          const dim3 grid((width + kTreeWarps - 1) / kTreeWarps), block(kTreeWarps * 32);
          if (grid.x > 0) {
            // built for 6 resident CTAs per SM (80 registers): faster than 4, 5, 7 or 8 at 4 096,
            // 8 192 and 32 768 games (profiles/r02_register_budget_final.txt)
            k_iterate<true, 6><<<grid, block, 0, st>>>(P, t->d_eval, t->d_probs, prs, pcs, nullptr, -1, it,
                                                       t->stagger_div);
            CB_LAUNCHED();
          }
        }
        CB_CUDA(cudaGetLastError());
      }
      ++t->iterations_done;
    }
    done_iters += batch;
    for (int g = 0; g < ng; ++g)
      if (active[g])
        CB_CUDA(cudaMemcpyAsync(t->h_gctr + g * 8, t->d_gctr + g * 8, 8 * sizeof(int32_t),
                                cudaMemcpyDeviceToHost, t->g_stream[g]));
    for (int g = 0; g < ng; ++g)
      if (active[g]) CB_CUDA(cudaStreamSynchronize(t->g_stream[g]));
    if (t->profiling) {
      int rc = prof_drain(t);
      if (rc != CB200_OK) return rc;
    }
    const int par = t->iterations_done & 1;
    long long live = 0;
    for (int g = 0; g < ng; ++g) {
      if (!active[g]) continue;
      const int32_t *c = t->h_gctr + g * 8;
      if (c[4] != 0)
        return set_error(c[4], "a game overflowed its node arena / path / sample buffer (raise "
                               "CB200_ARENA_NODES) or reached an impossible state");
      if (c[2 + par] == 0 && c[par] == 0) active[g] = 0;
      group_live[g] = c[2 + par];
      live += c[2 + par];
    }
    live_games = live;
    t->lockstep_wall_ms += lap_ms();
    if (live == 0) {
      result = 1;
      break;
    }
    const int er = emit_finished(t, false);
    if (er != CB200_OK) return er;
  }
  return result;
}

int cb200_trainer_run_selfplay(cb200_trainer *t, int max_iterations, int stagger) {
  int rc = guard(t);
  if (rc) return rc;
  const bool testing = t->P.testing != 0;
  if (t->precision[0] < 0 || (testing && t->precision[1] < 0))
    return set_error(CB200_ERR_STATE, "cb200_trainer_run_selfplay: set weights first");
  const int saved_div = t->stagger_div;
  if (!stagger) t->stagger_div = 0;
  if (!testing) {
    if (t->profiling) {  // counters may have been reset since the last mark
      int64_t c4[4];
      if ((rc = cb200_trainer_counters(t, c4)) != CB200_OK) return rc;
      t->searches_mark = t->searches_now, t->evals_mark = c4[2];
    }
    rc = run_selfplay_groups(t, max_iterations);
    if (rc >= 0 && t->profiling) {
      const int mr = prof_mark(t, !t->ps_active);
      if (mr != CB200_OK) return mr;
    }
    t->stagger_div = saved_div;
    if (rc >= 0) {
      const int lr = drain_logs(t);
      if (lr != CB200_OK) return lr;
    }
    return rc;
  }
  // two-model (gating match) mode. With both networks on the tensor cores (same operand format)
  // and every game resident at <= 16 per SM, the whole match runs in the persistent kernel
  // (persistent.cuh; each game's requests go to the row region of the model that owns its side).
  if ((t->iterations_done == 0 || t->ps_active) && t->precision[0] == 1 && t->precision[1] == 1 &&
      t->nettc[0].mode == t->nettc[1].mode && t->P.spe <= kPsRowsPerGame &&
      t->P.num_games <= t->ps_ctas * (t->nettc[0].mode == 2 ? 8 : 16) && !getenv("CB200_NO_PERSISTENT")) {
    CB_CUDA(cudaStreamSynchronize(cur_stream()));
    if (!t->ps_active) {
      if ((rc = ps_list_games(t)) != CB200_OK) return rc;
      t->ps_active = true, t->ps_from_lockstep = false;
    }
    int rounds = 0;
    bool all_done = false;
    rc = run_persistent(t, max_iterations > 0 ? max_iterations : (1 << 30), &rounds, &all_done);
    t->stagger_div = saved_div;
    if (rc == CB200_OK) rc = drain_logs(t);
    return rc != CB200_OK ? rc : (all_done ? 1 : 0);
  }
  // otherwise: single lock-step group, requests packed per side
  const int n_max = (int)t->cap;
  int done_iters = 0;
  int result = 0;
  while (max_iterations <= 0 || done_iters < max_iterations) {
    int batch = 32;
    if (max_iterations > 0 && max_iterations - done_iters < batch) batch = max_iterations - done_iters;
    for (int i = 0; i < batch && rc == CB200_OK; ++i) {
      for (int tp = 0; tp < 2 && rc == CB200_OK; ++tp) {  // model 0 = "new" serves to_play 0
        rc = scan(t, tp);
        if (rc == CB200_OK) rc = pack(t, tp, nullptr, t->d_packed);
        if (rc == CB200_OK) rc = run_net(t, tp == 0 ? 0 : 1, t->d_packed, t->d_summary, 0, n_max);
        if (rc == CB200_OK) rc = iterate(t, t->d_eval, t->d_probs, tp, t->precision[tp == 0 ? 0 : 1] == 1);
      }
      ++t->iterations_done;
    }
    done_iters += batch;
    if (rc == CB200_OK) rc = scan(t, -1);
    if (rc == CB200_OK) rc = fetch_summary(t);
    if (rc != CB200_OK) break;
    if (t->h_summary[1] == 0) {
      result = 1;
      break;
    }
  }
  t->stagger_div = saved_div;
  if (rc == CB200_OK) rc = drain_logs(t);
  return rc != CB200_OK ? rc : result;
}

int cb200_trainer_dump_tree(cb200_trainer *t, int game, int player, int64_t out[8],
                            uint32_t *words, int cap) {
  int rc = guard(t);
  if (rc) return rc;
  if (game < 0 || game >= t->P.num_games || player < 0 || player > 1)
    return set_error(CB200_ERR_ARG, "bad game/player");
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  int32_t tw[kTreeCtlWords], cw[kCtlWords];
  CB_CUDA(cudaMemcpy(tw, t->P.tree + ((size_t)game * 2 + player) * kTreeCtlWords, sizeof(tw), cudaMemcpyDeviceToHost));
  CB_CUDA(cudaMemcpy(cw, t->P.ctl + (size_t)game * kCtlWords, sizeof(cw), cudaMemcpyDeviceToHost));
  out[0] = tw[TW_HAS_ROOT], out[1] = (uint32_t)tw[TW_USED], out[2] = tw[TW_ROOT_VISITS];
  out[3] = tw[TW_ROOT_RESULT], out[4] = tw[TW_ROOT_ALLV], out[5] = tw[TW_SEARCHES_DONE];
  out[6] = (uint32_t)tw[TW_ROOT_EVAL];
  out[7] = (int64_t)cw[CW_TO_PLAY] | ((int64_t)(uint32_t)tw[TW_ROOT_OFF] << 8);
  const int used = tw[TW_USED];
  if (tw[TW_HAS_ROOT] && words && cap > 0) {
    const int n = used < cap ? used : cap;
    CB_CUDA(cudaMemcpy(words, t->P.arenas + ((size_t)game * 3 + tw[TW_ARENA]) * t->P.arena_words,
                       (size_t)n * 4, cudaMemcpyDeviceToHost));
  }
  return used;
}


// ==============================================================================================
// A device-resident network of the fused tourney (one per model id) and of the analysis. The
// weights stay on the host until the first run that needs them uploads them (the device state may
// not exist when they are set). Same weight layout and precision codes as cb200_trainer_set_weights.
struct ResidentNet {
  std::vector<float> host;
  int precision = -1;  // -1 = no weights set
  bool uploaded = false;
  NetF32 f32;
  NetTC tc;
};

static void resident_net_set(ResidentNet &n, const float *weights, int precision) {
  n.host.assign(weights, weights + kNetWeightFloats);
  n.precision = precision;
  n.uploaded = false;
}

static int resident_net_upload(ResidentNet &n) {
  if (n.uploaded) return CB200_OK;
  // tensor-core operand modes: precision 1 -> bf16, 2 -> fp16, 3 -> bf16x3 (hi + lo operands)
  const int rc = n.precision == 0 ? net_f32_upload(n.f32, n.host.data())
                                  : net_tc_upload(n.tc, n.host.data(), n.precision == 1 ? 0 : (n.precision == 2 ? 1 : 2));
  if (rc == CB200_OK) n.uploaded = true;
  return rc;
}

static void resident_net_free(ResidentNet &n) {
  cudaFree(n.f32.w);
  n.f32.w = nullptr;
  net_tc_free(n.tc);
}

// Evaluate the leaf cstates packed[0 .. t->d_summary[0]) into t's answer buffers on the current
// stream. The answer of row k for move m is then at d_probs[k * prs + m * pcs]: row-major from the
// fp32 kernel, move-major (leading dimension cap + kAnswerSlack) from the tensor-core kernel.
static int resident_net_launch(const ResidentNet &n, cb200_trainer *t, const ulonglong2 *packed, long &prs,
                               long &pcs) {
  if (n.precision == 0) {
    prs = CB200_NUM_MOVES, pcs = 1;
    return launch_mlp_f32(n.f32, packed, t->d_summary, 0, (int)t->cap, t->d_eval, t->d_probs);
  }
  prs = 1, pcs = (long)(t->cap + kAnswerSlack);
  return launch_mlp_tc(n.tc, packed, t->d_summary, 0, (int)t->cap, t->d_eval, t->d_probs,
                       (int)(t->cap + kAnswerSlack));
}

// ==============================================================================================
// Tourney (corintho_ai/cpp/include/tourney.h:12-46) over Match (match.h:33-101); device side in
// match.cuh. The matches share the per-game storage of a trainer created when the first call
// needs the device (all players and matches must have been added by then).
struct cb200_tourney {
  int num_threads = 1;
  std::string log_folder;
  std::map<int, MatchSide> players;
  std::vector<std::pair<int, int>> matches;
  std::vector<char> logging;  // per match (Tourney::addMatch, tourney.cpp:80-96)
  std::vector<std::unique_ptr<std::ofstream>> log_files;  // per logged match; null = not opened
  std::vector<int> log_written;
  cb200_trainer *t = nullptr;
  MatchSide *d_sides = nullptr;
  int32_t *d_pack_offs = nullptr, *d_iter_offs = nullptr;
  // fused mode (cb200_tourney_set_weights / cb200_tourney_run): one device-resident network per
  // model id, evaluated in the first-seen order of the ids like rating/tourney.pyx:112-173
  std::vector<int> model_order;
  std::map<int, ResidentNet> nets;
};

static int tourney_ready_build(cb200_tourney *T, cb200_trainer *t, const std::vector<MatchSide> &sides,
                               int n_log) {
  const int n = (int)T->matches.size();
  int rc = fetch_ctl(t);
  if (rc != CB200_OK) return rc;
  const CState st = start_state();
  for (int g = 0; g < n; ++g) {
    int32_t *c = t->h_ctl.data() + (size_t)g * kCtlWords;
    c[MW_ROOT0] = (int32_t)(uint32_t)st.w0, c[MW_ROOT1] = (int32_t)(uint32_t)(st.w0 >> 32);
    c[MW_ROOT2] = (int32_t)(uint32_t)st.w1, c[MW_ROOT3] = (int32_t)(uint32_t)(st.w1 >> 32);
    c[MW_DEPTH] = 0;
  }
  CB_CUDA(cudaMemcpy(t->P.ctl, t->h_ctl.data(), t->h_ctl.size() * 4, cudaMemcpyHostToDevice));
  if ((rc = dmalloc(&T->d_sides, sides.size())) != CB200_OK ||
      (rc = dmalloc(&T->d_pack_offs, (size_t)n)) != CB200_OK ||
      (rc = dmalloc(&T->d_iter_offs, (size_t)n)) != CB200_OK)
    return rc;
  CB_CUDA(cudaMemcpy(T->d_sides, sides.data(), sides.size() * sizeof(MatchSide), cudaMemcpyHostToDevice));
  if (n_log > 0) {  // the trainer owns (and frees) the log areas
    if ((rc = dmalloc(&t->P.log_buf, (size_t)n_log * kLogMaxMoves * kLogWords)) != CB200_OK ||
        (rc = dmalloc(&t->P.log_count, (size_t)n_log)) != CB200_OK)
      return rc;
    CB_CUDA(cudaMemset(t->P.log_count, 0, (size_t)n_log * sizeof(int32_t)));
  }
  return CB200_OK;
}

static int tourney_ready(cb200_tourney *T) {
  if (!T) return set_error(CB200_ERR_ARG, "null tourney");
  if (T->t) return CB200_OK;
  last_error_ref().clear();
  const int n = (int)T->matches.size();
  if (n == 0) return set_error(CB200_ERR_STATE, "tourney has no matches");
  int max_ms = 1, max_spe = 1;
  std::vector<MatchSide> sides(2 * (size_t)n);
  int n_log = 0;
  T->log_files.clear();
  for (int i = 0; i < n; ++i) {
    const int pid[2] = {T->matches[i].first, T->matches[i].second};
    for (int s = 0; s < 2; ++s) {
      sides[2 * i + s] = T->players[pid[s]];
      sides[2 * i + s].log_slot = -1;
      if (sides[2 * i + s].max_searches > max_ms) max_ms = sides[2 * i + s].max_searches;
      if (sides[2 * i + s].spe > max_spe) max_spe = sides[2 * i + s].spe;
    }
    if (T->logging[i]) {  // log_folder/match_<p1>_<p2>_<index>.txt (tourney.cpp:88-93)
      sides[2 * i].log_slot = n_log++;
      auto f = std::make_unique<std::ofstream>(T->log_folder + "/match_" + std::to_string(pid[0]) + "_" +
                                                   std::to_string(pid[1]) + "_" + std::to_string(i) + ".txt",
                                               std::ofstream::out);
      if (!f->is_open()) f.reset();
      T->log_files.push_back(std::move(f));
    }
  }
  T->log_written.assign(n_log, 0);
  if (max_spe > max_ms) max_ms = max_spe;
  // match seeds = successive draws of a default-seeded std::mt19937 (tourney.h:42, tourney.cpp:86)
  cb200_trainer *t = cb200_trainer_create_shard(n, 0, n, T->log_folder.c_str(), 5489, max_ms, max_spe,
                                                1.0f, 0.25f, 0, 1);
  if (!t) return CB200_ERR_CUDA;
  // the tourney becomes usable (T->t set) only when every buffer exists; a failure on the way
  // releases the partial allocations so that a later call starts over instead of launching
  // kernels with null side / offset pointers
  const int rc = tourney_ready_build(T, t, sides, n_log);
  if (rc != CB200_OK) {
    const std::string msg = last_error_ref();
    cudaFree(T->d_sides), cudaFree(T->d_pack_offs), cudaFree(T->d_iter_offs);
    T->d_sides = nullptr, T->d_pack_offs = nullptr, T->d_iter_offs = nullptr;
    cb200_trainer_destroy(t);
    last_error_ref() = msg;
    return rc;
  }
  T->t = t;
  return CB200_OK;
}

// append the records the matches wrote since the last call to their log files
static int tourney_drain_logs(cb200_tourney *T) {
  const int n_log = (int)T->log_written.size();
  if (n_log == 0) return CB200_OK;
  cb200_trainer *t = T->t;
  t->h_log_count.resize(n_log);
  CB_CUDA(cudaMemcpy(t->h_log_count.data(), t->P.log_count, (size_t)n_log * sizeof(int32_t), cudaMemcpyDeviceToHost));
  for (int g = 0; g < n_log; ++g) {
    const int have = t->h_log_count[g], done = T->log_written[g];
    if (have <= done) continue;
    T->log_written[g] = have;
    if (!T->log_files[g]) continue;
    t->h_log_rec.resize((size_t)(have - done) * kLogWords);
    CB_CUDA(cudaMemcpy(t->h_log_rec.data(), t->P.log_buf + ((size_t)g * kLogMaxMoves + done) * kLogWords,
                       t->h_log_rec.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (int k = 0; k < have - done; ++k)
      format_log_record(*T->log_files[g], t->h_log_rec.data() + (size_t)k * kLogWords);
    T->log_files[g]->flush();
  }
  return CB200_OK;
}

// offsets + summary for one model id; h_summary = {requests, live matches, error, rows read}
static int tourney_scan(cb200_tourney *T, int id) {
  cb200_trainer *t = T->t;
  k_match_scan<<<1, 1024, 0, cur_stream()>>>(t->P, T->d_sides, id, T->d_pack_offs, T->d_iter_offs,
                                         t->d_summary);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  return fetch_summary(t);
}

cb200_tourney *cb200_tourney_create(int num_threads, const char *log_folder) {
  if (num_threads <= 0) {
    set_error(CB200_ERR_ARG, "cb200_tourney_create: num_threads must be positive");
    return nullptr;
  }
  cb200_tourney *T = new cb200_tourney();
  T->num_threads = num_threads;
  T->log_folder = log_folder ? log_folder : "";
  return T;
}

void cb200_tourney_destroy(cb200_tourney *T) {
  if (!T) return;
  cudaFree(T->d_sides), cudaFree(T->d_pack_offs), cudaFree(T->d_iter_offs);
  for (auto &kv : T->nets) resident_net_free(kv.second);
  if (T->t) cb200_trainer_destroy(T->t);
  delete T;
}

int cb200_tourney_add_player(cb200_tourney *T, int player_id, int model_id, int max_searches,
                             int searches_per_eval, float c_puct, float epsilon, int random) {
  if (!T) return set_error(CB200_ERR_ARG, "null tourney");
  if (T->t) return set_error(CB200_ERR_STATE, "players must be added before the first iteration");
  if (!random && (max_searches <= 0 || searches_per_eval <= 0 || searches_per_eval > 64 ||
                  !(c_puct > 0.0f) || !(epsilon >= 0.0f) || !(epsilon <= 1.0f)))
    return set_error(CB200_ERR_ARG, "cb200_tourney_add_player: invalid search parameters");
  MatchSide s;
  s.model_id = model_id, s.max_searches = max_searches > 0 ? max_searches : 1;
  s.spe = searches_per_eval > 0 ? searches_per_eval : 1, s.random = random ? 1 : 0;
  s.c_puct = c_puct, s.epsilon = epsilon, s.player_id = player_id, s.log_slot = -1;
  T->players[player_id] = s;
  if (std::find(T->model_order.begin(), T->model_order.end(), model_id) == T->model_order.end())
    T->model_order.push_back(model_id);
  return CB200_OK;
}

int cb200_tourney_add_match(cb200_tourney *T, int player1, int player2, int logging) {
  if (!T) return set_error(CB200_ERR_ARG, "null tourney");
  if (T->t) return set_error(CB200_ERR_STATE, "matches must be added before the first iteration");
  if (!T->players.count(player1) || !T->players.count(player2))
    return set_error(CB200_ERR_ARG, "cb200_tourney_add_match: unknown player id");
  T->matches.emplace_back(player1, player2);
  T->logging.push_back(logging ? 1 : 0);
  return CB200_OK;
}

int cb200_tourney_all_done(cb200_tourney *T) {
  int rc = tourney_ready(T);
  if (rc) return rc;
  if ((rc = tourney_scan(T, 0x7fffffff)) != CB200_OK) return rc;
  return T->t->h_summary[1] == 0 ? 1 : 0;
}

int cb200_tourney_num_requests(cb200_tourney *T, int id) {
  int rc = tourney_ready(T);
  if (rc) return rc;
  if ((rc = tourney_scan(T, id)) != CB200_OK) return rc;
  return T->t->h_summary[0];
}

int cb200_tourney_write_requests(cb200_tourney *T, float *game_states, int id) {
  int rc = tourney_ready(T);
  if (rc) return rc;
  if (!game_states) return set_error(CB200_ERR_ARG, "null game_states");
  if ((rc = tourney_scan(T, id)) != CB200_OK) return rc;
  cb200_trainer *t = T->t;
  const int n = t->h_summary[0];
  if (n <= 0) return CB200_OK;
  k_match_pack<<<(t->P.num_games + 7) / 8, 256, 0, cur_stream()>>>(t->P, T->d_sides, id,
                                                                 T->d_pack_offs, t->d_rows, nullptr);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  CB_CUDA(cudaMemcpyAsync(game_states, t->d_rows, (size_t)n * CB200_STATE_SIZE * sizeof(float),
                          cudaMemcpyDeviceToHost, cur_stream()));
  CB_CUDA(cudaStreamSynchronize(cur_stream()));
  return CB200_OK;
}

int cb200_tourney_do_iteration(cb200_tourney *T, const float *eval, const float *probs, int rows,
                               int id) {
  int rc = tourney_ready(T);
  if (rc) return rc;
  if ((rc = tourney_scan(T, id)) != CB200_OK) return rc;
  cb200_trainer *t = T->t;
  const int need = t->h_summary[3];  // rows the matches will read (reference offset rule)
  if (need > 0) {
    if (!eval || !probs) return set_error(CB200_ERR_ARG, "requests pending but eval/probs null");
    if (need > rows || (size_t)need > t->cap)
      return set_error(CB200_ERR_ARG, "cb200_tourney_do_iteration: the answer offsets of "
                                      "tourney.cpp:54-62 reach past the caller's buffers");
    CB_CUDA(cudaMemcpyAsync(t->d_eval, eval, (size_t)need * sizeof(float), cudaMemcpyHostToDevice,
                            cur_stream()));
    CB_CUDA(cudaMemcpyAsync(t->d_probs, probs, (size_t)need * CB200_NUM_MOVES * sizeof(float),
                            cudaMemcpyHostToDevice, cur_stream()));
  }
  const int grid = (t->P.num_games + kTreeWarps - 1) / kTreeWarps;
  k_match_iterate<<<grid, kTreeWarps * 32, 0, cur_stream()>>>(t->P, T->d_sides, t->d_eval, t->d_probs,
                                                            T->d_iter_offs, id, CB200_NUM_MOVES, 1);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  if ((rc = tourney_scan(T, id)) != CB200_OK) return rc;
  if (t->h_summary[2] != 0)
    return set_error(t->h_summary[2], "a match overflowed its node arena / path buffer (raise "
                                      "CB200_ARENA_NODES) or reached an impossible state");
  ++t->iterations_done;
  return tourney_drain_logs(T);
}

// ---- fused tourney: the per-model evaluation of rating/tourney.pyx:139-155 on the device ------
int cb200_tourney_set_weights(cb200_tourney *T, int model_id, const float *weights, size_t n_floats,
                              int precision) {
  last_error_ref().clear();
  if (!T) return set_error(CB200_ERR_ARG, "null tourney");
  if (model_id < 0 || !weights || n_floats != kNetWeightFloats || precision < 0 || precision > 3)
    return set_error(CB200_ERR_ARG, "cb200_tourney_set_weights: bad arguments (model id >= 0, 127997 floats, "
                                    "precision 0|1|2|3)");
  resident_net_set(T->nets[model_id], weights, precision);
  return CB200_OK;
}

int cb200_tourney_run(cb200_tourney *T, int max_rounds) {
  int rc = tourney_ready(T);
  if (rc) return rc;
  cb200_trainer *t = T->t;
  if ((rc = guard(t)) != CB200_OK) return rc;
  for (int id : T->model_order) {
    if (id < 0) continue;  // random players: no network (tourney.pyx feeds them no evaluation)
    auto it = T->nets.find(id);
    if (it == T->nets.end() || it->second.precision < 0)
      return set_error(CB200_ERR_STATE, "cb200_tourney_run: no weights set for model " + std::to_string(id));
    if ((rc = resident_net_upload(it->second)) != CB200_OK) return rc;
  }
  cudaStream_t st = cur_stream();
  const int grid = (t->P.num_games + kTreeWarps - 1) / kTreeWarps;
  int rounds = 0;
  for (;;) {
    // all_done() check (tourney.pyx:118) every few rounds: one small read-back
    k_match_scan<<<1, 1024, 0, st>>>(t->P, T->d_sides, 0x7fffffff, T->d_pack_offs, T->d_iter_offs, t->d_summary);
    CB_LAUNCHED();
    CB_CUDA(cudaGetLastError());
    if ((rc = fetch_summary(t)) != CB200_OK) return rc;
    if (t->h_summary[1] == 0) return tourney_drain_logs(T) != CB200_OK ? CB200_ERR_CUDA : 1;
    if (max_rounds > 0 && rounds >= max_rounds) break;
    int batch = 8;
    if (max_rounds > 0 && max_rounds - rounds < batch) batch = max_rounds - rounds;
    for (int r = 0; r < batch; ++r) {
      for (int id : T->model_order) {
        // offsets of both kinds + request count of this model (summary[0], read by the network)
        k_match_scan<<<1, 1024, 0, st>>>(t->P, T->d_sides, id, T->d_pack_offs, T->d_iter_offs, t->d_summary);
        CB_LAUNCHED();
        long prs = CB200_NUM_MOVES, pcs = 1;
        if (id >= 0) {
          k_match_pack<<<(t->P.num_games + 7) / 8, 256, 0, st>>>(t->P, T->d_sides, id, T->d_pack_offs, nullptr,
                                                                 t->d_packed);
          CB_LAUNCHED();
          if ((rc = resident_net_launch(T->nets[id], t, t->d_packed, prs, pcs)) != CB200_OK) return rc;
        }
        k_match_iterate<<<grid, kTreeWarps * 32, 0, st>>>(t->P, T->d_sides, t->d_eval, t->d_probs, T->d_iter_offs,
                                                          id, prs, pcs);
        CB_LAUNCHED();
        CB_CUDA(cudaGetLastError());
      }
      ++t->iterations_done;
    }
    rounds += batch;
  }
  rc = tourney_drain_logs(T);
  return rc != CB200_OK ? rc : 0;
}

// Tourney::writeScores (tourney.cpp:34-42): "<player1> <player2> <score>" per finished match
int cb200_tourney_write_scores(cb200_tourney *T, const char *file) {
  int rc = tourney_ready(T);
  if (rc) return rc;
  if (!file) return set_error(CB200_ERR_ARG, "null file name");
  cb200_trainer *t = T->t;
  if ((rc = fetch_ctl(t)) != CB200_OK) return rc;
  std::ofstream f(file, std::ofstream::out);
  if (!f) return set_error(CB200_ERR_ARG, std::string("cannot open ") + file);
  for (int g = 0; g < t->P.num_games; ++g) {
    const int32_t *c = t->h_ctl.data() + (size_t)g * kCtlWords;
    if (!c[CW_DONE]) continue;
    f << T->matches[g].first << ' ' << T->matches[g].second << ' ' << game_score(c[CW_RESULT]) << '\n';
  }
  return CB200_OK;
}

int cb200_tourney_counters(cb200_tourney *T, int64_t out[4]) {
  int rc = tourney_ready(T);
  if (rc) return rc;
  return cb200_trainer_counters(T->t, out);
}

// ==============================================================================================
// Analysis (the reference's DockerMC, dockermc.cpp, for a batch of given positions); device side
// in analysis.cuh. The positions use the per-game storage of an internal testing-mode trainer, one
// "game" per position, created with the analysis object; every run re-seeds and resets it.

// The structural invariants of a cstate that the engine accepts from a caller (checked over the
// reachable positions of 1 000 000 random play-outs by tests/test_oracle_analysis.py): side to move
// 0 or 1, byte 7 zero, at most 4 pieces of a kind in a hand, frozen squares occupied, and every
// piece of a kind either on the board or in a hand (8 of each kind).
static bool valid_state(uint64_t w0, uint64_t w1) {
  if (((w1 >> 48) & 0xff) > 1 || (w1 >> 56) != 0) return false;
  const uint32_t base = (uint32_t)(w0 & 0xffff), column = (uint32_t)((w0 >> 16) & 0xffff);
  const uint32_t capital = (uint32_t)((w0 >> 32) & 0xffff), frozen = (uint32_t)(w0 >> 48);
  if (frozen & ~(base | column | capital)) return false;
  const uint32_t plane[3] = {base, column, capital};
  for (int t = 0; t < 3; ++t) {
    const int h0 = (int)((w1 >> (8 * t)) & 0xff), h1 = (int)((w1 >> (8 * (3 + t))) & 0xff);
    if (h0 > 4 || h1 > 4 || __builtin_popcount(plane[t]) != 8 - h0 - h1) return false;
  }
  return true;
}

int64_t cb200_check_states(int64_t n, const uint64_t *states, uint8_t *valid) {
  if (n < 0 || (n > 0 && !states)) return set_error(CB200_ERR_ARG, "cb200_check_states: bad arguments");
  int64_t bad = 0;
  for (int64_t i = 0; i < n; ++i) {
    const bool ok = valid_state(states[2 * i], states[2 * i + 1]);
    if (valid) valid[i] = ok ? 1 : 0;
    bad += ok ? 0 : 1;
  }
  return bad;
}

struct cb200_analysis {
  int max_positions = 0, max_searches = 0;
  cb200_trainer *t = nullptr;  // trainer max_searches = max(max_searches, spe): it sizes the arenas only
  ulonglong2 *d_roots = nullptr;   // [max_positions] the positions of the current run
  int32_t *d_moves = nullptr, *d_results = nullptr, *d_visits = nullptr;
  float *d_values = nullptr, *d_evals = nullptr;
  ResidentNet net;
  int64_t counters[2] = {0, 0};    // {simulations, leaf evaluations} of the last run
};

cb200_analysis *cb200_analysis_create(int max_positions, int max_searches, int searches_per_eval, float c_puct,
                                      float epsilon) {
  last_error_ref().clear();
  // the validation of cb200_tourney_add_player
  if (max_positions <= 0 || max_searches <= 0 || searches_per_eval <= 0 || searches_per_eval > 64 ||
      !(c_puct > 0.0f) || !(epsilon >= 0.0f) || !(epsilon <= 1.0f)) {
    set_error(CB200_ERR_ARG, "cb200_analysis_create: invalid argument");
    return nullptr;
  }
  cb200_trainer *t = cb200_trainer_create_shard(max_positions, 0, max_positions, "", 0,
                                                std::max(max_searches, searches_per_eval), searches_per_eval,
                                                c_puct, epsilon, 0, 1);
  if (!t) return nullptr;
  cb200_analysis *A = new cb200_analysis();
  A->max_positions = max_positions, A->max_searches = max_searches, A->t = t;
  const size_t n = (size_t)max_positions;
  if (dmalloc(&A->d_roots, n) != CB200_OK || dmalloc(&A->d_moves, n) != CB200_OK ||
      dmalloc(&A->d_results, n) != CB200_OK || dmalloc(&A->d_values, n) != CB200_OK ||
      dmalloc(&A->d_visits, n * CB200_NUM_MOVES) != CB200_OK ||
      dmalloc(&A->d_evals, n * CB200_NUM_MOVES) != CB200_OK) {
    const std::string msg = last_error_ref();
    cb200_analysis_destroy(A);
    last_error_ref() = msg;
    return nullptr;
  }
  return A;
}

void cb200_analysis_destroy(cb200_analysis *A) {
  if (!A) return;
  if (A->t) cudaSetDevice(A->t->device);
  cudaFree(A->d_roots), cudaFree(A->d_moves), cudaFree(A->d_results), cudaFree(A->d_values);
  cudaFree(A->d_visits), cudaFree(A->d_evals);
  resident_net_free(A->net);
  if (A->t) cb200_trainer_destroy(A->t);
  delete A;
}

int cb200_analysis_set_weights(cb200_analysis *A, const float *weights, size_t n_floats, int precision) {
  last_error_ref().clear();
  if (!A) return set_error(CB200_ERR_ARG, "null analysis");
  if (!weights || n_floats != kNetWeightFloats || precision < 0 || precision > 3)
    return set_error(CB200_ERR_ARG, "cb200_analysis_set_weights: bad arguments (127997 floats, precision 0|1|2|3)");
  resident_net_set(A->net, weights, precision);
  return CB200_OK;
}

int cb200_analysis_run(cb200_analysis *A, int n, const uint64_t *states, int seed, int32_t *moves,
                       int32_t *results, float *values, int32_t *visits, float *evals) {
  last_error_ref().clear();
  if (!A) return set_error(CB200_ERR_ARG, "null analysis");
  if (n <= 0 || n > A->max_positions)
    return set_error(CB200_ERR_ARG, "cb200_analysis_run: n must be in [1, max_positions]");
  if (!states || !moves || !results || !values || !visits)
    return set_error(CB200_ERR_ARG, "cb200_analysis_run: null states / moves / results / values / visits");
  for (int i = 0; i < n; ++i)
    if (!valid_state(states[2 * i], states[2 * i + 1]))
      return set_error(CB200_ERR_ARG, "cb200_analysis_run: state " + std::to_string(i) + " is not a valid cstate");
  if (A->net.precision < 0) return set_error(CB200_ERR_STATE, "cb200_analysis_run: no weights set");
  cb200_trainer *t = A->t;
  int rc = guard(t);
  if (rc != CB200_OK) return rc;
  if ((rc = resident_net_upload(A->net)) != CB200_OK) return rc;
  A->counters[0] = A->counters[1] = 0;
  // positions [0, n) become games [0, n) of the trainer: seeds = outputs 0 .. n-1 of mt19937(seed),
  // fresh control blocks and trees (the kernel builds each root on its first round)
  t->P.num_games = n;
  if ((rc = cb200_trainer_reset(t, seed)) != CB200_OK) return rc;
  cudaStream_t st = cur_stream();
  CB_CUDA(cudaMemcpyAsync(A->d_roots, states, (size_t)n * sizeof(ulonglong2), cudaMemcpyHostToDevice, st));
  const AnalysisOut out{A->d_moves, A->d_results, A->d_values, A->d_visits, evals ? A->d_evals : nullptr};
  const int grid = (n + kTreeWarps - 1) / kTreeWarps;
  // every round completes at least one search or the turn of each live position
  const int max_rounds = A->max_searches + 8;
  for (int round = 0;; ++round) {
    // request offsets of every live position (contiguous packing) and the live count
    k_scan_requests<<<1, 1024, 0, st>>>(t->P, -1, t->d_offs, t->d_summary);
    CB_LAUNCHED();
    if (round % 8 == 0) {  // one small read-back every few rounds
      if ((rc = fetch_summary(t)) != CB200_OK) return rc;
      if (t->h_summary[1] == 0) break;
      if (round > max_rounds) return set_error(CB200_ERR_STATE, "cb200_analysis_run: the searches did not finish");
    }
    k_pack_requests<<<(n + 7) / 8, 256, 0, st>>>(t->P, -1, t->d_offs, nullptr, t->d_packed);
    CB_LAUNCHED();
    long prs = 0, pcs = 0;
    if ((rc = resident_net_launch(A->net, t, t->d_packed, prs, pcs)) != CB200_OK) return rc;
    k_analysis_iterate<<<grid, kTreeWarps * 32, 0, st>>>(t->P, A->max_searches, A->d_roots, t->d_eval,
                                                          t->d_probs, prs, pcs, t->d_offs, out);
    CB_LAUNCHED();
    CB_CUDA(cudaGetLastError());
    ++t->iterations_done;
  }
  CB_CUDA(cudaMemcpyAsync(moves, A->d_moves, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CB_CUDA(cudaMemcpyAsync(results, A->d_results, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CB_CUDA(cudaMemcpyAsync(values, A->d_values, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, st));
  CB_CUDA(cudaMemcpyAsync(visits, A->d_visits, (size_t)n * CB200_NUM_MOVES * sizeof(int32_t),
                          cudaMemcpyDeviceToHost, st));
  if (evals)
    CB_CUDA(cudaMemcpyAsync(evals, A->d_evals, (size_t)n * CB200_NUM_MOVES * sizeof(float),
                            cudaMemcpyDeviceToHost, st));
  int64_t c4[4];
  if ((rc = cb200_trainer_counters(t, c4)) != CB200_OK) return rc;  // synchronises the stream
  A->counters[0] = c4[0], A->counters[1] = c4[2];
  return CB200_OK;
}

int cb200_analysis_counters(cb200_analysis *A, int64_t out[2]) {
  last_error_ref().clear();
  if (!A || !out) return set_error(CB200_ERR_ARG, "null analysis / out");
  out[0] = A->counters[0], out[1] = A->counters[1];
  return CB200_OK;
}

}  // extern "C"
