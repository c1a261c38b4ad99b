// Test harness for the tree search's arithmetic (tests/test_gpu_tree_kernels.py): puct_u and
// puct_bounds one thread per slot, fast_rcp over an array, select_slot one warp per constructed
// node record, and receive_eval on one constructed game, so that tests reach the exact pass, the
// n > 64 branch and degenerate evaluator outputs that self-play almost never produces.
#include <cmath>
#include <vector>

#include "../corintho_ai_b200/csrc/tree.cuh"

using namespace cb200;

namespace {

__global__ void k_puct(int n, const uint4 *slots, const float *den, const float *vs, float *u, float *lo,
                       float *hi, int *inexact, int *divided) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  bool dv;
  u[i] = puct_u(slots[i], den[i], vs[i], dv);
  divided[i] = dv ? 1 : 0;
  inexact[i] = puct_bounds(slots[i], den[i], vs[i], lo[i], hi[i]) ? 1 : 0;
}

__global__ void k_rcp(long n, const double *x, double *r) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    r[i] = fast_rcp(x[i]);
}

// iota variant: r[i] = fast_rcp(first + i), so that a range of 2^24 integers needs no input array
__global__ void k_rcp_iota(long n, double first, double *r) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    r[i] = fast_rcp(first + (double)i);
}

// one warp per case: the slots of record words + off[k] are loaded as search() loads them
__global__ void k_select(int ncase, const uint32_t *words, const int *off, const int *visits, const float *c_puct,
                         const float *const *tables, int *choice, int *exact) {
  const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (k >= ncase) return;
  Ctx c;
  TreeParams P;
  P.c_puct = c_puct[k];
  P.vsqrt = tables[k];
  const uint32_t *r = words + off[k];
  const int n = (int)(r[4] & 0xffu);
  constexpr int kS = 2;
  const uint4 zero4 = make_uint4(0, 0, 0, kS3Has | kS3Allv);
  uint4 s[kS];
#pragma unroll
  for (int j = 0; j < kS; ++j) s[j] = c.lane + 32 * j < n ? ld4(r + 8 + 4 * (c.lane + 32 * j)) : zero4;
  bool none, ex;
  const int e = select_slot(c, P, r, s, n, __uint_as_float(r[5]), visits[k], none, ex);
  if (c.lane == 0) choice[k] = none ? -1 : e, exact[k] = ex ? 1 : 0;
}

// one warp, one game: receive_eval with the pending records, evaluations and probabilities given
__global__ void k_ingest(uint32_t *arena, uint32_t *pending, int n_pending, const float *eval, const float *probs,
                         long prs, long pcs, uint32_t *mt, int *state, float *root_eval, float epsilon) {
  __shared__ WarpSm sm;
  Ctx c;
  TreeParams P;
  P.epsilon = epsilon;
  c.n_pending = n_pending;
  c.pending = pending;
  c.base = arena;
  c.mt = mt;
  c.mt_idx = state[0];
  c.root_eval = *root_eval;
  c.root_allv = 1;
  c.error = 0;
  c.d_evals = 0;
  receive_eval(c, P, sm, eval, probs, prs, pcs);
  if (c.lane == 0) state[0] = c.mt_idx, state[1] = c.error, *root_eval = c.root_eval;
}

// device allocations of one entry point, freed on every return path
struct DevAllocs {
  std::vector<void *> ptrs;
  ~DevAllocs() {
    for (void *p : ptrs) cudaFree(p);
  }
  template <class T>
  int alloc(T **d, size_t n) {
    *d = nullptr;
    CB_CUDA(cudaMalloc((void **)d, (n ? n : 1) * sizeof(T)));
    ptrs.push_back((void *)*d);
    return CB200_OK;
  }
  template <class T>
  int upload(T **d, const T *h, size_t n) {
    const int rc = alloc(d, n);
    if (rc != CB200_OK) return rc;
    if (n) CB_CUDA(cudaMemcpy((void *)*d, h, n * sizeof(T), cudaMemcpyHostToDevice));
    return CB200_OK;
  }
};
template <class T>
int download(T *h, const T *d, size_t n) {
  if (n) CB_CUDA(cudaMemcpy(h, d, n * sizeof(T), cudaMemcpyDeviceToHost));
  return CB200_OK;
}
int finish(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return set_error(CB200_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  return CB200_OK;
}
#define TK_TRY(expr)                     \
  do {                                   \
    const int _rc = (expr);              \
    if (_rc != CB200_OK) return _rc;     \
  } while (0)
}  // namespace

extern "C" {

const char *tk_last_error() { return last_error_ref().c_str(); }

// slots [n][4] words, den / vs [n] -> u, lo, hi [n], inexact [n] (puct_bounds' interval is not a
// single point), divided [n] (puct_u took the two IEEE divisions)
int tk_puct(int n, const uint32_t *slots, const float *den, const float *vs, float *u, float *lo, float *hi,
            int *inexact, int *divided) {
  DevAllocs g;
  uint4 *d_s;
  float *d_den, *d_vs, *d_out;
  int *d_in;
  TK_TRY(g.upload(&d_s, reinterpret_cast<const uint4 *>(slots), n));
  TK_TRY(g.upload(&d_den, den, n));
  TK_TRY(g.upload(&d_vs, vs, n));
  TK_TRY(g.alloc(&d_out, 3 * (size_t)n));
  TK_TRY(g.alloc(&d_in, 2 * (size_t)n));
  k_puct<<<(n + 127) / 128 + 1, 128>>>(n, d_s, d_den, d_vs, d_out, d_out + n, d_out + 2 * n, d_in, d_in + n);
  TK_TRY(finish("tk_puct"));
  TK_TRY(download(u, d_out, n));
  TK_TRY(download(lo, d_out + n, n));
  TK_TRY(download(hi, d_out + 2 * n, n));
  TK_TRY(download(inexact, d_in, n));
  TK_TRY(download(divided, d_in + n, n));
  return CB200_OK;
}

// r[i] = fast_rcp(x[i]); with x == null, r[i] = fast_rcp(first + i)
int tk_rcp(long n, const double *x, double first, double *r) {
  DevAllocs g;
  double *d_x, *d_r;
  TK_TRY(g.alloc(&d_r, n));
  if (x) {
    TK_TRY(g.upload(&d_x, x, n));
    k_rcp<<<1184, 256>>>(n, d_x, d_r);
  } else {
    k_rcp_iota<<<1184, 256>>>(n, first, d_r);
  }
  TK_TRY(finish("tk_rcp"));
  TK_TRY(download(r, d_r, n));
  return CB200_OK;
}

// ncase node records in words [nwords], case k at word off[k]; table[k] != 0: the c_puct * sqrt
// table of the engine (filled with the host expression of cb200_trainer_create) for c_puct[k].
// choice[k] = the selected slot or -1, exact[k] = the level went to the exact pass.
int tk_select(int ncase, const uint32_t *words, long nwords, const int *off, const int *visits,
              const float *c_puct, const int *table, int *choice, int *exact) {
  DevAllocs g;
  uint32_t *d_w;
  int *d_off, *d_vis, *d_out;
  float *d_c, *d_tab;
  const float **d_tp;
  std::vector<float> tab((size_t)ncase * kVsqrtCap);
  for (int k = 0; k < ncase; ++k)
    for (int i = 0; i < kVsqrtCap; ++i)
      tab[(size_t)k * kVsqrtCap + i] = (float)((double)c_puct[k] * sqrt((double)(float)i));
  TK_TRY(g.upload(&d_w, words, nwords));
  TK_TRY(g.upload(&d_off, off, ncase));
  TK_TRY(g.upload(&d_vis, visits, ncase));
  TK_TRY(g.upload(&d_c, c_puct, ncase));
  TK_TRY(g.upload(&d_tab, tab.data(), tab.size()));
  std::vector<const float *> tp(ncase);
  for (int k = 0; k < ncase; ++k) tp[k] = table[k] ? d_tab + (size_t)k * kVsqrtCap : nullptr;
  TK_TRY(g.upload(&d_tp, tp.data(), ncase));
  TK_TRY(g.alloc(&d_out, 2 * (size_t)ncase));
  k_select<<<(ncase + 3) / 4, 128>>>(ncase, d_w, d_off, d_vis, d_c, d_tp, d_out, d_out + ncase);
  TK_TRY(finish("tk_select"));
  TK_TRY(download(choice, d_out, ncase));
  TK_TRY(download(exact, d_out + ncase, ncase));
  return CB200_OK;
}

// One game's receive_eval. arena [nwords] and pending [n_pending][kPendWords] (leaf offset, path
// length | n_legal << 8, path) as search() writes them; probs element (row k, move m) =
// probs[k * prs + m * pcs] over nprobs floats. arena, mt [624], state {mt_idx, error} and
// root_eval are updated in place.
int tk_ingest(uint32_t *arena, long nwords, const uint32_t *pending, int n_pending, const float *eval,
              const float *probs, long nprobs, long prs, long pcs, uint32_t *mt, int *state, float *root_eval,
              float epsilon) {
  // this module's own gamma table: ensure_tables() keeps its "done" flag in an inline function's
  // static, which the dynamic linker shares with libcorintho_b200.so once both are loaded
  CB_CUDA(cudaMemcpyToSymbol(d_gamma, kCGammaBits, sizeof(kCGammaBits)));
  DevAllocs g;
  uint32_t *d_a, *d_p, *d_mt;
  float *d_e, *d_pr, *d_re;
  int *d_st;
  TK_TRY(g.upload(&d_a, (const uint32_t *)arena, nwords));
  TK_TRY(g.upload(&d_p, pending, (size_t)n_pending * kPendWords));
  TK_TRY(g.upload(&d_e, eval, n_pending));
  TK_TRY(g.upload(&d_pr, probs, nprobs));
  TK_TRY(g.upload(&d_mt, (const uint32_t *)mt, 624));
  TK_TRY(g.upload(&d_st, (const int *)state, 2));
  TK_TRY(g.upload(&d_re, (const float *)root_eval, 1));
  k_ingest<<<1, 32>>>(d_a, d_p, n_pending, d_e, d_pr, prs, pcs, d_mt, d_st, d_re, epsilon);
  TK_TRY(finish("tk_ingest"));
  TK_TRY(download(arena, d_a, nwords));
  TK_TRY(download(mt, d_mt, 624));
  TK_TRY(download(state, d_st, 2));
  TK_TRY(download(root_eval, d_re, 1));
  return CB200_OK;
}

}  // extern "C"
