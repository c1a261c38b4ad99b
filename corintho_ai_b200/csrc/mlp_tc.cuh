// K5 (tensor-core variant): the policy/value network on tcgen05 with TMEM accumulators.
// Architecture = corintho_ai/python/wrapper.py:256-271 (BatchNorm folded by the caller):
// 70 -> 12 x [Dense 100, ReLU] -> {tanh value, softmax 96 policy}; replaces the Keras predict
// call of the reference loop (corintho_ai/python/main.pyx:70-83).
//
// One CTA (256 threads = 2 warpgroups) pushes TWO tiles of 128 positions through all 13
// layers without touching HBM in between:
//   * A operand (activations, bf16) lives in shared memory in the UMMA canonical K-major
//     no-swizzle layout: 16-byte k-chunks (8 bf16) of all 128 rows are contiguous
//     (chunk stride 2048 B = LBO, 8-row core-matrix stride 128 B = SBO);
//   * B operand (weights of one layer, bf16, [N=112][K=112] K-major, same canonical layout
//     with chunk stride 1792 B, bias rows included) is ONE 24.5 KB image per layer, fetched by
//     a single cp.async.bulk (UBLKCP) per layer into a double buffer, mbarrier-tracked;
//   * D (fp32) lives in TMEM: 112 columns per tile, 7 x tcgen05.mma (M128 N112 K16) per layer,
//     issued by one thread per warpgroup and committed to an mbarrier;
//   * epilogue: batched tcgen05.ld (32 lanes x 32 columns) -> ReLU + bf16 pack -> written straight
//     back as the next layer's A operand. Input encoding (game.cpp:45-58) is expanded from
//     the packed cstate inside the kernel; tanh / softmax are done from TMEM in the last layer.
// All dimensions are padded with zeros: K 70/100 -> 112, N 100/97 -> 112.
// The bias rides in the GEMM: activation columns 100 and 101 are constant 1 (kept alive through
// the layers by unit weights), and weight rows 100/101 hold the bias split into bf16 hi + lo
// parts (~16 significant bits), so the hidden epilogue is just ReLU + bf16 packing
// (cvt.rn.relu.bf16x2.f32) on batched TMEM loads.
//
// Operand modes (template parameter kMode): 0 = bf16, 1 = fp16, 2 = "bf16x3": activations and
// weights are both carried as a bf16 hi + lo pair (16 significant bits) and every k-step issues
// three MMAs into the same accumulator (a_hi*w_hi + a_hi*w_lo + a_lo*w_hi; the lo*lo term is
// below fp32 round-off). Trained checkpoints need it: their folded BatchNorm scales make the
// outputs so sensitive to operand rounding that single bf16 / fp16 operands miss the 2e-2 bar
// (value error up to 0.24 / 0.033), while bf16x3 stays below 1e-3 (tests/test_gpu_net.py).
#ifndef CORINTHO_B200_MLP_TC_CUH
#define CORINTHO_B200_MLP_TC_CUH

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstring>
#include <vector>

#include "common.cuh"

namespace cb200 {

constexpr int kTcLayers = 13;
constexpr int kTcN = 112;                                // padded out features
constexpr int kTcChunks = 14;                            // padded in features / 8
constexpr int kTcAChunkBytes = 128 * 16;                 // 2048: one k-chunk of 128 rows
constexpr int kTcWChunkBytes = kTcN * 16;                // 1792: one k-chunk of 112 rows
constexpr int kTcABytes = kTcChunks * kTcAChunkBytes;    // 28672
constexpr int kTcWBytes = kTcChunks * kTcWChunkBytes;    // 25088
constexpr int kTcLayerBytes = kTcWBytes;                 // 25088 (bias folded into rows 100/101)
constexpr int kTcOnes = 100;                             // activation columns 100,101 == 1
constexpr int kTcThreads = 256;
constexpr int kTcTmemCols = 256;                         // 2 tiles x 128 columns
// shared memory of a network CTA: `tiles` activation tiles (128 positions each) and two weight
// buffers, everything in `parts` copies (bf16x3: hi and lo), four mbarriers, the TMEM slot
__host__ __device__ constexpr size_t tc_smem_bytes(int tiles, int parts) {
  return (size_t)tiles * parts * kTcABytes + 2 * (size_t)parts * kTcLayerBytes + 64;
}
constexpr size_t kTcSmemBytes = tc_smem_bytes(2, 1);    // 107 584
constexpr size_t kTcSmemBytesX3 = tc_smem_bytes(2, 2);  // 215 104
// instruction descriptor (cute/arch/mma_sm100_desc.hpp InstrDescriptor): D=F32 (bits 4-5 = 1),
// A=B=BF16 (bits 7-9, 10-12 = 1), both K-major, N>>3 at bit 17, M>>4 at bit 24
constexpr uint32_t kTcIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kTcN >> 3) << 17) |
                              ((uint32_t)(128 >> 4) << 24);
// same with A = B = F16 (format code 0): 8x finer mantissa than bf16, range +-65504 -- needed for
// trained checkpoints whose folded BatchNorm scales make the network sensitive to operand rounding
constexpr uint32_t kTcIdescF16 = (1u << 4) | ((uint32_t)(kTcN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

struct NetTC {
  void *w = nullptr;  // device: kTcLayers images of kTcLayerBytes (mode 2: hi image + lo image each)
  bool ready = false;
  bool fp16 = false;  // operand format of the images: false = bf16, true = fp16
  int mode = 0;       // 0 bf16, 1 fp16, 2 bf16x3 (hi + lo operands, three MMAs per k-step)
  size_t w_bytes = 0;
};

// ---- raw PTX helpers -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes,
                                         uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor), K-major,
// SWIZZLE_NONE: start>>4 [0,14), LBO>>4 [16,30) = k-chunk stride, SBO>>4 [32,46) = 8-row group
// stride, version 1 at [46,48)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t v[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t v[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t v[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
// tcgen05.wait::ld that also "touches" the 16 destination registers of the load it completes, so
// that the compiler cannot move their first use above the wait
__device__ __forceinline__ void tmem_wait_ld16(uint32_t v[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]),
                 "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]),
                 "+r"(v[14]), "+r"(v[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t v[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
      "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
      "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]),
      "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),
      "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t v[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
      "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// two fp32 -> packed 16-bit pair (bf16 or fp16) with ReLU, `lo` in bits 0-15. fp16 saturates at
// +-65504: a plain round would give inf past it, and the next layer's inf * 0 would put NaN into
// every output.
template <bool kFp16>
__device__ __forceinline__ uint32_t relu_pack16(uint32_t lo, uint32_t hi) {
  uint32_t d;
  if (kFp16)
    asm("cvt.rn.satfinite.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(__uint_as_float(hi)), "f"(__uint_as_float(lo)));
  else
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(__uint_as_float(hi)), "f"(__uint_as_float(lo)));
  return d;
}
template <bool kFp16>
__device__ __forceinline__ uint32_t pack16(float a, float b) {
  if (kFp16) {  // saturating like relu_pack16
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
  }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t *>(&h);
}

// Barrier of the 256 threads that run the network (named barrier 1, so that a larger CTA can keep
// its other warps out of it; in k_mlp_tc it is the whole CTA).
__device__ __forceinline__ void tc_sync(int nthreads) {
  asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// Per-CTA state of the tensor-core network: barriers, TMEM allocation and the phase counters of
// the mbarriers, so that tc_forward() can be called any number of times between tc_setup() and
// tc_teardown() (once per tile pair in k_mlp_tc, once per round in the persistent self-play kernel).
struct TcState {
  uint8_t *sA, *sW;
  uint32_t wbar0, mbar0, tmem_base;
  int nthreads;        // threads running the network: 256 (two tiles) or 128 (one tile)
  int parts;           // operand copies in shared memory: 1, or 2 (hi + lo) in bf16x3 mode
  uint32_t tmem_cols;  // 128 TMEM columns per tile
  uint32_t wcount[2];  // completed waits per weight buffer
  uint32_t mcount;     // completed waits on this warpgroup's MMA barrier
};
constexpr size_t kTcStateSmemBytes = kTcSmemBytes;  // sA[2] | sW[2] | 4 mbarriers | tmem slot

__device__ __forceinline__ void tc_setup(TcState &S, uint8_t *smem, int nthreads = kTcThreads,
                                         int parts = 1) {
  S.nthreads = nthreads;
  S.parts = parts;
  S.tmem_cols = nthreads == kTcThreads ? kTcTmemCols : kTcTmemCols / 2;
  const int tiles = nthreads / 128;
  S.sA = smem;                                 // tiles x parts x kTcABytes
  S.sW = smem + tiles * parts * kTcABytes;     // 2 buffers x parts x kTcLayerBytes
  uint64_t *bars = reinterpret_cast<uint64_t *>(S.sW + 2 * parts * kTcLayerBytes);  // wbar[2], mbar[2]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 4);
  const int t = threadIdx.x, warp = t >> 5;
  S.wbar0 = smem_u32(bars), S.mbar0 = smem_u32(bars + 2);
  if (t == 0) {
    mbar_init(S.wbar0, 1), mbar_init(S.wbar0 + 8, 1);
    mbar_init(S.mbar0, 1), mbar_init(S.mbar0 + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"(S.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  tc_sync(S.nthreads);
  tc_fence_after();
  S.tmem_base = *tmem_slot;
  S.wcount[0] = S.wcount[1] = 0;
  S.mcount = 0;
}

__device__ __forceinline__ void tc_teardown(TcState &S) {
  tc_fence_before();
  tc_sync(S.nthreads);
  if ((threadIdx.x >> 5) == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(S.tmem_base),
                 "r"(S.tmem_cols)
                 : "memory");
  }
}

// One pair of 128-position tiles (positions [pair * 256, pair * 256 + 256) of `states`, n valid
// positions in total) through all 13 layers. Called by all 256 threads of the CTA.
// kMode: 0 bf16, 1 fp16, 2 bf16x3 operands (see the file header).
template <int kMode>
__device__ __forceinline__ void tc_forward(TcState &S, const uint8_t *__restrict__ W,
                                           const ulonglong2 *__restrict__ states, int n, int pair,
                                           float *__restrict__ eval, float *__restrict__ probs,
                                           int probs_ld) {
  constexpr bool kFp16 = kMode == 1;
  constexpr int kParts = kMode == 2 ? 2 : 1;              // operand copies (hi, lo)
  constexpr int kBufBytes = kParts * kTcLayerBytes;       // one layer's weights in shared / global memory
  constexpr int kTileBytes = kParts * kTcABytes;          // one tile's activations
  const int t = threadIdx.x, warp = t >> 5;
  const int wg = t >> 7;    // warpgroup = tile within the CTA
  const int row = t & 127;  // row of the tile owned by this thread
  uint8_t *const sW = S.sW;
  const uint32_t wbar0 = S.wbar0, mbar0 = S.mbar0;
  const uint32_t tmem_tile = S.tmem_base + (uint32_t)wg * 128u;                  // column offset
  const uint32_t tmem_row = tmem_tile + ((uint32_t)((warp & 3) * 32) << 16);     // lane offset
  uint8_t *myA = S.sA + wg * kTileBytes;  // hi copy; the lo copy (bf16x3) follows at + kTcABytes
  const uint32_t aaddr = smem_u32(myA);
  uint32_t wc0 = S.wcount[0], wc1 = S.wcount[1];  // scalars: a dynamically indexed array would live in local memory
  uint32_t mcount = S.mcount;
  if (t == 0) {  // both weight buffers are free here: fetch layers 0 and 1
    for (int b = 0; b < 2; ++b) {
      mbar_expect_tx(wbar0 + 8 * b, kBufBytes);
      bulk_g2s(smem_u32(sW + b * kBufBytes), W + (size_t)b * kBufBytes, kBufBytes, wbar0 + 8 * b);
    }
  }
  // ---- input encoding straight from the packed state into the A operand (bf16 exact)
  const int p = pair * 256 + wg * 128 + row;
  // a warpgroup whose tile holds no position (small batches) only keeps the barriers company
  const bool tile_live = pair * 256 + wg * 128 < n;
  if (tile_live) {
    CState st{0, 0};
    if (p < n) {
      const ulonglong2 v = states[p];
      st.w0 = v.x, st.w1 = v.y;
    }
#pragma unroll
    for (int c = 0; c < kTcChunks; ++c) {
      uint32_t q[4];
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int j = 8 * c + 2 * h;
        const float a = j < CB200_STATE_SIZE ? encode_elem(st, j) : (j == kTcOnes ? 1.0f : 0.0f);
        const float b = j + 1 < CB200_STATE_SIZE ? encode_elem(st, j + 1)
                                                 : (j + 1 == kTcOnes + 1 ? 1.0f : 0.0f);
        q[h] = pack16<kFp16>(a, b);
      }
      *reinterpret_cast<uint4 *>(myA + c * kTcAChunkBytes + row * 16) =
          make_uint4(q[0], q[1], q[2], q[3]);
      if (kParts == 2)  // the encoding (0, 1/4, ..., 1) is exact in bf16: no lo part
        *reinterpret_cast<uint4 *>(myA + kTcABytes + c * kTcAChunkBytes + row * 16) = make_uint4(0, 0, 0, 0);
    }
  }
  // make this thread's generic-proxy writes of A visible to the tensor core, then sync
  fence_proxy_async();
  tc_fence_before();
  tc_sync(S.nthreads);
  tc_fence_after();
  for (int layer = 0; layer < kTcLayers; ++layer) {
    const int b = layer & 1;
    uint8_t *wbuf = sW + b * kBufBytes;
    mbar_wait(wbar0 + 8 * b, (b ? wc1 : wc0) & 1);
    wc0 += b ? 0u : 1u, wc1 += b ? 1u : 0u;
    if (tile_live) {
    if (row == 0) {  // one thread per warpgroup issues the MMAs of its tile
      const uint32_t waddr = smem_u32(wbuf);
      const uint32_t idesc = kFp16 ? kTcIdescF16 : kTcIdesc;
#pragma unroll
      for (int kk = 0; kk < kTcChunks / 2; ++kk) {
        const uint64_t ad = umma_desc(aaddr + kk * 2 * kTcAChunkBytes, kTcAChunkBytes, 128);
        const uint64_t bd = umma_desc(waddr + kk * 2 * kTcWChunkBytes, kTcWChunkBytes, 128);
        umma_bf16(tmem_tile, ad, bd, idesc, kk > 0 ? 1u : 0u);
        if (kParts == 2) {  // + a_hi * w_lo + a_lo * w_hi
          const uint64_t adl = umma_desc(aaddr + kTcABytes + kk * 2 * kTcAChunkBytes, kTcAChunkBytes, 128);
          const uint64_t bdl = umma_desc(waddr + kTcLayerBytes + kk * 2 * kTcWChunkBytes, kTcWChunkBytes, 128);
          umma_bf16(tmem_tile, ad, bdl, idesc, 1u);
          umma_bf16(tmem_tile, adl, bd, idesc, 1u);
        }
      }
      umma_commit(mbar0 + 8 * wg);
    }
    mbar_wait(mbar0 + 8 * wg, mcount & 1);
    mcount += 1;
    tc_fence_after();
    if (layer < kTcLayers - 1) {
      // ---- hidden-layer epilogue: ReLU + 16-bit pack (bias already in the accumulator), the
      // result becomes the next A operand. Seven 16-column TMEM loads, software-pipelined over two
      // register buffers: the next load is in flight while the current columns are converted
      // (32 registers of accumulator data at a time -- no local-memory spills).
      uint32_t va[16], vb[16];
      tmem_ld16_nowait(tmem_row, va);
#pragma unroll
      for (int c = 0; c < kTcN / 16; ++c) {
        uint32_t *cur = (c & 1) ? vb : va;
        tmem_wait_ld16(cur);
        if (c + 1 < kTcN / 16) tmem_ld16_nowait(tmem_row + 16 * (c + 1), (c & 1) ? va : vb);
#pragma unroll
        for (int h8 = 0; h8 < 2; ++h8) {
          const uint32_t *x = cur + 8 * h8;
          uint32_t hi[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) hi[q] = relu_pack16<kFp16>(x[2 * q], x[2 * q + 1]);
          uint8_t *dst = myA + (2 * c + h8) * kTcAChunkBytes + row * 16;
          *reinterpret_cast<uint4 *>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          if (kParts == 2) {  // lo = bf16(relu(x) - hi)
            uint32_t lo[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float r0 = fmaxf(__uint_as_float(x[2 * q]), 0.0f) - __uint_as_float(hi[q] << 16);
              const float r1 = fmaxf(__uint_as_float(x[2 * q + 1]), 0.0f) - __uint_as_float(hi[q] & 0xffff0000u);
              lo[q] = pack16<false>(r0, r1);
            }
            *reinterpret_cast<uint4 *>(dst + kTcABytes) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
      }
    } else {
      // ---- heads: column 0 = value (tanh), columns 1..96 = policy logits (softmax).
      // Pass 1 finds the row maximum, pass 2 writes e = exp(x - max) back into TMEM over the
      // logits while summing, pass 3 normalises and stores: one exponential per logit.
      // Columns come in batches of 16: batch 0 holds the value in column 0, batches 1-5 are all
      // logits, batch 6 holds the last logit (column 96) and padding.
      float mx = -INFINITY, v0 = 0.0f;
      {
        uint32_t v[16];
        tmem_ld16(tmem_row, v);
        v0 = __uint_as_float(v[0]);
#pragma unroll
        for (int h = 1; h < 16; ++h) mx = fmaxf(mx, __uint_as_float(v[h]));
#pragma unroll 1
        for (int c0 = 16; c0 < 96; c0 += 16) {
          tmem_ld16(tmem_row + c0, v);
#pragma unroll
          for (int h = 0; h < 16; ++h) mx = fmaxf(mx, __uint_as_float(v[h]));
        }
        tmem_ld16(tmem_row + 96, v);
        mx = fmaxf(mx, __uint_as_float(v[0]));
      }
      float sum = 0.0f;
      {
        uint32_t v[16];
        tmem_ld16(tmem_row, v);
#pragma unroll
        for (int h = 1; h < 16; ++h) {
          const float e = __expf(__uint_as_float(v[h]) - mx);
          sum += e, v[h] = __float_as_uint(e);
        }
        tmem_st16(tmem_row, v);
#pragma unroll 1
        for (int c0 = 16; c0 < 96; c0 += 16) {
          tmem_ld16(tmem_row + c0, v);
#pragma unroll
          for (int h = 0; h < 16; ++h) {
            const float e = __expf(__uint_as_float(v[h]) - mx);
            sum += e, v[h] = __float_as_uint(e);
          }
          tmem_st16(tmem_row + c0, v);
        }
        tmem_ld16(tmem_row + 96, v);
        const float e = __expf(__uint_as_float(v[0]) - mx);
        sum += e, v[0] = __float_as_uint(e);
        tmem_st16(tmem_row + 96, v);
        tmem_wait_st();
      }
      const float inv = 1.0f / sum;
      if (p < n) eval[p] = tanhf(v0);
      {
        // probabilities are written move-major ([96][ld]) so that a warp's stores coalesce;
        // the TMEM loads are warp-collective, only the stores are per-row
        const bool wr = p < n;
        float *pp = probs + p;
        uint32_t v[16];
        tmem_ld16(tmem_row, v);
#pragma unroll
        for (int h = 1; h < 16; ++h, pp += probs_ld)
          if (wr) *pp = __uint_as_float(v[h]) * inv;
#pragma unroll 1
        for (int c0 = 16; c0 < 96; c0 += 16) {
          tmem_ld16(tmem_row + c0, v);
#pragma unroll
          for (int h = 0; h < 16; ++h, pp += probs_ld)
            if (wr) *pp = __uint_as_float(v[h]) * inv;
        }
        tmem_ld16(tmem_row + 96, v);
        if (wr) *pp = __uint_as_float(v[0]) * inv;
      }
    }
    }  // tile_live
    // A (next layer's operand) is written, both tiles are done with this layer's
    // weights/bias: publish, sync, refill the weight buffer two layers ahead
    fence_proxy_async();
    tc_fence_before();
    tc_sync(S.nthreads);
    tc_fence_after();
    if (t == 0 && layer + 2 < kTcLayers) {
      mbar_expect_tx(wbar0 + 8 * b, kBufBytes);
      bulk_g2s(smem_u32(wbuf), W + (size_t)(layer + 2) * kBufBytes, kBufBytes, wbar0 + 8 * b);
    }
  }
  S.wcount[0] = wc0, S.wcount[1] = wc1;
  S.mcount = mcount;
}

template <int kMode>
__global__ void __launch_bounds__(kTcThreads, kMode == 2 ? 1 : 2)
    k_mlp_tc(const uint8_t *__restrict__ W, const ulonglong2 *__restrict__ states,
             const int32_t *__restrict__ n_ptr, int n_static, float *__restrict__ eval,
             float *__restrict__ probs, int probs_ld, int32_t *__restrict__ zero2) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int n = n_ptr ? *n_ptr : n_static;
  if (zero2 && blockIdx.x == 0 && threadIdx.x == 0) zero2[0] = 0, zero2[2] = 0;  // next parity's counters
  TcState S;
  tc_setup(S, smem, kTcThreads, kMode == 2 ? 2 : 1);
  const int n_pairs = (n + 255) / 256;
  for (int pair = blockIdx.x; pair < n_pairs; pair += gridDim.x)
    tc_forward<kMode>(S, W, states, n, pair, eval, probs, probs_ld);
  tc_teardown(S);
}

// One tile per CTA (128 threads; bf16 / fp16: 13 K registers and 77 KB of shared memory): small enough
// to share an SM with five 80-register game-step CTAs, so that one stream group's network overlaps
// the other groups' tree work. bf16x3: 154 KB, beside two game-step CTAs.
template <int kMode>
__global__ void __maxnreg__(kMode == 2 ? 168 : 104)
    k_mlp_tc1(const uint8_t *__restrict__ W, const ulonglong2 *__restrict__ states,
              const int32_t *__restrict__ n_ptr, int n_static, float *__restrict__ eval,
              float *__restrict__ probs, int probs_ld, int32_t *__restrict__ zero2) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int n = n_ptr ? *n_ptr : n_static;
  if (zero2 && blockIdx.x == 0 && threadIdx.x == 0) zero2[0] = 0, zero2[2] = 0;
  TcState S;
  tc_setup(S, smem, 128, kMode == 2 ? 2 : 1);
  for (int tile = blockIdx.x; tile * 128 < n; tile += gridDim.x) {
    const int rows = n - tile * 128 < 128 ? n - tile * 128 : 128;
    tc_forward<kMode>(S, W, states + tile * 128, rows, 0, eval + tile * 128, probs + tile * 128, probs_ld);
  }
  tc_teardown(S);
}

// Re-layout the C-ABI weight vector into per-layer UMMA images (16-bit operands, zero padded) and
// upload. mode 0 bf16, 1 fp16, 2 bf16x3: every layer is a hi image followed by a lo image
// (w = hi + lo to 16 significant bits; the bias rows carry a third part in the lo image).
inline int net_tc_upload(NetTC &net, const float *weights, int mode) {
  const bool fp16 = mode == 1;
  const int parts = mode == 2 ? 2 : 1;
  net.fp16 = fp16;
  net.mode = mode;
  const size_t layer_bytes = (size_t)parts * kTcLayerBytes;
  std::vector<uint8_t> host((size_t)kTcLayers * layer_bytes, 0);
  auto rnd = [&](float v) -> float {  // value of the 16-bit operand nearest to v
    return fp16 ? __half2float(__float2half_rn(v)) : __bfloat162float(__float2bfloat16_rn(v));
  };
  const float *src = weights;
  for (int l = 0; l < kTcLayers; ++l) {
    const int K = l == 0 ? CB200_STATE_SIZE : 100;
    const int N = l == kTcLayers - 1 ? 97 : 100;
    uint8_t *img = host.data() + (size_t)l * layer_bytes;
    // B operand is [N][K] K-major: chunk k/8, row o, element k%8; part 0 = hi image, 1 = lo image
    auto put = [&](int part, int k, int o, float v) {
      uint8_t *dst = img + (size_t)part * kTcLayerBytes + (size_t)(k >> 3) * kTcWChunkBytes + (size_t)o * 16 +
                     (k & 7) * 2;
      if (fp16) {
        const __half h = __float2half_rn(v);
        memcpy(dst, &h, 2);
      } else {
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        memcpy(dst, &h, 2);
      }
    };
    for (int k = 0; k < K; ++k)
      for (int o = 0; o < N; ++o) {
        const float w = src[(size_t)k * N + o];
        put(0, k, o, w);
        if (parts == 2) put(1, k, o, w - rnd(w));
      }
    src += (size_t)K * N;
    for (int o = 0; o < N; ++o) {  // bias = hi + lo (+ lo2), multiplied by the constant-one columns
      const float b = src[o];
      const float hi = rnd(b), lo = rnd(b - hi);
      put(0, kTcOnes, o, hi);
      put(0, kTcOnes + 1, o, lo);
      if (parts == 2) put(1, kTcOnes, o, b - hi - lo);
    }
    if (l < kTcLayers - 1) {  // keep the ones columns alive: out[:,100] = out[:,101] = 1
      put(0, kTcOnes, kTcOnes, 1.0f);
      put(0, kTcOnes, kTcOnes + 1, 1.0f);
    }
    src += N;
  }
  if (net.w && net.w_bytes != host.size()) {
    cudaFree(net.w);
    net.w = nullptr;
  }
  if (!net.w) CB_CUDA(cudaMalloc(&net.w, host.size()));
  net.w_bytes = host.size();
  CB_CUDA(cudaMemcpy(net.w, host.data(), host.size(), cudaMemcpyHostToDevice));
  net.ready = true;
  return CB200_OK;
}

inline void net_tc_free(NetTC &net) {
  if (net.w) cudaFree(net.w);
  net.w = nullptr;
}

inline int launch_mlp_tc(const NetTC &net, const ulonglong2 *d_states, const int32_t *d_n,
                         int n_static, int n_max, float *d_eval, float *d_probs, int probs_ld,
                         int32_t *zero2 = nullptr, cudaStream_t stream = nullptr,
                         bool use_stream = false, bool single_tile = false) {
  static bool attr_set[16] = {false};
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (dev < 16 && !attr_set[dev]) {
    CB_CUDA(cudaFuncSetAttribute(k_mlp_tc<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kTcSmemBytes));
    CB_CUDA(cudaFuncSetAttribute(k_mlp_tc<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kTcSmemBytes));
    CB_CUDA(cudaFuncSetAttribute(k_mlp_tc<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kTcSmemBytesX3));
    attr_set[dev] = true;
  }
  if (n_max <= 0) return CB200_OK;
  cudaStream_t st = use_stream ? stream : cur_stream();
  if (net.mode == 2 && !single_tile) {  // bf16x3, two tiles: 210 KB of shared memory, one CTA per SM
    const int pairs = (n_max + 255) / 256;
    k_mlp_tc<2><<<pairs < sms ? pairs : sms, kTcThreads, kTcSmemBytesX3, st>>>(
        (const uint8_t *)net.w, d_states, d_n, n_static, d_eval, d_probs, probs_ld, zero2);
    CB_LAUNCHED();
    CB_CUDA(cudaGetLastError());
    return CB200_OK;
  }
  if (single_tile) {
    static bool attr1[16] = {false};
    if (dev < 16 && !attr1[dev]) {
      CB_CUDA(cudaFuncSetAttribute(k_mlp_tc1<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)tc_smem_bytes(1, 1)));
      CB_CUDA(cudaFuncSetAttribute(k_mlp_tc1<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)tc_smem_bytes(1, 1)));
      CB_CUDA(cudaFuncSetAttribute(k_mlp_tc1<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)tc_smem_bytes(1, 2)));
      attr1[dev] = true;
    }
    const int tiles = (n_max + 127) / 128;
    const int g1 = tiles < sms ? tiles : sms;
    if (net.mode == 2)
      k_mlp_tc1<2><<<g1, 128, tc_smem_bytes(1, 2), st>>>(
          (const uint8_t *)net.w, d_states, d_n, n_static, d_eval, d_probs, probs_ld, zero2);
    else if (net.fp16)
      k_mlp_tc1<1><<<g1, 128, tc_smem_bytes(1, 1), st>>>(
          (const uint8_t *)net.w, d_states, d_n, n_static, d_eval, d_probs, probs_ld, zero2);
    else
      k_mlp_tc1<0><<<g1, 128, tc_smem_bytes(1, 1), st>>>(
          (const uint8_t *)net.w, d_states, d_n, n_static, d_eval, d_probs, probs_ld, zero2);
    CB_LAUNCHED();
    CB_CUDA(cudaGetLastError());
    return CB200_OK;
  }
  const int pairs = (n_max + 255) / 256;
  const int grid = pairs < 2 * sms ? pairs : 2 * sms;
  if (net.fp16)
    k_mlp_tc<1><<<grid, kTcThreads, kTcSmemBytes, st>>>(
        (const uint8_t *)net.w, d_states, d_n, n_static, d_eval, d_probs, probs_ld, zero2);
  else
    k_mlp_tc<0><<<grid, kTcThreads, kTcSmemBytes, st>>>(
        (const uint8_t *)net.w, d_states, d_n, n_static, d_eval, d_probs, probs_ld, zero2);
  CB_LAUNCHED();
  CB_CUDA(cudaGetLastError());
  return CB200_OK;
}

}  // namespace cb200
#endif
