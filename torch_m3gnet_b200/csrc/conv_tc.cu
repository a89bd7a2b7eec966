// M3GNetConv gated MLP on edges for F = 64 on the 5th-gen tensor cores (tcgen05.mma kind::tf32, accumulators in
// TMEM), fp32-faithful through the 3xTF32 split  a·b ≈ a_hi·b_hi + a_lo·b_hi + a_hi·b_lo  (hi = top 19 bits).
//
// One persistent CTA per SM walks tiles of 128 edges.  Per tile (forward):
//   e rows -> smem X (hi|lo, K-major SWIZZLE_128B)      GEMM1: D1[128x128] = X · W1e^T      (dense | gate halves)
//   epilogue: z1 = D1 + P[src] + P[dst] -> SiLU -> X    GEMM2d: D2d[128x64] = a1d · W2d^T
//                                        (gate half)    GEMM2g: D2g[128x64] = a1g · W2g^T
//   epilogue: SiLU(D2d + b) * sigmoid(D2g + b) * (h · Wh^T) (+ e) -> y
// The weight images (hi|lo for W1e, W2d, W2g = 128 KB) stay resident in shared memory for the whole kernel; the
// activation operand buffer X (64 KB) is reused by the three GEMMs; MMA completion is tracked with one mbarrier.
// The backward kernel recomputes the forward GEMMs and runs the transposed products (dz2·W2, dz1·W1e) against
// K-major images of the transposed weights that are staged per tile through a 32 KB buffer (tf32 operands
// only admit the 32B-atom swizzle in MN-major form, so the forward images cannot be reused transposed).
#include <cstdlib>

#include "common.cuh"
#include "umma.cuh"

namespace m3g {

using namespace umma;

constexpr int TC_F = 64;
constexpr int TILE_M = 128;
constexpr int TC_THREADS = 256;

// image sizes in floats
constexpr int IMG_W1 = 128 * 64;  // W1e: 128 rows (dense|gate outputs) x 64 (e features)
constexpr int IMG_W2 = 64 * 64;
constexpr int WIMG_FLOATS = 2 * IMG_W1 + 4 * IMG_W2;  // 32768 floats = 128 KB

__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xffffe000u); }

__device__ __forceinline__ float silu_fast(float z) { return __fdividef(z, 1.0f + __expf(-z)); }
__device__ __forceinline__ float sigmoid_fast(float z) { return __fdividef(1.0f, 1.0f + __expf(-z)); }

// split 4 consecutive k of row r into the hi / lo operand images
__device__ __forceinline__ void store_split4(char* x_hi, char* x_lo, int r, int k, float4 v) {
  uint32_t off = sw128_offset(r, k, TILE_M);
  float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
  float4 lo = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
  *reinterpret_cast<float4*>(x_hi + off) = hi;
  *reinterpret_cast<float4*>(x_lo + off) = lo;
}

// D[128 x N] (+)= A[128 x K] · Bimg^T with A a K-major image (128 rows) and B a K-major image with N rows:
//   D[m][n] += sum_k A[m][k] * Bimg[n][k]        (3 passes: hi·hi, lo·hi, hi·lo).  Issued by ONE thread.
// Descriptors only differ in their start-address field (bits 0-13, in 16-byte units), so the loops advance the
// low word instead of rebuilding them; PASSES / N / K are compile-time so the issue stream is straight-line code.
template <int PASSES, int N, int K>
__device__ __forceinline__ void issue_gemm_t(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi,
                                             uint32_t b_lo, bool accumulate) {
  constexpr uint32_t idesc = make_idesc_tf32(TILE_M, N, 0);
  const uint64_t dah = make_desc(a_hi, 16, 1024), dal = make_desc(a_lo, 16, 1024);
  const uint64_t dbh = make_desc(b_hi, 16, 1024), dbl = make_desc(b_lo, 16, 1024);
#pragma unroll
  for (int pass = 0; pass < PASSES; ++pass) {
    const uint64_t da0 = (pass == 1) ? dal : dah;
    const uint64_t db0 = (pass == 2) ? dbl : dbh;
#pragma unroll
    for (int kk = 0; kk < K / 8; ++kk) {
      const uint64_t da = da0 + (uint64_t)(((kk >> 2) * (TILE_M * 128) + (kk & 3) * 32) >> 4);
      const uint64_t db = db0 + (uint64_t)(((kk >> 2) * (N * 128) + (kk & 3) * 32) >> 4);
      mma_tf32(tmem_d, da, db, idesc, (accumulate || pass > 0 || kk > 0) ? 1u : 0u);
    }
  }
}
__device__ __forceinline__ void issue_gemm(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi,
                                           uint32_t b_lo, int N, int K, bool accumulate, int passes) {
  // (N, K) is (128, 64), (64, 64), (64, 128) or (128, 128) on every call site
  if (passes == 3) {
    if (N == 128 && K == 64) issue_gemm_t<3, 128, 64>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
    else if (N == 64 && K == 64) issue_gemm_t<3, 64, 64>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
    else if (N == 64) issue_gemm_t<3, 64, 128>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
    else issue_gemm_t<3, 128, 128>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
  } else {
    if (N == 128 && K == 64) issue_gemm_t<1, 128, 64>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
    else if (N == 64 && K == 64) issue_gemm_t<1, 64, 64>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
    else if (N == 64) issue_gemm_t<1, 64, 128>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
    else issue_gemm_t<1, 128, 128>(tmem_d, a_hi, a_lo, b_hi, b_lo, accumulate);
  }
}

// Same product with the A operand in tensor memory: A_hi at columns [ta_hi, ta_hi+K), A_lo at [ta_lo, ta_lo+K)
// (row m in lane m, written with tcgen05.st by the epilogue threads).
template <int PASSES, int N, int K>
__device__ __forceinline__ void issue_gemm_ts_t(uint32_t tmem_d, uint32_t ta_hi, uint32_t ta_lo, uint32_t b_hi,
                                                uint32_t b_lo, bool accumulate) {
  constexpr uint32_t idesc = make_idesc_tf32(TILE_M, N, 0);
  const uint64_t dbh = make_desc(b_hi, 16, 1024), dbl = make_desc(b_lo, 16, 1024);
#pragma unroll
  for (int pass = 0; pass < PASSES; ++pass) {
    const uint32_t a = (pass == 1) ? ta_lo : ta_hi;
    const uint64_t db0 = (pass == 2) ? dbl : dbh;
#pragma unroll
    for (int kk = 0; kk < K / 8; ++kk) {
      const uint64_t db = db0 + (uint64_t)(((kk >> 2) * (N * 128) + (kk & 3) * 32) >> 4);
      mma_tf32_ts(tmem_d, a + 8 * kk, db, idesc, (accumulate || pass > 0 || kk > 0) ? 1u : 0u);
    }
  }
}
__device__ __forceinline__ void issue_gemm_ts(uint32_t tmem_d, uint32_t ta_hi, uint32_t ta_lo, uint32_t b_hi,
                                              uint32_t b_lo, int N, int K, bool accumulate, int passes) {
  if (passes == 3) {
    if (N == 128 && K == 64) issue_gemm_ts_t<3, 128, 64>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
    else if (N == 64 && K == 64) issue_gemm_ts_t<3, 64, 64>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
    else if (N == 64) issue_gemm_ts_t<3, 64, 128>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
    else issue_gemm_ts_t<3, 128, 128>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
  } else {
    if (N == 128 && K == 64) issue_gemm_ts_t<1, 128, 64>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
    else if (N == 64 && K == 64) issue_gemm_ts_t<1, 64, 64>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
    else if (N == 64) issue_gemm_ts_t<1, 64, 128>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
    else issue_gemm_ts_t<1, 128, 128>(tmem_d, ta_hi, ta_lo, b_hi, b_lo, accumulate);
  }
}

// --------------------------------------------------------------------------------------------------------
// weight image packing: W (rows x cols) row-major -> hi / lo SWIZZLE_128B images
__global__ void tc_pack_kernel(const float* __restrict__ W, int rows, int cols, float* __restrict__ img_hi,
                               float* __restrict__ img_lo) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  int r = idx / cols, k = idx - r * cols;
  float v = W[idx];
  float hi = tf32_hi(v);
  uint32_t off = sw128_offset(r, k, rows) >> 2;
  img_hi[off] = hi;
  img_lo[off] = v - hi;
}

// --------------------------------------------------------------------------------------------------------
// self test of the UMMA plumbing: one 128-row tile.
//   out[128 x rows] = A[128 x cols] · W^T   (W given as its packed K-major image, rows x cols)
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_selftest_kernel(const float* __restrict__ A, const float* __restrict__ img_hi, const float* __restrict__ img_lo,
                   int rows, int cols, int passes, int a_tmem, float* __restrict__ out) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = (char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  char* b_hi = smem;
  char* b_lo = smem + rows * cols * 4;
  char* x_hi = smem + 2 * rows * cols * 4;
  const int K = cols;
  const int N = rows;
  char* x_lo = x_hi + TILE_M * K * 4;
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < rows * cols / 4; i += TC_THREADS) {
    reinterpret_cast<float4*>(b_hi)[i] = reinterpret_cast<const float4*>(img_hi)[i];
    reinterpret_cast<float4*>(b_lo)[i] = reinterpret_cast<const float4*>(img_lo)[i];
  }
  for (int i = tid; i < TILE_M * K / 4; i += TC_THREADS) {
    int r = i / (K / 4), c = i - r * (K / 4);
    float4 v = reinterpret_cast<const float4*>(A)[i];
    // A image with K columns: generic offset (K may be 64 or 128)
    uint32_t off = sw128_offset(r, 4 * c, TILE_M);
    float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    *reinterpret_cast<float4*>(x_hi + off) = hi;
    *reinterpret_cast<float4*>(x_lo + off) = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
  }
  if (warp == 0) tmem_alloc<512>(&tmem_slot);
  if (tid == 0) {
    mbar_init(&bar, 1);
    mbar_fence_init();
  }
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  uint32_t tmem = tmem_slot;
  int q = warp & 3, hsel = warp >> 2;
  int r = 32 * q + lane;
  if (a_tmem) {
    // A (hi | lo) into tensor memory columns [128, 128+K) | [256, 256+K): row r in lane r
    for (int k0 = 32 * hsel; k0 < K; k0 += 64) {
      float hi[32], lo[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        float v = A[r * K + k0 + c];
        hi[c] = tf32_hi(v);
        lo[c] = v - hi[c];
      }
      tmem_st32(tmem + ((uint32_t)(32 * q) << 16) + 128 + k0, hi);
      tmem_st32(tmem + ((uint32_t)(32 * q) << 16) + 256 + k0, lo);
    }
    tmem_st_wait();
    fence_before_sync();
    __syncthreads();
  }
  if (tid == 0) {
    fence_after_sync();
    if (a_tmem)
      issue_gemm_ts(tmem, tmem + 128, tmem + 256, smem_u32(b_hi), smem_u32(b_lo), N, K, false, passes);
    else
      issue_gemm(tmem, smem_u32(x_hi), smem_u32(x_lo), smem_u32(b_hi), smem_u32(b_lo), N, K, false, passes);
    commit(&bar);
  }
  mbar_wait(&bar, 0);
  fence_after_sync();
  for (int c0 = 32 * hsel; c0 < N; c0 += 64) {
    float v[32];
    tmem_ld32(tmem + ((uint32_t)(32 * q) << 16) + c0, v);
    tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < 32; ++c) out[r * N + c0 + c] = v[c];
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

// --------------------------------------------------------------------------------------------------------
struct ConvTcParams {
  const float* P; int ldp; int po;
  const int32_t* src; const int32_t* dst;
  const float* e; const float* h;
  const float* wimg;  // [W1 hi | W1 lo | W2d hi | W2d lo | W2g hi | W2g lo]
  const float* b2d; const float* b2g; const float* WhT;
  int64_t E; int R; int mode; int passes;
  float* y;
  float* save;  // optional (variant 4): per-tile activations for m3g_conv_tc_bwd_saved, see save_offset()
};

// Activations kept for the backward pass (1 KB per edge): four 64-column blocks per 128-edge tile —
// 0: SiLU'(z1 dense), 1: SiLU'(z1 gate), 2: z2 dense, 3: z2 gate (pre-activations, biases included).  The layout is
// private to the kernel pair and "fragment-major": a thread's 16-column slice of its row is four float4 that land,
// together with the other 31 rows of the warp, in four fully coalesced 512-byte segments:
//   [tile][block 4][16-column chunk 4][row quadrant 4][float4 index 4][row in quadrant 32][4 floats]
// Measured alternative (round 2, removed again): SiLU'(z1) kept as 24-bit fixed point (absolute error <= 5.6e-8, 896
// instead of 1024 B per edge): the packing work and its narrower stores cost the forward 0.455 -> 0.515 ms per launch
// (part of it register spills) while the backward only gained 0.638 -> 0.629 ms.
constexpr int SAVE_TILE_WORDS = TILE_M * 256;
__device__ __forceinline__ int64_t save_offset(int64_t tile, int block, int chunk, int quadrant) {
  return tile * (int64_t)SAVE_TILE_WORDS + (((block * 4 + chunk) * 4 + quadrant) << 9);
}

constexpr int SMEM_W_BYTES = WIMG_FLOATS * 4;         // 131072
constexpr int SMEM_X_BYTES = 2 * TILE_M * TC_F * 4;   // 65536 (hi | lo)
constexpr int SMEM_MISC_FLOATS = 64 + 64 + M3G_MAX_RADIAL * 64;
constexpr int SMEM_FWD_BYTES = SMEM_W_BYTES + SMEM_X_BYTES + SMEM_MISC_FLOATS * 4 + 1024;

constexpr int TC2_THREADS = 512;  // two groups of 8 warps
constexpr int GRP_THREADS = 256;

// --------------------------------------------------------------------------------------------------------
// Coalesced global traffic for row-per-lane accumulators.  The accumulator layout is row-per-lane (tcgen05.ld
// 32x32b), so a naive epilogue gathers P[dst] and writes y with 32 different cache lines per warp instruction (ncu:
// the L1 wavefront queue, not the tensor pipe, paced the first tcgen05 version).  Every gather / scatter therefore
// goes through a private 2 KB per-warp staging tile:
//   P[dst] rows:  coalesced LDG.128 (8 rows x 64 B per instruction, dst indices broadcast by shuffle)
//                 -> staging (XOR-swizzled 16 B slots, conflict-free both ways) -> row-per-lane LDS.128
//   y rows:       row-per-lane -> staging -> coalesced STG.128 (+ the residual e rows, read coalesced)
// P[src] stays a direct row-per-lane load: edges are grouped by source atom, so the 32 rows of a warp share one or
// two source atoms and the load is (nearly) a broadcast.
constexpr int STG_WARP_BYTES = 32 * 16 * 4;  // 32 rows x 16 floats
constexpr int TC3_MAX_R = 4;

// 16-byte slot of (row r, 4-column group c4) in a 32 x 16 float staging tile
__device__ __forceinline__ uint32_t stg_off(int r, int c4) { return (uint32_t)((r * 4 + (c4 ^ ((r >> 1) & 3))) << 4); }

// --------------------------------------------------------------------------------------------------------
// Forward: two groups of 8 warps ping-pong two tiles; layer-2 A operands in TENSOR MEMORY.
// ncu on the version that staged activations in shared memory: the shared-memory data pipe is ~95 % busy (LSU wavefronts 69 % + tensor-core operand fetch
// 26 %), so the layer-1 activations no longer round-trip through shared memory: the epilogue threads write their
// hi / lo split with tcgen05.st into TMEM columns they own (the consumed D1 columns, and the idle D2g columns) and
// GEMM2d / GEMM2g read A from TMEM ([a_tmem] operand form).  Only the e tile still uses the shared operand buffer X,
// so the two groups hand X over once per tile (mbarrier of the other group's GEMM1) and each GEMM has its own
// mbarrier (one completion per tile -> parity = tile counter, no multi-phase bookkeeping).
// TMEM columns per group: [0,128) D1, then A_hi at [0,64); A_lo at [192,256) for the dense branch and [64,128) for
// the gate branch; [128,192) D2d; [192,256) D2g.  Every thread only ever overwrites columns it has already read.
constexpr int SMEM_MISC4_BYTES = (64 + 64 + TC3_MAX_R * 64) * 4 + 64;  // biases, Wh^T, 6 mbarriers + TMEM slot
constexpr int SMEM_FWD4_BYTES = SMEM_W_BYTES + SMEM_X_BYTES + SMEM_MISC4_BYTES + 16 * STG_WARP_BYTES + 1024;
static_assert(SMEM_FWD4_BYTES <= 232448, "variant-4 forward exceeds the 227 KB shared-memory limit");

__device__ __forceinline__ void store_split4_s(uint32_t x_hi, uint32_t x_lo, int r, int k, float4 v) {
  uint32_t off = sw128_offset(r, k, TILE_M);
  float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
  sts128(x_hi + off, hi);
  sts128(x_lo + off, make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w));
}

// hi / lo split of 32 activations into two 32-column TMEM slices of this thread's lane
__device__ __forceinline__ void tmem_put_split32(uint32_t t_hi, uint32_t t_lo, const float* a) {
#pragma unroll
  for (int h2 = 0; h2 < 2; ++h2) {
    float t[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) t[c] = tf32_hi(a[16 * h2 + c]);
    tmem_st16(t_hi + 16 * h2, t);
#pragma unroll
    for (int c = 0; c < 16; ++c) t[c] = a[16 * h2 + c] - t[c];
    tmem_st16(t_lo + 16 * h2, t);
  }
  tmem_st_wait();
}

__global__ void __launch_bounds__(TC2_THREADS, 1) conv_tc4_fwd_kernel(ConvTcParams p) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = (char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(smem);
  const uint32_t w1_hi = sbase, w1_lo = w1_hi + IMG_W1 * 4;
  const uint32_t w2d_hi = w1_lo + IMG_W1 * 4, w2d_lo = w2d_hi + IMG_W2 * 4;
  const uint32_t w2g_hi = w2d_lo + IMG_W2 * 4, w2g_lo = w2g_hi + IMG_W2 * 4;
  const uint32_t xh = sbase + SMEM_W_BYTES, xl = xh + TILE_M * TC_F * 4;
  float* misc = reinterpret_cast<float*>(smem + SMEM_W_BYTES + SMEM_X_BYTES);
  const uint32_t b2d_a = sbase + SMEM_W_BYTES + SMEM_X_BYTES, b2g_a = b2d_a + 256, wh_a = b2g_a + 256;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + 128 + TC3_MAX_R * 64);  // [g1 A,B | g2d A,B | g2g A,B]
  uint32_t* tmem_slot_p = reinterpret_cast<uint32_t*>(bars + 6);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int grp = warp >> 3, wg = warp & 7;
  const int q = wg & 3, hsel = wg >> 2;
  const int gtid = tid & (GRP_THREADS - 1);
  const int row = 32 * q + lane;
  const int c0 = 32 * hsel;
  const uint32_t stg = sbase + SMEM_W_BYTES + SMEM_X_BYTES + SMEM_MISC4_BYTES + warp * STG_WARP_BYTES;
  const int cr = lane >> 2, cc4 = lane & 3;  // coalesced layout: row 8*i + cr, 4-column group cc4

  for (int i = tid; i < WIMG_FLOATS / 4; i += TC2_THREADS)
    reinterpret_cast<float4*>(smem)[i] = reinterpret_cast<const float4*>(p.wimg)[i];
  if (tid < 64) { misc[tid] = p.b2d[tid]; misc[64 + tid] = p.b2g[tid]; }
  for (int i = tid; i < TC3_MAX_R * 64; i += TC2_THREADS) misc[128 + i] = (i < p.R * 64) ? p.WhT[i] : 0.0f;
  if (warp == 0) tmem_alloc<512>(tmem_slot_p);
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 6; ++i) mbar_init(&bars[i], 1);
    mbar_fence_init();
  }
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_p;
  const uint32_t tmem = tmem_base + grp * 256;
  const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
  const uint32_t D1 = 0, D2D = 128, D2G = 192;
  uint64_t* g1_own = &bars[grp];
  uint64_t* g1_other = &bars[grp ^ 1];
  uint64_t* g2d_own = &bars[2 + grp];
  uint64_t* g2g_own = &bars[4 + grp];
  const int bar_id = 1 + grp;

  const int64_t n_tiles = (p.E + TILE_M - 1) / TILE_M;
  const int64_t per_iter = 2 * (int64_t)gridDim.x;
  const int64_t n_iter = (n_tiles + per_iter - 1) / per_iter;
  // this row's bond indices, loaded one tile ahead: P[src] / P[dst] gathers no longer start behind an index load
  int d_next = 0, s_next = 0;
  {
    const int64_t t0 = (int64_t)blockIdx.x * 2 + grp;
    if (t0 < n_tiles) {
      d_next = __ldg(p.dst + min(t0 * TILE_M + row, p.E - 1));
      s_next = __ldg(p.src + min(t0 * TILE_M + row, p.E - 1));
    }
  }
  for (int64_t it = 0; it < n_iter; ++it) {
    const int64_t tile = (it * gridDim.x + blockIdx.x) * 2 + grp;
    if (tile >= n_tiles) break;  // tiles are dealt A,B,A,B,...: the other group never waits on a tile that is absent
    const uint32_t par = (uint32_t)(it & 1);
    const int64_t e0 = tile * TILE_M;
    // ---- prefetch the e rows of this tile into registers (coalesced: 2 rows x 256 B per warp instruction) ----
    float4 ev[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int idx = gtid + GRP_THREADS * i;
      int64_t eg_ = min(e0 + (idx >> 4), p.E - 1);
      ev[i] = __ldg(reinterpret_cast<const float4*>(p.e + eg_ * TC_F) + (idx & 15));
    }
    const int64_t eg = min(e0 + row, p.E - 1);
    const int d_row = d_next;
    const int s_atom = s_next;
    if (tile + per_iter < n_tiles) {
      const int64_t en_ = min((tile + per_iter) * TILE_M + row, p.E - 1);
      d_next = __ldg(p.dst + en_);
      s_next = __ldg(p.src + en_);
    }
    const float* Pi = p.P + (int64_t)s_atom * p.ldp + p.po;
    // mode 2: source atom of every row of this warp's 32-row block (-1 past the end), for the segmented message sum
    const int s_row = (e0 + row < p.E) ? s_atom : -1;
    {
      // pull this group's next tile (e rows, indices, h) into L2 while this tile computes
      const int64_t en = (tile + 2 * (int64_t)gridDim.x) * TILE_M;
      if (en < p.E) {
        prefetch_l2(p.e + min(en + gtid / 2, p.E - 1) * TC_F + (gtid & 1) * 32);
        if (gtid < 16) prefetch_l2(p.h + min(en * p.R + gtid * 32, p.E * p.R - 1));
        else if (gtid < 20) prefetch_l2(p.src + min(en + (gtid - 16) * 32, p.E - 1));
        else if (gtid < 24) prefetch_l2(p.dst + min(en + (gtid - 20) * 32, p.E - 1));
      }
    }
    // P[dst] row pointers of the four rows this lane serves in the coalesced layout
    // (32-bit float offsets into P: N * ldp < 2^31 is checked by the host entry; four registers instead of eight)
    const float* Pb = p.P + p.po + 128 + 4 * cc4;
    uint32_t Pj[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) Pj[i] = (uint32_t)__shfl_sync(FULL, d_row, 8 * i + cr) * (uint32_t)p.ldp;
    float4 pj[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) pj[i] = __ldg(reinterpret_cast<const float4*>(Pb + Pj[i] + c0));
    // ---- X hand-off: the other group's latest GEMM1 must have consumed X ----
    if (grp == 1) mbar_wait_warp(g1_other, par);
    else if (it > 0) mbar_wait_warp(g1_other, par ^ 1);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int idx = gtid + GRP_THREADS * i;
      store_split4_s(xh, xl, idx >> 4, 4 * (idx & 15), ev[i]);
    }
    fence_proxy_async();
    fence_before_sync();
    named_bar_sync(bar_id, GRP_THREADS);
    if (gtid == 0) {
      fence_after_sync();
      issue_gemm(tmem + D1, xh, xl, w1_hi, w1_lo, 128, 64, false, p.passes);
      commit(g1_own);
    }
    float act[32];
    // ---- layer-1 activations: four 16-column sub-chunks (dense c0, c0+16 ; gate c0, c0+16) ----
#pragma unroll
    for (int sc = 0; sc < 4; ++sc) {
      const int col = ((sc >> 1) << 6) + c0 + ((sc & 1) << 4);  // column inside the 128-wide z1 row
#pragma unroll
      for (int i = 0; i < 4; ++i) sts128(stg + stg_off(8 * i + cr, cc4), pj[i]);
      if (sc < 3) {
        const int ncol = (((sc + 1) >> 1) << 6) + c0 + (((sc + 1) & 1) << 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) pj[i] = __ldg(reinterpret_cast<const float4*>(Pb + Pj[i] + ncol));
      }
      float4 pi4[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) pi4[c] = __ldg(reinterpret_cast<const float4*>(Pi + col + 4 * c));
      __syncwarp();
      if (sc == 0) {  // own GEMM1
        mbar_wait_warp(g1_own, par);
        fence_after_sync();
      }
      float v[16];
      tmem_ld16(t_lane + D1 + col, v);
      tmem_ld_wait();
      float* sv = p.save ? p.save + save_offset(tile, sc >> 1, 2 * hsel + (sc & 1), q) + 4 * lane : nullptr;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 b = lds128(stg + stg_off(lane, c));
        const float z[4] = {v[4 * c] + pi4[c].x + b.x, v[4 * c + 1] + pi4[c].y + b.y, v[4 * c + 2] + pi4[c].z + b.z,
                            v[4 * c + 3] + pi4[c].w + b.w};
        float g[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float sg = sigmoid_fast(z[u]);
          act[16 * (sc & 1) + 4 * c + u] = z[u] * sg;
          g[u] = sg * (1.0f + z[u] * (1.0f - sg));  // SiLU'(z1), kept for the backward pass
        }
        if (sv) *reinterpret_cast<float4*>(sv + 128 * c) = make_float4(g[0], g[1], g[2], g[3]);
      }
      __syncwarp();
      if (sc == 1) {
        // dense branch: A_hi -> own D1 dense columns, A_lo -> own (idle) D2g columns ; GEMM2d
        tmem_put_split32(t_lane + D1 + c0, t_lane + D2G + c0, act);
        fence_before_sync();
        named_bar_sync(bar_id, GRP_THREADS);
        if (gtid == 0) {
          fence_after_sync();
          issue_gemm_ts(tmem + D2D, tmem + D1, tmem + D2G, w2d_hi, w2d_lo, 64, 64, false, p.passes);
          commit(g2d_own);
        }
      } else if (sc == 3) {
        // gate branch: GEMM2d must have consumed A ; A_hi -> D1 dense columns, A_lo -> own D1 gate columns ; GEMM2g
        mbar_wait_warp(g2d_own, par);
        fence_after_sync();
        tmem_put_split32(t_lane + D1 + c0, t_lane + D1 + 64 + c0, act);
        fence_before_sync();
        named_bar_sync(bar_id, GRP_THREADS);
        if (gtid == 0) {
          fence_after_sync();
          issue_gemm_ts(tmem + D2G, tmem + D1, tmem + D1 + 64, w2g_hi, w2g_lo, 64, 64, false, p.passes);
          commit(g2g_own);
        }
      }
    }
    // ---- output stage ----
    float hm[TC3_MAX_R];
#pragma unroll
    for (int m = 0; m < TC3_MAX_R; ++m) hm[m] = (m < p.R) ? __ldg(p.h + eg * p.R + m) : 0.0f;
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {
      float v[16];
      tmem_ld16(t_lane + D2D + c0 + 16 * h2, v);
      tmem_ld_wait();
      float* sv = p.save ? p.save + save_offset(tile, 2, 2 * hsel + h2, q) + 4 * lane : nullptr;
#pragma unroll
      for (int c = 0; c < 16; c += 4) {
        float4 b = lds128(b2d_a + 4 * (c0 + 16 * h2 + c));
        const float4 z = make_float4(v[c] + b.x, v[c + 1] + b.y, v[c + 2] + b.z, v[c + 3] + b.w);
        if (sv) *reinterpret_cast<float4*>(sv + 32 * c) = z;
        act[16 * h2 + c] = silu_fast(z.x);
        act[16 * h2 + c + 1] = silu_fast(z.y);
        act[16 * h2 + c + 2] = silu_fast(z.z);
        act[16 * h2 + c + 3] = silu_fast(z.w);
      }
    }
    mbar_wait_warp(g2g_own, par);
    fence_after_sync();
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {
      const int col = c0 + 16 * h2;
      // residual rows (mode 0), coalesced layout; issued before the TMEM read so that they overlap it
      float4 er[4];
      if (p.mode == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          int64_t er_ = min(e0 + 32 * q + 8 * i + cr, p.E - 1);
          er[i] = __ldg(reinterpret_cast<const float4*>(p.e + er_ * TC_F + col + 4 * cc4));
        }
      }
      float v[16];
      tmem_ld16(t_lane + D2G + col, v);
      tmem_ld_wait();
      float* svg = p.save ? p.save + save_offset(tile, 3, 2 * hsel + h2, q) + 4 * lane : nullptr;
#pragma unroll
      for (int c = 0; c < 16; c += 4) {
        float4 bg = lds128(b2g_a + 4 * (col + c));
        if (svg) *reinterpret_cast<float4*>(svg + 32 * c) = make_float4(v[c] + bg.x, v[c + 1] + bg.y, v[c + 2] + bg.z,
                                                                       v[c + 3] + bg.w);
        float bgv[4] = {bg.x, bg.y, bg.z, bg.w};
        float o[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) o[u] = 0.0f;
#pragma unroll
        for (int m = 0; m < TC3_MAX_R; ++m) {
          float4 w4 = lds128(wh_a + 4 * (m * 64 + col + c));
          o[0] += hm[m] * w4.x; o[1] += hm[m] * w4.y; o[2] += hm[m] * w4.z; o[3] += hm[m] * w4.w;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) o[u] *= act[16 * h2 + c + u] * sigmoid_fast(v[c + u] + bgv[u]);
        sts128(stg + stg_off(lane, c >> 2), make_float4(o[0], o[1], o[2], o[3]));
      }
      __syncwarp();
      if (p.mode != 2) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 r4 = lds128(stg + stg_off(8 * i + cr, cc4));
          if (p.mode == 0) { r4.x += er[i].x; r4.y += er[i].y; r4.z += er[i].z; r4.w += er[i].w; }
          int64_t er_ = e0 + 32 * q + 8 * i + cr;
          if (er_ < p.E) *reinterpret_cast<float4*>(p.y + er_ * TC_F + col + 4 * cc4) = r4;
        }
      } else {
        // messages are only ever summed per source atom (nn/conv.py:82-87) and the rows of an atom are contiguous:
        // reduce this warp's 32 rows per source atom here and write ONE partial row per (32-row block, atom) at the
        // block's first row of that atom; m3g_segment_sum_parts adds the (ascending) partials of an atom to x.
        // Order (stated): rows 8 i + cr for i = 0..3 in this lane, then a fixed xor tree over cr.
        float4 r4[4];
        int sa[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          r4[i] = lds128(stg + stg_off(8 * i + cr, cc4));
          sa[i] = __shfl_sync(FULL, s_row, 8 * i + cr);
        }
        int start = 0;
        while (start < 32) {
          const int a = __shfl_sync(FULL, s_row, start);
          if (a < 0) break;
          const int n_rows = __popc(__ballot_sync(FULL, s_row == a));
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (sa[i] == a) { acc.x += r4[i].x; acc.y += r4[i].y; acc.z += r4[i].z; acc.w += r4[i].w; }
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) {
            acc.x += __shfl_xor_sync(FULL, acc.x, o); acc.y += __shfl_xor_sync(FULL, acc.y, o);
            acc.z += __shfl_xor_sync(FULL, acc.z, o); acc.w += __shfl_xor_sync(FULL, acc.w, o);
          }
          if (cr == 0)
            *reinterpret_cast<float4*>(p.y + (e0 + 32 * q + start) * TC_F + col + 4 * cc4) = acc;
          start += n_rows;
        }
      }
      __syncwarp();
    }
    fence_before_sync();
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// --------------------------------------------------------------------------------------------------------
// Backward of one gated MLP on edges (forward recomputed on the tensor cores).
struct ConvTcBwdParams {
  const float* P; int ldp; int po;
  const int32_t* src; const int32_t* dst;
  const float* e; const float* h;
  const float* wimg;   // forward images (resident)
  const float* wimgT;  // [W2d^T hi|lo, W2g^T hi|lo, W1e_dense^T hi|lo, W1e_gate^T hi|lo], each 64x64 image pair (staged)
  const float* b2d; const float* b2g; const float* WhT;
  const float* g_up; const float* g_e_base;
  int64_t E; int R; int mode; int passes;
  float* g_e; float* g_z1; float* g_h;
};

constexpr int SMEM_S_BYTES = 2 * IMG_W2 * 4;  // 32768: one staged 64x64 image pair
constexpr int TC_BWD_MAX_R = 3;

__device__ __forceinline__ float silu_grad_fast(float z) {
  float s = sigmoid_fast(z);
  return s * (1.0f + z * (1.0f - s));
}


// --------------------------------------------------------------------------------------------------------
// Backward with the forward RECOMPUTED (used when no saved activations exist; M3G_TC_BWD_VARIANT=2).  One persistent
// CTA per SM, 16 warps (4 threads per edge row, 16-column slices), one 128-edge tile in flight:
//  * EVERY A operand lives in tensor memory: the epilogue threads write hi / lo splits with tcgen05.st into columns
//    they own, so no activation / adjoint tile round-trips through shared memory and the tensor core only fetches B
//    from shared memory.  The layer-1 SiLU derivative is stashed in the D1 columns for the later dz1 stage.
//  * every global gather / scatter (e, P[dst], g_up, g_e, g_z1) is coalesced through a private 2 KB per-warp staging
//    tile (see the forward kernel); outputs are written at the end of the tile, re-read from the TMEM operand copies.
//  * the four transposed 64x64 weight image pairs are streamed by cp.async.bulk (TMA 1-D, mbarrier byte counts)
//    through two 32 KB buffers instead of LDG+STS by all threads; forward images stay resident.
//  * four MMA sync points per tile (GEMM1 | GEMM2d+2g | GEMM3d+3g | GEMM4a+4b) instead of seven.
// TMEM columns: [0,128) D1 -> SiLU'(z1) stash -> D4 in [0,64) ; [128,192) D2d, [192,256) D2g -> operand A2 (hi|lo) ;
//               [256,320) | [320,384) operand A (hi|lo) ; [384,448) D3d, [448,512) D3g (before that: operand A' = a1g).
constexpr int TCB2_THREADS = 512;
constexpr int SMEM_B2_MISC = (64 + 64 + TC_BWD_MAX_R * 64) * 4 + 80;  // biases, Wh^T, 8 mbarriers, TMEM slot
constexpr int SMEM_BWD2_BYTES = SMEM_W_BYTES + 2 * SMEM_S_BYTES + 16 * STG_WARP_BYTES + SMEM_B2_MISC + 1024;
static_assert(SMEM_BWD2_BYTES <= 232448, "backward variant 2 exceeds the 227 KB shared-memory limit");

__device__ __forceinline__ void tmem_put_split16(uint32_t t_hi, uint32_t t_lo, const float* a) {
  float t[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) t[c] = tf32_hi(a[c]);
  tmem_st16(t_hi, t);
#pragma unroll
  for (int c = 0; c < 16; ++c) t[c] = a[c] - t[c];
  tmem_st16(t_lo, t);
}

// optional phase timing (build with M3G_EXTRA_NVCC_FLAGS=-DM3G_TC_TIMING): thread 0 of every CTA accumulates the
// cycles between consecutive phase marks of the backward kernel; read back with m3g_debug_tc_timing
__device__ unsigned long long g_tc_timing[16];
#ifdef M3G_TC_TIMING
#define TCT(k)                                                          \
  do {                                                                  \
    if (tid == 0) {                                                     \
      long long now__ = clock64();                                      \
      atomicAdd(&g_tc_timing[k], (unsigned long long)(now__ - tct_prev)); \
      tct_prev = now__;                                                 \
    }                                                                   \
  } while (0)
#else
#define TCT(k) do { } while (0)
#endif

__global__ void __launch_bounds__(TCB2_THREADS, 1) conv_tc_bwd2_kernel(ConvTcBwdParams p) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = (char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(smem);
  const uint32_t w1_hi = sbase, w1_lo = w1_hi + IMG_W1 * 4;
  const uint32_t w2d_hi = w1_lo + IMG_W1 * 4, w2d_lo = w2d_hi + IMG_W2 * 4;
  const uint32_t w2g_hi = w2d_lo + IMG_W2 * 4, w2g_lo = w2g_hi + IMG_W2 * 4;
  const uint32_t s0 = sbase + SMEM_W_BYTES, s1 = s0 + SMEM_S_BYTES;  // streamed image pairs (hi | lo)
  const uint32_t stg_all = s1 + SMEM_S_BYTES;
  char* misc_c = smem + SMEM_W_BYTES + 2 * SMEM_S_BYTES + 16 * STG_WARP_BYTES;
  float* misc = reinterpret_cast<float*>(misc_c);
  const uint32_t b2d_a = stg_all + 16 * STG_WARP_BYTES, b2g_a = b2d_a + 256, wh_a = b2g_a + 256;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + 128 + TC_BWD_MAX_R * 64);  // bar1..bar4, tb0, tb1
  uint32_t* tmem_slot_p = reinterpret_cast<uint32_t*>(bars + 8);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, cs = warp >> 2;
  const int row = 32 * q + lane;
  const int k0 = 16 * cs;  // this thread's 16-column slice of every 64-column block
  const uint32_t stg = stg_all + warp * STG_WARP_BYTES;
  const int cr = lane >> 2, cc4 = lane & 3;  // coalesced layout: row 8*i + cr, 4-column group cc4
  const int R = p.R;
  constexpr uint32_t PAIR_BYTES = 2 * IMG_W2 * 4;

  for (int i = tid; i < WIMG_FLOATS / 4; i += TCB2_THREADS)
    reinterpret_cast<float4*>(smem)[i] = reinterpret_cast<const float4*>(p.wimg)[i];
  if (tid < 64) { misc[tid] = p.b2d[tid]; misc[64 + tid] = p.b2g[tid]; }
  for (int i = tid; i < TC_BWD_MAX_R * 64; i += TCB2_THREADS) misc[128 + i] = (i < R * 64) ? p.WhT[i] : 0.0f;
  if (warp == 0) tmem_alloc<512>(tmem_slot_p);
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) mbar_init(&bars[i], 1);
    mbar_fence_init();
  }
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  // One CTA per SM owns all 512 columns, so the allocation starts at lane 0 / column 0; using the literal keeps every
  // MMA operand address a compile-time uniform value (otherwise each tcgen05.mma costs two R2UR round trips and the
  // single issuing thread, not the tensor core, paces the 64-wide GEMMs).
  if (*tmem_slot_p != 0u) __trap();
  constexpr uint32_t tmem = 0u;
  const uint32_t t_lane = ((uint32_t)(32 * q) << 16);
  constexpr uint32_t Z1 = 0, D2D = 128, D2G = 192, AH = 256, AL = 320, D3D = 384, D3G = 448;
  uint64_t *bar1 = &bars[0], *bar2 = &bars[1], *bar3 = &bars[2], *bar4 = &bars[3], *tb0 = &bars[4], *tb1 = &bars[5];
  uint64_t *bar3a = &bars[6], *bar4a = &bars[7];  // GEMM3d / GEMM4a alone: their weight buffer can be refilled early

  const int64_t n_tiles = (p.E + TILE_M - 1) / TILE_M;
  if (tid == 0 && (int64_t)blockIdx.x < n_tiles) {
    mbar_arrive_expect_tx(tb0, PAIR_BYTES);
    bulk_g2s(s0, p.wimgT + 0 * 2 * IMG_W2, PAIR_BYTES, tb0);  // W2d^T
    mbar_arrive_expect_tx(tb1, PAIR_BYTES);
    bulk_g2s(s1, p.wimgT + 1 * 2 * IMG_W2, PAIR_BYTES, tb1);  // W2g^T
  }
  uint32_t par = 0;
#ifdef M3G_TC_TIMING
  long long tct_prev = clock64();
#endif
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, par ^= 1) {
    TCT(0);
    const int64_t e0 = tile * TILE_M;
    const int64_t eg = min(e0 + row, p.E - 1);
    const bool live = (e0 + row) < p.E;
    const int s_atom = __ldg(p.src + eg);
    const int d_atom = __ldg(p.dst + eg);
    {
      // pull the next tile's streamed rows (e, g_up / g_e_base, indices, h) into L2 while this tile computes
      const int64_t en = (tile + gridDim.x) * TILE_M;
      if (en < p.E) {
        const int64_t rn = min(en + (tid & 255) / 2, p.E - 1);  // 2 x 128-byte lines per 64-float row
        const int half = (tid & 1) * 32;
        if (tid < 256) {
          prefetch_l2(p.e + rn * TC_F + half);
          if (p.g_e_base) prefetch_l2(p.g_e_base + rn * TC_F + half);
        } else {
          if (p.mode == 0) prefetch_l2(p.g_up + rn * TC_F + half);
          if (tid < 256 + 16) prefetch_l2(p.h + min(en * R + (tid - 256) * 32, p.E * R - 1));
          else if (tid < 256 + 20) prefetch_l2(p.src + min(en + (tid - 272) * 32, p.E - 1));
          else if (tid < 256 + 24) prefetch_l2(p.dst + min(en + (tid - 276) * 32, p.E - 1));
        }
      }
    }
    // rows this lane serves in the coalesced layout
    int64_t erow[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) erow[i] = e0 + 32 * q + 8 * i + cr;
    float4 c4v[4];
    // ---- T1: e slice -> staging -> row-per-lane -> hi|lo -> operand A in TMEM ; GEMM1 ----
#pragma unroll
    for (int i = 0; i < 4; ++i)
      c4v[i] = __ldg(reinterpret_cast<const float4*>(p.e + min(erow[i], p.E - 1) * TC_F + k0 + 4 * cc4));
#pragma unroll
    for (int i = 0; i < 4; ++i) sts128(stg + stg_off(8 * i + cr, cc4), c4v[i]);
    __syncwarp();
    {
      float t[16];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 b = lds128(stg + stg_off(lane, c));
        t[4 * c] = b.x; t[4 * c + 1] = b.y; t[4 * c + 2] = b.z; t[4 * c + 3] = b.w;
      }
      tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, t);
    }
    __syncwarp();
    tmem_st_wait();
    fence_before_sync();
    __syncthreads();
    TCT(1);
    if (tid == 0) {
      fence_after_sync();
      issue_gemm_ts(tmem + Z1, tmem + AH, tmem + AL, w1_hi, w1_lo, 128, 64, false, p.passes);
      commit(bar1);
    }
    TCT(2);
    // ---- T2 (overlaps GEMM1): P[src] + P[dst] for the dense and gate slices ----
    float pz[32];
    {
      const float* Pi = p.P + (int64_t)s_atom * p.ldp + p.po;
      const float* Pj[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        Pj[i] = p.P + (int64_t)__shfl_sync(FULL, d_atom, 8 * i + cr) * p.ldp + p.po + 128 + k0 + 4 * cc4;
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
#pragma unroll
        for (int i = 0; i < 4; ++i) c4v[i] = __ldg(reinterpret_cast<const float4*>(Pj[i] + 64 * hb));
        float4 pi4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) pi4[c] = __ldg(reinterpret_cast<const float4*>(Pi + 64 * hb + k0 + 4 * c));
#pragma unroll
        for (int i = 0; i < 4; ++i) sts128(stg + stg_off(8 * i + cr, cc4), c4v[i]);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float4 b = lds128(stg + stg_off(lane, c));
          pz[16 * hb + 4 * c] = pi4[c].x + b.x;
          pz[16 * hb + 4 * c + 1] = pi4[c].y + b.y;
          pz[16 * hb + 4 * c + 2] = pi4[c].z + b.z;
          pz[16 * hb + 4 * c + 3] = pi4[c].w + b.w;
        }
        __syncwarp();
      }
    }
    // ---- T3: z1 -> a1 (operands A, A') and SiLU'(z1) (stash) ; GEMM2d + GEMM2g ----
    TCT(14);
    mbar_wait_warp(bar1, par);
    TCT(3);
    fence_after_sync();
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
      float v[16], g[16];
      tmem_ld16(t_lane + Z1 + 64 * hb + k0, v);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        float z = v[c] + pz[16 * hb + c];
        float sg = sigmoid_fast(z);
        v[c] = z * sg;
        g[c] = sg * (1.0f + z * (1.0f - sg));
      }
      tmem_st16(t_lane + Z1 + 64 * hb + k0, g);
      if (hb == 0) tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, v);
      else tmem_put_split16(t_lane + D3D + k0, t_lane + D3G + k0, v);
    }
    tmem_st_wait();
    fence_before_sync();
    __syncthreads();
    TCT(4);
    if (tid == 0) {
      fence_after_sync();
      issue_gemm_ts(tmem + D2D, tmem + AH, tmem + AL, w2d_hi, w2d_lo, 64, 64, false, p.passes);
      issue_gemm_ts(tmem + D2G, tmem + D3D, tmem + D3G, w2g_hi, w2g_lo, 64, 64, false, p.passes);
      commit(bar2);
    }
    TCT(5);
    // ---- T4 (overlaps GEMM2): upstream gradient slice, h ----
    float gu[16];
    if (p.mode == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        c4v[i] = __ldg(reinterpret_cast<const float4*>(p.g_up + min(erow[i], p.E - 1) * TC_F + k0 + 4 * cc4));
#pragma unroll
      for (int i = 0; i < 4; ++i) sts128(stg + stg_off(8 * i + cr, cc4), c4v[i]);
      __syncwarp();
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 b = lds128(stg + stg_off(lane, c));
        gu[4 * c] = b.x; gu[4 * c + 1] = b.y; gu[4 * c + 2] = b.z; gu[4 * c + 3] = b.w;
      }
      __syncwarp();
    } else {
      const float* gr = p.g_up + (int64_t)s_atom * TC_F + k0;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 b = __ldg(reinterpret_cast<const float4*>(gr + 4 * c));
        gu[4 * c] = b.x; gu[4 * c + 1] = b.y; gu[4 * c + 2] = b.z; gu[4 * c + 3] = b.w;
      }
    }
    float hm[TC_BWD_MAX_R], ghp[TC_BWD_MAX_R];
#pragma unroll
    for (int m = 0; m < TC_BWD_MAX_R; ++m) {
      hm[m] = (m < R) ? __ldg(p.h + eg * R + m) : 0.0f;
      ghp[m] = 0.0f;
    }
    // ---- T5: output-stage adjoint -> dz2d (operand A), dz2g (operand A2) ; GEMM3d + GEMM3g ----
    TCT(14);
    mbar_wait_warp(bar2, par);
    TCT(6);
    fence_after_sync();
    {
      float vd[16], vg[16];
      tmem_ld16(t_lane + D2D + k0, vd);
      tmem_ld16(t_lane + D2G + k0, vg);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 16; c += 4) {
        float4 bd = lds128(b2d_a + 4 * (k0 + c));
        float4 bg = lds128(b2g_a + 4 * (k0 + c));
        float bdv[4] = {bd.x, bd.y, bd.z, bd.w}, bgv[4] = {bg.x, bg.y, bg.z, bg.w};
        float whv[TC_BWD_MAX_R][4];
#pragma unroll
        for (int m = 0; m < TC_BWD_MAX_R; ++m) {
          float4 w4 = lds128(wh_a + 4 * (m * 64 + k0 + c));
          whv[m][0] = w4.x; whv[m][1] = w4.y; whv[m][2] = w4.z; whv[m][3] = w4.w;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float zd = vd[c + u] + bdv[u];
          float sgm = sigmoid_fast(zd);
          float sd = zd * sgm;
          float sgr = sgm * (1.0f + zd * (1.0f - sgm));
          float sg = sigmoid_fast(vg[c + u] + bgv[u]);
          float s = 0.0f;
#pragma unroll
          for (int m = 0; m < TC_BWD_MAX_R; ++m) s += hm[m] * whv[m][u];
          float gs = gu[c + u] * sd * sg;
#pragma unroll
          for (int m = 0; m < TC_BWD_MAX_R; ++m) ghp[m] += gs * whv[m][u];
          float gphi = gu[c + u] * s;
          vd[c + u] = gphi * sg * sgr;               // dz2d
          vg[c + u] = gphi * sd * sg * (1.0f - sg);  // dz2g
        }
      }
      tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, vd);
      tmem_put_split16(t_lane + D2D + k0, t_lane + D2G + k0, vg);
    }
    // g_h partial sums of the three other column slices of this row travel through their warps' own (idle)
    // staging tiles: slot `lane` of warp q + 4*cs
    if (cs != 0) sts128(stg + lane * 16, make_float4(ghp[0], ghp[1], ghp[2], 0.0f));
    tmem_st_wait();
    fence_before_sync();
    __syncthreads();
    TCT(7);
    if (tid == 0) {
      fence_after_sync();
      mbar_wait(tb0, 0);
      issue_gemm_ts(tmem + D3D, tmem + AH, tmem + AL, s0, s0 + IMG_W2 * 4, 64, 64, false, p.passes);
      commit(bar3a);
      mbar_wait(tb1, 0);
      issue_gemm_ts(tmem + D3G, tmem + D2D, tmem + D2G, s1, s1 + IMG_W2 * 4, 64, 64, false, p.passes);
      commit(bar3);
      // GEMM3d finished while GEMM3g was being issued: its buffer takes W1e(dense rows)^T now
      mbar_wait(bar3a, par);
      mbar_arrive_expect_tx(tb0, PAIR_BYTES);
      bulk_g2s(s0, p.wimgT + 2 * 2 * IMG_W2, PAIR_BYTES, tb0);
    }
    TCT(8);
    if (cs == 0) {
      float4 g1 = lds128(stg + 4 * STG_WARP_BYTES + lane * 16);
      float4 g2 = lds128(stg + 8 * STG_WARP_BYTES + lane * 16);
      float4 g3 = lds128(stg + 12 * STG_WARP_BYTES + lane * 16);
      if (live) {
        float tot[3] = {((ghp[0] + g1.x) + g2.x) + g3.x, ((ghp[1] + g1.y) + g2.y) + g3.y,
                        ((ghp[2] + g1.z) + g2.z) + g3.z};
#pragma unroll
        for (int m = 0; m < TC_BWD_MAX_R; ++m)
          if (m < R) p.g_h[eg * R + m] += tot[m];
      }
    }
    // ---- T6: dz1 = D3 * SiLU'(z1) -> operands A (dense), A2 (gate) ; GEMM4a + GEMM4b ----
    TCT(15);
    mbar_wait_warp(bar3, par);
    TCT(9);
    fence_after_sync();
    if (tid == 0) {
      mbar_arrive_expect_tx(tb1, PAIR_BYTES);
      bulk_g2s(s1, p.wimgT + 3 * 2 * IMG_W2, PAIR_BYTES, tb1);  // W1e(gate rows)^T
    }
    float dz1[32];
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
      float g[16];
      tmem_ld16(t_lane + (hb ? D3G : D3D) + k0, dz1 + 16 * hb);
      tmem_ld16(t_lane + Z1 + 64 * hb + k0, g);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 16; ++c) dz1[16 * hb + c] *= g[c];
      if (hb == 0) tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, dz1);
      else tmem_put_split16(t_lane + D2D + k0, t_lane + D2G + k0, dz1 + 16);
    }
    tmem_st_wait();
    fence_before_sync();
    __syncthreads();
    TCT(10);
    if (tid == 0) {
      fence_after_sync();
      mbar_wait(tb0, 1);
      issue_gemm_ts(tmem + Z1, tmem + AH, tmem + AL, s0, s0 + IMG_W2 * 4, 64, 64, false, p.passes);
      commit(bar4a);
      mbar_wait(tb1, 1);
      issue_gemm_ts(tmem + Z1, tmem + D2D, tmem + D2G, s1, s1 + IMG_W2 * 4, 64, 64, true, p.passes);
      commit(bar4);
      if (tile + gridDim.x < n_tiles) {  // the next tile's W2d^T
        mbar_wait(bar4a, par);
        mbar_arrive_expect_tx(tb0, PAIR_BYTES);
        bulk_g2s(s0, p.wimgT + 0 * 2 * IMG_W2, PAIR_BYTES, tb0);
      }
    }
    // residual gradient rows for the final g_e store (coalesced layout; L2-resident thanks to the tile prefetch)
    float4 gb[4];
    if (p.g_e_base) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        gb[i] = __ldg(reinterpret_cast<const float4*>(p.g_e_base + min(erow[i], p.E - 1) * TC_F + k0 + 4 * cc4));
    }
    // g_z1 rows straight from registers (overlaps GEMM4), coalesced through the staging tile
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        sts128(stg + stg_off(lane, c), make_float4(dz1[16 * hb + 4 * c], dz1[16 * hb + 4 * c + 1],
                                                   dz1[16 * hb + 4 * c + 2], dz1[16 * hb + 4 * c + 3]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 r4 = lds128(stg + stg_off(8 * i + cr, cc4));
        if (erow[i] < p.E) *reinterpret_cast<float4*>(p.g_z1 + erow[i] * 128 + 64 * hb + k0 + 4 * cc4) = r4;
      }
      __syncwarp();
    }
    TCT(11);
    // ---- T7: outputs (g_e, g_z1), coalesced through the staging tile ----
    TCT(15);
    mbar_wait_warp(bar4, par);
    TCT(12);
    fence_after_sync();
    if (tid == 0 && tile + gridDim.x < n_tiles) {
      mbar_arrive_expect_tx(tb1, PAIR_BYTES);
      bulk_g2s(s1, p.wimgT + 1 * 2 * IMG_W2, PAIR_BYTES, tb1);
    }
    {
      float v[16];
      tmem_ld16(t_lane + Z1 + k0, v);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 4; ++c)
        sts128(stg + stg_off(lane, c), make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 r4 = lds128(stg + stg_off(8 * i + cr, cc4));
        if (erow[i] < p.E) {
          if (p.g_e_base) { r4.x += gb[i].x; r4.y += gb[i].y; r4.z += gb[i].z; r4.w += gb[i].w; }
          *reinterpret_cast<float4*>(p.g_e + erow[i] * TC_F + k0 + 4 * cc4) = r4;
        }
      }
      __syncwarp();
    }
    fence_before_sync();
    TCT(13);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

// --------------------------------------------------------------------------------------------------------
// Backward from SAVED activations (pairs with conv_tc4_fwd_kernel(save != NULL)).  The recompute version above
// spends 43 % of its MMA instructions, both P gathers, the e load and half of its MUFU work on rebuilding z1 / z2;
// here the forward leaves SiLU'(z1) and z2 behind (1 KB per edge, fragment-major so that both sides use plain coalesced
// float4 accesses) and the backward is just   output adjoint -> GEMM3d/3g -> dz1 -> GEMM4a/4b -> outputs:
// two MMA sync points per tile, no forward weights, all four transposed weight image pairs resident in shared memory.
// Measured alternative (round 2, removed again): MMA batches issued by warps 15 / 14 (no g_h duty) instead of warp 0,
// with the issuing warp's SiLU' loads put in flight before it starts issuing — 0.640 vs 0.627 ms: slower, although
// the phase marks of warp 0 suggest that the issuing warp reaches both barriers ~2 k cycles after the others.
// Measured alternative (round 2, removed again): two tiles in flight with two groups of 8 warps and 256 tensor-memory
// columns per tile (one operand region refilled before each of four 64x64 GEMMs, dz2g parked in the idle D3g columns,
// D4 aliasing D3d, the four MMA batches issued by four different warps) — bit-identical g_e / g_z1, 0.651 vs 0.638 ms
// per launch at C2: the chain of one tile is not what bounds the kernel (tools/tc_timing.py: loads 2.5 k + 1.6 k, math
// 3.7 k, MMA issue 3.3 k + 3.2 k, stores 2.0 k of 18.4 k cycles per tile), the memory system's response to its six
// concurrent row streams is (ncu: long-scoreboard is the top stall, DRAM 60 %, no pipe above 50 %).
// TMEM columns: A [0,64)|[64,128) hi|lo, A2 [128,192)|[192,256), D3d [256,320), D3g [320,384), D4 [384,448).
struct ConvTcBwdSParams {
  const int32_t* src; const float* h;
  const float* wimgT;  // [W2d^T hi|lo, W2g^T hi|lo, W1e_dense^T hi|lo, W1e_gate^T hi|lo]
  const float* WhT; const float* save;
  const float* g_up; const float* g_e_base;
  int64_t E; int R; int mode; int passes;
  float* g_e; float* g_z1; float* g_h;
  int gh_store;  // 1: g_h rows are stored (the caller sums per-launch slices), 0: added to the rows already there
};
constexpr int SMEM_BS_MISC = TC_BWD_MAX_R * 64 * 4 + 32;  // Wh^T, 3 mbarriers, TMEM slot
constexpr int SMEM_Z2_BYTES = 2 * 16 * 2048;           // blocks 2, 3 of one tile
constexpr int SMEM_BWDS_BYTES = SMEM_W_BYTES + 16 * STG_WARP_BYTES + SMEM_Z2_BYTES + SMEM_BS_MISC + 1024;
static_assert(SMEM_BWDS_BYTES <= 232448, "saved-activation backward exceeds the 227 KB shared-memory limit");

__global__ void __launch_bounds__(TCB2_THREADS, 1) conv_tc_bwds_kernel(ConvTcBwdSParams p) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = (char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(smem);
  const uint32_t wt[4] = {sbase, sbase + SMEM_S_BYTES, sbase + 2 * SMEM_S_BYTES, sbase + 3 * SMEM_S_BYTES};
  const uint32_t stg_all = sbase + SMEM_W_BYTES;
  const uint32_t z2buf = stg_all + 16 * STG_WARP_BYTES;  // this tile's saved z2 blocks (64 KB), bulk-copied one tile ahead
  float* misc = reinterpret_cast<float*>(smem + SMEM_W_BYTES + 16 * STG_WARP_BYTES + SMEM_Z2_BYTES);
  const uint32_t wh_a = z2buf + SMEM_Z2_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + TC_BWD_MAX_R * 64);
  uint32_t* tmem_slot_p = reinterpret_cast<uint32_t*>(bars + 3);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, cs = warp >> 2;
  const int row = 32 * q + lane;
  const int k0 = 16 * cs;
  const uint32_t stg = stg_all + warp * STG_WARP_BYTES;
  const int cr = lane >> 2, cc4 = lane & 3;
  const int R = p.R;

  for (int i = tid; i < WIMG_FLOATS / 4; i += TCB2_THREADS)
    reinterpret_cast<float4*>(smem)[i] = reinterpret_cast<const float4*>(p.wimgT)[i];
  for (int i = tid; i < TC_BWD_MAX_R * 64; i += TCB2_THREADS) misc[i] = (i < R * 64) ? p.WhT[i] : 0.0f;
  if (warp == 0) tmem_alloc<512>(tmem_slot_p);
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    mbar_fence_init();
  }
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  if (*tmem_slot_p != 0u) __trap();  // one CTA per SM owns all 512 columns: literal operand addresses (see bwd2)
  constexpr uint32_t tmem = 0u;
  const uint32_t t_lane = ((uint32_t)(32 * q) << 16);
  constexpr uint32_t AH = 0, AL = 64, A2H = 128, A2L = 192, D3D = 256, D3G = 320, D4 = 384;
  uint64_t *bar3 = &bars[0], *bar4 = &bars[1], *zb = &bars[2];

  const int64_t n_tiles = (p.E + TILE_M - 1) / TILE_M;
  // blocks 2 and 3 (z2 dense | gate) of a tile are 64 KB contiguous in the save layout
  if (tid == 0 && (int64_t)blockIdx.x < n_tiles) {
    mbar_arrive_expect_tx(zb, SMEM_Z2_BYTES);
    bulk_g2s(z2buf, p.save + save_offset(blockIdx.x, 2, 0, 0), SMEM_Z2_BYTES, zb);
  }
  uint32_t par = 0;
  // mode 1 (g_up indexed by source atom): the row's source index is loaded one tile ahead — ncu showed the dependent
  // chain src[row] -> g_up[src] (a cold 512-byte line per tile, then the gather) as the largest single stall of the
  // node-MLP launches
  int s_cur = 0;
  if (p.mode != 0 && (int64_t)blockIdx.x < n_tiles) s_cur = __ldg(p.src + min((int64_t)blockIdx.x * TILE_M + row, p.E - 1));
  // the upstream-gradient pieces of a tile (four float4 per thread: the coalesced layout in mode 0, this row's slice of
  // g_up[src] in mode 1) are requested one tile ahead, while the previous tile's last stores drain: T0 starts with them
  // in registers instead of an L2 round trip (tools/tc_timing.py: "T0 loads" 2.1 k cycles per tile before)
  float4 gnext[4];
  auto load_upstream = [&](int64_t t, int s_atom) {
    if (p.mode == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int64_t r = min(t * TILE_M + 32 * q + 8 * i + cr, p.E - 1);
        gnext[i] = __ldg(reinterpret_cast<const float4*>(p.g_up + r * TC_F + k0 + 4 * cc4));
      }
    } else {
      const float* gr = p.g_up + (int64_t)s_atom * TC_F + k0;
#pragma unroll
      for (int c = 0; c < 4; ++c) gnext[c] = __ldg(reinterpret_cast<const float4*>(gr + 4 * c));
    }
  };
  if ((int64_t)blockIdx.x < n_tiles) load_upstream(blockIdx.x, s_cur);
#ifdef M3G_TC_TIMING
  long long tct_prev = clock64();
#endif
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, par ^= 1) {
    TCT(0);
    const int64_t e0 = tile * TILE_M;
    const int64_t eg = min(e0 + row, p.E - 1);
    const bool live = (e0 + row) < p.E;
    if (p.mode != 0 && tile + gridDim.x < n_tiles) s_cur = __ldg(p.src + min((tile + gridDim.x) * TILE_M + row, p.E - 1));
    const int64_t ebase = e0 + 32 * q + cr;  // rows ebase + 8 i (i = 0..3): this lane's rows in the coalesced layout
    {
      // next tile: saved activations (128 KB = 1024 lines), upstream rows, residual rows, h into L2
      const int64_t tn = tile + gridDim.x;
      if (tn < n_tiles) {
        const float* sv = p.save + tn * (int64_t)SAVE_TILE_WORDS;
        prefetch_l2(sv + tid * 32);  // blocks 0, 1 (SiLU'(z1)); blocks 2, 3 arrive by bulk copy
        const int64_t en = tn * TILE_M;
        const int64_t rn = min(en + (tid & 255) / 2, p.E - 1);
        const int half = (tid & 1) * 32;
        if (tid < 256) {
          if (p.mode == 0) prefetch_l2(p.g_up + rn * TC_F + half);
        } else {
          if (p.g_e_base) prefetch_l2(p.g_e_base + rn * TC_F + half);
          if (tid < 256 + 16) prefetch_l2(p.h + min(en * R + (tid - 256) * 32, p.E * R - 1));
        }
      }
    }
    // ---- T0: upstream gradient slice (requested one tile ago), saved z2 slices, h ----
    float zd[16], zg[16], gu[16];
    if (p.mode == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) sts128(stg + stg_off(8 * i + cr, cc4), gnext[i]);
      __syncwarp();
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 b = lds128(stg + stg_off(lane, c));
        gu[4 * c] = b.x; gu[4 * c + 1] = b.y; gu[4 * c + 2] = b.z; gu[4 * c + 3] = b.w;
      }
      __syncwarp();
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        gu[4 * c] = gnext[c].x; gu[4 * c + 1] = gnext[c].y; gu[4 * c + 2] = gnext[c].z; gu[4 * c + 3] = gnext[c].w;
      }
    }
    {
      mbar_wait_warp(zb, par);  // the bulk copy issued one tile ago has landed
      const uint32_t s2 = z2buf + ((cs * 4 + q) << 11) + 16 * lane;
      const uint32_t s3 = s2 + (16 << 11);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 a = lds128(s2 + 512 * c);
        float4 b = lds128(s3 + 512 * c);
        zd[4 * c] = a.x; zd[4 * c + 1] = a.y; zd[4 * c + 2] = a.z; zd[4 * c + 3] = a.w;
        zg[4 * c] = b.x; zg[4 * c + 1] = b.y; zg[4 * c + 2] = b.z; zg[4 * c + 3] = b.w;
      }
    }
    float hm[TC_BWD_MAX_R], ghp[TC_BWD_MAX_R];
#pragma unroll
    for (int m = 0; m < TC_BWD_MAX_R; ++m) {
      hm[m] = (m < R) ? __ldg(p.h + eg * R + m) : 0.0f;
      ghp[m] = 0.0f;
    }
    TCT(1);
    // ---- T5: output-stage adjoint -> dz2d (operand A), dz2g (operand A2) ; GEMM3d + GEMM3g ----
#pragma unroll
    for (int c = 0; c < 16; c += 4) {
      float whv[TC_BWD_MAX_R][4];
#pragma unroll
      for (int m = 0; m < TC_BWD_MAX_R; ++m) {
        float4 w4 = lds128(wh_a + 4 * (m * 64 + k0 + c));
        whv[m][0] = w4.x; whv[m][1] = w4.y; whv[m][2] = w4.z; whv[m][3] = w4.w;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float z = zd[c + u];
        const float sgm = sigmoid_fast(z);
        const float sd = z * sgm;
        const float sgr = sgm * (1.0f + z * (1.0f - sgm));
        const float sg = sigmoid_fast(zg[c + u]);
        float s = 0.0f;
#pragma unroll
        for (int m = 0; m < TC_BWD_MAX_R; ++m) s += hm[m] * whv[m][u];
        const float gs = gu[c + u] * sd * sg;
#pragma unroll
        for (int m = 0; m < TC_BWD_MAX_R; ++m) ghp[m] += gs * whv[m][u];
        const float gphi = gu[c + u] * s;
        zd[c + u] = gphi * sg * sgr;               // dz2d
        zg[c + u] = gphi * sd * sg * (1.0f - sg);  // dz2g
      }
    }
    tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, zd);
    tmem_put_split16(t_lane + A2H + k0, t_lane + A2L + k0, zg);
    if (cs != 0) sts128(stg + lane * 16, make_float4(ghp[0], ghp[1], ghp[2], 0.0f));
    tmem_st_wait();
    fence_before_sync();
    TCT(2);
    __syncthreads();
    TCT(3);
    if (tid == 0) {
      fence_after_sync();
      if (tile + gridDim.x < n_tiles) {  // every thread has consumed this tile's z2: refill for the next tile
        fence_proxy_async();
        mbar_arrive_expect_tx(zb, SMEM_Z2_BYTES);
        bulk_g2s(z2buf, p.save + save_offset(tile + gridDim.x, 2, 0, 0), SMEM_Z2_BYTES, zb);
      }
      issue_gemm_ts(tmem + D3D, tmem + AH, tmem + AL, wt[0], wt[0] + IMG_W2 * 4, 64, 64, false, p.passes);
      issue_gemm_ts(tmem + D3G, tmem + A2H, tmem + A2L, wt[1], wt[1] + IMG_W2 * 4, 64, 64, false, p.passes);
      commit(bar3);
    }
    TCT(4);
    if (cs == 0) {
      float4 g1 = lds128(stg + 4 * STG_WARP_BYTES + lane * 16);
      float4 g2 = lds128(stg + 8 * STG_WARP_BYTES + lane * 16);
      float4 g3 = lds128(stg + 12 * STG_WARP_BYTES + lane * 16);
      if (live) {
        float tot[3] = {((ghp[0] + g1.x) + g2.x) + g3.x, ((ghp[1] + g1.y) + g2.y) + g3.y,
                        ((ghp[2] + g1.z) + g2.z) + g3.z};
        // (store form: no read-modify-write round trip in the four warps every other warp waits for at the next barrier)
        if (p.gh_store) {
#pragma unroll
          for (int m = 0; m < TC_BWD_MAX_R; ++m)
            if (m < R) p.g_h[eg * R + m] = tot[m];
        } else {
#pragma unroll
          for (int m = 0; m < TC_BWD_MAX_R; ++m)
            if (m < R) p.g_h[eg * R + m] += tot[m];
        }
      }
    }
    // saved SiLU'(z1) slices (dense -> zd, gate -> zg), in flight while GEMM3 runs
    {
      const float* s0 = p.save + save_offset(tile, 0, cs, q) + 4 * lane;
      const float* s1 = p.save + save_offset(tile, 1, cs, q) + 4 * lane;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 a = __ldg(reinterpret_cast<const float4*>(s0 + 128 * c));
        float4 b = __ldg(reinterpret_cast<const float4*>(s1 + 128 * c));
        zd[4 * c] = a.x; zd[4 * c + 1] = a.y; zd[4 * c + 2] = a.z; zd[4 * c + 3] = a.w;
        zg[4 * c] = b.x; zg[4 * c + 1] = b.y; zg[4 * c + 2] = b.z; zg[4 * c + 3] = b.w;
      }
    }
    TCT(5);
    // ---- T6: dz1 = D3 * SiLU'(z1) -> operands A (dense), A2 (gate) ; GEMM4a + GEMM4b ----
    mbar_wait_warp(bar3, par);
    TCT(6);
    fence_after_sync();
    {
      float v[16];
      tmem_ld16(t_lane + D3D + k0, v);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 16; ++c) zd[c] *= v[c];
      tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, zd);
      tmem_ld16(t_lane + D3G + k0, v);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 16; ++c) zg[c] *= v[c];
      tmem_put_split16(t_lane + A2H + k0, t_lane + A2L + k0, zg);
    }
    tmem_st_wait();
    fence_before_sync();
    TCT(8);
    __syncthreads();
    TCT(9);
    if (tid == 0) {
      fence_after_sync();
      issue_gemm_ts(tmem + D4, tmem + AH, tmem + AL, wt[2], wt[2] + IMG_W2 * 4, 64, 64, false, p.passes);
      issue_gemm_ts(tmem + D4, tmem + A2H, tmem + A2L, wt[3], wt[3] + IMG_W2 * 4, 64, 64, true, p.passes);
      commit(bar4);
    }
    TCT(10);
    float4 gb[4];
    if (p.g_e_base) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        gb[i] = __ldg(reinterpret_cast<const float4*>(p.g_e_base + min(ebase + 8 * i, p.E - 1) * TC_F + k0 + 4 * cc4));
    }
    // g_z1 rows straight from registers (overlaps GEMM4), coalesced through the staging tile; skipped when the caller
    // has no use for them (first block of the model: its node features do not depend on the positions)
    if (p.g_z1 != nullptr) {
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
        const float* dz = hb ? zg : zd;
#pragma unroll
        for (int c = 0; c < 4; ++c)
          sts128(stg + stg_off(lane, c), make_float4(dz[4 * c], dz[4 * c + 1], dz[4 * c + 2], dz[4 * c + 3]));
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 r4 = lds128(stg + stg_off(8 * i + cr, cc4));
          if (ebase + 8 * i < p.E) *reinterpret_cast<float4*>(p.g_z1 + (ebase + 8 * i) * 128 + 64 * hb + k0 + 4 * cc4) = r4;
        }
        __syncwarp();
      }
    }
    TCT(11);
    if (tile + gridDim.x < n_tiles) load_upstream(tile + gridDim.x, s_cur);
    // ---- T7: g_e ----
    mbar_wait_warp(bar4, par);
    TCT(12);
    fence_after_sync();
    {
      float v[16];
      tmem_ld16(t_lane + D4 + k0, v);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 4; ++c)
        sts128(stg + stg_off(lane, c), make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 r4 = lds128(stg + stg_off(8 * i + cr, cc4));
        if (ebase + 8 * i < p.E) {
          if (p.g_e_base) { r4.x += gb[i].x; r4.y += gb[i].y; r4.z += gb[i].z; r4.w += gb[i].w; }
          *reinterpret_cast<float4*>(p.g_e + (ebase + 8 * i) * TC_F + k0 + 4 * cc4) = r4;
        }
      }
      __syncwarp();
    }
    fence_before_sync();
    TCT(13);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

// --------------------------------------------------------------------------------------------------------
// Node AND edge adjoint of one conv block in one launch: per 128-edge tile, the node MLP phase (mode 1 above) and
// then the edge MLP phase (mode 0) on the same rows.  The node phase's output ge2 = D4 + g_e2 (dL/de2) is the edge
// phase's upstream gradient and residual base; it is parked in the idle TMEM columns [448,512) (row-per-lane, exactly
// the layout the edge phase reads its upstream slice in) instead of being written to and read back from HBM (768 B
// per bond).  Per row, the MMAs and fp32 adds are those of the two conv_tc_bwds_kernel launches, in the same order, so
// every output is bitwise identical to theirs.
// Both MLPs' transposed images (2 x 128 KB) do not fit beside the z2 buffer and the staging tiles, so they stream
// through a ring of two 64 KB slots (slot 0: W2d^T | W2g^T for GEMM3, slot 1: W1e_dense^T | W1e_gate^T for GEMM4),
// refilled by cp.async.bulk from L2 as soon as the GEMM that read a slot has completed: node images, edge images, node
// images of the next tile, ...  The z2 buffer alternates the same way (node z2 of tile t, edge z2 of t, node z2 of the
// next tile).  Every barrier completes once per phase, so one parity bit (flipped per phase) serves all of them.
struct ConvTcBlockBwdParams {
  const int32_t* src; const float* h;
  const float* wimgT[2];  // [node, edge], each as ConvTcBwdSParams::wimgT
  const float* WhT[2]; const float* save[2];
  const float* g_x2; const float* g_e2;
  int64_t E; int R; int passes;
  float* g_e; float* g_z1[2]; float* g_h[2];
  int gh_mode;  // 0: node / edge g_h rows stored into g_h[0] / g_h[1]; 1: fl(node + edge) stored into g_h[0]
};
constexpr int SMEM_RING_SLOT = 2 * SMEM_S_BYTES;                   // 65536: the image pairs of one GEMM pair
constexpr int SMEM_BB_MISC = 2 * TC_BWD_MAX_R * 64 * 4 + 64;  // Wh^T of both MLPs, 5 mbarriers, TMEM slot, image pointers
constexpr int SMEM_BLOCK_BWD_BYTES = 2 * SMEM_RING_SLOT + 16 * STG_WARP_BYTES + SMEM_Z2_BYTES + SMEM_BB_MISC + 1024;
static_assert(SMEM_BLOCK_BWD_BYTES <= 232448, "fused block backward exceeds the 227 KB shared-memory limit");

__global__ void __launch_bounds__(TCB2_THREADS, 1) conv_tc_block_bwd_kernel(ConvTcBlockBwdParams p) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = (char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(smem);
  const uint32_t ring0 = sbase, ring1 = sbase + SMEM_RING_SLOT;
  const uint32_t stg_all = sbase + 2 * SMEM_RING_SLOT;
  const uint32_t z2buf = stg_all + 16 * STG_WARP_BYTES;
  float* misc = reinterpret_cast<float*>(smem + 2 * SMEM_RING_SLOT + 16 * STG_WARP_BYTES + SMEM_Z2_BYTES);
  const uint32_t wh_a = z2buf + SMEM_Z2_BYTES;  // [node | edge] Wh^T
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + 2 * TC_BWD_MAX_R * 64);
  uint32_t* tmem_slot_p = reinterpret_cast<uint32_t*>(bars + 5);
  // [node, edge] image addresses, re-read from shared memory by the refilling thread: as loop invariants held in
  // registers they would be spilled
  const float** wsrc = reinterpret_cast<const float**>(bars + 6);
  auto image_src = [&](int m) {
    uint64_t a;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(a) : "r"(smem_u32(wsrc + m)));
    return reinterpret_cast<const float*>(a);
  };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, cs = warp >> 2;
  const int row = 32 * q + lane;
  const int k0 = 16 * cs;
  const uint32_t stg = stg_all + warp * STG_WARP_BYTES;
  const int cr = lane >> 2, cc4 = lane & 3;
  const int R = p.R;
  constexpr uint32_t HALF_IMG_FLOATS = SMEM_RING_SLOT / 4;

  for (int i = tid; i < 2 * TC_BWD_MAX_R * 64; i += TCB2_THREADS) {
    const int j = i % (TC_BWD_MAX_R * 64);
    misc[i] = (j < R * 64) ? p.WhT[i / (TC_BWD_MAX_R * 64)][j] : 0.0f;
  }
  if (warp == 0) tmem_alloc<512>(tmem_slot_p);
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 5; ++i) mbar_init(&bars[i], 1);
    mbar_fence_init();
  }
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  if (*tmem_slot_p != 0u) __trap();  // one CTA per SM owns all 512 columns: literal operand addresses (see bwd2)
  constexpr uint32_t tmem = 0u;
  const uint32_t t_lane = ((uint32_t)(32 * q) << 16);
  constexpr uint32_t AH = 0, AL = 64, A2H = 128, A2L = 192, D3D = 256, D3G = 320, D4 = 384, GE2 = 448;
  uint64_t *bar3 = &bars[0], *bar4 = &bars[1], *zb = &bars[2], *rb0 = &bars[3], *rb1 = &bars[4];

  const int n_tiles = (int)((p.E + TILE_M - 1) / TILE_M);
  if (tid == 0 && (int)blockIdx.x < n_tiles) {
    wsrc[0] = p.wimgT[0];
    wsrc[1] = p.wimgT[1];
    const float* w = image_src(0);
    mbar_arrive_expect_tx(rb0, SMEM_RING_SLOT);
    bulk_g2s(ring0, w, SMEM_RING_SLOT, rb0);
    mbar_arrive_expect_tx(rb1, SMEM_RING_SLOT);
    bulk_g2s(ring1, w + HALF_IMG_FLOATS, SMEM_RING_SLOT, rb1);
    mbar_arrive_expect_tx(zb, SMEM_Z2_BYTES);
    bulk_g2s(z2buf, p.save[0] + save_offset(blockIdx.x, 2, 0, 0), SMEM_Z2_BYTES, zb);
  }
  uint32_t par = 0;
  // the node phase's upstream slice g_x2[src] of the next tile is requested one tile ahead (see conv_tc_bwds_kernel)
  float4 gnext[4];
  auto load_upstream = [&](int s_atom) {
    const float* gr = p.g_x2 + (int64_t)s_atom * TC_F + k0;
#pragma unroll
    for (int c = 0; c < 4; ++c) gnext[c] = __ldg(reinterpret_cast<const float4*>(gr + 4 * c));
  };
  if ((int)blockIdx.x < n_tiles) load_upstream(__ldg(p.src + min((int64_t)blockIdx.x * TILE_M + row, p.E - 1)));
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t e0 = (int64_t)tile * TILE_M;
    const int eg = (int)min(e0 + row, p.E - 1);  // E * R < 2^31 (checked by the host entry)
    const bool live = (e0 + row) < p.E;
    const bool more = tile + (int)gridDim.x < n_tiles;
    const int64_t ebase = e0 + 32 * q + cr;
#pragma unroll
    for (int m = 0; m < 2; ++m) {  // m = 0: node MLP (upstream g_x2[src]), m = 1: edge MLP (upstream ge2)
      const bool node = m == 0;
      const bool next_phase = node || more;
      {
        // next phase's SiLU'(z1) blocks into L2 (its z2 blocks arrive by bulk copy); the node phase also pulls the
        // next tile's g_e2 rows and h
        const int tn = node ? tile : tile + (int)gridDim.x;
        if (tn < n_tiles) prefetch_l2(p.save[m ^ 1] + (int64_t)tn * SAVE_TILE_WORDS + tid * 32);
        if (node && more) {
          const int64_t en = (int64_t)(tile + gridDim.x) * TILE_M;
          const int64_t rn = min(en + (tid & 255) / 2, p.E - 1);
          if (tid < 256) {
            if (p.g_e2) prefetch_l2(p.g_e2 + rn * TC_F + (tid & 1) * 32);
          } else if (tid < 256 + 16) {
            prefetch_l2(p.h + min(en * R + (tid - 256) * 32, p.E * R - 1));
          }
        }
      }
      // ---- T0: upstream gradient slice, saved z2 slices, h ----
      float zd[16], zg[16], gu[16];
      if (node) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          gu[4 * c] = gnext[c].x; gu[4 * c + 1] = gnext[c].y; gu[4 * c + 2] = gnext[c].z; gu[4 * c + 3] = gnext[c].w;
        }
      } else {
        tmem_ld16(t_lane + GE2 + k0, gu);  // written by this thread in the node phase
        tmem_ld_wait();
      }
      {
        mbar_wait_warp(zb, par);
        const uint32_t s2 = z2buf + ((cs * 4 + q) << 11) + 16 * lane;
        const uint32_t s3 = s2 + (16 << 11);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float4 a = lds128(s2 + 512 * c);
          float4 b = lds128(s3 + 512 * c);
          zd[4 * c] = a.x; zd[4 * c + 1] = a.y; zd[4 * c + 2] = a.z; zd[4 * c + 3] = a.w;
          zg[4 * c] = b.x; zg[4 * c + 1] = b.y; zg[4 * c + 2] = b.z; zg[4 * c + 3] = b.w;
        }
      }
      float hm[TC_BWD_MAX_R], ghp[TC_BWD_MAX_R];
#pragma unroll
      for (int mm = 0; mm < TC_BWD_MAX_R; ++mm) {
        hm[mm] = (mm < R) ? __ldg(p.h + eg * R + mm) : 0.0f;
        ghp[mm] = 0.0f;
      }
      // ---- T5: output-stage adjoint -> dz2d (operand A), dz2g (operand A2) ; GEMM3d + GEMM3g ----
      const uint32_t whm = wh_a + m * (TC_BWD_MAX_R * 64 * 4);
#pragma unroll
      for (int c = 0; c < 16; c += 4) {
        float whv[TC_BWD_MAX_R][4];
#pragma unroll
        for (int mm = 0; mm < TC_BWD_MAX_R; ++mm) {
          float4 w4 = lds128(whm + 4 * (mm * 64 + k0 + c));
          whv[mm][0] = w4.x; whv[mm][1] = w4.y; whv[mm][2] = w4.z; whv[mm][3] = w4.w;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float z = zd[c + u];
          const float sgm = sigmoid_fast(z);
          const float sd = z * sgm;
          const float sgr = sgm * (1.0f + z * (1.0f - sgm));
          const float sg = sigmoid_fast(zg[c + u]);
          float s = 0.0f;
#pragma unroll
          for (int mm = 0; mm < TC_BWD_MAX_R; ++mm) s += hm[mm] * whv[mm][u];
          const float gs = gu[c + u] * sd * sg;
#pragma unroll
          for (int mm = 0; mm < TC_BWD_MAX_R; ++mm) ghp[mm] += gs * whv[mm][u];
          const float gphi = gu[c + u] * s;
          zd[c + u] = gphi * sg * sgr;               // dz2d
          zg[c + u] = gphi * sd * sg * (1.0f - sg);  // dz2g
        }
      }
      tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, zd);
      tmem_put_split16(t_lane + A2H + k0, t_lane + A2L + k0, zg);
      if (cs != 0) sts128(stg + lane * 16, make_float4(ghp[0], ghp[1], ghp[2], 0.0f));
      tmem_st_wait();
      fence_before_sync();
      __syncthreads();
      if (tid == 0) {
        fence_after_sync();
        if (next_phase) {  // every thread has consumed this phase's z2: refill for the next phase
          fence_proxy_async();
          mbar_arrive_expect_tx(zb, SMEM_Z2_BYTES);
          bulk_g2s(z2buf, p.save[m ^ 1] + save_offset(node ? tile : tile + (int)gridDim.x, 2, 0, 0), SMEM_Z2_BYTES, zb);
        }
        mbar_wait(rb0, par);
        issue_gemm_ts(tmem + D3D, tmem + AH, tmem + AL, ring0, ring0 + IMG_W2 * 4, 64, 64, false, p.passes);
        issue_gemm_ts(tmem + D3G, tmem + A2H, tmem + A2L, ring0 + SMEM_S_BYTES, ring0 + SMEM_S_BYTES + IMG_W2 * 4, 64,
                      64, false, p.passes);
        commit(bar3);
      }
      if (cs == 0) {
        float4 g1 = lds128(stg + 4 * STG_WARP_BYTES + lane * 16);
        float4 g2 = lds128(stg + 8 * STG_WARP_BYTES + lane * 16);
        float4 g3 = lds128(stg + 12 * STG_WARP_BYTES + lane * 16);
        if (live) {
          float tot[3] = {((ghp[0] + g1.x) + g2.x) + g3.x, ((ghp[1] + g1.y) + g2.y) + g3.y,
                          ((ghp[2] + g1.z) + g2.z) + g3.z};
          float* gh = p.g_h[p.gh_mode ? 0 : m];
          if (p.gh_mode && !node) {  // this thread stored the node rows in this tile's node phase
#pragma unroll
            for (int mm = 0; mm < TC_BWD_MAX_R; ++mm)
              if (mm < R) gh[eg * R + mm] += tot[mm];
          } else {
#pragma unroll
            for (int mm = 0; mm < TC_BWD_MAX_R; ++mm)
              if (mm < R) gh[eg * R + mm] = tot[mm];
          }
        }
      }
      // saved SiLU'(z1) slices (dense -> zd, gate -> zg), in flight while GEMM3 runs
      int s_next = 0;  // edge phase: source atom of this row in the next tile
      if (!node && more) s_next = __ldg(p.src + min((int64_t)(tile + gridDim.x) * TILE_M + row, p.E - 1));
      {
        const float* s0 = p.save[m] + save_offset(tile, 0, cs, q) + 4 * lane;
        const float* s1 = p.save[m] + save_offset(tile, 1, cs, q) + 4 * lane;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float4 a = __ldg(reinterpret_cast<const float4*>(s0 + 128 * c));
          float4 b = __ldg(reinterpret_cast<const float4*>(s1 + 128 * c));
          zd[4 * c] = a.x; zd[4 * c + 1] = a.y; zd[4 * c + 2] = a.z; zd[4 * c + 3] = a.w;
          zg[4 * c] = b.x; zg[4 * c + 1] = b.y; zg[4 * c + 2] = b.z; zg[4 * c + 3] = b.w;
        }
      }
      // ---- T6: dz1 = D3 * SiLU'(z1) -> operands A (dense), A2 (gate) ; GEMM4a + GEMM4b ----
      mbar_wait_warp(bar3, par);
      fence_after_sync();
      if (tid == 0 && next_phase) {  // GEMM3 has read slot 0: the next phase's GEMM3 images
        mbar_arrive_expect_tx(rb0, SMEM_RING_SLOT);
        bulk_g2s(ring0, image_src(m ^ 1), SMEM_RING_SLOT, rb0);
      }
      {
        float v[16];
        tmem_ld16(t_lane + D3D + k0, v);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 16; ++c) zd[c] *= v[c];
        tmem_put_split16(t_lane + AH + k0, t_lane + AL + k0, zd);
        tmem_ld16(t_lane + D3G + k0, v);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 16; ++c) zg[c] *= v[c];
        tmem_put_split16(t_lane + A2H + k0, t_lane + A2L + k0, zg);
      }
      tmem_st_wait();
      fence_before_sync();
      __syncthreads();
      if (tid == 0) {
        fence_after_sync();
        mbar_wait(rb1, par);
        issue_gemm_ts(tmem + D4, tmem + AH, tmem + AL, ring1, ring1 + IMG_W2 * 4, 64, 64, false, p.passes);
        issue_gemm_ts(tmem + D4, tmem + A2H, tmem + A2L, ring1 + SMEM_S_BYTES, ring1 + SMEM_S_BYTES + IMG_W2 * 4, 64,
                      64, true, p.passes);
        commit(bar4);
      }
      float4 gb[4];
      if (node && p.g_e2) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          gb[i] = __ldg(reinterpret_cast<const float4*>(p.g_e2 + min(ebase + 8 * i, p.E - 1) * TC_F + k0 + 4 * cc4));
      }
      float* gz = p.g_z1[m];
      if (gz != nullptr) {
#pragma unroll
        for (int hb = 0; hb < 2; ++hb) {
          const float* dz = hb ? zg : zd;
#pragma unroll
          for (int c = 0; c < 4; ++c)
            sts128(stg + stg_off(lane, c), make_float4(dz[4 * c], dz[4 * c + 1], dz[4 * c + 2], dz[4 * c + 3]));
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float4 r4 = lds128(stg + stg_off(8 * i + cr, cc4));
            if (ebase + 8 * i < p.E) *reinterpret_cast<float4*>(gz + (ebase + 8 * i) * 128 + 64 * hb + k0 + 4 * cc4) = r4;
          }
          __syncwarp();
        }
      }
      if (!node && more) load_upstream(s_next);
      // ---- T7: ge2 = D4 + g_e2 into TMEM (node) | g_e = D4 + ge2 (edge) ----
      mbar_wait_warp(bar4, par);
      fence_after_sync();
      if (tid == 0 && next_phase) {  // GEMM4 has read slot 1: the next phase's GEMM4 images
        mbar_arrive_expect_tx(rb1, SMEM_RING_SLOT);
        bulk_g2s(ring1, image_src(m ^ 1) + HALF_IMG_FLOATS, SMEM_RING_SLOT, rb1);
      }
      if (node) {
        float v[16];
        tmem_ld16(t_lane + D4 + k0, v);
        tmem_ld_wait();
        if (p.g_e2) {
#pragma unroll
          for (int i = 0; i < 4; ++i) sts128(stg + stg_off(8 * i + cr, cc4), gb[i]);
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float4 b = lds128(stg + stg_off(lane, c));
            v[4 * c] += b.x; v[4 * c + 1] += b.y; v[4 * c + 2] += b.z; v[4 * c + 3] += b.w;
          }
          __syncwarp();
        }
        tmem_st16(t_lane + GE2 + k0, v);
        tmem_st_wait();
      } else {
        float v[16], b[16];
        tmem_ld16(t_lane + D4 + k0, v);
        tmem_ld16(t_lane + GE2 + k0, b);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 4; ++c)
          sts128(stg + stg_off(lane, c), make_float4(v[4 * c] + b[4 * c], v[4 * c + 1] + b[4 * c + 1],
                                                     v[4 * c + 2] + b[4 * c + 2], v[4 * c + 3] + b[4 * c + 3]));
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 r4 = lds128(stg + stg_off(8 * i + cr, cc4));
          if (ebase + 8 * i < p.E) *reinterpret_cast<float4*>(p.g_e + (ebase + 8 * i) * TC_F + k0 + 4 * cc4) = r4;
        }
        __syncwarp();
      }
      fence_before_sync();
      par ^= 1;
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

// --------------------------------------------------------------------------------------------------------
// debug: issue rate of tcgen05.mma kind::tf32 M=128 for a given N, A from shared (0) or tensor memory (1)
template <int N, int ATMEM>
__global__ void __launch_bounds__(128, 1) mma_rate_kernel(int n_rep, long long* out) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = (char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  for (int i = threadIdx.x; i < (64 + 128) * 1024 / 4; i += blockDim.x) reinterpret_cast<float*>(smem)[i] = 1.0f;
  if (threadIdx.x < 32) tmem_alloc<512>(&tmem_slot);
  if (threadIdx.x == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  if (tmem_slot != 0u) __trap();
  if (threadIdx.x == 0) {
    constexpr uint32_t idesc = make_idesc_tf32(TILE_M, N, 0);
    const uint32_t a = smem_u32(smem), b = a + 64 * 1024;
    const uint64_t da0 = make_desc(a, 16, 1024), db0 = make_desc(b, 16, 1024);
    long long t0 = clock64();
    for (int r = 0; r < n_rep; ++r) {
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const uint64_t db = db0 + (uint64_t)(((kk >> 2) * (N * 128) + (kk & 3) * 32) >> 4);
        if (ATMEM) {
          mma_tf32_ts(0u, 256u + 8 * kk, db, idesc, 1u);
        } else {
          const uint64_t da = da0 + (uint64_t)(((kk >> 2) * (TILE_M * 128) + (kk & 3) * 32) >> 4);
          mma_tf32(0u, da, db, idesc, 1u);
        }
      }
    }
    long long t1 = clock64();
    commit(&bar);
    mbar_wait(&bar, 0);
    long long t2 = clock64();
    out[0] = t1 - t0;
    out[1] = t2 - t0;
  }
  fence_before_sync();
  __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc<512>(0u);
}


// --------------------------------------------------------------------------------------------------------
// debug: issue rate of tcgen05.mma.cta_group::2 kind::tf32 (M = 256 over a CTA pair, each SM computes its own 128
// rows against the full N; each CTA holds N/2 rows of B).  Only the leader CTA issues; the commit is multicast to the
// mbarrier at the same shared-memory offset in both CTAs.
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int N>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1) mma_rate2_kernel(int n_rep, long long* out) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = (char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  uint32_t rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  for (int i = threadIdx.x; i < (64 + 64) * 1024 / 4; i += blockDim.x) reinterpret_cast<float*>(smem)[i] = 1.0f;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  fence_proxy_async();
  cluster_sync_all();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  cluster_sync_all();
  long long t0 = 0;
  if (rank == 0 && threadIdx.x == 0) {
    constexpr uint32_t idesc = make_idesc_tf32(256, N, 0);
    const uint32_t a = smem_u32(smem), b = a + 64 * 1024;
    const uint64_t da0 = make_desc(a, 16, 1024), db0 = make_desc(b, 16, 1024);
    t0 = clock64();
    for (int r = 0; r < n_rep; ++r) {
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const uint64_t db = db0 + (uint64_t)(((kk >> 2) * ((N / 2) * 128) + (kk & 3) * 32) >> 4);
        const uint64_t da = da0 + (uint64_t)(((kk >> 2) * (TILE_M * 128) + (kk & 3) * 32) >> 4);
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
            "}\n" ::"r"(0u),
            "l"(da), "l"(db), "r"(idesc), "r"(1u)
            : "memory");
      }
    }
    long long t1 = clock64();
    out[0] = t1 - t0;
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(&bar)),
        "h"((uint16_t)3)
        : "memory");
  }
  if (threadIdx.x == 0) {
    mbar_wait(&bar, 0);
    if (rank == 0) out[1] = clock64() - t0;
  }
  fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(0u), "n"(512) : "memory");
}

}  // namespace m3g

using namespace m3g;

extern "C" {

int m3g_debug_mma_rate(int N, int a_tmem, int n_mma, int64_t* cycles2, void* stream) {
  M3G_REQUIRE(cycles2 && (N == 64 || N == 128 || N == 256) && n_mma >= 8, "m3g_debug_mma_rate: bad arguments");
  int smem = (64 + 128) * 1024 + 1024;
  long long* out = (long long*)cycles2;
#define RATE_(N_, A_)                                                                                         \
  do {                                                                                                        \
    cudaFuncSetAttribute(mma_rate_kernel<N_, A_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);         \
    mma_rate_kernel<N_, A_><<<1, 128, smem, as_stream(stream)>>>(n_mma / 8, out);                             \
  } while (0)
  if (N == 64 && !a_tmem) RATE_(64, 0);
  else if (N == 64) RATE_(64, 1);
  else if (N == 128 && !a_tmem) RATE_(128, 0);
  else if (N == 128) RATE_(128, 1);
  else if (!a_tmem) RATE_(256, 0);
  else RATE_(256, 1);
#undef RATE_
  M3G_LAUNCH_CHECK("m3g_debug_mma_rate");
  return M3G_OK;
}

int m3g_debug_mma_rate2(int N, int n_mma, int64_t* cycles2, void* stream) {
  M3G_REQUIRE(cycles2 && (N == 64 || N == 128 || N == 256) && n_mma >= 8, "m3g_debug_mma_rate2: bad arguments");
  int smem = (64 + 64) * 1024 + 1024;
  long long* out = (long long*)cycles2;
#define RATE2_(N_)                                                                                       \
  do {                                                                                                   \
    cudaFuncSetAttribute(mma_rate2_kernel<N_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);       \
    mma_rate2_kernel<N_><<<2, 128, smem, as_stream(stream)>>>(n_mma / 8, out);                           \
  } while (0)
  if (N == 64) RATE2_(64); else if (N == 128) RATE2_(128); else RATE2_(256);
#undef RATE2_
  M3G_LAUNCH_CHECK("m3g_debug_mma_rate2");
  return M3G_OK;
}

int m3g_debug_tc_timing(int64_t* out16, int reset, void* stream) {
  M3G_REQUIRE(out16, "m3g_debug_tc_timing: null pointer");
  cudaError_t err = cudaStreamSynchronize(as_stream(stream));
  if (err == cudaSuccess) err = cudaMemcpyFromSymbol(out16, g_tc_timing, 16 * sizeof(unsigned long long));
  if (err == cudaSuccess && reset) {
    unsigned long long z[16] = {0};
    err = cudaMemcpyToSymbol(g_tc_timing, z, sizeof(z));
  }
  if (err != cudaSuccess) {
    set_error("m3g_debug_tc_timing: %s", cudaGetErrorString(err));
    return M3G_ERR_CUDA;
  }
  return M3G_OK;
}

int m3g_tc_pack_b(const float* W, int rows, int cols, float* img_hi, float* img_lo, void* stream) {
  M3G_REQUIRE(W && img_hi && img_lo, "m3g_tc_pack_b: null pointer");
  M3G_REQUIRE(rows % 8 == 0 && cols % 32 == 0, "m3g_tc_pack_b: rows %% 8 and cols %% 32 must be 0");
  tc_pack_kernel<<<blocks_for((int64_t)rows * cols, 256), 256, 0, as_stream(stream)>>>(W, rows, cols, img_hi, img_lo);
  M3G_LAUNCH_CHECK("m3g_tc_pack_b");
  return M3G_OK;
}

int m3g_tc_selftest(const float* A, const float* img_hi, const float* img_lo, int rows, int cols, int passes,
                    int a_tmem, float* out, void* stream) {
  M3G_REQUIRE(A && img_hi && img_lo && out, "m3g_tc_selftest: null pointer");
  M3G_REQUIRE((rows == 64 || rows == 128) && (cols == 64 || cols == 128), "m3g_tc_selftest: rows/cols in {64,128}");
  M3G_REQUIRE(passes == 1 || passes == 3, "m3g_tc_selftest: passes must be 1 or 3");
  size_t smem = 2 * (size_t)rows * cols * 4 + 2 * (size_t)TILE_M * cols * 4 + 1024;
  cudaError_t err = cudaFuncSetAttribute(tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) {
    set_error("m3g_tc_selftest: cudaFuncSetAttribute: %s", cudaGetErrorString(err));
    return M3G_ERR_CUDA;
  }
  tc_selftest_kernel<<<1, TC_THREADS, smem, as_stream(stream)>>>(A, img_hi, img_lo, rows, cols, passes, a_tmem, out);
  M3G_LAUNCH_CHECK("m3g_tc_selftest");
  return M3G_OK;
}

int64_t m3g_conv_tc_save_floats(int64_t E) { return ((E + TILE_M - 1) / TILE_M) * (int64_t)SAVE_TILE_WORDS; }

int m3g_conv_tc_fwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                    const float* h, const float* wimg, const float* b2d, const float* b2g, const float* WhT, int64_t E,
                    int R, int mode, int passes, int n_sm, float* y, float* save, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(P && src && dst && e && h && wimg && b2d && b2g && WhT && y, "m3g_conv_tc_fwd: null pointer");
  M3G_REQUIRE(R >= 1 && R <= TC3_MAX_R, "m3g_conv_tc_fwd: R=%d unsupported (max %d)", R, TC3_MAX_R);
  M3G_REQUIRE(passes == 1 || passes == 3, "m3g_conv_tc_fwd: passes must be 1 or 3");
  M3G_REQUIRE(ldp % 4 == 0 && po % 4 == 0, "m3g_conv_tc_fwd: P rows must be 16-byte aligned");
  cudaError_t err =
      cudaFuncSetAttribute(conv_tc4_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_FWD4_BYTES);
  if (err != cudaSuccess) {
    set_error("m3g_conv_tc_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(err));
    return M3G_ERR_CUDA;
  }
  ConvTcParams p{P, ldp, po, src, dst, e, h, wimg, b2d, b2g, WhT, E, R, mode, passes, y, save};
  int64_t n_tiles = (E + TILE_M - 1) / TILE_M;
  int64_t pairs = (n_tiles + 1) / 2;
  unsigned grid = (unsigned)((pairs < n_sm) ? pairs : n_sm);
  conv_tc4_fwd_kernel<<<grid, TC2_THREADS, SMEM_FWD4_BYTES, as_stream(stream)>>>(p);
  M3G_LAUNCH_CHECK("m3g_conv_tc_fwd");
  return M3G_OK;
}

int m3g_conv_tc_bwd_saved(const int32_t* src, const float* h, const float* wimgT, const float* WhT, const float* save,
                          const float* g_up, const float* g_e_base, int64_t E, int R, int mode, int passes, int n_sm,
                          float* g_e, float* g_z1, float* g_h, int gh_store, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(src && h && wimgT && WhT && save && g_up && g_e && g_h, "m3g_conv_tc_bwd_saved: null pointer");
  M3G_REQUIRE(R >= 1 && R <= TC_BWD_MAX_R, "m3g_conv_tc_bwd_saved: R=%d unsupported (max %d)", R, TC_BWD_MAX_R);
  M3G_REQUIRE(passes == 1 || passes == 3, "m3g_conv_tc_bwd_saved: passes must be 1 or 3");
  cudaError_t err =
      cudaFuncSetAttribute(conv_tc_bwds_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BWDS_BYTES);
  if (err != cudaSuccess) {
    set_error("m3g_conv_tc_bwd_saved: cudaFuncSetAttribute: %s", cudaGetErrorString(err));
    return M3G_ERR_CUDA;
  }
  ConvTcBwdSParams p{src, h, wimgT, WhT, save, g_up, g_e_base, E, R, mode, passes, g_e, g_z1, g_h, gh_store};
  int64_t n_tiles = (E + TILE_M - 1) / TILE_M;
  unsigned grid = (unsigned)((n_tiles < n_sm) ? n_tiles : n_sm);
  conv_tc_bwds_kernel<<<grid, TCB2_THREADS, SMEM_BWDS_BYTES, as_stream(stream)>>>(p);
  M3G_LAUNCH_CHECK("m3g_conv_tc_bwd_saved");
  return M3G_OK;
}

int m3g_conv_tc_block_bwd(const int32_t* src, const float* h, const float* n_wimgT, const float* n_WhT,
                          const float* save_n, const float* e_wimgT, const float* e_WhT, const float* save_e,
                          const float* g_x2, const float* g_e2, int64_t E, int R, int passes, int n_sm, float* g_e,
                          float* gz_node, float* gz_edge, float* g_h_node, float* g_h_edge, int gh_mode, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(gh_mode == 0 || gh_mode == 1, "m3g_conv_tc_block_bwd: gh_mode must be 0 or 1");
  M3G_REQUIRE(src && h && n_wimgT && n_WhT && save_n && e_wimgT && e_WhT && save_e && g_x2 && g_e && g_h_node &&
                  (gh_mode == 1 || g_h_edge),
              "m3g_conv_tc_block_bwd: null pointer");
  M3G_REQUIRE(R >= 1 && R <= TC_BWD_MAX_R, "m3g_conv_tc_block_bwd: R=%d unsupported (max %d)", R, TC_BWD_MAX_R);
  M3G_REQUIRE(E * R < ((int64_t)1 << 31), "m3g_conv_tc_block_bwd: E * R must be below 2^31");
  M3G_REQUIRE(passes == 1 || passes == 3, "m3g_conv_tc_block_bwd: passes must be 1 or 3");
  cudaError_t err =
      cudaFuncSetAttribute(conv_tc_block_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BLOCK_BWD_BYTES);
  if (err != cudaSuccess) {
    set_error("m3g_conv_tc_block_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(err));
    return M3G_ERR_CUDA;
  }
  ConvTcBlockBwdParams p{src, h, {n_wimgT, e_wimgT}, {n_WhT, e_WhT}, {save_n, save_e}, g_x2, g_e2, E, R, passes,
                         g_e, {gz_node, gz_edge}, {g_h_node, g_h_edge}, gh_mode};
  int64_t n_tiles = (E + TILE_M - 1) / TILE_M;
  unsigned grid = (unsigned)((n_tiles < n_sm) ? n_tiles : n_sm);
  conv_tc_block_bwd_kernel<<<grid, TCB2_THREADS, SMEM_BLOCK_BWD_BYTES, as_stream(stream)>>>(p);
  M3G_LAUNCH_CHECK("m3g_conv_tc_block_bwd");
  return M3G_OK;
}

int m3g_conv_tc_bwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                    const float* h, const float* wimg, const float* wimgT, const float* b2d, const float* b2g,
                    const float* WhT, const float* g_up, const float* g_e_base, int64_t E, int R, int mode, int passes,
                    int n_sm, float* g_e, float* g_z1, float* g_h, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(P && src && dst && e && h && wimg && wimgT && b2d && b2g && WhT && g_up && g_e && g_z1 && g_h,
              "m3g_conv_tc_bwd: null pointer");
  M3G_REQUIRE(R >= 1 && R <= TC_BWD_MAX_R, "m3g_conv_tc_bwd: R=%d unsupported (max %d)", R, TC_BWD_MAX_R);
  M3G_REQUIRE(passes == 1 || passes == 3, "m3g_conv_tc_bwd: passes must be 1 or 3");
  M3G_REQUIRE(ldp % 4 == 0 && po % 4 == 0, "m3g_conv_tc_bwd: P rows must be 16-byte aligned");
  cudaError_t err =
      cudaFuncSetAttribute(conv_tc_bwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BWD2_BYTES);
  if (err != cudaSuccess) {
    set_error("m3g_conv_tc_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(err));
    return M3G_ERR_CUDA;
  }
  ConvTcBwdParams p{P, ldp, po, src, dst, e, h, wimg, wimgT, b2d, b2g, WhT, g_up, g_e_base, E, R, mode, passes,
                    g_e, g_z1, g_h};
  int64_t n_tiles = (E + TILE_M - 1) / TILE_M;
  unsigned grid = (unsigned)((n_tiles < n_sm) ? n_tiles : n_sm);
  conv_tc_bwd2_kernel<<<grid, TCB2_THREADS, SMEM_BWD2_BYTES, as_stream(stream)>>>(p);
  M3G_LAUNCH_CHECK("m3g_conv_tc_bwd");
  return M3G_OK;
}

}  // extern "C"
