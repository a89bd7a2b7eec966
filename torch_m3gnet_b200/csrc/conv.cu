// M3GNetConv (nn/conv.py:63-97) — generic-width fp32 kernels: one warp owns EPW edges (rows), lanes own
// output features, weights stream through L1 in (in,out) layout so that every weight load is coalesced
// and reused for EPW rows.  The first GatedMLP layer is split algebraically
//   [x_i, x_j, e] W1 = x_i W1_i + x_j W1_j + e W1_e
// so the x parts are per-atom projections (m3g_linear_fwd) gathered per edge; this halves the per-edge FLOPs.
// The F=64 tensor-core path lives in conv_tc.cu; this file is the reference-width-agnostic path (F <= 128).
#include "common.cuh"

namespace m3g {

constexpr int EPW = 4;           // rows per warp
constexpr int WARPS_PER_BLOCK = 4;

// acc[q][j] += sum_k xs[q][k] * Wt[k*ldw + lane + 32 j]
template <int NJ>
__device__ __forceinline__ void warp_matvec(const float* xs, int xs_stride, int K, const float* __restrict__ Wt,
                                            int ldw, int ncols, int lane, float (&acc)[EPW][NJ]) {
  for (int k = 0; k < K; ++k) {
    float w[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      int col = lane + 32 * j;
      w[j] = (col < ncols) ? Wt[(int64_t)k * ldw + col] : 0.0f;
    }
#pragma unroll
    for (int q = 0; q < EPW; ++q) {
      float xv = xs[q * xs_stride + k];
#pragma unroll
      for (int j = 0; j < NJ; ++j) acc[q][j] += xv * w[j];
    }
  }
}

// out (n,M) = base + in (n,K) Wt (K,M) + bias.  K is consumed in chunks of KC staged through shared memory.
constexpr int LIN_KC = 128;
__global__ void linear_kernel(const float* __restrict__ in, const float* __restrict__ Wt,
                              const float* __restrict__ bias, const float* __restrict__ base, int64_t n, int K, int M,
                              float* __restrict__ out) {
  __shared__ float xs_all[WARPS_PER_BLOCK][EPW][LIN_KC];
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t row0 = ((int64_t)blockIdx.x * WARPS_PER_BLOCK + warp) * EPW;
  if (row0 >= n) return;
  float(*xs)[LIN_KC] = xs_all[warp];
  for (int c0 = 0; c0 < M; c0 += 128) {
    float acc[EPW][4];
#pragma unroll
    for (int q = 0; q < EPW; ++q)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[q][j] = 0.0f;
    for (int k0 = 0; k0 < K; k0 += LIN_KC) {
      int kc = min(LIN_KC, K - k0);
      __syncwarp();
      for (int q = 0; q < EPW; ++q) {
        int64_t row = min(row0 + q, n - 1);
        for (int k = lane; k < kc; k += 32) xs[q][k] = in[row * K + k0 + k];
      }
      __syncwarp();
      warp_matvec<4>(&xs[0][0], LIN_KC, kc, Wt + (int64_t)k0 * M + c0, M, M - c0, lane, acc);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int col = c0 + lane + 32 * j;
      if (col < M) {
        float b = bias ? bias[col] : 0.0f;
#pragma unroll
        for (int q = 0; q < EPW; ++q) {
          int64_t row = row0 + q;
          if (row < n) out[row * M + col] = acc[q][j] + b + (base ? base[row * M + col] : 0.0f);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Shared-memory tiled fp32 GEMM for the per-atom projections: out (n,M) = base + in (n,K) Wt (K,M) + bias, with
// K % 32 == 0 and M % 64 == 0.  Block tile BM x 64, K chunks of 32 staged in shared memory (A transposed so that
// both operands are read as float4), thread tile (BM/16) x 4, k ascending per output (deterministic order).
template <int BM>
__global__ void __launch_bounds__(256) linear_tiled_kernel(const float* __restrict__ in, const float* __restrict__ Wt,
                                                           const float* __restrict__ bias,
                                                           const float* __restrict__ base, int64_t n, int K, int M,
                                                           float* __restrict__ out) {
  constexpr int BN = 64, BK = 32, TM = BM / 16;
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // 16 column groups x 16 row groups
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int col0 = blockIdx.y * BN;
  float acc[TM][4];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  for (int k0 = 0; k0 < K; k0 += BK) {
    // A chunk (BM x 32): each thread loads float4 along k and stores it transposed
#pragma unroll
    for (int i = 0; i < BM / 32; ++i) {
      int idx = tid + 256 * i;
      int r = idx >> 3, c4 = idx & 7;
      int64_t row = min(row0 + r, n - 1);
      float4 v = __ldg(reinterpret_cast<const float4*>(in + row * K + k0) + c4);
      As[4 * c4 + 0][r] = v.x; As[4 * c4 + 1][r] = v.y; As[4 * c4 + 2][r] = v.z; As[4 * c4 + 3][r] = v.w;
    }
    // B chunk (32 x 64)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int idx = tid + 256 * i;
      int r = idx >> 4, c4 = idx & 15;
      *reinterpret_cast<float4*>(&Bs[r][4 * c4]) =
          __ldg(reinterpret_cast<const float4*>(Wt + (int64_t)(k0 + r) * M + col0) + c4);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM];
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        float4 t = *reinterpret_cast<const float4*>(&As[k][TM * ty + i]);
        a[i] = t.x; a[i + 1] = t.y; a[i + 2] = t.z; a[i + 3] = t.w;
      }
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][4 * tx]);
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        acc[i][0] += a[i] * b.x; acc[i][1] += a[i] * b.y; acc[i][2] += a[i] * b.z; acc[i][3] += a[i] * b.w;
      }
    }
    __syncthreads();
  }
  float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias) bv = __ldg(reinterpret_cast<const float4*>(bias + col0) + tx);
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int64_t row = row0 + TM * ty + i;
    if (row >= n) continue;
    float4 r4 = make_float4(acc[i][0] + bv.x, acc[i][1] + bv.y, acc[i][2] + bv.z, acc[i][3] + bv.w);
    if (base) {
      float4 b4 = __ldg(reinterpret_cast<const float4*>(base + row * M + col0) + tx);
      r4.x += b4.x; r4.y += b4.y; r4.z += b4.z; r4.w += b4.w;
    }
    reinterpret_cast<float4*>(out + row * M + col0)[tx] = r4;
  }
}

static inline bool launch_linear_tiled(const float* in, const float* Wt, const float* bias, const float* base,
                                       int64_t n, int K, int M, float* out, cudaStream_t stream) {
  if (K % 32 != 0 || M % 64 != 0) return false;
  if (M >= 256) {
    dim3 grid((unsigned)((n + 127) / 128), (unsigned)(M / 64));
    linear_tiled_kernel<128><<<grid, 256, 0, stream>>>(in, Wt, bias, base, n, K, M, out);
  } else {
    dim3 grid((unsigned)((n + 63) / 64), (unsigned)(M / 64));
    linear_tiled_kernel<64><<<grid, 256, 0, stream>>>(in, Wt, bias, base, n, K, M, out);
  }
  return true;
}

// ---------------------------------------------------------------------------------------------------
// forward of one gated MLP on edges
template <int NJ>
__global__ void conv_mlp_fwd_kernel(const float* __restrict__ P, int ldp, int po, const int32_t* __restrict__ src,
                                    const int32_t* __restrict__ dst, const float* __restrict__ e,
                                    const float* __restrict__ h, const float* __restrict__ W1eT,
                                    const float* __restrict__ W2dT, const float* __restrict__ b2d,
                                    const float* __restrict__ W2gT, const float* __restrict__ b2g,
                                    const float* __restrict__ WhT, int64_t E, int F, int R, int mode,
                                    float* __restrict__ y) {
  extern __shared__ float smem[];
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t e0 = ((int64_t)blockIdx.x * WARPS_PER_BLOCK + warp) * EPW;
  if (e0 >= E) return;
  const int F2 = 2 * F;
  float* in_s = smem + warp * (EPW * 3 * F);  // [EPW][F]
  float* a1_s = in_s + EPW * F;               // [EPW][2F]
  int64_t eq[EPW];
#pragma unroll
  for (int q = 0; q < EPW; ++q) eq[q] = min(e0 + q, E - 1);
  for (int q = 0; q < EPW; ++q)
    for (int k = lane; k < F; k += 32) in_s[q * F + k] = e[eq[q] * F + k];
  __syncwarp();
  // layer 1 (2F columns: dense | gate)
  {
    float acc[EPW][2 * NJ];
#pragma unroll
    for (int q = 0; q < EPW; ++q) {
      const float* Pi = P + (int64_t)src[eq[q]] * ldp + po;
      const float* Pj = P + (int64_t)dst[eq[q]] * ldp + po + F2;
#pragma unroll
      for (int j = 0; j < 2 * NJ; ++j) {
        int col = lane + 32 * j;
        acc[q][j] = (col < F2) ? Pi[col] + Pj[col] : 0.0f;
      }
    }
    warp_matvec<2 * NJ>(in_s, F, F, W1eT, F2, F2, lane, acc);
#pragma unroll
    for (int q = 0; q < EPW; ++q)
#pragma unroll
      for (int j = 0; j < 2 * NJ; ++j) {
        int col = lane + 32 * j;
        if (col < F2) a1_s[q * F2 + col] = silu_acc(acc[q][j]);
      }
  }
  __syncwarp();
  // layer 2
  float ad[EPW][NJ], ag[EPW][NJ];
#pragma unroll
  for (int q = 0; q < EPW; ++q)
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      int col = lane + 32 * j;
      ad[q][j] = (col < F) ? b2d[col] : 0.0f;
      ag[q][j] = (col < F) ? b2g[col] : 0.0f;
    }
  warp_matvec<NJ>(a1_s, F2, F, W2dT, F, F, lane, ad);
  warp_matvec<NJ>(a1_s + F, F2, F, W2gT, F, F, lane, ag);
#pragma unroll
  for (int q = 0; q < EPW; ++q) {
    if (e0 + q < E) {
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        int col = lane + 32 * j;
        if (col < F) {
          float s = 0.0f;
          for (int m = 0; m < R; ++m) s += h[eq[q] * R + m] * WhT[m * F + col];
          float out = silu_acc(ad[q][j]) * sigmoid_acc(ag[q][j]) * s;
          y[eq[q] * F + col] = (mode == 0) ? in_s[q * F + col] + out : out;
        }
      }
    }
  }
}

// out[i] = base[i] + sum over the atom's edge segment (ascending edge order), one warp per atom
__global__ void segment_sum_add_kernel(const float* __restrict__ base, const float* __restrict__ msg,
                                       const int32_t* __restrict__ edge_ptr, int64_t N, int F,
                                       float* __restrict__ out) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (i >= N) return;
  int b = edge_ptr[i], en = edge_ptr[i + 1];
  for (int col = lane; col < F; col += 32) {
    float acc = 0.0f;
    for (int e = b; e < en; ++e) acc += msg[(int64_t)e * F + col];
    out[i * F + col] = base[i * F + col] + acc;
  }
}

// out[i] = base[i] + sum of the per-(32-row block, atom) partial message rows that m3g_conv_tc_fwd(mode 2) left at the
// block's first row of the atom: rows max(b, 32 k) for k = b / 32 .. (en - 1) / 32, ascending.  One warp per atom, F = 64.
__global__ void segment_sum_parts_kernel(const float* __restrict__ base, const float* __restrict__ part,
                                         const int32_t* __restrict__ edge_ptr, int64_t N, float* __restrict__ out) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (i >= N) return;
  const int b = edge_ptr[i], en = edge_ptr[i + 1];
  float2 acc = make_float2(0.f, 0.f);
  if (en > b) {
    for (int k = b >> 5; k <= (en - 1) >> 5; ++k) {
      const int row = max(b, k << 5);
      const float2 v = __ldg(reinterpret_cast<const float2*>(part + (int64_t)row * 64) + lane);
      acc.x += v.x; acc.y += v.y;
    }
  }
  const float2 x = __ldg(reinterpret_cast<const float2*>(base + i * 64) + lane);
  reinterpret_cast<float2*>(out + i * 64)[lane] = make_float2(x.x + acc.x, x.y + acc.y);
}

// ---------------------------------------------------------------------------------------------------
// adjoint of one gated MLP on edges (forward recomputed)
template <int NJ>
__global__ void conv_mlp_bwd_kernel(const float* __restrict__ P, int ldp, int po, const int32_t* __restrict__ src,
                                    const int32_t* __restrict__ dst, const float* __restrict__ e,
                                    const float* __restrict__ h, const float* __restrict__ W1eT,
                                    const float* __restrict__ W2dT, const float* __restrict__ b2d,
                                    const float* __restrict__ W2gT, const float* __restrict__ b2g,
                                    const float* __restrict__ WhT, const float* __restrict__ W1e,
                                    const float* __restrict__ W2d, const float* __restrict__ W2g,
                                    const float* __restrict__ g_up, const float* __restrict__ g_e_base, int64_t E,
                                    int F, int R, int mode, float* __restrict__ g_e, float* __restrict__ g_z1,
                                    float* __restrict__ g_h) {
  extern __shared__ float smem[];
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t e0 = ((int64_t)blockIdx.x * WARPS_PER_BLOCK + warp) * EPW;
  if (e0 >= E) return;
  const int F2 = 2 * F;
  float* in_s = smem + warp * (EPW * 5 * F);  // [EPW][F]   e rows
  float* z1_s = in_s + EPW * F;               // [EPW][2F]  pre-activations, later dz1
  float* a1_s = z1_s + EPW * F2;              // [EPW][2F]  activations, later dz2
  int64_t eq[EPW];
#pragma unroll
  for (int q = 0; q < EPW; ++q) eq[q] = min(e0 + q, E - 1);
  for (int q = 0; q < EPW; ++q)
    for (int k = lane; k < F; k += 32) in_s[q * F + k] = e[eq[q] * F + k];
  __syncwarp();
  {
    float acc[EPW][2 * NJ];
#pragma unroll
    for (int q = 0; q < EPW; ++q) {
      const float* Pi = P + (int64_t)src[eq[q]] * ldp + po;
      const float* Pj = P + (int64_t)dst[eq[q]] * ldp + po + F2;
#pragma unroll
      for (int j = 0; j < 2 * NJ; ++j) {
        int col = lane + 32 * j;
        acc[q][j] = (col < F2) ? Pi[col] + Pj[col] : 0.0f;
      }
    }
    warp_matvec<2 * NJ>(in_s, F, F, W1eT, F2, F2, lane, acc);
#pragma unroll
    for (int q = 0; q < EPW; ++q)
#pragma unroll
      for (int j = 0; j < 2 * NJ; ++j) {
        int col = lane + 32 * j;
        if (col < F2) {
          z1_s[q * F2 + col] = acc[q][j];
          a1_s[q * F2 + col] = silu_acc(acc[q][j]);
        }
      }
  }
  __syncwarp();
  float ad[EPW][NJ], ag[EPW][NJ];
#pragma unroll
  for (int q = 0; q < EPW; ++q)
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      int col = lane + 32 * j;
      ad[q][j] = (col < F) ? b2d[col] : 0.0f;
      ag[q][j] = (col < F) ? b2g[col] : 0.0f;
    }
  warp_matvec<NJ>(a1_s, F2, F, W2dT, F, F, lane, ad);
  warp_matvec<NJ>(a1_s + F, F2, F, W2gT, F, F, lane, ag);
  __syncwarp();  // everyone is done reading a1_s before it is overwritten with dz2
  // output stage adjoint
  float gh_part[EPW][M3G_MAX_RADIAL];
#pragma unroll
  for (int q = 0; q < EPW; ++q)
#pragma unroll
    for (int m = 0; m < M3G_MAX_RADIAL; ++m) gh_part[q][m] = 0.0f;
#pragma unroll
  for (int q = 0; q < EPW; ++q) {
    const float* gu_row = (mode == 0) ? g_up + eq[q] * F : g_up + (int64_t)src[eq[q]] * F;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      int col = lane + 32 * j;
      float dzd = 0.0f, dzg = 0.0f;
      if (col < F) {
        float gu = gu_row[col];
        float s = 0.0f;
        for (int m = 0; m < R; ++m) s += h[eq[q] * R + m] * WhT[m * F + col];
        float zd = ad[q][j], zg = ag[q][j];
        float sd = silu_acc(zd), sg = sigmoid_acc(zg);
        float phi = sd * sg;
        float gs = gu * phi;
#pragma unroll
        for (int m = 0; m < M3G_MAX_RADIAL; ++m)
          if (m < R) gh_part[q][m] += gs * WhT[m * F + col];
        float gphi = gu * s;
        dzd = gphi * sg * silu_grad(zd);
        dzg = gphi * sd * sg * (1.0f - sg);
        a1_s[q * F2 + col] = dzd;
        a1_s[q * F2 + F + col] = dzg;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < EPW; ++q)
#pragma unroll
    for (int m = 0; m < M3G_MAX_RADIAL; ++m)
      if (m < R) {
        float t = warp_sum(gh_part[q][m]);
        if (lane == 0 && e0 + q < E) g_h[eq[q] * R + m] += t;
      }
  __syncwarp();
  // layer-2 adjoint: da1[k] = sum_f dz2[f] W2[f][k]  (W2 in (out,in) layout → coalesced over k)
  {
    float dd[EPW][NJ], dg[EPW][NJ];
#pragma unroll
    for (int q = 0; q < EPW; ++q)
#pragma unroll
      for (int j = 0; j < NJ; ++j) { dd[q][j] = 0.0f; dg[q][j] = 0.0f; }
    warp_matvec<NJ>(a1_s, F2, F, W2d, F, F, lane, dd);
    warp_matvec<NJ>(a1_s + F, F2, F, W2g, F, F, lane, dg);
    // dz1 = da1 * SiLU'(z1): each lane rewrites exactly the z1_s entries it reads
#pragma unroll
    for (int q = 0; q < EPW; ++q)
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        int col = lane + 32 * j;
        if (col < F) {
          float v0 = dd[q][j] * silu_grad(z1_s[q * F2 + col]);
          float v1 = dg[q][j] * silu_grad(z1_s[q * F2 + F + col]);
          z1_s[q * F2 + col] = v0;
          z1_s[q * F2 + F + col] = v1;
          if (e0 + q < E) {
            g_z1[eq[q] * F2 + col] = v0;
            g_z1[eq[q] * F2 + F + col] = v1;
          }
        }
      }
  }
  __syncwarp();
  // layer-1 adjoint w.r.t. e: g_e[k] = base + sum_c dz1[c] W1e[c][k]   (W1e (2F,F) in (out,in) layout)
  {
    float ge[EPW][NJ];
#pragma unroll
    for (int q = 0; q < EPW; ++q)
#pragma unroll
      for (int j = 0; j < NJ; ++j) ge[q][j] = 0.0f;
    warp_matvec<NJ>(z1_s, F2, F2, W1e, F, F, lane, ge);
#pragma unroll
    for (int q = 0; q < EPW; ++q)
      if (e0 + q < E) {
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          int col = lane + 32 * j;
          if (col < F) g_e[eq[q] * F + col] = ge[q][j] + (g_e_base ? g_e_base[eq[q] * F + col] : 0.0f);
        }
      }
  }
}

// g_P[i][po .. po+2F) = sum_{out(i)} g_z1 ; g_P[i][po+2F .. po+4F) = sum_{in(i)} g_z1 (ascending edge order)
__global__ void conv_gather_gz_kernel(const float* __restrict__ g_z1, const int32_t* __restrict__ edge_ptr,
                                      const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_perm,
                                      int64_t N, int F2, int ldp, int po, float* __restrict__ g_P) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (i >= N) return;
  int ob = edge_ptr[i], oe = edge_ptr[i + 1];
  int ib = in_ptr[i], ie = in_ptr[i + 1];
  for (int col = lane; col < F2; col += 32) {
    float a = 0.0f;
    for (int e = ob; e < oe; ++e) a += g_z1[(int64_t)e * F2 + col];
    g_P[i * ldp + po + col] = a;
    float b = 0.0f;
    for (int p = ib; p < ie; ++p) b += g_z1[(int64_t)in_perm[p] * F2 + col];
    g_P[i * ldp + po + F2 + col] = b;
  }
}

// F2 == 128: one float4 per lane covers the whole row (512-byte warp loads), 8 rows in flight per step; every column
// still adds its rows one by one in ascending edge order (the loads are batched, the adds are not reordered).  One warp
// per (atom, side): the source-side and the destination-side sums are independent latency chains, so they run in
// different warps (ncu on the one-warp-per-atom version: 22 long-scoreboard stalls per issue at 34 % occupancy).
__global__ void __launch_bounds__(256, 4)
conv_gather_gz128_kernel(const float* __restrict__ g_z1, const int32_t* __restrict__ edge_ptr,
                         const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_perm, int64_t N, int ldp,
                         int po, float* __restrict__ g_P) {
  constexpr int U = 8;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t i = w >> 1;
  const int side = (int)(w & 1);
  int lane = threadIdx.x & 31;
  if (i >= N) return;
  const float4* gz = reinterpret_cast<const float4*>(g_z1);
  if (side == 0) {
    const int ob = edge_ptr[i], oe = edge_ptr[i + 1];
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e0 = ob; e0 < oe; e0 += U) {
      float4 r[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (e0 + u < oe) r[u] = __ldg(gz + (int64_t)(e0 + u) * 32 + lane);
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (e0 + u < oe) { a.x += r[u].x; a.y += r[u].y; a.z += r[u].z; a.w += r[u].w; }
    }
    reinterpret_cast<float4*>(g_P + i * ldp + po)[lane] = a;
  } else {
    const int ib = in_ptr[i], ie = in_ptr[i + 1];
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p0 = ib; p0 < ie; p0 += U) {
      int idx[U];
#pragma unroll
      for (int u = 0; u < U; ++u) idx[u] = (p0 + u < ie) ? __ldg(in_perm + p0 + u) : 0;
      float4 r[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (p0 + u < ie) r[u] = __ldg(gz + (int64_t)idx[u] * 32 + lane);
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (p0 + u < ie) { b.x += r[u].x; b.y += r[u].y; b.z += r[u].z; b.w += r[u].w; }
    }
    reinterpret_cast<float4*>(g_P + i * ldp + po + 128)[lane] = b;
  }
}

template <typename K>
static int set_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (err != cudaSuccess) {
      set_error("cudaFuncSetAttribute(%zu B): %s", bytes, cudaGetErrorString(err));
      return M3G_ERR_CUDA;
    }
  }
  return M3G_OK;
}

}  // namespace m3g

using namespace m3g;

extern "C" {

int m3g_linear_fwd(const float* in, const float* Wt, const float* bias, int64_t n, int K, int M, float* out,
                   void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(in && Wt && out && K > 0 && M > 0, "m3g_linear_fwd: bad argument");
  if (!launch_linear_tiled(in, Wt, bias, nullptr, n, K, M, out, as_stream(stream)))
    linear_kernel<<<blocks_for(n, WARPS_PER_BLOCK * EPW), WARPS_PER_BLOCK * 32, 0, as_stream(stream)>>>(
        in, Wt, bias, nullptr, n, K, M, out);
  M3G_LAUNCH_CHECK("m3g_linear_fwd");
  return M3G_OK;
}

int m3g_linear_bwd_input(const float* g, const float* W, const float* base, int64_t n, int K, int M, float* out,
                         void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(g && W && out && K > 0 && M > 0, "m3g_linear_bwd_input: bad argument");
  // out (n,K) = base + g (n,M) · W (M,K): the same kernel with the roles of K and M exchanged
  if (!launch_linear_tiled(g, W, nullptr, base, n, M, K, out, as_stream(stream)))
    linear_kernel<<<blocks_for(n, WARPS_PER_BLOCK * EPW), WARPS_PER_BLOCK * 32, 0, as_stream(stream)>>>(
        g, W, nullptr, base, n, M, K, out);
  M3G_LAUNCH_CHECK("m3g_linear_bwd_input");
  return M3G_OK;
}

int m3g_conv_mlp_fwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                     const float* h, const float* W1eT, const float* W2dT, const float* b2d, const float* W2gT,
                     const float* b2g, const float* WhT, int64_t E, int F, int R, int mode, float* y, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(P && src && dst && e && h && W1eT && W2dT && b2d && W2gT && b2g && WhT && y,
              "m3g_conv_mlp_fwd: null pointer");
  M3G_REQUIRE(F >= 1 && F <= M3G_MAX_F, "m3g_conv_mlp_fwd: F=%d outside [1,%d]", F, M3G_MAX_F);
  M3G_REQUIRE(R >= 1 && R <= M3G_MAX_RADIAL, "m3g_conv_mlp_fwd: R=%d unsupported", R);
  size_t smem = (size_t)WARPS_PER_BLOCK * EPW * 3 * F * sizeof(float);
  unsigned grid = blocks_for(E, WARPS_PER_BLOCK * EPW);
  int nj = (F + 31) / 32;
#define LAUNCH_(NJ)                                                                                             \
  do {                                                                                                          \
    int rc = set_smem(conv_mlp_fwd_kernel<NJ>, smem);                                                           \
    if (rc) return rc;                                                                                          \
    conv_mlp_fwd_kernel<NJ><<<grid, WARPS_PER_BLOCK * 32, smem, as_stream(stream)>>>(                           \
        P, ldp, po, src, dst, e, h, W1eT, W2dT, b2d, W2gT, b2g, WhT, E, F, R, mode, y);                         \
  } while (0)
  if (nj == 1) LAUNCH_(1); else if (nj == 2) LAUNCH_(2); else if (nj == 3) LAUNCH_(3); else LAUNCH_(4);
#undef LAUNCH_
  M3G_LAUNCH_CHECK("m3g_conv_mlp_fwd");
  return M3G_OK;
}

int m3g_segment_sum_add(const float* base, const float* msg, const int32_t* edge_ptr, int64_t N, int F, float* out,
                        void* stream) {
  if (N == 0) return M3G_OK;
  M3G_REQUIRE(base && msg && edge_ptr && out, "m3g_segment_sum_add: null pointer");
  M3G_REQUIRE(F >= 1 && F <= M3G_MAX_F, "m3g_segment_sum_add: F=%d outside [1,%d]", F, M3G_MAX_F);
  segment_sum_add_kernel<<<blocks_for(N * 32, 256), 256, 0, as_stream(stream)>>>(base, msg, edge_ptr, N, F, out);
  M3G_LAUNCH_CHECK("m3g_segment_sum_add");
  return M3G_OK;
}

int m3g_segment_sum_parts(const float* base, const float* part, const int32_t* edge_ptr, int64_t N, int F,
                          float* out, void* stream) {
  if (N == 0) return M3G_OK;
  M3G_REQUIRE(base && part && edge_ptr && out, "m3g_segment_sum_parts: null pointer");
  M3G_REQUIRE(F == 64, "m3g_segment_sum_parts: F=%d (the tensor-core forward that writes the partial rows is F = 64)", F);
  segment_sum_parts_kernel<<<blocks_for(N * 32, 256), 256, 0, as_stream(stream)>>>(base, part, edge_ptr, N, out);
  M3G_LAUNCH_CHECK("m3g_segment_sum_parts");
  return M3G_OK;
}

int m3g_conv_mlp_bwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                     const float* h, const float* W1eT, const float* W2dT, const float* b2d, const float* W2gT,
                     const float* b2g, const float* WhT, const float* W1e, const float* W2d, const float* W2g,
                     const float* Wh, const float* g_up, const float* g_e_base, int64_t E, int F, int R, int mode,
                     float* g_e, float* g_z1, float* g_h, void* stream) {
  (void)Wh;
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(P && src && dst && e && h && W1eT && W2dT && b2d && W2gT && b2g && WhT && W1e && W2d && W2g && g_up &&
                  g_e && g_z1 && g_h,
              "m3g_conv_mlp_bwd: null pointer");
  M3G_REQUIRE(F >= 1 && F <= M3G_MAX_F, "m3g_conv_mlp_bwd: F=%d outside [1,%d]", F, M3G_MAX_F);
  M3G_REQUIRE(R >= 1 && R <= M3G_MAX_RADIAL, "m3g_conv_mlp_bwd: R=%d unsupported", R);
  size_t smem = (size_t)WARPS_PER_BLOCK * EPW * 5 * F * sizeof(float);
  unsigned grid = blocks_for(E, WARPS_PER_BLOCK * EPW);
  int nj = (F + 31) / 32;
#define LAUNCH_(NJ)                                                                                             \
  do {                                                                                                          \
    int rc = set_smem(conv_mlp_bwd_kernel<NJ>, smem);                                                           \
    if (rc) return rc;                                                                                          \
    conv_mlp_bwd_kernel<NJ><<<grid, WARPS_PER_BLOCK * 32, smem, as_stream(stream)>>>(                           \
        P, ldp, po, src, dst, e, h, W1eT, W2dT, b2d, W2gT, b2g, WhT, W1e, W2d, W2g, g_up, g_e_base, E, F, R,    \
        mode, g_e, g_z1, g_h);                                                                                  \
  } while (0)
  if (nj == 1) LAUNCH_(1); else if (nj == 2) LAUNCH_(2); else if (nj == 3) LAUNCH_(3); else LAUNCH_(4);
#undef LAUNCH_
  M3G_LAUNCH_CHECK("m3g_conv_mlp_bwd");
  return M3G_OK;
}

int m3g_conv_gather_gz(const float* g_z1, const int32_t* edge_ptr, const int32_t* in_ptr, const int32_t* in_perm,
                       int64_t N, int F, int ldp, int po, float* g_P, void* stream) {
  if (N == 0) return M3G_OK;
  M3G_REQUIRE(g_z1 && edge_ptr && in_ptr && in_perm && g_P, "m3g_conv_gather_gz: null pointer");
  M3G_REQUIRE(F >= 1 && F <= M3G_MAX_F, "m3g_conv_gather_gz: F=%d outside [1,%d]", F, M3G_MAX_F);
  if (F == 64 && ldp % 4 == 0 && po % 4 == 0)
    conv_gather_gz128_kernel<<<blocks_for(N * 64, 256), 256, 0, as_stream(stream)>>>(g_z1, edge_ptr, in_ptr, in_perm, N,
                                                                                     ldp, po, g_P);
  else
    conv_gather_gz_kernel<<<blocks_for(N * 32, 256), 256, 0, as_stream(stream)>>>(g_z1, edge_ptr, in_ptr, in_perm, N,
                                                                                  2 * F, ldp, po, g_P);
  M3G_LAUNCH_CHECK("m3g_conv_gather_gz");
  return M3G_OK;
}

}  // extern "C"
