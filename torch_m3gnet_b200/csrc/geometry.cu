// Geometry, radial basis, embedding and edge-feature initialisation kernels (HBM-bound elementwise /
// gather work: one coalesced pass per tensor, no shared memory needed).
#include "common.cuh"

namespace m3g {

__global__ void scale_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t n, float ls) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __fdiv_rn(in[i], ls);
}

// nn/invariant.py:44-59.  Contraction is disabled (explicit _rn ops) so that distances round exactly like
// the reference's separate mul / sum / add / sub tensor ops.
__global__ void geometry_fwd_kernel(const float* __restrict__ pos, const float* __restrict__ lattice,
                                    const int32_t* __restrict__ batch, const int32_t* __restrict__ src,
                                    const int32_t* __restrict__ dst, const int32_t* __restrict__ shift, int64_t E,
                                    float4* __restrict__ vec4, float* __restrict__ dist) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int i = src[e], j = dst[e];
  const float* Lm = lattice + (int64_t)batch[i] * 9;
  float s0 = (float)shift[e * 3 + 0], s1 = (float)shift[e * 3 + 1], s2 = (float)shift[e * 3 + 2];
  float v[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float sh = __fadd_rn(__fadd_rn(__fmul_rn(s0, Lm[0 + a]), __fmul_rn(s1, Lm[3 + a])), __fmul_rn(s2, Lm[6 + a]));
    v[a] = __fsub_rn(__fadd_rn(pos[(int64_t)j * 3 + a], sh), pos[(int64_t)i * 3 + a]);
  }
  float r2 = __fadd_rn(__fadd_rn(__fmul_rn(v[0], v[0]), __fmul_rn(v[1], v[1])), __fmul_rn(v[2], v[2]));
  float r = __fsqrt_rn(r2);
  vec4[e] = make_float4(v[0], v[1], v[2], r);
  dist[e] = r;
}

__global__ void angles_fwd_kernel(const float4* __restrict__ vec4, const int64_t* __restrict__ tri, int64_t T,
                                  float* __restrict__ cos_out) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  float4 a = vec4[tri[t]];
  float4 b = vec4[tri[T + t]];
  float dot = __fadd_rn(__fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fmul_rn(a.z, b.z));
  float c = __fdiv_rn(dot, __fmul_rn(a.w, b.w));
  cos_out[t] = fminf(fmaxf(c, -1.0f), 1.0f);
}

__global__ void angles_bwd_kernel(const float4* __restrict__ vec4, const int64_t* __restrict__ tri,
                                  const float* __restrict__ g_cos, int64_t T, float* __restrict__ g_vec4) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  int64_t e1 = tri[t], e2 = tri[T + t];
  float4 a = vec4[e1];
  float4 b = vec4[e2];
  // c rounded exactly as angles_fwd_kernel forms it: the clamp passes the gradient where the forward's unclamped c lies
  // in [-1, 1] (torch.clamp takes its mask from its input); a contracted dot * (1 / (|a||b|)) can land an ulp across
  // the bound at collinear bonds
  float dot = __fadd_rn(__fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fmul_rn(a.z, b.z));
  float c = __fdiv_rn(dot, __fmul_rn(a.w, b.w));
  if (!(c >= -1.0f && c <= 1.0f)) return;
  float inv = 1.0f / (a.w * b.w);
  float g = g_cos[t];
  atomicAdd(&g_vec4[e1 * 4 + 0], g * b.x * inv);
  atomicAdd(&g_vec4[e1 * 4 + 1], g * b.y * inv);
  atomicAdd(&g_vec4[e1 * 4 + 2], g * b.z * inv);
  atomicAdd(&g_vec4[e1 * 4 + 3], -g * c / a.w);
  atomicAdd(&g_vec4[e2 * 4 + 0], g * a.x * inv);
  atomicAdd(&g_vec4[e2 * 4 + 1], g * a.y * inv);
  atomicAdd(&g_vec4[e2 * 4 + 2], g * a.z * inv);
  atomicAdd(&g_vec4[e2 * 4 + 3], -g * c / b.w);
}

// One warp per atom: g_pos[i] = scale * (sum_{in(i)} g_e - sum_{out(i)} g_e),
// g_e = g_vec4.xyz + (g_vec4.w + g_dist) * v / r
__global__ void geometry_bwd_kernel(const float4* __restrict__ vec4, const float4* __restrict__ g_vec4,
                                    const float* __restrict__ g_dist, const int32_t* __restrict__ edge_ptr,
                                    const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_perm,
                                    int64_t N, float scale, float* __restrict__ g_pos) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (i >= N) return;
  float ax = 0.f, ay = 0.f, az = 0.f;
  for (int p = in_ptr[i] + lane; p < in_ptr[i + 1]; p += 32) {
    int e = in_perm[p];
    float4 v = vec4[e];
    float4 g = g_vec4 ? g_vec4[e] : make_float4(0.f, 0.f, 0.f, 0.f);
    float gr = g.w + (g_dist ? g_dist[e] : 0.0f);
    float s = gr / v.w;
    ax += g.x + s * v.x;
    ay += g.y + s * v.y;
    az += g.z + s * v.z;
  }
  for (int e = edge_ptr[i] + lane; e < edge_ptr[i + 1]; e += 32) {
    float4 v = vec4[e];
    float4 g = g_vec4 ? g_vec4[e] : make_float4(0.f, 0.f, 0.f, 0.f);
    float gr = g.w + (g_dist ? g_dist[e] : 0.0f);
    float s = gr / v.w;
    ax -= g.x + s * v.x;
    ay -= g.y + s * v.y;
    az -= g.z + s * v.z;
  }
  ax = warp_sum(ax);
  ay = warp_sum(ay);
  az = warp_sum(az);
  if (lane == 0) {
    g_pos[i * 3 + 0] = ax * scale;
    g_pos[i * 3 + 1] = ay * scale;
    g_pos[i * 3 + 2] = az * scale;
  }
}

// normalised sinc of torch (quirk Q2): sin(pi a)/(pi a), 1 at a == 0
__device__ __forceinline__ float sinc_n(float a) {
  if (a == 0.0f) return 1.0f;
  float p = 3.14159265358979323846f * a;
  return sinf(p) / p;
}
__device__ __forceinline__ float sinc_n_grad(float a) {
  if (a == 0.0f) return 0.0f;
  float p = 3.14159265358979323846f * a;
  return (cosf(p) - sinf(p) / p) / a;
}

// consts: [k_0..k_R | coeff_0.. | a_0.. | b_0..]
__global__ void radial_fwd_kernel(const float* __restrict__ dist, const float* __restrict__ consts, int64_t E, int R,
                                  float* __restrict__ h) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const float* k = consts;
  const float* coeff = consts + (R + 1);
  const float* am = coeff + R;
  const float* bm = am + R;
  float r = dist[e];
  float s_prev = sinc_n(k[0] * r);
  float h_prev = 0.0f;
  for (int m = 0; m < R; ++m) {
    float s_next = sinc_n(k[m + 1] * r);
    float f = coeff[m] * (s_prev + s_next);
    float hm = (m == 0) ? f : (f + am[m] * h_prev) / bm[m];
    h[e * R + m] = hm;
    h_prev = hm;
    s_prev = s_next;
  }
}

__global__ void radial_bwd_kernel(const float* __restrict__ dist, const float* __restrict__ consts,
                                  const float* __restrict__ g_h, int64_t E, int R, float* __restrict__ g_dist) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const float* k = consts;
  const float* coeff = consts + (R + 1);
  const float* am = coeff + R;
  const float* bm = am + R;
  float r = dist[e];
  float d_prev = sinc_n_grad(k[0] * r) * k[0];
  float dh_prev = 0.0f;
  float acc = 0.0f;
  for (int m = 0; m < R; ++m) {
    float d_next = sinc_n_grad(k[m + 1] * r) * k[m + 1];
    float df = coeff[m] * (d_prev + d_next);
    float dh = (m == 0) ? df : (df + am[m] * dh_prev) / bm[m];
    acc += g_h[e * R + m] * dh;
    dh_prev = dh;
    d_prev = d_next;
  }
  g_dist[e] = acc;
}

__global__ void atomref_kernel(const float* __restrict__ table, const int32_t* __restrict__ types, int64_t N,
                               float* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) out[i] = table[types[i]];
}

__global__ void embed_kernel(const float* __restrict__ W, const int32_t* __restrict__ types, int64_t N, int F,
                             int num_types, float* __restrict__ x) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * F) return;
  int64_t i = idx / F;
  int f = (int)(idx - i * F);
  x[idx] = W[(int64_t)f * num_types + types[i]];
}

__global__ void edge_adjust_fwd_kernel(const float* __restrict__ h, const float* __restrict__ Wt, int64_t E, int R,
                                       int F, float* __restrict__ e0) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= E * F) return;
  int64_t e = idx / F;
  int f = (int)(idx - e * F);
  float z = 0.0f;
  for (int m = 0; m < R; ++m) z += h[e * R + m] * Wt[m * F + f];
  e0[idx] = silu_acc(z);
}

// exp2 / reciprocal on the special-function unit, as in the gated-MLP epilogues (csrc/conv_tc.cu): relative error of a
// few 1e-7, an order of magnitude below the tolerances on edge_attr (the accurate expf + IEEE division cost ~3x the
// instructions and made these two kernels issue-bound at 40 % of the HBM rate)
__device__ __forceinline__ float sigmoid_q(float z) { return __fdividef(1.0f, 1.0f + __expf(-z)); }
__device__ __forceinline__ float silu_q(float z) { return z * sigmoid_q(z); }
__device__ __forceinline__ float silu_grad_q(float z) {
  const float s = sigmoid_q(z);
  return s * (1.0f + z * (1.0f - s));
}

// F % 4 == 0: one thread per 4 consecutive features (float4 stores, the h row is a broadcast inside the row's threads)
template <int RC>
__global__ void edge_adjust_fwd4_kernel(const float* __restrict__ h, const float* __restrict__ Wt, int64_t E, int R,
                                        int F, float* __restrict__ e0) {
  const int F4 = F >> 2;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= E * F4) return;
  int64_t e = idx / F4;
  int f = 4 * (int)(idx - e * F4);
  float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int m = 0; m < RC; ++m) {
    if (m < R) {
      float hv = __ldg(h + e * R + m);
      float4 w = __ldg(reinterpret_cast<const float4*>(Wt + m * F + f));
      z.x += hv * w.x; z.y += hv * w.y; z.z += hv * w.z; z.w += hv * w.w;
    }
  }
  reinterpret_cast<float4*>(e0 + e * F)[f >> 2] = make_float4(silu_q(z.x), silu_q(z.y), silu_q(z.z), silu_q(z.w));
}

// one warp per edge
__global__ void edge_adjust_bwd_kernel(const float* __restrict__ h, const float* __restrict__ Wt,
                                       const float* __restrict__ g_e0, int64_t E, int R, int F,
                                       float* __restrict__ g_h) {
  int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (e >= E) return;
  float acc[M3G_MAX_RADIAL];
#pragma unroll
  for (int m = 0; m < M3G_MAX_RADIAL; ++m) acc[m] = 0.0f;
  for (int f = lane; f < F; f += 32) {
    float z = 0.0f;
    for (int m = 0; m < R; ++m) z += h[e * R + m] * Wt[m * F + f];
    float gz = g_e0[e * F + f] * silu_grad(z);
#pragma unroll
    for (int m = 0; m < M3G_MAX_RADIAL; ++m)
      if (m < R) acc[m] += gz * Wt[m * F + f];
  }
#pragma unroll
  for (int m = 0; m < M3G_MAX_RADIAL; ++m) {
    if (m < R) {
      float s = warp_sum(acc[m]);
      if (lane == 0) g_h[e * R + m] = s;
    }
  }
}

// F == 64, R <= 4: 16 lanes per edge, one float4 of the upstream row per lane, butterfly over the 16 lanes
template <int RC>
__global__ void edge_adjust_bwd64_kernel(const float* __restrict__ h, const float* __restrict__ Wt,
                                         const float* __restrict__ g_e0, int64_t E, int R, float* __restrict__ g_h) {
  constexpr int F = 64;
  int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  const int gl = threadIdx.x & 15;
  const bool valid = e < E;
  const int64_t ec = valid ? e : (E - 1);
  float hv[RC];
  float4 w[RC];
#pragma unroll
  for (int m = 0; m < RC; ++m) {
    hv[m] = (m < R) ? __ldg(h + ec * R + m) : 0.0f;
    w[m] = (m < R) ? __ldg(reinterpret_cast<const float4*>(Wt + m * F) + gl) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float4 g = __ldg(reinterpret_cast<const float4*>(g_e0 + ec * F) + gl);
  float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int m = 0; m < RC; ++m) { z.x += hv[m] * w[m].x; z.y += hv[m] * w[m].y; z.z += hv[m] * w[m].z; z.w += hv[m] * w[m].w; }
  const float gx = g.x * silu_grad_q(z.x), gy = g.y * silu_grad_q(z.y), gz = g.z * silu_grad_q(z.z),
              gw = g.w * silu_grad_q(z.w);
#pragma unroll
  for (int m = 0; m < RC; ++m) {
    float a = ((gx * w[m].x + gy * w[m].y) + gz * w[m].z) + gw * w[m].w;
    a = group_sum<16>(a);
    if (valid && gl == 0 && m < R) g_h[e * R + m] = a;
  }
}

// forces = -g_pos; virial per structure (one warp per structure)
__global__ void forces_kernel(const float* __restrict__ g_pos, int64_t n, float* __restrict__ forces) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) forces[i] = -g_pos[i];
}

__global__ void virial_kernel(const float* __restrict__ pos, const float* __restrict__ forces,
                              const float* __restrict__ lattice, const int32_t* __restrict__ atom_ptr, int64_t B,
                              float* __restrict__ stresses) {
  int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (b >= B) return;
  // Voigt order of nn/gradient.py:50-59: xx, yy, zz, yz, zx, xy with s[a][c] = sum pos_a F_c
  float s[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = atom_ptr[b] + lane; i < atom_ptr[b + 1]; i += 32) {
    float px = pos[i * 3 + 0], py = pos[i * 3 + 1], pz = pos[i * 3 + 2];
    float fx = forces[i * 3 + 0], fy = forces[i * 3 + 1], fz = forces[i * 3 + 2];
    s[0] += px * fx;
    s[1] += py * fy;
    s[2] += pz * fz;
    s[3] += py * fz;
    s[4] += pz * fx;
    s[5] += px * fy;
  }
  const float* Lm = lattice + b * 9;
  // a . (b x c)
  float cx = Lm[4] * Lm[8] - Lm[5] * Lm[7];
  float cy = Lm[5] * Lm[6] - Lm[3] * Lm[8];
  float cz = Lm[3] * Lm[7] - Lm[4] * Lm[6];
  float vol = fabsf(Lm[0] * cx + Lm[1] * cy + Lm[2] * cz);
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    float t = warp_sum(s[k]);
    if (lane == 0) stresses[b * 6 + k] = t / vol;
  }
}

// Cell stress as the strain derivative of the energy (no reference counterpart): W_b = sum_{e in b} v_e (x) g_e with
// g_e = g_vec4.xyz + (g_vec4.w + g_dist) v/r, sigma_b = W_b / |det lattice_b|.  Deterministic two-stage reduction in
// float64.  Stage 1: block c owns the bonds [c*CH, (c+1)*CH) and writes one partial per (structure b, chunk c) segment
// at slot b + c (both indices are non-decreasing along the bonds and never repeat together, so slots are distinct).
// Stage 2: one warp per structure sums its slots b + c0 .. b + c1 in a fixed order.
constexpr int kVirialThreads = 256;
constexpr int kVirialChunk = 2048;

__device__ __forceinline__ int64_t structure_first_bond(const int32_t* edge_ptr, const int32_t* atom_ptr, int64_t b) {
  return edge_ptr[atom_ptr[b]];
}

__global__ void __launch_bounds__(kVirialThreads) bond_virial_partial_kernel(
    const float4* __restrict__ vec4, const float4* __restrict__ g_vec4, const float* __restrict__ g_dist,
    const int32_t* __restrict__ edge_ptr, const int32_t* __restrict__ atom_ptr, int64_t E, int64_t B,
    double* __restrict__ part) {
  __shared__ double red[kVirialThreads / 32][9];
  __shared__ int64_t seg[2];
  const int64_t c = blockIdx.x;
  const int64_t c_begin = c * kVirialChunk;
  const int64_t c_end = min(c_begin + (int64_t)kVirialChunk, E);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t start = c_begin;
  while (start < c_end) {
    if (threadIdx.x == 0) {
      // structure of bond `start`: last b with first_bond(b) <= start (empty structures share their first bond with
      // the next one, so the search lands on the structure that owns the bond)
      int64_t lo = 0, hi = B - 1;
      while (lo < hi) {
        int64_t mid = (lo + hi + 1) >> 1;
        if (structure_first_bond(edge_ptr, atom_ptr, mid) <= start) lo = mid;
        else hi = mid - 1;
      }
      seg[0] = lo;
      seg[1] = min((int64_t)edge_ptr[atom_ptr[lo + 1]], c_end);
    }
    __syncthreads();
    const int64_t b = seg[0], stop = seg[1];
    double w[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) w[k] = 0.0;
    for (int64_t e = start + threadIdx.x; e < stop; e += kVirialThreads) {
      const float4 v = vec4[e];
      const float4 g = g_vec4 ? g_vec4[e] : make_float4(0.f, 0.f, 0.f, 0.f);
      const float s = (g.w + (g_dist ? g_dist[e] : 0.0f)) / v.w;
      const double ge[3] = {(double)(g.x + s * v.x), (double)(g.y + s * v.y), (double)(g.z + s * v.z)};
      const double vv[3] = {(double)v.x, (double)v.y, (double)v.z};
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int k = 0; k < 3; ++k) w[3 * a + k] += vv[a] * ge[k];
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      double t = w[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (lane == 0) red[warp][k] = t;
    }
    __syncthreads();
    if (threadIdx.x < 9) {
      double t = 0.0;
#pragma unroll
      for (int q = 0; q < kVirialThreads / 32; ++q) t += red[q][threadIdx.x];
      part[(b + c) * 9 + threadIdx.x] = t;
    }
    start = stop;
    __syncthreads();  // seg / red are rewritten by the next segment
  }
}

__global__ void bond_virial_finish_kernel(const double* __restrict__ part, const int32_t* __restrict__ edge_ptr,
                                          const int32_t* __restrict__ atom_ptr, const float* __restrict__ lattice,
                                          int64_t B, float* __restrict__ sigma) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const int64_t s = edge_ptr[atom_ptr[b]], t = edge_ptr[atom_ptr[b + 1]];
  double w[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) w[k] = 0.0;
  if (t > s) {
    const int64_t c0 = s / kVirialChunk, c1 = (t - 1) / kVirialChunk;
    for (int64_t c = c0 + lane; c <= c1; c += 32)
#pragma unroll
      for (int k = 0; k < 9; ++k) w[k] += part[(b + c) * 9 + k];
  }
  const float* Lm = lattice + b * 9;
  const double vol = fabs((double)Lm[0] * ((double)Lm[4] * Lm[8] - (double)Lm[5] * Lm[7]) +
                          (double)Lm[1] * ((double)Lm[5] * Lm[6] - (double)Lm[3] * Lm[8]) +
                          (double)Lm[2] * ((double)Lm[3] * Lm[7] - (double)Lm[4] * Lm[6]));
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    double x = w[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) sigma[b * 9 + k] = (float)(x / vol);
  }
}

}  // namespace m3g

using namespace m3g;

extern "C" {

int m3g_scale_fwd(const float* in, float* out, int64_t n, float length_scale, void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(in && out, "m3g_scale_fwd: null pointer");
  scale_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(in, out, n, length_scale);
  M3G_LAUNCH_CHECK("m3g_scale_fwd");
  return M3G_OK;
}

int m3g_geometry_fwd(const float* pos, const float* lattice, const int32_t* batch, const int32_t* src,
                     const int32_t* dst, const int32_t* shift, int64_t E, float* vec4, float* dist, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(pos && lattice && batch && src && dst && shift && vec4 && dist, "m3g_geometry_fwd: null pointer");
  geometry_fwd_kernel<<<blocks_for(E, 256), 256, 0, as_stream(stream)>>>(pos, lattice, batch, src, dst, shift, E,
                                                                         (float4*)vec4, dist);
  M3G_LAUNCH_CHECK("m3g_geometry_fwd");
  return M3G_OK;
}

int m3g_angles_fwd(const float* vec4, const int64_t* tri_index, int64_t T, float* cos_out, void* stream) {
  if (T == 0) return M3G_OK;
  M3G_REQUIRE(vec4 && tri_index && cos_out, "m3g_angles_fwd: null pointer");
  angles_fwd_kernel<<<blocks_for(T, 256), 256, 0, as_stream(stream)>>>((const float4*)vec4, tri_index, T, cos_out);
  M3G_LAUNCH_CHECK("m3g_angles_fwd");
  return M3G_OK;
}

int m3g_angles_bwd(const float* vec4, const int64_t* tri_index, const float* g_cos, int64_t T, float* g_vec4,
                   void* stream) {
  if (T == 0) return M3G_OK;
  M3G_REQUIRE(vec4 && tri_index && g_cos && g_vec4, "m3g_angles_bwd: null pointer");
  angles_bwd_kernel<<<blocks_for(T, 256), 256, 0, as_stream(stream)>>>((const float4*)vec4, tri_index, g_cos, T,
                                                                       g_vec4);
  M3G_LAUNCH_CHECK("m3g_angles_bwd");
  return M3G_OK;
}

int m3g_geometry_bwd(const float* vec4, const float* g_vec4, const float* g_dist, const int32_t* edge_ptr,
                     const int32_t* in_ptr, const int32_t* in_perm, int64_t N, float scale, float* g_pos,
                     void* stream) {
  if (N == 0) return M3G_OK;
  M3G_REQUIRE(vec4 && edge_ptr && in_ptr && in_perm && g_pos, "m3g_geometry_bwd: null pointer");
  geometry_bwd_kernel<<<blocks_for(N * 32, 256), 256, 0, as_stream(stream)>>>(
      (const float4*)vec4, (const float4*)g_vec4, g_dist, edge_ptr, in_ptr, in_perm, N, scale, g_pos);
  M3G_LAUNCH_CHECK("m3g_geometry_bwd");
  return M3G_OK;
}

int m3g_radial_fwd(const float* dist, const float* consts, int64_t E, int R, float* h, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(dist && consts && h, "m3g_radial_fwd: null pointer");
  M3G_REQUIRE(R >= 1 && R <= M3G_MAX_RADIAL, "m3g_radial_fwd: n_max=%d outside [1,%d]", R, M3G_MAX_RADIAL);
  radial_fwd_kernel<<<blocks_for(E, 256), 256, 0, as_stream(stream)>>>(dist, consts, E, R, h);
  M3G_LAUNCH_CHECK("m3g_radial_fwd");
  return M3G_OK;
}

int m3g_radial_bwd(const float* dist, const float* consts, const float* g_h, int64_t E, int R, float* g_dist,
                   void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(dist && consts && g_h && g_dist, "m3g_radial_bwd: null pointer");
  M3G_REQUIRE(R >= 1 && R <= M3G_MAX_RADIAL, "m3g_radial_bwd: n_max=%d outside [1,%d]", R, M3G_MAX_RADIAL);
  radial_bwd_kernel<<<blocks_for(E, 256), 256, 0, as_stream(stream)>>>(dist, consts, g_h, E, R, g_dist);
  M3G_LAUNCH_CHECK("m3g_radial_bwd");
  return M3G_OK;
}

int m3g_atomref_fwd(const float* table, const int32_t* types, int64_t N, float* out, void* stream) {
  if (N == 0) return M3G_OK;
  M3G_REQUIRE(table && types && out, "m3g_atomref_fwd: null pointer");
  atomref_kernel<<<blocks_for(N, 256), 256, 0, as_stream(stream)>>>(table, types, N, out);
  M3G_LAUNCH_CHECK("m3g_atomref_fwd");
  return M3G_OK;
}

int m3g_embed_fwd(const float* weight, const int32_t* types, int64_t N, int F, int num_types, float* x,
                  void* stream) {
  if (N == 0) return M3G_OK;
  M3G_REQUIRE(weight && types && x && F > 0 && num_types > 0, "m3g_embed_fwd: bad argument");
  embed_kernel<<<blocks_for(N * F, 256), 256, 0, as_stream(stream)>>>(weight, types, N, F, num_types, x);
  M3G_LAUNCH_CHECK("m3g_embed_fwd");
  return M3G_OK;
}

int m3g_edge_adjust_fwd(const float* h, const float* Wt, int64_t E, int R, int F, float* e0, void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(h && Wt && e0, "m3g_edge_adjust_fwd: null pointer");
  M3G_REQUIRE(R >= 1 && R <= M3G_MAX_RADIAL, "m3g_edge_adjust_fwd: n_max=%d outside [1,%d]", R, M3G_MAX_RADIAL);
  M3G_REQUIRE(F >= 1 && F <= M3G_MAX_F, "m3g_edge_adjust_fwd: F=%d outside [1,%d]", F, M3G_MAX_F);
  if (F % 4 == 0 && R == 3)
    edge_adjust_fwd4_kernel<3><<<blocks_for(E * (F / 4), 256), 256, 0, as_stream(stream)>>>(h, Wt, E, R, F, e0);
  else if (F % 4 == 0 && R <= 4)
    edge_adjust_fwd4_kernel<4><<<blocks_for(E * (F / 4), 256), 256, 0, as_stream(stream)>>>(h, Wt, E, R, F, e0);
  else
    edge_adjust_fwd_kernel<<<blocks_for(E * F, 256), 256, 0, as_stream(stream)>>>(h, Wt, E, R, F, e0);
  M3G_LAUNCH_CHECK("m3g_edge_adjust_fwd");
  return M3G_OK;
}

int m3g_edge_adjust_bwd(const float* h, const float* Wt, const float* g_e0, int64_t E, int R, int F, float* g_h,
                        void* stream) {
  if (E == 0) return M3G_OK;
  M3G_REQUIRE(h && Wt && g_e0 && g_h, "m3g_edge_adjust_bwd: null pointer");
  M3G_REQUIRE(R >= 1 && R <= M3G_MAX_RADIAL, "m3g_edge_adjust_bwd: n_max=%d outside [1,%d]", R, M3G_MAX_RADIAL);
  M3G_REQUIRE(F >= 1 && F <= M3G_MAX_F, "m3g_edge_adjust_bwd: F=%d outside [1,%d]", F, M3G_MAX_F);
  if (F == 64 && R == 3)
    edge_adjust_bwd64_kernel<3><<<blocks_for(E * 16, 256), 256, 0, as_stream(stream)>>>(h, Wt, g_e0, E, R, g_h);
  else if (F == 64 && R <= 4)
    edge_adjust_bwd64_kernel<4><<<blocks_for(E * 16, 256), 256, 0, as_stream(stream)>>>(h, Wt, g_e0, E, R, g_h);
  else
    edge_adjust_bwd_kernel<<<blocks_for(E * 32, 256), 256, 0, as_stream(stream)>>>(h, Wt, g_e0, E, R, F, g_h);
  M3G_LAUNCH_CHECK("m3g_edge_adjust_bwd");
  return M3G_OK;
}

int m3g_forces_virial(const float* pos, const float* g_pos, const float* lattice, const int32_t* atom_ptr,
                      int64_t N, int64_t B, float* forces, float* stresses, void* stream) {
  M3G_REQUIRE(pos && g_pos && lattice && atom_ptr && forces && stresses, "m3g_forces_virial: null pointer");
  if (N > 0) forces_kernel<<<blocks_for(N * 3, 256), 256, 0, as_stream(stream)>>>(g_pos, N * 3, forces);
  if (B > 0)
    virial_kernel<<<blocks_for(B * 32, 128), 128, 0, as_stream(stream)>>>(pos, forces, lattice, atom_ptr, B, stresses);
  M3G_LAUNCH_CHECK("m3g_forces_virial");
  return M3G_OK;
}

int64_t m3g_bond_virial_work_elems(int64_t E, int64_t B) {
  return 9 * (B + (E + kVirialChunk - 1) / kVirialChunk);
}

int m3g_bond_virial(const float* vec4, const float* g_vec4, const float* g_dist, const int32_t* edge_ptr,
                    const int32_t* atom_ptr, int64_t E, int64_t B, const float* lattice, double* work, float* sigma,
                    void* stream) {
  if (B == 0) return M3G_OK;
  M3G_REQUIRE(edge_ptr && atom_ptr && lattice && work && sigma, "m3g_bond_virial: null pointer");
  M3G_REQUIRE(E == 0 || vec4, "m3g_bond_virial: null vec4");
  const int64_t chunks = (E + kVirialChunk - 1) / kVirialChunk;
  // a chunk-less batch (no bonds) still takes one (empty) stage-1 block: two launches per call, always
  bond_virial_partial_kernel<<<chunks > 0 ? chunks : 1, kVirialThreads, 0, as_stream(stream)>>>(
      (const float4*)vec4, (const float4*)g_vec4, g_dist, edge_ptr, atom_ptr, E, B, work);
  bond_virial_finish_kernel<<<blocks_for(B * 32, 128), 128, 0, as_stream(stream)>>>(work, edge_ptr, atom_ptr, lattice,
                                                                                    B, sigma);
  M3G_LAUNCH_CHECK("m3g_bond_virial");
  return M3G_OK;
}

}  // extern "C"
