// Batched climbing-image NEB step (extension, no reference counterpart): one FIRE step of every running band of a
// ragged batch, with the improved tangent of Henkelman & Jonsson (J. Chem. Phys. 113, 9978 (2000)) and the climbing
// image of Henkelman, Uberuaga & Jonsson (ibid. 9901), as ASE's NEB(method="improvedtangent") under FIRE.  A band is
// images 0 .. M+1 of one structure; 0 and M+1 are fixed endpoints, the M interior images move.  One CTA per band:
//   1. per interior image, five sums over its atoms in the fixed thread-row map and tree: |t+|^2, |t-|^2, t+.t-, F.t+
//      and F.t- (t+ = R_{i+1} - R_i, t- = R_i - R_{i-1}, raw differences);
//   2. thread 0 picks each image's tangent t = c+ t+ + c- t- from the energies, the climbing image and the two
//      coefficients of G_i = F_i + alpha_i t+ + beta_i t- (DESIGN.md §8);
//   3. fire.cuh's FIRE step over the band's M n rows as one vector, forming G row by row from F and the neighbouring
//      images' positions;
//   4. the position update from the new velocities.  Positions are read in 1-3 and written only in 4, after a barrier,
//      so no image reads a neighbour that has already moved.
// The result depends only on the band's own rows; there are no atomics and no scratch.
#include "fire.cuh"

namespace m3g {

constexpr int kNebMaxImages = M3G_NEB_MAX_IMAGES;
constexpr int kNebSums = 5;

struct NebArgs {
  const float *forces, *energy;
  const int32_t *row_ptr, *image_ptr, *end_ptr;
  const double *ends, *e_end, *k;
  int climb;
  FireParams q;
  double *pos, *v;
  FireState s;
  int32_t* i_climb;
  double* e_frame;
};

// block_sum of K values at once: each in common.cuh's tree (xor butterfly, then the warps in order); sh holds
// K * kWarps doubles
template <int K, int kWarps>
__device__ __forceinline__ void block_sums(double (&t)[K], double* sh) {
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t[k] += __shfl_xor_sync(FULL, t[k], o);
  if ((threadIdx.x & 31) == 0)
#pragma unroll
    for (int k = 0; k < K; ++k) sh[k * kWarps + (threadIdx.x >> 5)] = t[k];
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < kWarps; ++q) s += sh[k * kWarps + q];
    t[k] = s;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kFireThreads) neb_step_kernel(NebArgs p) {
  const int64_t b = blockIdx.x;
  if (p.s.status[b] != kFireRunning) return;  // finished bands stay bit-untouched
  __shared__ double sh[kNebSums * kFireWarps];
  __shared__ double sums[kNebSums * kNebMaxImages];
  __shared__ double coef[2 * kNebMaxImages];  // alpha_j, beta_j of interior image j (band image j + 1)
  __shared__ int bfail;
  const int tid = threadIdx.x;
  const int64_t r0 = p.row_ptr[b], i0 = p.image_ptr[b], e0 = p.end_ptr[b];
  const int M = p.image_ptr[b + 1] - p.image_ptr[b];
  const int n = (p.end_ptr[b + 1] - p.end_ptr[b]) / 2;
  if (M < 1 || M > kNebMaxImages) {  // the host rejects these; a band that gets here anyway fails, untouched
    if (tid == 0) p.s.status[b] = kFireFailed, p.s.fmax[b] = INFINITY;
    return;
  }
  const double* first = p.ends + e0 * 3;
  const double* last = p.ends + (e0 + n) * 3;
  // atom a of band image i (0 .. M + 1)
  auto image_row = [&](int i, int a) -> const double* {
    return i == 0 ? first + a * 3 : i == M + 1 ? last + a * 3 : p.pos + (r0 + (int64_t)(i - 1) * n + a) * 3;
  };

  // pass 1: the five sums of every interior image
  for (int j = 0; j < M; ++j) {
    double t[kNebSums] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int a = tid; a < n; a += kFireThreads) {
      const double *pm = image_row(j, a), *pc = image_row(j + 1, a), *pn = image_row(j + 2, a);
      const float* f = p.forces + (r0 + (int64_t)j * n + a) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double tp = pn[c] - pc[c], tm = pc[c] - pm[c], fc = f[c];
        t[0] += tp * tp;
        t[1] += tm * tm;
        t[2] += tp * tm;
        t[3] += fc * tp;
        t[4] += fc * tm;
      }
    }
    block_sums<kNebSums, kFireWarps>(t, sh);
    if (tid == 0)
#pragma unroll
      for (int k = 0; k < kNebSums; ++k) sums[j * kNebSums + k] = t[k];
  }

  // pass 2: tangents, climbing image and the G coefficients
  if (tid == 0) {
    const double* ee = p.e_end + b * 2;
    auto E = [&](int i) -> double { return i == 0 ? ee[0] : i == M + 1 ? ee[1] : (double)p.energy[i0 + i - 1]; };
    int fail = !(isfinite(ee[0]) && isfinite(ee[1]));
    int ic = 1;
    for (int i = 1; i <= M; ++i) {
      const double e = E(i);
      p.e_frame[i0 + i - 1] = e;
      fail |= !isfinite(e);
      if (e > E(ic)) ic = i;  // ties go to the lowest index
    }
    p.i_climb[b] = ic;
    const double kb = p.k[b];
    for (int i = 1; i <= M; ++i) {
      const double El = E(i - 1), Ei = E(i), Er = E(i + 1);
      double cp, cm;
      if (Er > Ei && Ei > El) {
        cp = 1.0, cm = 0.0;
      } else if (Er < Ei && Ei < El) {
        cp = 0.0, cm = 1.0;
      } else {
        const double dmax = fmax(fabs(Er - Ei), fabs(El - Ei)), dmin = fmin(fabs(Er - Ei), fabs(El - Ei));
        if (dmax == 0.0) {
          cp = 1.0, cm = 1.0;  // flat triplet: the limit of the mixed branch
        } else if (Er > El) {
          cp = dmax, cm = dmin;
        } else {
          cp = dmin, cm = dmax;
        }
      }
      const double* S = sums + (i - 1) * kNebSums;
      const double tn = sqrt(cp * cp * S[0] + 2.0 * cp * cm * S[2] + cm * cm * S[1]);
      fail |= !(tn > 0.0 && isfinite(tn));
      const double ft = (cp * S[3] + cm * S[4]) / tn;  // F . t^
      const double sc = (p.climb && i == ic) ? -2.0 * ft : -ft + kb * (sqrt(S[0]) - sqrt(S[1]));
      coef[2 * (i - 1)] = sc * cp / tn;
      coef[2 * (i - 1) + 1] = sc * cm / tn;
    }
    if (fail) p.s.status[b] = kFireFailed, p.s.fmax[b] = INFINITY;
    bfail = fail;
  }
  __syncthreads();
  if (bfail) return;

  // pass 3: FIRE on the band's rows, G formed on the fly
  const int rows = M * n;
  auto gen = [&](int r, double* g) {
    const int j = r / n, a = r - j * n;
    const double *pm = image_row(j, a), *pc = image_row(j + 1, a), *pn = image_row(j + 2, a);
    const float* f = p.forces + (r0 + r) * 3;
    const double al = coef[2 * j], be = coef[2 * j + 1];
#pragma unroll
    for (int c = 0; c < 3; ++c) g[c] = (double)f[c] + al * (pn[c] - pc[c]) + be * (pc[c] - pm[c]);
  };
  auto vel = [&](int r) -> double* { return p.v + (r0 + r) * 3; };
  FireMove step_of;
  if (!fire_advance(p.q, p.s, b, rows, gen, vel, sh, &step_of)) return;

  // pass 4: positions (fire_advance ends in a barrier, after the last read of a neighbour's positions)
  for (int r = tid; r < rows; r += kFireThreads) {
    const double* v = p.v + (r0 + r) * 3;
    double* x = p.pos + (r0 + r) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) x[c] = x[c] + step_of(v[c]);
  }
}

}  // namespace m3g

using namespace m3g;

extern "C" {

int m3g_neb_step(const float* forces, const float* energy, const int32_t* row_ptr, const int32_t* image_ptr,
                 const int32_t* end_ptr, int64_t B, int max_images, const double* ends, const double* e_end,
                 const double* k, int climb, double dt_max, double max_move, int n_min, double f_inc, double f_dec,
                 double a_start, double f_a, double fmax_target, int max_steps, double* pos, double* v, double* dt,
                 double* a, int32_t* n_pos, int32_t* n_steps, int32_t* status, double* fmax, int32_t* i_climb,
                 double* e_frame, void* stream) {
  if (B == 0) return M3G_OK;
  M3G_REQUIRE(forces && energy && row_ptr && image_ptr && end_ptr && ends && e_end && k && pos && v && dt && a &&
                  n_pos && n_steps && status && fmax && i_climb && e_frame,
              "m3g_neb_step: null pointer");
  M3G_REQUIRE(max_images >= 1 && max_images <= kNebMaxImages,
              "m3g_neb_step: %d interior images per band, expected 1 .. %d", max_images, kNebMaxImages);
  M3G_REQUIRE(B <= 0x7fffffff, "m3g_neb_step: B=%lld too large", (long long)B);
  NebArgs p{forces, energy, row_ptr, image_ptr, end_ptr, ends, e_end, k, climb,
            FireParams{dt_max, max_move, f_inc, f_dec, a_start, f_a, fmax_target, n_min, max_steps},
            pos, v, FireState{dt, a, fmax, n_pos, n_steps, status}, i_climb, e_frame};
  neb_step_kernel<<<(unsigned)B, kFireThreads, 0, as_stream(stream)>>>(p);
  M3G_LAUNCH_CHECK("m3g_neb_step");
  return M3G_OK;
}

}  // extern "C"
