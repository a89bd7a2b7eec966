// Batched harmonic phonons (extension, no reference counterpart): finite-displacement force constants, dynamical
// matrices, their eigenvalues and the harmonic thermal properties of many structures at once.  Everything is float64.
// Every sum runs in a fixed order that depends only on the structure's own data (no atomics), so a structure's output
// is bitwise the same whatever else is in the batch.
//   m3g_phonon_force_constants  one 256-thread block per structure: central differences, then `symmetrize` rounds of
//                               the index-permuted transpose average and the acoustic sum rule (ASE's
//                               Phonons.read(symmetrize=k, acoustic=True) order);
//   m3g_phonon_dynmat           D(q) of every (structure, q) into global memory (tests, cuSOLVER comparison);
//   m3g_phonon_frequencies      one block per (structure, q): D(q) built by the same device function into shared
//                               memory, its Hermitian part, eigenvalues by a cyclic complex Jacobi method with
//                               round-robin pair ordering (3n/2 disjoint rotations per round), sorted;
//   m3g_phonon_thermal          one block per (structure, temperature): F, S, Cv and E as block_sum reductions over the
//                               structure's mesh frequencies, n_imaginary and the lowest frequency.
#include "common.cuh"

namespace m3g {

constexpr int kPhThreads = 256;
constexpr int kPhWarps = kPhThreads / 32;
constexpr int kPhMaxAtoms = M3G_PHONON_MAX_ATOMS;
constexpr int kPhMaxDim = 3 * kPhMaxAtoms;
constexpr int kPhMaxSweeps = 30;
constexpr double kPhTol = 1e-13;  // converged: off-diagonal Frobenius norm <= kPhTol ||D||_F

struct PhCell {
  int n, r1, r2, r3, L, N;
  int64_t pair0;  // first (kappa, j) pair of the structure (fc rows of 9, sv_ptr entries)
};

__device__ __forceinline__ PhCell ph_cell(const int32_t* atom_ptr, const int32_t* reps, const int64_t* pair_ptr,
                                          int64_t b) {
  PhCell c;
  c.n = atom_ptr[b + 1] - atom_ptr[b];
  c.r1 = reps[3 * b], c.r2 = reps[3 * b + 1], c.r3 = reps[3 * b + 2];
  c.L = c.r1 * c.r2 * c.r3;
  c.N = c.n * c.L;
  c.pair0 = pair_ptr[b];
  return c;
}

// the structure whose q range [q_ptr[b], q_ptr[b+1]) holds q (q_ptr ascending, B + 1 entries)
__device__ __forceinline__ int64_t ph_owner(const int32_t* q_ptr, int64_t B, int64_t q) {
  int64_t lo = 0, hi = B;  // invariant: q_ptr[lo] <= q < q_ptr[hi]
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (q_ptr[mid] <= q) lo = mid; else hi = mid;
  }
  return lo;
}

// ------------------------------------------------------------------------------------------------------------------
// force constants
// ------------------------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kPhThreads) phonon_fc_kernel(const float* __restrict__ forces,
                                                               const int64_t* __restrict__ row_ptr,
                                                               const int32_t* __restrict__ atom_ptr,
                                                               const int32_t* __restrict__ reps,
                                                               const int64_t* __restrict__ pair_ptr, double h,
                                                               int symmetrize, double* __restrict__ fc,
                                                               int32_t* __restrict__ status,
                                                               double* __restrict__ residual) {
  __shared__ double sh[kPhWarps];
  __shared__ double rowsum[9 * kPhMaxAtoms];
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x;
  const PhCell c = ph_cell(atom_ptr, reps, pair_ptr, b);
  const float* F = forces + row_ptr[b] * 3;
  const int64_t N = c.N, rows = (6 * (int64_t)c.n + 1) * N;
  double* P = fc + c.pair0 * 9;
  const int64_t E = (int64_t)c.n * N * 9;

  int bad = 0;
  double fm = 0.0;
  for (int64_t r = tid; r < rows; r += kPhThreads) {
    const double x = F[3 * r], y = F[3 * r + 1], z = F[3 * r + 2];
    bad |= !(isfinite(x) && isfinite(y) && isfinite(z));
    if (r < N) fm = fmax(fm, sqrt(x * x + y * y + z * z));
  }
  bad = __syncthreads_or(bad);
  fm = block_max<kPhWarps>(fm, sh);
  if (bad) {
    for (int64_t e = tid; e < E; e += kPhThreads) P[e] = NAN;
    if (tid == 0) status[b] = 1, residual[b] = NAN;
    return;
  }
  if (tid == 0) status[b] = 0, residual[b] = fm;

  // Phi(0 kappa alpha; j beta) = -(F_j beta(+h) - F_j beta(-h)) / 2h; supercell 1 + 2 (3 kappa + alpha) is +h
  const double inv2h = 1.0 / (2.0 * h);
  for (int64_t e = tid; e < E; e += kPhThreads) {
    const int64_t kj = e / 9;
    const int ab = (int)(e - kj * 9), al = ab / 3, be = ab - 3 * al;
    const int64_t kap = kj / N, j = kj - kap * N;
    const int64_t sp = 1 + 2 * (3 * kap + al);
    const double fp = F[(sp * N + j) * 3 + be], fmn = F[((sp + 1) * N + j) * 3 + be];
    P[e] = -(fp - fmn) * inv2h;
  }
  __syncthreads();

  for (int round = 0; round < symmetrize; ++round) {
    // Phi(0k; l k')_ab <- (Phi(0k; l k')_ab + Phi(0k'; -l k)_ba) / 2, each pair of entries by one thread
    for (int64_t e = tid; e < E; e += kPhThreads) {
      const int64_t kj = e / 9;
      const int ab = (int)(e - kj * 9), al = ab / 3, be = ab - 3 * al;
      const int64_t kap = kj / N, j = kj - kap * N;
      const int64_t l = j / c.n, kp = j - l * c.n;
      const int i3 = (int)(l % c.r3), i2 = (int)((l / c.r3) % c.r2), i1 = (int)(l / ((int64_t)c.r3 * c.r2));
      const int m1 = (c.r1 - i1) % c.r1, m2 = (c.r2 - i2) % c.r2, m3 = (c.r3 - i3) % c.r3;
      const int64_t ml = ((int64_t)m1 * c.r2 + m2) * c.r3 + m3;
      const int64_t e2 = ((kp * N + ml * c.n + kap) * 3 + be) * 3 + al;
      if (e < e2) {
        const double avg = 0.5 * (P[e] + P[e2]);
        P[e] = avg;
        P[e2] = avg;
      }
    }
    __syncthreads();
    // acoustic sum rule: the self block Phi(0k; 0k) loses the row sum over every j (taken before the subtraction)
    for (int t = tid; t < 9 * c.n; t += kPhThreads) {
      const int kap = t / 9, ab = t - 9 * kap;
      const double* row = P + (int64_t)kap * N * 9 + ab;
      double s = 0.0;
      for (int64_t j = 0; j < N; ++j) s += row[j * 9];
      rowsum[t] = s;
    }
    __syncthreads();
    for (int t = tid; t < 9 * c.n; t += kPhThreads) {
      const int kap = t / 9, ab = t - 9 * kap;
      P[((int64_t)kap * N + kap) * 9 + ab] -= rowsum[t];
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------------------------
// dynamical matrix
// ------------------------------------------------------------------------------------------------------------------

// 1 / m for an image count m >= 1: a float estimate and two Newton steps (relative error far below 1e-16), without
// the division's slow-path call, whose register clobbers made the dynamical-matrix loop spill
__device__ __forceinline__ double ph_recip_count(int64_t m) {
  const double x = (double)m;
  double r = (double)__frcp_rn((float)m);
  r = fma(r, fma(-x, r, 1.0), r);
  return fma(r, fma(-x, r, 1.0), r);
}

// D_{k a, k' b}(q) = sum_l Phi(0k; l k')_ab (1/|M|) sum_{v in M(k, l k')} exp(2 pi i q.v) / sqrt(m_k m_k'), into
// D[i * ld + j] (i = 3k + a, j = 3k' + b); one thread per entry, l and the images in ascending order
template <typename Ptr>
__device__ __forceinline__ void ph_build_dynmat(const double* __restrict__ P, const int64_t* __restrict__ sv_ptr,
                                                const double* __restrict__ sv, const double* __restrict__ mass,
                                                const PhCell& c, double q0, double q1, double q2, Ptr D, int ld) {
  const int dim = 3 * c.n;
  for (int t = threadIdx.x; t < dim * dim; t += kPhThreads) {
    const int i = t / dim, jj = t - i * dim;
    const int k = i / 3, a = i - 3 * k, kp = jj / 3, bb = jj - 3 * kp;
    double re = 0.0, im = 0.0;
    for (int l = 0; l < c.L; ++l) {
      const int64_t p = (int64_t)k * c.N + (int64_t)l * c.n + kp;
      const int64_t m0 = sv_ptr[c.pair0 + p], m1 = sv_ptr[c.pair0 + p + 1];
      double cs = 0.0, sn = 0.0;
      for (int64_t m = m0; m < m1; ++m) {
        const double* v = sv + 3 * m;
        double s, co;
        sincospi(2.0 * (q0 * v[0] + q1 * v[1] + q2 * v[2]), &s, &co);
        cs += co;
        sn += s;
      }
      const double w = ph_recip_count(m1 - m0);
      const double phi = P[(c.pair0 + p) * 9 + 3 * a + bb];
      re += phi * (cs * w);
      im += phi * (sn * w);
    }
    const double scale = rsqrt(mass[k] * mass[kp]);
    D[i * ld + jj] = make_double2(re * scale, im * scale);
  }
}

__global__ void __launch_bounds__(kPhThreads) phonon_dynmat_kernel(
    const double* __restrict__ fc, const int32_t* __restrict__ atom_ptr, const int32_t* __restrict__ reps,
    const int64_t* __restrict__ pair_ptr, const int64_t* __restrict__ sv_ptr, const double* __restrict__ sv,
    const double* __restrict__ mass, const double* __restrict__ q, const int32_t* __restrict__ q_ptr, int64_t B,
    int ld, double2* __restrict__ dmat) {
  const int64_t iq = blockIdx.x;
  const int64_t b = ph_owner(q_ptr, B, iq);
  const PhCell c = ph_cell(atom_ptr, reps, pair_ptr, b);
  double2* D = dmat + iq * ld * ld;
  ph_build_dynmat(fc, sv_ptr, sv, mass + atom_ptr[b], c, q[3 * iq], q[3 * iq + 1], q[3 * iq + 2], D, ld);
  const int dim = 3 * c.n;
  for (int t = threadIdx.x; t < ld * ld; t += kPhThreads)
    if (t / ld >= dim || t % ld >= dim) D[t] = make_double2(0.0, 0.0);
}

// ------------------------------------------------------------------------------------------------------------------
// eigenvalues: cyclic complex Jacobi
// ------------------------------------------------------------------------------------------------------------------

struct PhRot {
  int p, q;          // p < q; p < 0: no rotation this round (the dummy index of an odd dimension)
  double c, s;       // the real rotation after the phase
  double er, ei;     // e^{i phi}, phi = arg A_pq
  double dp, dq;     // the new diagonal entries
};

// partner of slot k in round r of the circle method over M (even) players: player 0 stays, the others rotate
__device__ __forceinline__ int ph_player(int r, int slot, int M) {
  return slot == 0 ? 0 : (slot - 1 + r) % (M - 1) + 1;
}

__global__ void __launch_bounds__(kPhThreads) phonon_freq_kernel(
    const double* __restrict__ fc, const int32_t* __restrict__ atom_ptr, const int32_t* __restrict__ reps,
    const int64_t* __restrict__ pair_ptr, const int64_t* __restrict__ sv_ptr, const double* __restrict__ sv,
    const double* __restrict__ mass, const int32_t* __restrict__ status, const double* __restrict__ q,
    const int32_t* __restrict__ q_ptr, const int64_t* __restrict__ f_ptr, int64_t B, double thz,
    double* __restrict__ eig, double* __restrict__ freq, int32_t* __restrict__ sweeps,
    int32_t* __restrict__ q_status) {
  extern __shared__ double2 A[];  // dim x dim, row-major
  __shared__ double sh[kPhWarps];
  __shared__ PhRot rot[kPhMaxDim / 2];
  __shared__ double lam[kPhMaxDim];
  const int64_t iq = blockIdx.x;
  const int tid = threadIdx.x;
  const int64_t b = ph_owner(q_ptr, B, iq);
  const PhCell c = ph_cell(atom_ptr, reps, pair_ptr, b);
  const int dim = 3 * c.n;
  const int64_t o = f_ptr[b] + (iq - q_ptr[b]) * dim;

  auto fail = [&](int n_sweeps) {
    for (int i = tid; i < dim; i += kPhThreads) eig[o + i] = NAN, freq[o + i] = NAN;
    if (tid == 0) sweeps[iq] = n_sweeps, q_status[iq] = 1;
  };
  if (status[b] != 0) {  // a failed structure: NaN, without building anything
    fail(0);
    return;
  }

  ph_build_dynmat(fc, sv_ptr, sv, mass + atom_ptr[b], c, q[3 * iq], q[3 * iq + 1], q[3 * iq + 2], A, dim);
  __syncthreads();
  // Hermitian part (D + D^H) / 2, each pair of entries by one thread
  for (int t = tid; t < dim * dim; t += kPhThreads) {
    const int i = t / dim, j = t - i * dim;
    if (i < j) {
      const double2 x = A[i * dim + j], y = A[j * dim + i];
      const double re = 0.5 * (x.x + y.x), im = 0.5 * (x.y - y.y);
      A[i * dim + j] = make_double2(re, im);
      A[j * dim + i] = make_double2(re, -im);
    } else if (i == j) {
      A[t].y = 0.0;
    }
  }
  __syncthreads();
  double t2 = 0.0;
  for (int t = tid; t < dim * dim; t += kPhThreads) t2 += A[t].x * A[t].x + A[t].y * A[t].y;
  const double norm2 = block_sum<kPhWarps>(t2, sh);
  if (!isfinite(norm2)) {
    fail(0);
    return;
  }
  const double tol2 = kPhTol * kPhTol * norm2;
  const int M = dim + (dim & 1), half = M / 2;
  int n_sweeps = 0;
  for (;;) {
    double off = 0.0;
    for (int t = tid; t < dim * dim; t += kPhThreads)
      if (t / dim != t % dim) off += A[t].x * A[t].x + A[t].y * A[t].y;
    off = block_sum<kPhWarps>(off, sh);
    if (off <= tol2) break;
    if (n_sweeps == kPhMaxSweeps || !isfinite(off)) {
      fail(n_sweeps);
      return;
    }
    for (int r = 0; r < M - 1; ++r) {
      if (tid < half) {
        int p = ph_player(r, tid, M), qq = ph_player(r, M - 1 - tid, M);
        if (p > qq) { const int s = p; p = qq; qq = s; }
        PhRot R;
        R.p = qq < dim ? p : -1, R.q = qq;
        R.c = 1.0, R.s = 0.0, R.er = 1.0, R.ei = 0.0;
        if (R.p >= 0) {
          const double2 apq = A[p * dim + qq];
          const double app = A[p * dim + p].x, aqq = A[qq * dim + qq].x;
          const double g = hypot(apq.x, apq.y);
          R.dp = app, R.dq = aqq;
          if (g > 0.0) {
            R.er = apq.x / g, R.ei = apq.y / g;
            // Golub & Van Loan's symmetric Schur 2x2 on [app g; g aqq]
            const double tau = (aqq - app) / (2.0 * g);
            const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + hypot(1.0, tau));
            R.c = 1.0 / sqrt(1.0 + t * t);
            R.s = t * R.c;
            R.dp = app - t * g, R.dq = aqq + t * g;
          }
        }
        rot[tid] = R;
      }
      __syncthreads();
      // rows: A <- G^H A, G = diag(1, e^{-i phi}) [c s; -s c] on (p, q)
      for (int t = tid; t < half * dim; t += kPhThreads) {
        const int k = t / dim, col = t - k * dim;
        const PhRot R = rot[k];
        if (R.p < 0) continue;
        const double2 x = A[R.p * dim + col], y = A[R.q * dim + col];
        const double2 ey = make_double2(R.er * y.x - R.ei * y.y, R.er * y.y + R.ei * y.x);  // e^{i phi} a_qk
        A[R.p * dim + col] = make_double2(R.c * x.x - R.s * ey.x, R.c * x.y - R.s * ey.y);
        A[R.q * dim + col] = make_double2(R.s * x.x + R.c * ey.x, R.s * x.y + R.c * ey.y);
      }
      __syncthreads();
      // columns: A <- A G; the rotated pair's own 2x2 block takes its exact diagonal form
      for (int t = tid; t < half * dim; t += kPhThreads) {
        const int k = t / dim, row = t - k * dim;
        const PhRot R = rot[k];
        if (R.p < 0) continue;
        if (row == R.p || row == R.q) {
          const bool isp = row == R.p;
          A[row * dim + R.p] = make_double2(isp ? R.dp : 0.0, 0.0);
          A[row * dim + R.q] = make_double2(isp ? 0.0 : R.dq, 0.0);
          continue;
        }
        const double2 x = A[row * dim + R.p], y = A[row * dim + R.q];
        const double2 ey = make_double2(R.er * y.x + R.ei * y.y, R.er * y.y - R.ei * y.x);  // e^{-i phi} a_kq
        A[row * dim + R.p] = make_double2(R.c * x.x - R.s * ey.x, R.c * x.y - R.s * ey.y);
        A[row * dim + R.q] = make_double2(R.s * x.x + R.c * ey.x, R.s * x.y + R.c * ey.y);
      }
      __syncthreads();
    }
    ++n_sweeps;
  }
  for (int i = tid; i < dim; i += kPhThreads) lam[i] = A[i * dim + i].x;
  __syncthreads();
  // ascending by rank, ties by index
  for (int i = tid; i < dim; i += kPhThreads) {
    const double x = lam[i];
    int rank = 0;
    for (int j = 0; j < dim; ++j) rank += (lam[j] < x) || (lam[j] == x && j < i);
    eig[o + rank] = x;
    freq[o + rank] = copysign(sqrt(fabs(x)), x) * thz;
  }
  if (tid == 0) sweeps[iq] = n_sweeps, q_status[iq] = 0;
}

// ------------------------------------------------------------------------------------------------------------------
// thermal properties
// ------------------------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kPhThreads) phonon_thermal_kernel(
    const double* __restrict__ freq, const int64_t* __restrict__ f_ptr, const int32_t* __restrict__ q_ptr,
    const int32_t* __restrict__ status, const double* __restrict__ temps, int64_t T, double kB, double h_thz,
    double cutoff, double* __restrict__ out, int32_t* __restrict__ n_imag, double* __restrict__ fmin) {
  __shared__ double sh[kPhWarps];
  const int64_t b = blockIdx.x, it = blockIdx.y;
  const int tid = threadIdx.x;
  double* o = out + (b * T + it) * 4;
  if (status[b] != 0) {
    if (tid < 4) o[tid] = NAN;
    if (it == 0 && tid == 0) n_imag[b] = -1, fmin[b] = NAN;
    return;
  }
  const double* f = freq + f_ptr[b];
  const int64_t cnt = f_ptr[b + 1] - f_ptr[b];
  const double nq = (double)(q_ptr[b + 1] - q_ptr[b]);
  const double kT = kB * temps[it];
  double sF = 0.0, sS = 0.0, sC = 0.0, sE = 0.0;
  for (int64_t i = tid; i < cnt; i += kPhThreads) {
    const double fi = f[i];
    if (fi < cutoff) continue;  // NaN stays in (and makes the sums NaN)
    const double e = h_thz * fi;
    if (kT > 0.0) {
      const double x = e / kT, em = exp(-x), lg = log1p(-em), d = expm1(-x);
      sF += 0.5 * e + kT * lg;
      sS += kB * (x / expm1(x) - lg);
      sC += kB * x * x * em / (d * d);
      sE += e * (0.5 + 1.0 / expm1(x));
    } else {
      sF += 0.5 * e;
      sE += 0.5 * e;
    }
  }
  sF = block_sum<kPhWarps>(sF, sh);
  sS = block_sum<kPhWarps>(sS, sh);
  sC = block_sum<kPhWarps>(sC, sh);
  sE = block_sum<kPhWarps>(sE, sh);
  if (tid == 0) o[0] = sF / nq, o[1] = sS / nq, o[2] = sC / nq, o[3] = sE / nq;
  if (it != 0) return;
  double ni = 0.0, nn = 0.0, lo = -INFINITY;
  for (int64_t i = tid; i < cnt; i += kPhThreads) {
    const double fi = f[i];
    ni += fi < -cutoff;
    nn += isnan(fi);
    lo = fmax(lo, -fi);
  }
  ni = block_sum<kPhWarps>(ni, sh);
  nn = block_sum<kPhWarps>(nn, sh);
  lo = block_max<kPhWarps>(lo, sh);
  if (tid == 0) n_imag[b] = (int32_t)ni, fmin[b] = nn > 0.0 ? NAN : -lo;
}

}  // namespace m3g

using namespace m3g;

extern "C" {

int m3g_phonon_force_constants(const float* forces, const int64_t* row_ptr, const int32_t* atom_ptr,
                               const int32_t* reps, const int64_t* pair_ptr, int64_t B, int max_atoms, double h,
                               int symmetrize, double* fc, int32_t* status, double* residual, void* stream) {
  if (B == 0) return M3G_OK;
  M3G_REQUIRE(forces && row_ptr && atom_ptr && reps && pair_ptr && fc && status && residual,
              "m3g_phonon_force_constants: null pointer");
  M3G_REQUIRE(max_atoms >= 1 && max_atoms <= kPhMaxAtoms,
              "m3g_phonon_force_constants: %d atoms per unit cell, expected 1 .. %d", max_atoms, kPhMaxAtoms);
  M3G_REQUIRE(h > 0.0 && isfinite(h), "m3g_phonon_force_constants: displacement %g", h);
  M3G_REQUIRE(symmetrize >= 0, "m3g_phonon_force_constants: symmetrize=%d", symmetrize);
  M3G_REQUIRE(B <= 0x7fffffff, "m3g_phonon_force_constants: B=%lld too large", (long long)B);
  phonon_fc_kernel<<<(unsigned)B, kPhThreads, 0, as_stream(stream)>>>(forces, row_ptr, atom_ptr, reps, pair_ptr, h,
                                                                        symmetrize, fc, status, residual);
  M3G_LAUNCH_CHECK("m3g_phonon_force_constants");
  return M3G_OK;
}

int m3g_phonon_dynmat(const double* fc, const int32_t* atom_ptr, const int32_t* reps, const int64_t* pair_ptr,
                      const int64_t* sv_ptr, const double* sv, const double* mass, const double* q,
                      const int32_t* q_ptr, int64_t B, int64_t Q, int max_atoms, int ld, double* dmat, void* stream) {
  if (Q == 0) return M3G_OK;
  M3G_REQUIRE(fc && atom_ptr && reps && pair_ptr && sv_ptr && sv && mass && q && q_ptr && dmat,
              "m3g_phonon_dynmat: null pointer");
  M3G_REQUIRE(max_atoms >= 1 && max_atoms <= kPhMaxAtoms,
              "m3g_phonon_dynmat: %d atoms per unit cell, expected 1 .. %d", max_atoms, kPhMaxAtoms);
  M3G_REQUIRE(ld >= 3 * max_atoms, "m3g_phonon_dynmat: ld=%d < 3 x %d", ld, max_atoms);
  M3G_REQUIRE(B >= 1 && Q <= 0x7fffffff, "m3g_phonon_dynmat: B=%lld Q=%lld", (long long)B, (long long)Q);
  phonon_dynmat_kernel<<<(unsigned)Q, kPhThreads, 0, as_stream(stream)>>>(
      fc, atom_ptr, reps, pair_ptr, sv_ptr, sv, mass, q, q_ptr, B, ld, reinterpret_cast<double2*>(dmat));
  M3G_LAUNCH_CHECK("m3g_phonon_dynmat");
  return M3G_OK;
}

int m3g_phonon_frequencies(const double* fc, const int32_t* atom_ptr, const int32_t* reps, const int64_t* pair_ptr,
                           const int64_t* sv_ptr, const double* sv, const double* mass, const int32_t* status,
                           const double* q, const int32_t* q_ptr, const int64_t* f_ptr, int64_t B, int64_t Q,
                           int max_atoms, double thz, double* eig, double* freq, int32_t* sweeps, int32_t* q_status,
                           void* stream) {
  if (Q == 0) return M3G_OK;
  M3G_REQUIRE(fc && atom_ptr && reps && pair_ptr && sv_ptr && sv && mass && status && q && q_ptr && f_ptr && eig &&
                  freq && sweeps && q_status,
              "m3g_phonon_frequencies: null pointer");
  M3G_REQUIRE(max_atoms >= 1 && max_atoms <= kPhMaxAtoms,
              "m3g_phonon_frequencies: %d atoms per unit cell, expected 1 .. %d", max_atoms, kPhMaxAtoms);
  M3G_REQUIRE(B >= 1 && Q <= 0x7fffffff, "m3g_phonon_frequencies: B=%lld Q=%lld", (long long)B, (long long)Q);
  const size_t smem = sizeof(double2) * 9 * (size_t)max_atoms * max_atoms;
  if (smem > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(phonon_freq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)smem);
    M3G_REQUIRE(err == cudaSuccess, "m3g_phonon_frequencies: %zu B of shared memory: %s", smem,
                cudaGetErrorString(err));
  }
  phonon_freq_kernel<<<(unsigned)Q, kPhThreads, smem, as_stream(stream)>>>(
      fc, atom_ptr, reps, pair_ptr, sv_ptr, sv, mass, status, q, q_ptr, f_ptr, B, thz, eig, freq, sweeps, q_status);
  M3G_LAUNCH_CHECK("m3g_phonon_frequencies");
  return M3G_OK;
}

int m3g_phonon_thermal(const double* freq, const int64_t* f_ptr, const int32_t* q_ptr, const int32_t* status,
                       int64_t B, const double* temps, int64_t T, double kB, double h_thz, double cutoff, double* out,
                       int32_t* n_imag, double* fmin, void* stream) {
  if (B == 0 || T == 0) return M3G_OK;
  M3G_REQUIRE(freq && f_ptr && q_ptr && status && temps && out && n_imag && fmin, "m3g_phonon_thermal: null pointer");
  M3G_REQUIRE(B <= 0x7fffffff && T <= 65535, "m3g_phonon_thermal: B=%lld T=%lld", (long long)B, (long long)T);
  phonon_thermal_kernel<<<dim3((unsigned)B, (unsigned)T), kPhThreads, 0, as_stream(stream)>>>(
      freq, f_ptr, q_ptr, status, temps, T, kB, h_thz, cutoff, out, n_imag, fmin);
  M3G_LAUNCH_CHECK("m3g_phonon_thermal");
  return M3G_OK;
}

}  // extern "C"
