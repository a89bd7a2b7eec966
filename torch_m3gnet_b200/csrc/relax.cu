// Batched FIRE relaxation step (extension, no reference counterpart): calculator.py::Fire.step / Fire.run applied to
// every structure of a ragged batch at once, with per-structure FIRE state, on ASE UnitCellFilter coordinates when the
// cell relaxes.  One CTA per structure: its rows (N_b atoms, then 3 cell rows) are visited by a fixed thread-row map
// (thread t owns rows t, t + 256, ... counted from the structure's first row) and every sum ends in the same fixed tree
// (xor butterfly in each warp, then the 8 warp results in warp order).  The result therefore depends only on the
// structure's own rows, never on its offset in the batch or its neighbours, and there are no atomics.
#include "fire.cuh"

namespace m3g {

struct FireArgs {
  const float *forces, *sigma, *energy;
  const int32_t* atom_ptr;
  double dt_max, max_move, f_inc, f_dec, a_start, f_a, fmax_target, pressure;
  int n_min, max_steps;
  const double* cell_factor;
  double *x, *xc, *v, *vc, *dt, *a;
  int32_t *n_pos, *n_steps, *status;
  const double* L0;
  double *lattice, *pos, *fmax, *e_frame, *sigma_frame;
};

// inverse of a row-major 3x3 matrix (adjugate / determinant)
__device__ void inverse3(const double* m, double* inv) {
  const double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
  const double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
  inv[0] = c00 / det;
  inv[1] = (m[2] * m[7] - m[1] * m[8]) / det;
  inv[2] = (m[1] * m[5] - m[2] * m[4]) / det;
  inv[3] = c01 / det;
  inv[4] = (m[0] * m[8] - m[2] * m[6]) / det;
  inv[5] = (m[2] * m[3] - m[0] * m[5]) / det;
  inv[6] = c02 / det;
  inv[7] = (m[1] * m[6] - m[0] * m[7]) / det;
  inv[8] = (m[0] * m[4] - m[1] * m[3]) / det;
}

__device__ __forceinline__ double det3(const double* m) {
  return m[0] * (m[4] * m[8] - m[5] * m[7]) + m[1] * (m[5] * m[6] - m[3] * m[8]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
}

__global__ void __launch_bounds__(kFireThreads) fire_step_kernel(FireArgs p) {
  const int64_t b = blockIdx.x;
  if (p.status[b] != kFireRunning) return;  // finished structures stay bit-untouched
  __shared__ double sh[kFireWarps];
  __shared__ double D[9];      // deformation gradient D = solve(L0, L)^T, row-major
  __shared__ double Dn[9];     // D of the updated cell rows, xc / cell_factor
  __shared__ double cellf[9];  // generalised forces of the 3 cell rows
  const int64_t r0 = p.atom_ptr[b];
  const int n = p.atom_ptr[b + 1] - p.atom_ptr[b];
  const bool cell = p.sigma != nullptr;
  const int tid = threadIdx.x;

  if (cell && tid == 0) {
    double L0[9], L[9], inv0[9], Dinv[9], vir[9];
    for (int k = 0; k < 9; ++k) {
      L0[k] = p.L0[b * 9 + k];
      L[k] = p.lattice[b * 9 + k];
    }
    inverse3(L0, inv0);
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c)  // (L0^-1 L)[r][c] is D[c][r]
        D[c * 3 + r] = inv0[r * 3 + 0] * L[0 * 3 + c] + inv0[r * 3 + 1] * L[1 * 3 + c] + inv0[r * 3 + 2] * L[2 * 3 + c];
    const double vol = fabs(det3(L));
    for (int k = 0; k < 9; ++k) {
      const double s = (double)p.sigma[b * 9 + k];
      p.sigma_frame[b * 9 + k] = s;
      vir[k] = -vol * (k % 4 == 0 ? s + p.pressure : s);
    }
    inverse3(D, Dinv);
    const double cf = p.cell_factor[b];
    // -V (sigma + p I) D^-T / cell_factor
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c)
        cellf[r * 3 + c] = (vir[r * 3 + 0] * Dinv[c * 3 + 0] + vir[r * 3 + 1] * Dinv[c * 3 + 1] +
                            vir[r * 3 + 2] * Dinv[c * 3 + 2]) / cf;
  }
  if (tid == 0 && p.e_frame) p.e_frame[b] = (double)p.energy[b];
  __syncthreads();

  const int rows = n + (cell ? 3 : 0);
  // generalised force of row r: F D for an atom (F itself without the cell filter), the cell force for r >= n
  auto gen = [&](int r, double* g) {
    if (r < n) {
      const float* f = p.forces + (r0 + r) * 3;
      const double f0 = f[0], f1 = f[1], f2 = f[2];
      if (cell) {
#pragma unroll
        for (int c = 0; c < 3; ++c) g[c] = f0 * D[c] + f1 * D[3 + c] + f2 * D[6 + c];
      } else {
        g[0] = f0, g[1] = f1, g[2] = f2;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) g[c] = cellf[(r - n) * 3 + c];
    }
  };
  auto vel = [&](int r) -> double* { return r < n ? p.v + (r0 + r) * 3 : p.vc + b * 9 + (r - n) * 3; };

  const FireParams q{p.dt_max, p.max_move, p.f_inc, p.f_dec, p.a_start, p.f_a, p.fmax_target, p.n_min, p.max_steps};
  const FireState s{p.dt, p.a, p.fmax, p.n_pos, p.n_steps, p.status};
  FireMove step_of;
  if (!fire_advance(q, s, b, rows, gen, vel, sh, &step_of)) return;

  // pass 3: x <- x + dr, then back to Cartesian positions and lattice
  if (!cell) {
    for (int r = tid; r < n; r += kFireThreads) {
      const double* v = p.v + (r0 + r) * 3;
      double* x = p.pos + (r0 + r) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) x[c] = x[c] + step_of(v[c]);
    }
    return;
  }
  if (tid < 3) {
    const double* v = p.vc + b * 9 + tid * 3;
    double* x = p.xc + b * 9 + tid * 3;
    const double cf = p.cell_factor[b];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      x[c] = x[c] + step_of(v[c]);
      Dn[tid * 3 + c] = x[c] / cf;
    }
  }
  __syncthreads();
  if (tid < 9) {  // L = L0 D^T
    const int r = tid / 3, c = tid % 3;
    const double* L0 = p.L0 + b * 9;
    p.lattice[b * 9 + tid] = L0[r * 3 + 0] * Dn[c * 3 + 0] + L0[r * 3 + 1] * Dn[c * 3 + 1] + L0[r * 3 + 2] * Dn[c * 3 + 2];
  }
  for (int r = tid; r < n; r += kFireThreads) {
    const double* v = p.v + (r0 + r) * 3;
    double* x = p.x + (r0 + r) * 3;
    double* q = p.pos + (r0 + r) * 3;
    double xn[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) xn[c] = x[c] + step_of(v[c]);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      x[c] = xn[c];
      q[c] = xn[0] * Dn[c * 3 + 0] + xn[1] * Dn[c * 3 + 1] + xn[2] * Dn[c * 3 + 2];
    }
  }
}

}  // namespace m3g

using namespace m3g;

extern "C" {

int m3g_fire_step(const float* forces, const float* sigma, const float* energy, const int32_t* atom_ptr, int64_t B,
                  double dt_max, double max_move, int n_min, double f_inc, double f_dec, double a_start, double f_a,
                  double fmax_target, int max_steps, double pressure, const double* cell_factor, double* x, double* xc,
                  double* v, double* vc, double* dt, double* a, int32_t* n_pos, int32_t* n_steps, int32_t* status,
                  const double* L0, double* lattice, double* pos, double* fmax, double* e_frame, double* sigma_frame,
                  void* stream) {
  if (B == 0) return M3G_OK;
  M3G_REQUIRE(forces && atom_ptr && v && dt && a && n_pos && n_steps && status && pos && fmax,
              "m3g_fire_step: null pointer");
  M3G_REQUIRE(!e_frame || energy, "m3g_fire_step: e_frame needs energy");
  M3G_REQUIRE(!sigma || (cell_factor && x && xc && vc && L0 && lattice && sigma_frame),
              "m3g_fire_step: the cell filter needs cell_factor, x, xc, vc, L0, lattice and sigma_frame");
  M3G_REQUIRE(B <= 0x7fffffff, "m3g_fire_step: B=%lld too large", (long long)B);
  FireArgs p{forces, sigma, energy, atom_ptr, dt_max, max_move, f_inc, f_dec, a_start, f_a, fmax_target, pressure,
             n_min, max_steps, cell_factor, x, xc, v, vc, dt, a, n_pos, n_steps, status, L0, lattice, pos, fmax,
             e_frame, sigma_frame};
  fire_step_kernel<<<(unsigned)B, kFireThreads, 0, as_stream(stream)>>>(p);
  M3G_LAUNCH_CHECK("m3g_fire_step");
  return M3G_OK;
}

}  // extern "C"
