// Batched Langevin molecular dynamics (extension, no reference counterpart; torch_m3gnet_b200/md.py::BatchMD): one
// BAOAB step for every running structure of a ragged batch, optionally with a stochastic cell-rescaling barostat
// (Bernetti & Bussi 2020) for constant pressure, the Maxwell-Boltzmann draw of starting velocities, and the
// counter-based Philox4x64-10 generator all of them take their noise from.
//
// One CTA per structure with relax.cu's thread-row map (thread t owns atoms t, t + 256, ... of its structure) and its
// fixed reduction tree (block_sum / block_max, common.cuh).  The noise of atom i is keyed to (i, the structure's stream
// id, the step), not to its batch row, so a structure's new state depends only on its own rows and stream id, never on
// its offset in the batch or its neighbours; no atomics, no scratch.
#include "common.cuh"

namespace m3g {

constexpr int kMdThreads = 256;
constexpr int kMdWarps = kMdThreads / 32;
constexpr double kBoltzmann = 8.617333262e-5;  // eV/K

enum MdStatus { kMdRunning = 0, kMdFailed = 1 };
enum NoiseTag : uint64_t { kTagLangevin = 0, kTagVelocities = 1, kTagBarostat = 2 };
enum Coupling { kIsotropic = 0, kPerAxis = 1 };

// Philox4x64-10 (Salmon et al., SC'11; Random123's philox4x64, numpy.random.Philox): ten rounds on the counter c, the
// key bumped by the Weyl constants before every round but the first
__device__ __forceinline__ void philox4x64_10(uint64_t c[4], uint64_t k0, uint64_t k1) {
  constexpr uint64_t M0 = 0xD2E7470EE14C6C93ull, M1 = 0xCA5A826395121157ull;
  constexpr uint64_t W0 = 0x9E3779B97F4A7C15ull, W1 = 0xBB67AE8584CAA73Bull;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {
      k0 += W0;
      k1 += W1;
    }
    const uint64_t lo0 = M0 * c[0], hi0 = __umul64hi(M0, c[0]);
    const uint64_t lo1 = M1 * c[2], hi1 = __umul64hi(M1, c[2]);
    const uint64_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0;
    c[1] = lo1;
    c[2] = n2;
    c[3] = lo0;
  }
}

// ((w >> 11) + 0.5) 2^-53: in (0, 1), never 0, exact in float64
__device__ __forceinline__ double uniform53(uint64_t w) { return ((double)(w >> 11) + 0.5) * 0x1.0p-53; }

// three standard normals from one Philox call on the counter (i, s, k, tag) under the key (seed, 0), Box-Muller:
// (x, y) = sqrt(-2 ln u0) (cos, sin)(2 pi u1), z = sqrt(-2 ln u2) cos(2 pi u3).  sincospi takes 2 u exactly, with no
// argument reduction (and no local-memory slow path)
__device__ __forceinline__ void normal3(uint64_t i, uint64_t s, uint64_t k, uint64_t tag, uint64_t seed, double xi[3]) {
  uint64_t c[4] = {i, s, k, tag};
  philox4x64_10(c, seed, 0);
  const double r0 = sqrt(-2.0 * log(uniform53(c[0]))), r2 = sqrt(-2.0 * log(uniform53(c[2])));
  double sn, cs;
  sincospi(2.0 * uniform53(c[1]), &sn, &cs);
  xi[0] = r0 * cs;
  xi[1] = r0 * sn;
  xi[2] = r2 * cospi(2.0 * uniform53(c[3]));
}

struct LangevinArgs {
  const float *forces, *energy;
  const int32_t* atom_ptr;
  int64_t B;
  double dt, max_step_move;
  uint64_t seed;
  int advance, slot;
  const double *inv_mass, *c1, *c2, *kT;
  const int64_t* sid;
  double *pos, *v;
  int32_t *step, *status;
  double *bath, *obs;
};

// the barostat's inputs (m3g_langevin_npt_step); not read by the fixed-cell instance
struct BarostatArgs {
  const float* sigma;  // (B,3,3) cell stress of frame k, eV/A^3, ASE sign
  double* lattice;     // (B,3,3) row-major, rows are lattice vectors; L_k in, L_{k+1} out
  const double *P0, *beta_T, *tau_p;
  int coupling;
  double max_step_strain;
};

// Stochastic cell rescaling on thread 0 after pass 1: V = |det L|, the pressure P_int = 2 K / (3 V) - tr(sigma) / 3 (and
// per axis P_a = 2 K_aa / V - sigma_aa), and the log-strain step of Ito Euler-Maruyama in ln V (isotropic) or in the
// log axis scales (per axis), d eps = -(beta_T dt / tau_p) (P0 - P) + sqrt(2 kT beta_T dt / (V tau_p)) xi with xi from
// counter (0, s, k, tag 2).  mu = the axis scale factors.  False (the structure fails) on a non-finite stress or volume or
// a log-scale step beyond max_step_strain.
__device__ bool barostat(const BarostatArgs& q, int64_t b, double ek, const double ka[3], double kT, double dt,
                         uint64_t s, uint64_t k, uint64_t seed, double* vol, double* pint, double pa[3],
                         double mu[3]) {
  const double* L = q.lattice + b * 9;
  const float* sg = q.sigma + b * 9;
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 9; ++i) ok &= isfinite(sg[i]);
  const double V = fabs(L[0] * (L[4] * L[8] - L[5] * L[7]) - L[1] * (L[3] * L[8] - L[5] * L[6]) +
                        L[2] * (L[3] * L[7] - L[4] * L[6]));
  const double s00 = sg[0], s11 = sg[4], s22 = sg[8];
  *vol = V;
  *pint = 2.0 * ek / (3.0 * V) - (s00 + s11 + s22) / 3.0;
  pa[0] = 2.0 * ka[0] / V - s00;
  pa[1] = 2.0 * ka[1] / V - s11;
  pa[2] = 2.0 * ka[2] / V - s22;
  double xi[3];
  normal3(0, s, k, kTagBarostat, seed, xi);
  const double P0 = q.P0[b], drift = q.beta_T[b] * dt / q.tau_p[b];
  const double diff = sqrt(2.0 * kT * q.beta_T[b] * dt / (V * q.tau_p[b]));
  double le[3];
  if (q.coupling == kIsotropic) {
    le[0] = le[1] = le[2] = (-drift * (P0 - *pint) + diff * xi[0]) / 3.0;
  } else {
#pragma unroll
    for (int a = 0; a < 3; ++a) le[a] = -drift * (P0 - pa[a]) + diff * xi[a];
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    ok &= fabs(le[a]) <= q.max_step_strain;  // false on NaN too
    mu[a] = exp(le[a]);
  }
  return ok && isfinite(V);
}

// kNpt: with the barostat (BarostatArgs); otherwise the fixed-cell step, which reads nothing of q
template <bool kNpt>
__global__ void __launch_bounds__(kMdThreads) langevin_step_kernel(LangevinArgs p, BarostatArgs q) {
  const int64_t b = blockIdx.x;
  if (p.status[b] != kMdRunning) return;  // failed structures stay frozen at the frame that failed
  __shared__ double sh[kMdWarps];
  __shared__ double vcom[3];
  __shared__ double mu[3], rmu[3];  // barostat scale factors and their inverses
  __shared__ int bgo;
  const int64_t r0 = p.atom_ptr[b];
  const int n = p.atom_ptr[b + 1] - p.atom_ptr[b];
  const int tid = threadIdx.x;
  const int k = p.step[b];
  const double h = 0.5 * p.dt;
  const bool closing = k > 0;  // frame 0 has no half kick to close

  // v_k of atom r: the closing half kick B of step k - 1 on the stored velocity
  auto v_frame = [&](int r, const float* f, double im, double* w) {
    const double* v = p.v + (r0 + r) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) w[c] = closing ? v[c] + h * ((double)f[c] * im) : v[c];
  };

  // pass 1: v_k, finiteness, max |v_k|^2, kinetic energy (and per axis with the barostat) and total mass (in units of
  // 1 / ACC_UNIT)
  double ek = 0.0, vmax2 = 0.0, mass = 0.0, ka[3] = {0.0, 0.0, 0.0};
  int bad = 0;
  for (int r = tid; r < n; r += kMdThreads) {
    const float* f = p.forces + (r0 + r) * 3;
    const double im = p.inv_mass[r0 + r];
    double w[3];
    v_frame(r, f, im, w);
    const double w2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    bad |= !(isfinite(f[0]) && isfinite(f[1]) && isfinite(f[2]) && isfinite(w2));
    ek += w2 / im;
    if constexpr (kNpt) {
#pragma unroll
      // (w / im) w, not w w / im: a shared w w product would let the compiler rebuild w2 without its fmas and move
      // E_kin off the fixed-cell step's bits
      for (int c = 0; c < 3; ++c) ka[c] += (w[c] / im) * w[c];
    }
    vmax2 = fmax(vmax2, w2);
    mass += 1.0 / im;
  }
  bad = __syncthreads_or(bad);
  ek = 0.5 * block_sum<kMdWarps>(ek, sh);
  vmax2 = block_max<kMdWarps>(vmax2, sh);
  mass = block_sum<kMdWarps>(mass, sh);
  if constexpr (kNpt) {
#pragma unroll
    for (int c = 0; c < 3; ++c) ka[c] = 0.5 * block_sum<kMdWarps>(ka[c], sh);
  }

  if (tid == 0) {
    const double e = (double)p.energy[b];
    bool fail = bad || !isfinite(e) || !(sqrt(vmax2) * p.dt <= p.max_step_move);
    double vol = 0.0, pint = 0.0, pa[3], m[3];
    if constexpr (kNpt) {
      fail |= !barostat(q, b, ek, ka, p.kT[b], p.dt, (uint64_t)p.sid[b], (uint64_t)k, p.seed, &vol, &pint, pa, m);
    }
    if (fail) {
      p.status[b] = kMdFailed;
    } else if (p.slot >= 0) {
      // obs rows: 4 columns fixed-cell; with the barostat 6 (+ V, P_int), per axis 9 (+ P_x, P_y, P_z)
      const int width = !kNpt ? 4 : q.coupling == kIsotropic ? 6 : 9;
      double* o = p.obs + ((int64_t)p.slot * p.B + b) * width;
      o[0] = e;
      o[1] = ek;
      o[2] = 2.0 * ek / ((3.0 * n - 3.0) * kBoltzmann);
      o[3] = p.bath[b];
      if constexpr (kNpt) {
        o[4] = vol;
        o[5] = pint;
        if (q.coupling != kIsotropic) {
          o[6] = pa[0];
          o[7] = pa[1];
          o[8] = pa[2];
        }
      }
    }
    if constexpr (kNpt) {
      if (!fail && p.advance) {  // L_{k+1} = L_k diag(mu)
        double* L = q.lattice + b * 9;
#pragma unroll
        for (int i = 0; i < 9; ++i) L[i] *= m[i % 3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          mu[a] = m[a];
          rmu[a] = 1.0 / m[a];
        }
      }
    }
    bgo = !fail;
  }
  __syncthreads();
  if (!bgo) return;

  if (!p.advance) {  // the final frame: v_k is the result
    for (int r = tid; r < n; r += kMdThreads) {
      double w[3];
      v_frame(r, p.forces + (r0 + r) * 3, p.inv_mass[r0 + r], w);
      double* v = p.v + (r0 + r) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c] = w[c];
    }
    return;
  }

  // pass 2: B (v_k + dt/2 F_k / m), A (x + dt/2 v), O (c1 v + c2 sqrt(kT / m) xi); kinetic energy before O and the
  // momentum after it
  const double c1 = p.c1[b], c2 = p.c2[b], kT = p.kT[b];
  const uint64_t s = (uint64_t)p.sid[b];
  double ke0 = 0.0, px = 0.0, py = 0.0, pz = 0.0;
  for (int r = tid; r < n; r += kMdThreads) {
    const float* f = p.forces + (r0 + r) * 3;
    const double im = p.inv_mass[r0 + r];
    double w[3], xi[3];
    v_frame(r, f, im, w);
    normal3((uint64_t)r, s, (uint64_t)k, kTagLangevin, p.seed, xi);
    const double sigma = sqrt(kT * im);
    double* x = p.pos + (r0 + r) * 3;
    double* v = p.v + (r0 + r) * 3;
    double u2 = 0.0, o[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const double u = w[c] + h * ((double)f[c] * im);
      u2 += u * u;
      x[c] = x[c] + h * u;
      o[c] = c1 * u + c2 * (sigma * xi[c]);
      v[c] = o[c];
    }
    ke0 += u2 / im;
    px += o[0] / im;
    py += o[1] / im;
    pz += o[2] / im;
  }
  ke0 = 0.5 * block_sum<kMdWarps>(ke0, sh);
  px = block_sum<kMdWarps>(px, sh);
  py = block_sum<kMdWarps>(py, sh);
  pz = block_sum<kMdWarps>(pz, sh);
  if (tid == 0) {
    vcom[0] = px / mass;
    vcom[1] = py / mass;
    vcom[2] = pz / mass;
  }
  __syncthreads();

  // pass 3: centre-of-mass velocity removed, A (x + dt/2 v) -> x_{k+1}; kinetic energy after the thermostat (before the
  // barostat, which then scales x_{k+1} by mu and v by 1 / mu)
  double ke1 = 0.0;
  for (int r = tid; r < n; r += kMdThreads) {
    const double im = p.inv_mass[r0 + r];
    double* x = p.pos + (r0 + r) * 3;
    double* v = p.v + (r0 + r) * 3;
    double u2 = 0.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const double u = v[c] - vcom[c];
      u2 += u * u;
      if constexpr (kNpt) {
        v[c] = u * rmu[c];
        x[c] = (x[c] + h * u) * mu[c];
      } else {
        v[c] = u;
        x[c] = x[c] + h * u;
      }
    }
    ke1 += u2 / im;
  }
  ke1 = 0.5 * block_sum<kMdWarps>(ke1, sh);
  if (tid == 0) {
    p.bath[b] += ke1 - ke0;
    p.step[b] = k + 1;
  }
}

// (min. 1 block per SM: with the thread bound alone ptxas caps this kernel at 64 registers and spills)
__global__ void __launch_bounds__(kMdThreads, 1)
    maxwell_boltzmann_kernel(const int32_t* atom_ptr, uint64_t seed, const double* inv_mass, const double* kT,
                             const int64_t* sid, double* v) {
  const int64_t b = blockIdx.x;
  __shared__ double sh[kMdWarps];
  __shared__ double vcom[3];
  const int64_t r0 = atom_ptr[b];
  const int n = atom_ptr[b + 1] - atom_ptr[b];
  const int tid = threadIdx.x;
  const double t = kT[b];
  const uint64_t s = (uint64_t)sid[b];
  double px = 0.0, py = 0.0, pz = 0.0, mass = 0.0;
  for (int r = tid; r < n; r += kMdThreads) {
    const double im = inv_mass[r0 + r];
    double xi[3];
    normal3((uint64_t)r, s, 0, kTagVelocities, seed, xi);
    const double sigma = sqrt(t * im);
    const double w0 = sigma * xi[0], w1 = sigma * xi[1], w2 = sigma * xi[2];
    double* w = v + (r0 + r) * 3;
    w[0] = w0;
    w[1] = w1;
    w[2] = w2;
    px += w0 / im;
    py += w1 / im;
    pz += w2 / im;
    mass += 1.0 / im;
  }
  px = block_sum<kMdWarps>(px, sh);
  py = block_sum<kMdWarps>(py, sh);
  pz = block_sum<kMdWarps>(pz, sh);
  mass = block_sum<kMdWarps>(mass, sh);
  if (tid == 0) {
    vcom[0] = px / mass;
    vcom[1] = py / mass;
    vcom[2] = pz / mass;
  }
  __syncthreads();
  for (int r = tid; r < n; r += kMdThreads) {
    double* w = v + (r0 + r) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) w[c] = w[c] - vcom[c];
  }
}

__global__ void philox_kernel(const uint64_t* ctr, const uint64_t* key, int64_t n, uint64_t* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t c[4] = {ctr[i * 4], ctr[i * 4 + 1], ctr[i * 4 + 2], ctr[i * 4 + 3]};
  philox4x64_10(c, key[i * 2], key[i * 2 + 1]);
#pragma unroll
  for (int q = 0; q < 4; ++q) out[i * 4 + q] = c[q];
}

}  // namespace m3g

using namespace m3g;

extern "C" {

int m3g_langevin_step(const float* forces, const float* energy, const int32_t* atom_ptr, int64_t B, double dt,
                      double max_step_move, int64_t seed, int advance, int slot, const double* inv_mass,
                      const double* c1, const double* c2, const double* kT, const int64_t* sid, double* pos, double* v,
                      int32_t* step, int32_t* status, double* bath, double* obs, void* stream) {
  if (B == 0) return M3G_OK;
  M3G_REQUIRE(forces && energy && atom_ptr && inv_mass && c1 && c2 && kT && sid && pos && v && step && status && bath,
              "m3g_langevin_step: null pointer");
  M3G_REQUIRE(slot < 0 || obs, "m3g_langevin_step: slot %d needs obs", slot);
  M3G_REQUIRE(B <= 0x7fffffff, "m3g_langevin_step: B=%lld too large", (long long)B);
  LangevinArgs p{forces, energy, atom_ptr, B, dt, max_step_move, (uint64_t)seed, advance, slot, inv_mass, c1, c2, kT,
                 sid, pos, v, step, status, bath, obs};
  langevin_step_kernel<false><<<(unsigned)B, kMdThreads, 0, as_stream(stream)>>>(p, BarostatArgs{});
  M3G_LAUNCH_CHECK("m3g_langevin_step");
  return M3G_OK;
}

int m3g_langevin_npt_step(const float* forces, const float* energy, const int32_t* atom_ptr, int64_t B, double dt,
                          double max_step_move, int64_t seed, int advance, int slot, const double* inv_mass,
                          const double* c1, const double* c2, const double* kT, const int64_t* sid, double* pos,
                          double* v, int32_t* step, int32_t* status, double* bath, double* obs, const float* sigma,
                          double* lattice, const double* P0, const double* beta_T, const double* tau_p, int coupling,
                          double max_step_strain, void* stream) {
  if (B == 0) return M3G_OK;
  M3G_REQUIRE(forces && energy && atom_ptr && inv_mass && c1 && c2 && kT && sid && pos && v && step && status && bath &&
                  sigma && lattice && P0 && beta_T && tau_p,
              "m3g_langevin_npt_step: null pointer");
  M3G_REQUIRE(slot < 0 || obs, "m3g_langevin_npt_step: slot %d needs obs", slot);
  M3G_REQUIRE(coupling == kIsotropic || coupling == kPerAxis, "m3g_langevin_npt_step: coupling %d", coupling);
  M3G_REQUIRE(B <= 0x7fffffff, "m3g_langevin_npt_step: B=%lld too large", (long long)B);
  LangevinArgs p{forces, energy, atom_ptr, B, dt, max_step_move, (uint64_t)seed, advance, slot, inv_mass, c1, c2, kT,
                 sid, pos, v, step, status, bath, obs};
  BarostatArgs q{sigma, lattice, P0, beta_T, tau_p, coupling, max_step_strain};
  langevin_step_kernel<true><<<(unsigned)B, kMdThreads, 0, as_stream(stream)>>>(p, q);
  M3G_LAUNCH_CHECK("m3g_langevin_npt_step");
  return M3G_OK;
}

int m3g_md_maxwell_boltzmann(const int32_t* atom_ptr, int64_t B, int64_t seed, const double* inv_mass,
                             const double* kT, const int64_t* sid, double* v, void* stream) {
  if (B == 0) return M3G_OK;
  M3G_REQUIRE(atom_ptr && inv_mass && kT && sid && v, "m3g_md_maxwell_boltzmann: null pointer");
  M3G_REQUIRE(B <= 0x7fffffff, "m3g_md_maxwell_boltzmann: B=%lld too large", (long long)B);
  maxwell_boltzmann_kernel<<<(unsigned)B, kMdThreads, 0, as_stream(stream)>>>(atom_ptr, (uint64_t)seed, inv_mass, kT,
                                                                             sid, v);
  M3G_LAUNCH_CHECK("m3g_md_maxwell_boltzmann");
  return M3G_OK;
}

int m3g_debug_philox4x64(const int64_t* ctr, const int64_t* key, int64_t n, int64_t* out, void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(ctr && key && out, "m3g_debug_philox4x64: null pointer");
  philox_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const uint64_t*>(ctr), reinterpret_cast<const uint64_t*>(key), n,
      reinterpret_cast<uint64_t*>(out));
  M3G_LAUNCH_CHECK("m3g_debug_philox4x64");
  return M3G_OK;
}

}  // extern "C"
