// The FIRE step of one structure inside a one-CTA-per-structure kernel (relax.cu's m3g_fire_step, neb.cu's
// m3g_neb_step): checks the frame, takes the FIRE decision and updates the velocities; the caller then moves its
// positions with the returned FireMove.  Rows are visited by the fixed thread-row map (thread t owns rows t, t + 256,
// ...) and every sum ends in common.cuh's fixed block_sum / block_max tree, so the result depends only on the
// structure's own rows.
#pragma once
#include "common.cuh"

namespace m3g {

constexpr int kFireThreads = 256;
constexpr int kFireWarps = kFireThreads / 32;

enum FireStatus { kFireRunning = 0, kFireConverged = 1, kFireNotConverged = 2, kFireFailed = 3 };

struct FireParams {
  double dt_max, max_move, f_inc, f_dec, a_start, f_a, fmax_target;
  int n_min, max_steps;
};

// per-structure FIRE state, indexed by the structure
struct FireState {
  double *dt, *a, *fmax;
  int32_t *n_pos, *n_steps, *status;
};

// the position step of a row component from its new velocity w: dt w, scaled down to max_move over the structure
struct FireMove {
  double dt, scale;
  bool clip;
  __device__ __forceinline__ double operator()(double w) const {
    const double d = dt * w;
    return clip ? d * scale : d;
  }
};

// gen(r, g) writes the generalised force of row r to g[3]; vel(r) points to row r's velocity.  Returns false when the
// structure stops at this frame (status and fmax written, velocities untouched); otherwise the velocities are updated
// and *mv holds the position step.  Every thread of the block must call it; sh holds kFireWarps doubles.
template <class Gen, class Vel>
__device__ __forceinline__ bool fire_advance(const FireParams& q, const FireState& s, int64_t b, int rows, Gen gen,
                                             Vel vel, double* sh, FireMove* mv) {
  __shared__ double bc[4];  // broadcast: 1 - a, a |v|, max(|g|, 1e-30), dt
  __shared__ int bmode;     // 0 = stop, 1 = step with the velocity mix, 2 = step from zero velocity
  const int tid = threadIdx.x;

  // pass 1: power, |g|^2, |v|^2, max row |g|^2, finiteness
  double P = 0.0, gg = 0.0, vv = 0.0, gmax2 = 0.0;
  int bad = 0;
  for (int r = tid; r < rows; r += kFireThreads) {
    double g[3];
    gen(r, g);
    const double* v = vel(r);
    const double g2 = g[0] * g[0] + g[1] * g[1] + g[2] * g[2];
    P += g[0] * v[0] + g[1] * v[1] + g[2] * v[2];
    gg += g2;
    vv += v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    gmax2 = fmax(gmax2, g2);
    bad |= !(isfinite(g[0]) && isfinite(g[1]) && isfinite(g[2]));
  }
  bad = __syncthreads_or(bad);
  P = block_sum<kFireWarps>(P, sh);
  gg = block_sum<kFireWarps>(gg, sh);
  vv = block_sum<kFireWarps>(vv, sh);
  gmax2 = block_max<kFireWarps>(gmax2, sh);

  if (tid == 0) {
    const double fm = sqrt(gmax2);
    s.fmax[b] = bad ? (double)INFINITY : fm;
    int mode = 0;
    if (bad) {
      s.status[b] = kFireFailed;
    } else if (fm < q.fmax_target) {
      s.status[b] = kFireConverged;
    } else if (s.n_steps[b] >= q.max_steps) {
      s.status[b] = kFireNotConverged;
    } else {
      double a = s.a[b], dt = s.dt[b];
      int n_pos = s.n_pos[b];
      if (P > 0.0) {
        mode = 1;
        bc[0] = 1.0 - a;
        bc[1] = a * sqrt(vv);
        bc[2] = fmax(sqrt(gg), 1e-30);
        if (n_pos > q.n_min) {
          dt = fmin(dt * q.f_inc, q.dt_max);
          a *= q.f_a;
        }
        n_pos += 1;
      } else {
        mode = 2;
        a = q.a_start;
        dt *= q.f_dec;
        n_pos = 0;
      }
      s.a[b] = a;
      s.dt[b] = dt;
      s.n_pos[b] = n_pos;
      s.n_steps[b] += 1;
      bc[3] = dt;
    }
    bmode = mode;
  }
  __syncthreads();
  const int mode = bmode;
  if (mode == 0) return false;
  const double dt = bc[3];

  // pass 2: v <- (1 - a) v + a |v| g / |g|  (or 0), v <- v + dt g; |dr|^2 with dr = dt v
  double dr2 = 0.0;
  for (int r = tid; r < rows; r += kFireThreads) {
    double g[3];
    gen(r, g);
    double* v = vel(r);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      double w = mode == 1 ? bc[0] * v[c] + bc[1] * g[c] / bc[2] : 0.0;
      w = w + dt * g[c];
      v[c] = w;
      const double d = dt * w;
      dr2 += d * d;
    }
  }
  const double norm = sqrt(block_sum<kFireWarps>(dr2, sh));
  mv->dt = dt;
  mv->clip = norm > q.max_move;
  mv->scale = mv->clip ? q.max_move / norm : 1.0;
  return true;
}

}  // namespace m3g
