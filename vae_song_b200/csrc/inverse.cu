// inverse.cu -- left inverse of the Brenier map x = T(z) = grad(psi + kappa|z|^2) by batched Newton steps (d <= 4).
//
// z* = T^{-1}(x) is the unique minimiser of  f(z) = Phi(z) - <x, z>,  Phi = psi + kappa|z|^2, which is convex (2 kappa-
// strongly convex for kappa > 0).  Its gradient is r(z) = xhat(z) - x and, with the LeakyReLU masks fixed, its Hessian is the
// Brenier map's exact Jacobian J = A0^T diag(2 s0^2 gx1) A0 + 2 kappa I (symmetric, >= 2 kappa I).  b200vae_icnn_decode_jac
// returns both from one fused forward, so one ROUND of the solver is one decode_jac call at every row's trial point followed
// by one launch of the step kernel below.  One thread per row, fp64 inside; the per-row state persists in a caller-owned
// buffer between rounds; rows never interact except through the integer count of unfinished rows.
//
// Per row:
//   direction   p = -J^{-1} r by Cholesky at the accepted z (a pivot <= kPivotRel * max diag: SINGULAR -- only possible at
//               kappa = 0 with A0 rank-deficient on the active units).
//   line search on xhat only.  psi is NOT used: it reaches 1e10 at the toy scale, and fp32 rounding of psi then swamps an
//               Armijo decrease test near convergence.  Along the line phi'(t) = r(z + t p)^T p is non-decreasing (the
//               gradient is monotone) and phi'(0) = -r^T J^{-1} r < 0.  t = 1 is tried first and accepted when ||r|| <= tol
//               or phi'(1) <= 0 (then f decreased: f(t) - f(0) = int phi' <= t phi'(t)).  Otherwise [lo, hi] is bisected
//               on the sign of phi'; a t with phi'(t) <= 0 is accepted once phi'(t) >= -kEta |phi'(0)|.  The residual
//               and Jacobian of the evaluation at the accepted t are kept, so the next direction costs no round.
//   kinks       after kMaxHalvings halvings the line minimum lies within 2^-12 of a jump of phi' (a LeakyReLU kink of h1 /
//               h2: the gradient is discontinuous there).  Accepting lo, as a smooth line search would, leaves z just
//               before the kink, and the next direction -- from the same piece's Jacobian -- runs into the same kink at
//               once (measured on the fp64 oracle: rows that converge otherwise stall, at 20 wasted rounds a kink).  The
//               solver therefore CROSSES: the next trial point is z + hi p, just past the kink, and it becomes z once the
//               next round has evaluated it (unconditionally: f may rise there, by at most (hi - lo) phi'(hi)).  z
//               only ever moves to an evaluated point, so ||r|| -- and the error bound -- always belong to the z that
//               is returned, also when the caller stops in between.
//   statuses    CONVERGED ||r|| <= tol;  STALLED the bracket collapsed again with lo = 0 right after a crossing (both
//               one-sided Newton directions point across the kink: x lies in a jump of the gradient, or at a kink where
//               the minimum runs along the kink surface), or the next trial point rounds to z in fp32;  MAXITER the
//               caller's last round ended with the row unfinished;  SINGULAR;  NONFINITE
//               x or z0 not finite, or xhat not finite at an accepted z (a non-finite xhat at a trial point only halves t).
//               A finished row keeps its z; its trial point stays equal to z.
//   error bound ||z - z*|| <= ||r(z)|| / (2 kappa) at the accepted z (+inf at kappa = 0): f is 2 kappa-strongly convex and
//               xhat(z) is a subgradient of Phi at z, also on a kink.
//   tolerance   tol = tol_rel ||x|| + tol_abs, fixed at init.
//
// Trial points are the fp32 points fp32(z + t p) the decode sees; an accepted z is that same point, so z stays
// fp32-representable.  This file is compiled with -fmad=false (Makefile) and its fp64 operations run in the order of the
// fp64 oracle oracle/inverse_oracle.py, which therefore takes the same decisions bit for bit.
//
// State (b200vae_brenier_inverse_state_bytes): a 256-byte header -- int32 active[2], the count of unfinished rows after a
// round goes to active[round & 1], and the step kernel zeroes the other slot for the next round -- followed by kInvFields
// fp64 arrays of B values (structure of arrays: field f of row b at rows[f * B + b]).
#include <math_constants.h>

#include "icnn.cuh"

namespace b200vae {

constexpr int kInvMaxD = 4;
constexpr int kMaxHalvings = 12;
constexpr double kEta = 0.5;
constexpr double kPivotRel = 1e-12;
constexpr size_t kInvHeaderBytes = 256;
// field offsets of the per-row state (fp64); oracle/inverse_oracle.py mirrors them
enum : int {
  F_Z = 0,        // accepted z [4]
  F_P = 4,        // Newton direction [4]
  F_T = 8,        // trial step; 0 = the trial point is z itself (first round only)
  F_LO = 9, F_HI = 10, F_PHI0 = 11, F_TOL = 12,
  F_RNORM = 13,   // ||r|| at the accepted z
  F_STATUS = 14, F_NSTEP = 15, F_NHALF = 16,
  F_CROSSED = 17, // 2: the trial point z + hi p crosses a kink; 1: z was reached by a crossing and no line search has
                  // succeeded since; 0 otherwise
  kInvFields = 18
};

size_t inverse_state_bytes(int B) { return kInvHeaderBytes + (size_t)kInvFields * B * sizeof(double); }

namespace {

__device__ __forceinline__ double dadd_mul(double z, double t, double p) { return __dadd_rn(z, __dmul_rn(t, p)); }

template <int D>
struct Row {
  double z[D], p[D];
  double t, lo, hi, phi0, tol, rnorm, status, nstep, nhalf, crossed;
};

// Cholesky solve of J p = -r; false when a pivot is <= kPivotRel * max diag or not finite
template <int D>
__device__ bool newton_dir(const double (&J)[D][D], const double (&r)[D], double (&p)[D]) {
  double L[D][D], dmax = 0.0;
#pragma unroll
  for (int i = 0; i < D; ++i) dmax = fmax(dmax, J[i][i]);
#pragma unroll
  for (int j = 0; j < D; ++j) {
    double s = J[j][j];
#pragma unroll
    for (int k = 0; k < j; ++k) s -= L[j][k] * L[j][k];
    if (!(s > kPivotRel * dmax)) return false;
    L[j][j] = sqrt(s);
#pragma unroll
    for (int i = j + 1; i < D; ++i) {
      double u = J[i][j];
#pragma unroll
      for (int k = 0; k < j; ++k) u -= L[i][k] * L[j][k];
      L[i][j] = u / L[j][j];
    }
  }
  double y[D];
#pragma unroll
  for (int i = 0; i < D; ++i) {
    double u = -r[i];
#pragma unroll
    for (int k = 0; k < i; ++k) u -= L[i][k] * y[k];
    y[i] = u / L[i][i];
  }
#pragma unroll
  for (int i = D - 1; i >= 0; --i) {
    double u = y[i];
#pragma unroll
    for (int k = i + 1; k < D; ++k) u -= L[k][i] * p[k];
    p[i] = u / L[i][i];
  }
  return true;
}

template <int D>
__device__ double norm_of(const double (&v)[D]) {
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < D; ++i) s += v[i] * v[i];
  return sqrt(s);
}

// move to the evaluated point z + t p (t = 0: z itself) and take the Newton direction from its residual and Jacobian
template <int D>
__device__ void accept(Row<D>& s, double t, const double (&r)[D], const double (&J)[D][D]) {
  if (t != 0.0) {
#pragma unroll
    for (int i = 0; i < D; ++i) s.z[i] = (double)(float)dadd_mul(s.z[i], t, s.p[i]);
    s.nstep += 1.0;
    s.crossed = 0.0;
  }
  s.rnorm = norm_of(r);
  if (!(s.rnorm <= s.tol)) {
    bool fin = isfinite(s.rnorm);
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
      for (int k = 0; k < D; ++k) fin = fin && isfinite(J[i][k]);
    if (!fin) { s.status = B200VAE_INV_NONFINITE; return; }
  } else {
    s.status = B200VAE_INV_CONVERGED;
    return;
  }
  if (!newton_dir(J, r, s.p)) { s.status = B200VAE_INV_SINGULAR; return; }
  double phi0 = 0.0;
#pragma unroll
  for (int i = 0; i < D; ++i) phi0 += r[i] * s.p[i];
  s.phi0 = phi0;
  s.t = 1.0; s.lo = 0.0; s.hi = 1.0; s.nhalf = 0.0;
}

}  // namespace

template <int D>
__global__ void __launch_bounds__(128) inverse_init_kernel(const float* __restrict__ x, const float* __restrict__ z0, int B,
                                                           float tol_rel, float tol_abs, double* __restrict__ rows,
                                                           int* __restrict__ active, float* __restrict__ ztrial,
                                                           float* __restrict__ zout, int* __restrict__ status,
                                                           float* __restrict__ err) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) { active[0] = 0; active[1] = 0; }
  if (b >= B) return;
  auto at = [&](int f) -> double& { return rows[(size_t)f * B + b]; };
  double xn = 0.0;
  bool fin = true;
  float zi[D];
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const double xi = x[(size_t)b * D + i];
    xn += xi * xi;
    zi[i] = z0 ? z0[(size_t)b * D + i] : 0.f;
    fin = fin && isfinite(xi) && isfinite(zi[i]);
  }
  const int st = fin ? B200VAE_INV_ACTIVE : B200VAE_INV_NONFINITE;
#pragma unroll
  for (int i = 0; i < kInvMaxD; ++i) {
    at(F_Z + i) = i < D ? (double)zi[i] : 0.0;
    at(F_P + i) = 0.0;
  }
  at(F_T) = 0.0; at(F_LO) = 0.0; at(F_HI) = 1.0; at(F_PHI0) = 0.0;
  at(F_TOL) = (double)tol_rel * sqrt(xn) + (double)tol_abs;
  at(F_RNORM) = CUDART_INF;
  at(F_STATUS) = st; at(F_NSTEP) = 0.0; at(F_NHALF) = 0.0; at(F_CROSSED) = 0.0;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    ztrial[(size_t)b * D + i] = fin ? zi[i] : 0.f;      // the decode never sees a non-finite input
    zout[(size_t)b * D + i] = zi[i];
  }
  status[b] = st;
  err[b] = CUDART_INF_F;
}

template <int D>
__global__ void __launch_bounds__(128, 1) newton_step_kernel(const float* __restrict__ x, const float* __restrict__ xhat,
                                                          const float* __restrict__ jac, int B, float kappa, int slot,
                                                          int final_round, double* __restrict__ rows, int* __restrict__ active,
                                                          float* __restrict__ ztrial, float* __restrict__ zout,
                                                          int* __restrict__ status, float* __restrict__ err) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) active[slot ^ 1] = 0;                     // the next round's slot; nobody adds to it during this round
  bool live = false;
  if (b < B) {
    auto at = [&](int f) -> double& { return rows[(size_t)f * B + b]; };
    Row<D> s;
#pragma unroll
    for (int i = 0; i < D; ++i) { s.z[i] = at(F_Z + i); s.p[i] = at(F_P + i); }
    s.t = at(F_T); s.lo = at(F_LO); s.hi = at(F_HI); s.phi0 = at(F_PHI0); s.tol = at(F_TOL); s.rnorm = at(F_RNORM);
    s.status = at(F_STATUS); s.nstep = at(F_NSTEP); s.nhalf = at(F_NHALF); s.crossed = at(F_CROSSED);
    if (s.status == B200VAE_INV_ACTIVE) {
      double r[D], J[D][D];
#pragma unroll
      for (int i = 0; i < D; ++i) {
        r[i] = (double)xhat[(size_t)b * D + i] - (double)x[(size_t)b * D + i];
#pragma unroll
        for (int k = 0; k < D; ++k) J[i][k] = jac[((size_t)b * D + i) * D + k];
      }
      bool fin = true;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        fin = fin && isfinite(r[i]);
#pragma unroll
        for (int k = 0; k < D; ++k) fin = fin && isfinite(J[i][k]);
      }
      if (s.t == 0.0) {
        accept(s, 0.0, r, J);                            // first round: the evaluation at z itself
      } else if (s.crossed == 2.0) {                     // the evaluation at a kink crossing z + hi p: it becomes z
        if (fin) {
          accept(s, s.t, r, J);
          s.crossed = 1.0;
        } else {
          s.status = B200VAE_INV_STALLED;               // keep the last evaluated z and its bound
        }
      } else {
        bool bisect = true;
        if (!fin) {
          s.hi = s.t;
        } else {
          double ph = 0.0;
#pragma unroll
          for (int i = 0; i < D; ++i) ph += r[i] * s.p[i];
          if (norm_of(r) <= s.tol || (ph <= 0.0 && (s.t == 1.0 || ph >= -kEta * fabs(s.phi0)))) {
            accept(s, s.t, r, J);
            bisect = false;
          } else if (ph <= 0.0) {
            s.lo = s.t;
          } else {
            s.hi = s.t;
          }
        }
        if (bisect) {
          s.nhalf += 1.0;
          if (s.nhalf <= kMaxHalvings) {
            s.t = 0.5 * (s.lo + s.hi);
          } else if (s.lo == 0.0 && s.crossed == 1.0) {
            s.status = B200VAE_INV_STALLED;
          } else {                                       // cross the kink: the next trial point is z + hi p
            s.t = s.hi;
            s.crossed = 2.0;
          }
        }
      }
      // the next trial point; a step that no longer moves z in fp32 cannot make progress
      float zt[D];
      bool moved = false;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        zt[i] = (float)dadd_mul(s.z[i], s.t, s.p[i]);
        moved = moved || zt[i] != (float)s.z[i];
      }
      if (s.status == B200VAE_INV_ACTIVE && !moved) s.status = B200VAE_INV_STALLED;
      if (s.status == B200VAE_INV_ACTIVE && final_round) s.status = B200VAE_INV_MAXITER;
      const bool act = s.status == B200VAE_INV_ACTIVE;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        ztrial[(size_t)b * D + i] = act ? zt[i] : (float)s.z[i];
        zout[(size_t)b * D + i] = (float)s.z[i];
        at(F_Z + i) = s.z[i];
        at(F_P + i) = s.p[i];
      }
      at(F_T) = s.t; at(F_LO) = s.lo; at(F_HI) = s.hi; at(F_PHI0) = s.phi0; at(F_RNORM) = s.rnorm;
      at(F_STATUS) = s.status; at(F_NSTEP) = s.nstep; at(F_NHALF) = s.nhalf; at(F_CROSSED) = s.crossed;
      status[b] = (int)s.status;
      err[b] = kappa > 0.f ? (float)(s.rnorm / (2.0 * (double)kappa)) : CUDART_INF_F;
      live = act;
    }
  }
  const unsigned m = __ballot_sync(0xffffffffu, live);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(active + slot, __popc(m));
}

int brenier_inverse_init(const float* x, const float* z0, int B, int d, float tol_rel, float tol_abs, void* state,
                         float* ztrial, float* z, int* status, float* err, cudaStream_t st) {
  int* active = reinterpret_cast<int*>(state);
  double* rows = reinterpret_cast<double*>(reinterpret_cast<char*>(state) + kInvHeaderBytes);
  const int grid = (B + 127) / 128;
  switch (d) {
#define B200VAE_INV_CASE(D)                                                                                         \
  case D: inverse_init_kernel<D><<<grid, 128, 0, st>>>(x, z0, B, tol_rel, tol_abs, rows, active, ztrial, z, status, err); \
    break;
    B200VAE_INV_CASE(1) B200VAE_INV_CASE(2) B200VAE_INV_CASE(3) B200VAE_INV_CASE(4)
#undef B200VAE_INV_CASE
    default: return B200VAE_EUNSUP;
  }
  return check_launch();
}

int brenier_newton_step(const float* x, const float* xhat, const float* jac, int B, int d, float kappa, int round,
                        int final_round, void* state, float* ztrial, float* z, int* status, float* err, cudaStream_t st) {
  int* active = reinterpret_cast<int*>(state);
  double* rows = reinterpret_cast<double*>(reinterpret_cast<char*>(state) + kInvHeaderBytes);
  const int grid = (B + 127) / 128;
  const int slot = round & 1;
  switch (d) {
#define B200VAE_INV_CASE(D)                                                                                          \
  case D: newton_step_kernel<D><<<grid, 128, 0, st>>>(x, xhat, jac, B, kappa, slot, final_round, rows, active, ztrial, z, \
                                                      status, err);                                                   \
    break;
    B200VAE_INV_CASE(1) B200VAE_INV_CASE(2) B200VAE_INV_CASE(3) B200VAE_INV_CASE(4)
#undef B200VAE_INV_CASE
    default: return B200VAE_EUNSUP;
  }
  return check_launch();
}

}  // namespace b200vae
