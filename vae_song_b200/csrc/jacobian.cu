// jacobian.cu -- the decoder's Jacobian from the two Brenier maps' Jacobians, and its singular values.
//
// LIDVAE.decode (model.py:818-830) is y = T2(M . T1(z)) with T_i = grad(psi_i + kappa|.|^2) and M = eye(Dx, D) (or the
// user's B buffer), so J = J2(x) . M . J1(z).  b200vae_icnn_decode_jac gives J1 and J2; this kernel multiplies them and
// takes the singular values, one thread per sample, in fp64: one-sided (Hestenes) Jacobi on the columns of J (or of J^T
// when Dx < D), a fixed number of sweeps.  Column norms after orthogonalisation are the singular values with small relative
// error, which is what a lower bound sigma_min >= (inverse Lipschitz constant) needs.
#include "icnn.cuh"

namespace b200vae {

constexpr int kJacMaxDim = 4;
constexpr int kJacobiSweeps = 12;     // 4 x 4: quadratic convergence reaches fp64 rounding within ~5 sweeps

__global__ void __launch_bounds__(128) jacobian_chain_kernel(const float* __restrict__ J2, const float* __restrict__ M,
                                                             const float* __restrict__ J1, int B, int Dx, int D,
                                                             float* __restrict__ J, float* __restrict__ svals) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* j2 = J2 + (size_t)b * Dx * Dx;
  const float* j1 = J1 + (size_t)b * D * D;
  double MJ1[kJacMaxDim][kJacMaxDim], A[kJacMaxDim][kJacMaxDim];     // A = J2 . M . J1  [Dx][D]
  for (int r = 0; r < Dx; ++r)
    for (int c = 0; c < D; ++c) {
      double s = 0.0;
      for (int k = 0; k < D; ++k) s += (double)M[r * D + k] * (double)j1[k * D + c];
      MJ1[r][c] = s;
    }
  for (int r = 0; r < Dx; ++r)
    for (int c = 0; c < D; ++c) {
      double s = 0.0;
      for (int k = 0; k < Dx; ++k) s += (double)j2[r * Dx + k] * MJ1[k][c];
      A[r][c] = s;
      if (J) J[((size_t)b * Dx + r) * D + c] = (float)s;
    }
  if (!svals) return;
  // columns to orthogonalise: those of A (m = Dx rows, n = D columns) or of A^T; n = min(Dx, D)
  const bool tr = Dx < D;
  const int m = tr ? D : Dx, n = tr ? Dx : D;
  double U[kJacMaxDim][kJacMaxDim];    // U[col][row]
  for (int c = 0; c < n; ++c)
    for (int r = 0; r < m; ++r) U[c][r] = tr ? A[c][r] : A[r][c];
  for (int sweep = 0; sweep < kJacobiSweeps; ++sweep)
    for (int p = 0; p < n - 1; ++p)
      for (int q = p + 1; q < n; ++q) {
        double al = 0.0, be = 0.0, ga = 0.0;
        for (int r = 0; r < m; ++r) { al += U[p][r] * U[p][r]; be += U[q][r] * U[q][r]; ga += U[p][r] * U[q][r]; }
        if (ga == 0.0 || fabs(ga) <= 1e-300 + 1e-17 * sqrt(al * be)) continue;
        const double zeta = (be - al) / (2.0 * ga);
        const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
        for (int r = 0; r < m; ++r) {
          const double up = U[p][r], uq = U[q][r];
          U[p][r] = c * up - s * uq;
          U[q][r] = s * up + c * uq;
        }
      }
  double sv[kJacMaxDim];
  for (int c = 0; c < n; ++c) {
    double s = 0.0;
    for (int r = 0; r < m; ++r) s += U[c][r] * U[c][r];
    sv[c] = sqrt(s);
  }
  for (int i = 1; i < n; ++i)          // descending insertion sort
    for (int k = i; k > 0 && sv[k] > sv[k - 1]; --k) { const double t = sv[k]; sv[k] = sv[k - 1]; sv[k - 1] = t; }
  for (int c = 0; c < n; ++c) svals[(size_t)b * n + c] = (float)sv[c];
}

int jacobian_chain(const float* J2, const float* M, const float* J1, int B, int Dx, int D, float* J, float* svals,
                   cudaStream_t st) {
  jacobian_chain_kernel<<<(B + 127) / 128, 128, 0, st>>>(J2, M, J1, B, Dx, D, J, svals);
  return check_launch();
}

}  // namespace b200vae

using namespace b200vae;

extern "C" int b200vae_jacobian_chain(const float* J2, const float* M, const float* J1, int B, int Dx, int D, float* J,
                                      float* svals, void* stream) {
  if (B <= 0 || Dx <= 0 || D <= 0) return B200VAE_ESHAPE;
  if (Dx > kJacMaxDim || D > kJacMaxDim) return B200VAE_EUNSUP;
  if (!J2 || !M || !J1) return B200VAE_EALIGN;
  if (!J && !svals) return B200VAE_OK;
  return jacobian_chain(J2, M, J1, B, Dx, D, J, svals, (cudaStream_t)stream);
}
