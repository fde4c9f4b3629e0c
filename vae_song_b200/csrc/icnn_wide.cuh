// icnn_wide.cuh -- host interface of the wide-input ICNN path (d > 4) behind b200vae_icnn_wide_*: the one workspace layout,
// the tensor-core drivers (icnn_wide_tc.cu) and the small kernels both paths launch (icnn_wide.cu).
#pragma once
#include "common.cuh"

namespace b200vae {

// ---- workspace layout --------------------------------------------------------------------------------------------------
// Offsets in floats from the workspace base; every region starts 256 B aligned (TMA maps are built on the tensor-core ones).
// mt = B/128, nt = H/128 (rounded up), w = max(H, d).  A call runs one path, so the workspace holds one path's regions.
//  FP32 tile GEMMs (icnn_wide.cu; also the psi-gradient backward of every precision):
//   P0 [H][H], P0T [H][H], P1 [H], A0T [d][H], A1T [d][H]    positive weights and transposed A*w (unpadded)
//   part    [B][nt]               row partials of P1.sigma(h1)
//   for_backward:
//   colpart [mt][w]               per-128-row column partials (dP1, db0, dA2)
//   slabs   [splits][H][w]        split-batch partial products of dA0, dA1, dP0 (splits <= 32)
//  tcgen05 (icnn_wide_tc.cu):
//   P0 hi,lo [H][H], P0T hi,lo [H][H], A0 hi,lo [H][d], A1 hi,lo [H][d], A0T hi,lo [d][H], A1T hi,lo [d][H]   tf32 splits
//   P1 [H], g1b [B][H] (P1*sigma'(h1): the A operand of gx1), part [B][2*nt]
//   for_backward:
//   colpart [mt][w]
//   g0T, t0T, g1T [H][ldb], vT hi,lo [d][ldb], zT hi,lo [d][ldb] (nz <= d rows used), q1T hi,lo [H][ldb]   ldb = B rounded
//                                 up to 4: the batch-reduction operands with the batch as their contiguous K dimension
//   slabs   [splits][H][w]        split-K slabs of dA0, dA1, dP0 (splits <= 16)
struct WideLayout {
  size_t P0, P0T, A0T, A1T;                                          // FP32
  size_t P0hi, P0lo, P0Thi, P0Tlo, A0hi, A0lo, A1hi, A1lo, A0Thi, A0Tlo, A1Thi, A1Tlo, g1b;    // tcgen05
  size_t g0T, t0T, g1T, vThi, vTlo, zThi, zTlo, q1Thi, q1Tlo;       // tcgen05, for_backward
  size_t P1, part, colpart, slabs, end;
  int mt, nt, splits, ldb;
};
WideLayout wide_ws_layout(int B, int d, int H, bool tc, bool for_backward);

// The tcgen05 kernels store float4 groups and their TMA maps need 16-byte row strides: d, nz, H multiples of 4.
inline bool wide_tc_supported(int d, int nz, int H, int precision) {
  return (precision == B200VAE_PREC_TF32 || precision == B200VAE_PREC_TF32X3) && d % 4 == 0 && nz % 4 == 0 && H % 4 == 0;
}

// ---- kernels both paths launch (icnn_wide.cu) ----------------------------------------------------------------------------
// h2 = sum_t part[row][t] + A2.z + b2 -> psi (may be null), s2   (z is [B, nz])
int wide_row(const float* part, int npart, const float* z, const b200vae_icnn_params* p, int B, int nz, float* psi, float* s2,
             cudaStream_t st);
// out[c] = chain(sum_t colpart[t][c]) for c < w:  chain 0 none, 1 * P[c], 2 * [W[c] >= 1e-2]
int wide_col_finalize(const float* colpart, int mt, int w, int chain, const float* P, const float* W, float* out,
                      cudaStream_t st);
// out[i] = chain(sum_s slabs[s][i]) for i < n:  chain 0 none, 1 * exp(W[i]) (dW = dP * P), 2 * [W[i] >= 1e-2]
int wide_slab_finalize(const float* slabs, int splits, size_t n, int chain, const float* W, float* out, cudaStream_t st);

// ---- tcgen05 drivers (icnn_wide_tc.cu); the entry has validated everything and chosen this path ---------------------------
// forward: h0, mask1, s2 saved in the FP32 path's format; g0 [B,H] scratch
int wide_tc_fwd(const float* z, int B, int d, int nz, int H, const b200vae_icnn_params* p, int mode, float kappa, float* psi,
                float* xhat, float* h0, uint8_t* mask1, float* s2, float* g0, float* ws, const WideLayout& L, int precision,
                cudaStream_t st);
// sample-stationary GEMMs of the backward: u0, q1 -> w1 -> dW1;  gx1 -> g0, t0 -> db0;  dz.  Runs the prepare.
int wide_tc_bwd_rows(const float* v, const float* h0, const uint8_t* mask1, const float* s2, int B, int d, int nz, int H,
                     const b200vae_icnn_params* p, int mode, float kappa, float* dz, float* u0, float* q1, float* g0, float* t0,
                     float* dW1, float* db0, float* ws, const WideLayout& L, int precision, cudaStream_t st);
// batch-reduction GEMMs of the backward: dA0 = g0^T v + t0^T z, dA1 = g1^T v, dP0 = g1^T q1 (-> dW0); after wide_tc_bwd_rows
int wide_tc_bwd_tn(const float* z, const float* v, const uint8_t* mask1, const float* s2, const float* q1, const float* g0,
                   const float* t0, int B, int d, int nz, int H, const b200vae_icnn_params* p, int mode, float* dA0w, float* dA1w,
                   float* dW0, float* ws, const WideLayout& L, int precision, cudaStream_t st);

}  // namespace b200vae
