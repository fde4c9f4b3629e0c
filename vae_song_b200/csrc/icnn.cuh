// icnn.cuh -- host interface of the d <= 4 ICNN path behind api.cu: the one workspace layout of b200vae_icnn_* and the
// entry points of the FP32 kernels (icnn_simt.cu) and of the tensor-core pair kernels (icnn_tc3.cu).
#pragma once
#include "common.cuh"

namespace b200vae {

constexpr int kTc3MaxHq = 1024;           // tensor-core precisions: H rounded up to 256 (a row of mask bits and the operand
                                          // tables must fit the pair kernels' shared memory); wider ICNNs take FP32
constexpr int kTc3MaxTiles = 16384;       // 256-row tiles of one pair-kernel forward (unit counters in the workspace)
constexpr int kTc3MaxClusters = 80;
constexpr size_t k3ScrFloatsPerCta = (size_t)128 * 256;

// ---- workspace layout ------------------------------------------------------------------------------------------------
// Offsets in floats from the 256 B aligned workspace base; every region starts 256 B aligned (TMA maps are built on some).
// Hp = H rounded up to 128, Hq = H rounded up to 256, Bp = B rounded up to 256.  What prepare writes comes first and does
// not depend on B; the forward's scratch follows, then (for_backward) the backward's.
//  every precision:
//   P0   [Hp,Hp]  P0[k][n] = positive(W0)[k][n]                (B operand of  gx1 = g1 . P0)
//   P0T  [Hp,Hp]  P0T[n][k] = P0[k][n]                         (B operand of  h1  = x1 . P0^T)
//   P1   [Hp]
//   A0p  [Hp][d+1]  (A0w[n][0..d-1], A0b[n])
//   A1p  [Hp][d+1]  (A1w[n][0..d-1], A1b[n])
//   A2p  [d+1]      (A2w[0][0..d-1], A2b[0])     (padded to 16 floats)
//  tensor-core precisions, per-unit tables in natural unit order:
//   A0q, A1q  float4[Hq] = (w0, w1, w2, bias)     (A1q: P1 in the spare lane when d <= 2)    P1q [Hq]
//  tensor-core precisions, pair kernels.  K1 = Hq + 16: GEMM1's B operand carries one extra 16-wide K-block holding A1/b1
//  (split hi/lo) so that the affine part of h1 is accumulated by the tensor core.  F16X3 keeps fp16 copies in the same regions.
//   B1a hi,lo [Hq][K1]   B1a[o][i] = P[o][i] (i < Hq);  B1a[o][Hq + m] = lin-block column m (see tc3_prepare_kernel)
//   B2g hi,lo [Hq][Hq]   B2g[i][o] = 0.2 * P1[o] * P[o][i]        (GEMM2: A operand = 1 + 4*maskbit, exact in tf32)
//   A0g  float4[Hq]      (A0w0, A0w1, A0w2, A0b) in generator order: unit 16*kb + 4*c + e sits at 16*kb + 4*e + c
//   E1   float4[Hq]      (P1[o], P1[o]*A1w[o][0..2])
//   sumV [64]            sum_o P1[o]*A1w[o][j]; scales of the FP16 mode
//   cnt  [2*kTc3MaxTiles] u32 per-(tile, cta rank) unit counters: zeroed by prepare, left zero by every launch
//   -- B dependent --
//   scr1 float4 [Bp][NP][2]  (h2 partial, tpos_0..2) per (row, pass, column half);  scr2 float4 same shape (X_0..2)
//   imask u32 [Bp][Hq/32]    LeakyReLU bits of h1 when the caller does not ask for mask1
//   cscr float4 [clusters][2 CTAs][2 halves][32][128 rows]   hi/lo modes: running sums of the K-chunked accumulation.  The
//                            tensor core adds into its fp32 accumulator with truncation, a downward bias that grows with the
//                            SQUARE of the accumulated K (measured on psi at H = 1024: 7.8e-6 / 1.2e-5 in one piece, 4.3e-6 /
//                            5.6e-6 in chunks of 512, 2.1e-6 / 2.8e-6 in chunks of 256 -- "mixed" / "default" weights); the
//                            forward therefore accumulates K in chunks of kTc3ChunkK, each in a fresh accumulator, and the
//                            epilogue warps add the chunks with round-to-nearest FP32 adds.  A thread re-reads only what it
//                            wrote itself; 256 KB per cluster, L2 resident.  Cost: the drain is a read-modify-write with
//                            dependent L2 round trips (~8 us per chunk) and the MMA warp runs at most one chunk ahead, so a
//                            chunk must outlast its predecessor's drain: 512-wide GEMM1 chunks do (12.5 us, +1 %), 256-wide
//                            ones do not (+16 %).  Hence 512 (north_star's 1e-5 is met with 1.8x margin), GEMM1 only.
//  for_backward, every precision: the FP32 backward (it also serves the psi-gradient path of the tensor-core precisions)
//   colpart [n_mtiles][Hp][2d+3]  per-CTA column partials: dA0w(d) dA0b dA1w(d) dP1 (+1 pad)
//   a2part  [n_mtiles][d+1]
//   dP0part [splits][Hp][Hp]
//  for_backward, tensor-core precisions:
//   partA, partB [Bp/256*8][d+1][Hq]   ordered column partials of the rows kernel (A0 side, A1 / P1 side)
//   a2part_tc    [Bp/256][d]
//   dP0part_tc   [dp0_splits][Hq][Hq]  ordered split-K slabs of the dP0 kernel
//   dzpart float4 [Bp][NP][2]          dz partials per (row, pass, column half)
//   accsave      [Bp][Hq]              3xTF32 / F16X3 only: the forward's GEMM2 accumulators, kept for the backward
struct WsLayout {
  int B, d, H, Hp, Hq, K1, NP, Bp;
  int n_mtiles, splits;     // FP32 kernels: 128-row tiles, dP0 slabs
  int dp0_splits;           // dP0 slabs of the pair kernels (for_backward, tensor-core precisions)
  size_t P0, P0T, P1, A0p, A1p, A2p;
  size_t A0q, A1q, P1q, B1ahi, B1alo, B2ghi, B2glo, A0g, E1, sumV, cnt, scr1, scr2, imask, cscr;
  size_t colpart, a2part, dP0part;
  size_t partA, partB, a2part_tc, dP0part_tc, dzpart;
  size_t accsave;           // 0: no such region
  size_t end;
};
WsLayout icnn_ws_layout(int B, int d, int H, int precision, bool for_backward);

// dP0 slabs of the pair kernels: one wave of long-running clusters, (Hq/256) x ceil(Hq/512) of them per slab, and at least
// 256 samples per slab.  The workspace holds the count for sm_count() / 2 clusters; a launch passes the clusters its kernel
// can keep resident and takes at most the workspace's count.
inline int dp0_splits(int B, int Hq, int clusters) {
  int s = clusters / ((Hq / 256) * ((Hq + 511) / 512));
  const int maxs = (B + 255) / 256;
  if (s > maxs) s = maxs;
  return s < 1 ? 1 : s;
}

// ---- entry points (shapes validated by api.cu) -------------------------------------------------------------------------
// FP32 kernels, icnn_simt.cu
int simt_prepare(const b200vae_icnn_params* p, const WsLayout& L, int mode, float* ws, cudaStream_t st);
int simt_fwd(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
             const float* ws, cudaStream_t st);
int simt_fwd_jac(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
                 float* jac, const float* ws, cudaStream_t st);
int simt_bwd(const float* z, const float* v, const float* gpsi, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L,
             const b200vae_icnn_params* p, int mode, float kappa, const b200vae_icnn_grads* g, float* dz, float* ws,
             cudaStream_t st);
int finalize_W0_launch(const float* part, int splits, int H, int Hp, int ldp, const float* P0, const float* P1,
                       const float* W0raw, int mode, float scale, float* dW0, cudaStream_t st);
// tensor-core pair kernels, icnn_tc3.cu (after simt_prepare has written the FP32 arrays)
int tc3_prepare(const WsLayout& L, int precision, float* ws, cudaStream_t st);
int tc3_fwd(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
            int precision, float* ws, float* accsave, cudaStream_t st);
// the same forward, also writing jac [B,d,d]; jscr: tc3_jac_slots(d) float4 per (row, pass, column half), Bp x NP x 2 of them
inline int tc3_jac_slots(int d) { return d <= 2 ? 1 : 2; }
int tc3_fwd_jac(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
                float* jac, float4* jscr, int precision, float* ws, cudaStream_t st);
// chain + singular values of the decoder's Jacobian, jacobian.cu
int jacobian_chain(const float* J2, const float* M, const float* J1, int B, int Dx, int D, float* J, float* svals,
                   cudaStream_t st);
// Newton left inverse of the Brenier map, inverse.cu
size_t inverse_state_bytes(int B);
int brenier_inverse_init(const float* x, const float* z0, int B, int d, float tol_rel, float tol_abs, void* state,
                         float* ztrial, float* z, int* status, float* err, cudaStream_t st);
int brenier_newton_step(const float* x, const float* xhat, const float* jac, int B, int d, float kappa, int round,
                        int final_round, void* state, float* ztrial, float* z, int* status, float* err, cudaStream_t st);
int tc_bwd(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L,
           const b200vae_icnn_params* p, int mode, float kappa, const b200vae_icnn_grads* g, float* dz, int precision,
           float* ws, const float* accsave, int phase, cudaStream_t st);

}  // namespace b200vae
