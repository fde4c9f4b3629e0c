// icnn_simt.cu -- FP32-SIMT kernels of the fused ICNN potential / Brenier map and its double-backward.
//
// Algebra: SURVEY.md Appendix A (verified against reference autograd, oracle/icnn_oracle.py).
// Reference lines replaced: module.py:108-114 (PositiveLinear), module.py:142-148 (ICNN.forward),
// model.py:820-822 / 826-828 (psi + kappa|z|^2 and autograd.grad -> xhat) and the autograd
// double-backward those create (lipschitz.py:41).
//
// Kernels (all operate on the PREPARED workspace, see icnn.cuh::WsLayout):
//   prepare_kernel        P0 = positive(W0) (+ transpose), P1, packed/padded A0,A1,A2
//   icnn_fwd_kernel<D>    one CTA = 128 samples: GEMM1 h1 = x1.P0^T (+A1 z+b1) -> mask bits, h2 -> psi;
//                         GEMM2 gx1 = g1.P0 -> g0 -> xhat.   Nothing but z, psi, xhat, masks touches HBM.
//   icnn_bwd_rows_kernel<D>  sample-stationary: gx1 (GEMM), w1 = u1 + P0 q1 (GEMM) (+ h1 GEMM if gpsi)
//                         -> dz, per-CTA column partials of dA0,db0,dA1,db1,dP1,dA2,db2
//   icnn_bwd_dP0_kernel<D>   output-stationary, split over the batch: dP0 = g1^T q1
//   finalize kernels      fixed-order reduction of the partials + chain through exp / clamp
// All reductions are ordered (no float atomics): results are bit-reproducible run to run.
#include "gemm_simt.cuh"
#include "icnn.cuh"

namespace b200vae {

// ------------------------------------------------------------------------------------- prepare
__global__ void prepare_kernel(const float* __restrict__ W0, const float* __restrict__ W1,
                               const float* __restrict__ A0w, const float* __restrict__ A0b,
                               const float* __restrict__ A1w, const float* __restrict__ A1b,
                               const float* __restrict__ A2w, const float* __restrict__ A2b, int d, int H,
                               int Hp, int mode, float* __restrict__ P0, float* __restrict__ P0T,
                               float* __restrict__ P1, float* __restrict__ A0p, float* __restrict__ A1p,
                               float* __restrict__ A2p) {
  __shared__ float tile[32][33];
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;   // bx: n (col of W0), by: k (row of W0)
  const int tx = threadIdx.x, ty = threadIdx.y;           // 32 x 8
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int k = by + r, n = bx + tx;
    float p = 0.f;
    if (k < H && n < H) {
      const float w = W0[(size_t)k * H + n];
      p = (mode == B200VAE_WEIGHT_EXP) ? expf(w) : fmaxf(w, kClampMin);
    }
    P0[(size_t)k * Hp + n] = p;
    tile[r][tx] = p;
  }
  __syncthreads();
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int n = bx + r, k = by + tx;
    P0T[(size_t)n * Hp + k] = tile[tx][r];
  }
  if (blockIdx.y == 0 && ty == 0) {
    const int n = bx + tx;
    const bool in = n < H;
    float p1 = 0.f;
    if (in) {
      const float w = W1[n];
      p1 = (mode == B200VAE_WEIGHT_EXP) ? expf(w) : fmaxf(w, kClampMin);
    }
    P1[n] = p1;
    for (int j = 0; j < d; ++j) {
      A0p[(size_t)n * (d + 1) + j] = in ? A0w[(size_t)n * d + j] : 0.f;
      A1p[(size_t)n * (d + 1) + j] = in ? A1w[(size_t)n * d + j] : 0.f;
    }
    A0p[(size_t)n * (d + 1) + d] = in ? A0b[n] : 0.f;
    A1p[(size_t)n * (d + 1) + d] = in ? A1b[n] : 0.f;
    if (blockIdx.x == 0 && tx < 16) A2p[tx] = (tx < d) ? A2w[tx] : (tx == d ? A2b[0] : 0.f);
  }
}

// ------------------------------------------------------------------------------ shared memory map
// [GemmSmem 32 KB][A0s Hp*(D+1)][A1s Hp*(D+1)][P1s Hp][A2s 16][zs 128*D][vs 128*D][ws 128][s2s 128]
// [colb Hp (bwd only)][maskb 128*(Hp/8+4) bytes]
template <int D>
struct SmemMap {
  GemmSmem* gs;
  float *A0s, *A1s, *P1s, *A2s, *zs, *vs, *wsv, *s2s, *colb;
  uint8_t* maskb;
  int MS;
  __device__ __forceinline__ SmemMap(unsigned char* raw, int Hp) {
    gs = reinterpret_cast<GemmSmem*>(raw);
    A0s = reinterpret_cast<float*>(raw + sizeof(GemmSmem));
    A1s = A0s + Hp * (D + 1);
    P1s = A1s + Hp * (D + 1);
    A2s = P1s + Hp;
    zs = A2s + 16;
    vs = zs + 128 * D;
    wsv = vs + 128 * D;
    s2s = wsv + 128;
    colb = s2s + 128;
    maskb = reinterpret_cast<uint8_t*>(colb + Hp);
    MS = Hp / 8 + 4;
  }
  static size_t bytes(int Hp) {
    return sizeof(GemmSmem) + sizeof(float) * ((size_t)Hp * (2 * (D + 1) + 2) + 16 + 256 * D + 256) +
           (size_t)128 * (Hp / 8 + 4);
  }
};

// A tile generators ------------------------------------------------------------------------------
// x1[m,k] = leaky(A0[k].z[m] + b0[k])^2                       (module.py:143)
template <int D>
struct AGenX1 {
  const float* A0s;
  float zg[D];
  int m, kgrp;
  __device__ __forceinline__ void post(int, float (*)[kBM]) {}
  __device__ __forceinline__ void pre(int kt, float (*As)[kBM]) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float* a = A0s + (kt * kBK + kgrp * 8 + e) * (D + 1);
      float h = a[D];
#pragma unroll
      for (int j = 0; j < D; ++j) h = fmaf(a[j], zg[j], h);
      const float a0 = h > 0.f ? h : kSlope * h;
      As[kgrp * 8 + e][m] = a0 * a0;
    }
  }
};

// g1[m,k] = s2[m] * P1[k] * s1[m,k]    (reverse sweep through layer 2 and the LeakyReLU of layer 1)
template <int D, bool kAccumA1>
struct AGenG1 {
  const float* P1s;
  const float* A1s;
  const uint8_t* maskrow;
  float s2, xa[D];
  int m, kgrp;
  bool first;
  __device__ __forceinline__ void post(int, float (*)[kBM]) {}
  __device__ __forceinline__ void pre(int kt, float (*As)[kBM]) {
    const unsigned byte = maskrow[kt * 2 + kgrp];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = kt * kBK + kgrp * 8 + e;
      const float g1 = (s2 * P1s[k]) * (((byte >> e) & 1u) ? 1.f : kSlope);
      As[kgrp * 8 + e][m] = g1;
      if (kAccumA1 && first) {
#pragma unroll
        for (int j = 0; j < D; ++j) xa[j] = fmaf(A1s[k * (D + 1) + j], g1, xa[j]);
      }
    }
  }
};

// q1[m,n] = u0 * 2 a0 s0 (+ gpsi * a0^2),  u0 = A0[n].v[m]      (Appendix A; gpsi term: dP0 += dh1^T x1)
template <int D>
struct AGenQ1 {
  const float* A0s;
  float zg[D], vg[D], wg;
  int m, kgrp;
  __device__ __forceinline__ void post(int, float (*)[kBM]) {}
  __device__ __forceinline__ void pre(int kt, float (*As)[kBM]) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float* a = A0s + (kt * kBK + kgrp * 8 + e) * (D + 1);
      float h = a[D], u = 0.f;
#pragma unroll
      for (int j = 0; j < D; ++j) { h = fmaf(a[j], zg[j], h); u = fmaf(a[j], vg[j], u); }
      const float s0 = slope_of(h), a0 = h * s0;
      As[kgrp * 8 + e][m] = u * (2.f * a0) * s0;
    }
  }
};

// deterministic cross-warp row reduction: every thread holds partial sums for its 8 rows x NV values;
// scratch [8 warps][128 rows][NV] (aliases the GEMM tiles, which are idle here).
template <int NV>
__device__ __forceinline__ void row_reduce_store(float (&part)[8][NV], float* scratch, const TileCoord& tc) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int q = 0; q < NV; ++q) {
      float v = part[i][q];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      if (tc.txl == 0) scratch[(tc.w * 128 + tc.row(i)) * NV + q] = v;
    }
}
template <int NV>
__device__ __forceinline__ float row_reduce_load(const float* scratch, int row, int q) {
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += scratch[(w * 128 + row) * NV + q];
  return s;
}

// ------------------------------------------------------------------------------------- forward
// kJac: also the Jacobian of the Brenier map, J = dxhat/dz = A0^T diag(2 s0^2 gx1) A0 + 2 kappa I (jac [B][D][D]).  With the
// masks fixed xhat is affine in z; gx1 = g1 . P0 is the phase-2 accumulator, so J costs D(D+1)/2 FMAs per (sample, unit).
template <int D>
constexpr int kJacPairs = D * (D + 1) / 2;      // upper triangle, row-major: (0,0) (0,1) .. (0,D-1) (1,1) ..

template <int D, bool kJac>
__device__ __forceinline__ void icnn_fwd_body(const float* __restrict__ z, int B, int Hp, float kappa,
                                              const float* __restrict__ P0, const float* __restrict__ P0T,
                                              const float* __restrict__ P1, const float* __restrict__ A0p,
                                              const float* __restrict__ A1p, const float* __restrict__ A2p,
                                              float* __restrict__ psi, float* __restrict__ xhat,
                                              uint32_t* __restrict__ mask1, uint8_t* __restrict__ mask2,
                                              float* __restrict__ jac) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemMap<D> S(smem_raw, Hp);
  const TileCoord tc;
  const int tid = threadIdx.x, m0 = blockIdx.x * 128;
  const int KT = Hp / kBK, MS = S.MS;

  for (int i = tid; i < Hp * (D + 1); i += kThreads) { S.A0s[i] = A0p[i]; S.A1s[i] = A1p[i]; }
  for (int i = tid; i < Hp; i += kThreads) S.P1s[i] = P1[i];
  if (tid < 16) S.A2s[tid] = A2p[tid];
  for (int i = tid; i < 128 * D; i += kThreads) S.zs[i] = (m0 + i / D < B) ? z[(size_t)m0 * D + i] : 0.f;
  __syncthreads();

  float zr[8][D];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < D; ++j) zr[i][j] = S.zs[tc.row(i) * D + j];

  float acc[8][8];
  const int mg = tid & 127, kgrp = tid >> 7;

  // ---- phase 1: h1 = x1 . P0^T + A1 z + b1 -> mask bits, h2 partial ------------------------------
  float h2p[8][1];
#pragma unroll
  for (int i = 0; i < 8; ++i) h2p[i][0] = 0.f;
  {
    AGenX1<D> ag;
    ag.A0s = S.A0s; ag.m = mg; ag.kgrp = kgrp;
#pragma unroll
    for (int j = 0; j < D; ++j) ag.zg[j] = S.zs[mg * D + j];
    for (int n0 = 0; n0 < Hp; n0 += kBN) {
      BFromMatrix bl{P0T + n0, Hp};
      gemm_tile(acc, *S.gs, KT, ag, bl, tc);
      unsigned nib_lo = 0, nib_hi = 0;   // 8 rows x 4 bits for column group 0 / 1
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int n = n0 + tc.col(j);
        const float* a1 = S.A1s + n * (D + 1);
        const float p1 = S.P1s[n];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float lin = a1[D];
#pragma unroll
          for (int jj = 0; jj < D; ++jj) lin = fmaf(a1[jj], zr[i][jj], lin);
          const float h1 = acc[i][j] + lin;
          const bool pos = h1 > 0.f;
          const float x2 = pos ? h1 : kSlope * h1;
          h2p[i][0] = fmaf(p1, x2, h2p[i][0]);
          if (pos) {
            if (j < 4) nib_lo |= 1u << (i * 4 + j); else nib_hi |= 1u << (i * 4 + (j - 4));
          }
        }
      }
      const unsigned o_lo = __shfl_xor_sync(0xffffffffu, nib_lo, 1);
      const unsigned o_hi = __shfl_xor_sync(0xffffffffu, nib_hi, 1);
      if (tc.txl == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          uint8_t* rowp = S.maskb + tc.row(i) * MS + n0 / 8 + tc.w;
          rowp[0] = (uint8_t)(((nib_lo >> (i * 4)) & 0xFu) | (((o_lo >> (i * 4)) & 0xFu) << 4));
          rowp[8] = (uint8_t)(((nib_hi >> (i * 4)) & 0xFu) | (((o_hi >> (i * 4)) & 0xFu) << 4));
        }
      }
    }
  }
  float* scratch = reinterpret_cast<float*>(S.gs);   // GEMM tiles are idle between phases
  row_reduce_store<1>(h2p, scratch, tc);
  __syncthreads();
  if (tid < 128) {
    float h2 = row_reduce_load<1>(scratch, tid, 0);
    float lin = S.A2s[D];
#pragma unroll
    for (int j = 0; j < D; ++j) lin = fmaf(S.A2s[j], S.zs[tid * D + j], lin);
    h2 += lin;
    const bool pos = h2 > 0.f;
    S.s2s[tid] = pos ? 1.f : kSlope;
    if (m0 + tid < B) {
      if (psi) psi[m0 + tid] = pos ? h2 : kSlope * h2;
      if (mask2) mask2[m0 + tid] = pos ? 1 : 0;
    }
  }
  __syncthreads();
  if (mask1) {
    const int Hw = Hp / 32;
    for (int i = tid; i < 128 * Hw; i += kThreads) {
      const int r = i / Hw, wd = i - r * Hw;
      if (m0 + r < B) mask1[(size_t)(m0 + r) * Hw + wd] = *reinterpret_cast<const uint32_t*>(S.maskb + r * MS + wd * 4);
    }
  }
  if (xhat == nullptr) return;

  // ---- phase 2: gx1 = g1 . P0 -> g0 -> xhat --------------------------------------------------------
  float xh[8][D];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < D; ++j) xh[i][j] = 0.f;
  constexpr int NJ = kJac ? kJacPairs<D> : 1;
  float yj[8][NJ];                               // kJac: sum_n A0[n,a] A0[n,b] s0^2 gx1 over my columns
  if constexpr (kJac) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int q = 0; q < NJ; ++q) yj[i][q] = 0.f;
  }
  AGenG1<D, true> ag;
  ag.P1s = S.P1s; ag.A1s = S.A1s; ag.maskrow = S.maskb + mg * MS; ag.s2 = S.s2s[mg]; ag.m = mg; ag.kgrp = kgrp;
#pragma unroll
  for (int j = 0; j < D; ++j) ag.xa[j] = 0.f;
  for (int n0 = 0; n0 < Hp; n0 += kBN) {
    ag.first = (n0 == 0);
    BFromMatrix bl{P0 + n0, Hp};
    gemm_tile(acc, *S.gs, KT, ag, bl, tc);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float* a = S.A0s + (n0 + tc.col(j)) * (D + 1);
      float aa[NJ];
      if constexpr (kJac) {
#pragma unroll
        for (int ja = 0, q = 0; ja < D; ++ja)
#pragma unroll
          for (int jb = ja; jb < D; ++jb, ++q) aa[q] = a[ja] * a[jb];
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float h = a[D];
#pragma unroll
        for (int jj = 0; jj < D; ++jj) h = fmaf(a[jj], kJac ? S.zs[tc.row(i) * D + jj] : zr[i][jj], h);
        const float s0 = slope_of(h), a0 = h * s0;
        const float g0 = acc[i][j] * (2.f * a0) * s0;
#pragma unroll
        for (int jj = 0; jj < D; ++jj) xh[i][jj] = fmaf(a[jj], g0, xh[i][jj]);
        if constexpr (kJac) {
          const float w = (s0 * s0) * acc[i][j];
#pragma unroll
          for (int q = 0; q < NJ; ++q) yj[i][q] = fmaf(aa[q], w, yj[i][q]);
        }
      }
    }
  }
  row_reduce_store<D>(xh, scratch, tc);
  float* xas = scratch + 8 * 128 * D;   // [2][128][D]
#pragma unroll
  for (int j = 0; j < D; ++j) xas[(kgrp * 128 + mg) * D + j] = ag.xa[j];
  __syncthreads();
  for (int i = tid; i < 128 * D; i += kThreads) {
    const int r = i / D, j = i - r * D;
    if (m0 + r < B) {
      float x = row_reduce_load<D>(scratch, r, j);
      x += xas[r * D + j] + xas[(128 + r) * D + j];
      x = fmaf(S.s2s[r], S.A2s[j], x);
      x = fmaf(2.f * kappa, S.zs[i], x);
      xhat[(size_t)(m0 + r) * D + j] = x;
    }
  }
  if constexpr (kJac) {
    // the same ordered cross-warp reduction, in chunks of NCH pairs (8 x 128 x NCH floats of the 32 KB scratch)
    constexpr int NCH = NJ <= 8 ? NJ : NJ / 2;
    static_assert(NJ % NCH == 0 && NCH <= 8, "Jacobian chunks must tile the pairs and fit the scratch");
#pragma unroll
    for (int c0 = 0; c0 < NJ; c0 += NCH) {
      __syncthreads();
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int q = 0; q < NCH; ++q) {
          float v = yj[i][c0 + q];
          v += __shfl_xor_sync(0xffffffffu, v, 1);
          if (tc.txl == 0) scratch[(tc.w * 128 + tc.row(i)) * NCH + q] = v;
        }
      __syncthreads();
      for (int i = tid; i < 128 * NCH; i += kThreads) {
        const int r = i / NCH, q = i - r * NCH;
        if (m0 + r >= B) continue;
        int ja = 0, jb = c0 + q;                       // pair index -> (ja, jb), ja <= jb
        while (jb >= D - ja) { jb -= D - ja; ++ja; }
        jb += ja;
        const float y = row_reduce_load<NCH>(scratch, r, q);
        const float v = ja == jb ? fmaf(2.f, y, 2.f * kappa) : 2.f * y;
        float* J = jac + (size_t)(m0 + r) * D * D;
        J[ja * D + jb] = v;
        J[jb * D + ja] = v;
      }
    }
  }
}

template <int D>
__global__ void __launch_bounds__(kThreads, 2)
icnn_fwd_kernel(const float* __restrict__ z, int B, int Hp, float kappa, const float* __restrict__ P0,
                const float* __restrict__ P0T, const float* __restrict__ P1, const float* __restrict__ A0p,
                const float* __restrict__ A1p, const float* __restrict__ A2p, float* __restrict__ psi,
                float* __restrict__ xhat, uint32_t* __restrict__ mask1, uint8_t* __restrict__ mask2) {
  icnn_fwd_body<D, false>(z, B, Hp, kappa, P0, P0T, P1, A0p, A1p, A2p, psi, xhat, mask1, mask2, nullptr);
}

// one CTA per SM: the 8 x D(D+1)/2 Jacobian accumulators need the register file of the whole SM share (no spills)
template <int D>
__global__ void __launch_bounds__(kThreads, 1)
icnn_fwd_jac_kernel(const float* __restrict__ z, int B, int Hp, float kappa, const float* __restrict__ P0,
                    const float* __restrict__ P0T, const float* __restrict__ P1, const float* __restrict__ A0p,
                    const float* __restrict__ A1p, const float* __restrict__ A2p, float* __restrict__ psi,
                    float* __restrict__ xhat, uint32_t* __restrict__ mask1, uint8_t* __restrict__ mask2,
                    float* __restrict__ jac) {
  icnn_fwd_body<D, true>(z, B, Hp, kappa, P0, P0T, P1, A0p, A1p, A2p, psi, xhat, mask1, mask2, jac);
}

// ----------------------------------------------------------------------- backward, sample-stationary
// colpart layout per (mtile, n): [0..D-1] dA0w  [D] dA0b  [D+1..2D] dA1w  [2D+1] dA1b  [2D+2] dP1
template <int D, bool kGpsi>
__global__ void __launch_bounds__(kThreads, 1)
icnn_bwd_rows_kernel(const float* __restrict__ z, const float* __restrict__ v, const float* __restrict__ gpsi,
                     const uint32_t* __restrict__ mask1, const uint8_t* __restrict__ mask2, int B, int Hp,
                     float kappa, const float* __restrict__ P0, const float* __restrict__ P0T,
                     const float* __restrict__ P1, const float* __restrict__ A0p, const float* __restrict__ A1p,
                     const float* __restrict__ A2p, float* __restrict__ dz, float* __restrict__ colpart,
                     float* __restrict__ a2part) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemMap<D> S(smem_raw, Hp);
  const TileCoord tc;
  const int tid = threadIdx.x, m0 = blockIdx.x * 128;
  const int KT = Hp / kBK, MS = S.MS, Hw = Hp / 32;
  constexpr int NF = 2 * D + 3;
  float* cp = colpart + (size_t)blockIdx.x * Hp * NF;

  for (int i = tid; i < Hp * (D + 1); i += kThreads) { S.A0s[i] = A0p[i]; S.A1s[i] = A1p[i]; }
  for (int i = tid; i < Hp; i += kThreads) { S.P1s[i] = P1[i]; S.colb[i] = 0.f; }
  if (tid < 16) S.A2s[tid] = A2p[tid];
  for (int i = tid; i < 128 * D; i += kThreads) {
    const bool in = (m0 + i / D < B);
    S.zs[i] = in ? z[(size_t)m0 * D + i] : 0.f;
    S.vs[i] = (in && v) ? v[(size_t)m0 * D + i] : 0.f;
  }
  if (tid < 128) {
    const bool in = (m0 + tid < B);
    S.wsv[tid] = (kGpsi && in) ? gpsi[m0 + tid] : 0.f;
    S.s2s[tid] = (in && mask2[m0 + tid]) ? 1.f : kSlope;
  }
  for (int i = tid; i < 128 * Hw; i += kThreads) {
    const int r = i / Hw, wd = i - r * Hw;
    *reinterpret_cast<uint32_t*>(S.maskb + r * MS + wd * 4) = (m0 + r < B) ? mask1[(size_t)(m0 + r) * Hw + wd] : 0u;
  }
  __syncthreads();

  float zr[8][D], vr[8][D], wr[8], s2r[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = tc.row(i);
#pragma unroll
    for (int j = 0; j < D; ++j) { zr[i][j] = S.zs[r * D + j]; vr[i][j] = S.vs[r * D + j]; }
    wr[i] = S.wsv[r];
    s2r[i] = S.s2s[r];
  }
  float acc[8][8];
  float dzp[8][D];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < D; ++j) dzp[i][j] = 0.f;
  const int mg = tid & 127, kgrp = tid >> 7;

  // ---- phase 0 (only when psi carries gradient): h1 again -> x2 -> dP1 += sum_m gpsi s2 x2 --------
  if (kGpsi) {
    AGenX1<D> ag;
    ag.A0s = S.A0s; ag.m = mg; ag.kgrp = kgrp;
#pragma unroll
    for (int j = 0; j < D; ++j) ag.zg[j] = S.zs[mg * D + j];
    for (int n0 = 0; n0 < Hp; n0 += kBN) {
      BFromMatrix bl{P0T + n0, Hp};
      gemm_tile(acc, *S.gs, KT, ag, bl, tc);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int n = n0 + tc.col(j);
        const float* a1 = S.A1s + n * (D + 1);
        float cs = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float lin = a1[D];
#pragma unroll
          for (int jj = 0; jj < D; ++jj) lin = fmaf(a1[jj], zr[i][jj], lin);
          const float h1 = acc[i][j] + lin;
          const unsigned byte = S.maskb[tc.row(i) * MS + n / 8];
          const float x2 = ((byte >> (n & 7)) & 1u) ? h1 : kSlope * h1;
          cs = fmaf(wr[i] * s2r[i], x2, cs);
        }
        cs = colsum16(cs);
        if (tc.ty == 0) S.colb[n] = cs;
      }
    }
    __syncthreads();
  }

  // ---- phase 1: gx1 = g1 . P0 ; column partials dA0w, dA0b ; row partial dz -------------------------
  {
    AGenG1<D, false> ag;
    ag.P1s = S.P1s; ag.A1s = S.A1s; ag.maskrow = S.maskb + mg * MS; ag.s2 = S.s2s[mg]; ag.m = mg; ag.kgrp = kgrp;
    ag.first = false;
    for (int n0 = 0; n0 < Hp; n0 += kBN) {
      BFromMatrix bl{P0 + n0, Hp};
      gemm_tile(acc, *S.gs, KT, ag, bl, tc);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int n = n0 + tc.col(j);
        const float* a = S.A0s + n * (D + 1);
        float cA[D], cb = 0.f;
#pragma unroll
        for (int jj = 0; jj < D; ++jj) cA[jj] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float h = a[D], u0 = 0.f;
#pragma unroll
          for (int jj = 0; jj < D; ++jj) { h = fmaf(a[jj], zr[i][jj], h); u0 = fmaf(a[jj], vr[i][jj], u0); }
          const float s0 = slope_of(h), a0 = h * s0, gx1 = acc[i][j];
          const float g0 = gx1 * (2.f * a0) * s0;
          float del = u0 * (2.f * gx1) * s0 * s0;        // t0
          if (kGpsi) del = fmaf(wr[i], g0, del);           // + gpsi * g0 (first-order dh0)
          cb += del;
#pragma unroll
          for (int jj = 0; jj < D; ++jj) {
            cA[jj] = fmaf(g0, vr[i][jj], cA[jj]);
            cA[jj] = fmaf(del, zr[i][jj], cA[jj]);
            dzp[i][jj] = fmaf(a[jj], del, dzp[i][jj]);
          }
        }
        cb = colsum16(cb);
#pragma unroll
        for (int jj = 0; jj < D; ++jj) cA[jj] = colsum16(cA[jj]);
        if (tc.ty == 0) {
          float* o = cp + (size_t)n * NF;
#pragma unroll
          for (int jj = 0; jj < D; ++jj) o[jj] = cA[jj];
          o[D] = cb;
        }
      }
    }
  }

  // ---- phase 2: w1 = u1 + q1 . P0^T ; column partials dP1, dA1w, dA1b ; row partial dz (gpsi) -------
  {
    AGenQ1<D> ag;
    ag.A0s = S.A0s; ag.m = mg; ag.kgrp = kgrp; ag.wg = 0.f;
#pragma unroll
    for (int j = 0; j < D; ++j) { ag.zg[j] = S.zs[mg * D + j]; ag.vg[j] = S.vs[mg * D + j]; }
    for (int n0 = 0; n0 < Hp; n0 += kBN) {
      BFromMatrix bl{P0T + n0, Hp};
      gemm_tile(acc, *S.gs, KT, ag, bl, tc);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = n0 + tc.col(j);
        const float* a1 = S.A1s + k * (D + 1);
        const float p1 = S.P1s[k];
        float cA[D], cb = 0.f, cp1 = 0.f;
#pragma unroll
        for (int jj = 0; jj < D; ++jj) cA[jj] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float u1 = 0.f;
#pragma unroll
          for (int jj = 0; jj < D; ++jj) u1 = fmaf(a1[jj], vr[i][jj], u1);
          const unsigned byte = S.maskb[tc.row(i) * MS + k / 8];
          const float s1 = ((byte >> (k & 7)) & 1u) ? 1.f : kSlope;
          const float w1 = acc[i][j] + u1;
          cp1 = fmaf(s2r[i] * s1, w1, cp1);
          const float g1 = (s2r[i] * p1) * s1;
#pragma unroll
          for (int jj = 0; jj < D; ++jj) cA[jj] = fmaf(g1, vr[i][jj], cA[jj]);
          if (kGpsi) {
            const float dh1 = wr[i] * g1;
            cb += dh1;
#pragma unroll
            for (int jj = 0; jj < D; ++jj) {
              cA[jj] = fmaf(dh1, zr[i][jj], cA[jj]);
              dzp[i][jj] = fmaf(a1[jj], dh1, dzp[i][jj]);
            }
          }
        }
        cp1 = colsum16(cp1);
        cb = colsum16(cb);
#pragma unroll
        for (int jj = 0; jj < D; ++jj) cA[jj] = colsum16(cA[jj]);
        if (tc.ty == 0) {
          float* o = cp + (size_t)k * NF + D + 1;
#pragma unroll
          for (int jj = 0; jj < D; ++jj) o[jj] = cA[jj];
          o[D] = cb;
          o[D + 1] = cp1 + S.colb[k];
        }
      }
    }
  }

  // ---- rows: dz = A0^T t0 + 2 kappa v (+ gpsi * (xhat - 2 kappa z)) ; dA2 ---------------------------
  float* scratch = reinterpret_cast<float*>(S.gs);
  row_reduce_store<D>(dzp, scratch, tc);
  __syncthreads();
  float* a2s = scratch + 8 * 128 * D;   // [128][D+1]
  if (tid < 128) {
    const int r = tid;
    const float s2 = S.s2s[r], w = S.wsv[r];
#pragma unroll
    for (int j = 0; j < D; ++j) {
      float g = row_reduce_load<D>(scratch, r, j);
      g = fmaf(2.f * kappa, S.vs[r * D + j], g);
      if (kGpsi) g = fmaf(w * s2, S.A2s[j], g);
      if (dz && m0 + r < B) dz[(size_t)(m0 + r) * D + j] = g;
      a2s[r * (D + 1) + j] = s2 * S.vs[r * D + j] + (kGpsi ? w * s2 * S.zs[r * D + j] : 0.f);
    }
    a2s[r * (D + 1) + D] = kGpsi ? w * s2 : 0.f;
    if (m0 + r >= B) {
#pragma unroll
      for (int j = 0; j <= D; ++j) a2s[r * (D + 1) + j] = 0.f;
    }
  }
  __syncthreads();
  if (tid <= D) {
    float s = 0.f;
    for (int r = 0; r < 128; ++r) s += a2s[r * (D + 1) + tid];
    a2part[(size_t)blockIdx.x * (D + 1) + tid] = s;
  }
}

// ----------------------------------------------------------------------- backward, output-stationary
// dP0part[split][k][n] = sum_{b in split} s2[b] s1[b,k] * (q1[b,n] + gpsi[b] x1[b,n])   (P1[k] applied later)
struct AGenMaskT {
  const uint32_t* mask1;
  const uint8_t* mask2;
  int Hw, b0, b1, kword, kbit, kl, bgrp;
  uint32_t wreg[8];
  uint32_t s2reg;
  __device__ __forceinline__ void pre(int kt, float (*)[kBM]) {
    s2reg = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int b = b0 + kt * kBK + bgrp * 8 + e;
      const bool in = b < b1;
      wreg[e] = in ? __ldg(mask1 + (size_t)b * Hw + kword) : 0u;
      const unsigned s2 = in ? (unsigned)__ldg(mask2 + b) : 2u;   // 2 = row out of range
      s2reg |= s2 << (2 * e);
    }
  }
  __device__ __forceinline__ void post(int, float (*As)[kBM]) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const unsigned s2 = (s2reg >> (2 * e)) & 3u;
      float val = (s2 == 1u) ? 1.f : kSlope;
      val *= ((wreg[e] >> kbit) & 1u) ? 1.f : kSlope;
      As[bgrp * 8 + e][kl] = (s2 == 2u) ? 0.f : val;
    }
  }
};

template <int D, bool kGpsi>
struct BGenQ1T {
  const float *z, *v, *gpsi;
  int b0, b1, nl, bgrp;
  float aw[D], ab;
  float zr[8][D], vr[8][D], wr[8];
  __device__ __forceinline__ void pre(int kt, float (*)[kBN]) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int b = b0 + kt * kBK + bgrp * 8 + e;
      const bool in = b < b1;
#pragma unroll
      for (int j = 0; j < D; ++j) {
        zr[e][j] = in ? __ldg(z + (size_t)b * D + j) : 0.f;
        vr[e][j] = (in && v) ? __ldg(v + (size_t)b * D + j) : 0.f;
      }
      wr[e] = (kGpsi && in) ? __ldg(gpsi + b) : 0.f;
    }
  }
  __device__ __forceinline__ void post(int, float (*Bs)[kBN]) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float h = ab, u = 0.f;
#pragma unroll
      for (int j = 0; j < D; ++j) { h = fmaf(aw[j], zr[e][j], h); u = fmaf(aw[j], vr[e][j], u); }
      const float s0 = slope_of(h), a0 = h * s0;
      float q = u * (2.f * a0) * s0;
      if (kGpsi) q = fmaf(wr[e], a0 * a0, q);
      Bs[bgrp * 8 + e][nl] = q;
    }
  }
};

template <int D, bool kGpsi>
__global__ void __launch_bounds__(kThreads, 1)
icnn_bwd_dP0_kernel(const float* __restrict__ z, const float* __restrict__ v, const float* __restrict__ gpsi,
                    const uint32_t* __restrict__ mask1, const uint8_t* __restrict__ mask2, int B, int Hp,
                    int rows_per_split, const float* __restrict__ A0p, float* __restrict__ dP0part) {
  __shared__ GemmSmem gs;
  const TileCoord tc;
  const int tid = threadIdx.x;
  const int n0 = blockIdx.x * kBN, k0 = blockIdx.y * kBM, split = blockIdx.z;
  const int b0 = split * rows_per_split;
  const int b1 = min(B, b0 + rows_per_split);
  const int KT = (max(b1 - b0, 0) + kBK - 1) / kBK;

  AGenMaskT ag;
  ag.mask1 = mask1; ag.mask2 = mask2; ag.Hw = Hp / 32; ag.b0 = b0; ag.b1 = b1;
  ag.kl = tid & 127; ag.bgrp = tid >> 7;
  ag.kword = (k0 + ag.kl) >> 5; ag.kbit = (k0 + ag.kl) & 31;
  BGenQ1T<D, kGpsi> bg;
  bg.z = z; bg.v = v; bg.gpsi = gpsi; bg.b0 = b0; bg.b1 = b1; bg.nl = tid & 127; bg.bgrp = tid >> 7;
  {
    const float* a = A0p + (size_t)(n0 + bg.nl) * (D + 1);
#pragma unroll
    for (int j = 0; j < D; ++j) bg.aw[j] = a[j];
    bg.ab = a[D];
  }
  float acc[8][8];
  gemm_tile(acc, gs, KT, ag, bg, tc);
  float* out = dP0part + ((size_t)split * Hp + k0) * Hp + n0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float* o = out + (size_t)tc.row(i) * Hp;
    *reinterpret_cast<float4*>(o + tc.tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    *reinterpret_cast<float4*>(o + 64 + tc.tx * 4) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
  }
}

// ------------------------------------------------------------------------------------- finalize
__global__ void finalize_W0_kernel(const float* __restrict__ part, int splits, int H, int Hp, int ldp,
                                   const float* __restrict__ P0, const float* __restrict__ P1,
                                   const float* __restrict__ W0raw, int mode, float scale, float* __restrict__ dW0) {
  // part: [splits][ldp][ldp] ordered split-K partials of sum_b s2*s1[b,k] * q1[b,n] / scale; scale*P1[k] is applied here
  const int n = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
  if (n >= H) return;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += part[((size_t)sp * ldp + k) * ldp + n];
  const float dP = (scale * P1[k]) * s;
  float g;
  if (mode == B200VAE_WEIGHT_EXP) g = dP * P0[(size_t)k * Hp + n];
  else g = (W0raw[(size_t)k * H + n] >= kClampMin) ? dP : 0.f;
  dW0[(size_t)k * H + n] = g;
}

__global__ void finalize_small_kernel(const float* __restrict__ colpart, const float* __restrict__ a2part,
                                      int n_mtiles, int d, int H, int Hp, const float* __restrict__ P1,
                                      const float* __restrict__ W1raw, int mode, b200vae_icnn_grads g) {
  const int NF = 2 * d + 3;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < H * NF) {
    const int n = idx / NF, f = idx - n * NF;
    float s = 0.f;
    for (int mt = 0; mt < n_mtiles; ++mt) s += colpart[((size_t)mt * Hp + n) * NF + f];
    if (f < d) { if (g.A0w) g.A0w[(size_t)n * d + f] = s; }
    else if (f == d) { if (g.A0b) g.A0b[n] = s; }
    else if (f <= 2 * d) { if (g.A1w) g.A1w[(size_t)n * d + (f - d - 1)] = s; }
    else if (f == 2 * d + 1) { if (g.A1b) g.A1b[n] = s; }
    else if (g.W1) {
      g.W1[n] = (mode == B200VAE_WEIGHT_EXP) ? s * P1[n] : (W1raw[n] >= kClampMin ? s : 0.f);
    }
  }
  if (idx <= d) {
    float s = 0.f;
    for (int mt = 0; mt < n_mtiles; ++mt) s += a2part[(size_t)mt * (d + 1) + idx];
    if (idx < d) { if (g.A2w) g.A2w[idx] = s; }
    else if (g.A2b) g.A2b[0] = s;
  }
}

// ------------------------------------------------------------------------------------- host side
template <int D>
static int launch_fwd(const float* z, int B, const WsLayout& L, const float* ws, float kappa, float* psi,
                      float* xhat, uint32_t* mask1, uint8_t* mask2, cudaStream_t st) {
  const size_t smem = SmemMap<D>::bytes(L.Hp);
  static bool attr_done = false;
  if (!attr_done) {
    cudaFuncSetAttribute(icnn_fwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_done = true;
  }
  if (smem > 200 * 1024) return B200VAE_EUNSUP;
  icnn_fwd_kernel<D><<<L.n_mtiles, kThreads, smem, st>>>(z, B, L.Hp, kappa, ws + L.P0, ws + L.P0T, ws + L.P1,
                                                          ws + L.A0p, ws + L.A1p, ws + L.A2p, psi, xhat, mask1, mask2);
  return check_launch();
}

template <int D>
static int launch_fwd_jac(const float* z, int B, const WsLayout& L, const float* ws, float kappa, float* psi,
                          float* xhat, uint32_t* mask1, uint8_t* mask2, float* jac, cudaStream_t st) {
  const size_t smem = SmemMap<D>::bytes(L.Hp);
  static bool attr_done = false;
  if (!attr_done) {
    cudaFuncSetAttribute(icnn_fwd_jac_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_done = true;
  }
  if (smem > 200 * 1024) return B200VAE_EUNSUP;
  icnn_fwd_jac_kernel<D><<<L.n_mtiles, kThreads, smem, st>>>(z, B, L.Hp, kappa, ws + L.P0, ws + L.P0T, ws + L.P1,
                                                              ws + L.A0p, ws + L.A1p, ws + L.A2p, psi, xhat, mask1,
                                                              mask2, jac);
  return check_launch();
}

template <int D, bool G>
static int launch_bwd(const float* z, const float* v, const float* gpsi, const uint32_t* mask1,
                      const uint8_t* mask2, int B, const WsLayout& L, float* ws, float kappa, float* dz,
                      bool need_W0, cudaStream_t st) {
  const size_t smem = SmemMap<D>::bytes(L.Hp);
  static bool attr_done = false;
  if (!attr_done) {
    cudaFuncSetAttribute(icnn_bwd_rows_kernel<D, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_done = true;
  }
  if (smem > 200 * 1024) return B200VAE_EUNSUP;
  icnn_bwd_rows_kernel<D, G><<<L.n_mtiles, kThreads, smem, st>>>(
      z, v, gpsi, mask1, mask2, B, L.Hp, kappa, ws + L.P0, ws + L.P0T, ws + L.P1, ws + L.A0p, ws + L.A1p,
      ws + L.A2p, dz, ws + L.colpart, ws + L.a2part);
  int rc = check_launch();
  if (rc) return rc;
  if (need_W0) {
    int rows = (B + L.splits - 1) / L.splits;
    rows = round_up(rows, kBK);
    dim3 grid(L.Hp / kBN, L.Hp / kBM, L.splits);
    icnn_bwd_dP0_kernel<D, G><<<grid, kThreads, 0, st>>>(z, v, gpsi, mask1, mask2, B, L.Hp, rows, ws + L.A0p,
                                                          ws + L.dP0part);
    rc = check_launch();
  }
  return rc;
}

int finalize_W0_launch(const float* part, int splits, int H, int Hp, int ldp, const float* P0, const float* P1,
                       const float* W0raw, int mode, float scale, float* dW0, cudaStream_t st) {
  dim3 grid((H + 255) / 256, H);
  finalize_W0_kernel<<<grid, 256, 0, st>>>(part, splits, H, Hp, ldp, P0, P1, W0raw, mode, scale, dW0);
  return check_launch();
}

int simt_prepare(const b200vae_icnn_params* p, const WsLayout& L, int mode, float* ws, cudaStream_t st) {
  dim3 grid(L.Hp / 32, L.Hp / 32), block(32, 8);
  prepare_kernel<<<grid, block, 0, st>>>(p->W0, p->W1, p->A0w, p->A0b, p->A1w, p->A1b, p->A2w, p->A2b, L.d, L.H, L.Hp,
                                         mode, ws + L.P0, ws + L.P0T, ws + L.P1, ws + L.A0p, ws + L.A1p, ws + L.A2p);
  return check_launch();
}

int simt_fwd(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
             const float* ws, cudaStream_t st) {
  const int B = L.B;
  switch (L.d) {
    case 1: return launch_fwd<1>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, st);
    case 2: return launch_fwd<2>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, st);
    case 3: return launch_fwd<3>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, st);
    case 4: return launch_fwd<4>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, st);
    default: return B200VAE_EUNSUP;
  }
}

int simt_fwd_jac(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
                 float* jac, const float* ws, cudaStream_t st) {
  const int B = L.B;
  switch (L.d) {
    case 1: return launch_fwd_jac<1>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, jac, st);
    case 2: return launch_fwd_jac<2>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, jac, st);
    case 3: return launch_fwd_jac<3>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, jac, st);
    case 4: return launch_fwd_jac<4>(z, B, L, ws, kappa, psi, xhat, mask1, mask2, jac, st);
    default: return B200VAE_EUNSUP;
  }
}

int simt_bwd(const float* z, const float* v, const float* gpsi, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L,
             const b200vae_icnn_params* p, int mode, float kappa, const b200vae_icnn_grads* g, float* dz, float* ws,
             cudaStream_t st) {
  const int B = L.B, d = L.d, H = L.H;
  const bool need_W0 = g && g->W0;
  int rc;
#define B200VAE_BWD(DD)                                                                                   \
  rc = gpsi ? launch_bwd<DD, true>(z, v, gpsi, mask1, mask2, B, L, ws, kappa, dz, need_W0, st)           \
            : launch_bwd<DD, false>(z, v, gpsi, mask1, mask2, B, L, ws, kappa, dz, need_W0, st)
  switch (d) {
    case 1: B200VAE_BWD(1); break;
    case 2: B200VAE_BWD(2); break;
    case 3: B200VAE_BWD(3); break;
    case 4: B200VAE_BWD(4); break;
    default: return B200VAE_EUNSUP;
  }
#undef B200VAE_BWD
  if (rc) return rc;
  if (!g) return B200VAE_OK;
  if (need_W0) {
    dim3 grid((H + 255) / 256, H);
    finalize_W0_kernel<<<grid, 256, 0, st>>>(ws + L.dP0part, L.splits, H, L.Hp, L.Hp, ws + L.P0, ws + L.P1, p->W0, mode, 1.f, g->W0);
    rc = check_launch();
    if (rc) return rc;
  }
  const int total = H * (2 * d + 3);
  finalize_small_kernel<<<(total + 255) / 256, 256, 0, st>>>(ws + L.colpart, ws + L.a2part, L.n_mtiles, d, H, L.Hp,
                                                             ws + L.P1, p->W1, mode, *g);
  return check_launch();
}

}  // namespace b200vae
