// icnn_wide.cu -- fused FP32 kernels for WIDE-input ICNNs (d > 4): the MNIST-shaped LIDVAE decoder of BASELINE
// configs[3], ICNN(32,512) + ICNN(784,1024) (model.py:766-805, module.py:117-148).  Also the b200vae_icnn_wide_* entries:
// validation, the workspace size, and the choice between these kernels and the tcgen05 drivers of icnn_wide_tc.cu.
//
// For wide inputs the thin products A.z are dense [B,d]x[d,H] contractions too, so per-sample activations no longer fit in
// registers.  The path is a short chain of 128x128x16 FP32 tile GEMMs (gemm_simt.cuh) whose A operands are GENERATED while
// loading (x1 = sigma(h0)^2 from h0; g1 = s2*P1*sigma'(h1) from the saved byte mask) and whose epilogues do all the
// elementwise work, so only h0, the mask, g0 (and u0,q1,t0 in the backward) ever touch HBM:
//   forward   lin : h0 = z A0^T + b0                                        (store h0)
//             hid : h1 = x1 P0^T + z A1^T + b1  -> mask1, row partials of P1.sigma(h1)
//             row : h2 = sum partials + A2 z + b2 -> psi, s2
//             gx1 : gx1 = g1 P0 -> g0 = gx1*2a0*s0                           (store g0)
//             out : xhat = g0 A0 + g1 A1 + s2 A2 + 2 kappa z
//   backward  lin : u0 = v A0^T -> q1 = u0*2a0*s0                            (store u0, q1)
//             hid : w1 = q1 P0^T + v A1^T -> column partials of s2*s1*w1     (dP1)
//             gx1 : gx1 -> g0, t0 = u0*2gx1*s0^2, column partials of t0      (store g0, t0; db0)
//             out : dz = t0 A0 + 2 kappa v
//             tn  : dA0 = g0^T v + t0^T z,  dA1 = g1^T v,  dP0 = g1^T q1     (split over the batch, ordered slabs)
// Algebra: SURVEY.md Appendix A (oracle/icnn_oracle.py).  All reductions are ordered: bit-reproducible.
#include "gemm_simt.cuh"
#include "icnn_wide.cuh"

namespace b200vae {

enum { XF_ID = 0, XF_X1 = 1, XF_G1 = 2 };

// ---- accumulate variant of the tile core (two-phase GEMMs share one accumulator) ---------------------------------------
template <class AGen, class BGen>
__device__ __forceinline__ void gemm_tile_acc(float (&acc)[8][8], GemmSmem& sm, int KT, AGen& a, BGen& b,
                                              const TileCoord& tc) {
  if (KT <= 0) return;
  a.pre(0, sm.As[0]); b.pre(0, sm.Bs[0]);
  a.post(0, sm.As[0]); b.post(0, sm.Bs[0]);
  cp_async_commit();
  for (int kt = 0; kt < KT; ++kt) {
    const int cur = kt & 1;
    cp_async_wait_all();
    __syncthreads();
    const bool more = (kt + 1 < KT);
    if (more) { b.pre(kt + 1, sm.Bs[cur ^ 1]); a.pre(kt + 1, sm.As[cur ^ 1]); cp_async_commit(); }
    float(*As)[kBM] = sm.As[cur];
    float(*Bs)[kBN] = sm.Bs[cur];
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][tc.ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][64 + tc.ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tc.tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tc.tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (more) {
      a.post(kt + 1, sm.As[cur ^ 1]);
      b.post(kt + 1, sm.Bs[cur ^ 1]);
    }
  }
  __syncthreads();
}
__device__ __forceinline__ void zero_acc(float (&acc)[8][8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
}

// ---- operand generators -------------------------------------------------------------------------------------------------------
// A[m][k] = xf(src[(m0+m)*ld + k]), rows = samples.  Thread: row m = t&127, 8 consecutive k.
struct ARow {
  const float* src; const uint8_t* mask; const float* P1; int ld, M, K, m0, xf; float s2row;
  float r[8];
  __device__ __forceinline__ void init(const float* src_, int ld_, int M_, int K_, int m0_, int xf_, const uint8_t* mask_ = nullptr,
                                       const float* P1_ = nullptr, const float* s2 = nullptr) {
    src = src_; ld = ld_; M = M_; K = K_; m0 = m0_; xf = xf_; mask = mask_; P1 = P1_;
    const int row = m0 + (threadIdx.x & 127);
    s2row = (s2 && row < M) ? s2[row] : 0.f;
  }
  __device__ __forceinline__ void pre(int kt, float (*)[kBM]) {
    const int row = m0 + (threadIdx.x & 127), kb = kt * kBK + (threadIdx.x >> 7) * 8;
    const bool rv = row < M;
    if (xf == XF_G1) {
      const uint8_t* mp = mask + (size_t)row * ld + kb;
#pragma unroll
      for (int e = 0; e < 8; ++e) r[e] = (rv && kb + e < K) ? (mp[e] ? 1.f : kSlope) * __ldg(P1 + kb + e) : 0.f;
    } else {
      const float* sp = src + (size_t)row * ld + kb;
      if (rv && kb + 7 < K && ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15u) == 0)) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(sp)), b = __ldg(reinterpret_cast<const float4*>(sp) + 1);
        r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w; r[4] = b.x; r[5] = b.y; r[6] = b.z; r[7] = b.w;
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) r[e] = (rv && kb + e < K) ? __ldg(sp + e) : 0.f;
      }
    }
  }
  __device__ __forceinline__ void post(int, float (*As)[kBM]) {
    const int m = threadIdx.x & 127, kg = threadIdx.x >> 7;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float x = r[e];
      if (xf == XF_X1) { const float a = x * slope_of(x); x = a * a; }
      else if (xf == XF_G1) x *= s2row;
      As[kg * 8 + e][m] = x;
    }
  }
};

// A[m][k] = xf(src[(kbeg + k)*ld + m0 + m]): k runs over SAMPLES (batch-reduction GEMMs).  Thread: 2 sample rows x 4 columns.
struct ACol {
  const float* src; const uint8_t* mask; const float* P1; const float* s2; int ld, Mdim, kbeg, kend, m0, xf;
  float r[2][4];
  __device__ __forceinline__ void pre(int kt, float (*)[kBM]) {
    const int rr = threadIdx.x >> 5, c4 = (threadIdx.x & 31) * 4;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int b = kbeg + kt * kBK + rr + 8 * h;
      const bool bv = b < kend;
      const float sc = (xf == XF_G1 && bv) ? __ldg(s2 + b) : 1.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int m = m0 + c4 + j;
        float x = 0.f;
        if (bv && m < Mdim) {
          const size_t idx = (size_t)b * ld + m;
          x = (xf == XF_G1) ? sc * (mask[idx] ? 1.f : kSlope) * __ldg(P1 + m) : __ldg(src + idx);
        }
        r[h][j] = x;
      }
    }
  }
  __device__ __forceinline__ void post(int, float (*As)[kBM]) {
    const int rr = threadIdx.x >> 5, c4 = (threadIdx.x & 31) * 4;
#pragma unroll
    for (int h = 0; h < 2; ++h)
      *reinterpret_cast<float4*>(&As[rr + 8 * h][c4]) = make_float4(r[h][0], r[h][1], r[h][2], r[h][3]);
  }
};

// B[k][n] = Mx[(kbeg + k)*ld + n0 + n], guarded (k < kend, n < N): cp.async when the 16-byte chunk is whole and aligned.
struct BMat {
  const float* Mx; int ld, kbeg, kend, N, n0;
  __device__ __forceinline__ void post(int, float (*)[kBN]) {}
  __device__ __forceinline__ void pre(int kt, float (*Bs)[kBN]) {
    const int rr = threadIdx.x >> 5, c4 = (threadIdx.x & 31) * 4;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int k = kbeg + kt * kBK + rr + 8 * h, n = n0 + c4;
      const float* sp = Mx + (size_t)k * ld + n;
      if (k < kend && n + 3 < N && ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(Mx) & 15u) == 0)) {
        cp_async16(&Bs[rr + 8 * h][c4], sp);
      } else {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < kend) {
          if (n < N) v.x = __ldg(sp);
          if (n + 1 < N) v.y = __ldg(sp + 1);
          if (n + 2 < N) v.z = __ldg(sp + 2);
          if (n + 3 < N) v.w = __ldg(sp + 3);
        }
        *reinterpret_cast<float4*>(&Bs[rr + 8 * h][c4]) = v;
      }
    }
  }
};
__device__ __forceinline__ BMat make_bmat(const float* Mx, int ld, int kbeg, int kend, int N, int n0) {
  BMat b; b.Mx = Mx; b.ld = ld; b.kbeg = kbeg; b.kend = kend; b.N = N; b.n0 = n0; return b;
}
__device__ __forceinline__ int ktiles(int K) { return (K + kBK - 1) / kBK; }

// ---- prepare: P0, P0^T, P1, A0^T, A1^T (unpadded; the generators guard the edges) ------------------------------------------------
__global__ void wide_prepare_kernel(const float* __restrict__ W0, const float* __restrict__ W1, const float* __restrict__ A0w,
                                    const float* __restrict__ A1w, int d, int H, int mode, float* __restrict__ P0,
                                    float* __restrict__ P0T, float* __restrict__ P1, float* __restrict__ A0T,
                                    float* __restrict__ A1T) {
  const size_t HH = (size_t)H * H, dH = (size_t)d * H, tot = HH + H + dH, gstride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += gstride) {
    if (i < HH) {
      const float w = W0[i];
      const float p = (mode == B200VAE_WEIGHT_EXP) ? expf(w) : fmaxf(w, kClampMin);
      const size_t n = i / H, k = i - n * H;
      P0[i] = p; P0T[k * H + n] = p;
    } else if (i < HH + H) {
      const float w = W1[i - HH];
      P1[i - HH] = (mode == B200VAE_WEIGHT_EXP) ? expf(w) : fmaxf(w, kClampMin);
    } else {
      const size_t j = i - HH - H, n = j / d, c = j - n * d;    // A*w[n][c]
      A0T[c * H + n] = A0w[j]; A1T[c * H + n] = A1w[j];
    }
  }
}

// ---- lin: out = src[B,d] . WT[d,H] (+ bias);  mode 0: store h0;  mode 1: store u0 and q1 = u0 * c0(h0) ------------------------------
__global__ void __launch_bounds__(kThreads, 2)
wide_lin_kernel(const float* __restrict__ src, const float* __restrict__ WT, const float* __restrict__ bias, int B, int d, int H,
                int mode, const float* __restrict__ h0, float* __restrict__ out0, float* __restrict__ out1) {
  __shared__ GemmSmem sm;
  const TileCoord tc;
  const int m0 = blockIdx.x * kBM, n0 = blockIdx.y * kBN;
  float acc[8][8];
  zero_acc(acc);
  ARow a; a.init(src, d, B, d, m0, XF_ID);
  BMat b = make_bmat(WT, H, 0, d, H, n0);
  gemm_tile_acc(acc, sm, ktiles(d), a, b, tc);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = m0 + tc.row(i);
    if (row >= B) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = n0 + tc.col(j);
      if (col >= H) continue;
      const size_t idx = (size_t)row * H + col;
      if (mode == 0) {
        out0[idx] = acc[i][j] + bias[col];
      } else {
        const float h = h0[idx], s = slope_of(h);
        out0[idx] = acc[i][j];
        out1[idx] = acc[i][j] * (2.f * h * s * s);
      }
    }
  }
}

// ---- hid: acc = xf(src1[B,H]) . P0T[H,H] + src2[B,d] . A1T[d,H] ------------------------------------------------------------------
//   mode 0 (forward): h1 = acc + b1 -> mask1, part[row][nt] = sum_cols P1*sigma(h1)
//   mode 1 (backward): colpart[mt][col] = sum_rows s2*s1*acc
//   mode 2 (psi-gradient backward): colpart[mt][col] = sum_rows s2[row]*sigma(acc + b1)   (s2 = gpsi*s2: dP1 of dL/dpsi)
__global__ void __launch_bounds__(kThreads, 2)
wide_hid_kernel(const float* __restrict__ src1, int xf1, const float* __restrict__ P0T, const float* __restrict__ src2,
                const float* __restrict__ A1T, const float* __restrict__ b1, const float* __restrict__ P1, int B, int d, int H,
                int mode, uint8_t* __restrict__ mask1, const float* __restrict__ s2, float* __restrict__ part,
                float* __restrict__ colpart) {
  __shared__ GemmSmem sm;
  const TileCoord tc;
  const int m0 = blockIdx.x * kBM, n0 = blockIdx.y * kBN;
  float acc[8][8];
  zero_acc(acc);
  {
    ARow a; a.init(src1, H, B, H, m0, xf1);
    BMat b = make_bmat(P0T, H, 0, H, H, n0);
    gemm_tile_acc(acc, sm, ktiles(H), a, b, tc);
  }
  {
    ARow a; a.init(src2, d, B, d, m0, XF_ID);
    BMat b = make_bmat(A1T, H, 0, d, H, n0);
    gemm_tile_acc(acc, sm, ktiles(d), a, b, tc);
  }
  if (mode == 0) {
    float* red = &sm.As[0][0][0];                         // [128 rows][16 tx]
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = m0 + tc.row(i);
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int col = n0 + tc.col(j);
        if (row < B && col < H) {
          const float h = acc[i][j] + b1[col];
          mask1[(size_t)row * H + col] = h > 0.f ? 1 : 0;
          s = fmaf(P1[col], h * slope_of(h), s);
        }
      }
      red[tc.row(i) * 16 + tc.tx] = s;
    }
    __syncthreads();
    if (threadIdx.x < kBM && m0 + threadIdx.x < B) {
      float s = 0.f;
#pragma unroll
      for (int t = 0; t < 16; ++t) s += red[threadIdx.x * 16 + t];
      part[(size_t)(m0 + threadIdx.x) * gridDim.y + blockIdx.y] = s;
    }
  } else {
    float cs[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) cs[j] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = m0 + tc.row(i);
      if (row >= B) continue;
      const float sr = s2[row];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int col = n0 + tc.col(j);
        if (col >= H) continue;
        if (mode == 1) {
          cs[j] = fmaf(sr * (mask1[(size_t)row * H + col] ? 1.f : kSlope), acc[i][j], cs[j]);
        } else {
          const float h = acc[i][j] + b1[col];
          cs[j] = fmaf(sr, h * slope_of(h), cs[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float s = colsum16(cs[j]);
      const int col = n0 + tc.col(j);
      if (tc.ty == 0 && col < H) colpart[(size_t)blockIdx.x * H + col] = s;
    }
  }
}

// ---- row: h2 = sum_nt part + A2.z + b2 -> psi, s2 ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
wide_row_kernel(const float* __restrict__ part, int nt, const float* __restrict__ z, const float* __restrict__ A2w,
                const float* __restrict__ A2b, int B, int d /* = nz: columns of z */, float* __restrict__ psi,
                float* __restrict__ s2) {
  const int lane = threadIdx.x & 31, row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= B) return;
  float s = 0.f;
  for (int c = lane; c < d; c += 32) s = fmaf(__ldg(A2w + c), z[(size_t)row * d + c], s);
  s = warp_sum(s);
  if (lane == 0) {
    float h2 = s + A2b[0];
    for (int t = 0; t < nt; ++t) h2 += part[(size_t)row * nt + t];
    const float sl = slope_of(h2);
    if (psi) psi[row] = h2 * sl;
    s2[row] = sl;
  }
}

// ---- gx1: gx1 = g1 . P0 -> g0 = gx1*c0(h0); backward also t0 = u0*2*gx1*s0^2 and its column partials (db0); with t0 == null
//      and colpart != null the column partials are those of g0 itself (psi-gradient backward) --------------------------------------
__global__ void __launch_bounds__(kThreads, 2)
wide_gx1_kernel(const uint8_t* __restrict__ mask1, const float* __restrict__ s2, const float* __restrict__ P1,
                const float* __restrict__ P0, const float* __restrict__ h0, const float* __restrict__ u0, int B, int H,
                float* __restrict__ g0, float* __restrict__ t0, float* __restrict__ colpart) {
  __shared__ GemmSmem sm;
  const TileCoord tc;
  const int m0 = blockIdx.x * kBM, n0 = blockIdx.y * kBN;
  float acc[8][8];
  zero_acc(acc);
  ARow a; a.init(nullptr, H, B, H, m0, XF_G1, mask1, P1, s2);
  BMat b = make_bmat(P0, H, 0, H, H, n0);
  gemm_tile_acc(acc, sm, ktiles(H), a, b, tc);
  float cs[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) cs[j] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = m0 + tc.row(i);
    if (row >= B) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = n0 + tc.col(j);
      if (col >= H) continue;
      const size_t idx = (size_t)row * H + col;
      const float h = h0[idx], s = slope_of(h), gx = acc[i][j];
      const float gv = gx * (2.f * h * s * s);
      g0[idx] = gv;
      if (t0) {
        const float t = u0[idx] * (2.f * gx) * s * s;
        t0[idx] = t;
        cs[j] += t;
      } else if (colpart) {
        cs[j] += gv;                                        // psi-gradient backward: db0 = column sums of gpsi*g0
      }
    }
  }
  if (colpart) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float s = colsum16(cs[j]);
      const int col = n0 + tc.col(j);
      if (tc.ty == 0 && col < H) colpart[(size_t)blockIdx.x * H + col] = s;
    }
  }
}

// ---- out: out[B,d] = srcA[B,H] . A0w[H,d] (+ g1 . A1w[H,d] + s2*A2w) + 2 kappa * zv ---------------------------------------------------
__global__ void __launch_bounds__(kThreads, 2)
wide_out_kernel(const float* __restrict__ srcA, const float* __restrict__ A0w, int with_g1, const uint8_t* __restrict__ mask1,
                const float* __restrict__ s2, const float* __restrict__ P1, const float* __restrict__ A1w,
                const float* __restrict__ A2w, const float* __restrict__ zv, int zv_ld, int zv_cols, float kappa2, int B,
                int d, int N /* output columns computed (<= d) */, int H, float* __restrict__ out) {
  __shared__ GemmSmem sm;
  const TileCoord tc;
  const int m0 = blockIdx.x * kBM, n0 = blockIdx.y * kBN;
  float acc[8][8];
  zero_acc(acc);
  {
    ARow a; a.init(srcA, H, B, H, m0, XF_ID);
    BMat b = make_bmat(A0w, d, 0, H, N, n0);
    gemm_tile_acc(acc, sm, ktiles(H), a, b, tc);
  }
  if (with_g1) {
    ARow a; a.init(nullptr, H, B, H, m0, XF_G1, mask1, P1, s2);
    BMat b = make_bmat(A1w, d, 0, H, N, n0);
    gemm_tile_acc(acc, sm, ktiles(H), a, b, tc);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = m0 + tc.row(i);
    if (row >= B) continue;
    const float sr = with_g1 ? s2[row] : 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = n0 + tc.col(j);
      if (col >= N) continue;
      float o = acc[i][j];
      if (col < zv_cols) o = fmaf(kappa2, zv[(size_t)row * zv_ld + col], o);
      if (with_g1) o = fmaf(sr, A2w[col], o);
      out[(size_t)row * N + col] = o;
    }
  }
}

// ---- tn: slab[split][m][n] = sum_{b in split} xfA(srcA)[b][m] * B1[b][n]  (+ second pair) -----------------------------------------
struct TnArgs {
  const float* a1; int xf1; const float* b1;     // first product  (a1 unused for XF_G1)
  const float* a2; const float* b2; int N2;      // optional second product (identity A), b2 [B,N2], N2 <= N; may be null
  const uint8_t* mask1; const float* s2; const float* P1;
  int B, Mdim, N, rows_per_split;
  int N1;                                        // columns (= row stride) of b1; 0 = N.  Output columns >= N1 get no first product
};
__global__ void __launch_bounds__(kThreads, 2)
wide_tn_kernel(TnArgs p, float* __restrict__ slabs) {
  __shared__ GemmSmem sm;
  const TileCoord tc;
  const int m0 = blockIdx.x * kBM, n0 = blockIdx.y * kBN;
  const int kbeg = blockIdx.z * p.rows_per_split, kend = min(p.B, kbeg + p.rows_per_split);
  float acc[8][8];
  zero_acc(acc);
  const int KT = kend > kbeg ? ktiles(kend - kbeg) : 0;
  {
    ACol a; a.src = p.a1; a.mask = p.mask1; a.P1 = p.P1; a.s2 = p.s2; a.ld = p.Mdim; a.Mdim = p.Mdim; a.kbeg = kbeg; a.kend = kend;
    a.m0 = m0; a.xf = p.xf1;
    const int n1 = p.N1 > 0 ? p.N1 : p.N;
    BMat b = make_bmat(p.b1, n1, kbeg, kend, n1, n0);
    gemm_tile_acc(acc, sm, KT, a, b, tc);
  }
  if (p.a2) {
    ACol a; a.src = p.a2; a.mask = nullptr; a.P1 = nullptr; a.s2 = nullptr; a.ld = p.Mdim; a.Mdim = p.Mdim; a.kbeg = kbeg; a.kend = kend;
    a.m0 = m0; a.xf = XF_ID;
    BMat b = make_bmat(p.b2, p.N2, kbeg, kend, p.N2, n0);
    gemm_tile_acc(acc, sm, KT, a, b, tc);
  }
  float* out = slabs + (size_t)blockIdx.z * p.Mdim * p.N;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + tc.row(i);
    if (m >= p.Mdim) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = n0 + tc.col(j);
      if (n < p.N) out[(size_t)m * p.N + n] = acc[i][j];
    }
  }
}
// chain 1 recomputes P = exp(W): the tensor-core path keeps no fp32 copy of P0, and expf gives the prepare's bits
__global__ void wide_slab_finalize_kernel(const float* __restrict__ slabs, int splits, size_t n, int chain,
                                          const float* __restrict__ W, float* __restrict__ out) {
  const size_t gstride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gstride) {
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += slabs[(size_t)k * n + i];
    if (chain == 1) s *= expf(W[i]);
    else if (chain == 2) s = W[i] >= kClampMin ? s : 0.f;
    out[i] = s;
  }
}
// column sums of s2[b]*v[b][c] over 128-row blocks -> colpart[mt][c]   (dA2w)
__global__ void __launch_bounds__(256)
wide_a2_kernel(const float* __restrict__ v, const float* __restrict__ s2, int B, int d, float* __restrict__ colpart) {
  const int m0 = blockIdx.x * 128, m1 = min(B, m0 + 128);
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float s = 0.f;
    for (int b = m0; b < m1; ++b) s = fmaf(s2[b], v[(size_t)b * d + c], s);
    colpart[(size_t)blockIdx.x * d + c] = s;
  }
}
__global__ void wide_col_finalize_kernel(const float* __restrict__ colpart, int mt, int w, int chain, const float* __restrict__ P,
                                         const float* __restrict__ W, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= w) return;
  float s = 0.f;
  for (int t = 0; t < mt; ++t) s += colpart[(size_t)t * w + c];
  if (chain == 1) s *= P[c];
  else if (chain == 2) s = W[c] >= kClampMin ? s : 0.f;
  out[c] = s;
}
__global__ void wide_zero_kernel(float* __restrict__ p, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0.f;
}

// ---- psi-gradient backward helpers --------------------------------------------------------------------------------------------
// s2g[b] = gpsi[b]*s2[b];  x1[b][n] = sigma(h0[b][n])^2 (B operand of dP0 = (gpsi g1)^T x1)
__global__ void wide_psi_pre_kernel(const float* __restrict__ gpsi, const float* __restrict__ s2, const float* __restrict__ h0,
                                    int B, size_t n, float* __restrict__ s2g, float* __restrict__ x1) {
  const size_t gstride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gstride) {
    if (i < (size_t)B) s2g[i] = gpsi[i] * s2[i];
    const float h = h0[i], a = h * slope_of(h);
    x1[i] = a * a;
  }
}
// colpart[mt][c] = sum over the 128-row block of sc[b] * sigma'(h1[b][c])   (db1 / P1[c] of dL/dpsi)
__global__ void __launch_bounds__(256)
wide_maskcol_kernel(const uint8_t* __restrict__ mask1, const float* __restrict__ sc, int B, int H, float* __restrict__ colpart) {
  const int m0 = blockIdx.x * 128, m1 = min(B, m0 + 128);
  for (int c = blockIdx.y * 256 + threadIdx.x; c < H; c += gridDim.y * 256) {
    float s = 0.f;
    for (int b = m0; b < m1; ++b) s = fmaf(sc[b], mask1[(size_t)b * H + c] ? 1.f : kSlope, s);
    colpart[(size_t)blockIdx.x * H + c] = s;
  }
}
// out[0] = sum_b x[b], fixed order (one block)
__global__ void __launch_bounds__(256)
wide_sum_kernel(const float* __restrict__ x, int B, float* __restrict__ out) {
  __shared__ float red[8];
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += 256) s += x[b];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    out[0] = t;
  }
}
// out[r][c] (row stride ld) = sum_s slabs[s][r][c] for c < cols, 0 for cols <= c < ld
__global__ void wide_slab_finalize_ld_kernel(const float* __restrict__ slabs, int splits, int rows, int cols, int ld,
                                             float* __restrict__ out) {
  const size_t n = (size_t)rows * ld, gstride = (size_t)gridDim.x * blockDim.x, slab = (size_t)rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gstride) {
    const size_t r = i / ld, c = i - r * ld;
    float s = 0.f;
    if (c < (size_t)cols)
      for (int k = 0; k < splits; ++k) s += slabs[(size_t)k * slab + r * cols + c];
    out[i] = s;
  }
}

// ---- launchers of the kernels the tensor-core path shares (icnn_wide.cuh) ------------------------------------------------------
int wide_row(const float* part, int npart, const float* z, const b200vae_icnn_params* p, int B, int nz, float* psi, float* s2,
             cudaStream_t st) {
  wide_row_kernel<<<(B + 7) / 8, 256, 0, st>>>(part, npart, z, p->A2w, p->A2b, B, nz, psi, s2);
  return check_launch();
}
int wide_col_finalize(const float* colpart, int mt, int w, int chain, const float* P, const float* W, float* out,
                      cudaStream_t st) {
  wide_col_finalize_kernel<<<(w + 255) / 256, 256, 0, st>>>(colpart, mt, w, chain, P, W, out);
  return check_launch();
}
int wide_slab_finalize(const float* slabs, int splits, size_t n, int chain, const float* W, float* out, cudaStream_t st) {
  wide_slab_finalize_kernel<<<148 * 4, 256, 0, st>>>(slabs, splits, n, chain, W, out);
  return check_launch();
}

// ---- workspace layout (map: icnn_wide.cuh) ---------------------------------------------------------------------------------
// slabs of a split-batch GEMM: enough to give `ctas` CTAs over `tiles` output tiles, at least `rows` samples per slab
static int wide_splits(int B, int tiles, int ctas, int rows, int cap) {
  int s = (ctas + tiles - 1) / tiles, maxs = (B + rows - 1) / rows;
  s = s < maxs ? s : maxs;
  return s < 1 ? 1 : (s > cap ? cap : s);
}
WideLayout wide_ws_layout(int B, int d, int H, bool tc, bool for_backward) {
  WideLayout L = {};
  L.mt = (B + 127) / 128; L.nt = (H + 127) / 128;
  L.splits = 1;
  const size_t HH = (size_t)H * H, dH = (size_t)d * H, w = H > d ? H : d;
  size_t o = 0;
  auto take = [&](size_t n) { const size_t at = o; o += (n + 63) / 64 * 64; return at; };
  if (!tc) {
    L.P0 = take(HH); L.P0T = take(HH); L.P1 = take(H); L.A0T = take(dH); L.A1T = take(dH);
    L.part = take((size_t)B * L.nt);
    if (for_backward) {
      L.colpart = take(L.mt * w);
      L.splits = wide_splits(B, L.nt * L.nt, 148 * 2, 128, 32);
      L.slabs = take(L.splits * H * w);
    }
  } else {
    L.P0hi = take(HH); L.P0lo = take(HH); L.P0Thi = take(HH); L.P0Tlo = take(HH);
    L.A0hi = take(dH); L.A0lo = take(dH); L.A1hi = take(dH); L.A1lo = take(dH);
    L.A0Thi = take(dH); L.A0Tlo = take(dH); L.A1Thi = take(dH); L.A1Tlo = take(dH);
    L.P1 = take(H); L.g1b = take((size_t)B * H);
    L.part = take((size_t)B * L.nt * 2);                  // two per 128-column (3xTF32) / 256-column (TF32) tile
    if (for_backward) {
      L.colpart = take(L.mt * w);
      L.ldb = (B + 3) / 4 * 4;
      const size_t HB = (size_t)H * L.ldb, dB = (size_t)d * L.ldb;
      L.g0T = take(HB); L.t0T = take(HB); L.g1T = take(HB);
      L.vThi = take(dB); L.vTlo = take(dB); L.zThi = take(dB); L.zTlo = take(dB); L.q1Thi = take(HB); L.q1Tlo = take(HB);
      L.splits = wide_splits(B, L.nt * ((H + 255) / 256), 148, 256, 16);
      L.slabs = take(L.splits * H * w);
    }
  }
  L.end = o;
  return L;
}

// every wide entry's and the size query's check: shapes, and a precision id the wide kernels run (2 is reserved)
static int wide_shape_ok(int B, int d, int nz, int H, int precision) {
  if (B <= 0 || d <= 0 || H <= 0 || nz <= 0 || nz > d) return B200VAE_ESHAPE;
  if (precision != B200VAE_PREC_FP32 && precision != B200VAE_PREC_TF32 && precision != B200VAE_PREC_TF32X3 &&
      precision != B200VAE_PREC_F16X3)
    return B200VAE_EUNSUP;
  return B200VAE_OK;
}
// The wide kernels read their operands from HBM and have no fp16 variant: F16X3 runs as TF32X3.
static int wide_precision(int precision) {
  return precision == B200VAE_PREC_F16X3 ? B200VAE_PREC_TF32X3 : precision;
}

static int wide_prepare(const b200vae_icnn_params* p, int d, int H, int mode, float* ws, const WideLayout& L, cudaStream_t st) {
  wide_prepare_kernel<<<148 * 4, 256, 0, st>>>(p->W0, p->W1, p->A0w, p->A1w, d, H, mode, ws + L.P0, ws + L.P0T, ws + L.P1,
                                              ws + L.A0T, ws + L.A1T);
  return check_launch();
}
static bool wide_params_ok(const b200vae_icnn_params* p) {
  return p && p->A0w && p->A0b && p->A1w && p->A1b && p->A2w && p->A2b && p->W0 && p->W1;
}

}  // namespace b200vae

using namespace b200vae;

// A tensor-core precision gets the larger of the two paths' layouts: the query sees neither nz nor the parameters'
// alignment, and either can send a call to the FP32 kernels.
extern "C" size_t b200vae_icnn_wide_workspace_bytes(int B, int d, int H, int precision, int for_backward) {
  if (wide_shape_ok(B, d, d, H, precision)) return 0;
  size_t n = wide_ws_layout(B, d, H, false, for_backward != 0).end;
  if (precision != B200VAE_PREC_FP32) {
    const size_t t = wide_ws_layout(B, d, H, true, for_backward != 0).end;
    if (t > n) n = t;
  }
  return n * sizeof(float);
}

#define WIDE_CHECK() do { rc = check_launch(); if (rc) return rc; } while (0)

extern "C" int b200vae_icnn_wide_fwd(const float* z, int B, int d, int nz, int H, const b200vae_icnn_params* p, int weight_mode,
                                     float kappa, float* psi, float* xhat, float* h0, uint8_t* mask1, float* s2, float* g0,
                                     int precision, void* workspace, size_t ws_bytes, void* stream) {
  int rc = wide_shape_ok(B, d, nz, H, precision);
  if (rc) return rc;
  if (!z || !wide_params_ok(p) || !h0 || !mask1 || !s2 || !workspace || (xhat && !g0)) return B200VAE_EALIGN;
  if (weight_mode != B200VAE_WEIGHT_EXP && weight_mode != B200VAE_WEIGHT_CLAMP) return B200VAE_EUNSUP;
  if (ws_bytes < b200vae_icnn_wide_workspace_bytes(B, d, H, precision, 0)) return B200VAE_EWS;
  if (!aligned16(workspace) || !aligned16(z) || !aligned16(h0) || !aligned4(p->A0w) || !aligned4(p->A1w) ||
      (g0 && !aligned16(g0)) || (xhat && !aligned16(xhat)))
    return B200VAE_EALIGN;
  precision = wide_precision(precision);
  // the tcgen05 epilogues read b0, b1, A2 with 16-byte loads; parameters at odd offsets take the FP32 kernels
  const bool tc = wide_tc_supported(d, nz, H, precision) && aligned16(p->A0b) && aligned16(p->A1b) && aligned16(p->A2w);
  const WideLayout L = wide_ws_layout(B, d, H, tc, false);
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
  if (tc) return wide_tc_fwd(z, B, d, nz, H, p, weight_mode, kappa, psi, xhat, h0, mask1, s2, g0, ws, L, precision, st);
  rc = wide_prepare(p, d, H, weight_mode, ws, L, st);
  if (rc) return rc;
  const dim3 gH(L.mt, L.nt), gD(L.mt, (d + 127) / 128);
  // z is [B,nz]: the input is z zero-padded to d columns, so every product with z runs over nz only
  wide_lin_kernel<<<gH, kThreads, 0, st>>>(z, ws + L.A0T, p->A0b, B, nz, H, 0, nullptr, h0, nullptr);
  WIDE_CHECK();
  wide_hid_kernel<<<gH, kThreads, 0, st>>>(h0, XF_X1, ws + L.P0T, z, ws + L.A1T, p->A1b, ws + L.P1, B, nz, H, 0, mask1, nullptr,
                                          ws + L.part, nullptr);
  WIDE_CHECK();
  rc = wide_row(ws + L.part, L.nt, z, p, B, nz, psi, s2, st);
  if (rc || !xhat) return rc;
  wide_gx1_kernel<<<gH, kThreads, 0, st>>>(mask1, s2, ws + L.P1, ws + L.P0, h0, nullptr, B, H, g0, nullptr, nullptr);
  WIDE_CHECK();
  wide_out_kernel<<<gD, kThreads, 0, st>>>(g0, p->A0w, 1, mask1, s2, ws + L.P1, p->A1w, p->A2w, z, nz, nz, 2.f * kappa, B, d, d, H,
                                          xhat);
  WIDE_CHECK();
  return B200VAE_OK;
}

extern "C" int b200vae_icnn_wide_bwd(const float* z, const float* v, const float* h0, const uint8_t* mask1, const float* s2,
                                     int B, int d, int nz, int H, const b200vae_icnn_params* p, int weight_mode, float kappa,
                                     const b200vae_icnn_grads* g, float* dz, float* u0, float* q1, float* g0, float* t0,
                                     int precision, void* workspace, size_t ws_bytes, void* stream) {
  int rc = wide_shape_ok(B, d, nz, H, precision);
  if (rc) return rc;
  if (!z || !v || !h0 || !mask1 || !s2 || !wide_params_ok(p) || !u0 || !q1 || !g0 || !t0 || !workspace) return B200VAE_EALIGN;
  if (weight_mode != B200VAE_WEIGHT_EXP && weight_mode != B200VAE_WEIGHT_CLAMP) return B200VAE_EUNSUP;
  if (ws_bytes < b200vae_icnn_wide_workspace_bytes(B, d, H, precision, 1)) return B200VAE_EWS;
  if (!aligned16(workspace) || !aligned16(z) || !aligned16(v) || !aligned16(h0) || !aligned16(u0) || !aligned16(q1) ||
      !aligned16(g0) || !aligned16(t0) || !aligned4(p->A0w) || !aligned4(p->A1w) || (dz && !aligned16(dz)))
    return B200VAE_EALIGN;
  precision = wide_precision(precision);
  const bool tc = wide_tc_supported(d, nz, H, precision);
  const WideLayout L = wide_ws_layout(B, d, H, tc, true);
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
  const int chain = weight_mode == B200VAE_WEIGHT_EXP ? 1 : 2;
  const dim3 gH(L.mt, L.nt);
  if (tc) {
    rc = wide_tc_bwd_rows(v, h0, mask1, s2, B, d, nz, H, p, weight_mode, kappa, dz, u0, q1, g0, t0, g ? g->W1 : nullptr,
                          g ? g->A0b : nullptr, ws, L, precision, st);
    if (rc) return rc;
  } else {
    rc = wide_prepare(p, d, H, weight_mode, ws, L, st);
    if (rc) return rc;
    // u0 = v A0^T, q1 = u0 * c0
    wide_lin_kernel<<<gH, kThreads, 0, st>>>(v, ws + L.A0T, nullptr, B, d, H, 1, h0, u0, q1);
    WIDE_CHECK();
    // w1 = q1 P0^T + v A1^T -> dP1 (column partials) -> dW1
    wide_hid_kernel<<<gH, kThreads, 0, st>>>(q1, XF_ID, ws + L.P0T, v, ws + L.A1T, nullptr, ws + L.P1, B, d, H, 1,
                                            const_cast<uint8_t*>(mask1), s2, nullptr, ws + L.colpart);
    WIDE_CHECK();
    if (g && g->W1) {
      rc = wide_col_finalize(ws + L.colpart, L.mt, H, chain, ws + L.P1, p->W1, g->W1, st);
      if (rc) return rc;
    }
    // gx1 -> g0, t0, db0 partials
    wide_gx1_kernel<<<gH, kThreads, 0, st>>>(mask1, s2, ws + L.P1, ws + L.P0, h0, u0, B, H, g0, t0, ws + L.colpart);
    WIDE_CHECK();
    if (g && g->A0b) {
      rc = wide_col_finalize(ws + L.colpart, L.mt, H, 0, nullptr, nullptr, g->A0b, st);
      if (rc) return rc;
    }
    if (dz) {
      // dz [B,nz]: only the gradient w.r.t. the real (unpadded) input columns is formed
      wide_out_kernel<<<dim3(L.mt, (nz + 127) / 128), kThreads, 0, st>>>(t0, p->A0w, 0, nullptr, nullptr, nullptr, nullptr,
                                                                        nullptr, v, d, nz, 2.f * kappa, B, d, nz, H, dz);
      WIDE_CHECK();
    }
  }
  if (!g) return B200VAE_OK;
  if (g->A2w) {
    wide_a2_kernel<<<L.mt, 256, 0, st>>>(v, s2, B, d, ws + L.colpart);
    WIDE_CHECK();
    rc = wide_col_finalize(ws + L.colpart, L.mt, d, 0, nullptr, nullptr, g->A2w, st);
    if (rc) return rc;
  }
  if (g->A1b) { wide_zero_kernel<<<(H + 255) / 256, 256, 0, st>>>(g->A1b, H); WIDE_CHECK(); }   // sigma'' = 0: exact zeros
  if (g->A2b) { wide_zero_kernel<<<1, 32, 0, st>>>(g->A2b, 1); WIDE_CHECK(); }
  if (tc)
    return wide_tc_bwd_tn(z, v, mask1, s2, q1, g0, t0, B, d, nz, H, p, weight_mode, g->A0w, g->A1w, g->W0, ws, L, precision, st);
  TnArgs t;
  t.N1 = 0;
  t.mask1 = mask1; t.s2 = s2; t.P1 = ws + L.P1; t.B = B; t.Mdim = H;
  t.rows_per_split = round_up((B + L.splits - 1) / L.splits, kBK);
  if (g->A0w) {   // dA0 = g0^T v + t0^T z
    t.a1 = g0; t.xf1 = XF_ID; t.b1 = v; t.a2 = t0; t.b2 = z; t.N2 = nz; t.N = d;
    wide_tn_kernel<<<dim3(L.nt, (d + 127) / 128, L.splits), kThreads, 0, st>>>(t, ws + L.slabs);
    WIDE_CHECK();
    rc = wide_slab_finalize(ws + L.slabs, L.splits, (size_t)H * d, 0, nullptr, g->A0w, st);
    if (rc) return rc;
  }
  if (g->A1w) {   // dA1 = g1^T v
    t.a1 = nullptr; t.xf1 = XF_G1; t.b1 = v; t.a2 = nullptr; t.b2 = nullptr; t.N2 = 0; t.N = d;
    wide_tn_kernel<<<dim3(L.nt, (d + 127) / 128, L.splits), kThreads, 0, st>>>(t, ws + L.slabs);
    WIDE_CHECK();
    rc = wide_slab_finalize(ws + L.slabs, L.splits, (size_t)H * d, 0, nullptr, g->A1w, st);
    if (rc) return rc;
  }
  if (g->W0) {    // dP0 = g1^T q1 -> dW0
    t.a1 = nullptr; t.xf1 = XF_G1; t.b1 = q1; t.a2 = nullptr; t.b2 = nullptr; t.N2 = 0; t.N = H;
    wide_tn_kernel<<<dim3(L.nt, L.nt, L.splits), kThreads, 0, st>>>(t, ws + L.slabs);
    WIDE_CHECK();
    return wide_slab_finalize(ws + L.slabs, L.splits, (size_t)H * H, chain, p->W0, g->W0, st);
  }
  return B200VAE_OK;
}

// First-order backward of psi for wide inputs (SURVEY Appendix A, last line): gradients of L = sum_b gpsi[b]*psi[b].  With
// delta2 = gpsi*s2, delta1 = delta2*P1*sigma'(h1) (= gpsi*g1), delta0 = (delta1 P0)*2a0s0 (= gpsi*g0):
//   dA2 = delta2^T z, db2 = sum delta2, dP1 = delta2^T sigma(h1), dA1 = delta1^T z, db1 = sum delta1, dP0 = delta1^T x1,
//   dA0 = delta0^T z, db0 = sum delta0, dz = delta0 A0 + delta1 A1 + delta2 A2.
// Every product reuses the FP32 tile kernels above with s2 replaced by s2g = gpsi*s2 (g1 and g0 scale with it).
extern "C" int b200vae_icnn_wide_bwd_psi(const float* z, const float* gpsi, const float* h0, const uint8_t* mask1,
                                         const float* s2, int B, int d, int nz, int H, const b200vae_icnn_params* p,
                                         int weight_mode, const b200vae_icnn_grads* g, float* dz, float* x1, float* g0,
                                         float* s2g, void* workspace, size_t ws_bytes, void* stream) {
  int rc = wide_shape_ok(B, d, nz, H, B200VAE_PREC_FP32);
  if (rc) return rc;
  if (!z || !gpsi || !h0 || !mask1 || !s2 || !wide_params_ok(p) || !x1 || !g0 || !s2g || !workspace) return B200VAE_EALIGN;
  if (weight_mode != B200VAE_WEIGHT_EXP && weight_mode != B200VAE_WEIGHT_CLAMP) return B200VAE_EUNSUP;
  const WideLayout L = wide_ws_layout(B, d, H, false, true);
  if (ws_bytes < b200vae_icnn_wide_workspace_bytes(B, d, H, B200VAE_PREC_FP32, 1)) return B200VAE_EWS;
  if (!aligned16(workspace) || !aligned16(z) || !aligned16(h0) || !aligned16(x1) || !aligned16(g0) || !aligned4(p->A0w) ||
      !aligned4(p->A1w) || (dz && !aligned16(dz)))
    return B200VAE_EALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
  const int chain = weight_mode == B200VAE_WEIGHT_EXP ? 1 : 2;
  rc = wide_prepare(p, d, H, weight_mode, ws, L, st);
  if (rc) return rc;
  const dim3 gH(L.mt, L.nt);
  wide_psi_pre_kernel<<<148 * 4, 256, 0, st>>>(gpsi, s2, h0, B, (size_t)B * H, s2g, x1);
  WIDE_CHECK();
  // dP1 = delta2^T sigma(h1): h1 recomputed (x1 P0^T + z A1^T + b1), weighted column sums in the epilogue
  if (g && g->W1) {
    wide_hid_kernel<<<gH, kThreads, 0, st>>>(h0, XF_X1, ws + L.P0T, z, ws + L.A1T, p->A1b, ws + L.P1, B, nz, H, 2, nullptr, s2g,
                                            nullptr, ws + L.colpart);
    WIDE_CHECK();
    rc = wide_col_finalize(ws + L.colpart, L.mt, H, chain, ws + L.P1, p->W1, g->W1, st);
    if (rc) return rc;
  }
  // delta0 = (delta1 P0) * 2 a0 s0 -> g0 buffer, column sums = db0
  wide_gx1_kernel<<<gH, kThreads, 0, st>>>(mask1, s2g, ws + L.P1, ws + L.P0, h0, nullptr, B, H, g0, nullptr, ws + L.colpart);
  WIDE_CHECK();
  if (g && g->A0b) {
    rc = wide_col_finalize(ws + L.colpart, L.mt, H, 0, nullptr, nullptr, g->A0b, st);
    if (rc) return rc;
  }
  if (dz) {
    wide_out_kernel<<<dim3(L.mt, (nz + 127) / 128), kThreads, 0, st>>>(g0, p->A0w, 1, mask1, s2g, ws + L.P1, p->A1w, p->A2w, nullptr,
                                                                      0, 0, 0.f, B, d, nz, H, dz);
    WIDE_CHECK();
  }
  if (!g) return B200VAE_OK;
  if (g->A1b) {       // db1[c] = P1[c] * sum_b delta2[b] sigma'(h1[b][c])
    wide_maskcol_kernel<<<dim3(L.mt, (H + 255) / 256), 256, 0, st>>>(mask1, s2g, B, H, ws + L.colpart);
    WIDE_CHECK();
    rc = wide_col_finalize(ws + L.colpart, L.mt, H, 1, ws + L.P1, nullptr, g->A1b, st);
    if (rc) return rc;
  }
  if (g->A2w) {       // dA2[c] = sum_b delta2[b] z[b][c] for c < nz, 0 beyond (the padded inputs are zero)
    wide_a2_kernel<<<L.mt, 256, 0, st>>>(z, s2g, B, nz, ws + L.colpart);
    WIDE_CHECK();
    rc = wide_col_finalize(ws + L.colpart, L.mt, nz, 0, nullptr, nullptr, g->A2w, st);
    if (rc) return rc;
    if (d > nz) { wide_zero_kernel<<<(d - nz + 255) / 256, 256, 0, st>>>(g->A2w + nz, d - nz); WIDE_CHECK(); }
  }
  if (g->A2b) { wide_sum_kernel<<<1, 256, 0, st>>>(s2g, B, g->A2b); WIDE_CHECK(); }
  TnArgs t;
  t.mask1 = mask1; t.s2 = s2g; t.P1 = ws + L.P1; t.B = B; t.Mdim = H; t.a2 = nullptr; t.b2 = nullptr; t.N2 = 0;
  const int splits = L.splits;
  t.rows_per_split = round_up((B + splits - 1) / splits, kBK);
  if (g->A0w) {       // dA0 = delta0^T z   ([H, nz] block of [H, d])
    t.a1 = g0; t.xf1 = XF_ID; t.b1 = z; t.N = nz; t.N1 = nz;
    wide_tn_kernel<<<dim3(L.nt, (nz + 127) / 128, splits), kThreads, 0, st>>>(t, ws + L.slabs);
    WIDE_CHECK();
    wide_slab_finalize_ld_kernel<<<148 * 4, 256, 0, st>>>(ws + L.slabs, splits, H, nz, d, g->A0w);
    WIDE_CHECK();
  }
  if (g->A1w) {       // dA1 = delta1^T z
    t.a1 = nullptr; t.xf1 = XF_G1; t.b1 = z; t.N = nz; t.N1 = nz;
    wide_tn_kernel<<<dim3(L.nt, (nz + 127) / 128, splits), kThreads, 0, st>>>(t, ws + L.slabs);
    WIDE_CHECK();
    wide_slab_finalize_ld_kernel<<<148 * 4, 256, 0, st>>>(ws + L.slabs, splits, H, nz, d, g->A1w);
    WIDE_CHECK();
  }
  if (g->W0) {        // dP0 = delta1^T x1 -> dW0
    t.a1 = nullptr; t.xf1 = XF_G1; t.b1 = x1; t.N = H; t.N1 = H;
    wide_tn_kernel<<<dim3(L.nt, L.nt, splits), kThreads, 0, st>>>(t, ws + L.slabs);
    WIDE_CHECK();
    return wide_slab_finalize(ws + L.slabs, splits, (size_t)H * H, chain, p->W0, g->W0, st);
  }
  return B200VAE_OK;
}
