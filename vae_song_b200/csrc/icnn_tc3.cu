// icnn_tc3.cu -- persistent CTA-pair (tcgen05 cta_group::2) fused ICNN potential + Brenier map (forward).
//
// Why this design: ncu showed round 1's single-CTA kernel (one 256-row tile per CTA, since deleted) to be ISSUE bound, not tensor bound
// (about 2000 warp instructions per 16-wide K-block against 512 tensor cycles), with the epilogue exposed
// (D[256x256] fills TMEM) and 256 tiles on 148 SMs.  This kernel removes all three:
//   * lean operand generators.  GEMM1's A = leaky(A0 z + b0)^2 is computed with packed f32x2 FMAs and rounded to
//     tf32 with ONE integer add (the tensor core ignores the low 13 bits).  GEMM2's A operand is no longer
//     g1 = s2*P1*s1 but the bare LeakyReLU slope pattern 1 + 4*bit (1.0 / 5.0, exact in tf32): P1 and the factor
//     0.2 are folded into the B operand (B2g = 0.2*P1[o]*P[o][i], prepared once), s2 is a per-row scalar applied
//     at the very end.  The affine part A1 z + b1 of h1 rides in one extra K-block of GEMM1 (z and A1 split hi/lo,
//     so it is fp32-accurate in every precision) and xhat's A1^T g1 term is a predicated add in GEMM1's epilogue.
//   * CTA pairs: one tcgen05.mma.cta_group::2 (M=256, N=256, K=8) drives both SMs, each SM holds 128 sample rows
//     (A tile + accumulator) and half of every B tile: half the shared-memory operand traffic per MMA, and the
//     512 TMEM columns hold TWO accumulators, so 8 epilogue warps drain unit i while 8 generator warps feed unit i+1.
//   * persistent scheduling over fine units.  Unit = (256-row tile, GEMM, 256-column pass); 74 clusters walk the
//     unit list round-robin (all GEMM1 units first).  Cross-unit data (mask bits, per-pass partial sums) goes
//     through an L2-resident scratch; a per-(tile, rank) counter orders GEMM2 after GEMM1 and elects the last
//     unit of a tile to combine the partials in a FIXED order (bit-reproducible, no float atomics).
// Reference lines replaced: module.py:142-148 (ICNN.forward) and model.py:820-822 / 826-828 (grad of psi).
#include <mutex>
#include <unordered_map>

#include <cuda_fp16.h>

#include "icnn.cuh"
#include "tc_common.cuh"

namespace b200vae {

// Arithmetic of the pair kernels.  kTf32: one kind::tf32 MMA per product.  kX3: 3xTF32 (operands split tf32 hi/lo).
// kF16: operands split into FP16 hi/lo pairs and fed to kind::f16 MMAs (a_lo.b_hi + a_hi.b_lo + a_hi.b_hi): an fp16 pair
// carries 22 mantissa bits like a tf32 pair, but kind::f16 runs at twice the tf32 rate and the operand bytes halve, so
// the fp32-grade contraction costs 1.5 instead of 3 tf32-MMA times.  FP16 has a 5-bit exponent, so every operand is
// scaled by a power of two (exact) into the fp16 range and the accumulator is unscaled in the epilogue:
//   * prepared B operands: one scale per tensor, from the tensor's maximum (tc3_rowmax_kernel), maximum -> [2^14, 2^15);
//   * generated A operands: one scale per sample row, from an upper bound of the row's largest element computed from
//     (z, v) and max |A0| -- the generator and the epilogue evaluate the same function (row_scale_*, explicit intrinsics
//     so that both sites round identically).
// An element more than 2^17 below its row / tensor maximum lands in the fp16 subnormal range and keeps an ABSOLUTE error
// of 2^-25 (scaled units), i.e. < 2^-39 of the maximum: far below fp32 rounding of the sum.
constexpr int kTf32 = 0, kX3 = 1, kF16 = 2;

constexpr int k3Rows = 128;                       // sample rows per CTA
constexpr int k3Threads = 18 * 32;                // 8 epilogue warps, 8 generator warps, TMA warp, MMA warp
constexpr int k3TileBytes = k3Rows * 64;          // 128 rows x 64 B = 8 KB (A tile, and this CTA's half of a B tile)
constexpr int k3MaskStride = 36;                  // words per row of the shared mask buffer (16 B aligned, conflict free)
static_assert(kTc3MaxHq / 32 <= k3MaskStride, "a row of mask bits must fit the shared mask buffer");
constexpr int kTc3ChunkK = 512;                   // K per accumulation chunk of the hi/lo modes (WsLayout::cscr, icnn.cuh)
constexpr uint32_t k3ParkNs = 2000;               // suspend-time hint of the epilogue warps' accumulator waits
constexpr uint32_t k3Idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

__device__ __forceinline__ uint32_t cluster_rank3() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id3() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t num_clusters3() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync3() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa3(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t lead_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(lead_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(k3Idesc), "r"(acc) : "memory");
}
constexpr uint32_t k3IdescF16 = (1u << 4) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);   // A = B = F16, D = F32
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(k3IdescF16), "r"(acc) : "memory");
}
template <bool F16>
__device__ __forceinline__ void umma_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t acc) {
  if (F16) umma_f16_pair(tmem_d, adesc, bdesc, acc);
  else umma_tf32_pair(tmem_d, adesc, bdesc, acc);
}
// ---- FP16 hi/lo operands --------------------------------------------------------------------------------------------
// (a, b) -> packed fp16 pairs: hi = rn16(x), lo = rn16(x - hi); a in the low half (lower address = lower k)
__device__ __forceinline__ void split_f16(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// two LeakyReLU bits (bit 0, bit 1 of w) -> packed fp16 (1.0 | 5.0, 1.0 | 5.0): 0x3C00 + 0x0900 = 0x4500
__device__ __forceinline__ uint32_t pat2_f16(uint32_t w) { return 0x3C003C00u + ((w & 1u) | ((w & 2u) << 15)) * 0x0900u; }
// biased exponent of a non-negative float, clamped
__device__ __forceinline__ uint32_t bexp_of(float x, uint32_t lo, uint32_t hi) {
  const uint32_t e = (__float_as_uint(x) >> 23) & 0xffu;
  return min(max(e, lo), hi);
}
// upper bound of max_k |A0 z + b0|_k:  am = (max|A0w_0|, max|A0w_1|, max|A0w_2|, max|A0b|)
template <int D>
__device__ __forceinline__ float h0_bound(const float (&z)[D], const float4 am) {
  float b = fmaf(am.x, fabsf(z[0]), am.w);
  if (D > 1) b = fmaf(am.y, fabsf(z[D > 1 ? 1 : 0]), b);
  if (D > 2) b = fmaf(am.z, fabsf(z[D > 2 ? 2 : 0]), b);
  return b;
}
// GEMM1 rows: h0 is scaled by t = 2^(6 - floor(log2 bound)) so that x1 = leaky(h0)^2 t^2 < 2^14; inv = t^-2
template <int D>
__device__ __forceinline__ void row_scale_x1(const float (&z)[D], const float4 am, float& t, float& inv) {
  const uint32_t e = bexp_of(h0_bound<D>(z, am), 70u, 196u);
  t = __uint_as_float((260u - e) << 23);
  inv = __uint_as_float((2u * e - 139u) << 23);
}
// backward B-units: q1 = 2 (A0 v) h0 s0^2 is bounded by (sum_j max|A0w_j| |2 v_j|) * bound(h0); t = 2^(13 - floor(log2 bound))
template <int D>
__device__ __forceinline__ void row_scale_q1(const float (&z)[D], const float (&v)[D], const float4 am, float& t, float& inv) {
  float bu = __fmul_rn(am.x, fabsf(2.f * v[0]));
  if (D > 1) bu = fmaf(am.y, fabsf(2.f * v[D > 1 ? 1 : 0]), bu);
  if (D > 2) bu = fmaf(am.z, fabsf(2.f * v[D > 2 ? 2 : 0]), bu);
  const uint32_t e = bexp_of(__fmul_rn(bu, h0_bound<D>(z, am)), 30u, 220u);
  t = __uint_as_float((267u - e) << 23);
  inv = __uint_as_float((e - 13u) << 23);
}
// tensor scale from the bit pattern of the tensor's maximum: maximum * s in [2^14, 2^15)
__device__ __forceinline__ void tensor_scale(uint32_t maxbits, float& s, float& inv) {
  const uint32_t e = min(max((maxbits >> 23) & 0xffu, 15u), 253u);
  s = __uint_as_float((268u - e) << 23);
  inv = __uint_as_float((e - 14u) << 23);
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ int round_up_dev(int x, int m) { return (x + m - 1) / m * m; }
// float offset of the saved-accumulator block (tile, cta rank, pass, column half, 32-column chunk): [32 columns][128 rows]
__device__ __forceinline__ size_t k3_save_block(int tile, int rank, int NP, int pass, int chalf, int cc) {
  return ((((size_t)(tile * 2 + rank) * NP + pass) * 2 + chalf) * 4 + cc) * (size_t)(32 * 128);
}
__device__ __forceinline__ void bar_epi() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ void bar_gen() { asm volatile("bar.sync 2, 256;" ::: "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ------------------------------------------------------------------------------------ prepare
// grid (ceil(K1/256), Hq): row r, column c of the four operand copies; row 0 also packs the per-unit parameter tables
__global__ void tc3_prepare_kernel(const float* __restrict__ P0, const float* __restrict__ P0T, const float* __restrict__ P1,
                                   const float* __restrict__ A0p, const float* __restrict__ A1p, int d, int Hp, int Hq,
                                   int K1, int want_lo, float* __restrict__ B1ahi, float* __restrict__ B1alo,
                                   float* __restrict__ B2ghi, float* __restrict__ B2glo, float4* __restrict__ A0g,
                                   float4* __restrict__ E1) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= K1) return;
  const bool rin = r < Hp;
  if (c < Hq) {
    const bool in = rin && c < Hp;
    const float a = in ? P0[(size_t)r * Hp + c] : 0.f;                              // P[o=r][i=c]
    const float b = in ? (kSlope * P1[c]) * P0T[(size_t)r * Hp + c] : 0.f;          // 0.2 * P1[o=c] * P[o=c][i=r]
    const float ah = to_tf32(a), bh = to_tf32(b);
    B1ahi[(size_t)r * K1 + c] = ah;
    B2ghi[(size_t)r * Hq + c] = bh;
    if (want_lo) {
      B1alo[(size_t)r * K1 + c] = to_tf32(a - ah);
      B2glo[(size_t)r * Hq + c] = to_tf32(b - bh);
    }
    if (r == 0) {
      const bool inr = c < Hp;
      float w[4] = {0.f, 0.f, 0.f, 0.f}, u[4] = {0.f, 0.f, 0.f, 0.f};
      if (inr) {
        const float p1 = P1[c];
        for (int j = 0; j < d; ++j) { w[j] = A0p[(size_t)c * (d + 1) + j]; u[1 + j] = p1 * A1p[(size_t)c * (d + 1) + j]; }
        w[3] = A0p[(size_t)c * (d + 1) + d];
        u[0] = p1;
      }
      const int pos = (c & ~15) | ((c & 3) << 2) | ((c >> 2) & 3);                  // unit 16kb+4cc+e -> slot 16kb+4e+cc
      A0g[pos] = make_float4(w[0], w[1], w[2], w[3]);
      E1[c] = make_float4(u[0], u[1], u[2], u[3]);
    }
  } else {
    // lin block, column m: m = 3j -> A1w_j hi, 3j+1 -> A1w_j hi, 3j+2 -> A1w_j lo, 3d -> b1 hi, 3d+1 -> b1 lo.
    // The generator writes (z_j hi, z_j lo, z_j hi, ..., 1, 1): the sum is A1.z + b1 to ~2^-22 relative.
    const int m = c - Hq;
    float val = 0.f;
    if (rin && m < 3 * d + 2) {
      const int j = m < 3 * d ? m / 3 : d, t = m < 3 * d ? m % 3 : (m - 3 * d == 0 ? 0 : 2);
      const float x = A1p[(size_t)r * (d + 1) + j];
      const float xh = to_tf32(x);
      val = (t == 2) ? to_tf32(x - xh) : xh;
    }
    B1ahi[(size_t)r * K1 + c] = val;
    if (want_lo) B1alo[(size_t)r * K1 + c] = 0.f;
  }
}
// sumV[j] = sum_o E1[o].(y,z,w)[j]  (fixed order: one warp, strided partials then a shuffle tree);
// sumV[24..27] = (max |A0w_0|, max |A0w_1|, max |A0w_2|, max |A0b|) for the row scales of the FP16 mode
__global__ void tc3_sumv_kernel(const float4* __restrict__ E1, const float4* __restrict__ A0g, int Hq, float* __restrict__ sumV) {
  float s[3] = {0.f, 0.f, 0.f}, m[4] = {0.f, 0.f, 0.f, 0.f};
  for (int o = threadIdx.x; o < Hq; o += 32) {
    const float4 q = E1[o];
    s[0] += q.y; s[1] += q.z; s[2] += q.w;
    const float4 w = A0g[o];                                 // generator order: a maximum does not care
    m[0] = fmaxf(m[0], fabsf(w.x)); m[1] = fmaxf(m[1], fabsf(w.y)); m[2] = fmaxf(m[2], fabsf(w.z)); m[3] = fmaxf(m[3], fabsf(w.w));
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) s[j] = warp_sum(s[j]);
#pragma unroll
  for (int j = 0; j < 4; ++j) m[j] = warp_max(m[j]);
  if (threadIdx.x == 0) {
    sumV[0] = s[0]; sumV[1] = s[1]; sumV[2] = s[2]; sumV[3] = 0.f;
    sumV[24] = m[0]; sumV[25] = m[1]; sumV[26] = m[2]; sumV[27] = m[3];
  }
}

// ---- FP16 mode: the prepared B operands as fp16 hi/lo pairs, scaled per tensor ---------------------------------------
// mx[0] = max P0, mx[1] = max_{o,i} (0.2 P1[o]) P0[o][i] as bit patterns (non-negative floats order like unsigned ints, and a
// maximum is order independent: deterministic).  One block per output unit o; mx zeroed before the launch.
__global__ void __launch_bounds__(256) tc3_rowmax_kernel(const float* __restrict__ P0, const float* __restrict__ P1, int Hp,
                                                         uint32_t* __restrict__ mx) {
  __shared__ float red[8];
  const int o = blockIdx.x;
  float m = 0.f;
  for (int c = threadIdx.x; c < Hp; c += 256) m = fmaxf(m, P0[(size_t)o * Hp + c]);
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    atomicMax(mx, __float_as_uint(m));
    atomicMax(mx + 1, __float_as_uint((kSlope * P1[o]) * m));
  }
}
// grid (Hq/256, Hq): B1[o=r][i=c] = P[o][i] s1,  B2[i=r][o=c] = 0.2 P1[o] P[o][i] s2;  row 0 also packs the tables
// (A0g in the FP16 generator order: unit 32kb + 8cc + e sits at 32kb + 4e + cc) and the scale constants scl = (s1, 1/s1, s2, 1/s2)
__global__ void tc3_prepare_f16_kernel(const float* __restrict__ P0, const float* __restrict__ P0T, const float* __restrict__ P1,
                                       const float* __restrict__ A0p, const float* __restrict__ A1p, int d, int Hp, int Hq,
                                       const uint32_t* __restrict__ mx, __half* __restrict__ B1hi, __half* __restrict__ B1lo,
                                       __half* __restrict__ B2hi, __half* __restrict__ B2lo, float4* __restrict__ A0g,
                                       float4* __restrict__ E1, float* __restrict__ scl) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= Hq) return;
  float s1, i1, s2, i2;
  tensor_scale(mx[0], s1, i1);
  tensor_scale(mx[1], s2, i2);
  const bool in = r < Hp && c < Hp;
  const float a = in ? P0[(size_t)r * Hp + c] * s1 : 0.f;
  const float b = in ? ((kSlope * P1[c]) * P0T[(size_t)r * Hp + c]) * s2 : 0.f;
  const __half ah = __float2half_rn(a), bh = __float2half_rn(b);
  B1hi[(size_t)r * Hq + c] = ah;
  B1lo[(size_t)r * Hq + c] = __float2half_rn(a - __half2float(ah));
  B2hi[(size_t)r * Hq + c] = bh;
  B2lo[(size_t)r * Hq + c] = __float2half_rn(b - __half2float(bh));
  if (r == 0) {
    const bool inr = c < Hp;
    float w[4] = {0.f, 0.f, 0.f, 0.f}, u[4] = {0.f, 0.f, 0.f, 0.f};
    if (inr) {
      const float p1 = P1[c];
      for (int j = 0; j < d; ++j) { w[j] = A0p[(size_t)c * (d + 1) + j]; u[1 + j] = p1 * A1p[(size_t)c * (d + 1) + j]; }
      w[3] = A0p[(size_t)c * (d + 1) + d];
      u[0] = p1;
    }
    const int pos = (c & ~31) | ((c & 7) << 2) | ((c >> 3) & 3);
    A0g[pos] = make_float4(w[0], w[1], w[2], w[3]);
    E1[c] = make_float4(u[0], u[1], u[2], u[3]);
    if (c == 0) { scl[0] = s1; scl[1] = i1; scl[2] = s2; scl[3] = i2; }
  }
}

// ------------------------------------------------------------------------------------ the kernel
struct alignas(64) Tc3Args {
  CUtensorMap b1hi, b1lo, b2hi, b2lo;             // boxes of 16 x 128 (this CTA's half of a 256-row B tile)
  const float* z;
  const float4 *A0g, *E1, *A0q;
  const float4* A1q;                              // FP16 mode: (A1w0, A1w1, A1w2 | spare, A1b) per unit (WsLayout::A1q)
  const float* P1q;                               // FP16 mode: P1 per unit (WsLayout::P1q)
  const float *sumV, *A2p;                        // sumV[16..19] = (s1, 1/s1, s2, 1/s2), sumV[24..27] = max |A0| (FP16 mode)
  float *psi, *xhat;
  uint32_t* maskg;                                // mask1 of the caller or the internal scratch (null: psi-only, no masks)
  uint8_t* mask2;
  float4 *scr1, *scr2;
  uint32_t* cnt;
  float* accsave;                                 // GEMM2 accumulators (gx1 / s2) kept for the backward, or null.  Bp x Hq floats in
                                                  // blocks [tile][cta rank][pass][column half][32-column chunk] of [32 columns][128
                                                  // rows] (k3SaveBlock): the TMEM-native order, so that a warp's store of one
                                                  // column is ONE 128-byte line (row-major rows made every 256-bit store touch 32
                                                  // lines: a quarter of the LSU's time during a GEMM2 unit)
  float4* cscr;                                   // K-chunk running sums (WsLayout::cscr), used when NC > 1
  int B, Hq, T, NP, mask_stride, mask_rows, want_x;
  int NC;                                         // K-chunks per unit (hi/lo modes: Hq / kTc3ChunkK; 1 = plain accumulation)
  float kappa;
};

template <int MODE>
struct Tc3Cfg {
  static constexpr bool HL = MODE != kTf32;                               // operands come as hi/lo pairs
  static constexpr bool F16 = MODE == kF16;
  static constexpr int KBE = F16 ? 32 : 16;                               // K elements per K-block (64-byte rows)
  // K-blocks per stage: a generator thread produces 32 elements per stage either way (two 16-wide tf32 blocks or one 32-wide
  // fp16 block) -- all of them computed BEFORE it waits for the stage to drain, so that only the stores follow the wait
  static constexpr int KPS = F16 ? 1 : 2;
  static constexpr int S = F16 ? 4 : (HL ? 2 : 4);                        // stages
  static constexpr int kSubBytes = (HL ? 4 : 2) * k3TileBytes;            // one K-block: A(hi[,lo]) + B half (hi[,lo])
  static constexpr int kStageBytes = KPS * kSubBytes;
  static constexpr int kOffAlo = k3TileBytes, kOffB = (HL ? 2 : 1) * k3TileBytes, kOffBlo = 3 * k3TileBytes;
};
template <int MODE>
constexpr size_t tc3_smem_bytes(int Hq) {
  using C = Tc3Cfg<MODE>;
  return (size_t)C::S * C::kStageBytes + (size_t)Hq * (C::F16 ? 52 : 48) + 2 * k3Rows * k3MaskStride * 4 + (2 * C::S + 4) * 8 +
         64 + 1024;
}
static_assert(tc3_smem_bytes<kTf32>(kTc3MaxHq) <= 227 * 1024 && tc3_smem_bytes<kX3>(kTc3MaxHq) <= 227 * 1024 &&
                  tc3_smem_bytes<kF16>(kTc3MaxHq) <= 227 * 1024,
              "pair kernels: the per-unit tables of every mode fit in shared memory up to kTc3MaxHq");

struct Unit { int g, t, p; };
__device__ __forceinline__ Unit decode_unit(int u, int T, int NP) {
  Unit x;
  const int per = T * NP;
  x.g = u >= per ? 1 : 0;
  const int rem = u - x.g * per;
  x.t = rem / NP;
  x.p = rem - x.t * NP;
  return x;
}

// JAC: also the Brenier map's Jacobian (icnn_simt.cu, icnn_fwd_body): GEMM2 units accumulate Y[a][b] = sum_o A0[o,a] A0[o,b]
// s0^2 r (a <= b; r = gx1 / s2) beside X, publish them to jscr like scr2, and the finalizing unit writes J = 2 s2 Y + 2 kappa I.
template <int D, int MODE, bool JAC>
__device__ __forceinline__ void tc3_fwd_body(const Tc3Args& a, float4* __restrict__ jscr, float* __restrict__ jac) {
  using C = Tc3Cfg<MODE>;
  constexpr int S = C::S;
  constexpr bool X3 = C::HL, F16 = C::F16;                                 // X3: hi/lo operands, three (two) MMAs per K step
  constexpr int KBE = C::KBE, KPS = C::KPS;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* stages = smem;
  const int Hq = a.Hq;
  float4* A0gs = reinterpret_cast<float4*>(smem + S * C::kStageBytes);     // generator order
  float4* E1s = A0gs + Hq;                                                 // FP16 mode: A1q = (A1w, A1b) instead
  float4* A0qs = E1s + Hq;
  float* P1s = reinterpret_cast<float*>(A0qs + Hq);                        // FP16 mode only
  uint32_t* maskbuf = reinterpret_cast<uint32_t*>(P1s + (F16 ? Hq : 0));   // [2][128][36]
  uint64_t* bars = reinterpret_cast<uint64_t*>(maskbuf + 2 * k3Rows * k3MaskStride);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 4);
  volatile int* flags = reinterpret_cast<volatile int*>(tmem_slot + 1);   // [0] finalize (epilogue), [1] prefetch ok (generators)
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + S), accfull0 = smem_u32(bars + 2 * S),
                 accempty0 = smem_u32(bars + 2 * S + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);     // provably warp-uniform role index
  const uint32_t rank = cluster_rank3();
  const int cid = (int)cluster_id3(), G = (int)num_clusters3();
  const int T = a.T, NP = a.NP, NKB = Hq / KBE;
  const int U = (a.want_x ? 2 : 1) * T * NP;
  const uint32_t target = (uint32_t)((a.want_x ? 2 : 1) * NP);
  // FP16 mode: tensor scales of the prepared operands and max |A0| (row scales)
  const float inv_s1 = F16 ? a.sumV[17] : 1.f, inv_s2 = F16 ? a.sumV[19] : 1.f;
  const float4 amax = F16 ? make_float4(a.sumV[24], a.sumV[25], a.sumV[26], a.sumV[27]) : make_float4(0.f, 0.f, 0.f, 0.f);

  if (tid == 0) {
    // full: 4 generator warps (one group owns a whole stage) x 2 CTAs + the leader's TMA arrivals (one per K-block)
    for (int s = 0; s < S; ++s) { mbar_init(full0 + 8 * s, 8 + C::KPS); mbar_init(empty0 + 8 * s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(accfull0 + 8 * b, 1); mbar_init(accempty0 + 8 * b, 16); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 16) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
  }
  for (int i = tid; i < Hq; i += k3Threads) {
    A0gs[i] = a.A0g[i]; E1s[i] = F16 ? a.A1q[i] : a.E1[i]; A0qs[i] = a.A0q[i];
    if (F16) P1s[i] = a.P1q[i];
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync3();                         // peer barriers initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lead_full0 = mapa3(full0, 0), lead_accempty0 = mapa3(accempty0, 0);

  if (warp_u < 8) {
    // =========================== epilogue warps: my row, 128 of the unit's 256 columns ===========================
    const int row = (warp & 3) * 32 + lane, chalf = warp >> 2;
    const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(chalf * 128);
    // K-chunked accumulation (NC > 1): chunks 0 .. NC-2 of a unit are only drained and added (round to nearest) into the
    // running sums in `mysum` -- slot q of this thread = its columns 4q .. 4q+3, laid out [q][row] so that a warp's
    // accesses are contiguous; nobody else touches these slots -- and the last chunk's epilogue starts from those sums.
    const int NC = X3 ? a.NC : 1;
    float4* mysum = a.cscr + ((size_t)((cid * 2 + (int)rank) * 2 + chalf) * 32) * k3Rows + row;
    int i = 0;
    for (int u = cid; u < U; u += G, ++i) {
      const Unit un = decode_unit(u, T, NP);
      // only GEMM1 (h1: its sign bits and psi inherit the accumulation bias) is chunked; GEMM2's accumulator enters xhat
      // linearly and its one-piece error (2 MMAs per K step) stays below 2e-6
      const int nck = un.g ? 1 : NC;
      for (int ck = 0; ck + 1 < nck; ++ck, ++i) {
        const int pbuf = i & 1;
        mbar_wait_parked(accfull0 + 8 * pbuf, (i >> 1) & 1, k3ParkNs);
        tc_fence_after();
#pragma unroll 1
        for (int cc = 0; cc < 4; ++cc) {
          uint32_t r[32];
          tmem_ld32(taddr + pbuf * 256 + cc * 32, r);
          tmem_ld_wait();
          float4* slot = mysum + (size_t)(cc * 8) * k3Rows;
          // loads batched four at a time: interleaved with the stores they would serialise into one L2 round trip each
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float4 t[4];
            if (ck > 0) {
#pragma unroll
              for (int q = 0; q < 4; ++q) t[q] = __ldcg(slot + (size_t)(4 * h + q) * k3Rows);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int e = 4 * (4 * h + q);
              float4 s = make_float4(__uint_as_float(r[e]), __uint_as_float(r[e + 1]), __uint_as_float(r[e + 2]),
                                     __uint_as_float(r[e + 3]));
              if (ck > 0) { s.x += t[q].x; s.y += t[q].y; s.z += t[q].z; s.w += t[q].w; }
              __stcg(slot + (size_t)(4 * h + q) * k3Rows, s);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(lead_accempty0 + 8 * pbuf);
      }
      const int buf = i & 1;
      const int grow = un.t * 256 + (int)rank * k3Rows + row;
      const size_t sidx = ((size_t)grow * NP + un.p) * 2 + chalf;
      float zr[D];
      if (un.g || F16) {
#pragma unroll
        for (int j = 0; j < D; ++j) zr[j] = grow < a.B ? a.z[(size_t)grow * D + j] : 0.f;
      }
      float cinv = 1.f;                                       // FP16 mode, GEMM1: acc = h1 (without its affine part) / cinv
      if (F16 && !un.g) {
        float t_r, inv_x;
        row_scale_x1<D>(zr, amax, t_r, inv_x);
        cinv = inv_x * inv_s1;
      }
      mbar_wait_parked(accfull0 + 8 * buf, (i >> 1) & 1, k3ParkNs);
      tc_fence_after();
      // r = TMEM accumulator columns [32 cc, 32 cc + 32) of my row (+ the running sums of the earlier chunks)
      auto load_acc = [&](uint32_t (&r)[32], int cc) {
        tmem_ld32(taddr + buf * 256 + cc * 32, r);
        tmem_ld_wait();
        if (nck > 1) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 t = __ldcg(mysum + (size_t)(cc * 8 + q) * k3Rows);
            r[4 * q] = __float_as_uint(__uint_as_float(r[4 * q]) + t.x);
            r[4 * q + 1] = __float_as_uint(__uint_as_float(r[4 * q + 1]) + t.y);
            r[4 * q + 2] = __float_as_uint(__uint_as_float(r[4 * q + 2]) + t.z);
            r[4 * q + 3] = __float_as_uint(__uint_as_float(r[4 * q + 3]) + t.w);
          }
        }
      };
      if (!un.g) {
        float h2p = 0.f, tp[3] = {0.f, 0.f, 0.f};
        uint32_t words[4];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          uint32_t r[32];
          load_acc(r, cc);
          const int nb = un.p * 256 + chalf * 128 + cc * 32;
          uint32_t word = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (F16) {
              const float4 q = E1s[nb + j];                     // (A1w0, A1w1, A1w2 | spare, A1b)
              const float p1 = P1s[nb + j];
              const float h1 = fmaf(__uint_as_float(r[j]), cinv, lin_of<D>(q, zr));   // unscale, affine part in FP32
              h2p = fmaf(p1, fmaxf(h1, kSlope * h1), h2p);
              if (h1 > 0.f) {
                tp[0] = fmaf(p1, q.x, tp[0]);
                if (D > 1) tp[1] = fmaf(p1, q.y, tp[1]);
                if (D > 2) tp[2] = fmaf(p1, q.z, tp[2]);
                word |= 1u << j;
              }
            } else {
              const float4 q = E1s[nb + j];                     // (P1, P1*A1w0, P1*A1w1, P1*A1w2)
              const float h1 = __uint_as_float(r[j]);           // affine part included by the lin K-block
              const bool pos = h1 > 0.f;
              h2p = fmaf(q.x, fmaxf(h1, kSlope * h1), h2p);     // leaky(h) = max(h, 0.2 h)
              if (pos) {
                tp[0] += q.y;
                if (D > 1) tp[1] += q.z;
                if (D > 2) tp[2] += q.w;
                word |= 1u << j;
              }
            }
          }
          words[cc] = word;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(lead_accempty0 + 8 * buf);
        a.scr1[sidx] = make_float4(h2p, tp[0], tp[1], tp[2]);
        const int w0 = un.p * 8 + chalf * 4;
        if (a.maskg != nullptr && grow < a.mask_rows && w0 < a.mask_stride)
          *reinterpret_cast<uint4*>(a.maskg + (size_t)grow * a.mask_stride + w0) = make_uint4(words[0], words[1], words[2], words[3]);
      } else {
        float X[3] = {0.f, 0.f, 0.f};
        float Y[JAC ? (D * (D + 1)) / 2 : 1];
        if constexpr (JAC) {
#pragma unroll
          for (int q = 0; q < (D * (D + 1)) / 2; ++q) Y[q] = 0.f;
        }
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          uint32_t r[32];
          load_acc(r, cc);
          const int nb = un.p * 256 + chalf * 128 + cc * 32;
          if (F16) {                             // undo the tensor scale of B2g
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) * inv_s2);
          }
          if (a.accsave != nullptr) {            // training: the backward reads this back instead of redoing GEMM2
            float* dst = a.accsave + k3_save_block(un.t, (int)rank, NP, un.p, chalf, cc) + row;
#pragma unroll
            for (int j = 0; j < 32; ++j) __stcs(dst + j * k3Rows, __uint_as_float(r[j]));    // lane = row: coalesced
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float4 q = A0qs[nb + j];
            const float h0 = lin_of<D>(q, zr);
            const float f0 = fmaxf(h0, (kSlope * kSlope) * h0);   // a0*s0 = h0*s0^2
            const float wv = f0 * __uint_as_float(r[j]);
#pragma unroll
            for (int jj = 0; jj < D; ++jj) X[jj] = fmaf(comp(q, jj), wv, X[jj]);
            if constexpr (JAC) {
              const float yv = (h0 > 0.f ? 1.f : kSlope * kSlope) * __uint_as_float(r[j]);
#pragma unroll
              for (int ja = 0, p = 0; ja < D; ++ja)
#pragma unroll
                for (int jb = ja; jb < D; ++jb, ++p) Y[p] = fmaf(comp(q, ja) * comp(q, jb), yv, Y[p]);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(lead_accempty0 + 8 * buf);
        a.scr2[sidx] = make_float4(X[0], X[1], X[2], 0.f);
        if constexpr (JAC) {
          if constexpr (D == 1) {
            jscr[sidx] = make_float4(Y[0], 0.f, 0.f, 0.f);
          } else if constexpr (D == 2) {
            jscr[sidx] = make_float4(Y[0], Y[1], Y[2], 0.f);
          } else {
            jscr[2 * sidx] = make_float4(Y[0], Y[1], Y[2], Y[3]);
            jscr[2 * sidx + 1] = make_float4(Y[4], Y[5], 0.f, 0.f);
          }
        }
      }
      // ---- publish the unit; the last unit of this (tile, rank) combines all partials in a fixed order ----
      __threadfence();
      bar_epi();
      uint32_t* cp = a.cnt + (un.t * 2 + (int)rank);
      if (tid == 0) flags[0] = (atomicAdd(cp, 1u) + 1u == target) ? 1 : 0;
      bar_epi();
      if (flags[0]) {
        __threadfence();
        if (tid < k3Rows) {
          const int fr = un.t * 256 + (int)rank * k3Rows + tid;
          if (fr < a.B) {
            float zf[D];
#pragma unroll
            for (int j = 0; j < D; ++j) zf[j] = a.z[(size_t)fr * D + j];
            float h2 = 0.f, tp[3] = {0.f, 0.f, 0.f}, X[3] = {0.f, 0.f, 0.f};
            for (int q = 0; q < 2 * NP; ++q) {
              const float4 s1 = __ldcg(a.scr1 + (size_t)fr * NP * 2 + q);
              h2 += s1.x; tp[0] += s1.y; tp[1] += s1.z; tp[2] += s1.w;
            }
            float lin = a.A2p[D];
#pragma unroll
            for (int j = 0; j < D; ++j) lin = fmaf(a.A2p[j], zf[j], lin);
            h2 += lin;
            const bool pos2 = h2 > 0.f;
            const float s2 = pos2 ? 1.f : kSlope;
            if (a.psi) a.psi[fr] = pos2 ? h2 : kSlope * h2;
            if (a.mask2) a.mask2[fr] = pos2 ? 1 : 0;
            if (a.want_x) {
              for (int q = 0; q < 2 * NP; ++q) {
                const float4 s2v = __ldcg(a.scr2 + (size_t)fr * NP * 2 + q);
                X[0] += s2v.x; X[1] += s2v.y; X[2] += s2v.z;
              }
#pragma unroll
              for (int j = 0; j < D; ++j) {
                // xhat = A0^T g0 + A1^T g1 + s2 A2 + 2 kappa z;  g1 = s2 P1 (0.2 + 0.8 bit),  A0^T g0 = 2 s2 X
                const float a1 = fmaf(0.8f, tp[j], kSlope * a.sumV[j]);
                const float inner = fmaf(2.f, X[j], a1) + a.A2p[j];
                a.xhat[(size_t)fr * D + j] = fmaf(2.f * a.kappa, zf[j], s2 * inner);
              }
              if constexpr (JAC) {
                // same fixed order as scr2; J = 2 s2 Y + 2 kappa I, both triangles
                constexpr int NS = D <= 2 ? 1 : 2;
                float Yf[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                for (int q = 0; q < 2 * NP; ++q) {
#pragma unroll
                  for (int k = 0; k < NS; ++k) {
                    const float4 v = __ldcg(jscr + ((size_t)fr * NP * 2 + q) * NS + k);
                    Yf[4 * k] += v.x; Yf[4 * k + 1] += v.y; Yf[4 * k + 2] += v.z; Yf[4 * k + 3] += v.w;
                  }
                }
                float* J = jac + (size_t)fr * D * D;
#pragma unroll
                for (int ja = 0, p = 0; ja < D; ++ja)
#pragma unroll
                  for (int jb = ja; jb < D; ++jb, ++p) {
                    const float v = ja == jb ? fmaf(2.f * s2, Yf[p], 2.f * a.kappa) : (2.f * s2) * Yf[p];
                    J[ja * D + jb] = v;
                    J[jb * D + ja] = v;
                  }
              }
            }
          }
        }
        if (tid == 0) *cp = 0u;                               // leave the counter ready for the next launch
      }
    }
  } else if (warp_u < 16) {
    // =========================== generator warps: A tiles for every stage ===========================
    // thread = (16-byte chunk c of 4 consecutive k, base row rb): it writes its chunk of rows rb, rb+32, rb+64, rb+96 of
    // BOTH K-blocks of a stage; the two groups (warps 8-11 / 12-15) take alternate stages, so each has two stage-times
    // per stage and pays one proxy fence + one barrier arrival per 32 generated elements.
    const int t2 = tid - 256, kh = t2 >> 7, c = t2 & 3, rb = (t2 >> 2) & 31;
    const uint32_t goff = (uint32_t)rb * 64u + ((uint32_t)(c ^ ((rb >> 1) & 3)) << 4);
    uint32_t stg = 0;                                          // stages since kernel start (same sequence in every role)
    int n2 = 0;                                                // GEMM2 units seen (mask buffer parity)
    bool prefetched = false;
    auto stage_ptr = [&](uint32_t sg) { return stages + (sg % S) * C::kStageBytes + goff; };
    auto wait_stage = [&](uint32_t sg) { mbar_wait(empty0 + 8 * (sg % S), ((sg / S) & 1) ^ 1); };
    auto publish = [&](uint32_t sg) {
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(lead_full0 + 8 * (sg % S));
    };
    auto load_masks = [&](int tile, int mb) {                  // 128 rows x Hq/32 words -> maskbuf[mb] (cp.async, 16 B chunks)
      const int cpr = Hq / 128;                                // 16-byte chunks per row
      uint32_t* dst0 = maskbuf + mb * (k3Rows * k3MaskStride);
      for (int id = t2; id < k3Rows * cpr; id += 256) {
        const int r = id / cpr, ch = id - r * cpr;
        const int gr = tile * 256 + (int)rank * k3Rows + r;
        uint32_t* dst = dst0 + r * k3MaskStride + ch * 4;
        if (gr < a.mask_rows && ch * 4 < a.mask_stride) cp_async16(dst, a.maskg + (size_t)gr * a.mask_stride + ch * 4);
        else *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
      }
      cp_async_commit();
    };
    const int NST = NKB / KPS;                                 // full stages per unit
    for (int u = cid; u < U; u += G) {
      const Unit un = decode_unit(u, T, NP);
      const int m0 = un.t * 256 + (int)rank * k3Rows;
      if (!un.g) {
        // ---------------- GEMM1: x1 = leaky(A0 z + b0)^2, then the lin block (z hi/lo, 1, 1) ----------------
        float z4[4][D];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int j = 0; j < D; ++j) z4[r][j] = (m0 + rb + 32 * r < a.B) ? a.z[(size_t)(m0 + rb + 32 * r) * D + j] : 0.f;
        float2 zp[2][D];
#pragma unroll
        for (int pr = 0; pr < 2; ++pr)
#pragma unroll
          for (int j = 0; j < D; ++j) zp[pr][j] = make_float2(z4[2 * pr][j], z4[2 * pr + 1][j]);
        if constexpr (F16) {
          // FP16 hi/lo operands: thread = 16-byte chunk c (8 consecutive k) of rows rb + 32r, both K-blocks of its stages.
          // h0 is scaled per row by a power of two (exact): x1 t^2 < 2^14
          float2 tq[2];
#pragma unroll
          for (int pr = 0; pr < 2; ++pr) {
            float t0, t1, iv;
            row_scale_x1<D>(z4[2 * pr], amax, t0, iv);
            row_scale_x1<D>(z4[2 * pr + 1], amax, t1, iv);
            tq[pr] = make_float2(t0, t1);
#pragma unroll
            for (int j = 0; j < D; ++j) zp[pr][j] = __fmul2_rn(zp[pr][j], tq[pr]);
          }
          for (int st = (int)((stg ^ (uint32_t)kh) & 1u); st < NST; st += 2) {
            uint4 hi[4], lo[4];
            {
              float x[4][8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const float4 q = A0gs[st * KBE + e * 4 + c];
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                  float2 h = __ffma2_rn(make_float2(q.x, q.x), zp[pr][0], __fmul2_rn(make_float2(q.w, q.w), tq[pr]));
                  if (D > 1) h = __ffma2_rn(make_float2(q.y, q.y), zp[pr][D > 1 ? 1 : 0], h);
                  if (D > 2) h = __ffma2_rn(make_float2(q.z, q.z), zp[pr][D > 2 ? 2 : 0], h);
                  const float2 l = __fmul2_rn(h, make_float2(kSlope, kSlope));
                  const float2 a0 = make_float2(fmaxf(h.x, l.x), fmaxf(h.y, l.y));
                  const float2 xx = __fmul2_rn(a0, a0);
                  x[2 * pr][e] = xx.x; x[2 * pr + 1][e] = xx.y;
                }
              }
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                split_f16(x[r][0], x[r][1], hi[r].x, lo[r].x);
                split_f16(x[r][2], x[r][3], hi[r].y, lo[r].y);
                split_f16(x[r][4], x[r][5], hi[r].z, lo[r].z);
                split_f16(x[r][6], x[r][7], hi[r].w, lo[r].w);
              }
            }
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              *reinterpret_cast<uint4*>(At + r * 2048) = hi[r];
              *reinterpret_cast<uint4*>(At + C::kOffAlo + r * 2048) = lo[r];
            }
            publish(stg + st);
          }
          stg += NST;
        } else {
          int st = (int)((stg ^ (uint32_t)kh) & 1u);           // my first stage of this unit
          for (; st < NST; st += 2) {
            float v[2][4][4];
#pragma unroll
            for (int sub = 0; sub < 2; ++sub)
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float4 q = A0gs[(2 * st + sub) * kKB + e * 4 + c];
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                  float2 h = __ffma2_rn(make_float2(q.x, q.x), zp[pr][0], make_float2(q.w, q.w));
                  if (D > 1) h = __ffma2_rn(make_float2(q.y, q.y), zp[pr][D > 1 ? 1 : 0], h);
                  if (D > 2) h = __ffma2_rn(make_float2(q.z, q.z), zp[pr][D > 2 ? 2 : 0], h);
                  const float2 l = __fmul2_rn(h, make_float2(kSlope, kSlope));
                  const float2 a0 = make_float2(fmaxf(h.x, l.x), fmaxf(h.y, l.y));
                  const float2 x = __fmul2_rn(a0, a0);
                  v[sub][2 * pr][e] = x.x; v[sub][2 * pr + 1][e] = x.y;
                }
              }
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int sub = 0; sub < 2; ++sub)
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                unsigned char* dst = At + sub * C::kSubBytes + r * 2048;
                if (X3) {
                  const float4 hi = make_float4(rn_tf32_masked(v[sub][r][0]), rn_tf32_masked(v[sub][r][1]),
                                                rn_tf32_masked(v[sub][r][2]), rn_tf32_masked(v[sub][r][3]));
                  *reinterpret_cast<float4*>(dst) = hi;
                  *reinterpret_cast<float4*>(dst + C::kOffAlo) =
                      make_float4(rn_tf32_fast(v[sub][r][0] - hi.x), rn_tf32_fast(v[sub][r][1] - hi.y),
                                  rn_tf32_fast(v[sub][r][2] - hi.z), rn_tf32_fast(v[sub][r][3] - hi.w));
                } else {
                  *reinterpret_cast<float4*>(dst) = make_float4(rn_tf32_fast(v[sub][r][0]), rn_tf32_fast(v[sub][r][1]),
                                                                rn_tf32_fast(v[sub][r][2]), rn_tf32_fast(v[sub][r][3]));
                }
              }
            publish(stg + st);
          }
          if (st == NST) {
            // last stage of the unit: the lin block in K-block 0; K-block 1 is a dummy the MMA warp skips
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              float col[16];
#pragma unroll
              for (int m = 0; m < 16; ++m) col[m] = 0.f;
#pragma unroll
              for (int j = 0; j < D; ++j) {
                const float zh = rn_tf32_masked(z4[r][j]);
                col[3 * j] = zh; col[3 * j + 1] = rn_tf32_masked(z4[r][j] - zh); col[3 * j + 2] = zh;
              }
              col[3 * D] = 1.f; col[3 * D + 1] = 1.f;
#pragma unroll
              for (int cc = 0; cc < 4; ++cc)
                if (cc == c) {
                  *reinterpret_cast<float4*>(At + r * 2048) = make_float4(col[4 * cc], col[4 * cc + 1], col[4 * cc + 2], col[4 * cc + 3]);
                  if (X3) *reinterpret_cast<float4*>(At + C::kOffAlo + r * 2048) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            publish(stg + st);
          }
          stg += NST + 1;
        }
      } else {
        // ---------------- GEMM2: A = 1 + 4*bit (LeakyReLU slope / 0.2), exact in tf32 ----------------
        const int mb = n2 & 1;
        ++n2;
        if (!prefetched) {
          if (t2 == 0) {
            const uint32_t* cp = a.cnt + (un.t * 2 + (int)rank);
            while (ld_acquire_u32(cp) < (uint32_t)NP) {}       // all GEMM1 passes of this tile have published their bits
          }
          bar_gen();
          load_masks(un.t, mb);
        }
        cp_async_wait_all();
        if (t2 == 0) {                                         // can the next unit's bits be fetched while this one runs?
          int ok = 0;
          if (u + G < U) {
            const Unit nx = decode_unit(u + G, T, NP);
            ok = (nx.g && ld_acquire_u32(a.cnt + (nx.t * 2 + (int)rank)) >= (uint32_t)NP) ? 1 : 0;
          }
          flags[1] = ok;
        }
        bar_gen();                                             // masks of this unit visible; flags[1] valid
        prefetched = flags[1] != 0;
        if (prefetched) load_masks(decode_unit(u + G, T, NP).t, mb ^ 1);
        const uint32_t* mrow = maskbuf + mb * (k3Rows * k3MaskStride) + rb * k3MaskStride;
        for (int st = (int)((stg ^ (uint32_t)kh) & 1u); st < NST; st += 2) {
          if constexpr (F16) {
            uint4 pat[4];                                      // word st of my 4 rows = K-block st (32 bits), my byte c of it
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const uint32_t w = mrow[r * 32 * k3MaskStride + st] >> (c * 8);
              pat[r] = make_uint4(pat2_f16(w), pat2_f16(w >> 2), pat2_f16(w >> 4), pat2_f16(w >> 6));
            }
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int r = 0; r < 4; ++r) *reinterpret_cast<uint4*>(At + r * 2048) = pat[r];
          } else {
            uint32_t w4[4];                                    // word st of my 4 rows: bits of K-blocks 2st (low half), 2st+1
#pragma unroll
            for (int r = 0; r < 4; ++r) w4[r] = mrow[r * 32 * k3MaskStride + st] >> (c * 4);
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int sub = 0; sub < 2; ++sub)
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                const uint32_t w = w4[r] >> (16 * sub);
                *reinterpret_cast<float4*>(At + sub * C::kSubBytes + r * 2048) =
                    make_float4((w & 1u) ? 5.f : 1.f, (w & 2u) ? 5.f : 1.f, (w & 4u) ? 5.f : 1.f, (w & 8u) ? 5.f : 1.f);
              }
          }
          publish(stg + st);
        }
        stg += NST;
        bar_gen();                                             // everybody is done with maskbuf[mb] before it is refilled
      }
    }
    cp_async_wait_all();
  } else if (warp_u == 16) {
    // =========================== TMA producer: this CTA's half of every B tile ===========================
    // The whole warp walks the loop converged (warp-uniform state); one elected lane issues.
    uint32_t it = 0;
    for (int u = cid; u < U; u += G) {
      const Unit un = decode_unit(u, T, NP);
      const CUtensorMap* mhi = un.g ? &a.b2hi : &a.b1hi;
      const CUtensorMap* mlo = un.g ? &a.b2lo : &a.b1lo;
      const int nreal = (un.g || F16) ? NKB : NKB + 1, npad = round_up_dev(nreal, KPS);   // FP16 mode has no lin block
      const int rowc = un.p * 256 + (int)rank * k3Rows;
      for (int kb = 0; kb < npad; kb += KPS, it += KPS) {              // one stage = KPS K-blocks
        const uint32_t s = (it / KPS) % S, ph = ((it / KPS) / S) & 1;
        mbar_wait(empty0 + 8 * s, ph ^ 1);
        if (elect_one()) {
          const uint32_t bar = lead_full0 + 8 * s;
          const uint32_t dst = smem_u32(stages + s * C::kStageBytes);
#pragma unroll
          for (int sub = 0; sub < KPS; ++sub) {
            const bool real = kb + sub < nreal;                         // (the block after a lin block is a dummy)
            if (rank == 0) {                                            // expect both CTAs' halves of the K-block
              if (real) mbar_arrive_expect_tx(full0 + 8 * s, 2 * (X3 ? 2 : 1) * k3TileBytes);
              else mbar_arrive(full0 + 8 * s);
            }
            if (real) {
              tma_load_2d_pair(dst + sub * C::kSubBytes + C::kOffB, mhi, bar, (kb + sub) * KBE, rowc);
              if (X3) tma_load_2d_pair(dst + sub * C::kSubBytes + C::kOffBlo, mlo, bar, (kb + sub) * KBE, rowc);
            }
          }
        }
        __syncwarp();
      }
    }
  } else if (rank == 0) {
    // =========================== MMA issuer (leader CTA only) ===========================
    // Converged warp, one elected lane issues.  Descriptors advance by constants: +2 (32 B) per K=8 step,
    // +kSubBytes/16 per K-block, +kStageBytes/16 per stage.
    const uint64_t descA0 = make_desc_sw64(smem_u32(stages));
    const int NC = X3 ? a.NC : 1, kb_per_chunk = NKB / NC;                       // chunks of whole stages
    uint32_t it = 0;
    int i = 0;
    for (int u = cid; u < U; u += G) {
      const Unit un = decode_unit(u, T, NP);
      const int nreal = (un.g || F16) ? NKB : NKB + 1, npad = round_up_dev(nreal, KPS);
      int kb = 0;
      const int nck = un.g ? 1 : NC;                                    // GEMM1 units only (see the epilogue warps)
      for (int ck = 0; ck < nck; ++ck, ++i) {                           // one accumulator per K-chunk
        const int buf = i & 1;
        const int kb0 = kb, kb1 = (ck == nck - 1) ? npad : kb + kb_per_chunk;
        mbar_wait(accempty0 + 8 * buf, ((i >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_t = tmem_base + (uint32_t)(buf * 256);
        for (; kb < kb1; kb += KPS, it += KPS) {
          const uint32_t s = (it / KPS) % S, ph = ((it / KPS) / S) & 1;
          mbar_wait(full0 + 8 * s, ph);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t a0 = descA0 + (uint64_t)(s * (C::kStageBytes >> 4));
#pragma unroll
            for (int sub = 0; sub < KPS; ++sub) {
              if (kb + sub >= nreal) break;                             // dummy block of a GEMM1 unit
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) {
                const uint64_t a_hi = a0 + (uint64_t)(sub * (C::kSubBytes >> 4) + ks * 2);
                const uint64_t b_hi = a_hi + (uint64_t)(C::kOffB >> 4);
                const uint32_t acc = ((kb - kb0) | sub | ks) ? 1u : 0u;
                if (X3) {
                  const uint64_t b_lo = a_hi + (uint64_t)(C::kOffBlo >> 4);
                  if (!un.g) {                                          // GEMM2's A operand is exact: no a_lo term
                    umma_pair<F16>(d_t, a_hi + (uint64_t)(C::kOffAlo >> 4), b_hi, acc);
                    umma_pair<F16>(d_t, a_hi, b_lo, 1u);
                  } else {
                    umma_pair<F16>(d_t, a_hi, b_lo, acc);
                  }
                  umma_pair<F16>(d_t, a_hi, b_hi, 1u);
                } else {
                  umma_pair<F16>(d_t, a_hi, b_hi, acc);
                }
              }
            }
            umma_commit_pair(empty0 + 8 * s);                           // frees the stage in both CTAs
            if (kb + KPS >= kb1) umma_commit_pair(accfull0 + 8 * buf);  // chunk complete
          }
          __syncwarp();
        }
      }
    }
  }
  // teardown: nobody may leave (or free TMEM) while the peer can still touch this CTA's smem / TMEM
  tc_fence_before();
  __syncthreads();
  cluster_sync3();
  if (warp == 16) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

template <int D, int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(k3Threads, 1)
icnn_tc3_fwd_kernel(const __grid_constant__ Tc3Args a) {
  tc3_fwd_body<D, MODE, false>(a, nullptr, nullptr);
}

template <int D, int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(k3Threads, 1)
icnn_tc3_fwd_jac_kernel(const __grid_constant__ Tc3Args a, float4* __restrict__ jscr, float* __restrict__ jac) {
  tc3_fwd_body<D, MODE, true>(a, jscr, jac);
}

// =====================================================================================================
// Backward (double-backward of the Brenier map), sample-stationary part, same persistent pair framework.
//   A-units: acc = (1 + 4 bit) . B2g  (= gx1 / s2, the forward's GEMM2 recomputed from the saved mask bits)
//            epilogue: t0, g0 -> row-local dz partials; column sums dA0w_j = sum_b (g0 v_j + t0 z_j), db0 = sum_b t0
//   B-units: w1 = A1 v + P q1  (q1 = 2 (A0 v) a0 s0 generated; A1 v rides in the lin K-block with v instead of z)
//            epilogue: column sums dP1 = sum_b s2 s1 w1, dA1w_j = P1 sum_b s2 s1 v_j
// All units are independent.  The epilogue reads TMEM with the 16x256b shape: a thread then owns 4 rows x 8 columns
// of every 32-column chunk, so per-column parameters are loaded once per 4 rows and a column sum needs 3 in-thread
// adds plus a 3-step transposing shuffle reduction over the 8 lanes that share the columns (instead of 5 steps over
// 32 lanes).  Column partials go to ordered slots part[(tile*8 + rank*4 + quarter)][f][Hq] (summed in fixed order by
// tc_finalize_small_kernel); dz partials per (row, pass, column half) are combined by tc3_bwd_dz_kernel.
struct alignas(64) Tc3BwdArgs {
  CUtensorMap b1hi, b1lo, b2hi, b2lo;
  const float *z, *v;
  const uint32_t* mask1;
  const uint8_t* mask2;
  const float4 *A0g, *E1, *A0q;
  const float4* A1q;                              // FP16 mode: (A1w, A1b) per unit, read from global memory by the B-part
  const float* sumV;                              // FP16 mode: scale constants (see Tc3Args)
  float *partA, *partB;
  float4* dzpart;
  const float* accsave;                           // SV kernels: the forward's GEMM2 accumulators [T*256][Hq]
  int B, Hq, T, NP, Hw_in;
};

__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
// vals[c*NF + f] (c = 0..7 column slots) summed over the 8 lanes with equal (lane & 3): afterwards vals[0..NF) of a
// lane hold the sums for column slot (lane >> 2) & 7.  NV = 8*NF values, 7*NF shuffles.
template <int NV>
__device__ __forceinline__ void fold8(float (&vals)[NV], int lane) {
#pragma unroll
  for (int step = 0; step < 3; ++step) {
    const int off = 16 >> step, n = NV >> step, half = n / 2;
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = up ? vals[i] : vals[i + half];
      const float keep = up ? vals[i + half] : vals[i];
      vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
}

// SV ("saved") variant: the forward kept its GEMM2 accumulators (Tc3Args::accsave), so the A-units need no tensor work at
// all.  The unit list is then the B-units only; for each one the epilogue warps FIRST do the A-part of the same
// (tile, pass) from global memory -- while the B-unit's MMAs are in flight -- and then drain the B accumulator.  At 3xTF32
// the kernel is tensor bound, so dropping 2 of the 5 MMAs per element pair shortens it by ~40 %; HBM is idle anyway.
template <int D, int MODE, bool SV>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(k3Threads, 1)
icnn_tc3_bwd_kernel(const __grid_constant__ Tc3BwdArgs a) {
  using C = Tc3Cfg<MODE>;
  constexpr int S = C::S;
  constexpr bool X3 = C::HL, F16 = C::F16;
  constexpr int KBE = C::KBE, KPS = C::KPS;
  constexpr int NF = D + 1;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* stages = smem;
  const int Hq = a.Hq;
  float4* A0gs = reinterpret_cast<float4*>(smem + S * C::kStageBytes);     // generator order
  float4* E1s = A0gs + Hq;
  float4* A0qs = E1s + Hq;
  uint32_t* maskbuf = reinterpret_cast<uint32_t*>(A0qs + Hq);              // [2][128][36]
  uint64_t* bars = reinterpret_cast<uint64_t*>(maskbuf + 2 * k3Rows * k3MaskStride);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 4);
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + S), accfull0 = smem_u32(bars + 2 * S),
                 accempty0 = smem_u32(bars + 2 * S + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
  const uint32_t rank = cluster_rank3();
  const int cid = (int)cluster_id3(), G = (int)num_clusters3();
  const int T = a.T, NP = a.NP, NKB = Hq / KBE;
  const int U = (SV ? 1 : 2) * T * NP;
  const float inv_s1 = F16 ? a.sumV[17] : 1.f, inv_s2 = F16 ? a.sumV[19] : 1.f;
  const float4 amax = F16 ? make_float4(a.sumV[24], a.sumV[25], a.sumV[26], a.sumV[27]) : make_float4(0.f, 0.f, 0.f, 0.f);
  auto unit_of = [&](int u) {
    if (SV) { Unit x; x.g = 1; x.t = u / NP; x.p = u - x.t * NP; return x; }
    return decode_unit(u, T, NP);
  };

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full0 + 8 * s, 8 + C::KPS); mbar_init(empty0 + 8 * s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(accfull0 + 8 * b, 1); mbar_init(accempty0 + 8 * b, 16); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 16) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
  }
  for (int i = tid; i < Hq; i += k3Threads) { A0gs[i] = a.A0g[i]; E1s[i] = a.E1[i]; A0qs[i] = a.A0q[i]; }
  tc_fence_before();
  __syncthreads();
  cluster_sync3();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lead_full0 = mapa3(full0, 0), lead_accempty0 = mapa3(accempty0, 0);

  if (warp_u < 8) {
    // =========================== epilogue warps ===========================
    // warp -> TMEM lane quarter q (32 rows) and column half; lane -> rows (lane>>2) + 8r, columns 8n + 2(lane&3) + e
    const int q4 = warp & 3, chalf = warp >> 2;
    const int r0 = q4 * 32 + (lane >> 2), cp2 = 2 * (lane & 3);
    const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(chalf * 128);
    int i = 0;
    for (int u = cid; u < U; u += G, ++i) {
      const Unit un = unit_of(u);
      const int buf = i & 1;
      const int m0 = un.t * 256 + (int)rank * k3Rows;
      float zr[4][D], vr[4][D], s2r[4];
      uint4 mw[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int gr = m0 + r0 + 8 * r;
        const bool in = gr < a.B;
#pragma unroll
        for (int j = 0; j < D; ++j) {
          zr[r][j] = in ? a.z[(size_t)gr * D + j] : 0.f;
          vr[r][j] = in ? a.v[(size_t)gr * D + j] : 0.f;
        }
        s2r[r] = in ? (a.mask2[gr] ? 1.f : kSlope) : 0.f;      // 0 kills every term of padded rows
        const int w0 = un.p * 8 + chalf * 4;
        mw[r] = (un.g && in && w0 < a.Hw_in) ? *reinterpret_cast<const uint4*>(a.mask1 + (size_t)gr * a.Hw_in + w0)
                                              : make_uint4(0u, 0u, 0u, 0u);
      }
      float qinv[4] = {1.f, 1.f, 1.f, 1.f};                    // FP16 mode, B-part: P q1 = acc * qinv (row and tensor scales)
      if (F16 && un.g) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          float t_r, iv;
          row_scale_q1<D>(zr[r], vr[r], amax, t_r, iv);
          qinv[r] = iv * inv_s1;
        }
      }
      // one part of the unit: isB = B-unit maths (w1 column sums) else A-unit maths (t0, g0, dz);  from_global = the
      // accumulator comes from the forward's saved GEMM2 output instead of TMEM (SV kernels, A-part only)
      // the per-element maths runs on packed f32x2 instructions over ROW PAIRS (rows r0 + 8r, r = (0,1) and (2,3): the two halves
      // of ra / rb): the kernel is issue bound (60 % of the issue slots at 73 % tensor activity), and packing halves the
      // floating-point instructions of the epilogue
      float2 zp[2][D], vp[2][D], s2p[2], qinvp[2];
#pragma unroll
      for (int pr = 0; pr < 2; ++pr) {
#pragma unroll
        for (int j = 0; j < D; ++j) {
          zp[pr][j] = make_float2(zr[2 * pr][j], zr[2 * pr + 1][j]);
          vp[pr][j] = make_float2(vr[2 * pr][j], vr[2 * pr + 1][j]);
        }
        s2p[pr] = make_float2(s2r[2 * pr], s2r[2 * pr + 1]);
        qinvp[pr] = make_float2(qinv[2 * pr], qinv[2 * pr + 1]);
      }
      auto do_part = [&](const bool isB, const bool from_global) {
        float* part = (isB ? a.partB : a.partA) + (size_t)((un.t * 8 + (int)rank * 4 + q4) * NF) * Hq;
        float2 dzp[2][D];
#pragma unroll
        for (int pr = 0; pr < 2; ++pr)
#pragma unroll
          for (int j = 0; j < D; ++j) dzp[pr][j] = make_float2(0.f, 0.f);
        float2 s2x2p[2];                                       // 2 s2 (and the tensor scale of B2g when the accumulator is raw)
#pragma unroll
        for (int pr = 0; pr < 2; ++pr) {
          const float k2 = (F16 && !from_global) ? 2.f * inv_s2 : 2.f;
          s2x2p[pr] = __fmul2_rn(s2p[pr], make_float2(k2, k2));
        }
        if (!from_global) {
          mbar_wait_parked(accfull0 + 8 * buf, (i >> 1) & 1, k3ParkNs);
          tc_fence_after();
        }
#pragma unroll 1
        for (int cc = 0; cc < 4; ++cc) {
          uint32_t ra[16], rb[16];
          const int nb = un.p * 256 + chalf * 128 + cc * 32;
          if (from_global) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const float* src = a.accsave + k3_save_block(un.t, (int)rank, NP, un.p, chalf, cc) + (size_t)cp2 * k3Rows + r0 + 8 * r;
#pragma unroll
              for (int n = 0; n < 4; ++n) {
                (r < 2 ? ra : rb)[4 * n + 2 * (r & 1)] = __float_as_uint(__ldcs(src + (8 * n) * k3Rows));
                (r < 2 ? ra : rb)[4 * n + 2 * (r & 1) + 1] = __float_as_uint(__ldcs(src + (8 * n + 1) * k3Rows));
              }
            }
          } else {
            tmem_ld_16x256b_x4(taddr + buf * 256 + cc * 32, ra);
            tmem_ld_16x256b_x4(taddr + (16u << 16) + buf * 256 + cc * 32, rb);
            tmem_ld_wait();
          }
          float vals[8 * NF];
          uint32_t wsh[4];                                         // my rows' mask words of this chunk, my column pair at bit 0
#pragma unroll
          for (int r = 0; r < 4; ++r)
            wsh[r] = (cc == 0 ? mw[r].x : (cc == 1 ? mw[r].y : (cc == 2 ? mw[r].z : mw[r].w))) >> cp2;
          if (!isB) {
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const float4 q = A0qs[nb + 8 * n + cp2 + e];
                float2 ef[NF];
#pragma unroll
                for (int f = 0; f < NF; ++f) ef[f] = make_float2(0.f, 0.f);
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                  const uint32_t* rr = pr ? rb : ra;
                  const float2 acc = make_float2(__uint_as_float(rr[4 * n + e]), __uint_as_float(rr[4 * n + 2 + e]));
                  float2 h0 = __ffma2_rn(make_float2(q.x, q.x), zp[pr][0], make_float2(q.w, q.w));
                  float2 u0 = __fmul2_rn(make_float2(q.x, q.x), vp[pr][0]);
                  if (D > 1) {
                    h0 = __ffma2_rn(make_float2(q.y, q.y), zp[pr][D > 1 ? 1 : 0], h0);
                    u0 = __ffma2_rn(make_float2(q.y, q.y), vp[pr][D > 1 ? 1 : 0], u0);
                  }
                  if (D > 2) {
                    h0 = __ffma2_rn(make_float2(q.z, q.z), zp[pr][D > 2 ? 2 : 0], h0);
                    u0 = __ffma2_rn(make_float2(q.z, q.z), vp[pr][D > 2 ? 2 : 0], u0);
                  }
                  const float2 s0sq = make_float2(h0.x > 0.f ? 1.f : kSlope * kSlope, h0.y > 0.f ? 1.f : kSlope * kSlope);
                  const float2 mc = __fmul2_rn(__fmul2_rn(acc, s2x2p[pr]), s0sq);         // 2 s2 s0^2 acc
                  const float2 t0 = __fmul2_rn(mc, u0);                                   // u0 2 gx1 s0^2
#pragma unroll
                  for (int j = 0; j < D; ++j) {
                    const float qj = comp(q, j);
                    dzp[pr][j] = __ffma2_rn(make_float2(qj, qj), t0, dzp[pr][j]);
                    ef[j] = __ffma2_rn(mc, __ffma2_rn(h0, vp[pr][j], __fmul2_rn(u0, zp[pr][j])), ef[j]);   // g0 v_j + t0 z_j
                  }
                  ef[D] = __fadd2_rn(ef[D], t0);
                }
#pragma unroll
                for (int f = 0; f < NF; ++f) vals[(2 * n + e) * NF + f] = ef[f].x + ef[f].y;
              }
          } else {
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const uint32_t bit = 1u << (8 * n + e);                    // (shifted by cp2 below: cp2 is a run-time lane value)
                float2 ef[NF];
#pragma unroll
                for (int f = 0; f < NF; ++f) ef[f] = make_float2(0.f, 0.f);
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                  const uint32_t* rr = pr ? rb : ra;
                  const float2 w1 = make_float2(__uint_as_float(rr[4 * n + e]), __uint_as_float(rr[4 * n + 2 + e]));
                  const float2 c1 = make_float2((wsh[2 * pr] & bit) ? s2p[pr].x : kSlope * s2p[pr].x,
                                                (wsh[2 * pr + 1] & bit) ? s2p[pr].y : kSlope * s2p[pr].y);   // s2 s1
#pragma unroll
                  for (int j = 0; j < D; ++j) ef[j] = __ffma2_rn(c1, vp[pr][j], ef[j]);
                  // FP16 mode: the accumulator holds P q1 only (scaled); the A1 v part of w1 is added after the fold
                  ef[D] = __ffma2_rn(F16 ? __fmul2_rn(c1, qinvp[pr]) : c1, w1, ef[D]);
                }
#pragma unroll
                for (int f = 0; f < NF; ++f) vals[(2 * n + e) * NF + f] = ef[f].x + ef[f].y;
              }
          }
          fold8<8 * NF>(vals, lane);
          const int cs = (lane >> 2) & 7;                          // my column slot after the fold
          const int col = nb + 8 * (cs >> 1) + cp2 + (cs & 1);
          const float p1 = isB ? E1s[col].x : 1.f;                 // dA1w carries P1 (g1 = s2 P1 s1)
          if (F16 && isB) {                                        // sum_b s2 s1 (A1 v)[col] = sum_j A1w[col][j] sum_b s2 s1 v_j
            const float4 q1w = a.A1q[col];
            vals[D] = fmaf(q1w.x, vals[0], vals[D]);
            if (D > 1) vals[D] = fmaf(q1w.y, vals[D > 1 ? 1 : 0], vals[D]);
            if (D > 2) vals[D] = fmaf(q1w.z, vals[D > 2 ? 2 : 0], vals[D]);
          }
#pragma unroll
          for (int f = 0; f < NF; ++f) part[(size_t)f * Hq + col] = (f < D) ? vals[f] * p1 : vals[f];
        }
        if (!from_global) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(lead_accempty0 + 8 * buf);
        }
        if (!isB) {
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            float o[3] = {0.f, 0.f, 0.f};
#pragma unroll
            for (int j = 0; j < D; ++j) {
              float t = (r & 1) ? dzp[r >> 1][j].y : dzp[r >> 1][j].x;
              t += __shfl_xor_sync(0xffffffffu, t, 1);
              t += __shfl_xor_sync(0xffffffffu, t, 2);
              o[j] = t;
            }
            if ((lane & 3) == 0)
              a.dzpart[((size_t)(m0 + r0 + 8 * r) * NP + un.p) * 2 + chalf] = make_float4(o[0], o[1], o[2], 0.f);
          }
        }
      };
      if (SV) {
        do_part(false, true);       // A-part from the saved accumulators, overlapping this unit's MMAs
        do_part(true, false);
      } else {
        do_part(un.g != 0, false);
      }
    }
  } else if (warp_u < 16) {
    // =========================== generator warps ===========================
    const int t2 = tid - 256, kh = t2 >> 7, c = t2 & 3, rb = (t2 >> 2) & 31;
    const uint32_t goff = (uint32_t)rb * 64u + ((uint32_t)(c ^ ((rb >> 1) & 3)) << 4);
    uint32_t stg = 0;
    int n2 = 0;
    bool prefetched = false;
    auto stage_ptr = [&](uint32_t sg) { return stages + (sg % S) * C::kStageBytes + goff; };
    auto wait_stage = [&](uint32_t sg) { mbar_wait(empty0 + 8 * (sg % S), ((sg / S) & 1) ^ 1); };
    auto publish = [&](uint32_t sg) {
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(lead_full0 + 8 * (sg % S));
    };
    auto load_masks = [&](int tile, int mb) {
      const int cpr = Hq / 128;
      uint32_t* dst0 = maskbuf + mb * (k3Rows * k3MaskStride);
      for (int id = t2; id < k3Rows * cpr; id += 256) {
        const int r = id / cpr, ch = id - r * cpr;
        const int gr = tile * 256 + (int)rank * k3Rows + r;
        uint32_t* dst = dst0 + r * k3MaskStride + ch * 4;
        if (gr < a.B && ch * 4 < a.Hw_in) cp_async16(dst, a.mask1 + (size_t)gr * a.Hw_in + ch * 4);
        else *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
      }
      cp_async_commit();
    };
    const int NST = NKB / KPS;
    for (int u = cid; u < U; u += G) {
      const Unit un = unit_of(u);
      const int m0 = un.t * 256 + (int)rank * k3Rows;
      if (!un.g) {
        // ---------------- A-units: bits -> 1 + 4*bit ----------------
        const int mb = n2 & 1;
        ++n2;
        if (!prefetched) load_masks(un.t, mb);
        cp_async_wait_all();
        bar_gen();
        prefetched = (u + G < U) && (decode_unit(u + G, T, NP).g == 0);
        if (prefetched) load_masks(decode_unit(u + G, T, NP).t, mb ^ 1);
        const uint32_t* mrow = maskbuf + mb * (k3Rows * k3MaskStride) + rb * k3MaskStride;
        for (int st = (int)((stg ^ (uint32_t)kh) & 1u); st < NST; st += 2) {
          if constexpr (F16) {
            uint4 pat[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const uint32_t w = mrow[r * 32 * k3MaskStride + st] >> (c * 8);
              pat[r] = make_uint4(pat2_f16(w), pat2_f16(w >> 2), pat2_f16(w >> 4), pat2_f16(w >> 6));
            }
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int r = 0; r < 4; ++r) *reinterpret_cast<uint4*>(At + r * 2048) = pat[r];
          } else {
            uint32_t w4[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) w4[r] = mrow[r * 32 * k3MaskStride + st] >> (c * 4);
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int sub = 0; sub < 2; ++sub)
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                const uint32_t w = w4[r] >> (16 * sub);
                *reinterpret_cast<float4*>(At + sub * C::kSubBytes + r * 2048) =
                    make_float4((w & 1u) ? 5.f : 1.f, (w & 2u) ? 5.f : 1.f, (w & 4u) ? 5.f : 1.f, (w & 8u) ? 5.f : 1.f);
              }
          }
          publish(stg + st);
        }
        stg += NST;
        bar_gen();
      } else {
        // ---------------- B-units: q1 = 2 (A0 v) a0 s0, then the lin block (v hi/lo, bias columns off) ----------------
        float z4[4][D], v4[4][D];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int j = 0; j < D; ++j) {
            const bool in = m0 + rb + 32 * r < a.B;
            z4[r][j] = in ? a.z[(size_t)(m0 + rb + 32 * r) * D + j] : 0.f;
            v4[r][j] = in ? a.v[(size_t)(m0 + rb + 32 * r) * D + j] : 0.f;
          }
        float2 zp[2][D], vp[2][D];
#pragma unroll
        for (int pr = 0; pr < 2; ++pr)
#pragma unroll
          for (int j = 0; j < D; ++j) {
            zp[pr][j] = make_float2(z4[2 * pr][j], z4[2 * pr + 1][j]);
            vp[pr][j] = make_float2(2.f * v4[2 * pr][j], 2.f * v4[2 * pr + 1][j]);
          }
        if constexpr (F16) {
          // FP16 hi/lo operands; q1 is scaled per row by a power of two (through v): |q1| t < 2^14
#pragma unroll
          for (int pr = 0; pr < 2; ++pr) {
            float t0, t1, iv;
            row_scale_q1<D>(z4[2 * pr], v4[2 * pr], amax, t0, iv);
            row_scale_q1<D>(z4[2 * pr + 1], v4[2 * pr + 1], amax, t1, iv);
#pragma unroll
            for (int j = 0; j < D; ++j) vp[pr][j] = __fmul2_rn(vp[pr][j], make_float2(t0, t1));
          }
          for (int st = (int)((stg ^ (uint32_t)kh) & 1u); st < NST; st += 2) {
            uint4 hi[4], lo[4];
            {
              float x[4][8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const float4 q = A0gs[st * KBE + e * 4 + c];
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                  float2 h = __ffma2_rn(make_float2(q.x, q.x), zp[pr][0], make_float2(q.w, q.w));
                  float2 uu = __fmul2_rn(make_float2(q.x, q.x), vp[pr][0]);
                  if (D > 1) {
                    h = __ffma2_rn(make_float2(q.y, q.y), zp[pr][D > 1 ? 1 : 0], h);
                    uu = __ffma2_rn(make_float2(q.y, q.y), vp[pr][D > 1 ? 1 : 0], uu);
                  }
                  if (D > 2) {
                    h = __ffma2_rn(make_float2(q.z, q.z), zp[pr][D > 2 ? 2 : 0], h);
                    uu = __ffma2_rn(make_float2(q.z, q.z), vp[pr][D > 2 ? 2 : 0], uu);
                  }
                  const float2 l = __fmul2_rn(h, make_float2(kSlope * kSlope, kSlope * kSlope));
                  const float2 f0 = make_float2(fmaxf(h.x, l.x), fmaxf(h.y, l.y));        // a0 s0 = h0 s0^2
                  const float2 xx = __fmul2_rn(uu, f0);
                  x[2 * pr][e] = xx.x; x[2 * pr + 1][e] = xx.y;
                }
              }
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                split_f16(x[r][0], x[r][1], hi[r].x, lo[r].x);
                split_f16(x[r][2], x[r][3], hi[r].y, lo[r].y);
                split_f16(x[r][4], x[r][5], hi[r].z, lo[r].z);
                split_f16(x[r][6], x[r][7], hi[r].w, lo[r].w);
              }
            }
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              *reinterpret_cast<uint4*>(At + r * 2048) = hi[r];
              *reinterpret_cast<uint4*>(At + C::kOffAlo + r * 2048) = lo[r];
            }
            publish(stg + st);
          }
          stg += NST;
        } else {
          int st = (int)((stg ^ (uint32_t)kh) & 1u);
          for (; st < NST; st += 2) {
            float vv[2][4][4];
#pragma unroll
            for (int sub = 0; sub < 2; ++sub)
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float4 q = A0gs[(2 * st + sub) * kKB + e * 4 + c];
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                  float2 h = __ffma2_rn(make_float2(q.x, q.x), zp[pr][0], make_float2(q.w, q.w));
                  float2 uu = __fmul2_rn(make_float2(q.x, q.x), vp[pr][0]);
                  if (D > 1) {
                    h = __ffma2_rn(make_float2(q.y, q.y), zp[pr][D > 1 ? 1 : 0], h);
                    uu = __ffma2_rn(make_float2(q.y, q.y), vp[pr][D > 1 ? 1 : 0], uu);
                  }
                  if (D > 2) {
                    h = __ffma2_rn(make_float2(q.z, q.z), zp[pr][D > 2 ? 2 : 0], h);
                    uu = __ffma2_rn(make_float2(q.z, q.z), vp[pr][D > 2 ? 2 : 0], uu);
                  }
                  const float2 l = __fmul2_rn(h, make_float2(kSlope * kSlope, kSlope * kSlope));
                  const float2 f0 = make_float2(fmaxf(h.x, l.x), fmaxf(h.y, l.y));        // a0 s0 = h0 s0^2
                  const float2 x = __fmul2_rn(uu, f0);
                  vv[sub][2 * pr][e] = x.x; vv[sub][2 * pr + 1][e] = x.y;
                }
              }
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int sub = 0; sub < 2; ++sub)
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                unsigned char* dst = At + sub * C::kSubBytes + r * 2048;
                if (X3) {
                  const float4 hi = make_float4(rn_tf32_masked(vv[sub][r][0]), rn_tf32_masked(vv[sub][r][1]),
                                                rn_tf32_masked(vv[sub][r][2]), rn_tf32_masked(vv[sub][r][3]));
                  *reinterpret_cast<float4*>(dst) = hi;
                  *reinterpret_cast<float4*>(dst + C::kOffAlo) =
                      make_float4(rn_tf32_fast(vv[sub][r][0] - hi.x), rn_tf32_fast(vv[sub][r][1] - hi.y),
                                  rn_tf32_fast(vv[sub][r][2] - hi.z), rn_tf32_fast(vv[sub][r][3] - hi.w));
                } else {
                  *reinterpret_cast<float4*>(dst) = make_float4(rn_tf32_fast(vv[sub][r][0]), rn_tf32_fast(vv[sub][r][1]),
                                                                rn_tf32_fast(vv[sub][r][2]), rn_tf32_fast(vv[sub][r][3]));
                }
              }
            publish(stg + st);
          }
          if (st == NST) {
            wait_stage(stg + st);
            unsigned char* At = stage_ptr(stg + st);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              float col[16];
#pragma unroll
              for (int m = 0; m < 16; ++m) col[m] = 0.f;
#pragma unroll
              for (int j = 0; j < D; ++j) {
                const float vh = rn_tf32_masked(v4[r][j]);
                col[3 * j] = vh; col[3 * j + 1] = rn_tf32_masked(v4[r][j] - vh); col[3 * j + 2] = vh;
              }
#pragma unroll
              for (int cc = 0; cc < 4; ++cc)
                if (cc == c) {
                  *reinterpret_cast<float4*>(At + r * 2048) = make_float4(col[4 * cc], col[4 * cc + 1], col[4 * cc + 2], col[4 * cc + 3]);
                  if (X3) *reinterpret_cast<float4*>(At + C::kOffAlo + r * 2048) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            publish(stg + st);
          }
          stg += NST + 1;
        }
      }
    }
    cp_async_wait_all();
  } else if (warp_u == 16) {
    // =========================== TMA producer ===========================
    uint32_t it = 0;
    for (int u = cid; u < U; u += G) {
      const Unit un = unit_of(u);
      const CUtensorMap* mhi = un.g ? &a.b1hi : &a.b2hi;
      const CUtensorMap* mlo = un.g ? &a.b1lo : &a.b2lo;
      const int nreal = (un.g && !F16) ? NKB + 1 : NKB, npad = round_up_dev(nreal, KPS);
      const int rowc = un.p * 256 + (int)rank * k3Rows;
      for (int kb = 0; kb < npad; kb += KPS, it += KPS) {
        const uint32_t s = (it / KPS) % S, ph = ((it / KPS) / S) & 1;
        mbar_wait(empty0 + 8 * s, ph ^ 1);
        if (elect_one()) {
          const uint32_t bar = lead_full0 + 8 * s;
          const uint32_t dst = smem_u32(stages + s * C::kStageBytes);
#pragma unroll
          for (int sub = 0; sub < KPS; ++sub) {
            const bool real = kb + sub < nreal;                         // (the block after a lin block is a dummy)
            if (rank == 0) {                                            // expect both CTAs' halves of the K-block
              if (real) mbar_arrive_expect_tx(full0 + 8 * s, 2 * (X3 ? 2 : 1) * k3TileBytes);
              else mbar_arrive(full0 + 8 * s);
            }
            if (real) {
              tma_load_2d_pair(dst + sub * C::kSubBytes + C::kOffB, mhi, bar, (kb + sub) * KBE, rowc);
              if (X3) tma_load_2d_pair(dst + sub * C::kSubBytes + C::kOffBlo, mlo, bar, (kb + sub) * KBE, rowc);
            }
          }
        }
        __syncwarp();
      }
    }
  } else if (rank == 0) {
    // =========================== MMA issuer (leader CTA only) ===========================
    const uint64_t descA0 = make_desc_sw64(smem_u32(stages));
    uint32_t it = 0;
    int i = 0;
    for (int u = cid; u < U; u += G, ++i) {
      const Unit un = unit_of(u);
      const int buf = i & 1;
      const int nreal = (un.g && !F16) ? NKB + 1 : NKB, npad = round_up_dev(nreal, KPS);
      mbar_wait(accempty0 + 8 * buf, ((i >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_t = tmem_base + (uint32_t)(buf * 256);
      for (int kb = 0; kb < npad; kb += KPS, it += KPS) {
        const uint32_t s = (it / KPS) % S, ph = ((it / KPS) / S) & 1;
        mbar_wait(full0 + 8 * s, ph);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t a0 = descA0 + (uint64_t)(s * (C::kStageBytes >> 4));
#pragma unroll
          for (int sub = 0; sub < KPS; ++sub) {
            if (kb + sub >= nreal) break;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              const uint64_t a_hi = a0 + (uint64_t)(sub * (C::kSubBytes >> 4) + ks * 2);
              const uint64_t b_hi = a_hi + (uint64_t)(C::kOffB >> 4);
              const uint32_t acc = (kb | sub | ks) ? 1u : 0u;
              if (X3) {
                const uint64_t b_lo = a_hi + (uint64_t)(C::kOffBlo >> 4);
                if (un.g) {                                             // A-units' operand is exact: no a_lo term
                  umma_pair<F16>(d_t, a_hi + (uint64_t)(C::kOffAlo >> 4), b_hi, acc);
                  umma_pair<F16>(d_t, a_hi, b_lo, 1u);
                } else {
                  umma_pair<F16>(d_t, a_hi, b_lo, acc);
                }
                umma_pair<F16>(d_t, a_hi, b_hi, 1u);
              } else {
                umma_pair<F16>(d_t, a_hi, b_hi, acc);
              }
            }
          }
          umma_commit_pair(empty0 + 8 * s);
          if (kb + KPS >= npad) umma_commit_pair(accfull0 + 8 * buf);
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync3();
  if (warp == 16) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// dz[b] = sum of the A-units' partials + 2 kappa v;  a2part[tile][j] = sum_{b in tile} s2 v_j (fixed order).  One block per
// 256-row tile.
__global__ void __launch_bounds__(256)
tc3_bwd_dz_kernel(const float4* __restrict__ dzpart, const float* __restrict__ v, const uint8_t* __restrict__ mask2, int B,
                  int NP, int d, float kappa, float* __restrict__ dz, float* __restrict__ a2part) {
  __shared__ float red[8][4];
  const int row = blockIdx.x * 256 + threadIdx.x, lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const bool in = row < B;
  float acc[3] = {0.f, 0.f, 0.f}, sv[3] = {0.f, 0.f, 0.f};
  if (in) {
    for (int q = 0; q < 2 * NP; ++q) {
      const float4 t = dzpart[(size_t)row * NP * 2 + q];
      acc[0] += t.x; acc[1] += t.y; acc[2] += t.z;
    }
    const float s2 = mask2[row] ? 1.f : kSlope;
    for (int j = 0; j < d; ++j) {
      const float vj = v[(size_t)row * d + j];
      if (dz) dz[(size_t)row * d + j] = fmaf(2.f * kappa, vj, acc[j]);
      sv[j] = s2 * vj;
    }
  }
  for (int j = 0; j < 3; ++j) {
    const float t = warp_sum(sv[j]);
    if (lane == 0) red[wp][j] = t;
  }
  __syncthreads();
  if (threadIdx.x < d) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    a2part[(size_t)blockIdx.x * d + threadIdx.x] = t;
  }
}

// one thread per hidden unit: (A0w, A0b), (A1w | P1 in the spare lane, A1b), P1 in natural unit order, zero padded to Hq
__global__ void tc_prepare_kernel(const float* __restrict__ P1, const float* __restrict__ A0p, const float* __restrict__ A1p,
                                  int d, int Hp, int Hq, float4* __restrict__ A0q, float4* __restrict__ A1q,
                                  float* __restrict__ P1q) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Hq) return;
  const bool inr = c < Hp;
  float w[4] = {0.f, 0.f, 0.f, 0.f}, u[4] = {0.f, 0.f, 0.f, 0.f};
  if (inr) {
    for (int j = 0; j < d; ++j) { w[j] = A0p[(size_t)c * (d + 1) + j]; u[j] = A1p[(size_t)c * (d + 1) + j]; }
    w[3] = A0p[(size_t)c * (d + 1) + d]; u[3] = A1p[(size_t)c * (d + 1) + d];
  }
  if (d <= 2) u[2] = inr ? P1[c] : 0.f;     // spare lane of the float4: P1 rides along
  A0q[c] = make_float4(w[0], w[1], w[2], w[3]);
  A1q[c] = make_float4(u[0], u[1], u[2], u[3]);
  P1q[c] = inr ? P1[c] : 0.f;
}

// ordered reduction of the row-kernel partials + chain through the positive reparam for W1.
// grid (Hq/32, NF, 2): one block of 1024 threads sums all `nslots` partial rows of 32 columns (32 slot lanes x 32 columns,
// coalesced 128-byte reads, fixed summation order -> deterministic).
__global__ void __launch_bounds__(1024)
tc_finalize_small_kernel(const float* __restrict__ partA, const float* __restrict__ partB,
                         const float* __restrict__ a2part, int nslots, int nmt, int d, int H, int Hq,
                         const float* __restrict__ P1, const float* __restrict__ W1raw, int mode, b200vae_icnn_grads g) {
  __shared__ float red[32][33];
  const int NF = d + 1;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + tx, f = blockIdx.y, which = blockIdx.z;
  const float* part = (which ? partB : partA) + (size_t)f * Hq + n;
  // 16 independent partial sums per thread, 32 slot lanes per block: the kernel is latency bound (2048 slots x 128-byte
  // rows per block at B = 65536), so the number of loads in flight is what sets its duration (8 slot lanes: 21 us)
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  int sl = ty;
  const size_t stride = (size_t)NF * Hq;
  for (; sl + 480 < nslots; sl += 512) {
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] += part[(size_t)(sl + 32 * i) * stride];
  }
  for (; sl < nslots; sl += 32) acc[0] += part[(size_t)sl * stride];
#pragma unroll
  for (int w = 8; w >= 1; w >>= 1)
#pragma unroll
    for (int i = 0; i < w; ++i) acc[i] += acc[i + w];
  red[ty][tx] = acc[0];
  __syncthreads();
  if (ty == 0 && n < H) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 32; ++q) s += red[q][tx];
    if (!which) {
      if (f < d) { if (g.A0w) g.A0w[(size_t)n * d + f] = s; }
      else if (g.A0b) g.A0b[n] = s;
    } else {
      if (f < d) { if (g.A1w) g.A1w[(size_t)n * d + f] = s; }
      else if (g.W1) g.W1[n] = (mode == B200VAE_WEIGHT_EXP) ? s * P1[n] : (W1raw[n] >= kClampMin ? s : 0.f);
      if (f == 0 && g.A1b) g.A1b[n] = 0.f;                   // exact zeros on the <v, xhat> path (Appendix A)
    }
  }
  if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) {
    if (threadIdx.x < d) {
      float s = 0.f;
      for (int mt = 0; mt < nmt; ++mt) s += a2part[(size_t)mt * d + threadIdx.x];
      if (g.A2w) g.A2w[threadIdx.x] = s;
    }
    if (threadIdx.x == 0 && g.A2b) g.A2b[0] = 0.f;
  }
}

// ------------------------------------------------------------------------------------ host side
// arithmetic of the pair kernels for an ABI precision id
static int tc3_mode(int precision) {
  return precision == B200VAE_PREC_F16X3 ? kF16 : precision == B200VAE_PREC_TF32X3 ? kX3 : kTf32;
}
// the per-unit tables and the pair kernels' operands, from the FP32 arrays simt_prepare wrote
int tc3_prepare(const WsLayout& L, int precision, float* ws, cudaStream_t st) {
  tc_prepare_kernel<<<(L.Hq + 255) / 256, 256, 0, st>>>(ws + L.P1, ws + L.A0p, ws + L.A1p, L.d, L.Hp, L.Hq,
                                                       reinterpret_cast<float4*>(ws + L.A0q),
                                                       reinterpret_cast<float4*>(ws + L.A1q), ws + L.P1q);
  int rc = check_launch();
  if (rc) return rc;
  const int mode = tc3_mode(precision);
  if (mode == kF16) {
    // the fp16 copies live in the (larger) fp32 operand regions: hi/lo of B1 [Hq][Hq], hi/lo of B2g [Hq][Hq]
    uint32_t* mx = reinterpret_cast<uint32_t*>(ws + L.sumV + 8);
    if (cudaMemsetAsync(mx, 0, 2 * sizeof(uint32_t), st) != cudaSuccess) return B200VAE_ECUDA;
    tc3_rowmax_kernel<<<L.Hp, 256, 0, st>>>(ws + L.P0, ws + L.P1, L.Hp, mx);
    rc = check_launch();
    if (rc) return rc;
    dim3 grid((L.Hq + 255) / 256, L.Hq);
    tc3_prepare_f16_kernel<<<grid, 256, 0, st>>>(
        ws + L.P0, ws + L.P0T, ws + L.P1, ws + L.A0p, ws + L.A1p, L.d, L.Hp, L.Hq, mx, reinterpret_cast<__half*>(ws + L.B1ahi),
        reinterpret_cast<__half*>(ws + L.B1alo), reinterpret_cast<__half*>(ws + L.B2ghi), reinterpret_cast<__half*>(ws + L.B2glo),
        reinterpret_cast<float4*>(ws + L.A0g), reinterpret_cast<float4*>(ws + L.E1), ws + L.sumV + 16);
  } else {
    dim3 grid((L.K1 + 255) / 256, L.Hq);
    tc3_prepare_kernel<<<grid, 256, 0, st>>>(ws + L.P0, ws + L.P0T, ws + L.P1, ws + L.A0p, ws + L.A1p, L.d, L.Hp, L.Hq, L.K1,
                                             mode == kX3 ? 1 : 0, ws + L.B1ahi, ws + L.B1alo, ws + L.B2ghi, ws + L.B2glo,
                                             reinterpret_cast<float4*>(ws + L.A0g), reinterpret_cast<float4*>(ws + L.E1));
  }
  rc = check_launch();
  if (rc) return rc;
  tc3_sumv_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const float4*>(ws + L.E1), reinterpret_cast<const float4*>(ws + L.A0g),
                                    L.Hq, ws + L.sumV);
  rc = check_launch();
  if (rc) return rc;
  if (cudaMemsetAsync(ws + L.cnt, 0, (size_t)2 * kTc3MaxTiles * sizeof(uint32_t), st) != cudaSuccess) return B200VAE_ECUDA;
  return B200VAE_OK;
}

struct Tc3Maps { CUtensorMap b1hi, b1lo, b2hi, b2lo; };
static int get_maps3(const float* ws, const WsLayout& L, int mode, Tc3Maps* out) {
  static std::mutex mu;
  static std::unordered_map<uint64_t, Tc3Maps> cache;       // tensor maps only encode (address, shape, element type)
  std::lock_guard<std::mutex> lk(mu);
  const uint64_t key = reinterpret_cast<uint64_t>(ws + L.B1ahi) ^ ((uint64_t)L.Hq << 48) ^ ((uint64_t)mode << 62);
  auto itc = cache.find(key);
  if (itc != cache.end()) { *out = itc->second; return B200VAE_OK; }
  Tc3Maps mp;
  const bool hl = mode != kTf32, f16 = mode == kF16;
  const int K1 = f16 ? L.Hq : L.K1;
  int rc = tma_map_2d(&mp.b1hi, ws + L.B1ahi, K1, L.Hq, K1, k3Rows, f16);
  if (!rc) rc = tma_map_2d(&mp.b1lo, ws + (hl ? L.B1alo : L.B1ahi), K1, L.Hq, K1, k3Rows, f16);
  if (!rc) rc = tma_map_2d(&mp.b2hi, ws + L.B2ghi, L.Hq, L.Hq, L.Hq, k3Rows, f16);
  if (!rc) rc = tma_map_2d(&mp.b2lo, ws + (hl ? L.B2glo : L.B2ghi), L.Hq, L.Hq, L.Hq, k3Rows, f16);
  if (rc) return rc;
  if (cache.size() > 256) cache.clear();
  cache.emplace(key, mp);
  *out = mp;
  return B200VAE_OK;
}

// =====================================================================================================
// dP0 (batch-reduced gradient of the H x H weight) on CTA pairs:  dP0part[split][o][n] = sum_{m in split} (1 + 4 bit[m,o]) s2[m] q1[m,n]
// Round 1's single-CTA kernel (since deleted) turned out to be bound by SHARED-MEMORY BYTES, not by generator
// instructions or the tensor pipe (ncu: issue 36 %, tensor 45 / 69 % active; an n-stationary single-CTA variant with fewer
// generator instructions but more generated bytes was slower): per 16-sample K-block an SM wrote 32 / 48 KB of generated
// operands and the MMAs read 48 / 96 KB (TF32 / 3xTF32) against ~730 / 1460 tensor cycles x 128 B/clk.  Here
//   * one tcgen05.mma.cta_group::2 (M = 256, N = 256, K = 8) drives both SMs: an SM reads 4 KB of A and only ITS 4 KB half
//     of B per MMA (8 KB instead of 12 KB);
//   * the EXPENSIVE operand q1 (packed FMAs, tf32 hi/lo split) is the A operand -- each SM generates it for its own 128 n's
//     only -- and the cheap exact slope pattern 1 + 4*bit is the B operand: two accumulators (all 512 TMEM columns) cover
//     512 o's, of which each SM generates 2 x 128.  Generated bytes per K-block and SM: 24 / 32 KB; MMA reads 32 / 64 KB.
// D[n][o] is written transposed by the epilogue (thread = n lane, one coalesced 128-byte store per o column).
// Both operands MN-major, SWIZZLE_128B_BASE32B atoms of 4 k-rows x 128 B; every tile is 128 MN wide: LBO 512 B, SBO 2 KB.
constexpr int kDpWarps = 16;                                   // generator / epilogue warps (+ 1 MMA / TMEM warp)
constexpr int kDpThreads3 = (kDpWarps + 1) * 32;
constexpr int kDpTile = 16 * 128 * 4;                          // 16 k x 128 MN x 4 B = 8 KB
constexpr uint32_t k3IdescMN = k3Idesc | (1u << 15) | (1u << 16);
__device__ __forceinline__ uint64_t make_desc_mn128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(512 >> 4) << 16) | ((uint64_t)(2048 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)1 << 61);           // layout type 1 = SWIZZLE_128B_BASE32B
}
__device__ __forceinline__ void umma_tf32_pair_mn(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(k3IdescMN), "r"(acc) : "memory");
}
__device__ __forceinline__ void bar_dp() { asm volatile("bar.sync 1, %0;" ::"n"(kDpWarps * 32) : "memory"); }
template <bool X3>
struct DpCfg {
  static constexpr int S = X3 ? 5 : 6;
  static constexpr int kOffQlo = kDpTile, kOffO = (X3 ? 2 : 1) * kDpTile;
  static constexpr int kStage = kOffO + 2 * kDpTile;           // 24 KB / 32 KB
};
template <int D, bool X3>
constexpr size_t dp3_smem_bytes() {
  return (size_t)DpCfg<X3>::S * DpCfg<X3>::kStage + (size_t)2 * 256 * (2 * D + 1) * 4 + 2 * 8 * 256 * 4 +
         (2 * DpCfg<X3>::S + 1) * 8 + 16 + 1024;
}

template <int D, bool X3>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kDpThreads3, 1)
icnn_tc3_dP0_kernel(const float* __restrict__ z, const float* __restrict__ v, const uint32_t* __restrict__ mask1,
                    const uint8_t* __restrict__ mask2, int B, int Hq, int Hw_in, int rows_per_split,
                    const float4* __restrict__ A0q_g, float* __restrict__ dP0part) {
  using C = DpCfg<X3>;
  constexpr int S = C::S;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* stages = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* samp = reinterpret_cast<float*>(stages + S * C::kStage);            // [2][2D+1][256]  z, v, s2 per sample
  uint32_t* sampw = reinterpret_cast<uint32_t*>(samp + 2 * 256 * (2 * D + 1));    // [2][8][256] this CTA's mask words
  uint64_t* bars = reinterpret_cast<uint64_t*>(sampw + 2 * 8 * 256);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 1);
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + S), accfull = smem_u32(bars + 2 * S);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
  const uint32_t rank = cluster_rank3();
  const int n0 = (blockIdx.x >> 1) * 256 + (int)rank * 128;  // my 128 n's (rows of D)
  const int o0 = blockIdx.y * 512, split = blockIdx.z;
  const bool two = o0 + 256 < Hq;                            // Hq is a multiple of 256: the last o-tile may be half
  const int b0 = split * rows_per_split;
  const int b1 = min(B, b0 + rows_per_split);
  const int NKB = (max(b1 - b0, 0) + kKB - 1) / kKB;

  if (tid == 0) {
    // full (leader's copy is the one in use): one arrival per generator warp of BOTH CTAs
    for (int s = 0; s < S; ++s) { mbar_init(full0 + 8 * s, 2 * kDpWarps); mbar_init(empty0 + 8 * s, 1); }
    mbar_init(accfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kDpWarps) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync3();                         // peer barriers initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lead_full0 = mapa3(full0, 0);

  if (warp_u < kDpWarps) {
    // thread -> (sample ks of the stage, 4 consecutive MN elements).  A quarter warp (8 lanes = 4 k-rows x 2 halves of one
    // 32-byte swizzle unit) stores 128 distinct bytes: conflict-free 16-byte stores (the k-groups g4 share banks, so they
    // sit in different quarters); a warp owns one 8-wide MN unit (blk, qd) for all 16 samples
    const int g4 = lane >> 3, hf = (lane >> 2) & 1, kr = lane & 3;   // group of 4 k, 4-wide half, k-row inside the atom
    const int ks = g4 * 4 + kr;
    const int blk = warp >> 2, qd = warp & 3;                // 32-wide block, 8-wide quarter (swizzle unit)
    const uint32_t off = (uint32_t)((g4 * 4 + blk) * 512 + kr * 128) + ((uint32_t)(qd ^ kr) << 5) + (uint32_t)(hf * 16);
    const int bsh = qd * 8 + hf * 4;                         // my 4 bits inside mask word `blk` (of either accumulator)
    float2 qx2[2], qy2[2], qz2[2], qw2[2];                   // my 4 n's as two packed pairs: (w0, w1, w2, bias)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int n = n0 + blk * 32 + qd * 8 + hf * 4 + 2 * i;
      const float4 qa = A0q_g[n], qb = A0q_g[n + 1];
      qx2[i] = make_float2(qa.x, qb.x); qy2[i] = make_float2(qa.y, qb.y);
      qz2[i] = make_float2(qa.z, qb.z); qw2[i] = make_float2(qa.w, qb.w);
    }
    // per-sample inputs (z, v, s2, this CTA's 8 mask words: o's [t*256 + rank*128, +128) of accumulator t = 0, 1) are staged
    // through shared memory in chunks of 256 samples, fetched one chunk ahead (register staged)
    constexpr int CH = 256, ZV = 2 * D + 1;
    const int nchunk = (NKB * kKB + CH - 1) / CH;
    float pre_f[ZV];
    uint32_t pre_w[4];
    auto fetch = [&](int c) {                                // thread -> sample (tid&255), accumulator t = tid>>8
      const int mrow = b0 + c * CH + (tid & 255);
      const bool in = mrow < b1;
      if (tid < CH) {
#pragma unroll
        for (int j = 0; j < D; ++j) {
          pre_f[j] = in ? __ldg(z + (size_t)mrow * D + j) : 0.f;
          pre_f[D + j] = in ? __ldg(v + (size_t)mrow * D + j) : 0.f;
        }
        pre_f[2 * D] = in ? (__ldg(mask2 + mrow) ? 1.f : kSlope) : 0.f;
      }
      const int w0 = (o0 >> 5) + (tid >> 8) * 8 + (int)rank * 4;
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) pre_w[q4] = (in && w0 + q4 < Hw_in) ? __ldg(mask1 + (size_t)mrow * Hw_in + w0 + q4) : 0u;
    };
    auto stash = [&](int buf) {
      float* zf = samp + buf * (CH * ZV);
      uint32_t* mw = sampw + buf * (CH * 8);
      if (tid < CH) {
#pragma unroll
        for (int j = 0; j < ZV; ++j) zf[j * CH + tid] = pre_f[j];
      }
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) mw[((tid >> 8) * 4 + q4) * CH + (tid & 255)] = pre_w[q4];
    };
    if (nchunk > 0) { fetch(0); stash(0); }
    bar_dp();
    for (int kb = 0; kb < NKB; ++kb) {
      const int c = kb >> 4, buf = c & 1, sl = (kb & 15) * kKB + ks;       // sample slot inside the chunk
      if ((kb & 15) == 0 && c + 1 < nchunk) fetch(c + 1);
      const float* zf = samp + buf * (CH * ZV);
      float zr[D], vr[D];
#pragma unroll
      for (int j = 0; j < D; ++j) { zr[j] = zf[j * CH + sl]; vr[j] = zf[(D + j) * CH + sl]; }
      const float s2f = zf[2 * D * CH + sl];
      const uint32_t bits0 = sampw[buf * (CH * 8) + blk * CH + sl] >> bsh;
      const uint32_t bits1 = sampw[buf * (CH * 8) + (4 + blk) * CH + sl] >> bsh;
      // A = s2 q1 = (2 s2 A0 v) . max(h0, 0.04 h0) for my 4 n's, two per packed instruction
      float qv[4];
      float sv[D];
#pragma unroll
      for (int j = 0; j < D; ++j) sv[j] = (2.f * s2f) * vr[j];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        float2 h = __ffma2_rn(qx2[i], make_float2(zr[0], zr[0]), qw2[i]);
        float2 uu = __fmul2_rn(qx2[i], make_float2(sv[0], sv[0]));
        if (D > 1) {
          h = __ffma2_rn(qy2[i], make_float2(zr[D > 1 ? 1 : 0], zr[D > 1 ? 1 : 0]), h);
          uu = __ffma2_rn(qy2[i], make_float2(sv[D > 1 ? 1 : 0], sv[D > 1 ? 1 : 0]), uu);
        }
        if (D > 2) {
          h = __ffma2_rn(qz2[i], make_float2(zr[D > 2 ? 2 : 0], zr[D > 2 ? 2 : 0]), h);
          uu = __ffma2_rn(qz2[i], make_float2(sv[D > 2 ? 2 : 0], sv[D > 2 ? 2 : 0]), uu);
        }
        const float2 l = __fmul2_rn(h, make_float2(kSlope * kSlope, kSlope * kSlope));
        const float2 x = __fmul2_rn(uu, make_float2(fmaxf(h.x, l.x), fmaxf(h.y, l.y)));
        qv[2 * i] = x.x; qv[2 * i + 1] = x.y;
      }
      if ((kb & 15) == 15 && c + 1 < nchunk) {               // next chunk's buffer was last read 16 stages ago
        bar_dp();
        stash(buf ^ 1);
        bar_dp();
      }
      const uint32_t s = kb % S, ph = (kb / S) & 1;
      mbar_wait(empty0 + 8 * s, ph ^ 1);
      unsigned char* st = stages + s * C::kStage + off;
      if (X3) {
        const float4 hi = make_float4(rn_tf32_masked(qv[0]), rn_tf32_masked(qv[1]), rn_tf32_masked(qv[2]), rn_tf32_masked(qv[3]));
        *reinterpret_cast<float4*>(st) = hi;
        *reinterpret_cast<float4*>(st + C::kOffQlo) =
            make_float4(rn_tf32_fast(qv[0] - hi.x), rn_tf32_fast(qv[1] - hi.y), rn_tf32_fast(qv[2] - hi.z), rn_tf32_fast(qv[3] - hi.w));
      } else {
        *reinterpret_cast<float4*>(st) =
            make_float4(rn_tf32_masked(qv[0]), rn_tf32_masked(qv[1]), rn_tf32_masked(qv[2]), rn_tf32_masked(qv[3]));
      }
      // B = 1 + 4*bit (the LeakyReLU slope / 0.2, exact in tf32; 0.2 and P1 are applied by finalize_W0)
      *reinterpret_cast<float4*>(st + C::kOffO) =
          make_float4((bits0 & 1u) ? 5.f : 1.f, (bits0 & 2u) ? 5.f : 1.f, (bits0 & 4u) ? 5.f : 1.f, (bits0 & 8u) ? 5.f : 1.f);
      *reinterpret_cast<float4*>(st + C::kOffO + kDpTile) =
          make_float4((bits1 & 1u) ? 5.f : 1.f, (bits1 & 2u) ? 5.f : 1.f, (bits1 & 4u) ? 5.f : 1.f, (bits1 & 8u) ? 5.f : 1.f);
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(lead_full0 + 8 * s);
    }
    // epilogue: TMEM lane = my n, column = o (512 of them).  Warp w: lane quadrant w & 3, the 128 columns of group w >> 2.
    const int q = warp & 3, cg = warp >> 2;
    const int n = n0 + q * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * 128);
    if (two || cg < 2) {
      float* out = dP0part + ((size_t)split * Hq + o0 + cg * 128) * Hq + n;
      if (NKB > 0) {
        mbar_wait_parked(accfull, 0, k3ParkNs);
        tc_fence_after();
#pragma unroll 1
        for (int cc = 0; cc < 4; ++cc) {
          uint32_t r[32];
          tmem_ld32(taddr + cc * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) out[(size_t)(cc * 32 + j) * Hq] = __uint_as_float(r[j]);
        }
      } else {
        for (int j = 0; j < 128; ++j) out[(size_t)j * Hq] = 0.f;
      }
    }
  } else if (rank == 0) {
    // MMA issuer (leader CTA only): whole converged warp, one elected lane issues; descriptors advance by constants
    const uint64_t desc0 = make_desc_mn128(smem_u32(stages));
    for (int kb = 0; kb < NKB; ++kb) {
      const uint32_t s = kb % S, ph = (kb / S) & 1;
      mbar_wait(full0 + 8 * s, ph);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t sa = desc0 + (uint64_t)((s * C::kStage) >> 4);
#pragma unroll
        for (int g = 0; g < 2; ++g) {                                            // K = 8 = two 4-k groups (2 x SBO)
          const uint64_t a_hi = sa + (uint64_t)((g * 4096) >> 4);
          const uint32_t acc = (kb | g) ? 1u : 0u;
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            if (t == 1 && !two) break;
            const uint32_t d_t = tmem_base + (uint32_t)(t * 256);
            const uint64_t b = sa + (uint64_t)((C::kOffO + t * kDpTile + g * 4096) >> 4);
            if (X3) {                                                            // B is exact: a_lo.b + a_hi.b
              umma_tf32_pair_mn(d_t, a_hi + (uint64_t)(C::kOffQlo >> 4), b, acc);
              umma_tf32_pair_mn(d_t, a_hi, b, 1u);
            } else {
              umma_tf32_pair_mn(d_t, a_hi, b, acc);
            }
          }
        }
        umma_commit_pair(empty0 + 8 * s);                                        // frees the stage in both CTAs
        if (kb == NKB - 1) umma_commit_pair(accfull);
      }
      __syncwarp();
    }
  }
  // teardown: nobody may leave (or free TMEM) while the peer can still touch this CTA's smem / TMEM
  tc_fence_before();
  __syncthreads();
  cluster_sync3();
  if (warp == kDpWarps) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// ---- dP0 in the FP16 mode ----------------------------------------------------------------------------------------------
// Same CTA-pair scheme on kind::f16 MMAs (M = 256, N = 256, K = 16): the expensive operand s2 q1 as an FP16 hi/lo pair (two
// MMAs per accumulator and K step: half the tensor time of the 3xTF32 instantiation, whose tensor pipe is 95 % busy), the slope
// pattern 1 | 5 exact in fp16.  FP16 range: the samples are the K dimension here, so a per-sample scale could not be undone
// after the sum; instead every CTA first scans ITS samples for the largest bound of |s2 q1| (the bound of row_scale_q1) and
// scales the whole operand by ONE power of two G (exact), |s2 q1| G < 2^14, undone in the epilogue.  A sample far below the
// split's maximum keeps an absolute error of 2^-25 / G -- 2^-39 of the largest element, nothing against the fp32 rounding of
// the sum.  Both CTAs of a pair scan the same samples, so they agree on G.
// 16-bit MN-major operands: SWIZZLE_128B atoms of 8 k-rows x 128 B (64 MN elements), the 16-byte chunks of a row XOR-ed with
// the k-row; a tile is 128 MN wide: LBO = 1 KB between the two atoms, SBO = 2 KB between groups of 8 k.  A stage holds 32
// samples (two K = 16 steps): A hi, A lo, B (accumulator 0), B (accumulator 1), 8 KB each.
constexpr int kDpTile16 = 32 * 128 * 2;                        // 32 k x 128 MN x 2 B = 8 KB
constexpr int kDpStage16 = 4 * kDpTile16;
constexpr int kDpS16 = 5;
constexpr uint32_t k3IdescF16MN = k3IdescF16 | (1u << 15) | (1u << 16);
__device__ __forceinline__ uint64_t make_desc_mn128_b16(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(1024 >> 4) << 16) | ((uint64_t)(2048 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);           // layout type 2 = SWIZZLE_128B
}
__device__ __forceinline__ void umma_f16_pair_mn(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(k3IdescF16MN), "r"(acc) : "memory");
}
template <int D>
constexpr size_t dp3_f16_smem_bytes() {
  return (size_t)kDpS16 * kDpStage16 + (size_t)2 * 256 * (2 * D + 1) * 4 + 2 * 8 * 256 * 4 + (2 * kDpS16 + 1) * 8 + 16 + 64 + 1024;
}

template <int D>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kDpThreads3, 1)
icnn_tc3_dP0_f16_kernel(const float* __restrict__ z, const float* __restrict__ v, const uint32_t* __restrict__ mask1,
                        const uint8_t* __restrict__ mask2, int B, int Hq, int Hw_in, int rows_per_split,
                        const float4* __restrict__ A0q_g, const float* __restrict__ sumV, float* __restrict__ dP0part) {
  constexpr int S = kDpS16, KS = 32;                         // samples per stage
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* stages = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* samp = reinterpret_cast<float*>(stages + S * kDpStage16);           // [2][2D+1][256]  z, v, s2 per sample
  uint32_t* sampw = reinterpret_cast<uint32_t*>(samp + 2 * 256 * (2 * D + 1));    // [2][8][256] this CTA's mask words
  uint64_t* bars = reinterpret_cast<uint64_t*>(sampw + 2 * 8 * 256);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 1);
  float* redmax = reinterpret_cast<float*>(tmem_slot + 2);                   // [16] per-warp maxima of the scale scan
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + S), accfull = smem_u32(bars + 2 * S);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
  const uint32_t rank = cluster_rank3();
  const int n0 = (blockIdx.x >> 1) * 256 + (int)rank * 128;  // my 128 n's (rows of D)
  const int o0 = blockIdx.y * 512, split = blockIdx.z;
  const bool two = o0 + 256 < Hq;                            // Hq is a multiple of 256: the last o-tile may be half
  const int b0 = split * rows_per_split;
  const int b1 = min(B, b0 + rows_per_split);
  const int NSG = (max(b1 - b0, 0) + KS - 1) / KS;           // stages

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full0 + 8 * s, 2 * kDpWarps); mbar_init(empty0 + 8 * s, 1); }
    mbar_init(accfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kDpWarps) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync3();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lead_full0 = mapa3(full0, 0);

  if (warp_u < kDpWarps) {
    // thread -> (sample ks of the stage, 8 consecutive MN elements = one 16-byte chunk).  The 8 lanes of a quarter warp hold the
    // 8 chunks of one 128-byte row (conflict-free 16-byte stores); a warp covers the k-rows kr of all four 8-k groups.
    const int ncl = lane & 7, kg = lane >> 3, atom = warp & 1, kr = warp >> 1;
    const int ks = kg * 8 + kr;
    const uint32_t off = (uint32_t)(kg * 2048 + atom * 1024 + kr * 128) + ((uint32_t)(ncl ^ kr) << 4);
    const int wsel = atom * 2 + (ncl >> 2), bsh = (ncl & 3) * 8;   // my 8 bits: word wsel of either accumulator's 4 words
    float2 qx2[4], qy2[4], qz2[4], qw2[4];                   // my 8 n's as four packed pairs: (w0, w1, w2, bias)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int n = n0 + atom * 64 + ncl * 8 + 2 * i;
      const float4 qa = A0q_g[n], qb = A0q_g[n + 1];
      qx2[i] = make_float2(qa.x, qb.x); qy2[i] = make_float2(qa.y, qb.y);
      qz2[i] = make_float2(qa.z, qb.z); qw2[i] = make_float2(qa.w, qb.w);
    }
    // ---- the split's scale: largest bound of |s2 q1| over my samples -> one power of two for the whole accumulation ----
    const float4 amax = make_float4(sumV[24], sumV[25], sumV[26], sumV[27]);
    float bmax = 0.f;
    for (int m = b0 + tid; m < b1; m += kDpWarps * 32) {
      float zr[D], vr[D];
#pragma unroll
      for (int j = 0; j < D; ++j) { zr[j] = __ldg(z + (size_t)m * D + j); vr[j] = __ldg(v + (size_t)m * D + j); }
      float bu = __fmul_rn(amax.x, fabsf(2.f * vr[0]));
      if (D > 1) bu = fmaf(amax.y, fabsf(2.f * vr[D > 1 ? 1 : 0]), bu);
      if (D > 2) bu = fmaf(amax.z, fabsf(2.f * vr[D > 2 ? 2 : 0]), bu);
      bmax = fmaxf(bmax, __fmul_rn(bu, h0_bound<D>(zr, amax)));
    }
    bmax = warp_max(bmax);
    if (lane == 0) redmax[warp] = bmax;
    bar_dp();
#pragma unroll
    for (int w = 0; w < kDpWarps; ++w) bmax = fmaxf(bmax, redmax[w]);
    const uint32_t eb = bexp_of(bmax, 30u, 220u);
    const float G = __uint_as_float((267u - eb) << 23), invG = __uint_as_float((eb - 13u) << 23);

    constexpr int CH = 256, ZV = 2 * D + 1, SPC = CH / KS;   // stages per staged chunk of samples
    const int nchunk = (NSG * KS + CH - 1) / CH;
    float pre_f[ZV];
    uint32_t pre_w[4];
    auto fetch = [&](int c) {                                // thread -> sample (tid&255), accumulator t = tid>>8
      const int mrow = b0 + c * CH + (tid & 255);
      const bool in = mrow < b1;
      if (tid < CH) {
#pragma unroll
        for (int j = 0; j < D; ++j) {
          pre_f[j] = in ? __ldg(z + (size_t)mrow * D + j) : 0.f;
          pre_f[D + j] = in ? __ldg(v + (size_t)mrow * D + j) : 0.f;
        }
        pre_f[2 * D] = in ? (__ldg(mask2 + mrow) ? 1.f : kSlope) : 0.f;
      }
      const int w0 = (o0 >> 5) + (tid >> 8) * 8 + (int)rank * 4;
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) pre_w[q4] = (in && w0 + q4 < Hw_in) ? __ldg(mask1 + (size_t)mrow * Hw_in + w0 + q4) : 0u;
    };
    auto stash = [&](int buf) {
      float* zf = samp + buf * (CH * ZV);
      uint32_t* mw = sampw + buf * (CH * 8);
      if (tid < CH) {
#pragma unroll
        for (int j = 0; j < ZV; ++j) zf[j * CH + tid] = pre_f[j];
      }
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) mw[((tid >> 8) * 4 + q4) * CH + (tid & 255)] = pre_w[q4];
    };
    if (nchunk > 0) { fetch(0); stash(0); }
    bar_dp();
    for (int sg = 0; sg < NSG; ++sg) {
      const int c = sg / SPC, buf = c & 1, sl = (sg % SPC) * KS + ks;      // sample slot inside the chunk
      if ((sg % SPC) == 0 && c + 1 < nchunk) fetch(c + 1);
      const float* zf = samp + buf * (CH * ZV);
      float zr[D], vr[D];
#pragma unroll
      for (int j = 0; j < D; ++j) { zr[j] = zf[j * CH + sl]; vr[j] = zf[(D + j) * CH + sl]; }
      const float s2f = zf[2 * D * CH + sl];
      const uint32_t bits0 = sampw[buf * (CH * 8) + wsel * CH + sl] >> bsh;
      const uint32_t bits1 = sampw[buf * (CH * 8) + (4 + wsel) * CH + sl] >> bsh;
      // A = G s2 q1 = (2 G s2 A0 v) . max(h0, 0.04 h0) for my 8 n's, two per packed instruction
      float qv[8];
      float sv[D];
#pragma unroll
      for (int j = 0; j < D; ++j) sv[j] = ((2.f * s2f) * G) * vr[j];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float2 h = __ffma2_rn(qx2[i], make_float2(zr[0], zr[0]), qw2[i]);
        float2 uu = __fmul2_rn(qx2[i], make_float2(sv[0], sv[0]));
        if (D > 1) {
          h = __ffma2_rn(qy2[i], make_float2(zr[D > 1 ? 1 : 0], zr[D > 1 ? 1 : 0]), h);
          uu = __ffma2_rn(qy2[i], make_float2(sv[D > 1 ? 1 : 0], sv[D > 1 ? 1 : 0]), uu);
        }
        if (D > 2) {
          h = __ffma2_rn(qz2[i], make_float2(zr[D > 2 ? 2 : 0], zr[D > 2 ? 2 : 0]), h);
          uu = __ffma2_rn(qz2[i], make_float2(sv[D > 2 ? 2 : 0], sv[D > 2 ? 2 : 0]), uu);
        }
        const float2 l = __fmul2_rn(h, make_float2(kSlope * kSlope, kSlope * kSlope));
        const float2 x = __fmul2_rn(uu, make_float2(fmaxf(h.x, l.x), fmaxf(h.y, l.y)));
        qv[2 * i] = x.x; qv[2 * i + 1] = x.y;
      }
      if ((sg % SPC) == SPC - 1 && c + 1 < nchunk) {          // next chunk's buffer was last read SPC stages ago
        bar_dp();
        stash(buf ^ 1);
        bar_dp();
      }
      const uint32_t s = sg % S, ph = (sg / S) & 1;
      mbar_wait(empty0 + 8 * s, ph ^ 1);
      unsigned char* st = stages + s * kDpStage16 + off;
      uint4 hi, lo;
      split_f16(qv[0], qv[1], hi.x, lo.x);
      split_f16(qv[2], qv[3], hi.y, lo.y);
      split_f16(qv[4], qv[5], hi.z, lo.z);
      split_f16(qv[6], qv[7], hi.w, lo.w);
      *reinterpret_cast<uint4*>(st) = hi;
      *reinterpret_cast<uint4*>(st + kDpTile16) = lo;
      // B = 1 + 4*bit (the LeakyReLU slope / 0.2, exact in fp16; 0.2 and P1 are applied by finalize_W0)
      *reinterpret_cast<uint4*>(st + 2 * kDpTile16) = make_uint4(pat2_f16(bits0), pat2_f16(bits0 >> 2), pat2_f16(bits0 >> 4), pat2_f16(bits0 >> 6));
      *reinterpret_cast<uint4*>(st + 3 * kDpTile16) = make_uint4(pat2_f16(bits1), pat2_f16(bits1 >> 2), pat2_f16(bits1 >> 4), pat2_f16(bits1 >> 6));
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(lead_full0 + 8 * s);
    }
    // epilogue: TMEM lane = my n, column = o (512 of them).  Warp w: lane quadrant w & 3, the 128 columns of group w >> 2.
    const int q = warp & 3, cg = warp >> 2;
    const int n = n0 + q * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * 128);
    if (two || cg < 2) {
      float* out = dP0part + ((size_t)split * Hq + o0 + cg * 128) * Hq + n;
      if (NSG > 0) {
        mbar_wait_parked(accfull, 0, k3ParkNs);
        tc_fence_after();
#pragma unroll 1
        for (int cc = 0; cc < 4; ++cc) {
          uint32_t r[32];
          tmem_ld32(taddr + cc * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) out[(size_t)(cc * 32 + j) * Hq] = __uint_as_float(r[j]) * invG;
        }
      } else {
        for (int j = 0; j < 128; ++j) out[(size_t)j * Hq] = 0.f;
      }
    }
  } else if (rank == 0) {
    const uint64_t desc0 = make_desc_mn128_b16(smem_u32(stages));
    for (int sg = 0; sg < NSG; ++sg) {
      const uint32_t s = sg % S, ph = (sg / S) & 1;
      mbar_wait(full0 + 8 * s, ph);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t sa = desc0 + (uint64_t)((s * kDpStage16) >> 4);
#pragma unroll
        for (int g = 0; g < 2; ++g) {                                            // K = 16 = two 8-k groups (2 x SBO = 4 KB)
          const uint64_t a_hi = sa + (uint64_t)((g * 4096) >> 4);
          const uint32_t acc = (sg | g) ? 1u : 0u;
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            if (t == 1 && !two) break;
            const uint32_t d_t = tmem_base + (uint32_t)(t * 256);
            const uint64_t b = sa + (uint64_t)(((2 + t) * kDpTile16 + g * 4096) >> 4);
            umma_f16_pair_mn(d_t, a_hi + (uint64_t)(kDpTile16 >> 4), b, acc);     // B is exact: a_lo.b + a_hi.b
            umma_f16_pair_mn(d_t, a_hi, b, 1u);
          }
        }
        umma_commit_pair(empty0 + 8 * s);
        if (sg == NSG - 1) umma_commit_pair(accfull);
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync3();
  if (warp == kDpWarps) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// clusters of two CTAs of `fn` that can be resident at once
static int max_clusters_for(const void* fn, size_t smem, int threads) {
  cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * 74); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at;
  at.id = cudaLaunchAttributeClusterDimension;
  at.val.clusterDim.x = 2; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
  cfg.attrs = &at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, fn, &cfg) != cudaSuccess || n <= 0) {
    (void)cudaGetLastError();
    n = sm_count() / 2;
  }
  return n;
}

// dP0 launches: one wave of long-running clusters, never more slabs than the workspace holds
template <int D, bool X3>
static int launch_tc3_dp0(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L,
                          const float4* A0q, float* part, int* splits_out, cudaStream_t st) {
  constexpr size_t smem = dp3_smem_bytes<D, X3>();
  static_assert(smem <= 227 * 1024, "dP0 pair kernel: shared memory");
  static int max_clusters = 0;
  if (max_clusters == 0)
    max_clusters = max_clusters_for(reinterpret_cast<const void*>(icnn_tc3_dP0_kernel<D, X3>), smem, kDpThreads3);
  int splits = dp0_splits(L.B, L.Hq, max_clusters);
  if (splits > L.dp0_splits) splits = L.dp0_splits;
  const int rows = round_up((L.B + splits - 1) / splits, kKB);
  dim3 grid(2 * (L.Hq / 256), (L.Hq + 511) / 512, splits);
  icnn_tc3_dP0_kernel<D, X3><<<grid, kDpThreads3, smem, st>>>(z, v, mask1, mask2, L.B, L.Hq, L.Hp / 32, rows, A0q, part);
  *splits_out = splits;
  return check_launch();
}
template <int D>
static int launch_tc3_dp0_f16(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L,
                              const float4* A0q, const float* sumV, float* part, int* splits_out, cudaStream_t st) {
  constexpr size_t smem = dp3_f16_smem_bytes<D>();
  static_assert(smem <= 227 * 1024, "dP0 pair kernel (fp16): shared memory");
  static int max_clusters = 0;
  if (max_clusters == 0)
    max_clusters = max_clusters_for(reinterpret_cast<const void*>(icnn_tc3_dP0_f16_kernel<D>), smem, kDpThreads3);
  int splits = dp0_splits(L.B, L.Hq, max_clusters);
  if (splits > L.dp0_splits) splits = L.dp0_splits;
  const int rows = round_up((L.B + splits - 1) / splits, 32);
  dim3 grid(2 * (L.Hq / 256), (L.Hq + 511) / 512, splits);
  icnn_tc3_dP0_f16_kernel<D><<<grid, kDpThreads3, smem, st>>>(z, v, mask1, mask2, L.B, L.Hq, L.Hp / 32, rows, A0q, sumV, part);
  *splits_out = splits;
  return check_launch();
}
// dP0part_tc: [splits][Hq][Hq] ordered split-K slabs (reduced by finalize_W0_kernel)
static int tc3_dp0(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L, int precision,
                   float* ws, int* splits_out, cudaStream_t st) {
  const float4* q = reinterpret_cast<const float4*>(ws + L.A0q);
  float* part = ws + L.dP0part_tc;
  if (precision == B200VAE_PREC_F16X3) {
    const float* sumV = ws + L.sumV;                         // max |A0| for the FP16 mode's scale
    switch (L.d) {
      case 1: return launch_tc3_dp0_f16<1>(z, v, mask1, mask2, L, q, sumV, part, splits_out, st);
      case 2: return launch_tc3_dp0_f16<2>(z, v, mask1, mask2, L, q, sumV, part, splits_out, st);
      default: return launch_tc3_dp0_f16<3>(z, v, mask1, mask2, L, q, sumV, part, splits_out, st);
    }
  }
  const bool x3 = precision == B200VAE_PREC_TF32X3;
#define B200VAE_TC3D(DD)                                                                          \
  return x3 ? launch_tc3_dp0<DD, true>(z, v, mask1, mask2, L, q, part, splits_out, st)            \
            : launch_tc3_dp0<DD, false>(z, v, mask1, mask2, L, q, part, splits_out, st)
  switch (L.d) {
    case 1: B200VAE_TC3D(1);
    case 2: B200VAE_TC3D(2);
    default: B200VAE_TC3D(3);
  }
#undef B200VAE_TC3D
}

template <int D, int MODE, bool SV>
static int launch_tc3_bwd(const Tc3BwdArgs& args, cudaStream_t st) {
  const size_t smem = tc3_smem_bytes<MODE>(args.Hq);
  static int max_clusters = 0;
  if (max_clusters == 0)
    max_clusters = max_clusters_for(reinterpret_cast<const void*>(icnn_tc3_bwd_kernel<D, MODE, SV>), smem, k3Threads);
  const int units = (SV ? 1 : 2) * args.T * args.NP;
  const int G = units < max_clusters ? units : max_clusters;
  icnn_tc3_bwd_kernel<D, MODE, SV><<<2 * G, k3Threads, smem, st>>>(args);
  return check_launch();
}

// rows part of the backward: fills partA / partB [T*8][d+1][Hq], a2part_tc [T][d], dz [B,d]
static int tc3_bwd_rows(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L,
                        float kappa, float* dz, int precision, float* ws, const float* accsave, cudaStream_t st) {
  const int mode = tc3_mode(precision);
  Tc3Maps mp;
  int rc = get_maps3(ws, L, mode, &mp);
  if (rc) return rc;
  Tc3BwdArgs args;
  args.b1hi = mp.b1hi; args.b1lo = mp.b1lo; args.b2hi = mp.b2hi; args.b2lo = mp.b2lo;
  args.z = z; args.v = v; args.mask1 = mask1; args.mask2 = mask2;
  args.A0g = reinterpret_cast<const float4*>(ws + L.A0g);
  args.E1 = reinterpret_cast<const float4*>(ws + L.E1);
  args.A0q = reinterpret_cast<const float4*>(ws + L.A0q);
  args.A1q = reinterpret_cast<const float4*>(ws + L.A1q);
  args.sumV = ws + L.sumV;
  args.partA = ws + L.partA; args.partB = ws + L.partB;
  args.dzpart = reinterpret_cast<float4*>(ws + L.dzpart);
  args.accsave = accsave;
  args.B = L.B; args.Hq = L.Hq; args.T = L.Bp / 256; args.NP = L.NP; args.Hw_in = L.Hp / 32;
  // the saved-accumulator kernels pay off where the kernel is tensor bound (3xTF32); at 1xTF32 the epilogue warps are the
  // bottleneck either way and recomputing GEMM2 is free
#define B200VAE_TC3B(DD)                                                                                                  \
  rc = mode == kF16 ? (accsave ? launch_tc3_bwd<DD, kF16, true>(args, st) : launch_tc3_bwd<DD, kF16, false>(args, st))    \
       : mode == kX3 ? (accsave ? launch_tc3_bwd<DD, kX3, true>(args, st) : launch_tc3_bwd<DD, kX3, false>(args, st))     \
                     : launch_tc3_bwd<DD, kTf32, false>(args, st)
  switch (L.d) {
    case 1: B200VAE_TC3B(1); break;
    case 2: B200VAE_TC3B(2); break;
    default: B200VAE_TC3B(3); break;
  }
#undef B200VAE_TC3B
  if (rc) return rc;
  tc3_bwd_dz_kernel<<<args.T, 256, 0, st>>>(args.dzpart, v, mask2, L.B, args.NP, L.d, kappa, dz, ws + L.a2part_tc);
  return check_launch();
}

// phase 0: everything; 1: the rows part only (dz + the ordered column partials in the workspace); 2: the parameter
// gradients only (dP0 + the finalize kernels), from the partials a phase-1 call left in the SAME workspace
int tc_bwd(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2, const WsLayout& L,
           const b200vae_icnn_params* p, int mode, float kappa, const b200vae_icnn_grads* g, float* dz, int precision,
           float* ws, const float* accsave, int phase, cudaStream_t st) {
  int rc = B200VAE_OK;
  if (phase != 2) rc = tc3_bwd_rows(z, v, mask1, mask2, L, kappa, dz, precision, ws, accsave, st);
  if (rc || !g || phase == 1) return rc;
  if (g->W0) {
    int splits = 0;
    rc = tc3_dp0(z, v, mask1, mask2, L, precision, ws, &splits, st);
    if (rc) return rc;
    rc = finalize_W0_launch(ws + L.dP0part_tc, splits, L.H, L.Hp, L.Hq, ws + L.P0, ws + L.P1, p->W0, mode, kSlope, g->W0, st);
    if (rc) return rc;
  }
  const int T = L.Bp / 256;
  dim3 fgrid(L.Hq / 32, L.d + 1, 2);
  tc_finalize_small_kernel<<<fgrid, 1024, 0, st>>>(ws + L.partA, ws + L.partB, ws + L.a2part_tc, T * 8, T, L.d, L.H, L.Hq,
                                                  ws + L.P1, p->W1, mode, *g);
  return check_launch();
}

template <int D, int MODE>
static int launch_tc3(const Tc3Args& args, int units, cudaStream_t st) {
  const size_t smem = tc3_smem_bytes<MODE>(args.Hq);
  static int max_clusters = 0;
  if (max_clusters == 0)
    max_clusters = max_clusters_for(reinterpret_cast<const void*>(icnn_tc3_fwd_kernel<D, MODE>), smem, k3Threads);
  // every cluster must be resident (GEMM2 units wait for GEMM1 units of other clusters): never exceed one wave
  const int G = units < max_clusters ? units : max_clusters;
  icnn_tc3_fwd_kernel<D, MODE><<<2 * G, k3Threads, smem, st>>>(args);
  return check_launch();
}

template <int D, int MODE>
static int launch_tc3_jac(const Tc3Args& args, int units, float4* jscr, float* jac, cudaStream_t st) {
  const size_t smem = tc3_smem_bytes<MODE>(args.Hq);
  static int max_clusters = 0;
  if (max_clusters == 0)
    max_clusters = max_clusters_for(reinterpret_cast<const void*>(icnn_tc3_fwd_jac_kernel<D, MODE>), smem, k3Threads);
  const int G = units < max_clusters ? units : max_clusters;
  icnn_tc3_fwd_jac_kernel<D, MODE><<<2 * G, k3Threads, smem, st>>>(args, jscr, jac);
  return check_launch();
}

// the arguments of one pair-kernel forward (both variants); returns the unit count, or a negative error code
static int tc3_fwd_args(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1,
                        uint8_t* mask2, int mode, float* ws, float* accsave, Tc3Args& args) {
  if (L.Bp / 256 > kTc3MaxTiles) return B200VAE_EUNSUP;
  {
    Tc3Maps mp;
    int rc = get_maps3(ws, L, mode, &mp);
    if (rc) return rc;
    args.b1hi = mp.b1hi; args.b1lo = mp.b1lo; args.b2hi = mp.b2hi; args.b2lo = mp.b2lo;
  }
  args.z = z;
  args.A0g = reinterpret_cast<const float4*>(ws + L.A0g);
  args.E1 = reinterpret_cast<const float4*>(ws + L.E1);
  args.A0q = reinterpret_cast<const float4*>(ws + L.A0q);
  args.A1q = reinterpret_cast<const float4*>(ws + L.A1q);
  args.P1q = ws + L.P1q;
  args.sumV = ws + L.sumV;
  args.A2p = ws + L.A2p;
  args.psi = psi; args.xhat = xhat; args.mask2 = mask2;
  args.want_x = xhat != nullptr ? 1 : 0;
  if (mask1) { args.maskg = mask1; args.mask_stride = L.Hp / 32; args.mask_rows = L.B; }
  else if (args.want_x) { args.maskg = reinterpret_cast<uint32_t*>(ws + L.imask); args.mask_stride = L.Hq / 32; args.mask_rows = L.Bp; }
  else { args.maskg = nullptr; args.mask_stride = 0; args.mask_rows = 0; }
  args.scr1 = reinterpret_cast<float4*>(ws + L.scr1);
  args.scr2 = reinterpret_cast<float4*>(ws + L.scr2);
  args.cnt = reinterpret_cast<uint32_t*>(ws + L.cnt);
  args.accsave = args.want_x ? accsave : nullptr;
  args.B = L.B; args.Hq = L.Hq; args.T = L.Bp / 256; args.NP = L.NP; args.kappa = kappa;
  // hi/lo modes: accumulate K in chunks of kTc3ChunkK where it divides Hq.  FP16 mode at H = 1024, default-init weights: psi
  // error 8.7e-6 in one piece (0.453 ms), 4.0e-6 in two chunks (0.474 ms, wherever the split point lies -- 512 ... 768
  // measured; the 21 us are the drain's L2 traffic: 14 us its stores, 6 us the loads of the last chunk's epilogue --
  // measured by leaving each out), 2.0e-6 in four (0.544 ms)
  args.cscr = reinterpret_cast<float4*>(ws + L.cscr);
  args.NC = (mode != kTf32 && L.Hq % kTc3ChunkK == 0) ? L.Hq / kTc3ChunkK : 1;
  return (args.want_x ? 2 : 1) * args.T * args.NP;
}

int tc3_fwd(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
            int precision, float* ws, float* accsave, cudaStream_t st) {
  const int mode = tc3_mode(precision);
  Tc3Args args;
  const int units = tc3_fwd_args(z, L, kappa, psi, xhat, mask1, mask2, mode, ws, accsave, args);
  if (units < 0) return units;
#define B200VAE_TC3(DD)                                                       \
  return mode == kF16 ? launch_tc3<DD, kF16>(args, units, st)                 \
         : mode == kX3 ? launch_tc3<DD, kX3>(args, units, st) : launch_tc3<DD, kTf32>(args, units, st)
  switch (L.d) {
    case 1: B200VAE_TC3(1);
    case 2: B200VAE_TC3(2);
    default: B200VAE_TC3(3);
  }
#undef B200VAE_TC3
}

int tc3_fwd_jac(const float* z, const WsLayout& L, float kappa, float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
                float* jac, float4* jscr, int precision, float* ws, cudaStream_t st) {
  const int mode = tc3_mode(precision);
  Tc3Args args;
  const int units = tc3_fwd_args(z, L, kappa, psi, xhat, mask1, mask2, mode, ws, nullptr, args);
  if (units < 0) return units;
#define B200VAE_TC3J(DD)                                                                    \
  return mode == kF16 ? launch_tc3_jac<DD, kF16>(args, units, jscr, jac, st)                \
         : mode == kX3 ? launch_tc3_jac<DD, kX3>(args, units, jscr, jac, st)                \
                       : launch_tc3_jac<DD, kTf32>(args, units, jscr, jac, st)
  switch (L.d) {
    case 1: B200VAE_TC3J(1);
    case 2: B200VAE_TC3J(2);
    default: B200VAE_TC3J(3);
  }
#undef B200VAE_TC3J
}

}  // namespace b200vae
