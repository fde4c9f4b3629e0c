// icnn_wide_tc.cu -- tcgen05 forward (decode: psi + Brenier map) AND backward (dL/dxhat) for wide-input ICNNs (d > 4): the
// MNIST-shaped decoder ICNN(32,512) + ICNN(784,1024) of BASELINE configs[3] (model.py:766-805, module.py:142-148,
// model.py:820-828).  b200vae_icnn_wide_fwd / _bwd (icnn_wide.cu) call these drivers at TF32 / TF32X3 (and F16X3, which
// runs as TF32X3) when wide_tc_supported holds -- and, for the forward, b0, b1, A2 are 16-byte aligned; the psi-gradient
// backward always runs on the FP32 kernels.
//
// For wide inputs every product of the sweep is a dense contraction, so every GEMM of both directions is a launch of ONE
// generic tensor-core GEMM kernel  C[M,N] = xf(A1)[M,K1] . B1[N,K1]^T (+ A2[M,K2] . B2[N,K2]^T)  with different epilogues.
// The forward:
//   lin : h0 = z A0^T + b0                                   (store h0)
//   hid : h1 = sigma(h0)^2 P0^T + z A1^T + b1 -> byte mask, g1b = P1*sigma'(h1) (fp32), row partials of P1.sigma(h1)
//   row : h2 = sum partials + A2 z + b2 -> psi, s2            (small SIMT kernel)
//   gx1 : g0' = (g1b P0) * 2 a0 s0                            (s2 factored out: it is a per-row scalar)
//   out : xhat = s2 * (g0' A0 + g1b A1 + A2) + 2 kappa z
// Kernel: CTA tile 128 x 256, K in 16-float blocks (64-byte rows, SWIZZLE_64B), 6- / 8-stage ring.  Warp 8 streams BOTH
// operands with TMA (out-of-bounds rows/columns are zero filled: ragged B, d, H need no special cases); warps 0-7 apply
// the elementwise transform to the raw A tile IN PLACE in shared memory (the swizzle does not matter for an elementwise
// pass) and split it into tf32 hi / lo; warp 9 issues tcgen05.mma.kind::tf32 (3 MMAs per product at 3xTF32, B hi/lo
// prepared once per forward); the accumulator (128 lanes x 256 columns of TMEM) is drained by warps 0-7 with
// tcgen05.ld.32x32b: one thread = one sample row x 128 columns, so row partials need no shuffles and stores are
// row-contiguous.  The saved activations (h0, byte mask, s2) have the FP32 path's format, so either backward runs on them.
// The backward runs the sample-stationary GEMMs (u0, w1, gx1, dz) with fused epilogues, then transposes its operands so
// that the batch becomes K and runs the batch-reduction GEMMs (dA0, dA1, dP0) split over K into ordered slabs.
#include <string.h>

#include "icnn_wide.cuh"
#include "tc_common.cuh"

namespace b200vae {

constexpr int kWtThreads = 10 * 32;
constexpr int kWtATile = 128 * 64;
// Accumulation accuracy at 3xTF32.  tcgen05 adds into its fp32 accumulator with truncation: a downward bias that grows with
// the number of MMAs per accumulator times the accumulator's magnitude (measured on psi of ICNN(784,1024): 3.0e-5 with the
// 3 MMAs of every K step in ONE accumulator).  The 3xTF32 kernel therefore uses 128-column tiles and all four 128-column
// accumulators that fit in TMEM: the hi*hi products of the first / second / last third of K go to accumulators 0 / 1 / 2
// and ALL lo-order products (2^-11 smaller, so their truncation is negligible) to accumulator 3; the epilogue adds the four
// with round-to-nearest FP32 adds.  A third of the truncating adds per accumulator, each on a third of the magnitude: 1/9 of
// the bias.  The 1xTF32 kernel keeps one 256-column accumulator (its error is the operand rounding).
constexpr int kWtMainChunks = 3;

enum { WT_XF_ID = 0, WT_XF_X1 = 1 };
enum { WT_EPI_LIN = 0, WT_EPI_HID = 1, WT_EPI_GX1 = 2, WT_EPI_OUT = 3, WT_EPI_U = 4, WT_EPI_W1 = 5, WT_EPI_GXB = 6, WT_EPI_DZ = 7, WT_EPI_SLAB = 8 };

struct alignas(64) WtArgs {
  CUtensorMap a1, b1hi, b1lo, a2, b2hi, b2lo;
  int nkb1, nkb2, xf1, M, N, epi;
  const float* bias;     // LIN: b0, HID: b1
  const float* P1;       // HID
  const float* h0;       // GX1
  const float* s2;       // OUT
  const float* A2w;      // OUT
  const float* z;        // OUT: [M, nz]
  int nz;
  float kappa2;
  float* out0;           // LIN: h0, HID: g1b, GX1: g0', OUT: xhat   (row stride N)
  uint8_t* mask;         // HID (written); W1 (read)
  float* part;           // HID: [M][npart]
  int npart;
  // backward epilogues
  float* out1;           // U: q1, GXB: t0
  const float* u0;       // GXB
  const float* v;        // DZ: [M, ldv]
  int ldv;
  int kb_per_split;      // > 0: split-K over blockIdx.z (both phases share the K range); SLAB epilogue stores partial tiles
};

template <bool X3>
struct WtCfg {
  static constexpr int NT = X3 ? 128 : 256;                      // tile / accumulator width (columns)
  static constexpr int kBTile = NT * 64;
  static constexpr int kStage = kWtATile * (X3 ? 2 : 1) + kBTile * (X3 ? 2 : 1);
  static constexpr int kOffAlo = kWtATile, kOffB = kWtATile * (X3 ? 2 : 1), kOffBlo = kOffB + kBTile;
  static constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  // ring depth (template parameter of the kernel): as many stages as fit -- 6 x 32 KB / 8 x 24 KB -- where the grid is at
  // most one wave: at the configs' own batch (256 rows = 2 row tiles) a GEMM is a latency chain TMA -> transform -> MMA per
  // K-block and its time is (K-blocks / stages) x that latency (B = 256 decode 0.344 -> 0.309 ms).  Larger 3xTF32 grids keep
  // 4 stages: the deep ring leaves ~30 KB of L1 for the epilogue's parameter reads (B = 8192 decode 0.58 -> 0.82 ms with 6).
  static constexpr int kDeep = X3 ? 6 : 8, kShallow = X3 ? 4 : 8;
};
inline int wt_tile_n(bool x3) { return x3 ? 128 : 256; }
template <bool X3>
static size_t wt_smem_bytes(int S) { return (size_t)S * WtCfg<X3>::kStage + (3 * S + 1) * 8 + 16 + 1024; }

template <bool X3, int S>
__global__ void __launch_bounds__(kWtThreads, 1)
wide_tc_gemm_kernel(const __grid_constant__ WtArgs a) {
  using C = WtCfg<X3>;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* stages = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S * C::kStage);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * S + 1);
  const uint32_t full0 = smem_u32(bars), ready0 = smem_u32(bars + S), empty0 = smem_u32(bars + 2 * S),
                 accfull = smem_u32(bars + 3 * S);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
  constexpr int NT = C::NT;
  const int m0 = blockIdx.x * 128, n0 = blockIdx.y * NT;
  const int nkb = a.nkb1 + a.nkb2;
  const int kb_off = a.kb_per_split > 0 ? (int)blockIdx.z * a.kb_per_split : 0;   // split-K: first K-block of this CTA

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(ready0 + 8 * s, 8); mbar_init(empty0 + 8 * s, 1); }
    mbar_init(accfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(X3 ? 512 : 256));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp_u < 8) {
    // =========================== transform warps, then epilogue ===========================
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S;
      mbar_wait(full0 + 8 * s, (kb / S) & 1);
      const bool x1 = (kb < a.nkb1) && (a.xf1 == WT_XF_X1);
      unsigned char* At = stages + s * C::kStage;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float4* p = reinterpret_cast<float4*>(At + (tid + 256 * h) * 16);
        float4 v = *p;
        if (x1) {
          float t;
          t = fmaxf(v.x, kSlope * v.x); v.x = t * t;
          t = fmaxf(v.y, kSlope * v.y); v.y = t * t;
          t = fmaxf(v.z, kSlope * v.z); v.z = t * t;
          t = fmaxf(v.w, kSlope * v.w); v.w = t * t;
        }
        if (X3) {
          const float4 hi = make_float4(rn_tf32_masked(v.x), rn_tf32_masked(v.y), rn_tf32_masked(v.z), rn_tf32_masked(v.w));
          *p = hi;
          *reinterpret_cast<float4*>(At + C::kOffAlo + (tid + 256 * h) * 16) =
              make_float4(rn_tf32_fast(v.x - hi.x), rn_tf32_fast(v.y - hi.y), rn_tf32_fast(v.z - hi.z), rn_tf32_fast(v.w - hi.w));
        } else {
          *p = make_float4(rn_tf32_fast(v.x), rn_tf32_fast(v.y), rn_tf32_fast(v.z), rn_tf32_fast(v.w));
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(ready0 + 8 * s);
    }
    // ---- epilogue: my row, one half of the tile's columns ----
    const int q4 = warp & 3, chalf = warp >> 2;
    const int row = m0 + q4 * 32 + lane;
    const bool rin = row < a.M;
    const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(chalf * (NT / 2));
    mbar_wait_parked(accfull, 0, 1000);
    tc_fence_after();
    float rowsum = 0.f;
    const float s2r = ((a.epi == WT_EPI_OUT || a.epi == WT_EPI_W1 || a.epi == WT_EPI_GXB) && rin) ? a.s2[row] : 0.f;
#pragma unroll 1
    for (int cc = 0; cc < NT / 64; ++cc) {
      uint32_t r[32];
      tmem_ld32(taddr + cc * 32, r);
      tmem_ld_wait();
      if (X3) {                                              // + the other K-chunk accumulators in use, then the lo-order one
        const int nchunks = min(kWtMainChunks, nkb);
#pragma unroll 1
        for (int k = 1; k <= nchunks; ++k) {
          uint32_t r2[32];
          tmem_ld32(taddr + (k < nchunks ? k : kWtMainChunks) * NT + cc * 32, r2);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
        }
      }
      const int c0 = n0 + chalf * (NT / 2) + cc * 32;
      if (!rin || c0 >= a.N) continue;
      const int nv = min(32, a.N - c0);                    // N % 4 == 0: whole float4 groups
      float* orow = a.out0 + (size_t)row * a.N + c0;
      if (a.epi == WT_EPI_SLAB) {              // split-K partial tile -> slab[blockIdx.z]
        float* srow = orow + (size_t)blockIdx.z * a.M * a.N;
        for (int j = 0; j < nv; j += 4)
          *reinterpret_cast<uint4*>(srow + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
      } else if (a.epi == WT_EPI_LIN) {
        for (int j = 0; j < nv; j += 4) {
          const float4 b = *reinterpret_cast<const float4*>(a.bias + c0 + j);
          *reinterpret_cast<float4*>(orow + j) = make_float4(__uint_as_float(r[j]) + b.x, __uint_as_float(r[j + 1]) + b.y,
                                                             __uint_as_float(r[j + 2]) + b.z, __uint_as_float(r[j + 3]) + b.w);
        }
      } else if (a.epi == WT_EPI_HID) {
        uint8_t* mrow = a.mask + (size_t)row * a.N + c0;
        for (int j = 0; j < nv; j += 4) {
          const float4 b = *reinterpret_cast<const float4*>(a.bias + c0 + j);
          const float4 p1 = *reinterpret_cast<const float4*>(a.P1 + c0 + j);
          const float h[4] = {__uint_as_float(r[j]) + b.x, __uint_as_float(r[j + 1]) + b.y, __uint_as_float(r[j + 2]) + b.z,
                              __uint_as_float(r[j + 3]) + b.w};
          const float pp[4] = {p1.x, p1.y, p1.z, p1.w};
          float g[4];
          uint32_t mb = 0;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const bool pos = h[e] > 0.f;
            rowsum = fmaf(pp[e], pos ? h[e] : kSlope * h[e], rowsum);
            g[e] = pos ? pp[e] : kSlope * pp[e];
            mb |= (pos ? 1u : 0u) << (8 * e);
          }
          *reinterpret_cast<float4*>(orow + j) = make_float4(g[0], g[1], g[2], g[3]);
          *reinterpret_cast<uint32_t*>(mrow + j) = mb;
        }
      } else if (a.epi == WT_EPI_GX1) {
        const float* hrow = a.h0 + (size_t)row * a.N + c0;
        for (int j = 0; j < nv; j += 4) {
          const float4 hv = *reinterpret_cast<const float4*>(hrow + j);
          const float h[4] = {hv.x, hv.y, hv.z, hv.w};
          float g[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float sl = h[e] > 0.f ? 1.f : kSlope;
            g[e] = __uint_as_float(r[j + e]) * (2.f * h[e] * sl * sl);
          }
          *reinterpret_cast<float4*>(orow + j) = make_float4(g[0], g[1], g[2], g[3]);
        }
      } else if (a.epi == WT_EPI_U) {          // u0 = acc, q1 = u0 * 2 a0 s0
        const float* hrow = a.h0 + (size_t)row * a.N + c0;
        float* qrow = a.out1 + (size_t)row * a.N + c0;
        for (int j = 0; j < nv; j += 4) {
          const float4 hv = *reinterpret_cast<const float4*>(hrow + j);
          const float h[4] = {hv.x, hv.y, hv.z, hv.w};
          float u[4], q[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float sl = h[e] > 0.f ? 1.f : kSlope;
            u[e] = __uint_as_float(r[j + e]);
            q[e] = u[e] * (2.f * h[e] * sl * sl);
          }
          *reinterpret_cast<float4*>(orow + j) = make_float4(u[0], u[1], u[2], u[3]);
          *reinterpret_cast<float4*>(qrow + j) = make_float4(q[0], q[1], q[2], q[3]);
        }
      } else if (a.epi == WT_EPI_W1) {         // e1 = s2 s1 w1 (its column sums are dP1)
        const uint8_t* mrow = a.mask + (size_t)row * a.N + c0;
        for (int j = 0; j < nv; j += 4) {
          const uint32_t mb = *reinterpret_cast<const uint32_t*>(mrow + j);
          float o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) o[e] = __uint_as_float(r[j + e]) * (((mb >> (8 * e)) & 0xffu) ? s2r : kSlope * s2r);
          *reinterpret_cast<float4*>(orow + j) = make_float4(o[0], o[1], o[2], o[3]);
        }
      } else if (a.epi == WT_EPI_GXB) {        // gx1 = s2 acc;  g0 = gx1 2 a0 s0;  t0 = u0 2 gx1 s0^2
        const float* hrow = a.h0 + (size_t)row * a.N + c0;
        const float* urow = a.u0 + (size_t)row * a.N + c0;
        float* trow = a.out1 + (size_t)row * a.N + c0;
        for (int j = 0; j < nv; j += 4) {
          const float4 hv = *reinterpret_cast<const float4*>(hrow + j);
          const float4 uv = *reinterpret_cast<const float4*>(urow + j);
          const float h[4] = {hv.x, hv.y, hv.z, hv.w}, u[4] = {uv.x, uv.y, uv.z, uv.w};
          float g[4], t[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float sl = h[e] > 0.f ? 1.f : kSlope, gx = s2r * __uint_as_float(r[j + e]);
            g[e] = gx * (2.f * h[e] * sl * sl);
            t[e] = u[e] * (2.f * gx) * sl * sl;
          }
          *reinterpret_cast<float4*>(orow + j) = make_float4(g[0], g[1], g[2], g[3]);
          *reinterpret_cast<float4*>(trow + j) = make_float4(t[0], t[1], t[2], t[3]);
        }
      } else if (a.epi == WT_EPI_DZ) {         // dz = acc + 2 kappa v
        for (int j = 0; j < nv; j += 4) {
          const float4 vv = *reinterpret_cast<const float4*>(a.v + (size_t)row * a.ldv + c0 + j);
          *reinterpret_cast<float4*>(orow + j) = make_float4(fmaf(a.kappa2, vv.x, __uint_as_float(r[j])), fmaf(a.kappa2, vv.y, __uint_as_float(r[j + 1])),
                                                             fmaf(a.kappa2, vv.z, __uint_as_float(r[j + 2])), fmaf(a.kappa2, vv.w, __uint_as_float(r[j + 3])));
        }
      } else {   // WT_EPI_OUT
        for (int j = 0; j < nv; j += 4) {
          const float4 a2 = *reinterpret_cast<const float4*>(a.A2w + c0 + j);
          float o[4] = {s2r * (__uint_as_float(r[j]) + a2.x), s2r * (__uint_as_float(r[j + 1]) + a2.y),
                        s2r * (__uint_as_float(r[j + 2]) + a2.z), s2r * (__uint_as_float(r[j + 3]) + a2.w)};
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (c0 + j + e < a.nz) o[e] = fmaf(a.kappa2, a.z[(size_t)row * a.nz + c0 + j + e], o[e]);
          *reinterpret_cast<float4*>(orow + j) = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    if (a.epi == WT_EPI_HID && rin) a.part[(size_t)row * a.npart + blockIdx.y * 2 + chalf] = rowsum;
    tc_fence_before();
  } else if (warp_u == 8) {
    // =========================== TMA producer: A (raw) and B (hi, lo) tiles ===========================
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S;
      mbar_wait(empty0 + 8 * s, ((kb / S) & 1) ^ 1);
      if (elect_one()) {
        const bool p2 = kb >= a.nkb1;
        const int k0 = (kb_off + (p2 ? kb - a.nkb1 : kb)) * kKB;
        const uint32_t bar = full0 + 8 * s;
        const uint32_t dst = smem_u32(stages + s * C::kStage);
        mbar_arrive_expect_tx(bar, kWtATile + C::kBTile * (X3 ? 2 : 1));
        tma_load_2d(dst, p2 ? &a.a2 : &a.a1, bar, k0, m0);
        tma_load_2d(dst + C::kOffB, p2 ? &a.b2hi : &a.b1hi, bar, k0, n0);
        if (X3) tma_load_2d(dst + C::kOffBlo, p2 ? &a.b2lo : &a.b1lo, bar, k0, n0);
      }
      __syncwarp();
    }
  } else {
    // =========================== MMA issuer ===========================
    const uint64_t desc0 = make_desc_sw64(smem_u32(stages));
    const int nchunks = X3 ? min(kWtMainChunks, nkb) : 1;    // K-chunks in use (every one gets at least one K-block)
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S;
      mbar_wait(ready0 + 8 * s, (kb / S) & 1);
      tc_fence_after();
      const int chunk = (kb * nchunks) / nkb;
      const bool chunk_first = kb == 0 || ((kb - 1) * nchunks) / nkb != chunk;
      if (elect_one()) {
        const uint64_t a0 = desc0 + (uint64_t)(s * (C::kStage >> 4));
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          const uint64_t a_hi = a0 + (uint64_t)(ks * 2);
          const uint64_t b_hi = a_hi + (uint64_t)(C::kOffB >> 4);
          if (X3) {
            const uint32_t d_main = tmem_base + (uint32_t)(chunk * NT), d_lo = tmem_base + (uint32_t)(kWtMainChunks * NT);
            const uint64_t a_lo = a_hi + (uint64_t)(C::kOffAlo >> 4), b_lo = a_hi + (uint64_t)(C::kOffBlo >> 4);
            umma_tf32(d_lo, a_lo, b_hi, C::kIdesc, (kb | ks) ? 1u : 0u);
            umma_tf32(d_lo, a_hi, b_lo, C::kIdesc, 1u);
            umma_tf32(d_main, a_hi, b_hi, C::kIdesc, (chunk_first && ks == 0) ? 0u : 1u);
          } else {
            umma_tf32(tmem_base, a_hi, b_hi, C::kIdesc, (kb | ks) ? 1u : 0u);
          }
        }
        umma_commit(empty0 + 8 * s);
        if (kb + 1 == nkb) umma_commit(accfull);
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(X3 ? 512 : 256));
  }
}

// ---- prepare: positive weights and all operand copies, split into tf32 hi / lo ------------------------------------------------
__device__ __forceinline__ void split_store(float x, float* hi, float* lo, size_t i) {
  const float h = rn_tf32_masked(x);
  hi[i] = h; lo[i] = rn_tf32_masked(x - h);
}
__global__ void wide_tc_prepare_kernel(const float* __restrict__ W0, const float* __restrict__ W1, const float* __restrict__ A0w,
                                       const float* __restrict__ A1w, int d, int H, int mode, float* __restrict__ ws,
                                       WideLayout L) {
  const size_t HH = (size_t)H * H, dH = (size_t)d * H, tot = HH + H + dH, gstride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += gstride) {
    if (i < HH) {
      const float w = W0[i];
      const float p = (mode == B200VAE_WEIGHT_EXP) ? expf(w) : fmaxf(w, kClampMin);
      const size_t n = i / H, k = i - n * H;
      split_store(p, ws + L.P0hi, ws + L.P0lo, i);
      split_store(p, ws + L.P0Thi, ws + L.P0Tlo, k * H + n);
    } else if (i < HH + H) {
      const float w = W1[i - HH];
      ws[L.P1 + i - HH] = (mode == B200VAE_WEIGHT_EXP) ? expf(w) : fmaxf(w, kClampMin);
    } else {
      const size_t j = i - HH - H, n = j / d, c = j - n * d;    // A*w[n][c]
      split_store(A0w[j], ws + L.A0hi, ws + L.A0lo, j);
      split_store(A1w[j], ws + L.A1hi, ws + L.A1lo, j);
      split_store(A0w[j], ws + L.A0Thi, ws + L.A0Tlo, c * H + n);
      split_store(A1w[j], ws + L.A1Thi, ws + L.A1Tlo, c * H + n);
    }
  }
}
// g1b[b][n] = P1[n] * sigma'(h1[b][n]) from the saved byte mask (A operand of the backward's gx1 GEMM)
__global__ void wide_tc_g1b_kernel(const uint8_t* __restrict__ mask, const float* __restrict__ P1, size_t n, int H,
                                   float* __restrict__ g1b) {
  const size_t gstride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gstride)
    g1b[i] = P1[i % H] * (mask[i] ? 1.f : kSlope);
}
// ordered column sums of a [B][H] matrix: colpart[mt][H] over 128-row blocks (wide_col_finalize adds them in fixed order)
__global__ void __launch_bounds__(256)
wide_tc_colsum_kernel(const float* __restrict__ x, int B, int H, float* __restrict__ colpart) {
  const int c = blockIdx.y * 256 + threadIdx.x, r0 = blockIdx.x * 128, r1 = min(B, r0 + 128);
  if (c >= H) return;
  float s = 0.f;
  for (int r = r0; r < r1; ++r) s += x[(size_t)r * H + c];
  colpart[(size_t)blockIdx.x * H + c] = s;
}

// Transpose [B][C] -> [C][ldo] (ldo >= B) so that the BATCH index becomes the contiguous K dimension of the batch-reduction
// GEMMs.  mode 0: plain; mode 1: g1 = s2[b]*P1[c]*sigma'(h1) from the byte mask.  `lo` != null: also the tf32 residual.
__global__ void __launch_bounds__(256)
wide_tc_transpose_kernel(const float* __restrict__ src, const uint8_t* __restrict__ mask, const float* __restrict__ s2,
                         const float* __restrict__ P1, int mode, int B, int Ccols, int ldo, float* __restrict__ hi,
                         float* __restrict__ lo) {
  __shared__ float tile[32][33];
  const int b0 = blockIdx.x * 32, c0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int b = b0 + r, c = c0 + tx;
    float x = 0.f;
    if (b < B && c < Ccols) {
      const size_t i = (size_t)b * Ccols + c;
      x = mode == 1 ? s2[b] * P1[c] * (mask[i] ? 1.f : kSlope) : src[i];
    }
    tile[r][tx] = x;
  }
  __syncthreads();
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, b = b0 + tx;
    if (c < Ccols && b < B) {
      const float x = tile[tx][r];
      const size_t o = (size_t)c * ldo + b;
      if (lo) { const float h = rn_tf32_masked(x); hi[o] = h; lo[o] = rn_tf32_masked(x - h); }
      else hi[o] = x;
    }
  }
}
// ---- host side ---------------------------------------------------------------------------------------------------------------
template <bool X3, int S>
static int wt_launch_s(const WtArgs& args, dim3 grid, cudaStream_t st) {
  static bool attr_done = false;
  if (!attr_done) {
    cudaFuncSetAttribute(wide_tc_gemm_kernel<X3, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    attr_done = true;
  }
  wide_tc_gemm_kernel<X3, S><<<grid, kWtThreads, wt_smem_bytes<X3>(S), st>>>(args);
  return check_launch();
}
template <bool X3>
static int wt_launch(const WtArgs& args, int splits, cudaStream_t st) {
  constexpr int NT = WtCfg<X3>::NT;
  dim3 grid((args.M + 127) / 128, (args.N + NT - 1) / NT, splits);
  const bool one_wave = (long long)grid.x * grid.y * grid.z <= sm_count();
  if (WtCfg<X3>::kDeep != WtCfg<X3>::kShallow && !one_wave) return wt_launch_s<X3, WtCfg<X3>::kShallow>(args, grid, st);
  return wt_launch_s<X3, WtCfg<X3>::kDeep>(args, grid, st);
}
static int wt_run(const WtArgs& args, bool x3, cudaStream_t st, int splits = 1) {
  return x3 ? wt_launch<true>(args, splits, st) : wt_launch<false>(args, splits, st);
}

int wide_tc_fwd(const float* z, int B, int d, int nz, int H, const b200vae_icnn_params* p, int mode, float kappa, float* psi,
                float* xhat, float* h0, uint8_t* mask1, float* s2, float* g0, float* ws, const WideLayout& L, int precision,
                cudaStream_t st) {
  const bool x3 = precision == B200VAE_PREC_TF32X3;
  const int bn = wt_tile_n(x3);                         // rows of a B-operand TMA box = the kernel's tile width
  wide_tc_prepare_kernel<<<148 * 4, 256, 0, st>>>(p->W0, p->W1, p->A0w, p->A1w, d, H, mode, ws, L);
  int rc = check_launch();
  if (rc) return rc;
  const int kb = kKB;
  auto nkb = [&](int K) { return (K + kb - 1) / kb; };
  WtArgs a;
  memset(&a, 0, sizeof(a));
  // ---- lin: h0 = z A0^T + b0   (A0w is [H][d]; only its first nz columns meet non-zero inputs)
  rc = tma_map_2d(&a.a1, z, nz, B, nz, 128);
  if (!rc) rc = tma_map_2d(&a.b1hi, ws + L.A0hi, nz, H, d, wt_tile_n(true));
  if (!rc) rc = tma_map_2d(&a.b1lo, ws + L.A0lo, nz, H, d, wt_tile_n(true));
  if (rc) return rc;
  a.a2 = a.a1; a.b2hi = a.b1hi; a.b2lo = a.b1lo;
  a.nkb1 = nkb(nz); a.nkb2 = 0; a.xf1 = WT_XF_ID; a.M = B; a.N = H; a.epi = WT_EPI_LIN; a.bias = p->A0b; a.out0 = h0;
  rc = wt_run(a, true, st);     // always 3xTF32: K = nz is tiny, and h0 feeds a square (its error would be amplified)
  if (rc) return rc;
  // ---- hid: h1 = x1 P0^T + z A1^T + b1
  WtArgs b;
  memset(&b, 0, sizeof(b));
  rc = tma_map_2d(&b.a1, h0, H, B, H, 128);
  if (!rc) rc = tma_map_2d(&b.b1hi, ws + L.P0hi, H, H, H, bn);
  if (!rc) rc = tma_map_2d(&b.b1lo, ws + (x3 ? L.P0lo : L.P0hi), H, H, H, bn);
  if (!rc) rc = tma_map_2d(&b.b2hi, ws + L.A1hi, nz, H, d, bn);
  if (!rc) rc = tma_map_2d(&b.b2lo, ws + (x3 ? L.A1lo : L.A1hi), nz, H, d, bn);
  if (rc) return rc;
  b.a2 = a.a1;
  b.nkb1 = nkb(H); b.nkb2 = nkb(nz); b.xf1 = WT_XF_X1; b.M = B; b.N = H; b.epi = WT_EPI_HID; b.bias = p->A1b; b.P1 = ws + L.P1;
  b.out0 = ws + L.g1b; b.mask = mask1; b.part = ws + L.part; b.npart = ((H + bn - 1) / bn) * 2;
  rc = wt_run(b, x3, st);
  if (rc) return rc;
  rc = wide_row(ws + L.part, b.npart, z, p, B, nz, psi, s2, st);
  if (rc || !xhat) return rc;
  // ---- gx1: g0' = (g1b P0) * c0(h0)      B^T[k'][n] = P0[n][k'] = P0T
  WtArgs c;
  memset(&c, 0, sizeof(c));
  rc = tma_map_2d(&c.a1, ws + L.g1b, H, B, H, 128);
  if (!rc) rc = tma_map_2d(&c.b1hi, ws + L.P0Thi, H, H, H, bn);
  if (!rc) rc = tma_map_2d(&c.b1lo, ws + (x3 ? L.P0Tlo : L.P0Thi), H, H, H, bn);
  if (rc) return rc;
  c.a2 = c.a1; c.b2hi = c.b1hi; c.b2lo = c.b1lo;
  c.nkb1 = nkb(H); c.nkb2 = 0; c.xf1 = WT_XF_ID; c.M = B; c.N = H; c.epi = WT_EPI_GX1; c.h0 = h0; c.out0 = g0;
  rc = wt_run(c, x3, st);
  if (rc) return rc;
  // ---- out: xhat = s2 (g0' A0 + g1b A1 + A2) + 2 kappa z      B^T[c][n] = A*w[n][c] = A*wT  ([d][H])
  WtArgs e;
  memset(&e, 0, sizeof(e));
  rc = tma_map_2d(&e.a1, g0, H, B, H, 128);
  if (!rc) rc = tma_map_2d(&e.b1hi, ws + L.A0Thi, H, d, H, bn);
  if (!rc) rc = tma_map_2d(&e.b1lo, ws + (x3 ? L.A0Tlo : L.A0Thi), H, d, H, bn);
  if (!rc) rc = tma_map_2d(&e.b2hi, ws + L.A1Thi, H, d, H, bn);
  if (!rc) rc = tma_map_2d(&e.b2lo, ws + (x3 ? L.A1Tlo : L.A1Thi), H, d, H, bn);
  if (rc) return rc;
  e.a2 = c.a1;
  e.nkb1 = nkb(H); e.nkb2 = nkb(H); e.xf1 = WT_XF_ID; e.M = B; e.N = d; e.epi = WT_EPI_OUT; e.s2 = s2; e.A2w = p->A2w; e.z = z;
  e.nz = nz; e.kappa2 = 2.f * kappa; e.out0 = xhat;
  return wt_run(e, x3, st);
}

// Sample-stationary part of the backward (SURVEY Appendix A): u0, q1 -> w1 -> dP1;  gx1 -> g0, t0 -> db0;  dz.
// Leaves u0, q1, g0, t0 [B,H] filled for wide_tc_bwd_tn.  dW1 / db0 / dz may be null.
int wide_tc_bwd_rows(const float* v, const float* h0, const uint8_t* mask1, const float* s2, int B, int d, int nz, int H,
                     const b200vae_icnn_params* p, int mode, float kappa, float* dz, float* u0, float* q1, float* g0, float* t0,
                     float* dW1, float* db0, float* ws, const WideLayout& L, int precision, cudaStream_t st) {
  const bool x3 = precision == B200VAE_PREC_TF32X3;
  const int bn = wt_tile_n(x3);                         // rows of a B-operand TMA box = the kernel's tile width
  wide_tc_prepare_kernel<<<148 * 4, 256, 0, st>>>(p->W0, p->W1, p->A0w, p->A1w, d, H, mode, ws, L);
  int rc = check_launch();
  if (rc) return rc;
  wide_tc_g1b_kernel<<<148 * 8, 256, 0, st>>>(mask1, ws + L.P1, (size_t)B * H, H, ws + L.g1b);
  rc = check_launch();
  if (rc) return rc;
  auto nkb = [&](int K) { return (K + kKB - 1) / kKB; };
  const dim3 cgrid(L.mt, (H + 255) / 256);
  const int chain = mode == B200VAE_WEIGHT_EXP ? 1 : 2;
  // ---- u0 = v A0^T, q1 = u0 * c0
  WtArgs a;
  memset(&a, 0, sizeof(a));
  rc = tma_map_2d(&a.a1, v, d, B, d, 128);
  if (!rc) rc = tma_map_2d(&a.b1hi, ws + L.A0hi, d, H, d, bn);
  if (!rc) rc = tma_map_2d(&a.b1lo, ws + (x3 ? L.A0lo : L.A0hi), d, H, d, bn);
  if (rc) return rc;
  a.a2 = a.a1; a.b2hi = a.b1hi; a.b2lo = a.b1lo;
  a.nkb1 = nkb(d); a.nkb2 = 0; a.xf1 = WT_XF_ID; a.M = B; a.N = H; a.epi = WT_EPI_U; a.h0 = h0; a.out0 = u0; a.out1 = q1;
  rc = wt_run(a, x3, st);
  if (rc) return rc;
  // ---- e1 = s2 s1 (q1 P0^T + v A1^T)  -> column sums = dP1   (e1 parked in the g0 buffer)
  WtArgs b;
  memset(&b, 0, sizeof(b));
  rc = tma_map_2d(&b.a1, q1, H, B, H, 128);
  if (!rc) rc = tma_map_2d(&b.b1hi, ws + L.P0hi, H, H, H, bn);
  if (!rc) rc = tma_map_2d(&b.b1lo, ws + (x3 ? L.P0lo : L.P0hi), H, H, H, bn);
  if (!rc) rc = tma_map_2d(&b.b2hi, ws + L.A1hi, d, H, d, bn);
  if (!rc) rc = tma_map_2d(&b.b2lo, ws + (x3 ? L.A1lo : L.A1hi), d, H, d, bn);
  if (rc) return rc;
  b.a2 = a.a1;
  b.nkb1 = nkb(H); b.nkb2 = nkb(d); b.xf1 = WT_XF_ID; b.M = B; b.N = H; b.epi = WT_EPI_W1; b.s2 = s2;
  b.mask = const_cast<uint8_t*>(mask1); b.out0 = g0;
  rc = wt_run(b, x3, st);
  if (rc) return rc;
  if (dW1) {
    wide_tc_colsum_kernel<<<cgrid, 256, 0, st>>>(g0, B, H, ws + L.colpart);
    rc = check_launch();
    if (!rc) rc = wide_col_finalize(ws + L.colpart, L.mt, H, chain, ws + L.P1, p->W1, dW1, st);
    if (rc) return rc;
  }
  // ---- gx1 = s2 (g1b P0) -> g0, t0
  WtArgs c;
  memset(&c, 0, sizeof(c));
  rc = tma_map_2d(&c.a1, ws + L.g1b, H, B, H, 128);
  if (!rc) rc = tma_map_2d(&c.b1hi, ws + L.P0Thi, H, H, H, bn);
  if (!rc) rc = tma_map_2d(&c.b1lo, ws + (x3 ? L.P0Tlo : L.P0Thi), H, H, H, bn);
  if (rc) return rc;
  c.a2 = c.a1; c.b2hi = c.b1hi; c.b2lo = c.b1lo;
  c.nkb1 = nkb(H); c.nkb2 = 0; c.xf1 = WT_XF_ID; c.M = B; c.N = H; c.epi = WT_EPI_GXB; c.h0 = h0; c.u0 = u0; c.s2 = s2;
  c.out0 = g0; c.out1 = t0;
  rc = wt_run(c, x3, st);
  if (rc) return rc;
  if (db0) {
    wide_tc_colsum_kernel<<<cgrid, 256, 0, st>>>(t0, B, H, ws + L.colpart);
    rc = check_launch();
    if (!rc) rc = wide_col_finalize(ws + L.colpart, L.mt, H, 0, nullptr, nullptr, db0, st);
    if (rc) return rc;
  }
  if (!dz) return B200VAE_OK;
  // ---- dz [B,nz] = t0 A0[:, :nz] + 2 kappa v[:, :nz]
  WtArgs e;
  memset(&e, 0, sizeof(e));
  rc = tma_map_2d(&e.a1, t0, H, B, H, 128);
  if (!rc) rc = tma_map_2d(&e.b1hi, ws + L.A0Thi, H, nz, H, bn);
  if (!rc) rc = tma_map_2d(&e.b1lo, ws + (x3 ? L.A0Tlo : L.A0Thi), H, nz, H, bn);
  if (rc) return rc;
  e.a2 = e.a1; e.b2hi = e.b1hi; e.b2lo = e.b1lo;
  e.nkb1 = nkb(H); e.nkb2 = 0; e.xf1 = WT_XF_ID; e.M = B; e.N = nz; e.epi = WT_EPI_DZ; e.v = v; e.ldv = d; e.kappa2 = 2.f * kappa;
  e.out0 = dz;
  return wt_run(e, x3, st);
}

// Batch-reduction GEMMs of the backward on tcgen05:  dA0 = g0^T v + t0^T z,  dA1 = g1^T v,  dP0 = g1^T q1 (-> dW0).
// The operands are transposed first (batch -> contiguous K; B operands split hi/lo on the way), then each product is the
// generic GEMM with M = H, K = B, split over K into L.splits slabs that are summed in fixed order.
int wide_tc_bwd_tn(const float* z, const float* v, const uint8_t* mask1, const float* s2, const float* q1, const float* g0,
                   const float* t0, int B, int d, int nz, int H, const b200vae_icnn_params* p, int mode, float* dA0w, float* dA1w,
                   float* dW0, float* ws, const WideLayout& L, int precision, cudaStream_t st) {
  const bool x3 = precision == B200VAE_PREC_TF32X3;
  const int ldb = L.ldb, bn = wt_tile_n(x3);
  int rc;
  auto transpose = [&](const float* src, int md, int C, float* hi, float* lo) {
    dim3 grid((B + 31) / 32, (C + 31) / 32);
    wide_tc_transpose_kernel<<<grid, 256, 0, st>>>(src, mask1, s2, ws + L.P1, md, B, C, ldb, hi, lo);
    return check_launch();
  };
  const int nkb_all = (B + kKB - 1) / kKB, per = (nkb_all + L.splits - 1) / L.splits;
  const int chain = mode == B200VAE_WEIGHT_EXP ? 1 : 2;
  auto gemm = [&](const float* At, const float* Bhi, const float* Blo, int N, const float* At2, const float* B2hi,
                  const float* B2lo, int N2) {
    WtArgs a;
    memset(&a, 0, sizeof(a));
    int r = tma_map_2d(&a.a1, At, B, H, ldb, 128);
    if (!r) r = tma_map_2d(&a.b1hi, Bhi, B, N, ldb, bn);
    if (!r) r = tma_map_2d(&a.b1lo, x3 ? Blo : Bhi, B, N, ldb, bn);
    if (!r && At2) {
      r = tma_map_2d(&a.a2, At2, B, H, ldb, 128);
      if (!r) r = tma_map_2d(&a.b2hi, B2hi, B, N2, ldb, bn);
      if (!r) r = tma_map_2d(&a.b2lo, x3 ? B2lo : B2hi, B, N2, ldb, bn);
    } else if (!r) {
      a.a2 = a.a1; a.b2hi = a.b1hi; a.b2lo = a.b1lo;
    }
    if (r) return r;
    a.nkb1 = per; a.nkb2 = At2 ? per : 0; a.xf1 = WT_XF_ID; a.M = H; a.N = N; a.epi = WT_EPI_SLAB; a.out0 = ws + L.slabs;
    a.kb_per_split = per;
    return wt_run(a, x3, st, L.splits);
  };
  auto finalize = [&](size_t n, int ch, const float* W, float* out) {
    return wide_slab_finalize(ws + L.slabs, L.splits, n, ch, W, out, st);
  };
  if (dA0w || dA1w) { rc = transpose(v, 0, d, ws + L.vThi, x3 ? ws + L.vTlo : nullptr); if (rc) return rc; }
  if (dA1w || dW0) { rc = transpose(nullptr, 1, H, ws + L.g1T, nullptr); if (rc) return rc; }
  if (dA0w) {
    rc = transpose(g0, 0, H, ws + L.g0T, nullptr); if (rc) return rc;
    rc = transpose(t0, 0, H, ws + L.t0T, nullptr); if (rc) return rc;
    rc = transpose(z, 0, nz, ws + L.zThi, x3 ? ws + L.zTlo : nullptr); if (rc) return rc;
    rc = gemm(ws + L.g0T, ws + L.vThi, ws + L.vTlo, d, ws + L.t0T, ws + L.zThi, ws + L.zTlo, nz); if (rc) return rc;
    rc = finalize((size_t)H * d, 0, nullptr, dA0w); if (rc) return rc;
  }
  if (dA1w) {
    rc = gemm(ws + L.g1T, ws + L.vThi, ws + L.vTlo, d, nullptr, nullptr, nullptr, 0); if (rc) return rc;
    rc = finalize((size_t)H * d, 0, nullptr, dA1w); if (rc) return rc;
  }
  if (dW0) {
    rc = transpose(q1, 0, H, ws + L.q1Thi, x3 ? ws + L.q1Tlo : nullptr); if (rc) return rc;
    rc = gemm(ws + L.g1T, ws + L.q1Thi, ws + L.q1Tlo, H, nullptr, nullptr, nullptr, 0); if (rc) return rc;
    rc = finalize((size_t)H * H, chain, p->W0, dW0); if (rc) return rc;
  }
  return B200VAE_OK;
}

}  // namespace b200vae
