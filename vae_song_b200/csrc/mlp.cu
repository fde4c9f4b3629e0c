// mlp.cu -- fused [Linear -> BatchNorm1d -> LeakyReLU] encoder stack (SURVEY.md section 8(f) rank 1).
//
// The reference's 1-D encoders (model.py:711-734 LIDVAE.make_encoder_1d, model.py:186-208 FlexibleVAE MLP) are chains
// of narrow (width <= 128) Linear+BN+LeakyReLU(0.01) blocks: in eager PyTorch each block is ~6 launches forward and ~8
// backward on [B, w] tensors (cuBLAS picks split-K sgemm kernels for the [B,2]x[2,2] products).  Here one layer is
//   forward : y = act(prev) W^T + b   with act = LeakyReLU(BN(prev)) applied while loading, per-column (count, mean, M2)
//             partials per CTA (Chan-combined in fixed order -> deterministic batch statistics);
//   backward: (1) dyhat = da * lrelu'(.) + per-column sums S1 = sum dyhat, S2 = sum dyhat*xhat,
//             (2) da_prev = dy W  and  dW = dy^T act(prev)  with dy = gamma*invstd*(dyhat - S1/N - xhat*S2/N) formed on
//                 the fly, both on the 128x128x16 FP32 tile core (gemm_simt.cuh).
// Everything but y / dyhat / da stays on chip; cross-rank BatchNorm only needs the tiny (count,mean,M2) / (S1,S2)
// vectors exchanged: the *_peer finalize kernels publish them straight into the other GPUs' memory over NVLink and
// combine in rank order (peer.cuh), so a sharded step has no NCCL call and no torch glue per BatchNorm layer.
#include <string.h>

#include "gemm_simt.cuh"
#include "peer.cuh"

namespace b200vae {

struct ActSrc {          // how a layer input a[b][k] is obtained from the previous layer's pre-BN output
  const float* y;        // [B, w]
  const float* mean;     // [w]; nullptr => identity (raw network input)
  const float* invstd;
  const float* gamma;
  const float* beta;
  int w;
  float slope;
};

__host__ __device__ __forceinline__ ActSrc make_src(const float* y, const float* stats, const float* gamma,
                                                    const float* beta, int w, float slope) {
  ActSrc s;
  s.y = y; s.w = w; s.slope = slope;
  s.mean = stats; s.invstd = stats ? stats + 2 * w : nullptr; s.gamma = gamma; s.beta = beta;
  return s;
}

struct ActSmem {
  float mean[128], invstd[128], gamma[128], beta[128];
  __device__ __forceinline__ void load(const ActSrc& s) {
    if (s.mean && threadIdx.x < 128) {
      const int k = threadIdx.x;
      const bool in = k < s.w;
      mean[k] = in ? s.mean[k] : 0.f; invstd[k] = in ? s.invstd[k] : 0.f;
      gamma[k] = in ? s.gamma[k] : 0.f; beta[k] = in ? s.beta[k] : 0.f;
    }
  }
  __device__ __forceinline__ float xhat(float yv, int k) const { return (yv - mean[k]) * invstd[k]; }
  __device__ __forceinline__ float act(bool has_bn, float slope, float yv, int k) const {
    if (!has_bn) return yv;
    const float t = fmaf(xhat(yv, k), gamma[k], beta[k]);
    return t > 0.f ? t : slope * t;
  }
};

// A tile from activations: As[kk][m] = act(prev[m0+m][k0+kk])
// (pre() only issues the global loads; post() -- after the FMA block of the previous K-step -- finishes and stores)
struct AGenAct {
  ActSrc s; const ActSmem* sm; int m0, B;
  float r[8];
  __device__ __forceinline__ void pre(int kt, float (*)[kBM]) {
    const int m = threadIdx.x & 127, kg = threadIdx.x >> 7, row = m0 + m;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = kt * kBK + kg * 8 + e;
      r[e] = (row < B && k < s.w) ? __ldg(s.y + (size_t)row * s.w + k) : 0.f;
    }
  }
  __device__ __forceinline__ void post(int kt, float (*As)[kBM]) {
    const int m = threadIdx.x & 127, kg = threadIdx.x >> 7, row = m0 + m;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = kt * kBK + kg * 8 + e;
      As[kg * 8 + e][m] = (row < B && k < s.w) ? sm->act(s.mean != nullptr, s.slope, r[e], k) : 0.f;
    }
  }
};
// B tile from a small row-major weight: Bs[kk][n] = W[n][k0+kk] (transposed read) or W[k0+kk][n] (direct)
template <bool kTransposed>
struct BGenW {
  const float* W; int rows, cols;     // W is [rows][cols]
  __device__ __forceinline__ void post(int, float (*)[kBN]) {}
  __device__ __forceinline__ void pre(int kt, float (*Bs)[kBN]) {
    const int n = threadIdx.x & 127, kg = threadIdx.x >> 7;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = kt * kBK + kg * 8 + e;
      float v = 0.f;
      if (kTransposed) { if (n < rows && k < cols) v = __ldg(W + (size_t)n * cols + k); }
      else             { if (k < rows && n < cols) v = __ldg(W + (size_t)k * cols + n); }
      Bs[kg * 8 + e][n] = v;
    }
  }
};

// ----------------------------------------------------------------------------------------- fused finalize ("last block")
// Single-GPU layers fold the finalize step into the producing kernel: every CTA publishes its ordered partials, takes a
// ticket, and the CTA that draws the last ticket combines ALL partials -- in the same fixed order as the stand-alone
// finalize kernels, so the results stay bit-reproducible -- instead of a second launch per layer (the encoder of BASELINE
// configs[1] went from 42 to 25 launches per step, the 8-layer encoder of configs[2] from 56 to 33).  The ticket lives at
// the end of the caller's scratch (b200vae_mlp_scratch_bytes): zero before the first call, reset by the last block.  The
// cross-rank (peer) layers keep their own finalize kernel: it is the one that talks to the other GPUs.
__device__ __forceinline__ bool last_block_arrives(unsigned* ticket) {
  __shared__ int s_last;
  __threadfence();                               // this thread's partials are visible device-wide
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(ticket, 1u);
    s_last = (t + 1u == gridDim.x) ? 1 : 0;
    if (s_last) *ticket = 0u;                    // everyone has drawn: ready for the next launch
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last != 0;
}
// `peer` != 0: the last CTA also runs the cross-rank exchange (peer.cuh) -- publishes this rank's per-column values to every
// GPU, waits for theirs and combines in rank order -- so a sharded layer needs no finalize launch either.  `stage`: global
// staging for the exchange ([128*3] mine + [world][128*3] all, part of the caller's scratch).
struct StatsFin {      // stats == nullptr: no fused finalize (a finalize kernel follows)
  float* stats; float* running_mean; float* running_var; float eps, momentum; unsigned* ticket;
  int peer, slot; float* stage; PeerComm comm;
};
struct SumsFin { float* sums; unsigned* ticket; int peer, slot; float* sums_global; float* stage; PeerComm comm; };
struct DwFin { float* dW; unsigned* ticket; };

// The merged (count, mean, M2) of column n -> stats[4][w] = mean, biased var, invstd, count, and (with running_mean) the
// momentum update of the running statistics.  The update is written with explicit roundings: left to the compiler, the
// products were contracted into an FMA differently depending on the kernel this is inlined into.
__device__ __forceinline__ void stats_store(const StatsFin& f, int w, int n, float cnt, float mean, float m2) {
  const float var = m2 / cnt;
  f.stats[n] = mean; f.stats[w + n] = var; f.stats[2 * w + n] = rsqrtf(var + f.eps); f.stats[3 * w + n] = cnt;
  if (f.running_mean) {
    const float keep = __fsub_rn(1.f, f.momentum);
    f.running_mean[n] = __fmaf_rn(f.momentum, mean, __fmul_rn(keep, f.running_mean[n]));
    f.running_var[n] = __fmaf_rn(f.momentum, m2 / fmaxf(cnt - 1.f, 1.f), __fmul_rn(keep, f.running_var[n]));
  }
}

// ----------------------------------------------------------------------------------------- forward
// part: [nCTA][128][3] = (count, mean, M2) of this CTA's rows per output column
__device__ __forceinline__ void chan_merge(float& cnt, float& mean, float& m2, float nb, float mb, float m2b);
__device__ __forceinline__ void stats_finalize_block(const float* __restrict__ part, int ncta, int w, const StatsFin& f);

__global__ void __launch_bounds__(kThreads, 2)
mlp_fwd_kernel(ActSrc src, const float* __restrict__ W, const float* __restrict__ bias, int B, int wo,
               float* __restrict__ y_out, float* __restrict__ part, int do_stats, StatsFin fin) {
  __shared__ GemmSmem gs;
  __shared__ ActSmem am;
  const TileCoord tc;
  const int m0 = blockIdx.x * kBM;
  am.load(src);
  __syncthreads();
  AGenAct ag{src, &am, m0, B};
  BGenW<true> bg{W, wo, src.w};
  float acc[8][8];
  gemm_tile(acc, gs, (src.w + kBK - 1) / kBK, ag, bg, tc);
  const int nvalid = min(kBM, B - m0);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int n = tc.col(j);
    const float bj = (n < wo && bias) ? bias[n] : 0.f;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = m0 + tc.row(i);
      const float yv = acc[i][j] + bj;
      acc[i][j] = yv;
      if (row < B && n < wo) { y_out[(size_t)row * wo + n] = yv; s += yv; }
    }
    if (do_stats) {
      s = colsum16(s);
      const float mean_c = s / (float)nvalid;
      float m2 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float dlt = acc[i][j] - mean_c;
        if (m0 + tc.row(i) < B) m2 = fmaf(dlt, dlt, m2);
      }
      m2 = colsum16(m2);
      if (tc.ty == 0 && n < wo) {
        float* o = part + ((size_t)blockIdx.x * 128 + n) * 3;
        o[0] = (float)nvalid; o[1] = mean_c; o[2] = m2;
      }
    }
  }
  if (do_stats && fin.stats && last_block_arrives(fin.ticket)) stats_finalize_block(part, (int)gridDim.x, wo, fin);
}

// Chan et al. combination of the per-CTA (count, mean, M2): one WARP per column, lanes stride over the CTAs (independent
// loads in flight), then a fixed-order shuffle tree -> deterministic.  stats: [4][w] = mean, biased var, invstd, count
__device__ __forceinline__ void chan_merge(float& cnt, float& mean, float& m2, float nb, float mb, float m2b) {
  const float tot = cnt + nb;
  if (tot > 0.f) {
    const float dlt = mb - mean;
    mean += dlt * (nb / tot);
    m2 += m2b + dlt * dlt * (cnt * nb / tot);
  }
  cnt = tot;
}
// the fixed-order shuffle tree: lane 0 ends with the merge of the warp's 32 triples
__device__ __forceinline__ void chan_warp_merge(float& cnt, float& mean, float& m2) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const float nb = __shfl_down_sync(0xffffffffu, cnt, off), mb = __shfl_down_sync(0xffffffffu, mean, off),
                m2b = __shfl_down_sync(0xffffffffu, m2, off);
    chan_merge(cnt, mean, m2, nb, mb, m2b);
  }
}
// column n by one warp: lanes stride over the CTAs' partials (L2 loads), fixed-order shuffle tree
__device__ __forceinline__ void stats_finalize_column(const float* __restrict__ part, int ncta, int w, int n,
                                                      const StatsFin& f) {
  const int lane = threadIdx.x & 31;
  float cnt = 0.f, mean = 0.f, m2 = 0.f;
  for (int c0 = lane; c0 < ncta; c0 += 4 * 32) {   // 4 partial triples per lane in flight per L2 round trip, merged in order
    float pc[4], pm[4], pq[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + 32 * j;
      const bool in = c < ncta;
      const float* p = part + ((size_t)(in ? c : c0) * 128 + n) * 3;
      pc[j] = in ? __ldcg(p) : 0.f; pm[j] = in ? __ldcg(p + 1) : 0.f; pq[j] = in ? __ldcg(p + 2) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) chan_merge(cnt, mean, m2, pc[j], pm[j], pq[j]);     // a zero count is the identity
  }
  chan_warp_merge(cnt, mean, m2);
  if (lane == 0) stats_store(f, w, n, cnt, mean, m2);
}
__global__ void __launch_bounds__(256)
mlp_stats_finalize_kernel(const float* __restrict__ part, int ncta, int w, StatsFin fin) {
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (n >= w) return;
  stats_finalize_column(part, ncta, w, n, fin);
}
// the same, executed by ONE CTA (all its warps, columns round-robin): the last CTA of the producing kernel, or the
// stand-alone cross-rank finalize below
__device__ __forceinline__ void stats_finalize_block(const float* __restrict__ part, int ncta, int w, const StatsFin& f) {
  if (f.peer) {                // cross-rank: local (count, mean, M2) per column -> exchange -> Chan merge in rank order
    float* mine = f.stage;
    float* all = f.stage + 3 * 128;
    const int lane = threadIdx.x & 31;
    for (int n = threadIdx.x >> 5; n < w; n += (int)(blockDim.x >> 5)) {
      float cnt = 0.f, mean = 0.f, m2 = 0.f;
      for (int c = lane; c < ncta; c += 32) {
        const float* p = part + ((size_t)c * 128 + n) * 3;
        chan_merge(cnt, mean, m2, __ldcg(p), __ldcg(p + 1), __ldcg(p + 2));
      }
      chan_warp_merge(cnt, mean, m2);
      if (lane == 0) { mine[n] = cnt; mine[w + n] = mean; mine[2 * w + n] = m2; }
    }
    __syncthreads();
    peer_exchange(f.comm, f.slot, mine, 3 * w, all);
    for (int n = threadIdx.x; n < w; n += (int)blockDim.x) {
      float cnt = 0.f, mean = 0.f, m2 = 0.f;
      for (int r = 0; r < f.comm.world; ++r) {
        const float* a = all + (size_t)r * 3 * w;
        chan_merge(cnt, mean, m2, a[n], a[w + n], a[2 * w + n]);
      }
      stats_store(f, w, n, cnt, mean, m2);
    }
    return;
  }
  if (ncta <= 64) {            // few partials (small batches): a THREAD per column, partials merged in CTA order
    for (int n = threadIdx.x; n < w; n += (int)blockDim.x) {
      float cnt = 0.f, mean = 0.f, m2 = 0.f;
      for (int c0 = 0; c0 < ncta; c0 += 8) {       // 8 partial triples in flight per L2 round trip, merged in CTA order
        float pc[8], pm[8], pq[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const bool in = c0 + j < ncta;
          const float* p = part + ((size_t)(in ? c0 + j : c0) * 128 + n) * 3;
          pc[j] = in ? __ldcg(p) : 0.f; pm[j] = in ? __ldcg(p + 1) : 0.f; pq[j] = in ? __ldcg(p + 2) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) chan_merge(cnt, mean, m2, pc[j], pm[j], pq[j]);   // a zero count is the identity
      }
      stats_store(f, w, n, cnt, mean, m2);
    }
    return;
  }
  for (int n = threadIdx.x >> 5; n < w; n += (int)(blockDim.x >> 5)) stats_finalize_column(part, ncta, w, n, f);
}

// Cross-rank finalize when it is not fused into the producing kernel: ONE CTA of 32 warps, staging in f.stage.
__global__ void __launch_bounds__(1024)
mlp_stats_finalize_peer_kernel(const float* __restrict__ part, int ncta, int w, StatsFin fin) {
  stats_finalize_block(part, ncta, w, fin);
}

// column n of the (S1, S2) sums by one warp (lanes stride over the blocks' partials, fixed shuffle tree)
__device__ __forceinline__ void sums_finalize_column(const float* __restrict__ part, int nblk, int w, int n,
                                                     float* __restrict__ sums /*[2][w]*/) {
  const int lane = threadIdx.x & 31;
  float a = 0.f, b = 0.f;
#pragma unroll 4
  for (int c = lane; c < nblk; c += 32) {          // unrolled: four float2 loads per lane go out together
    const float2 t = __ldcg(reinterpret_cast<const float2*>(part + ((size_t)c * 128 + n) * 2));
    a += t.x; b += t.y;
  }
  a = warp_sum(a); b = warp_sum(b);
  if (lane == 0) { sums[n] = a; sums[w + n] = b; }
}

// ----------------------------------------------------------------------------------------- backward (1): reduce
// dyhat = da * lrelu'(gamma*xhat+beta) ; S1 = sum dyhat ; S2 = sum dyhat*xhat.  w must divide 256 (power of two <= 128).
__global__ void __launch_bounds__(256)
mlp_bwd_reduce_kernel(const float* __restrict__ da, ActSrc cur, int has_bn, long long n_elem, long long per_block,
                      float* __restrict__ dyhat, float* __restrict__ part /*[nblk][128][2]*/, SumsFin fin) {
  __shared__ ActSmem am;
  __shared__ float red[256][2];
  am.load(cur);
  __syncthreads();
  const int w = cur.w, n = threadIdx.x % w;
  const long long e0 = (long long)blockIdx.x * per_block, e1 = min(n_elem, e0 + per_block);
  float s1 = 0.f, s2 = 0.f;
  for (long long i = e0 + threadIdx.x; i < e1; i += 256) {
    float g = da[i];
    if (has_bn) {
      const float xh = am.xhat(cur.y[i], n);
      const float t = fmaf(xh, am.gamma[n], am.beta[n]);
      g = t > 0.f ? g : cur.slope * g;
      s2 = fmaf(g, xh, s2);
    }
    s1 += g;
    dyhat[i] = g;
  }
  red[threadIdx.x][0] = s1; red[threadIdx.x][1] = s2;
  __syncthreads();
  if (threadIdx.x < w) {
    float a = 0.f, b = 0.f;
    for (int t = threadIdx.x; t < 256; t += w) { a += red[t][0]; b += red[t][1]; }
    part[((size_t)blockIdx.x * 128 + threadIdx.x) * 2 + 0] = a;
    part[((size_t)blockIdx.x * 128 + threadIdx.x) * 2 + 1] = b;
  }
  if (fin.peer && last_block_arrives(fin.ticket)) {       // cross-rank: local sums -> exchange -> rank-ordered global sums
    const int nblk = (int)gridDim.x, lane = threadIdx.x & 31;
    float* mine = fin.stage;
    float* all = fin.stage + 2 * 128;
    for (int n = threadIdx.x >> 5; n < w; n += 8) {
      float a = 0.f, b = 0.f;
      for (int c = lane; c < nblk; c += 32) { a += __ldcg(part + ((size_t)c * 128 + n) * 2); b += __ldcg(part + ((size_t)c * 128 + n) * 2 + 1); }
      a = warp_sum(a); b = warp_sum(b);
      if (lane == 0) { mine[n] = a; mine[w + n] = b; }
    }
    __syncthreads();
    peer_exchange(fin.comm, fin.slot, mine, 2 * w, all);
    for (int i = threadIdx.x; i < 2 * w; i += 256) {
      float sacc = 0.f;
      for (int r = 0; r < fin.comm.world; ++r) sacc += all[(size_t)r * 2 * w + i];
      fin.sums_global[i] = sacc;
      if (fin.sums) fin.sums[i] = mine[i];
    }
  } else if (!fin.peer && last_block_arrives(fin.ticket)) {
    const int nblk = (int)gridDim.x;
    if (nblk <= 64) {          // few partials: a thread per column, block order
      if (threadIdx.x < w) {
        float a = 0.f, b = 0.f;
        for (int c = 0; c < nblk; ++c) {
          a += __ldcg(part + ((size_t)c * 128 + threadIdx.x) * 2);
          b += __ldcg(part + ((size_t)c * 128 + threadIdx.x) * 2 + 1);
        }
        fin.sums[threadIdx.x] = a; fin.sums[w + threadIdx.x] = b;
      }
    } else {
      for (int n = threadIdx.x >> 5; n < w; n += 8) sums_finalize_column(part, nblk, w, n, fin.sums);
    }
  }
}

// dy[b][o] formed on the fly from dyhat, y, stats and the (global) sums
struct DyCtx {
  const float* dyhat; ActSrc cur; const float* sums; float invN; int has_bn;
  __device__ __forceinline__ void fetch(long long idx, float& g, float& yv) const {
    g = __ldg(dyhat + idx);
    yv = has_bn ? __ldg(cur.y + idx) : 0.f;
  }
  __device__ __forceinline__ float dy(const ActSmem& am, const float* s1, const float* s2, float g, float yv, int o) const {
    if (!has_bn) return g;
    const float xh = am.xhat(yv, o);
    return am.gamma[o] * am.invstd[o] * (g - s1[o] * invN - xh * (s2[o] * invN));
  }
};

// ----------------------------------------------------------------------------------------- backward (2a): da_prev = dy W
struct AGenDy {
  DyCtx c; const ActSmem* am; const float* s1; const float* s2; int m0, B;
  float g[8], yv[8];
  __device__ __forceinline__ void pre(int kt, float (*)[kBM]) {
    const int m = threadIdx.x & 127, kg = threadIdx.x >> 7, row = m0 + m, wo = c.cur.w;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int o = kt * kBK + kg * 8 + e;
      g[e] = 0.f; yv[e] = 0.f;
      if (row < B && o < wo) c.fetch((long long)row * wo + o, g[e], yv[e]);
    }
  }
  __device__ __forceinline__ void post(int kt, float (*As)[kBM]) {
    const int m = threadIdx.x & 127, kg = threadIdx.x >> 7, row = m0 + m, wo = c.cur.w;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int o = kt * kBK + kg * 8 + e;
      As[kg * 8 + e][m] = (row < B && o < wo) ? c.dy(*am, s1, s2, g[e], yv[e], o) : 0.f;
    }
  }
};
__global__ void __launch_bounds__(kThreads, 2)
mlp_bwd_gemm_kernel(DyCtx c, const float* __restrict__ W /*[wo][wi]*/, int B, int wi, float* __restrict__ da_prev) {
  __shared__ GemmSmem gs;
  __shared__ ActSmem am;
  __shared__ float s1[128], s2[128];
  const TileCoord tc;
  const int m0 = blockIdx.x * kBM, wo = c.cur.w;
  am.load(c.cur);
  if (threadIdx.x < 128) {
    s1[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[threadIdx.x] : 0.f;
    s2[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[wo + threadIdx.x] : 0.f;
  }
  __syncthreads();
  AGenDy ag{c, &am, s1, s2, m0, B};
  BGenW<false> bg{W, wo, wi};
  float acc[8][8];
  gemm_tile(acc, gs, (wo + kBK - 1) / kBK, ag, bg, tc);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = m0 + tc.row(i);
    if (row >= B) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = tc.col(j);
      if (n < wi) da_prev[(size_t)row * wi + n] = acc[i][j];
    }
  }
}

// ----------------------------------------------------------------------------------------- backward (2b): dW = dy^T act(prev)
struct AGenDyT {   // As[kk = sample][m = o]
  DyCtx c; const ActSmem* am; const float* s1; const float* s2; int b0, b1;
  float g[8], yv[8];
  __device__ __forceinline__ void pre(int kt, float (*)[kBM]) {
    const int o = threadIdx.x & 127, kg = threadIdx.x >> 7, wo = c.cur.w;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int b = b0 + kt * kBK + kg * 8 + e;
      g[e] = 0.f; yv[e] = 0.f;
      if (b < b1 && o < wo) c.fetch((long long)b * wo + o, g[e], yv[e]);
    }
  }
  __device__ __forceinline__ void post(int kt, float (*As)[kBM]) {
    const int o = threadIdx.x & 127, kg = threadIdx.x >> 7, wo = c.cur.w;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int b = b0 + kt * kBK + kg * 8 + e;
      As[kg * 8 + e][o] = (b < b1 && o < wo) ? c.dy(*am, s1, s2, g[e], yv[e], o) : 0.f;
    }
  }
};
struct BGenActT {  // Bs[kk = sample][n = i]
  ActSrc s; const ActSmem* sm; int b0, b1;
  float r[8];
  __device__ __forceinline__ void pre(int kt, float (*)[kBN]) {
    const int i = threadIdx.x & 127, kg = threadIdx.x >> 7;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int b = b0 + kt * kBK + kg * 8 + e;
      r[e] = (b < b1 && i < s.w) ? __ldg(s.y + (size_t)b * s.w + i) : 0.f;
    }
  }
  __device__ __forceinline__ void post(int kt, float (*Bs)[kBN]) {
    const int i = threadIdx.x & 127, kg = threadIdx.x >> 7;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int b = b0 + kt * kBK + kg * 8 + e;
      Bs[kg * 8 + e][i] = (b < b1 && i < s.w) ? sm->act(s.mean != nullptr, s.slope, r[e], i) : 0.f;
    }
  }
};
__device__ __forceinline__ void dw_finalize_block(const float* __restrict__ part, int nsplit, int n, float* __restrict__ dW);
__global__ void __launch_bounds__(kThreads, 2)
mlp_bwd_dw_kernel(DyCtx c, ActSrc prev, int B, int rows_per_split, float* __restrict__ part /*[nsplit][wo][wi]*/, DwFin fin) {
  __shared__ GemmSmem gs;
  __shared__ ActSmem am, pm;
  __shared__ float s1[128], s2[128];
  const TileCoord tc;
  const int wo = c.cur.w, wi = prev.w;
  am.load(c.cur);
  pm.load(prev);
  if (threadIdx.x < 128) {
    s1[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[threadIdx.x] : 0.f;
    s2[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[wo + threadIdx.x] : 0.f;
  }
  __syncthreads();
  const int b0 = blockIdx.x * rows_per_split, b1 = min(B, b0 + rows_per_split);
  AGenDyT ag{c, &am, s1, s2, b0, b1};
  BGenActT bg{prev, &pm, b0, b1};
  float acc[8][8];
  gemm_tile(acc, gs, (max(b1 - b0, 0) + kBK - 1) / kBK, ag, bg, tc);
  float* out = part + (size_t)blockIdx.x * wo * wi;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int o = tc.row(i);
    if (o >= wo) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = tc.col(j);
      if (n < wi) out[(size_t)o * wi + n] = acc[i][j];
    }
  }
  if (fin.dW && last_block_arrives(fin.ticket)) dw_finalize_block(part, (int)gridDim.x, wo * wi, fin.dW);
}
__device__ __forceinline__ void dw_finalize_elem(const float* __restrict__ part, int nsplit, int n, int i, float* __restrict__ dW) {
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int c = lane; c < nsplit; c += 32) s += __ldcg(part + (size_t)c * n + i);
  s = warp_sum(s);
  if (lane == 0) dW[i] = s;
}
// all n elements by ONE CTA (the last block of the producing kernel): few partials -> a thread per element (coalesced
// over e), many partials -> a warp per element
__device__ __forceinline__ void dw_finalize_block(const float* __restrict__ part, int nsplit, int n, float* __restrict__ dW) {
  if (nsplit <= 32) {
    for (int e = threadIdx.x; e < n; e += (int)blockDim.x) {
      float s = 0.f;
#pragma unroll 8
      for (int c = 0; c < nsplit; ++c) s += __ldcg(part + (size_t)c * n + e);     // unrolled: the loads go out together
      dW[e] = s;
    }
  } else {
    for (int e = threadIdx.x >> 5; e < n; e += (int)(blockDim.x >> 5)) dw_finalize_elem(part, nsplit, n, e, dW);
  }
}
__global__ void __launch_bounds__(256)
mlp_dw_finalize_kernel(const float* __restrict__ part, int nsplit, int n, float* __restrict__ dW) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= n) return;
  dw_finalize_elem(part, nsplit, n, i, dW);
}

// ----------------------------------------------------------------------------------------- narrow layers (w <= 8)
// The default LID-VAE encoder is 2-2-2-2-2-4-4 wide: a 128x128 tile per 128 rows wastes >99 % of its FMAs and is
// latency bound.  For wi, wo <= 8 one THREAD owns a row (row = blockIdx*256 + tid, stride gridDim*256): vector load,
// BN+LeakyReLU, wo x wi FMAs, vector store; statistics / weight gradients are Chan- / sum-reduced warp -> block -> ordered
// per-block partials.  The bodies below serve both the per-layer kernels and the whole-stack kernels, so the two paths
// compute the same bits from the same partition of the rows.  Weights are staged zero-padded to 8 x 8.
__device__ __forceinline__ void stage_w8(float (*Ws)[8], float* bs, const float* W, const float* bias, int wi, int wo, int e) {
  const int o = e >> 3, k = e & 7;
  Ws[o][k] = (o < wo && k < wi) ? W[o * wi + k] : 0.f;
  if (bs && k == 0) bs[o] = (o < wo && bias) ? bias[o] : 0.f;
}

// per-CTA sums of v[R][C] over the 256 threads: warp_sum, then warps 0..7 in order.  Thread i < R*C returns the sum of
// element i (row-major).
template <int R, int C>
__device__ __forceinline__ float cta_sum(const float (&v)[R][C], float* red /*[8][R*C]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < R; ++i)
#pragma unroll
    for (int j = 0; j < C; ++j) {
      const float s = warp_sum(v[i][j]);
      if (lane == 0) red[(warp * R + i) * C + j] = s;
    }
  __syncthreads();
  float s = 0.f;
  if (threadIdx.x < R * C)
    for (int w8 = 0; w8 < 8; ++w8) s += red[w8 * R * C + threadIdx.x];
  return s;
}

// ro_in: the layer input is not written by the launch that runs the body, so it may be read through the read-only
// cache (the stack kernel reads rows it wrote itself for the previous layer).
__device__ __forceinline__ float ld_in(bool ro_in, const float* p) { return ro_in ? __ldg(p) : *p; }

// Forward rows: y = act(src) W^T + b.  head > 0: the layer's output is also split into mu = cols [0, head) and
// softplus(cols [head, 2 head)) (torch.nn.functional.softplus, beta 1, threshold 20, ATen's expression).  do_stats: this
// CTA's (count, mean, M2) per column -> part[blockIdx][128][3].
template <int WI, int WO>
__device__ __forceinline__ void narrow_fwd_rows(const ActSrc& src, bool ro_in, const ActSmem& am, int B, int wo,
                                                const float (*Ws)[8],
                                                const float* bs, float* y, bool head, int nh, float* mu, float* lv,
                                                bool do_stats, float (*red)[8][3], float* part) {
  const int wi = src.w;
  const bool has_bn = src.mean != nullptr;
  float cnt = 0.f, mean[WO], m2[WO];
#pragma unroll
  for (int o = 0; o < WO; ++o) { mean[o] = 0.f; m2[o] = 0.f; }
  for (int row = blockIdx.x * 256 + threadIdx.x; row < B; row += gridDim.x * 256) {
    float a[WI];
#pragma unroll
    for (int k = 0; k < WI; ++k) a[k] = (k < wi) ? am.act(has_bn, src.slope, ld_in(ro_in, src.y + (size_t)row * wi + k), k) : 0.f;
    cnt += 1.f;
#pragma unroll
    for (int o = 0; o < WO; ++o) {
      float yv = bs[o];
#pragma unroll
      for (int k = 0; k < WI; ++k) yv = fmaf(a[k], Ws[o][k], yv);
      if (o < wo) {
        y[(size_t)row * wo + o] = yv;
        if (head) {
          if (o < nh) mu[(size_t)row * nh + o] = yv;
          else lv[(size_t)row * nh + o - nh] = yv > 20.f ? yv : log1pf(expf(yv));
        }
      }
      const float dlt = yv - mean[o];                    // Welford
      mean[o] += dlt / cnt;
      m2[o] = fmaf(dlt, yv - mean[o], m2[o]);
    }
  }
  if (!do_stats) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 0; o < WO; ++o) {
    float c = cnt, mu_o = mean[o], q = m2[o];
    chan_warp_merge(c, mu_o, q);
    if (lane == 0) { red[warp][o][0] = c; red[warp][o][1] = mu_o; red[warp][o][2] = q; }
  }
  __syncthreads();
  if (threadIdx.x < wo) {
    float c = 0.f, mu_o = 0.f, q = 0.f;
    for (int w8 = 0; w8 < 8; ++w8) chan_merge(c, mu_o, q, red[w8][threadIdx.x][0], red[w8][threadIdx.x][1], red[w8][threadIdx.x][2]);
    float* o = part + ((size_t)blockIdx.x * 128 + threadIdx.x) * 3;
    o[0] = c; o[1] = mu_o; o[2] = q;
  }
}

template <int WI, int WO>
__global__ void __launch_bounds__(256)
mlp_narrow_fwd_kernel(ActSrc src, const float* __restrict__ W, const float* __restrict__ bias, int B, int wo,
                      float* __restrict__ y_out, float* __restrict__ part, int do_stats, StatsFin fin) {
  __shared__ ActSmem am;
  __shared__ float Ws[8][8], bs[8];
  __shared__ float red[8][8][3];
  am.load(src);
  if (threadIdx.x < 64) stage_w8(Ws, bs, W, bias, src.w, wo, threadIdx.x);
  __syncthreads();
  narrow_fwd_rows<WI, WO>(src, true, am, B, wo, Ws, bs, y_out, false, 0, nullptr, nullptr, do_stats, red, part);
  if (do_stats && fin.stats && last_block_arrives(fin.ticket)) stats_finalize_block(part, (int)gridDim.x, wo, fin);
}

// da_prev = dy W and per-block partial of dW = dy^T act(prev), one row per thread.  stack_bwd_layer runs the same row
// loop and reduction; sharing them (cta_sum included) raised the register count here and in the stack kernels (the
// 8-wide stack kernel spilled).
template <int WI, int WO>
__global__ void __launch_bounds__(256)
mlp_narrow_bwd_kernel(DyCtx c, ActSrc prev, const float* __restrict__ W, int B, float* __restrict__ da_prev,
                      float* __restrict__ part /*[nblk][wo*wi]*/, DwFin fin) {
  __shared__ ActSmem am, pm;
  __shared__ float Ws[WO][WI], s1[WO], s2[WO];
  __shared__ float red[8 * WO * WI];
  const int wo = c.cur.w, wi = prev.w;
  am.load(c.cur);
  pm.load(prev);
  if (threadIdx.x < WO * WI) {
    const int o = threadIdx.x / WI, k = threadIdx.x % WI;
    Ws[o][k] = (o < wo && k < wi) ? W[o * wi + k] : 0.f;
  }
  if (threadIdx.x < WO) {
    s1[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[threadIdx.x] : 0.f;
    s2[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[wo + threadIdx.x] : 0.f;
  }
  __syncthreads();
  const bool prev_bn = prev.mean != nullptr;
  float acc[WO][WI];
#pragma unroll
  for (int o = 0; o < WO; ++o)
#pragma unroll
    for (int k = 0; k < WI; ++k) acc[o][k] = 0.f;
  for (int row = blockIdx.x * 256 + threadIdx.x; row < B; row += gridDim.x * 256) {
    float dy[WO], a[WI], dap[WI];
#pragma unroll
    for (int o = 0; o < WO; ++o) {
      dy[o] = 0.f;
      if (o < wo) {
        float g, yv;
        c.fetch((long long)row * wo + o, g, yv);
        dy[o] = c.dy(am, s1, s2, g, yv, o);
      }
    }
#pragma unroll
    for (int k = 0; k < WI; ++k) {
      a[k] = (k < wi) ? pm.act(prev_bn, prev.slope, __ldg(prev.y + (size_t)row * wi + k), k) : 0.f;
      dap[k] = 0.f;
    }
#pragma unroll
    for (int o = 0; o < WO; ++o)
#pragma unroll
      for (int k = 0; k < WI; ++k) { dap[k] = fmaf(dy[o], Ws[o][k], dap[k]); acc[o][k] = fmaf(dy[o], a[k], acc[o][k]); }
    if (da_prev) {
#pragma unroll
      for (int k = 0; k < WI; ++k) if (k < wi) da_prev[(size_t)row * wi + k] = dap[k];
    }
  }
  if (!part) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 0; o < WO; ++o)
#pragma unroll
    for (int k = 0; k < WI; ++k) {
      const float v = warp_sum(acc[o][k]);
      if (lane == 0) red[warp * WO * WI + o * WI + k] = v;
    }
  __syncthreads();
  if (threadIdx.x < WO * WI) {
    const int o = threadIdx.x / WI, k = threadIdx.x % WI;
    float v = 0.f;
    for (int w8 = 0; w8 < 8; ++w8) v += red[w8 * WO * WI + threadIdx.x];
    if (o < wo && k < wi) part[(size_t)blockIdx.x * wo * wi + o * wi + k] = v;
  }
  if (fin.dW && last_block_arrives(fin.ticket)) dw_finalize_block(part, (int)gridDim.x, wo * wi, fin.dW);
}

// Calls FN<WI, WO> ARGS for the width classes (ci, co) of a narrow layer; ARGS is an argument list in parentheses, or a
// kernel launch's <<<...>>>(...).  kMaxC: the widest class compiled (4: only the (2|4) x (2|4) bodies, which keeps the
// register count of the stack kernels -- and what they leave to concurrent kernels -- low).
#define B200VAE_NARROW_DISPATCH(kMaxC, FN, ci, co, ...)                                                  \
  do {                                                                                                    \
    if (ci == 2 && co == 2) FN<2, 2> __VA_ARGS__; else if (ci == 2 && co == 4) FN<2, 4> __VA_ARGS__;     \
    else if (ci == 4 && co == 2) FN<4, 2> __VA_ARGS__; else if (ci == 4 && co == 4) FN<4, 4> __VA_ARGS__; \
    else if constexpr (kMaxC == 8) {                                                                      \
      if (ci == 2) FN<2, 8> __VA_ARGS__; else if (ci == 4) FN<4, 8> __VA_ARGS__;                          \
      else if (co == 2) FN<8, 2> __VA_ARGS__; else if (co == 4) FN<8, 4> __VA_ARGS__;                     \
      else FN<8, 8> __VA_ARGS__;                                                                          \
    }                                                                                                     \
  } while (0)

// ----------------------------------------------------------------------------------------- small batches (B <= kRowsMaxB)
// At the batch sizes of BASELINE configs[2] / [3] (256) the 128x128x16 tile core runs a layer on 2 CTAs that walk up to 8
// DEPENDENT K-tiles, each exposing a full global-load latency: 20 us per layer forward, 27 us for the two backward GEMMs
// (warm-cache ncu, profiles/r02_launches_c3_warm.csv) -- half of the whole train step.  Here a CTA owns kRowsRT sample rows
// and the WHOLE weight matrix sits in shared memory (<= 128 x 129 floats), loaded with all requests in flight at once; the
// activations of the row tile are formed once (BN + LeakyReLU while loading) and every output is a dot product out of
// shared memory.  B = 256 -> 16 CTAs, one latency per layer.
constexpr int kRowsRT = 16;
constexpr int kRowsMaxB = 2048;
constexpr int kRowsLdw = 129;                      // padded row stride of W in shared memory (conflict-free across o)
static size_t rows_smem_bytes(bool bwd) {
  // W [128][129] + act tile [RT][128] (+ bwd: dy tile [RT][128])
  return (size_t)(128 * kRowsLdw + kRowsRT * 128 * (bwd ? 2 : 1)) * sizeof(float);
}

// forward: y = act(prev) W^T + b for rows [r0, r0 + RT); per-column (count, mean, M2) partial of the tile; fused finalize
__global__ void __launch_bounds__(256)
mlp_rows_fwd_kernel(ActSrc src, const float* __restrict__ W, const float* __restrict__ bias, int B, int wo,
                    float* __restrict__ y_out, float* __restrict__ part, int do_stats, StatsFin fin) {
  extern __shared__ float rsm[];
  float* Ws = rsm;                                 // [wo][kRowsLdw]
  float* As = rsm + 128 * kRowsLdw;                // [RT][128]: activations, later the output tile
  __shared__ ActSmem am;
  const int wi = src.w, r0 = blockIdx.x * kRowsRT, nrows = min(kRowsRT, B - r0);
  am.load(src);
  for (int e = threadIdx.x; e < wo * wi; e += 256) { const int o = e / wi, k = e - o * wi; Ws[o * kRowsLdw + k] = __ldg(W + e); }
  float pre[(kRowsRT * 128) / 256];                // raw inputs first (loads in flight with the W loads), act after the sync
#pragma unroll
  for (int q = 0; q < (kRowsRT * 128) / 256; ++q) {
    const int e = threadIdx.x + 256 * q, r = e >> 7, k = e & 127;
    pre[q] = (r < nrows && k < wi) ? __ldg(src.y + (size_t)(r0 + r) * wi + k) : 0.f;
  }
  __syncthreads();
  const bool has_bn = src.mean != nullptr;
#pragma unroll
  for (int q = 0; q < (kRowsRT * 128) / 256; ++q) {
    const int e = threadIdx.x + 256 * q, r = e >> 7, k = e & 127;
    As[e] = (r < nrows && k < wi) ? am.act(has_bn, src.slope, pre[q], k) : 0.f;
  }
  __syncthreads();
  // thread -> column o = tid & 127, rows (tid >> 7) + 2 j: 8 dot products sharing every W element
  const int o = threadIdx.x & 127, rb = threadIdx.x >> 7;
  float acc[kRowsRT / 2];
#pragma unroll
  for (int j = 0; j < kRowsRT / 2; ++j) acc[j] = 0.f;
  if (o < wo) {
    const float* wrow = Ws + o * kRowsLdw;
    for (int k = 0; k < wi; ++k) {
      const float wv = wrow[k];
#pragma unroll
      for (int j = 0; j < kRowsRT / 2; ++j) acc[j] = fmaf(As[(rb + 2 * j) * 128 + k], wv, acc[j]);
    }
  }
  __syncthreads();                                 // everyone is done reading As: it becomes the output tile
  if (o < wo) {
    const float bj = bias ? bias[o] : 0.f;
#pragma unroll
    for (int j = 0; j < kRowsRT / 2; ++j) {
      const int r = rb + 2 * j;
      const float yv = acc[j] + bj;
      As[r * 128 + o] = yv;
      if (r < nrows) y_out[(size_t)(r0 + r) * wo + o] = yv;
    }
  }
  if (!do_stats) return;
  __syncthreads();
  if (threadIdx.x < wo) {                          // column statistics of this tile, rows in order
    float sum = 0.f;
    for (int r = 0; r < nrows; ++r) sum += As[r * 128 + threadIdx.x];
    const float mean_c = sum / (float)nrows;
    float m2 = 0.f;
    for (int r = 0; r < nrows; ++r) { const float dlt = As[r * 128 + threadIdx.x] - mean_c; m2 = fmaf(dlt, dlt, m2); }
    float* po = part + ((size_t)blockIdx.x * 128 + threadIdx.x) * 3;
    po[0] = (float)nrows; po[1] = mean_c; po[2] = m2;
  }
  if (fin.stats && last_block_arrives(fin.ticket)) stats_finalize_block(part, (int)gridDim.x, wo, fin);
}

// backward: dy formed on the fly for the row tile; da_prev = dy W (may be null) and the tile's partial dW = dy^T act(prev)
__global__ void __launch_bounds__(256)
mlp_rows_bwd_kernel(DyCtx c, ActSrc prev, const float* __restrict__ W, int B, float* __restrict__ da_prev,
                    float* __restrict__ part /*[nCTA][wo*wi] or null*/) {
  extern __shared__ float rsm[];
  float* Ws = rsm;                                 // [wo][kRowsLdw]
  float* As = rsm + 128 * kRowsLdw;                // [RT][128] act(prev)
  float* Ds = As + kRowsRT * 128;                  // [RT][128] dy
  __shared__ ActSmem am, pm;
  __shared__ float s1[128], s2[128];
  const int wo = c.cur.w, wi = prev.w, r0 = blockIdx.x * kRowsRT, nrows = min(kRowsRT, B - r0);
  am.load(c.cur);
  pm.load(prev);
  if (threadIdx.x < 128) {
    s1[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[threadIdx.x] : 0.f;
    s2[threadIdx.x] = (c.has_bn && threadIdx.x < wo) ? c.sums[wo + threadIdx.x] : 0.f;
  }
  for (int e = threadIdx.x; e < wo * wi; e += 256) { const int o = e / wi, k = e - o * wi; Ws[o * kRowsLdw + k] = __ldg(W + e); }
  constexpr int Q = (kRowsRT * 128) / 256;
  float pa[Q], pg[Q], py[Q];
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int e = threadIdx.x + 256 * q, r = e >> 7, k = e & 127;
    pa[q] = (r < nrows && k < wi) ? __ldg(prev.y + (size_t)(r0 + r) * wi + k) : 0.f;
    pg[q] = 0.f; py[q] = 0.f;
    if (r < nrows && k < wo) c.fetch((long long)(r0 + r) * wo + k, pg[q], py[q]);
  }
  __syncthreads();
  const bool prev_bn = prev.mean != nullptr;
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int e = threadIdx.x + 256 * q, r = e >> 7, k = e & 127;
    As[e] = (r < nrows && k < wi) ? pm.act(prev_bn, prev.slope, pa[q], k) : 0.f;
    Ds[e] = (r < nrows && k < wo) ? c.dy(am, s1, s2, pg[q], py[q], k) : 0.f;
  }
  __syncthreads();
  if (da_prev) {                                   // thread -> input column k = tid & 127, rows (tid >> 7) + 2 j
    const int k = threadIdx.x & 127, rb = threadIdx.x >> 7;
    if (k < wi) {
      float acc[kRowsRT / 2];
#pragma unroll
      for (int j = 0; j < kRowsRT / 2; ++j) acc[j] = 0.f;
      for (int o = 0; o < wo; ++o) {
        const float wv = Ws[o * kRowsLdw + k];
#pragma unroll
        for (int j = 0; j < kRowsRT / 2; ++j) acc[j] = fmaf(Ds[(rb + 2 * j) * 128 + o], wv, acc[j]);
      }
#pragma unroll
      for (int j = 0; j < kRowsRT / 2; ++j) {
        const int r = rb + 2 * j;
        if (r < nrows) da_prev[(size_t)(r0 + r) * wi + k] = acc[j];
      }
    }
  }
  if (part) {                                      // dW partial of the tile: element (o, k), rows in order
    float* out = part + (size_t)blockIdx.x * wo * wi;
    for (int e = threadIdx.x; e < wo * wi; e += 256) {
      const int o = e / wi, k = e - o * wi;
      float s = 0.f;
#pragma unroll
      for (int r = 0; r < kRowsRT; ++r) s = fmaf(Ds[r * 128 + o], As[r * 128 + k], s);
      out[e] = s;
    }
  }
}

__host__ __device__ __forceinline__ int narrow_class(int w) { return w <= 2 ? 2 : (w <= 4 ? 4 : (w <= 8 ? 8 : 0)); }
static int narrow_grid(int B) { int g = (B + 255) / 256; return g > 592 ? 592 : (g < 1 ? 1 : g); }

// ----------------------------------------------------------------------------------------- narrow stacks, one launch
// When every layer of a stack is narrow the per-layer kernels above are bound by their chain of dependent launches (one
// or two per layer and direction, each ending in a last-block finalize), not by the few MFLOP they do.  The stack kernels
// run all layers in ONE cooperative launch: rows keep the thread mapping of mlp_narrow_*_kernel (row = blockIdx*256 +
// tid, stride gridDim*256), and where the per-layer path finalises in the last block, every CTA waits at a grid barrier
// and then combines the same ordered per-CTA partials itself, in the same fixed order, so all CTAs hold identical
// statistics and the forward results are bit-identical to the per-layer path at the same grid.
constexpr int kStackMaxLayers = 16;
constexpr int kStackMaxGrid = 592;
constexpr size_t kStackPartFloats = (size_t)2 * kStackMaxGrid * 128 * 3;      // two alternating partial buffers
constexpr size_t kStackDwFloats = (size_t)kStackMaxGrid * 64 * kStackMaxLayers; // per-CTA dW partials of every layer
constexpr size_t kStackDbFloats = (size_t)kStackMaxGrid * 8;                    // per-CTA bias-gradient partials, last layer
static size_t stack_scratch_floats(int B) { return kStackPartFloats + kStackDwFloats + kStackDbFloats + (size_t)B * 8; }

struct StackArgs {
  b200vae_mlp_layer_t L[kStackMaxLayers];
  b200vae_mlp_grad_t G[kStackMaxLayers];
  int nl, B, training, head;   // head > 0: the last layer's output is (mu = cols [0, head), softplus(cols [head, 2 head)))
  float slope;
  const float* x;              // [B][L[0].wi]
  float* out0; float* out1;    // forward: mu, lv (head) ; backward: unused
  const float* g0; const float* g1;   // backward: g_mu, g_lv (head; either may be null = zero) or g_out in g0
  float* dx;                   // backward: [B][L[0].wi] or null
  float* scratch;
  unsigned* bar;               // [0] barrier arrivals, [1] exit ticket: zero before the launch, left zero
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Grid-wide barrier.  Only valid in a cooperative launch (all CTAs co-resident).  The arrival counter only grows during a
// launch (`epoch` = arrivals expected so far); stack_exit() resets it once every CTA is past its last barrier.
__device__ __forceinline__ void grid_barrier(unsigned* count, unsigned& epoch) {
  __syncthreads();
  epoch += gridDim.x;
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(count, 1u);
    while (ld_acquire_gpu(count) < epoch) __nanosleep(32);
    __threadfence();
  }
  __syncthreads();
}
__device__ __forceinline__ bool stack_exit(unsigned* bar) {
  const bool last = last_block_arrives(bar + 1);
  if (last && threadIdx.x == 0) bar[0] = 0u;
  return last;
}

// Forward of a whole narrow stack.  Training: per BatchNorm layer one grid barrier, then every CTA combines the layer's
// (count, mean, M2) partials with stats_finalize_block (the per-layer path's last-block code) into shared memory; CTA 0
// also stores the statistics and updates running_mean / running_var / num_batches_tracked.  Eval: the statistics are read
// from L[l].stats and no CTA waits for another.
// the input of layer l: the raw input, or LeakyReLU(BN(y of layer l - 1)) with that layer's stored statistics
__device__ __forceinline__ ActSrc stack_in(const StackArgs& A, int l) {
  if (l == 0) return make_src(A.x, nullptr, nullptr, nullptr, A.L[0].wi, A.slope);
  const b200vae_mlp_layer_t& P = A.L[l - 1];
  return make_src(P.y, P.stats, P.gamma, P.beta, P.wo, A.slope);
}

template <int kMaxC>
__global__ void __launch_bounds__(256, kMaxC == 8 ? 2 : 4) mlp_stack_fwd_kernel(const StackArgs A) {
  __shared__ ActSmem am;
  __shared__ float Ws[kStackMaxLayers][8][8], bs[kStackMaxLayers][8];
  __shared__ float red[8][8][3];
  __shared__ float st[4 * 8];
  for (int e = threadIdx.x; e < A.nl * 64; e += 256) {      // every layer's weights
    const int l = e >> 6;
    stage_w8(Ws[l], bs[l], A.L[l].W, A.L[l].bias, A.L[l].wi, A.L[l].wo, e & 63);
  }
  unsigned epoch = 0;
  for (int l = 0; l < A.nl; ++l) {
    const b200vae_mlp_layer_t& L = A.L[l];
    const bool last = l == A.nl - 1;
    __syncthreads();                                          // weights loaded / previous layer's ActSmem in place
    const bool do_stats = A.training && !last;
    float* part = A.scratch + (size_t)(l & 1) * kStackMaxGrid * 128 * 3;
    const ActSrc src = stack_in(A, l);
    B200VAE_NARROW_DISPATCH(kMaxC, narrow_fwd_rows, narrow_class(L.wi), narrow_class(L.wo),
                            (src, false, am, A.B, L.wo, Ws[l], bs[l], L.y, last && A.head > 0, A.head, A.out0, A.out1, do_stats, red, part));
    if (last) break;
    const int wo = L.wo;
    if (do_stats) {
      grid_barrier(A.bar, epoch);
      StatsFin f;
      f.stats = st; f.eps = L.eps; f.momentum = L.momentum; f.peer = 0;
      f.running_mean = blockIdx.x == 0 ? L.running_mean : nullptr;
      f.running_var = blockIdx.x == 0 ? L.running_var : nullptr;
      stats_finalize_block(part, (int)gridDim.x, wo, f);
      __syncthreads();
      if (blockIdx.x == 0) {
        if (threadIdx.x < 4 * wo) L.stats[threadIdx.x] = st[threadIdx.x];
        if (threadIdx.x == 0 && L.num_batches_tracked) *L.num_batches_tracked += 1;
      }
    } else if (threadIdx.x < 4 * wo) {
      st[threadIdx.x] = L.stats[threadIdx.x];
    }
    __syncthreads();
    am.load(make_src(L.y, st, L.gamma, L.beta, wo, A.slope));   // the next layer's input transform
  }
  if (A.training) stack_exit(A.bar);
}

// Backward, phase 1 of layer l: dyhat = da * lrelu'(.) and the per-CTA (S1, S2) partials.  da of the last layer comes
// from the caller's gradients (softplus' applied to the lv half, the expression of ATen's softplus_backward); the
// others from the rows buffer that phase 2 of layer l + 1 filled (each thread only touches its own rows).
template <int WO>
__device__ __forceinline__ void stack_dyhat(const StackArgs& A, int l, const ActSmem& am, int row, float (&g)[WO],
                                            float (&xh)[WO]) {
  const b200vae_mlp_layer_t& L = A.L[l];
  const int wo = L.wo;
  const bool has_bn = l < A.nl - 1;
  const float* da_rows = A.scratch + kStackPartFloats + kStackDwFloats + kStackDbFloats;
#pragma unroll
  for (int o = 0; o < WO; ++o) {
    float d = 0.f, yv = 0.f;
    if (o < wo) {
      if (has_bn) yv = L.y[(size_t)row * wo + o];
      if (l < A.nl - 1) {
        d = da_rows[(size_t)row * 8 + o];
      } else if (A.head == 0) {
        d = A.g0[(size_t)row * wo + o];
      } else if (o < A.head) {
        d = A.g0 ? A.g0[(size_t)row * A.head + o] : 0.f;
      } else {
        const float gl = A.g1 ? A.g1[(size_t)row * A.head + o - A.head] : 0.f;
        const float x = L.y[(size_t)row * wo + o], z = expf(x);
        d = x > 20.f ? gl : gl * z / (z + 1.f);
      }
    }
    xh[o] = 0.f;
    if (has_bn) {
      xh[o] = am.xhat(yv, o);
      const float t = fmaf(xh[o], am.gamma[o], am.beta[o]);
      d = t > 0.f ? d : A.slope * d;
    }
    g[o] = d;
  }
}

template <int WO>
__device__ __forceinline__ void stack_bwd_sums(const StackArgs& A, int l, const ActSmem& am, float* red, float* part) {
  float s[WO][2];                                             // S1, S2 of column o
#pragma unroll
  for (int o = 0; o < WO; ++o) { s[o][0] = 0.f; s[o][1] = 0.f; }
  for (int row = blockIdx.x * 256 + threadIdx.x; row < A.B; row += gridDim.x * 256) {
    float g[WO], xh[WO];
    stack_dyhat<WO>(A, l, am, row, g, xh);
#pragma unroll
    for (int o = 0; o < WO; ++o) { s[o][0] += g[o]; s[o][1] = fmaf(g[o], xh[o], s[o][1]); }
  }
  const float v = cta_sum(s, red);
  if (threadIdx.x < 2 * A.L[l].wo) part[(size_t)blockIdx.x * 256 + threadIdx.x] = v;
}

// Backward, phase 2 of layer l: dy from dyhat and the global sums, da_prev = dy W into the rows buffer (or dx), and the
// per-CTA dW partial.  The row loop is mlp_narrow_bwd_kernel's, with dy from stack_dyhat.
template <int WI, int WO>
__device__ __forceinline__ void stack_bwd_layer(const StackArgs& A, int l, const ActSmem& am, const ActSmem& pm,
                                                const float (*Ws)[8], const float* s1, const float* s2, float invN,
                                                float* red) {
  const b200vae_mlp_layer_t& L = A.L[l];
  const int wo = L.wo, wi = L.wi;
  const bool has_bn = l < A.nl - 1;
  const float* src = l == 0 ? A.x : A.L[l - 1].y;
  float* da_rows = A.scratch + kStackPartFloats + kStackDwFloats + kStackDbFloats;
  float acc[WO][WI];
#pragma unroll
  for (int o = 0; o < WO; ++o)
#pragma unroll
    for (int k = 0; k < WI; ++k) acc[o][k] = 0.f;
  for (int row = blockIdx.x * 256 + threadIdx.x; row < A.B; row += gridDim.x * 256) {
    float g[WO], xh[WO], dy[WO], a[WI], dap[WI];
    stack_dyhat<WO>(A, l, am, row, g, xh);
#pragma unroll
    for (int o = 0; o < WO; ++o)
      dy[o] = (o < wo && has_bn) ? am.gamma[o] * am.invstd[o] * (g[o] - s1[o] * invN - xh[o] * (s2[o] * invN)) : g[o];
#pragma unroll
    for (int k = 0; k < WI; ++k) {
      a[k] = (k < wi) ? pm.act(l > 0, A.slope, src[(size_t)row * wi + k], k) : 0.f;
      dap[k] = 0.f;
    }
#pragma unroll
    for (int o = 0; o < WO; ++o)
#pragma unroll
      for (int k = 0; k < WI; ++k) { dap[k] = fmaf(dy[o], Ws[o][k], dap[k]); acc[o][k] = fmaf(dy[o], a[k], acc[o][k]); }
    if (l > 0) {
#pragma unroll
      for (int k = 0; k < WI; ++k) if (k < wi) da_rows[(size_t)row * 8 + k] = dap[k];
    } else if (A.dx) {
#pragma unroll
      for (int k = 0; k < WI; ++k) if (k < wi) A.dx[(size_t)row * wi + k] = dap[k];
    }
  }
  const float v = cta_sum(acc, red);
  if (threadIdx.x < WO * WI) {
    const int o = threadIdx.x / WI, k = threadIdx.x % WI;
    float* part = A.scratch + kStackPartFloats + (size_t)l * kStackMaxGrid * 64;
    if (o < wo && k < wi) part[(size_t)blockIdx.x * wo * wi + o * wi + k] = v;
  }
}

// Backward of a whole narrow stack, layers in reverse.  Per BatchNorm layer one grid barrier between the (S1, S2)
// partials and their fixed-order combine (sums_finalize_column, in every CTA); CTA 0 stores dbeta = S1, dgamma = S2 and
// the exactly-zero gradient of the bias that feeds the BatchNorm.  dW of every layer and the last layer's bias gradient
// are reduced once, by the last CTA to leave, in fixed order (dw_finalize_block).
template <int kMaxC>
__global__ void __launch_bounds__(256, kMaxC == 8 ? 2 : 4) mlp_stack_bwd_kernel(const StackArgs A) {
  __shared__ ActSmem am, pm;
  __shared__ float Ws[8][8], s1[8], s2[8], sums[2 * 8];
  __shared__ float red[8 * 64];
  unsigned epoch = 0;
  const float invN = 1.f / (float)A.B;
  float* dbpart = A.scratch + kStackPartFloats + kStackDwFloats;
  for (int l = A.nl - 1; l >= 0; --l) {
    const b200vae_mlp_layer_t& L = A.L[l];
    const int wo = L.wo, wi = L.wi;
    const bool has_bn = l < A.nl - 1;
    __syncthreads();                                          // the previous layer is done with the shared arrays
    if (has_bn) am.load(stack_in(A, l + 1));
    pm.load(stack_in(A, l));
    if (threadIdx.x < 64) stage_w8(Ws, nullptr, L.W, nullptr, wi, wo, threadIdx.x);
    __syncthreads();
    float* part = A.scratch + (size_t)(l & 1) * kStackMaxGrid * 128 * 2;
    const int co = narrow_class(wo);
    if (co == 2) stack_bwd_sums<2>(A, l, am, red, part);
    else if (co == 4) stack_bwd_sums<4>(A, l, am, red, part);
    else if constexpr (kMaxC == 8) stack_bwd_sums<8>(A, l, am, red, part);
    if (has_bn) {
      grid_barrier(A.bar, epoch);
      for (int n = threadIdx.x >> 5; n < wo; n += 8) sums_finalize_column(part, (int)gridDim.x, wo, n, sums);
      __syncthreads();
      if (threadIdx.x < wo) {
        const int n = threadIdx.x;
        if (blockIdx.x == 0) { A.G[l].dbeta[n] = sums[n]; A.G[l].dgamma[n] = sums[wo + n]; A.G[l].db[n] = 0.f; }
        s1[n] = A.training ? sums[n] : 0.f;          // eval-mode BatchNorm is affine: dy = gamma*invstd*dyhat
        s2[n] = A.training ? sums[wo + n] : 0.f;
      }
    } else {
      __syncthreads();
      if (threadIdx.x < wo) dbpart[(size_t)blockIdx.x * wo + threadIdx.x] = part[((size_t)blockIdx.x * 128 + threadIdx.x) * 2];
    }
    __syncthreads();
    B200VAE_NARROW_DISPATCH(kMaxC, stack_bwd_layer, narrow_class(wi), co, (A, l, am, pm, Ws, s1, s2, invN, red));
  }
  if (stack_exit(A.bar)) {
    for (int l = 0; l < A.nl; ++l) {
      const float* part = A.scratch + kStackPartFloats + (size_t)l * kStackMaxGrid * 64;
      dw_finalize_block(part, (int)gridDim.x, A.L[l].wo * A.L[l].wi, A.G[l].dW);
    }
    const int wo = A.L[A.nl - 1].wo;
    dw_finalize_block(dbpart, (int)gridDim.x, wo, A.G[A.nl - 1].db);
  }
}

static bool pow2_le128(int w) { return w >= 1 && w <= 128 && (w & (w - 1)) == 0; }

}  // namespace b200vae

using namespace b200vae;

static size_t mlp_scratch_floats(int B) {
  const size_t ncta = (size_t)(B + 127) / 128;
  const size_t a = (ncta > 592 ? ncta : 592) * 128 * 3, b = (size_t)296 * 128 * 2, c = (size_t)296 * 128 * 128;
  size_t m = a > b ? a : b;
  if (c > m) m = c;
  const size_t s = stack_scratch_floats(B);
  return s > m ? s : m;
}
// partials, then 64 floats holding the last-block ticket (must be zero before the first call; every call leaves it zero),
// then the staging area of the fused cross-rank exchange (this rank's values + every rank's)
constexpr size_t kMlpStageFloats = (size_t)(kPeerMaxWorld + 1) * 3 * 128;
extern "C" size_t b200vae_mlp_scratch_bytes(int B) { return (mlp_scratch_floats(B) + 64 + kMlpStageFloats) * sizeof(float); }
static unsigned* mlp_ticket(void* scratch, int B) { return reinterpret_cast<unsigned*>((float*)scratch + mlp_scratch_floats(B)); }
static float* mlp_stage(void* scratch, int B) { return (float*)scratch + mlp_scratch_floats(B) + 64; }
// one CTA finalising n outputs from `nparts` partials each: worth fusing while that is a few thousand loads per warp
static bool fuse_finalize(long long nparts, long long n) { return nparts * n <= (long long)1 << 16; }

static int mlp_layer_fwd_impl(const float* in_y, const float* in_stats, const float* in_gamma, const float* in_beta,
                              float slope, const float* W, const float* bias, int B, int wi, int wo, float* y_out,
                              float* stats_out, float eps, float* running_mean, float* running_var, float momentum,
                              void* scratch, const b200vae_peer_t* comm, int slot, void* stream) {
  if (!in_y || !W || !y_out || !scratch) return B200VAE_EALIGN;
  if (B <= 0 || wi < 1 || wi > 128 || wo < 1 || wo > 128) return B200VAE_ESHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  int ncta = (B + 127) / 128;
  const ActSrc src = make_src(in_y, in_stats, in_gamma, in_beta, wi, slope);
  const int ci = narrow_class(wi), co = narrow_class(wo);
  const bool rows = !(ci && co) && B <= kRowsMaxB;          // small batch, wide layer: row-tile kernel, W in shared memory
  if (ci && co) ncta = narrow_grid(B);
  else if (rows) ncta = (B + kRowsRT - 1) / kRowsRT;
  // single GPU: the last CTA of the layer kernel finalises the statistics itself (no second launch)
  const bool fused = stats_out && fuse_finalize(ncta, wo);
  StatsFin fin;
  fin.stats = fused ? stats_out : nullptr; fin.running_mean = running_mean; fin.running_var = running_var; fin.eps = eps;
  fin.momentum = momentum; fin.ticket = mlp_ticket(scratch, B);
  fin.peer = comm ? 1 : 0; fin.slot = slot; fin.stage = mlp_stage(scratch, B);
  if (comm) fin.comm = make_peer(comm); else memset(&fin.comm, 0, sizeof(fin.comm));
  if (ci && co) {
    B200VAE_NARROW_DISPATCH(8, mlp_narrow_fwd_kernel, ci, co,
                            <<<ncta, 256, 0, st>>>(src, W, bias, B, wo, y_out, (float*)scratch, stats_out ? 1 : 0, fin));
  } else if (rows) {
    static bool attr_done = false;
    if (!attr_done) { cudaFuncSetAttribute(mlp_rows_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem_bytes(false)); attr_done = true; }
    mlp_rows_fwd_kernel<<<ncta, 256, rows_smem_bytes(false), st>>>(src, W, bias, B, wo, y_out, (float*)scratch, stats_out ? 1 : 0, fin);
  } else {
    mlp_fwd_kernel<<<ncta, kThreads, 0, st>>>(src, W, bias, B, wo, y_out, (float*)scratch, stats_out ? 1 : 0, fin);
  }
  int rc = check_launch();
  if (rc || !stats_out || fused) return rc;
  fin.stats = stats_out;
  if (comm) mlp_stats_finalize_peer_kernel<<<1, 1024, 0, st>>>((const float*)scratch, ncta, wo, fin);
  else mlp_stats_finalize_kernel<<<(wo + 7) / 8, 256, 0, st>>>((const float*)scratch, ncta, wo, fin);
  return check_launch();
}
extern "C" int b200vae_mlp_layer_fwd(const float* in_y, const float* in_stats, const float* in_gamma, const float* in_beta,
                                     float slope, const float* W, const float* bias, int B, int wi, int wo, float* y_out,
                                     float* stats_out, float eps, float* running_mean, float* running_var, float momentum,
                                     void* scratch, void* stream) {
  return mlp_layer_fwd_impl(in_y, in_stats, in_gamma, in_beta, slope, W, bias, B, wi, wo, y_out, stats_out, eps,
                            running_mean, running_var, momentum, scratch, nullptr, 0, stream);
}
extern "C" int b200vae_mlp_layer_fwd_peer(const float* in_y, const float* in_stats, const float* in_gamma,
                                          const float* in_beta, float slope, const float* W, const float* bias, int B,
                                          int wi, int wo, float* y_out, float* stats_out, float eps, float* running_mean,
                                          float* running_var, float momentum, void* scratch, const b200vae_peer_t* comm,
                                          int slot, void* stream) {
  if (!peer_ok(comm, slot) || !stats_out) return B200VAE_EALIGN;
  return mlp_layer_fwd_impl(in_y, in_stats, in_gamma, in_beta, slope, W, bias, B, wi, wo, y_out, stats_out, eps,
                            running_mean, running_var, momentum, scratch, comm, slot, stream);
}

static int mlp_layer_bwd_reduce_impl(const float* da, const float* y, const float* stats, const float* gamma,
                                     const float* beta, float slope, int B, int w, float* dyhat, float* sums,
                                     float* sums_global, void* scratch, const b200vae_peer_t* comm, int slot,
                                     void* stream) {
  if (!da || !dyhat || !(sums || sums_global) || !scratch) return B200VAE_EALIGN;
  if (B <= 0 || !pow2_le128(w)) return B200VAE_EUNSUP;
  cudaStream_t st = (cudaStream_t)stream;
  const long long n = (long long)B * w;
  int nblk = (int)((n + 256 * 4 - 1) / (256 * 4));
  if (nblk > 296) nblk = 296;
  if (nblk < 1) nblk = 1;
  long long per = (n + nblk - 1) / nblk;
  per = (per + 255) / 256 * 256;                       // keeps (element index % w) == (thread index % w)
  const ActSrc cur = make_src(y, stats, gamma, beta, w, slope);
  SumsFin fin;
  fin.sums = sums; fin.ticket = mlp_ticket(scratch, B);
  fin.peer = comm ? 1 : 0; fin.slot = slot; fin.sums_global = sums_global; fin.stage = mlp_stage(scratch, B);
  if (comm) fin.comm = make_peer(comm); else memset(&fin.comm, 0, sizeof(fin.comm));
  mlp_bwd_reduce_kernel<<<nblk, 256, 0, st>>>(da, cur, stats ? 1 : 0, n, per, dyhat, (float*)scratch, fin);
  return check_launch();
}
extern "C" int b200vae_mlp_layer_bwd_reduce(const float* da, const float* y, const float* stats, const float* gamma,
                                            const float* beta, float slope, int B, int w, float* dyhat, float* sums,
                                            void* scratch, void* stream) {
  if (!sums) return B200VAE_EALIGN;
  return mlp_layer_bwd_reduce_impl(da, y, stats, gamma, beta, slope, B, w, dyhat, sums, nullptr, scratch, nullptr, 0, stream);
}
extern "C" int b200vae_mlp_layer_bwd_reduce_peer(const float* da, const float* y, const float* stats, const float* gamma,
                                                 const float* beta, float slope, int B, int w, float* dyhat,
                                                 float* sums_local, float* sums_global, void* scratch,
                                                 const b200vae_peer_t* comm, int slot, void* stream) {
  if (!peer_ok(comm, slot) || !sums_global) return B200VAE_EALIGN;
  return mlp_layer_bwd_reduce_impl(da, y, stats, gamma, beta, slope, B, w, dyhat, sums_local, sums_global, scratch, comm,
                                   slot, stream);
}

extern "C" int b200vae_mlp_layer_bwd(const float* dyhat, const float* y, const float* stats, const float* gamma,
                                     const float* beta, const float* sums, float inv_n, float slope, const float* W,
                                     const float* prev_y, const float* prev_stats, const float* prev_gamma,
                                     const float* prev_beta, int B, int wo, int wi, float* da_prev, float* dW,
                                     void* scratch, void* stream) {
  if (!dyhat || !W || !prev_y || !scratch) return B200VAE_EALIGN;
  if (B <= 0 || wi < 1 || wi > 128 || wo < 1 || wo > 128) return B200VAE_ESHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  DyCtx c;
  c.dyhat = dyhat; c.cur = make_src(y, stats, gamma, beta, wo, slope); c.sums = sums; c.invN = inv_n; c.has_bn = stats ? 1 : 0;
  if (c.has_bn && !sums) return B200VAE_EALIGN;
  int rc = B200VAE_OK;
  const int ci = narrow_class(wi), co = narrow_class(wo);
  if (ci && co) {
    const int grid = narrow_grid(B);
    const ActSrc prev = make_src(prev_y, prev_stats, prev_gamma, prev_beta, wi, slope);
    DwFin fin;
    fin.dW = dW; fin.ticket = mlp_ticket(scratch, B);        // <= 64 outputs from <= 592 partials: always fused
    B200VAE_NARROW_DISPATCH(8, mlp_narrow_bwd_kernel, ci, co,
                            <<<grid, 256, 0, st>>>(c, prev, W, B, da_prev, dW ? (float*)scratch : nullptr, fin));
    return check_launch();
  }
  if (B <= kRowsMaxB) {            // small batch: ONE row-tile kernel for da_prev and the dW partials (W in shared memory)
    static bool attr_done = false;
    if (!attr_done) { cudaFuncSetAttribute(mlp_rows_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem_bytes(true)); attr_done = true; }
    const ActSrc prev = make_src(prev_y, prev_stats, prev_gamma, prev_beta, wi, slope);
    const int ncta = (B + kRowsRT - 1) / kRowsRT, n = wo * wi;
    mlp_rows_bwd_kernel<<<ncta, 256, rows_smem_bytes(true), st>>>(c, prev, W, B, da_prev, dW ? (float*)scratch : nullptr);
    rc = check_launch();
    if (rc || !dW) return rc;
    mlp_dw_finalize_kernel<<<(n + 7) / 8, 256, 0, st>>>((const float*)scratch, ncta, n, dW);
    return check_launch();
  }
  if (da_prev) {
    mlp_bwd_gemm_kernel<<<(B + 127) / 128, kThreads, 0, st>>>(c, W, B, wi, da_prev);
    rc = check_launch();
    if (rc) return rc;
  }
  if (dW) {
    // split the batch (the K dimension of dW = dy^T act(prev)) over CTAs: 256 samples each at large B; at small B one
    // 16-sample K-tile each, so that a batch-256 layer runs on 16 SMs instead of ONE CTA walking 16 dependent K-tiles
    // (measured at B = 256: 80-114 us per layer before)
    int nsplit = (B + 255) / 256;
    if (nsplit < 64) { const int fine = (B + kBK - 1) / kBK; nsplit = fine < 64 ? fine : 64; }
    if (nsplit > 296) nsplit = 296;
    int rows = (B + nsplit - 1) / nsplit;
    rows = round_up(rows, kBK);
    const ActSrc prev = make_src(prev_y, prev_stats, prev_gamma, prev_beta, wi, slope);
    const int n = wo * wi;
    DwFin fin;
    fin.dW = fuse_finalize(nsplit, n) ? dW : nullptr; fin.ticket = mlp_ticket(scratch, B);
    mlp_bwd_dw_kernel<<<nsplit, kThreads, 0, st>>>(c, prev, B, rows, (float*)scratch, fin);
    rc = check_launch();
    if (rc || fin.dW) return rc;
    mlp_dw_finalize_kernel<<<(n + 7) / 8, 256, 0, st>>>((const float*)scratch, nsplit, n, dW);
    rc = check_launch();
  }
  return rc;
}

// ----------------------------------------------------------------------------------------- narrow stacks
static bool stack_shape_ok(const b200vae_mlp_layer_t* L, int nl, int B) {
  if (!L || nl < 1 || nl > kStackMaxLayers || B <= 0) return false;
  for (int l = 0; l < nl; ++l) {
    if (L[l].wi < 1 || L[l].wi > 8 || L[l].wo < 1 || L[l].wo > 8) return false;
    if (l > 0 && L[l].wi != L[l - 1].wo) return false;
    if (!L[l].W || !L[l].bias || !L[l].y) return false;
    if (l < nl - 1 && (!L[l].gamma || !L[l].beta || !L[l].stats)) return false;
  }
  return true;
}
static int stack_max_class(const b200vae_mlp_layer_t* L, int nl) {
  int c = 2;
  for (int l = 0; l < nl; ++l) c = max(c, max(narrow_class(L[l].wi), narrow_class(L[l].wo)));
  return c;
}
// The grid of the per-layer narrow kernels (so the statistics are combined from the same partials), clamped to what
// the occupancy API says fits co-resident: the grid barrier needs every CTA running at once.
template <int kMaxC>
static int stack_grid(int B) {
  static int cap = 0;
  if (cap == 0) {
    int f = 0, b = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&f, mlp_stack_fwd_kernel<kMaxC>, 256, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, mlp_stack_bwd_kernel<kMaxC>, 256, 0);
    cap = (f < b ? f : b) * sm_count();
    if (cap <= 0) return 0;
  }
  const int g = narrow_grid(B);
  return g < cap ? g : cap;
}
template <typename Kernel>
static int stack_launch(Kernel kernel, const StackArgs& A, int grid, void* stream) {
  if (grid <= 0) return B200VAE_ECUDA;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative; attr[0].val.cooperative = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, A);
  if (e != cudaSuccess) { g_last_cuda_error = (int)e; ++g_launch_count; return B200VAE_ECUDA; }
  return check_launch();
}
static StackArgs stack_args(const b200vae_mlp_layer_t* layers, int nl, const float* x, int B, float slope, int training,
                            int head, void* scratch) {
  StackArgs A;
  memset(&A, 0, sizeof(A));
  for (int l = 0; l < nl; ++l) A.L[l] = layers[l];
  A.nl = nl; A.B = B; A.training = training ? 1 : 0; A.head = head; A.slope = slope; A.x = x;
  A.scratch = (float*)scratch; A.bar = mlp_ticket(scratch, B) + 1;    // [0] stays the layer kernels' last-block ticket
  return A;
}

extern "C" int b200vae_mlp_stack_fwd(const b200vae_mlp_layer_t* layers, int nl, const float* x, int B, float slope,
                                     int training, int head, float* mu, float* lv, void* scratch, void* stream) {
  if (!x || !scratch) return B200VAE_EALIGN;
  if (!stack_shape_ok(layers, nl, B)) return B200VAE_ESHAPE;
  if (head < 0 || (head > 0 && (2 * head != layers[nl - 1].wo || !mu || !lv))) return B200VAE_ESHAPE;
  StackArgs A = stack_args(layers, nl, x, B, slope, training, head, scratch);
  A.out0 = mu; A.out1 = lv;
  if (stack_max_class(layers, nl) == 8) return stack_launch(mlp_stack_fwd_kernel<8>, A, stack_grid<8>(B), stream);
  return stack_launch(mlp_stack_fwd_kernel<4>, A, stack_grid<4>(B), stream);
}

extern "C" int b200vae_mlp_stack_bwd(const b200vae_mlp_layer_t* layers, const b200vae_mlp_grad_t* grads, int nl,
                                     const float* x, int B, float slope, int training, int head, const float* g0,
                                     const float* g1, float* dx, void* scratch, void* stream) {
  if (!x || !scratch || !grads) return B200VAE_EALIGN;
  if (!stack_shape_ok(layers, nl, B)) return B200VAE_ESHAPE;
  if (head < 0 || (head > 0 && 2 * head != layers[nl - 1].wo) || (head == 0 && !g0)) return B200VAE_ESHAPE;
  for (int l = 0; l < nl; ++l)
    if (!grads[l].dW || !grads[l].db || (l < nl - 1 && (!grads[l].dgamma || !grads[l].dbeta))) return B200VAE_EALIGN;
  StackArgs A = stack_args(layers, nl, x, B, slope, training, head, scratch);
  for (int l = 0; l < nl; ++l) A.G[l] = grads[l];
  A.g0 = g0; A.g1 = g1; A.dx = dx;
  if (stack_max_class(layers, nl) == 8) return stack_launch(mlp_stack_bwd_kernel<8>, A, stack_grid<8>(B), stream);
  return stack_launch(mlp_stack_bwd_kernel<4>, A, stack_grid<4>(B), stream);
}
