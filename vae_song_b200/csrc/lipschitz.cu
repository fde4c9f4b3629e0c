// lipschitz.cu -- pairwise |f(x)-f(y)| / |x-y| estimators.
//   pairs kernel    : reference semantics, utils.py:544-562 (random index pairs given by the caller,
//                     rows flattened, p=2 norms, both norms clamped at eps)
//   all-pairs kernels: north_star kernel 4 -- 64x64 tiles of the upper triangle, 4x4 pairs per thread, one MUFU op per
//                     pair, warp-shuffle max / min / sum, ordered per-CTA partials + last-block reduce (no float atomics),
//                     optional log2 histogram (shared-memory bins flushed once per CTA).
//   select kernels   : exact quantiles of the same keys over every pair: the all-pairs tile walks with a counting sink (a
//                     3-pass radix select on the key bits, integer histograms only) + a one-CTA locate kernel per pass.
#include "common.cuh"

namespace b200vae {

// one warp per pair; lanes stride over the feature dimension
__global__ void __launch_bounds__(256)
lipschitz_pairs_kernel(const float* __restrict__ X, const float* __restrict__ Y, const int64_t* __restrict__ i1,
                       const int64_t* __restrict__ i2, int P, int N, int dx, int dy, float eps,
                       float* __restrict__ ratio) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int p = warp; p < P; p += nwarps) {
    long long a = i1[p], b = i2[p];
    a = a < 0 ? 0 : (a >= N ? N - 1 : a);
    b = b < 0 ? 0 : (b >= N ? N - 1 : b);
    float sx = 0.f, sy = 0.f;
    for (int j = lane; j < dx; j += 32) { const float t = X[a * dx + j] - X[b * dx + j]; sx = fmaf(t, t, sx); }
    for (int j = lane; j < dy; j += 32) { const float t = Y[a * dy + j] - Y[b * dy + j]; sy = fmaf(t, t, sy); }
    sx = warp_sum(sx); sy = warp_sum(sy);
    if (lane == 0) ratio[p] = fmaxf(sqrtf(sy), eps) / fmaxf(sqrtf(sx), eps);
  }
}

constexpr int kTile = 64;                      // pair tile: 64 x 64 points (ABI: b200vae_lipschitz_num_tiles)
constexpr int kApThreads = 256;                // 16 x 16 threads, 4 x 4 pairs each
constexpr int kApMaxBlocks = 148 * 8;
constexpr int kApMaxSmemBins = 2048;

// (ti, tj) of tile t, row-major over the upper triangle (ti <= tj): row r starts at r*T - r*(r-1)/2.  A float estimate of
// the row, made exact by integer fix-up steps.
__device__ __forceinline__ void tile_coords(long long t, int T, int& ti, int& tj) {
  const float b = 2.f * (float)T + 1.f;
  int r = (int)((b - sqrtf(fmaxf(b * b - 8.f * (float)t, 0.f))) * 0.5f);
  r = r < 0 ? 0 : (r > T - 1 ? T - 1 : r);
  auto start = [T](long long q) { return q * T - q * (q - 1) / 2; };
  while (r > 0 && start(r) > t) --r;
  while (r + 1 < T && start(r + 1) <= t) ++r;
  ti = r;
  tj = r + (int)(t - start(r));
}

struct ApAcc {
  float vmax, vmin, sum;                       // running max / min / sum of the ratios of this thread
  unsigned cnt;
};

// ratio = clamp(|dy|, eps) / clamp(|dx|, eps) = sqrt(max(sy, eps^2) / max(sx, eps^2)) with ONE MUFU op per pair:
// r = a * rsqrt(a * b), a = max(sy, eps^2), b = max(sx, eps^2) (utils.py:560-562 semantics, ~2 ulp).  The product a*b can leave
// the fp32 range (then r is 0, inf or NaN -- a true ratio is a positive finite number): callers check the min / max of a
// group of pairs once and redo the group with ap_ratio_safe (rare).
__device__ __forceinline__ float ap_ratio(float sx, float sy, float eps2) {
  const float a = fmaxf(sy, eps2), b = fmaxf(sx, eps2);
  return a * rsqrtf(a * b);
}
__device__ __noinline__ float ap_ratio_safe(float sx, float sy, float eps2) {
  return sqrtf(fmaxf(sy, eps2)) / sqrtf(fmaxf(sx, eps2));
}
__device__ __forceinline__ bool ap_valid(float rmin, float rmax) { return rmin > 0.f && rmax < 3.0e38f; }   // false for NaN too
__device__ __forceinline__ void ap_take(ApAcc& acc, float r) {
  acc.vmax = fmaxf(acc.vmax, r);
  acc.vmin = fminf(acc.vmin, r);
  acc.sum += r;
}

// Block-level combine into ordered per-CTA slots + last-block reduce in a FIXED order (no float atomics: results are
// bit-reproducible).  scratch: [kApMaxBlocks][4] floats, then a self-resetting ticket.
__device__ __forceinline__ void ap_finish(ApAcc acc, float* __restrict__ scratch, double* __restrict__ stats) {
  __shared__ float red[3][8];
  __shared__ unsigned cnt_red[8];
  __shared__ int last;
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
  const float vmax = warp_max(acc.vmax), vmin = warp_min(acc.vmin), vsum = warp_sum(acc.sum);
  const unsigned cnt = __reduce_add_sync(0xffffffffu, acc.cnt);
  if (l == 0) { red[0][w] = vmax; red[1][w] = vmin; red[2][w] = vsum; cnt_red[w] = cnt; }
  __syncthreads();
  unsigned* ticket = reinterpret_cast<unsigned*>(scratch + (size_t)kApMaxBlocks * 4);
  if (tid == 0) {
    float a = red[0][0], b = red[1][0], c = red[2][0];
    unsigned n = cnt_red[0];
    for (int q = 1; q < 8; ++q) { a = fmaxf(a, red[0][q]); b = fminf(b, red[1][q]); c += red[2][q]; n += cnt_red[q]; }
    float* slot = scratch + (size_t)blockIdx.x * 4;
    slot[0] = a; slot[1] = b; slot[2] = c; slot[3] = __uint_as_float(n);
    __threadfence();
    last = (atomicAdd(ticket, 1u) + 1u == gridDim.x) ? 1 : 0;
  }
  __syncthreads();
  if (last && w == 0) {
    __threadfence();
    float a = 0.f, b = 3.4e38f;
    double c = 0.0, n = 0.0;
    for (int q = l; q < (int)gridDim.x; q += 32) {            // lane-strided, then a fixed shuffle tree
      const float* slot = scratch + (size_t)q * 4;
      a = fmaxf(a, __ldcg(slot)); b = fminf(b, __ldcg(slot + 1)); c += (double)__ldcg(slot + 2);
      n += (double)__float_as_uint(__ldcg(slot + 3));
    }
    a = warp_max(a); b = warp_min(b);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { c += __shfl_xor_sync(0xffffffffu, c, o); n += __shfl_xor_sync(0xffffffffu, n, o); }
    if (l == 0) {
      const bool any = n > 0.0;
      stats[0] = any ? (double)a : 0.0;
      stats[1] = any ? (double)b : 1.7976931348623157e308;
      stats[2] = c;
      stats[3] = n;
      *ticket = 0u;                                          // ready for the next launch
    }
  }
}

__device__ __forceinline__ void ap_hist_add(uint32_t* hs, float r, int nbins, float hist_lo, float hscale) {
  int bin = (int)floorf((__log2f(r) - hist_lo) * hscale);
  bin = bin < 0 ? 0 : (bin >= nbins ? nbins - 1 : bin);
  atomicAdd(hs + bin, 1u);
}

// ---- per-pair sinks.  The tile walks below own tile enumeration, loads, masking and the key of a pair (ap_ratio when
// ap_valid holds for it, else ap_ratio_safe); a Sink decides what happens to the keys.  Interface:
//   Sink(args, hs)          prologue (hs: the kernel's dynamic shared memory)
//   take(r)                 one key
//   kTile                   whether interior 4x4 groups take the fast path below (else every pair goes through take())
//   tile_key(ii, jj, r)     the 16 ap_ratio values of an interior group, in order; then
//   tile_end(rlo, rhi)      with their min / max: takes the group and returns true, or returns false (taking nothing) when
//                           the group is not ap_valid -- the caller then redoes it pair by pair with take()
//   finish()                epilogue
enum ApHist { kHistNone, kHistShared, kHistGlobal };

// max / min / sum / count, and optionally the log2 histogram: kHistShared = per-CTA shared bins when nbins <=
// kApMaxSmemBins (else global atomics), kHistGlobal = global atomics when args.hist != NULL
template <ApHist H>
struct ApStatsSink {
  struct Args {
    float* scratch;
    double* stats;
    uint32_t* hist;
    int nbins;
    float hist_lo, hist_hi;
  };
  static constexpr bool kTile = H == kHistNone;
  const Args a;
  float hscale, rs;
  uint32_t* hdst;
  ApAcc acc;
  __device__ __forceinline__ ApStatsSink(const Args& args, uint32_t* hs)
      : a(args), hscale(0.f), hdst(hs), acc{0.f, 3.4e38f, 0.f, 0u} {
    if (H == kHistShared) {
      hscale = (float)a.nbins / (a.hist_hi - a.hist_lo);
      if (a.nbins <= kApMaxSmemBins) {
        for (int q = threadIdx.x; q < a.nbins; q += kApThreads) hs[q] = 0u;
        __syncthreads();
      } else {
        hdst = a.hist;
      }
    } else if (H == kHistGlobal) {
      hscale = a.hist ? (float)a.nbins / (a.hist_hi - a.hist_lo) : 0.f;
    }
  }
  __device__ __forceinline__ void take(float r) {
    ap_take(acc, r);
    ++acc.cnt;
    if (H == kHistShared) ap_hist_add(hdst, r, a.nbins, a.hist_lo, hscale);
    if (H == kHistGlobal && a.hist) ap_hist_add(a.hist, r, a.nbins, a.hist_lo, hscale);
  }
  __device__ __forceinline__ void tile_key(int ii, int jj, float r) { rs = (ii | jj) ? rs + r : r; }   // r0 == 0 + r0
  __device__ __forceinline__ bool tile_end(float rlo, float rhi) {
    if (!ap_valid(rlo, rhi)) return false;
    acc.vmin = fminf(acc.vmin, rlo); acc.vmax = fmaxf(acc.vmax, rhi); acc.sum += rs; acc.cnt += 16u;
    return true;
  }
  __device__ __forceinline__ void finish() {
    if (H == kHistShared && a.nbins <= kApMaxSmemBins) {
      __syncthreads();
      for (int q = threadIdx.x; q < a.nbins; q += kApThreads) { const uint32_t c = hdst[q]; if (c) atomicAdd(a.hist + q, c); }
    }
    ap_finish(acc, a.scratch, a.stats);
  }
};

// ---- exact order statistics: a 3-pass radix select on the key's bit pattern.  Keys are positive floats, so their u32
// patterns order like their values (bit 31 is 0).  Pass 0 histograms bits [30:20] (2048 bins), pass 1 bits [19:10] and pass
// 2 bits [9:0] (1024 bins per slot) of the keys whose higher bits equal a slot's prefix.  Up to 4 targets (ranks k and k+1
// of two quantiles); targets with the same prefix share a slot, i.e. bins.
constexpr int kSelTargets = 4;
constexpr int kSelBins = kSelTargets * 1024;   // histogram: [slot][1024] (pass 0: 2048 bins of slot 0)
constexpr int kSelPasses = 3;
constexpr uint32_t kSelNoSlot = 0xffffffffu;   // unused slot: no key prefix (at most 21 bits) equals it

struct SelState {                              // caller-owned device state between passes (b200vae_lipschitz_select_state_bytes)
  unsigned long long rank[kSelTargets];        // residual rank of each target among the keys that share its prefix
  uint32_t prefix[kSelTargets];                // key bits located so far
  uint32_t slot_prefix[kSelTargets];           // the count pass's slots: distinct target prefixes, kSelNoSlot if unused
  int slot[kSelTargets];                       // target -> slot
  double w[2];                                 // interpolation weights of the two quantiles
};
constexpr size_t kSelStateBytes = 128;
static_assert(sizeof(SelState) <= kSelStateBytes, "SelState outgrew its ABI size");

// torch.quantile's "linear" rule with the rank arithmetic in fp64: pos = q (n - 1), k = floor(pos), w = pos - k
__host__ __device__ __forceinline__ void quantile_rank(long long n, double q, long long& k, double& w) {
  const double pos = q * (double)(n - 1);
  long long kk = (long long)floor(pos);
  kk = kk < 0 ? 0 : (kk > n - 1 ? n - 1 : kk);
  k = kk;
  w = pos - (double)kk;
}

struct ApSelectSink {
  struct Args {
    const SelState* state;
    unsigned long long* hist;
    int pass;
  };
  static constexpr bool kTile = true;
  uint32_t* bins;
  unsigned long long* hist;
  uint32_t p0, p1, p2, p3;                     // slot prefixes
  int hi_sh, lo_sh, nbins;
  uint32_t fmask;
  float r[4][4];                               // the keys of an interior group
  __device__ __forceinline__ ApSelectSink(const Args& a, uint32_t* hs) : bins(hs), hist(a.hist) {
    if (a.pass == 0) {
      p0 = 0u; p1 = p2 = p3 = kSelNoSlot;
      hi_sh = 31; lo_sh = 20; fmask = 2047u; nbins = 2048;
    } else {
      p0 = a.state->slot_prefix[0]; p1 = a.state->slot_prefix[1];
      p2 = a.state->slot_prefix[2]; p3 = a.state->slot_prefix[3];
      hi_sh = a.pass == 1 ? 20 : 10; lo_sh = hi_sh - 10; fmask = 1023u; nbins = kSelBins;
    }
    for (int q = threadIdx.x; q < nbins; q += kApThreads) bins[q] = 0u;
    __syncthreads();
  }
  __device__ __forceinline__ int bin_of(float r) const {
    const uint32_t key = __float_as_uint(r), hi = key >> hi_sh, f = (key >> lo_sh) & fmask;
    return hi == p0 ? (int)f : hi == p1 ? 1024 + (int)f : hi == p2 ? 2048 + (int)f : hi == p3 ? 3072 + (int)f : -1;
  }
  __device__ __forceinline__ void take(float r) {
    const int b = bin_of(r);
    if (b >= 0) atomicAdd(bins + b, 1u);
  }
  __device__ __forceinline__ void tile_key(int ii, int jj, float key) { r[ii][jj] = key; }
  // One shared atomic per counted key.  Ratios concentrate in a few pass-0 bins (a factor 2 of ratio spans 8 of them), but
  // aggregating the lanes of a warp that share a bin (__match_any_sync, one add per distinct bin) made pass 0 twice as slow
  // on a B200 (N = 50000: 3.19 vs 1.54 ms), so the plain atomic stays.
  __device__ __forceinline__ bool tile_end(float rlo, float rhi) {
    if (!ap_valid(rlo, rhi)) return false;
#pragma unroll
    for (int ii = 0; ii < 4; ++ii)
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) take(r[ii][jj]);
    return true;
  }
  __device__ __forceinline__ void finish() {
    __syncthreads();
    for (int q = threadIdx.x; q < nbins; q += kApThreads) {
      const uint32_t c = bins[q];
      if (c) atomicAdd(hist + q, (unsigned long long)c);
    }
  }
};

// ---- small feature widths (DX, DY <= 4): everything in registers, operands straight from global memory (L1 / L2
// resident: N*(DX+DY)*4 bytes).  A CTA owns a CONTIGUOUS range of tile indices, i.e. it walks along a tile row: the 4 i-points
// of a thread (i0 + 4 ta + ii) stay in registers while only its 4 j-points (j0 + 4 tb + jj, contiguous -> wide loads) are
// reloaded per tile, and the tile coordinates advance incrementally.  Interior tiles (every pair valid) take the fast path:
// 16 ratios handed to the sink at once; diagonal and edge tiles (and sinks without a fast path) the masked, exact-division path.
template <int DX, int DY, class Sink>
__global__ void __launch_bounds__(kApThreads, 4)
lipschitz_allpairs_small_kernel(const float* __restrict__ X, const float* __restrict__ Y, int N, float eps,
                                long long tile_begin, long long tile_end, const typename Sink::Args args, int vec_ok) {
  extern __shared__ uint32_t hs[];               // the sink's per-CTA bins, if any
  const int T = (N + kTile - 1) / kTile;
  const int tid = threadIdx.x, ta = tid >> 4, tb = tid & 15;
  const float eps2 = eps * eps;
  Sink sink(args, hs);
  // 4 consecutive points: vector loads when all four exist (g0 is a multiple of 4, so 4*DIM floats are 16-byte aligned if
  // the base pointer is), else clamped scalar loads (out-of-range points are masked by the slow path)
  auto load4 = [&](const float* __restrict__ F, int g0, auto& f) {
    constexpr int DIM = sizeof(f[0]) / sizeof(float);
    if (vec_ok && g0 + 3 < N) {
      const float4* src = reinterpret_cast<const float4*>(F + (size_t)g0 * DIM);
      float flat[4 * DIM];
#pragma unroll
      for (int q = 0; q < DIM; ++q) {
        const float4 t = __ldg(src + q);
        flat[4 * q] = t.x; flat[4 * q + 1] = t.y; flat[4 * q + 2] = t.z; flat[4 * q + 3] = t.w;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int q = 0; q < DIM; ++q) f[k][q] = flat[k * DIM + q];
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int gc = g0 + k < N ? g0 + k : N - 1;
#pragma unroll
        for (int q = 0; q < DIM; ++q) f[k][q] = __ldg(F + (size_t)gc * DIM + q);
      }
    }
  };
  const long long nt = tile_end - tile_begin;
  const long long per = (nt + gridDim.x - 1) / gridDim.x;
  const long long t0 = tile_begin + (long long)blockIdx.x * per;
  const long long t1 = t0 + per < tile_end ? t0 + per : tile_end;
  int ti = 0, tj = 0;
  float xi[4][DX], yi[4][DY];
  if (t0 < t1) {
    tile_coords(t0, T, ti, tj);
    load4(X, ti * kTile + 4 * ta, xi); load4(Y, ti * kTile + 4 * ta, yi);
  }
  for (long long t = t0; t < t1; ++t) {
    const int i0 = ti * kTile + 4 * ta, j0 = tj * kTile + 4 * tb;
    float xj[4][DX], yj[4][DY];
    load4(X, j0, xj); load4(Y, j0, yj);
    auto sq = [&](int ii, int jj, float& ax, float& ay) {
      ax = 0.f; ay = 0.f;
#pragma unroll
      for (int q = 0; q < DX; ++q) { const float d = xi[ii][q] - xj[jj][q]; ax = fmaf(d, d, ax); }
#pragma unroll
      for (int q = 0; q < DY; ++q) { const float d = yi[ii][q] - yj[jj][q]; ay = fmaf(d, d, ay); }
    };
    const bool full = (ti != tj) && (tj * kTile + kTile <= N);  // every pair valid (i < j, both in range)
    bool done = false;
    if (full && Sink::kTile) {
      float rlo = 3.4e38f, rhi = 0.f;
#pragma unroll
      for (int ii = 0; ii < 4; ++ii)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          float ax, ay;
          sq(ii, jj, ax, ay);
          const float r = ap_ratio(ax, ay, eps2);
          rlo = fminf(rlo, r); rhi = fmaxf(rhi, r);
          sink.tile_key(ii, jj, r);
        }
      done = sink.tile_end(rlo, rhi);
    }
    if (!done) {                                                // diagonal / edge tile, histogram, or a*b out of range
#pragma unroll
      for (int ii = 0; ii < 4; ++ii)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj)
          if (i0 + ii < j0 + jj && j0 + jj < N) {
            float ax, ay;
            sq(ii, jj, ax, ay);
            float r = ap_ratio(ax, ay, eps2);
            if (!ap_valid(r, r)) r = ap_ratio_safe(ax, ay, eps2);
            sink.take(r);
          }
    }
    if (++tj == T) {                                            // next tile row: its first tile is the diagonal one
      ++ti; tj = ti;
      if (t + 1 < t1) { load4(X, ti * kTile + 4 * ta, xi); load4(Y, ti * kTile + 4 * ta, yi); }
    }
  }
  sink.finish();
}

// ---- any feature widths: 64 x 64 tile, the feature axis staged through shared memory in chunks of kApChunk, [q][point]
// layout (conflict-free: a warp reads 2 broadcast i-rows and 16 consecutive j-points), 4 x 4 accumulator pairs per thread.
constexpr int kApChunk = 32;
template <class Sink>
__global__ void __launch_bounds__(kApThreads)
lipschitz_allpairs_wide_kernel(const float* __restrict__ X, const float* __restrict__ Y, int N, int dx, int dy, float eps,
                               long long tile_begin, long long tile_end, const typename Sink::Args args) {
  __shared__ float Fi[kApChunk][kTile + 1], Fj[kApChunk][kTile + 1];
  extern __shared__ uint32_t hs[];               // the sink's per-CTA bins, if any
  const int T = (N + kTile - 1) / kTile;
  const int tid = threadIdx.x, ta = tid >> 4, tb = tid & 15;
  const float eps2 = eps * eps;
  Sink sink(args, hs);
  for (long long t = tile_begin + blockIdx.x; t < tile_end; t += gridDim.x) {
    int ti, tj;
    tile_coords(t, T, ti, tj);
    const int i0 = ti * kTile, j0 = tj * kTile;
    float s[2][4][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int ii = 0; ii < 4; ++ii)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) s[m][ii][jj] = 0.f;
#pragma unroll 1
    for (int m = 0; m < 2; ++m) {                              // m = 0: X (sx), m = 1: Y (sy)
      const float* F = m ? Y : X;
      const int dim = m ? dy : dx;
      for (int c0 = 0; c0 < dim; c0 += kApChunk) {
        const int cw = min(kApChunk, dim - c0);
        __syncthreads();
        for (int id = tid; id < kTile * kApChunk; id += kApThreads) {
          const int pt = id / kApChunk, q = id - pt * kApChunk;          // consecutive threads: consecutive features
          const bool inq = q < cw;
          Fi[q][pt] = (inq && i0 + pt < N) ? __ldg(F + (size_t)(i0 + pt) * dim + c0 + q) : 0.f;
          Fj[q][pt] = (inq && j0 + pt < N) ? __ldg(F + (size_t)(j0 + pt) * dim + c0 + q) : 0.f;
        }
        __syncthreads();
        for (int q = 0; q < cw; ++q) {
          float fi[4], fj[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) { fi[k] = Fi[q][ta + 16 * k]; fj[k] = Fj[q][tb + 16 * k]; }
#pragma unroll
          for (int ii = 0; ii < 4; ++ii)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const float d = fi[ii] - fj[jj];
              if (m == 0) s[0][ii][jj] = fmaf(d, d, s[0][ii][jj]);
              else s[1][ii][jj] = fmaf(d, d, s[1][ii][jj]);
            }
        }
      }
    }
#pragma unroll
    for (int ii = 0; ii < 4; ++ii)
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const int gi = i0 + ta + 16 * ii, gj = j0 + tb + 16 * jj;
        if (gi < gj && gj < N) {
          float r = ap_ratio(s[0][ii][jj], s[1][ii][jj], eps2);
          if (!ap_valid(r, r)) r = ap_ratio_safe(s[0][ii][jj], s[1][ii][jj], eps2);
          sink.take(r);
        }
      }
  }
  sink.finish();
}

// One CTA, after each count pass: warp t finds the bin that holds target t's residual rank in its slot's bins, then the
// prefix grows by that bin and the rank becomes the residual within it.  Pass 0 first sets the targets from (N, q0, q1);
// the last pass writes out = (v(q0), v(q1), key[k0], key[k0 + 1], key[k1], key[k1 + 1]) in fp64.
__global__ void __launch_bounds__(128)
lipschitz_select_locate_kernel(int N, double q0, double q1, int pass, const unsigned long long* __restrict__ hist,
                               SelState* __restrict__ state, double* __restrict__ out) {
  __shared__ unsigned long long bins[kSelBins];
  __shared__ SelState S;
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
  if (tid == 0) {
    if (pass == 0) {
      const long long n = (long long)N * (N - 1) / 2;
      long long k0, k1;
      quantile_rank(n, q0, k0, S.w[0]);
      quantile_rank(n, q1, k1, S.w[1]);
      S.rank[0] = k0; S.rank[1] = k0 + 1 < n ? k0 + 1 : n - 1;
      S.rank[2] = k1; S.rank[3] = k1 + 1 < n ? k1 + 1 : n - 1;
      for (int t = 0; t < kSelTargets; ++t) { S.prefix[t] = 0u; S.slot[t] = 0; S.slot_prefix[t] = t ? kSelNoSlot : 0u; }
    } else {
      S = *state;
    }
  }
  const int nb = pass == 0 ? 2048 : kSelBins;
  for (int q = tid; q < nb; q += blockDim.x) bins[q] = __ldcg(hist + q);
  __syncthreads();
  if (w < kSelTargets) {
    const int width = pass == 0 ? 2048 : 1024, base = S.slot[w] * 1024;
    const unsigned long long rank = S.rank[w];
    unsigned long long run = 0ull;
    int bin = width - 1;
    unsigned long long res = 0ull;
    for (int c0 = 0; c0 < width; c0 += 32) {
      const unsigned long long c = bins[base + c0 + l];
      unsigned long long incl = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
        if (l >= o) incl += v;
      }
      const unsigned long long tot = __shfl_sync(0xffffffffu, incl, 31);
      if (run + tot > rank) {                                  // warp-uniform
        const unsigned hit = __ballot_sync(0xffffffffu, run + incl > rank);
        const int src = __ffs(hit) - 1;
        bin = c0 + src;
        res = rank - (run + __shfl_sync(0xffffffffu, incl - c, src));
        break;
      }
      run += tot;
    }
    if (l == 0) {
      S.rank[w] = res;
      S.prefix[w] = (S.prefix[w] << (pass == 0 ? 11 : 10)) | (uint32_t)bin;
    }
  }
  __syncthreads();
  if (tid == 0) {
    int ns = 0;                                                 // the next pass's slots, in target order
    for (int t = 0; t < kSelTargets; ++t) {
      int s = 0;
      while (s < ns && S.slot_prefix[s] != S.prefix[t]) ++s;
      if (s == ns) S.slot_prefix[ns++] = S.prefix[t];
      S.slot[t] = s;
    }
    for (int s = ns; s < kSelTargets; ++s) S.slot_prefix[s] = kSelNoSlot;
    *state = S;
    if (pass == kSelPasses - 1) {
      double key[kSelTargets];
      for (int t = 0; t < kSelTargets; ++t) { key[t] = (double)__uint_as_float(S.prefix[t]); out[2 + t] = key[t]; }
      // key_k + w (key_k+1 - key_k), rounded step by step (no contraction into an FMA)
      out[0] = __dadd_rn(key[0], __dmul_rn(S.w[0], __dsub_rn(key[1], key[0])));
      out[1] = __dadd_rn(key[2], __dmul_rn(S.w[1], __dsub_rn(key[3], key[2])));
    }
  }
}

}  // namespace b200vae

using namespace b200vae;

extern "C" int b200vae_lipschitz_pairs(const float* X, const float* Y, const int64_t* i1, const int64_t* i2, int P,
                                       int N, int dx, int dy, float eps, float* ratio, void* stream) {
  if (!X || !Y || !i1 || !i2 || !ratio) return B200VAE_EALIGN;
  if (P <= 0 || N <= 0 || dx <= 0 || dy <= 0) return B200VAE_ESHAPE;
  int blocks = (P + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  lipschitz_pairs_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(X, Y, i1, i2, P, N, dx, dy, eps, ratio);
  return check_launch();
}

extern "C" long long b200vae_lipschitz_num_tiles(int N) {
  const long long T = (N + kTile - 1) / kTile;
  return T * (T + 1) / 2;
}

extern "C" size_t b200vae_lipschitz_scratch_bytes(void) { return ((size_t)kApMaxBlocks * 4 + 4) * sizeof(float); }

// one wave of resident CTAs (4 per SM: __launch_bounds__(256, 4)); a CTA walks a contiguous range of tiles, so at least ~2
// tiles per CTA keep the per-CTA prologue / epilogue amortised
static int ap_blocks(long long nt) {
  const int per_sm = 4;
  long long want = nt < 1 ? 1 : (nt + 1) / 2;
  const long long cap = (long long)sm_count() * per_sm;
  return (int)(want < cap ? want : (cap < kApMaxBlocks ? cap : kApMaxBlocks));
}

// One launch of the small-width tile walk over [tb, te) with `Sink` (dx, dy <= 4) ...
template <class Sink>
static int launch_ap_small(const float* X, const float* Y, int N, int dx, int dy, float eps, long long tb, long long te,
                           const typename Sink::Args& args, size_t smem, int blocks, cudaStream_t st) {
  const int vec_ok = (aligned16(X) && aligned16(Y)) ? 1 : 0;
#define B200VAE_AP(DX_, DY_)                                                                                          \
  lipschitz_allpairs_small_kernel<DX_, DY_, Sink><<<blocks, kApThreads, smem, st>>>(X, Y, N, eps, tb, te, args, vec_ok); \
  return check_launch()
#define B200VAE_APX(DX_) \
  switch (dy) { case 1: B200VAE_AP(DX_, 1); case 2: B200VAE_AP(DX_, 2); case 3: B200VAE_AP(DX_, 3); default: B200VAE_AP(DX_, 4); }
  switch (dx) {
    case 1: B200VAE_APX(1)
    case 2: B200VAE_APX(2)
    case 3: B200VAE_APX(3)
    default: B200VAE_APX(4)
  }
#undef B200VAE_APX
#undef B200VAE_AP
}
// ... and of the any-width one
template <class Sink>
static int launch_ap_wide(const float* X, const float* Y, int N, int dx, int dy, float eps, long long tb, long long te,
                          const typename Sink::Args& args, size_t smem, int blocks, cudaStream_t st) {
  lipschitz_allpairs_wide_kernel<Sink><<<blocks, kApThreads, smem, st>>>(X, Y, N, dx, dy, eps, tb, te, args);
  return check_launch();
}

extern "C" int b200vae_lipschitz_allpairs(const float* X, const float* Y, int N, int dx, int dy, float eps,
                                          long long tile_begin, long long tile_end, double* stats, uint32_t* hist,
                                          int nbins, float hist_lo, float hist_hi, void* scratch, void* stream) {
  if (!X || !Y || !stats || !scratch || !aligned16(scratch)) return B200VAE_EALIGN;
  if (N <= 0 || dx <= 0 || dy <= 0 || tile_begin < 0 || tile_end < tile_begin ||
      tile_end > b200vae_lipschitz_num_tiles(N))
    return B200VAE_ESHAPE;
  if (hist && (nbins <= 0 || !(hist_hi > hist_lo))) return B200VAE_ESHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  if (hist && cudaMemsetAsync(hist, 0, (size_t)nbins * sizeof(uint32_t), st) != cudaSuccess) return B200VAE_ECUDA;
  // one launch, even for an empty tile range (the kernel then only writes the neutral statistics)
  const int blocks = ap_blocks(tile_end - tile_begin);
  float* scr = reinterpret_cast<float*>(scratch);
  if (dx <= 4 && dy <= 4) {
    if (hist) {
      const size_t smem = nbins <= kApMaxSmemBins ? (size_t)nbins * 4 : 0;
      return launch_ap_small<ApStatsSink<kHistShared>>(X, Y, N, dx, dy, eps, tile_begin, tile_end,
                                                       {scr, stats, hist, nbins, hist_lo, hist_hi}, smem, blocks, st);
    }
    return launch_ap_small<ApStatsSink<kHistNone>>(X, Y, N, dx, dy, eps, tile_begin, tile_end,
                                                   {scr, stats, hist, nbins, hist_lo, hist_hi}, 0, blocks, st);
  }
  return launch_ap_wide<ApStatsSink<kHistGlobal>>(X, Y, N, dx, dy, eps, tile_begin, tile_end,
                                                  {scr, stats, hist, nbins, hist_lo, hist_hi}, 0, blocks, st);
}

// ---- exact quantiles of the keys: count (shardable) / locate, three passes
extern "C" size_t b200vae_lipschitz_select_state_bytes(void) { return kSelStateBytes; }
extern "C" size_t b200vae_lipschitz_select_hist_bytes(void) { return (size_t)kSelBins * sizeof(uint64_t); }

extern "C" int b200vae_lipschitz_quantile_ranks(long long n, double q, long long* k, double* w) {
  if (!k || !w) return B200VAE_EALIGN;
  if (n < 1 || !(q >= 0.0 && q <= 1.0)) return B200VAE_ESHAPE;
  quantile_rank(n, q, *k, *w);
  return B200VAE_OK;
}

extern "C" int b200vae_lipschitz_select_count(const float* X, const float* Y, int N, int dx, int dy, float eps,
                                              long long tile_begin, long long tile_end, int pass, const void* state,
                                              uint64_t* hist, void* stream) {
  if (!X || !Y || !state || !hist || !aligned16(state) || !aligned16(hist)) return B200VAE_EALIGN;
  if (N < 2 || dx <= 0 || dy <= 0 || !(eps > 0.f) || pass < 0 || pass >= kSelPasses || tile_begin < 0 ||
      tile_end < tile_begin || tile_end > b200vae_lipschitz_num_tiles(N))
    return B200VAE_ESHAPE;
  const long long nt = tile_end - tile_begin;
  const int blocks = ap_blocks(nt);
  // the per-CTA shared bins are uint32: one CTA may see at most 2^32 - 1 pairs (every N below ~2 million points)
  if ((nt + blocks - 1) / blocks * (long long)(kTile * kTile) > 0xffffffffLL) return B200VAE_EUNSUP;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(hist, 0, b200vae_lipschitz_select_hist_bytes(), st) != cudaSuccess) return B200VAE_ECUDA;
  const size_t smem = (size_t)(pass == 0 ? 2048 : kSelBins) * sizeof(uint32_t);
  const ApSelectSink::Args args{reinterpret_cast<const SelState*>(state), reinterpret_cast<unsigned long long*>(hist), pass};
  if (dx <= 4 && dy <= 4) return launch_ap_small<ApSelectSink>(X, Y, N, dx, dy, eps, tile_begin, tile_end, args, smem, blocks, st);
  return launch_ap_wide<ApSelectSink>(X, Y, N, dx, dy, eps, tile_begin, tile_end, args, smem, blocks, st);
}

extern "C" int b200vae_lipschitz_select_locate(int N, double q0, double q1, int pass, const uint64_t* hist, void* state,
                                               double* out, void* stream) {
  if (!hist || !state || !out || !aligned16(state) || !aligned16(hist) || (reinterpret_cast<uintptr_t>(out) & 7u))
    return B200VAE_EALIGN;
  if (N < 2 || !(q0 >= 0.0 && q0 <= 1.0) || !(q1 >= 0.0 && q1 <= 1.0) || pass < 0 || pass >= kSelPasses)
    return B200VAE_ESHAPE;
  lipschitz_select_locate_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(N, q0, q1, pass,
                                                                      reinterpret_cast<const unsigned long long*>(hist),
                                                                      reinterpret_cast<SelState*>(state), out);
  return check_launch();
}
