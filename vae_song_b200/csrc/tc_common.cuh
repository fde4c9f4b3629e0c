// tc_common.cuh -- PTX wrappers (mbarrier, TMA, tcgen05, TMEM) and small helpers shared by the tensor-core kernels.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace b200vae {

constexpr int kKB = 16;           // K elements per block (64 B rows, SWIZZLE_64B)

// ------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
// long waits (epilogue warps waiting for a whole accumulator pass): let the hardware park the warp for up to
// `ns` nanoseconds per try instead of re-issuing the poll every few dozen cycles next to the MMA-issuing warp
__device__ __forceinline__ void mbar_wait_parked(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity), "r"(ns) : "memory");
  } while (!ok);
}
// one lane of a CONVERGED warp (CUTLASS elect_one_sync): inside `if (elect_one())` the compiler knows a single lane
// is active, so the uniform-register operands of UTCHMMA / UTMALDG need no ELECT + R2UR.BROADCAST retry loops
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

// round-to-nearest (ties away) to tf32 in one integer add: tcgen05 kind::tf32 ignores the 13 low mantissa bits
__device__ __forceinline__ float rn_tf32_fast(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }
__device__ __forceinline__ float rn_tf32_masked(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }

// K-major, SWIZZLE_64B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO(1)<<16 |
// SBO(512 B >> 4)<<32 | version(1)<<46 | layout SWIZZLE_64B(4)<<61.  8-row atoms of 64-byte rows.
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)4 << 61);
}

// ------------------------------------------------------------------------------------ host: TMA descriptors
// 2-D tensor [rows][K] of fp32 (or fp16) elements, row stride `ld` elements; boxes of 64 bytes of K x box_rows rows,
// 64-byte swizzle, zero fill outside the tensor.  The driver entry point is looked up through the runtime (no -lcuda).
inline int tma_map_2d(CUtensorMap* m, const void* base, int K, int rows, int ld, int box_rows, bool f16 = false) {
  typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static const EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess;
    return ok ? reinterpret_cast<EncodeTiledFn>(p) : nullptr;
  }();
  if (!fn) return B200VAE_ECUDA;
  const size_t esize = f16 ? 2 : sizeof(float);
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * esize};
  const cuuint32_t box[2] = {(cuuint32_t)(64 / esize), (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { g_last_cuda_error = 100000 + (int)r; return B200VAE_ECUDA; }
  return B200VAE_OK;
}

template <int D>
__device__ __forceinline__ float lin_of(const float4 q, const float (&z)[D]) {
  float h = q.w;
  h = fmaf(q.x, z[0], h);
  if (D > 1) h = fmaf(q.y, z[D > 1 ? 1 : 0], h);
  if (D > 2) h = fmaf(q.z, z[D > 2 ? 2 : 0], h);
  return h;
}
__device__ __forceinline__ float comp(const float4 q, int j) { return j == 0 ? q.x : (j == 1 ? q.y : q.z); }

}  // namespace b200vae
