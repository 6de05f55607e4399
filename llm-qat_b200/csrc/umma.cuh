// umma.cuh — PTX wrappers shared by the tcgen05 kernels of libqat_b200 (sm_100a):
// mbarriers, TMA (cp.async.bulk.tensor), tcgen05.mma / commit / ld / st, TMEM
// allocation, shared-memory matrix descriptors and instruction descriptors.
// Used by tcgen05_gemm.cuh (the GEMM pipeline of qlinear_gemm.cu and gemm_bf16.cu)
// and attention.cu (QK^T / PV and their backward, kind::f16).
#pragma once
#include <cuda.h>

#include <cstdio>
#include <mutex>

#include "common.cuh"

namespace qat {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> launch failure the host reports)
// instead of hanging the GPU.  ~4 s at 2 GHz; never reached in a correct run.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try(bar, parity)) {
    if (clock64() - t0 > 8000000000ll) {
      printf("libqat_b200: mbarrier timeout (block %d,%d thread %d bar 0x%x parity %u)\n", blockIdx.x,
             blockIdx.y, threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// cta_group::2: executed by both CTAs of the pair; the mbarrier operand has the
// peer bit (24) of its shared::cluster address cleared, so the transaction
// bytes land on the LEADER CTA's barrier wherever the data lands.
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                                 int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(rank)
      : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// generic-proxy shared-memory writes -> visible to the async proxy (tcgen05.mma / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// arrives (once the MMAs issued so far retire) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, int8 x int8 -> s32
template <int CG>
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  if (CG == 1) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> f32
template <int CG>
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  if (CG == 1) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),
        "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),
        "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]),
        "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_cg1(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_cg1(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}

// ---- shared-memory matrix descriptors (version 1 = sm_100, SWIZZLE_128B) --------------------
// K-major operand tile whose rows are 128 bytes (one swizzle atom wide, what a TMA box of
// {128 B, rows} with CU_TENSOR_MAP_SWIZZLE_128B writes): 8-row groups are 1024 bytes apart
// (SBO); LBO is unused for swizzled K-major layouts (encoded 1, as CUTLASS does).  One MMA
// consumes 32 bytes of K: advance the start-address field by 2 per UMMA_K step.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffffu) >> 4);   // [0,14)  start address >> 4
  d |= (uint64_t)1 << 16;                      // [16,30) leading byte offset >> 4
  d |= (uint64_t)(1024u >> 4) << 32;           // [32,46) stride byte offset >> 4
  d |= (uint64_t)1 << 46;                      // [46,48) descriptor version
  d |= (uint64_t)2 << 61;                      // [61,64) SWIZZLE_128B
  return d;
}
// MN-major operand tile (16-bit elements): the contraction index runs over ROWS of 128 bytes
// (64 consecutive M/N elements), i.e. what a TMA box of {64 elements of M/N, rows of K} writes from a
// row-major [K, MN] matrix.  Canonical layout (CUTLASS make_umma_desc<Major::MN>, SW128), in
// 16-byte units: ((8, n), (8, k)) : ((1, LBO), (8, SBO)) — a swizzle atom is 8 K-rows x 128 B;
// SBO = bytes between consecutive groups of 8 K-rows (1024 when the box rows are contiguous),
// LBO = bytes between consecutive 64-element chunks of M/N (= one whole box).  One MMA (K = 16)
// consumes 16 rows = 2048 B: advance the start-address field by 128 per UMMA_K step.
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffffu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::i8 instruction descriptor: s32 accumulate, signed int8 A and B, both K-major
__host__ __device__ constexpr uint32_t make_idesc_i8(int m, int n) {
  return (2u << 4)                  // c_format  = S32
         | (1u << 7) | (1u << 10)   // a_format = b_format = INT8 (signed)
         | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// kind::f16 instruction descriptor: f32 accumulate, bf16 A and B; a_mn / b_mn = 1 for an MN-major operand
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n, int a_mn, int b_mn) {
  return (1u << 4)                  // c_format  = F32
         | (1u << 7) | (1u << 10)   // a_format = b_format = BF16
         | ((uint32_t)(a_mn & 1) << 15) | ((uint32_t)(b_mn & 1) << 16)
         | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---- host: cuTensorMapEncodeTiled through the runtime (no link against libcuda) ------------
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                              const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                              CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                              CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled is a DRIVER call: it fails with CUDA_ERROR_INVALID_CONTEXT on a thread that has not
// touched the runtime yet (autograd's backward thread, when a tensor-map encode is the first CUDA call it
// makes).  cudaFree(0) binds the device's primary context to the calling thread; ~100 ns once bound.
inline void bind_context() { (void)cudaFree(nullptr); }

inline EncodeFn get_encode() {
  bind_context();
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  });
  return fn;
}

// Row-major matrix [rows, cols] of bf16 (elem_bytes = 2) or int8 (elem_bytes = 1) with a row pitch
// of `pitch_elems` -> 2-D map with a {128 B, box_rows} box, 128B swizzle.  OOB reads fill zeros.
inline int make_map_2d(CUtensorMap* map, int elem_bytes, const void* ptr, int64_t rows, int64_t cols,
                       int64_t pitch_elems, int box_rows) {
  EncodeFn enc = get_encode();
  if (enc == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return QAT_ERR_UNSUPPORTED;
  }
  const bool bf16 = elem_bytes == 2;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * elem_bytes};
  cuuint32_t box[2] = {128u / elem_bytes, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2,
                   const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) for %s [%lld, %lld] pitch %lld box_rows %d", (int)r,
              bf16 ? "bf16" : "int8", (long long)rows, (long long)cols, (long long)pitch_elems, box_rows);
    return QAT_ERR_BAD_ARG;
  }
  return QAT_OK;
}

// The opt-in to more than 48 KB of dynamic shared memory is per function AND per device.  `done`
// is the caller's per-kernel record of the devices already opted in (a benign race: idempotent).
template <typename Kern>
int opt_in_smem(Kern kern, uint32_t bytes, bool (&done)[64], const char* name) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  if (dev < 0 || dev >= 64 || !done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      char what[96];
      snprintf(what, sizeof(what), "cudaFuncSetAttribute(%s)", name);
      return cuda_fail(e, what);
    }
    if (dev >= 0 && dev < 64) done[dev] = true;
  }
  return QAT_OK;
}

}  // namespace umma
}  // namespace qat
