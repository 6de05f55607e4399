// gemm_bf16.cu — the two backward contractions of QuantizeLinear on tcgen05 (kind::f16).
//
// Replaces what autograd runs for /root/reference/models/utils_quant.py:250
// `F.linear(x_q, W_q)` in backward — two cuBLAS bf16 GEMMs — followed by the STE clip
// masks of utils_quant.py:83-87 (clone + 2 compares + 2 masked fills per operand):
//     dgrad:  gx[T, K] = mask_x .* ( g[T, N] . W_q[N, K] )       A K-major,  B MN-major
//     wgrad:  gw[N, K] = mask_w .* ( g[T, N]^T . x_q[T, K] )     A MN-major, B MN-major
// Both read their operands exactly as they lie in HBM (no transposed copies): the
// contraction index of an MN-major operand runs over rows of the row-major matrix,
// which is what tcgen05's MN-major shared-memory descriptor consumes (umma.cuh).
// The packed STE mask the forward emitted (1 bit per element) is applied in the
// epilogue, on the fp32 accumulator, so no separate masking pass exists.
//
// C[M, N] = sum_k A(m, k) * B(n, k), fp32 accumulation in TMEM:
//   A_MN = false: A is row-major [M, K];   A_MN = true: A is row-major [K, M]
//   B_MN = false: B is row-major [N, K];   B_MN = true: B is row-major [K, N]
// Structure = K4's (qlinear_gemm.cu): persistent, one CTA per SM, warp 0 TMA producer,
// warp 1 single-thread MMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue overlapped
// with the next tile through a double-buffered accumulator; CG = 2 pairs the two CTAs
// of a cluster on one 256x256 tile (tcgen05.mma.cta_group::2).
// Tensor-bound: 2*M*N*K flops against the bf16 dense peak.
#define QAT_PDL_FAMILY 5   // bit of QAT_B200_PDL_MASK (common.cuh)
#include <cstdlib>

#include "umma.cuh"

namespace qat {
namespace {
using namespace umma;

constexpr int BLOCK_M = 128;   // accumulator rows per CTA (TMEM lanes)
constexpr int BLOCK_N = 256;   // accumulator columns per tile
constexpr int BLOCK_K = 64;    // bf16 elements per k-block: 128 bytes, one swizzle row
constexpr int UMMA_K = 16;     // elements per tcgen05.mma.kind::f16
constexpr int kAccStages = 2;
constexpr int kTmemCols = kAccStages * BLOCK_N;   // 512
constexpr int kThreads = 256;
constexpr int kEpiWarp0 = 4;
constexpr int kEpiWarps = 4;
constexpr uint32_t kChunkBytes = 64 * BLOCK_K * 2;   // one MN-major TMA box: 64 K-rows x 128 B = 8 KB

template <int CG>
struct Cfg {
  static constexpr int kStages = CG == 1 ? 4 : 6;
  static constexpr int kTileM = BLOCK_M * CG;
  static constexpr int kBRows = BLOCK_N / CG;                     // B rows (N) staged by each CTA
  static constexpr uint32_t kABytes = BLOCK_M * BLOCK_K * 2;      // 16 KB
  static constexpr uint32_t kBBytes = kBRows * BLOCK_K * 2;       // 32 KB | 16 KB
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static __host__ __device__ constexpr uint32_t a(int s) { return (uint32_t)s * kStageBytes; }
  static __host__ __device__ constexpr uint32_t b(int s) { return (uint32_t)s * kStageBytes + kABytes; }
  static constexpr uint32_t bars = kStages * kStageBytes;
  static __host__ __device__ constexpr uint32_t full(int s) { return bars + 8u * s; }
  static __host__ __device__ constexpr uint32_t empty(int s) { return bars + 8u * (kStages + s); }
  static __host__ __device__ constexpr uint32_t tfull(int a) { return bars + 8u * (2 * kStages + a); }
  static __host__ __device__ constexpr uint32_t tempty(int a) { return bars + 8u * (2 * kStages + kAccStages + a); }
  static constexpr uint32_t tmem_ptr = bars + 8u * (2 * kStages + 2 * kAccStages);
  static constexpr uint32_t total = tmem_ptr + 16;
  static constexpr uint32_t kSmemBytes = total + 1024;
};
static_assert(Cfg<1>::kSmemBytes <= 232448 && Cfg<2>::kSmemBytes <= 232448, "over the 227 KB per-CTA limit");

struct Params {
  void* out;             // [M, N] row-major, bf16 or fp32
  const uint8_t* mask;   // optional packed pass-mask over the flattened [M, N] output (bit i%8 of byte i/8)
  int64_t M, N, K;
  int out_dtype;
  int m_blocks, n_blocks, k_blocks;
};

// 32 consecutive mask bits starting at flat element index i0 (any alignment)
__device__ __forceinline__ uint32_t mask_bits32(const uint8_t* mask, int64_t i0, int64_t nbytes) {
  const int64_t b0 = i0 >> 3;
  uint64_t w = 0;
#pragma unroll
  for (int j = 0; j < 5; ++j)
    if (b0 + j < nbytes) w |= (uint64_t)mask[b0 + j] << (8 * j);
  return (uint32_t)(w >> (i0 & 7));
}

__device__ __forceinline__ void store_chunk(const Params& p, int64_t row, int64_t col0, const uint32_t (&acc)[32],
                                            bool vec_ok) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
  if (p.mask != nullptr) {
    const uint32_t bits = mask_bits32(p.mask, row * p.N + col0, (p.M * p.N + 7) >> 3);
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (!((bits >> j) & 1u)) v[j] = 0.f;
  }
  if (p.out_dtype == QAT_BF16) {
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + row * p.N + col0;
    if (vec_ok && col0 + 32 <= p.N) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint4 o;
        o.x = pack_bf16x2(v[j], v[j + 1]);
        o.y = pack_bf16x2(v[j + 2], v[j + 3]);
        o.z = pack_bf16x2(v[j + 4], v[j + 5]);
        o.w = pack_bf16x2(v[j + 6], v[j + 7]);
        *reinterpret_cast<uint4*>(dst + j) = o;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < p.N) dst[j] = __float2bfloat16_rn(v[j]);
    }
  } else {
    float* dst = reinterpret_cast<float*>(p.out) + row * p.N + col0;
    if (vec_ok && col0 + 32 <= p.N) {
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < p.N) dst[j] = v[j];
    }
  }
}

template <int CG>
__device__ __forceinline__ void tma_any(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1) {
  if (CG == 1) tma_load_2d(dst, map, bar, c0, c1); else tma_load_2d_pair(dst, map, bar, c0, c1);
}

template <bool A_MN, bool B_MN, int CG>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const Params p) {
  using C = Cfg<CG>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;
  const int unit = (CG == 2) ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int num_units = (CG == 2) ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int num_tiles = p.m_blocks * p.n_blocks;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
  }
  if (warp == 1 && lane == 0) {
#pragma unroll
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(base + C::full(s), 1);
      mbar_init(base + C::empty(s), 1);
    }
#pragma unroll
    for (int a = 0; a < kAccStages; ++a) {
      mbar_init(base + C::tfull(a), 1);
      mbar_init(base + C::tempty(a), CG * kEpiWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (CG == 1) tmem_alloc_cg1<kTmemCols>(base + C::tmem_ptr); else tmem_alloc_cg2<kTmemCols>(base + C::tmem_ptr);
  }
  tcgen05_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(base_ptr + C::tmem_ptr);
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    // ===================== TMA producer (every CTA loads its own rows of A and of B) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = unit; tile < num_tiles; tile += num_units) {
        const int m_blk = tile % p.m_blocks, n_blk = tile / p.m_blocks;
        const int32_t a_row = m_blk * C::kTileM + (int)rank * BLOCK_M;
        const int32_t b_row = n_blk * BLOCK_N + (int)rank * C::kBRows;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(base + C::empty(stage), phase ^ 1u);
          const uint32_t full = base + C::full(stage);
          if (CG == 1) mbar_expect_tx(full, C::kStageBytes);
          else if (rank == 0) mbar_expect_tx(full, 2 * C::kStageBytes);
          const int32_t k0 = kb * BLOCK_K;
          if (!A_MN) {
            tma_any<CG>(base + C::a(stage), &map_a, full, k0, a_row);              // box {64 k, 128 m}
          } else {
#pragma unroll
            for (int c = 0; c < BLOCK_M / 64; ++c)                                 // boxes {64 m, 64 k}
              tma_any<CG>(base + C::a(stage) + c * kChunkBytes, &map_a, full, a_row + 64 * c, k0);
          }
          if (!B_MN) {
            tma_any<CG>(base + C::b(stage), &map_b, full, k0, b_row);              // box {64 k, kBRows n}
          } else {
#pragma unroll
            for (int c = 0; c < C::kBRows / 64; ++c)                               // boxes {64 n, 64 k}
              tma_any<CG>(base + C::b(stage) + c * kChunkBytes, &map_b, full, b_row + 64 * c, k0);
          }
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (single thread of the leader CTA) =====================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(C::kTileM, BLOCK_N, A_MN ? 1 : 0, B_MN ? 1 : 0);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int tile = unit; tile < num_tiles; tile += num_units) {
        mbar_wait(base + C::tempty(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(base + C::full(stage), phase);
          tcgen05_fence_after();
          const uint64_t adesc = A_MN ? make_smem_desc_mn(base + C::a(stage), kChunkBytes, 1024u)
                                      : make_smem_desc(base + C::a(stage));
          const uint64_t bdesc = B_MN ? make_smem_desc_mn(base + C::b(stage), kChunkBytes, 1024u)
                                      : make_smem_desc(base + C::b(stage));
          // per UMMA_K = 16 elements: K-major +32 B inside the swizzle row; MN-major +16 rows = 2048 B
          constexpr uint64_t a_step = A_MN ? (16u * 128u) >> 4 : 2u;
          constexpr uint64_t b_step = B_MN ? (16u * 128u) >> 4 : 2u;
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
            umma_f16<CG>(tmem_d, adesc + a_step * k, bdesc + b_step * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          if (CG == 1) umma_commit(base + C::empty(stage)); else umma_commit_pair(base + C::empty(stage));
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (CG == 1) umma_commit(base + C::tfull(acc)); else umma_commit_pair(base + C::tfull(acc));
        if (++acc == kAccStages) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
  } else if (warp >= kEpiWarp0 && warp < kEpiWarp0 + kEpiWarps) {
    // ===================== epilogue: TMEM -> registers -> STE mask -> global =====================
    const int quad = warp & 3;
    const bool vec_ok = (p.out_dtype == QAT_BF16) ? (p.N % 8 == 0) : (p.N % 4 == 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = unit; tile < num_tiles; tile += num_units) {
      const int m_blk = tile % p.m_blocks, n_blk = tile / p.m_blocks;
      const int64_t row = (int64_t)m_blk * C::kTileM + (int64_t)rank * BLOCK_M + quad * 32 + lane;
      const int64_t col_base = (int64_t)n_blk * BLOCK_N;
      mbar_wait(base + C::tfull(acc), acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BLOCK_N);
#pragma unroll 1
      for (int c = 0; c < BLOCK_N / 32; ++c) {
        if (col_base + c * 32 >= p.N) break;   // warp-uniform
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + (uint32_t)(c * 32), r);
        tmem_ld_wait();
        if (row < p.M) store_chunk(p, row, col_base + c * 32, r, vec_ok);
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG == 1) mbar_arrive(base + C::tempty(acc)); else mbar_arrive_remote(base + C::tempty(acc), 0u);
      }
      if (++acc == kAccStages) {
        acc = 0;
        acc_phase ^= 1u;
      }
    }
  }

  tcgen05_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    if (CG == 1) tmem_dealloc_cg1<kTmemCols>(tmem_base); else tmem_dealloc_cg2<kTmemCols>(tmem_base);
  }
}

template <bool A_MN, bool B_MN, int CG>
int launch(const CUtensorMap& ma, const CUtensorMap& mb, const Params& p, cudaStream_t st) {
  using C = Cfg<CG>;
  static bool attr_set[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(gemm_bf16_kernel<A_MN, B_MN, CG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)C::kSmemBytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(gemm_bf16_kernel)");
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const int tiles = p.m_blocks * p.n_blocks;
  int units = num_sms() / CG;
  if (units > tiles) units = tiles;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(units * CG));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = C::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = pdl_enabled(QAT_PDL_FAMILY) ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_bf16_kernel<A_MN, B_MN, CG>, ma, mb, p);
  if (e != cudaSuccess) return cuda_fail(e, "gemm_bf16_kernel launch");
  QAT_CHECK_LAUNCH("gemm_bf16_kernel");
  return QAT_OK;
}

int g_forced_cg = -1;
int pick_cg(int64_t M, int64_t N) {
  if (g_forced_cg < 0) {
    const char* v = getenv("QAT_B200_GEMM_CG");
    g_forced_cg = (v && (v[0] == '1' || v[0] == '2')) ? v[0] - '0' : 0;
  }
  if (g_forced_cg) return g_forced_cg;
  if (num_sms() % 2) return 1;
  const int64_t pair_tiles = ((M + 255) / 256) * ((N + BLOCK_N - 1) / BLOCK_N);
  return pair_tiles >= num_sms() / 2 ? 2 : 1;
}

}  // namespace
}  // namespace qat

extern "C" int qat_gemm_bf16(const void* a, const void* b, void* out, const uint8_t* mask, int64_t M, int64_t N,
                             int64_t K, int a_mn_major, int b_mn_major, int out_dtype, int cta_group,
                             void* stream) {
  using namespace qat;
  QAT_CHECK_ARG(out_dtype == QAT_F32 || out_dtype == QAT_BF16, "out_dtype must be QAT_F32 or QAT_BF16");
  QAT_CHECK_ARG(M >= 0 && N >= 0 && K > 0, "bad GEMM shape [%lld, %lld, %lld]", (long long)M, (long long)N,
                (long long)K);
  if (M == 0 || N == 0) return QAT_OK;
  QAT_CHECK_ARG(a && b && out, "NULL operand");
  QAT_CHECK_ARG(((uintptr_t)a & 15) == 0 && ((uintptr_t)b & 15) == 0 && ((uintptr_t)out & 15) == 0,
                "operands must be 16-byte aligned");
  QAT_CHECK_ARG(M < (1ll << 31) && N < (1ll << 31) && K < (1ll << 31), "dimension too large");
  // TMA: the row pitch of every operand must be a multiple of 16 bytes
  QAT_CHECK_ARG((a_mn_major ? M : K) % 8 == 0, "A's contiguous dimension must be a multiple of 8 elements");
  QAT_CHECK_ARG((b_mn_major ? N : K) % 8 == 0, "B's contiguous dimension must be a multiple of 8 elements");
  QAT_CHECK_ARG(cta_group == 0 || cta_group == 1 || cta_group == 2, "cta_group must be 0 (automatic), 1 or 2");
  const int cg = cta_group ? cta_group : pick_cg(M, N);
  CUtensorMap ma, mb;
  int rc = a_mn_major ? make_map_bf16_2d(&ma, a, K, M, M, 64) : make_map_bf16_2d(&ma, a, M, K, K, BLOCK_M);
  if (rc != QAT_OK) return rc;
  rc = b_mn_major ? make_map_bf16_2d(&mb, b, K, N, N, 64) : make_map_bf16_2d(&mb, b, N, K, K, BLOCK_N / cg);
  if (rc != QAT_OK) return rc;
  Params p{};
  p.out = out;
  p.mask = mask;
  p.M = M;
  p.N = N;
  p.K = K;
  p.out_dtype = out_dtype;
  p.m_blocks = (int)((M + BLOCK_M * cg - 1) / (BLOCK_M * cg));
  p.n_blocks = (int)((N + BLOCK_N - 1) / BLOCK_N);
  p.k_blocks = (int)((K + BLOCK_K - 1) / BLOCK_K);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int sel = (a_mn_major ? 4 : 0) | (b_mn_major ? 2 : 0) | (cg == 2 ? 1 : 0);
  switch (sel) {
    case 0: return launch<false, false, 1>(ma, mb, p, st);
    case 1: return launch<false, false, 2>(ma, mb, p, st);
    case 2: return launch<false, true, 1>(ma, mb, p, st);
    case 3: return launch<false, true, 2>(ma, mb, p, st);
    case 4: return launch<true, false, 1>(ma, mb, p, st);
    case 5: return launch<true, false, 2>(ma, mb, p, st);
    case 6: return launch<true, true, 1>(ma, mb, p, st);
    default: return launch<true, true, 2>(ma, mb, p, st);
  }
}
