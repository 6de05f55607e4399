// tcgen05_gemm.cuh — the persistent tcgen05 GEMM pipeline shared by qlinear_gemm.cu (K4,
// kind::i8) and gemm_bf16.cu (dgrad / wgrad, kind::f16).
//
// C[M, N] = sum_k A(m, k) * B(n, k), accumulated in TMEM.  Each GEMM supplies an `Op` traits
// struct (MMA kind and instruction descriptor, k-block size, operand majors, epilogue hooks) and
// a one-line __global__ that calls gemm_body<Op, CG>.  CG = CTAs per MMA, the PTX cta_group:
//   * persistent grid, one CTA per SM, static round-robin over output tiles (m fastest);
//   * CG == 2 (large problems): the two CTAs of a cluster (one TPC) own one 256x256 tile.  Each
//     CTA stages its own 128 rows of A and its own 128-row half of B (32 KB per k-block instead
//     of 48 KB) and holds 128 rows of the accumulator in its TMEM; the leader CTA issues
//     tcgen05.mma.cta_group::2, which reads B from both CTAs' shared memory.  Per SM the operand
//     read rate drops from 96 to 64 B/clk — below the 128 B/clk shared-memory port — which is
//     what lets the tensor pipe stay busy (DESIGN.md "K4").
//   * CG == 1: one CTA per 128x256 tile (small problems, odd SM counts).
//   * warp 0   : TMA producer  (cp.async.bulk.tensor.2d, 128B swizzle; with CG == 2 both CTAs'
//                               loads complete on the leader's mbarrier)
//   * warp 1   : MMA issuer    (one thread of the leader CTA; tcgen05.commit multicasts
//                               "stage free" / "accumulator full" to both CTAs)
//   * warp 2   : TMEM allocator (512 columns = 2 accumulator stages)
//   * warps 4-7: epilogue      (tcgen05.ld 32x32b.x32 -> Op::store), overlapped with the next
//                               tile's MMAs.
//   * smem: CG1 4 x (16 KB A + 32 KB B), CG2 6 x (16 KB A + 16 KB B), plus Op::kEpiBytes.
// Every operand row of a k-block is 128 bytes (one swizzle row): 128 int8 or 64 bf16 elements.
#pragma once
#include "umma.cuh"

namespace qat {

// CTAs per MMA for an [M, N] output: pairs pay off once there are enough 256-row tiles to fill
// the machine.  qat_set_gemm_cta_group() / QAT_B200_GEMM_CG=1|2 force a choice for both GEMMs;
// the state lives in qlinear_gemm.cu.
int pick_cta_group(int64_t M, int64_t N);

namespace {
using namespace umma;

constexpr int BLOCK_M = 128;             // accumulator rows per CTA (TMEM lanes)
constexpr int BLOCK_N = 256;             // accumulator columns per tile
constexpr uint32_t kRowBytes = 128;      // bytes of K per operand row and k-block: one 128B swizzle row
constexpr int kAccStages = 2;
constexpr int kTmemCols = kAccStages * BLOCK_N;  // 512
constexpr int kThreads = 256;
constexpr int kEpiWarp0 = 4;  // warps 4..7; (warp % 4) selects the TMEM lane quadrant
constexpr int kEpiThreads = 128;
constexpr int kEpiWarps = kEpiThreads / 32;
constexpr uint32_t kChunkBytes = 64 * kRowBytes;  // one MN-major TMA box: 64 K-rows x 128 B = 8 KB

// Per-CTA shared-memory plan.  CG CTAs cooperate on one (CG*128) x 256 tile; EPI_BYTES is the
// Op's own epilogue region.
template <int CG, uint32_t EPI_BYTES>
struct Cfg {
  static constexpr int kStages = CG == 1 ? 4 : 6;
  static constexpr int kTileM = BLOCK_M * CG;                    // output rows per tile
  static constexpr int kBRows = BLOCK_N / CG;                    // B rows staged by each CTA
  static constexpr uint32_t kABytes = BLOCK_M * kRowBytes;       // 16 KB
  static constexpr uint32_t kBBytes = kBRows * kRowBytes;        // 32 KB | 16 KB
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  // offsets from the 1024-byte aligned base (identical in both CTAs of a pair)
  static __host__ __device__ constexpr uint32_t a(int s) { return (uint32_t)s * kStageBytes; }
  static __host__ __device__ constexpr uint32_t b(int s) { return (uint32_t)s * kStageBytes + kABytes; }
  static constexpr uint32_t epi = kStages * kStageBytes;
  static constexpr uint32_t bars = epi + EPI_BYTES;              // 8-byte aligned
  static __host__ __device__ constexpr uint32_t full(int s) { return bars + 8u * s; }
  static __host__ __device__ constexpr uint32_t empty(int s) { return bars + 8u * (kStages + s); }
  static __host__ __device__ constexpr uint32_t tfull(int a) { return bars + 8u * (2 * kStages + a); }
  static __host__ __device__ constexpr uint32_t tempty(int a) { return bars + 8u * (2 * kStages + kAccStages + a); }
  static constexpr uint32_t tmem_ptr = bars + 8u * (2 * kStages + 2 * kAccStages);
  static constexpr uint32_t total = tmem_ptr + 16;
  static constexpr uint32_t kSmemBytes = total + 1024;  // slack for manual 1024B alignment
  static_assert(EPI_BYTES % 8 == 0, "mbarriers need 8-byte alignment");
  static_assert(kSmemBytes <= 232448, "over the 227 KB per-CTA limit");
};

template <int CG>
__device__ __forceinline__ void tma_any(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1) {
  if (CG == 1) tma_load_2d(dst, map, bar, c0, c1); else tma_load_2d_pair(dst, map, bar, c0, c1);
}

// One operand's k-block: K-major is one box {128 B of K, ROWS}; MN-major is ROWS/64 boxes
// {64 elements of M/N, 64 rows of K}, kChunkBytes apart.
template <bool MN, int ROWS, int CG>
__device__ __forceinline__ void load_operand(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t k0,
                                             int32_t row) {
  if (!MN) {
    tma_any<CG>(dst, map, bar, k0, row);
  } else {
#pragma unroll
    for (int c = 0; c < ROWS / 64; ++c) tma_any<CG>(dst + c * kChunkBytes, map, bar, row + 64 * c, k0);
  }
}

// 32 consecutive fp32 values of one output row -> bf16 or fp32 at out[row, col0..], 16-byte
// stores when the row pitch allows (vec_ok) and the chunk lies inside N, else element by element.
__device__ __forceinline__ void store_row32(void* out, bool bf16, int64_t row, int64_t col0, int64_t N,
                                            const float (&v)[32], bool vec_ok) {
  if (bf16) {
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(out) + row * N + col0;
    if (vec_ok && col0 + 32 <= N) {
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
        if (col0 + j < N) dst[j] = __float2bfloat16_rn(v[j]);
    }
  } else {
    float* dst = reinterpret_cast<float*>(out) + row * N + col0;
    if (vec_ok && col0 + 32 <= N) {
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < N) dst[j] = v[j];
    }
  }
}

// The kernel body.  Op provides:
//   Params                       with fields N, m_blocks, n_blocks, k_blocks
//   kBlockK, kUmmaK              elements per k-block (128 B) and per MMA
//   kAMN, kBMN                   operand majors (MN-major needs 16-bit elements)
//   kEpiBytes                    its shared-memory epilogue region
//   kStopPastN                   leave the chunk loop at the first chunk past N (else store() guards)
//   idesc(m), mma<CG>(...)       instruction descriptor and tcgen05.mma
//   out_bf16(p)                  output type (bf16 or fp32)
//   tile_prologue(p, epi, acc, row, col_base) -> Tile, run by the epilogue warps before each tile's wait
//   store(p, tile, row, col0, c, acc[32], vec_ok)    one 32-column chunk of the TMEM accumulator
template <class Op, int CG>
__device__ __forceinline__ void gemm_body(const CUtensorMap& map_a, const CUtensorMap& map_b,
                                          const typename Op::Params& p) {
  using C = Cfg<CG, Op::kEpiBytes>;
  extern __shared__ uint8_t smem_raw[];
  // the dynamic window starts at the same shared::cta offset in every CTA of the
  // kernel, so `base` — and with it every barrier / tile offset — is identical
  // in both CTAs of a pair (the multicast commit and the peer-bit trick need it)
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;   // 0 = leader (issues the MMAs)
  const int unit = (CG == 2) ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;   // CTA (pair) index
  const int num_units = (CG == 2) ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int num_tiles = p.m_blocks * p.n_blocks;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
  }
  if (warp == 1 && lane == 0) {
#pragma unroll
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(base + C::full(s), 1);    // the leader's producer: arrive.expect_tx (bytes of both CTAs)
      mbar_init(base + C::empty(s), 1);   // one tcgen05.commit arrival (multicast to both CTAs when CG == 2)
    }
#pragma unroll
    for (int a = 0; a < kAccStages; ++a) {
      mbar_init(base + C::tfull(a), 1);
      mbar_init(base + C::tempty(a), CG * kEpiWarps);   // one arrival per epilogue warp of every CTA
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (CG == 1) tmem_alloc_cg1<kTmemCols>(base + C::tmem_ptr); else tmem_alloc_cg2<kTmemCols>(base + C::tmem_ptr);
  }
  tcgen05_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();   // peers touch our barriers: cluster-wide
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(base_ptr + C::tmem_ptr);
  // barrier init, TMEM allocation and descriptor prefetch above overlap the previous
  // kernel's tail; its results are read only from here on
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
          mbar_wait(base + C::empty(stage), phase ^ 1u);   // own copy: the commit is multicast
          const uint32_t full = base + C::full(stage);
          if (CG == 1) mbar_expect_tx(full, C::kStageBytes);
          else if (rank == 0) mbar_expect_tx(full, 2 * C::kStageBytes);
          const int32_t k0 = kb * Op::kBlockK;
          load_operand<Op::kAMN, BLOCK_M, CG>(base + C::a(stage), &map_a, full, k0, a_row);
          load_operand<Op::kBMN, C::kBRows, CG>(base + C::b(stage), &map_b, full, k0, b_row);
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
      constexpr uint32_t idesc = Op::idesc(C::kTileM);
      // per MMA: K-major +32 B inside the swizzle row (+2 in the >>4 address field);
      // MN-major +kUmmaK rows of 128 B
      constexpr uint64_t a_step = Op::kAMN ? (Op::kUmmaK * kRowBytes) >> 4 : 2u;
      constexpr uint64_t b_step = Op::kBMN ? (Op::kUmmaK * kRowBytes) >> 4 : 2u;
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int tile = unit; tile < num_tiles; tile += num_units) {
        mbar_wait(base + C::tempty(acc), acc_phase ^ 1u);  // every epilogue warp drained this stage
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(base + C::full(stage), phase);
          tcgen05_fence_after();
          const uint64_t adesc = Op::kAMN ? make_smem_desc_mn(base + C::a(stage), kChunkBytes, 1024u)
                                          : make_smem_desc(base + C::a(stage));
          const uint64_t bdesc = Op::kBMN ? make_smem_desc_mn(base + C::b(stage), kChunkBytes, 1024u)
                                          : make_smem_desc(base + C::b(stage));
#pragma unroll
          for (int k = 0; k < Op::kBlockK / Op::kUmmaK; ++k)
            Op::template mma<CG>(tmem_d, adesc + a_step * k, bdesc + b_step * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          // frees the smem stage (in both CTAs) when the MMAs retire
          if (CG == 1) umma_commit(base + C::empty(stage)); else umma_commit_pair(base + C::empty(stage));
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        // accumulator complete -> epilogue (of both CTAs)
        if (CG == 1) umma_commit(base + C::tfull(acc)); else umma_commit_pair(base + C::tfull(acc));
        if (++acc == kAccStages) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ===================== epilogue (4 warps, 128 threads, own 128 accumulator rows) =====================
    const int quad = warp & 3;   // TMEM lane quadrant this warp may read
    const bool vec_ok = Op::out_bf16(p) ? (p.N % 8 == 0) : (p.N % 4 == 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = unit; tile < num_tiles; tile += num_units) {
      const int m_blk = tile % p.m_blocks, n_blk = tile / p.m_blocks;
      const int64_t row = (int64_t)m_blk * C::kTileM + (int64_t)rank * BLOCK_M + quad * 32 + lane;
      const int64_t col_base = (int64_t)n_blk * BLOCK_N;
      const typename Op::Tile t = Op::tile_prologue(p, base_ptr + C::epi, acc, row, col_base);
      mbar_wait(base + C::tfull(acc), acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BLOCK_N);
#pragma unroll 1
      for (int c = 0; c < BLOCK_N / 32; ++c) {
        if (Op::kStopPastN && col_base + c * 32 >= p.N) break;   // warp-uniform
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + (uint32_t)(c * 32), r);
        tmem_ld_wait();
        Op::store(p, t, row, col_base + c * 32, c, r, vec_ok);
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
  if (CG == 2) cluster_sync_all(); else __syncthreads();   // nobody leaves while its peer may still use it
  if (warp == 2) {
    tcgen05_fence_after();
    if (CG == 1) tmem_dealloc_cg1<kTmemCols>(tmem_base); else tmem_dealloc_cg2<kTmemCols>(tmem_base);
  }
}

// Persistent cluster launch of one gemm_body kernel: one CTA (pair) per SM (TPC), at most one per
// tile, programmatic launch when `pdl_family` is enabled in QAT_B200_PDL_MASK.
template <class Op, int CG, class Params>
int launch_gemm(void (*kernel)(CUtensorMap, CUtensorMap, Params), const char* name, const CUtensorMap& ma,
                const CUtensorMap& mb, const Params& p, cudaStream_t st, int pdl_family) {
  constexpr uint32_t smem = Cfg<CG, Op::kEpiBytes>::kSmemBytes;
  static bool opted_in[64] = {};  // per kernel
  int rc = opt_in_smem(kernel, smem, opted_in, name);
  if (rc != QAT_OK) return rc;
  const int tiles = p.m_blocks * p.n_blocks;
  int units = num_sms() / CG;
  if (units > tiles) units = tiles;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(units * CG));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = pdl_enabled(pdl_family) ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, ma, mb, p);
  if (e != cudaSuccess) {
    char what[96];
    snprintf(what, sizeof(what), "%s launch", name);
    return cuda_fail(e, what);
  }
  QAT_CHECK_LAUNCH(name);
  return QAT_OK;
}

}  // namespace
}  // namespace qat
