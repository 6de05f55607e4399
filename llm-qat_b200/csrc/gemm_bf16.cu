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
// The pipeline is tcgen05_gemm.cuh's (kind::f16, fp32 accumulators in TMEM); what is specific
// here is the MN-major operand loads and descriptors, the STE mask in the epilogue and the output
// type, which is read at run time (one instance per operand layout, not per output type).
// Tensor-bound: 2*M*N*K flops against the bf16 dense peak.
#define QAT_PDL_FAMILY 5   // bit of QAT_B200_PDL_MASK (common.cuh)

#include "tcgen05_gemm.cuh"

namespace qat {
namespace {

constexpr int BLOCK_K = 64;    // bf16 elements per k-block: 128 bytes, one swizzle row

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

template <bool A_MN, bool B_MN>
struct Bf16Op {
  using Params = qat::Params;
  static constexpr int kBlockK = BLOCK_K;
  static constexpr int kUmmaK = 16;   // elements per tcgen05.mma.kind::f16
  static constexpr bool kAMN = A_MN, kBMN = B_MN;
  static constexpr uint32_t kEpiBytes = 0;
  static constexpr bool kStopPastN = true;
  static __host__ __device__ constexpr uint32_t idesc(int m) {
    return make_idesc_bf16(m, BLOCK_N, A_MN ? 1 : 0, B_MN ? 1 : 0);
  }
  template <int CG>
  static __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    umma_f16<CG>(d, a, b, idesc, acc);
  }
  static __device__ __forceinline__ bool out_bf16(const Params& p) { return p.out_dtype == QAT_BF16; }

  struct Tile {};
  static __device__ __forceinline__ Tile tile_prologue(const Params&, uint8_t*, int, int64_t, int64_t) { return {}; }
  static __device__ __forceinline__ void store(const Params& p, const Tile&, int64_t row, int64_t col0, int,
                                               const uint32_t (&acc)[32], bool vec_ok) {
    if (row >= p.M) return;
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
    if (p.mask != nullptr) {
      const uint32_t bits = mask_bits32(p.mask, row * p.N + col0, (p.M * p.N + 7) >> 3);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (!((bits >> j) & 1u)) v[j] = 0.f;
    }
    store_row32(p.out, p.out_dtype == QAT_BF16, row, col0, p.N, v, vec_ok);
  }
};

template <bool A_MN, bool B_MN, int CG>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const Params p) {
  gemm_body<Bf16Op<A_MN, B_MN>, CG>(map_a, map_b, p);
}

template <bool A_MN, bool B_MN, int CG>
int launch(const CUtensorMap& ma, const CUtensorMap& mb, const Params& p, cudaStream_t st) {
  return launch_gemm<Bf16Op<A_MN, B_MN>, CG>(gemm_bf16_kernel<A_MN, B_MN, CG>, "gemm_bf16_kernel", ma, mb, p, st,
                                             QAT_PDL_FAMILY);
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
  const int cg = cta_group ? cta_group : pick_cta_group(M, N);
  CUtensorMap ma, mb;
  int rc = a_mn_major ? make_map_2d(&ma, 2, a, K, M, M, 64) : make_map_2d(&ma, 2, a, M, K, K, BLOCK_M);
  if (rc != QAT_OK) return rc;
  rc = b_mn_major ? make_map_2d(&mb, 2, b, K, N, N, 64) : make_map_2d(&mb, 2, b, N, K, K, BLOCK_N / cg);
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
