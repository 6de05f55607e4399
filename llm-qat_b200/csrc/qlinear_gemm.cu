// qlinear_gemm.cu — K4: the QuantizeLinear contraction on the integer grid.
//
// Replaces /root/reference/models/utils_quant.py:250  F.linear(x_q, W_q)  (a
// cuBLAS bf16 GEMM over two *dequantized* tensors) with
//     out[t, n] = (sum_k qx[t,k] * qw[n,k]) * (1/ex[t]) * (1/ew[n])
// where qx / qw are the int8 codes and ex / ew the dequant divisors that K1
// emits in its codes-only mode.  The integer dot product is exact (s32
// accumulators), so the result is at least as accurate as the reference's.
//
// The pipeline is tcgen05_gemm.cuh's (kind::i8, s32 accumulators in TMEM, both operands
// K-major); what is specific to K4 is the dual-scale epilogue: the epilogue warps stage 1/ew for
// the tile's 256 columns in shared memory while the MMAs run, then each 32-column chunk goes
// I2F -> x 1/ex[row] -> x 1/ew[col] -> bf16/fp32.  The output type is a template parameter.
// Tensor-bound: 2*T*N*K integer ops; see DESIGN.md "K4".
#define QAT_PDL_FAMILY 4   // bit of QAT_B200_PDL_MASK (common.cuh)
#include <cstdlib>

#include "tcgen05_gemm.cuh"

namespace qat {
namespace {

constexpr int BLOCK_K = 128;  // bytes == int8 elements: one 128B swizzle row

struct GemmParams {
  const float* ex;  // [T] dequant divisors of the activation rows
  const float* ew;  // [N] dequant divisors of the weight rows
  void* out;
  int64_t T, N, K;
  int m_blocks, n_blocks, k_blocks;
};

template <int OUT_DT>
struct I8Op {
  using Params = GemmParams;
  static constexpr int kBlockK = BLOCK_K;
  static constexpr int kUmmaK = 32;   // elements per tcgen05.mma.kind::i8
  static constexpr bool kAMN = false, kBMN = false;
  static constexpr uint32_t kEpiBytes = kAccStages * BLOCK_N * 4;   // 1/ew of each accumulator stage's columns
  static constexpr bool kStopPastN = false;
  static __host__ __device__ constexpr uint32_t idesc(int m) { return make_idesc_i8(m, BLOCK_N); }
  template <int CG>
  static __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    umma_i8<CG>(d, a, b, idesc, acc);
  }
  static __device__ __forceinline__ bool out_bf16(const Params&) { return OUT_DT == QAT_BF16; }

  struct Tile {
    const float* colscale;  // smem, 256 entries
    float row_scale;
  };
  static __device__ __forceinline__ Tile tile_prologue(const Params& p, uint8_t* epi, int acc, int64_t row,
                                                       int64_t col_base) {
    const int et = threadIdx.x - kEpiWarp0 * 32;  // 0..127
    float* colscale = reinterpret_cast<float*>(epi) + acc * BLOCK_N;
    // stage 1/ew for this tile's 256 columns (2 per thread) while the MMAs run
#pragma unroll
    for (int j = et; j < BLOCK_N; j += kEpiThreads) {
      const int64_t c = col_base + j;
      colscale[j] = (c < p.N) ? __frcp_rn(p.ew[c]) : 0.f;
    }
    const float row_scale = (row < p.T) ? __frcp_rn(p.ex[row]) : 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");  // colscale visible to the 4 warps
    return {colscale, row_scale};
  }
  static __device__ __forceinline__ void store(const Params& p, const Tile& t, int64_t row, int64_t col0, int c,
                                               const uint32_t (&acc)[32], bool vec_ok) {
    if (row < p.T && col0 < p.N) {
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j)
        v[j] = __fmul_rn(__fmul_rn((float)(int32_t)acc[j], t.row_scale), t.colscale[c * 32 + j]);
      store_row32(p.out, OUT_DT == QAT_BF16, row, col0, p.N, v, vec_ok);
    }
  }
};

template <int OUT_DT, int CG>
__global__ void __launch_bounds__(kThreads, 1)
qlinear_i8_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                  const GemmParams p) {
  gemm_body<I8Op<OUT_DT>, CG>(map_a, map_b, p);
}

template <int OUT_DT, int CG>
int launch(const CUtensorMap& ma, const CUtensorMap& mb, const GemmParams& p, cudaStream_t st) {
  return launch_gemm<I8Op<OUT_DT>, CG>(qlinear_i8_kernel<OUT_DT, CG>, "qlinear_i8_kernel", ma, mb, p, st,
                                       QAT_PDL_FAMILY);
}

// 0: automatic; -1: not yet read from the environment
int g_forced_cg = -1;

}  // namespace

int pick_cta_group(int64_t M, int64_t N) {
  if (g_forced_cg < 0) {
    const char* v = getenv("QAT_B200_GEMM_CG");
    g_forced_cg = (v && (v[0] == '1' || v[0] == '2')) ? v[0] - '0' : 0;
  }
  if (g_forced_cg) return g_forced_cg;
  if (num_sms() % 2) return 1;
  const int64_t pair_tiles = ((M + 255) / 256) * ((N + BLOCK_N - 1) / BLOCK_N);
  return pair_tiles >= num_sms() / 2 ? 2 : 1;
}

}  // namespace qat

extern "C" int qat_set_gemm_cta_group(int cta_group) {
  using namespace qat;
  QAT_CHECK_ARG(cta_group == 0 || cta_group == 1 || cta_group == 2, "cta_group must be 0 (automatic), 1 or 2");
  g_forced_cg = cta_group;
  return QAT_OK;
}

extern "C" int qat_qlinear_i8_fwd(const int8_t* qx, const int8_t* qw, const float* ex, const float* ew,
                                  void* out, int64_t T, int64_t N, int64_t K, int out_dtype, void* stream) {
  using namespace qat;
  QAT_CHECK_ARG(out_dtype == QAT_F32 || out_dtype == QAT_BF16, "out_dtype must be QAT_F32 or QAT_BF16");
  QAT_CHECK_ARG(T >= 0 && N >= 0 && K > 0, "bad GEMM shape [%lld, %lld, %lld]", (long long)T, (long long)N,
                (long long)K);
  if (T == 0 || N == 0) return QAT_OK;
  QAT_CHECK_ARG(qx && qw && ex && ew && out, "NULL operand");
  QAT_CHECK_ARG(K % 16 == 0, "K must be a multiple of 16 (TMA row pitch), got %lld", (long long)K);
  QAT_CHECK_ARG(((uintptr_t)qx & 15) == 0 && ((uintptr_t)qw & 15) == 0, "code pointers must be 16-byte aligned");
  QAT_CHECK_ARG(((uintptr_t)out & 15) == 0, "out must be 16-byte aligned");
  QAT_CHECK_ARG(T < (1ll << 31) && N < (1ll << 31) && K < (1ll << 31), "dimension too large");
  const int cg = pick_cta_group(T, N);
  CUtensorMap ma, mb;
  int rc = make_map_2d(&ma, 1, qx, T, K, K, BLOCK_M);
  if (rc != QAT_OK) return rc;
  rc = make_map_2d(&mb, 1, qw, N, K, K, BLOCK_N / cg);
  if (rc != QAT_OK) return rc;
  GemmParams p{};
  p.ex = ex;
  p.ew = ew;
  p.out = out;
  p.T = T;
  p.N = N;
  p.K = K;
  p.m_blocks = (int)((T + BLOCK_M * cg - 1) / (BLOCK_M * cg));
  p.n_blocks = (int)((N + BLOCK_N - 1) / BLOCK_N);
  p.k_blocks = (int)((K + BLOCK_K - 1) / BLOCK_K);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (cg == 2) return out_dtype == QAT_BF16 ? launch<QAT_BF16, 2>(ma, mb, p, st) : launch<QAT_F32, 2>(ma, mb, p, st);
  return out_dtype == QAT_BF16 ? launch<QAT_BF16, 1>(ma, mb, p, st) : launch<QAT_F32, 1>(ma, mb, p, st);
}

// One call for QuantizeLinear.forward's main path (utils_quant.py:197-201,244-250):
// K1 (codes-only) on the activations, K1 on the weights, then the tcgen05 GEMM.
// `reuse_x` / `reuse_w` skip a quantization whose outputs the caller still holds
// (q/k/v share one input; weights only change at optimizer steps).
extern "C" int qat_qlinear_fused_fwd(const void* x, const void* w, void* out, int8_t* qx, float* ex,
                                     uint8_t* mx, int8_t* qw, float* ew, uint8_t* mw, int64_t T, int64_t N,
                                     int64_t K, int dtype, int a_bits, int w_bits, float clip_lo,
                                     float clip_hi, int reuse_x, int reuse_w, void* stream) {
  using namespace qat;
  QAT_CHECK_ARG(qx && ex && qw && ew, "code / scale buffers must be provided");
  QAT_CHECK_ARG(a_bits >= 2 && a_bits <= 8 && w_bits >= 2 && w_bits <= 8, "int8 grid needs 2 <= bits <= 8");
  if (!reuse_x) {
    int rc = sym_fwd_feed(x, qx, ex, mx, clip_lo, clip_hi, T, K, dtype, a_bits, stream);
    if (rc != QAT_OK) return rc;
  }
  if (!reuse_w) {
    int rc = sym_fwd_feed(w, qw, ew, mw, clip_lo, clip_hi, N, K, dtype, w_bits, stream);
    if (rc != QAT_OK) return rc;
  }
  // under autocast the reference's F.linear runs, and returns, bf16
  return qat_qlinear_i8_fwd(qx, qw, ex, ew, out, T, N, K, dtype == QAT_BF16_AMP ? QAT_BF16 : dtype, stream);
}
