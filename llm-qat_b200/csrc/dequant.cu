// dequant.cu — rebuild the fake-quantized tensor from K1's int8 codes:
//     out[r, c] = fl_dtype(codes[r, c] / e[r])
// which is bit-identical to SymQuantizer's forward output
// (/root/reference/models/utils_quant.py:72) wherever the int8 feed did not
// saturate.  QuantizeLinear's backward uses it for the dgrad/wgrad operands, so
// the forward can save 1 B/elem of codes instead of the reference's two
// dequantized tensors.  HBM-bound: 1 + sizeof(T) bytes per element.
#define QAT_PDL_FAMILY 2   // bit of QAT_B200_PDL_MASK (common.cuh)
#include <type_traits>

#include "common.cuh"

namespace qat {
namespace {

constexpr int kThreads = 256;

// Tile = kThreads * unroll code groups, all loaded before use; ONE CTA PER TILE (no grid-stride cap).  Measured
// (profiles/r02_dequant_ste_tune.json): the former cap of 8 CTAs per SM assumed an
// occupancy the 40-64 register kernels do not have (5-6 CTAs per SM), so a second, ragged wave of CTAs each
// walked 4-5 tiles on a third of the slots: 0.77 of the HBM peak at [11008, 4096]; uncapped, the block scheduler
// balances tile by tile: 0.85.  Large tensors take 8 groups per thread (fp32 divisors: 26.7 -> 24.7 us), small
// ones 2 (more CTAs than slots even at [2048, 4096]).
constexpr int64_t kLargeGroups = 4ll << 20;   // >= this many groups: unroll 8, else 2
constexpr int kCtasPerSmDefault = 0;          // 0 = one CTA per tile

// Each thread turns one group of G = 16 / sizeof(out element) codes (8 for bf16, 4 for fp32) into
// exactly ONE 16-byte store, so that every store instruction of a warp writes 512 contiguous
// bytes — whole 32-byte sectors.  (A first version took 16 codes per thread and issued two
// stores per thread, i.e. half sectors per instruction: 0.63 of the HBM peak at [11008, 4096];
// the traffic is write-dominated, 1 B in : 2 B out.)
template <int DT>
struct Group {
  static constexpr int kCodes = 16 / Num<DT>::kBytes;                 // 8 | 4
  using load_t = typename std::conditional<DT == QAT_BF16, uint2, uint32_t>::type;
};

template <int DT>
__device__ __forceinline__ uint4 dequant_group(typename Group<DT>::load_t c, float e) {
  const bool fast = recip_range_ok(e);
  const float r = __frcp_rn(e);
  // bf16 output and a bf16-valued divisor (what K1 emits for bf16 tensors): one multiply is
  // exact — see SymScale::mulq in common.cuh
  const bool mulq = DT == QAT_BF16 && fast && Num<QAT_BF16>::fl(e) == e;
  constexpr int G = Group<DT>::kCodes;
  uint32_t w[2];
  if constexpr (DT == QAT_BF16) {
    w[0] = c.x;
    w[1] = c.y;
  } else {
    w[0] = c;
    w[1] = 0u;
  }
  float y[G];
#pragma unroll
  for (int k = 0; k < G; ++k) y[k] = (float)(int)(int8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xffu);
  // one (nearly always warp-uniform) branch per group, not a select per element: the exact
  // division's slow path is a long instruction sequence that must stay out of the common stream
  if (mulq) {
#pragma unroll
    for (int k = 0; k < G; ++k) y[k] = __fmul_rn(y[k], r);
  } else if (fast) {
#pragma unroll
    for (int k = 0; k < G; ++k) y[k] = div_code_by_recip(y[k], e, r);
  } else {
#pragma unroll
    for (int k = 0; k < G; ++k) y[k] = __fdiv_rn(y[k], e);
  }
  if constexpr (DT == QAT_BF16)
    return make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4 % G], y[5 % G]),
                      pack_bf16x2(y[6 % G], y[7 % G]));
  else
    return make_uint4(__float_as_uint(y[0]), __float_as_uint(y[1]), __float_as_uint(y[2]), __float_as_uint(y[3]));
}

// IDX32: the group index fits 32 bits, so the row lookup is a multiply-high by a host-computed
// magic number (exact for every j < 2^32: Granlund-Montgomery round-up method with a 33-bit
// multiplier) instead of a 64-bit division (~60 instructions per group).
struct Magic {
  uint32_t mul;   // low 32 bits of the 33-bit multiplier
  uint32_t shift; // post-shift
  uint32_t pow2;  // divisor is a power of two: row = j >> shift
};
__device__ __forceinline__ uint32_t magic_div(uint32_t j, const Magic& m) {
  if (m.pow2) return j >> m.shift;
  const uint32_t t = __umulhi(j, m.mul);
  return (t + ((j - t) >> 1)) >> m.shift;   // (j * (2^32 + mul)) >> (33 + shift) without overflow
}

template <int DT, bool IDX32, int kUnroll>
__global__ void __launch_bounds__(kThreads) dequant_codes_kernel(const int8_t* __restrict__ codes,
                                                                 const float* __restrict__ row_e,
                                                                 void* __restrict__ out, int64_t ngroups,
                                                                 int groups_per_row, const Magic magic) {
  using L = typename Group<DT>::load_t;
  constexpr int64_t kTile = (int64_t)kThreads * kUnroll;
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t base = (int64_t)blockIdx.x * kTile; base < ngroups; base += (int64_t)gridDim.x * kTile) {
    L c[kUnroll];
    float e[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t j = base + (int64_t)u * kThreads + threadIdx.x;
      if (j < ngroups) {
        c[u] = __ldg(reinterpret_cast<const L*>(codes) + j);
        e[u] = row_e[IDX32 ? (int64_t)magic_div((uint32_t)j, magic) : j / groups_per_row];
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t j = base + (int64_t)u * kThreads + threadIdx.x;
      if (j < ngroups) stg_stream(reinterpret_cast<uint4*>(out) + j, dequant_group<DT>(c[u], e[u]));
    }
  }
}

}  // namespace
}  // namespace qat

extern "C" int qat_dequant_codes(const int8_t* codes, const float* row_e, void* out, int64_t rows,
                                 int64_t cols, int dtype, void* stream) {
  using namespace qat;
  QAT_CHECK_ARG(dtype == QAT_F32 || dtype == QAT_BF16, "dtype must be QAT_F32 or QAT_BF16 (got %d)", dtype);
  QAT_CHECK_ARG(rows >= 0 && cols >= 0, "negative shape");
  if (rows == 0 || cols == 0) return QAT_OK;
  QAT_CHECK_ARG(codes && row_e && out, "NULL operand");
  QAT_CHECK_ARG(cols % 16 == 0, "cols must be a multiple of 16 (got %lld)", (long long)cols);
  QAT_CHECK_ARG(((uintptr_t)codes & 15) == 0 && ((uintptr_t)out & 15) == 0, "pointers must be 16-byte aligned");
  const int per = dtype == QAT_BF16 ? 8 : 4;    // codes per thread-iteration == one 16-byte store
  const int64_t ngroups = rows * cols / per;
  QAT_CHECK_ARG(cols / per < (1ll << 31), "row too long");
  const int unroll = ngroups >= kLargeGroups ? 8 : 2;
  int64_t grid = (ngroups + kThreads * unroll - 1) / (kThreads * unroll);
  const int64_t cap = kCtasPerSmDefault > 0 ? (int64_t)num_sms() * kCtasPerSmDefault : (int64_t)0x7fffffff;
  if (grid > cap) grid = cap;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool idx32 = ngroups < (1ll << 32);
  const int gpr = (int)(cols / per);
  Magic magic{};
  {
    const uint32_t d = (uint32_t)gpr;
    if ((d & (d - 1)) == 0) {
      magic.pow2 = 1;
      while ((1u << magic.shift) < d) ++magic.shift;
    } else {
      uint32_t l = 0;
      while ((1ull << l) < d) ++l;                                    // l = ceil(log2 d), d not a power of two
      const unsigned __int128 one = 1;
      const uint64_t m = (uint64_t)(((one << (32 + l)) / d) + 1);    // 2^32 <= m < 2^33
      magic.mul = (uint32_t)(m - (1ull << 32));
      magic.shift = l - 1;
    }
  }
  const dim3 g((unsigned)grid), b(kThreads);
#define QAT_DEQUANT_LAUNCH(DT, IDX, U) \
  (void)launch_pdl(dequant_codes_kernel<DT, IDX, U>, g, b, 0, st, codes, row_e, out, ngroups, gpr, magic)
#define QAT_DEQUANT_UNROLL(DT, IDX)                 \
  do {                                              \
    if (unroll == 8) QAT_DEQUANT_LAUNCH(DT, IDX, 8); \
    else QAT_DEQUANT_LAUNCH(DT, IDX, 2);             \
  } while (0)
  if (dtype == QAT_BF16) {
    if (idx32) QAT_DEQUANT_UNROLL(QAT_BF16, true);
    else QAT_DEQUANT_UNROLL(QAT_BF16, false);
  } else {
    if (idx32) QAT_DEQUANT_UNROLL(QAT_F32, true);
    else QAT_DEQUANT_UNROLL(QAT_F32, false);
  }
#undef QAT_DEQUANT_UNROLL
#undef QAT_DEQUANT_LAUNCH
  QAT_CHECK_LAUNCH("dequant_codes_kernel");
  return QAT_OK;
}
