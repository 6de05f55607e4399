// lowbit.cu — QuantizeLinear's w_bits in {1, 2} weight path (secondary; no
// BASELINE config exercises it).  Replaces the eager chain at
// /root/reference/models/utils_quant.py:202-242:
//   1-bit : sf = mean|w|      ; q = sf * sign(w / sf)
//   2-bit : sf = 2 * mean|w|  ; q = sf * (round(clamp(w/sf, -0.99, 0.99) * 2 - 0.5) + 0.5) / 2
//   forward value = (q - w) + w           (gradient is the identity)
// The mean is per output row, or over the whole tensor when layerwise.
//
// Row-wise mode (and layerwise below 32768 elements): ONE pass, one CTA per row with the row staged in
// shared memory, mean|w| summed in the exact order of torch's CPU reduction (torch_sum_order.cuh) so that
// the scale — and every element scaled by it — carries the reference's bits in fp32 and bf16: 2e B/elem.
// Larger layerwise tensors (torch splits that reduction over its threads: no portable bit contract) and
// rows beyond one CTA's shared memory: two launches, a double-precision sum merged with atomics, then a
// pass that re-reads w and applies (3e B/elem).
#define QAT_PDL_FAMILY 3   // bit of QAT_B200_PDL_MASK (common.cuh)
#include <algorithm>
#include <atomic>
#include <type_traits>

#include "common.cuh"
#include "torch_sum_order.cuh"

namespace qat {
namespace {

constexpr int kThreads = 256;

struct LowbitParams {
  const void* w;
  void* out;
  double* sums;  // [rows] or [1]
  int64_t rows, cols;
  int64_t chunk;  // elements of a row per CTA
  int w_bits;
  int layerwise;
};

template <int DT>
__device__ __forceinline__ float load_elem(const void* p, int64_t i) {
  if (DT == QAT_F32) return reinterpret_cast<const float*>(p)[i];
  return bf16lo(reinterpret_cast<const uint16_t*>(p)[i]);
}

// (q - w) + w for one element, every op rounded to the tensor dtype — :205-242
// `rsf`: RN(1/sf) when the quotient may be taken as one multiply (bf16 tensors, sf in the proven
// window: oracle/proofs/bf16_quotient_by_reciprocal.c "anyratio", every bf16 numerator x every
// bf16 divisor, 0 mismatches), else 0 -> exact IEEE division.
template <int DT>
__device__ __forceinline__ float lowbit_eff(float w, float sf, float rsf, float clip, int w_bits) {
  using N = Num<DT>;
  const float r = N::fl((DT == QAT_BF16 && rsf != 0.f) ? __fmul_rn(w, rsf) : __fdiv_rn(w, sf));
  float q;
  if (w_bits == 1) {
    const float sgn = (r > 0.f) ? 1.f : (r < 0.f) ? -1.f : 0.f;  // torch.sign: NaN -> 0
    q = N::fl(__fmul_rn(sf, sgn));                               // :211-213
  } else {
    float t = (r != r) ? r : fminf(fmaxf(r, -clip), clip);       // clamp keeps NaN (:229-231)
    t = N::fl(__fsub_rn(N::fl(__fmul_rn(t, 2.0f)), 0.5f));       // :232-233
    t = N::fl(__fadd_rn(rintf(t), 0.5f));                        // :228,235
    q = N::fl(__fmul_rn(N::fl(__fmul_rn(sf, t)), 0.5f));         // :226-237  (/ 2 == * 0.5 exactly)
  }
  return N::fl(__fadd_rn(N::fl(__fsub_rn(q, w)), w));            // :240-242
}

template <int DT>
__global__ void __launch_bounds__(kThreads) lowbit_sum_kernel(const LowbitParams p) {
  __shared__ double sm[kThreads / 32];
  const int64_t row = blockIdx.y;
  const int64_t j0 = (int64_t)blockIdx.x * p.chunk;
  const int64_t j1 = min(j0 + p.chunk, p.cols);
  double acc = 0.0;
  for (int64_t j = j0 + threadIdx.x; j < j1; j += kThreads)
    acc += (double)fabsf(load_elem<DT>(p.w, row * p.cols + j));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) t += sm[i];
    atomicAdd(p.sums + (p.layerwise ? 0 : row), t);
  }
}

template <int DT>
__global__ void __launch_bounds__(kThreads) lowbit_apply_kernel(const LowbitParams p) {
  using N = Num<DT>;
  const int64_t row = blockIdx.y;
  const int64_t j0 = (int64_t)blockIdx.x * p.chunk;
  const int64_t j1 = min(j0 + p.chunk, p.cols);
  const double count = p.layerwise ? (double)p.rows * (double)p.cols : (double)p.cols;
  const float mean_abs = N::fl((float)(p.sums[p.layerwise ? 0 : row] / count));  // :205-210 / :219-224
  const float sf = (p.w_bits == 1) ? mean_abs : N::fl(__fmul_rn(2.0f, mean_abs));
  const float clip = N::fl(0.99f);  // 1 - 1e-2, cast to the tensor dtype by clamp (:218)
  const float rsf = (DT == QAT_BF16 && recip_range_ok(sf)) ? __frcp_rn(sf) : 0.f;
  for (int64_t j = j0 + threadIdx.x; j < j1; j += kThreads) {
    const int64_t i = row * p.cols + j;
    const float eff = lowbit_eff<DT>(load_elem<DT>(p.w, i), sf, rsf, clip, p.w_bits);
    if (DT == QAT_F32)
      reinterpret_cast<float*>(p.out)[i] = eff;
    else
      reinterpret_cast<__nv_bfloat16*>(p.out)[i] = __float2bfloat16_rn(eff);
  }
}

// bf16, two elements per instruction wherever the op exists packed: mul/add/sub.rn.bf16x2 round
// once where the reference rounds twice, which is identical for bf16 operands (products are
// exact in fp32; sums: oracle/proofs "addsub"); rint(t) for t in [-2.5, 1.5] is (t + 192) - 192
// in bf16 arithmetic (spacing 1 in [128, 256), ties to even; the lost sign of -0 dies in + 0.5).
__device__ __forceinline__ uint32_t lowbit_pair_bf16(uint32_t w2, float sf, float rsf, uint32_t sf2, uint32_t clip2,
                                                     int w_bits) {
  const float r0 = __fmul_rn(bf16lo(w2), rsf), r1 = __fmul_rn(bf16hi(w2), rsf);   // w / sf  (one multiply: "anyratio")
  uint32_t q2;
  if (w_bits == 1) {
    // sf * sign(r) on the pair: sign = (r > 0) - (r < 0) as packed compares (1.0 / 0.0 each; NaN compares false,
    // like torch.sign(NaN) = 0 here), fl_bf16 of the quotient first because it may round to zero
    const uint32_t rb = pack_bf16x2(r0, r1);
    const __nv_bfloat162 r2 = *reinterpret_cast<const __nv_bfloat162*>(&rb);
    const __nv_bfloat162 zero = __floats2bfloat162_rn(0.f, 0.f);
    const __nv_bfloat162 sg = __hsub2(__hgt2(r2, zero), __hlt2(r2, zero));
    q2 = mul_bf16x2(sf2, *reinterpret_cast<const uint32_t*>(&sg));                  // :211-213
  } else {
    const uint32_t k2 = 0x40004000u, kh = 0x3f003f00u, k192 = 0x43404340u;        // 2.0, 0.5, 192.0 as bf16x2
    uint32_t t2 = clamp_nan_bf16x2(pack_bf16x2(r0, r1), clip2 ^ 0x80008000u, clip2);  // :229-231
    t2 = sub_bf16x2(mul_bf16x2(t2, k2), kh);                                      // :232-233  * 2 - 0.5
    t2 = sub_bf16x2(add_bf16x2(t2, k192), k192);                                  // :228      round
    t2 = add_bf16x2(t2, kh);                                                      // :235      + 0.5
    q2 = mul_bf16x2(mul_bf16x2(sf2, t2), kh);                                     // :226-237  sf * t / 2
  }
  return add_bf16x2(sub_bf16x2(q2, w2), w2);                                      // :240-242  (q - w) + w
}

// One CTA per row, the row staged ONCE in shared memory (any width, any alignment): one HBM read, one HBM
// write.  mean|w| follows torch's own summation order (torch_sum_order.cuh): the 32 chains of ATen's
// vectorised cascade sum are the 32 lanes of a warp, the independent 16-step groups of a chain are spread over
// the CTA's warps (phase A), warp 0 folds the group sums through the cascade levels (phase B) and thread 0 does
// the final fold over vectors, tail and lanes — the bits of `w.abs().mean(dim=-1)` on the reference's CPU,
// fp32 and bf16 alike.
// VEC (both base pointers 16-byte aligned): global memory is touched in aligned 16-byte chunks whatever the row
// pitch — a row that starts `off` bytes into a chunk is staged `off` bytes into the buffer, so chunk j of the
// row's span is chunk j of shared memory, input and output rows have the same phase, and only the (at most two)
// chunks a row shares with its neighbours are handled element by element.  !VEC: element accesses throughout.
template <int DT, bool VEC>
__global__ void __launch_bounds__(512) lowbit_exact_kernel(const void* __restrict__ w, void* __restrict__ out,
                                                           int64_t cols, int w_bits, uint32_t gs_offset) {
  using N = Num<DT>;
  using Elem = typename std::conditional<DT == QAT_F32, float, uint16_t>::type;
  constexpr int kPer = N::kPerVec;   // elements per 16-byte chunk
  extern __shared__ uint4 smem16[];
  float* gs = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(smem16) + gs_offset);   // [groups][32]
  const int64_t row = blockIdx.x;
  const uint32_t tid = threadIdx.x, nthr = blockDim.x;
  const int lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
  const int64_t steps = tso::chain_steps(cols), groups = steps / tso::kGroup;
  float* chain = gs + groups * tso::kChains;   // [32]
  float* total = chain + tso::kChains;         // [1]
  // the row's span in aligned chunks (VEC); element e of the row sits at srow[e] either way
  const int64_t elem0 = row * cols;                                   // first element, counted from the base pointer
  const uint32_t off = VEC ? (uint32_t)(elem0 % kPer) : 0u;           // elements into its first chunk
  const int64_t chunk0 = VEC ? elem0 / kPer : 0;
  const uint32_t nchunks = VEC ? (uint32_t)((off + cols + kPer - 1) / kPer) : 0u;
  const uint32_t full_lo = off ? 1u : 0u;                             // chunks [full_lo, full_hi) belong to this row alone
  const bool shared_last = VEC && ((off + cols) % kPer) != 0;
  const uint32_t full_hi = shared_last ? nchunks - 1u : nchunks;
  const int64_t head = off ? min((int64_t)(kPer - off), cols) : 0;    // elements of a shared first chunk
  const int64_t tail0 = shared_last ? max(head, (int64_t)full_hi * kPer - off) : cols;   // first element of a shared last chunk
  Elem* srow = reinterpret_cast<Elem*>(smem16) + off;
  pdl_wait();
  pdl_launch_dependents();
  if constexpr (VEC) {
    const uint4* src = reinterpret_cast<const uint4*>(w) + chunk0;
    for (uint32_t j0 = full_lo + tid; j0 < full_hi; j0 += 4u * nthr) {   // four loads in flight per thread
      uint4 r[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t j = j0 + (uint32_t)u * nthr;
        if (j < full_hi) r[u] = ldg_stream(src + j);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t j = j0 + (uint32_t)u * nthr;
        if (j < full_hi) smem16[j] = r[u];
      }
    }
    const Elem* srcE = reinterpret_cast<const Elem*>(w) + elem0;
    if (tid < head) srow[tid] = srcE[tid];
    if (tail0 + tid < cols) srow[tail0 + tid] = srcE[tail0 + tid];
  } else {
    const Elem* srcE = reinterpret_cast<const Elem*>(w) + elem0;
    for (int64_t j = tid; j < cols; j += nthr) srow[j] = srcE[j];
  }
  __syncthreads();
  auto mag = [srow](int64_t e) -> float {
    if constexpr (DT == QAT_F32) return fabsf(srow[e]);
    else return fabsf(bf16lo((uint32_t)srow[e]));
  };
  if (cols >= tso::kLanes) {
    for (int64_t g = warp; g < groups; g += nwarps) gs[g * tso::kChains + lane] = tso::group_sum(mag, g, lane);
    __syncthreads();
    if (warp == 0) {
      chain[lane] = tso::chain_sum(mag, [gs, lane](int64_t g) { return gs[g * tso::kChains + lane]; }, steps, lane);
      __syncwarp();
      if (lane == 0) total[0] = tso::finalize(mag, [chain](int c) { return chain[c]; }, cols);
    }
  } else if (tid == 0) {
    total[0] = tso::short_row_sum(mag, cols);
  }
  __syncthreads();
  const float mean_abs = N::fl(__fdiv_rn(total[0], (float)cols));            // :205-210 / :219-224 (mean_out: sum / K)
  const float sf = (w_bits == 1) ? mean_abs : N::fl(__fmul_rn(2.0f, mean_abs));
  const float clip = N::fl(0.99f);  // 1 - 1e-2, cast to the tensor dtype by clamp (:218)
  const float rsf = (DT == QAT_BF16 && recip_range_ok(sf)) ? __frcp_rn(sf) : 0.f;
  Elem* outE = reinterpret_cast<Elem*>(out) + elem0;
  auto one = [&](int64_t c) {   // element c of the row, the scalar chain (exact division unless rsf allows the multiply)
    if constexpr (DT == QAT_F32) {
      outE[c] = lowbit_eff<DT>(srow[c], sf, 0.f, clip, w_bits);
    } else {
      const __nv_bfloat16 y = __float2bfloat16_rn(lowbit_eff<DT>(bf16lo((uint32_t)srow[c]), sf, rsf, clip, w_bits));
      outE[c] = *reinterpret_cast<const uint16_t*>(&y);
    }
  };
  if (!VEC || (DT == QAT_BF16 && rsf == 0.f)) {
    // element accesses; also bf16 rows whose scale is 0 / inf / NaN / outside the proven window (all-zero or
    // overflowed rows): exact IEEE division — rare, and kept out of the unrolled path (its slow path is a call)
#pragma unroll 1
    for (int64_t c = tid; c < cols; c += nthr) one(c);
    return;
  }
  if constexpr (VEC) {
    uint4* dst = reinterpret_cast<uint4*>(out) + chunk0;
    if constexpr (DT == QAT_BF16) {
      const uint32_t sf2 = pack_bf16x2(sf, sf), clip2 = pack_bf16x2(clip, clip);
      for (uint32_t j = full_lo + tid; j < full_hi; j += nthr) {   // the packed chain
        const uint4 v = smem16[j];
        stg_stream(dst + j, make_uint4(lowbit_pair_bf16(v.x, sf, rsf, sf2, clip2, w_bits),
                                       lowbit_pair_bf16(v.y, sf, rsf, sf2, clip2, w_bits),
                                       lowbit_pair_bf16(v.z, sf, rsf, sf2, clip2, w_bits),
                                       lowbit_pair_bf16(v.w, sf, rsf, sf2, clip2, w_bits)));
      }
    } else {
      for (uint32_t j = full_lo + tid; j < full_hi; j += nthr) {
        const uint4 v = smem16[j];
        stg_stream(dst + j, make_uint4(__float_as_uint(lowbit_eff<DT>(__uint_as_float(v.x), sf, 0.f, clip, w_bits)),
                                       __float_as_uint(lowbit_eff<DT>(__uint_as_float(v.y), sf, 0.f, clip, w_bits)),
                                       __float_as_uint(lowbit_eff<DT>(__uint_as_float(v.z), sf, 0.f, clip, w_bits)),
                                       __float_as_uint(lowbit_eff<DT>(__uint_as_float(v.w), sf, 0.f, clip, w_bits))));
      }
    }
    if (tid < head) one(tid);
    if (tail0 + tid < cols) one(tail0 + tid);
  }
}

constexpr size_t kMaxDynSmem = 227 * 1024;

// shared memory of one CTA: the row (16-byte padded), the level-0 group sums, 32 chain sums, the total
inline size_t exact_smem_bytes(int64_t cols, int elem_bytes, uint32_t* gs_offset) {
  const size_t row_bytes = (((size_t)cols * elem_bytes + 15) & ~(size_t)15) + 16;   // + the row's phase within a chunk
  const size_t groups = (size_t)(tso::chain_steps(cols) / tso::kGroup);
  *gs_offset = (uint32_t)row_bytes;
  return row_bytes + (groups * tso::kChains + tso::kChains + 4) * sizeof(float);
}

template <int DT, bool VEC>
cudaError_t launch_exact_variant(const void* w, void* out, int64_t rows, int64_t cols, int w_bits, size_t smem,
                                 uint32_t gs_offset, int threads, cudaStream_t st) {
  static std::atomic<bool> raised{false};   // > 48 KB of dynamic shared memory is an opt-in, once per kernel
  if (smem > 48 * 1024 && !raised.load(std::memory_order_acquire)) {
    cudaError_t e = cudaFuncSetAttribute(lowbit_exact_kernel<DT, VEC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kMaxDynSmem);
    if (e != cudaSuccess) return e;
    raised.store(true, std::memory_order_release);
  }
  return launch_pdl(lowbit_exact_kernel<DT, VEC>, dim3((unsigned)rows), dim3((unsigned)threads), smem, st, w, out, cols,
                    w_bits, gs_offset);
}

// false: the row does not fit one CTA's shared memory (the caller falls back to the two-pass kernels)
template <int DT>
bool launch_exact(const void* w, void* out, int64_t rows, int64_t cols, int w_bits, cudaStream_t st, cudaError_t* err) {
  const int eb = Num<DT>::kBytes;
  uint32_t gs_offset = 0;
  const size_t smem = exact_smem_bytes(cols, eb, &gs_offset);
  if (smem > kMaxDynSmem || rows > 0x7fffffffLL || cols >= (1LL << 24)) return false;
  // one round of four 16-byte loads per thread where the row allows it: a CTA's lifetime is what the last,
  // partly filled wave of rows costs, so it is kept short rather than the CTA small (profiles/r02_lowbit_exact.json)
  const int64_t chunks = ((int64_t)cols * eb + 15) / 16;
  const int threads = (int)std::min<int64_t>(512, std::max<int64_t>(128, ((chunks + 3) / 4 + 63) / 64 * 64));
  const bool vec = ((uintptr_t)w & 15) == 0 && ((uintptr_t)out & 15) == 0;
  *err = vec ? launch_exact_variant<DT, true>(w, out, rows, cols, w_bits, smem, gs_offset, threads, st)
             : launch_exact_variant<DT, false>(w, out, rows, cols, w_bits, smem, gs_offset, threads, st);
  return true;
}

}  // namespace
}  // namespace qat

extern "C" {

size_t qat_lowbit_workspace_bytes(int64_t rows, int layerwise) {
  if (rows <= 0) return 0;
  return (size_t)(layerwise ? 1 : rows) * sizeof(double);
}

int qat_lowbit_weight_fwd(const void* w, void* w_eff, int64_t rows, int64_t cols, int dtype,
                          int w_bits, int layerwise, void* workspace, size_t workspace_bytes,
                          void* stream) {
  using namespace qat;
  QAT_CHECK_ARG(dtype == QAT_F32 || dtype == QAT_BF16, "dtype must be QAT_F32 or QAT_BF16 (got %d)", dtype);
  QAT_CHECK_ARG(w_bits == 1 || w_bits == 2, "low-bit path handles w_bits 1 or 2 (got %d)", w_bits);
  QAT_CHECK_ARG(rows >= 0 && cols >= 0, "negative shape");
  if (rows == 0 || cols == 0) return QAT_OK;
  QAT_CHECK_ARG(w != nullptr && w_eff != nullptr && w != w_eff, "w / w_eff NULL or aliased");
  const size_t need = qat_lowbit_workspace_bytes(rows, layerwise);
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("low-bit weight path needs %zu bytes of workspace (got %zu)", need, workspace_bytes);
    return QAT_ERR_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // Per-row scales, and the layerwise scale of a tensor below 32768 elements (which torch reduces as ONE serial
  // cascade over the flattened tensor): one pass, mean|w| in torch's own order.  A larger layerwise tensor is
  // split over torch's intra-op threads — the reference's bits depend on its machine — and takes the
  // order-independent double-precision sum below, like rows too long for one CTA's shared memory.
  const bool flat = layerwise && rows * cols < 32768;
  if (!layerwise || flat) {
    const int64_t r = flat ? 1 : rows, c = flat ? rows * cols : cols;
    cudaError_t le = cudaSuccess;
    const bool done = dtype == QAT_F32 ? launch_exact<QAT_F32>(w, w_eff, r, c, w_bits, st, &le)
                                       : launch_exact<QAT_BF16>(w, w_eff, r, c, w_bits, st, &le);
    if (done) {
      if (le != cudaSuccess) return cuda_fail(le, "lowbit_exact_kernel");
      QAT_CHECK_LAUNCH("lowbit_exact_kernel");
      return QAT_OK;
    }
  }
  if (rows > 65535) {
    set_error("low-bit weight path: two-pass kernels support at most 65535 rows (got %lld)", (long long)rows);
    return QAT_ERR_UNSUPPORTED;
  }
  cudaError_t e = cudaMemsetAsync(workspace, 0, need, st);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
  LowbitParams p{};
  p.w = w;
  p.out = w_eff;
  p.sums = reinterpret_cast<double*>(workspace);
  p.rows = rows;
  p.cols = cols;
  p.w_bits = w_bits;
  p.layerwise = layerwise ? 1 : 0;
  p.chunk = 8192;
  dim3 grid((unsigned)((cols + p.chunk - 1) / p.chunk), (unsigned)rows);
  if (dtype == QAT_F32) {
    lowbit_sum_kernel<QAT_F32><<<grid, kThreads, 0, st>>>(p);
    QAT_CHECK_LAUNCH("lowbit_sum_kernel");
    lowbit_apply_kernel<QAT_F32><<<grid, kThreads, 0, st>>>(p);
    QAT_CHECK_LAUNCH("lowbit_apply_kernel");
  } else {
    lowbit_sum_kernel<QAT_BF16><<<grid, kThreads, 0, st>>>(p);
    QAT_CHECK_LAUNCH("lowbit_sum_kernel");
    lowbit_apply_kernel<QAT_BF16><<<grid, kThreads, 0, st>>>(p);
    QAT_CHECK_LAUNCH("lowbit_apply_kernel");
  }
  return QAT_OK;
}

}  // extern "C"
