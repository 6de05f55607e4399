// ste.cu — K3: straight-through-estimator backward with its clip mask.
//
// Replaces /root/reference/models/utils_quant.py:83-87 and :158-162
//   grad_input = grad_output.clone(); grad_input[x >= hi] = 0; grad_input[x <= lo] = 0
// (5 ATen kernels: clone + 2 bool-mask compares + 2 masked fills) with one
// streaming pass: read g, read x (or a forward-emitted packed mask), write gx.
// HBM-bound: 3*sizeof(T) B/elem from x, 2*sizeof(T) + 1/8 B/elem from a mask.
#define QAT_PDL_FAMILY 1   // bit of QAT_B200_PDL_MASK (common.cuh)
#include "common.cuh"

namespace qat {
namespace {

constexpr uint32_t kFull = 0xffffffffu;
constexpr int kThreads = 256;
constexpr int kUnroll = 4;  // 16-byte vectors per thread per tile, all loaded before use
// Grid of the vector kernel: ONE CTA PER TILE (0 = no cap).  The former cap of 8 CTAs per SM assumed an occupancy
// the 48-register bf16 kernel does not have (5 per SM), leaving a ragged second wave of grid-striding CTAs:
// bf16 [8192, 4096] 35.1 -> 33.1 us (0.89 -> 0.94 of the HBM peak), from a mask 0.92 -> 0.98, fp32 0.96 -> 1.03
// (profiles/r02_dequant_ste_tune.json; outputs bit-identical for every grid).
constexpr int kCtasPerSmDefault = 0;

struct BwdParams {
  const void* g;
  const void* x;          // nullptr when driven by `mask_in`
  const uint8_t* mask_in;  // packed pass-mask from the forward
  void* gx;
  uint8_t* mask_out;  // optional
  float lo, hi;       // rounded to the tensor dtype on the host
  const float* clip_dev;  // optional: {lo, hi} in device memory (a CUDA clip_val), read in-kernel
  int64_t n;          // elements
  int64_t nvec;       // full 16-byte vectors
};

template <int DT>
__device__ __forceinline__ uint32_t pass_bits(const uint4& xv, float lo, float hi) {
  uint32_t pass = 0;
#pragma unroll
  for (int i = 0; i < Num<DT>::kPerVec; ++i) {
    const float xf = vec_get<DT>(xv, i);
    pass |= ((xf >= hi || xf <= lo) ? 0u : 1u) << i;  // NaN: both compares false => passes
  }
  return pass;
}

template <int DT>
__device__ __forceinline__ uint4 apply_pass(const uint4& gv, uint32_t pass) {
  uint4 o;
  if (DT == QAT_F32) {
    o.x = (pass & 1u) ? gv.x : 0u;
    o.y = (pass & 2u) ? gv.y : 0u;
    o.z = (pass & 4u) ? gv.z : 0u;
    o.w = (pass & 8u) ? gv.w : 0u;
  } else {
    // 2 mask bits -> 0x0000ffff / 0xffff0000 lanes
    auto m2 = [](uint32_t b) { return ((b & 1u) ? 0x0000ffffu : 0u) | ((b & 2u) ? 0xffff0000u : 0u); };
    o.x = gv.x & m2(pass);
    o.y = gv.y & m2(pass >> 2);
    o.z = gv.z & m2(pass >> 4);
    o.w = gv.w & m2(pass >> 6);
  }
  return o;
}

// grid-stride over tiles of kThreads*kUnroll vectors; trip counts are uniform
// per CTA so the nibble-pairing shuffle below is convergent.
template <int DT, bool FROM_MASK>
__global__ void __launch_bounds__(kThreads) ste_bwd_kernel(const BwdParams p) {
  constexpr int N = Num<DT>::kPerVec;
  constexpr int64_t kTile = (int64_t)kThreads * kUnroll;
  const char* g = reinterpret_cast<const char*>(p.g);
  const char* x = reinterpret_cast<const char*>(p.x);
  char* gx = reinterpret_cast<char*>(p.gx);
  pdl_wait();
  pdl_launch_dependents();
  float lo = p.lo, hi = p.hi;
  if (!FROM_MASK && p.clip_dev != nullptr) {  // compared in x's dtype, like x.ge(clip_val[1])
    lo = Num<DT>::fl(p.clip_dev[0]);
    hi = Num<DT>::fl(p.clip_dev[1]);
  }
  for (int64_t base = (int64_t)blockIdx.x * kTile; base < p.nvec; base += (int64_t)gridDim.x * kTile) {
    uint4 gv[kUnroll], xv[kUnroll];
    uint32_t mb[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t j = base + (int64_t)u * kThreads + threadIdx.x;
      if (j < p.nvec) {
        gv[u] = ldg_stream(g + j * 16);
        if (FROM_MASK) {
          const uint32_t b = p.mask_in[(j * N) >> 3];
          mb[u] = (N == 8) ? b : ((j & 1) ? (b >> 4) : (b & 0xfu));
        } else {
          xv[u] = ldg_stream(x + j * 16);
        }
      } else {
        gv[u] = make_uint4(0u, 0u, 0u, 0u);
        xv[u] = make_uint4(0u, 0u, 0u, 0u);
        mb[u] = 0u;
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t j = base + (int64_t)u * kThreads + threadIdx.x;
      const bool valid = j < p.nvec;
      const uint32_t pass = FROM_MASK ? mb[u] : pass_bits<DT>(xv[u], lo, hi);
      if (valid) stg_stream(gx + j * 16, apply_pass<DT>(gv[u], pass));
      if (!FROM_MASK && p.mask_out != nullptr) {
        if (N == 8) {
          if (valid) p.mask_out[j] = (uint8_t)pass;
        } else {
          const uint32_t mine = valid ? pass : 0u;
          const uint32_t other = __shfl_xor_sync(kFull, mine, 1);
          // an odd last vector shares its byte with the scalar tail, which owns it
          const bool tail_owns = (p.nvec & 1) && (p.nvec * N < p.n) && (j == p.nvec - 1);
          if (valid && !(threadIdx.x & 1) && !tail_owns)
            p.mask_out[j >> 1] = (uint8_t)(mine | (other << 4));
        }
      }
    }
  }
  // tail: n % N trailing elements, one thread each (block 0 only)
  const int64_t tail0 = p.nvec * N;
  if (blockIdx.x == 0) {
    const int64_t i = tail0 + threadIdx.x;
    if (i < p.n) {
      bool pass;
      if (FROM_MASK) {
        pass = (p.mask_in[i >> 3] >> (i & 7)) & 1u;
      } else {
        const float xf = (DT == QAT_F32) ? reinterpret_cast<const float*>(p.x)[i]
                                         : bf16lo(reinterpret_cast<const uint16_t*>(p.x)[i]);
        pass = !(xf >= hi || xf <= lo);
      }
      if (DT == QAT_F32) {
        const uint32_t gvb = reinterpret_cast<const uint32_t*>(p.g)[i];
        reinterpret_cast<uint32_t*>(p.gx)[i] = pass ? gvb : 0u;
      } else {
        const uint16_t gvb = reinterpret_cast<const uint16_t*>(p.g)[i];
        reinterpret_cast<uint16_t*>(p.gx)[i] = pass ? gvb : (uint16_t)0;
      }
    }
    if (!FROM_MASK && p.mask_out != nullptr && threadIdx.x == 0 && tail0 < p.n) {
      // tail0 is a multiple of N; when N == 4 and nvec is odd the tail shares
      // its byte with the last vector's nibble, so this thread rebuilds the
      // whole byte (the vector loop skips it, see tail_owns).
      const int64_t byte0 = tail0 >> 3;
      const int64_t nbytes = (p.n + 7) >> 3;
      for (int64_t b = byte0; b < nbytes; ++b) {
        uint32_t bits = 0;
        for (int k = 0; k < 8; ++k) {
          const int64_t i2 = b * 8 + k;
          if (i2 >= p.n) break;
          const float xf = (DT == QAT_F32) ? reinterpret_cast<const float*>(p.x)[i2]
                                           : bf16lo(reinterpret_cast<const uint16_t*>(p.x)[i2]);
          bits |= ((xf >= hi || xf <= lo) ? 0u : 1u) << k;
        }
        p.mask_out[b] = (uint8_t)bits;
      }
    }
  }
}

// unaligned pointers: one element per thread
template <int DT, bool FROM_MASK>
__global__ void __launch_bounds__(kThreads) ste_bwd_scalar_kernel(const BwdParams p) {
  float lo = p.lo, hi = p.hi;
  if (!FROM_MASK && p.clip_dev != nullptr) {
    lo = Num<DT>::fl(p.clip_dev[0]);
    hi = Num<DT>::fl(p.clip_dev[1]);
  }
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < p.n;
       i += (int64_t)gridDim.x * kThreads) {
    bool pass;
    if (FROM_MASK) {
      pass = (p.mask_in[i >> 3] >> (i & 7)) & 1u;
    } else {
      const float xf = (DT == QAT_F32) ? reinterpret_cast<const float*>(p.x)[i]
                                       : bf16lo(reinterpret_cast<const uint16_t*>(p.x)[i]);
      pass = !(xf >= hi || xf <= lo);
    }
    if (DT == QAT_F32) {
      const uint32_t gvb = reinterpret_cast<const uint32_t*>(p.g)[i];
      reinterpret_cast<uint32_t*>(p.gx)[i] = pass ? gvb : 0u;
    } else {
      const uint16_t gvb = reinterpret_cast<const uint16_t*>(p.g)[i];
      reinterpret_cast<uint16_t*>(p.gx)[i] = pass ? gvb : (uint16_t)0;
    }
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <bool FROM_MASK>
int bwd_entry(const void* g, const void* x, const uint8_t* mask_in, void* gx, uint8_t* mask_out,
              float lo, float hi, int64_t n, int dtype, void* stream, const float* clip_dev = nullptr) {
  QAT_CHECK_ARG(dtype == QAT_F32 || dtype == QAT_BF16, "dtype must be QAT_F32 or QAT_BF16 (got %d)", dtype);
  QAT_CHECK_ARG(n >= 0, "negative element count");
  if (n == 0) return QAT_OK;
  QAT_CHECK_ARG(g != nullptr && gx != nullptr, "g / gx is NULL");
  QAT_CHECK_ARG(FROM_MASK ? mask_in != nullptr : x != nullptr, "x / mask is NULL");
  QAT_CHECK_ARG(gx != g && gx != x, "gx must not alias g or x");
  BwdParams p{};
  p.g = g;
  p.x = x;
  p.mask_in = mask_in;
  p.gx = gx;
  p.mask_out = mask_out;
  p.lo = dtype == QAT_F32 ? lo : __bfloat162float(__float2bfloat16_rn(lo));
  p.hi = dtype == QAT_F32 ? hi : __bfloat162float(__float2bfloat16_rn(hi));
  p.clip_dev = clip_dev;
  p.n = n;
  const int per = dtype == QAT_F32 ? 4 : 8;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool vec = aligned16(g) && aligned16(gx) && (FROM_MASK || aligned16(x));
  const int sms = num_sms();
  if (vec) {
    p.nvec = n / per;
    const int64_t tile = (int64_t)kThreads * kUnroll;
    int64_t grid = (p.nvec + tile - 1) / tile;
    const int64_t cap = kCtasPerSmDefault > 0 ? (int64_t)sms * kCtasPerSmDefault : (int64_t)0x7fffffff;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    if (dtype == QAT_F32)
      (void)launch_pdl(ste_bwd_kernel<QAT_F32, FROM_MASK>, dim3((unsigned)grid), dim3(kThreads), 0, st, p);
    else
      (void)launch_pdl(ste_bwd_kernel<QAT_BF16, FROM_MASK>, dim3((unsigned)grid), dim3(kThreads), 0, st, p);
    QAT_CHECK_LAUNCH("ste_bwd_kernel");
  } else {
    if (mask_out != nullptr) {
      set_error("packed-mask output needs 16-byte aligned g/x/gx");
      return QAT_ERR_UNSUPPORTED;
    }
    int64_t grid = (n + kThreads - 1) / kThreads;
    const int64_t cap = (int64_t)sms * 8;
    if (grid > cap) grid = cap;
    if (dtype == QAT_F32)
      ste_bwd_scalar_kernel<QAT_F32, FROM_MASK><<<(unsigned)grid, kThreads, 0, st>>>(p);
    else
      ste_bwd_scalar_kernel<QAT_BF16, FROM_MASK><<<(unsigned)grid, kThreads, 0, st>>>(p);
    QAT_CHECK_LAUNCH("ste_bwd_scalar_kernel");
  }
  return QAT_OK;
}

}  // namespace
}  // namespace qat

extern "C" {

int qat_ste_bwd(const void* g, const void* x, void* gx, uint8_t* mask_out, float clip_lo,
                float clip_hi, int64_t n, int dtype, void* stream) {
  return qat::bwd_entry<false>(g, x, nullptr, gx, mask_out, clip_lo, clip_hi, n, dtype, stream);
}

int qat_ste_bwd_devclip(const void* g, const void* x, void* gx, uint8_t* mask_out, const float* clip_dev,
                        int64_t n, int dtype, void* stream) {
  if (clip_dev == nullptr) {
    qat::set_error("clip_dev is NULL");
    return QAT_ERR_BAD_ARG;
  }
  return qat::bwd_entry<false>(g, x, nullptr, gx, mask_out, 0.f, 0.f, n, dtype, stream, clip_dev);
}

int qat_ste_bwd_from_mask(const void* g, const uint8_t* mask, void* gx, int64_t n, int dtype,
                          void* stream) {
  return qat::bwd_entry<true>(g, nullptr, mask, gx, nullptr, 0.f, 0.f, n, dtype, stream);
}

}  // extern "C"
