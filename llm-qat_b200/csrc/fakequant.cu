// fakequant.cu — K1 (Sym), K2 (Asym) and K5 (long-row / layerwise) forward
// kernels of the fake-quantization hot path, hand-written for sm_100a.
//
// Replaces the eager ATen chains of /root/reference/models/utils_quant.py:50-72
// (9 kernels, ~18 tensor passes) and :110-147 (3 reductions + 9 elementwise)
// with ONE pass: each row is read from HBM exactly once with 128-bit streaming
// loads, held in registers across the abs-max / min-max warp-shuffle tree, then
// quantized, dequantized and written back with 128-bit streaming stores.
// Optional side outputs (integer codes for the tcgen05 GEMM, row scales, packed
// STE mask) come out of the same pass.
//
// HBM-bound: algorithmic traffic = 2*sizeof(T) bytes per element (+1/8 B with
// the mask, +1 or 2 B with codes).  See DESIGN.md section "K1/K2".
#define QAT_PDL_FAMILY 0   // bit of QAT_B200_PDL_MASK (common.cuh)
#include <cstdlib>

#include "common.cuh"

namespace qat {
namespace {

constexpr uint32_t kFull = 0xffffffffu;

struct FwdParams {
  const void* x;
  void* y;
  void* codes;
  int codes_kind;
  float* st0;  // Sym: s      Asym: a (= alpha + 1e-8)
  float* st1;  // Sym: e      Asym: beta
  uint8_t* mask;
  float lo, hi;  // already rounded to the tensor dtype by the host wrapper
  int64_t rows;
  int64_t cols;
  int64_t nvec;  // vectors (VEC) or elements (scalar path) per row
  float qmax;    // Sym: Q = 2^(bits-1)-1     Asym: S = 2^bits-1, negated in the QAT_ASYM_DIV_RECIP mode
  int group;     // threads cooperating on one row (power of two, >= 32)
  int log2_group;
  // long-row path
  uint32_t* ws;
  int64_t chunk;  // vectors per CTA
  int poison_inf;  // Sym GEMM feed: e = NaN for rows whose abs-max is +inf (see sym_fwd_feed)
};

// ---- reductions --------------------------------------------------------------
__device__ __forceinline__ void warp_reduce(RowStat& r, bool sym) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    if (sym) {
      r.amax_bits = max(r.amax_bits, __shfl_xor_sync(kFull, r.amax_bits, o));
    } else {
      r.mx = fmaxf(r.mx, __shfl_xor_sync(kFull, r.mx, o));
      r.mn = fminf(r.mn, __shfl_xor_sync(kFull, r.mn, o));
      r.nan |= __shfl_xor_sync(kFull, r.nan, o);
    }
  }
}

__device__ __forceinline__ RowStat stat_identity() {
  RowStat r;
  r.amax_bits = 0u;
  r.mx = -INFINITY;
  r.mn = INFINITY;
  r.nan = 0u;
  return r;
}

// Reduce over `group` consecutive threads of the CTA (group % 32 == 0); every
// thread of the group receives the result.  One __syncthreads when group > 32.
template <bool SYM>
__device__ __forceinline__ void group_reduce(RowStat& r, int group, uint32_t* sm_u, float* sm_mx,
                                             float* sm_mn) {
  warp_reduce(r, SYM);
  if (group > 32) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
      if (SYM) {
        sm_u[warp] = r.amax_bits;
      } else {
        sm_mx[warp] = r.mx;
        sm_mn[warp] = r.mn;
        sm_u[warp] = r.nan;
      }
    }
    __syncthreads();
    const int nw = group >> 5;
    const int base = (warp / nw) * nw;
    RowStat t = stat_identity();
    if (lane < nw) {
      if (SYM) {
        t.amax_bits = sm_u[base + lane];
      } else {
        t.mx = sm_mx[base + lane];
        t.mn = sm_mn[base + lane];
        t.nan = sm_u[base + lane];
      }
    }
    warp_reduce(t, SYM);
    r = t;
  }
}

template <int DT, bool SYM>
__device__ __forceinline__ void accumulate_vec(RowStat& r, const uint4& v) {
  if (SYM) {
    if (DT == QAT_F32) {
      r.amax_bits = max(r.amax_bits, v.x & 0x7fffffffu);
      r.amax_bits = max(r.amax_bits, v.y & 0x7fffffffu);
      r.amax_bits = max(r.amax_bits, v.z & 0x7fffffffu);
      r.amax_bits = max(r.amax_bits, v.w & 0x7fffffffu);
    } else {
      // packed |bf16| maxima; r.amax_bits holds two u16 lanes until finalised
      r.amax_bits = __vmaxu2(r.amax_bits, v.x & 0x7fff7fffu);
      r.amax_bits = __vmaxu2(r.amax_bits, v.y & 0x7fff7fffu);
      r.amax_bits = __vmaxu2(r.amax_bits, v.z & 0x7fff7fffu);
      r.amax_bits = __vmaxu2(r.amax_bits, v.w & 0x7fff7fffu);
    }
  } else {
#pragma unroll
    for (int i = 0; i < Num<DT>::kPerVec; ++i) {
      float f = vec_get<DT>(v, i);
      r.mx = fmaxf(r.mx, f);
      r.mn = fminf(r.mn, f);
      r.nan |= (f != f) ? 1u : 0u;
    }
  }
}

template <int DT, bool SYM>
__device__ __forceinline__ void accumulate_scalar(RowStat& r, float f) {
  if (SYM) {
    r.amax_bits = max(r.amax_bits, __float_as_uint(f) & 0x7fffffffu);
  } else {
    r.mx = fmaxf(r.mx, f);
    r.mn = fminf(r.mn, f);
    r.nan |= (f != f) ? 1u : 0u;
  }
}

// bf16 Sym keeps two u16 lanes while accumulating; fold them into fp32 |x| bits
template <int DT, bool SYM, bool VEC>
__device__ __forceinline__ void finalize_thread_stat(RowStat& r) {
  if (SYM && VEC && DT != QAT_F32) {
    uint32_t m = max(r.amax_bits & 0xffffu, r.amax_bits >> 16);
    r.amax_bits = m << 16;
  }
}

template <int DT>
__device__ __forceinline__ float load_scalar(const void* x, int64_t i) {
  if (DT == QAT_F32) return reinterpret_cast<const float*>(x)[i];
  return bf16lo(reinterpret_cast<const uint16_t*>(x)[i]);
}

// AsymScale's packed-bf16 chain, callable from code that is also instantiated for SymScale
template <int DT>
__device__ __forceinline__ bool sc_packed(const AsymScale<DT>& sc) { return sc.packed; }
template <int DT>
__device__ __forceinline__ bool sc_packed(const SymScale<DT>&) { return false; }
template <int DT>
__device__ __forceinline__ uint32_t sc_pair(const AsymScale<DT>& sc, uint32_t w, float* c0, float* c1) {
  return sc.pair_bf16(w, c0, c1);
}
template <int DT>
__device__ __forceinline__ uint32_t sc_pair(const SymScale<DT>&, uint32_t w, float*, float*) { return w; }

// ---- per-vector quantize + all outputs ------------------------------------
// `e0` = flat element index of the vector's first element.
template <int DT, bool SYM, bool FAST, typename Scale>
__device__ __forceinline__ void emit_vec(const FwdParams& p, const Scale& sc, const uint4& v,
                                         int64_t e0, bool valid) {
  constexpr int N = Num<DT>::kPerVec;
  float yv[N], qv[N];
  if constexpr (SYM && DT == QAT_BF16) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t pw = mul_bf16x2(w[j], sc.s2);  // fl_bf16(x * s), two elements
      yv[(2 * j) % N] = sc.template apply_p<FAST>(bf16lo(pw), &qv[(2 * j) % N]);
      yv[(2 * j + 1) % N] = sc.template apply_p<FAST>(bf16hi(pw), &qv[(2 * j + 1) % N]);
    }
  } else if (!SYM && DT == QAT_BF16 && FAST && sc_packed(sc)) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t yw = sc_pair(sc, w[j], &qv[(2 * j) % N], &qv[(2 * j + 1) % N]);
      yv[(2 * j) % N] = bf16lo(yw);
      yv[(2 * j + 1) % N] = bf16hi(yw);
    }
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) yv[i] = sc.template apply<FAST>(vec_get<DT>(v, i), &qv[i]);
  }
  if (p.y != nullptr && valid) {
    char* dst = reinterpret_cast<char*>(p.y) + e0 * Num<DT>::kOutBytes;
    if (Num<DT>::kOutBytes == 4) {
#pragma unroll
      for (int k = 0; k < N / 4; ++k)   // one store for fp32 input, two for bf16 input with fp32 y
        stg_stream(dst + 16 * k, make_uint4(__float_as_uint(yv[4 * k]), __float_as_uint(yv[4 * k + 1]),
                                            __float_as_uint(yv[4 * k + 2]), __float_as_uint(yv[4 * k + 3])));
    } else {
      uint4 o;
      o.x = pack_bf16x2(yv[0], yv[1]);
      o.y = pack_bf16x2(yv[2 % N], yv[3 % N]);
      o.z = pack_bf16x2(yv[4 % N], yv[5 % N]);
      o.w = pack_bf16x2(yv[6 % N], yv[7 % N]);
      stg_stream(dst, o);
    }
  }
  if (p.codes != nullptr && valid) {
    if (p.codes_kind == QAT_CODES_I8) {
      uint32_t w[N / 4];
#pragma unroll
      for (int i = 0; i < N / 4; ++i) w[i] = pack_codes4<SYM>(qv[4 * i], qv[4 * i + 1], qv[4 * i + 2], qv[4 * i + 3]);
      uint8_t* dst = reinterpret_cast<uint8_t*>(p.codes) + e0;
      if (N == 4) {
        *reinterpret_cast<uint32_t*>(dst) = w[0];
      } else {
        *reinterpret_cast<uint2*>(dst) = make_uint2(w[0], w[(N / 4) - 1]);
      }
    } else {
      uint32_t w[N / 2];
#pragma unroll
      for (int i = 0; i < N / 2; ++i)
        w[i] = (uint32_t)(uint16_t)code_i16(qv[2 * i]) |
               ((uint32_t)(uint16_t)code_i16(qv[2 * i + 1]) << 16);
      int16_t* dst = reinterpret_cast<int16_t*>(p.codes) + e0;
      if (N == 4) {
        *reinterpret_cast<uint2*>(dst) = make_uint2(w[0], w[1]);
      } else {
        *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2 % (N / 2)], w[3 % (N / 2)]);
      }
    }
  }
  if (p.mask != nullptr) {  // uniform branch; host guarantees (rows*cols) byte alignment rules
    uint32_t pass = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const float xf = vec_get<DT>(v, i);
      pass |= ((xf >= p.hi || xf <= p.lo) ? 0u : 1u) << i;  // utils_quant.py:85-86
    }
    if (N == 8) {
      if (valid) p.mask[e0 >> 3] = (uint8_t)pass;
    } else {
      // two adjacent lanes hold the two nibbles of one byte
      uint32_t mine = valid ? pass : 0u;
      uint32_t other = __shfl_xor_sync(kFull, mine, 1);
      if (valid && !(threadIdx.x & 1)) p.mask[e0 >> 3] = (uint8_t)(mine | (other << 4));
    }
  }
}

template <int DT, bool SYM, bool FAST, typename Scale>
__device__ __forceinline__ void emit_scalar(const FwdParams& p, const Scale& sc, float xf,
                                            int64_t e0) {
  float q;
  float yf = sc.template apply<FAST>(xf, &q);
  if (p.y != nullptr) {
    if (Num<DT>::kOutBytes == 4)
      reinterpret_cast<float*>(p.y)[e0] = yf;
    else
      reinterpret_cast<__nv_bfloat16*>(p.y)[e0] = __float2bfloat16_rn(yf);
  }
  if (p.codes != nullptr) {
    if (p.codes_kind == QAT_CODES_I8)
      reinterpret_cast<uint8_t*>(p.codes)[e0] = code_i8<SYM>(q);
    else
      reinterpret_cast<int16_t*>(p.codes)[e0] = code_i16(q);
  }
}

template <int DT, bool SYM>
struct ScaleOf;
template <int DT>
struct ScaleOf<DT, true> {
  using type = SymScale<DT>;
  static __device__ __forceinline__ type make(const RowStat& r, float qmax) {
    type s;
    s.derive(__uint_as_float(r.amax_bits), qmax);
    return s;
  }
  static __device__ __forceinline__ float st0(const type& s) { return s.s; }
  static __device__ __forceinline__ float st1(const type& s) { return s.e; }
};
template <int DT>
struct ScaleOf<DT, false> {
  using type = AsymScale<DT>;
  static __device__ __forceinline__ type make(const RowStat& r, float qmax) {
    type s;
    // a negative qmax carries the "multiply by fl(1/S)" mode of qat_set_asym_div (FwdParams::qmax)
    s.derive(r.mx, r.mn, r.nan != 0u, fabsf(qmax));
    s.mulS = qmax < 0.f;
    return s;
  }
  static __device__ __forceinline__ float st0(const type& s) { return s.a; }
  static __device__ __forceinline__ float st1(const type& s) { return s.beta; }
};

// =============================================================================
// K1 / K2: one row per thread group, the row lives in registers between the
// reduction and the quantize pass => exactly one HBM read + one HBM write.
//   grid  = ceil(rows / (blockDim / group)),  block = max(group, 256)
//   ITERS = 16-byte vectors per thread, compile-time unrolled so all loads of a
//           row are in flight before the first use.
//   OUT   = which outputs exist, resolved at compile time so the element loop
//           carries no branches:  OUT_Y (y [+ scales]) is Quantizer.apply;
//           OUT_FEED (int8 codes + scales [+ mask], no y) feeds the tcgen05 GEMM;
//           OUT_ANY keeps every output optional at run time.
// The kernel is instruction-issue bound in bf16 (4 B/elem of traffic), hence:
// 32-bit in-row indexing, one lane per warp derives the scale (two frcp.rn) and
// shuffles it, packed bf16x2 multiply and packed sign restoration.
// =============================================================================
constexpr int OUT_Y = 0, OUT_FEED = 1, OUT_ANY = 2;

template <int DT, bool SYM>
__device__ __forceinline__ typename ScaleOf<DT, SYM>::type warp_derive_scale(const RowStat& st, float qmax) {
  using SO = ScaleOf<DT, SYM>;
  typename SO::type sc;
  const int lane = threadIdx.x & 31;
  if (lane == 0) sc = SO::make(st, qmax);
  if constexpr (SYM) {
    sc.s = __shfl_sync(kFull, sc.s, 0);
    sc.e = __shfl_sync(kFull, sc.e, 0);
    sc.r = __shfl_sync(kFull, sc.r, 0);
    sc.finish(qmax);
  } else {
    sc.a = __shfl_sync(kFull, sc.a, 0);
    sc.beta = __shfl_sync(kFull, sc.beta, 0);
    sc.ra.r1 = __shfl_sync(kFull, sc.ra.r1, 0);
    sc.S = fabsf(qmax);
    sc.mulS = qmax < 0.f;
    sc.rS = __shfl_sync(kFull, sc.rS, 0);
    sc.ra_rn = __shfl_sync(kFull, sc.ra_rn, 0);
    sc.finish();
  }
  return sc;
}

// y for one 16-byte vector, no side outputs (the Quantizer.apply hot loop)
// o[0] (and o[1] when y elements are twice as wide as x elements) receive the output vectors
template <int DT, bool SYM, bool FAST, typename Scale>
__device__ __forceinline__ void quant_vec_y(const Scale& sc, const uint4& v,
                                            uint4 (&oo)[Num<DT>::kOutBytes / Num<DT>::kBytes]) {
  uint4 o;
  if constexpr (SYM && DT == QAT_BF16) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t ow[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t pw = mul_bf16x2(w[j], sc.s2);  // fl_bf16(x * s), two elements
      const float c0 = rintf(bf16lo(pw)), c1 = rintf(bf16hi(pw));
      if (FAST && sc.mulq) {
        ow[j] = pack_bf16x2(__fmul_rn(c0, sc.r), __fmul_rn(c1, sc.r));   // == fl_bf16(c / e), see SymScale
      } else if (FAST) {
        // sign(y) == sign(p) always (e > 0); restoring it on the packed pair also
        // turns the +0 that the remainder step gives for c = -0 back into -0.
        ow[j] = pack_bf16x2(div_code_by_recip(c0, sc.e, sc.r), div_code_by_recip(c1, sc.e, sc.r)) |
                (pw & 0x80008000u);
      } else {
        ow[j] = pack_bf16x2(__fdiv_rn(c0, sc.e), __fdiv_rn(c1, sc.e));
      }
    }
    o = make_uint4(ow[0], ow[1], ow[2], ow[3]);
  } else if (!SYM && DT == QAT_BF16 && FAST && sc_packed(sc)) {
    float c0, c1;
    o = make_uint4(sc_pair(sc, v.x, &c0, &c1), sc_pair(sc, v.y, &c0, &c1), sc_pair(sc, v.z, &c0, &c1),
                   sc_pair(sc, v.w, &c0, &c1));
  } else {
    constexpr int N = Num<DT>::kPerVec;
    float yv[N], q;
#pragma unroll
    for (int i = 0; i < N; ++i) yv[i] = sc.template apply<FAST>(vec_get<DT>(v, i), &q);
    if (Num<DT>::kOutBytes == 4) {
#pragma unroll
      for (int k = 0; k < N / 4; ++k)
        oo[k % (Num<DT>::kOutBytes / Num<DT>::kBytes)] =
            make_uint4(__float_as_uint(yv[4 * k]), __float_as_uint(yv[4 * k + 1]), __float_as_uint(yv[4 * k + 2]),
                       __float_as_uint(yv[4 * k + 3]));
      return;
    } else {
      o = make_uint4(pack_bf16x2(yv[0], yv[1]), pack_bf16x2(yv[2 % N], yv[3 % N]),
                     pack_bf16x2(yv[4 % N], yv[5 % N]), pack_bf16x2(yv[6 % N], yv[7 % N]));
    }
  }
  oo[0] = o;
}

// int8 codes (+ optional packed mask) for one vector: the GEMM feed.  Only the
// code is needed, so Sym does no division at all.
template <int DT, bool SYM, bool FAST, typename Scale>
__device__ __forceinline__ void quant_vec_feed(const FwdParams& p, const Scale& sc, const uint4& v,
                                               uint8_t* codes_row, uint8_t* mask_row, uint32_t j,
                                               bool valid) {
  constexpr int N = Num<DT>::kPerVec;
  float qv[N];
  if constexpr (SYM && DT == QAT_BF16) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {   // p = fl_bf16(x*s); pack_codes4 rounds it half-to-even
      const uint32_t pw = mul_bf16x2(w[k], sc.s2);
      qv[(2 * k) % N] = bf16lo(pw);
      qv[(2 * k + 1) % N] = bf16hi(pw);
    }
  } else if constexpr (SYM) {
#pragma unroll
    for (int i = 0; i < N; ++i) qv[i] = Num<DT>::fl(__fmul_rn(vec_get<DT>(v, i), sc.s));
  } else if (DT == QAT_BF16 && FAST && sc_packed(sc)) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) (void)sc_pair(sc, w[k], &qv[(2 * k) % N], &qv[(2 * k + 1) % N]);
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) (void)sc.template apply<FAST>(vec_get<DT>(v, i), &qv[i]);
  }
  uint32_t cw[N / 4];
#pragma unroll
  for (int i = 0; i < N / 4; ++i)
    cw[i] = pack_codes4<SYM, DT == QAT_BF16>(qv[4 * i], qv[4 * i + 1], qv[4 * i + 2], qv[4 * i + 3]);
  if (valid) {
    if (N == 4)
      *reinterpret_cast<uint32_t*>(codes_row + (size_t)j * N) = cw[0];
    else
      *reinterpret_cast<uint2*>(codes_row + (size_t)j * N) = make_uint2(cw[0], cw[(N / 4) - 1]);
  }
  if (mask_row != nullptr) {
    uint32_t pass = 0;
    if (p.lo == -p.hi) {   // the model's clip is always [-c, c]: one compare on |x| (NaN passes, inf is masked)
#pragma unroll
      for (int i = 0; i < N; ++i) pass |= ((fabsf(vec_get<DT>(v, i)) >= p.hi) ? 0u : 1u) << i;
    } else {
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const float xf = vec_get<DT>(v, i);
        pass |= ((xf >= p.hi || xf <= p.lo) ? 0u : 1u) << i;  // utils_quant.py:85-86
      }
    }
    if (N == 8) {
      if (valid) mask_row[j] = (uint8_t)pass;
    } else {
      const uint32_t mine = valid ? pass : 0u;
      const uint32_t other = __shfl_xor_sync(kFull, mine, 1);
      if (valid && !(threadIdx.x & 1)) mask_row[j >> 1] = (uint8_t)(mine | (other << 4));
    }
  }
}

template <int DT, int ITERS, bool SYM, int OUT>
__global__ void __launch_bounds__(1024) rowquant_vec_kernel(const FwdParams p) {
  __shared__ uint32_t sm_u[32];
  __shared__ float sm_mx[32], sm_mn[32];

  const uint32_t lg = (uint32_t)p.log2_group;
  const uint32_t group = 1u << lg;
  const uint32_t t = threadIdx.x & (group - 1u);
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> lg) + (threadIdx.x >> lg);
  const bool row_ok = row < p.rows;
  const uint32_t nvec = row_ok ? (uint32_t)p.nvec : 0u;  // fused rows hold <= 8192 vectors
  const uint4* xrow = reinterpret_cast<const uint4*>(p.x) + row * p.nvec;
  // keep the 64-bit row base in registers: without this the compiler re-derives
  // row * nvec under every load's predicate (5 extra instructions per vector)
  asm volatile("" : "+l"(xrow));
  pdl_wait();               // the previous grid's results are visible from here on
  pdl_launch_dependents();  // the next kernel's CTAs may queue up behind this grid's

  uint4 v[ITERS];
#pragma unroll
  for (int i = 0; i < ITERS; ++i) {
    const uint32_t j = t + (uint32_t)i * group;
    v[i] = (j < nvec) ? ldg_stream(xrow + j) : make_uint4(0u, 0u, 0u, 0u);
  }
  RowStat st = stat_identity();
#pragma unroll
  for (int i = 0; i < ITERS; ++i) {
    const uint32_t j = t + (uint32_t)i * group;
    if (SYM || j < nvec) accumulate_vec<DT, SYM>(st, v[i]);  // zero vectors are neutral for max|x|
  }
  finalize_thread_stat<DT, SYM, true>(st);
  group_reduce<SYM>(st, (int)group, sm_u, sm_mx, sm_mn);
  using SO = ScaleOf<DT, SYM>;
  const typename SO::type sc = warp_derive_scale<DT, SYM>(st, p.qmax);
  if (t == 0 && row_ok) {
    if (p.st0 != nullptr) p.st0[row] = SO::st0(sc);
    if (p.st1 != nullptr) {
      float st1 = SO::st1(sc);
      if (SYM && OUT == OUT_FEED && p.poison_inf && st.amax_bits == 0x7f800000u) st1 = __int_as_float(0x7fc00000);
      p.st1[row] = st1;
    }
  }

  if constexpr (OUT == OUT_Y) {
    constexpr int OV = Num<DT>::kOutBytes / Num<DT>::kBytes;  // output vectors per input vector
    uint4* yrow = reinterpret_cast<uint4*>(p.y) + row * p.nvec * OV;
    asm volatile("" : "+l"(yrow));
    if constexpr (OV == 1) {
      if (sc.fast) {  // row-uniform => warp-uniform: a warp never spans two rows
#pragma unroll
        for (int i = 0; i < ITERS; ++i) {
          const uint32_t j = t + (uint32_t)i * group;
          uint4 o[1];
          quant_vec_y<DT, SYM, true>(sc, v[i], o);
          if (j < nvec) stg_stream(yrow + j, o[0]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < ITERS; ++i) {
          const uint32_t j = t + (uint32_t)i * group;
          uint4 o[1];
          quant_vec_y<DT, SYM, false>(sc, v[i], o);
          if (j < nvec) stg_stream(yrow + j, o[0]);
        }
      }
    } else {
      // y elements are twice as wide as x elements: a lane holds 32 consecutive output bytes.
      // Storing them as two 16-byte pieces per lane would make every store instruction write
      // HALF of each 32-byte sector (measured: the L2 then handles twice the write transactions
      // and the kernel ran at 0.71 of the HBM peak).  The warp's 64 pieces go through a
      // bank-conflict-free swizzled shared-memory exchange instead, so that each store
      // instruction writes 512 contiguous bytes.
      __shared__ uint4 stage[2048];                        // 64 pieces per warp, up to 32 warps
      uint4* ws = stage + (threadIdx.x >> 5) * 64;
      const uint32_t lane = threadIdx.x & 31u;
      const uint32_t w0 = 2u * lane, w1 = 2u * lane + 1u;  // pieces this lane produces
      const uint32_t r0 = lane, r1 = 32u + lane;           // pieces this lane stores
      auto sw = [](uint32_t c) { return c ^ ((c >> 3) & 1u); };
#pragma unroll
      for (int i = 0; i < ITERS; ++i) {
        const uint32_t j = t + (uint32_t)i * group;
        const uint32_t jw = j - lane;                      // the warp's first vector of this step
        uint4 o[OV];
        if (sc.fast)
          quant_vec_y<DT, SYM, true>(sc, v[i], o);
        else
          quant_vec_y<DT, SYM, false>(sc, v[i], o);
        ws[sw(w0)] = o[0];
        ws[sw(w1)] = o[1];
        __syncwarp();
        const uint4 a = ws[sw(r0)], b = ws[sw(r1)];
        __syncwarp();
        if (jw + (r0 >> 1) < nvec) stg_stream(yrow + (size_t)jw * OV + r0, a);
        if (jw + (r1 >> 1) < nvec) stg_stream(yrow + (size_t)jw * OV + r1, b);
      }
    }
  } else if constexpr (OUT == OUT_FEED) {
    uint8_t* codes_row = reinterpret_cast<uint8_t*>(p.codes) + row * p.cols;
    uint8_t* mask_row = p.mask != nullptr ? p.mask + ((row * p.cols) >> 3) : nullptr;
    if (sc.fast) {
#pragma unroll
      for (int i = 0; i < ITERS; ++i) {
        const uint32_t j = t + (uint32_t)i * group;
        quant_vec_feed<DT, SYM, true>(p, sc, v[i], codes_row, mask_row, j, j < nvec);
      }
    } else {
#pragma unroll
      for (int i = 0; i < ITERS; ++i) {
        const uint32_t j = t + (uint32_t)i * group;
        quant_vec_feed<DT, SYM, false>(p, sc, v[i], codes_row, mask_row, j, j < nvec);
      }
    }
  } else {
    const int64_t row_e0 = row * p.cols;
    if (sc.fast) {
#pragma unroll
      for (int i = 0; i < ITERS; ++i) {
        const uint32_t j = t + (uint32_t)i * group;
        emit_vec<DT, SYM, true>(p, sc, v[i], row_e0 + (int64_t)j * Num<DT>::kPerVec, j < nvec);
      }
    } else {
#pragma unroll
      for (int i = 0; i < ITERS; ++i) {
        const uint32_t j = t + (uint32_t)i * group;
        emit_vec<DT, SYM, false>(p, sc, v[i], row_e0 + (int64_t)j * Num<DT>::kPerVec, j < nvec);
      }
    }
  }
}

// scalar path (misaligned pointers or row pitch not a multiple of 16 bytes):
// same structure, one element per thread-iteration, every output optional.
template <int DT, int ITERS, bool SYM>
__global__ void __launch_bounds__(1024) rowquant_scalar_kernel(const FwdParams p) {
  __shared__ uint32_t sm_u[32];
  __shared__ float sm_mx[32], sm_mn[32];

  const int group = p.group;
  const int t = threadIdx.x & (group - 1);
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x / group) + (threadIdx.x / group);
  const bool row_ok = row < p.rows;
  const int64_t row_e0 = row * p.cols;
  RowStat st = stat_identity();
  using SO = ScaleOf<DT, SYM>;
  float v[ITERS];
#pragma unroll
  for (int i = 0; i < ITERS; ++i) {
    const int64_t j = t + (int64_t)i * group;
    v[i] = (row_ok && j < p.nvec) ? load_scalar<DT>(p.x, row_e0 + j) : 0.f;
  }
#pragma unroll
  for (int i = 0; i < ITERS; ++i) {
    const int64_t j = t + (int64_t)i * group;
    if (row_ok && j < p.nvec) accumulate_scalar<DT, SYM>(st, v[i]);
  }
  group_reduce<SYM>(st, group, sm_u, sm_mx, sm_mn);
  const typename SO::type sc = SO::make(st, p.qmax);
  if (t == 0 && row_ok) {
    if (p.st0 != nullptr) p.st0[row] = SO::st0(sc);
    if (p.st1 != nullptr) p.st1[row] = SO::st1(sc);
  }
#pragma unroll
  for (int i = 0; i < ITERS; ++i) {
    const int64_t j = t + (int64_t)i * group;
    if (row_ok && j < p.nvec) {
      if (sc.fast)
        emit_scalar<DT, SYM, true>(p, sc, v[i], row_e0 + j);
      else
        emit_scalar<DT, SYM, false>(p, sc, v[i], row_e0 + j);
    }
  }
}

// =============================================================================
// K5: rows too long for one CTA's registers (layerwise mode: the whole tensor
// is one row).  Phase 1 reduces chunks and merges with atomics on an ordered
// key; phase 2 re-reads (L2-resident up to ~100 MB) and applies.
//   ws[4*row + 0] = Sym |x| max bits / Asym ordered-key max
//   ws[4*row + 1] = Asym ordered-key min     ws[4*row + 2] = Asym NaN flag
// =============================================================================
__global__ void ws_init_kernel(uint32_t* ws, int64_t rows) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < rows) {
    ws[4 * r + 0] = 0u;
    ws[4 * r + 1] = 0xffffffffu;
    ws[4 * r + 2] = 0u;
    ws[4 * r + 3] = 0u;
  }
}

template <int DT, bool SYM, bool VEC>
__global__ void __launch_bounds__(256) longrow_stats_kernel(const FwdParams p) {
  __shared__ uint32_t sm_u[32];
  __shared__ float sm_mx[32], sm_mn[32];
  const int64_t row = blockIdx.y;
  const int64_t row_e0 = row * p.cols;
  const int64_t j0 = (int64_t)blockIdx.x * p.chunk;
  const int64_t j1 = min(j0 + p.chunk, p.nvec);
  RowStat st = stat_identity();
  if (VEC) {
    const char* xrow = reinterpret_cast<const char*>(p.x) + row_e0 * Num<DT>::kBytes;
    int64_t j = j0 + threadIdx.x;
    for (; j + 3 * 256 < j1; j += 4 * 256) {
      uint4 a = ldg_stream(xrow + j * 16);
      uint4 b = ldg_stream(xrow + (j + 256) * 16);
      uint4 c = ldg_stream(xrow + (j + 512) * 16);
      uint4 d = ldg_stream(xrow + (j + 768) * 16);
      accumulate_vec<DT, SYM>(st, a);
      accumulate_vec<DT, SYM>(st, b);
      accumulate_vec<DT, SYM>(st, c);
      accumulate_vec<DT, SYM>(st, d);
    }
    for (; j < j1; j += 256) {
      uint4 a = ldg_stream(xrow + j * 16);
      accumulate_vec<DT, SYM>(st, a);
    }
  } else {
    for (int64_t j = j0 + threadIdx.x; j < j1; j += 256)
      accumulate_scalar<DT, SYM>(st, load_scalar<DT>(p.x, row_e0 + j));
  }
  finalize_thread_stat<DT, SYM, VEC>(st);
  group_reduce<SYM>(st, 256, sm_u, sm_mx, sm_mn);
  if (threadIdx.x == 0) {
    uint32_t* w = p.ws + 4 * row;
    if (SYM) {
      atomicMax(w, st.amax_bits);
    } else {
      if (st.mx >= st.mn) {  // at least one non-NaN value seen
        atomicMax(w, ordered_key(st.mx));
        atomicMin(w + 1, ordered_key(st.mn));
      }
      if (st.nan) atomicOr(w + 2, 1u);
    }
  }
}

template <int DT, bool SYM, bool VEC>
__global__ void __launch_bounds__(256) longrow_apply_kernel(const FwdParams p) {
  const int64_t row = blockIdx.y;
  const int64_t row_e0 = row * p.cols;
  const int64_t j0 = (int64_t)blockIdx.x * p.chunk;
  const int64_t j1 = min(j0 + p.chunk, p.nvec);
  const uint32_t* w = p.ws + 4 * row;
  RowStat st;
  st.amax_bits = w[0];
  st.mx = SYM ? 0.f : ordered_unkey(w[0]);
  st.mn = SYM ? 0.f : ordered_unkey(w[1]);
  st.nan = w[2];
  using SO = ScaleOf<DT, SYM>;
  const typename SO::type sc = SO::make(st, p.qmax);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (p.st0 != nullptr) p.st0[row] = SO::st0(sc);
    if (p.st1 != nullptr) p.st1[row] = SO::st1(sc);
  }
  if (VEC) {
    const char* xrow = reinterpret_cast<const char*>(p.x) + row_e0 * Num<DT>::kBytes;
    // whole-CTA trip count so the mask shuffle inside emit_vec stays convergent
    for (int64_t jb = j0; jb < j1; jb += 256) {
      const int64_t j = jb + threadIdx.x;
      const bool valid = j < j1;
      uint4 v = valid ? ldg_stream(xrow + j * 16) : make_uint4(0u, 0u, 0u, 0u);
      if (sc.fast)
        emit_vec<DT, SYM, true>(p, sc, v, row_e0 + j * Num<DT>::kPerVec, valid);
      else
        emit_vec<DT, SYM, false>(p, sc, v, row_e0 + j * Num<DT>::kPerVec, valid);
    }
  } else {
    for (int64_t j = j0 + threadIdx.x; j < j1; j += 256) {
      if (sc.fast)
        emit_scalar<DT, SYM, true>(p, sc, load_scalar<DT>(p.x, row_e0 + j), row_e0 + j);
      else
        emit_scalar<DT, SYM, false>(p, sc, load_scalar<DT>(p.x, row_e0 + j), row_e0 + j);
    }
  }
}

// ---- host-side dispatch -----------------------------------------------------
constexpr int kMaxIters = 8;
constexpr int kMaxGroup = 1024;

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct Plan {
  bool vec;
  bool fused;  // row fits registers
  int64_t nvec;
  int group, iters, block;
  int64_t chunk, chunks;
};

Plan make_plan(const void* x, const void* y, int64_t rows, int64_t cols, int dtype) {
  Plan pl{};
  const int esz = dtype == QAT_F32 ? 4 : 2;
  const int per = 16 / esz;
  pl.vec = (cols % per == 0) && aligned16(x) && (y == nullptr || aligned16(y));
  pl.nvec = pl.vec ? cols / per : cols;
  // Threads per row (power of two >= 32) and vectors per thread (<= 8).  Per-thread
  // fixed work (reduction tree, scale broadcast, addressing) is ~200 instructions,
  // so prefer many vectors per thread; among candidates take the one with the
  // fewest idle vector slots, ties to the smaller group.
  int best_group = 0;
  int64_t best_iters = 0, best_slots = 0;
  for (int group = 32; group <= kMaxGroup; group <<= 1) {
    const int64_t iters = (pl.nvec + group - 1) / group;
    if (iters > kMaxIters) continue;
    const int64_t slots = iters * group;
    if (best_group == 0 || slots < best_slots) {
      best_group = group;
      best_iters = iters;
      best_slots = slots;
    }
  }
  pl.fused = best_group != 0;
  if (!pl.fused) {  // does not fit: the cap below only sizes the long-row path
    best_group = kMaxGroup;
    best_iters = kMaxIters;
  }
  pl.group = best_group;
  pl.iters = (int)best_iters;
  if (!pl.vec) pl.iters = best_iters <= 2 ? 2 : best_iters <= 4 ? 4 : 8;  // scalar kernels: 3 instantiations
  pl.block = best_group < 256 ? 256 : best_group;
  if (!pl.fused) {
    int64_t chunk = (pl.nvec + 4095) / 4096;
    if (chunk < 2048) chunk = 2048;
    chunk = (chunk + 255) / 256 * 256;  // multiple of the CTA width (keeps lane parity for the mask)
    pl.chunk = chunk;
    pl.chunks = (pl.nvec + chunk - 1) / chunk;
  }
  return pl;
}

template <int DT, bool SYM, int ITERS>
void launch_vec_iters(const FwdParams& p, const Plan& pl, unsigned grid, int out, cudaStream_t st) {
  if (out == OUT_Y)
    (void)launch_pdl(rowquant_vec_kernel<DT, ITERS, SYM, OUT_Y>, dim3(grid), dim3(pl.block), 0, st, p);
  else if (out == OUT_FEED)
    (void)launch_pdl(rowquant_vec_kernel<DT, ITERS, SYM, OUT_FEED>, dim3(grid), dim3(pl.block), 0, st, p);
  else
    (void)launch_pdl(rowquant_vec_kernel<DT, ITERS, SYM, OUT_ANY>, dim3(grid), dim3(pl.block), 0, st, p);
}

template <int DT, bool SYM, bool VEC>
int launch_fused(const FwdParams& p, const Plan& pl, cudaStream_t st) {
  const int rows_per_cta = pl.block / pl.group;
  const int64_t grid64 = (p.rows + rows_per_cta - 1) / rows_per_cta;
  if (grid64 > 0x7fffffffLL) {
    set_error("too many rows (%lld)", (long long)p.rows);
    return QAT_ERR_UNSUPPORTED;
  }
  const unsigned grid = (unsigned)grid64;
  if (VEC) {
    int out = OUT_ANY;
    if (p.y != nullptr && p.codes == nullptr && p.mask == nullptr) out = OUT_Y;
    if (p.y == nullptr && p.codes != nullptr && p.codes_kind == QAT_CODES_I8) out = OUT_FEED;
    switch (pl.iters) {
      case 1: launch_vec_iters<DT, SYM, 1>(p, pl, grid, out, st); break;
      case 2: launch_vec_iters<DT, SYM, 2>(p, pl, grid, out, st); break;
      case 3: launch_vec_iters<DT, SYM, 3>(p, pl, grid, out, st); break;
      case 4: launch_vec_iters<DT, SYM, 4>(p, pl, grid, out, st); break;
      case 5: launch_vec_iters<DT, SYM, 5>(p, pl, grid, out, st); break;
      case 6: launch_vec_iters<DT, SYM, 6>(p, pl, grid, out, st); break;
      case 7: launch_vec_iters<DT, SYM, 7>(p, pl, grid, out, st); break;
      default: launch_vec_iters<DT, SYM, 8>(p, pl, grid, out, st); break;
    }
    QAT_CHECK_LAUNCH("rowquant_vec_kernel");
  } else {
    switch (pl.iters) {
      case 2: rowquant_scalar_kernel<DT, 2, SYM><<<grid, pl.block, 0, st>>>(p); break;
      case 4: rowquant_scalar_kernel<DT, 4, SYM><<<grid, pl.block, 0, st>>>(p); break;
      default: rowquant_scalar_kernel<DT, 8, SYM><<<grid, pl.block, 0, st>>>(p); break;
    }
    QAT_CHECK_LAUNCH("rowquant_scalar_kernel");
  }
  return QAT_OK;
}

template <int DT, bool SYM, bool VEC>
int launch_longrow(const FwdParams& p, const Plan& pl, cudaStream_t st) {
  if (p.rows > 65535) {
    set_error("long-row path supports at most 65535 rows (got %lld)", (long long)p.rows);
    return QAT_ERR_UNSUPPORTED;
  }
  ws_init_kernel<<<(unsigned)((p.rows + 255) / 256), 256, 0, st>>>(p.ws, p.rows);
  QAT_CHECK_LAUNCH("ws_init_kernel");
  dim3 grid((unsigned)pl.chunks, (unsigned)p.rows);
  longrow_stats_kernel<DT, SYM, VEC><<<grid, 256, 0, st>>>(p);
  QAT_CHECK_LAUNCH("longrow_stats_kernel");
  longrow_apply_kernel<DT, SYM, VEC><<<grid, 256, 0, st>>>(p);
  QAT_CHECK_LAUNCH("longrow_apply_kernel");
  return QAT_OK;
}

template <int DT, bool SYM>
int dispatch(const FwdParams& p, const Plan& pl, cudaStream_t st) {
  if (pl.fused)
    return pl.vec ? launch_fused<DT, SYM, true>(p, pl, st) : launch_fused<DT, SYM, false>(p, pl, st);
  return pl.vec ? launch_longrow<DT, SYM, true>(p, pl, st) : launch_longrow<DT, SYM, false>(p, pl, st);
}

float round_to_dtype(float v, int dtype) {
  if (dtype == QAT_F32) return v;
  return __bfloat162float(__float2bfloat16_rn(v));
}

// AsymQuantizer's `.div(S)`: 0 = true division (torch CPU), 1 = multiply by fl(1/S) (ATen CUDA).
// -1: read QAT_B200_ASYM_DIV ("cuda" selects 1) on first use.
int g_asym_div = -1;
int asym_div_mode() {
  if (g_asym_div < 0) {
    const char* v = getenv("QAT_B200_ASYM_DIV");
    g_asym_div = (v != nullptr && (v[0] == 'c' || v[0] == 'C') && (v[1] == 'u' || v[1] == 'U')) ? 1 : 0;
  }
  return g_asym_div;
}

template <bool SYM>
int fwd_entry(const void* x, void* y, void* codes, int codes_kind, float* st0, float* st1,
              uint8_t* mask, float lo, float hi, int64_t rows, int64_t cols, int dtype, int bits,
              void* workspace, size_t workspace_bytes, void* stream, int poison_inf = 0) {
  QAT_CHECK_ARG(dtype == QAT_F32 || dtype == QAT_BF16 || (SYM && (dtype == QAT_BF16_AMP || dtype == QAT_BF16_AMP_CAST)),
                "dtype must be QAT_F32, QAT_BF16 or (Sym only) QAT_BF16_AMP / QAT_BF16_AMP_CAST (got %d)", dtype);
  QAT_CHECK_ARG(rows >= 0 && cols >= 0, "negative shape [%lld, %lld]", (long long)rows, (long long)cols);
  QAT_CHECK_ARG(SYM ? (bits >= 2 && bits <= 31) : (bits >= 1 && bits <= 31), "unsupported num_bits %d", bits);
  QAT_CHECK_ARG(!(codes != nullptr && codes_kind == QAT_CODES_I16 && bits > (SYM ? 16 : 15)),
                "int16 codes need num_bits <= %d (got %d)", SYM ? 16 : 15, bits);
  if (rows == 0 || cols == 0) return QAT_OK;
  QAT_CHECK_ARG(x != nullptr, "x is NULL");
  QAT_CHECK_ARG(y != nullptr || codes != nullptr || st0 != nullptr || st1 != nullptr || mask != nullptr,
                "no output requested");
  QAT_CHECK_ARG(codes == nullptr || codes_kind == QAT_CODES_I8 || codes_kind == QAT_CODES_I16,
                "codes_kind must be QAT_CODES_I8 or QAT_CODES_I16 when codes != NULL");
  QAT_CHECK_ARG(!(codes != nullptr && codes_kind == QAT_CODES_I8 && bits > 8),
                "int8 codes need num_bits <= 8 (got %d)", bits);
  QAT_CHECK_ARG(x != y, "y must not alias x");

  Plan pl = make_plan(x, y, rows, cols, dtype);
  if (codes != nullptr && pl.vec) {
    // code stores are vectorised with the same element grouping
    const int per = dtype == QAT_F32 ? 4 : 8;
    const uintptr_t need = (uintptr_t)(codes_kind == QAT_CODES_I8 ? per : 2 * per);
    QAT_CHECK_ARG((reinterpret_cast<uintptr_t>(codes) & (need - 1)) == 0, "codes pointer misaligned");
  }
  if (mask != nullptr) {
    if (!pl.vec || (cols % 8 != 0 && rows != 1)) {
      set_error("packed-mask output needs 16-byte aligned rows with cols %% 8 == 0 (cols=%lld)",
                (long long)cols);
      return QAT_ERR_UNSUPPORTED;
    }
    if (dtype == QAT_F32 && (cols % 8 != 0)) {
      set_error("packed-mask output needs cols %% 8 == 0 for fp32 (cols=%lld)", (long long)cols);
      return QAT_ERR_UNSUPPORTED;
    }
  }
  FwdParams p{};
  p.x = x;
  p.y = y;
  p.codes = codes;
  p.codes_kind = codes_kind;
  p.st0 = st0;
  p.st1 = st1;
  p.mask = mask;
  p.lo = round_to_dtype(lo, dtype);
  p.hi = round_to_dtype(hi, dtype);
  p.rows = rows;
  p.cols = cols;
  p.nvec = pl.nvec;
  // the reference's Python int, converted to the fp32 op scalar (round to nearest)
  p.qmax = SYM ? (float)((1ll << (bits - 1)) - 1) : (float)((1ll << bits) - 1);
  if (!SYM && asym_div_mode() == 1) p.qmax = -p.qmax;   // see ScaleOf<DT, false>::make
  p.group = pl.group;
  p.log2_group = 0;
  while ((1 << p.log2_group) < pl.group) ++p.log2_group;
  p.ws = reinterpret_cast<uint32_t*>(workspace);
  p.chunk = pl.chunk;
  p.poison_inf = poison_inf;
  if (!pl.fused) {
    const size_t need = (size_t)rows * 16;
    if (workspace == nullptr || workspace_bytes < need) {
      set_error("row length %lld needs %zu bytes of workspace (got %zu)", (long long)cols, need,
                workspace_bytes);
      return QAT_ERR_WORKSPACE;
    }
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == QAT_F32) return dispatch<QAT_F32, SYM>(p, pl, st);
  if constexpr (SYM) {
    if (dtype == QAT_BF16_AMP) return dispatch<QAT_BF16_AMP, true>(p, pl, st);
    if (dtype == QAT_BF16_AMP_CAST) return dispatch<QAT_BF16_AMP_CAST, true>(p, pl, st);
  }
  return dispatch<QAT_BF16, SYM>(p, pl, st);
}

}  // namespace

int sym_fwd_feed(const void* x, void* codes, float* row_e, uint8_t* mask, float clip_lo, float clip_hi,
                 int64_t rows, int64_t cols, int dtype, int bits, void* stream) {
  // the feed's codes do not depend on the final cast: QAT_BF16_AMP names the autocast chain here
  QAT_CHECK_ARG(dtype != QAT_BF16_AMP_CAST, "QAT_BF16_AMP_CAST is a qat_sym_fwd output mode");
  return fwd_entry<true>(x, nullptr, codes, QAT_CODES_I8, nullptr, row_e, mask, clip_lo, clip_hi, rows, cols,
                         dtype, bits, nullptr, 0, stream, /*poison_inf=*/1);
}
}  // namespace qat

extern "C" {

size_t qat_fwd_workspace_bytes(int64_t rows, int64_t cols, int dtype) {
  if (rows <= 0 || cols <= 0) return 0;
  // worst case (scalar path): one element per thread-iteration
  (void)dtype;
  // the scalar path may be chosen at run time when a pointer is misaligned, so
  // size for it: fused iff cols <= kMaxGroup * kMaxIters elements.
  if (cols <= (int64_t)qat::kMaxGroup * qat::kMaxIters) return 0;
  return (size_t)rows * 16;
}

int qat_sym_fwd(const void* x, void* y, void* codes, int codes_kind, float* row_s, float* row_e,
                uint8_t* mask, float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                int bits, void* workspace, size_t workspace_bytes, void* stream) {
  return qat::fwd_entry<true>(x, y, codes, codes_kind, row_s, row_e, mask, clip_lo, clip_hi, rows,
                              cols, dtype, bits, workspace, workspace_bytes, stream);
}

int qat_asym_fwd(const void* x, void* y, void* codes, int codes_kind, float* row_a, float* row_b,
                 uint8_t* mask, float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                 int bits, void* workspace, size_t workspace_bytes, void* stream) {
  return qat::fwd_entry<false>(x, y, codes, codes_kind, row_a, row_b, mask, clip_lo, clip_hi, rows,
                               cols, dtype, bits, workspace, workspace_bytes, stream);
}

int qat_sym_feed(const void* x, int8_t* codes, float* row_e, uint8_t* mask, float clip_lo, float clip_hi,
                 int64_t rows, int64_t cols, int dtype, int bits, void* stream) {
  QAT_CHECK_ARG(codes != nullptr && row_e != nullptr, "codes / row_e must be provided");
  QAT_CHECK_ARG(bits >= 2 && bits <= 8, "int8 codes need 2 <= bits <= 8 (got %d)", bits);
  return qat::sym_fwd_feed(x, codes, row_e, mask, clip_lo, clip_hi, rows, cols, dtype, bits, stream);
}

int qat_set_asym_div(int mode) {
  QAT_CHECK_ARG(mode == QAT_ASYM_DIV_TRUE || mode == QAT_ASYM_DIV_RECIP, "mode must be QAT_ASYM_DIV_TRUE or QAT_ASYM_DIV_RECIP");
  qat::g_asym_div = mode;
  return QAT_OK;
}

}  // extern "C"
