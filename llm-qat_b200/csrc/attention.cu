// attention.cu — fused causal attention, forward and backward, on tcgen05 (kind::f16, bf16 in,
// fp32 accumulation in TMEM).  SURVEY.md section 8(f)-4.
//
// Replaces the eager block of /root/reference/models/modeling_llama_quant.py:352-377:
//     attn_weights = Q K^T / sqrt(d);  + attention_mask;  max(., finfo.min);
//     softmax(dim=-1, dtype=float32).to(bf16);  attn_output = attn_weights V
// (6 kernels, a materialised [b, 32, s, s] score tensor in bf16 and fp32) and autograd's
// backward of it, for the causal mask the model builds (:60-92).  K and V arrive already
// fake-quantized (per token, :320-327) and rotated; this kernel consumes them as they are.
//
// Layout: Q, K, V, O, dO, dQ, dK, dV are bf16 [B, S, H, D] (the projections' own layout:
// [b, s, hidden] viewed as heads — no transposes), D == 128.  LSE and delta are fp32 [B, H, S].
//
// Forward, one CTA per (128-query tile, head, batch), 384 threads:
//   warp 0 / 11 TMA producers: Q once and the K tiles / the V tiles (128 keys, 2-stage rings each)
//   warp 1   MMA issuer:   S[b] = Q K_j^T  (M128 N128 K128, both K-major), up to two tiles ahead
//   warp 10  MMA issuer:   O[b] += P_j V_j (A = P from shared memory, B = V MN-major),  b = j % 2
//   warps 2-5, 6-9         two softmax warpgroups, tile parity b each: one thread per query row (a TMEM
//                          lane): tcgen05.ld S, running max / sum in registers (no shuffles), P -> bf16 ->
//                          128B-swizzled shared memory, lazy rescale of O[b] in TMEM (only when the row max
//                          grew by > 2^8); the two partial soft-maxes are merged in the epilogue.
//   TMEM: S0 | S1 | O0 | O1 = 512 columns.
// Backward: attn_delta (rowsum(dO * O)), then two kernels without atomics —
//   attn_bwd_dq   (query-stationary, 64-key steps):  S, dP -> dS -> dQ += dS K
//   attn_bwd_dkv  (key-stationary, 64-query steps):  S^T, dP^T -> P^T, dS^T -> dV += P^T dO, dK += dS^T Q
// each recomputing P from the saved LSE (7 GEMMs of 128x128x64-ish tiles instead of the
// minimal 5; deterministic, and every accumulator fits TMEM double-buffered).
// 4 S^2 D H B / 2 flops forward (causal), x3.5 backward; measured limits (tests/gpu_attn_trace.py): the exponentials
// (MUFU, 16 ex2 per clock) in the forward, shared-memory operand bandwidth of the N = 64 MMAs in the backward.
#define QAT_PDL_FAMILY 6   // bit of QAT_B200_PDL_MASK (common.cuh)
#include <cmath>

#include "umma.cuh"

namespace qat {
namespace {
using namespace umma;

constexpr int D = 128;            // head dim
constexpr int BM = 128;           // rows per CTA tile (TMEM lanes)
constexpr float kLog2e = 1.4426950408889634f;

// ---- shared helpers -------------------------------------------------------------------------
// K-major operand [rows][128 d] staged as two 64-element (128 B) chunks, `chunk_stride` apart.
// k-step j (16 elements) lives in chunk j/4 at byte (j%4)*32.
__device__ __forceinline__ uint64_t desc_k_step(uint32_t base, uint32_t chunk_stride, int j) {
  return make_smem_desc(base + (uint32_t)(j >> 2) * chunk_stride + (uint32_t)(j & 3) * 32u);
}
// MN-major operand: [k rows][N] staged as 64-element chunks of N, `lbo` apart; k-step j = rows 16j..16j+15
__device__ __forceinline__ uint64_t desc_mn_step(uint32_t base, uint32_t lbo, int j) {
  return make_smem_desc_mn(base + (uint32_t)j * 2048u, lbo, 1024u);
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// byte offset of 16-byte unit `u` (0..7) of row `r` inside a 128B-swizzled [rows][128 B] chunk
__device__ __forceinline__ uint32_t swz(uint32_t r, uint32_t u) { return r * 128u + ((u ^ (r & 7u)) << 4); }
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int n) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int n) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory");
}

// Debug hook (tests/gpu_attn_trace.py): when set, CTA (0,0,0) of attn_fwd_kernel records clock64() at its
// phase boundaries — slots [role][tile][event] of a device buffer — so the per-tile critical path can be
// read off instead of guessed.  NULL in normal operation (one predictable branch per event).
long long* g_attn_trace = nullptr;
constexpr int kTraceTiles = 16, kTraceEvents = 8;

struct AttnParams {
  long long* trace;
  void* o;             // fwd: O [B,S,H,D] bf16
  float* lse;          // [B,H,S] natural-log LSE of the scaled scores
  const float* delta;  // bwd: rowsum(dO * O) [B,H,S]
  void* dq;            // bwd outputs, bf16 [B,S,H,D]
  void* dk;
  void* dv;
  int B, S, H;
  float scale;         // 1 / sqrt(D)
  int causal;
};

// =============================================================================================
// forward
// =============================================================================================
// Two softmax warpgroups per CTA, each with its OWN running (max, sum), S buffer, P buffer and O
// accumulator: warpgroup b takes the key tiles j with j % 2 == b, so its soft-max of tile j runs
// while the tensor core does Q K_{j+1}^T and P_{j-1} V_{j-1} of the other warpgroup, and the two
// partial results are merged once at the end (split-KV inside the CTA).  One thread per query
// row: row max / sum never leave registers.
namespace fwd {
constexpr int kThreads = 384;                       // warp 0 TMA (Q, K), warp 1 QK^T issuer, warps 2-5 WG0, warps 6-9 WG1,
                                                    // warp 10 PV issuer, warp 11 TMA (V)
constexpr uint32_t kTile = BM * D * 2;              // 32 KB: [128][128] bf16 as 2 chunks of 16 KB
constexpr uint32_t kChunk = BM * 128;               // 16 KB
constexpr uint32_t oQ = 0, oK = kTile, oV = 3 * kTile, oP = 5 * kTile, oBar = 7 * kTile;
enum { bQ = 0, bKfull = 1, bKempty = 3, bVfull = 5, bVempty = 7, bSfull = 9, bSfree = 11, bPfull = 13, bPVdone = 15,
       nBars = 17 };
constexpr uint32_t oTmem = oBar + 8 * nBars;
constexpr uint32_t kSmem = oTmem + 16 + 1024;
static_assert(kSmem <= 232448, "smem");
// TMEM columns: S0 [0,128) S1 [128,256) O0 [256,384) O1 [384,512)
}  // namespace fwd

__global__ void __launch_bounds__(fwd::kThreads, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                const __grid_constant__ CUtensorMap map_v, const AttnParams p) {
  using namespace fwd;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q_tile = (int)gridDim.x - 1 - (int)blockIdx.x;   // heaviest (most key tiles) first
  const int h = blockIdx.y, b = blockIdx.z;
  const int q0 = q_tile * BM;
  const int n_kv = p.causal ? min((q0 + BM + BM - 1) / BM, (p.S + BM - 1) / BM) : (p.S + BM - 1) / BM;
  auto bar = [&](int i) { return base + oBar + 8u * (uint32_t)i; };
  const bool tracing = p.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
  // role 0 = MMA thread, 1 = warpgroup 0 (thread 64), 2 = warpgroup 1 (thread 192)
  auto trace = [&](int role, int tile, int ev) {
    if (tracing && tile < kTraceTiles) p.trace[(role * kTraceTiles + tile) * kTraceEvents + ev] = clock64();
  };

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&map_q);
    prefetch_tensormap(&map_k);
    prefetch_tensormap(&map_v);
    mbar_init(bar(bQ), 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar(bKfull + s), 1);
      mbar_init(bar(bKempty + s), 1);
      mbar_init(bar(bVfull + s), 1);
      mbar_init(bar(bVempty + s), 1);
      mbar_init(bar(bSfull + s), 1);
      mbar_init(bar(bSfree + s), 128);
      mbar_init(bar(bPfull + s), 128);
      mbar_init(bar(bPVdone + s), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc_cg1<512>(base + oTmem);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(base_ptr + oTmem);
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    if (lane == 0) {
      const int32_t col = h * D;
      mbar_expect_tx(bar(bQ), kTile);
      tma_load_3d(base + oQ, &map_q, bar(bQ), col, q0, b);
      tma_load_3d(base + oQ + kChunk, &map_q, bar(bQ), col + 64, q0, b);
      // K and V have their own producer threads (this one and warp 11): K_j is wanted two tiles ahead of V_j
      // (Q K^T is issued two tiles early, P V only after the soft-max) and its stage frees as soon as
      // Q K_{j-2}^T retires, whereas V's stage frees only after P V of tile j-2.  One in-order producer made
      // the K loads queue behind V stages still in use: 1300-2600 cycles of exposed TMA latency per tile
      // (tests/gpu_attn_trace.py).
      for (int j = 0; j < n_kv; ++j) {
        const int s = j & 1;
        mbar_wait(bar(bKempty + s), (uint32_t)((j >> 1) & 1) ^ 1u);
        mbar_expect_tx(bar(bKfull + s), kTile);
        tma_load_3d(base + oK + s * kTile, &map_k, bar(bKfull + s), col, j * BM, b);
        tma_load_3d(base + oK + s * kTile + kChunk, &map_k, bar(bKfull + s), col + 64, j * BM, b);
      }
    }
  } else if (warp == 11) {
    if (lane == 0) {
      const int32_t col = h * D;
      for (int j = 0; j < n_kv; ++j) {
        const int s = j & 1;
        mbar_wait(bar(bVempty + s), (uint32_t)((j >> 1) & 1) ^ 1u);
        mbar_expect_tx(bar(bVfull + s), kTile);
        tma_load_3d(base + oV + s * kTile, &map_v, bar(bVfull + s), col, j * BM, b);
        tma_load_3d(base + oV + s * kTile + kChunk, &map_v, bar(bVfull + s), col + 64, j * BM, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_qk = make_idesc_bf16(BM, BM, 0, 0);
      // tile j uses K/V stage, S buffer, P buffer and O accumulator (j & 1); its use count is j >> 1
      auto issue_qk = [&](int j) {
        const int s = j & 1;
        const uint32_t ph = (uint32_t)((j >> 1) & 1);
        trace(0, j, 0);
        mbar_wait(bar(bKfull + s), ph);
        trace(0, j, 1);
        mbar_wait(bar(bSfree + s), ph ^ 1u);     // the warpgroup drained this S buffer's previous use
        tcgen05_fence_after();
        trace(0, j, 2);
        const uint32_t d_s = tmem + (uint32_t)(s * BM);
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_f16<1>(d_s, desc_k_step(base + oQ, kChunk, k), desc_k_step(base + oK + s * kTile, kChunk, k),
                      idesc_qk, k > 0 ? 1u : 0u);
        umma_commit(bar(bKempty + s));
        umma_commit(bar(bSfull + s));
        trace(0, j, 3);
      };
      // Q K^T and P V are issued by two different threads (this one and warp 10): each blocks only on its
      // own barriers, so a late P_j never holds back Q K_{j+2}^T and a late K tile never holds back P V
      // (one issuer spent ~500 of every 2000 cycles per tile in barrier round trips: tests/gpu_attn_trace.py)
      mbar_wait(bar(bQ), 0);
      for (int j = 0; j < n_kv; ++j) issue_qk(j);
    }
  } else if (warp == 10) {
    if (lane == 0) {
      constexpr uint32_t idesc_pv = make_idesc_bf16(BM, D, 0, 1);
      for (int j = 0; j < n_kv; ++j) {
        const int s = j & 1;
        const uint32_t ph = (uint32_t)((j >> 1) & 1);
        trace(0, j, 4);
        mbar_wait(bar(bVfull + s), ph);
        trace(0, j, 5);
        mbar_wait(bar(bPfull + s), ph);
        tcgen05_fence_after();
        trace(0, j, 6);
        const uint32_t d_o = tmem + 2u * BM + (uint32_t)(s * D);
#pragma unroll
        for (int k = 0; k < BM / 16; ++k)
          umma_f16<1>(d_o, desc_k_step(base + oP + s * kTile, kChunk, k), desc_mn_step(base + oV + s * kTile, kChunk, k),
                      idesc_pv, (j > 1 || k > 0) ? 1u : 0u);
        umma_commit(bar(bVempty + s));
        umma_commit(bar(bPVdone + s));
        trace(0, j, 7);
      }
    }
  } else {
    // ===================== two softmax warpgroups: one thread per query row =====================
    const int wg = (warp - 2) >> 2;                 // 0 | 1: takes the key tiles j with (j & 1) == wg
    const int quad = warp & 3;                      // TMEM lane quadrant this warp may access
    const int r = quad * 32 + lane;                 // row inside the tile == TMEM lane
    const int q_idx = q0 + r;
    const uint32_t t_lane = tmem + ((uint32_t)(quad * 32) << 16);
    const uint32_t t_s = t_lane + (uint32_t)(wg * BM), t_o = t_lane + 2u * BM + (uint32_t)(wg * D);
    const uint32_t p_buf = base + oP + (uint32_t)wg * kTile;
    const float c = p.scale * kLog2e;
    float m_run = -INFINITY;   // running max of the raw scores (the one the exponent is taken against)
    float l_run = 0.f;
    int uses = 0;
    const bool tr = (threadIdx.x == 64 || threadIdx.x == 192);
    // exp token: warpgroup 0 goes first (warpgroup 1 hands it the token up front); the turns alternate strictly
    // — tile 0, 1, 2, ... — which is also the order the S tiles are produced in
    const bool pingpong = n_kv > 1;
    if (pingpong && wg == 1) named_bar_arrive(2, 256);
    for (int j = wg; j < n_kv; j += 2, ++uses) {
      const uint32_t ph = (uint32_t)(uses & 1);
      if (tr) trace(1 + wg, j, 0);
      mbar_wait(bar(bSfull + wg), ph);
      tcgen05_fence_after();
      if (tr) trace(1 + wg, j, 1);
      uint32_t sv[128];
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t(&dst)[32] = *reinterpret_cast<uint32_t(*)[32]>(&sv[ch * 32]);
        tmem_ld_32x32b_x32(t_s + (uint32_t)(ch * 32), dst);
      }
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(bar(bSfree + wg));
      if (tr) trace(1 + wg, j, 2);
      const int k0 = j * BM;
      const bool edge = (p.causal && k0 + BM - 1 > q0) || (k0 + BM > p.S);
      if (edge) {
#pragma unroll
        for (int i = 0; i < 128; ++i) {
          const int k_idx = k0 + i;
          const bool dead = k_idx >= p.S || (p.causal && k_idx > q_idx);
          if (dead) sv[i] = 0xff800000u;   // -inf
        }
      }
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};   // four chains: 32 dependent max ops, not 128
#pragma unroll
      for (int i = 0; i < 128; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(sv[i]));
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      // lazy rescale: keep the stale max unless the new one exceeds it by more than 2^8 in the
      // exponent (p <= 256 stays exact enough in bf16 and far from fp32 overflow)
      if (tr) trace(1 + wg, j, 3);
      const float m_new = fmaxf(m_run, mx);
      const bool grow = (m_new - m_run) * c > 8.0f;     // true on this warpgroup's first tile (m_run = -inf)
      const float m_use = grow ? m_new : m_run;
      const float alpha = grow ? ex2f((m_run - m_use) * c) : 1.0f;   // first tile: ex2(-inf) = 0
      const float mc = m_use * c;
      // The exponentials are what bounds a tile (16384 ex2 at the SM's 16 per clock = 1024 cycles): the two
      // warpgroups take turns at them (named barriers 2 / 3 as a token), so that one warpgroup's TMEM loads,
      // row max, P stores and barrier waits run under the other's exponentials instead of both halving each
      // other's MUFU rate and then both leaving the unit idle (tests/gpu_attn_trace.py).
      if (pingpong) named_bar_sync(2 + wg, 256);
      float sum2[2] = {0.f, 0.f};
      uint32_t pk[64];
#pragma unroll
      for (int i = 0; i < 128; i += 2) {
        const float p0 = ex2f(fmaf(__uint_as_float(sv[i]), c, -mc));
        const float p1 = ex2f(fmaf(__uint_as_float(sv[i + 1]), c, -mc));
        sum2[(i >> 1) & 1] += p0 + p1;
        pk[i >> 1] = pack_bf16x2(p0, p1);
      }
      if (pingpong) named_bar_arrive(3 - wg, 256);
      l_run = l_run * alpha + (sum2[0] + sum2[1]);
      m_run = m_use;
      if (tr) trace(1 + wg, j, 4);
      if (uses > 0) {
        mbar_wait(bar(bPVdone + wg), ph ^ 1u);      // this warpgroup's O is quiescent, its P buffer free
        tcgen05_fence_after();
        if (__any_sync(0xffffffffu, grow)) {
#pragma unroll 1
          for (int ch = 0; ch < 4; ++ch) {
            uint32_t o[32];
            tmem_ld_32x32b_x32(t_o + (uint32_t)(ch * 32), o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_32x32b_x32(t_o + (uint32_t)(ch * 32), o);
          }
          tmem_st_wait();
        }
      }
      if (tr) trace(1 + wg, j, 5);
#pragma unroll
      for (int u = 0; u < 16; ++u)
        sts128(p_buf + (uint32_t)(u >> 3) * kChunk + swz((uint32_t)r, (uint32_t)(u & 7)), pk[4 * u], pk[4 * u + 1],
               pk[4 * u + 2], pk[4 * u + 3]);
      if (tr) trace(1 + wg, j, 6);
      fence_proxy_async_smem();
      tcgen05_fence_before();
      mbar_arrive(bar(bPfull + wg));
      if (tr) trace(1 + wg, j, 7);
    }
    // ---- merge the two warpgroups' partial soft-maxes: stats through shared memory (their own, now idle,
    //      P buffers), then warpgroup b writes output columns [64 b, 64 b + 64)
    if (uses > 0) {
      mbar_wait(bar(bPVdone + wg), (uint32_t)((uses - 1) & 1));
      tcgen05_fence_after();
    }
    float2* stats = reinterpret_cast<float2*>(base_ptr + oP + (uint32_t)wg * kTile);
    stats[r] = make_float2(m_run, l_run);
    named_bar_sync(1, 256);
    const float2 other = reinterpret_cast<const float2*>(base_ptr + oP + (uint32_t)(wg ^ 1) * kTile)[r];
    const float m0 = wg == 0 ? m_run : other.x, l0 = wg == 0 ? l_run : other.y;
    const float m1 = wg == 0 ? other.x : m_run, l1 = wg == 0 ? other.y : l_run;
    const bool has1 = n_kv > 1;                      // warpgroup 1 saw at least one tile (its O1 is defined)
    const float m = has1 ? fmaxf(m0, m1) : m0;
    const float w0 = ex2f((m0 - m) * c), w1 = has1 ? ex2f((m1 - m) * c) : 0.f;
    const float l = l0 * w0 + l1 * w1;
    const float f0 = w0 / l, f1 = w1 / l;
    const bool live = q_idx < p.S;
    __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(p.o) + (((int64_t)b * p.S + q_idx) * p.H + h) * D + wg * 64;
#pragma unroll 1
    for (int ch = 0; ch < 2; ++ch) {
      uint32_t o0[32], o1[32];
      tmem_ld_32x32b_x32(t_lane + (uint32_t)(2 * BM + wg * 64 + ch * 32), o0);
      if (has1) tmem_ld_32x32b_x32(t_lane + (uint32_t)(2 * BM + D + wg * 64 + ch * 32), o1);
      tmem_ld_wait();
      if (live) {
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          v[i] = __uint_as_float(o0[i]) * f0;
          if (has1) v[i] = fmaf(__uint_as_float(o1[i]), f1, v[i]);
        }
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 q4;
          q4.x = pack_bf16x2(v[i], v[i + 1]);
          q4.y = pack_bf16x2(v[i + 2], v[i + 3]);
          q4.z = pack_bf16x2(v[i + 4], v[i + 5]);
          q4.w = pack_bf16x2(v[i + 6], v[i + 7]);
          *reinterpret_cast<uint4*>(orow + ch * 32 + i) = q4;
        }
      }
    }
    if (wg == 0 && live && p.lse != nullptr)
      p.lse[((int64_t)b * p.H + h) * p.S + q_idx] = m * p.scale + logf(l);
    tcgen05_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_cg1<512>(tmem);
  }
}

// =============================================================================================
// backward: delta = rowsum(dO * O)
// =============================================================================================
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ o,
                                                         const __nv_bfloat16* __restrict__ d_o,
                                                         float* __restrict__ delta, int B, int S, int H) {
  pdl_wait();
  pdl_launch_dependents();
  // one warp per (b, s, h) row of 128 elements: lane reads 4 elements (8 B) of each
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= (int64_t)B * S * H) return;
  const uint2 a = *reinterpret_cast<const uint2*>(o + row * D + lane * 4);
  const uint2 g = *reinterpret_cast<const uint2*>(d_o + row * D + lane * 4);
  float acc = bf16lo(a.x) * bf16lo(g.x) + bf16hi(a.x) * bf16hi(g.x) + bf16lo(a.y) * bf16lo(g.y) +
              bf16hi(a.y) * bf16hi(g.y);
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o2);
  if (lane == 0) {
    const int64_t bs = row / H;
    const int hh = (int)(row % H);
    const int64_t bb = bs / S, ss = bs % S;
    delta[(bb * H + hh) * S + ss] = acc;
  }
}

// =============================================================================================
// backward: dQ  (query-stationary; 64-key steps)
// =============================================================================================
namespace bq {
constexpr int kThreads = 320;                        // warp 0 TMA, warp 1 MMA, warps 2-5 / 6-9: two warpgroups, each thread
                                                     // owns one query row and HALF of the step's 64 key columns
constexpr int BN = 64;                               // keys per step
constexpr uint32_t kTileQ = BM * D * 2;              // 32 KB (2 chunks of 16 KB)
constexpr uint32_t kChunkQ = BM * 128;               // 16 KB
constexpr uint32_t kTileK = BN * D * 2;              // 16 KB (2 chunks of 8 KB)
constexpr uint32_t kChunkK = BN * 128;               // 8 KB
constexpr uint32_t kTileS = BM * BN * 2;             // 16 KB: dS [128][64] bf16, one chunk
constexpr int KS = 4;                                // K / V ring depth: K_j is held until dQ += dS_j K_j retires,
                                                     // i.e. through the whole soft-max of step j
constexpr uint32_t oQ = 0, oDO = kTileQ, oK = 2 * kTileQ, oV = oK + KS * kTileK, oDS = oV + KS * kTileK,
                   oBar = oDS + 2 * kTileS;
enum { bQ = 0, bKfull = 1, bKempty = bKfull + KS, bVfull = bKempty + KS, bVempty = bVfull + KS, bSPfull = bVempty + KS,
       bSPfree = bSPfull + 2, bDSfull = bSPfree + 2, bDSfree = bDSfull + 2, bDone = bDSfree + 2, nBars = bDone + 1 };
constexpr uint32_t oTmem = oBar + 8 * nBars;
constexpr uint32_t kSmem = oTmem + 16 + 1024;
static_assert(kSmem <= 232448, "smem");
// TMEM columns: S0 [0,64) dP0 [64,128) S1 [128,192) dP1 [192,256) dQ [256,384)
}  // namespace bq

__global__ void __launch_bounds__(bq::kThreads, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                   const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do,
                   const AttnParams p) {
  using namespace bq;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q_tile = (int)gridDim.x - 1 - (int)blockIdx.x;
  const int h = blockIdx.y, b = blockIdx.z;
  const int q0 = q_tile * BM;
  const int kv_end = p.causal ? min(q0 + BM, p.S) : p.S;       // keys [0, kv_end)
  const int n_steps = (kv_end + BN - 1) / BN;
  auto bar = [&](int i) { return base + oBar + 8u * (uint32_t)i; };
  // debug trace (qat_attn_debug_trace): slots [384, 768) of the buffer, role 0 = MMA thread, 1 / 2 = warpgroups
  const bool tracing = p.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
  auto trace = [&](int role, int step, int ev) {
    if (tracing && step < kTraceTiles) p.trace[384 + (role * kTraceTiles + step) * kTraceEvents + ev] = clock64();
  };

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&map_q);
    prefetch_tensormap(&map_k);
    prefetch_tensormap(&map_v);
    prefetch_tensormap(&map_do);
    mbar_init(bar(bQ), 1);
    for (int s = 0; s < KS; ++s) {
      mbar_init(bar(bKfull + s), 1);
      mbar_init(bar(bKempty + s), 1);
      mbar_init(bar(bVfull + s), 1);
      mbar_init(bar(bVempty + s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar(bSPfull + s), 1);
      mbar_init(bar(bSPfree + s), 256);
      mbar_init(bar(bDSfull + s), 256);
      mbar_init(bar(bDSfree + s), 1);
    }
    mbar_init(bar(bDone), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc_cg1<512>(base + oTmem);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(base_ptr + oTmem);
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    if (lane == 0) {
      const int32_t col = h * D;
      mbar_expect_tx(bar(bQ), 2 * kTileQ);
      tma_load_3d(base + oQ, &map_q, bar(bQ), col, q0, b);
      tma_load_3d(base + oQ + kChunkQ, &map_q, bar(bQ), col + 64, q0, b);
      tma_load_3d(base + oDO, &map_do, bar(bQ), col, q0, b);
      tma_load_3d(base + oDO + kChunkQ, &map_do, bar(bQ), col + 64, q0, b);
      for (int j = 0; j < n_steps; ++j) {
        const int ks = j % KS;
        const uint32_t ph = (uint32_t)((j / KS) & 1);
        // K[ks] is read by S_j (K-major) and by dQ += dS_j K_j (MN-major): free after the latter
        mbar_wait(bar(bKempty + ks), ph ^ 1u);
        mbar_expect_tx(bar(bKfull + ks), kTileK);
        tma_load_3d(base + oK + ks * kTileK, &map_k, bar(bKfull + ks), col, j * BN, b);
        tma_load_3d(base + oK + ks * kTileK + kChunkK, &map_k, bar(bKfull + ks), col + 64, j * BN, b);
        mbar_wait(bar(bVempty + ks), ph ^ 1u);
        mbar_expect_tx(bar(bVfull + ks), kTileK);
        tma_load_3d(base + oV + ks * kTileK, &map_v, bar(bVfull + ks), col, j * BN, b);
        tma_load_3d(base + oV + ks * kTileK + kChunkK, &map_v, bar(bVfull + ks), col + 64, j * BN, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(BM, BN, 0, 0);      // S / dP: M128 N64, K-major x K-major
      constexpr uint32_t idesc_dq = make_idesc_bf16(BM, D, 0, 1);      // dQ: M128 N128, B = K MN-major
      auto issue_sp = [&](int j) {
        const int s = j & 1, ks = j % KS;
        const uint32_t ph = (uint32_t)((j >> 1) & 1), kph = (uint32_t)((j / KS) & 1);
        trace(0, j, 0);
        mbar_wait(bar(bKfull + ks), kph);
        mbar_wait(bar(bVfull + ks), kph);
        trace(0, j, 1);
        mbar_wait(bar(bSPfree + s), ph ^ 1u);
        tcgen05_fence_after();
        trace(0, j, 2);
        const uint32_t d_s = tmem + (uint32_t)(s * 128), d_p = d_s + 64u;
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_f16<1>(d_s, desc_k_step(base + oQ, kChunkQ, k), desc_k_step(base + oK + ks * kTileK, kChunkK, k),
                      idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_f16<1>(d_p, desc_k_step(base + oDO, kChunkQ, k), desc_k_step(base + oV + ks * kTileK, kChunkK, k),
                      idesc_s, k > 0 ? 1u : 0u);
        umma_commit(bar(bVempty + ks));
        umma_commit(bar(bSPfull + s));
        trace(0, j, 3);
      };
      mbar_wait(bar(bQ), 0);
      issue_sp(0);
      for (int j = 0; j < n_steps; ++j) {
        if (j + 1 < n_steps) issue_sp(j + 1);
        const int s = j & 1, ks = j % KS;
        trace(0, j, 4);
        mbar_wait(bar(bDSfull + s), (uint32_t)((j >> 1) & 1));
        tcgen05_fence_after();
        trace(0, j, 5);
        const uint32_t d_q = tmem + 256u;
#pragma unroll
        for (int k = 0; k < BN / 16; ++k)
          umma_f16<1>(d_q, make_smem_desc(base + oDS + s * kTileS + (uint32_t)k * 32u),
                      desc_mn_step(base + oK + ks * kTileK, kChunkK, k), idesc_dq, (j > 0 || k > 0) ? 1u : 0u);
        umma_commit(bar(bKempty + ks));
        umma_commit(bar(bDSfree + s));
        trace(0, j, 6);
      }
      umma_commit(bar(bDone));
    }
  } else {
    const int wg = (warp - 2) >> 2;                 // which half of the step's key columns
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const int q_idx = q0 + r;
    const bool live = q_idx < p.S;
    const uint32_t t_lane = tmem + ((uint32_t)(quad * 32) << 16);
    const float c = p.scale * kLog2e;
    const int64_t stat = ((int64_t)b * p.H + h) * p.S + q_idx;
    const float lse_c = live ? p.lse[stat] * kLog2e : 0.f;
    const float dlt = live ? p.delta[stat] : 0.f;
    const int c0 = wg * 32;
    const bool tr = (threadIdx.x == 64 || threadIdx.x == 192);
    for (int j = 0; j < n_steps; ++j) {
      const int s = j & 1;
      const uint32_t ph = (uint32_t)((j >> 1) & 1);
      if (tr) trace(1 + wg, j, 0);
      mbar_wait(bar(bSPfull + s), ph);
      tcgen05_fence_after();
      if (tr) trace(1 + wg, j, 1);
      uint32_t sv[32], dp[32];
      tmem_ld_32x32b_x32(t_lane + (uint32_t)(s * 128 + c0), sv);
      tmem_ld_32x32b_x32(t_lane + (uint32_t)(s * 128 + 64 + c0), dp);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(bar(bSPfree + s));
      if (tr) trace(1 + wg, j, 2);
      const int k0 = j * BN + c0;
      const bool edge = (p.causal && j * BN + BN - 1 > q0) || (j * BN + BN > p.S) || (q0 + BM > p.S);
      uint32_t pk[16];
      if (edge) {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          float ds[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int k_idx = k0 + i + e;
            const bool dead = !live || k_idx >= p.S || (p.causal && k_idx > q_idx);
            const float pr = ex2f(fmaf(__uint_as_float(sv[i + e]), c, -lse_c));
            ds[e] = dead ? 0.f : pr * (__uint_as_float(dp[i + e]) - dlt) * p.scale;
          }
          pk[i >> 1] = pack_bf16x2(ds[0], ds[1]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float p0 = ex2f(fmaf(__uint_as_float(sv[i]), c, -lse_c));
          const float p1 = ex2f(fmaf(__uint_as_float(sv[i + 1]), c, -lse_c));
          pk[i >> 1] = pack_bf16x2(p0 * (__uint_as_float(dp[i]) - dlt) * p.scale,
                                   p1 * (__uint_as_float(dp[i + 1]) - dlt) * p.scale);
        }
      }
      if (tr) trace(1 + wg, j, 3);
      mbar_wait(bar(bDSfree + s), ph ^ 1u);        // the dQ MMA that read this dS buffer two steps ago is done
      if (tr) trace(1 + wg, j, 4);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        sts128(base + oDS + s * kTileS + swz((uint32_t)r, (uint32_t)(wg * 4 + u)), pk[4 * u], pk[4 * u + 1],
               pk[4 * u + 2], pk[4 * u + 3]);
      fence_proxy_async_smem();
      mbar_arrive(bar(bDSfull + s));
      if (tr) trace(1 + wg, j, 5);
    }
    mbar_wait(bar(bDone), 0);
    tcgen05_fence_after();
    __nv_bfloat16* row = reinterpret_cast<__nv_bfloat16*>(p.dq) + (((int64_t)b * p.S + q_idx) * p.H + h) * D + wg * 64;
#pragma unroll 1
    for (int ch = 0; ch < 2; ++ch) {
      uint32_t o[32];
      tmem_ld_32x32b_x32(t_lane + (uint32_t)(256 + wg * 64 + ch * 32), o);
      tmem_ld_wait();
      if (live) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 v;
          v.x = pack_bf16x2(__uint_as_float(o[i]), __uint_as_float(o[i + 1]));
          v.y = pack_bf16x2(__uint_as_float(o[i + 2]), __uint_as_float(o[i + 3]));
          v.z = pack_bf16x2(__uint_as_float(o[i + 4]), __uint_as_float(o[i + 5]));
          v.w = pack_bf16x2(__uint_as_float(o[i + 6]), __uint_as_float(o[i + 7]));
          *reinterpret_cast<uint4*>(row + ch * 32 + i) = v;
        }
      }
    }
    tcgen05_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_cg1<512>(tmem);
  }
}

// =============================================================================================
// backward: dK, dV  (key-stationary; 64-query steps)
// =============================================================================================
namespace bk {
constexpr int kThreads = 320;                        // as attn_bwd_dq: two warpgroups split the step's 64 query columns
constexpr int BN = 64;                               // queries per step
constexpr uint32_t kTileK = BM * D * 2;              // 32 KB
constexpr uint32_t kChunkK = BM * 128;               // 16 KB
constexpr uint32_t kTileQ = BN * D * 2;              // 16 KB (2 chunks of 8 KB)
constexpr uint32_t kChunkQ = BN * 128;               // 8 KB
constexpr uint32_t kTileS = BM * BN * 2;             // 16 KB: P^T / dS^T [128 keys][64 q]
constexpr int QS = 3;                                // Q / dO ring depth (held until dV / dK of the step retire)
constexpr uint32_t oK = 0, oV = kTileK, oQ = 2 * kTileK, oDO = oQ + QS * kTileQ, oPT = oDO + QS * kTileQ,
                   oDST = oPT + 2 * kTileS, oStat = oDST + 2 * kTileS, oBar = oStat + 2 * 2 * BN * 4;
enum { bKV = 0, bQfull = 1, bQempty = bQfull + QS, bSPfull = bQempty + QS, bSPfree = bSPfull + 2, bPfull = bSPfree + 2,
       bPfree = bPfull + 2, bDone = bPfree + 2, nBars = bDone + 1 };
constexpr uint32_t oTmem = oBar + 8 * nBars;
constexpr uint32_t kSmem = oTmem + 16 + 1024;
static_assert(kSmem <= 232448, "smem");
// TMEM columns: S^T0 [0,64) dP^T0 [64,128) S^T1 [128,192) dP^T1 [192,256) dK [256,384) dV [384,512)
}  // namespace bk

__global__ void __launch_bounds__(bk::kThreads, 1)
attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do,
                    const AttnParams p) {
  using namespace bk;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kv_tile = blockIdx.x;                     // tile 0 has the most query steps under the causal mask
  const int h = blockIdx.y, b = blockIdx.z;
  const int k0 = kv_tile * BM;
  const int q_begin = p.causal ? (k0 / BN) * BN : 0;  // first query that can see a key of this tile
  const int n_steps = (p.S - q_begin + BN - 1) / BN;
  auto bar = [&](int i) { return base + oBar + 8u * (uint32_t)i; };

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&map_q);
    prefetch_tensormap(&map_k);
    prefetch_tensormap(&map_v);
    prefetch_tensormap(&map_do);
    mbar_init(bar(bKV), 1);
    for (int s = 0; s < QS; ++s) {
      mbar_init(bar(bQfull + s), 1);
      mbar_init(bar(bQempty + s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar(bSPfull + s), 1);
      mbar_init(bar(bSPfree + s), 256);
      mbar_init(bar(bPfull + s), 256);
      mbar_init(bar(bPfree + s), 1);
    }
    mbar_init(bar(bDone), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc_cg1<512>(base + oTmem);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(base_ptr + oTmem);
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    if (lane == 0) {
      const int32_t col = h * D;
      mbar_expect_tx(bar(bKV), 2 * kTileK);
      tma_load_3d(base + oK, &map_k, bar(bKV), col, k0, b);
      tma_load_3d(base + oK + kChunkK, &map_k, bar(bKV), col + 64, k0, b);
      tma_load_3d(base + oV, &map_v, bar(bKV), col, k0, b);
      tma_load_3d(base + oV + kChunkK, &map_v, bar(bKV), col + 64, k0, b);
      for (int i = 0; i < n_steps; ++i) {
        const int s = i % QS;
        const uint32_t ph = (uint32_t)((i / QS) & 1);
        mbar_wait(bar(bQempty + s), ph ^ 1u);
        mbar_expect_tx(bar(bQfull + s), 2 * kTileQ);
        const int32_t qr = q_begin + i * BN;
        tma_load_3d(base + oQ + s * kTileQ, &map_q, bar(bQfull + s), col, qr, b);
        tma_load_3d(base + oQ + s * kTileQ + kChunkQ, &map_q, bar(bQfull + s), col + 64, qr, b);
        tma_load_3d(base + oDO + s * kTileQ, &map_do, bar(bQfull + s), col, qr, b);
        tma_load_3d(base + oDO + s * kTileQ + kChunkQ, &map_do, bar(bQfull + s), col + 64, qr, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(BM, BN, 0, 0);      // S^T / dP^T: M128 (keys) N64 (queries)
      constexpr uint32_t idesc_acc = make_idesc_bf16(BM, D, 0, 1);     // dV / dK: M128 N128, B MN-major
      auto issue_sp = [&](int i) {
        const int s = i & 1, qs = i % QS;
        const uint32_t ph = (uint32_t)((i >> 1) & 1);
        mbar_wait(bar(bQfull + qs), (uint32_t)((i / QS) & 1));
        mbar_wait(bar(bSPfree + s), ph ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_s = tmem + (uint32_t)(s * 128), d_p = d_s + 64u;
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_f16<1>(d_s, desc_k_step(base + oK, kChunkK, k), desc_k_step(base + oQ + qs * kTileQ, kChunkQ, k),
                      idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_f16<1>(d_p, desc_k_step(base + oV, kChunkK, k), desc_k_step(base + oDO + qs * kTileQ, kChunkQ, k),
                      idesc_s, k > 0 ? 1u : 0u);
        umma_commit(bar(bSPfull + s));
      };
      mbar_wait(bar(bKV), 0);
      issue_sp(0);
      for (int i = 0; i < n_steps; ++i) {
        if (i + 1 < n_steps) issue_sp(i + 1);
        const int s = i & 1, qs = i % QS;
        mbar_wait(bar(bPfull + s), (uint32_t)((i >> 1) & 1));
        tcgen05_fence_after();
        const uint32_t d_k = tmem + 256u, d_v = tmem + 384u;
#pragma unroll
        for (int k = 0; k < BN / 16; ++k)
          umma_f16<1>(d_v, make_smem_desc(base + oPT + s * kTileS + (uint32_t)k * 32u),
                      desc_mn_step(base + oDO + qs * kTileQ, kChunkQ, k), idesc_acc, (i > 0 || k > 0) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < BN / 16; ++k)
          umma_f16<1>(d_k, make_smem_desc(base + oDST + s * kTileS + (uint32_t)k * 32u),
                      desc_mn_step(base + oQ + qs * kTileQ, kChunkQ, k), idesc_acc, (i > 0 || k > 0) ? 1u : 0u);
        umma_commit(bar(bQempty + qs));
        umma_commit(bar(bPfree + s));
      }
      umma_commit(bar(bDone));
    }
  } else {
    const int wg = (warp - 2) >> 2;                   // which half of the step's query columns
    const int quad = warp & 3;
    const int r = quad * 32 + lane;                   // key row
    const int st = threadIdx.x - 64;                  // 0..255 among the softmax threads
    const int k_idx = k0 + r;
    const bool live = k_idx < p.S;
    const uint32_t t_lane = tmem + ((uint32_t)(quad * 32) << 16);
    const float c = p.scale * kLog2e;
    const int64_t stat0 = ((int64_t)b * p.H + h) * p.S;
    const int c0 = wg * 32;
    for (int i = 0; i < n_steps; ++i) {
      const int s = i & 1;
      const uint32_t ph = (uint32_t)((i >> 1) & 1);
      const int qr = q_begin + i * BN;
      // stage this step's 64 LSE (x log2 e) and 64 delta values: thread t < 64 -> lse, 64 <= t < 128 -> delta
      float* stat = reinterpret_cast<float*>(base_ptr + oStat) + s * 2 * BN;
      if (st < 128) {
        const int qi = qr + (st & 63);
        float v = 0.f;
        if (qi < p.S) v = (st < 64) ? p.lse[stat0 + qi] * kLog2e : p.delta[stat0 + qi];
        stat[st] = v;
      }
      named_bar_sync(1, 256);
      mbar_wait(bar(bSPfull + s), ph);
      tcgen05_fence_after();
      uint32_t sv[32], dp[32];
      tmem_ld_32x32b_x32(t_lane + (uint32_t)(s * 128 + c0), sv);
      tmem_ld_32x32b_x32(t_lane + (uint32_t)(s * 128 + 64 + c0), dp);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(bar(bSPfree + s));
      const bool edge = (p.causal && k0 + BM - 1 > qr) || (qr + BN > p.S) || (k0 + BM > p.S);
      uint32_t ppk[16], dpk[16];
#pragma unroll
      for (int q = 0; q < 32; q += 4) {
        const float4 l4 = *reinterpret_cast<const float4*>(stat + c0 + q);
        const float4 d4 = *reinterpret_cast<const float4*>(stat + BN + c0 + q);
        const float ls[4] = {l4.x, l4.y, l4.z, l4.w};
        const float dl[4] = {d4.x, d4.y, d4.z, d4.w};
        float pr[4], ds[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float pv = ex2f(fmaf(__uint_as_float(sv[q + e]), c, -ls[e]));
          bool dead = false;
          if (edge) {
            const int q_idx = qr + c0 + q + e;
            dead = !live || q_idx >= p.S || (p.causal && k_idx > q_idx);
          }
          pr[e] = dead ? 0.f : pv;
          ds[e] = dead ? 0.f : pv * (__uint_as_float(dp[q + e]) - dl[e]) * p.scale;
        }
        ppk[q >> 1] = pack_bf16x2(pr[0], pr[1]);
        ppk[(q >> 1) + 1] = pack_bf16x2(pr[2], pr[3]);
        dpk[q >> 1] = pack_bf16x2(ds[0], ds[1]);
        dpk[(q >> 1) + 1] = pack_bf16x2(ds[2], ds[3]);
      }
      mbar_wait(bar(bPfree + s), ph ^ 1u);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        sts128(base + oPT + s * kTileS + swz((uint32_t)r, (uint32_t)(wg * 4 + u)), ppk[4 * u], ppk[4 * u + 1],
               ppk[4 * u + 2], ppk[4 * u + 3]);
        sts128(base + oDST + s * kTileS + swz((uint32_t)r, (uint32_t)(wg * 4 + u)), dpk[4 * u], dpk[4 * u + 1],
               dpk[4 * u + 2], dpk[4 * u + 3]);
      }
      fence_proxy_async_smem();
      mbar_arrive(bar(bPfull + s));
    }
    mbar_wait(bar(bDone), 0);
    tcgen05_fence_after();
    // warpgroup 0 stores dK, warpgroup 1 stores dV
    const int64_t off = (((int64_t)b * p.S + k_idx) * p.H + h) * D;
    __nv_bfloat16* row = reinterpret_cast<__nv_bfloat16*>(wg == 0 ? p.dk : p.dv) + off;
#pragma unroll 1
    for (int ch = 0; ch < 4; ++ch) {
      uint32_t o[32];
      tmem_ld_32x32b_x32(t_lane + (uint32_t)(256 + wg * 128 + ch * 32), o);
      tmem_ld_wait();
      if (live) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 v;
          v.x = pack_bf16x2(__uint_as_float(o[i]), __uint_as_float(o[i + 1]));
          v.y = pack_bf16x2(__uint_as_float(o[i + 2]), __uint_as_float(o[i + 3]));
          v.z = pack_bf16x2(__uint_as_float(o[i + 4]), __uint_as_float(o[i + 5]));
          v.w = pack_bf16x2(__uint_as_float(o[i + 6]), __uint_as_float(o[i + 7]));
          *reinterpret_cast<uint4*>(row + ch * 32 + i) = v;
        }
      }
    }
    tcgen05_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_cg1<512>(tmem);
  }
}

// ---- host -------------------------------------------------------------------------------------
// bf16 [B, S, H*D] viewed as a 3-D tensor {H*D, S, B}; box {64, box_rows, 1}, 128B swizzle, zero fill
int make_map_bshd(CUtensorMap* map, const void* ptr, int B, int S, int H, int box_rows) {
  EncodeFn enc = get_encode();
  if (enc == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return QAT_ERR_UNSUPPORTED;
  }
  const cuuint64_t hd = (cuuint64_t)H * D;
  cuuint64_t dims[3] = {hd, (cuuint64_t)S, (cuuint64_t)B};
  cuuint64_t strides[2] = {hd * 2, hd * 2 * (cuuint64_t)S};
  cuuint32_t box[3] = {64u, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) for bf16 [%d, %d, %d, %d]", (int)r, B, S, H, D);
    return QAT_ERR_BAD_ARG;
  }
  return QAT_OK;
}

int check_common(const void* q, const void* k, const void* v, int B, int S, int H, int Dh) {
  QAT_CHECK_ARG(Dh == D, "head_dim must be %d (got %d)", D, Dh);
  QAT_CHECK_ARG(B > 0 && S > 0 && H > 0, "bad shape B=%d S=%d H=%d", B, S, H);
  QAT_CHECK_ARG(B <= 65535 && H <= 65535, "B and H must fit a grid dimension");
  QAT_CHECK_ARG(q && k && v, "NULL operand");
  QAT_CHECK_ARG((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v) & 15) == 0, "operands must be 16-byte aligned");
  return QAT_OK;
}

}  // namespace
}  // namespace qat

extern "C" int qat_attn_debug_trace(long long* dev_buffer) {   // 2 kernels x 3 roles x 16 steps x 8 events (int64), or NULL: off
  qat::g_attn_trace = dev_buffer;
  return QAT_OK;
}

extern "C" int qat_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int B, int S, int H,
                            int head_dim, float softmax_scale, int causal, void* stream) {
  using namespace qat;
  int rc = check_common(q, k, v, B, S, H, head_dim);
  if (rc != QAT_OK) return rc;
  QAT_CHECK_ARG(o != nullptr && ((uintptr_t)o & 15) == 0, "o must be a 16-byte aligned device pointer");
  CUtensorMap mq, mk, mv;
  if ((rc = make_map_bshd(&mq, q, B, S, H, BM)) != QAT_OK) return rc;
  if ((rc = make_map_bshd(&mk, k, B, S, H, BM)) != QAT_OK) return rc;
  if ((rc = make_map_bshd(&mv, v, B, S, H, BM)) != QAT_OK) return rc;
  static bool opted_in[64] = {};
  if ((rc = opt_in_smem(attn_fwd_kernel, fwd::kSmem, opted_in, "attention kernel")) != QAT_OK) return rc;
  AttnParams p{};
  p.trace = g_attn_trace;
  p.o = o;
  p.lse = lse;
  p.B = B;
  p.S = S;
  p.H = H;
  p.scale = softmax_scale;
  p.causal = causal ? 1 : 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const dim3 grid((unsigned)((S + BM - 1) / BM), (unsigned)H, (unsigned)B);
  cudaError_t e = launch_pdl(attn_fwd_kernel, grid, dim3(fwd::kThreads), fwd::kSmem, st, mq, mk, mv, p);
  if (e != cudaSuccess) return cuda_fail(e, "attn_fwd_kernel launch");
  QAT_CHECK_LAUNCH("attn_fwd_kernel");
  return QAT_OK;
}

extern "C" int qat_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o,
                            const float* lse, float* delta, void* dq, void* dk, void* dv, int B, int S, int H,
                            int head_dim, float softmax_scale, int causal, void* stream) {
  using namespace qat;
  int rc = check_common(q, k, v, B, S, H, head_dim);
  if (rc != QAT_OK) return rc;
  QAT_CHECK_ARG(o && d_o && lse && delta && dq && dk && dv, "NULL operand");
  QAT_CHECK_ARG((((uintptr_t)o | (uintptr_t)d_o | (uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) & 15) == 0,
                "operands must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  {
    const int64_t rows = (int64_t)B * S * H;
    cudaError_t e = launch_pdl(attn_delta_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, st,
                               reinterpret_cast<const __nv_bfloat16*>(o), reinterpret_cast<const __nv_bfloat16*>(d_o),
                               delta, B, S, H);
    if (e != cudaSuccess) return cuda_fail(e, "attn_delta_kernel launch");
    QAT_CHECK_LAUNCH("attn_delta_kernel");
  }
  AttnParams p{};
  p.trace = g_attn_trace;
  p.lse = const_cast<float*>(lse);
  p.delta = delta;
  p.dq = dq;
  p.dk = dk;
  p.dv = dv;
  p.B = B;
  p.S = S;
  p.H = H;
  p.scale = softmax_scale;
  p.causal = causal ? 1 : 0;
  {
    CUtensorMap mq, mk, mv, mdo;
    if ((rc = make_map_bshd(&mq, q, B, S, H, BM)) != QAT_OK) return rc;
    if ((rc = make_map_bshd(&mdo, d_o, B, S, H, BM)) != QAT_OK) return rc;
    if ((rc = make_map_bshd(&mk, k, B, S, H, bq::BN)) != QAT_OK) return rc;
    if ((rc = make_map_bshd(&mv, v, B, S, H, bq::BN)) != QAT_OK) return rc;
    static bool opted_in[64] = {};
    if ((rc = opt_in_smem(attn_bwd_dq_kernel, bq::kSmem, opted_in, "attention kernel")) != QAT_OK) return rc;
    const dim3 grid((unsigned)((S + BM - 1) / BM), (unsigned)H, (unsigned)B);
    cudaError_t e = launch_pdl(attn_bwd_dq_kernel, grid, dim3(bq::kThreads), bq::kSmem, st, mq, mk, mv, mdo, p);
    if (e != cudaSuccess) return cuda_fail(e, "attn_bwd_dq_kernel launch");
    QAT_CHECK_LAUNCH("attn_bwd_dq_kernel");
  }
  {
    CUtensorMap mq, mk, mv, mdo;
    if ((rc = make_map_bshd(&mq, q, B, S, H, bk::BN)) != QAT_OK) return rc;
    if ((rc = make_map_bshd(&mdo, d_o, B, S, H, bk::BN)) != QAT_OK) return rc;
    if ((rc = make_map_bshd(&mk, k, B, S, H, BM)) != QAT_OK) return rc;
    if ((rc = make_map_bshd(&mv, v, B, S, H, BM)) != QAT_OK) return rc;
    static bool opted_in[64] = {};
    if ((rc = opt_in_smem(attn_bwd_dkv_kernel, bk::kSmem, opted_in, "attention kernel")) != QAT_OK) return rc;
    const dim3 grid((unsigned)((S + BM - 1) / BM), (unsigned)H, (unsigned)B);
    cudaError_t e = launch_pdl(attn_bwd_dkv_kernel, grid, dim3(bk::kThreads), bk::kSmem, st, mq, mk, mv, mdo, p);
    if (e != cudaSuccess) return cuda_fail(e, "attn_bwd_dkv_kernel launch");
    QAT_CHECK_LAUNCH("attn_bwd_dkv_kernel");
  }
  return QAT_OK;
}
