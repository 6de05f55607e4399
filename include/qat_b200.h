/*
 * qat_b200.h — C ABI of libqat_b200.so: hand-written sm_100a kernels for
 * LLM-QAT's fake-quantization hot path.
 *
 * The reference (JingyangXiang/LLM-QAT) has no FFI: its hot path is eager
 * PyTorch in models/utils_quant.py.  This header is the thin layer that a
 * drop-in `models/utils_quant.py` binds with ctypes (see INTEGRATION.md); each
 * entry point names the reference lines it replaces.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer owned by the
 *     caller unless the name ends in `_host`;
 *   - tensors are dense row-major `[rows, cols]`; one row == one reduction set
 *     (per-token / per-output-channel / per-(b,h) / whole tensor — the caller
 *     flattens exactly as utils_quant.py:50-70 does);
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous on
 *     it, the library never synchronises and never allocates;
 *   - return value: 0 on success, a QAT_ERR_* or cudaError_t otherwise;
 *     qat_last_error() returns a thread-local message;
 *   - outputs must not alias inputs;
 *   - arithmetic follows the reference's op order bit-for-bit (SURVEY.md
 *     appendix A): no FMA contraction, IEEE division, round-half-even, and in
 *     bf16 one rounding to bf16 after every op.
 */
#ifndef QAT_B200_H_
#define QAT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QAT_B200_VERSION 100 /* major*10000 + minor*100 + patch */

/* element types of x / y / g / gx */
#define QAT_F32 0
#define QAT_BF16 1
/* SymQuantizer on a bf16 tensor inside torch.autocast — the context HF's Trainer runs the step in
 * (kd_trainer.py:106).  Autocast executes `Q / (max + 1e-6)` (Tensor.__rtruediv__ = reciprocal * Q)
 * in fp32, so the reference's chain becomes: max|x| and `max + 1e-6` in bf16, then the reciprocal, the
 * scale, x * s, round, s + 1e-6 and the division all in fp32, and the result is an fp32 tensor
 * (measured on the GPU box: tests/gpu_autocast_probe.py).  qat_sym_fwd only: x bf16, y fp32. */
#define QAT_BF16_AMP 2
/* The QAT_BF16_AMP chain followed by the cast autocast's F.linear applies to its operand
 * (utils_quant.py:250): y = bf16(y_fp32), one more round-to-nearest-even.  This is the exact bf16
 * operand the reference hands its GEMM under autocast, written at 2 B/elem instead of 4 and without a
 * separate cast pass.  qat_sym_fwd only: x bf16, y bf16 (codes and mask as for QAT_BF16_AMP). */
#define QAT_BF16_AMP_CAST 3

/* optional integer-code output */
#define QAT_CODES_NONE 0
#define QAT_CODES_I8 1  /* saturating to [-128,127] (Sym) / [0,255] as uint8 (Asym); NaN -> 0.  GEMM feed. */
#define QAT_CODES_I16 2 /* exact; NaN -> INT16_MIN.  What parity tests compare. */

/* error codes (cudaError_t values are passed through unchanged, all < 1000) */
#define QAT_OK 0
#define QAT_ERR_BAD_ARG 1001
#define QAT_ERR_UNSUPPORTED 1002
#define QAT_ERR_WORKSPACE 1003
#define QAT_ERR_NO_DEVICE 1004

int qat_version(void);
const char* qat_last_error(void);
/* Number of kernels this library has launched in the calling process (all
 * threads); bench.py reports the delta over its timed region. */
uint64_t qat_launch_count(void);
/* 0 when a CUDA device with compute capability 10.x is current, else an error. */
int qat_check_device(void);

/*
 * Workspace (bytes) the forward entry points need for a [rows, cols] tensor.
 * Rows that fit one CTA's registers (the per-token / per-channel case) need
 * none; longer rows (layerwise mode: rows == 1, cols == numel) use a two-phase
 * reduce-then-apply and need 16 bytes per row.
 */
size_t qat_fwd_workspace_bytes(int64_t rows, int64_t cols, int dtype);

/*
 * SymQuantizer.forward — utils_quant.py:37-74.
 *   m = max|x_row|; s = fl(fl(1/fl(m+1e-6)) * Q), Q = 2^(bits-1)-1;
 *   q = rint(fl(x*s)); y = fl(q / fl(s+1e-6)).
 * y      [rows, cols] dtype, may be NULL (codes-only mode for the GEMM feed)
 * codes  [rows, cols] int8 / int16 per `codes_kind`, may be NULL
 * row_s  [rows] float (s), row_e [rows] float (the dequant divisor), may be NULL
 * mask   packed STE mask, bit i%8 of byte i/8 = (lo < x_i < hi), may be NULL;
 *        lo/hi are only read when mask != NULL (utils_quant.py:85-86).
 */
int qat_sym_fwd(const void* x, void* y, void* codes, int codes_kind, float* row_s, float* row_e,
                uint8_t* mask, float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                int bits, void* workspace, size_t workspace_bytes, void* stream);

/*
 * AsymQuantizer.forward — utils_quant.py:96-149.
 *   a = fl(fl(max-min)+1e-8); b = min; S = 2^bits-1;
 *   q = rint(fl(fl(fl(x-b)/a)*S)); y = fl(fl(fl(q/S)*a)+b).
 * codes: uint8 (QAT_CODES_I8, bits<=8) or int16; row_a / row_b [rows] float.
 */
int qat_asym_fwd(const void* x, void* y, void* codes, int codes_kind, float* row_a, float* row_b,
                 uint8_t* mask, float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                 int bits, void* workspace, size_t workspace_bytes, void* stream);

/*
 * How AsymQuantizer divides the code by S = 2^bits - 1 (utils_quant.py:146, `.div(s)` with a Python
 * int): QAT_ASYM_DIV_TRUE (default) is the IEEE division torch's CPU kernel performs — BASELINE
 * configs[0] names torch CPU, and the oracle follows it; QAT_ASYM_DIV_RECIP multiplies by fl(1/S), which
 * is what ATen's CUDA kernel does for a CPU-scalar divisor, so fp32 results then match the reference
 * run eagerly on a GPU bit for bit (33 % of fp32 elements differ between the two; bf16 results are
 * identical for bits <= 8).  Process-wide; also settable once through QAT_B200_ASYM_DIV=cpu|cuda.
 */
#define QAT_ASYM_DIV_TRUE 0
#define QAT_ASYM_DIV_RECIP 1
int qat_set_asym_div(int mode);

/*
 * SymQuantizer.backward / AsymQuantizer.backward — utils_quant.py:77-87, 152-162.
 *   gx_i = (x_i >= hi || x_i <= lo) ? 0 : g_i      (bounds compared in x's dtype)
 * mask_out (optional) receives the packed pass-mask; n = number of elements.
 */
int qat_ste_bwd(const void* g, const void* x, void* gx, uint8_t* mask_out, float clip_lo,
                float clip_hi, int64_t n, int dtype, void* stream);

/* Same backward with the clip bounds {lo, hi} read in-kernel from DEVICE memory (two floats):
 * a CUDA clip_val costs no host synchronisation (the reference indexes clip_val[0] / [1] as
 * 0-dim tensors, utils_quant.py:85-86).  Bounds are rounded to x's dtype, like x.ge(clip_val[1]). */
int qat_ste_bwd_devclip(const void* g, const void* x, void* gx, uint8_t* mask_out, const float* clip_dev,
                        int64_t n, int dtype, void* stream);

/* Same backward, driven by a forward-emitted packed mask instead of x
 * (reads 2e + 1/8 bytes per element instead of 3e). */
int qat_ste_bwd_from_mask(const void* g, const uint8_t* mask, void* gx, int64_t n, int dtype,
                          void* stream);

/*
 * QuantizeLinear low-bit weight path — utils_quant.py:202-242 (w_bits in {1,2}).
 * w_eff = fl(fl(q - w) + w) with q the 1-bit sign / 2-bit 4-level quantization
 * scaled by the row (or tensor) mean |w|.  rows = out_features.
 * The row mean is summed in the order of torch's CPU reduction (csrc/torch_sum_order.cuh), so w_eff
 * carries the reference's bits in fp32 and bf16 for any width and alignment (rows up to ~220 KB; one
 * pass).  Layerwise: exact below 32768 elements; above, torch splits the reduction over its threads
 * (no machine-independent result exists) and a double-precision sum is used — like for longer rows —
 * through `workspace` (two passes).  w and w_eff must not alias.
 */
size_t qat_lowbit_workspace_bytes(int64_t rows, int layerwise); /* 8 B per row, or 8 B layerwise */
int qat_lowbit_weight_fwd(const void* w, void* w_eff, int64_t rows, int64_t cols, int dtype,
                          int w_bits, int layerwise, void* workspace, size_t workspace_bytes,
                          void* stream);

/*
 * QuantizeLinear.forward contraction — utils_quant.py:250 on integer-grid
 * operands:  out[t, n] = (sum_k qx[t,k] * qw[n,k]) / (ex[t] * ew[n]).
 * tcgen05 (kind::i8, s32 accumulators in TMEM), TMA-fed, dual-scale epilogue.
 *   qx [T, K] int8, qw [N, K] int8 (both K-major), ex [T], ew [N] float,
 *   out [T, N] in `out_dtype`.  K % 16 == 0 required (TMA row pitch).
 */
int qat_qlinear_i8_fwd(const int8_t* qx, const int8_t* qw, const float* ex, const float* ew,
                       void* out, int64_t T, int64_t N, int64_t K, int out_dtype, void* stream);

/* Programmatic dependent launch for the hot kernels (K1-K4, dequant): 1 (default) lets a
 * kernel's CTAs be scheduled while the previous kernel of the stream drains — no memory is
 * touched before that grid has completed (griddepcontrol.wait); 0 = plain stream order.
 * Also settable once through the environment, QAT_B200_PDL=0. */
int qat_set_pdl(int enabled);

/* Tuning knob of the contraction: CTAs per tcgen05.mma.  2 = CTA pairs on 256x256
 * tiles (cta_group::2), 1 = single CTAs on 128x256 tiles, 0 = choose per problem
 * (the default; also settable once through the environment, QAT_B200_GEMM_CG). */
int qat_set_gemm_cta_group(int cta_group);

/*
 * QuantizeLinear.forward main path in one call (utils_quant.py:197-201,244-250):
 * qat_sym_fwd (codes-only) on x [T,K] and on w [N,K], then qat_qlinear_i8_fwd.
 * qx/ex/mx and qw/ew/mw receive the int8 codes, dequant divisors and packed STE
 * masks (mx / mw may be NULL); reuse_x / reuse_w != 0 skip a quantization whose
 * outputs the caller still holds.  K % 16 == 0, 2 <= bits <= 8.
 * Deviation from the reference, plain-bf16 8-bit operands only: bf16 rounding of x*s can give the
 * code +128 for a row's largest elements (fp32 tensors and dtype QAT_BF16_AMP — the recipe's
 * autocast chain — cannot); the int8 feed carries 127 for them (-128 is exact), i.e. a 1/128 change
 * of those terms of the dot product.  qat_sym_fwd with QAT_CODES_I16 returns the exact codes.
 */
int qat_qlinear_fused_fwd(const void* x, const void* w, void* out, int8_t* qx, float* ex, uint8_t* mx,
                          int8_t* qw, float* ew, uint8_t* mw, int64_t T, int64_t N, int64_t K, int dtype,
                          int a_bits, int w_bits, float clip_lo, float clip_hi, int reuse_x, int reuse_w,
                          void* stream);

/*
 * The GEMM feed of a [rows, cols] tensor alone — what qat_qlinear_fused_fwd runs on each operand:
 * SymQuantizer's codes (int8), dequant divisors e = fl(s + 1e-6) (NaN for a row whose abs-max is inf, so
 * that the contraction returns NaN like the reference) and the packed STE mask (may be NULL).  Used to
 * quantize a weight by output-channel shard: rows are independent, so a row range of W gives the same
 * bits as the same rows of the full call (BASELINE configs[4]).
 */
int qat_sym_feed(const void* x, int8_t* codes, float* row_e, uint8_t* mask, float clip_lo, float clip_hi,
                 int64_t rows, int64_t cols, int dtype, int bits, void* stream);

/*
 * Rebuild the fake-quantized tensor from K1's int8 codes and row divisors:
 * out[r,c] = fl(codes[r,c] / row_e[r]) — bit-identical to qat_sym_fwd's y
 * (utils_quant.py:72) wherever the int8 feed did not saturate.  cols % 16 == 0.
 * Used by QuantizeLinear's backward for the dgrad / wgrad operands.
 */
int qat_dequant_codes(const int8_t* codes, const float* row_e, void* out, int64_t rows, int64_t cols,
                      int dtype, void* stream);

/*
 * QuantizeLinear backward contractions — what autograd runs for utils_quant.py:250
 * (two cuBLAS GEMMs) with the STE clip mask of utils_quant.py:83-87 fused into the epilogue.
 *   out[m, n] = pass(m, n) * sum_k A(m, k) * B(n, k)          bf16 operands, fp32 accumulation
 * a_mn_major = 0: A is row-major [M, K];  1: A is row-major [K, M]   (read in place, no transpose)
 * b_mn_major = 0: B is row-major [N, K];  1: B is row-major [K, N]
 *   dgrad  gx[T,K] = g[T,N] . Wq[N,K]    -> M=T, N=K_in, K=N_out, a_mn_major=0, b_mn_major=1
 *   wgrad  gw[N,K] = g[T,N]^T . xq[T,K]  -> M=N_out, N=K_in, K=T, a_mn_major=1, b_mn_major=1
 * mask (optional): packed pass-mask over the flattened [M, N] output, bit i%8 of byte i/8 (what
 * qat_sym_fwd emits); masked-out elements are written as 0.  out: bf16 or fp32 per out_dtype.
 * The contiguous dimension of each operand must be a multiple of 8 elements (TMA pitch).
 * cta_group: 0 = choose, 1 = 128x256 tiles, 2 = CTA pairs on 256x256 tiles.
 * tcgen05.mma kind::f16, TMEM accumulators, TMA-fed (MN-major shared-memory descriptors).
 */
int qat_gemm_bf16(const void* a, const void* b, void* out, const uint8_t* mask, int64_t M, int64_t N,
                  int64_t K, int a_mn_major, int b_mn_major, int out_dtype, int cta_group, void* stream);

/*
 * Fused causal attention on tcgen05 — replaces the eager block of
 * models/modeling_llama_quant.py:352-377 (QK^T / sqrt(d), + mask, max(finfo.min), fp32 softmax,
 * cast, . V) and its autograd backward, for the causal mask of :60-92; no [b, h, s, s] tensor is
 * materialised.  K and V are consumed as the K/V fake-quant (:320-327) and RoPE left them.
 *   q, k, v, o, d_o, dq, dk, dv : bf16 [B, S, H, head_dim] (== [b, s, hidden] of the projections), head_dim == 128
 *   lse   : fp32 [B, H, S], natural-log sum-exp of the scaled scores (saved for backward; may be NULL in fwd)
 *   delta : fp32 [B, H, S] scratch of the backward (rowsum(dO * O))
 *   causal != 0: key j is visible to query i iff j <= i;  0: every key is visible
 * Scores, softmax and accumulation are fp32; P is rounded to bf16 before P.V like the reference's
 * `.to(query_states.dtype)`.  Agreement with the eager chain: <= 1e-2 relative (bf16).
 */
int qat_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int B, int S, int H,
                 int head_dim, float softmax_scale, int causal, void* stream);
/* Test hook: clock64() trace of one CTA of the forward kernel (3 roles x 16 tiles x 8 events, int64). */
int qat_attn_debug_trace(long long* dev_buffer);
int qat_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                 float* delta, void* dq, void* dk, void* dv, int B, int S, int H, int head_dim,
                 float softmax_scale, int causal, void* stream);

/*
 * Logit-distillation loss — utils/kd_trainer.py:42-48:
 *   loss = KLDivLoss(reduction="batchmean")(log_softmax(student, dim=2), softmax(teacher, dim=2))
 *        = (1 / batch) * sum over rows and vocabulary of p_t (log p_t - log q_s),   fp32 arithmetic.
 * student / teacher: [rows, V] logits (rows = batch * seq), fp32 or bf16 per `dtype`.
 * fwd: loss (1 float), row_kl [rows] and row_stat [rows * 4] (scratch kept for bwd); one read of both.
 * bwd: grad_student[r, v] = (softmax(student) - softmax(teacher)) * (*grad_loss) / batch, in `dtype`;
 *      grad_loss is a DEVICE float (NULL = 1.0): no host synchronisation.
 * Summation order differs from eager PyTorch's: agreement <= 1e-5 relative on the loss.
 */
int qat_kd_loss_fwd(const void* student, const void* teacher, float* loss, float* row_kl, float* row_stat,
                    int64_t rows, int64_t V, int64_t batch, int dtype, void* stream);
int qat_kd_loss_bwd(const void* student, const void* teacher, const float* row_stat, const float* grad_loss,
                    void* grad_student, int64_t rows, int64_t V, int64_t batch, int dtype, void* stream);

/*
 * Producers of QuantizeLinear's inputs, fused with the per-token fake-quantization of what they produce
 * (bf16 tensors; dtype = QAT_BF16, or QAT_BF16_AMP inside torch.autocast — see above).  codes / row_e / mask
 * are exactly what qat_sym_fwd's GEMM-feed mode emits for the produced tensor (NULL codes: producer only).
 *
 * LlamaRMSNorm.forward — models/modeling_llama_quant.py:121-129:
 *   y = weight * bf16( x * rsqrt(mean(x^2) + eps) );  rstd [rows] (fp32) is kept for the backward.
 * qat_rmsnorm_bwd: grad_x [rows, cols] bf16, grad_weight [cols] bf16 (fixed-order column sums through
 *   `workspace`, qat_rmsnorm_bwd_workspace_bytes).  cols % 8 == 0, cols <= 8192.
 */
int qat_rmsnorm_feed_fwd(const void* x, const void* weight, void* y, float* rstd, int8_t* codes, float* row_e,
                         uint8_t* mask, float clip_lo, float clip_hi, int64_t rows, int64_t cols, float eps,
                         int dtype, int bits, void* stream);
size_t qat_rmsnorm_bwd_workspace_bytes(int64_t rows, int64_t cols);
int qat_rmsnorm_bwd(const void* grad_y, const void* x, const void* weight, const float* rstd, void* grad_x,
                    void* grad_weight, void* workspace, size_t workspace_bytes, int64_t rows, int64_t cols,
                    void* stream);
/*
 * LlamaMLP.forward's act_fn(gate_proj(x)) * up_proj(x) — models/modeling_llama_quant.py:235 (SiLU):
 *   act = bf16(silu(gate)) * up, with the feed of `act` for down_proj.  cols % 8 == 0, cols <= 16384.
 * qat_swiglu_bwd: elementwise, n = number of elements (multiple of 8).
 */
int qat_swiglu_feed_fwd(const void* gate, const void* up, void* act, int8_t* codes, float* row_e, uint8_t* mask,
                        float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype, int bits, void* stream);
int qat_swiglu_bwd(const void* grad_act, const void* gate, const void* up, void* grad_gate, void* grad_up, int64_t n,
                   void* stream);
/*
 * The K/V fake-quant call site and the rotary embedding in one launch —
 * models/modeling_llama_quant.py:320-341: key / value = SymQuantizer.apply(k_proj / v_proj output,
 * [-2, 2], kv_bits, False) per token over all heads' channels (skipped when kv_bits >= 32), then
 * apply_rotary_pos_emb on query and key (:174-196).  q, k, v and the outputs: bf16 [tokens, heads * 128];
 * cos_table / sin_table: fp32 [max_pos, 128] (LlamaRotaryEmbedding's caches); position_ids int64 [tokens]:
 * negative ids count from the end of the table like the reference's `cos[position_ids]`, ids >= max_pos (an
 * IndexError there) are clamped to the last row — no launch reads outside the tables.
 * k_mask / v_mask receive the packed STE pass-masks of the unquantized K / V.  The fake-quantized values
 * are bit-identical to qat_sym_fwd's (same chain); under QAT_BF16_AMP K is rotated in fp32 and rounded
 * once to bf16, as autocast's matmul cast does.
 * qat_qkv_prep_bwd: gradients of the three inputs from those of the three outputs (RoPE transpose, STE masks).
 */
int qat_qkv_prep_fwd(const void* q, const void* k, const void* v, void* q_out, void* k_out, void* v_out,
                     uint8_t* k_mask, uint8_t* v_mask, const float* cos_table, const float* sin_table,
                     const int64_t* position_ids, int64_t max_pos, int64_t tokens, int heads, int head_dim,
                     int kv_bits, float clip_lo, float clip_hi, int dtype, void* stream);
int qat_qkv_prep_bwd(const void* dq_rot, const void* dk_rot, const void* dv_q, const uint8_t* k_mask,
                     const uint8_t* v_mask, const float* cos_table, const float* sin_table,
                     const int64_t* position_ids, int64_t max_pos, void* dq, void* dk, void* dv, int64_t tokens,
                     int heads, int head_dim, void* stream);

/* Host-buffer convenience entry points (pinned or pageable host memory):
 * copy in, run, copy out on `stream`; `dev_scratch` must hold
 * qat_host_scratch_bytes(...) bytes of device memory. */
size_t qat_host_scratch_bytes(int64_t rows, int64_t cols, int dtype, int with_backward);
int qat_sym_fwd_bwd_host(const void* x_host, const void* g_host, void* y_host, void* gx_host,
                         float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                         int bits, void* dev_scratch, size_t dev_scratch_bytes, void* stream);
int qat_asym_fwd_bwd_host(const void* x_host, const void* g_host, void* y_host, void* gx_host,
                          float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                          int bits, void* dev_scratch, size_t dev_scratch_bytes, void* stream);

/*
 * Device self-test of the hoisted-reciprocal divisions K1/K2 use in place of a
 * per-element div.rn (see csrc/common.cuh): `rows` random divisors, `per_row`
 * numerators each.  dev_counters[6] (caller-zeroed device u64):
 * {general-numerator mismatches, tested}  divisor in [2^-27, 2^100] (the Asym
 *                                         row guard), quotient in [2^-41, 1];
 * {integer-code mismatches, tested}       |q| <= 32767, divisor in [2^-100, 2^100];
 * {wide-domain mismatches, tested}        informational: numerators down to the
 *                                         denormal boundary, outside what the
 *                                         kernels rely on.
 */
int qat_selftest_fastdiv(uint64_t seed, int64_t rows, int per_row, int bf16_operands,
                         uint64_t* dev_counters, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* QAT_B200_H_ */
