"""ctypes binding of libqat_b200.so (the C ABI declared in include/qat_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is
missing, or a kernel call fails, this raises.  ``check(rc)`` turns a non-zero
return code into ``RuntimeError`` with the library's thread-local message.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "lib", "libqat_b200.so")

QAT_F32, QAT_BF16, QAT_BF16_AMP, QAT_BF16_AMP_CAST = 0, 1, 2, 3
CODES_NONE, CODES_I8, CODES_I16 = 0, 1, 2
ERR_UNSUPPORTED = 1002

_lib = None


def _declare(lib):
    P, I, L, F, Z = c_void_p, c_int, c_int64, c_float, c_size_t
    sig = {
        "qat_version": (I, []),
        "qat_last_error": (c_char_p, []),
        "qat_launch_count": (c_uint64, []),
        "qat_check_device": (I, []),
        "qat_fwd_workspace_bytes": (Z, [L, L, I]),
        # x, y, codes, codes_kind, st0, st1, mask, lo, hi, rows, cols, dtype, bits, ws, ws_bytes, stream
        "qat_sym_fwd": (I, [P, P, P, I, P, P, P, F, F, L, L, I, I, P, Z, P]),
        "qat_asym_fwd": (I, [P, P, P, I, P, P, P, F, F, L, L, I, I, P, Z, P]),
        # g, x, gx, mask_out, lo, hi, n, dtype, stream
        "qat_ste_bwd": (I, [P, P, P, P, F, F, L, I, P]),
        # g, x, gx, mask_out, clip_dev, n, dtype, stream
        "qat_ste_bwd_devclip": (I, [P, P, P, P, P, L, I, P]),
        # g, mask, gx, n, dtype, stream
        "qat_ste_bwd_from_mask": (I, [P, P, P, L, I, P]),
        "qat_lowbit_workspace_bytes": (Z, [L, I]),
        # w, w_eff, rows, cols, dtype, w_bits, layerwise, ws, ws_bytes, stream
        "qat_lowbit_weight_fwd": (I, [P, P, L, L, I, I, I, P, Z, P]),
        # qx, qw, ex, ew, out, T, N, K, out_dtype, stream
        "qat_qlinear_i8_fwd": (I, [P, P, P, P, P, L, L, L, I, P]),
        "qat_set_gemm_cta_group": (I, [I]),
        "qat_set_pdl": (I, [I]),
        "qat_set_asym_div": (I, [I]),
        # x, codes, row_e, mask, lo, hi, rows, cols, dtype, bits, stream
        "qat_sym_feed": (I, [P, P, P, P, F, F, L, L, I, I, P]),
        # seed, rows, per_row, bf16_operands, dev_counters, stream
        "qat_selftest_fastdiv": (I, [c_uint64, L, I, I, P, P]),
        # x, w, out, qx, ex, mx, qw, ew, mw, T, N, K, dtype, a_bits, w_bits, lo, hi, reuse_x, reuse_w, stream
        "qat_qlinear_fused_fwd": (I, [P, P, P, P, P, P, P, P, P, L, L, L, I, I, I, F, F, I, I, P]),
        # codes, row_e, out, rows, cols, dtype, stream
        "qat_dequant_codes": (I, [P, P, P, L, L, I, P]),
        # a, b, out, mask, M, N, K, a_mn, b_mn, out_dtype, cta_group, stream
        "qat_gemm_bf16": (I, [P, P, P, P, L, L, L, I, I, I, I, P]),
        # q, k, v, o, lse, B, S, H, D, scale, causal, stream
        "qat_attn_fwd": (I, [P, P, P, P, P, I, I, I, I, F, I, P]),
        # q, k, v, o, do, lse, delta, dq, dk, dv, B, S, H, D, scale, causal, stream
        "qat_attn_bwd": (I, [P, P, P, P, P, P, P, P, P, P, I, I, I, I, F, I, P]),
        # student, teacher, loss, row_kl, row_stat, rows, V, batch, dtype, stream
        "qat_kd_loss_fwd": (I, [P, P, P, P, P, L, L, L, I, P]),
        # student, teacher, row_stat, grad_loss, grad_student, rows, V, batch, dtype, stream
        "qat_kd_loss_bwd": (I, [P, P, P, P, P, L, L, L, I, P]),
        # x, w, y, rstd, codes, row_e, mask, lo, hi, rows, cols, eps, dtype, bits, stream
        "qat_rmsnorm_feed_fwd": (I, [P, P, P, P, P, P, P, F, F, L, L, F, I, I, P]),
        "qat_rmsnorm_bwd_workspace_bytes": (Z, [L, L]),
        # gy, x, w, rstd, gx, gw, ws, ws_bytes, rows, cols, stream
        "qat_rmsnorm_bwd": (I, [P, P, P, P, P, P, P, Z, L, L, P]),
        # gate, up, act, codes, row_e, mask, lo, hi, rows, cols, dtype, bits, stream
        "qat_swiglu_feed_fwd": (I, [P, P, P, P, P, P, F, F, L, L, I, I, P]),
        # g, gate, up, d_gate, d_up, n, stream
        "qat_swiglu_bwd": (I, [P, P, P, P, P, L, P]),
        # q, k, v, qo, ko, vo, kmask, vmask, cos, sin, pos, tokens, heads, head_dim, kv_bits, lo, hi, dtype, stream
        "qat_qkv_prep_fwd": (I, [P, P, P, P, P, P, P, P, P, P, P, L, L, I, I, I, F, F, I, P]),
        # dq_rot, dk_rot, dv_q, kmask, vmask, cos, sin, pos, dq, dk, dv, tokens, heads, head_dim, stream
        "qat_qkv_prep_bwd": (I, [P, P, P, P, P, P, P, P, L, P, P, P, L, I, I, P]),
        "qat_attn_debug_trace": (I, [P]),
        "qat_host_scratch_bytes": (Z, [L, L, I, I]),
        # x_host, g_host, y_host, gx_host, lo, hi, rows, cols, dtype, bits, scratch, scratch_bytes, stream
        "qat_sym_fwd_bwd_host": (I, [P, P, P, P, F, F, L, L, I, I, P, Z, P]),
        "qat_asym_fwd_bwd_host": (I, [P, P, P, P, F, F, L, L, I, I, P, Z, P]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale: fail loudly
        fn.restype = res
        fn.argtypes = args
    return sig


# Programmatic dependent launch x CUPTI.  With a CUPTI activity trace attached (torch.profiler / kineto),
# a stream of PDL launches of this library's persistent one-CTA-per-SM kernels can stop making progress:
# tests/gpu_pdl_profiler_soak.py reproduces it on B200 / driver 580 (1 of 20 traces of a decoder layer's
# fwd+bwd never returned from cudaDeviceSynchronize with PDL forced on; 0 of 20 with plain stream order;
# never without a tracer).  PDL buys ~1.5 us per launch and nothing else, so it is switched off for as long
# as a torch profiler is active (checked on every entry to lib(): one C++ bool read) and when the process
# was started under an injected profiler (Nsight Systems / Compute set CUDA_INJECTION64_PATH).
# QAT_B200_PDL=0 always off, =force never auto-disabled (what the soak tool uses to reproduce the hang).
_pdl_mode = os.environ.get("QAT_B200_PDL", "1").strip().lower()
_pdl_user_on = _pdl_mode != "0"
_pdl_auto = _pdl_user_on and _pdl_mode != "force"
_pdl_suppressed = False
_INJECTED = any(os.environ.get(k) for k in ("CUDA_INJECTION64_PATH", "NSYS_PROFILING_SESSION_ID",
                                             "NV_COMPUTE_PROFILER_PERFWORKS_DIR"))
try:
    from torch.autograd import _profiler_enabled as _torch_profiler_enabled
except Exception:  # pragma: no cover - torch without the symbol
    def _torch_profiler_enabled():
        return False


def _sync_pdl_with_profiler(handle) -> None:
    global _pdl_suppressed
    want_off = _INJECTED or _torch_profiler_enabled()
    if want_off != _pdl_suppressed:
        handle.qat_set_pdl(0 if want_off else 1)
        _pdl_suppressed = want_off


def lib():
    """The loaded library; raises ImportError with build instructions if absent."""
    global _lib
    if _lib is not None:
        if _pdl_auto:
            _sync_pdl_with_profiler(_lib)
        return _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing. Build it with `python llm-qat_b200/build.py` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
                "llm-qat_b200 has no CPU or PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        _declare(handle)
        if _pdl_mode == "force":
            handle.qat_set_pdl(1)
        _lib = handle
        if _pdl_auto:
            _sync_pdl_with_profiler(_lib)
    return _lib


def exported_symbols():
    """Names the header declares and the binding expects (used by the CPU tests)."""
    return list(_declare(lib()).keys())


def last_error() -> str:
    msg = lib().qat_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, what: str = "libqat_b200") -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")


def launch_count() -> int:
    return int(lib().qat_launch_count())
