"""Drop-in replacement for the reference's ``models/utils_quant.py``.

Same three public names, same signatures, no new parameters or buffers:

* ``SymQuantizer.apply(input, clip_val, num_bits, layerwise)``   (reference utils_quant.py:31-87)
* ``AsymQuantizer.apply(input, clip_val, num_bits, layerwise)``  (reference utils_quant.py:90-162)
* ``QuantizeLinear(in, out, symmetric=True, bias=False, w_bits=32, a_bits=32,
  act_layerwise=False, weight_layerwise=False)``                 (reference utils_quant.py:165-254)

Every tensor op of the reference's eager chains runs here as one hand-written
sm_100a kernel reached through the C ABI in ``include/qat_b200.h``.  Inputs must
be CUDA tensors (fp32 or bf16): there is no CPU fallback.

Install under the reference's import name before its model file is imported::

    import llm_qat_b200; llm_qat_b200.install()      # sys.modules["models.utils_quant"] = this module
    from models.modeling_llama_quant import LlamaForCausalLM

Run-time knobs (environment; signatures stay the reference's):
  QAT_B200_CACHE=0|1|2        1 (default): a module's weight codes are reused only by the checkpoint
                              recompute of the SAME step (forward re-entered from inside a backward
                              pass — weights cannot have changed), and q/k/v (gate/up) share the codes
                              of their common input tensor.  2: weights are frozen (evaluation, gradient
                              accumulation): also reuse across plain forwards, keyed on the parameter's
                              (data_ptr, _version) — NOT safe under wrappers that rewrite parameter
                              storage behind that key (FSDP use_orig_params=True).  0: no reuse.
  QAT_B200_WEIGHT_REUSE=0|1   0: never keep a module's weight codes between its forward and its
                              backward (1.125 B per weight element per live layer — under FSDP
                              full_shard that is unsharded memory); q/k/v and gate/up still share
                              their activation codes.  Default 1.
  QAT_B200_FUSED_LINEAR=0|1   QuantizeLinear uses the integer-grid tcgen05 GEMM (default 1, taken
                              when shapes/dtypes allow) or the fake-quant kernels + F.linear (0).
                              The int8 operand feed holds codes in [-128, 127]: a plain-bf16 (no
                              autocast) 8-bit activation row whose largest element rounds to the code
                              +128 (bf16 arithmetic can produce it, fp32 and the autocast chain cannot)
                              carries 127 for that element — at most the row's maxima, a 1/128 change of
                              one term of the dot product.  0 gives the reference's operands exactly.
  QAT_B200_ASYM_DIV=cpu|cuda  AsymQuantizer's `.div(S)` (utils_quant.py:146): "cpu" (default) is the true
                              division torch's CPU kernel performs (BASELINE configs[0] names torch CPU);
                              "cuda" multiplies by fl(1/S) like ATen's CUDA kernel for a Python-scalar
                              divisor, reproducing the reference's eager-GPU bits for fp32 tensors
                              (bf16 results are identical under both).
"""
from __future__ import annotations

import os
import weakref

import torch
import torch.nn as nn

from . import _lib
from . import sharding as _sharding
from ._lib import CODES_I8, CODES_I16, CODES_NONE, QAT_BF16, QAT_BF16_AMP, QAT_BF16_AMP_CAST, QAT_F32, check

__all__ = ["SymQuantizer", "AsymQuantizer", "QuantizeLinear"]

_DTYPES = {torch.float32: QAT_F32, torch.bfloat16: QAT_BF16}


# ------------------------------------------------------------------ helpers
def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"llm-qat_b200 kernels take float32 or bfloat16 tensors, got {t.dtype}") from None


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{what}: expected a CUDA tensor, got device {t.device}. "
            "llm-qat_b200 runs only on B200 (sm_100a); there is no CPU fallback.")


def _sym_amp(t: torch.Tensor) -> bool:
    """SymQuantizer on a bf16 CUDA tensor inside torch.autocast (HF's Trainer runs the step in one,
    kd_trainer.py:106): autocast executes the reference's `Q / (max + 1e-6)` — a reciprocal — in fp32,
    so everything after it is fp32 and the fake-quantized tensor comes back as float32
    (tests/gpu_autocast_probe.py).  The kernels reproduce that chain as dtype QAT_BF16_AMP.
    AsymQuantizer contains no op autocast touches and is unchanged."""
    return t.dtype == torch.bfloat16 and t.is_cuda and torch.is_autocast_enabled("cuda")


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NO_GUARD = _NoGuard()


def _on(device):
    """Device guard for a launch: free when ``device`` is already current (the
    usual case — torch.cuda.device() costs ~10 us of host time per use)."""
    if device.index is None or torch.cuda.current_device() == device.index:
        return _NO_GUARD
    return torch.cuda.device(device)


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _clip_bounds(clip_val):
    """(lo, hi) as python floats.  The reference reads clip_val[0]/[1] as 0-dim
    tensors in backward (utils_quant.py:85-86); a CPU clip tensor (the only kind
    the model creates, :198,245) costs no device sync."""
    if isinstance(clip_val, torch.Tensor):
        lo, hi = clip_val.detach().reshape(-1)[:2].tolist()
        return float(lo), float(hi)
    lo, hi = clip_val
    return float(lo), float(hi)


def _reduction_view(input: torch.Tensor, layerwise: bool):
    """(rows, cols) with one row per reduction set — utils_quant.py:50-70."""
    if layerwise:
        return 1, input.numel()
    nd = input.dim()
    if nd <= 3:
        cols = input.shape[-1] if nd >= 1 else 1
        return (input.numel() // cols if cols else 0), cols
    if nd == 4:
        # the reference does input.view(d0, d1, -1): raise like it does when not viewable
        input.view(input.shape[0], input.shape[1], -1)
        return input.shape[0] * input.shape[1], input.shape[2] * input.shape[3]
    raise ValueError


def fake_quant_forward(input: torch.Tensor, num_bits: int, layerwise: bool, symmetric: bool, *,
                       want_y: bool = True, codes_kind: int = CODES_NONE, want_scales: bool = False,
                       mask_clip=None, amp: bool = False, cast: bool = False):
    """One launch of K1/K2 (or the two-phase K5 for long rows).

    Returns ``(y, codes, st0, st1, mask)``; entries not requested are ``None``.
    Sym: st0 = s, st1 = e (dequant divisor).  Asym: st0 = alpha + 1e-8, st1 = beta.
    ``amp`` with ``cast``: y is the autocast chain's fp32 result cast to bf16 (QAT_BF16_AMP_CAST).
    """
    _require_cuda(input, "fake-quant forward")
    dt = _dtype_code(input)
    if amp:
        if not (symmetric and dt == QAT_BF16):
            raise TypeError("the autocast variant exists for SymQuantizer on bfloat16 tensors only")
        dt = QAT_BF16_AMP_CAST if cast else QAT_BF16_AMP
    y_fp32 = amp and not cast
    rows, cols = _reduction_view(input, layerwise)
    if input.numel() == 0:
        # what the reference's torch.max does: an empty reduction set raises (IndexError for
        # max(dim=-1) over zero columns, RuntimeError for the layerwise max() of nothing), but zero
        # ROWS of a non-empty width are simply zero reductions and the result is an empty tensor
        if layerwise:
            raise RuntimeError("max(): Expected reduction dim to be specified for input.numel() == 0. "
                               "Specify the reduction dim with the 'dim' argument.")
        if cols == 0:
            raise IndexError("max(): Expected reduction dim to have non-zero size.")
        empty = torch.empty(input.shape, dtype=torch.float32 if y_fp32 else input.dtype, device=input.device)
        return (empty if want_y else None), None, None, None, None
    x = input.detach()
    if not x.is_contiguous():
        x = x.contiguous()
    dev = x.device
    y = (torch.empty(x.shape, dtype=torch.float32, device=dev) if y_fp32 else torch.empty_like(x)) if want_y else None
    codes = None
    if codes_kind == CODES_I8:
        codes = torch.empty(x.shape, dtype=torch.int8 if symmetric else torch.uint8, device=dev)
    elif codes_kind == CODES_I16:
        codes = torch.empty(x.shape, dtype=torch.int16, device=dev)
    st0 = torch.empty(rows, dtype=torch.float32, device=dev) if want_scales else None
    st1 = torch.empty(rows, dtype=torch.float32, device=dev) if want_scales else None
    mask = None
    lo = hi = 0.0
    if mask_clip is not None:
        lo, hi = mask_clip
        mask = torch.empty((x.numel() + 7) // 8, dtype=torch.uint8, device=dev)
    L = _lib.lib()
    ws_bytes = L.qat_fwd_workspace_bytes(rows, cols, dt)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
    fn = L.qat_sym_fwd if symmetric else L.qat_asym_fwd
    with _on(dev):
        rc = fn(x.data_ptr(), _ptr(y), _ptr(codes), codes_kind, _ptr(st0), _ptr(st1), _ptr(mask),
                lo, hi, rows, cols, dt, int(num_bits), _ptr(ws), ws_bytes, _stream_ptr(dev))
    check(rc, "qat_sym_fwd" if symmetric else "qat_asym_fwd")
    return y, codes, st0, st1, mask


def ste_backward(grad_output: torch.Tensor, input: torch.Tensor, clip_val, *, want_mask: bool = False):
    """K3: gx = g where clip[0] < x < clip[1] else 0 — utils_quant.py:83-87."""
    _require_cuda(grad_output, "STE backward")
    _require_cuda(input, "STE backward")
    if grad_output.dtype != input.dtype:
        raise TypeError(f"STE backward: grad dtype {grad_output.dtype} != input dtype {input.dtype}")
    if grad_output.shape != input.shape:
        raise RuntimeError(f"STE backward: grad shape {tuple(grad_output.shape)} != input shape {tuple(input.shape)}")
    dt = _dtype_code(input)
    g = grad_output if grad_output.is_contiguous() else grad_output.contiguous()
    x = input.detach()
    x = x if x.is_contiguous() else x.contiguous()
    gx = torch.empty_like(g)
    n = g.numel()
    if n == 0:
        return (gx, None) if want_mask else gx
    mask = torch.empty((n + 7) // 8, dtype=torch.uint8, device=g.device) if want_mask else None
    if isinstance(clip_val, torch.Tensor) and clip_val.is_cuda:
        # a CUDA clip_val is read by the kernel: no .item()/.tolist() synchronisation
        clip_dev = clip_val.detach().reshape(-1)[:2].to(device=g.device, dtype=torch.float32).contiguous()
        with _on(g.device):
            rc = _lib.lib().qat_ste_bwd_devclip(g.data_ptr(), x.data_ptr(), gx.data_ptr(), _ptr(mask),
                                                clip_dev.data_ptr(), n, dt, _stream_ptr(g.device))
        check(rc, "qat_ste_bwd_devclip")
        return (gx, mask) if want_mask else gx
    lo, hi = _clip_bounds(clip_val)
    with _on(g.device):
        rc = _lib.lib().qat_ste_bwd(g.data_ptr(), x.data_ptr(), gx.data_ptr(), _ptr(mask), lo, hi, n, dt,
                                    _stream_ptr(g.device))
    check(rc, "qat_ste_bwd")
    return (gx, mask) if want_mask else gx


def ste_backward_from_mask(grad_output: torch.Tensor, mask: torch.Tensor):
    """K3 driven by a forward-emitted packed mask (reads 1/8 B/elem instead of x)."""
    _require_cuda(grad_output, "STE backward")
    dt = _dtype_code(grad_output)
    g = grad_output if grad_output.is_contiguous() else grad_output.contiguous()
    gx = torch.empty_like(g)
    if g.numel() == 0:
        return gx
    with _on(g.device):
        rc = _lib.lib().qat_ste_bwd_from_mask(g.data_ptr(), mask.data_ptr(), gx.data_ptr(), g.numel(), dt,
                                              _stream_ptr(g.device))
    check(rc, "qat_ste_bwd_from_mask")
    return gx


# ------------------------------------------------------------------ quantizers
class SymQuantizer(torch.autograd.Function):
    """Symmetric abs-max fake-quant with STE backward (reference utils_quant.py:31-87)."""

    @staticmethod
    def forward(ctx, input, clip_val, num_bits, layerwise):
        ctx.save_for_backward(input, clip_val)
        y, *_ = fake_quant_forward(input, num_bits, layerwise, symmetric=True, amp=_sym_amp(input))
        return y

    @staticmethod
    def backward(ctx, grad_output):
        input, clip_val = ctx.saved_tensors
        if grad_output.dtype != input.dtype:
            # autocast variant: y (and its gradient) are fp32 while the input is bf16; the reference
            # masks the fp32 gradient and the autograd engine then casts it to the input's dtype —
            # casting first gives the same bits
            grad_output = grad_output.to(input.dtype)
        return ste_backward(grad_output, input, clip_val), None, None, None


class AsymQuantizer(torch.autograd.Function):
    """Min-max asymmetric fake-quant with STE backward (reference utils_quant.py:90-162)."""

    @staticmethod
    def forward(ctx, input, clip_val, num_bits, layerwise):
        ctx.save_for_backward(input, clip_val)
        y, *_ = fake_quant_forward(input, num_bits, layerwise, symmetric=False)
        return y

    @staticmethod
    def backward(ctx, grad_output):
        input, clip_val = ctx.saved_tensors
        return ste_backward(grad_output, input, clip_val), None, None, None


def lowbit_weight(weight: torch.Tensor, w_bits: int, layerwise: bool) -> torch.Tensor:
    """The effective weight (q - w) + w of w_bits in {1, 2} (reference utils_quant.py:202-242)."""
    _require_cuda(weight, "low-bit weight quant")
    dt = _dtype_code(weight)
    w = weight.detach()
    w = w if w.is_contiguous() else w.contiguous()
    out = torch.empty_like(w)
    rows, cols = w.shape
    L = _lib.lib()
    ws_bytes = int(L.qat_lowbit_workspace_bytes(rows, int(bool(layerwise))))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=w.device)
    with _on(w.device):
        rc = L.qat_lowbit_weight_fwd(w.data_ptr(), out.data_ptr(), rows, cols, dt, int(w_bits),
                                     int(bool(layerwise)), _ptr(ws), ws_bytes, _stream_ptr(w.device))
    check(rc, "qat_lowbit_weight_fwd")
    return out


class _LowBitWeight(torch.autograd.Function):
    """w_bits in {1, 2}: forward value (q - w) + w, identity gradient
    (reference utils_quant.py:202-242)."""

    @staticmethod
    def forward(ctx, weight, w_bits, layerwise):
        return lowbit_weight(weight, w_bits, layerwise)

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output, None, None


# ------------------------------------------------------------------ fused linear
# longest row qat_sym_fwd handles without a workspace (register-resident: 8192 16-byte vectors of
# fp32; bf16 rows could be twice as long — the smaller bound keeps one rule)
_MAX_FEED_COLS = 32768


def _fused_linear_enabled() -> bool:
    return os.environ.get("QAT_B200_FUSED_LINEAR", "1") != "0"


def _cache_mode() -> int:
    v = os.environ.get("QAT_B200_CACHE", "1")
    return 0 if v == "0" else 2 if v == "2" else 1


def _weight_reuse_enabled() -> bool:
    return os.environ.get("QAT_B200_WEIGHT_REUSE", "1") != "0"


def _in_backward_pass() -> bool:
    """True while autograd is executing a backward graph on this thread — i.e. this
    forward is a gradient-checkpoint recompute (torch.utils.checkpoint, reentrant or
    not).  Parameters are only updated between backward passes, so codes produced by
    the step's original forward are still those of the current weights."""
    return torch._C._current_graph_task_id() != -1


def _feed_layout(rows: int, cols: int):
    """Byte offsets of (codes int8 [rows, cols], divisors f32 [rows], packed mask) in one blob."""
    n = rows * cols
    off_e = (n + 255) & ~255
    off_m = off_e + ((rows * 4 + 255) & ~255)
    return off_e, off_m, off_m + (n + 7) // 8


def _feed_views(blob: torch.Tensor, rows: int, cols: int):
    off_e, off_m, total = _feed_layout(rows, cols)
    codes = blob[: rows * cols].view(torch.int8).view(rows, cols)
    e = blob[off_e: off_e + rows * 4].view(torch.float32)
    mask = blob[off_m: total]
    return codes, e, mask


# Single-slot memo of the last quantized activation per device: q/k/v (and gate/up)
# receive the very same tensor OBJECT, so its codes are produced once (SURVEY.md
# 8f-2).  A hit needs that identity (weak reference: a live tensor object keeps its
# storage) plus an unchanged data_ptr and _version.  The slot holds only the codes
# blob, never the activation, and is dropped by the first backward of the step.
_ACT_SLOT: dict = {}


def register_activation_feed(y: torch.Tensor, blob: torch.Tensor, rows: int, cols: int, dt: int, bits: int) -> None:
    """A producer kernel (fused_ops.rmsnorm / swiglu) already emitted the codes of ``y``: publish them in
    the activation slot so the QuantizeLinear layers that receive this very tensor object reuse them
    (SURVEY.md 8(f)-3) — same key a consumer would have stored after quantizing ``y`` itself."""
    dev = y.device
    key = (y.data_ptr(), y._version, rows, cols, dt, bits, _stream_ptr(dev))
    _ACT_SLOT[dev.index] = (key, None, blob, weakref.ref(y))


class _QuantLinearFn(torch.autograd.Function):
    """QuantizeLinear main path (3 <= w_bits <= 8, 3 <= a_bits <= 8, symmetric,
    per-row scales) on the integer grid — reference utils_quant.py:197-201,244-250.

    forward : ONE C call: K1 codes-only passes (int8 codes + row divisors + packed
              STE masks) -> tcgen05 int8 GEMM with the dual-scale epilogue (K4).
              The weight's codes are kept on the module and reused by the
              gradient-checkpoint recompute of the same step (see QAT_B200_CACHE).
    backward: dequantized operands are rebuilt from codes (q / e, bit-identical
              to the reference's fake-quant outputs); dgrad / wgrad run on this
              library's tcgen05 bf16 GEMM, which reads them in place (MN-major) and
              applies the STE masks saved by the forward in its epilogue.
    Saves 1 B/elem of codes + 1/8 B/elem of mask instead of the reference's two
    dequantized tensors plus two unquantized inputs.
    """

    @staticmethod
    def forward(ctx, input, weight, w_bits, a_bits, owner):
        K = input.shape[-1]
        N = weight.shape[0]
        if weight.dim() != 2 or weight.shape[1] != K:
            raise RuntimeError(f"QuantizeLinear: input features {K} do not match weight {tuple(weight.shape)}")
        x2 = input.detach()
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        w = weight.detach()
        if not w.is_contiguous():
            w = w.contiguous()
        T = x2.numel() // K
        dev = x2.device
        dt = QAT_BF16_AMP if _sym_amp(x2) else _DTYPES[x2.dtype]   # codes from the autocast chain under autocast
        stream = _stream_ptr(dev)
        mode = _cache_mode()

        xkey = (x2.data_ptr(), input._version, T, K, dt, a_bits, stream)
        slot = _ACT_SLOT.get(dev.index) if mode else None
        if slot is not None and slot[0] == xkey and slot[3]() is input:
            xblob, reuse_x = slot[2], 1
        else:
            xblob, reuse_x = torch.empty(_feed_layout(T, K)[2], dtype=torch.uint8, device=dev), 0
        wkey = (w.data_ptr(), weight._version, N, K, dt, w_bits, stream)
        cached = None
        if owner is not None and (mode == 2 or (mode == 1 and _in_backward_pass())):
            cached = getattr(owner, "_qat_wfeed", None)
        if cached is not None and cached[0] == wkey:
            wblob, reuse_w = cached[1], 1
        else:
            wblob, reuse_w = torch.empty(_feed_layout(N, K)[2], dtype=torch.uint8, device=dev), 0

        out = torch.empty((T, N), dtype=x2.dtype, device=dev)
        xe, xm, _ = _feed_layout(T, K)
        we, wm, _ = _feed_layout(N, K)
        xb, wb = xblob.data_ptr(), wblob.data_ptr()
        if not reuse_w:
            # never from inside a backward pass: a checkpoint recompute that missed the cache must not
            # interleave a collective with DDP's gradient all-reduces (rank-dependent order -> deadlock)
            sh = None if _in_backward_pass() else _sharding.weight_sharding()
            if sh is not None and _sharding.shardable(N, K, sh[1]):
                # BASELINE configs[4]: this rank quantizes its out/world output channels, then the codes,
                # divisors and masks (1.125 B/elem) are all-gathered over NVLink
                group, world, rank = sh
                n = N // world
                with _on(dev):
                    check(_lib.lib().qat_sym_feed(w.data_ptr() + rank * n * K * w.element_size(),
                                                  wb + rank * n * K, wb + we + rank * n * 4, wb + wm + rank * n * K // 8,
                                                  -2.0, 2.0, n, K, dt, int(w_bits), stream), "qat_sym_feed")
                _sharding.all_gather_feed(wblob, N, K, group, world, rank)
                reuse_w = 1
        with _on(dev):
            rc = _lib.lib().qat_qlinear_fused_fwd(
                x2.data_ptr(), w.data_ptr(), out.data_ptr(), xb, xb + xe, xb + xm, wb, wb + we, wb + wm,
                T, N, K, dt, int(a_bits), int(w_bits), -2.0, 2.0,  # clip: utils_quant.py:198,245
                reuse_x, reuse_w, stream)
        check(rc, "qat_qlinear_fused_fwd")
        if mode:
            _ACT_SLOT[dev.index] = (xkey, None, xblob, weakref.ref(input))
            # Weight codes are kept on the module only when a consumer can follow: a gradient-
            # checkpoint recompute of this step (mode 1: the module is training; cleared by its own
            # backward) or any later forward of frozen weights (mode 2).  Evaluation / no_grad
            # inference in mode 1 keeps nothing.
            if owner is not None and _weight_reuse_enabled() and (mode == 2 or owner.training):
                owner._qat_wfeed = (wkey, wblob)
            elif owner is not None and getattr(owner, "_qat_wfeed", None) is not None:
                owner._qat_wfeed = None
        ctx.save_for_backward(xblob, wblob)
        ctx.owner_ref = weakref.ref(owner) if (owner is not None and mode == 1) else None
        ctx.dims = (T, N, K)
        ctx.in_shape = input.shape
        ctx.dtype = input.dtype
        return out.view(*input.shape[:-1], N)

    @staticmethod
    def backward(ctx, grad_output):
        xblob, wblob = ctx.saved_tensors
        T, N, K = ctx.dims
        g2 = grad_output.reshape(T, N)
        if not g2.is_contiguous():
            g2 = g2.contiguous()
        dev, dtype = g2.device, ctx.dtype
        if g2.dtype != dtype:
            g2 = g2.to(dtype)
        dt = _DTYPES[dtype]
        L = _lib.lib()
        xb, wb = xblob.data_ptr(), wblob.data_ptr()
        xe, xm, _ = _feed_layout(T, K)
        we, wm, _ = _feed_layout(N, K)
        # bf16: both contractions run on this library's tcgen05 kernel (qat_gemm_bf16), reading the
        # operands where they lie (W_q [N,K] and x_q [T,K] as MN-major B, g [T,N] as K-major /
        # MN-major A) with the STE pass-mask applied to the fp32 accumulator in the epilogue.
        # fp32 modules keep the library GEMM + mask kernel.
        own = dtype == torch.bfloat16 and N % 8 == 0 and K % 8 == 0 and g2.data_ptr() % 16 == 0
        # The operands are rebuilt from the codes by one streaming pass each (qat_dequant_codes, 25 us for
        # [11008, 4096]).  QAT_B200_BWD_DEQUANT_PASS=0 selects the variant that rebuilds them INSIDE the GEMM
        # (converter warps, no dequantized tensor in HBM): bit-identical, but measured 2.1-2.5x slower at
        # T = 2048 (336 vs 133 + 25 us for dgrad [2048 x 11008] x [11008 x 4096]) — every weight tile is converted
        # T / 256 times instead of once and the converters, not the tensor pipe, pace the k-loop.
        from_codes = own and K % 16 == 0 and os.environ.get("QAT_B200_BWD_DEQUANT_PASS", "1") == "0"
        gx = gw = None
        with _on(dev):
            stream = _stream_ptr(dev)
            if ctx.needs_input_grad[0]:
                if from_codes:
                    gx = torch.empty((T, K), dtype=dtype, device=dev)
                    check(L.qat_gemm_bf16_codes(g2.data_ptr(), wb, wb + we, gx.data_ptr(), xb + xm, T, K, N, 0, dt, 0,
                                                stream), "qat_gemm_bf16_codes (dgrad)")
                else:
                    wq = torch.empty((N, K), dtype=dtype, device=dev)       # == the reference's fake-quant W
                    check(L.qat_dequant_codes(wb, wb + we, wq.data_ptr(), N, K, dt, stream), "qat_dequant_codes")
                    if own:
                        gx = torch.empty((T, K), dtype=dtype, device=dev)
                        check(L.qat_gemm_bf16(g2.data_ptr(), wq.data_ptr(), gx.data_ptr(), xb + xm, T, K, N, 0, 1,
                                              dt, 0, stream), "qat_gemm_bf16 (dgrad)")
                    else:
                        t = torch.mm(g2, wq)
                        gx = torch.empty_like(t)
                        check(L.qat_ste_bwd_from_mask(t.data_ptr(), xb + xm, gx.data_ptr(), T * K, dt, stream),
                              "qat_ste_bwd_from_mask")
                    del wq
                gx = gx.view(ctx.in_shape)
            if ctx.needs_input_grad[1]:
                if from_codes:
                    gw = torch.empty((N, K), dtype=dtype, device=dev)
                    check(L.qat_gemm_bf16_codes(g2.data_ptr(), xb, xb + xe, gw.data_ptr(), wb + wm, N, K, T, 1, dt, 0,
                                                stream), "qat_gemm_bf16_codes (wgrad)")
                else:
                    xq = torch.empty((T, K), dtype=dtype, device=dev)       # == the reference's fake-quant x
                    check(L.qat_dequant_codes(xb, xb + xe, xq.data_ptr(), T, K, dt, stream), "qat_dequant_codes")
                    if own:
                        gw = torch.empty((N, K), dtype=dtype, device=dev)
                        check(L.qat_gemm_bf16(g2.data_ptr(), xq.data_ptr(), gw.data_ptr(), wb + wm, N, K, T, 1, 1,
                                              dt, 0, stream), "qat_gemm_bf16 (wgrad)")
                    else:
                        t = torch.mm(g2.t(), xq)
                        gw = torch.empty_like(t)
                        check(L.qat_ste_bwd_from_mask(t.data_ptr(), wb + wm, gw.data_ptr(), N * K, dt, stream),
                              "qat_ste_bwd_from_mask")
                    del xq
        # mode 1 keeps a module's codes only from its forward to its backward (for the checkpoint
        # recompute in between): 1.125 B per weight element must not sit in HBM through the
        # optimizer step
        owner = ctx.owner_ref() if ctx.owner_ref is not None else None
        if owner is not None:
            owner._qat_wfeed = None
        # the shared activation codes are dead once a consumer's backward runs (the step's
        # forwards are over); do not pin the last blob past the step
        _ACT_SLOT.pop(dev.index, None)
        return gx, gw, None, None, None


# ------------------------------------------------------------------ the reference's operands on the own GEMM
# QuantizeLinear off the int8 grid (reference utils_quant.py:190-254): 16-bit activations (W4-A16), weight-only
# QAT (a_bits >= 32, W1/W2 included), activation-only (w_bits >= 32) and 9..31-bit weights.  Wider codes do not
# suit kind::i8 (two MMAs per k-block for 16-bit codes, s32 overflow of the sum), so this route produces the
# exact bf16 operands the reference hands F.linear and contracts them on qat_gemm_bf16, dgrad / wgrad with the
# STE masks in the epilogue.  It differs from the reference only in the order of the fp32 accumulation.
# Taken for modules that fuse_model marked (``_qat_operand_route``); the three kernel calls below are
# module-level functions so that a CPU test can put torch statements in their place.
def quant_operand(t: torch.Tensor, bits: int, amp: bool):
    """(SymQuantizer's output as the bf16 operand of F.linear, packed STE mask for clip [-2, 2]).
    Under autocast: the fp32 chain cast to bf16 in the same pass (QAT_BF16_AMP_CAST)."""
    y, _, _, _, mask = fake_quant_forward(t, bits, False, True, mask_clip=(-2.0, 2.0), amp=amp, cast=amp)
    return y, mask


def lowbit_operand(w: torch.Tensor, bits: int) -> torch.Tensor:
    """w_bits in {1, 2}: the effective weight; its gradient is the identity (no mask)."""
    return lowbit_weight(w, bits, False)


def gemm_bf16(a, b, mask, M: int, N: int, K: int, a_mn_major: int, b_mn_major: int,
              cta_group: int = 0) -> torch.Tensor:
    """out [M, N] bf16 = mask * (A . B^T) on qat_gemm_bf16 (layouts and cta_group: include/qat_b200.h)."""
    out = torch.empty((M, N), dtype=torch.bfloat16, device=a.device)
    with _on(a.device):
        rc = _lib.lib().qat_gemm_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), _ptr(mask), M, N, K,
                                      a_mn_major, b_mn_major, QAT_BF16, cta_group, _stream_ptr(a.device))
    check(rc, "qat_gemm_bf16")
    return out


def _route_device_ok(t: torch.Tensor) -> bool:
    """The route's kernels exist for CUDA tensors only (a CPU test patches this with emulated kernels)."""
    return t.is_cuda


def _stream_key(dev) -> int:
    return _stream_ptr(dev) if dev.type == "cuda" else 0


def operand_route_config(lin) -> bool:
    """The module configurations the operand route serves: symmetric, no layerwise flag, at least one operand
    quantized, both feature counts multiples of 8 (TMA pitch), and not on the int8 grid."""
    w, a = lin.w_bits, lin.a_bits
    quant_x = 2 < a < 32
    return (isinstance(lin, QuantizeLinear)
            and (quant_x or w < 32) and w >= 1
            and not (3 <= w <= 8 and 3 <= a <= 8)
            and (not quant_x or getattr(lin, "act_quantizer", None) is SymQuantizer)
            and not lin.act_layerwise and not lin.weight_layerwise
            and lin.in_features % 8 == 0 and lin.out_features % 8 == 0)


class _OperandLinearFn(torch.autograd.Function):
    """out = x_op . W_op^T with the reference's bf16 operands (see the section comment).

    forward : K1 writes each quantized operand (+ its packed STE mask); W1/W2 weights come from the low-bit
              kernel; an unquantized operand is the tensor itself.  The weight operand is kept for the
              checkpoint recompute like _QuantLinearFn's codes (QAT_B200_CACHE, QAT_B200_WEIGHT_REUSE) and the
              activation operand is shared through the activation slot (q/k/v, gate/up).
    backward: gx = mask_x * (g . W_op), gw = mask_w * (g^T . x_op), both on qat_gemm_bf16.
    """

    @staticmethod
    def forward(ctx, input, weight, w_bits, a_bits, owner):
        K = input.shape[-1]
        N = weight.shape[0]
        x2 = input.detach().reshape(-1, K)
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        w = weight.detach()
        if not w.is_contiguous():
            w = w.contiguous()
        T = x2.shape[0]
        dev = x2.device
        amp = torch.is_autocast_enabled("cuda")
        stream = _stream_key(dev)
        mode = _cache_mode()

        if 2 < a_bits < 32:
            xkey = ("operand", x2.data_ptr(), input._version, T, K, amp, a_bits, stream)
            slot = _ACT_SLOT.get(dev.index) if mode else None
            if slot is not None and slot[0] == xkey and slot[3]() is input:
                xq, xm = slot[2]
            else:
                xq, xm = quant_operand(x2, a_bits, amp)
            if mode:
                _ACT_SLOT[dev.index] = (xkey, None, (xq, xm), weakref.ref(input))
        else:
            xq, xm = x2, None

        if w_bits < 32:
            wkey = ("operand", w.data_ptr(), weight._version, N, K, amp, w_bits, stream)
            cached = None
            if owner is not None and (mode == 2 or (mode == 1 and _in_backward_pass())):
                cached = getattr(owner, "_qat_wfeed", None)
            if cached is not None and cached[0] == wkey:
                wq, wm = cached[1]
            elif w_bits >= 3:
                wq, wm = quant_operand(w, w_bits, amp)
            else:
                wq, wm = lowbit_operand(w, w_bits), None
            if mode:
                if owner is not None and _weight_reuse_enabled() and (mode == 2 or owner.training):
                    owner._qat_wfeed = (wkey, (wq, wm))
                elif owner is not None and getattr(owner, "_qat_wfeed", None) is not None:
                    owner._qat_wfeed = None
        else:
            wq, wm = w, None

        out = gemm_bf16(xq, wq, None, T, N, K, 0, 0)
        ctx.save_for_backward(xq, wq, xm, wm)
        ctx.owner_ref = weakref.ref(owner) if (owner is not None and mode == 1) else None
        ctx.dims = (T, N, K)
        ctx.in_shape = input.shape
        return out.view(*input.shape[:-1], N)

    @staticmethod
    def backward(ctx, grad_output):
        xq, wq, xm, wm = ctx.saved_tensors
        T, N, K = ctx.dims
        g2 = grad_output.reshape(T, N)
        if g2.dtype != torch.bfloat16:
            g2 = g2.to(torch.bfloat16)
        if not g2.is_contiguous() or g2.data_ptr() % 16:
            g2 = g2.contiguous() if not g2.is_contiguous() else g2.clone()
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gx = gemm_bf16(g2, wq, xm, T, K, N, 0, 1).view(ctx.in_shape)
        if ctx.needs_input_grad[1]:
            gw = gemm_bf16(g2, xq, wm, N, K, T, 1, 1)
        owner = ctx.owner_ref() if ctx.owner_ref is not None else None
        if owner is not None:
            owner._qat_wfeed = None
        _ACT_SLOT.pop(g2.device.index, None)
        return gx, gw, None, None, None


def dequant_codes(codes, row_e, dtype):
    """out[r, c] = codes[r, c] / row_e[r] in ``dtype`` (exact IEEE quotient, one rounding)."""
    rows, cols = codes.shape
    out = torch.empty((rows, cols), dtype=dtype, device=codes.device)
    with _on(codes.device):
        rc = _lib.lib().qat_dequant_codes(codes.data_ptr(), row_e.data_ptr(), out.data_ptr(), rows, cols,
                                          _DTYPES[dtype], _stream_ptr(codes.device))
    check(rc, "qat_dequant_codes")
    return out


def qlinear_i8(qx, qw, ex, ew, out_dtype):
    """K4: out[t, n] = (sum_k qx[t,k] qw[n,k]) / (ex[t] * ew[n]) on tcgen05 (kind::i8)."""
    T, K = qx.shape
    N = qw.shape[0]
    out = torch.empty((T, N), dtype=out_dtype, device=qx.device)
    with _on(qx.device):
        rc = _lib.lib().qat_qlinear_i8_fwd(qx.data_ptr(), qw.data_ptr(), ex.data_ptr(), ew.data_ptr(),
                                           out.data_ptr(), T, N, K, _DTYPES[out_dtype], _stream_ptr(qx.device))
    check(rc, "qat_qlinear_i8_fwd")
    return out


# ------------------------------------------------------------------ QuantizeLinear
class QuantizeLinear(nn.Linear):
    """nn.Linear whose weight and input are fake-quantized on every forward
    (reference utils_quant.py:165-254).  State dict == {"weight"}; bias is
    always None (the reference ignores the ``bias`` kwarg, :176)."""

    def __init__(
        self,
        *kargs,
        symmetric=True,
        bias=False,
        w_bits=32,
        a_bits=32,
        act_layerwise=False,
        weight_layerwise=False,
    ):
        super(QuantizeLinear, self).__init__(*kargs, bias=False)
        self.w_bits = w_bits
        self.a_bits = a_bits
        self.act_layerwise = act_layerwise
        self.weight_layerwise = weight_layerwise
        if self.a_bits < 32 and self.a_bits > 2:
            self.act_quantizer = SymQuantizer if symmetric else AsymQuantizer

    def _can_fuse(self, input_: torch.Tensor) -> bool:
        return (
            _fused_linear_enabled()
            and 3 <= self.w_bits <= 8
            and 3 <= self.a_bits <= 8
            and getattr(self, "act_quantizer", None) is SymQuantizer
            and not self.act_layerwise
            and not self.weight_layerwise
            and input_.is_cuda
            and input_.device == self.weight.device   # otherwise let F.linear raise its usual error
            and input_.dtype in _DTYPES
            and input_.dtype == self.weight.dtype
            and 1 <= input_.dim() <= 3
            and input_.shape[-1] % 16 == 0
            and input_.shape[-1] == self.weight.shape[1]   # else F.linear raises its usual shape error
            and input_.shape[-1] <= _MAX_FEED_COLS          # rows the feed kernel keeps in registers
            and input_.numel() > 0
            and input_.data_ptr() % 16 == 0 and self.weight.data_ptr() % 16 == 0
            # under autocast to another dtype the reference's F.linear casts its operands and
            # returns that dtype: leave that case to the unfused path, which does exactly that
            and not (torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") != input_.dtype)
        )

    def _can_route(self, input_: torch.Tensor) -> bool:
        """The operand route (_OperandLinearFn): modules fuse_model marked, bf16 CUDA operands."""
        return (
            self.__dict__.get("_qat_operand_route", False)
            and operand_route_config(self)
            and _route_device_ok(input_)
            and input_.device == self.weight.device
            and input_.dtype == torch.bfloat16
            and self.weight.dtype == torch.bfloat16
            and 1 <= input_.dim() <= 3
            and input_.numel() > 0
            and input_.shape[-1] == self.weight.shape[1]
            and input_.data_ptr() % 16 == 0 and self.weight.data_ptr() % 16 == 0
            and not (torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") != torch.bfloat16)
        )

    def forward(self, input_):
        assert len(self.weight.size()) == 2
        real_weights = self.weight

        if self._can_fuse(input_):
            return _QuantLinearFn.apply(input_, real_weights, self.w_bits, self.a_bits, self)
        if self._can_route(input_):
            return _OperandLinearFn.apply(input_, real_weights, self.w_bits, self.a_bits, self)

        if self.w_bits >= 32:
            weight = self.weight
        elif self.w_bits >= 3:
            weight_clip_val = torch.tensor([-2.0, 2.0])
            weight = SymQuantizer.apply(real_weights, weight_clip_val, self.w_bits, self.weight_layerwise)
        else:
            weight = _LowBitWeight.apply(real_weights, self.w_bits, self.weight_layerwise)
        if self.a_bits < 32 and self.a_bits > 2:
            act_clip_val = torch.tensor([-2.0, 2.0])
            input_ = self.act_quantizer.apply(input_, act_clip_val, self.a_bits, self.act_layerwise)

        out = nn.functional.linear(input_, weight)
        if self.bias is not None:
            out += self.bias.view(1, -1).expand_as(out)
        return out
