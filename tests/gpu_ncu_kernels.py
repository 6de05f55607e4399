#!/usr/bin/env python
"""GPU-box tool: launch each round-2 kernel a few times at its LLaMA-7B shape (T = 2048) so that
`ncu --set full -k regex:...` can capture it:  attention fwd / bwd, the bf16 dgrad / wgrad GEMMs,
qkv_prep, rmsnorm / swiglu feeds, KD loss.  Prints CUDA-event times (the roofline numerators)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import llm_qat_b200  # noqa: E402
from llm_qat_b200 import _lib, fused_ops as FO  # noqa: E402

L = _lib.lib()
dev = torch.device("cuda", 0)
REPS = int(os.environ.get("NCU_REPS", "3"))
out = {}


def timed(name, fn, flops=None, nbytes=None):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    e1.synchronize()
    us = e0.elapsed_time(e1) / REPS * 1e3
    r = {"us": round(us, 1)}
    if flops:
        r["TFLOPs"] = round(flops / us / 1e6, 1)
    if nbytes:
        r["GBps"] = round(nbytes / us / 1e3, 1)
    out[name] = r
    print(name, r, flush=True)


B, S, H = 1, 2048, 32
T, C, I, V = 2048, 4096, 11008, 32000
st = torch.cuda.current_stream().cuda_stream
q, k, v = (torch.randn(B, S, H, 128, device=dev).bfloat16().requires_grad_(True) for _ in range(3))
go = torch.randn(B, S, H, 128, device=dev).bfloat16()
fl = 4.0 * S * S * 128 * H * B / 2
timed("attn_fwd", lambda: FO.causal_attention(q, k, v), flops=fl)
o = FO.causal_attention(q, k, v)
timed("attn_bwd(delta+dq+dkv)", lambda: torch.autograd.grad(o, (q, k, v), go, retain_graph=True), flops=2.5 * fl)

g = torch.randn(T, I, device=dev).bfloat16()
wq = torch.randn(I, C, device=dev).bfloat16()
xq = torch.randn(T, C, device=dev).bfloat16()
gx, gw = torch.empty(T, C, device=dev).bfloat16(), torch.empty(I, C, device=dev).bfloat16()
mx = torch.randint(0, 255, (T * C // 8,), dtype=torch.uint8, device=dev)
mw = torch.randint(0, 255, (I * C // 8,), dtype=torch.uint8, device=dev)
timed("dgrad[2048x11008]x[11008x4096]", lambda: _lib.check(L.qat_gemm_bf16(
    g.data_ptr(), wq.data_ptr(), gx.data_ptr(), mx.data_ptr(), T, C, I, 0, 1, 1, 0, st)), flops=2.0 * T * C * I)
timed("wgrad[11008x2048]x[2048x4096]", lambda: _lib.check(L.qat_gemm_bf16(
    g.data_ptr(), xq.data_ptr(), gw.data_ptr(), mw.data_ptr(), I, C, T, 1, 1, 1, 0, st)), flops=2.0 * T * C * I)

wc = torch.randint(-7, 8, (I, C), dtype=torch.int8, device=dev)
we = torch.rand(I, device=dev) * 100 + 50
xc = torch.randint(-127, 128, (T, C), dtype=torch.int8, device=dev)
xe = torch.rand(T, device=dev) * 100 + 50
wq2, xq2 = torch.empty(I, C, device=dev).bfloat16(), torch.empty(T, C, device=dev).bfloat16()
timed("dequant_W[11008x4096]", lambda: _lib.check(L.qat_dequant_codes(wc.data_ptr(), we.data_ptr(), wq2.data_ptr(), I, C, 1, st)),
      nbytes=I * C * 3)
timed("dequant_x[2048x4096]", lambda: _lib.check(L.qat_dequant_codes(xc.data_ptr(), xe.data_ptr(), xq2.data_ptr(), T, C, 1, st)),
      nbytes=T * C * 3)

qkv = [torch.randn(B, S, H * 128, device=dev).bfloat16() for _ in range(3)]
cos = torch.randn(2048, 128, device=dev)
sin = torch.randn(2048, 128, device=dev)
pos = torch.arange(S, device=dev)[None]
with torch.autocast("cuda", dtype=torch.bfloat16):
    timed("qkv_prep", lambda: FO.qkv_prep(*qkv, cos, sin, pos, H, 4), nbytes=T * C * (12 + 0.25))
    x = torch.randn(T, C, device=dev).bfloat16()
    w = torch.ones(C, device=dev).bfloat16()
    timed("rmsnorm_feed", lambda: FO.rmsnorm(x, w, 1e-6, feed_bits=8), nbytes=T * C * 5.125)
    ga, up = torch.randn(T, I, device=dev).bfloat16(), torch.randn(T, I, device=dev).bfloat16()
    timed("swiglu_feed", lambda: FO.swiglu(ga, up, feed_bits=8), nbytes=T * I * 7.125)
sl = torch.randn(1, T, V, device=dev).bfloat16().requires_grad_(True)
tl = torch.randn(1, T, V, device=dev).bfloat16()
timed("kd_loss_fwd", lambda: FO.kd_loss(sl, tl), nbytes=T * V * 4)
loss = FO.kd_loss(sl, tl)
timed("kd_loss_bwd", lambda: torch.autograd.grad(loss, sl, retain_graph=True), nbytes=T * V * 6)
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(out, open(os.path.join(ROOT, "gpurun_out", "ncu_kernels_times.json"), "w"), indent=1)
