#!/usr/bin/env python
"""GPU-box tool: the two tcgen05 GEMMs alone, for both tile plans — K4 and the bf16 GEMM's dgrad (A K-major,
B MN-major) and wgrad (both MN-major) of a QuantizeLinear [T, K] -> [T, N] — at BASELINE config 2
(T=8192, K=4096, N=11008) and the LLaMA-7B layer shapes at T=2048.  argv: [reps] [cta_group]."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import torch
from llm_qat_b200 import _lib
from llm_qat_b200.utils_quant import gemm_bf16, qlinear_i8
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
groups = [int(sys.argv[2])] if len(sys.argv) > 2 else [1, 2]
shapes = [(8192, 4096, 11008)] if len(sys.argv) > 2 else [(8192, 4096, 11008), (2048, 4096, 4096),
                                                            (2048, 4096, 11008), (2048, 11008, 4096)]


def time_us(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


g = torch.Generator().manual_seed(0)
for T, K, N in shapes:
    qx = torch.randint(-127, 128, (T, K), generator=g, dtype=torch.int8).cuda()
    qw = torch.randint(-7, 8, (N, K), generator=g, dtype=torch.int8).cuda()
    ex = (torch.rand(T, generator=g) * 50 + 1).cuda()
    ew = (torch.rand(N, generator=g) * 300 + 10).cuda()
    gy = torch.randn(T, N, generator=g).bfloat16().cuda()
    w = torch.randn(N, K, generator=g).bfloat16().cuda()
    x = torch.randn(T, K, generator=g).bfloat16().cuda()
    for cg in groups:
        _lib.check(_lib.lib().qat_set_gemm_cta_group(cg))
        us = time_us(lambda: qlinear_i8(qx, qw, ex, ew, torch.bfloat16))
        print(f"qlinear_i8 cta_group={cg} {T}x{N}x{K}: {us:.1f} us  {2*T*N*K/us/1e6:.0f} TOP/s", flush=True)
        us = time_us(lambda: gemm_bf16(gy, w, None, T, K, N, 0, 1))
        print(f"gemm_bf16 dgrad cta_group={cg} {T}x{K}x{N}: {us:.1f} us  {2*T*N*K/us/1e6:.0f} TFLOP/s", flush=True)
        us = time_us(lambda: gemm_bf16(gy, x, None, N, K, T, 1, 1))
        print(f"gemm_bf16 wgrad cta_group={cg} {N}x{K}x{T}: {us:.1f} us  {2*T*N*K/us/1e6:.0f} TFLOP/s", flush=True)
_lib.check(_lib.lib().qat_set_gemm_cta_group(0))
