"""GPU probe for qat_gemm_bf16 (csrc/gemm_bf16.cu): every operand majorness x CTA-group plan against
an fp32 torch matmul, then timing against torch.mm (cuBLAS) at the QuantizeLinear backward shapes.
Run on the GPU box:  python tests/gpu_umma_probe.py
Prints one JSON line per case; exits non-zero if a case is wrong."""
from __future__ import annotations

import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import llm_qat_b200  # noqa: E402
from llm_qat_b200 import _lib  # noqa: E402

L = _lib.lib()
dev = torch.device("cuda", 0)


def gemm(a, b, M, N, K, a_mn, b_mn, cg, out_dtype=torch.bfloat16, mask=None):
    out = torch.empty(M, N, dtype=out_dtype, device=dev)
    rc = L.qat_gemm_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), 0 if mask is None else mask.data_ptr(), M, N, K,
                         a_mn, b_mn, 1 if out_dtype == torch.bfloat16 else 0, cg,
                         torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "qat_gemm_bf16")
    return out


def case(M, N, K, a_mn, b_mn, cg, masked=False, out_dtype=torch.bfloat16, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    A = torch.randn(M, K, generator=g).bfloat16().to(dev)      # logical [M, K]
    B = torch.randn(N, K, generator=g).bfloat16().to(dev)      # logical [N, K]
    a = A.t().contiguous() if a_mn else A
    b = B.t().contiguous() if b_mn else B
    mask = bits = None
    if masked:
        bits = torch.rand(M * N, generator=g) < 0.7
        pad = (-bits.numel()) % 8
        bb = torch.cat([bits, torch.zeros(pad, dtype=torch.bool)]).view(-1, 8).to(torch.uint8)
        mask = (bb * (1 << torch.arange(8, dtype=torch.uint8))).sum(1).to(torch.uint8).to(dev)
    out = gemm(a, b, M, N, K, a_mn, b_mn, cg, out_dtype, mask)
    torch.cuda.synchronize()
    ref = A.float() @ B.float().t()
    if masked:
        ref = ref * bits.view(M, N).to(dev)
    err = (out.float() - ref).norm() / ref.norm()
    return float(err)


def main():
    ok = True
    shapes = [(128, 256, 64), (256, 256, 128), (304, 520, 200), (2048, 4096, 1024), (1000, 776, 4096)]
    for a_mn in (0, 1):
        for b_mn in (0, 1):
            for cg in (1, 2):
                for (M, N, K) in shapes:
                    try:
                        err = case(M, N, K, a_mn, b_mn, cg)
                    except Exception as e:  # noqa: BLE001
                        err = float("nan")
                        print("EXC", repr(e)[:300], flush=True)
                    good = err == err and err < 5e-3
                    ok &= good
                    print(json.dumps({"a_mn": a_mn, "b_mn": b_mn, "cg": cg, "shape": [M, N, K],
                                      "rel_err": err, "ok": good}), flush=True)
    # masked epilogue + fp32 output
    for (M, N, K) in [(256, 512, 128), (304, 520, 200), (77, 40, 64)]:
        for od in (torch.bfloat16, torch.float32):
            err = case(M, N, K, 0, 1, 0, masked=True, out_dtype=od, seed=3)
            good = err < 5e-3
            ok &= good
            print(json.dumps({"masked": True, "shape": [M, N, K], "out": str(od), "rel_err": err, "ok": good}),
                  flush=True)

    # timing at the LLaMA-7B backward shapes (T = 2048 and 8192)
    def bench(fn, n=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / n * 1e3

    for T in (2048, 8192):
        for (No, Ki) in [(4096, 4096), (11008, 4096), (4096, 11008)]:
            g_ = torch.randn(T, No, device=dev).bfloat16()
            wq = torch.randn(No, Ki, device=dev).bfloat16()
            xq = torch.randn(T, Ki, device=dev).bfloat16()
            row = {"T": T, "N_out": No, "K_in": Ki}
            for cg in (1, 2):
                row[f"dgrad_cg{cg}_us"] = round(bench(lambda: gemm(g_, wq, T, Ki, No, 0, 1, cg)), 1)
                row[f"wgrad_cg{cg}_us"] = round(bench(lambda: gemm(g_, xq, No, Ki, T, 1, 1, cg)), 1)
            row["dgrad_cublas_us"] = round(bench(lambda: torch.mm(g_, wq)), 1)
            row["wgrad_cublas_us"] = round(bench(lambda: torch.mm(g_.t(), xq)), 1)
            fl = 2.0 * T * No * Ki
            row["dgrad_best_TF"] = round(fl / min(row["dgrad_cg1_us"], row["dgrad_cg2_us"]) / 1e6, 1)
            row["wgrad_best_TF"] = round(fl / min(row["wgrad_cg1_us"], row["wgrad_cg2_us"]) / 1e6, 1)
            row["cublas_dgrad_TF"] = round(fl / row["dgrad_cublas_us"] / 1e6, 1)
            row["cublas_wgrad_TF"] = round(fl / row["wgrad_cublas_us"] / 1e6, 1)
            print(json.dumps(row), flush=True)
    print("PROBE", "OK" if ok else "FAILED", flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
