#!/usr/bin/env python
"""GPU-box tool: the W1 / W2 weight kernel (lowbit_exact_kernel) alone — parity against the numpy oracle on the
LLaMA weight shapes and on ragged ones, then CUDA-event timings (rotating buffers > L2) with the HBM fraction.
`python tests/gpu_lowbit_probe.py [ncu]`: with `ncu`, only a few launches at [11008, 4096] (for a capture)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import qat_testutil as U  # noqa: E402
from llm_qat_b200 import _lib  # noqa: E402
from llm_qat_b200.utils_quant import _LowBitWeight  # noqa: E402
from oracle import quant_oracle as qo  # noqa: E402

PEAK = 6459.0
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:  # noqa: BLE001
    pass


def parity():
    g = torch.Generator().manual_seed(5)
    bad = 0
    for dtype, tdt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        for rows, cols in ((512, 4096), (256, 11008), (64, 13824), (3, 50000), (33, 1001), (17, 7), (9, 8), (5, 31),
                           (257, 4095), (129, 11007), (64, 4097), (2, 100000)):
            w = (torch.randn(rows, cols, generator=g) * 0.02).to(tdt)
            w[0] = 0.0                       # scale 0: the exact-division rows
            w[rows - 1, cols // 2] = 3e4      # an outlier: the sum's rounding depends on the order
            for bits in (1, 2):
                got = U.tensor_to_f32(_LowBitWeight.apply(w.cuda(), bits, False))
                ref = qo.lowbit_weight(U.tensor_to_f32(w), bits, False, dtype)["w_eff"]
                n = qo.count_mismatch(got, ref)
                fits = cols * (4 if dtype == "fp32" else 2) < 220 * 1024   # else: two-pass kernels, fp64 sum (tolerance)
                bad += n > 0 and fits
                print(f"{dtype} [{rows},{cols}] W{bits}: {n} mismatching elements" + ("" if fits else "  (row beyond one CTA's shared memory: two-pass path)"), flush=True)
    print("PARITY", "OK" if bad == 0 else f"FAILED ({bad} cases)")
    return bad


def timing(steps=30):
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(1)
    out = {}
    for dt_name, dt, tdt, esz in (("bf16", 1, torch.bfloat16, 2), ("fp32", 0, torch.float32, 4)):
        for rows, cols in ((11008, 4096), (4096, 11008), (4096, 4096), (11007, 4095)):
            n = rows * cols
            nbuf = max(3, -(-300_000_000 // (n * esz * 2)))
            ws = [(torch.randn(rows, cols, generator=g) * 0.02).to(tdt).cuda() for _ in range(2)]
            ws += [ws[i % 2].clone() for i in range(nbuf - 2)]
            outs = [torch.empty_like(t) for t in ws]
            wsp = torch.empty(int(L.qat_lowbit_workspace_bytes(rows, 0)), dtype=torch.uint8, device="cuda")
            for bits in (1, 2):
                def once(i):
                    _lib.check(L.qat_lowbit_weight_fwd(ws[i].data_ptr(), outs[i].data_ptr(), rows, cols, dt, bits, 0,
                                                       wsp.data_ptr(), wsp.numel(), st))
                for i in range(nbuf):
                    once(i)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for k in range(steps):
                    once(k % nbuf)
                e1.record()
                e1.synchronize()
                us = e0.elapsed_time(e1) / steps * 1e3
                gbs = n * esz * 2 / us / 1e3
                key = f"{dt_name}[{rows},{cols}] W{bits}"
                out[key] = {"us": round(us, 2), "GBps": round(gbs, 1), "frac": round(gbs / PEAK, 3)}
                print(f"{key}: {us:.1f} us  {gbs:.0f} GB/s  {gbs / PEAK:.3f} of peak", flush=True)
            del ws, outs
    print(json.dumps({"lowbit_exact_kernel": out, "hbm_peak_GBps": PEAK}))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "ncu":
        w = [(torch.randn(11008, 4096) * 0.02).bfloat16().cuda() for _ in range(3)]
        for i in range(6):
            _LowBitWeight.apply(w[i % 3], 1 + i % 2, False)
        torch.cuda.synchronize()
        print("ok")
    else:
        rc = parity()
        timing()
        sys.exit(1 if rc else 0)
