#!/usr/bin/env python
"""bench.py — the hot path's headline measurement (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], the QuantizeLinear up_proj operands):
    x  bf16 [8192, 4096]   A8 per-token   SymQuantizer forward + STE backward
    W  bf16 [11008, 4096]  W4 per-channel SymQuantizer forward + STE backward
One step = those four launches (K1 x, K1 W, K3 x, K3 W).  Algorithmic bytes per
step = 10 B/elem * (33,554,432 + 45,088,768) = 786.4 MB (SURVEY.md section 8d).

Metric: "fake-quant fwd+bwd GB/s" = algorithmic bytes of all ranks / max-over-ranks
device time.  Prints ONE JSON line (rank 0).  Extra objects on the same line:
roofline (dominant kernel, live CUDA-event timing), cpu_baseline (torch-eager
port of the reference on the host cores), e2e (host buffers through the C ABI's
host entry points, H2D + D2H inside the timed region; link_probe = the host link's
own ceiling with every rank copying at once), qlinear (K4 tcgen05 GEMM vs cuBLASLt
int8 and vs the reference's eager QuantizeLinear.forward), config1_fp32 (BASELINE
configs[0], each kernel with its roofline), config3_layer and qat_step (BASELINE
configs[2] / [3] / [4]: this library with fuse_model vs the quant path only vs the
reference's eager chain on the same GPU(s); 13b adds the output-channel-sharded arm), clocks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

T_TOK, K_IN, N_OUT = 8192, 4096, 11008
A_BITS, W_BITS = 8, 4
CLIP = (-2.0, 2.0)
ELEMS = T_TOK * K_IN + N_OUT * K_IN
BYTES_PER_ELEM_BF16 = 10  # fwd 2e + bwd 3e, e = 2 (SURVEY.md 8d)
STEP_BYTES = ELEMS * BYTES_PER_ELEM_BF16
METRIC = "fake-quant fwd+bwd GB/s"
WORKLOAD = ("configs[1]: QuantizeLinear up_proj operands, x bf16[8192,4096] A8 per-token + "
            "W bf16[11008,4096] W4 per-channel, SymQuantizer fwd + STE bwd")


def bench_config(world: int):
    """The `config` object — identical in the b200 and the reference arm (same workload, same partitioning)."""
    return {"workload": WORKLOAD, "bytes_per_step_per_gpu": STEP_BYTES,
            "l2": "inputs larger than L2 (x+W = 157 MB per step, 786 MB touched between re-reads)",
            "parallelism": f"dp{world}: every rank fake-quantizes its own 8192-token batch and weight replica; "
                           "rows are independent, no data-path collective"}


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed
# `ncu --set full` capture (profiles/): filled in from profiles/rNN_ncu_summary.json
def _ncu_summary():
    for tag in ("r02", "r01"):
        try:
            with open(os.path.join(ROOT, "profiles", f"{tag}_ncu_summary.json")) as f:
                return json.load(f)
        except Exception:
            continue
    return {}


def _load_ncu_traffic():
    return {k: v.get("dram_bytes_per_launch") for k, v in _ncu_summary().get("kernels", {}).items()}


NCU_TRAFFIC = _load_ncu_traffic()


def _load_ncu_gemm():
    return _ncu_summary().get("kernels", {}).get("qlinear_i8", {})


NCU_GEMM = _load_ncu_gemm()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


def make_inputs(seed: int):
    """Synthetic configs[1] tensors on the CPU (SURVEY.md 8d config 2 distributions)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(T_TOK, K_IN, generator=g)
    idx = torch.randint(0, x.numel(), (x.numel() // 1000,), generator=g)
    x.view(-1)[idx] *= 20.0
    w = torch.randn(N_OUT, K_IN, generator=g) * 0.02
    gx = torch.randn(T_TOK, K_IN, generator=g)
    gw = torch.randn(N_OUT, K_IN, generator=g)
    return [t.bfloat16() for t in (x, w, gx, gw)]


DUMP_ROWS = 512   # rows of each operand that --dump-outputs writes: 4 files of 512 x 4096 float32 = 32 MB


def dump_rows():
    """The fixed, seeded row indices of x and of W that --dump-outputs writes (sorted)."""
    g = torch.Generator().manual_seed(0)
    return (torch.randperm(T_TOK, generator=g)[:DUMP_ROWS].sort().values,
            torch.randperm(N_OUT, generator=g)[:DUMP_ROWS].sort().values)


def dump_outputs(out_dir: str, y_x, y_w, grad_x, grad_w):
    """--dump-outputs: what one step hands its caller (fake-quantized x and W, the STE gradients of both) as
    float32 DIR/<name>.npy.  Whole rows, the unit each scale is computed over, at the dump_rows() sample
    (the same rows for an output and its gradient), so that two builds or the two arms can be compared
    element for element."""
    import numpy as np

    rows_x, rows_w = dump_rows()
    os.makedirs(out_dir, exist_ok=True)
    for name, t, rows in (("y_x", y_x, rows_x), ("y_w", y_w, rows_w), ("grad_x", grad_x, rows_x),
                          ("grad_w", grad_w, rows_w)):
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, rows.to(t.device)).float().cpu().numpy())


# ----------------------------------------------------------------------------
# clocks sampler (pynvml; falls back to nvidia-smi)
# ----------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._th = None
        self._nv = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None
            return self
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()
        return self

    def _run(self):
        nv = self._nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                util = nv.nvmlDeviceGetUtilizationRates(self._h).gpu
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                self.samples.append((mhz, util))
                for bit, name in names.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def stop(self):
        self._stop.set()
        if self._th is not None:
            self._th.join(timeout=2)
        loaded = [m for m, u in self.samples if u > 0] or [m for m, _ in self.samples]
        return {"sm_mhz": statistics.median(loaded) if loaded else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------
class Step:
    """One hot-path step on preallocated device buffers, launched through the C
    ABI with raw pointers (what the Python boundary does, minus allocation)."""

    def __init__(self, x, w, gx, gw):
        from llm_qat_b200 import _lib

        self.L = _lib.lib()
        self.lib = _lib
        self.x, self.w, self.gx, self.gw = x, w, gx, gw
        self.yx, self.yw = torch.empty_like(x), torch.empty_like(w)
        self.dx, self.dw = torch.empty_like(x), torch.empty_like(w)
        self.names = ["sym_fwd_x_a8", "sym_fwd_w_w4", "ste_bwd_x", "ste_bwd_w"]
        self.kernel_bytes = [x.numel() * 4, w.numel() * 4, x.numel() * 6, w.numel() * 6]

    def launch(self, i, stream):
        L, BF16 = self.L, 1
        if i == 0:
            rc = L.qat_sym_fwd(self.x.data_ptr(), self.yx.data_ptr(), 0, 0, 0, 0, 0, 0.0, 0.0, T_TOK, K_IN, BF16,
                               A_BITS, 0, 0, stream)
        elif i == 1:
            rc = L.qat_sym_fwd(self.w.data_ptr(), self.yw.data_ptr(), 0, 0, 0, 0, 0, 0.0, 0.0, N_OUT, K_IN, BF16,
                               W_BITS, 0, 0, stream)
        elif i == 2:
            rc = L.qat_ste_bwd(self.gx.data_ptr(), self.x.data_ptr(), self.dx.data_ptr(), 0, CLIP[0], CLIP[1],
                               self.x.numel(), BF16, stream)
        else:
            rc = L.qat_ste_bwd(self.gw.data_ptr(), self.w.data_ptr(), self.dw.data_ptr(), 0, CLIP[0], CLIP[1],
                               self.w.numel(), BF16, stream)
        self.lib.check(rc, self.names[i])

    def run(self, stream):
        for i in range(4):
            self.launch(i, stream)


def time_config1_fp32(device, steps, pk):
    """BASELINE configs[0] on the GPU: fp32 [8192, 4096], SymQuantizer (W4 per-channel, A8 per-token) and
    AsymQuantizer (A8, A4), forward + STE backward, each kernel with its own roofline object (algorithmic
    bytes: fwd 2e, bwd 3e per element, e = 4; SURVEY.md 8d).  Two buffer sets alternate so that no launch
    re-reads what the previous one left in L2 (134 MB per tensor, 4 tensors per set)."""
    from llm_qat_b200 import _lib

    L = _lib.lib()
    g = torch.Generator().manual_seed(1234)
    sets = []
    for _ in range(2):
        x = (torch.randn(8192, 4096, generator=g) * 0.5).to(device)
        gr = torch.randn(8192, 4096, generator=g).to(device)
        sets.append((x, gr, torch.empty_like(x), torch.empty_like(x)))
    n = 8192 * 4096
    st = torch.cuda.current_stream().cuda_stream
    out = {}

    def timed(fn):
        for i in range(4):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / steps

    for name, fn, bits in (("sym_w4", L.qat_sym_fwd, 4), ("sym_a8", L.qat_sym_fwd, 8),
                           ("asym_a8", L.qat_asym_fwd, 8), ("asym_a4", L.qat_asym_fwd, 4)):
        def fwd(i):
            x, gr, y, dx = sets[i & 1]
            _lib.check(fn(x.data_ptr(), y.data_ptr(), 0, 0, 0, 0, 0, 0.0, 0.0, 8192, 4096, 0, bits, 0, 0, st))

        def bwd(i):
            x, gr, y, dx = sets[i & 1]
            _lib.check(L.qat_ste_bwd(gr.data_ptr(), x.data_ptr(), dx.data_ptr(), 0, -2.0, 2.0, n, 0, st))

        def both(i):
            fwd(i)
            bwd(i)
        ms_f, ms_b, ms = timed(fwd), timed(bwd), timed(both)

        def roof(bytes_, ms_):
            a = bytes_ / ms_ / 1e6
            return {"bound": "hbm", "achieved": round(a, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": round(a / pk["hbm_gbs"], 4), "bytes_per_launch": bytes_, "us_per_launch": round(ms_ * 1e3, 2)}
        out[name] = {"ms_fwd_bwd": round(ms, 4), "GBps": round(n * 20 / ms / 1e6, 1),
                     "frac_of_hbm_peak": round(n * 20 / ms / 1e6 / pk["hbm_gbs"], 4),
                     "roofline_fwd": roof(n * 8, ms_f), "roofline_bwd": roof(n * 12, ms_b)}
    out["workload"] = "configs[0]: fp32 [8192, 4096], Sym W4 / A8 and Asym A8 / A4, fwd + STE bwd (20 B/elem)"
    return out


def time_shape_sweep(device, steps, pk):
    """SURVEY.md 8d config 1, the rest of it: both dtypes, the LLaMA-7B operand shapes, forward
    alone and forward + backward, per quantizer.  Buffers rotate through > 2x L2 so that no
    launch re-reads what a previous one left in the 126 MB L2."""
    from llm_qat_b200 import _lib

    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    out = {}
    g = torch.Generator().manual_seed(1234)
    for dt_name, dt, tdt, esz in (("fp32", 0, torch.float32, 4), ("bf16", 1, torch.bfloat16, 2)):
        for rows, cols in ((8192, 4096), (11008, 4096), (4096, 11008), (2048, 4096)):
            n = rows * cols
            nbuf = max(2, -(-300_000_000 // (n * esz * 2)))
            xs = [(torch.randn(rows, cols, generator=g) * 0.5).to(tdt).to(device) for _ in range(min(nbuf, 2))]
            while len(xs) < nbuf:
                xs.append(xs[len(xs) % 2].clone())
            gs = [torch.randn(rows, cols, generator=g).to(tdt).to(device)] * 1
            gs = gs + [gs[0].clone() for _ in range(nbuf - 1)]
            ys = [torch.empty_like(t) for t in xs]
            ds = [torch.empty_like(t) for t in xs]
            for qname, fn, bits in (("sym4", L.qat_sym_fwd, 4), ("sym8", L.qat_sym_fwd, 8), ("asym8", L.qat_asym_fwd, 8)):
                res = {}
                for mode in ("fwd", "fwd_bwd"):
                    def once(i):
                        _lib.check(fn(xs[i].data_ptr(), ys[i].data_ptr(), 0, 0, 0, 0, 0, 0.0, 0.0, rows, cols, dt,
                                      bits, 0, 0, st))
                        if mode == "fwd_bwd":
                            _lib.check(L.qat_ste_bwd(gs[i].data_ptr(), xs[i].data_ptr(), ds[i].data_ptr(), 0, -2.0,
                                                     2.0, n, dt, st))
                    for i in range(nbuf):
                        once(i)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for k in range(steps):
                        once(k % nbuf)
                    e1.record()
                    e1.synchronize()
                    us = e0.elapsed_time(e1) / steps * 1e3
                    nbytes = n * esz * (2 if mode == "fwd" else 5)
                    res[mode] = {"us": round(us, 2), "GBps": round(nbytes / us / 1e3, 1),
                                 "frac": round(nbytes / us / 1e3 / pk["hbm_gbs"], 4)}
                out[f"{dt_name}[{rows},{cols}] {qname}"] = res
            del xs, gs, ys, ds
    # SymQuantizer inside torch.autocast: bf16 in, fp32 y (6 B/elem), and the GEMM feed (codes + mask: 3.125 B/elem)
    for rows, cols in ((8192, 4096), (11008, 4096), (2048, 4096)):
        n = rows * cols
        nbuf = max(2, -(-300_000_000 // (n * 6)))
        xs = [(torch.randn(rows, cols, generator=g) * 0.5).bfloat16().to(device) for _ in range(2)]
        xs += [xs[i % 2].clone() for i in range(nbuf - 2)]
        ys = [torch.empty(rows, cols, dtype=torch.float32, device=device) for _ in range(nbuf)]
        cs = [torch.empty(rows, cols, dtype=torch.int8, device=device) for _ in range(nbuf)]
        ms = [torch.empty(n // 8, dtype=torch.uint8, device=device) for _ in range(nbuf)]
        es = torch.empty(rows, dtype=torch.float32, device=device)
        for mode, nbytes in (("y_fp32", n * 6), ("feed", n * 3 + n // 8)):
            def once(i):
                if mode == "y_fp32":
                    rc = L.qat_sym_fwd(xs[i].data_ptr(), ys[i].data_ptr(), 0, 0, 0, 0, 0, 0.0, 0.0, rows, cols, 2, 8, 0, 0, st)
                else:
                    rc = L.qat_sym_fwd(xs[i].data_ptr(), 0, cs[i].data_ptr(), 1, 0, es.data_ptr(), ms[i].data_ptr(),
                                       -2.0, 2.0, rows, cols, 2, 8, 0, 0, st)
                _lib.check(rc)
            for i in range(nbuf):
                once(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(steps):
                once(k % nbuf)
            e1.record()
            e1.synchronize()
            us = e0.elapsed_time(e1) / steps * 1e3
            out[f"bf16_amp[{rows},{cols}] sym8 {mode}"] = {"fwd": {"us": round(us, 2), "GBps": round(nbytes / us / 1e3, 1),
                                                                  "frac": round(nbytes / us / 1e3 / pk["hbm_gbs"], 4)}}
        del xs, ys, cs, ms
    # the fused linear's backward helpers: rebuild bf16 operands from codes (3 B/elem) and the
    # mask-driven STE (4.125 B/elem)
    for rows, cols in ((11008, 4096), (8192, 4096), (2048, 4096)):
        n = rows * cols
        nbuf = max(2, -(-300_000_000 // (n * 4)))
        cs = [torch.randint(-7, 8, (rows, cols), generator=g, dtype=torch.int8).to(device) for _ in range(2)]
        cs += [cs[i % 2].clone() for i in range(nbuf - 2)]
        es = (torch.rand(rows, generator=g) * 300 + 10).bfloat16().float().to(device)
        outs = [torch.empty(rows, cols, dtype=torch.bfloat16, device=device) for _ in range(nbuf)]
        gs = [torch.randn(rows, cols, generator=g).bfloat16().to(device)]
        gs += [gs[0].clone() for _ in range(nbuf - 1)]
        ms = [torch.randint(0, 256, (n // 8,), generator=g, dtype=torch.uint8).to(device)]
        ms += [ms[0].clone() for _ in range(nbuf - 1)]
        for mode, nbytes in (("dequant_codes", n * 3), ("ste_from_mask", n * 4 + n // 8)):
            def once(i):
                if mode == "dequant_codes":
                    rc = L.qat_dequant_codes(cs[i].data_ptr(), es.data_ptr(), outs[i].data_ptr(), rows, cols, 1, st)
                else:
                    rc = L.qat_ste_bwd_from_mask(gs[i].data_ptr(), ms[i].data_ptr(), outs[i].data_ptr(), n, 1, st)
                _lib.check(rc)
            for i in range(nbuf):
                once(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(steps):
                once(k % nbuf)
            e1.record()
            e1.synchronize()
            us = e0.elapsed_time(e1) / steps * 1e3
            out[f"bf16[{rows},{cols}] {mode}"] = {"fwd": {"us": round(us, 2), "GBps": round(nbytes / us / 1e3, 1),
                                                         "frac": round(nbytes / us / 1e3 / pk["hbm_gbs"], 4)}}
        del cs, outs, gs, ms
    # QuantizeLinear's W1 / W2 weight path (utils_quant.py:202-242): mean|w| per row (torch's summation order),
    # then apply, in one pass with the row staged in shared memory: 2e B/elem
    for dt_name, dt, tdt, esz in (("bf16", 1, torch.bfloat16, 2), ("fp32", 0, torch.float32, 4)):
        rows, cols = 11008, 4096
        n = rows * cols
        ws_ = [(torch.randn(rows, cols, generator=g) * 0.02).to(tdt).to(device) for _ in range(2)]
        ws_ += [ws_[0].clone()]
        outs = [torch.empty_like(t) for t in ws_]
        wsp = torch.empty(int(L.qat_lowbit_workspace_bytes(rows, 0)), dtype=torch.uint8, device=device)
        for bits in (1, 2):
            def once(i):
                _lib.check(L.qat_lowbit_weight_fwd(ws_[i].data_ptr(), outs[i].data_ptr(), rows, cols, dt, bits, 0,
                                                   wsp.data_ptr(), wsp.numel(), st))
            for i in range(3):
                once(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(steps):
                once(k % 3)
            e1.record()
            e1.synchronize()
            us = e0.elapsed_time(e1) / steps * 1e3
            nbytes = n * esz * 2
            out[f"{dt_name}[{rows},{cols}] lowbit_w{bits}"] = {"fwd": {"us": round(us, 2), "GBps": round(nbytes / us / 1e3, 1),
                                                                      "frac": round(nbytes / us / 1e3 / pk["hbm_gbs"], 4)}}
        del ws_, outs
    return out


def time_qlinear(device, x, w, steps, pk):
    """K4: integer-grid tcgen05 GEMM at configs[1]; codes produced by K1."""
    from llm_qat_b200._lib import CODES_I8
    from llm_qat_b200.utils_quant import fake_quant_forward, qlinear_i8

    _, qw, _, ew, _ = fake_quant_forward(w, W_BITS, False, True, want_y=False, codes_kind=CODES_I8, want_scales=True)
    _, qx, _, ex, _ = fake_quant_forward(x, A_BITS, False, True, want_y=False, codes_kind=CODES_I8, want_scales=True)

    def gemm_only():
        return qlinear_i8(qx, qw, ex, ew, torch.bfloat16)

    def fwd():  # what QuantizeLinear.forward costs per call: quantize x, quantize W, GEMM
        _, qx2, _, ex2, _ = fake_quant_forward(x, A_BITS, False, True, want_y=False, codes_kind=CODES_I8,
                                               want_scales=True)
        _, qw2, _, ew2, _ = fake_quant_forward(w, W_BITS, False, True, want_y=False, codes_kind=CODES_I8,
                                               want_scales=True)
        return qlinear_i8(qx2, qw2, ex2, ew2, torch.bfloat16)

    res = {}
    flop = 2.0 * T_TOK * K_IN * N_OUT
    for name, fn in (("gemm", gemm_only), ("forward", fwd)):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / steps
        res[name] = {"ms": round(ms, 4), "TOPs": round(flop / ms / 1e9, 1), "tokens_per_s": round(T_TOK / ms * 1e3)}
    # comparators, measured in this run at the same shape:
    #  (1) the library int8 GEMM (torch._int_mm -> cuBLASLt, int32 output): the measured int8 tensor peak
    #      this kernel's roofline fraction is taken against;
    #  (2) the reference's own QuantizeLinear.forward, eager on this GPU (oracle/ref_module: 18 elementwise
    #      kernels + a cuBLAS bf16 GEMM on dequantized operands, utils_quant.py:190-254).
    lib_tops = None
    try:
        b_t = qw.t().contiguous()     # [K, N]; _int_mm wants a row-major second operand
        torch._int_mm(qx, b_t)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            torch._int_mm(qx, b_t)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / steps
        lib_tops = flop / ms / 1e9
        res["library_int8_gemm"] = {"ms": round(ms, 4), "TOPs": round(lib_tops, 1),
                                    "what": "torch._int_mm (cuBLASLt int8, s32 out) 8192x11008x4096"}
        del b_t
    except Exception as e:  # noqa: BLE001
        res["library_int8_gemm"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    try:
        from oracle import ref_module

        lin = ref_module.QuantizeLinear(K_IN, N_OUT, w_bits=W_BITS, a_bits=A_BITS).bfloat16().to(device)
        with torch.no_grad():
            lin.weight.copy_(w)
            for _ in range(2):
                lin(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n_ref = max(3, steps // 2)
            for _ in range(n_ref):
                lin(x)
            e1.record()
            e1.synchronize()
        ms = e0.elapsed_time(e1) / n_ref
        res["reference_eager"] = {"ms": round(ms, 4), "tokens_per_s": round(T_TOK / ms * 1e3),
                                  "what": "reference QuantizeLinear.forward op chain, eager on this GPU (bf16)",
                                  "speedup_of_forward": round(ms / res["forward"]["ms"], 2)}
        del lin
    except Exception as e:  # noqa: BLE001
        res["reference_eager"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    # tensor roofline: the measured library int8 GEMM when available (else twice the measured cuBLAS bf16
    # figure: kind::i8 retires 2x the MACs of kind::f16 per SM cycle), with the bf16 fraction beside it
    peak_i8 = lib_tops if lib_tops else 2.0 * pk["bf16_tflops"]
    res["roofline"] = {"bound": "tensor", "achieved": res["gemm"]["TOPs"], "peak": round(peak_i8, 1),
                       "unit": "TOP/s", "frac": round(res["gemm"]["TOPs"] / peak_i8, 4),
                       "frac_of_2x_bf16_peak": round(res["gemm"]["TOPs"] / (2.0 * pk["bf16_tflops"]), 4),
                       "frac_of_bf16_peak": round(res["gemm"]["TOPs"] / pk["bf16_tflops"], 4),
                       "peak_source": ("measured in this run: torch._int_mm (cuBLASLt int8) at the same shape" if lib_tops
                                       else "2 x bf16_tflops of " + pk["source"]),
                       "tensor_pipe_active_ncu": NCU_GEMM.get("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed"),
                       "traffic": NCU_GEMM.get("dram_bytes_per_launch"),
                       "kernel": "qlinear_i8_kernel<bf16, cta_group 2> 8192x11008x4096"}
    return res


def link_probe(device, h_src, h_dst, barrier, dist, reps=5):
    """Pinned-host copies only, every rank concurrently: STEP-sized H2D and D2H streams at once.
    Returns per-direction GB/s of this rank (max-over-ranks time) and the aggregate over ranks."""
    world = dist.get_world_size() if dist is not None else 1
    nbytes = ELEMS * 2 * 2                    # what one e2e step moves each way
    n_el = nbytes // h_src.element_size()
    reps_src = [h_src.view(-1)] * ((n_el + h_src.numel() - 1) // h_src.numel())
    d_in = torch.empty(h_src.numel(), dtype=h_src.dtype, device=device)
    d_out = torch.empty(h_dst.numel(), dtype=h_dst.dtype, device=device)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    chunks = len(reps_src)

    def run(n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s1.wait_stream(torch.cuda.current_stream())
        s2.wait_stream(torch.cuda.current_stream())
        for _ in range(n * chunks):
            with torch.cuda.stream(s1):
                d_in.copy_(h_src.view(-1), non_blocking=True)
            with torch.cuda.stream(s2):
                h_dst.view(-1).copy_(d_out, non_blocking=True)
        torch.cuda.current_stream().wait_stream(s1)
        torch.cuda.current_stream().wait_stream(s2)
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / n

    run(1)
    ms = run(reps)
    if dist is not None:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    moved = chunks * h_src.numel() * h_src.element_size()
    return {"ms_per_step_equivalent": round(ms * nbytes / moved, 3), "GBps_per_direction_per_gpu": round(moved / ms / 1e6, 1),
            "GBps_per_direction_aggregate": round(world * moved / ms / 1e6, 1), "ranks_concurrent": world,
            "what": "pinned H2D + D2H concurrently on every rank, no kernels: the ceiling of e2e on this host"}


def run_b200(args):
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; llm-qat_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=device)
    import llm_qat_b200
    from llm_qat_b200 import _lib
    from llm_qat_b200.host_api import fake_quant_fwd_bwd_host

    _lib.check(_lib.lib().qat_check_device(), "device check")
    pk = peaks()
    hx, hw, hgx, hgw = make_inputs(1234 + rank)   # each rank: its own token batch (data parallel)
    hx, hw, hgx, hgw = [t.pin_memory() for t in (hx, hw, hgx, hgw)]
    x, w, gx, gw = [t.to(device, non_blocking=True) for t in (hx, hw, hgx, hgw)]
    step = Step(x, w, gx, gw)
    torch.cuda.synchronize()
    K, W = args.steps, max(args.warmup, 3)
    stream = torch.cuda.current_stream().cuda_stream

    sampler = ClockSampler(local).start()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- region 1: K steps, launched as a CUDA graph of one step (device-resident inputs)
    for _ in range(W):
        step.run(stream)
    torch.cuda.synchronize()
    graph, used_graph = None, False
    try:
        cap = torch.cuda.Stream()
        cap.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(cap):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=cap):
                step.run(torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        for _ in range(W):
            graph.replay()
        used_graph = True
    except Exception as e:  # capture unsupported: fall back to direct launches
        print(f"bench.py: CUDA graph capture failed ({type(e).__name__}: {e}); timing direct launches", file=sys.stderr)
        graph = None
    barrier()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        if graph is not None:
            graph.replay()
        else:
            step.run(stream)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = (_lib.launch_count() - launches0) if graph is None else 4 * K
    if dist is not None:
        t = torch.tensor([ms_total], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / K
    value = world * STEP_BYTES / (ms_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:   # the buffers hold what the last timed step wrote
        dump_outputs(args.dump_outputs, step.yx, step.yw, step.dx, step.dw)

    # ---- region 2: per-kernel durations for the roofline.  An event record between
    # two kernels costs ~4 us of serialisation, so each kernel is timed as K
    # back-to-back launches inside ONE event pair, alternating between two buffer
    # sets so that consecutive launches never re-read what is still in L2
    # (smallest footprint: 2 x 134 MB > 126 MB L2).
    step_b = Step(x.clone(), w.clone(), gx.clone(), gw.clone())
    per_kernel_ms = []
    for i in range(4):
        for s_ in (step, step_b):
            s_.launch(i, stream)
        torch.cuda.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for k in range(K):
            (step if k % 2 == 0 else step_b).launch(i, stream)
        k1.record()
        k1.synchronize()
        per_kernel_ms.append(k0.elapsed_time(k1) / K)
    del step_b
    dom = max(range(4), key=lambda i: per_kernel_ms[i])
    achieved = step.kernel_bytes[dom] / (per_kernel_ms[dom] * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": step.names[dom], "achieved": round(achieved, 1), "peak": pk["hbm_gbs"],
        "unit": "GB/s", "frac": round(achieved / pk["hbm_gbs"], 4), "traffic": NCU_TRAFFIC.get(step.names[dom]),
        "peak_source": pk["source"], "bytes_per_launch": step.kernel_bytes[dom],
        "us_per_launch": round(per_kernel_ms[dom] * 1e3, 2),
        "timing": f"{K} back-to-back launches per kernel in one CUDA-event pair, alternating two buffer sets",
        "all_kernels": {n: {"us": round(ms * 1e3, 2), "GBps": round(b / ms / 1e6, 1),
                            "frac": round(b / ms / 1e6 / pk["hbm_gbs"], 4)}
                        for n, ms, b in zip(step.names, per_kernel_ms, step.kernel_bytes)},
        "sum_kernels_us": round(sum(per_kernel_ms) * 1e3, 2), "graph_step_us": round(ms_step * 1e3, 2),
    }

    if roofline["frac"] > 1.0:
        # not an error: MEASURED_PEAKS' HBM figure is a COPY (1 read : 1 write); the STE backward streams
        # 2 reads : 1 write, and a read-heavier mix pays fewer read/write bus turnarounds than a copy does
        # (the fp32 configs[0] kernels read 1.01-1.04 of the copy figure the same way)
        roofline["note"] = ("frac > 1: the peak is the measured copy bandwidth (1 read : 1 write); this kernel "
                            "streams 2 reads : 1 write, which HBM3e serves a few per cent faster than a copy")

    # ---- e2e: host (pinned) buffers through the C ABI host entry points
    Ke = max(3, min(K, 10))
    yx = torch.empty_like(hx).pin_memory()
    dxh = torch.empty_like(hx).pin_memory()
    yw = torch.empty_like(hw).pin_memory()
    dwh = torch.empty_like(hw).pin_memory()

    def e2e_step():
        fake_quant_fwd_bwd_host(hx, hgx, CLIP, A_BITS, symmetric=True, device=device, y=yx, gx=dxh)
        fake_quant_fwd_bwd_host(hw, hgw, CLIP, W_BITS, symmetric=True, device=device, y=yw, gx=dwh)

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(Ke):
        e2e_step()
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    if dist is not None:
        t = torch.tensor([e2e_ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e = {"value": round(world * STEP_BYTES * Ke / (e2e_ms * 1e-3) / 1e9, 2), "unit": "GB/s",
           "h2d_bytes_per_step": ELEMS * 2 * 2, "d2h_bytes_per_step": ELEMS * 2 * 2, "steps": Ke,
           "ms_per_step": round(e2e_ms / Ke, 3), "wall_ms_per_step": round(wall_ms / Ke, 3),
           "api": "llm_qat_b200.host_api.fake_quant_fwd_bwd_host -> qat_sym_fwd_bwd_host (pinned host buffers)"}

    # the host link's own ceiling with all ranks busy at once (plain pinned H2D + D2H of the same byte
    # counts, both directions concurrently): what the e2e figure is bounded by on this box
    try:
        e2e["link_probe"] = link_probe(device, hx, yx, barrier, dist)
    except Exception as e:  # noqa: BLE001
        e2e["link_probe"] = {"error": f"{type(e).__name__}: {e}"[:200]}

    extras = {}
    if rank == 0:
        try:
            extras["qlinear"] = time_qlinear(device, x, w, max(3, min(K, 20)), pk)
        except Exception as e:
            extras["qlinear"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            extras["config1_fp32"] = time_config1_fp32(device, max(4, min(K, 20)), pk)
        except Exception as e:
            extras["config1_fp32"] = {"error": f"{type(e).__name__}: {e}"}
        if args.shape_sweep:
            try:
                extras["shape_sweep"] = time_shape_sweep(device, max(3, min(K, 20)), pk)
            except Exception as e:
                extras["shape_sweep"] = {"error": f"{type(e).__name__}: {e}"}
    # ---- BASELINE configs[2] (decoder layer) and configs[3] / [4] (full QAT step, data-parallel), with the
    # comparator the north star names — the reference's eager-PyTorch GPU path (oracle/ref_module under the
    # same harness, same N, same autocast context) — measured in the same run.
    layer, qat = None, None
    if not args.no_qat_step:
        try:
            from harness import llama_qat as HQ
            from harness import qat_bench as QB
            from oracle import ref_module as RM

            if args.qat_model == "13b":   # BASELINE configs[4]: LLaMA-13B W4A8KV8 (180 GB/GPU sizing: DESIGN.md section 6)
                cfg7 = HQ.QatConfig.llama_13b(w_bits=4, a_bits=8, kv_bits=8)
                if args.qat_layers != 32:
                    cfg7.num_hidden_layers = args.qat_layers
            else:
                cfg7 = HQ.QatConfig.llama_7b(w_bits=4, a_bits=8, kv_bits=4, num_hidden_layers=args.qat_layers)
            del step, x, w, gx, gw
            torch.cuda.empty_cache()
            nst = max(3, min(K, 10))

            def reduce_max(ms):
                if dist is None:
                    return ms
                t = torch.tensor([ms], device=device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                return float(t.item())

            if rank == 0:   # configs[2]: one decoder layer fwd+bwd, seq 2048, inside autocast(bf16)
                layer = {"workload": f"configs[2]: LlamaDecoderLayer W{cfg7.w_bits}A{cfg7.a_bits}KV{cfg7.kv_bits} bf16, "
                                     f"hidden_states [1, 2048, {cfg7.hidden_size}], fwd + bwd, inside torch.autocast(bf16)"}
                for name, quant, fm in (("b200_fused_model", llm_qat_b200.utils_quant, True),
                                        ("b200_quant_path_only", llm_qat_b200.utils_quant, False),
                                        ("reference_eager_gpu", RM, False)):
                    layer[name] = QB.time_layer(quant, cfg7, warmup=3, steps=nst, device=device, autocast=True, fused=fm)
                layer["speedup_vs_reference_eager_gpu"] = round(layer["reference_eager_gpu"]["ms_fwd_bwd"] /
                                                                layer["b200_fused_model"]["ms_fwd_bwd"], 2)
            if dist is not None:
                dist.barrier()

            def qat_arm(quant, fm, steps_):
                QB.release_memory()
                if os.environ.get("BENCH_VERBOSE"):
                    print(f"[rank {rank}] arm start: {torch.cuda.memory_allocated(device) / 2**30:.1f} GiB allocated",
                          file=sys.stderr, flush=True)
                torch.cuda.reset_peak_memory_stats()
                r = QB.time_qat_step(quant, cfg7, seq=2048, bsz=1, warmup=3, steps=steps_, device=device, rank=rank,
                                     world=world, autocast=True,   # the recipe: HF's Trainer runs the step in autocast(bf16)
                                     fused=fm, bucket_cap_mb=args.bucket_cap_mb)
                ms = reduce_max(r["ms_per_step"])
                return dict(r, ms_per_step=round(ms, 2), tokens_per_s=round(world * 2048 / ms * 1e3), n_gpus=world)

            qat = qat_arm(llm_qat_b200.utils_quant, True, nst)
            qat["model"] = (("LLaMA-13B dims, random init, student W4A8KV8" if args.qat_model == "13b" else
                             "LLaMA-7B dims, random init, student W4A8KV4") + " + frozen FP teacher, KD (KL batchmean), "
                            "grad checkpointing, AdamW, bf16 inside torch.autocast(bf16) as kd_trainer.py:106 does; "
                            "llm_qat_b200.fuse_model + fused KD loss" + (", DDP/NCCL all-reduce" if world > 1 else ""))
            if world > 1 and (args.weight_shard or args.qat_model == "13b"):
                # BASELINE configs[4]: weights fake-quantized by output-channel shard (each rank quantizes
                # out/world channels of every QuantizeLinear) + all-gather of int8 codes / divisors / masks over
                # NVLink, against the replicated variant above (every rank quantizes every channel locally)
                from llm_qat_b200 import sharding as SH

                SH.enable_weight_sharding()
                try:
                    qat["weight_sharded"] = qat_arm(llm_qat_b200.utils_quant, True, nst)
                    qat["weight_sharded"]["what"] = (f"weights quantized by output-channel shard across {world} ranks, "
                                                     "codes all-gathered (1.125 B per weight element over NVLink)")
                except Exception as e:  # noqa: BLE001 - keep the arms already measured
                    qat["weight_sharded"] = {"error": f"{type(e).__name__}: {e}"[:300]}
                finally:
                    SH.disable_weight_sharding()
            if not args.no_comparators:
                try:
                    qat["quant_path_only"] = qat_arm(llm_qat_b200.utils_quant, False, max(3, nst // 2))
                    qat["reference_eager_gpu"] = qat_arm(RM, False, max(3, nst // 2))
                    qat["reference_eager_gpu"]["what"] = ("same harness, same N, the reference's eager op chain "
                                                          "(oracle/ref_module.py) on the GPU")
                    qat["speedup_vs_reference_eager_gpu"] = round(qat["reference_eager_gpu"]["ms_per_step"] / qat["ms_per_step"], 2)
                except Exception as e:  # noqa: BLE001
                    qat["comparators_error"] = f"{type(e).__name__}: {e}"[:300]
        except Exception as e:  # keep the headline line even if the big model cannot run
            qat = {"error": f"{type(e).__name__}: {e}"}
    torch.cuda.synchronize()
    clocks = sampler.stop()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = run_cpu_port(hx, hw, hgx, hgw, budget_s=12.0)

    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": "GB/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(ms_step, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": bench_config(world),
        "launch": "CUDA graph of one step, replayed K times" if used_graph else "direct launches",
        "gpu_launches": launches,
        "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu_baseline, "clocks": clocks,
    }
    line.update(extras)
    line["config3_layer"] = layer
    line["qat_step"] = qat
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------
# CPU port of the reference (cpu_baseline leg and --impl reference arm)
# ----------------------------------------------------------------------------
def run_cpu_port(hx, hw, hgx, hgw, budget_s: float, steps: int | None = None, warmup: int = 1, last=None):
    """Times oracle/torch_chain.py (the torch-eager port of utils_quant.py) on
    the host cores over the SAME workload; a step = fwd+bwd of x and of W.
    A dict passed as `last` receives the last step's (y, grad) of "x" and "w"."""
    from oracle import torch_chain as tc

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)

    def step():
        ox = tc.fwd_bwd(hx, hgx, A_BITS, True, CLIP)
        ow = tc.fwd_bwd(hw, hgw, W_BITS, True, CLIP)
        if last is not None:
            last["x"], last["w"] = ox, ow

    for _ in range(warmup):
        step()
    times = []
    t_start = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if steps is not None:
            if len(times) >= steps:
                break
        elif time.perf_counter() - t_start > budget_s or len(times) >= 50:
            break
    best = min(times)
    mean = statistics.mean(times)
    return {"value": round(STEP_BYTES / mean / 1e9, 3), "unit": "GB/s", "cores": cores, "kind": "port",
            "sample": f"full configs[1] step (x + W fwd+bwd, {ELEMS} bf16 elements) x {len(times)} "
                      f"repetitions, mean; best {STEP_BYTES / best / 1e9:.3f} GB/s",
            "ms_per_step": round(mean * 1e3, 1), "threads": torch.get_num_threads()}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    hx, hw, hgx, hgw = make_inputs(1234)
    K, W = args.steps, max(args.warmup, 3)      # the same K / W the b200 arm reports (~0.1-0.3 s per step)
    last = {} if args.dump_outputs else None
    cb = run_cpu_port(hx, hw, hgx, hgw, budget_s=0.0, steps=K, warmup=W, last=last)
    if last is not None:
        dump_outputs(args.dump_outputs, last["x"][0], last["w"][0], last["x"][1], last["w"][1])
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "GB/s",
        "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": bench_config(world),
        "arm_note": "reference's torch CPU path (oracle/torch_chain.py port; /root/reference cannot travel to the "
                    "GPU box), all host threads, rank 0 only",
        "gpu_launches": 0,
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-qat-step", action="store_true", help="skip the LLaMA-7B QAT-step extra (config 4)")
    ap.add_argument("--qat-layers", type=int, default=32)
    ap.add_argument("--no-comparators", action="store_true",
                    help="skip the reference-eager-GPU and quant-path-only arms of the QAT step")
    ap.add_argument("--bucket-cap-mb", type=int, default=None, help="DDP gradient bucket size of the QAT step")
    ap.add_argument("--weight-shard", action="store_true",
                    help="add the QAT-step arm with weights quantized by output-channel shard (default on for 13b)")
    ap.add_argument("--shape-sweep", action="store_true",
                    help="add per-shape / per-dtype / per-quantizer kernel timings (SURVEY.md 8d config 1)")
    ap.add_argument("--qat-model", default="7b", choices=["7b", "13b"],
                    help="model of the QAT-step extra: 7b = BASELINE configs[3], 13b = configs[4] (W4A8KV8)")
    ap.add_argument("--hang-dump-s", type=int, default=int(os.environ.get("BENCH_HANG_DUMP_S", "600")),
                    help="dump every thread's stack and exit if the run is still going after this many seconds")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (a fixed sample of "
                         f"{DUMP_ROWS} rows per operand) as float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import faulthandler

    # a stuck collective must not sit there until the driver's limit: report where each rank is and exit
    faulthandler.dump_traceback_later(args.hang_dump_s, exit=True)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
