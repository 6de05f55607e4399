#!/usr/bin/env python
"""GPU-box tool: the QuantizeLinear operand route (configurations off the int8 grid) on one B200.  Writes
profiles/r03_wide_linear.json (or the path given as argv[1]):

* K1 in QAT_BF16_AMP_CAST mode (y bf16 + packed mask) next to the QAT_BF16_AMP y (fp32) and GEMM-feed
  (int8 codes + divisors + mask) modes at the LLaMA-7B operand shapes: us, GB/s, share of the 7.7 TB/s
  HBM data-sheet bound.  Inputs rotate over > 256 MB of buffers, so every pass reads from HBM, not L2.
* a LLaMA-7B decoder layer fwd+bwd, seq 2048, under autocast (harness.qat_bench.time_layer) for the eight
  rows of the reference's accuracy table plus W4A32KV32 and W2A32KV32; four arms alternated in one process:
  route (fuse_model, linear=True), fuse_model(linear=False), the quant path only (no fuse_model) and the
  reference's eager chain (oracle/ref_module.py).  The route's and the linear=False outputs are compared at
  that size.
* one 32-layer W4A16KV16 QAT step (time_qat_step): fused against the reference eager chain, with peak memory.
(Test/bench infrastructure: may import oracle/.)"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from harness import llama_qat as H  # noqa: E402
from harness import qat_bench as B  # noqa: E402
from oracle import ref_module as R  # noqa: E402

HBM_BYTES_PER_S = 7.7e12      # HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip(),
            "torch_name": torch.cuda.get_device_name(0)}


def k1_modes():
    from llm_qat_b200 import utils_quant as uq
    from llm_qat_b200._lib import CODES_I8

    out = {}
    for rows, cols in ((2048, 4096), (2048, 11008), (11008, 4096)):
        n = rows * cols
        modes = {
            # name: (call, bytes moved per element)
            "amp_cast_y_bf16_mask": (lambda x: uq.fake_quant_forward(x, 4, False, True, amp=True, cast=True,
                                                                      mask_clip=(-2.0, 2.0)), 2 + 2 + 1 / 8),
            "amp_y_fp32": (lambda x: uq.fake_quant_forward(x, 4, False, True, amp=True), 2 + 4),
            "amp_feed_int8_mask": (lambda x: uq.fake_quant_forward(x, 4, False, True, amp=True, want_y=False,
                                                                   codes_kind=CODES_I8, want_scales=True,
                                                                   mask_clip=(-2.0, 2.0)), 2 + 1 + 1 / 8),
        }
        copies = max(2, -(-300 * 2 ** 20 // (n * 6)))
        xs = [torch.randn(rows, cols, device="cuda").bfloat16() for _ in range(copies)]
        res = {}
        for _ in range(2):          # alternate the modes twice, keep the better median
            for name, (fn, bpe) in modes.items():
                for i in range(copies):
                    fn(xs[i])
                torch.cuda.synchronize()
                times = []
                for rep in range(5):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for i in range(copies * 4):
                        fn(xs[i % copies])
                    e1.record()
                    e1.synchronize()
                    times.append(e0.elapsed_time(e1) * 1e3 / (copies * 4))
                us = statistics.median(times)
                if name not in res or us < res[name]["us"]:
                    gbs = n * bpe / (us * 1e-6) / 1e9
                    res[name] = {"us": round(us, 2), "GB_per_s": round(gbs, 1), "bytes_per_elem": round(bpe, 3),
                                 "share_of_hbm_bound": round(gbs * 1e9 / HBM_BYTES_PER_S, 3)}
        out[f"{rows}x{cols}"] = res
        print("k1", rows, cols, res, flush=True)
        del xs
    return out


ROWS = [(4, 8, 4), (4, 8, 8), (4, 6, 16), (4, 8, 16), (4, 16, 16), (8, 8, 4), (8, 8, 8), (8, 8, 16),
        (4, 32, 32), (2, 32, 32)]


def compare_route_and_unrouted(cfg):
    """Route vs fuse_model(linear=False) on one LLaMA-7B layer at seq 2048 under autocast: relative norms."""
    import llm_qat_b200

    torch.manual_seed(0)
    base = H.DecoderLayer(cfg, llm_qat_b200.utils_quant).bfloat16().cuda()
    with torch.no_grad():
        for p in base.parameters():
            if p.dim() == 2:
                p.normal_(0.0, cfg.initializer_range)
    g = torch.Generator().manual_seed(7)
    x0 = torch.randn(1, 2048, cfg.hidden_size, generator=g).bfloat16().cuda()
    go = torch.randn(1, 2048, cfg.hidden_size, generator=g).bfloat16().cuda()
    mask = H.causal_mask(1, 2048, torch.bfloat16, "cuda")
    llm_qat_b200.mark_causal_mask(mask)
    pos = torch.arange(2048, device="cuda")[None]
    res = []
    for linear in (True, False):
        llm_qat_b200.fuse_model(base, linear=linear)
        x = x0.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = base(x, mask, pos)
        y.backward(go)
        res.append([y.float(), x.grad.float()] + [p.grad.float() for p in base.parameters() if p.dim() == 2])
        for p in base.parameters():
            p.grad = None
    rel = [((a - b).norm() / b.norm()).item() for a, b in zip(*res)]
    del base, res
    B.release_memory()
    return {"rel_out": round(rel[0], 6), "rel_gx": round(rel[1], 6), "rel_gw_max": round(max(rel[2:]), 6),
            "within_4e-3": max(rel) <= 4e-3}


def layers():
    import llm_qat_b200

    arms = (("route", llm_qat_b200.utils_quant, dict(fused=True, linear=True)),
            ("linear_false", llm_qat_b200.utils_quant, dict(fused=True, linear=False)),
            ("quant_path_only", llm_qat_b200.utils_quant, dict(fused=False)),
            ("reference_eager_gpu", R, dict(fused=False)))
    out = {}
    for w, a, kv in ROWS:
        cfg = H.QatConfig.llama_7b(w_bits=w, a_bits=a, kv_bits=kv)
        row = {}
        for _ in range(2):           # arms alternated twice; the better median of each is kept
            for name, quant, kw in arms:
                r = B.time_layer(quant, cfg, autocast=True, warmup=3, steps=10, **kw)
                B.release_memory()
                if name not in row or r["ms_fwd_bwd"] < row[name]["ms_fwd_bwd"]:
                    row[name] = r
        entry = {name: row[name]["ms_fwd_bwd"] for name in row}
        entry["route_speedup_vs_linear_false"] = round(entry["linear_false"] / entry["route"], 3)
        entry["route_speedup_vs_reference"] = round(entry["reference_eager_gpu"] / entry["route"], 3)
        if not (3 <= w <= 8 and 3 <= a <= 8):
            entry["agreement_route_vs_linear_false"] = compare_route_and_unrouted(cfg)
        out[f"W{w}A{a}KV{kv}"] = entry
        print("layer", w, a, kv, entry, flush=True)
    return out


def qat_step():
    import llm_qat_b200

    cfg = H.QatConfig.llama_7b(w_bits=4, a_bits=16, kv_bits=16)
    out = {}
    for name, quant, fused in (("fused", llm_qat_b200.utils_quant, True), ("reference_eager_gpu", R, False)):
        torch.cuda.reset_peak_memory_stats()
        out[name] = B.time_qat_step(quant, cfg, autocast=True, fused=fused, warmup=2, steps=5)
        print("step", name, out[name], flush=True)
    out["speedup"] = round(out["reference_eager_gpu"]["ms_per_step"] / out["fused"]["ms_per_step"], 3)
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_wide_linear.json")
    result = {"card": card(), "k1_modes": k1_modes(), "layer_7b_seq2048_autocast_ms": layers(),
              "qat_step_7b_32_layers_W4A16KV16": qat_step()}
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
