"""Timing helpers for BASELINE configs 3 (decoder layer fwd+bwd) and 4/5 (full
QAT step with KD loss, data-parallel).  The quantization module is a parameter:
bench.py passes the product (llm_qat_b200.utils_quant); tests/gpu_layer_bench.py
also passes the oracle module to time the reference's eager GPU path."""
from __future__ import annotations

import contextlib
import statistics

import torch

from . import llama_qat as H


def release_memory():
    """DDP / autograd objects sit in reference cycles: without a collection the previous arm's 130 GB (13B)
    is still allocated when the next arm builds its models."""
    import gc

    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _timed(fn, warmup, steps):
    import os
    import sys
    import time

    verbose = bool(os.environ.get("BENCH_VERBOSE"))
    for i in range(warmup):
        t0 = time.perf_counter()
        fn()
        if verbose:
            torch.cuda.synchronize()
            print(f"[rank {os.environ.get('RANK', '0')}] warm-up step {i}: {time.perf_counter() - t0:.2f} s", file=sys.stderr, flush=True)
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return times


def time_layer(quant, cfg: H.QatConfig, seq=2048, bsz=1, warmup=3, steps=10, device="cuda", seed=1234,
               autocast=False, fused=False, linear=True):
    """Config 3: one LlamaDecoderLayer W4A8KV4 bf16, hidden_states [bsz, seq, H], fwd + bwd.
    ``fused``: llm_qat_b200.fuse_model on the layer (attention / MLP / RMSNorm kernels; ``linear``: its
    operand route for QuantizeLinear configurations off the int8 grid)."""
    torch.manual_seed(0)
    layer = H.DecoderLayer(cfg, quant).bfloat16().to(device)
    if fused:
        import llm_qat_b200

        llm_qat_b200.fuse_model(layer, linear=linear)
    with torch.no_grad():
        for p in layer.parameters():
            if p.dim() == 2:
                p.normal_(0.0, cfg.initializer_range)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(bsz, seq, cfg.hidden_size, generator=g).bfloat16().to(device).requires_grad_(True)
    go = torch.randn(bsz, seq, cfg.hidden_size, generator=g).bfloat16().to(device)
    mask = H.causal_mask(bsz, seq, torch.bfloat16, device)
    if fused:
        llm_qat_b200.mark_causal_mask(mask)
    pos = torch.arange(seq, device=device)[None].expand(bsz, seq)

    def step():
        with (torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()):
            y = layer(x, mask, pos)
        y.backward(go.to(y.dtype))
        x.grad = None
        for p in layer.parameters():
            p.grad = None

    t = _timed(step, warmup, steps)
    ms = statistics.median(t)
    return {"ms_fwd_bwd": round(ms, 3), "tokens_per_s": round(bsz * seq / ms * 1e3), "seq": seq, "bsz": bsz,
            "autocast": autocast, "fused_model": fused}


def time_qat_step(quant, cfg: H.QatConfig, seq=2048, bsz=1, warmup=3, steps=10, device="cuda", rank=0, world=1,
                  lr=2e-5, autocast=False, fused=False, bucket_cap_mb=None):
    """Config 4/5: student (quantized) + frozen FP teacher of identical init, KD loss,
    gradient checkpointing, AdamW; DDP (NCCL all-reduce of the gradients) when world > 1.
    Returns this rank's median step time; the caller reduces max over ranks."""
    torch.manual_seed(0)
    with torch.device(device):
        student = H.CausalLM(cfg, quant, fused=fused).bfloat16()
        teacher = H.build_teacher(cfg, fused=fused).bfloat16()
    teacher.load_state_dict(student.state_dict())
    student.train()
    model = student
    if world > 1:
        from torch.nn.parallel import DistributedDataParallel as DDP

        # one gradient bucket per decoder layer (~400 MB of bf16 gradients) instead of 25 MB ones: 34 all-reduces per
        # step instead of 540, less contention with the backward GEMMs; the model's only buffers are the rotary
        # tables, identical on every rank by construction, so the per-forward buffer broadcast is switched off
        model = DDP(student, device_ids=[torch.device(device).index], gradient_as_bucket_view=True,
                    bucket_cap_mb=400 if bucket_cap_mb is None else bucket_cap_mb, broadcast_buffers=False)
    opt = torch.optim.AdamW(student.parameters(), lr=lr)
    g = torch.Generator().manual_seed(1234 + rank)
    ids = torch.randint(0, cfg.vocab_size, (bsz, seq), generator=g).to(device)

    loss_fn = None
    if fused:
        import llm_qat_b200

        loss_fn = llm_qat_b200.fused_ops.kd_loss

    def step():
        H.qat_step(model, teacher, ids, opt, autocast=autocast, loss_fn=loss_fn)

    t = _timed(step, warmup, steps)
    ms = statistics.median(t)
    mem = torch.cuda.max_memory_allocated(device) / 2 ** 30
    del opt, model, student, teacher, step
    release_memory()
    return {"ms_per_step": round(ms, 2), "tokens_per_s_per_gpu": round(bsz * seq / ms * 1e3), "seq": seq,
            "bsz_per_gpu": bsz, "peak_mem_GiB": round(mem, 1), "layers": cfg.num_hidden_layers, "autocast": autocast,
            "fused_model": fused}
