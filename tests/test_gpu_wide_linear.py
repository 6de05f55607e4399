"""GPU (-m gpu): QuantizeLinear's operand route (utils_quant._OperandLinearFn) for configurations off the int8
grid — the reference's bf16 operands bit for bit, its contractions on qat_gemm_bf16, the new K1 output mode
QAT_BF16_AMP_CAST, and decoder layers / a short training run against the reference's eager chain."""
import functools

import numpy as np
import pytest
import torch

import qat_testutil as U
from harness import llama_qat as H
from oracle import ref_module as R

pytestmark = pytest.mark.gpu

CLIP = torch.tensor([-2.0, 2.0])


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert torch.cuda.is_available(), "these tests need a B200"
    import llm_qat_b200

    assert llm_qat_b200._lib.lib().qat_check_device() == 0, llm_qat_b200._lib.last_error()
    yield
    torch.cuda.synchronize()


def _uq():
    from llm_qat_b200 import utils_quant

    return utils_quant


def _pack(bits: torch.Tensor) -> torch.Tensor:
    return torch.from_numpy(np.packbits(bits.cpu().numpy().reshape(-1), bitorder="little")).cuda()


def _ref_mask(t):
    """utils_quant.py:85-86: the gradient is zeroed where x >= hi or x <= lo (NaN passes), packed."""
    return _pack(~((t >= 2.0) | (t <= -2.0)))


def _ref_operand(t, bits, amp):
    """What the reference hands F.linear for a SymQuantizer-quantized operand, and its packed STE mask."""
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        y = R.SymQuantizer.apply(t, CLIP, bits, False)
    return y.to(torch.bfloat16), _ref_mask(t)


def _direct_gemm(a, b, mask, M, N, K, a_mn, b_mn, cg):
    from llm_qat_b200 import _lib

    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    _lib.check(_lib.lib().qat_gemm_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), 0 if mask is None else mask.data_ptr(),
                                        M, N, K, a_mn, b_mn, 1, cg, torch.cuda.current_stream().cuda_stream), "qat_gemm_bf16")
    return out


def _marked(K, N, w_bits, a_bits, w0):
    import llm_qat_b200

    lin = _uq().QuantizeLinear(K, N, w_bits=w_bits, a_bits=a_bits).bfloat16().cuda()
    with torch.no_grad():
        lin.weight.copy_(w0)
    llm_qat_b200.fuse_model(lin)
    assert lin.__dict__.get("_qat_operand_route")
    return lin


# --------------------------------------------------------------- operands and contractions, bit for bit
@pytest.mark.parametrize("w_bits,a_bits", [(4, 16), (2, 32), (32, 16), (12, 32)])
@pytest.mark.parametrize("amp", [False, True])
@pytest.mark.parametrize("T,K,N", [(200, 1040, 264), (2048, 4096, 11008)])
@pytest.mark.parametrize("cg", [1, 2])
def test_route_is_the_library_gemm_on_the_reference_operands(w_bits, a_bits, amp, T, K, N, cg, monkeypatch):
    uq = _uq()
    monkeypatch.setattr(uq, "gemm_bf16", functools.partial(uq.gemm_bf16, cta_group=cg))
    gen = torch.Generator().manual_seed(T + w_bits)
    x0 = (torch.randn(T, K, generator=gen) * 1.3).bfloat16().cuda()
    w0 = (torch.randn(N, K, generator=gen) * 0.05).bfloat16().cuda()
    w0[0, :4] = torch.tensor([2.5, -2.0, 1.99, -3.0])   # clip edges of the weight's STE mask
    g0 = torch.randn(T, N, generator=gen).bfloat16().cuda()
    xq, xm = _ref_operand(x0, a_bits, amp) if 2 < a_bits < 32 else (x0, None)
    if w_bits >= 32:
        wq, wm = w0, None
    elif w_bits >= 3:
        wq, wm = _ref_operand(w0, w_bits, amp)
    else:
        wq, wm = uq.lowbit_weight(w0, w_bits, False), None       # _LowBitWeight's output, identity gradient
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            assert torch.equal(uq._LowBitWeight.apply(w0, w_bits, False), wq)
    lin = _marked(K, N, w_bits, a_bits, w0)
    x = x0.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        out = lin(x)
    out.backward(g0)
    assert out.dtype == torch.bfloat16
    assert torch.equal(out, _direct_gemm(xq, wq, None, T, N, K, 0, 0, cg))
    assert torch.equal(x.grad, _direct_gemm(g0, wq, xm, T, K, N, 0, 1, cg))
    assert torch.equal(lin.weight.grad, _direct_gemm(g0, xq, wm, N, K, T, 1, 1, cg))


# --------------------------------------------------------------- against the reference chain
_GRID = [(w, a) for w in (1, 2, 4, 8, 16, 32) for a in (4, 8, 16, 32)
         if not (w in (4, 8) and a in (4, 8)) and (w, a) != (32, 32)]


@pytest.mark.parametrize("w_bits,a_bits", _GRID)
@pytest.mark.parametrize("amp", [False, True])
def test_route_vs_reference_chain(w_bits, a_bits, amp):
    gen = torch.Generator().manual_seed(17)
    T, K, N = 384, 1024, 776
    x0 = (torch.randn(2, T // 2, K, generator=gen) * 1.3).bfloat16().cuda()
    w0 = (torch.randn(N, K, generator=gen) * 0.05).bfloat16().cuda()
    g0 = torch.randn(2, T // 2, N, generator=gen).bfloat16().cuda()
    res = []
    for lin in (R.QuantizeLinear(K, N, w_bits=w_bits, a_bits=a_bits).bfloat16().cuda(), _marked(K, N, w_bits, a_bits, w0)):
        with torch.no_grad():
            lin.weight.copy_(w0)
        x = x0.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            out = lin(x)
        out.backward(g0)
        res.append((out, x.grad, lin.weight.grad))
    for a, b in zip(*res):
        assert a.dtype == b.dtype and a.shape == b.shape
        rel = ((a.double() - b.double()).norm() / a.double().norm()).item()
        assert rel <= 4e-3, (w_bits, a_bits, amp, rel)


# --------------------------------------------------------------- launches
def test_w4a16_runs_only_own_kernels():
    from llm_qat_b200 import _lib

    gen = torch.Generator().manual_seed(9)
    T, K, N = 512, 1024, 1536
    x = (torch.randn(T, K, generator=gen) * 1.2).bfloat16().cuda().requires_grad_(True)
    lin = _marked(K, N, 4, 16, (torch.randn(N, K, generator=gen) * 0.02).bfloat16().cuda())
    g0 = torch.randn(T, N, generator=gen).bfloat16().cuda()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = lin(x)
        n1 = _lib.launch_count()
        out.backward(g0)
        torch.cuda.synchronize()
    assert (n1 - n0, _lib.launch_count() - n1) == (3, 2)       # 2 operands + 1 GEMM; dgrad + wgrad
    kernels = [e.key for e in prof.key_averages()]
    assert not any(("nvjet" in k or "gemm" in k.lower() or "cutlass" in k.lower()) and "gemm_bf16_kernel" not in k
                   for k in kernels), kernels
    assert not any("ste" in k.lower() for k in kernels), kernels       # masks are applied in the GEMM epilogue


def _three_consumers_with_checkpoint(amp):
    """q/k/v-like: three marked linears read one tensor, inside a checkpointed block."""
    gen = torch.Generator().manual_seed(21)
    K, N = 512, 512
    lins = [_marked(K, N, 4, 16, (torch.randn(N, K, generator=gen) * 0.05).bfloat16().cuda()) for _ in range(3)]
    x = (torch.randn(2, 96, K, generator=gen) * 1.2).bfloat16().cuda().requires_grad_(True)
    g = torch.randn(2, 96, N, generator=gen).bfloat16().cuda()

    def block(h):
        return sum(lin(h) for lin in lins)

    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        out = torch.utils.checkpoint.checkpoint(block, x, use_reentrant=False)
    out.backward(g)
    return [out, x.grad] + [lin.weight.grad for lin in lins]


@pytest.mark.parametrize("amp", [False, True])
def test_operand_reuse_and_cache_modes_give_equal_results(amp, monkeypatch):
    uq = _uq()
    calls = []
    orig = uq.quant_operand

    def counting(t, bits, a):
        calls.append(tuple(t.shape))
        return orig(t, bits, a)

    monkeypatch.setattr(uq, "quant_operand", counting)
    results = {}
    for mode in ("0", "1", "2"):
        monkeypatch.setenv("QAT_B200_CACHE", mode)
        calls.clear()
        results[mode] = _three_consumers_with_checkpoint(amp)
        n_x = sum(1 for c in calls if c == (192, 512))
        n_w = len(calls) - n_x
        if mode == "0":
            assert (n_x, n_w) == (6, 6), calls          # forward + recompute, every consumer for itself
        else:
            assert n_x <= 2 and n_w == 3, calls         # x once per pass; weights reused by the recompute
    for mode in ("1", "2"):
        for a, b in zip(results["0"], results[mode]):
            assert torch.equal(a, b)


# --------------------------------------------------------------- K1 in QAT_BF16_AMP_CAST mode
@pytest.mark.parametrize("bits", [3, 4, 8, 16, 24])
@pytest.mark.parametrize("shape", [(33, 7), (17, 1000), (9, 1023), (64, 4096), (3, 11008), (2, 40000)])
def test_k1_cast_mode_is_the_autocast_chain_then_cast(bits, shape):
    from llm_qat_b200 import SymQuantizer

    uq = _uq()
    gen = torch.Generator().manual_seed(bits * 7 + shape[1])
    x = (torch.randn(*shape, generator=gen) * 1.7).bfloat16()
    x[0] = 0.0
    if shape[0] > 3:
        x[1, 0], x[2, shape[1] // 2], x[3, -1] = float("nan"), float("inf"), -float("inf")
    x = x.cuda()
    want_mask = shape[1] % 8 == 0
    y, _, _, _, mask = uq.fake_quant_forward(x, bits, False, True, amp=True, cast=True,
                                             mask_clip=(-2.0, 2.0) if want_mask else None)
    assert y.dtype == torch.bfloat16
    with torch.autocast("cuda", dtype=torch.bfloat16):
        own = SymQuantizer.apply(x, CLIP, bits, False)
        ref = R.SymQuantizer.apply(x, CLIP, bits, False)
    assert own.dtype == torch.float32
    for other in (own.to(torch.bfloat16), ref.to(torch.bfloat16)):
        assert U.mismatches(U.tensor_bits(y), U.tensor_bits(other), "bf16") == 0
    if want_mask:
        assert torch.equal(mask, _ref_mask(x))


def test_k1_cast_mode_is_rejected_where_it_does_not_apply():
    from llm_qat_b200 import _lib

    L = _lib.lib()
    x = torch.randn(4, 64, device="cuda").bfloat16()
    codes = torch.empty(4, 64, dtype=torch.int8, device="cuda")
    e = torch.empty(4, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    assert L.qat_sym_feed(x.data_ptr(), codes.data_ptr(), e.data_ptr(), 0, -2.0, 2.0, 4, 64,
                          _lib.QAT_BF16_AMP_CAST, 4, st) == 1001
    y = torch.empty_like(x)
    assert L.qat_asym_fwd(x.data_ptr(), y.data_ptr(), 0, 0, 0, 0, 0, -2.0, 2.0, 4, 64, _lib.QAT_BF16_AMP_CAST, 4,
                          0, 0, st) == 1001


# --------------------------------------------------------------- K/V at 16 bits
@pytest.mark.parametrize("amp", [False, True])
def test_qkv_prep_at_kv16_equals_kv_fake_quant_then_rope(amp):
    import test_gpu_parity as P

    P.test_qkv_prep_equals_kv_fake_quant_then_rope(amp, 16)


# --------------------------------------------------------------- decoder layers and training
def _layer_pair(cfg, linear=True):
    import llm_qat_b200

    torch.manual_seed(0)
    ref = H.DecoderLayer(cfg, R).bfloat16().cuda()
    new = H.DecoderLayer(cfg, llm_qat_b200.utils_quant).bfloat16().cuda()
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() == 2:
                p.normal_(0.0, 0.02)
            else:
                p.uniform_(0.5, 1.5)
    new.load_state_dict(ref.state_dict())
    llm_qat_b200.fuse_model(new, linear=linear)
    return ref, new


def _run_layer(layer, x0, go, mask, pos, autocast):
    import llm_qat_b200

    x = x0.clone().requires_grad_(True)
    n0 = llm_qat_b200._lib.launch_count()
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        y = layer(x, mask, pos)
    y.backward(go)
    grads = {n: p.grad.float() for n, p in layer.named_parameters()}
    return y.float(), x.grad.float(), grads, llm_qat_b200._lib.launch_count() - n0


def _layer_inputs():
    g = torch.Generator().manual_seed(5)
    x0 = torch.randn(2, 256, 512, generator=g).bfloat16().cuda()
    go = torch.randn(2, 256, 512, generator=g).bfloat16().cuda()
    mask = H.causal_mask(2, 256, torch.bfloat16, "cuda")
    pos = torch.arange(256, device="cuda")[None].expand(2, 256)
    return x0, go, mask, pos


_LAYER_CFG = dict(hidden_size=512, intermediate_size=1376, num_attention_heads=4, num_hidden_layers=1,
                  max_position_embeddings=256)


@pytest.mark.parametrize("w_bits,a_bits,kv_bits", [(4, 16, 16), (4, 32, 32), (2, 32, 32), (8, 16, 8)])
@pytest.mark.parametrize("autocast", [False, True])
def test_fused_decoder_layer_off_the_grid_matches_reference_chain(w_bits, a_bits, kv_bits, autocast):
    import llm_qat_b200

    cfg = H.QatConfig(**_LAYER_CFG, w_bits=w_bits, a_bits=a_bits, kv_bits=kv_bits)
    ref, new = _layer_pair(cfg)
    assert all(m.__dict__.get("_qat_operand_route") for m in new.modules() if isinstance(m, llm_qat_b200.QuantizeLinear))
    x0, go, mask, pos = _layer_inputs()
    y_r, gx_r, gr_r, _ = _run_layer(ref, x0, go, mask, pos, autocast)
    llm_qat_b200.mark_causal_mask(mask)
    y, gx, gr, launches = _run_layer(new, x0, go, mask, pos, autocast)
    rel = lambda a, b: ((a - b).norm() / b.norm().clamp_min(1e-30)).item()  # noqa: E731
    assert rel(y, y_r) <= 1e-2, rel(y, y_r)
    assert rel(gx, gx_r) <= 3e-2, rel(gx, gx_r)
    for n in gr_r:
        assert rel(gr[n], gr_r[n]) <= 3e-2, (n, rel(gr[n], gr_r[n]))
    assert launches >= 30, launches


def test_grid_layer_issues_the_same_launches_with_and_without_the_route():
    import llm_qat_b200

    cfg = H.QatConfig(**_LAYER_CFG, w_bits=4, a_bits=8, kv_bits=8)
    x0, go, mask, pos = _layer_inputs()
    llm_qat_b200.mark_causal_mask(mask)
    counts, outs = [], []
    for linear in (True, False):
        _, new = _layer_pair(cfg, linear=linear)
        assert not any(m.__dict__.get("_qat_operand_route") for m in new.modules())
        y, gx, _, launches = _run_layer(new, x0, go, mask, pos, True)
        counts.append(launches)
        outs.append((y, gx))
    assert counts[0] == counts[1], counts
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_w4a16kv16_training_trajectory_tracks_the_reference_chain():
    import llm_qat_b200

    cfg = H.QatConfig(hidden_size=256, intermediate_size=688, num_attention_heads=2, num_hidden_layers=2,
                      vocab_size=512, max_position_embeddings=128, w_bits=4, a_bits=16, kv_bits=16)

    def run(quant, fused):
        torch.manual_seed(0)
        student = H.CausalLM(cfg, quant, fused=fused).bfloat16().cuda()
        teacher = H.build_teacher(cfg, fused=fused).bfloat16().cuda()
        teacher.load_state_dict(student.state_dict())
        with torch.no_grad():
            for p in student.parameters():
                p.add_(torch.randn(p.shape, generator=torch.Generator().manual_seed(p.numel())).to(p).mul_(0.01))
        opt = torch.optim.AdamW(student.parameters(), lr=1e-3)
        g = torch.Generator().manual_seed(99)
        losses = []
        for _ in range(30):
            ids = torch.randint(0, cfg.vocab_size, (2, 128), generator=g).cuda()
            losses.append(float(H.qat_step(student.train(), teacher, ids, opt, autocast=True,
                                           loss_fn=llm_qat_b200.fused_ops.kd_loss if fused else None)))
        return losses

    ref = run(R, False)
    fused = run(llm_qat_b200.utils_quant, True)
    assert all(np.isfinite(fused)) and fused[-1] < fused[0]
    rel = max(abs(a - b) / abs(b) for a, b in zip(fused, ref))
    assert rel < 0.15 and abs(fused[-1] - ref[-1]) / ref[-1] < 0.15, (rel, fused[-3:], ref[-3:])
