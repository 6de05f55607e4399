"""GPU (-m gpu): the CUDA path, called through the reference-shaped Python
boundary over the C ABI, against (i) the golden vectors generated from the live
reference and (ii) the oracle on seeded inputs, bit for bit."""
import numpy as np
import pytest
import torch

import qat_testutil as U
from oracle import quant_oracle as qo

pytestmark = pytest.mark.gpu

CLIP = torch.tensor([-2.0, 2.0])


def _q(name):
    from llm_qat_b200 import AsymQuantizer, SymQuantizer

    return SymQuantizer if name == "sym" else AsymQuantizer


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert torch.cuda.is_available(), "these tests need a B200"
    import llm_qat_b200

    assert llm_qat_b200._lib.lib().qat_check_device() == 0, llm_qat_b200._lib.last_error()
    yield
    torch.cuda.synchronize()


# --------------------------------------------------------------- golden vectors
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_forward_bit_exact_vs_reference_goldens(dtype):
    g = U.golden(dtype)
    bad = []
    for q, key, bits, lw in U.quant_cases(g):
        x = U.bits_to_tensor(g[f"in/{key}"], dtype, "cuda")
        y = _q(q).apply(x, CLIP, bits, lw)
        assert y.shape == x.shape and y.dtype == x.dtype and y.is_contiguous()
        ref = g[f"y/{q}/{key}/b{bits}/{'lw' if lw else 'row'}"]
        nm = U.mismatches(U.tensor_bits(y), ref, dtype)
        if nm:
            bad.append((q, key, bits, lw, nm, ref.size))
    assert not bad, bad


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_backward_bit_exact_vs_reference_goldens(dtype):
    g = U.golden(dtype)
    bad = []
    for q, key, lw, lo, hi, gk in U.clip_cases(g):
        x = U.bits_to_tensor(g[f"in/{key}"], dtype, "cuda").requires_grad_(True)
        gr = U.bits_to_tensor(g[f"grad/{key}"], dtype, "cuda")
        bits = 2 if q == "sym" else 3
        y = _q(q).apply(x, torch.tensor([lo, hi]), bits, lw)
        y.backward(gr)
        nm = U.mismatches(U.tensor_bits(x.grad), g[gk], dtype)
        if nm:
            bad.append((gk, nm))
    assert not bad, bad


# --------------------------------------------------------------- hoisted-reciprocal division
@pytest.mark.parametrize("bf16_operands", [0, 1])
def test_fast_division_matches_div_rn_on_device(bf16_operands):
    """K1/K2 replace the per-element div.rn by 3 FP ops on a per-row reciprocal;
    ~2.7e9 random operand pairs (x2 kinds) must agree with div.rn bit for bit."""
    import llm_qat_b200

    L = llm_qat_b200._lib.lib()
    counters = torch.zeros(6, dtype=torch.int64, device="cuda")
    for seed in (1, 2):
        rc = L.qat_selftest_fastdiv(seed * 7919, 1 << 20, 1280, bf16_operands, counters.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream)
        llm_qat_b200._lib.check(rc, "qat_selftest_fastdiv")
    bad, n, bad_i, n_i, bad_w, n_w = counters.tolist()
    print(f"fastdiv self-test: general {bad}/{n}, integer {bad_i}/{n_i}, wide (informational) {bad_w}/{n_w}")
    assert n > 2e9 and n_i > 2e9, (n, n_i)
    assert bad == 0 and bad_i == 0, (bad, n, bad_i, n_i)


# --------------------------------------------------------------- codes, scales, masks vs oracle
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("sym", [True, False])
def test_codes_scales_and_mask_bit_exact_vs_oracle(dtype, sym):
    from llm_qat_b200._lib import CODES_I8, CODES_I16
    from llm_qat_b200.utils_quant import fake_quant_forward

    gen = torch.Generator().manual_seed(5)
    x = (torch.randn(96, 1024, generator=gen) * 0.7)
    x[3] = 0.0
    x[5, 7] = 2.0
    x[5, 8] = -2.0
    x[7, ::5] = 3.0
    x = x.to(U.DTYPES[dtype])
    xn = U.tensor_to_f32(x)
    for bits in (4, 8):
        y, c16, st0, st1, mask = fake_quant_forward(x.cuda(), bits, False, sym, codes_kind=CODES_I16,
                                                    want_scales=True, mask_clip=(-2.0, 2.0))
        o = (qo.sym_forward if sym else qo.asym_forward)(xn, bits, False, dtype)
        assert qo.count_mismatch(U.tensor_to_f32(y), o["y"]) == 0
        np.testing.assert_array_equal(c16.cpu().numpy(), o["codes"].astype(np.int16))
        if sym:
            assert U.f32_mismatches(st0.cpu().numpy(), o["s"]) == 0
            assert U.f32_mismatches(st1.cpu().numpy(), o["e"]) == 0
        else:
            assert U.f32_mismatches(st0.cpu().numpy(), o["a"]) == 0
            assert U.f32_mismatches(st1.cpu().numpy(), o["beta"]) == 0
        ob = qo.ste_backward(np.ones_like(xn), xn, -2.0, 2.0, dtype)
        np.testing.assert_array_equal(mask.cpu().numpy(), qo.pack_mask(ob["mask"]))
        # int8 GEMM feed: exact wherever the code fits, saturated otherwise
        _, c8, _, _, _ = fake_quant_forward(x.cuda(), bits, False, sym, want_y=False, codes_kind=CODES_I8)
        lo8, hi8 = (-128, 127) if sym else (0, 255)
        np.testing.assert_array_equal(c8.cpu().numpy().astype(np.int32),
                                      np.clip(o["codes"], lo8, hi8).astype(np.int32))


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_backward_mask_variants_agree(dtype):
    from llm_qat_b200.utils_quant import fake_quant_forward, ste_backward, ste_backward_from_mask

    gen = torch.Generator().manual_seed(11)
    for shape in [(64, 4096), (33, 1000), (1, 8), (5, 12)]:
        x = (torch.randn(*shape, generator=gen) * 1.5).to(U.DTYPES[dtype]).cuda()
        g = torch.randn(*shape, generator=gen).to(U.DTYPES[dtype]).cuda()
        gx, mask = ste_backward(g, x, CLIP, want_mask=True)
        ob = qo.ste_backward(U.tensor_to_f32(g), U.tensor_to_f32(x), -2.0, 2.0, dtype)
        assert qo.count_mismatch(U.tensor_to_f32(gx), ob["gx"]) == 0
        np.testing.assert_array_equal(mask.cpu().numpy(), qo.pack_mask(ob["mask"]))
        gx2 = ste_backward_from_mask(g, mask)
        assert torch.equal(gx.view(torch.int16 if dtype == "bf16" else torch.int32),
                           gx2.view(torch.int16 if dtype == "bf16" else torch.int32))
        if shape[1] % 8 == 0:
            _, _, _, _, fmask = fake_quant_forward(x, 4, False, True, mask_clip=(-2.0, 2.0))
            assert torch.equal(fmask, mask)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_cuda_clip_val_is_read_in_kernel(dtype):
    """clip_val may live on the GPU (the reference indexes it as 0-dim tensors, :85-86): the kernel
    reads the two bounds itself — same result as the host-scalar path, for bounds that are and are
    not representable in the tensor dtype (x.ge(clip) compares in x's dtype)."""
    from llm_qat_b200 import AsymQuantizer, SymQuantizer

    gen = torch.Generator().manual_seed(9)
    x = (torch.randn(33, 1000, generator=gen) * 1.5).to(U.DTYPES[dtype])
    x.view(-1)[:6] = torch.tensor([2.0, -2.0, 1.703125, -1.296875, 1.7, -1.3]).to(x.dtype)
    g = torch.randn(33, 1000, generator=gen).to(U.DTYPES[dtype])
    for clip in ([-2.0, 2.0], [-1.3, 1.7]):
        outs = []
        for dev in ("cpu", "cuda"):
            for Q in (SymQuantizer, AsymQuantizer):
                xi = x.cuda().requires_grad_(True)
                Q.apply(xi, torch.tensor(clip, device=dev), 8, False).backward(g.cuda())
                outs.append(xi.grad)
        want = qo.ste_backward(U.tensor_to_f32(g), U.tensor_to_f32(x), clip[0], clip[1], dtype)["gx"]
        for o in outs:
            assert qo.count_mismatch(U.tensor_to_f32(o), want) == 0, (clip, dtype)


# --------------------------------------------------------------- shapes / modes at scale vs oracle
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("shape,lw", [
    ((512, 4096), False),        # activations: per token
    ((256, 11008), False),       # down_proj input / weight rows of 11008
    ((2, 64, 4096), False),      # K/V [b, s, hidden]
    ((3, 5, 7, 24), False),      # 4-D per (b, h)
    ((300, 4096), True),         # layerwise: two-phase long-row path
    ((4, 40000), False),         # rows too long for registers
    ((17, 8200), False),         # scalar-path long rows (8200*4 % 16 != 0 for bf16? -> vec for fp32)
    ((9, 1023), False),          # odd width -> scalar path
    ((1, 70001), True),
])
def test_shapes_and_modes_bit_exact_vs_oracle(dtype, shape, lw):
    gen = torch.Generator().manual_seed(hash(shape) % 1000)
    x = (torch.randn(*shape, generator=gen) * 0.5).to(U.DTYPES[dtype])
    x.view(-1)[::997] *= 9.0
    xn = U.tensor_to_f32(x)
    for q, fn in (("sym", qo.sym_forward), ("asym", qo.asym_forward)):
        for bits in (4, 8):
            y = _q(q).apply(x.cuda(), CLIP, bits, lw)
            nm = qo.count_mismatch(U.tensor_to_f32(y), fn(xn, bits, lw, dtype)["y"])
            assert nm == 0, (q, bits, shape, lw, nm)


def test_unaligned_and_noncontiguous_inputs():
    from llm_qat_b200 import SymQuantizer

    gen = torch.Generator().manual_seed(2)
    base = torch.randn(64 * 260 + 3, generator=gen).cuda()
    x = base[3:].view(64, 260)                       # 12-byte offset -> scalar path
    y = SymQuantizer.apply(x, CLIP, 4, False)
    assert qo.count_mismatch(U.tensor_to_f32(y), qo.sym_forward(U.tensor_to_f32(x), 4)["y"]) == 0
    xt = torch.randn(128, 96, generator=gen).cuda().t()   # non-contiguous 2-D: reduce over its last dim
    y = SymQuantizer.apply(xt, CLIP, 8, False)
    assert qo.count_mismatch(U.tensor_to_f32(y), qo.sym_forward(U.tensor_to_f32(xt), 8)["y"]) == 0
    with pytest.raises(ValueError):
        SymQuantizer.apply(torch.zeros(1, 1, 1, 1, 2).cuda(), CLIP, 4, False)
    with pytest.raises(RuntimeError):
        SymQuantizer.apply(torch.zeros(2, 3, 4, 8).cuda().transpose(1, 2), CLIP, 4, False)


# --------------------------------------------------------------- seeded fuzz: shapes x bits x dtypes
@pytest.mark.parametrize("seed", range(12))
def test_fuzz_forward_backward_bit_exact_vs_oracle(seed):
    """qat_testutil.fuzz_cases: random shapes x bit widths x dtypes x edge values (also the bit
    widths that leave the packed-bf16 and single-multiply fast paths): y and the STE gradient bit
    for bit against the oracle, which tests/test_oracle.py pins to the live reference on the
    very same cases."""
    for what, dtype, sym, bits, lw, x, g in U.fuzz_cases(seed):
        xi = x.cuda().requires_grad_(True)
        y = _q("sym" if sym else "asym").apply(xi, CLIP, bits, lw)
        y.backward(g.cuda())
        ref = (qo.sym_forward if sym else qo.asym_forward)(U.tensor_to_f32(x), bits, lw, dtype)["y"]
        assert qo.count_mismatch(U.tensor_to_f32(y), ref) == 0, what
        gref = qo.ste_backward(U.tensor_to_f32(g), U.tensor_to_f32(x), -2.0, 2.0, dtype)["gx"]
        assert qo.count_mismatch(U.tensor_to_f32(xi.grad), gref) == 0, what


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_wide_bit_widths_take_the_exact_division(dtype):
    """num_bits up to 31 (the reference accepts any): codes beyond 15/16 bits leave the proven range
    of the reciprocal-based quotient, so those rows divide exactly — still bit for bit."""
    gen = torch.Generator().manual_seed(17)
    x = (torch.randn(24, 1000, generator=gen) * 1.3).to(U.DTYPES[dtype])
    x[0] = 0.0
    x[1, :5] = torch.tensor([2.0, -2.0, -0.0, 1e-20, -3e4]).to(x.dtype)
    xn = U.tensor_to_f32(x)
    for q, fn, widths in (("sym", qo.sym_forward, (16, 17, 20, 24, 25, 31)), ("asym", qo.asym_forward, (15, 16, 20, 24, 31))):
        for bits in widths:
            y = _q(q).apply(x.cuda(), CLIP, bits, False)
            assert qo.count_mismatch(U.tensor_to_f32(y), fn(xn, bits, False, dtype)["y"]) == 0, (q, bits, dtype)


# --------------------------------------------------------------- dependent chains, no host sync in between
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_dependent_kernel_chain_without_syncs(dtype):
    """Every kernel is launched with programmatic dependent launch: its CTAs may be resident while
    the previous kernel of the stream still runs.  A chain in which each launch consumes what the
    previous one has just written (quantizer on quantizer output, K3 on fresh gradients, the GEMM
    on fresh codes), enqueued back to back many times without a host synchronisation, must give the
    oracle's bits — a misplaced griddepcontrol.wait would read half-written data."""
    from llm_qat_b200 import _lib
    from llm_qat_b200._lib import CODES_I8
    from llm_qat_b200.utils_quant import fake_quant_forward, qlinear_i8, ste_backward

    gen = torch.Generator().manual_seed(321)
    x0 = (torch.randn(512, 4096, generator=gen) * 0.7).to(U.DTYPES[dtype])
    g0 = torch.randn(512, 4096, generator=gen).to(U.DTYPES[dtype])
    w = (torch.randn(256, 4096, generator=gen) * 0.05).to(U.DTYPES[dtype]).cuda()
    xd, gd = x0.cuda(), g0.cuda()
    plan = [(True, 8), (False, 8), (True, 4), (False, 4), (True, 6)]
    finals = []
    for rep in range(30):
        t = xd
        for sym, bits in plan:                       # each stage reads the previous stage's output
            t = fake_quant_forward(t, bits, False, sym)[0]
        gx = ste_backward(gd, t, CLIP)               # K3 on the chain's fresh output
        gx = ste_backward(gx, xd, CLIP)              # and on K3's own fresh output
        _, qx, _, ex, _ = fake_quant_forward(t, 8, False, True, want_y=False, codes_kind=CODES_I8, want_scales=True)
        _, qw, _, ew, _ = fake_quant_forward(w, 4, False, True, want_y=False, codes_kind=CODES_I8, want_scales=True)
        out = qlinear_i8(qx, qw, ex, ew, torch.float32)   # GEMM on codes written by the two launches before it
        finals.append((t, gx, out))
    torch.cuda.synchronize()
    ref = U.tensor_to_f32(x0)
    for sym, bits in plan:
        ref = (qo.sym_forward if sym else qo.asym_forward)(ref, bits, False, dtype)["y"]
    gref = qo.ste_backward(U.tensor_to_f32(g0), ref, -2.0, 2.0, dtype)["gx"]
    gref = qo.ste_backward(gref, U.tensor_to_f32(x0), -2.0, 2.0, dtype)["gx"]
    o = qo.sym_forward(ref, 8, False, dtype)
    ow = qo.sym_forward(U.tensor_to_f32(w), 4, False, dtype)
    dot = np.clip(o["codes"], -128, 127).astype(np.float64) @ np.clip(ow["codes"], -128, 127).astype(np.float64).T
    oref = ((dot.astype(np.float32) * (np.float32(1) / o["e"].astype(np.float32))[:, None]) *
            (np.float32(1) / ow["e"].astype(np.float32))[None, :]).astype(np.float32)
    for t, gx, out in (finals[0], finals[-1], finals[13]):
        assert qo.count_mismatch(U.tensor_to_f32(t), ref) == 0
        assert qo.count_mismatch(U.tensor_to_f32(gx), gref) == 0
        assert qo.count_mismatch(out.cpu().numpy(), oref) == 0
    assert _lib.launch_count() > 0


# --------------------------------------------------------------- config 5: LLaMA-13B shapes, 8 shards
@pytest.mark.parametrize("shape,bits,what", [
    ((13824, 5120), 4, "gate/up_proj weight: sharded by output channel"),
    ((5120, 13824), 4, "down_proj weight: sharded by output channel"),
    ((1, 2048, 5120), 8, "K/V of one sequence, KV8: sharded by token"),
])
def test_config5_shards_reassemble_bit_exact(shape, bits, what):
    """BASELINE configs[4]: every statistic is row-local, so the 8 row shards a box of 8 GPUs
    would process (sharding.row_partition) must reproduce the unsharded tensor bit for bit —
    dequantized values, int8 codes, row divisors and STE masks alike (no data-path collective)."""
    from llm_qat_b200._lib import CODES_I8
    from llm_qat_b200.sharding import row_partition
    from llm_qat_b200.utils_quant import fake_quant_forward, ste_backward

    gen = torch.Generator().manual_seed(5)
    x = (torch.randn(*shape, generator=gen) * (0.02 if len(shape) == 2 else 1.0)).bfloat16().cuda()
    g = torch.randn(*shape, generator=gen).bfloat16().cuda()
    flat, gflat = x.reshape(-1, shape[-1]), g.reshape(-1, shape[-1])
    y, _, _, _, _ = fake_quant_forward(flat, bits, False, True)
    _, codes, _, e, mask = fake_quant_forward(flat, bits, False, True, want_y=False, codes_kind=CODES_I8,
                                              want_scales=True, mask_clip=(-2.0, 2.0))
    gx = ste_backward(gflat, flat, CLIP)
    world, rows = 8, flat.shape[0]
    ys, cs, es, ms, gs = [], [], [], [], []
    for rank in range(world):
        r0, n = row_partition(rows, world, rank)
        part = flat[r0:r0 + n]
        ys.append(fake_quant_forward(part, bits, False, True)[0])
        _, c, _, ee, m = fake_quant_forward(part, bits, False, True, want_y=False, codes_kind=CODES_I8,
                                            want_scales=True, mask_clip=(-2.0, 2.0))
        cs.append(c); es.append(ee); ms.append(m)
        gs.append(ste_backward(gflat[r0:r0 + n], part, CLIP))
    assert torch.equal(torch.cat(ys).view(torch.int16), y.view(torch.int16)), what
    assert torch.equal(torch.cat(cs), codes) and torch.equal(torch.cat(es), e), what
    assert torch.equal(torch.cat(ms), mask), what          # shard sizes are multiples of 8 elements
    assert torch.equal(torch.cat(gs).view(torch.int16), gx.view(torch.int16)), what
    # and the unsharded result is the oracle's
    assert qo.count_mismatch(U.tensor_to_f32(y[:64]), qo.sym_forward(U.tensor_to_f32(flat[:64]), bits, False, "bf16")["y"]) == 0


def test_empty_inputs_behave_like_the_reference():
    """Zero rows of a non-empty width: an empty result (and gradient); an empty reduction set
    (zero columns, or layerwise over nothing) raises what torch.max raises in the reference;
    QuantizeLinear on zero tokens returns [0, out]."""
    from llm_qat_b200 import AsymQuantizer, QuantizeLinear, SymQuantizer

    for Q in (SymQuantizer, AsymQuantizer):
        x = torch.zeros(0, 8, device="cuda", requires_grad=True)
        y = Q.apply(x, CLIP, 4, False)
        assert y.shape == (0, 8) and y.dtype == x.dtype
        y.sum().backward()
        assert x.grad.shape == (0, 8)
        assert Q.apply(torch.zeros(2, 0, 8, device="cuda"), CLIP, 4, False).shape == (2, 0, 8)
        with pytest.raises(IndexError):
            Q.apply(torch.zeros(4, 0, device="cuda"), CLIP, 4, False)
        with pytest.raises(RuntimeError):
            Q.apply(torch.zeros(0, 8, device="cuda"), CLIP, 4, True)
    # a 0-dim tensor is one row of one element
    for val in (1.7, -0.3, 0.0):
        y = SymQuantizer.apply(torch.tensor(val, device="cuda"), CLIP, 4, False)
        assert y.shape == () and qo.count_mismatch(U.tensor_to_f32(y).reshape(1), qo.sym_forward(np.float32([val]), 4)["y"]) == 0
    lin = QuantizeLinear(16, 4, w_bits=4, a_bits=8).bfloat16().cuda()
    assert lin(torch.zeros(0, 16, device="cuda", dtype=torch.bfloat16)).shape == (0, 4)
    assert lin(torch.zeros(2, 0, 16, device="cuda", dtype=torch.bfloat16)).shape == (2, 0, 4)


# --------------------------------------------------------------- full BASELINE sizes: properties
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_config1_full_size_properties(dtype):
    """[8192, 4096] (BASELINE config 1): size-independent properties + a sampled
    bit-exact check against the oracle."""
    from llm_qat_b200 import AsymQuantizer, SymQuantizer
    from llm_qat_b200._lib import CODES_I16
    from llm_qat_b200.utils_quant import fake_quant_forward

    gen = torch.Generator().manual_seed(1234)
    x = (torch.randn(8192, 4096, generator=gen) * 0.5).to(U.DTYPES[dtype]).cuda()
    g = torch.randn(8192, 4096, generator=gen).to(U.DTYPES[dtype]).cuda()
    for bits in (4, 8):
        xr = x.clone().requires_grad_(True)
        y = SymQuantizer.apply(xr, CLIP, bits, False)
        y.backward(g)
        Q = 2 ** (bits - 1) - 1
        _, codes, s, e, _ = fake_quant_forward(x, bits, False, True, want_y=False, codes_kind=CODES_I16,
                                               want_scales=True)
        assert int(codes.abs().max()) in ((Q, Q + 1) if dtype == "bf16" else (Q,))
        # linearity on the integer grid: y == codes / e exactly (fp32) — the dequant identity
        if dtype == "fp32":
            assert torch.equal(y.detach(), codes.float() / e[:, None])
        # row independence: quantizing a row subset gives the same rows
        sub = SymQuantizer.apply(x[1000:1064], CLIP, bits, False)
        assert torch.equal(sub, y.detach()[1000:1064])
        # checksum of the STE mask: gx is g where |x| < 2, else 0
        keep = (x.float().abs() < 2.0)
        assert torch.equal(xr.grad, torch.where(keep, g, torch.zeros_like(g)))
        # sampled rows vs the oracle
        rows = torch.arange(0, 8192, 257)
        o = qo.sym_forward(U.tensor_to_f32(x[rows]), bits, False, dtype)["y"]
        assert qo.count_mismatch(U.tensor_to_f32(y.detach()[rows]), o) == 0
        ya = AsymQuantizer.apply(x, CLIP, bits, False)
        oa = qo.asym_forward(U.tensor_to_f32(x[rows]), bits, False, dtype)["y"]
        assert qo.count_mismatch(U.tensor_to_f32(ya[rows]), oa) == 0
        # idempotence of the code grid: re-quantizing y keeps every code (fp32, sym)
        if dtype == "fp32" and bits == 4:
            _, codes2, _, _, _ = fake_quant_forward(y.detach(), bits, False, True, want_y=False,
                                                    codes_kind=CODES_I16)
            assert torch.equal(codes, codes2)


# --------------------------------------------------------------- QuantizeLinear
@pytest.mark.parametrize("dtype,tol", [("fp32", 5e-6), ("bf16", 1e-2)])
@pytest.mark.parametrize("fused", ["0", "1"])
def test_quantize_linear_vs_reference_goldens(dtype, tol, fused, monkeypatch):
    from llm_qat_b200 import QuantizeLinear

    monkeypatch.setenv("QAT_B200_FUSED_LINEAR", fused)
    g = U.golden(dtype)
    x0 = U.bits_to_tensor(g["lin/x"], dtype, "cuda")
    w0 = U.bits_to_tensor(g["lin/w"], dtype, "cuda")
    gr = U.bits_to_tensor(g["lin/g"], dtype, "cuda")
    tags = [k.split("/")[-1] for k in g.files if k.startswith("lin/out/")]
    for tag in tags:
        body = tag.replace("_wlw", "")
        w_bits = int(body[1:body.index("a")])
        rest = body[body.index("a") + 1:]
        a_bits, sym = int(rest[:-1]), rest[-1] == "s"
        lin = QuantizeLinear(192, 80, symmetric=sym, w_bits=w_bits, a_bits=a_bits,
                             weight_layerwise=tag.endswith("_wlw")).to(U.DTYPES[dtype]).cuda()
        with torch.no_grad():
            lin.weight.copy_(w0)
        x = x0.clone().requires_grad_(True)
        out = lin(x)
        out.backward(gr)
        for name, got in (("out", out), ("gx", x.grad), ("gw", lin.weight.grad)):
            ref = U.bits_to_f32(g[f"lin/{name}/{tag}"], dtype).astype(np.float64)
            got = U.tensor_to_f32(got).astype(np.float64)
            rel = np.linalg.norm(got - ref) / (np.linalg.norm(ref) + 1e-30)
            assert rel <= tol, (dtype, tag, name, rel, fused)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_lowbit_weight_vs_reference_goldens(dtype):
    from llm_qat_b200.utils_quant import _LowBitWeight

    g = U.golden(dtype)
    w = U.bits_to_tensor(g["lowbit/w"], dtype, "cuda")
    for k in [k for k in g.files if k.startswith("lowbit/weff/")]:
        tag = k.split("/")[-1]
        got = _LowBitWeight.apply(w, int(tag[1]), tag.endswith("_lw"))
        assert U.mismatches(U.tensor_bits(got), g[k], dtype) == 0, k   # fp32 too: mean|w| in torch's own order


def test_lowbit_weight_edge_rows_and_shapes_vs_oracle():
    """W1 / W2 weight path (qat_testutil.lowbit_edge_cases: edge rows, LLaMA-like and ragged shapes,
    row-wise and layerwise) through the one-pass row kernel, its packed-bf16 chain, the
    exact-division fallback (scale 0 / inf / NaN rows) and the two-pass path (odd width, layerwise)."""
    from llm_qat_b200.utils_quant import _LowBitWeight

    for dtype, w, bits, lw in U.lowbit_edge_cases():
        got = U.tensor_to_f32(_LowBitWeight.apply(w.cuda(), bits, lw))
        ref = qo.lowbit_weight(U.tensor_to_f32(w), bits, lw, dtype)["w_eff"]
        assert U.lowbit_close(got, ref, dtype, U.lowbit_exact(lw, w.numel())), (dtype, tuple(w.shape), bits, lw)


# --------------------------------------------------------------- K4: tcgen05 GEMM
@pytest.mark.parametrize("T,N,K", [(128, 256, 128), (256, 512, 4096), (200, 264, 1040), (8, 80, 192),
                                   (1024, 11008, 4096), (300, 520, 2064), (2048, 4096, 11008)])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("cta_group", [1, 2])
def test_qlinear_i8_gemm_exact_integer_dot(T, N, K, out_dtype, cta_group):
    """int8 x int8 -> s32 is exact, so the only rounding is the epilogue's:
    compare with an int64 reference scaled in float64.  Both tile plans (single
    CTAs on 128x256 tiles, CTA pairs on 256x256 tiles) on every shape, ragged
    ones included (rows/columns/K beyond the edge are TMA zero fill)."""
    from llm_qat_b200 import _lib
    from llm_qat_b200.utils_quant import qlinear_i8

    _lib.check(_lib.lib().qat_set_gemm_cta_group(cta_group))
    try:
        _qlinear_exact_case(qlinear_i8, T, N, K, out_dtype)
    finally:
        _lib.lib().qat_set_gemm_cta_group(0)


def _qlinear_exact_case(qlinear_i8, T, N, K, out_dtype):

    gen = torch.Generator().manual_seed(T + N + K)
    qx = torch.randint(-127, 128, (T, K), generator=gen, dtype=torch.int8)
    qw = torch.randint(-7, 8, (N, K), generator=gen, dtype=torch.int8)
    ex = (torch.rand(T, generator=gen) * 50 + 1).float()
    ew = (torch.rand(N, generator=gen) * 300 + 10).float()
    out = qlinear_i8(qx.cuda(), qw.cuda(), ex.cuda(), ew.cuda(), out_dtype)
    acc = qx.double() @ qw.double().t()            # exact: |acc| < 2^53
    ref = acc / (ex.double()[:, None] * ew.double()[None, :])
    got = out.double().cpu()
    tol = 2 ** -8 if out_dtype == torch.bfloat16 else 3e-7
    err = ((got - ref).abs() / (ref.abs() + 1e-12)).max().item()
    assert err <= tol, (T, N, K, out_dtype, err)


def test_quantize_linear_caches_are_transparent(monkeypatch):
    """QAT_B200_CACHE: 1 = weight codes reused only by the checkpoint recompute of the same step,
    activation codes shared by consecutive layers fed the same tensor object (q/k/v); 2 = weight
    codes also reused across plain forwards until the parameter's (data_ptr, _version) changes.
    No mode may change a result (0 = no reuse is the baseline)."""
    from torch.utils.checkpoint import checkpoint

    from llm_qat_b200 import QuantizeLinear, _lib

    gen = torch.Generator().manual_seed(77)
    x = torch.randn(4, 50, 256, generator=gen).bfloat16().cuda()
    go = torch.randn(4, 50, 384, generator=gen).bfloat16().cuda()
    ws = [(torch.randn(384, 256, generator=gen) * 0.05).bfloat16().cuda() for _ in range(3)]

    def run(cache):
        monkeypatch.setenv("QAT_B200_CACHE", cache)
        monkeypatch.setenv("QAT_B200_FUSED_LINEAR", "1")
        lins = [QuantizeLinear(256, 384, w_bits=4, a_bits=8).bfloat16().cuda() for _ in range(3)]
        res, launches = [], []
        for lin, w in zip(lins, ws):
            with torch.no_grad():
                lin.weight.copy_(w)
        xi = x.clone().requires_grad_(True)
        n0 = _lib.launch_count()
        outs = [lin(xi) for lin in lins]              # same input three times (q/k/v pattern)
        launches.append(_lib.launch_count() - n0)     # 3 GEMMs + 3 weight quantizations + 1 or 3 activation ones
        sum(o.float().mul(go.float()).sum() for o in outs).backward()
        res += [o.detach().clone() for o in outs] + [xi.grad.clone()] + [lin.weight.grad.clone() for lin in lins]
        # optimizer-style in-place update: stale codes must never be used
        with torch.no_grad():
            lins[0].weight.mul_(-1.5)
        res.append(lins[0](xi).detach().clone())
        n0 = _lib.launch_count()
        res.append(lins[0](xi).detach().clone())       # plain second forward: reuses the weight codes in mode 2 only
        launches.append(_lib.launch_count() - n0)
        # in-place change of the activation: the activation slot must miss
        with torch.no_grad():
            xi.mul_(0.5)
        res.append(lins[1](xi).detach().clone())
        # gradient checkpointing, both flavours: the recompute inside backward reuses the weight codes (modes 1, 2)
        for reentrant in (False, True):
            xc = x.clone().requires_grad_(True)
            lins[2].weight.grad = None
            y = checkpoint(lins[2], xc, use_reentrant=reentrant)
            n0 = _lib.launch_count()
            y.backward(go)
            launches.append(_lib.launch_count() - n0)
            res += [y.detach().clone(), xc.grad.clone(), lins[2].weight.grad.clone()]
        return res, launches

    (a, la), (b, lb), (c, lc) = run("1"), run("0"), run("2")
    assert len(a) == len(b) == len(c)
    for i, (u, v, w) in enumerate(zip(a, b, c)):
        assert torch.equal(u, v) and torch.equal(u, w), i
    assert torch.equal(a[7], a[8]) and not torch.equal(a[0], a[7])
    # what was actually skipped: [q/k/v forward, plain second forward, backward incl. recompute x2]
    assert lb[0] == 9 and la[0] == 7 and lc[0] == 7          # activation codes shared in modes 1 and 2
    assert lb[1] == 3 and la[1] == 2 and lc[1] == 1          # plain re-forward: activation slot hits (1, 2); only mode 2 trusts the weight's version key
    # recompute skips the weight quantization; the non-reentrant flavour re-enters with the very same
    # input tensor object, so the activation slot hits too
    assert la[2] == lb[2] - 2 and la[3] == lb[3] - 1
    assert lc[2] == la[2] and lc[3] == la[3]


@pytest.mark.parametrize("bits", [4, 8])
def test_sym_quantizer_under_autocast_is_the_fp32_scale_chain(bits):
    """Inside torch.autocast the reference's SymQuantizer on a bf16 tensor computes its scale in
    fp32 and returns float32 (autocast runs `reciprocal` in fp32).  Product == the restated chain
    under the same context == the numpy oracle's "bf16_amp" mode, bit for bit: forward values,
    codes / divisors / mask of the GEMM feed, and the gradient (which autograd casts to bf16)."""
    from llm_qat_b200 import SymQuantizer
    from llm_qat_b200._lib import CODES_I8
    from llm_qat_b200.utils_quant import fake_quant_forward
    from oracle import ref_module as R

    gen = torch.Generator().manual_seed(40 + bits)
    for shape in ((64, 4096), (3, 17, 1000), (5, 11008), (7, 172), (2, 3, 4, 24)):
        x = (torch.randn(*shape, generator=gen) * 0.8).bfloat16()
        x.view(-1)[:4] = torch.tensor([2.0, -2.0, 0.0, -0.0]).bfloat16()
        g = torch.randn(*shape, generator=gen)
        outs = []
        for Q in (R.SymQuantizer, SymQuantizer):
            xi = x.cuda().requires_grad_(True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = Q.apply(xi, CLIP, bits, False)
            assert y.dtype == torch.float32
            y.backward(g.cuda())
            assert xi.grad.dtype == torch.bfloat16
            outs.append((y.detach().cpu(), xi.grad.cpu()))
        assert torch.equal(outs[0][0].view(torch.int32), outs[1][0].view(torch.int32)), shape
        assert torch.equal(outs[0][1].view(torch.int16), outs[1][1].view(torch.int16)), shape
        o = qo.sym_forward(U.tensor_to_f32(x), bits, False, "bf16_amp")
        assert qo.count_mismatch(outs[1][0].numpy(), o["y"]) == 0, shape
        if len(shape) == 2 and shape[1] % 16 == 0:
            _, codes, _, e, _ = fake_quant_forward(x.cuda(), bits, False, True, want_y=False, codes_kind=CODES_I8,
                                                   want_scales=True, mask_clip=(-2.0, 2.0), amp=True)
            assert np.array_equal(codes.cpu().numpy().astype(np.float32), o["codes"])
            assert qo.count_mismatch(e.cpu().numpy(), o["e"]) == 0


def test_fused_linear_propagates_nonfinite_rows_like_the_reference():
    """An overflowed activation (or weight) row must not vanish: the reference's fake-quantized row
    holds NaN (inf * 0, or NaN itself) and so does its output row (column); the integer codes of
    NaN are 0, so the fused path carries the information in the row divisor instead."""
    from llm_qat_b200 import QuantizeLinear
    from oracle import ref_module as R

    gen = torch.Generator().manual_seed(8)
    x = torch.randn(64, 256, generator=gen).bfloat16()
    w = (torch.randn(128, 256, generator=gen) * 0.05).bfloat16()
    x[3, 17] = float("inf")
    x[9, 200] = float("nan")
    x[20, 5] = -float("inf")
    w[40, 3] = float("inf")
    w[77, 100] = float("nan")
    outs = []
    for mod in (R, None):
        lin = (mod.QuantizeLinear if mod else QuantizeLinear)(256, 128, w_bits=4, a_bits=8).bfloat16().cuda()
        with torch.no_grad():
            lin.weight.copy_(w.cuda())
            outs.append(lin(x.cuda()).float().cpu())
    ref, got = outs
    assert torch.equal(torch.isnan(ref), torch.isnan(got))
    assert torch.isnan(got[3]).all() and torch.isnan(got[:, 40]).all() and not torch.isnan(got[0, 0])
    ok = ~torch.isnan(ref)
    assert ((ref[ok] - got[ok]).norm() / ref[ok].norm()).item() <= 1e-2


@pytest.mark.parametrize("fused", ["0", "1"])
def test_quantize_linear_under_autocast_matches_reference_semantics(fused, monkeypatch):
    """HF's Trainer wraps the step in torch.autocast(bf16) (kd_trainer.py:106).  With fp32 modules the
    reference fake-quantizes in fp32 and its F.linear then runs — and returns — bf16; with bf16 modules
    its SymQuantizer switches to the fp32 scale chain and returns float32, which F.linear casts back.
    The product must give the same dtypes and values in both cases: bit-identical on the unfused path
    (same op chain, same library GEMM), within the GEMM tolerance on the integer-grid path."""
    from llm_qat_b200 import QuantizeLinear
    from oracle import ref_module as R

    monkeypatch.setenv("QAT_B200_FUSED_LINEAR", fused)
    gen = torch.Generator().manual_seed(3)
    x32 = torch.randn(6, 40, 256, generator=gen).cuda()
    w32 = (torch.randn(128, 256, generator=gen) * 0.05).cuda()
    go = torch.randn(6, 40, 128, generator=gen).cuda()
    for dtype in (torch.float32, torch.bfloat16):
        res = []
        for mod in (R, None):
            lin = (mod.QuantizeLinear if mod else QuantizeLinear)(256, 128, w_bits=4, a_bits=8).to(dtype).cuda()
            with torch.no_grad():
                lin.weight.copy_(w32.to(dtype))
            xi = x32.detach().clone().to(dtype).requires_grad_(True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = lin(xi)
            out.backward(go.to(out.dtype))
            res.append((out, xi.grad, lin.weight.grad))
        (o_ref, dx_ref, dw_ref), (o, dx, dw) = res
        assert o.dtype == o_ref.dtype == torch.bfloat16 and dx.dtype == dtype and dw.dtype == dtype
        for a, c in ((o_ref, o), (dx_ref, dx), (dw_ref, dw)):
            rel = ((a.double() - c.double()).norm() / a.double().norm()).item()
            assert rel <= 1e-2, (dtype, rel)
        if fused == "0" or dtype == torch.float32:   # the very same op chain as the reference
            assert torch.equal(o_ref, o) and torch.equal(dx_ref, dx) and torch.equal(dw_ref, dw), dtype


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_dequant_codes_reproduces_forward_output(dtype):
    from llm_qat_b200._lib import CODES_I8
    from llm_qat_b200.utils_quant import dequant_codes, fake_quant_forward

    gen = torch.Generator().manual_seed(21)
    x = (torch.randn(300, 1024, generator=gen) * 0.6).to(U.DTYPES[dtype]).cuda()
    for bits in (4, 8):
        y, c8, _, e, _ = fake_quant_forward(x, bits, False, True, codes_kind=CODES_I8, want_scales=True)
        back = dequant_codes(c8, e, x.dtype)
        # identical except -0 (codes carry no sign of zero) and the saturated +128 codes of bf16 A8
        sat = (y.float() * e[:, None]) > 127.5
        same = (back == y) | sat
        assert bool(same.all()), int((~same).sum())
        assert int(sat.sum()) <= (0 if dtype == "fp32" else 300)


def test_config2_quantize_linear_full_shape():
    """BASELINE config 2: x bf16 [8192, 4096], W bf16 [11008, 4096], W4A8; fused
    path vs the unfused (fake-quant kernels + library GEMM) path, rel <= 1e-2."""
    from llm_qat_b200 import QuantizeLinear
    import os

    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(8192, 4096, generator=gen)
    idx = torch.randint(0, x.numel(), (x.numel() // 1000,), generator=gen)
    x.view(-1)[idx] *= 20.0
    x = x.bfloat16().cuda()
    lin = QuantizeLinear(4096, 11008, w_bits=4, a_bits=8).bfloat16().cuda()
    with torch.no_grad():
        lin.weight.copy_((torch.randn(11008, 4096, generator=gen) * 0.02).bfloat16())
    outs = {}
    for fused in ("0", "1"):
        os.environ["QAT_B200_FUSED_LINEAR"] = fused
        with torch.no_grad():
            outs[fused] = lin(x).float()
    os.environ.pop("QAT_B200_FUSED_LINEAR")
    rel = (outs["1"] - outs["0"]).norm() / outs["0"].norm()
    assert rel.item() <= 1e-2, rel.item()
    rows = (outs["1"] - outs["0"]).norm(dim=1) / outs["0"].norm(dim=1)
    assert rows.max().item() <= 1e-2, rows.max().item()


# --------------------------------------------------------------- host-buffer entry points
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("sym", [True, False])
def test_host_entry_points_match_device_path(dtype, sym):
    from llm_qat_b200.host_api import fake_quant_fwd_bwd_host

    gen = torch.Generator().manual_seed(9)
    x = (torch.randn(3000, 4096, generator=gen) * 0.8).to(U.DTYPES[dtype]).pin_memory()
    g = torch.randn(3000, 4096, generator=gen).to(U.DTYPES[dtype]).pin_memory()
    y, gx = fake_quant_fwd_bwd_host(x, g, (-2.0, 2.0), 8, symmetric=sym)
    torch.cuda.synchronize()
    rows = torch.arange(0, 3000, 37)
    fn = qo.sym_forward if sym else qo.asym_forward
    assert qo.count_mismatch(U.tensor_to_f32(y[rows]), fn(U.tensor_to_f32(x[rows]), 8, False, dtype)["y"]) == 0
    ob = qo.ste_backward(U.tensor_to_f32(g), U.tensor_to_f32(x), -2.0, 2.0, dtype)
    assert qo.count_mismatch(U.tensor_to_f32(gx), ob["gx"]) == 0


# --------------------------------------------------------------- round 2: own backward GEMMs, parity knobs
def _pack_bits(bits: torch.Tensor) -> torch.Tensor:
    return torch.from_numpy(np.packbits(bits.cpu().numpy().reshape(-1), bitorder="little"))


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("shape", [(128, 256, 64), (304, 520, 200), (1000, 776, 1032)])
def test_gemm_bf16_every_operand_layout(a_mn, b_mn, cg, shape):
    """qat_gemm_bf16 (tcgen05 kind::f16, K-major / MN-major operands through TMA) vs fp32 matmul."""
    from llm_qat_b200 import _lib

    M, N, K = shape
    gen = torch.Generator().manual_seed(5)
    A = torch.randn(M, K, generator=gen).bfloat16().cuda()
    B = torch.randn(N, K, generator=gen).bfloat16().cuda()
    a = A.t().contiguous() if a_mn else A
    b = B.t().contiguous() if b_mn else B
    bits = torch.rand(M * N, generator=gen) < 0.7
    mask = _pack_bits(bits).cuda()
    for use_mask, od in ((False, torch.bfloat16), (True, torch.bfloat16), (True, torch.float32)):
        out = torch.empty(M, N, dtype=od, device="cuda")
        rc = _lib.lib().qat_gemm_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), mask.data_ptr() if use_mask else 0,
                                      M, N, K, a_mn, b_mn, 1 if od == torch.bfloat16 else 0, cg,
                                      torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "qat_gemm_bf16")
        ref = A.float() @ B.float().t()
        if use_mask:
            ref = ref * bits.view(M, N).cuda()
            assert bool((out[~bits.view(M, N).cuda()] == 0).all())     # masked elements are exactly 0
        rel = ((out.float() - ref).norm() / ref.norm()).item()
        assert rel <= (4e-3 if od == torch.bfloat16 else 1e-5), (a_mn, b_mn, cg, shape, use_mask, rel)


def test_quantize_linear_backward_runs_on_own_kernels(monkeypatch):
    """(f)-1: dgrad / wgrad of the fused QuantizeLinear are this library's tcgen05 kernel with the STE
    mask in the epilogue — no library GEMM, no separate mask pass — and equal the reference chain's
    gradients to bf16 rounding."""
    from llm_qat_b200 import QuantizeLinear, _lib
    from oracle import ref_module

    monkeypatch.setenv("QAT_B200_FUSED_LINEAR", "1")
    gen = torch.Generator().manual_seed(9)
    T, K, N = 512, 1024, 1536
    x0 = (torch.randn(T, K, generator=gen) * 1.2).bfloat16().cuda()
    w0 = (torch.randn(N, K, generator=gen) * 0.02).bfloat16().cuda()
    g0 = torch.randn(T, N, generator=gen).bfloat16().cuda()
    res = []
    for cls in (ref_module.QuantizeLinear, QuantizeLinear):
        lin = cls(K, N, w_bits=4, a_bits=8).bfloat16().cuda()
        with torch.no_grad():
            lin.weight.copy_(w0)
        x = x0.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = lin(x)
        n0 = _lib.launch_count()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            out.backward(g0)
            torch.cuda.synchronize()
        res.append((x.grad, lin.weight.grad, _lib.launch_count() - n0, [e.key for e in prof.key_averages()]))
    (gx_r, gw_r, _, _), (gx, gw, launches, kernels) = res
    assert launches == 4, launches                         # 2 operand rebuilds + 2 contractions
    assert not any("nvjet" in k or "gemm" in k.lower() and "qat" not in k for k in kernels
                   if "gemm_bf16_kernel" not in k), kernels
    for a, c in ((gx_r, gx), (gw_r, gw)):
        rel = ((a.double() - c.double()).norm() / a.double().norm()).item()
        assert rel <= 1e-2, rel
        assert bool(((a == 0) == (c == 0)).float().mean() > 0.999)    # same STE mask


def test_asym_div_mode_cuda_matches_reference_eager_on_gpu():
    """QAT_ASYM_DIV_RECIP reproduces, bit for bit, what the reference's op chain computes when it runs
    eagerly on CUDA (fp32: `.div(255)` is a multiply by fl(1/255) there); QAT_ASYM_DIV_TRUE (default)
    reproduces its CPU result."""
    from llm_qat_b200 import AsymQuantizer, _lib
    from oracle import torch_chain as tc

    gen = torch.Generator().manual_seed(17)
    x = (torch.randn(257, 1000, generator=gen) * 0.7)
    try:
        for bits in (4, 8):
            cpu_ref = tc.asym_forward(x, bits, False)
            cuda_ref = tc.asym_forward(x.cuda(), bits, False)
            _lib.check(_lib.lib().qat_set_asym_div(0))
            y_true = AsymQuantizer.apply(x.cuda(), CLIP, bits, False)
            _lib.check(_lib.lib().qat_set_asym_div(1))
            y_recip = AsymQuantizer.apply(x.cuda(), CLIP, bits, False)
            assert torch.equal(y_true.cpu(), cpu_ref)
            assert torch.equal(y_recip, cuda_ref)
            assert qo.count_mismatch(y_recip.cpu().numpy(), qo.asym_forward(x.numpy(), bits, False, "fp32", div="cuda")["y"]) == 0
            # bf16: both modes agree with each other and with the reference on either device
            xb = x.bfloat16()
            _lib.check(_lib.lib().qat_set_asym_div(0))
            yb0 = AsymQuantizer.apply(xb.cuda(), CLIP, bits, False)
            _lib.check(_lib.lib().qat_set_asym_div(1))
            yb1 = AsymQuantizer.apply(xb.cuda(), CLIP, bits, False)
            assert torch.equal(yb0, yb1) and torch.equal(yb0, tc.asym_forward(xb.cuda(), bits, False))
    finally:
        _lib.lib().qat_set_asym_div(0)


def test_int8_feed_keeps_minus_128_and_saturates_only_plus_128():
    """Plain-bf16 A8 rows whose extreme elements round to the codes +-128: -128 is carried exactly, +128
    becomes 127 (documented in qat_b200.h); the fused linear stays within 1e-2 of the reference chain and
    the deviation is bounded by the saturated terms."""
    from llm_qat_b200 import QuantizeLinear
    from llm_qat_b200._lib import CODES_I8, CODES_I16
    from llm_qat_b200.utils_quant import fake_quant_forward
    from oracle import ref_module

    gen = torch.Generator().manual_seed(23)
    x = torch.randn(2048, 1024, generator=gen).bfloat16().cuda()
    x[:, 7] = -x.abs().max(dim=1).values            # a unique negative extreme per row ...
    x[1::2, 7] = x[1::2, 7].neg()                   # ... or a positive one on odd rows
    _, c16, _, _, _ = fake_quant_forward(x, 8, False, True, want_y=False, codes_kind=CODES_I16)
    _, c8, _, _, _ = fake_quant_forward(x, 8, False, True, want_y=False, codes_kind=CODES_I8)
    c16, c8 = c16.cpu().int(), c8.cpu().int()
    assert int((c16 == -128).sum()) > 0 and int((c16 == 128).sum()) > 0       # the case is exercised
    assert torch.equal(c8[c16 != 128], c16[c16 != 128])                       # -128 kept exactly
    assert bool((c8[c16 == 128] == 127).all())
    assert int((c16 == 128).sum(dim=1).max()) <= 8
    w = (torch.randn(768, 1024, generator=gen) * 0.02).bfloat16().cuda()
    outs = []
    for cls in (ref_module.QuantizeLinear, QuantizeLinear):
        lin = cls(1024, 768, w_bits=4, a_bits=8).bfloat16().cuda()
        with torch.no_grad():
            lin.weight.copy_(w)
            outs.append(lin(x).float())
    rows = (outs[1] - outs[0]).norm(dim=1) / outs[0].norm(dim=1)
    assert rows.max().item() <= 1e-2, rows.max().item()


def test_config2_full_shape_vs_reference_chain():
    """BASELINE config 2 at full size against the reference's own op chain (oracle.ref_module, eager on
    the GPU): x bf16 [8192, 4096], W bf16 [11008, 4096], W4A8; plain bf16 and under autocast."""
    from llm_qat_b200 import QuantizeLinear
    from oracle import ref_module

    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(8192, 4096, generator=gen)
    idx = torch.randint(0, x.numel(), (x.numel() // 1000,), generator=gen)
    x.view(-1)[idx] *= 20.0
    x = x.bfloat16().cuda()
    w = (torch.randn(11008, 4096, generator=gen) * 0.02).bfloat16().cuda()
    for amp in (False, True):
        outs = []
        for cls in (ref_module.QuantizeLinear, QuantizeLinear):
            lin = cls(4096, 11008, w_bits=4, a_bits=8).bfloat16().cuda()
            with torch.no_grad():
                lin.weight.copy_(w)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
                    outs.append(lin(x).float())
            del lin
        rel = ((outs[1] - outs[0]).norm() / outs[0].norm()).item()
        rows = ((outs[1] - outs[0]).norm(dim=1) / outs[0].norm(dim=1)).max().item()
        assert rel <= 1e-2 and rows <= 1e-2, (amp, rel, rows)


# --------------------------------------------------------------- round 2: attention, KD loss, producers
def _eager_attention(q, k, v, causal=True):
    """modeling_llama_quant.py:352-377 on [B, S, H, D] inputs"""
    import math

    B, S, H, D = q.shape
    qh, kh, vh = (t.transpose(1, 2) for t in (q, k, v))
    w = torch.matmul(qh, kh.transpose(2, 3)) / math.sqrt(D)
    if causal:
        m = torch.full((S, S), torch.finfo(w.dtype).min, device=w.device, dtype=w.dtype).triu(1)
        w = torch.max(w + m[None, None], torch.tensor(torch.finfo(w.dtype).min, device=w.device))
    w = torch.softmax(w, dim=-1, dtype=torch.float32).to(qh.dtype)
    return torch.matmul(w, vh).transpose(1, 2)


@pytest.mark.parametrize("B,S,H,causal", [(1, 128, 1, True), (2, 320, 3, True), (1, 200, 2, True), (1, 72, 1, True),
                                          (1, 512, 2, False), (1, 2048, 2, True)])
def test_fused_attention_forward_backward_vs_reference_chain(B, S, H, causal):
    """tcgen05 attention (fwd + bwd) vs the reference's eager chain in bf16 and an fp32 statement of it:
    the fused kernel must be within 1e-2 of the fp32 result and at least as close to it as eager bf16."""
    from llm_qat_b200.fused_ops import causal_attention

    gen = torch.Generator().manual_seed(S + H)
    mk = lambda: torch.randn(B, S, H, 128, generator=gen).bfloat16().cuda().requires_grad_(True)  # noqa: E731
    q, k, v = mk(), mk(), mk()
    go = torch.randn(B, S, H, 128, generator=gen).bfloat16().cuda()
    o = causal_attention(q, k, v, causal=causal)
    o.backward(go)
    qf, kf, vf = (t.detach().float().requires_grad_(True) for t in (q, k, v))
    of = _eager_attention(qf, kf, vf, causal)
    of.backward(go.float())
    q2, k2, v2 = (t.detach().clone().requires_grad_(True) for t in (q, k, v))
    oe = _eager_attention(q2, k2, v2, causal)
    oe.backward(go)
    rel = lambda a, b: ((a.double() - b.double()).norm() / b.double().norm()).item()  # noqa: E731
    for name, mine, eager, exact in (("o", o, oe, of), ("dq", q.grad, q2.grad, qf.grad), ("dk", k.grad, k2.grad, kf.grad),
                                     ("dv", v.grad, v2.grad, vf.grad)):
        assert torch.isfinite(mine).all(), name
        assert rel(mine, exact) <= 1e-2, (name, rel(mine, exact))
        assert rel(mine, exact) <= 1.2 * rel(eager, exact) + 1e-4, (name, rel(mine, exact), rel(eager, exact))
        assert rel(mine, eager) <= 1e-2, (name, rel(mine, eager))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 64, 32000), (1, 33, 1000), (3, 5, 12)])
def test_fused_kd_loss_matches_kd_trainer_formula(dtype, shape):
    """utils/kd_trainer.py:42-48 — KL(batchmean) of log_softmax(student) vs softmax(teacher): loss to 1e-5
    relative, gradient to 1e-4 of its norm (fp32 arithmetic in both; summation order differs)."""
    from llm_qat_b200.fused_ops import kd_loss

    gen = torch.Generator().manual_seed(7)
    s0 = (torch.randn(*shape, generator=gen) * 3).to(dtype).cuda()
    t0 = (torch.randn(*shape, generator=gen) * 3).to(dtype).cuda()
    s1 = s0.clone().requires_grad_(True)
    s2 = s0.clone().requires_grad_(True)
    ref = torch.nn.functional.kl_div(torch.log_softmax(s1.float(), dim=2), torch.softmax(t0.float(), dim=2),
                                     reduction="batchmean")
    mine = kd_loss(s2, t0)
    assert mine.dtype == torch.float32 and mine.dim() == 0
    assert abs(mine.item() - ref.item()) <= 1e-5 * abs(ref.item()) + 1e-7, (mine.item(), ref.item())
    (ref * 0.5).backward()
    (mine * 0.5).backward()
    err = (s2.grad.float() - s1.grad.float()).norm() / s1.grad.float().norm()
    assert err.item() <= (1e-4 if dtype == torch.float32 else 6e-3), err.item()


@pytest.mark.parametrize("amp", [False, True])
def test_rmsnorm_and_swiglu_producers_emit_the_consumers_codes(amp):
    """(f)-3: y / act equal the eager ops' bits (RMSNorm up to the summation order of mean(x^2)), and the
    codes, divisors and STE mask emitted alongside are exactly what qat_sym_fwd's feed gives for them."""
    from llm_qat_b200 import fused_ops as FO
    from llm_qat_b200._lib import CODES_I8
    from llm_qat_b200.utils_quant import _ACT_SLOT, _feed_views, fake_quant_forward

    gen = torch.Generator().manual_seed(31)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        for C, T in ((4096, 300), (5120, 17), (1000, 64)):
            x = (torch.randn(T, C, generator=gen) * 2).bfloat16().cuda()
            w = (1 + 0.1 * torch.randn(C, generator=gen)).bfloat16().cuda()
            y = FO.rmsnorm(x, w, 1e-6, feed_bits=8)
            var = x.to(torch.float32).pow(2).mean(-1, keepdim=True)
            y_ref = w * (x * torch.rsqrt(var + 1e-6)).to(torch.bfloat16)
            assert (y != y_ref).float().mean().item() < 2e-3          # <= 1 bf16 ulp where rstd differs by 1 ulp
            assert ((y.float() - y_ref.float()).abs() <= 0.01 * y_ref.float().abs() + 1e-6).all()
            codes, e, mask = _feed_views(_ACT_SLOT[0][2], T, C)
            _, c8, _, e_ref, m_ref = fake_quant_forward(y, 8, False, True, want_y=False, codes_kind=CODES_I8,
                                                        want_scales=True, mask_clip=(-2.0, 2.0), amp=amp)
            assert torch.equal(codes, c8) and torch.equal(e, e_ref) and torch.equal(mask, m_ref)
        for C, T in ((11008, 100), (13824, 9), (2000, 33)):
            gate = (torch.randn(T, C, generator=gen) * 2).bfloat16().cuda()
            up = torch.randn(T, C, generator=gen).bfloat16().cuda()
            act = FO.swiglu(gate, up, feed_bits=8)
            ref = torch.nn.functional.silu(gate) * up
            assert (act != ref).float().mean().item() < 2e-2          # __expf vs expf: rare 1-ulp differences
            assert ((act.float() - ref.float()).abs() <= 0.01 * ref.float().abs() + 1e-6).all()
            codes, e, mask = _feed_views(_ACT_SLOT[0][2], T, C)
            _, c8, _, e_ref, m_ref = fake_quant_forward(act, 8, False, True, want_y=False, codes_kind=CODES_I8,
                                                        want_scales=True, mask_clip=(-2.0, 2.0), amp=amp)
            assert torch.equal(codes, c8) and torch.equal(e, e_ref) and torch.equal(mask, m_ref)


def test_producer_backward_kernels_vs_autograd():
    from llm_qat_b200 import fused_ops as FO

    gen = torch.Generator().manual_seed(37)
    T, C = 200, 1024
    x0 = torch.randn(T, C, generator=gen).bfloat16().cuda()
    w0 = (1 + 0.1 * torch.randn(C, generator=gen)).bfloat16().cuda()
    g0 = torch.randn(T, C, generator=gen).bfloat16().cuda()
    x1, w1 = x0.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    FO.rmsnorm(x1, w1, 1e-6).backward(g0)
    x2, w2 = x0.float().requires_grad_(True), w0.float().requires_grad_(True)
    var = x2.pow(2).mean(-1, keepdim=True)
    (w2 * (x2 * torch.rsqrt(var + 1e-6))).backward(g0.float())
    rel = lambda a, b: ((a.float() - b).norm() / b.norm()).item()  # noqa: E731
    assert rel(x1.grad, x2.grad) <= 6e-3 and rel(w1.grad, w2.grad) <= 6e-3, (rel(x1.grad, x2.grad), rel(w1.grad, w2.grad))
    a0 = torch.randn(T, C, generator=gen).bfloat16().cuda()
    u0 = torch.randn(T, C, generator=gen).bfloat16().cuda()
    a1, u1 = a0.clone().requires_grad_(True), u0.clone().requires_grad_(True)
    FO.swiglu(a1, u1).backward(g0)
    a2, u2 = a0.float().requires_grad_(True), u0.float().requires_grad_(True)
    (torch.nn.functional.silu(a2) * u2).backward(g0.float())
    assert rel(a1.grad, a2.grad) <= 8e-3 and rel(u1.grad, u2.grad) <= 8e-3, (rel(a1.grad, a2.grad), rel(u1.grad, u2.grad))


@pytest.mark.parametrize("amp", [False, True])
@pytest.mark.parametrize("kv_bits", [4, 8, 32])
def test_qkv_prep_equals_kv_fake_quant_then_rope(amp, kv_bits):
    """One launch == SymQuantizer.apply on K and V (bit-exact values: V is compared directly) followed by
    apply_rotary_pos_emb (modeling_llama_quant.py:320-341), forward and backward, vs the eager chain."""
    from harness import llama_qat as H
    from llm_qat_b200 import SymQuantizer
    from llm_qat_b200.fused_ops import qkv_prep

    B, S, nh = 2, 96, 3
    gen = torch.Generator().manual_seed(41)
    mk = lambda: (torch.randn(B, S, nh * 128, generator=gen) * 1.5).bfloat16().cuda()  # noqa: E731
    q0, k0, v0 = mk(), mk(), mk()
    gq, gk, gv = mk(), mk(), mk()
    rot = H.RotaryEmbedding(128, 256).cuda()
    pos = torch.arange(S, device="cuda")[None].expand(B, S)
    cos_t, sin_t = rot.cos_cached[0, 0].contiguous(), rot.sin_cached[0, 0].contiguous()
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        q1, k1, v1 = (t.clone().requires_grad_(True) for t in (q0, k0, v0))
        qr, kr, vq = qkv_prep(q1, k1, v1, cos_t, sin_t, pos, nh, kv_bits)
        torch.autograd.backward((qr, kr, vq), (gq, gk, gv))
        q2, k2, v2 = (t.clone().requires_grad_(True) for t in (q0, k0, v0))
        kq, vq2 = k2, v2
        if kv_bits < 32:
            kq = SymQuantizer.apply(k2, CLIP, kv_bits, False)
            vq2 = SymQuantizer.apply(v2, CLIP, kv_bits, False)
        sh = (B, S, nh, 128)
        qh, kh, vh = q2.view(sh).transpose(1, 2), kq.view(sh).transpose(1, 2), vq2.view(sh).transpose(1, 2)
        cos, sin = rot(vh, seq_len=S)
        qe, ke = H._apply_rotary_pos_emb(qh, kh, cos, sin, pos)
        qe, ke = (t.transpose(1, 2).reshape(B, S, nh * 128) for t in (qe, ke))
        torch.autograd.backward((qe, ke, vq2), (gq.to(qe.dtype), gk.to(ke.dtype), gv.to(vq2.dtype)))
    assert torch.equal(vq, vq2.to(torch.bfloat16))
    rel = lambda a, b: ((a.float() - b.float()).norm() / b.float().norm()).item()  # noqa: E731
    assert rel(qr, qe) <= 4e-3 and rel(kr, ke) <= 4e-3, (rel(qr, qe), rel(kr, ke))
    if not amp:
        assert torch.equal(qr, qe) and torch.equal(kr, ke)     # plain bf16: every op rounded like eager
    assert torch.equal(v1.grad, v2.grad)
    assert rel(q1.grad, q2.grad) <= 6e-3 and rel(k1.grad, k2.grad) <= 6e-3, (rel(q1.grad, q2.grad), rel(k1.grad, k2.grad))
    assert bool(((k1.grad == 0) == (k2.grad == 0)).float().mean() > 0.999)


def test_qkv_prep_position_ids_outside_the_tables_stay_in_bounds():
    """`cos[position_ids]` (modeling_llama_quant.py:189-190): negative ids count from the end of the table, like
    torch indexing; ids past the table raise IndexError in the reference — here they are clamped to the last
    row, so a bad id can never read outside the tables (forward and backward)."""
    from harness import llama_qat as H
    from llm_qat_b200.fused_ops import qkv_prep

    S, nh, max_pos = 64, 2, 80
    gen = torch.Generator().manual_seed(43)
    mk = lambda: torch.randn(1, S, nh * 128, generator=gen).bfloat16().cuda()  # noqa: E731
    q0, k0, v0, gq, gk, gv = mk(), mk(), mk(), mk(), mk(), mk()
    rot = H.RotaryEmbedding(128, max_pos).cuda()
    cos_t, sin_t = rot.cos_cached[0, 0].contiguous(), rot.sin_cached[0, 0].contiguous()
    assert cos_t.shape[0] == max_pos

    def run(pos):
        q, k, v = (t.clone().requires_grad_(True) for t in (q0, k0, v0))
        out = qkv_prep(q, k, v, cos_t, sin_t, pos, nh, 4)
        torch.autograd.backward(out, (gq, gk, gv))
        return [t.detach() for t in out] + [q.grad, k.grad, v.grad]

    good = torch.arange(S, device="cuda")[None] + 10                      # 10 .. 73
    wrapped = good - max_pos                                                # the same rows, counted from the end
    for a, b in zip(run(good), run(wrapped)):
        assert torch.equal(a, b)
    wild = good.clone()
    wild[0, ::3] = 10 ** 12
    wild[0, 1::3] = -(10 ** 12)
    clamped = good.clone()
    clamped[0, ::3] = max_pos - 1
    clamped[0, 1::3] = 0
    for a, b in zip(run(wild), run(clamped)):
        assert torch.equal(a, b)
    with pytest.raises(RuntimeError):
        qkv_prep(q0, k0[:, :32], v0, cos_t, sin_t, good, nh, 4)
    with pytest.raises(RuntimeError):
        qkv_prep(q0, k0, v0, cos_t.double(), sin_t, good, nh, 4)
