"""CPU: QuantizeLinear's operand route for configurations off the int8 grid (utils_quant._OperandLinearFn) —
which modules fuse_model marks, which calls take the route, and the route's glue with its three kernel calls
replaced by the torch statements of the reference (oracle/ref_module.py), bit for bit."""
import pytest
import torch
import torch.nn as nn

from oracle import ref_module, torch_chain as tc


def _uq():
    from llm_qat_b200 import utils_quant

    return utils_quant


@pytest.mark.parametrize("w_bits,a_bits,symmetric,act_lw,w_lw,k,n,eligible", [
    (4, 16, True, False, False, 64, 96, True),      # W4-A16
    (4, 32, True, False, False, 64, 96, True),      # weight-only
    (2, 32, True, False, False, 64, 96, True),      # W2 weight-only
    (1, 16, True, False, False, 64, 96, True),      # W1-A16
    (16, 16, True, False, False, 64, 96, True),
    (32, 8, True, False, False, 64, 96, True),      # activation-only
    (9, 8, True, False, False, 64, 96, True),
    (4, 2, True, False, False, 64, 96, True),       # a_bits <= 2: the activation is not quantized
    (4, 8, True, False, False, 64, 96, False),      # the int8 grid keeps its own path
    (8, 3, True, False, False, 64, 96, False),
    (32, 32, True, False, False, 64, 96, False),    # nothing quantized
    (4, 16, False, False, False, 64, 96, False),    # asymmetric activations
    (4, 32, False, False, False, 64, 96, True),     # `symmetric` only concerns the activation quantizer
    (4, 16, True, True, False, 64, 96, False),      # layerwise flags
    (4, 16, True, False, True, 64, 96, False),
    (4, 16, True, False, False, 60, 96, False),     # TMA pitch: features % 8
    (4, 16, True, False, False, 64, 92, False),
    (0, 16, True, False, False, 64, 96, False),
])
def test_eligibility_table(w_bits, a_bits, symmetric, act_lw, w_lw, k, n, eligible):
    uq = _uq()
    lin = uq.QuantizeLinear(k, n, symmetric=symmetric, w_bits=w_bits, a_bits=a_bits, act_layerwise=act_lw,
                            weight_layerwise=w_lw)
    assert uq.operand_route_config(lin) is eligible
    assert uq.operand_route_config(ref_module.QuantizeLinear(k, n, w_bits=w_bits, a_bits=a_bits)) is False


def test_fuse_model_marks_only_eligible_instances():
    import llm_qat_b200

    uq = _uq()
    model = nn.Sequential(uq.QuantizeLinear(64, 96, w_bits=4, a_bits=16), uq.QuantizeLinear(64, 96, w_bits=4, a_bits=8),
                          uq.QuantizeLinear(64, 96, w_bits=2, a_bits=32), uq.QuantizeLinear(64, 96, a_bits=16, symmetric=False),
                          nn.Linear(64, 96))
    state = {k: v.clone() for k, v in model.state_dict().items()}
    marked = lambda: [m.__dict__.get("_qat_operand_route", False) for m in model]  # noqa: E731
    assert marked() == [False] * 5
    llm_qat_b200.fuse_model(model)
    assert marked() == [True, False, True, False, False]
    llm_qat_b200.fuse_model(model)                       # idempotent
    assert marked() == [True, False, True, False, False]
    assert list(model.state_dict()) == list(state) and all(torch.equal(model.state_dict()[k], v) for k, v in state.items())
    assert "_qat_operand_route" not in dict(model[0].named_buffers()) and len(list(model[0].parameters())) == 1
    llm_qat_b200.fuse_model(model, linear=False)          # the "before" arm
    assert marked() == [False] * 5
    llm_qat_b200.fuse_model(model)
    llm_qat_b200.unfuse_model(model)
    assert marked() == [False] * 5


def test_cpu_tensors_never_take_the_route(monkeypatch):
    import llm_qat_b200

    uq = _uq()
    lin = uq.QuantizeLinear(64, 96, w_bits=4, a_bits=16).bfloat16()
    llm_qat_b200.fuse_model(lin)
    assert not lin._can_route(torch.randn(3, 64).bfloat16())
    monkeypatch.setattr(uq, "_route_device_ok", lambda t: True)
    assert lin._can_route(torch.randn(3, 64).bfloat16())
    assert not lin._can_route(torch.randn(3, 64))                     # fp32 input
    assert not lin._can_route(torch.randn(0, 64).bfloat16())          # empty
    assert not lin._can_route(torch.randn(1, 2, 3, 64).bfloat16())    # 4-D
    assert not lin._can_route(torch.randn(3, 32).bfloat16())          # shape mismatch: F.linear raises
    llm_qat_b200.unfuse_model(lin)
    assert not lin._can_route(torch.randn(3, 64).bfloat16())


def _emulate_kernels(monkeypatch, uq):
    """The route's three kernel calls as the reference's torch statements on CPU."""
    def quant_operand(t, bits, amp):
        assert not amp
        return tc.sym_forward(t, bits, False), (t > -2.0) & (t < 2.0)

    def lowbit_operand(w, bits):         # oracle/ref_module.py, w_bits < 3
        sf = w.abs().mean(dim=1, keepdim=True)
        if bits == 1:
            q = sf * torch.sign(w / sf)
        else:
            sf = 2 * sf
            q = sf * (torch.round(torch.clamp(w / sf, -(1 - 1e-2), 1 - 1e-2) * 2 ** (bits - 1) - 0.5) + 0.5) / 2 ** (bits - 1)
        return q - w + w

    def gemm_bf16(a, b, mask, M, N, K, a_mn, b_mn, cta_group=0):
        A = a.t() if a_mn else a
        B = b.t() if b_mn else b
        assert A.shape == (M, K) and B.shape == (N, K)
        out = torch.mm(A, B.t())
        return out if mask is None else out.masked_fill(~mask.view(M, N), 0)

    monkeypatch.setattr(uq, "quant_operand", quant_operand)
    monkeypatch.setattr(uq, "lowbit_operand", lowbit_operand)
    monkeypatch.setattr(uq, "gemm_bf16", gemm_bf16)
    monkeypatch.setattr(uq, "_route_device_ok", lambda t: True)


@pytest.mark.parametrize("w_bits,a_bits", [(4, 16), (2, 32), (32, 8), (16, 32)])
@pytest.mark.parametrize("shape", [(5, 64), (2, 7, 64)])
def test_route_glue_is_the_reference_forward_and_gradients_on_cpu(w_bits, a_bits, shape, monkeypatch):
    import llm_qat_b200

    uq = _uq()
    _emulate_kernels(monkeypatch, uq)
    gen = torch.Generator().manual_seed(3)
    x0 = (torch.randn(*shape, generator=gen) * 1.5).bfloat16()
    w0 = (torch.randn(96, 64, generator=gen) * 0.5).bfloat16()
    g0 = torch.randn(*shape[:-1], 96, generator=gen).bfloat16()
    res = []
    for cls in (ref_module.QuantizeLinear, uq.QuantizeLinear):
        lin = cls(64, 96, w_bits=w_bits, a_bits=a_bits).bfloat16()
        with torch.no_grad():
            lin.weight.copy_(w0)
        if cls is uq.QuantizeLinear:
            llm_qat_b200.fuse_model(lin)
            assert lin._can_route(x0)
        x = x0.clone().requires_grad_(True)
        out = lin(x)
        out.backward(g0)
        res.append((out, x.grad, lin.weight.grad))
    for a, b in zip(*res):
        assert a.dtype == b.dtype and a.shape == b.shape
        assert torch.equal(a, b)
    assert uq._ACT_SLOT.get(None) is None         # the first backward drops the shared activation operand
