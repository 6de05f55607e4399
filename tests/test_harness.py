"""The configs 3-5 harness (harness/llama_qat.py) and the oracle-side quant
module (oracle/ref_module.py).

CPU: both are pinned to the reference's stored outputs (tests/golden/) — ref_module
bit for bit against what models/utils_quant.py computed, the harness layer in bf16
against what the real LlamaDecoderLayer computed (layer_bf16.npz).  With a checkout
of the original project (QAT_B200_REFERENCE) also against its live code, which adds
the fp32 layer comparison and the model-file binding checks.
GPU: the harness on llm_qat_b200 vs the harness on the oracle module."""
import os
import sys

import numpy as np
import pytest
import torch

import qat_testutil as U
from harness import llama_qat as H
from oracle import grid_module as G
from oracle import ref_module as R

REF = U.REFERENCE
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = U.needs_reference


def _ref_modules():
    sys.dont_write_bytecode = True
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import importlib

    uq = importlib.import_module("models.utils_quant")
    assert uq.__file__.startswith(REF)
    return uq


@needs_reference
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ref_module_matches_live_reference(dtype):
    uq = _ref_modules()
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(2, 9, 96, generator=g) * 1.2).to(dtype)
    gr = torch.randn(2, 9, 96, generator=g).to(dtype)
    clip = torch.tensor([-2.0, 2.0])
    for mine, theirs in ((R.SymQuantizer, uq.SymQuantizer), (R.AsymQuantizer, uq.AsymQuantizer)):
        for bits in (4, 8):
            a = x.clone().requires_grad_(True)
            b = x.clone().requires_grad_(True)
            ya, yb = mine.apply(a, clip, bits, False), theirs.apply(b, clip, bits, False)
            ya.backward(gr)
            yb.backward(gr)
            assert torch.equal(ya, yb) and torch.equal(a.grad, b.grad)
    w = (torch.randn(40, 96, generator=g) * 0.05).to(dtype)
    go = torch.randn(2, 9, 40, generator=g).to(dtype)
    for kw in (dict(w_bits=4, a_bits=8), dict(w_bits=8, a_bits=8, symmetric=False), dict(w_bits=1, a_bits=8),
               dict(w_bits=2, a_bits=32, weight_layerwise=True), dict(w_bits=32, a_bits=4)):
        la, lb = R.QuantizeLinear(96, 40, **kw).to(dtype), uq.QuantizeLinear(96, 40, **kw).to(dtype)
        with torch.no_grad():
            la.weight.copy_(w)
            lb.weight.copy_(w)
        a = x.clone().requires_grad_(True)
        b = x.clone().requires_grad_(True)
        oa, ob = la(a), lb(b)
        oa.backward(go)
        ob.backward(go)
        assert torch.equal(oa, ob) and torch.equal(a.grad, b.grad) and torch.equal(la.weight.grad, lb.weight.grad), kw


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_ref_module_reproduces_the_reference_goldens(dtype):
    """ref_module (the eager comparator of the GPU tests and of bench.py) against what the original
    models/utils_quant.py computed on the CPU (tests/golden/quant_*.npz, oracle/gen_golden.py), bit for bit:
    both quantizers' forward on every stored case, their STE backward for every stored clip, and
    QuantizeLinear's output, input gradient and weight gradient for every stored bit-width combination,
    the W1 / W2 weight path included."""
    g = U.golden(dtype)
    tdt = U.DTYPES[dtype]
    t = lambda k: U.bits_to_tensor(g[k], dtype)  # noqa: E731
    quant = {"sym": R.SymQuantizer, "asym": R.AsymQuantizer}
    n = 0
    for q, key, bits, lw in U.quant_cases(g):
        y = quant[q].apply(t(f"in/{key}"), torch.tensor([-2.0, 2.0]), bits, lw)
        k = f"y/{q}/{key}/b{bits}/{'lw' if lw else 'row'}"
        assert U.mismatches(U.tensor_bits(y), g[k], dtype) == 0, k
        n += 1
    for q, key, lw, lo, hi, k in U.clip_cases(g):
        x = t(f"in/{key}").requires_grad_(True)      # bit widths as oracle/gen_golden.py ran the backward
        quant[q].apply(x, torch.tensor([lo, hi]), 2 if q == "sym" else 3, lw).backward(t(f"grad/{key}"))
        assert U.mismatches(U.tensor_bits(x.grad), g[k], dtype) == 0, k
        n += 1
    for tag in [k.split("/")[-1] for k in g.files if k.startswith("lin/out/")]:
        body = tag.replace("_wlw", "")
        w_bits, rest = int(body[1:body.index("a")]), body[body.index("a") + 1:]
        lin = R.QuantizeLinear(192, 80, symmetric=rest[-1] == "s", w_bits=w_bits, a_bits=int(rest[:-1]),
                               weight_layerwise=tag.endswith("_wlw")).to(tdt)
        with torch.no_grad():
            lin.weight.copy_(t("lin/w"))
        x = t("lin/x").requires_grad_(True)
        out = lin(x)
        out.backward(t("lin/g"))
        for what, v in (("out", out), ("gx", x.grad), ("gw", lin.weight.grad)):
            assert U.mismatches(U.tensor_bits(v), g[f"lin/{what}/{tag}"], dtype) == 0, (what, tag)
            n += 1
    for k in [k for k in g.files if k.startswith("lowbit/weff/")]:
        tag = k.split("/")[-1]
        lin = R.QuantizeLinear(192, 40, w_bits=int(tag[1]), a_bits=32, weight_layerwise=tag.endswith("_lw")).to(tdt)
        with torch.no_grad():
            lin.weight.copy_(t("lowbit/w"))
        w_eff = lin(torch.eye(192, dtype=tdt)).detach().t().contiguous()   # as oracle/gen_golden.py recovers it
        assert U.mismatches(U.tensor_bits(w_eff), g[k], dtype) == 0, k
        n += 1
    assert n == 178, n


@needs_reference
def test_harness_layer_matches_live_reference_layer():
    _ref_modules()
    from models.configuration_llama import LlamaConfig
    from models.modeling_llama_quant import LlamaDecoderLayer

    cfg = H.QatConfig.tiny(w_bits=4, a_bits=8, kv_bits=4)
    rcfg = LlamaConfig(hidden_size=cfg.hidden_size, intermediate_size=cfg.intermediate_size,
                       num_attention_heads=cfg.num_attention_heads, num_hidden_layers=1, vocab_size=cfg.vocab_size,
                       max_position_embeddings=cfg.max_position_embeddings, w_bits=4, a_bits=8, kv_bits=4)
    rcfg.kv_bits = 4
    torch.manual_seed(0)
    ref_layer = LlamaDecoderLayer(rcfg)
    mine = H.DecoderLayer(cfg, R)
    missing, unexpected = mine.load_state_dict(ref_layer.state_dict(), strict=False)
    assert not missing, missing
    g = torch.Generator().manual_seed(1)
    b, s = 2, 24
    x0 = torch.randn(b, s, cfg.hidden_size, generator=g)
    go = torch.randn(b, s, cfg.hidden_size, generator=g)
    mask = H.causal_mask(b, s, torch.float32, "cpu")
    pos = torch.arange(s)[None].expand(b, s)
    xa = x0.clone().requires_grad_(True)
    xb = x0.clone().requires_grad_(True)
    ya = mine(xa, mask, pos)
    yb = ref_layer(xb, attention_mask=mask, position_ids=pos)[0]
    ya.backward(go)
    yb.backward(go)
    torch.testing.assert_close(ya, yb, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(xa.grad, xb.grad, rtol=1e-4, atol=1e-5)
    for (n1, p1), (n2, p2) in zip(sorted(mine.named_parameters()), sorted(ref_layer.named_parameters())):
        assert n1 == n2
        torch.testing.assert_close(p1.grad, p2.grad, rtol=1e-4, atol=1e-5, msg=n1)


def test_kd_step_runs_on_cpu_oracle_module():
    cfg = H.QatConfig.tiny(w_bits=4, a_bits=8, kv_bits=4)
    torch.manual_seed(0)
    student = H.CausalLM(cfg, R)
    teacher = H.build_teacher(cfg)
    teacher.load_state_dict(student.state_dict())        # identical init, as train.py does
    opt = torch.optim.AdamW(student.parameters(), lr=1e-3)
    ids = torch.randint(0, cfg.vocab_size, (2, 16), generator=torch.Generator().manual_seed(5))
    losses = [float(H.qat_step(student.train(), teacher, ids, opt)) for _ in range(6)]
    # student == teacher up to quantization noise, so the KL starts near zero; the first
    # AdamW step perturbs it and the following steps must bring it back down
    assert all(np.isfinite(losses)) and losses[0] < 0.05 and losses[-1] < losses[1], losses


def test_grid_module_is_the_reference_up_to_operand_rounding():
    """oracle/grid_module.py (the K4 checker) vs oracle/ref_module.py on one linear:
    fp32 differs by accumulation order only, bf16 by the reference's rounding of each
    dequantized operand (<= 1e-2, the north-star GEMM tolerance); gradients share one code path."""
    g = torch.Generator().manual_seed(11)
    for dtype, tol in ((torch.float32, 5e-6), (torch.bfloat16, 1e-2)):
        x = torch.randn(3, 40, 256, generator=g).to(dtype)
        w = (torch.randn(96, 256, generator=g) * 0.05).to(dtype)
        go = torch.randn(3, 40, 96, generator=g).to(dtype)
        res = []
        for mod in (R, G):
            lin = mod.QuantizeLinear(256, 96, w_bits=4, a_bits=8).to(dtype)
            with torch.no_grad():
                lin.weight.copy_(w)
            xi = x.clone().requires_grad_(True)
            out = lin(xi)
            out.backward(go)
            res.append((out.double(), xi.grad.double(), lin.weight.grad.double()))
        for a, c in zip(*res):
            assert ((a - c).norm() / a.norm()).item() <= tol


def _layer_outputs(layer, x0, go, mask, pos):
    x = x0.clone().requires_grad_(True)
    y = layer(x, mask, pos)
    y.backward(go)
    return (y.float(), x.grad.float(), layer.mlp.down_proj.weight.grad.float(),
            layer.self_attn.q_proj.weight.grad.float())


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["0", "1"])
def test_harness_layer_on_b200_matches_oracle_module(fused, monkeypatch):
    """BASELINE config 3 in miniature: LLaMA decoder layer W4A8KV4 bf16 fwd+bwd, same weights
    and input, on three L1s: the reference's eager chain (oracle/ref_module.py), the integer-grid
    statement (oracle/grid_module.py) and the product."""
    import llm_qat_b200

    monkeypatch.setenv("QAT_B200_FUSED_LINEAR", fused)
    cfg = H.QatConfig(hidden_size=512, intermediate_size=1376, num_attention_heads=8, num_hidden_layers=1,
                      vocab_size=256, max_position_embeddings=256)
    torch.manual_seed(0)
    layers = {"ref": H.DecoderLayer(cfg, R).bfloat16().cuda(), "grid": H.DecoderLayer(cfg, G).bfloat16().cuda(),
              "mine": H.DecoderLayer(cfg, llm_qat_b200.utils_quant).bfloat16().cuda()}
    with torch.no_grad():
        for p in layers["ref"].parameters():
            if p.dim() == 2:
                p.normal_(0.0, 0.05)             # keeps the softmax out of its saturated (chaotic) regime
    for k in ("grid", "mine"):
        layers[k].load_state_dict(layers["ref"].state_dict())
    g = torch.Generator().manual_seed(2)
    b, s = 2, 128
    x0 = torch.randn(b, s, cfg.hidden_size, generator=g).bfloat16().cuda()
    go = torch.randn(b, s, cfg.hidden_size, generator=g).bfloat16().cuda()
    mask = H.causal_mask(b, s, torch.bfloat16, "cuda")
    pos = torch.arange(s, device="cuda")[None].expand(b, s)
    outs = {k: _layer_outputs(layer, x0, go, mask, pos) for k, layer in layers.items()}

    def rel(a, c):
        return [((x - y).norm() / x.norm()).item() for x, y in zip(outs[a], outs[c])]

    names = ("out", "dx", "dW_down", "dW_q")
    if fused == "0":
        # bit-identical quantizers + the same library GEMM on the same operands
        for name, r in zip(names, rel("ref", "mine")):
            assert r < 1e-2, (name, r)
        return
    # fused: K4 contracts the codes exactly; oracle/grid_module.py states that arithmetic, and the
    # product must agree with it to bf16 rounding through the whole layer, forward and backward.
    for name, r in zip(names, rel("grid", "mine")):
        assert r < 1e-2, (name, r, "vs the integer-grid statement")
    # Against the reference's eager chain the difference is the reference's own rounding of each
    # dequantized operand to bf16 before its GEMM (~1e-3 per linear); the 4-bit K/V and 8-bit
    # activation quantizers downstream turn that into whole-step code flips for a fraction of a
    # percent of the elements.  The floor is what the oracle-side grid statement itself shows
    # against the reference; the product must not be further away than that (x2 + 1e-2 slack).
    floor, mine = rel("ref", "grid"), rel("ref", "mine")
    for name, f, m in zip(names, floor, mine):
        assert m < 2 * f + 1e-2, (name, "product vs reference", m, "grid statement vs reference", f)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_fused_linear_is_the_grid_statement_bit_for_bit(dtype):
    """QuantizeLinear's fused path (K1 codes -> tcgen05 int8 GEMM -> dual-scale epilogue) against
    oracle/grid_module.py on the GPU, random shapes and bit widths: the forward output must be
    IDENTICAL (exact integer dot product, then the same two fp32 multiplies and one rounding);
    gradients go through the same library GEMM on operands that are bit-identical."""
    import llm_qat_b200

    rng = np.random.default_rng(7)
    gen = torch.Generator().manual_seed(7)
    for case in range(10):
        T = int(rng.choice([1, 5, 64, 200, 333, 1024]))
        K = 16 * int(rng.integers(1, 90))
        N = int(rng.choice([8, 24, 256, 264, 1000, 1376]))
        w_bits, a_bits = int(rng.integers(3, 9)), int(rng.integers(3, 9))
        x = (torch.randn(T, K, generator=gen) * float(10.0 ** rng.uniform(-1, 1))).to(dtype).cuda()
        w = (torch.randn(N, K, generator=gen) * 0.05).to(dtype).cuda()
        go = torch.randn(T, N, generator=gen).to(dtype).cuda()
        res = []
        for mod in (G, llm_qat_b200.utils_quant):
            lin = mod.QuantizeLinear(K, N, w_bits=w_bits, a_bits=a_bits).to(dtype).cuda()
            with torch.no_grad():
                lin.weight.copy_(w)
            xi = x.clone().requires_grad_(True)
            out = lin(xi)
            out.backward(go)
            res.append((out, xi.grad, lin.weight.grad))
        what = (case, T, K, N, w_bits, a_bits, dtype)
        assert torch.equal(res[0][0], res[1][0]), what
        for a, c in zip(res[0][1:], res[1][1:]):
            rel = ((a.double() - c.double()).norm() / a.double().norm().clamp_min(1e-30)).item()
            assert rel <= (1e-2 if dtype == torch.bfloat16 else 1e-5), what


@needs_reference
def test_reference_model_file_builds_on_the_product_module():
    """The drop-in claim at the import boundary: with llm_qat_b200 installed under the name
    `models.utils_quant`, the UNMODIFIED reference model file (modeling_llama_quant.py:51 imports
    QuantizeLinear and SymQuantizer from it) constructs its LLaMA with the product's classes, and
    its state dict keeps the reference's keys.  (No forward here: the product has no CPU path.)"""
    import importlib
    import subprocess

    code = r'''
import sys
sys.dont_write_bytecode = True
sys.path.insert(0, %r); sys.path.insert(0, %r)
import llm_qat_b200
import models                                   # the reference package
llm_qat_b200.install()                          # models.utils_quant -> the product
from models.configuration_llama import LlamaConfig
from models import modeling_llama_quant as M
assert M.QuantizeLinear is llm_qat_b200.QuantizeLinear and M.SymQuantizer is llm_qat_b200.SymQuantizer
cfg = LlamaConfig(hidden_size=64, intermediate_size=176, num_attention_heads=4, num_hidden_layers=2, vocab_size=128,
                  max_position_embeddings=64, w_bits=4, a_bits=8, kv_bits=4)
cfg.kv_bits = 4
model = M.LlamaForCausalLM(cfg)
lin = [m for m in model.modules() if isinstance(m, llm_qat_b200.QuantizeLinear)]
assert len(lin) == 2 * 7, len(lin)
att = model.model.layers[0].self_attn
assert att.act_quantizer_k is llm_qat_b200.SymQuantizer and att.kv_bits == 4
keys = sorted(model.state_dict().keys())
assert all(not k.endswith("_qat_wfeed") for k in keys) and "model.layers.0.mlp.up_proj.weight" in keys
print("ok", len(keys))
''' % (REF, ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("ok"), r.stdout + r.stderr[-3000:]


@pytest.mark.gpu
@pytest.mark.parametrize("autocast", [False, True])
def test_training_trajectory_matches_the_reference_chain(autocast, monkeypatch):
    """30 QAT steps (teacher forward, student forward, KL loss, backward through gradient
    checkpointing, AdamW) of a small LLaMA on three L1s with identical init and data.  Every kernel of
    the unfused product path is bit-exact and everything else is the same torch op on the same GPU,
    so its loss trajectory must be IDENTICAL to the reference chain's, step for step — with and
    without the Trainer's autocast context.  The integer-grid path must track it closely."""
    import llm_qat_b200

    cfg = H.QatConfig(hidden_size=256, intermediate_size=688, num_attention_heads=4, num_hidden_layers=2,
                      vocab_size=512, max_position_embeddings=128, w_bits=4, a_bits=8, kv_bits=4)

    def run(quant, fused):
        monkeypatch.setenv("QAT_B200_FUSED_LINEAR", fused)
        torch.manual_seed(0)
        student = H.CausalLM(cfg, quant).bfloat16().cuda()
        teacher = H.build_teacher(cfg).bfloat16().cuda()
        teacher.load_state_dict(student.state_dict())
        with torch.no_grad():                         # make the student differ from its teacher
            for p in student.parameters():
                p.add_(torch.randn(p.shape, generator=torch.Generator().manual_seed(p.numel())).to(p).mul_(0.01))
        opt = torch.optim.AdamW(student.parameters(), lr=1e-3)
        g = torch.Generator().manual_seed(99)
        losses = []
        for _ in range(30):
            ids = torch.randint(0, cfg.vocab_size, (2, 64), generator=g).cuda()
            losses.append(float(H.qat_step(student.train(), teacher, ids, opt, autocast=autocast)))
        return losses

    ref = run(R, "0")
    unfused = run(llm_qat_b200.utils_quant, "0")
    fused = run(llm_qat_b200.utils_quant, "1")
    assert all(np.isfinite(ref)) and ref[-1] < ref[0]          # it trains
    assert unfused == ref, [(i, a, b) for i, (a, b) in enumerate(zip(unfused, ref)) if a != b][:3]
    rel = max(abs(a - b) / abs(b) for a, b in zip(fused, ref))
    assert rel < 0.15 and abs(fused[-1] - ref[-1]) / ref[-1] < 0.15, (rel, fused[-3:], ref[-3:])


# --------------------------------------------------------------------------- round 2: fuse_model
@needs_reference
def test_fuse_model_binds_the_unmodified_reference_model():
    """llm_qat_b200.fuse_model on a LLaMA built from the UNMODIFIED reference model file: attention, MLP,
    RMSNorm and the model's mask builder are rebound on the instances (classes, parameters and state dict
    untouched), the causal mask the reference builds (:599-629) is recognised, a padded one is not, and
    unfuse_model restores everything.  (No product forward here: no CPU path.)"""
    import subprocess

    code = r'''
import sys
sys.dont_write_bytecode = True
sys.path.insert(0, %r); sys.path.insert(0, %r)
import torch
import llm_qat_b200
import models
llm_qat_b200.install()
from models.configuration_llama import LlamaConfig
from models import modeling_llama_quant as M
from llm_qat_b200 import model_patch as MP
cfg = LlamaConfig(hidden_size=256, intermediate_size=688, num_attention_heads=2, num_hidden_layers=2, vocab_size=128,
                  max_position_embeddings=64, w_bits=4, a_bits=8, kv_bits=4)
cfg.kv_bits = 4
model = M.LlamaForCausalLM(cfg)
keys = sorted(model.state_dict().keys())
cls_fwd = M.LlamaAttention.forward
llm_qat_b200.fuse_model(model)
llm_qat_b200.fuse_model(model)                       # idempotent
lay = model.model.layers[0]
assert lay.self_attn.forward.__func__ is MP._attention_forward and lay.self_attn.head_dim == 128
assert lay.mlp.forward.__func__ is MP._mlp_forward and lay.mlp._qat_feed_bits == 8
assert lay.input_layernorm.forward.__func__ is MP._rmsnorm_forward and lay.input_layernorm._qat_feed_bits == 8
assert model.model.norm.forward.__func__ is MP._rmsnorm_forward and model.model.norm._qat_feed_bits == 0
assert model.model.forward.__func__ is MP._model_forward
assert M.LlamaAttention.forward is cls_fwd and sorted(model.state_dict().keys()) == keys
# the mask the reference builds for "no attention_mask" is registered as causal ...
emb = torch.zeros(1, 8, 256)
model.model._qat_plain_causal = True
m = model.model._prepare_decoder_attention_mask(torch.ones(1, 8, dtype=torch.bool), (1, 8), emb, 0)
assert MP._is_causal(m) and m.shape == (1, 1, 8, 8)
assert MP._is_causal(m.detach().view(m.shape))        # same storage (what a checkpoint re-wrap passes on)
assert not MP._is_causal(m.clone())
# ... a padded one is not
model.model._qat_plain_causal = False
m2 = model.model._prepare_decoder_attention_mask(torch.tensor([[0, 1, 1, 1, 1, 1, 1, 1]]).bool(), (1, 8), emb, 0)
assert not MP._is_causal(m2) and MP._is_causal(m)     # m stays registered: it IS a causal mask and is kept alive
# several models' masks are live in one step (teacher, then student, then the student's recompute in backward)
m3 = MP.mark_causal_mask(torch.zeros(1, 1, 8, 8))
assert MP._is_causal(m) and MP._is_causal(m3) and len(MP._CAUSAL) == 2
MP.mark_causal_mask(m3); assert len(MP._CAUSAL) == 2              # re-registering is a no-op
for _ in range(MP._CAUSAL_KEEP):                                   # bounded: the oldest entries fall out
    MP.mark_causal_mask(torch.zeros(1, 1, 8, 8))
assert not MP._is_causal(m) and len(MP._CAUSAL) == MP._CAUSAL_KEEP
# a CPU call falls through to the reference's own forward code path selection (non-CUDA -> original)
assert lay.self_attn._qat_orig_forward.__func__ is cls_fwd
llm_qat_b200.unfuse_model(model)
assert "forward" not in lay.self_attn.__dict__ and "forward" not in model.model.__dict__
assert lay.self_attn.forward.__func__ is cls_fwd
print("ok")
''' % (REF, ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("ok"), r.stdout + r.stderr[-3000:]


def _layer_pair(cfg, seed=0):
    import llm_qat_b200

    torch.manual_seed(seed)
    ref = H.DecoderLayer(cfg, R).bfloat16().cuda()
    new = H.DecoderLayer(cfg, llm_qat_b200.utils_quant).bfloat16().cuda()
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() == 2:
                p.normal_(0.0, 0.02)
            else:
                p.uniform_(0.5, 1.5)
    new.load_state_dict(ref.state_dict())
    llm_qat_b200.fuse_model(new)
    return ref, new


@pytest.mark.gpu
@pytest.mark.parametrize("autocast", [False, True])
def test_fused_decoder_layer_matches_reference_chain(autocast):
    """(f)-3/(f)-4 at the layer level: a decoder layer on the product with fuse_model (RMSNorm+feed,
    qkv_prep, tcgen05 attention, SwiGLU+feed, own dgrad/wgrad) against the same layer on the reference's
    eager chain; forward and every gradient within bf16 tolerance of it, measured against what the
    integer-grid statement of the same layer (oracle.grid_module) deviates by."""
    cfg = H.QatConfig(hidden_size=512, intermediate_size=1376, num_attention_heads=4, num_hidden_layers=1,
                      max_position_embeddings=256, w_bits=4, a_bits=8, kv_bits=8)
    ref, new = _layer_pair(cfg)
    import llm_qat_b200

    g = torch.Generator().manual_seed(5)
    x0 = torch.randn(2, 256, 512, generator=g).bfloat16().cuda()
    go = torch.randn(2, 256, 512, generator=g).bfloat16().cuda()
    mask = H.causal_mask(2, 256, torch.bfloat16, "cuda")
    pos = torch.arange(256, device="cuda")[None].expand(2, 256)
    outs = []
    for layer in (ref, new):
        if layer is new:
            llm_qat_b200.mark_causal_mask(mask)
        x = x0.clone().requires_grad_(True)
        n0 = llm_qat_b200._lib.launch_count()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            y = layer(x, mask, pos)
        y.backward(go)
        grads = {n: p.grad.float() for n, p in layer.named_parameters()}
        outs.append((y.float(), x.grad.float(), grads, llm_qat_b200._lib.launch_count() - n0))
    (y_r, gx_r, gr_r, _), (y, gx, gr, launches) = outs
    rel = lambda a, b: ((a - b).norm() / b.norm().clamp_min(1e-30)).item()  # noqa: E731
    assert rel(y, y_r) <= 1e-2, rel(y, y_r)
    assert rel(gx, gx_r) <= 3e-2, rel(gx, gx_r)
    for n in gr_r:
        assert rel(gr[n], gr_r[n]) <= 3e-2, (n, rel(gr[n], gr_r[n]))
    assert launches >= 30, launches     # the layer really ran on this library's kernels


@pytest.mark.gpu
def test_fused_model_training_trajectory_tracks_the_reference_chain():
    """30 QAT steps with fuse_model + the fused KD loss against the reference chain (same init, data):
    the loss goes down and tracks the reference's trajectory."""
    import llm_qat_b200

    cfg = H.QatConfig(hidden_size=256, intermediate_size=688, num_attention_heads=2, num_hidden_layers=2,
                      vocab_size=512, max_position_embeddings=128, w_bits=4, a_bits=8, kv_bits=4)

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


# --------------------------------------------------------------------------- golden from the live model file
def _load_layer_golden():
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "layer_bf16.npz"))
    t = lambda a: torch.from_numpy(a.copy()).view(torch.bfloat16)  # noqa: E731
    b, s, hid, inter, heads, wb, ab, kvb = (int(v) for v in g["meta"])
    cfg = H.QatConfig(hidden_size=hid, intermediate_size=inter, num_attention_heads=heads, num_hidden_layers=1,
                      vocab_size=128, max_position_embeddings=128, w_bits=wb, a_bits=ab, kv_bits=kvb)
    weights = {k[2:]: t(g[k]) for k in g.files if k.startswith("w/")}
    grads = {k[2:]: t(g[k]) for k in g.files if k.startswith("g/")}
    return cfg, t(g["x"]), t(g["go"]), t(g["y"]), t(g["gx"]), weights, grads, (b, s)


def _run_layer_on(cfg, quant, weights, x0, go, device, fused):
    layer = H.DecoderLayer(cfg, quant).bfloat16()
    missing, unexpected = layer.load_state_dict(weights, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    layer = layer.to(device)
    b, s, _ = x0.shape
    mask = H.causal_mask(b, s, torch.bfloat16, device)
    if fused:
        import llm_qat_b200

        llm_qat_b200.fuse_model(layer)
        llm_qat_b200.mark_causal_mask(mask)
    pos = torch.arange(s, device=device)[None].expand(b, s)
    x = x0.to(device).clone().requires_grad_(True)
    y = layer(x, mask, pos)
    y.backward(go.to(device))
    return y.detach().float().cpu(), x.grad.float().cpu(), {n: p.grad.float().cpu() for n, p in layer.named_parameters()}


def test_harness_on_oracle_module_reproduces_the_live_layer_golden_on_cpu():
    """tests/golden/layer_bf16.npz was produced by the UNMODIFIED reference model file (oracle/gen_golden_layer.py);
    the harness layer on the oracle module must reproduce it bit for bit on the CPU (same ops, same order)."""
    cfg, x, go, y, gx, weights, grads, _ = _load_layer_golden()
    y2, gx2, gr2 = _run_layer_on(cfg, R, weights, x, go, "cpu", fused=False)
    assert torch.equal(y2, y.float()) and torch.equal(gx2, gx.float())
    for n, gref in grads.items():
        assert torch.equal(gr2[n], gref.float()), n


@pytest.mark.gpu
def test_fused_model_layer_vs_live_reference_golden():
    """The product with fuse_model (tcgen05 attention, K/V-quant + RoPE kernel, RMSNorm / SwiGLU producers, int8
    forward GEMMs, own backward GEMMs) against what the reference's own model file computed on the CPU:
    forward <= 2e-2 at the layer level, and every tensor within 1.5 x (+1e-2) of what the integer-grid statement of
    QuantizeLinear alone deviates by (bf16: 4-bit weight and 8-bit K/V codes flip on ties)."""
    import llm_qat_b200

    cfg, x, go, y, gx, weights, grads, _ = _load_layer_golden()
    n0 = llm_qat_b200._lib.launch_count()
    y2, gx2, gr2 = _run_layer_on(cfg, llm_qat_b200.utils_quant, weights, x, go, "cuda", fused=True)
    assert llm_qat_b200._lib.launch_count() - n0 >= 30
    # yardsticks against the same CPU golden: (i) the reference's OWN op chain run eagerly on this GPU — what merely
    # changing the device costs (6e-4: small); (ii) the integer-grid statement of QuantizeLinear (oracle/grid_module:
    # exact code dot product instead of a bf16 GEMM on bf16-rounded operands, everything else the reference's eager
    # layer) — the deviation the K4 design itself implies once the 4-/8-bit quantizers downstream amplify it
    # (CPU emulation: y 1.1e-2, gx 3.3e-2, up to 6.6e-2 on single weight gradients).  The fused model must stay
    # within 1.5 x of (ii): everything beyond the grid design (attention, producers, backward GEMMs) adds little.
    y3, gx3, gr3 = _run_layer_on(cfg, R, weights, x, go, "cuda", fused=False)
    y4, gx4, gr4 = _run_layer_on(cfg, G, weights, x, go, "cuda", fused=False)
    rel = lambda a, b_: ((a - b_.float()).norm() / b_.float().norm().clamp_min(1e-30)).item()  # noqa: E731
    errs = {"y": rel(y2, y), "gx": rel(gx2, gx), **{n: rel(gr2[n], gref) for n, gref in grads.items()}}
    base = {"y": rel(y3, y), "gx": rel(gx3, gx), **{n: rel(gr3[n], gref) for n, gref in grads.items()}}
    grid = {"y": rel(y4, y), "gx": rel(gx4, gx), **{n: rel(gr4[n], gref) for n, gref in grads.items()}}
    print("layer vs live-reference golden (fused model | reference chain on GPU | integer-grid statement):",
          {k: (round(v, 4), round(base[k], 4), round(grid[k], 4)) for k, v in errs.items()})
    assert errs["y"] <= 2e-2, errs
    assert max(base.values()) <= 5e-3, base
    for k, v in errs.items():
        assert v <= 1.5 * grid[k] + 1e-2, (k, v, grid[k])


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["7b", "13b"])
def test_fused_layer_is_bit_deterministic_over_back_to_back_iterations(model):
    """Race check for the tcgen05 pipelines (compute-sanitizer is closed on this pool): no kernel of the fused
    layer uses atomics, so 24 forward+backward passes issued back to back WITHOUT host synchronisation (kernels
    of consecutive iterations overlap at their edges) must give bit-identical outputs and gradients — at the
    LLaMA-7B and the LLaMA-13B shapes (the latter is where a launch-overlap stall was found and fixed)."""
    import llm_qat_b200

    cfg = (H.QatConfig.llama_13b(w_bits=4, a_bits=8, kv_bits=8) if model == "13b"
           else H.QatConfig.llama_7b(w_bits=4, a_bits=8, kv_bits=4))
    torch.manual_seed(0)
    layer = H.DecoderLayer(cfg, llm_qat_b200.utils_quant).bfloat16().cuda()
    llm_qat_b200.fuse_model(layer)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1, 2048, cfg.hidden_size, generator=g).bfloat16().cuda().requires_grad_(True)
    go = torch.randn(1, 2048, cfg.hidden_size, generator=g).bfloat16().cuda()
    mask = llm_qat_b200.mark_causal_mask(H.causal_mask(1, 2048, torch.bfloat16, "cuda"))
    pos = torch.arange(2048, device="cuda")[None]
    runs = []
    for _ in range(24):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = layer(x, mask, pos)
        y.backward(go)
        runs.append((y.detach(), x.grad.clone(), layer.mlp.up_proj.weight.grad.clone(),
                     layer.self_attn.k_proj.weight.grad.clone(), layer.input_layernorm.weight.grad.clone()))
        x.grad = None
        for p in layer.parameters():
            p.grad = None
    torch.cuda.synchronize()
    assert all(torch.isfinite(t).all() for t in runs[0])
    for i, r in enumerate(runs[1:], 1):
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b), (model, i, float((a.float() - b.float()).abs().max()))


@needs_reference
def test_fuse_model_glue_on_the_real_model_file_with_emulated_kernels():
    """The patched forwards (llm-qat_b200/model_patch.py) driven through the UNMODIFIED reference
    LlamaForCausalLM on the CPU, with the four fused ops replaced by eager restatements of the reference's own
    formulas: logits, cache tensors and gradients must equal the original forward's — i.e. the glue (mask
    recognition inside LlamaModel.forward, position ids, RoPE tables taken from LlamaRotaryEmbedding, kv_bits,
    clip values, output tuple, use_cache) is right against the real model file, not only the harness."""
    import subprocess

    code = r'''
import sys, math
sys.dont_write_bytecode = True
sys.path.insert(0, %r); sys.path.insert(0, %r)
import torch
import models
from oracle import ref_module as R
sys.modules["models.utils_quant"] = R; models.utils_quant = R      # CPU-capable quantizers under the reference's name
from models.configuration_llama import LlamaConfig
from models import modeling_llama_quant as M
import llm_qat_b200
from llm_qat_b200 import model_patch as MP

calls = {"attn": 0, "qkv": 0, "swiglu": 0, "rms": 0}
def qkv_prep(q, k, v, cos, sin, pos, heads, kv_bits, clip):
    calls["qkv"] += 1
    b, s, hid = q.shape
    c = torch.tensor(list(clip))
    if kv_bits < 32:
        k = R.SymQuantizer.apply(k, c, kv_bits, False); v = R.SymQuantizer.apply(v, c, kv_bits, False)
    sh = (b, s, heads, hid // heads)
    qh, kh = q.view(sh).transpose(1, 2), k.view(sh).transpose(1, 2)
    cs, sn = cos.to(v.dtype)[pos].unsqueeze(1), sin.to(v.dtype)[pos].unsqueeze(1)
    qe = (qh * cs) + (M.rotate_half(qh) * sn); ke = (kh * cs) + (M.rotate_half(kh) * sn)
    return qe.transpose(1, 2).reshape(b, s, hid), ke.transpose(1, 2).reshape(b, s, hid), v
def causal_attention(q, k, v, scale=None, causal=True):
    calls["attn"] += 1
    b, s, h, d = q.shape
    qh, kh, vh = (t.transpose(1, 2) for t in (q, k, v))
    w = torch.matmul(qh, kh.transpose(2, 3)) / math.sqrt(d)
    m = torch.full((s, s), torch.finfo(w.dtype).min, dtype=w.dtype).triu(1)
    w = torch.max(w + m[None, None], torch.tensor(torch.finfo(w.dtype).min))
    w = torch.nn.functional.softmax(w, dim=-1, dtype=torch.float32).to(qh.dtype)
    return torch.matmul(w, vh).transpose(1, 2)
def swiglu(gate, up, feed_bits=0):
    calls["swiglu"] += 1
    return torch.nn.functional.silu(gate) * up
def rmsnorm(x, w, eps, feed_bits=0):
    calls["rms"] += 1
    var = x.to(torch.float32).pow(2).mean(-1, keepdim=True)
    return w * (x * torch.rsqrt(var + eps)).to(w.dtype)
MP.F.qkv_prep, MP.F.causal_attention, MP.F.swiglu, MP.F.rmsnorm = qkv_prep, causal_attention, swiglu, rmsnorm
MP.F.swiglu_supported = lambda g, u: True
MP.F.rmsnorm_supported = lambda x, w: True
MP._on_gpu = lambda t: True

cfg = LlamaConfig(hidden_size=256, intermediate_size=688, num_attention_heads=2, num_hidden_layers=2, vocab_size=128,
                  max_position_embeddings=64, w_bits=4, a_bits=8, kv_bits=4)
cfg.kv_bits = 4
torch.manual_seed(0)
model = M.LlamaForCausalLM(cfg).bfloat16()
ids = torch.randint(0, 128, (2, 24), generator=torch.Generator().manual_seed(1))
def run(**kw):
    model.zero_grad()
    out = model(input_ids=ids, use_cache=True, **kw)
    out.logits.float().sum().backward()
    grads = {n: p.grad.clone() for n, p in model.named_parameters()}
    return out.logits.detach(), out.past_key_values, grads
l0, pkv0, g0 = run()
llm_qat_b200.fuse_model(model)
l1, pkv1, g1 = run()
assert calls["attn"] == 2 and calls["qkv"] == 2 and calls["swiglu"] == 2 and calls["rms"] == 5, calls
assert torch.equal(l0, l1), float((l0.float() - l1.float()).abs().max())
for (k0, v0), (k1, v1) in zip(pkv0, pkv1):
    assert k0.shape == k1.shape and torch.equal(k0, k1) and torch.equal(v0, v1)
for n in g0:
    assert torch.equal(g0[n], g1[n]), n
# an explicit all-ones mask is still recognised as causal; a padded one takes the reference's own attention
n_attn = calls["attn"]
l2, _, _ = run(attention_mask=torch.ones(2, 24, dtype=torch.long))
assert calls["attn"] == n_attn + 2 and torch.equal(l2, l0)
pad = torch.ones(2, 24, dtype=torch.long); pad[0, :5] = 0
model(input_ids=ids, attention_mask=pad)
assert calls["attn"] == n_attn + 2
llm_qat_b200.unfuse_model(model)
l3, _, _ = run()
assert torch.equal(l3, l0)
print("ok")
''' % (REF, ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-2000:] + r.stderr[-4000:]
