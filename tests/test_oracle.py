"""CPU: the oracle restatement vs the golden vectors generated from the live
reference (oracle/gen_golden.py), plus structural properties of the arithmetic."""
import os

import numpy as np
import pytest

from oracle import quant_oracle as qo
import qat_testutil as U


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_forward_matches_reference_goldens(dtype):
    g = U.golden(dtype)
    cases = U.quant_cases(g)
    assert len(cases) >= 80
    for q, key, bits, lw in cases:
        x = U.bits_to_f32(g[f"in/{key}"], dtype)
        fn = qo.sym_forward if q == "sym" else qo.asym_forward
        y = fn(x, bits, lw, dtype)["y"]
        ref = U.bits_to_f32(g[f"y/{q}/{key}/b{bits}/{'lw' if lw else 'row'}"], dtype)
        assert qo.count_mismatch(y, ref) == 0, (dtype, q, key, bits, lw)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_backward_matches_reference_goldens(dtype):
    g = U.golden(dtype)
    cases = U.clip_cases(g)
    assert len(cases) >= 40
    for q, key, lw, lo, hi, gk in cases:
        x = U.bits_to_f32(g[f"in/{key}"], dtype)
        gr = U.bits_to_f32(g[f"grad/{key}"], dtype)
        out = qo.ste_backward(gr, x, lo, hi, dtype)
        assert qo.count_mismatch(out["gx"], U.bits_to_f32(g[gk], dtype)) == 0, (dtype, gk)


@pytest.mark.parametrize("dtype,tol", [("fp32", 2e-6), ("bf16", 4e-3)])
def test_qlinear_matches_reference_goldens(dtype, tol):
    g = U.golden(dtype)
    x = U.bits_to_f32(g["lin/x"], dtype)
    w = U.bits_to_f32(g["lin/w"], dtype)
    tags = [k.split("/")[-1] for k in g.files if k.startswith("lin/out/")]
    assert len(tags) >= 8
    for tag in tags:
        body = tag.replace("_wlw", "")
        w_bits = int(body[1:body.index("a")])
        rest = body[body.index("a") + 1:]
        a_bits, sym = int(rest[:-1]), rest[-1] == "s"
        o = qo.qlinear_forward(x, w, w_bits, a_bits, False, tag.endswith("_wlw"), sym, dtype)["out"]
        ref = U.bits_to_f32(g[f"lin/out/{tag}"], dtype)
        rel = np.linalg.norm((o - ref).astype(np.float64)) / (np.linalg.norm(ref.astype(np.float64)) + 1e-30)
        assert rel <= tol, (dtype, tag, rel)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_lowbit_weight_matches_reference_goldens(dtype):
    g = U.golden(dtype)
    keys = [k for k in g.files if k.startswith("lowbit/weff/")]
    assert len(keys) == 4
    w = U.bits_to_f32(g["lowbit/w"], dtype)
    for k in keys:
        _, _, tag = k.split("/")
        w_bits, lw = int(tag[1]), tag.endswith("_lw")
        o = qo.lowbit_weight(w, w_bits, lw, dtype)["w_eff"]
        ref = U.bits_to_f32(g[k], dtype)
        # per-row scales and this small layerwise tensor (7680 elements) are bit contracts in both dtypes
        assert qo.count_mismatch(o, ref) == 0, k


def test_code_ranges_and_dequant_identity():
    rng = np.random.default_rng(7)
    x = (rng.standard_normal((64, 512)) * 0.5).astype(np.float32)
    for bits in (3, 4, 8):
        o = qo.sym_forward(x, bits)
        Q = 2 ** (bits - 1) - 1
        assert np.all(np.abs(o["codes"]) <= Q)
        # every row's abs-max element maps to +-Q
        assert np.all(np.max(np.abs(o["codes"]), axis=1) == Q)
        np.testing.assert_array_equal(o["y"], (o["codes"] / o["e"][:, None]).astype(np.float32))
        a = qo.asym_forward(x, bits)
        assert a["codes"].min() == 0 and a["codes"].max() == 2 ** bits - 1


def test_bf16_a8_codes_can_reach_128():
    """SURVEY.md section 7: bf16 rounding inflates the scale so |code| may be 128."""
    rng = np.random.default_rng(3)
    x = qo.bf16_round((rng.standard_normal((4096, 256))).astype(np.float32))
    codes = qo.sym_forward(x, 8, False, "bf16")["codes"]
    assert np.abs(codes).max() in (127.0, 128.0)
    assert np.abs(codes).max() == 128.0


def test_ste_mask_edges():
    x = np.array([2.0, -2.0, 1.9999999, -1.9999999, np.nan, np.inf, -np.inf, 0.0], dtype=np.float32)
    g = np.ones_like(x)
    out = qo.ste_backward(g, x, -2.0, 2.0)
    np.testing.assert_array_equal(out["mask"], [False, False, True, True, True, False, False, True])
    packed = qo.pack_mask(out["mask"])
    assert packed.tolist() == [0b10011100]


def test_reduction_view_shapes():
    assert qo.as_rows(np.zeros((2, 3, 8), np.float32), False).shape == (6, 8)
    assert qo.as_rows(np.zeros((2, 3, 4, 8), np.float32), False).shape == (6, 32)
    assert qo.as_rows(np.zeros((2, 3, 4, 8), np.float32), True).shape == (1, 192)
    with pytest.raises(ValueError):
        qo.as_rows(np.zeros((1, 1, 1, 1, 1), np.float32), False)


def test_bf16_round_is_nearest_even():
    # bf16 spacing at 1.0 is 2^-7: 1 + 2^-8 is a tie -> even (1.0); 1 + 3*2^-8 is a
    # tie -> even (1 + 2^-6); just above the first tie -> 1 + 2^-7
    v = np.array([1.0, 1.00390625, 1.01171875, 1.00390625 + 2.0 ** -12, np.inf, -0.0], dtype=np.float32)
    r = qo.bf16_round(v)
    np.testing.assert_array_equal(r[:4], np.array([1.0, 1.0, 1.015625, 1.0078125], dtype=np.float32))
    assert np.isinf(r[4]) and np.signbit(r[5])
    assert np.isnan(qo.bf16_round(np.array([np.nan], dtype=np.float32)))[0]


def test_bf16_reciprocal_quotient_proof(tmp_path):
    """The packed-bf16 AsymQuantizer chain of K2 replaces the reference's two divisions by
    multiplications with per-row reciprocals and its add/sub by single-rounding bf16x2
    instructions.  oracle/proofs/bf16_quotient_by_reciprocal.c checks both claims exhaustively
    (4.3e8 quotients; 4.26e9 add/sub pairs; 7.6e8 quotients of arbitrary ratio for the W1/W2 path): compile and run it."""
    import shutil
    import subprocess

    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    src = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "proofs",
                       "bf16_quotient_by_reciprocal.c")
    exe = str(tmp_path / "bf16q")
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", src, "-o", exe], check=True)
    for args in ([], ["addsub"], ["anyratio"]):
        r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and " 0 mismatches" in r.stdout, r.stdout + r.stderr


def _live_reference():
    """The original's models/utils_quant.py, imported read-only from the QAT_B200_REFERENCE checkout."""
    import importlib
    import sys

    sys.dont_write_bytecode = True
    if U.REFERENCE not in sys.path:
        sys.path.insert(0, U.REFERENCE)
    uq = importlib.import_module("models.utils_quant")
    assert uq.__file__.startswith(U.REFERENCE)
    return uq


def _fuzz_vs(uq):
    """The oracle against module `uq`'s SymQuantizer / AsymQuantizer on the seeded fuzz cases the GPU parity
    test uses: forward values and STE gradients, bit for bit."""
    import torch

    clip = torch.tensor([-2.0, 2.0])
    n = 0
    for seed in range(12):
        for what, dtype, sym, bits, lw, x, g in U.fuzz_cases(seed):
            xi = x.clone().requires_grad_(True)
            y = (uq.SymQuantizer if sym else uq.AsymQuantizer).apply(xi, clip, bits, lw)
            y.backward(g)
            ref = (qo.sym_forward if sym else qo.asym_forward)(U.tensor_to_f32(x), bits, lw, dtype)["y"]
            assert qo.count_mismatch(U.tensor_to_f32(y), ref) == 0, what
            gref = qo.ste_backward(U.tensor_to_f32(g), U.tensor_to_f32(x), -2.0, 2.0, dtype)["gx"]
            assert qo.count_mismatch(U.tensor_to_f32(xi.grad), gref) == 0, what
            n += 1
    assert n == 72


def _lowbit_edge_cases_vs(uq, monkeypatch):
    """The oracle's W1 / W2 weight path against module `uq`'s QuantizeLinear on the edge-row cases the GPU
    test uses; the effective weight is captured where QuantizeLinear.forward hands it to F.linear."""
    import torch
    import torch.nn as nn

    captured = {}
    orig = nn.functional.linear

    def capture(inp, weight, *a, **k):
        captured["w"] = weight.detach().clone()
        return orig(inp, weight, *a, **k)

    monkeypatch.setattr(nn.functional, "linear", capture)
    n = 0
    for dtype, w, bits, lw in U.lowbit_edge_cases():
        rows, cols = w.shape
        lin = uq.QuantizeLinear(cols, rows, w_bits=bits, a_bits=32, weight_layerwise=lw).to(w.dtype)
        with torch.no_grad():
            lin.weight.copy_(w)
        lin(torch.zeros(1, cols, dtype=w.dtype))
        ref = qo.lowbit_weight(U.tensor_to_f32(w), bits, lw, dtype)["w_eff"]
        assert U.lowbit_close(U.tensor_to_f32(captured["w"]), ref, dtype, U.lowbit_exact(lw, w.numel())), \
            (dtype, rows, cols, bits, lw)
        n += 1
    assert n == 72


@U.needs_reference
def test_oracle_fuzz_matches_live_reference():
    """The oracle against the UNMODIFIED reference (imported read-only) on the seeded fuzz cases."""
    _fuzz_vs(_live_reference())


@U.needs_reference
def test_oracle_lowbit_edge_cases_match_live_reference(monkeypatch):
    """The oracle's W1 / W2 weight path against the UNMODIFIED reference on the edge-row cases."""
    _lowbit_edge_cases_vs(_live_reference(), monkeypatch)


def test_oracle_fuzz_matches_ref_module():
    """The same fuzz cases against oracle/ref_module.py, which issues the reference's ATen op chain and is
    held bit for bit to the reference's stored outputs (test_harness.py::test_ref_module_reproduces_the_
    reference_goldens): the bit widths, widths, ranks and non-finite values the stored cases lack are
    checked on every machine."""
    from oracle import ref_module

    _fuzz_vs(ref_module)


def test_oracle_lowbit_edge_cases_match_ref_module(monkeypatch):
    """The W1 / W2 edge-row cases (shapes up to 40000 columns, layerwise included) against oracle/ref_module.py."""
    from oracle import ref_module

    _lowbit_edge_cases_vs(ref_module, monkeypatch)
