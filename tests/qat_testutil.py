"""Shared helpers for the parity tests: golden fixtures as raw bits, bit-level compares."""
from __future__ import annotations

import os

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
_cache = {}

# A checkout of the original LLM-QAT project (the directory holding its models/ package).  The tests that import
# its code run only where QAT_B200_REFERENCE names one; what it computed on the stored cases is in golden/.
REFERENCE = os.path.abspath(os.environ["QAT_B200_REFERENCE"]) if os.environ.get("QAT_B200_REFERENCE") else ""
needs_reference = pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "models"))),
                                     reason="needs the original project's source: set QAT_B200_REFERENCE to a checkout")


def golden(dtype: str):
    if dtype not in _cache:
        _cache[dtype] = np.load(os.path.join(GOLD, f"quant_{dtype}.npz"))
    return _cache[dtype]


def bits_to_f32(bits: np.ndarray, dtype: str) -> np.ndarray:
    """Stored raw bits -> float32 values (exact for both dtypes)."""
    if dtype == "bf16":
        return (bits.astype(np.uint32) << 16).view(np.float32)
    return bits.view(np.float32)


def bits_to_tensor(bits: np.ndarray, dtype: str, device="cpu") -> torch.Tensor:
    if dtype == "bf16":
        t = torch.from_numpy(bits.view(np.int16).copy()).view(torch.bfloat16)
    else:
        t = torch.from_numpy(bits.view(np.int32).copy()).view(torch.float32)
    return t.to(device)


def tensor_to_f32(t: torch.Tensor) -> np.ndarray:
    return t.detach().float().cpu().numpy()


def tensor_bits(t: torch.Tensor) -> np.ndarray:
    t = t.detach().cpu().contiguous()
    if t.dtype == torch.bfloat16:
        return t.view(torch.int16).numpy().view(np.uint16)
    return t.view(torch.int32).numpy().view(np.uint32)


def mismatches(a_bits: np.ndarray, b_bits: np.ndarray, dtype: str) -> int:
    """Elements whose bit patterns differ, treating any NaN == any NaN."""
    if a_bits.shape != b_bits.shape:
        return max(a_bits.size, b_bits.size)
    a, b = bits_to_f32(a_bits, dtype), bits_to_f32(b_bits, dtype)
    na, nb = np.isnan(a), np.isnan(b)
    return int(np.count_nonzero(((a_bits != b_bits) & ~(na & nb)) | (na != nb)))


def f32_mismatches(a: np.ndarray, b: np.ndarray) -> int:
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    return mismatches(a.view(np.uint32), b.view(np.uint32), "fp32")


def quant_cases(g):
    """[(quantizer, input key, bits, layerwise)] present in a golden file."""
    out = []
    for k in g.files:
        if k.startswith("y/"):
            _, q, key, b, mode = k.split("/")
            out.append((q, key, int(b[1:]), mode == "lw"))
    return out


def clip_cases(g):
    out = []
    for k in g.files:
        if k.startswith("gx/"):
            _, q, key, mode, clip = k.split("/")
            lo, hi = clip[4:].split("_")
            out.append((q, key, mode == "lw", float(lo), float(hi), k))
    return out


def fuzz_cases(seed: int, n_cases: int = 6):
    """Seeded random fake-quant cases shared by the CPU test that pins the oracle to the live
    reference and the GPU test that pins the kernels to the oracle: 1-D..4-D shapes (widths
    1..9000, odd ones included), Sym bits 2..16 / Asym bits 2..12, both dtypes, layerwise now
    and then, magnitudes 1e-3..1e3, injected +-2.0 / zeros / -0.0 / an all-zero row and, in the
    last case of a seed, one NaN or +-inf.  Yields (what, dtype, sym, bits, layerwise, x, g)."""
    rng = np.random.default_rng(1000 + seed)
    gen = torch.Generator().manual_seed(2000 + seed)
    for case in range(n_cases):
        dtype = ("fp32", "bf16")[int(rng.integers(2))]
        nd = int(rng.integers(1, 5))
        cols = int(rng.choice([1, 7, 8, 24, 100, 172, 256, 1000, 1023, 4096, int(rng.integers(1, 9000))]))
        lead = [int(rng.integers(1, 5)) for _ in range(nd - 1)]
        if nd == 4:   # reduction over the last two dims
            shape = (lead[0], lead[1], int(rng.integers(1, 9)), max(1, cols // 8))
        else:
            shape = tuple(lead) + (cols,)
        sym = bool(rng.integers(2))
        bits = int(rng.choice([2, 3, 4, 5, 6, 7, 8, 9, 12, 16] if sym else [2, 3, 4, 5, 7, 8, 9, 12]))
        lw = bool(rng.integers(5) == 0)
        scale = float(10.0 ** rng.uniform(-3, 3))
        x = torch.randn(*shape, generator=gen) * scale
        flat = x.view(-1)
        n = flat.numel()
        flat[::13] = 0.0
        if n > 4:
            flat[1], flat[2], flat[3] = 2.0, -2.0, -0.0
        if nd >= 2 and shape[-1] > 1 and not lw:
            x.view(-1, shape[-1])[0] = 0.0
        if case == n_cases - 1 and n > 16:
            flat[int(rng.integers(n))] = (float("nan"), float("inf"), -float("inf"))[seed % 3]
        x = x.to(DTYPES[dtype])
        g = torch.randn(*shape, generator=gen).to(DTYPES[dtype])
        what = (seed, case, dtype, shape, "sym" if sym else "asym", bits, lw, scale)
        yield what, dtype, sym, bits, lw, x, g


def lowbit_edge_cases():
    """Weights for the W1 / W2 path: LLaMA-like and ragged shapes with an all-zero row, +-inf, NaN,
    -0.0 and magnitudes spread over 2^40.  Yields (dtype, w, bits, layerwise); shared by the CPU test
    that pins the oracle to the live reference and the GPU test that pins the kernels to the oracle."""
    gen = torch.Generator().manual_seed(12)
    for dtype in ("fp32", "bf16"):
        for rows, cols in ((64, 4096), (16, 11008), (9, 1000), (5, 172), (7, 1023), (5, 7), (5, 20), (6, 33),
                           (5, 40000)):
            w = (torch.randn(rows, cols, generator=gen) * 0.02).to(DTYPES[dtype])
            w[0] = 0.0
            w[1, :6] = torch.tensor([float("inf"), -float("inf"), 1e-30, -1e-30, -0.0, 3.0]).to(w.dtype)
            w[2, 3] = float("nan")
            w[3, ::7] *= 1e6
            w[4, ::5] *= 1e-6
            for bits in (1, 2):
                for lw in (False, True):
                    yield dtype, w, bits, lw


def lowbit_exact(layerwise: bool, numel: int) -> bool:
    """Where the W1 / W2 effective weight is a bit contract: always for per-row scales; for the layerwise scale only
    below 32768 elements — from there on torch splits the full `mean()` over its threads and the reference's own
    bits depend on the machine (tests/test_torch_sum_order.py)."""
    return (not layerwise) or numel < 32768


def lowbit_close(got: np.ndarray, ref: np.ndarray, dtype: str, exact: bool = True) -> bool:
    """Bit for bit; with exact=False (large layerwise tensors, see lowbit_exact) bf16 stays bit for bit and fp32 is
    the same NaN / inf pattern and 2e-6 relative (the thread-dependent summation order of a full `mean()`)."""
    if exact or dtype == "bf16":
        return f32_mismatches(got, ref) == 0
    with np.errstate(all="ignore"):
        if not (np.array_equal(np.isnan(got), np.isnan(ref)) and np.array_equal(np.isfinite(got), np.isfinite(ref))):
            return False
        ok = np.isfinite(ref)
        return bool((np.abs(got[ok] - ref[ok]) / (np.abs(ref[ok]) + 1e-30)).max(initial=0.0) < 2e-6)
