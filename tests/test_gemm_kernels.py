"""The two tcgen05 GEMMs built on tcgen05_gemm.cuh: what the compiled library contains (CPU, cuobjdump on the
built library) and that the CTA-group setter reaches both of them (GPU)."""
import collections
import os
import re
import shutil
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "llm-qat_b200", "lib", "libqat_b200.so")


def _cuobjdump(*args):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    return subprocess.run([exe, *args, LIB], capture_output=True, text=True, check=True).stdout


def _gemm_kernels():
    """{mangled name: (family, Counter of SASS mnemonics, stack bytes)} for the two GEMM families."""
    fam = lambda n: next((f for f in ("qlinear_i8_kernel", "gemm_bf16_kernel") if f in n), None)
    stack = {}
    cur = None
    for ln in _cuobjdump("-res-usage").splitlines():
        m = re.match(r"\s*Function (\S+):", ln)
        if m:
            cur = m.group(1)
        elif cur and "STACK:" in ln:
            stack[cur] = int(re.search(r"STACK:(\d+)", ln).group(1))
            cur = None
    out = {}
    cur = None
    for ln in _cuobjdump("-sass").splitlines():
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            cur = m.group(1) if fam(m.group(1)) else None
            if cur:
                out[cur] = (fam(cur), collections.Counter(), stack[cur])
            continue
        m = cur and re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]+)", ln)
        if m:
            out[cur][1][m.group(1)] += 1
    return out


def test_gemm_instances_and_their_hardware_paths():
    kernels = _gemm_kernels()
    by_fam = collections.defaultdict(list)
    for name, (f, ops, stack) in kernels.items():
        by_fam[f].append((name, ops, stack))
    assert len(by_fam["qlinear_i8_kernel"]) == 4, sorted(kernels)
    assert len(by_fam["gemm_bf16_kernel"]) == 8, sorted(kernels)
    for name, ops, _ in by_fam["qlinear_i8_kernel"]:
        assert ops["UTCIMMA"] > 0 and ops["UTCHMMA"] == 0, (name, ops)
    for name, ops, _ in by_fam["gemm_bf16_kernel"]:
        assert ops["UTCHMMA"] > 0 and ops["UTMALDG"] > 0 and ops["LDTM"] > 0, (name, ops)
    # the only stack frame is the printf argument buffer of the mbarrier timeout (stored, never
    # loaded back): no spills
    for name, (_, ops, stack) in kernels.items():
        assert stack <= 24 and ops["LDL"] == 0, (name, stack, ops)


@pytest.mark.gpu
@pytest.mark.parametrize("cg", [1, 2])
def test_gemm_cta_group_setter_reaches_the_bf16_gemm(cg):
    """qat_set_gemm_cta_group() pins the tile plan of qat_gemm_bf16 with cta_group == 0 too."""
    from llm_qat_b200 import _lib

    M, N, K = 2048, 4096, 1024   # automatic choice would be CG = 2 here; CG = 1 must still be honoured
    gen = torch.Generator().manual_seed(3)
    a = torch.randn(M, K, generator=gen).bfloat16().cuda()
    b = torch.randn(N, K, generator=gen).bfloat16().cuda()
    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    _lib.check(_lib.lib().qat_set_gemm_cta_group(cg))
    try:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            _lib.check(_lib.lib().qat_gemm_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), 0, M, N, K, 0, 0, 1, 0,
                                                torch.cuda.current_stream().cuda_stream), "qat_gemm_bf16")
            torch.cuda.synchronize()
    finally:
        _lib.lib().qat_set_gemm_cta_group(0)
    ran = {m.group(1) for e in prof.key_averages()
           for m in [re.search(r"gemm_bf16_kernel<\w+, \w+, (\d)>", e.key)] if m}
    assert ran == {str(cg)}, [e.key for e in prof.key_averages()]
