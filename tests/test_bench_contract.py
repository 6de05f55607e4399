"""bench.py's reference arm runs without a GPU: check the JSON-line contract the driver parses
(one line, the metric/config keys, the cpu_baseline and e2e objects of the tier's reference arm)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1", *args], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "fake-quant fwd+bwd GB/s" and d["unit"] == "GB/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["steps"] == 2 and d["gpu_launches"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_nonzero_ranks_do_no_work():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, ("--gpus", "2")) == []


def test_dump_outputs_writes_the_last_step_of_the_workload(tmp_path):
    """--dump-outputs: float32 arrays of at most 64 MB in all, holding exactly what the port computes on the
    sampled rows of the seeded workload (quantization is per row, so a row sample is computed the same way)."""
    import numpy as np

    import bench
    from oracle import torch_chain as tc

    assert len(_run(args=("--dump-outputs", str(tmp_path / "out")))) == 1
    files = sorted(os.listdir(tmp_path / "out"))
    assert files == ["grad_w.npy", "grad_x.npy", "y_w.npy", "y_x.npy"]
    got = {f[:-4]: np.load(tmp_path / "out" / f) for f in files}
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    hx, hw, hgx, hgw = bench.make_inputs(1234)
    rx, rw = bench.dump_rows()
    y_x, grad_x = tc.fwd_bwd(hx[rx], hgx[rx], bench.A_BITS, True, bench.CLIP)
    y_w, grad_w = tc.fwd_bwd(hw[rw], hgw[rw], bench.W_BITS, True, bench.CLIP)
    for name, want in (("y_x", y_x), ("y_w", y_w), ("grad_x", grad_x), ("grad_w", grad_w)):
        assert got[name].dtype == np.float32 and got[name].shape == (bench.DUMP_ROWS, bench.K_IN), name
        assert np.array_equal(got[name], want.float().numpy()), name


@pytest.mark.gpu
def test_b200_arm_dump_equals_the_reference_arm_dump(tmp_path):
    """The b200 arm's --dump-outputs (the kernels' output buffers after the CUDA-graph replays of the timed steps)
    against the reference arm's on the same seeded workload.  The bf16 A8 / W4 SymQuantizer forward and the STE
    backward are bit-exact contracts, so every dumped element must be identical."""
    import numpy as np

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-qat-step",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "b200")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.splitlines()[-1])["steps"] == 2
    assert len(_run(args=("--dump-outputs", str(tmp_path / "ref")))) == 1
    for name in ("y_x", "y_w", "grad_x", "grad_w"):
        got, want = np.load(tmp_path / "b200" / f"{name}.npy"), np.load(tmp_path / "ref" / f"{name}.npy")
        assert got.dtype == want.dtype == np.float32 and got.shape == want.shape, name
        assert np.array_equal(got, want, equal_nan=True), (name, int((got != want).sum()))
