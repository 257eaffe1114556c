"""bench.py's command line: the reference arm prints one JSON line with the result keys, the b200 arm refuses to run
without a GPU, and --dump-outputs writes the last timed step's results (sampling on the CPU, the b200 arm on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "16"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "solves/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["vs_baseline"] is None and d["gpu_launches"] == 0 and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_b200_arm_refuses_to_run_without_a_gpu():
    # no CPU fallback: without CUDA the product arm must fail loudly, not print a number
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline", "--no-sub"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert not any(ln.strip().startswith("{") and '"value"' in ln for ln in r.stdout.splitlines())


def _dump_size(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_dump_outputs_keeps_one_seeded_sample_under_64_mb(tmp_path):
    # the headline's result arrays at 2^20 problems (fp32 q [15][n] alone is 63 MB): one sample of problems for all
    import torch
    import bench
    n = 1 << 20
    q = torch.arange(15 * n, dtype=torch.float32).reshape(15, n)
    arrays = {"q": q, "converged": (torch.arange(n) % 3 == 0).to(torch.uint8), "iterations": torch.arange(n, dtype=torch.int32),
              "residual": torch.arange(2 * n, dtype=torch.float64).reshape(2, n)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    assert _dump_size(tmp_path / "a") <= bench.DUMP_BYTES
    idx = np.load(tmp_path / "a" / "problem_index.npy")
    assert idx.dtype == np.float64 and n // 2 < len(idx) < n and (np.diff(idx) > 0).all()
    i = idx.astype(np.int64)
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in arrays}
    assert {k: v.dtype for k, v in got.items()} == {"q": np.float32, "converged": np.float32, "iterations": np.float32,
                                                   "residual": np.float64}
    for k, t in arrays.items():
        assert np.array_equal(got[k], t.double().numpy()[..., i]), k
        assert np.array_equal(got[k], np.load(tmp_path / "b" / f"{k}.npy")), k      # same sample every run
    # small outputs are written whole
    bench.dump_outputs(str(tmp_path / "c"), {"q": q[:, :1000]})
    assert np.array_equal(np.load(tmp_path / "c" / "q.npy"), q[:, :1000].numpy())
    assert np.array_equal(np.load(tmp_path / "c" / "problem_index.npy"), np.arange(1000.0))


@pytest.mark.gpu
@pytest.mark.parametrize("config,n,expected", [
    (2, 8192, {"q": ((15, 8192), np.float32), "converged": ((8192,), np.float32), "iterations": ((8192,), np.float32),
               "residual": ((2, 8192), np.float32)}),
    (3, 128, {"q_best": ((15, 128), np.float64), "converged": ((128,), np.float32), "restart": ((128,), np.float32)}),
    (4, 64, {"q_path": ((256, 15, 64), np.float32), "n_valid": ((64,), np.float32), "iterations": ((64,), np.float32)}),
])
def test_b200_arm_dumps_the_last_step_identically_every_run(tmp_path, config, n, expected):
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", str(config), "--steps", "2",
                            "--warmup", "1", "--n", str(n), "--no-cpu-baseline", "--no-e2e", "--no-sub",
                            "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == 2
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted([f"{k}.npy" for k in expected] + ["problem_index.npy"])
    for k, (shape, dtype) in expected.items():
        a = np.load(tmp_path / "a" / f"{k}.npy")
        assert a.shape == shape and a.dtype == dtype, k
    assert np.array_equal(np.load(tmp_path / "a" / "problem_index.npy"), np.arange(float(n)))
    if config == 4:
        nv = np.load(tmp_path / "a" / "n_valid.npy")
        assert ((nv >= 0) & (nv <= 256) & (nv == np.round(nv))).all() and nv.mean() > 1
    else:
        conv = np.load(tmp_path / "a" / "converged.npy")
        assert set(np.unique(conv)) <= {0.0, 1.0} and conv.mean() > 0.5
    for f in names:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
