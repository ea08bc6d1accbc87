"""bench.py --dump-outputs: the outputs of the last timed step, within the size budget, on inputs that repeat from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_keeps_a_fixed_particle_sample_within_budget(tmp_path):
    import bench
    H, M = 60, 131072
    particle = torch.arange(M, dtype=torch.float64).repeat(H, 1)[..., None]         # every entry holds its particle index
    arrays = {"states": particle.expand(H, M, 4).contiguous(), "inputs": -particle, "cost": torch.tensor(1.5, dtype=torch.float64),
              "grad_centers": torch.randn(200, 5, dtype=torch.float64, generator=torch.Generator().manual_seed(0))}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, per_particle=("states", "inputs"))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["cost.npy", "grad_centers.npy", "inputs.npy", "states.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert a["cost.npy"].shape == () and float(a["cost.npy"]) == 1.5
    np.testing.assert_array_equal(a["grad_centers.npy"], arrays["grad_centers"].numpy())
    kept = a["states.npy"].shape[1]
    assert a["states.npy"].shape == (H, kept, 4) and a["inputs.npy"].shape == (H, kept, 1) and 0 < kept < M
    # distinct particles in order, the same ones in both arrays and in both dumps
    idx = a["states.npy"][0, :, 0].astype(np.int64)
    assert (np.diff(idx) > 0).all()
    np.testing.assert_array_equal(a["states.npy"], arrays["states"].numpy()[:, idx])
    np.testing.assert_array_equal(a["inputs.npy"], arrays["inputs"].numpy()[:, idx])
    for f in files:
        np.testing.assert_array_equal(np.load(tmp_path / "b" / f), a[f])
    # below the budget nothing is sampled
    small = {k: (v[:, :1000] if v.dim() == 3 else v) for k, v in arrays.items()}
    bench.dump_outputs(str(tmp_path / "c"), small, per_particle=("states", "inputs"))
    np.testing.assert_array_equal(np.load(tmp_path / "c" / "states.npy"), small["states"].numpy())


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    H, M = 5, 64
    args = ["--steps", "2", "--warmup", "1", "--train-points", "256", "--particles-per-gpu", str(M), "--horizon", str(H), "--e2e-steps", "0",
            "--no-cpu-baseline", "--no-real-shapes", "--no-variants", "--no-forward-only"]
    runs = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(tmp_path / d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout)
        assert line["steps"] == 2
        out = {f[:-4]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)}
        assert set(out) == {"states", "inputs", "cost", "std_cost", "grad_log_lengthscales", "grad_centers", "grad_weight"}
        assert all(a.dtype == np.float64 for a in out.values())
        assert out["states"].shape == (H, M, 4) and out["inputs"].shape == (H, M, 1) and out["grad_centers"].shape == (200, 5)
        assert float(out["cost"]) == line["config"]["cost"]            # the step the JSON line reports
        runs.append(out)
    np.testing.assert_array_equal(runs[0]["states"][0], runs[1]["states"][0])   # same initial particles: same inputs in both runs
