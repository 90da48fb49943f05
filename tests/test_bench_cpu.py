"""CPU checks of bench.py: the reference arm (`--impl reference`, the reference's own host code on the host cores) runs
without a GPU and prints the contract's JSON line; the product arm refuses to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest
from conftest import ROOT
from oracle_bindings import have_ref


@pytest.mark.skipif(not have_ref(), reason="oracle/_ref not built")
def test_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "24",
                          "--steps", "1", "--warmup", "0", "--ref-iters", "2"], capture_output=True, text=True,
                         timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is False and line["unit"] == "s"
    assert line["metric"].startswith("amg_pcg_solve_seconds")
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["gpu_launches"] == 0 and line["value"] > 0


@pytest.mark.skipif(not have_ref(), reason="oracle/_ref not built")
def test_reference_arm_runs_a_converged_solve_in_its_warmup():
    """with --warmup >= 1 the reference arm runs ONE solve to convergence with the reference's own stopping rule and
    extrapolates its bounded samples with THAT iteration count (same config dict as the product arm)"""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "24",
                          "--steps", "2", "--warmup", "1", "--ref-iters", "2"], capture_output=True, text=True,
                         timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    conv = line["details"]["converged_solve"]
    assert conv["iterations"] >= 5 and conv["final_rel_residual"] <= 1e-8 and conv["seconds"] > 0
    assert abs(line["value"] - line["details"]["seconds_per_pcg_iteration"] * conv["iterations"]) < 1e-12
    assert set(line["config"]) == {"workload", "grid", "rows", "nnz"} and line["config"]["rows"] == 24 ** 3


def test_reference_arm_non_zero_ranks_do_nothing():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--gpus", "2", "--dump-outputs", "out"],
                                   ["--impl", "reference", "--dump-outputs", "out"]])
def test_unsupported_arguments_are_refused(tmp_path, extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                         timeout=120, cwd=tmp_path)
    assert out.returncode == 2 and "error:" in out.stderr
    assert not os.path.exists(tmp_path / "out")


def test_dump_outputs_samples_long_vectors(tmp_path):
    """above DUMP_ROWS rows every vector is written at the same seeded rows, listed in x_index.npy; 256^3 stays < 64 MB"""
    import numpy as np

    import bench

    n = bench.DUMP_ROWS + 1000
    x = np.arange(n, dtype=np.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"x": x, "x_e2e": -x}, [2.0, 1.0])
    got = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert set(got) == {"x.npy", "x_e2e.npy", "x_index.npy", "residual_history.npy"}
    assert all(v.dtype == np.float64 for v in got.values())
    idx = got["x_index.npy"]
    assert len(idx) == bench.DUMP_ROWS and np.all(np.diff(idx) > 0) and idx[-1] < n
    np.testing.assert_array_equal(got["x.npy"], idx)
    np.testing.assert_array_equal(got["x_e2e.npy"], -idx)
    np.testing.assert_array_equal(got["residual_history.npy"], [2.0, 1.0])
    for f, v in got.items():
        np.testing.assert_array_equal(np.load(tmp_path / "b" / f), v)
    assert 3 * 8 * bench.DUMP_ROWS <= 64 << 20


def test_product_arm_needs_a_gpu():
    try:
        import torch

        if torch.cuda.is_available():
            pytest.skip("GPU present")
    except ImportError:
        pass
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--grid", "24", "--no-cpu-baseline"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0  # fails loudly: there is no CPU path to fall back to
    assert "\"metric\"" not in out.stdout
