"""GPU check of bench.py --dump-outputs: the outputs of the last timed step land as float64 .npy files, and the same
arguments give the same inputs, hence the same solution, from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
from conftest import ROOT

pytestmark = pytest.mark.gpu


def run_bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--grid", "24", "--steps", str(steps), "--warmup", "0",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_dump_outputs_of_the_last_step(tmp_path, oracle):
    lines = {d: run_bench(tmp_path / d, steps) for d, steps in (("one", 1), ("two", 2))}
    assert lines["one"]["steps"] == 1 and lines["two"]["steps"] == 2
    A = oracle.gen_poisson3d(24, 24, 24)
    b = np.ones(A.nrow)
    got = {}
    for d, line in lines.items():
        files = {f[:-4]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)}
        assert set(files) == {"x", "x_e2e", "x_index", "residual_history"}
        assert all(v.dtype == np.float64 for v in files.values())
        np.testing.assert_array_equal(files["x_index"], np.arange(A.nrow))  # small enough to be written whole
        assert len(files["residual_history"]) == line["details"]["pcg_iterations"] + 1
        for name in ("x", "x_e2e"):
            assert np.linalg.norm(b - A.to_scipy() @ files[name]) <= 2e-8 * np.linalg.norm(b), name
        np.testing.assert_allclose(files["x_e2e"], files["x"], rtol=1e-10)
        got[d] = files
    for name in ("x", "x_e2e", "residual_history"):
        np.testing.assert_allclose(got["two"][name], got["one"][name], rtol=1e-10)
