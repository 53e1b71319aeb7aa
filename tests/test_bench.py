"""bench.py's command line: argument checks (no GPU needed) and one small run with --dump-outputs on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_bad_arguments(tmp_path, args):
    r = subprocess.run([sys.executable, BENCH, *args], cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "error:" in r.stderr and r.stdout == ""
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_bench_steps_and_dump_outputs(mplu, tmp_path):
    """--steps sets the timed steps; --dump-outputs writes the last step's solution, the same on a second run."""
    n = 4096
    xs = []
    for run in range(2):
        out = tmp_path / f"out{run}"
        cmd = [sys.executable, BENCH, "--gpus", "1", "--steps", str(2 + run), "--warmup", "3", "--n", str(n), "--no-e2e",
               "--no-cpu-baseline", "--extra-n", "0", "--dropin-n", "0", "--dump-outputs", str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = r.stdout.strip().splitlines()
        assert len(lines) == 1
        line = json.loads(lines[0])
        assert line["steps"] == 2 + run and line["config"]["n"] == n
        assert sorted(os.listdir(out)) == ["x.npy"]
        x = np.load(out / "x.npy")
        assert x.dtype == np.float64 and x.shape == (n,)
        assert np.abs(x - 1).max() == line["max_abs_err"] <= 1e-12
        xs.append(x)
    np.testing.assert_allclose(xs[0], xs[1], rtol=0, atol=1e-13)
