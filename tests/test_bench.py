"""bench.py as a program: `--steps` sets the number of timed steps, and `--dump-outputs` writes what the timed rollouts
returned (config 2 checked against the oracle on the same counter-RNG inputs)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT)


def test_rejects_zero_steps():
    r = run_bench("--gpus", "1", "--steps", "0", "--warmup", "1")
    assert r.returncode == 2 and "--steps must be >= 1" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_and_step_count(tmp_path, oracle):
    B, N, Bi, Ni, steps = 4096, 50, 2048, 40, 2
    r = run_bench("--gpus", "1", "--steps", str(steps), "--warmup", "1", "--traj", str(B), "--horizon", str(N),
                  "--id-samples", str(Bi), "--id-horizon", str(Ni), "--no-sens", "--no-e2e", "--no-cpu-baseline",
                  "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["steps"] == steps and res["gpu_launches"] == steps
    assert res["id_sweep"]["gpu_launches"] == steps
    assert sorted(os.listdir(tmp_path)) == ["config2_xf.npy", "config5_cost.npy", "config5_status.npy", "config5_xf.npy"]
    xf = np.load(tmp_path / "config2_xf.npy")
    assert xf.dtype == np.float64 and xf.shape == (13, B)
    ref = oracle.rollout(None, None, N, 1e-3, u_mode=3, traj0=0, n=B)
    assert_close(xf.T, ref, 1e-9, what="config-2 dump")
    xi, cost, st = (np.load(tmp_path / ("config5_%s.npy" % n)) for n in ("xf", "cost", "status"))
    assert st.shape == (Bi,) and st.dtype == np.float32
    n_ok = int((st == 0).sum())                       # final states and costs of the unflagged samples only
    assert n_ok > 0 and xi.shape == (13, n_ok) and cost.shape == (n_ok,) and (cost >= 0).all()
    for name in os.listdir(tmp_path):
        assert np.isfinite(np.load(tmp_path / name)).all(), name
