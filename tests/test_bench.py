"""bench.py's command line: the timed step count and --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", *args],
                          capture_output=True, text=True, timeout=900, cwd=ROOT)


def test_steps_below_one_rejected():
    r = _bench("--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """ap400: 3 warm-up + 2 timed bench steps of 20 MD steps each, chained from the seed-0 lattice, are
    100 MD steps; the dump holds every particle and is that state bit for bit, run after run."""
    from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
    from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        r = _bench("--steps", "2", "--warmup", "3", "--workload", "ap400", "--md-steps", "20",
                   "--no-cpu-baseline", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2 and line["warmup"] == 3
        assert sorted(os.listdir(d)) == ["positions.npy", "velocities.npy"]
        dumps.append({n: np.load(d / f"{n}.npy") for n in ("positions", "velocities")})
    for a in dumps[0].values():
        assert a.dtype == np.float32 and a.shape == (400, 2)
    for n in dumps[0]:
        assert np.array_equal(dumps[0][n], dumps[1][n])
    R, V, _ = lattice_jitter(400, seed=0)
    (R1, V1), _ = LJSimulation(400, rc=None, dt=1e-3, path="allpairs").run((R, V), 100)
    assert np.array_equal(dumps[0]["positions"], R1.numpy())
    assert np.array_equal(dumps[0]["velocities"], V1.numpy())


@pytest.mark.gpu
def test_dump_outputs_samples_large_systems(tmp_path):
    """cells4m (4 M particles): a fixed sample of 2^20 rows, 16 MiB in all."""
    r = _bench("--steps", "1", "--warmup", "0", "--workload", "cells4m", "--md-steps", "10",
               "--no-cpu-baseline", "--no-check", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    R = np.load(tmp_path / "positions.npy")
    V = np.load(tmp_path / "velocities.npy")
    assert R.dtype == V.dtype == np.float32 and R.shape == V.shape == (1 << 20, 2)
    assert np.isfinite(R).all() and np.isfinite(V).all() and R.min() >= 0.0
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20
