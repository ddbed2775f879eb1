"""Density modes on the GPU (ljmd_density_modes, csrc/sk.cu) and the structure factor built on them
(LJSimulation.structure_factor, driver --sk_kmax): against the fp64 CPU reference (tests/sk_reference.c) within the
derived bound, known answers, periodicity, determinism, the NaN rule, argument errors and the launch count."""
import os

import numpy as np
import pytest
import torch

from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation, structure_factor_vectors
from sk_reference import bound, c_density_modes

pytestmark = pytest.mark.gpu

E_INVALID = -1
LAUNCHES = 2                            # per batch of snapshots and vectors


def _sim(N, path="auto", **kw):
    return LJSimulation(N, rc=2.5, dt=0.005, path=path, device=0, **kw)


def _half_plane(nmax):
    """Every n with 0 < |n| <= nmax, one of each +-n pair."""
    v = [(x, y) for y in range(0, nmax + 1) for x in range(-nmax, nmax + 1)
         if (y > 0 or x > 0) and x * x + y * y <= nmax * nmax]
    return np.array(v, dtype=np.int32)


def modes(sim, R, nvec):
    """rho (S, K, 2) float64 on the host and the launches of the call."""
    l0 = sim.launch_count()
    rho = sim.density_modes(R, nvec).numpy()
    return rho, sim.launch_count() - l0


def _snapshots(sim, N, nsteps=30, every=10, seed=0):
    R, V, box = lattice_jitter(N, seed=seed)
    (_, _), traj = sim.run((R, V), nsteps, sample_every=every)
    return traj.numpy(), box


def _check_bound(got, ref, N, nvec, what):
    b = bound(N, nvec)
    err = np.abs(got - ref).max(axis=-1)                  # (S, K): worse of Re and Im
    ratio = (err / b).max()
    print(f"{what}: max |error| {err.max():.3e}, max error / bound {ratio:.3e}, "
          f"max error / (sqrt(N) eps_term) {(err / (np.sqrt(N) * 1.074e-6)).max():.2f}")
    assert np.isfinite(got).all() and ratio <= 1.0, what
    return ratio


@pytest.mark.parametrize("N", [400, 4096])
def test_snapshots_against_reference(N):
    sim = _sim(N)
    th, box = _snapshots(sim, N)
    nv = _half_plane(40)
    rho, launches = modes(sim, th, nv)
    assert rho.shape == (th.shape[0], nv.shape[0], 2) and launches == LAUNCHES
    _check_bound(rho, c_density_modes(th, box, nv), N, nv, f"N={N}, |n|<=40")


def test_large_n_against_reference():
    N = 4194304
    sim = _sim(N, path="cells")
    R, _, box = lattice_jitter(N, seed=3)
    nv = _half_plane(8)
    rho, launches = modes(sim, R, nv)
    assert launches == LAUNCHES
    ref = c_density_modes(R, box, nv)
    _check_bound(rho, ref, N, nv, "N=4194304, |n|<=8")


def test_square_lattice_bragg_peaks():
    m = 64
    N = m * m
    sim = _sim(N, box_size=float(m))
    ii, jj = np.meshgrid(np.arange(m), np.arange(m), indexing="ij")
    R = np.stack([ii.ravel(), jj.ravel()], axis=1).astype(np.float32)       # exact phase words
    nv = _half_plane(2 * m + 2)
    rho = modes(sim, R, nv)[0][0]
    bragg = (nv[:, 0] % m == 0) & (nv[:, 1] % m == 0)
    assert bragg.sum() == 6                                 # (64,0) (0,64) (+-64,64) (128,0) (0,128)
    b = bound(N, nv)
    assert np.all(np.abs(rho[bragg, 0] - N) <= b[bragg]) and np.all(np.abs(rho[bragg, 1]) <= b[bragg])
    assert np.all(np.abs(rho[~bragg]).max(axis=1) <= b[~bragg])


def test_uniform_random_points():
    N = 4096
    sim = _sim(N)
    box = float(sim.box_size)
    R = (np.random.default_rng(21).random((N, 2)) * box).astype(np.float32)
    nv, _ = structure_factor_vectors(box, 8.0)
    K = nv.shape[0]
    assert K >= 10000
    rho = modes(sim, R, nv)[0][0]
    s = (rho[:, 0] ** 2 + rho[:, 1] ** 2) / N
    assert abs(s.mean() - 1.0) <= 5.0 / np.sqrt(K), s.mean()


def test_large_wave_numbers():
    N = 400
    sim = _sim(N)
    th, box = _snapshots(sim, N, nsteps=10, every=10)
    rng = np.random.default_rng(5)
    nv = np.concatenate([np.array([[8192, 0], [0, 8192], [8192, -8192], [-8192, 8192], [5000, 7000],
                                   [8191, 1], [1, -8191]], np.int32),
                         rng.integers(-8192, 8193, size=(500, 2)).astype(np.int32)])
    rho = modes(sim, th, nv)[0]
    _check_bound(rho, c_density_modes(th, box, nv), N, nv, "N=400, |n_i|<=8192")


def _dyadic_state(N, box, seed):
    """Positions in [0, box) on multiples of 2^-17 (box = 64): x +- box and x + d stay exact in fp32."""
    rng = np.random.default_rng(seed)
    return (np.floor(rng.random((N, 2)) * box * 2 ** 17) / 2 ** 17).astype(np.float32)


def test_periodic_images_give_the_same_bits():
    N, box = 4096, 64.0
    sim = _sim(N, box_size=box)
    R = _dyadic_state(N, box, 1)
    imgs = np.stack([R, R + np.float32(box), R - np.float32(box),
                     R + np.array([box, -2 * box], np.float32)]).astype(np.float32)
    assert np.array_equal(imgs[1] - np.float32(box), R)                     # the shifts are exact
    assert np.array_equal(imgs[3] - np.array([box, -2 * box], np.float32), R)
    nv = _half_plane(30)
    rho = modes(sim, imgs, nv)[0]
    for s in range(1, 4):
        assert np.array_equal(rho[s], rho[0]), s


def test_translation_keeps_the_modulus():
    N, box = 4096, 64.0
    sim = _sim(N, box_size=box)
    R = _dyadic_state(N, box, 2)
    d = np.array([13.375, -7.5], np.float32)
    nv = _half_plane(30)
    rho = modes(sim, np.stack([R, (R + d).astype(np.float32)]), nv)[0]
    a = np.hypot(rho[0, :, 0], rho[0, :, 1])
    t = np.hypot(rho[1, :, 0], rho[1, :, 1])
    assert np.all(np.abs(a - t) <= 2 * np.sqrt(2) * bound(N, nv))


def test_deterministic_and_independent_of_the_batch():
    N = 4096
    sim = _sim(N)
    th, _ = _snapshots(sim, N, nsteps=50, every=10)
    nv = _half_plane(40)
    a = modes(sim, th, nv)[0]
    b = modes(sim, th, nv)[0]
    assert np.array_equal(a, b)
    for s in range(th.shape[0]):
        assert np.array_equal(modes(sim, th[s], nv)[0][0], a[s])
    # a vector's value does not depend on the other vectors either
    assert np.array_equal(modes(sim, th, nv[7:9])[0], a[:, 7:9])


def test_scratch_batches_give_the_single_batch_bits():
    """N = 2^20 has 1024 particle segments, so 16 KiB of scratch per (snapshot, vector): a call with more than
    32,768 vectors, or more snapshots than fit next to them in 512 MiB, is split into several batches."""
    N = 1 << 20
    sim = _sim(N, path="cells")
    R, _, box = lattice_jitter(N, seed=9)
    nv = _half_plane(160)[:40000]
    assert nv.shape[0] == 40000
    rho, launches = modes(sim, R, nv)
    assert launches == 2 * LAUNCHES                                          # two vector batches
    lo, l1 = modes(sim, R, nv[:20000])
    hi, l2 = modes(sim, R, nv[20000:])
    assert l1 == l2 == LAUNCHES
    assert np.array_equal(np.concatenate([lo, hi], axis=1), rho)
    # snapshots: 34 x 1000 vectors need two batches (32 snapshots fit)
    Rs = np.stack([R, lattice_jitter(N, seed=10)[0]] * 17)
    few = nv[:1000]
    rs, launches = modes(sim, Rs, few)
    assert launches == 2 * LAUNCHES
    for s in (0, 1, 31, 32, 33):
        assert np.array_equal(modes(sim, Rs[s], few)[0][0], rs[s]), s
    _check_bound(rs[:2, :200], c_density_modes(Rs[:2], box, few[:200]), N, few[:200], "N=2^20, batched")


def test_nan_snapshot_rows():
    N = 4096
    sim = _sim(N)
    th, _ = _snapshots(sim, N)
    nv = _half_plane(20)
    clean = modes(sim, th, nv)[0]
    for bad in (np.nan, np.inf, -np.inf):
        X = th.copy()
        X[1, 1234, 1] = bad
        rho = modes(sim, X, nv)[0]
        sim.check()
        assert sim.lib.ljmd_check(sim._h) == 0
        assert np.isnan(rho[1]).all()
        assert np.array_equal(rho[0], clean[0]) and np.array_equal(rho[2], clean[2])


def test_structure_factor_is_the_shell_mean():
    N = 4096
    sim = _sim(N)
    th, box = _snapshots(sim, N)
    k, S = sim.structure_factor(th, 4.0)
    nv, shell = structure_factor_vectors(float(box), 4.0)
    assert np.array_equal(sim.last_sk_nvec, nv) and np.array_equal(sim.last_sk_shell, shell)
    rho = modes(sim, th, nv)[0]
    p = (rho[..., 0] ** 2 + rho[..., 1] ** 2) / N
    assert np.allclose(sim.last_sk_power.numpy(), p, rtol=1e-14, atol=0)
    kmag = 2 * np.pi / float(box) * np.hypot(nv[:, 0], nv[:, 1])
    shells = np.unique(shell)
    want_S = np.array([p[:, shell == m].mean() for m in shells])
    want_k = np.array([kmag[shell == m].mean() for m in shells])
    assert k.shape == S.shape == (shells.size,) and k.dtype == S.dtype == torch.float64
    assert np.allclose(S.numpy(), want_S, rtol=1e-12, atol=0) and np.allclose(k.numpy(), want_k, rtol=1e-12)
    assert np.all(np.diff(k.numpy()) > 0) and k.numpy()[-1] <= 4.0
    # max_per_shell keeps at most M vectors per shell
    k2, S2 = sim.structure_factor(th, 4.0, max_per_shell=8)
    nv8, sh8 = structure_factor_vectors(float(box), 4.0, 8)
    assert np.array_equal(sim.last_sk_nvec, nv8) and nv8.shape[0] < nv.shape[0]
    assert np.bincount(sh8).max() == 8 and k2.shape == k.shape
    # a liquid-like lattice-jitter state: S(k) small at small k, a peak near 2 pi / a
    assert S.numpy()[0] < 1.0


def test_argument_errors_and_empty_calls():
    N = 400
    sim = _sim(N)
    lib, h = sim.lib, sim._h
    R = torch.zeros((2, N, 2), dtype=torch.float32, device="cuda")
    nv = torch.ones((3, 2), dtype=torch.int32, device="cuda")
    rho = torch.zeros((2, 3, 2), dtype=torch.float64, device="cuda")
    ok = (h, R.data_ptr(), 2, nv.data_ptr(), 3, rho.data_ptr())
    assert lib.ljmd_density_modes(*ok) == 0
    bad = [
        (None,) + ok[1:],
        ok[:1] + (None,) + ok[2:],
        ok[:3] + (None,) + ok[4:],
        ok[:5] + (None,),
        ok[:2] + (-1,) + ok[3:],
        ok[:4] + (-1,) + ok[5:],
        ok[:5] + (rho.data_ptr() + 8,),                                     # rho not 16-byte aligned
        ok[:3] + (nv.data_ptr() + 4,) + ok[4:],                             # nvec not 8-byte aligned
    ]
    for args in bad:
        assert lib.ljmd_density_modes(*args) == E_INVALID, args
        assert lib.ljmd_last_error()
    l0 = sim.launch_count()
    assert lib.ljmd_density_modes(h, None, 0, None, 3, None) == 0            # S == 0
    assert lib.ljmd_density_modes(h, None, 2, None, 0, None) == 0            # K == 0
    assert sim.launch_count() == l0
    assert sim.density_modes(np.zeros((0, N, 2), np.float32), np.ones((3, 2))).shape == (0, 3, 2)
    assert sim.density_modes(np.zeros((2, N, 2), np.float32), np.zeros((0, 2))).shape == (2, 0, 2)
    with pytest.raises(ValueError):
        sim.density_modes(np.zeros((2, N + 1, 2), np.float32), np.ones((3, 2)))


def test_all_pairs_and_cell_list_handles():
    N = 16384
    R, _, box = lattice_jitter(N, seed=2)
    nv = _half_plane(12)
    out = []
    for path in ("allpairs", "cells"):
        sim = _sim(N, path=path)
        rho, launches = modes(sim, R, nv)
        assert launches == LAUNCHES
        out.append(rho)
        sim.close()
    assert np.array_equal(out[0], out[1])
    _check_bound(out[0], c_density_modes(R, box, nv), N, nv, "N=16384")


def test_driver_sk_kmax(tmp_path, capsys):
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.parse_args(
        ["--N", "4096", "--rc", "2.5", "--ic", "lattice", "--eq_steps", "200", "--prod_steps", "300",
         "--sample_every", "100", "--sk_kmax", "8", "--sk_per_shell", "32", "--output", out])
    res = driver.main(args)
    k, S = res[3]
    text = capsys.readouterr().out
    assert "S(k) Analysis" in text and "S(k) first peak: k = " in text
    stem = str(tmp_path / "g_r_plot_sk")
    saved = np.load(stem + ".npy")
    assert np.array_equal(saved, np.stack([k, S]))
    assert np.allclose(np.loadtxt(stem + ".csv", delimiter=","), saved.T)
    assert np.isfinite(S).all() and k.max() <= 8.0
    i = int(np.argmax(S))
    assert 4.0 < k[i] < 8.0 and S[i] > 1.0                                 # the first peak, near 2 pi / a


def test_driver_sk_with_nan_positions(tmp_path, capsys):
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.parse_args(["--N", "400", "--eq_steps", "100", "--prod_steps", "200", "--sample_every", "100",
                              "--sk_kmax", "4", "--output", out])
    res = driver.main(args)
    assert len(res) == 4 and os.path.exists(str(tmp_path / "g_r_plot_sk.csv"))
    assert "S(k) Analysis" in capsys.readouterr().out
