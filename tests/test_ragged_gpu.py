"""The force / step kernels at particle counts that do not fill their tiles, and under every launch-shape setting.

Inputs are ``ragged_lattice`` states (tests/ragged_reference.py).  Forces are checked per particle against the
float64 reference: |F_i - F_ref,i|_inf <= 1e-5 S_i with S_i = sum_j |F_ij|, so a dropped or doubled in-cutoff pair
fails for every particle (tests/test_ragged_cpu.py checks that power).  Every case asserts the kernel it targets
(``allpairs_mode()``, ``cell_geometry()``) and that its N leaves the padding it is meant to reach.

The launch-shape settings are environment variables.  LJMD_AP_CHUNK, LJMD_CELLS_CHUNK and LJMD_CELLS_STATIC are read
per call, the others when the handle is created.  Where DESIGN.md promises results independent of the schedule
(§4.1: the tile mode's patch-indexed partials; §4.2: the cell list's unit-indexed energies and position-determined
sorted order), the settings must not change a bit."""
import functools

import numpy as np
import pytest
import torch

import bond_reference
from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation
from ragged_reference import check_forces, check_rows, forces_f64, ragged_lattice
from sk_reference import bound, c_density_modes
from virial_reference import c_virial

pytestmark = pytest.mark.gpu

TOL = 1e-5                   # per particle, in units of S_i
ENERGY_TOL = 1e-6
VIR_TOL = 2e-6               # as tests/test_virial_gpu.py
T3_BLK, J_UNIT, CL_UNIT = 64, 8, 32
KNOBS = ("LJMD_AP_IPT", "LJMD_AP_Q", "LJMD_AP_GRID", "LJMD_AP_CTAS_PER_SM", "LJMD_AP_CLUSTER_SIZE",
         "LJMD_AP_CLUSTER_NMAX", "LJMD_AP_CHUNK", "LJMD_CELLS_CHUNK", "LJMD_CELLS_STATIC", "LJMD_CELLS_CTAS_PER_SM")


@functools.lru_cache(maxsize=None)
def _state(N):
    return ragged_lattice(N)


@functools.lru_cache(maxsize=None)
def _ref(N, rc, rows=None):
    R, _, box = _state(N)
    return forces_f64(R, box, rc=rc, rows=rows)


def _env(monkeypatch, **knobs):
    """Exactly the given launch-shape settings (None: unset); every other one unset."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in knobs.items():
        if v is not None:
            monkeypatch.setenv(k, str(v))


def _sim(N, path="allpairs", **kw):
    kw.setdefault("rc", 2.5)
    return LJSimulation(N, path=path, device=0, **kw)


def _check(F, N, rc, what, rows=None):
    Fr, S, _ = _ref(N, rc, rows)
    ok, worst, i = check_forces(F, Fr, S, TOL)
    print(f"[ragged] {what}: max |dF_i| / S_i = {worst:.2e}")
    assert ok, f"{what}: |dF_i| / S_i = {worst:.3e} at particle {i + (rows[0] if rows else 0)} (S_i = {S[i]:.3g})"


def _pdist(a, b, box):
    d = np.abs(np.asarray(a) - np.asarray(b))
    return np.minimum(d, float(box) - d)


def _assert_padded(mode, N):
    """N leaves the padding of the kernel: a short cluster CTA (C in {8, 16}), a padded j unit of 8 and a partly
    filled i-block of 128 ipt, or a partly filled 64-particle block of the tile mode."""
    if mode == 4:
        assert N % 8 != 0
    elif mode in (1, 2):
        assert N % J_UNIT != 0 and N % (128 * mode) != 0
    else:
        assert N % T3_BLK != 0


def _run(sim, R, V, nsteps, sample_every=0, energy_every=0):
    (R1, V1), traj = sim.run((R, V), nsteps, sample_every=sample_every, energy_every=energy_every)
    e = sim.last_energies.numpy().copy() if energy_every else None
    return R1.numpy(), V1.numpy(), traj.numpy(), e


# ---------------------------------------------------------------------------------------------- a. dispatch
@pytest.mark.parametrize("N,mode", [(640, 4), (641, 1), (2047, 1), (2048, 3)])
def test_dispatch_boundaries(monkeypatch, N, mode):
    _env(monkeypatch)
    assert _sim(N).allpairs_mode() == mode


# ---------------------------------------------------------------------------------------------- b. per mode
MODE_CASES = ([(4, N) for N in (2, 3, 17, 31, 33, 401, 639)] + [(1, N) for N in (641, 1021, 2047)]
              + [(2, 641), (2, 2049)] + [(3, N) for N in (2049, 4097, 5003)])


@pytest.mark.parametrize("rc", [None, 2.5])
@pytest.mark.parametrize("mode,N", MODE_CASES)
def test_forces_energy_virial(monkeypatch, oracle, mode, N, rc):
    _env(monkeypatch, LJMD_AP_IPT=2 if mode == 2 else None)
    R, _, box = _state(N)
    sim = _sim(N, rc=rc)
    assert sim.allpairs_mode() == mode
    _assert_padded(mode, N)
    F = sim.force_fn(R).numpy()
    _check(F, N, rc, f"mode {mode} N={N} rc={rc}")
    F2, pe = sim.force_and_energy(R)
    assert np.array_equal(F2.numpy(), F)
    pe_ref = _ref(N, rc)[2]
    assert abs(float(pe) - pe_ref) <= ENERGY_TOL * abs(pe_ref), (float(pe), pe_ref)
    w_ref, wabs = c_virial(R, box, rc=rc)
    w = float(sim.virial_fn(R))
    assert abs(w - w_ref) <= VIR_TOL * wabs, (w, w_ref, wabs)


def _host_q(N, slots):
    """The tile mode's q rule of ap_create (csrc/allpairs.cu), single GPU."""
    blocks = -(-N // T3_BLK)
    q = 8
    while q > 1:
        npr = -(-blocks // (2 * q))
        if npr * (npr + 1) // 2 >= 4 * slots:
            break
        q //= 2
    return q


@pytest.mark.parametrize("N,q", [(33331, 2), (70001, 8)])
def test_tile_mode_large_rows(monkeypatch, oracle, N, q):
    """The host's q rule picks q = 2 and q = 8 at these N (148 SMs, 4 CTAs per SM); 4 row blocks of 256, the last
    rows among them, against the float64 reference, and the PE against the cell-grid oracle."""
    _env(monkeypatch)
    R, _, box = _state(N)
    sim = _sim(N)
    assert sim.allpairs_mode() == 3
    _assert_padded(3, N)
    assert _host_q(N, 4 * 148) == q
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    print(f"[ragged] N={N}: host rule q = {_host_q(N, 4 * sms)} at 4 CTAs on {sms} SMs")
    F, pe = sim.force_and_energy(R)
    F = F.numpy()
    for lo, hi in check_rows(N):
        _check(F[lo:hi], N, 2.5, f"mode 3 N={N} rows [{lo}, {hi})", rows=(lo, hi))
    _, pe_c = oracle.c_forces_cells(R, box, 2.5)
    assert abs(float(pe) - pe_c) <= ENERGY_TOL * abs(pe_c)


# ---------------------------------------------------------------------------------------------- c. q sweep
def _tile_outputs(N, R, V):
    sim = _sim(N, dt=0.005)
    assert sim.allpairs_mode() == 3
    F, pe = sim.force_and_energy(R)
    out = {"F": F.numpy(), "pe": np.float32(float(pe))}
    out["R"], out["V"], out["traj"], e = _run(sim, R, V, 30, sample_every=10, energy_every=5)
    out["KE"], out["PE"] = e[:, 0], e[:, 1]
    return out


@pytest.mark.parametrize("q", [1, 2, 4, 8])
@pytest.mark.parametrize("N", [2049, 5003])
def test_tile_mode_q_and_schedule(monkeypatch, N, q):
    """Every q against the reference.  For one q, the grid size and CTAs per SM only change which CTA draws which
    patch: forces, PE and a 30-step run (positions, velocities, samples, PE rows) are bit-identical (DESIGN §4.1).
    The KE rows are per-CTA sums over the CTA's particle range, so they move with the grid size in the last bits
    only.  Across q the summation order of the forces changes: only the tolerance applies."""
    R, V, _ = _state(N)
    blocks = -(-N // T3_BLK)
    npr = -(-blocks // (2 * q))
    if q == 8 and N == 2049:
        assert npr * 2 * q - blocks == 15           # 15 blocks of the last patch row hold only padding
    _env(monkeypatch, LJMD_AP_Q=q)
    base = _tile_outputs(N, R, V)
    _check(base["F"], N, 2.5, f"mode 3 N={N} q={q}")
    diffs = []
    for grid in (1, 3, None):
        for per_sm in (1, None):
            if grid is None and per_sm is None:
                continue
            _env(monkeypatch, LJMD_AP_Q=q, LJMD_AP_GRID=grid, LJMD_AP_CTAS_PER_SM=per_sm)
            got = _tile_outputs(N, R, V)
            diffs += [f"GRID={grid} CTAS_PER_SM={per_sm}: {k}" for k in base
                      if k != "KE" and not np.array_equal(got[k], base[k])]
            assert np.abs(got["KE"] - base["KE"]).max() <= 1e-6 * np.abs(base["KE"]).max()
    assert not diffs, diffs


# ---------------------------------------------------------------------------------------------- d. stream-K
@pytest.mark.parametrize("rc", [None, 2.5])
@pytest.mark.parametrize("grid", [1, 7, None])
@pytest.mark.parametrize("ipt", [1, 2])
@pytest.mark.parametrize("N", [641, 2047])
def test_ordered_modes_stream_k_split(monkeypatch, N, ipt, grid, rc):
    _env(monkeypatch, LJMD_AP_IPT=ipt, LJMD_AP_GRID=grid)
    R, _, _ = _state(N)
    sim = _sim(N, rc=rc)
    assert sim.allpairs_mode() == ipt
    _assert_padded(ipt, N)
    _check(sim.force_fn(R).numpy(), N, rc, f"mode {ipt} N={N} G={grid} rc={rc}")


# ---------------------------------------------------------------------------------------------- e. cluster sizes
@pytest.mark.parametrize("C", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("N", [17, 401, 639])
def test_cluster_sizes(monkeypatch, oracle, N, C):
    """C CTAs, S lanes per pair and the j slice length all follow the cluster size; forces against the reference
    and a 100-step trajectory against the C oracle (tolerances of test_short_trajectory_vs_oracle)."""
    _env(monkeypatch, LJMD_AP_CLUSTER_SIZE=C)
    R, V, box = _state(N)
    dt, rc = 0.005, 2.5
    sim = _sim(N, rc=rc, dt=dt)
    assert sim.allpairs_mode() == 4
    _check(sim.force_fn(R).numpy(), N, rc, f"mode 4 N={N} C<={C}")
    R1, _, traj, _ = _run(sim, R, V, 100, sample_every=50)
    Rc, _, traj_c, _ = oracle.c_run(R, V, box, dt, 100, sample_every=50, rc=rc)
    assert _pdist(R1, Rc, box).max() <= 1e-4
    assert _pdist(traj[0], traj_c[0], box).max() <= 1e-6


# ---------------------------------------------------------------------------------------------- f. steps
STEP_CASES = [(401, 4, None), (1021, 1, None), (2049, 2, 2), (4097, 3, None)]


@pytest.mark.parametrize("N,mode,ipt", STEP_CASES)
def test_step_chunking_and_thermostat(monkeypatch, oracle, N, mode, ipt):
    _env(monkeypatch, LJMD_AP_IPT=ipt)
    R, V, box = _state(N)
    dt, rc = 0.005, 2.5
    sim = _sim(N, rc=rc, dt=dt)
    assert sim.allpairs_mode() == mode
    _assert_padded(mode, N)
    # one step against the C oracle (as test_one_step_vs_oracle)
    R1, V1, _, e = _run(sim, R, V, 1, energy_every=1)
    Rc, Vc, _, e_c = oracle.c_run(R, V, box, dt, 1, rc=rc, energy_every=1)
    assert np.abs(R1 - Rc).max() <= 2e-6
    assert np.abs(V1 - Vc).max() <= 1e-5 * np.abs(Vc).max()
    assert abs(float(e[0, 0]) + float(e[0, 1]) - e_c[0].sum()) <= ENERGY_TOL * abs(e_c[0].sum())
    # a call cut into launches of 7 steps is one launch, bit for bit
    a = _run(sim, R, V, 45, sample_every=10, energy_every=5)
    monkeypatch.setenv("LJMD_AP_CHUNK", "7")
    b = _run(sim, R, V, 45, sample_every=10, energy_every=5)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    # the rescale thermostat reaches every particle, the padded tail included
    monkeypatch.delenv("LJMD_AP_CHUNK")
    th = _sim(N, rc=rc, dt=dt, thermostat_kT=0.7, thermostat_every=10)
    assert th.allpairs_mode() == mode
    _, Vt, _, _ = _run(th, R, V, 30)
    assert abs(0.5 * float((Vt.astype(np.float64) ** 2).sum()) / N - 0.7) < 1e-4


# ---------------------------------------------------------------------------------------------- g. cell list
CELL_CASES = [58, 75, 99, 401, 4097, 16385]
CELL_LAST_UNIT = {58: 26, 75: 11, 99: 3, 401: 17, 4097: 1, 16385: 1}


@pytest.mark.parametrize("N", CELL_CASES)
def test_cells_ragged(monkeypatch, oracle, N):
    _env(monkeypatch)
    R, V, box = _state(N)
    dt, rc, skin = 0.005, 2.5, 0.3
    sim = _sim(N, path="cells", rc=rc, dt=dt, skin=skin)
    assert sim.allpairs_mode() == 0
    nrows, nbx, _, inv_hy, inv_wx = sim.cell_geometry()
    assert (nrows == 3) == (N < 100)
    assert N % CL_UNIT == CELL_LAST_UNIT[N]
    cid, cnt = sim.cell_assign(R)
    cid_c, cnt_c = oracle.c_cell_assign(R, nrows, nbx, inv_hy, inv_wx)
    assert np.array_equal(cid.cpu().numpy(), cid_c) and np.array_equal(cnt.cpu().numpy(), cnt_c)
    for radius in (rc, rc + skin):
        assert np.array_equal(sim.neighbor_count(R, radius).cpu().numpy(), oracle.c_neighbor_count(R, box, radius))
    _check(sim.force_fn(R).numpy(), N, rc, f"cells N={N} rows={nrows}")

    base = _run(sim, R, V, 200, sample_every=50, energy_every=10)
    assert sim.last_rebuilds() >= 2
    if N <= 401:
        Rc, _, traj_c, _ = oracle.c_run(R, V, box, dt, 200, sample_every=50, rc=rc)
        assert _pdist(base[0], Rc, box).max() <= 1e-4
        assert _pdist(base[2][0], traj_c[0], box).max() <= 1e-6
    else:
        # as test_cells_matches_allpairs_dynamics: 60 steps, across rebuilds.  By 200 steps the rounding
        # differences of the two summation orders have grown chaotically to a few 1e-4 (measured at N = 16385).
        R2, _, _, e = _run(sim, R, V, 60, energy_every=20)
        assert sim.last_rebuilds() >= 2
        Ra, _, _, ea = _run(_sim(N, rc=rc, dt=dt), R, V, 60, energy_every=20)
        assert _pdist(R2, Ra, box).max() <= 1e-4
        assert np.abs(e.astype(np.float64).sum(1) - ea.sum(1)).max() <= 2e-6 * np.abs(ea.sum(1)).max()

    # the schedule: launches of 1 / 7 steps, all-static or all-dynamic units, one CTA per SM (DESIGN §4.2)
    diffs = []
    settings = [dict(LJMD_CELLS_CHUNK=c, LJMD_CELLS_STATIC=s) for c in (1, 7) for s in (0, 1)]
    settings.append(dict(LJMD_CELLS_CTAS_PER_SM=1, LJMD_CELLS_CHUNK=7))
    for kn in settings:
        _env(monkeypatch, **kn)
        s2 = _sim(N, path="cells", rc=rc, dt=dt, skin=skin) if "LJMD_CELLS_CTAS_PER_SM" in kn else sim
        got = _run(s2, R, V, 200, sample_every=50, energy_every=10)
        diffs += [f"{kn}: {name}" for name, x, y in zip(("R", "V", "traj", "energies"), got, base)
                  if not np.array_equal(x, y)]
    assert not diffs, diffs


# ---------------------------------------------------------------------------------------------- h. analysis
def _snapshots(N):
    R, V, box = _state(N)
    sim = _sim(N, path="auto", dt=0.005)
    _, _, traj, _ = _run(sim, R, V, 30, sample_every=10)
    return sim, traj, box


@pytest.mark.parametrize("N", [401, 2049])
def test_gr_and_bond_order_ragged(oracle, N):
    sim, th, box = _snapshots(N)
    r_half = np.float32(box / np.float32(2.0))
    for r_max, nbins, launches in ((r_half, int(r_half / 0.05), 1), (np.float32(5.0), 100, 4)):
        l0 = sim.launch_count()
        sim.calculate_g_r(th, N, box, nbins, r_max)
        assert sim.launch_count() - l0 == launches           # all-pairs histogram / cell grid
        counts = sim.last_gr_counts.numpy()
        for s in range(th.shape[0]):
            assert np.array_equal(counts[s], oracle.c_gr_hist(th[s], box, nbins, r_max)), (r_max, s)
    psi, n = sim.bond_order(th, 6, 1.5)
    psi, n = psi.numpy(), n.numpy()
    for s in range(th.shape[0]):
        p_ref, n_ref = bond_reference.bond_order(th[s], box, 6, 1.5)
        assert np.array_equal(n[s], n_ref)
        assert np.array_equal(psi[s].view(np.int64), p_ref.view(np.int64))


@pytest.mark.parametrize("N", [1025, 2049])
def test_density_modes_ragged(N):
    """N = 1025 and 2049 put one particle past the 1024-particle tile and segment boundaries of csrc/sk.cu."""
    sim, th, box = _snapshots(N)
    nv = np.array([(x, y) for y in range(0, 21) for x in range(-20, 21)
                   if (y > 0 or x > 0) and x * x + y * y <= 400], dtype=np.int32)
    rho = sim.density_modes(th, nv).numpy()
    err = np.abs(rho - c_density_modes(th, box, nv)).max(axis=-1)
    assert np.isfinite(rho).all() and (err / bound(N, nv)).max() <= 1.0
