"""GPU tests of the pair virial and the pressure (ljmd_virial / ljmd_run_virial) against the CPU reference
(tests/virial_reference.py).

Bound: |W_gpu - W_ref| <= 2e-6 * sum_{i<j} |w_ij| (fp32 pair terms with MUFU.RCP, fp32 partial sums).
The virial kernels are separate instantiations: with the virial on, positions, velocities, trajectory
and energies must stay bit for bit those of the same call without it.
"""
import ctypes

import numpy as np
import pytest
import torch

from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter

import virial_reference as vref   # tests/virial_reference.py

pytestmark = pytest.mark.gpu

VIR_TOL = 2e-6


def _sim(N, **kw):
    from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation
    return LJSimulation(N, **kw)


def _ref(oracle, R, box, rc, cells=False):
    return vref.c_virial_cells(R, box, rc) if cells else vref.c_virial(R, box, rc=rc)


@pytest.mark.parametrize("N,rc,path,mode", [
    (400, None, "allpairs", 4),          # the reference's default run: one thread-block cluster
    (400, 2.5, "allpairs", 4),
    (1024, 2.5, "allpairs", 1),          # ordered pairs
    (4096, 2.5, "allpairs", 3),          # Newton's-third-law tiles
    (16384, 2.5, "cells", 0),
    (4194304, 2.5, "cells", 0),
])
def test_virial_fn_vs_oracle(oracle, N, rc, path, mode):
    R, _, box = lattice_jitter(N, seed=0)
    sim = _sim(N, rc=rc, path=path)
    assert sim.allpairs_mode() == mode
    w = float(sim.virial_fn(R))
    w_ref, wabs = _ref(oracle, R, box, rc, cells=N > 65536)
    assert abs(w - w_ref) <= VIR_TOL * wabs, (w, w_ref, wabs)
    # the one-shot evaluation leaves the energy and force entry points as they were
    F, pe = sim.force_and_energy(R)
    assert float(sim.total_energy_fn(R)) == float(pe)


def test_forced_allpairs_modes_agree(oracle, monkeypatch):
    N = 4096
    R, _, box = lattice_jitter(N, seed=1)
    w_ref, wabs = vref.c_virial(R, box, rc=2.5)
    ws = []
    for ipt in (1, 2, 3):
        monkeypatch.setenv("LJMD_AP_IPT", str(ipt))
        sim = _sim(N, rc=2.5, path="allpairs")
        assert sim.allpairs_mode() == ipt
        ws.append(float(sim.virial_fn(R)))
        sim.close()
    monkeypatch.delenv("LJMD_AP_IPT")
    for w in ws:
        assert abs(w - w_ref) <= VIR_TOL * wabs
    assert max(ws) - min(ws) <= 2 * VIR_TOL * wabs


def _run_both(sim, R, V, nsteps, sample_every):
    (Ra, Va), ta = sim.run((R, V), nsteps, sample_every=sample_every, energy_every=1, virial=False)
    ea = sim.last_energies.numpy().copy()
    assert sim.last_virial is None and sim.last_pressure is None
    (Rb, Vb), tb = sim.run((R, V), nsteps, sample_every=sample_every, energy_every=1, virial=True)
    eb = sim.last_energies.numpy().copy()
    assert sim.last_virial.shape == (nsteps,) and sim.last_pressure.shape == (nsteps,)
    assert np.array_equal(Ra.numpy(), Rb.numpy()) and np.array_equal(Va.numpy(), Vb.numpy())
    assert np.array_equal(ta.numpy(), tb.numpy())
    assert np.array_equal(ea, eb)
    assert np.isfinite(sim.last_virial.numpy()).all()


@pytest.mark.parametrize("N,path,mode", [(400, "allpairs", 4), (1024, "allpairs", 1), (4096, "allpairs", 3),
                                         (16384, "cells", 0)])
def test_virial_changes_nothing_else(N, path, mode):
    R, V, box = lattice_jitter(N, seed=2)
    sim = _sim(N, rc=2.5, dt=0.005, path=path)
    assert sim.allpairs_mode() == mode
    _run_both(sim, R, V, 300, 25)
    if path == "cells":
        assert sim.last_rebuilds() > 0          # the calls crossed list rebuilds
    thermo = _sim(N, rc=2.5, dt=0.005, path=path, thermostat_kT=0.9, thermostat_every=7)
    _run_both(thermo, R, V, 50, 10)


@pytest.mark.parametrize("N,path", [(4096, "allpairs"), (16384, "cells")])
def test_trace_rows_vs_oracle(oracle, N, path):
    R, V, box = lattice_jitter(N, seed=3)
    sim = _sim(N, rc=2.5, dt=0.005, path=path)
    (_, _), traj = sim.run((R, V), 200, sample_every=20, energy_every=20, virial=True)
    w = sim.last_virial.numpy()
    t = traj.numpy()
    assert w.shape == (10,) and t.shape == (10, N, 2)
    if path == "cells":
        assert sim.last_rebuilds() > 0
    for s in range(t.shape[0]):
        w_ref, wabs = _ref(oracle, t[s], box, 2.5, cells=path == "cells")
        assert abs(float(w[s]) - w_ref) <= VIR_TOL * wabs, (s, float(w[s]), w_ref)


def test_pressure_formula(oracle):
    N = 1024
    R, V, box = lattice_jitter(N, seed=4)
    sim = _sim(N, rc=2.5, dt=0.005, path="allpairs")
    p = float(sim.pressure_fn((R, V)))
    w = float(sim.virial_fn(R))
    ke = oracle.kinetic_energy(torch.from_numpy(V))
    assert p == pytest.approx((ke + 0.5 * w) / float(box) ** 2, rel=1e-12)
    sim.run((R, V), 40, energy_every=4, virial=True)
    e = sim.last_energies.numpy().astype(np.float64)
    w_tr = sim.last_virial.numpy().astype(np.float64)
    P = sim.last_pressure.numpy()
    assert np.allclose(P, (e[:, 0] + 0.5 * w_tr) / float(box) ** 2, rtol=1e-12, atol=0)
    # the constructor's switch applies to equilibrate_fn / production_fn
    prod = _sim(N, rc=2.5, dt=0.005, path="allpairs", prod_steps=30, sample_every=10, energy_every=10,
                virial=True)
    prod.production_fn((R, V))
    assert prod.last_pressure.shape == (3,)


def test_argument_errors_leave_handle_usable():
    from jax_tpus_benchmark_physics_simulation_b200 import _lib
    N = 400
    R, V, box = lattice_jitter(N, seed=5)
    sim = _sim(N, rc=2.5, path="allpairs")
    w0 = float(sim.virial_fn(R))
    Rd = torch.from_numpy(R).cuda()
    Vd = torch.from_numpy(V).cuda()
    Ro, Vo = torch.empty_like(Rd), torch.empty_like(Vd)
    wbuf = torch.zeros(10, dtype=torch.float32, device="cuda")
    ke_pe = torch.zeros((10, 2), dtype=torch.float32, device="cuda")
    lib = sim.lib
    for ee, kp in ((1, None), (0, ke_pe.data_ptr())):       # w without ke_pe / without energy_every
        code = lib.ljmd_run_virial(sim._h, Rd.data_ptr(), Vd.data_ptr(), Ro.data_ptr(), Vo.data_ptr(), 10, 0,
                                   None, ee, kp, ctypes.c_float(0.0), 0, wbuf.data_ptr())
        assert code == -1
        with pytest.raises(_lib.LjmdError):
            _lib.check(code, "ljmd_run_virial")
    assert lib.ljmd_virial(sim._h, Rd.data_ptr(), None) == -1
    sim.check()
    assert float(sim.virial_fn(R)) == w0
    (R1, V1), _ = sim.run((R, V), 10, energy_every=1, virial=True)
    assert np.isfinite(sim.last_virial.numpy()).all()


def test_driver_pressure_flag(capsys, tmp_path):
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    args = driver.parse_args(["--N", "400", "--ic", "lattice", "--eq_steps", "200", "--prod_steps", "200",
                              "--sample_every", "50", "--energy_every", "10", "--pressure",
                              "--output", str(tmp_path / "g.png")])
    driver.main(args)
    out = capsys.readouterr().out
    line = [l for l in out.splitlines() if "Pressure (production)" in l]
    assert len(line) == 1
    mean = float(line[0].split("mean")[1].split()[0])
    assert np.isfinite(mean)
    with pytest.raises(SystemExit):
        driver.parse_args(["--pressure"])
