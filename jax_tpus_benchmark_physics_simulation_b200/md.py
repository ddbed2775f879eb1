"""Host-side mirror of the closures the reference defines inside ``main()``.

Reference: molecular_dynamics_jax_single-host_workload.py (MD:<line>).  The names, argument
meaning and return structure of ``periodic_displacement`` (MD:46-48), ``total_energy_fn``
(MD:50-62), ``force_fn`` (MD:64), ``verlet_step`` (MD:66-75), ``equilibrate_fn`` (MD:77-83),
``production_fn`` (MD:85-106) and ``calculate_g_r`` (MD:108-131) are kept, so the reference's
driver lines MD:138-165 run unchanged against an :class:`LJSimulation`.

All arithmetic on the path is done by hand-written sm_100a kernels in ``libljmd.so`` reached
through the C ABI of include/ljmd.h.  torch is only the device-buffer allocator and stream
owner.  There is no CPU fallback: without the built library or without a B200 the constructor
raises.
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .ic import box_size as _box_size

_PATHS = {"auto": _lib.LJMD_PATH_AUTO, "allpairs": _lib.LJMD_PATH_ALLPAIRS,
          "cells": _lib.LJMD_PATH_CELLS}


class DeviceArray:
    """Minimal jax.Array look-alike over a CUDA torch tensor: ``.block_until_ready()``
    (MD:145,152,163), ``.shape`` (MD:174), ``__array__`` for numpy/matplotlib (MD:181)."""

    __slots__ = ("tensor", "_check")

    def __init__(self, tensor: torch.Tensor, check=None):
        self.tensor = tensor
        # status hook of the simulation that produced the array: the kernels run asynchronously, so
        # device-side failures (Verlet-list / slab overflow, barrier timeout) can only be raised
        # where the caller synchronises - exactly where the reference blocks (MD:145,152,163)
        self._check = check

    def block_until_ready(self) -> "DeviceArray":
        torch.cuda.current_stream(self.tensor.device).synchronize()
        if self._check is not None:
            self._check()
        return self

    @property
    def shape(self):
        return tuple(self.tensor.shape)

    @property
    def dtype(self):
        return self.tensor.dtype

    def __len__(self):
        return self.tensor.shape[0]

    def __getitem__(self, idx):
        return DeviceArray(self.tensor[idx], self._check)

    def __array__(self, dtype=None, copy=None):
        if self._check is not None:
            self._check()
        a = self.tensor.detach().cpu().numpy()
        return a.astype(dtype) if dtype is not None else a

    def numpy(self) -> np.ndarray:
        return self.__array__()

    def __float__(self):
        if self._check is not None:
            self._check()
        return float(self.tensor.item())

    def __repr__(self):
        return f"DeviceArray(shape={self.shape}, device={self.tensor.device})"


class LJSimulation:
    """2-D Lennard-Jones NVE simulation bound to one B200 (one handle of the C ABI).

    Parameters mirror the reference's CLI / closure captures (MD:16-31,196-213).  ``rc=None``
    reproduces the reference (no cutoff).  ``thermostat_kT`` / ``energy_every`` are additions
    that default to the reference's behaviour (pure NVE, no energy output).  ``virial=True``
    (also an addition, off by default) makes ``equilibrate_fn`` / ``production_fn`` record the pair
    virial W on the energy rows: ``last_virial`` (ne,) and ``last_pressure`` (ne,) next to
    ``last_energies`` (ne, 2); ``run(..., virial=...)`` overrides it per call.
    """

    def __init__(self, N: int, rho: float = 0.8, dt: float = 1e-3, eq_steps: int = 10000,
                 prod_steps: int = 10000, sample_every: int = 100, sigma: float = 1.0,
                 epsilon: float = 1.0, rc: Optional[float] = None, path: str = "auto",
                 skin: float = 0.3, device: Optional[int] = None,
                 box_size: Optional[float] = None, thermostat_kT: float = 0.0,
                 thermostat_every: int = 0, energy_every: int = 0,
                 dist: Optional[Tuple[bytes, int, int]] = None, virial: bool = False):
        if not torch.cuda.is_available():
            raise _lib.LjmdError("no CUDA device: the LJ-MD hot path has no CPU fallback")
        self.lib = _lib.load()
        self.N = int(N)
        self.rho = float(rho)
        self.dt = float(dt)
        self.equilibration_steps = int(eq_steps)
        self.production_steps = int(prod_steps)
        self.sample_every = int(sample_every)
        self.sigma, self.epsilon = float(sigma), float(epsilon)
        self.rc = None if rc is None or not math.isfinite(rc) or rc <= 0 else float(rc)
        self.box_size = np.float32(box_size) if box_size is not None else _box_size(N, rho)  # MD:30
        self.thermostat_kT = float(thermostat_kT)
        self.thermostat_every = int(thermostat_every)
        self.energy_every = int(energy_every)
        self.virial = bool(virial)
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.last_energies: Optional[DeviceArray] = None
        self.last_virial: Optional[DeviceArray] = None
        self.last_pressure: Optional[DeviceArray] = None
        p = _lib.LjmdParams()
        p.N = self.N
        p.box = float(self.box_size)
        p.sigma, p.epsilon = self.sigma, self.epsilon
        p.rc = self.rc if self.rc is not None else float("inf")
        p.dt = self.dt
        p.skin = float(skin)
        p.path = _PATHS[path]
        p.device = self.device_index
        self._stream = torch.cuda.current_stream(self.device)
        p.stream = ctypes.c_void_p(self._stream.cuda_stream)
        self._h = ctypes.c_void_p()
        self._dist_rank = (0, 1) if dist is None else (int(dist[1]), int(dist[2]))
        if dist is None:
            _lib.check(self.lib.ljmd_create(ctypes.byref(self._h), ctypes.byref(p)), "ljmd_create")
        else:
            uid, rank, nranks = dist
            buf = ctypes.create_string_buffer(bytes(uid), 128)
            _lib.check(self.lib.ljmd_create_dist(ctypes.byref(self._h), ctypes.byref(p), buf,
                                                 rank, nranks), "ljmd_create_dist")
        self._pe = torch.empty(1, dtype=torch.float32, device=self.device)

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.ljmd_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self) -> None:
        """Block until the handle's stream is idle and raise :class:`LjmdError` if the last call
        flagged a device-side failure (ljmd_check, include/ljmd.h)."""
        if getattr(self, "_h", None) is None or not self._h.value:
            return                      # handle already destroyed: nothing left to ask
        _lib.check(self.lib.ljmd_check(self._h), "ljmd_check")

    def _arr(self, t: torch.Tensor) -> DeviceArray:
        return DeviceArray(t, self.check)

    def _dev(self, x, shape: Optional[Sequence[int]] = None) -> torch.Tensor:
        """Accept DeviceArray / torch (cpu or cuda) / numpy; return contiguous fp32 CUDA tensor."""
        if isinstance(x, DeviceArray):
            t = x.tensor
        elif isinstance(x, torch.Tensor):
            t = x
        else:
            t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        if t.device != self.device:
            t = t.to(self.device, dtype=torch.float32, non_blocking=True)
        t = t.to(torch.float32).contiguous()
        if shape is not None and tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    def _check_stream(self):
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream != self._stream.cuda_stream:
            # the handle enqueues on the stream captured at construction: order the two streams
            self._stream.wait_stream(cur)

    def _after(self):
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream != self._stream.cuda_stream:
            cur.wait_stream(self._stream)

    # ------------------------------------------------------------------ MD:46-48
    def periodic_displacement(self, dr, box_size=None):
        """dr - box * round(dr / box), elementwise on any shape (MD:46-48).  Stand-alone helper
        (the kernels apply the bit-identical min-image internally); plain device arithmetic."""
        box = torch.as_tensor(self.box_size if box_size is None else np.float32(box_size),
                              dtype=torch.float32, device=self.device)
        t = self._dev(dr)
        return DeviceArray(t - box * torch.round(t / box))

    # ------------------------------------------------------------------ MD:50-62
    def total_energy_fn(self, R) -> DeviceArray:
        R = self._dev(R, (self.N, 2))
        out = torch.empty(1, dtype=torch.float32, device=self.device)
        self._check_stream()
        _lib.check(self.lib.ljmd_energy(self._h, R.data_ptr(), out.data_ptr()), "ljmd_energy")
        self._after()
        return self._arr(out[0])

    # ------------------------------------------------------------------ MD:64
    def force_fn(self, R) -> DeviceArray:
        R = self._dev(R, (self.N, 2))
        F = torch.empty_like(R)
        self._check_stream()
        _lib.check(self.lib.ljmd_forces(self._h, R.data_ptr(), F.data_ptr(), None), "ljmd_forces")
        self._after()
        return self._arr(F)

    def force_and_energy(self, R) -> Tuple[DeviceArray, DeviceArray]:
        R = self._dev(R, (self.N, 2))
        F = torch.empty_like(R)
        pe = torch.empty(1, dtype=torch.float32, device=self.device)
        self._check_stream()
        _lib.check(self.lib.ljmd_forces(self._h, R.data_ptr(), F.data_ptr(), pe.data_ptr()),
                   "ljmd_forces")
        self._after()
        return self._arr(F), self._arr(pe[0])

    # ------------------------------------------------------------------ virial / pressure (new)
    def virial_fn(self, R) -> DeviceArray:
        """Pair virial W(R) = sum_{i<j, r < rc} r_ij . f_ij as a device scalar (ljmd_virial): the
        same pair set, minimum image and fp32 arithmetic as the force; no tail correction."""
        R = self._dev(R, (self.N, 2))
        out = torch.empty(1, dtype=torch.float32, device=self.device)
        self._check_stream()
        _lib.check(self.lib.ljmd_virial(self._h, R.data_ptr(), out.data_ptr()), "ljmd_virial")
        self._after()
        return self._arr(out[0])

    def _pressure(self, ke: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
        """P = (KE + W/2) / box^2 of the 2-D fluid (unit mass, k_B = 1), in float64."""
        box = float(self.box_size)
        return (ke.to(torch.float64) + 0.5 * w.to(torch.float64)) / (box * box)

    def pressure_fn(self, state) -> DeviceArray:
        """Instantaneous pressure (KE(V) + W(R)/2) / box^2 of state = (R, V), a float64 device scalar;
        KE = 0.5 sum |v|^2 with the centre-of-mass motion included (as the reference's energies)."""
        R, V = state
        V = self._dev(V, (self.N, 2))
        w = self.virial_fn(R).tensor
        ke = 0.5 * torch.sum(V.to(torch.float64) ** 2)
        return self._arr(self._pressure(ke, w))

    # ------------------------------------------------------------------ MD:66-106
    def _run(self, state, nsteps: int, sample_every: int = 0, energy_every: int = 0,
             virial: bool = False):
        R, V = state
        R = self._dev(R, (self.N, 2))
        V = self._dev(V, (self.N, 2))
        R_out = torch.empty_like(R)
        V_out = torch.empty_like(V)
        S = nsteps // sample_every if sample_every > 0 else 0
        traj = torch.empty((S, self.N, 2), dtype=torch.float32, device=self.device)
        ne = -(-nsteps // energy_every) if energy_every > 0 else 0
        ke_pe = torch.zeros((ne, 2), dtype=torch.float32, device=self.device) if ne else None
        w = torch.zeros(ne, dtype=torch.float32, device=self.device) if (virial and ne) else None
        self._check_stream()
        if w is None:
            _lib.check(self.lib.ljmd_run(
                self._h, R.data_ptr(), V.data_ptr(), R_out.data_ptr(), V_out.data_ptr(), nsteps,
                sample_every if S > 0 else 0, traj.data_ptr() if S > 0 else None,
                energy_every if ne else 0, ke_pe.data_ptr() if ne else None,
                self.thermostat_kT, self.thermostat_every), "ljmd_run")
        else:
            _lib.check(self.lib.ljmd_run_virial(
                self._h, R.data_ptr(), V.data_ptr(), R_out.data_ptr(), V_out.data_ptr(), nsteps,
                sample_every if S > 0 else 0, traj.data_ptr() if S > 0 else None,
                energy_every, ke_pe.data_ptr(), self.thermostat_kT, self.thermostat_every,
                w.data_ptr()), "ljmd_run_virial")
        self._after()
        self.last_energies = self._arr(ke_pe) if ne else None
        self.last_virial = self._arr(w) if w is not None else None
        self.last_pressure = self._arr(self._pressure(ke_pe[:, 0], w)) if w is not None else None
        return (self._arr(R_out), self._arr(V_out)), self._arr(traj)

    def verlet_step(self, state):
        """One velocity-Verlet step (MD:66-75)."""
        return self._run(state, 1)[0]

    def run(self, state, nsteps: int, sample_every: int = 0, energy_every: int = 0,
            virial: Optional[bool] = None):
        """nsteps velocity-Verlet steps in one device dispatch; returns (state, traj).
        ``virial`` (default: the constructor's) also records W and P on the energy rows."""
        virial = self.virial if virial is None else bool(virial)
        return self._run(state, int(nsteps), int(sample_every), int(energy_every), virial)

    def block_range(self) -> Tuple[int, int]:
        """Index block [lo, hi) of this rank in the block-distributed convention of run_blocked."""
        rank, nranks = self._dist_rank
        return slab_range(self.N, rank, nranks)

    def run_blocked(self, state_block, nsteps: int, energy_every: int = 0):
        """nsteps steps with BLOCK-DISTRIBUTED state (multi-GPU handles; ljmd_run_blocked): this rank
        passes and receives only the particles of its index block ``block_range()`` as (N/P, 2)
        arrays, so a step's host<->device traffic is 1/P of the state.  Returns (R_block, V_block)."""
        lo, hi = self.block_range()
        R = self._dev(state_block[0], (hi - lo, 2))
        V = self._dev(state_block[1], (hi - lo, 2))
        R_out, V_out = torch.empty_like(R), torch.empty_like(V)
        ne = -(-nsteps // energy_every) if energy_every > 0 else 0
        ke_pe = torch.zeros((ne, 2), dtype=torch.float32, device=self.device) if ne else None
        self._check_stream()
        _lib.check(self.lib.ljmd_run_blocked(
            self._h, R.data_ptr(), V.data_ptr(), R_out.data_ptr(), V_out.data_ptr(), int(nsteps),
            energy_every if ne else 0, ke_pe.data_ptr() if ne else None), "ljmd_run_blocked")
        self._after()
        self.last_energies = self._arr(ke_pe) if ne else None
        return self._arr(R_out), self._arr(V_out)

    def equilibrate_fn(self, initial_state):
        """fori_loop(0, equilibration_steps, verlet_step) — one dispatch, NVE (MD:77-83)."""
        return self._run(initial_state, self.equilibration_steps, 0, self.energy_every, self.virial)[0]

    def production_fn(self, initial_state):
        """production_steps steps, snapshot after step i when i % sample_every == 0 into row
        i // sample_every of R_history (S, N, 2), S = production_steps // sample_every
        (MD:85-106)."""
        return self._run(initial_state, self.production_steps, self.sample_every,
                         self.energy_every, self.virial)

    # ------------------------------------------------------------------ MD:108-131
    def calculate_g_r(self, R_history, N_local=None, box_size_local=None, nbins=None, r_max=None):
        """Radial distribution function (MD:108-129).  The O(S N^2) pair-distance histogram runs
        on the GPU (ljmd_gr_hist); the nbins-long normalisation is host arithmetic in fp32 as in
        the reference."""
        N = self.N if N_local is None else int(N_local)
        if N != self.N:
            raise ValueError("calculate_g_r: N must match the simulation")
        box = np.float32(self.box_size if box_size_local is None else box_size_local)
        r_max = np.float32(box / np.float32(2.0)) if r_max is None else np.float32(r_max)
        nbins = int(r_max / 0.05) if nbins is None else int(nbins)               # MD:158-159
        Rh = self._dev(R_history)
        if Rh.dim() == 2:
            Rh = Rh[None]
        S = Rh.shape[0]
        r_bins = np.linspace(0, r_max, nbins + 1, dtype=np.float32)              # MD:110
        centers = (r_bins[:-1] + r_bins[1:]) / np.float32(2.0)                    # MD:111
        shell = np.float32(np.pi) * (r_bins[1:] ** 2 - r_bins[:-1] ** 2)          # MD:112
        rho_pairs = np.float32(N * (N - 1) / 2.0) / (box ** 2)                    # MD:113
        ideal = rho_pairs * shell                                                 # MD:115
        edges = torch.from_numpy(r_bins).to(self.device)
        counts = torch.empty((S, nbins), dtype=torch.int64, device=self.device)
        self._check_stream()
        _lib.check(self.lib.ljmd_gr_hist(self._h, Rh.data_ptr(), S, nbins, edges.data_ptr(),
                                         counts.data_ptr()), "ljmd_gr_hist")
        self._after()
        self.last_gr_counts = DeviceArray(counts)
        avg = counts.to(torch.float32).mean(dim=0) if S else torch.zeros(nbins, device=self.device)
        g = avg / torch.from_numpy(ideal.astype(np.float32)).to(self.device)      # MD:126-128
        return DeviceArray(torch.from_numpy(centers).to(self.device)), DeviceArray(g)

    # ------------------------------------------------------------------ cell-list introspection
    def cell_geometry(self):
        """(nrows, nbins_x, kbins, inv_row_height, inv_bin_width) of the strip-cell grid."""
        nr, nb, kb = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        ih, iw = ctypes.c_float(), ctypes.c_float()
        _lib.check(self.lib.ljmd_cell_geometry(self._h, ctypes.byref(nr), ctypes.byref(nb),
                                               ctypes.byref(kb), ctypes.byref(ih), ctypes.byref(iw)),
                   "ljmd_cell_geometry")
        return nr.value, nb.value, kb.value, np.float32(ih.value), np.float32(iw.value)

    def cell_assign(self, R):
        R = self._dev(R, (self.N, 2))
        nr, nb, _, _, _ = self.cell_geometry()
        cid = torch.empty(self.N, dtype=torch.int32, device=self.device)
        cnt = torch.empty(nr * nb, dtype=torch.int32, device=self.device)
        self._check_stream()
        _lib.check(self.lib.ljmd_cell_assign(self._h, R.data_ptr(), cid.data_ptr(), cnt.data_ptr()),
                   "ljmd_cell_assign")
        self._after()
        return cid, cnt

    def neighbor_count(self, R, radius: float):
        R = self._dev(R, (self.N, 2))
        out = torch.empty(self.N, dtype=torch.int32, device=self.device)
        self._check_stream()
        _lib.check(self.lib.ljmd_neighbor_count(self._h, R.data_ptr(), float(radius),
                                                out.data_ptr()), "ljmd_neighbor_count")
        self._after()
        return out

    def last_rebuilds(self) -> int:
        v = ctypes.c_int64()
        _lib.check(self.lib.ljmd_last_rebuilds(self._h, ctypes.byref(v)), "ljmd_last_rebuilds")
        return v.value

    # ------------------------------------------------------------------ measurement
    def last_run_ms(self) -> float:
        v = ctypes.c_float()
        _lib.check(self.lib.ljmd_last_run_ms(self._h, ctypes.byref(v)), "ljmd_last_run_ms")
        return v.value

    def allpairs_mode(self) -> int:
        """1 / 2: every ordered pair evaluated; 3: Newton's-third-law tiles (each unordered pair
        once); 4: ordered pairs in one thread-block cluster (small N); 0: cell-list path."""
        v = ctypes.c_int32()
        _lib.check(self.lib.ljmd_allpairs_mode(self._h, ctypes.byref(v)), "ljmd_allpairs_mode")
        return v.value

    def launch_count(self) -> int:
        v = ctypes.c_int64()
        _lib.check(self.lib.ljmd_launch_count(self._h, ctypes.byref(v)), "ljmd_launch_count")
        return v.value


def slab_range(N: int, rank: int, nranks: int) -> Tuple[int, int]:
    """Atom decomposition of the all-pairs path: rank p owns i-rows [p*N/P, (p+1)*N/P)
    (SURVEY.md §8e).  N must be divisible by the rank count."""
    if nranks < 1 or not (0 <= rank < nranks):
        raise ValueError(f"bad rank {rank} / nranks {nranks}")
    if N % nranks != 0:
        raise ValueError(f"N={N} is not divisible by nranks={nranks}")
    n = N // nranks
    return rank * n, (rank + 1) * n


def row_slab_range(nrows: int, rank: int, nranks: int) -> Tuple[int, int]:
    """Slab decomposition of the cell-list path: rank p owns the contiguous block of strip-cell
    rows [g0, g0 + nloc), blocks as even as possible (the first nrows % P ranks own one more), and
    holds one halo row on each side (csrc/cells.cu::cells_create).  Needs 2 rows per rank."""
    if nranks < 1 or not (0 <= rank < nranks):
        raise ValueError(f"bad rank {rank} / nranks {nranks}")
    if nranks > 1 and nrows < 2 * nranks:
        raise ValueError(f"{nrows} rows cannot be split over {nranks} ranks (need 2 rows per rank)")
    base, extra = divmod(nrows, nranks)
    g0 = rank * base + min(rank, extra)
    return g0, base + (1 if rank < extra else 0)


def broadcast_unique_id(rank: int, get_uid=None) -> bytes:
    """Rank 0 creates the 128-byte NCCL unique id (ljmd_get_unique_id) and broadcasts it over the
    already-initialised torch.distributed group (any backend: gloo on CPU, nccl on GPUs)."""
    import torch.distributed as dist
    if get_uid is None:
        def get_uid():
            buf = ctypes.create_string_buffer(128)
            _lib.check(_lib.load().ljmd_get_unique_id(buf), "ljmd_get_unique_id")
            return buf.raw
    box = [get_uid() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    uid = bytes(box[0])
    if len(uid) != 128:
        raise _lib.LjmdError(f"NCCL unique id must be 128 bytes, got {len(uid)}")
    return uid


def make_dist_arg(rank: int, nranks: int):
    """(uid, rank, nranks) for ``LJSimulation(dist=...)``: one handle per rank / GPU."""
    return broadcast_unique_id(rank), rank, nranks


def fp32_peak_probe(device: int = 0, packed: bool = False) -> float:
    """Measured FP32 CUDA-core ceiling in TFLOP/s (FFMA or FFMA2 dependent chains)."""
    v = ctypes.c_float()
    _lib.check(_lib.load().ljmd_fp32_peak_probe(device, int(packed), ctypes.byref(v)),
               "ljmd_fp32_peak_probe")
    return v.value
