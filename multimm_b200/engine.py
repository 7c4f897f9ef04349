"""Engine — Python face of one mmm_handle.

This is the object that stands where ``openmm.System`` + ``Simulation`` + ``Context`` stand in the
reference (model.py:763-764, 876-889).  It only marshals numpy arrays across the C-ABI; all
numerics run in libmultimm_b200.so on the GPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import Error, MdReport, MinReport, NUM_TERMS, TERM, TERM_NAMES  # noqa: F401  (re-exported)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _arr(a, dt):
    return None if a is None else np.ascontiguousarray(a, dtype=dt)


class Engine:
    """One system on one CUDA device.  Not thread-safe; independent of other engines."""

    def __init__(self, n_beads: int, device: int = 0):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        self.n = int(n_beads)
        self.device = int(device)
        rc = self._lib.mmm_create(self.device, self.n, C.byref(self._h))
        if rc != 0:
            msg = self._lib.mmm_last_error(None).decode()
            self._h = C.c_void_p()
            self._raise(rc, msg)

    # -- plumbing ---------------------------------------------------------------------------
    @staticmethod
    def _raise(rc: int, msg: str):
        if rc == -1:
            raise ValueError(msg)  # unknown form / bad argument: the reference raises ValueError too
        raise Error(rc, msg)

    def _ck(self, rc: int):
        if rc != 0:
            self._raise(rc, self._lib.mmm_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.mmm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- topology / parameters (model.py add_* methods) --------------------------------------------
    def set_bonds(self, i, j, r0, k):
        i, j = _arr(i, np.int32), _arr(j, np.int32)
        r0 = np.broadcast_to(np.asarray(r0, dtype=np.float64), i.shape)
        k = np.broadcast_to(np.asarray(k, dtype=np.float64), i.shape)
        r0, k = _arr(r0, np.float64), _arr(k, np.float64)
        self._ck(self._lib.mmm_set_bonds(self._h, _p(i), _p(j), _p(r0), _p(k), len(i)))

    def set_loops(self, i, j, r0, k, form: int = 0):
        i, j = _arr(i, np.int32), _arr(j, np.int32)
        r0 = _arr(np.broadcast_to(np.asarray(r0, dtype=np.float64), i.shape), np.float64)
        k = _arr(np.broadcast_to(np.asarray(k, dtype=np.float64), i.shape), np.float64)
        self._ck(self._lib.mmm_set_loops(self._h, _p(i), _p(j), _p(r0), _p(k), len(i), int(form)))

    def set_angles(self, i, j, k, theta0, k_theta):
        i, j, k = _arr(i, np.int32), _arr(j, np.int32), _arr(k, np.int32)
        t0 = _arr(np.broadcast_to(np.asarray(theta0, dtype=np.float64), i.shape), np.float64)
        kt = _arr(np.broadcast_to(np.asarray(k_theta, dtype=np.float64), i.shape), np.float64)
        self._ck(self._lib.mmm_set_angles(self._h, _p(i), _p(j), _p(k), _p(t0), _p(kt), len(i)))

    def set_bead_params(self, s=None, chrom=None, chrom_strength=None):
        s, chrom, cs = _arr(s, np.int8), _arr(chrom, np.int32), _arr(chrom_strength, np.float64)
        for a in (s, chrom, cs):
            if a is not None and a.shape != (self.n,):
                raise ValueError("per-bead parameter arrays must have shape (N,)")
        self._ck(self._lib.mmm_set_bead_params(self._h, _p(s), _p(chrom), _p(cs)))

    def set_pair_term(self, term, form: int, globals_=()):
        t = TERM[term] if isinstance(term, str) else int(term)
        g = np.ascontiguousarray(list(globals_) if len(globals_) else [0.0], dtype=np.float64)
        self._ck(self._lib.mmm_set_pair_term(self._h, t, int(form), _p(g), len(globals_)))

    def set_external_term(self, term, form: int, globals_=()):
        t = TERM[term] if isinstance(term, str) else int(term)
        g = np.ascontiguousarray(list(globals_) if len(globals_) else [0.0], dtype=np.float64)
        self._ck(self._lib.mmm_set_external_term(self._h, t, int(form), _p(g), len(globals_)))

    def set_cutoff(self, rc_nm: float):
        self._ck(self._lib.mmm_set_cutoff(self._h, float(rc_nm)))

    # -- state ------------------------------------------------------------------------------
    def set_positions(self, xyz_nm):
        x = _arr(xyz_nm, np.float64)
        if x.shape != (self.n, 3):
            raise ValueError(f"positions must have shape ({self.n}, 3)")
        self._ck(self._lib.mmm_set_positions(self._h, _p(x)))

    def get_positions(self) -> np.ndarray:
        out = np.empty((self.n, 3), dtype=np.float64)
        self._ck(self._lib.mmm_get_positions(self._h, _p(out)))
        return out

    def set_positions_tensor(self, t):
        """Hand a CUDA float64 (N,3) torch tensor on this engine's device to the engine (no host copy of x)."""
        if not (t.is_cuda and t.dtype.is_floating_point and t.element_size() == 8 and t.is_contiguous()):
            raise ValueError("expected a contiguous CUDA float64 tensor")
        if tuple(t.shape) != (self.n, 3) or t.device.index != self.device:
            raise ValueError("tensor shape/device mismatch")
        self._ck(self._lib.mmm_set_positions_device(self._h, C.c_void_p(t.data_ptr())))

    def get_positions_tensor(self, out):
        if tuple(out.shape) != (self.n, 3) or not out.is_cuda or out.element_size() != 8 or not out.is_contiguous():
            raise ValueError("expected a contiguous CUDA float64 (N,3) tensor")
        self._ck(self._lib.mmm_get_positions_device(self._h, C.c_void_p(out.data_ptr())))
        return out

    def hilbert_init(self, p: int = 8, spacing_nm: float = 0.1):
        self._ck(self._lib.mmm_hilbert_init(self._h, int(p), float(spacing_nm)))

    def hilbert_points(self, p: int = 8) -> np.ndarray:
        out = np.empty((self.n, 3), dtype=np.int32)
        self._ck(self._lib.mmm_hilbert_points(self._h, int(p), _p(out)))
        return out

    # -- evaluation -------------------------------------------------------------------------
    def energy_forces(self, want_forces: bool = True, out=None):
        """Per-term energies (10,) kJ/mol and forces (N,3) kJ/mol/nm at the current positions.
        ``out``: optional preallocated C-contiguous float64 (N,3) array for the forces (e.g. pinned)."""
        e = np.zeros(NUM_TERMS)
        if out is not None and (out.shape != (self.n, 3) or out.dtype != np.float64 or not out.flags.c_contiguous):
            raise ValueError("out must be a C-contiguous float64 (N, 3) array")
        f = (out if out is not None else np.empty((self.n, 3))) if want_forces else None
        self._ck(self._lib.mmm_energy_forces(self._h, _p(e), _p(f)))
        return e, f

    def evaluate_n(self, n: int):
        self._ck(self._lib.mmm_evaluate_n(self._h, int(n)))

    def evaluate_timed(self, n: int, flush_l2: bool = True):
        """n evaluations timed on the device; returns (total_ms, summed pair-kernel ms)."""
        tot, pair = C.c_float(), C.c_float()
        self._ck(self._lib.mmm_evaluate_timed(self._h, int(n), int(bool(flush_l2)), C.byref(tot), C.byref(pair)))
        return float(tot.value), float(pair.value)

    def last_result(self):
        """Per-term energies (10,) and forces (N,3) of the most recent evaluation, read back
        without evaluating again (e.g. the last of ``evaluate_timed``'s evaluations)."""
        e = np.zeros(NUM_TERMS)
        f = np.empty((self.n, 3))
        self._ck(self._lib.mmm_last_result(self._h, _p(e), _p(f)))
        return e, f

    def minimize(self, tol: float = 10.0, max_iter: int = 0) -> dict:
        """L-BFGS to OpenMM's default tolerance (10 kJ/mol/nm RMS force), unlimited iterations."""
        rep = MinReport()
        self._ck(self._lib.mmm_minimize(self._h, float(tol), int(max_iter), C.byref(rep)))
        return {k: getattr(rep, k) for k, _ in MinReport._fields_}

    def mean_pair_distance(self) -> float:
        """np.mean(cdist(V, V)) at the current positions, computed on the device."""
        out = C.c_double()
        self._ck(self._lib.mmm_mean_pair_distance(self._h, C.byref(out)))
        return float(out.value)

    # -- MD relaxation ----------------------------------------------------------------------------
    def md_configure(self, integrator="langevin", dt_ps=0.001, temperature_k=310.0, friction_per_ps=0.5,
                     mass_amu=16427.889, seed=0, amd_alpha=None, amd_e=None):
        """amd_alpha / amd_e: the two globals of mm.amd.AMDIntegrator (model.py:796-800), kJ/mol; used by
        the "amd" integrator only (a handle starts with the reference's defaults, 100 and 1000)."""
        kind = _lib.MD_INTEGRATORS.get(integrator, integrator) if isinstance(integrator, str) else int(integrator)
        if not isinstance(kind, int):
            raise ValueError(f"Unknown SIM_INTEGRATOR_TYPE: {integrator} (supported: {', '.join(_lib.MD_INTEGRATORS)})")
        self._ck(self._lib.mmm_md_configure(self._h, kind, float(dt_ps), float(temperature_k), float(friction_per_ps),
                                            float(mass_amu), int(seed)))
        if amd_alpha is not None or amd_e is not None:
            self._ck(self._lib.mmm_md_set_amd(self._h, float(100.0 if amd_alpha is None else amd_alpha),
                                              float(1000.0 if amd_e is None else amd_e)))

    def set_velocities_to_temperature(self, temperature_k: float, seed: int = 0):
        self._ck(self._lib.mmm_set_velocities_to_temperature(self._h, float(temperature_k), int(seed)))

    def set_velocities(self, v):
        v = _arr(v, np.float64)
        if v.shape != (self.n, 3):
            raise ValueError(f"velocities must have shape ({self.n}, 3)")
        self._ck(self._lib.mmm_set_velocities(self._h, _p(v)))

    def get_velocities(self) -> np.ndarray:
        out = np.empty((self.n, 3), dtype=np.float64)
        self._ck(self._lib.mmm_get_velocities(self._h, _p(out)))
        return out

    def md_run(self, n_steps: int, want_report: bool = True) -> dict | None:
        """n steps enqueued back to back.  want_report: one more force evaluation at the end for the potential
        energy, the kinetic energy and a host read of both; without it nothing is evaluated or read back."""
        if not want_report:
            self._ck(self._lib.mmm_md_run(self._h, int(n_steps), None))
            return None
        rep = MdReport()
        self._ck(self._lib.mmm_md_run(self._h, int(n_steps), C.byref(rep)))
        return {k: getattr(rep, k) for k, _ in MdReport._fields_}

    # -- one system on several GPUs (exact mode) ------------------------------------------------
    @staticmethod
    def dist_unique_id() -> bytes:
        """NCCL unique id (rank 0 creates it and ships it to the other ranks)."""
        lib = _lib.load()
        buf = C.create_string_buffer(128)
        rc = lib.mmm_dist_unique_id(buf, 128)
        if rc != 0:
            raise Error(rc, lib.mmm_last_error(None).decode())
        return buf.raw

    def dist_init(self, rank: int, world: int, unique_id: bytes | None):
        """Join a group of `world` engines (one per GPU / process) that share the pair work of ONE system."""
        buf = C.create_string_buffer(unique_id, 128) if unique_id else None
        self._ck(self._lib.mmm_dist_init(self._h, int(rank), int(world), buf, 128 if unique_id else 0))

    def dist_emulate(self, world: int):
        """Tests: run the shares of `world` ranks one after another on this GPU."""
        self._ck(self._lib.mmm_dist_emulate(self._h, int(world)))

    @property
    def dist_queue_mode(self) -> int:
        """1: all ranks draw work items from one queue over NVLink peer memory; 0: static round-robin dealing."""
        return int(self._lib.mmm_dist_queue_mode(self._h))

    @property
    def last_collective_ms(self) -> float:
        """ms of the exchange step of the most recent evaluation on this rank (0 without a communicator)."""
        ms = C.c_float()
        self._ck(self._lib.mmm_dist_last_exchange_ms(self._h, C.byref(ms)))
        return float(ms.value)

    # -- introspection ----------------------------------------------------------------------
    @property
    def launch_count(self) -> int:
        return int(self._lib.mmm_launch_count(self._h))

    def set_pair_kernel(self, which: int):
        """0 = automatic (Newton-3 kernel for the default forms), 1 = always the gather kernel."""
        self._ck(self._lib.mmm_set_pair_kernel(self._h, int(which)))

    def set_chb_surrogate(self, on: bool):
        """Cut-off mode only: CHB between cluster centroids instead of the exact same-chromosome pass
        (coarse stage of the two-stage minimisation; not the reference's potential)."""
        self._ck(self._lib.mmm_set_chb_surrogate(self._h, int(bool(on))))

    def set_graph(self, on: bool):
        """minimize(): replay a captured CUDA graph per evaluation (default) or launch kernel by kernel."""
        self._ck(self._lib.mmm_set_graph(self._h, int(bool(on))))

    @property
    def pair_kernel_in_use(self) -> int:
        """0 none, 1 gather, 2 Newton-3, 3 cut-off cell list (kernel of the last evaluation)."""
        return int(self._lib.mmm_pair_kernel_in_use(self._h))

    @property
    def last_pair_kernel_ms(self) -> float:
        ms = C.c_float()
        self._ck(self._lib.mmm_last_pair_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def cell_list(self):
        order = np.empty(self.n, dtype=np.int32)
        keys = np.empty(self.n, dtype=np.uint32)
        self._ck(self._lib.mmm_get_cell_list(self._h, _p(order), _p(keys)))
        return order, keys

    def cell_grid(self) -> dict:
        """Grid of the last cut-off evaluation and the number of unordered pairs inside the cut-off."""
        cell, dim, origin, pairs = C.c_float(), C.c_int(), C.c_float(), C.c_int64()
        self._ck(self._lib.mmm_get_cell_grid(self._h, C.byref(cell), C.byref(dim), C.byref(origin), C.byref(pairs)))
        return dict(cell=float(cell.value), dim=int(dim.value), origin=float(origin.value), pairs=int(pairs.value))


def measure_fp32_peak(device: int = 0):
    """(FP32 TFLOP/s, MUFU Tera-op/s) measured by micro-benchmark on this GPU."""
    lib = _lib.load()
    a, b = C.c_double(), C.c_double()
    rc = lib.mmm_measure_fp32_peak(int(device), C.byref(a), C.byref(b))
    if rc != 0:
        raise Error(rc, "CUDA error: FP32 peak micro-benchmark failed")
    return a.value, b.value
