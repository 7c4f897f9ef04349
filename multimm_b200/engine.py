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

    def contacts(self, rc_nm: float, bin_of_bead=None, n_bins: int = 1, want_sep: bool = True):
        """Contacts (FP64 d2 < rc^2, see mmm_contacts) at the current positions, counted on the device.
        Returns (map, sep, pairs): map (n_bins, n_bins) uint64, symmetric, of the contacts between the bins
        of ``bin_of_bead`` (int[N], -1 = left out), or None without ``bin_of_bead``; sep (N,) uint64,
        same-chromosome contacts by index separation j - i, or None if not ``want_sep``; pairs, all contacts."""
        n_bins = int(n_bins)
        bins = None
        if bin_of_bead is not None:
            bins = _arr(bin_of_bead, np.int32)
            if bins.shape != (self.n,):
                raise ValueError(f"bin_of_bead must have shape ({self.n},)")
        cmap = np.empty((n_bins, n_bins), dtype=np.uint64) if bins is not None and 1 <= n_bins <= 4096 else None
        sep = np.empty(self.n, dtype=np.uint64) if want_sep else None
        pairs = C.c_int64()
        self._ck(self._lib.mmm_contacts(self._h, float(rc_nm), _p(bins), n_bins, _p(cmap), _p(sep), C.byref(pairs)))
        return cmap, sep, int(pairs.value)

    def contacts_sparse(self, rc_nm: float, bin_of_bead, n_bins: int):
        """The contact map of ``contacts`` stored sparse, for any int32 number of bins (mmm_contacts_sparse).
        Returns (rows int32, cols int32, vals uint64, pairs): the nonzero entries of the upper triangle
        sorted by (row, col), row <= col, counting the contacts between bins row and col of ``bin_of_bead``
        (int[N], -1 = left out); pairs, all contacts."""
        bins = _arr(bin_of_bead, np.int32)
        if bins.shape != (self.n,):
            raise ValueError(f"bin_of_bead must have shape ({self.n},)")
        n_entries, pairs = C.c_int64(), C.c_int64()
        self._ck(self._lib.mmm_contacts_sparse(self._h, float(rc_nm), _p(bins), int(n_bins), C.byref(n_entries),
                                               C.byref(pairs)))
        e = int(n_entries.value)
        rows, cols, vals = np.empty(e, np.int32), np.empty(e, np.int32), np.empty(e, np.uint64)
        self._ck(self._lib.mmm_contacts_sparse_read(self._h, _p(rows), _p(cols), _p(vals)))
        return rows, cols, vals, int(pairs.value)

    def contacts_stats(self) -> dict:
        """Of the last contacts() or contacts_sparse() call: bead pairs tested in FP64 (those that survived box culling) and the
        device time of its kernels in ms (CUDA events on the engine's stream)."""
        cand, ms = C.c_int64(), C.c_float()
        self._ck(self._lib.mmm_contacts_stats(self._h, C.byref(cand), C.byref(ms)))
        return dict(candidates=int(cand.value), device_ms=float(ms.value))

    def distance_map(self, bin_of_bead, n_bins: int):
        """Sums of the quantised distance and squared distance over every bead pair i < j, binned by
        ``bin_of_bead`` (int[N], -1 = left out), at the current positions (mmm_distance_map).  Returns
        (dist_sum, dist2_sum): uint64 (n_bins, n_bins), symmetric, in units of Q = 2^-24 nm and nm^2."""
        n_bins = int(n_bins)
        bins = _arr(bin_of_bead, np.int32)
        if bins is None or bins.shape != (self.n,):
            raise ValueError(f"bin_of_bead must have shape ({self.n},)")
        shape = (n_bins, n_bins) if 1 <= n_bins <= 4096 else (0, 0)
        dsum, d2sum = np.empty(shape, np.uint64), np.empty(shape, np.uint64)
        ms = C.c_float()
        self._ck(self._lib.mmm_distance_map(self._h, _p(bins), n_bins, _p(dsum), _p(d2sum), C.byref(ms)))
        self._distance_ms = float(ms.value)
        return dsum, d2sum

    def distance_stats(self) -> dict:
        """Of the last distance_map() call: the device time of its pass in ms (CUDA events on the engine's
        stream)."""
        return dict(device_ms=getattr(self, "_distance_ms", 0.0))

    # -- trajectory maps (sums over many structures) --------------------------------------------------
    def sampler_configure(self, rc_nm: float = 0.2, contact_bins=None, n_contact_bins: int = 0, fine_bins=None,
                          n_fine_bins: int = 0, distance_bins=None, n_distance_bins: int = 0):
        """Clear the sampler and set its maps (mmm_sampler_configure): the dense contact map, sep and pairs of
        ``contacts`` over ``contact_bins``, the sparse map of ``contacts_sparse`` over ``fine_bins`` (needs
        ``contact_bins``), the sums of ``distance_map`` over ``distance_bins``; None switches a map off."""
        tabs = []
        for bins in (contact_bins, fine_bins, distance_bins):
            b = _arr(bins, np.int32)
            if b is not None and b.shape != (self.n,):
                raise ValueError(f"bin tables must have shape ({self.n},)")
            tabs.append(b)
        self._ck(self._lib.mmm_sampler_configure(self._h, float(rc_nm), _p(tabs[0]), int(n_contact_bins), _p(tabs[1]),
                                                 int(n_fine_bins), _p(tabs[2]), int(n_distance_bins)))
        self._sampler = (None if tabs[0] is None else int(n_contact_bins), None if tabs[1] is None else int(n_fine_bins),
                         None if tabs[2] is None else int(n_distance_bins))

    def sample(self):
        """Add the structure at the current positions to every map of the sampler (mmm_sample)."""
        self._ck(self._lib.mmm_sample(self._h))

    def sampler_read(self) -> dict:
        """The sampler's sums (mmm_sampler_read, mmm_sampler_read_fine): ``samples``; ``counts`` (B, B), ``sep``
        (N,) uint64 and ``pairs``; the fine map ``rows``, ``cols`` int32, ``vals`` uint64 (sorted upper
        triangle); ``dist_sum``, ``dist2_sum`` (B, B) uint64; ``device_ms`` of all samples.  The entries of a
        map that is off are None."""
        nc, nf, nd = getattr(self, "_sampler", (None, None, None))
        counts = np.empty((nc, nc), np.uint64) if nc else None
        sep = np.empty(self.n, np.uint64) if nc else None
        dsum = np.empty((nd, nd), np.uint64) if nd else None
        d2sum = np.empty((nd, nd), np.uint64) if nd else None
        samples, pairs, entries, ms = C.c_int64(), C.c_int64(), C.c_int64(), C.c_float()
        self._ck(self._lib.mmm_sampler_read(self._h, C.byref(samples), _p(counts), _p(sep), C.byref(pairs),
                                            C.byref(entries), _p(dsum), _p(d2sum), C.byref(ms)))
        out = dict(samples=int(samples.value), counts=counts, sep=sep, pairs=int(pairs.value) if nc else None,
                   rows=None, cols=None, vals=None, dist_sum=dsum, dist2_sum=d2sum, device_ms=float(ms.value))
        if nf:
            e = int(entries.value)
            out["rows"], out["cols"], out["vals"] = np.empty(e, np.int32), np.empty(e, np.int32), np.empty(e, np.uint64)
            self._ck(self._lib.mmm_sampler_read_fine(self._h, _p(out["rows"]), _p(out["cols"]), _p(out["vals"])))
        return out

    # -- loop readout (per-loop sums and APA over many structures) -------------------------------------
    def loops_configure(self, rc_nm: float, window: int, bead_lo, bead_hi, first_lo, end_lo, first_hi, end_hi,
                        group):
        """Clear the loop accumulator and set its rows (mmm_loops_configure): anchor beads ``bead_lo`` <
        ``bead_hi``, the chromosome block [first, end) of each, ``group`` 0 (enforced) or 1 (held out); the
        contact radius and the APA window W in [0, 25].  loops.device_rows gives these for a member."""
        cols = [_arr(a, np.int32) for a in (bead_lo, bead_hi, first_lo, end_lo, first_hi, end_hi)]
        grp = _arr(group, np.int8)
        r = len(cols[0])
        if any(c.shape != (r,) for c in cols) or grp.shape != (r,):
            raise ValueError("loop rows: every array must have the same length")
        self._ck(self._lib.mmm_loops_configure(self._h, float(rc_nm), int(window), r, *(_p(c) for c in cols), _p(grp)))
        self._loops = (r, int(window))

    def loops_add(self):
        """Add the structure at the current positions to the loop sums (mmm_loops_add)."""
        self._ck(self._lib.mmm_loops_add(self._h))

    def loops_read(self) -> dict:
        """The loop sums (mmm_loops_read): ``samples``; ``contacts``, ``dist_sum``, ``dist2_sum`` uint64[rows];
        ``apa_contacts``, ``apa_dist_sum`` uint64 [2][2W+1][2W+1]; ``device_ms`` of all adds."""
        r, w = getattr(self, "_loops", (0, 0))
        span = 2 * w + 1
        out = {k: np.zeros(r, np.uint64) for k in ("contacts", "dist_sum", "dist2_sum")}
        out.update(apa_contacts=np.zeros((2, span, span), np.uint64), apa_dist_sum=np.zeros((2, span, span), np.uint64))
        samples, ms = C.c_int64(), C.c_float()
        self._ck(self._lib.mmm_loops_read(self._h, C.byref(samples), _p(out["contacts"]), _p(out["dist_sum"]),
                                          _p(out["dist2_sum"]), _p(out["apa_contacts"]), _p(out["apa_dist_sum"]),
                                          C.byref(ms)))
        out.update(samples=int(samples.value), device_ms=float(ms.value))
        return out

    # -- three-way contact map (bead triples in mutual contact, summed over many structures) -----------
    def triplets_configure(self, rc_nm: float, bin_of_bead, n_bins: int, max_chunk_keys: int = 0):
        """Clear the three-way accumulator and set its bins (mmm_triplets_configure): ``bin_of_bead`` (int[N],
        -1 = left out) of ``n_bins`` <= 2^20 bins, the contact radius, and the most binned triples of one
        structure sorted at a time (0 = 2^26)."""
        bins = _arr(bin_of_bead, np.int32)
        if bins is not None and bins.shape != (self.n,):
            raise ValueError(f"bin_of_bead must have shape ({self.n},)")
        self._ck(self._lib.mmm_triplets_configure(self._h, float(rc_nm), _p(bins), int(n_bins), int(max_chunk_keys)))
        self._triplet_bins = int(n_bins)

    def triplets_add(self):
        """Add the three-way contacts of the structure at the current positions (mmm_triplets_add)."""
        self._ck(self._lib.mmm_triplets_add(self._h))

    def triplets_read(self) -> dict:
        """The three-way sums (mmm_triplets_read, mmm_triplets_read_entries): ``samples``; ``triples``, all
        three-way contacts; ``p`` <= ``q`` <= ``r`` (int32) and ``vals`` (uint64), the entries sorted by key
        (p * B + q) * B + r; ``chunks`` and ``device_ms`` of all adds."""
        samples, triples, entries, chunks, ms = C.c_int64(), C.c_uint64(), C.c_int64(), C.c_int64(), C.c_float()
        self._ck(self._lib.mmm_triplets_read(self._h, C.byref(samples), C.byref(triples), C.byref(entries),
                                             C.byref(chunks), C.byref(ms)))
        e = int(entries.value)
        keys, vals = np.empty(e, np.uint64), np.empty(e, np.uint64)
        self._ck(self._lib.mmm_triplets_read_entries(self._h, _p(keys), _p(vals)))
        b = np.uint64(getattr(self, "_triplet_bins", 1))
        pq, r = keys // b, keys % b
        return dict(samples=int(samples.value), triples=int(triples.value), chunks=int(chunks.value),
                    device_ms=float(ms.value), p=(pq // b).astype(np.int32), q=(pq % b).astype(np.int32),
                    r=r.astype(np.int32), vals=vals)

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
