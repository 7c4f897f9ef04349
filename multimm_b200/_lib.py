"""ctypes binding of libmultimm_b200.so (the C-ABI in include/multimm_b200.h).

The library is the product; there is no CPU or PyTorch fallback.  If it is missing or cannot be
loaded, importing the engine fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, os.environ.get("MMM_LIB_NAME", "libmultimm_b200.so"))  # MMM_LIB_NAME: experiments only

NUM_TERMS = 10
TERM_NAMES = ("EV", "COB", "SCB", "CHB", "SC", "LAM", "CF", "BOND", "LOOP", "ANGLE")
TERM = {name: i for i, name in enumerate(TERM_NAMES)}
FORM_OFF = -1

# functional-form enumerations (mirrors of the MMM_* macros)
EV_FORMS = {"powerlaw": 0, "gaussian_core": 1}
BLOCK_FORMS = {"gaussian": 0, "yukawa": 1, "theta": 2}
CHB_FORMS = {"polynomial": 0, "gaussian": 1, "saturating": 2}
LAM_FORMS = {"sin": 0, "gaussian_shell": 1, "harmonic_shell": 2, "logistic_shell": 3}
CF_FORMS = {"harmonic": 0, "gaussian": 1, "logistic": 2}
LOOP_FORMS = {"harmonic": 0, "fene_soft": 1, "gaussian_tether": 2}

# every symbol include/multimm_b200.h declares
EXPORTS = (
    "mmm_abi_version", "mmm_create", "mmm_destroy", "mmm_last_error",
    "mmm_set_bonds", "mmm_set_loops", "mmm_set_angles", "mmm_set_bead_params",
    "mmm_set_pair_term", "mmm_set_external_term", "mmm_set_cutoff",
    "mmm_set_positions", "mmm_get_positions", "mmm_set_positions_device", "mmm_get_positions_device",
    "mmm_hilbert_init", "mmm_hilbert_points",
    "mmm_energy_forces", "mmm_energy_forces_device", "mmm_evaluate_n", "mmm_evaluate_timed", "mmm_last_result",
    "mmm_minimize",
    "mmm_launch_count", "mmm_set_graph", "mmm_set_chb_surrogate", "mmm_set_pair_kernel", "mmm_pair_kernel_in_use", "mmm_last_pair_kernel_ms", "mmm_get_cell_list", "mmm_get_cell_grid", "mmm_measure_fp32_peak",
    "mmm_dist_unique_id", "mmm_dist_init", "mmm_dist_emulate", "mmm_dist_last_exchange_ms", "mmm_dist_queue_mode",
    "mmm_mean_pair_distance", "mmm_contact_map", "mmm_contacts", "mmm_contacts_sparse", "mmm_contacts_sparse_read", "mmm_contacts_stats", "mmm_distance_map", "mmm_sampler_configure", "mmm_sample", "mmm_sampler_read", "mmm_sampler_read_fine", "mmm_loops_configure", "mmm_loops_add", "mmm_loops_read", "mmm_triplets_configure", "mmm_triplets_add", "mmm_triplets_read", "mmm_triplets_read_entries", "mmm_dynamics_configure", "mmm_dynamics_add", "mmm_dynamics_read", "mmm_dynamics_read_runs", "mmm_disthist_configure", "mmm_disthist_add", "mmm_disthist_read", "mmm_gam_configure", "mmm_gam_add", "mmm_gam_read", "mmm_md_configure", "mmm_md_set_amd", "mmm_set_velocities_to_temperature", "mmm_set_velocities", "mmm_get_velocities", "mmm_md_run",
)


class MinReport(C.Structure):
    _fields_ = [
        ("iterations", C.c_int64), ("evaluations", C.c_int64),
        ("e_initial", C.c_double), ("e_final", C.c_double), ("rms_force", C.c_double),
        ("wall_seconds", C.c_double), ("converged", C.c_int32), ("ls_status", C.c_int32),
    ]


class MdReport(C.Structure):
    _fields_ = [("step", C.c_int64), ("potential", C.c_double), ("kinetic", C.c_double), ("temperature", C.c_double)]


MD_INTEGRATORS = {"langevin": 0, "verlet": 1, "brownian": 2, "amd": 3}


class Error(RuntimeError):
    """Engine failure (replaces openmm.OpenMMException for callers in the style of bridge.py:65-84).
    Device failures keep the substring "CUDA error" in the message."""

    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


_lib = None


def load():
    """Load the shared library once.  Raises if it has not been built (python -m multimm_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m multimm_b200.build` "
            "(nvcc, sm_100a). The engine has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
    sigs = {
        "mmm_abi_version": (i32, []),
        "mmm_create": (i32, [i32, i64, C.POINTER(vp)]),
        "mmm_destroy": (i32, [vp]),
        "mmm_last_error": (C.c_char_p, [vp]),
        "mmm_set_bonds": (i32, [vp, vp, vp, vp, vp, i64]),
        "mmm_set_loops": (i32, [vp, vp, vp, vp, vp, i64, i32]),
        "mmm_set_angles": (i32, [vp, vp, vp, vp, vp, vp, i64]),
        "mmm_set_bead_params": (i32, [vp, vp, vp, vp]),
        "mmm_set_pair_term": (i32, [vp, i32, i32, vp, i32]),
        "mmm_set_external_term": (i32, [vp, i32, i32, vp, i32]),
        "mmm_set_cutoff": (i32, [vp, dbl]),
        "mmm_set_positions": (i32, [vp, vp]),
        "mmm_get_positions": (i32, [vp, vp]),
        "mmm_set_positions_device": (i32, [vp, vp]),
        "mmm_get_positions_device": (i32, [vp, vp]),
        "mmm_hilbert_init": (i32, [vp, i32, dbl]),
        "mmm_hilbert_points": (i32, [vp, i32, vp]),
        "mmm_energy_forces": (i32, [vp, vp, vp]),
        "mmm_energy_forces_device": (i32, [vp, vp, vp]),
        "mmm_evaluate_n": (i32, [vp, i32]),
        "mmm_evaluate_timed": (i32, [vp, i32, i32, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
        "mmm_last_result": (i32, [vp, vp, vp]),
        "mmm_minimize": (i32, [vp, dbl, i64, C.POINTER(MinReport)]),
        "mmm_launch_count": (i64, [vp]),
        "mmm_set_pair_kernel": (i32, [vp, i32]),
        "mmm_set_graph": (i32, [vp, i32]),
        "mmm_set_chb_surrogate": (i32, [vp, i32]),
        "mmm_pair_kernel_in_use": (i32, [vp]),
        "mmm_last_pair_kernel_ms": (i32, [vp, C.POINTER(C.c_float)]),
        "mmm_get_cell_list": (i32, [vp, vp, vp]),
        "mmm_get_cell_grid": (i32, [vp, C.POINTER(C.c_float), C.POINTER(i32), C.POINTER(C.c_float), C.POINTER(i64)]),
        "mmm_measure_fp32_peak": (i32, [i32, C.POINTER(dbl), C.POINTER(dbl)]),
        "mmm_dist_unique_id": (i32, [vp, i32]),
        "mmm_dist_init": (i32, [vp, i32, i32, vp, i32]),
        "mmm_dist_emulate": (i32, [vp, i32]),
        "mmm_dist_last_exchange_ms": (i32, [vp, C.POINTER(C.c_float)]),
        "mmm_dist_queue_mode": (i32, [vp]),
        "mmm_mean_pair_distance": (i32, [vp, C.POINTER(dbl)]),
        "mmm_contact_map": (i32, [i32, vp, i64, i32, i32, vp, C.POINTER(dbl)]),
        "mmm_contacts": (i32, [vp, dbl, vp, i32, vp, vp, C.POINTER(i64)]),
        "mmm_contacts_sparse": (i32, [vp, dbl, vp, i32, C.POINTER(i64), C.POINTER(i64)]),
        "mmm_contacts_sparse_read": (i32, [vp, vp, vp, vp]),
        "mmm_contacts_stats": (i32, [vp, C.POINTER(i64)]),
        "mmm_distance_map": (i32, [vp, vp, i32, vp, vp, C.POINTER(C.c_float)]),
        "mmm_sampler_configure": (i32, [vp, dbl, vp, i32, vp, i32, vp, i32]),
        "mmm_sample": (i32, [vp]),
        "mmm_sampler_read": (i32, [vp, C.POINTER(i64), vp, vp, C.POINTER(i64), C.POINTER(i64), vp, vp,
                                   C.POINTER(C.c_float)]),
        "mmm_sampler_read_fine": (i32, [vp, vp, vp, vp]),
        "mmm_loops_configure": (i32, [vp, dbl, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
        "mmm_loops_add": (i32, [vp]),
        "mmm_loops_read": (i32, [vp, C.POINTER(i64), vp, vp, vp, vp, vp, C.POINTER(C.c_float)]),
        "mmm_triplets_configure": (i32, [vp, dbl, vp, i32, i64]),
        "mmm_triplets_add": (i32, [vp]),
        "mmm_triplets_read": (i32, [vp, C.POINTER(i64), C.POINTER(C.c_uint64), C.POINTER(i64), C.POINTER(i64),
                                    C.POINTER(C.c_float)]),
        "mmm_triplets_read_entries": (i32, [vp, vp, vp]),
        "mmm_dynamics_configure": (i32, [vp, dbl, vp, i32, vp, i32, i32, vp, vp, vp]),
        "mmm_dynamics_add": (i32, [vp]),
        "mmm_dynamics_read": (i32, [vp, C.POINTER(i64), vp, vp, C.POINTER(C.c_float)]),
        "mmm_dynamics_read_runs": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "mmm_disthist_configure": (i32, [vp, vp, i32, vp, i32]),
        "mmm_disthist_add": (i32, [vp]),
        "mmm_disthist_read": (i32, [vp, C.POINTER(i64), vp, C.POINTER(C.c_float)]),
        "mmm_gam_configure": (i32, [vp, vp, i32, i32]),
        "mmm_gam_add": (i32, [vp, vp, i32, dbl]),
        "mmm_gam_read": (i32, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), vp, C.POINTER(C.c_float)]),
        "mmm_md_configure": (i32, [vp, i32, dbl, dbl, dbl, dbl, C.c_uint64]),
        "mmm_md_set_amd": (i32, [vp, dbl, dbl]),
        "mmm_set_velocities_to_temperature": (i32, [vp, dbl, C.c_uint64]),
        "mmm_set_velocities": (i32, [vp, vp]),
        "mmm_get_velocities": (i32, [vp, vp]),
        "mmm_md_run": (i32, [vp, i64, C.POINTER(MdReport)]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.mmm_abi_version() != 1:
        raise ImportError("libmultimm_b200.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib
