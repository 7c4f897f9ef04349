"""Cut-off mode's device code against FP64 / bit-exact references:

* the cell-list gather kernel (mmm_cells.cu) for every functional form and both fast instantiations,
  against the oracle with the same truncation, and its grid, keys and order against tests/cells_ref.py;
* the cell edge: a 0.1 nm lattice puts in-cut pairs exactly on cell boundaries (tests/cells_ref.py's
  stencil_misses), where a grid of edge rc would lose them to the 27-cell walk;
* the far field on cluster centroids (mmm_chb_clusters.cu) against tests/far_field_ref.py;
* switching modes on one handle, as the two-stage minimisation does every round.

Bars: per-term energies 1e-5 relative and per-bead forces 1e-4 against the oracle (BASELINE.json north
star); integer outputs bit-exact."""
import numpy as np
import pytest

import cells_ref as CR
import far_field_ref as FR
from common import O, force_rel_err, make_case, to_engine, to_oracle

pytestmark = pytest.mark.gpu

E_TOL = 1e-5
F_TOL = 1e-4
U = 2.0 ** -53  # unit round-off of FP64

ALL_TERMS = ("EV", "COB", "SCB", "CHB", "SC", "LAM", "CF", "BOND", "LOOP", "ANGLE")


def _assert_energies(e, e_ref, what=""):
    for t in range(10):
        assert abs(e[t] - e_ref[t]) <= E_TOL * max(abs(e_ref[t]), 1e-12) + 1e-9, (what, O.TERM_NAMES[t], e[t], e_ref[t])


def _check_cells(case, rc, force_cells=False):
    """One cut-off evaluation on the cell-list kernel against the oracle and cells_ref; returns the grid."""
    eng = to_engine(case, cutoff=rc)
    if force_cells:
        eng.set_pair_kernel(1)
    e, f = eng.energy_forces()
    assert eng.pair_kernel_in_use == 3
    grid = eng.cell_grid()
    order, keys = eng.cell_list()
    e2, f2 = eng.energy_forces()
    eng.close()
    sysd = to_oracle(case, cutoff=rc)
    n_ref = O.count_pairs(sysd, case["x"])
    assert grid["pairs"] == n_ref, ("pairs inside the cut-off", grid["pairs"], n_ref)
    e_ref, f_ref = O.energy_forces(sysd, case["x"])
    _assert_energies(e, e_ref, rc)
    assert force_rel_err(f, f_ref) <= F_TOL
    xc = CR.centred(case["x"])
    keys_ref, order_ref, (cell, dim, origin) = CR.cell_list(xc, rc)
    assert (grid["cell"], grid["dim"], grid["origin"]) == (float(cell), dim, float(origin)), (grid, cell, dim, origin)
    assert np.array_equal(order, order_ref) and np.array_equal(keys, keys_ref)
    assert np.array_equal(e, e2) and np.array_equal(f, f2)
    return grid


def _form_case(forms, terms=ALL_TERMS, ev_power=6.0):
    return make_case(1500, n_chrom=3, seed=11, forms=forms, chb_de=1.0, terms=terms, ev_power=ev_power)


def _cob_rc_differs():
    case = make_case(1500, n_chrom=3, seed=12, terms=("EV", "COB", "SCB", "BOND"))
    form, g = case["cob"]
    case["cob"] = (form, [g[0] * 1.3, *g[1:]])
    return case


# (case builder, set_pair_kernel(1) needed): the pair forms of the last three form sets are the defaults,
# which cut-off mode would give to the Morton kernel
FORM_CASES = {
    "ev_gaussian_core": (lambda: _form_case({"EV": 1}), False),  # CHB polynomial: Newton-3 CHB pass beside
    "cob_scb_yukawa": (lambda: _form_case({"COB": 1, "SCB": 1}), False),
    "cob_scb_theta": (lambda: _form_case({"COB": 2, "SCB": 2}), False),
    "chb_gaussian": (lambda: _form_case({"CHB": 1}), False),  # CHB-only gather pass beside
    "chb_rational": (lambda: _form_case({"CHB": 2}), False),
    "ext_forms_1": (lambda: _form_case({"LAM": 1, "CF": 1, "LOOP": 1}), True),
    "ext_forms_2": (lambda: _form_case({"LAM": 2, "CF": 2, "LOOP": 2}), True),
    "lam_3": (lambda: _form_case({"LAM": 3}), True),
    "ev_power_4.5": (lambda: _form_case({}, terms=("EV", "SCB", "CHB", "BOND"), ev_power=4.5), False),
    "ev_off_scb_on": (lambda: _form_case({}, terms=("SCB", "COB", "BOND")), False),
    "cob_rc_ne_scb_rc": (_cob_rc_differs, False),
}


@pytest.mark.parametrize("rc", [0.25, 0.45])
@pytest.mark.parametrize("name", list(FORM_CASES))
def test_cell_list_kernel_every_form(built_lib, name, rc):
    build, force_cells = FORM_CASES[name]
    grid = _check_cells(build(), rc, force_cells)
    assert grid["dim"] > 3  # several cells per axis: neighbours really are walked


@pytest.mark.parametrize("ev_power", [6.0, 3.0])
@pytest.mark.parametrize("terms", [("EV",), ("EV", "SCB"), ("EV", "COB"), ("EV", "COB", "SCB")])
def test_cell_list_kernel_fast_instantiations(built_lib, ev_power, terms):
    """Default forms forced onto the cell-list kernel: k_pair_cells<EVP = 6 | 3, GK = 0..3>."""
    case = make_case(2000, n_chrom=2, seed=13, terms=terms + ("BOND",), ev_power=ev_power)
    _check_cells(case, 0.35, force_cells=True)


def lattice_case(side=24, terms=("EV", "SCB"), ev_power=6.0):
    """A cubic lattice of 0.1 nm: pairs at 0.1, 0.2, 0.3 nm sit exactly on the boundaries of cells of
    edge 0.2 or 0.3 nm."""
    case = make_case(side ** 3, n_chrom=2, seed=17, terms=terms, ev_power=ev_power)
    g = np.arange(side) * 0.1
    case["x"] = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) + np.array([0.013, -0.4, 2.0])
    return case


@pytest.mark.parametrize("kernel", ["cells_generic", "cells_fast", "morton"])
@pytest.mark.parametrize("rc", [0.2, 0.3])
def test_lattice_pairs_on_cell_boundaries(built_lib, rc, kernel):
    """Every in-cut pair of the lattice is found, however close to a cell boundary it sits."""
    case = lattice_case(ev_power=4.5 if kernel == "cells_generic" else 6.0)
    xc = CR.centred(case["x"])
    predicted = len(CR.stencil_misses(xc, rc)[0])
    assert predicted > 0  # the case still puts pairs two cells apart on a grid of edge rc
    eng = to_engine(case, cutoff=rc)
    if kernel == "cells_fast":
        eng.set_pair_kernel(1)
    e, f = eng.energy_forces()
    grid = eng.cell_grid()
    eng.close()
    sysd = to_oracle(case, cutoff=rc)
    n_ref = O.count_pairs(sysd, case["x"])
    assert grid["pairs"] == n_ref, (f"{kernel}: {n_ref - grid['pairs']} pairs inside the cut-off missed "
                                    f"({predicted} lie two cells apart on a grid of edge rc)")
    if kernel != "morton":
        assert grid["cell"] == float(CR.grid(xc, rc)[0]) and grid["cell"] > np.float32(rc)
    e_ref, f_ref = O.energy_forces(sysd, case["x"])
    _assert_energies(e, e_ref, kernel)
    assert force_rel_err(f, f_ref) <= F_TOL


def test_full_size_kernels_count_the_same_pairs(built_lib):
    """The genome-wide Hilbert start (N = 2e5, rc = 0.3 nm) has thousands of in-cut pairs on cell
    boundaries: the cell-list and Morton kernels on one handle count the same pairs, forces agree."""
    case = make_case(200000, n_chrom=22, seed=2024, terms=("EV", "SCB"), noise=0.0)
    eng = to_engine(case, cutoff=0.3)
    e_m, f_m = eng.energy_forces()
    p_m = eng.cell_grid()["pairs"]
    eng.set_pair_kernel(1)
    e_c, f_c = eng.energy_forces()
    p_c = eng.cell_grid()["pairs"]
    eng.close()
    assert p_c == p_m, ("cell-list kernel pairs short of the Morton kernel's", p_m - p_c)
    assert force_rel_err(f_c, f_m) <= F_TOL
    for t in range(3):
        assert abs(e_c[t] - e_m[t]) <= E_TOL * max(abs(e_m[t]), 1e-12), (O.TERM_NAMES[t], e_c[t], e_m[t])


@pytest.mark.parametrize("n", [2, 3, 31, 33, 255, 257, 1023])
def test_ragged_sizes_in_cutoff_mode(built_lib, n):
    terms = ("EV", "SCB", "CHB", "SC", "LAM", "CF", "BOND", "ANGLE") if n >= 40 else ("EV", "SCB", "CHB", "SC", "LAM", "CF")
    case = make_case(n, n_chrom=1 if n < 40 else 2, seed=n, terms=terms)
    rc = 0.25
    sysd = to_oracle(case, cutoff=rc)
    n_ref = O.count_pairs(sysd, case["x"])
    e_ref, f_ref = O.energy_forces(sysd, case["x"])
    for pref in (0, 1):  # Morton kernel, cell-list kernel
        eng = to_engine(case, cutoff=rc)
        eng.set_pair_kernel(pref)
        e, f = eng.energy_forces()
        assert eng.pair_kernel_in_use == 3
        grid = eng.cell_grid()
        order, keys = eng.cell_list()
        eng.close()
        assert grid["pairs"] == n_ref, (pref, grid["pairs"], n_ref)
        _assert_energies(e, e_ref, pref)
        assert force_rel_err(f, f_ref) <= F_TOL
        if pref == 1:
            keys_ref, order_ref, g = CR.cell_list(CR.centred(case["x"]), rc)
            assert (grid["cell"], grid["dim"], grid["origin"]) == (float(g[0]), g[1], float(g[2]))
            assert np.array_equal(order, order_ref) and np.array_equal(keys, keys_ref)


def _outlier_case():
    case = make_case(5000, n_chrom=2, seed=41, terms=("EV", "SCB", "BOND", "ANGLE"))
    case["x"] = case["x"].copy()
    case["x"][1234] += np.array([100.0, -60.0, 30.0])
    return case, 0.5


def _wide_case():
    case = make_case(8000, n_chrom=2, seed=43, terms=("EV", "SCB"))
    case["x"] = np.random.default_rng(43).uniform(-3.5, 3.5, size=(8000, 3))  # 7 nm across
    return case, 0.1


@pytest.mark.parametrize("build", [_outlier_case, _wide_case], ids=["outlier_100nm", "small_rc"])
def test_coarse_grid_branch(built_lib, build):
    """More than 64 cells of rc per axis: the grid becomes 64 cells of extent / 63."""
    case, rc = build()
    grid = _check_cells(case, rc, force_cells=True)
    xc = CR.centred(case["x"])
    extent = np.float32(np.float32(xc.max()) - np.float32(xc.min()))
    assert grid["dim"] == 64 and grid["cell"] == float(np.float32(extent / np.float32(63)))
    assert grid["pairs"] > 100


# ---- far field on cluster centroids ---------------------------------------------------------------

def _far_case(ev_power, chb):
    """~20 000 beads in chromosomes of 1-69 beads: ~1 300 clusters (5 chunks of 256 in k_cl_forces), among
    them one-bead clusters; n % 32 != 0 and n_clusters % 8 != 0."""
    n = 20011
    terms = ("EV", "CHB") if chb else ("EV",)
    case = make_case(n, n_chrom=1, seed=91, terms=terms, chb_de=5.0, ev_power=ev_power)
    rng = np.random.default_rng(92)
    chrom = np.zeros(n, np.int32)
    pos, cid = 0, 0
    while pos < n:
        ln = 1 if cid == 5 else int(rng.integers(1, 70))
        chrom[pos:pos + ln] = cid
        pos, cid = pos + ln, cid + 1
    case["chrom"] = chrom
    start, _ = FR.clusters(chrom)
    sizes = np.diff(start)
    assert n % 32 != 0 and len(sizes) > 3 * 256 and len(sizes) % 8 != 0 and sizes.min() == 1
    assert (np.bincount(chrom) < 32).any()
    return case


@pytest.mark.parametrize("ev_power,chb", [(6.0, True), (3.0, True), (6.0, False)], ids=["ev6_chb", "ev3_chb", "ev6_chb_off"])
def test_far_field_against_fp64_reference(built_lib, ev_power, chb):
    """Energies and per-bead forces of the far field against far_field_ref.

    Bars, from the FP64 arithmetic of both sides:
    * CHB (slot 3) is a sum of positive terms (kC R^4 - R^3 + R^2 > 0 for kC = 0.3); the device sums
      ~1.3e3 per cluster in a different order, with rsqrt good to a few ulp: relative error below ~1e-13.
      Held to 1e-11.
    * EV tail: e[0] with the surrogate minus e[0] without.  The truncated pass's slot leaves fixed point
      with the same bits both times (asserted), and k_finalize_energy adds it to ~ncl / 256 cluster
      slots and then 8 tree levels: at most ~16 roundings of size U |e_trunc + tail|, so the bar is
      1e-11 |tail| + 16 U (|e_trunc| + |tail|).
    * Force: with the surrogate, a bead's force is fl(truncated + cluster) and the truncated part alone
      is what the evaluation with CHB off returns, so their difference is the cluster force up to one
      rounding of the total (U |f_i|).  The cluster force itself is an FP64 sum over ~1.3e3 clusters;
      where neighbours cancel its error relative to max(|f_i|, RMS) stays near 1e-12.  Held to 1e-9 of
      max(|f_ref_i|, RMS |f_ref|), plus 4 U |f_i|."""
    case = _far_case(ev_power, chb)
    rc = 0.4
    ev = (100.0, 0.05, 0.1, ev_power)
    ref = FR.far_field(case["x"], case["chrom"], rc, ev, (0.3, 5.0) if chb else None)
    assert ref["n_below"] > 0 and ref["n_band"] > 0 and ref["n_above"] > 0, ref
    eng = to_engine(case, cutoff=rc)
    eng.set_chb_surrogate(True)
    e_s, f_s = eng.energy_forces()
    assert eng.pair_kernel_in_use == 3
    eng.set_chb_surrogate(False)
    e_p, f_p = eng.energy_forces()
    if chb:
        eng.set_pair_term("CHB", -1)
        e_c, f_c = eng.energy_forces()
        assert e_c[0] == e_p[0]  # the truncated pass gives the same bits with or without CHB
    else:
        e_c, f_c = e_p, f_p
    eng.close()
    if chb:
        assert abs(e_s[3] - ref["e_chb"]) <= 1e-11 * abs(ref["e_chb"]), (e_s[3], ref["e_chb"])
    else:
        assert e_s[3] == 0.0
    tail = e_s[0] - e_p[0]
    bar = 1e-11 * abs(ref["e_ev"]) + 16 * U * (abs(e_p[0]) + abs(ref["e_ev"]))
    assert abs(tail - ref["e_ev"]) <= bar, (tail, ref["e_ev"], bar)
    f_far = f_s - f_c
    f_ref = ref["force"]
    mag = np.linalg.norm(f_ref, axis=1)
    den = np.maximum(mag, np.sqrt((mag ** 2).mean()))
    err = np.linalg.norm(f_far - f_ref, axis=1)
    worst = int(np.argmax(err / (1e-9 * den + 4 * U * np.linalg.norm(f_s, axis=1))))
    assert (err <= 1e-9 * den + 4 * U * np.linalg.norm(f_s, axis=1)).all(), (worst, f_far[worst], f_ref[worst])


# ---- switching modes on one handle ----------------------------------------------------------------

def test_switching_modes_replays_fresh_handles(built_lib):
    """The two-stage minimisation switches one handle between exact mode, the Morton cut-off pass with and
    without the far field, and back, every round; the cell-list kernel shares d_keys, d_keys_tmp,
    d_order and d_cell_grid with the Morton pass at other sizes.  Every evaluation must be the bits of a
    fresh handle set up the same way."""
    case = make_case(5000, n_chrom=3, seed=61, terms=("EV", "SCB", "CHB", "BOND", "ANGLE"), chb_de=5.0)
    steps = [(0.0, False, 0), (0.5, False, 0), (0.5, True, 0), (0.5, False, 1), (0.3, False, 1),
             (0.3, False, 0), (0.3, True, 0), (0.0, False, 0)]
    eng = to_engine(case)
    for rc, far, kernel in steps:
        eng.set_cutoff(rc)
        eng.set_chb_surrogate(far)
        eng.set_pair_kernel(kernel)
        e, f = eng.energy_forces()
        got = [e, f]
        if rc > 0:
            got += [eng.cell_grid(), *eng.cell_list()]
        fresh = to_engine(case, cutoff=rc)
        fresh.set_chb_surrogate(far)
        fresh.set_pair_kernel(kernel)
        e0, f0 = fresh.energy_forces()
        want = [e0, f0]
        if rc > 0:
            want += [fresh.cell_grid(), *fresh.cell_list()]
        fresh.close()
        step = (rc, far, kernel)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), step
        if rc > 0:
            assert got[2] == want[2], (step, got[2], want[2])
            assert np.array_equal(got[3], want[3]) and np.array_equal(got[4], want[4]), step
    eng.close()
