"""mmm_contacts on the device against the numpy restatement (tests/contacts_ref.py), exactly: maps,
separation counts and totals, at the threshold, at full size; determinism and invariance; no side effects
on evaluations, minimisation or mmm_last_result; argument errors; the SAVE_CONTACTS driver paths."""
import os
import tarfile
import tempfile

import numpy as np
import pytest

import contacts_ref as R
from common import make_case, to_engine

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")
BED = os.path.join(GOLD, "synthetic_subcompartments.bed")


def _globule(n, seed=0, radius=None):
    """Random points in a ball at ~200 beads / nm^3 (about 7 contacts per bead at rc = 0.2 nm)."""
    rng = np.random.default_rng(seed)
    radius = radius or (3.0 * n / (4.0 * np.pi * 200.0)) ** (1.0 / 3.0)
    v = rng.normal(size=(n, 3))
    v *= (radius * rng.random(n) ** (1.0 / 3.0) / np.linalg.norm(v, axis=1))[:, None]
    return v + np.array([1.5, -0.7, 3.2])


def _engine(x, chrom=None):
    from multimm_b200.engine import Engine

    eng = Engine(len(x))
    if chrom is not None:
        eng.set_bead_params(chrom=np.asarray(chrom, np.int32))
    eng.set_positions(x)
    return eng


def _check(eng, x, rc, bins, n_bins, chrom):
    got = eng.contacts(rc, bins, n_bins)
    want = R.contact_counts(x, rc, bins, n_bins, chrom)
    if bins is not None:
        assert got[0].dtype == np.uint64 and np.array_equal(got[0], want[0])
    assert np.array_equal(got[1], want[1])
    assert got[2] == want[2]
    return got


@pytest.mark.parametrize("n,n_bins,with_chrom", [(3000, 97, True), (3000, 1, False), (2013, 4096, True),
                                                 (1000 + 7, 13, False), (33, 5, True)])
def test_kernel_matches_reference(built_lib, n, n_bins, with_chrom):
    rng = np.random.default_rng(n + n_bins)
    x = _globule(n, seed=n)
    bins = rng.integers(-1, n_bins, size=n).astype(np.int32)  # includes beads left out of the map
    chrom = np.repeat(np.arange(4), [n // 4, n // 3, n // 5, n - n // 4 - n // 3 - n // 5]) * 7 if with_chrom else None
    with _engine(x, chrom) as eng:
        for rc in (0.2, 0.35):
            cmap, sep, pairs = _check(eng, x, rc, bins, n_bins, chrom)
            assert pairs > n and np.array_equal(cmap, cmap.T)
            st = eng.contacts_stats()
            assert pairs <= st["candidates"] <= n * (n - 1) // 2 and st["device_ms"] > 0
        _check(eng, x, 0.2, None, 1, chrom)


def test_hilbert_lattice_at_the_threshold(built_lib):
    """Lattice neighbours sit at 0.1 nm: the FP64 verdict at rc = 0.1 and 0.1 (1 + 1e-12) decides each of them."""
    from multimm_b200.engine import Engine

    n = 6000
    with Engine(n) as eng:
        eng.hilbert_init(8, 0.1)
        x = eng.get_positions()
        bins = (np.arange(n) // 61).astype(np.int32)
        nb = int(bins.max()) + 1
        counts = []
        for rc in (0.1, 0.1 * (1 + 1e-12), 0.1 * (1 - 1e-12)):
            counts.append(_check(eng, x, rc, bins, nb, None)[2])
        assert counts[1] >= n - 1 and counts[1] > counts[0] >= counts[2]


def test_pairs_at_the_threshold_far_apart_in_index(built_lib):
    """Bead pairs placed at rc (1 -/+ 1e-12), in different tiles and stages, in a sparse cloud: a culling
    margin that is too tight would drop the inner ones."""
    rng = np.random.default_rng(3)
    n, rc = 4099, 0.2
    x = rng.uniform(-8.0, 8.0, size=(n, 3))
    for k, i in enumerate(range(0, 1800, 9)):
        j = n - 1 - i - 517 * (k % 3)
        u = rng.normal(size=3)
        u /= np.linalg.norm(u)
        x[j] = x[i] + u * rc * (1 - 1e-12 if k % 2 == 0 else 1 + 1e-12)
    i_ref, j_ref = R.contact_pairs(x, rc)
    with _engine(x) as eng:
        _check(eng, x, rc, (np.arange(n) % 41).astype(np.int32), 41, None)
    assert np.count_nonzero(j_ref - i_ref > 256) >= 80


def test_full_size_genome_wide_after_40_iterations(built_lib, tmp_path):
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    from multimm_b200 import contacts

    m = bench.build_model("gw", 0, 0, str(tmp_path))
    try:
        m.engine.minimize(tol=10.0, max_iter=40)
        x = m.engine.get_positions()
        gb = contacts.genome_bins(m.layout, 0, n_beads=len(x))
        chrom = m.chrom_spin.astype(np.int32)
        cmap, sep, pairs = _check(m.engine, x, 0.2, gb.bins, gb.n_bins, chrom)
        assert pairs > len(x) and int(sep.sum()) > 0
    finally:
        m.close()


def test_deterministic_and_invariant(built_lib):
    n = 3000
    case = make_case(n, n_chrom=4, seed=9)
    x, chrom, ce = case["x"], case["chrom"], case["chr_ends"]
    bins = (np.arange(n) * 50 // n).astype(np.int32)
    with _engine(x, chrom) as eng:
        a = eng.contacts(0.2, bins, 50)
        b = eng.contacts(0.2, bins, 50)
        assert all(np.array_equal(u, v) for u, v in zip(a[:2], b[:2])) and a[2] == b[2]
        assert eng.contacts(0.2, bins % 7, 7)[2] == a[2]  # another n_bins, the same contacts
    # whole chromosome blocks permuted, bins carried along: the same map and P(s) counts
    perm = np.concatenate([np.arange(ce[k], ce[k + 1]) for k in (2, 0, 3, 1)])
    with _engine(x[perm], chrom[perm]) as eng:
        c = eng.contacts(0.2, bins[perm], 50)
    assert np.array_equal(c[0], a[0]) and np.array_equal(c[1], a[1]) and c[2] == a[2]


@pytest.mark.parametrize("cutoff", [0.0, 1.2])
def test_no_side_effects_on_evaluation(built_lib, cutoff):
    case = make_case(3000, n_chrom=3, seed=4)
    bins = (np.arange(3000) // 100).astype(np.int32)
    ref = to_engine(case, cutoff=cutoff)
    eng = to_engine(case, cutoff=cutoff)
    try:
        for _ in range(2):
            e0, f0 = ref.energy_forces()
            e1, f1 = eng.energy_forces()
            assert np.array_equal(e0, e1) and np.array_equal(f0, f1)
            eng.contacts(0.3, bins, 30)
            le, lf = eng.last_result()  # still the evaluation before the contacts call
            assert np.array_equal(le, e1) and np.array_equal(lf, f1)
    finally:
        ref.close()
        eng.close()


def test_no_side_effects_on_minimisation(built_lib):
    case = make_case(3000, n_chrom=3, seed=5)
    bins = (np.arange(3000) // 100).astype(np.int32)
    ref, eng = to_engine(case), to_engine(case)
    try:
        r0 = ref.minimize(tol=10.0, max_iter=15)
        eng.contacts(0.2, bins, 30)
        r1 = eng.minimize(tol=10.0, max_iter=15)
        eng.contacts(0.2, bins, 30)
        assert r0["iterations"] == r1["iterations"] and r0["e_final"] == r1["e_final"]
        assert np.array_equal(ref.get_positions(), eng.get_positions())
        r0 = ref.minimize(tol=10.0, max_iter=10)
        r1 = eng.minimize(tol=10.0, max_iter=10)
        assert r0["e_final"] == r1["e_final"] and np.array_equal(ref.get_positions(), eng.get_positions())
    finally:
        ref.close()
        eng.close()


def test_argument_errors(built_lib):
    from multimm_b200.engine import Engine, Error

    n = 100
    x = _globule(n)
    with Engine(n) as eng:
        with pytest.raises(Error, match="positions"):
            eng.contacts(0.2, np.zeros(n, np.int32), 1)
        eng.set_positions(x)
        ok = np.zeros(n, np.int32)
        for rc in (0.0, -0.1, float("nan"), float("inf")):
            with pytest.raises(ValueError, match="rc"):
                eng.contacts(rc, ok, 1)
        for nb in (0, 4097):
            with pytest.raises(ValueError, match="n_bins"):
                eng.contacts(0.2, ok, nb)
        for bad in (-2, 5):
            b = ok.copy()
            b[37] = bad
            with pytest.raises(ValueError, match="bin id"):
                eng.contacts(0.2, b, 5)
        assert eng.contacts(0.2, np.full(n, -1, np.int32), 4)[0].sum() == 0


# ---- driver -------------------------------------------------------------------------------------------
def _ini(tmp_path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=3000, LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "out"), SAVE_PLOTS=False,
                SIM_RUN_MD=False, MIN_MAX_ITERATIONS=150, SAVE_CONTACTS=True)
    base.update(fields)
    path = tmp_path / "config.ini"
    path.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items()))
    return str(path), base["OUT_PATH"]


KEYS = ("counts", "members", "radius_nm", "resolution_bp", "bin_chrom", "bin_start_bp", "sep_contacts", "sep_pairs",
        "pairs")


def test_single_run_writes_contacts(built_lib, tmp_path):
    from multimm_b200 import cif, contacts, run

    ini, out = _ini(tmp_path, COMPARTMENT_PATH=BED, SCB_USE_SUBCOMPARTMENT_BLOCKS=True, SHUFFLE_CHROMS=True)
    assert run.main(["-c", ini]) == 0
    d = contacts.load(os.path.join(out, "analysis", "contacts.npz"))
    assert set(KEYS) <= set(d) and int(d["members"]) == 1 and float(d["radius_nm"]) == 0.2
    assert d["counts"].dtype == np.uint64 and np.array_equal(d["counts"], d["counts"].T)
    assert d["counts"].shape[0] <= 1000 and int(d["pairs"]) > 3000
    x = cif.read_cif_coordinates(os.path.join(out, "model/MultiMM_minimized.cif"), include_hetatm=True) / 10.0
    _, _, pairs = R.contact_counts(x, 0.2)
    assert abs(pairs - int(d["pairs"])) <= R.near_threshold_pairs(x, 0.2, 2e-5)


def _ensemble(tmp_path, n, devices, name):
    from multimm_b200 import run

    d = tmp_path / name
    d.mkdir()
    ini, out = _ini(d, N_BEADS=4000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=n, SHUFFLE_CHROMS=True, COMPARTMENT_PATH=BED,
                    SCB_USE_SUBCOMPARTMENT_BLOCKS=True, MIN_MAX_ITERATIONS=100)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=devices)
    return out


def test_ensemble_contacts_sum_members_and_match_reference(built_lib, tmp_path):
    from multimm_b200 import cif, contacts, loaders

    out = _ensemble(tmp_path, 3, [0], "e1")
    ens = contacts.load(os.path.join(out, "ensemble_contacts.npz"))
    members = [contacts.load(os.path.join(out, "contacts", f"member_{i}.npz")) for i in range(3)]
    assert int(ens["members"]) == 3
    assert np.array_equal(ens["counts"], sum(m["counts"] for m in members))
    assert np.array_equal(ens["sep_contacts"], sum(m["sep_contacts"] for m in members))
    assert int(ens["pairs"]) == sum(int(m["pairs"]) for m in members)
    assert np.array_equal(ens["counts"], ens["counts"].T)
    for i, m in enumerate(members):
        # the member's bins rebuilt from its loaders; its map against numpy on the minimised CIF read back
        lay = {}
        loaders.import_mns_from_bedpe(BEDPE, N_beads=4000, path=None, shuffle=True, seed=i, layout=lay)
        gb = contacts.genome_bins(lay, int(m["resolution_bp"]), n_beads=4000)
        assert np.array_equal(gb.bin_start_bp, m["bin_start_bp"])
        with tarfile.open(os.path.join(out, f"run_{i}.tar.gz")) as t, tempfile.TemporaryDirectory() as td:
            t.extract(f"run_{i}/model/MultiMM_minimized.cif", td)
            x = cif.read_cif_coordinates(os.path.join(td, f"run_{i}/model/MultiMM_minimized.cif"), include_hetatm=True) / 10.0
        cmap, _, pairs = R.contact_counts(x, 0.2, gb.bins, gb.n_bins)
        amb = R.near_threshold_pairs(x, 0.2, 2e-5)  # the only pairs the CIF's 1e-5 nm rounding can flip
        assert abs(pairs - int(m["pairs"])) <= amb
        diff = np.abs(cmap.astype(np.int64) - m["counts"].astype(np.int64))
        assert int(np.triu(diff).sum()) <= amb


def test_ensemble_contacts_same_bits_on_two_gpus(built_lib, tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from multimm_b200 import contacts

    one = contacts.load(os.path.join(_ensemble(tmp_path, 4, [0], "g1"), "ensemble_contacts.npz"))
    two = contacts.load(os.path.join(_ensemble(tmp_path, 4, [0, 1], "g2"), "ensemble_contacts.npz"))
    for k in KEYS:
        assert one[k].dtype == two[k].dtype and one[k].tobytes() == two[k].tobytes(), k
