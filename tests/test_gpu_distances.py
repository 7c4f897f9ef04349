"""mmm_distance_map on the device against the numpy restatement (tests/distances_ref.py), exactly: random
globules and the Hilbert lattice over bead, coarse, shuffled, random and partial bin sets; exact coarsening;
the FP32 mean pair distance; the full genome-wide model; determinism, no side effects on evaluations,
minimisation or mmm_last_result; argument, state and overflow-guard errors; the SAVE_DISTANCES driver
paths."""
import os
import tarfile
import tempfile

import numpy as np
import pytest

import distances_ref as R
from common import make_case, to_engine

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")
BED = os.path.join(GOLD, "synthetic_subcompartments.bed")


def _globule(n, seed=0):
    """Random points in a ball at ~200 beads / nm^3, off the origin."""
    rng = np.random.default_rng(seed)
    radius = (3.0 * n / (4.0 * np.pi * 200.0)) ** (1.0 / 3.0)
    v = rng.normal(size=(n, 3))
    v *= (radius * rng.random(n) ** (1.0 / 3.0) / np.linalg.norm(v, axis=1))[:, None]
    return v + np.array([1.5, -0.7, 3.2])


def _engine(x):
    from multimm_b200.engine import Engine

    eng = Engine(len(x))
    eng.set_positions(x)
    return eng


def _bin_sets(n, seed):
    """name -> (bins, n_bins): bead level (n <= 4096), one bin, 7 and 300 contiguous bins, shuffled blocks of
    contiguous bins, random ids, and 10 % of beads left out."""
    rng = np.random.default_rng(seed)
    out = {}
    if n <= 4096:
        out["bead"] = (np.arange(n, dtype=np.int32), n)
    for nb in (1, 7, 300):
        out[f"blocks{nb}"] = ((np.arange(n) * nb // n).astype(np.int32), nb)
    perm = rng.permutation(300)
    out["shuffled"] = (perm[np.arange(n) * 300 // n].astype(np.int32), 300)
    out["random"] = (rng.integers(0, 97, size=n).astype(np.int32), 97)
    left = (np.arange(n) * 50 // n).astype(np.int32)
    left[rng.random(n) < 0.1] = -1
    out["partial"] = (left, 50)
    return out


def _check(eng, x, bins, nb):
    got = eng.distance_map(bins, nb)
    want = R.distance_sums(x, bins, nb)
    for g, w in zip(got, want):
        assert g.dtype == np.uint64 and g.shape == (nb, nb)
        assert np.array_equal(g, w)
    return got


@pytest.mark.parametrize("n", [33, 1007, 3000])
def test_kernel_matches_reference(built_lib, n):
    x = _globule(n, seed=n)
    with _engine(x) as eng:
        for name, (bins, nb) in _bin_sets(n, n).items():
            d, d2 = _check(eng, x, bins, nb)
            assert np.array_equal(d, d.T) and np.array_equal(d2, d2.T), name
            assert eng.distance_stats()["device_ms"] > 0


def test_kernel_matches_reference_12345(built_lib):
    n = 12345  # not a multiple of 32: a partial last tile; more than 4096 beads: no bead-level map
    x = _globule(n, seed=5)
    sets = _bin_sets(n, 7)
    with _engine(x) as eng:
        for name in ("blocks7", "shuffled", "partial"):
            _check(eng, x, *sets[name])
        # the others against the restatement on sampled entries
        for name in ("blocks1", "blocks300", "random"):
            bins, nb = sets[name]
            d, d2 = eng.distance_map(bins, nb)
            rng = np.random.default_rng(len(name))
            for p, q in [(0, 0), (nb - 1, 0)] + [tuple(rng.integers(0, nb, 2)) for _ in range(6)]:
                assert (int(d[p, q]), int(d2[p, q])) == R.block_sums(x, bins, p, q), (name, p, q)


def test_hilbert_lattice_ties(built_lib):
    """On the 0.1 nm lattice many pairs sit at exactly equal distances (and d2 values with .5 ties after
    scaling are possible): the rounding must agree for every one."""
    from multimm_b200.engine import Engine

    n = 3000
    with Engine(n) as eng:
        eng.hilbert_init(8, 0.1)
        x = eng.get_positions()
        for bins, nb in ((np.arange(n, dtype=np.int32), n), ((np.arange(n) // 61).astype(np.int32), 50)):
            _check(eng, x, bins, nb)


def test_coarsening_is_exact(built_lib):
    n = 2500
    x = _globule(n, seed=11)
    rng = np.random.default_rng(2)
    with _engine(x) as eng:
        fine = eng.distance_map(np.arange(n, dtype=np.int32), n)
        totals = set()
        for nb in (1, 13, 250, 2500):
            cmap = rng.permutation(n) % nb  # any bead -> bin mapping
            coarse = eng.distance_map(cmap.astype(np.int32), nb)
            for f, c in zip(fine, coarse):
                want = np.zeros((nb, nb), np.uint64)
                # every ordered bead pair (i, j) into (bin_i, bin_j): an off-diagonal entry receives each of its
                # pairs once, a diagonal entry each of its pairs twice, where the device map holds it once
                np.add.at(want, (cmap[:, None], cmap[None, :]), f)
                want[np.diag_indices(nb)] //= np.uint64(2)
                assert np.array_equal(c, want)
            totals.add(int(np.triu(coarse[0]).sum(dtype=np.uint64)))
        assert len(totals) == 1 and totals == {int(np.triu(fine[0]).sum(dtype=np.uint64))}


def test_cross_check_with_fp32_mean_pair_distance(built_lib):
    n = 5000
    x = _globule(n, seed=3)
    with _engine(x) as eng:
        d, _ = eng.distance_map(np.zeros(n, np.int32), 1)
        mean = 2.0 * 2.0 ** -24 * float(int(d[0, 0])) / (n * n)
        assert abs(mean / eng.mean_pair_distance() - 1.0) < 1e-5


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
        d, d2 = m.engine.distance_map(gb.bins, gb.n_bins)  # the overflow guard stays silent
        assert np.array_equal(d, d.T) and np.array_equal(d2, d2.T)
        rng = np.random.default_rng(0)
        occupied = np.flatnonzero(np.bincount(gb.bins, minlength=gb.n_bins) > 1)
        pairs = [(p, p) for p in occupied[:8]] + [tuple(rng.choice(occupied, 2)) for _ in range(56)]
        for p, q in pairs:
            assert (int(d[p, q]), int(d2[p, q])) == R.block_sums(x, gb.bins, p, q), (p, q)
        assert np.all(np.diag(d)[occupied] > 0)
    finally:
        m.close()


def test_deterministic_and_scratch_growth(built_lib):
    n = 3000
    x = _globule(n, seed=8)
    bins = (np.arange(n) * 40 // n).astype(np.int32)
    with _engine(x) as eng:
        a = eng.distance_map(bins, 40)
        big = eng.distance_map(np.arange(n, dtype=np.int32), n)  # grows the maps
        b = eng.distance_map(bins, 40)  # a smaller map in the grown scratch
        c = eng.distance_map(bins, 40)
        assert all(np.array_equal(u, v) and np.array_equal(u, w) for u, v, w in zip(a, b, c))
        assert int(np.triu(big[0]).sum(dtype=np.uint64)) == int(np.triu(a[0]).sum(dtype=np.uint64))


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
            eng.distance_map(bins, 30)
            le, lf = eng.last_result()  # still the evaluation before the distance call
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
        eng.distance_map(bins, 30)
        r1 = eng.minimize(tol=10.0, max_iter=15)
        eng.distance_map(bins, 30)
        assert r0["iterations"] == r1["iterations"] and r0["e_final"] == r1["e_final"]
        assert np.array_equal(ref.get_positions(), eng.get_positions())
        r0 = ref.minimize(tol=10.0, max_iter=10)
        r1 = eng.minimize(tol=10.0, max_iter=10)
        assert r0["e_final"] == r1["e_final"] and np.array_equal(ref.get_positions(), eng.get_positions())
    finally:
        ref.close()
        eng.close()


def test_argument_state_and_overflow_errors(built_lib):
    from multimm_b200 import distances
    from multimm_b200.engine import Engine, Error

    n = 100
    x = _globule(n)
    ok = np.zeros(n, np.int32)
    with Engine(n) as eng:
        with pytest.raises(Error, match="positions"):
            eng.distance_map(ok, 1)
        eng.set_positions(x)
        for nb in (0, 4097):
            with pytest.raises(ValueError, match="n_bins"):
                eng.distance_map(ok, nb)
        for bad in (-2, 5):
            b = ok.copy()
            b[37] = bad
            with pytest.raises(ValueError, match="bin id"):
                eng.distance_map(b, 5)
        with pytest.raises(ValueError, match="shape"):
            eng.distance_map(ok[:-1], 1)
        d, d2 = eng.distance_map(np.full(n, -1, np.int32), 4)
        assert d.sum() == 0 and d2.sum() == 0
    # far spread: 100 beads over 2e4 nm (about 2e16 Q nm^2 per pair) at B = 1, 4950 pairs in one entry, would
    # overflow int64: refused, not wrapped
    far = np.random.default_rng(1).uniform(-1e4, 1e4, size=(n, 3))
    with pytest.raises(ValueError, match="overflow"):
        distances.distance_sums(far, ok, 1)
    # the same spread over bead-level bins fits (one pair per entry)
    d, d2 = distances.distance_sums(far[:40], np.arange(40, dtype=np.int32), 40)
    want = R.distance_sums(far[:40], np.arange(40), 40)
    assert np.array_equal(d, want[0]) and np.array_equal(d2, want[1])


# ---- driver -------------------------------------------------------------------------------------------
def _ini(tmp_path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=3000, LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "out"), SAVE_PLOTS=False,
                SIM_RUN_MD=False, MIN_MAX_ITERATIONS=150, SAVE_DISTANCES=True)
    base.update(fields)
    for k in [k for k, v in base.items() if v is None]:
        del base[k]
    path = tmp_path / "config.ini"
    path.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items()))
    return str(path), base["OUT_PATH"]


def _means_match_cif(d, x, bins):
    """Mean distances of a member file against numpy on the CIF positions: within the CIF's rounding
    (coordinates to 1e-4 Angstrom, 5e-6 nm each: at most 1.8e-5 nm on a distance)."""
    from multimm_b200 import distances

    nb = len(d["bin_beads"])
    ds, d2s = R.distance_sums(x, bins, nb)
    ref = dict(d, dist_sum=ds, dist2_sum=d2s)
    got, want = distances.mean_distance(d), distances.mean_distance(ref)
    ok = ~np.isnan(want)
    assert np.array_equal(ok, ~np.isnan(got)) and ok.sum() > 0
    assert np.max(np.abs(got[ok] - want[ok])) <= 2e-5


def test_single_run_writes_distances(built_lib, tmp_path):
    from multimm_b200 import cif, contacts, distances, loaders, run

    ini, out = _ini(tmp_path, COMPARTMENT_PATH=BED, SCB_USE_SUBCOMPARTMENT_BLOCKS=True, SHUFFLE_CHROMS=True,
                    DISTANCE_RESOLUTION=2_000_000)
    assert run.main(["-c", ini]) == 0
    d = distances.load(os.path.join(out, "analysis", "distances.npz"))
    assert int(d["members"]) == 1 and int(d["quantum_log2"]) == -24 and int(d["resolution_bp"]) == 2_000_000
    assert d["dist_sum"].dtype == np.uint64 and np.array_equal(d["dist_sum"], d["dist_sum"].T)
    assert int(d["bin_beads"].sum()) == 3000
    assert not os.path.exists(os.path.join(out, "analysis", "contacts.npz"))
    x = cif.read_cif_coordinates(os.path.join(out, "model/MultiMM_minimized.cif"), include_hetatm=True) / 10.0
    lay = {}
    loaders.import_mns_from_bedpe(BEDPE, N_beads=3000, path=None, shuffle=True, seed=0, layout=lay)
    gb = contacts.genome_bins(lay, 2_000_000, n_beads=3000)
    assert np.array_equal(gb.bin_start_bp, d["bin_start_bp"])
    _means_match_cif(d, x, gb.bins)
    mean, std = distances.radial_profile(d)
    assert np.all(np.isfinite(mean[d["bin_beads"] > 0])) and np.all(std[d["bin_beads"] > 0] >= 0)


def test_ensemble_writes_member_and_summed_distances(built_lib, tmp_path):
    from multimm_b200 import cif, contacts, distances, loaders, run

    d = tmp_path / "e"
    d.mkdir()
    ini, out = _ini(d, N_BEADS=4000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=3, SHUFFLE_CHROMS=True, COMPARTMENT_PATH=BED,
                    SCB_USE_SUBCOMPARTMENT_BLOCKS=True, MIN_MAX_ITERATIONS=100)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=[0])
    paths = [os.path.join(out, "distances", f"member_{i}.npz") for i in range(3)]
    ens = distances.load(os.path.join(out, "ensemble_distances.npz"))
    agg = distances.aggregate(paths[::-1])
    for k in distances.KEYS:
        assert ens[k].dtype == agg[k].dtype and ens[k].tobytes() == agg[k].tobytes(), k
    assert int(ens["members"]) == 3
    for i in range(3):
        m = distances.load(paths[i])
        lay = {}
        loaders.import_mns_from_bedpe(BEDPE, N_beads=4000, path=None, shuffle=True, seed=i, layout=lay)
        gb = contacts.genome_bins(lay, int(m["resolution_bp"]), n_beads=4000)
        with tarfile.open(os.path.join(out, f"run_{i}.tar.gz")) as t, tempfile.TemporaryDirectory() as td:
            names = t.getnames()
            assert not any("distances" in s for s in names)  # the member file lives outside the archive
            t.extract(f"run_{i}/model/MultiMM_minimized.cif", td)
            x = cif.read_cif_coordinates(os.path.join(td, f"run_{i}/model/MultiMM_minimized.cif"), include_hetatm=True) / 10.0
        _means_match_cif(m, x, gb.bins)


def test_run_without_the_settings_writes_no_distance_files(built_lib, tmp_path):
    from multimm_b200 import run

    ini, out = _ini(tmp_path, SAVE_DISTANCES=None, MIN_MAX_ITERATIONS=20)
    assert run.main(["-c", ini]) == 0
    written = [os.path.join(r, f) for r, _, fs in os.walk(out) for f in fs]
    assert written and not any("distances" in p for p in written)
