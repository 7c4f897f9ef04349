"""mmm_contacts_sparse on the device against the numpy restatement (contacts_ref.contact_pairs, then
np.unique of the packed keys), exactly: random globules over several bin sets up to 62-bit keys, the
Hilbert lattice at the threshold, full size; the dense map of mmm_contacts at the same positions;
determinism, scratch growth and no side effects; argument and state errors; the fine-map driver paths."""
import os
import tarfile
import tempfile

import numpy as np
import pytest

import contacts_ref as R
from common import make_case, to_engine

pytestmark = pytest.mark.gpu

MMM_ERR_STATE = -3  # include/multimm_b200.h
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


def _engine(x):
    from multimm_b200.engine import Engine

    eng = Engine(len(x))
    eng.set_positions(x)
    return eng


def sparse_ref(x, rc, bins, n_bins):
    """(rows, cols, vals, pairs) of the sparse map, restated in numpy."""
    i, j = R.contact_pairs(x, rc)
    bins = np.asarray(bins, np.int64)
    bi, bj = bins[i], bins[j]
    ok = (bi >= 0) & (bj >= 0)
    p, q = np.minimum(bi[ok], bj[ok]), np.maximum(bi[ok], bj[ok])
    keys, vals = np.unique(p * np.int64(n_bins) + q, return_counts=True)
    return ((keys // n_bins).astype(np.int32), (keys % n_bins).astype(np.int32), vals.astype(np.uint64),
            int(len(i)))


def _check(eng, x, rc, bins, n_bins):
    got = eng.contacts_sparse(rc, bins, n_bins)
    want = sparse_ref(x, rc, bins, n_bins)
    assert got[0].dtype == np.int32 and got[1].dtype == np.int32 and got[2].dtype == np.uint64
    for g, w in zip(got[:3], want[:3]):
        assert np.array_equal(g, w)
    assert got[3] == want[3]
    return got


def _bin_sets(n, rng):
    """bins = bead index, coarse sets, blocks shuffled (bins not monotone in bead index), a huge n_bins."""
    yield np.arange(n, dtype=np.int32), n
    for nb in (1, 7, 300):
        yield (np.arange(n) * nb // n).astype(np.int32), nb
    blocks = rng.permutation(64)
    yield blocks[np.arange(n) * 64 // n].astype(np.int32), 64
    big = 2**31 - 1
    ids = rng.choice(np.int64(big), size=97, replace=False)
    yield ids[rng.integers(0, 97, size=n)].astype(np.int32), big


@pytest.mark.parametrize("n,left_out", [(33, False), (1000 + 7, True), (3000, False), (12_345, True)])
def test_kernel_matches_reference(built_lib, n, left_out):
    rng = np.random.default_rng(n)
    x = _globule(n, seed=n)
    with _engine(x) as eng:
        for bins, nb in _bin_sets(n, rng):
            if left_out:
                bins = np.where(rng.random(n) < 0.1, -1, bins).astype(np.int32)
            for rc in (0.2, 0.35):
                rows, cols, vals, pairs = _check(eng, x, rc, bins, nb)
                assert np.all(rows <= cols) and np.all(vals > 0)
                st = eng.contacts_stats()
                assert pairs <= st["candidates"] and st["device_ms"] > 0


def test_hilbert_lattice_at_the_threshold(built_lib):
    from multimm_b200.engine import Engine

    n = 6000
    with Engine(n) as eng:
        eng.hilbert_init(8, 0.1)
        x = eng.get_positions()
        counts = []
        for rc in (0.1, 0.1 * (1 + 1e-12), 0.1 * (1 - 1e-12)):
            counts.append(_check(eng, x, rc, np.arange(n, dtype=np.int32), n)[3])
            _check(eng, x, rc, (np.arange(n) // 61).astype(np.int32), (n - 1) // 61 + 1)
        assert counts[1] >= n - 1 and counts[1] > counts[0] >= counts[2]


def test_full_size_genome_wide_after_40_iterations(built_lib, tmp_path):
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    m = bench.build_model("gw", 0, 0, str(tmp_path))
    try:
        m.engine.minimize(tol=10.0, max_iter=40)
        x = m.engine.get_positions()
        n = len(x)
        rows, cols, vals, pairs = _check(m.engine, x, 0.2, np.arange(n, dtype=np.int32), n)
        assert pairs > n and len(vals) == pairs and np.all(vals == 1)  # bead bins: the entries are the pairs
    finally:
        m.close()


def _densify(rows, cols, vals, nb):
    d = np.zeros((nb, nb), np.uint64)
    d[rows, cols] = vals
    d[cols, rows] = vals
    return d


def test_equals_dense_map(built_lib):
    n = 5000
    rng = np.random.default_rng(11)
    x = _globule(n, seed=11)
    with _engine(x) as eng:
        for nb in (1, 13, 500, 4096):
            bins = rng.integers(-1, nb, size=n).astype(np.int32)
            cmap, _, dpairs = eng.contacts(0.25, bins, nb)
            rows, cols, vals, pairs = eng.contacts_sparse(0.25, bins, nb)
            assert pairs == dpairs
            assert np.array_equal(_densify(rows, cols, vals, nb), cmap)


def test_deterministic_scratch_growth_and_empty(built_lib):
    n = 4000
    x = _globule(n, seed=3)
    bins = np.arange(n, dtype=np.int32)
    with _engine(x) as eng:
        a = eng.contacts_sparse(0.15, bins, n)
        b = eng.contacts_sparse(0.15, bins, n)
        assert all(u.tobytes() == v.tobytes() for u, v in zip(a[:3], b[:3])) and a[3] == b[3]
        big = _check(eng, x, 0.4, bins, n)  # more contacts than before: the scratch grows
        assert big[3] > 4 * a[3]
        _check(eng, x, 0.15, bins, n)       # and serves a smaller call again
        rows, cols, vals, pairs = eng.contacts_sparse(1e-6, bins, n)
        assert pairs == 0 and len(rows) == len(cols) == len(vals) == 0
        rows, cols, vals, pairs = eng.contacts_sparse(0.2, np.full(n, -1, np.int32), 5)
        assert pairs > 0 and len(vals) == 0


@pytest.mark.parametrize("cutoff", [0.0, 1.2])
def test_no_side_effects_on_evaluation(built_lib, cutoff):
    case = make_case(3000, n_chrom=3, seed=4)
    bins = np.arange(3000, dtype=np.int32)
    ref = to_engine(case, cutoff=cutoff)
    eng = to_engine(case, cutoff=cutoff)
    try:
        for _ in range(2):
            e0, f0 = ref.energy_forces()
            e1, f1 = eng.energy_forces()
            assert np.array_equal(e0, e1) and np.array_equal(f0, f1)
            eng.contacts_sparse(0.3, bins, 3000)
            le, lf = eng.last_result()
            assert np.array_equal(le, e1) and np.array_equal(lf, f1)
    finally:
        ref.close()
        eng.close()


def test_no_side_effects_on_minimisation(built_lib):
    case = make_case(3000, n_chrom=3, seed=5)
    bins = np.arange(3000, dtype=np.int32)
    ref, eng = to_engine(case), to_engine(case)
    try:
        r0 = ref.minimize(tol=10.0, max_iter=15)
        eng.contacts_sparse(0.2, bins, 3000)
        r1 = eng.minimize(tol=10.0, max_iter=15)
        eng.contacts_sparse(0.2, bins, 3000)
        assert r0["iterations"] == r1["iterations"] and r0["e_final"] == r1["e_final"]
        assert np.array_equal(ref.get_positions(), eng.get_positions())
        r0 = ref.minimize(tol=10.0, max_iter=10)
        r1 = eng.minimize(tol=10.0, max_iter=10)
        assert r0["e_final"] == r1["e_final"] and np.array_equal(ref.get_positions(), eng.get_positions())
    finally:
        ref.close()
        eng.close()


def test_argument_and_state_errors(built_lib):
    import ctypes as C

    from multimm_b200 import _lib
    from multimm_b200.engine import Engine, Error

    n = 100
    x = _globule(n)
    ok = np.zeros(n, np.int32)
    with Engine(n) as eng:
        lib = _lib.load()
        assert lib.mmm_contacts_sparse_read(eng._h, None, None, None) == MMM_ERR_STATE
        with pytest.raises(Error, match="positions"):
            eng.contacts_sparse(0.2, ok, 1)
        eng.set_positions(x)
        for rc in (0.0, -0.1, float("nan"), float("inf")):
            with pytest.raises(ValueError, match="rc"):
                eng.contacts_sparse(rc, ok, 1)
        for nb in (0, -5):
            with pytest.raises(ValueError, match="n_bins"):
                eng.contacts_sparse(0.2, ok, nb)
        for bad in (-2, 5):
            b = ok.copy()
            b[37] = bad
            with pytest.raises(ValueError, match="bin id"):
                eng.contacts_sparse(0.2, b, 5)
        assert lib.mmm_contacts_sparse_read(eng._h, None, None, None) == MMM_ERR_STATE  # failed calls only
        e, p = C.c_int64(), C.c_int64()
        assert lib.mmm_contacts_sparse(eng._h, 0.2, ok.ctypes.data_as(C.c_void_p), 1, C.byref(e), C.byref(p)) == 0
        assert e.value == 1 and p.value > 0
        assert lib.mmm_contacts_sparse_read(eng._h, None, None, None) == 0


# ---- driver -------------------------------------------------------------------------------------------
def _ini(tmp_path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=3000, LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "out"), SAVE_PLOTS=False,
                SIM_RUN_MD=False, MIN_MAX_ITERATIONS=150, SAVE_CONTACTS=True)
    base.update(fields)
    path = tmp_path / "config.ini"
    path.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items()))
    return str(path), base["OUT_PATH"]


def test_single_run_writes_fine_and_dense(built_lib, tmp_path):
    from multimm_b200 import cif, contacts, run

    ini, out = _ini(tmp_path, COMPARTMENT_PATH=BED, SCB_USE_SUBCOMPARTMENT_BLOCKS=True, SHUFFLE_CHROMS=True,
                    CONTACT_RESOLUTION=5_000_000, CONTACT_FINE_RESOLUTION=50_000)
    assert run.main(["-c", ini]) == 0
    dense = contacts.load(os.path.join(out, "analysis", "contacts.npz"))
    fine = contacts.load_fine(os.path.join(out, "analysis", "contacts_fine.npz"))
    assert set(fine) == set(contacts.FINE_KEYS) and int(fine["resolution_bp"]) == 50_000
    assert int(fine["n_bins"]) > contacts.MAX_BINS and int(fine["pairs"]) == int(dense["pairs"])
    assert np.array_equal(contacts.coarsen(fine, 5_000_000), dense["counts"])
    with pytest.raises(ValueError, match="load_fine"):
        contacts.load(os.path.join(out, "analysis", "contacts_fine.npz"))
    x = cif.read_cif_coordinates(os.path.join(out, "model/MultiMM_minimized.cif"), include_hetatm=True) / 10.0
    _, _, pairs = R.contact_counts(x, 0.2)
    assert abs(pairs - int(fine["pairs"])) <= R.near_threshold_pairs(x, 0.2, 2e-5)


def _ensemble(tmp_path, n, devices, name):
    from multimm_b200 import run

    d = tmp_path / name
    d.mkdir()
    ini, out = _ini(d, N_BEADS=4000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=n, SHUFFLE_CHROMS=True, COMPARTMENT_PATH=BED,
                    SCB_USE_SUBCOMPARTMENT_BLOCKS=True, MIN_MAX_ITERATIONS=100, CONTACT_FINE_RESOLUTION=20_000)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=devices)
    return out


def _signed_sum(maps, nb):
    """Union of sparse maps (rows, cols, vals, sign) as (keys, int64 sums); never dense (~1.6e5 bins here)."""
    keys = np.concatenate([r.astype(np.int64) * nb + c for r, c, _, _ in maps])
    vals = np.concatenate([sg * v.astype(np.int64) for _, _, v, sg in maps])
    u, inv = np.unique(keys, return_inverse=True)
    out = np.zeros(len(u), np.int64)
    np.add.at(out, inv, vals)
    return u, out


def test_ensemble_fine_sums_members_and_matches_reference(built_lib, tmp_path):
    from multimm_b200 import cif, contacts, loaders

    out = _ensemble(tmp_path, 3, [0], "e1")
    ens = contacts.load_fine(os.path.join(out, "ensemble_contacts_fine.npz"))
    members = [contacts.load_fine(os.path.join(out, "contacts", f"member_{i}_fine.npz")) for i in range(3)]
    nb = int(ens["n_bins"])
    assert nb > contacts.MAX_BINS
    assert int(ens["members"]) == 3 and int(ens["pairs"]) == sum(int(m["pairs"]) for m in members)
    keys, total = _signed_sum([(m["rows"], m["cols"], m["vals"], 1) for m in members], nb)
    assert np.array_equal(ens["rows"].astype(np.int64) * nb + ens["cols"], keys)
    assert np.array_equal(ens["vals"].astype(np.int64), total)
    for i, m in enumerate(members):
        lay = {}
        loaders.import_mns_from_bedpe(BEDPE, N_beads=4000, path=None, shuffle=True, seed=i, layout=lay)
        gb = contacts.genome_bins(lay, 20_000, n_beads=4000, max_bins=contacts.MAX_FINE_BINS)
        assert np.array_equal(gb.bin_start_bp, m["bin_start_bp"])
        with tarfile.open(os.path.join(out, f"run_{i}.tar.gz")) as t, tempfile.TemporaryDirectory() as td:
            t.extract(f"run_{i}/model/MultiMM_minimized.cif", td)
            x = cif.read_cif_coordinates(os.path.join(td, f"run_{i}/model/MultiMM_minimized.cif"), include_hetatm=True) / 10.0
        rows, cols, vals, pairs = sparse_ref(x, 0.2, gb.bins, gb.n_bins)
        amb = R.near_threshold_pairs(x, 0.2, 2e-5)  # the only pairs the CIF's 1e-5 nm rounding can flip
        assert abs(pairs - int(m["pairs"])) <= amb
        _, diff = _signed_sum([(rows, cols, vals, 1), (m["rows"], m["cols"], m["vals"], -1)], nb)
        assert int(np.abs(diff).sum()) <= amb


def test_ensemble_fine_same_bits_on_two_gpus(built_lib, tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from multimm_b200 import contacts

    one = contacts.load_fine(os.path.join(_ensemble(tmp_path, 4, [0], "g1"), "ensemble_contacts_fine.npz"))
    two = contacts.load_fine(os.path.join(_ensemble(tmp_path, 4, [0, 1], "g2"), "ensemble_contacts_fine.npz"))
    for k in contacts.FINE_KEYS:
        assert one[k].dtype == two[k].dtype and one[k].tobytes() == two[k].tobytes(), k
