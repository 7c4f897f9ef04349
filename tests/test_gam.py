"""Genome architecture mapping on the host: the numpy restatement (tests/gam_ref.py) against brute force, beads on
the slab boundary, the diagonal and the bounds of the co-segregation table, invariance under bead order within a
bin, the slice geometry of gam.slice_planes, the GAM file format, its exact aggregation, the readers (D, D', NPMI)
on hand-built tables, and the SAVE_GAM / GAM_RESOLUTION / GAM_SLICES / GAM_SLICE_FRACTION settings."""
import os

import numpy as np
import pytest

import gam_ref as GR
from multimm_b200 import contacts, gam, loaders
from triplets_ref import globule

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


def _gb(n=4000, res=20_000_000):
    lay = {}
    loaders.import_mns_from_bedpe(BEDPE, N_beads=n, chrom=None, coords=None, path=None, shuffle=False, seed=0,
                                  layout=lay)
    return contacts.genome_bins(lay, res, n_beads=n)


def _planes(x, bins, count, fraction, seed):
    return gam.slice_planes(x, np.zeros(3), bins, count, fraction, np.random.default_rng(seed))


# ---- the restatement -------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,nb,count,seed", [(1, 1, 5, 0), (40, 6, 33, 1), (90, 9, 64, 2)])
def test_restatement_equals_brute_force(n, nb, count, seed):
    rng = np.random.default_rng(seed)
    x = globule(n, 30, seed)
    bins = rng.integers(-1, nb, size=n).astype(np.int32)
    bins[0] = 0
    planes, h = _planes(x, bins, count, 0.2, seed)
    planes[::3, :3] *= 2.5  # normals need not be unit length
    c, e = GR.gam_add(x, bins, nb, planes, h)
    cb, eb = GR.brute_gam(x, bins, nb, planes, h)
    assert c.dtype == np.uint64 and np.array_equal(c, cb) and e == eb
    det = GR.detection(x, bins, nb, planes, h, block_slices=7)
    assert np.array_equal(det, GR.detection(x, bins, nb, planes, h))


def test_a_bead_on_the_boundary_is_inside():
    # dyadic coordinates, planes and h: every s is exact, and beads sit exactly at |s| = h
    x = np.array([[0.5, 0.0, 0.0], [-0.5, 0.0, 0.0], [0.0, 0.75, 0.0], [0.0, 0.0, 0.25]])
    bins = np.array([0, 1, 2, 3], np.int32)
    planes = np.array([[1.0, 0.0, 0.0, 0.0],     # |s| = 0.5, 0.5, 0, 0: all four in at h = 0.5
                       [0.0, 1.0, 0.0, 0.25],    # s = -0.25, -0.25, 0.5, -0.25: all four in
                       [0.0, 0.0, 2.0, 1.0],     # s = -1, -1, -1, -0.5: only bead 3 (on the boundary)
                       [1.0, 0.0, 0.0, 1.0 + 2.0 ** -40]])  # s = -0.5 - 2^-40 and below: none
    c, e = GR.gam_add(x, bins, 4, planes, 0.5)
    det = GR.detection(x, bins, 4, planes, 0.5)
    assert det.tolist() == [[True] * 4, [True] * 4, [False, False, False, True], [False] * 4]
    assert e == 1
    assert c.tolist() == [2, 2, 2, 2, 2, 2, 2, 2, 2, 3]
    assert np.array_equal(c, GR.brute_gam(x, bins, 4, planes, 0.5)[0])
    # just below h, every bead at |s| = 0.5 leaves its slice
    below = GR.detection(x, bins, 4, planes, np.nextafter(0.5, 0.0))
    assert below.tolist() == [[False, False, True, True], [True, True, False, True], [False] * 4, [False] * 4]
    assert GR.gam_add(x, bins, 4, planes, np.nextafter(0.5, 0.0))[1] == 2


def test_diagonal_is_detection_and_bounds_hold():
    n = 4000
    gb = _gb(n)
    x = globule(n, 680, 3)
    planes, h = _planes(x, gb.bins, 300, 0.025, 3)
    c, e = GR.gam_add(x, gb.bins, gb.n_bins, planes, h)
    det = GR.detection(x, gb.bins, gb.n_bins, planes, h)
    d = gam._dense(c, gb.n_bins)
    fp = det.sum(axis=0)
    assert np.array_equal(np.diagonal(d), fp)
    assert np.all(d <= np.minimum(fp[:, None], fp[None, :]))
    assert e == np.count_nonzero(~det.any(axis=1)) and 0 < fp.sum()


def test_counts_do_not_depend_on_the_bead_order_within_a_bin():
    n = 4000
    gb = _gb(n)
    x = globule(n, 680, 4)
    planes, h = _planes(x, gb.bins, 200, 0.05, 4)
    want = GR.gam_add(x, gb.bins, gb.n_bins, planes, h)
    rng = np.random.default_rng(5)
    perm = np.arange(n)
    for b in range(gb.n_bins):  # permute the beads of every bin among themselves
        idx = np.flatnonzero(gb.bins == b)
        perm[idx] = rng.permutation(idx)
    got = GR.gam_add(x[perm], gb.bins, gb.n_bins, planes, h)
    assert np.array_equal(got[0], want[0]) and got[1] == want[1]


# ---- slice geometry --------------------------------------------------------------------------------------
def test_slice_planes_geometry_and_seeding():
    x = globule(3000, 680, 6) + np.array([1.0, -2.0, 0.5])
    bins = (np.arange(3000) % 7 - 1).astype(np.int32)  # some beads without a bin
    c = np.array([1.1, -1.9, 0.4])
    state = np.random.get_state()
    a, ha = gam.slice_planes(x, c, bins, 500, 0.025, np.random.default_rng([3, 1]))
    b, hb = gam.slice_planes(x, c, bins, 500, 0.025, np.random.default_rng([3, 1]))
    after = np.random.get_state()
    assert state[0] == after[0] and np.array_equal(state[1], after[1]) and state[2:] == after[2:]
    assert np.array_equal(a, b) and ha == hb
    other, _ = gam.slice_planes(x, c, bins, 500, 0.025, np.random.default_rng([3, 2]))
    assert not np.array_equal(a, other)
    assert a.shape == (500, 4) and a.dtype == np.float64
    assert np.allclose(np.linalg.norm(a[:, :3], axis=1), 1.0, rtol=0, atol=1e-12)
    d = x[bins >= 0] - c
    r = np.sqrt(np.max(np.sum(d * d, axis=1)))
    assert abs(ha - 0.025 * r) <= 1e-12 * r
    off = a[:, 3] - a[:, :3] @ c
    assert np.all(np.abs(off) <= r * (1 + 1e-12))
    assert off.min() < -0.8 * r and off.max() > 0.8 * r  # uniform over [-R, R]
    # isotropic: the mean normal is near zero, the mean of n n^T near I / 3
    assert np.all(np.abs(a[:, :3].mean(axis=0)) < 0.1)
    assert np.allclose(a[:, :3].T @ a[:, :3] / 500, np.eye(3) / 3, atol=0.06)
    with pytest.raises(ValueError, match="no bead has a bin"):
        gam.slice_planes(x, c, np.full(3000, -1), 5, 0.025, np.random.default_rng(0))


# ---- files -----------------------------------------------------------------------------------------------
def _member(x, gb, seed=0, count=200, fraction=0.025):
    planes, h = _planes(x, gb.bins, count, fraction, seed)
    c, e = GR.gam_add(x, gb.bins, gb.n_bins, planes, h)
    return gam.result(dict(counts=c, structures=1, slices=count, empty=e), gb, fraction)


def test_file_round_trip(tmp_path):
    gb = _gb()
    d = _member(globule(4000, 680, 1), gb)
    path = str(tmp_path / "g.npz")
    gam.save(path, d)
    got = gam.load(path)
    assert set(got) == set(gam.KEYS)
    for k in gam.KEYS:
        assert np.array_equal(got[k], d[k]) and got[k].dtype == np.asarray(d[k]).dtype, k
    assert got["counts"].dtype == np.uint64 and got["counts"].shape == (gb.n_bins * (gb.n_bins + 1) // 2,)
    np.savez(str(tmp_path / "other.npz"), counts=np.zeros(1))
    with pytest.raises(ValueError, match="not a GAM file"):
        gam.load(str(tmp_path / "other.npz"))


def test_aggregate_exact_and_order_independent(tmp_path):
    gb = _gb()
    xs = [globule(4000, 680, s) for s in range(3)]
    paths, parts = [], []
    for s, x in enumerate(xs):
        paths.append(str(tmp_path / f"m{s}.npz"))
        parts.append(_member(x, gb, seed=s))
        gam.save(paths[-1], parts[-1])
    a = gam.aggregate(paths)
    for order in (paths[::-1], [paths[1], paths[2], paths[0]]):
        b = gam.aggregate(order)
        for k in gam.KEYS:
            assert np.array_equal(a[k], b[k]) and a[k].dtype == b[k].dtype, k
    assert np.array_equal(a["counts"], sum(p["counts"] for p in parts))
    assert int(a["structures"]) == 3 and int(a["slices"]) == 600
    assert int(a["empty"]) == sum(int(p["empty"]) for p in parts)


@pytest.mark.parametrize("key", ["slice_fraction", "resolution_bp", "bin_start_bp", "bin_chrom"])
def test_aggregate_refuses_mismatches(tmp_path, key):
    gb = _gb()
    d = _member(globule(4000, 680, 1), gb)
    gam.save(str(tmp_path / "a.npz"), d)
    e = dict(d)
    e[key] = np.asarray(d[key] + 1, np.asarray(d[key]).dtype)
    gam.save(str(tmp_path / "b.npz"), e)
    with pytest.raises(ValueError, match=f"b.npz: {key}"):
        gam.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])


def test_aggregate_refuses_overflow_and_nothing(tmp_path):
    gb = _gb()
    d = _member(globule(4000, 680, 1), gb)
    e = dict(d)
    e["counts"] = d["counts"].copy()
    e["counts"][0] = np.uint64(2**64 - 1)
    d["counts"][0] = 1
    gam.save(str(tmp_path / "a.npz"), d)
    gam.save(str(tmp_path / "b.npz"), e)
    with pytest.raises(ValueError, match="b.npz: counts would overflow"):
        gam.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])
    with pytest.raises(ValueError, match="no GAM files"):
        gam.aggregate([])


# ---- readers ---------------------------------------------------------------------------------------------
def _table(det, empty_extra=0):
    """A GAM result from a hand-written detection table (bool [S, B]) plus ``empty_extra`` empty slices."""
    det = np.asarray(det, bool)
    b = det.shape[1]
    d = det.astype(np.int64)
    counts = (d.T @ d)[np.triu_indices(b)].astype(np.uint64)
    empty = int(np.count_nonzero(~det.any(axis=1))) + empty_extra
    gb = contacts.GenomeBins(np.arange(b, dtype=np.int32), np.zeros(b, np.int32), np.arange(b, dtype=np.int64) * 10, 10)
    return gam.result(dict(counts=counts, structures=1, slices=det.shape[0] + empty_extra, empty=empty), gb, 0.025)


def test_identical_windows_give_one():
    # bins 0 and 1 detected in exactly the same 3 of 8 slices, bin 2 in others
    det = np.zeros((8, 3), bool)
    det[[0, 2, 5], 0] = det[[0, 2, 5], 1] = True
    det[[1, 2, 3, 6], 2] = True
    d = _table(det)
    assert gam.normalized_linkage(d)[0, 1] == pytest.approx(1.0, abs=1e-15)
    assert gam.npmi(d)[0, 1] == pytest.approx(1.0, abs=1e-15)
    assert np.allclose(np.diagonal(gam.npmi(d)), 1.0)


def test_exclusive_windows_give_minus_one():
    det = np.zeros((6, 2), bool)
    det[[0, 1], 0] = True
    det[[2, 3, 4], 1] = True
    d = _table(det)
    assert gam.cosegregation(d)[0, 1] == 0.0
    assert gam.npmi(d)[0, 1] == -1.0 and gam.npmi(d)[1, 0] == -1.0
    assert gam.normalized_linkage(d)[0, 1] == pytest.approx(-1.0, abs=1e-15)  # D = -f_p f_q = -D_max


def test_a_product_table_has_no_linkage():
    # every combination of a 4-slice pattern of bin 0 (detected in 2) and a 4-slice pattern of bin 1 (in 1):
    # f_pq = f_p f_q exactly, with dyadic frequencies; bin 2, detected in every slice, leaves no slice empty
    det = np.array([[a, b, 1] for a in (1, 1, 0, 0) for b in (1, 0, 0, 0)], bool)
    d = _table(det)
    f = gam.detection_frequency(d)
    assert f.tolist() == [0.5, 0.25, 1.0] and int(d["empty"]) == 0
    assert gam.linkage(d)[0, 1] == 0.0 and gam.normalized_linkage(d)[0, 1] == 0.0 and gam.npmi(d)[0, 1] == 0.0


def test_empty_slices_are_left_out_of_the_denominators():
    det = np.zeros((4, 3), bool)
    det[[0, 1], 0] = det[[1, 2], 1] = True
    det[3, 2] = True
    a, b = _table(det), _table(det, empty_extra=5)
    assert int(b["slices"]) == 9 and int(b["empty"]) == 5
    for fn in (gam.cosegregation, gam.detection_frequency, gam.linkage, gam.normalized_linkage, gam.npmi):
        assert np.array_equal(fn(a), fn(b), equal_nan=True), fn.__name__
    assert np.allclose(gam.detection_frequency(b), [0.5, 0.5, 0.25])


def test_undetected_windows_and_no_hits_are_nan():
    det = np.zeros((4, 3), bool)
    det[[0, 1], 0] = True
    det[:, 1] = True  # detected in every slice: D_max = 0 with every other window
    d = _table(det)
    m = gam.npmi(d)
    assert np.all(np.isnan(m[2])) and np.all(np.isnan(m[:, 2]))
    assert m[1, 1] == 1.0 and m[0, 1] == pytest.approx(0.0, abs=1e-15)  # f_pq = f_p, f_q = 1
    dn = gam.normalized_linkage(d)
    assert np.isnan(dn[0, 1]) and np.isnan(dn[2, 0])
    for fn in (gam.cosegregation, gam.npmi, gam.normalized_linkage):
        m = fn(d)
        assert np.array_equal(m, m.T, equal_nan=True)
    none = _table(np.zeros((0, 3), bool), empty_extra=4)
    assert np.all(np.isnan(gam.detection_frequency(none))) and np.all(np.isnan(gam.npmi(none)))


# ---- settings --------------------------------------------------------------------------------------------
def _cfg(tmp_path, **kw):
    from multimm_b200.config import SimulationConfig

    base = dict(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    base.update(kw)
    return SimulationConfig(**base)


def test_settings_are_extras_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import EXTRA_FIELDS, GAM_FIELDS, SimulationConfig, contact_setting

    assert set(GAM_FIELDS) == {"SAVE_GAM", "GAM_RESOLUTION", "GAM_SLICES", "GAM_SLICE_FRACTION"}
    assert set(GAM_FIELDS) <= set(EXTRA_FIELDS) and not set(GAM_FIELDS) & set(SimulationConfig.model_fields)
    plain = _cfg(tmp_path)
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert contact_setting(plain, "SAVE_GAM") is False
    assert contact_setting(plain, "GAM_RESOLUTION") == 0
    assert contact_setting(plain, "GAM_SLICES") == 1024
    assert contact_setting(plain, "GAM_SLICE_FRACTION") == 0.025
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\nSAVE_GAM = True\nGAM_SLICES = 64\n")
    args, _ = run.get_config(["-c", str(ini), "--gam_resolution", "5000000", "--gam_slice_fraction", "0.1"])
    assert contact_setting(args, "SAVE_GAM") is True
    assert contact_setting(args, "GAM_RESOLUTION") == 5_000_000
    assert contact_setting(args, "GAM_SLICES") == 64
    assert contact_setting(args, "GAM_SLICE_FRACTION") == 0.1


def _dumps(tmp_path, name):
    """(config_auto.ini, parameters.txt) bytes of a config without the GAM settings."""
    import types

    from multimm_b200 import run
    from multimm_b200.model import MultiMM

    ini = tmp_path / f"{name}.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / name}\nSAVE_CONTACTS = true\n")
    args, _ = run.get_config(["-c", str(ini)])
    params = tmp_path / f"{name}_parameters.txt"
    MultiMM.save_args_to_txt(types.SimpleNamespace(args=args), str(params))
    auto = (tmp_path / name / "metadata" / "config_auto.ini").read_bytes()
    return auto.replace(str(tmp_path / name).encode(), b"OUT"), params.read_bytes().replace(str(tmp_path / name).encode(), b"OUT")


def test_dumps_without_the_settings_are_unchanged(tmp_path, monkeypatch):
    from multimm_b200 import config

    with_fields = _dumps(tmp_path, "a")
    for word in (b"save_gam", b"gam_resolution", b"gam_slices", b"gam_slice_fraction"):
        assert word not in with_fields[0].lower() + with_fields[1].lower()
    for k in config.GAM_FIELDS:
        monkeypatch.delitem(config.EXTRA_FIELDS, k)
    assert _dumps(tmp_path, "b") == with_fields


@pytest.mark.parametrize("fields,match", [
    (dict(GAM_RESOLUTION=-1), "GAM_RESOLUTION"),
    (dict(GAM_RESOLUTION=100_000), "GAM_RESOLUTION"),   # 3.1e4 bins genome-wide
    (dict(GAM_RESOLUTION=2_000, CHROM="chr1", LOC_START=0, LOC_END=50_000_000), "GAM_RESOLUTION"),
    (dict(GAM_SLICES=0), "GAM_SLICES"),
    (dict(GAM_SLICES=65537), "GAM_SLICES"),
    (dict(GAM_SLICE_FRACTION=0.0), "GAM_SLICE_FRACTION"),
    (dict(GAM_SLICE_FRACTION=-0.1), "GAM_SLICE_FRACTION"),
    (dict(GAM_SLICE_FRACTION=1.5), "GAM_SLICE_FRACTION"),
    (dict(GAM_SLICE_FRACTION=float("nan")), "GAM_SLICE_FRACTION"),
    (dict(GAM_SLICE_FRACTION=float("inf")), "GAM_SLICE_FRACTION"),
    (dict(SHUFFLING_SEED=-1), "SHUFFLING_SEED"),
])
def test_bad_gam_fields_refused_before_any_output(tmp_path, fields, match):
    from multimm_b200 import run

    with pytest.raises(ValueError, match=match):
        run.args_tests(_cfg(tmp_path, SAVE_GAM=True, **fields))
    assert not (tmp_path / "o").exists()


def test_gam_fields_valid_values(tmp_path):
    from multimm_b200 import run

    for res in (0, 1_000_000, 3_000_000):
        run.args_tests(_cfg(tmp_path, SAVE_GAM=True, GAM_RESOLUTION=res))
    run.args_tests(_cfg(tmp_path, SAVE_GAM=True, GAM_SLICES=1, GAM_SLICE_FRACTION=1.0))
    run.args_tests(_cfg(tmp_path, SAVE_GAM=True, GAM_SLICES=65536, GAM_RESOLUTION=5_000, CHROM="chr1", LOC_START=0,
                        LOC_END=50_000_000))
    assert not (tmp_path / "o").exists()
    b = gam.MAX_BINS
    assert b * (b + 1) // 2 <= gam.MAX_ROWS < (b + 1) * (b + 2) // 2


def test_md_sampling_accepts_gam_alone(tmp_path):
    from multimm_b200 import run

    run.args_tests(_cfg(tmp_path, SAVE_GAM=True, SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100,
                        MD_SAMPLE_STEP=200))
    with pytest.raises(ValueError, match="SAVE_GAM"):
        run.args_tests(_cfg(tmp_path, SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100, MD_SAMPLE_STEP=200))
