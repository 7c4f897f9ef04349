"""Three-way contact maps on the host: the numpy restatement (tests/triplets_ref.py) against brute force and
against trace(A^3) / 6, the triplets file format, its exact aggregation, the coarsen and viewpoint views, and the
SAVE_TRIPLETS / TRIPLET_RESOLUTION settings and their checks."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

import contacts_ref as CR
import triplets_ref as TR
from multimm_b200 import contacts, loaders, triplets

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


def _layout(n=4000):
    lay = {}
    loaders.import_mns_from_bedpe(BEDPE, N_beads=n, chrom=None, coords=None, path=None, shuffle=False, seed=0,
                                  layout=lay)
    return lay


def _sorted(t):
    o = np.lexsort(t[::-1])
    return tuple(a[o] for a in t)


# ---- the restatement -------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,rc,seed", [(3, 1.0, 0), (40, 0.3, 1), (60, 0.25, 2), (90, 0.2, 3)])
def test_restatement_equals_brute_force(n, rc, seed):
    x = TR.globule(n, 680, seed)
    want = TR.brute_triangles(x, rc)
    got = _sorted(TR.triangles_from_pairs(n, *CR.contact_pairs(x, rc)))
    assert all(np.array_equal(a, b) for a, b in zip(got, want)) and len(want[0]) > 0
    # binning with left-out beads: every triple with a bead at -1 drops out, the others sort their bins
    rng = np.random.default_rng(seed)
    bins = rng.integers(-1, 5, size=n).astype(np.int32)
    d = TR.binned(*want, bins, 5)
    want_keys = []
    for i, j, k in zip(*want):
        b = sorted((bins[i], bins[j], bins[k]))
        if b[0] >= 0:
            want_keys.append((b[0] * 5 + b[1]) * 5 + b[2])
    u, c = np.unique(np.asarray(want_keys, np.int64), return_counts=True)
    assert np.array_equal((d[0].astype(np.int64) * 5 + d[1]) * 5 + d[2], u) and np.array_equal(d[3], c)
    assert np.all(d[0] <= d[1]) and np.all(d[1] <= d[2])


def test_restatement_total_equals_trace_of_a_cubed():
    n = 20_000
    x = TR.globule(n, 680, 5)
    i, j = CR.contact_pairs(x, 0.3)
    a = sp.csr_matrix((np.ones(len(i), np.int64), (i, j)), shape=(n, n))
    a = a + a.T
    want = int((a @ a).multiply(a).sum()) // 6
    d = TR.triplet_sums(x, 0.3, np.zeros(n, np.int32), 1)
    assert d["triples"] == want > 10 * n and int(d["vals"].sum()) == want  # one bin: every triple at (0, 0, 0)


# ---- files -----------------------------------------------------------------------------------------------
def _member(x, rc, gb, members=1):
    return triplets.result(TR.triplet_sums(x, rc, gb.bins, gb.n_bins), rc, gb, members)


def _gb(n=4000, res=2_000_000):
    return contacts.genome_bins(_layout(n), res, n_beads=n, max_bins=triplets.MAX_BINS)


def test_file_round_trip(tmp_path):
    gb = _gb()
    d = _member(TR.globule(4000, 680, 1), 0.3, gb, members=3)
    path = str(tmp_path / "t.npz")
    triplets.save(path, d)
    got = triplets.load(path)
    assert set(got) == set(triplets.KEYS)
    for k in triplets.KEYS:
        assert np.array_equal(got[k], d[k]) and got[k].dtype == np.asarray(d[k]).dtype, k
    assert int(got["members"]) == 3 and got["triples"].dtype == np.uint64
    np.savez(str(tmp_path / "other.npz"), rows=np.zeros(1))
    with pytest.raises(ValueError, match="not a triplets file"):
        triplets.load(str(tmp_path / "other.npz"))


def test_aggregate_exact_and_order_independent(tmp_path):
    gb = _gb()
    xs = [TR.globule(4000, 680, s) for s in range(3)]
    paths = []
    for s, x in enumerate(xs):
        paths.append(str(tmp_path / f"m{s}.npz"))
        triplets.save(paths[-1], _member(x, 0.3, gb))
    a = triplets.aggregate(paths)
    b = triplets.aggregate(paths[::-1])
    c = triplets.aggregate([paths[1], paths[2], paths[0]])
    for k in triplets.KEYS:
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c[k]) and a[k].dtype == b[k].dtype, k
    # the sum of the members' triangles, binned once
    tri = [TR.triangles_from_pairs(4000, *CR.contact_pairs(x, 0.3)) for x in xs]
    want = TR.binned(*(np.concatenate([t[m] for t in tri]) for m in range(3)), gb.bins, gb.n_bins)
    for k, w in zip(("p", "q", "r", "vals"), want):
        assert np.array_equal(a[k], w) and a[k].dtype == w.dtype, k
    assert int(a["members"]) == 3 and int(a["triples"]) == sum(len(t[0]) for t in tri)


@pytest.mark.parametrize("key,value", [("radius_nm", 0.25), ("resolution_bp", 1), ("n_bins", 7),
                                       ("bin_start_bp", None)])
def test_aggregate_refuses_mismatches(tmp_path, key, value):
    gb = _gb()
    d = _member(TR.globule(4000, 680, 1), 0.3, gb)
    triplets.save(str(tmp_path / "a.npz"), d)
    e = dict(d)
    e[key] = d[key] + 1 if value is None else np.asarray(value, np.asarray(d[key]).dtype)
    triplets.save(str(tmp_path / "b.npz"), e)
    with pytest.raises(ValueError, match=key):
        triplets.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])


# ---- views -----------------------------------------------------------------------------------------------
def test_coarsen_equals_the_restatement_at_the_coarse_bins():
    n = 4000
    lay = _layout(n)
    fine = contacts.genome_bins(lay, 100_000, n_beads=n, max_bins=triplets.MAX_BINS)
    coarse = contacts.genome_bins(lay, 5_000_000, n_beads=n)
    x = TR.globule(n, 680, 7)
    d = _member(x, 0.3, fine, members=2)
    got = triplets.coarsen(d, 5_000_000)
    want = _member(x, 0.3, coarse, members=2)
    for k in triplets.KEYS:
        assert np.array_equal(got[k], want[k]) and got[k].dtype == np.asarray(want[k]).dtype, k
    assert len(got["vals"]) < len(d["vals"]) and int(got["vals"].sum()) == int(d["vals"].sum())
    with pytest.raises(ValueError, match="multiple"):
        triplets.coarsen(d, 150_000)
    with pytest.raises(ValueError, match="bins"):
        triplets.coarsen(d, 200_000)  # over 4096 bins genome-wide


def test_viewpoint_is_symmetric_and_consistent_with_the_entries():
    gb = _gb(4000, 20_000_000)
    d = _member(TR.globule(4000, 680, 3), 0.25, gb)
    nb = gb.n_bins
    full = np.zeros((nb, nb, nb), np.uint64)  # the count of every ordered bin triple
    for p, q, r, v in zip(d["p"], d["q"], d["r"], d["vals"]):
        for a, b, c in {(p, q, r), (p, r, q), (q, p, r), (q, r, p), (r, p, q), (r, q, p)}:
            full[a, b, c] = v
    seen = 0
    for v in range(nb):
        m = triplets.viewpoint(d, v)
        assert m.dtype == np.uint64 and np.array_equal(m, m.T)
        assert np.array_equal(m, full[v])
        seen += int(m.sum() > 0)
    assert seen > nb // 2
    with pytest.raises(ValueError):
        triplets.viewpoint(d, nb)


# ---- settings --------------------------------------------------------------------------------------------
def _cfg(tmp_path, **kw):
    from multimm_b200.config import SimulationConfig

    base = dict(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    base.update(kw)
    return SimulationConfig(**base)


def test_settings_are_extras_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import EXTRA_FIELDS, SimulationConfig, TRIPLET_FIELDS, contact_setting

    assert set(TRIPLET_FIELDS) == {"SAVE_TRIPLETS", "TRIPLET_RESOLUTION"} and set(TRIPLET_FIELDS) <= set(EXTRA_FIELDS)
    assert not set(TRIPLET_FIELDS) & set(SimulationConfig.model_fields)
    plain = _cfg(tmp_path)
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert contact_setting(plain, "SAVE_TRIPLETS") is False and contact_setting(plain, "TRIPLET_RESOLUTION") == 0
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\nSAVE_TRIPLETS = True\n")
    args, _ = run.get_config(["-c", str(ini), "--triplet_resolution", "5000"])
    assert contact_setting(args, "SAVE_TRIPLETS") is True and contact_setting(args, "TRIPLET_RESOLUTION") == 5000


def _dumps(tmp_path, name):
    """(config_auto.ini, parameters.txt) bytes of a config without the three-way settings."""
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
    for word in (b"save_triplets", b"triplet_resolution"):
        assert word not in with_fields[0].lower() + with_fields[1].lower()
    for k in config.TRIPLET_FIELDS:
        monkeypatch.delitem(config.EXTRA_FIELDS, k)
    assert _dumps(tmp_path, "b") == with_fields


@pytest.mark.parametrize("fields", [dict(TRIPLET_RESOLUTION=-1), dict(TRIPLET_RESOLUTION=2_000),
                                    dict(TRIPLET_RESOLUTION=40, CHROM="chr1", LOC_START=0, LOC_END=50_000_000)])
def test_bad_triplet_fields_refused_before_any_output(tmp_path, fields):
    from multimm_b200 import run

    with pytest.raises(ValueError, match="TRIPLET_RESOLUTION"):
        run.args_tests(_cfg(tmp_path, SAVE_TRIPLETS=True, **fields))
    assert not (tmp_path / "o").exists()


def test_triplet_fields_valid_values(tmp_path):
    from multimm_b200 import run

    for res in (0, 5_000, 1_000_000):  # 5 kb: about 5.8e5 bins genome-wide
        run.args_tests(_cfg(tmp_path, SAVE_TRIPLETS=True, TRIPLET_RESOLUTION=res))
    run.args_tests(_cfg(tmp_path, SAVE_TRIPLETS=True, TRIPLET_RESOLUTION=50, CHROM="chr1", LOC_START=0,
                        LOC_END=50_000_000))  # 10^6 bins
    assert not (tmp_path / "o").exists()


def test_md_sampling_accepts_the_three_way_map_alone(tmp_path):
    from multimm_b200 import run

    run.args_tests(_cfg(tmp_path, SAVE_TRIPLETS=True, SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100,
                        MD_SAMPLE_STEP=200))
    with pytest.raises(ValueError, match="SAVE_CONTACTS or SAVE_DISTANCES"):
        run.args_tests(_cfg(tmp_path, SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100, MD_SAMPLE_STEP=200))
