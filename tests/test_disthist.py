"""Distance distributions on the host: the numpy restatement (tests/disthist_ref.py) against brute force, against
the distance map's pair counts and the contact map at every edge, the distance-histogram file format, its exact
aggregation, the readers, and the SAVE_DISTANCE_HIST / DISTANCE_HIST_RESOLUTION / DISTANCE_HIST_EDGES settings."""
import os

import numpy as np
import pytest

import contacts_ref as CR
import disthist_ref as HR
from multimm_b200 import contacts, disthist, distances, loaders
from triplets_ref import globule

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")
EDGES = disthist.parse_edges(disthist.DEFAULT_EDGES)


def _layout(n=4000):
    lay = {}
    loaders.import_mns_from_bedpe(BEDPE, N_beads=n, chrom=None, coords=None, path=None, shuffle=False, seed=0,
                                  layout=lay)
    return lay


def _gb(n=4000, res=20_000_000):
    return contacts.genome_bins(_layout(n), res, n_beads=n)


def lattice(n, step=0.5, seed=0):
    """n beads on a cubic lattice of spacing ``step`` (shuffled): many pairs sit exactly at multiples of step, whose
    squares are exact in FP64 when step is a power of two."""
    rng = np.random.default_rng(seed)
    side = int(np.ceil(n ** (1.0 / 3.0))) + 1
    g = np.stack(np.meshgrid(*(np.arange(side),) * 3, indexing="ij"), -1).reshape(-1, 3)
    return step * g[rng.permutation(len(g))[:n]].astype(np.float64)


# ---- the restatement -------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,seed", [(2, 0), (45, 1), (80, 2)])
def test_restatement_equals_brute_force(n, seed):
    rng = np.random.default_rng(seed)
    x = globule(n, 30, seed)
    bins = rng.integers(-1, 6, size=n).astype(np.int32)
    for edges in (EDGES, [0.3], np.linspace(0.05, 3.15, 63)):
        assert np.array_equal(HR.hist_counts(x, bins, 6, edges, block_pairs=97), HR.brute_hist(x, bins, 6, edges))


def test_a_pair_on_an_edge_counts_in_the_upper_cell():
    x = np.array([[0.0, 0.0, 0.0], [0.5, 0.0, 0.0], [0.0, 1.0, 0.0], [0.25, 0.0, 0.0]])
    c = HR.hist_counts(x, np.zeros(4, np.int32), 1, [0.25, 0.5, 1.0])
    # pairs: 0.5 (on e_2), 1.0 (on e_3), 0.25 (on e_1), sqrt(1.25), 0.25 (on e_1), sqrt(1.0625)
    assert c.tolist() == [[0, 2, 1, 3]]
    assert np.array_equal(c, HR.brute_hist(x, np.zeros(4, np.int32), 1, [0.25, 0.5, 1.0]))
    assert disthist.cells_of([0.25, np.nextafter(0.25, 0.0)], [0.5]).tolist() == [1, 0]


def test_lattice_pairs_on_the_edges():
    x = lattice(300)
    bins = (np.arange(300) % 4).astype(np.int32)
    edges = [0.5, 1.0, 1.5, 2.0]
    d = x[:, None, :] - x[None, :, :]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    on_edge = np.isin(d2[np.triu_indices(300, 1)], np.asarray(edges) ** 2).sum()
    assert on_edge > 1000
    assert np.array_equal(HR.hist_counts(x, bins, 4, edges), HR.brute_hist(x, bins, 4, edges))


def test_restatement_sums_to_the_pair_counts_and_the_contact_maps():
    n = 4000
    gb = _gb(n)
    x = globule(n, 680, 3)
    c = HR.hist_counts(x, gb.bins, gb.n_bins, EDGES)
    d = disthist.result(c, EDGES, gb)
    pairs, _ = distances._counts(gb)
    assert np.array_equal(disthist.pair_counts(d), pairs)
    iu = np.triu_indices(gb.n_bins)
    cum = np.cumsum(c, axis=1, dtype=np.uint64)
    for k, e in enumerate(EDGES[:8]):
        cmap, _, _ = CR.contact_counts(x, float(e), gb.bins, gb.n_bins)
        assert np.array_equal(cum[:, k], cmap[iu]), e


# ---- files -----------------------------------------------------------------------------------------------
def _member(x, gb, edges=EDGES, members=1):
    return disthist.result(HR.hist_counts(x, gb.bins, gb.n_bins, edges), edges, gb, members)


def test_file_round_trip(tmp_path):
    gb = _gb()
    d = _member(globule(4000, 680, 1), gb, members=3)
    path = str(tmp_path / "h.npz")
    disthist.save(path, d)
    got = disthist.load(path)
    assert set(got) == set(disthist.KEYS)
    for k in disthist.KEYS:
        assert np.array_equal(got[k], d[k]) and got[k].dtype == np.asarray(d[k]).dtype, k
    assert got["counts"].dtype == np.uint64 and got["counts"].shape == (gb.n_bins * (gb.n_bins + 1) // 2, 20)
    np.savez(str(tmp_path / "other.npz"), rows=np.zeros(1))
    with pytest.raises(ValueError, match="not a distance-histogram file"):
        disthist.load(str(tmp_path / "other.npz"))


def test_aggregate_exact_and_order_independent(tmp_path):
    gb = _gb()
    xs = [globule(4000, 680, s) for s in range(3)]
    paths = []
    for s, x in enumerate(xs):
        paths.append(str(tmp_path / f"m{s}.npz"))
        disthist.save(paths[-1], _member(x, gb))
    a = disthist.aggregate(paths)
    for order in (paths[::-1], [paths[1], paths[2], paths[0]]):
        b = disthist.aggregate(order)
        for k in disthist.KEYS:
            assert np.array_equal(a[k], b[k]) and a[k].dtype == b[k].dtype, k
    want = sum(HR.hist_counts(x, gb.bins, gb.n_bins, EDGES) for x in xs)
    assert np.array_equal(a["counts"], want) and int(a["members"]) == 3
    assert np.array_equal(a["bin_beads"], 3 * np.bincount(gb.bins[gb.bins >= 0], minlength=gb.n_bins))


@pytest.mark.parametrize("key", ["edges_nm", "resolution_bp", "bin_start_bp", "bin_chrom"])
def test_aggregate_refuses_mismatches(tmp_path, key):
    gb = _gb()
    d = _member(globule(4000, 680, 1), gb)
    disthist.save(str(tmp_path / "a.npz"), d)
    e = dict(d)
    e[key] = np.asarray(d[key] + 1, np.asarray(d[key]).dtype)
    disthist.save(str(tmp_path / "b.npz"), e)
    with pytest.raises(ValueError, match=f"b.npz: {key}"):
        disthist.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])


def test_aggregate_refuses_overflow(tmp_path):
    gb = _gb()
    d = _member(globule(4000, 680, 1), gb)
    disthist.save(str(tmp_path / "a.npz"), d)
    e = dict(d)
    e["counts"] = d["counts"].copy()
    e["counts"][0, 0] = np.uint64(2**64 - 1)
    disthist.save(str(tmp_path / "b.npz"), e)
    d["counts"][0, 0] = 1
    disthist.save(str(tmp_path / "a.npz"), d)
    with pytest.raises(ValueError, match="b.npz: counts would overflow"):
        disthist.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])


# ---- readers ---------------------------------------------------------------------------------------------
def _hand(counts, edges=(1.0, 2.0, 4.0)):
    """A histogram of two bins from hand-written rows (0, 0), (0, 1), (1, 1)."""
    gb = contacts.GenomeBins(np.array([0, 1], np.int32), np.zeros(2, np.int32), np.array([0, 10], np.int64), 10)
    return disthist.result(np.asarray(counts, np.uint64), np.asarray(edges, np.float64), gb)


def test_readers_on_a_hand_built_histogram():
    d = _hand([[2, 2, 0, 0],     # (0, 0): two pairs in [0, 1), two in [1, 2)
               [0, 0, 0, 0],     # (0, 1): no pair
               [0, 1, 1, 2]])    # (1, 1): one in [1, 2), one in [2, 4), two in [4, inf)
    pc = disthist.pair_counts(d)
    assert pc.dtype == np.uint64 and pc.tolist() == [[4, 0], [0, 4]]
    cum = disthist.cumulative_probability(d)
    assert cum.shape == (2, 2, 3)
    assert np.allclose(cum[0, 0], [0.5, 1.0, 1.0]) and np.allclose(cum[1, 1], [0.0, 0.25, 0.5])
    assert np.all(np.isnan(cum[0, 1])) and np.all(np.isnan(cum[1, 0]))
    assert np.allclose(disthist.contact_probability(d, 2.0), [[1.0, np.nan], [np.nan, 0.25]], equal_nan=True)
    with pytest.raises(ValueError, match="not one of the histogram's edges"):
        disthist.contact_probability(d, 1.5)
    med = disthist.median_distance(d)
    # (0, 0), (1, 1): the median (2 of 4 pairs) is the upper edge of cell 0 and of cell 2
    assert med[0, 0] == 1.0 and med[1, 1] == 4.0 and np.isnan(med[0, 1])
    assert np.isnan(disthist.quantile_distance(d, 0.6)[1, 1])  # 2.4 of 4 pairs: in the open last cell
    q = disthist.quantile_distance(d, 0.25)
    assert q[0, 0] == 0.5 and q[1, 1] == 2.0  # 1 of 4 pairs: half-way through cell 0; the end of cell 1
    assert disthist.quantile_distance(d, 0.375)[1, 1] == 3.0  # 1.5 of 4: half-way through [2, 4)
    assert disthist.quantile_distance(d, 0.0)[1, 1] == 1.0  # the lower edge of the first cell with pairs
    assert disthist.quantile_distance(d, 0.75)[0, 0] == 1.5
    for m in (med, q):
        assert np.array_equal(m, m.T, equal_nan=True)
    with pytest.raises(ValueError, match="outside"):
        disthist.quantile_distance(d, 1.5)


def test_median_matches_the_sample_median_within_a_cell():
    rng = np.random.default_rng(4)
    dist = rng.uniform(0.0, 10.0, 100_001)
    edges = np.arange(0.5, 10.5, 0.5)
    counts = np.bincount(np.searchsorted(edges, dist, side="right"), minlength=len(edges) + 1)
    d = _hand(np.stack([counts, np.zeros_like(counts), counts]), edges)
    med = disthist.median_distance(d)
    assert abs(med[0, 0] - np.median(dist)) < 0.01 and abs(med[1, 1] - med[0, 0]) == 0.0


# ---- settings --------------------------------------------------------------------------------------------
def _cfg(tmp_path, **kw):
    from multimm_b200.config import SimulationConfig

    base = dict(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    base.update(kw)
    return SimulationConfig(**base)


def test_settings_are_extras_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import DISTANCE_HIST_FIELDS, EXTRA_FIELDS, SimulationConfig, contact_setting

    assert set(DISTANCE_HIST_FIELDS) == {"SAVE_DISTANCE_HIST", "DISTANCE_HIST_RESOLUTION", "DISTANCE_HIST_EDGES"}
    assert set(DISTANCE_HIST_FIELDS) <= set(EXTRA_FIELDS) and not set(DISTANCE_HIST_FIELDS) & set(SimulationConfig.model_fields)
    plain = _cfg(tmp_path)
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert contact_setting(plain, "SAVE_DISTANCE_HIST") is False
    assert contact_setting(plain, "DISTANCE_HIST_RESOLUTION") == 0
    assert contact_setting(plain, "DISTANCE_HIST_EDGES") == disthist.DEFAULT_EDGES
    # the default edges hold the default contact radius, so the contact map can be read off the histogram
    assert float(contact_setting(plain, "CONTACT_RADIUS")) in disthist.parse_edges(disthist.DEFAULT_EDGES)
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\nSAVE_DISTANCE_HIST = True\n"
                   "DISTANCE_HIST_EDGES = 0.2,0.4\n")
    args, _ = run.get_config(["-c", str(ini), "--distance_hist_resolution", "5000000"])
    assert contact_setting(args, "SAVE_DISTANCE_HIST") is True
    assert contact_setting(args, "DISTANCE_HIST_RESOLUTION") == 5_000_000
    assert contact_setting(args, "DISTANCE_HIST_EDGES") == "0.2,0.4"


def _dumps(tmp_path, name):
    """(config_auto.ini, parameters.txt) bytes of a config without the distance-histogram settings."""
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
    for word in (b"save_distance_hist", b"distance_hist_resolution", b"distance_hist_edges"):
        assert word not in with_fields[0].lower() + with_fields[1].lower()
    for k in config.DISTANCE_HIST_FIELDS:
        monkeypatch.delitem(config.EXTRA_FIELDS, k)
    assert _dumps(tmp_path, "b") == with_fields


@pytest.mark.parametrize("fields,match", [
    (dict(DISTANCE_HIST_RESOLUTION=-1), "DISTANCE_HIST_RESOLUTION"),
    (dict(DISTANCE_HIST_RESOLUTION=100_000), "DISTANCE_HIST_RESOLUTION"),   # 3.1e4 bins genome-wide
    (dict(DISTANCE_HIST_RESOLUTION=2_000, CHROM="chr1", LOC_START=0, LOC_END=50_000_000), "DISTANCE_HIST_RESOLUTION"),
    (dict(DISTANCE_HIST_EDGES="0.2,0.1"), "strictly increasing"),
    (dict(DISTANCE_HIST_EDGES="0.2,0.2"), "strictly increasing"),
    (dict(DISTANCE_HIST_EDGES="0,0.2"), "finite and > 0"),
    (dict(DISTANCE_HIST_EDGES="-1"), "finite and > 0"),
    (dict(DISTANCE_HIST_EDGES="0.1,inf"), "finite and > 0"),
    (dict(DISTANCE_HIST_EDGES="0.1,nan"), "finite and > 0"),
    (dict(DISTANCE_HIST_EDGES="1e200"), "finite and > 0"),
    (dict(DISTANCE_HIST_EDGES="0.1,x"), "comma-separated"),
    (dict(DISTANCE_HIST_EDGES=""), "comma-separated"),
    (dict(DISTANCE_HIST_EDGES=",".join(str(0.1 * k) for k in range(1, 65))), "1 to 63 edges"),
])
def test_bad_distance_hist_fields_refused_before_any_output(tmp_path, fields, match):
    from multimm_b200 import run

    with pytest.raises(ValueError, match=match):
        run.args_tests(_cfg(tmp_path, SAVE_DISTANCE_HIST=True, **fields))
    assert not (tmp_path / "o").exists()


def test_distance_hist_fields_valid_values(tmp_path):
    from multimm_b200 import run

    for res in (0, 1_000_000, 3_000_000):
        run.args_tests(_cfg(tmp_path, SAVE_DISTANCE_HIST=True, DISTANCE_HIST_RESOLUTION=res))
    run.args_tests(_cfg(tmp_path, SAVE_DISTANCE_HIST=True, DISTANCE_HIST_EDGES="0.5",
                        DISTANCE_HIST_RESOLUTION=50_000, CHROM="chr1", LOC_START=0, LOC_END=50_000_000))
    run.args_tests(_cfg(tmp_path, SAVE_DISTANCE_HIST=True,
                        DISTANCE_HIST_EDGES=",".join(str(0.1 * k) for k in range(1, 64))))
    assert not (tmp_path / "o").exists()
    assert disthist.max_bins(19) == 3663 and 3663 * 3664 // 2 * 20 <= 2**27 < 3664 * 3665 // 2 * 20


def test_md_sampling_accepts_the_distance_histograms_alone(tmp_path):
    from multimm_b200 import run

    run.args_tests(_cfg(tmp_path, SAVE_DISTANCE_HIST=True, SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100,
                        MD_SAMPLE_STEP=200))
    with pytest.raises(ValueError, match="SAVE_CONTACTS or SAVE_DISTANCES"):
        run.args_tests(_cfg(tmp_path, SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100, MD_SAMPLE_STEP=200))
