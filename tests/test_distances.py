"""Distance maps on the host: the numpy restatement (distances_ref.py) against brute force, the
SAVE_DISTANCES / DISTANCE_RESOLUTION settings, the file format and its exact aggregation over ensemble
members, and the mean / RMS / std / radial helpers."""
import os

import numpy as np
import pytest

import distances_ref as R
from multimm_b200 import contacts, distances

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


# ---- the numpy restatement ----------------------------------------------------------------------------
@pytest.mark.parametrize("n,n_bins,scale", [(40, 1, 1.0), (75, 6, 3.0), (123, 123, 0.4)])
def test_reference_matches_brute_force(n, n_bins, scale):
    rng = np.random.default_rng(n)
    x = rng.uniform(-scale, scale, size=(n, 3))
    bins = rng.integers(-1, n_bins, size=n) if n_bins > 1 else np.zeros(n, np.int64)
    got = R.distance_sums(x, bins, n_bins, block_pairs=97)  # many small blocks
    want = R.brute_distance_sums(x, bins, n_bins)
    for g, w in zip(got, want):
        assert g.dtype == np.uint64 and np.array_equal(g, w) and np.array_equal(g, g.T)
    p, q = int(bins.max()), int(bins[bins >= 0].min())
    assert R.block_sums(x, bins, p, q) == (int(want[0][p, q]), int(want[1][p, q]))


def test_reference_rounds_half_to_even():
    """Distances whose scaled value ends in exactly .5: rint, like __double2ll_rn, rounds to even."""
    x = np.array([[0.0, 0.0, 0.0], [2.5 * 2.0 ** -24, 0.0, 0.0], [3.5 * 2.0 ** -24, 0.0, 0.0]])
    d, _ = R.distance_sums(x, np.zeros(3, np.int64), 1)
    assert int(d[0, 0]) == 2 + 4 + 1  # 2.5 -> 2, 3.5 -> 4, 1.0 -> 1


# ---- settings ------------------------------------------------------------------------------------------
def test_distance_settings_are_extras_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import DISTANCE_FIELDS, EXTRA_FIELDS, SimulationConfig, contact_setting

    assert set(DISTANCE_FIELDS) <= set(EXTRA_FIELDS) and not set(DISTANCE_FIELDS) & set(SimulationConfig.model_fields)
    plain = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert [contact_setting(plain, k) for k in DISTANCE_FIELDS] == [False, 0]
    given = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), SAVE_DISTANCES="yes",
                             DISTANCE_RESOLUTION="3000000")
    again = SimulationConfig(**given.model_dump())
    assert [contact_setting(again, k) for k in DISTANCE_FIELDS] == [True, 3_000_000]
    with pytest.raises(ValueError):
        SimulationConfig(LOOPS_PATH=BEDPE, DISTANCE_RESOLUTION="fine")
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\nSAVE_DISTANCES = true\n")
    args, _ = run.get_config(["-c", str(ini), "--distance_resolution", "2000000"])
    assert contact_setting(args, "SAVE_DISTANCES") is True and contact_setting(args, "DISTANCE_RESOLUTION") == 2_000_000
    assert "save_distances = True" in (tmp_path / "cli" / "metadata" / "config_auto.ini").read_text()


def _dumps(tmp_path, name):
    """(config_auto.ini, parameters.txt) bytes of a config without the distance settings."""
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
    """config_auto.ini and parameters.txt of a config without the distance settings are the bytes of the
    same config read by a package that does not know them."""
    from multimm_b200 import config

    with_fields = _dumps(tmp_path, "a")
    for word in (b"save_distances", b"distance_resolution"):
        assert word not in with_fields[0].lower() + with_fields[1].lower()
    for k in config.DISTANCE_FIELDS:
        monkeypatch.delitem(config.EXTRA_FIELDS, k)
    assert _dumps(tmp_path, "b") == with_fields


@pytest.mark.parametrize("fields", [dict(DISTANCE_RESOLUTION=-1), dict(DISTANCE_RESOLUTION=100_000),
                                    dict(DISTANCE_RESOLUTION=10_000, CHROM="chr1", LOC_START=0, LOC_END=50_000_000)])
def test_bad_distance_fields_refused_before_any_output(tmp_path, fields):
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    out = tmp_path / "out"
    args = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(out), SAVE_DISTANCES=True, **fields)
    with pytest.raises(ValueError, match="DISTANCE_RESOLUTION"):
        run.args_tests(args)
    assert not out.exists()


def test_distance_fields_valid_values(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    for res in (0, 1_000_000, 800_000):  # 800 kb: about 3900 bins genome-wide
        run.args_tests(SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), SAVE_DISTANCES="yes",
                                        DISTANCE_RESOLUTION=res))
    assert not (tmp_path / "o").exists()


# ---- files, aggregation, helpers ---------------------------------------------------------------------------
def _member(rng, b=6, members=1, bin_beads=None, lo=0, hi=10**9):
    m = rng.integers(lo, hi, size=(b, b), dtype=np.uint64)
    m = np.triu(m) + np.triu(m, 1).T
    m2 = rng.integers(lo, hi, size=(b, b), dtype=np.uint64)
    m2 = np.triu(m2) + np.triu(m2, 1).T
    n = np.asarray(bin_beads if bin_beads is not None else [3, 1, 0, 5, 2, 4], np.uint64)
    pc = np.outer(n, n)
    pc[np.diag_indices(b)] = n * (n - np.uint64(1)) // np.uint64(2)
    return dict(dist_sum=m, dist2_sum=m2, pair_count=pc, bin_beads=n, radial_sum=rng.integers(lo, hi, size=b, dtype=np.uint64),
                radial2_sum=rng.integers(lo, hi, size=b, dtype=np.uint64), members=np.int64(members),
                resolution_bp=np.int64(7), bin_chrom=np.arange(b, dtype=np.int32) // 3,
                bin_start_bp=np.arange(b, dtype=np.int64) * 7, quantum_log2=np.int64(-24))


def _save(tmp_path, members):
    paths = []
    for k, d in enumerate(members):
        p = str(tmp_path / "distances" / f"member_{k}.npz")
        distances.save(p, d)
        paths.append(p)
    return paths


def test_file_round_trip_and_format(tmp_path):
    d = _member(np.random.default_rng(0))
    p = _save(tmp_path, [d])[0]
    with np.load(p) as z:
        assert set(z.files) == set(distances.KEYS)
        iu = np.triu_indices(6)
        assert z["dist_sum"].dtype == np.uint64 and np.array_equal(z["dist_sum"], d["dist_sum"][iu])
        assert int(z["quantum_log2"]) == -24
    back = distances.load(p)
    for k in distances.KEYS:
        assert back[k].dtype == np.asarray(d[k]).dtype and np.array_equal(back[k], d[k]), k
    assert not os.path.exists(p + ".tmp.npz")
    np.savez(str(tmp_path / "other.npz"), counts=np.zeros((2, 2)))
    with pytest.raises(ValueError, match="not a distances file"):
        distances.load(str(tmp_path / "other.npz"))


def test_aggregate_exact_and_order_independent(tmp_path):
    rng = np.random.default_rng(1)
    members = [_member(rng, lo=2**58, hi=2**59) for _ in range(5)]  # sums beyond 2^53: float would round
    paths = _save(tmp_path, members)
    agg = distances.aggregate(paths)
    assert int(agg["members"]) == 5
    for k in ("dist_sum", "dist2_sum", "pair_count", "bin_beads", "radial_sum", "radial2_sum"):
        want = np.array(sum(np.asarray(d[k], object) for d in members), dtype=object)
        assert agg[k].dtype == np.uint64 and (agg[k].astype(object) == want).all(), k
    out = []
    for order in (paths, paths[::-1], [paths[k] for k in (3, 0, 4, 2, 1)]):
        p = str(tmp_path / f"ens_{len(out)}.npz")
        distances.save(p, distances.aggregate(order))
        with np.load(p) as z:
            out.append({k: z[k].tobytes() for k in z.files})
    assert out[0] == out[1] == out[2]


@pytest.mark.parametrize("key,value", [("resolution_bp", np.int64(8)), ("quantum_log2", np.int64(-20)),
                                       ("bin_start_bp", np.arange(6, dtype=np.int64) * 9),
                                       ("bin_chrom", np.zeros(6, np.int32))])
def test_aggregate_refuses_mismatched_members(tmp_path, key, value):
    rng = np.random.default_rng(2)
    a, b = _member(rng), _member(rng)
    b[key] = value
    paths = _save(tmp_path, [a, b])
    with pytest.raises(ValueError, match=f"member_1.npz: {key}"):
        distances.aggregate(paths)


def test_aggregate_refuses_uint64_overflow(tmp_path):
    rng = np.random.default_rng(3)
    a, b = _member(rng), _member(rng)
    a["dist2_sum"][2, 4] = a["dist2_sum"][4, 2] = np.uint64(2**64 - 5)
    b["dist2_sum"][2, 4] = b["dist2_sum"][4, 2] = np.uint64(5)
    paths = _save(tmp_path, [a, b])
    with pytest.raises(ValueError, match="member_1.npz: dist2_sum would overflow"):
        distances.aggregate(paths)


def test_mean_rms_std_and_pair_counts(tmp_path):
    """Three members whose beads per bin differ by one at a bin edge (as shuffled members' do): [2, 1, 0, 3],
    [3, 0, 0, 3], [2, 1, 0, 3].  Written, aggregated and read back, the helpers match the plain definitions
    over every pair of every member, the diagonal counts n (n - 1) / 2 pairs, and entries without pairs are
    NaN."""
    rng = np.random.default_rng(4)
    layouts = [np.array([0, 0, 1, 3, 3, 3]), np.array([0, 0, 0, 3, 3, 3]), np.array([0, 0, 1, 3, 3, 3])]
    center = np.array([0.3, -0.2, 0.1])
    xs = [rng.normal(size=(6, 3)) for _ in range(3)]
    paths = []
    for k, (x, bins) in enumerate(zip(xs, layouts)):
        gb = contacts.GenomeBins(bins.astype(np.int32), np.zeros(4, np.int32), np.arange(4, dtype=np.int64) * 5, 5)
        dsum, d2sum = R.distance_sums(x, bins, 4)
        paths.append(str(tmp_path / f"member_{k}.npz"))
        distances.save(paths[-1], distances.result(dsum, d2sum, gb, x, center))
    acc = distances.aggregate(paths)
    assert list(acc["bin_beads"]) == [7, 2, 0, 9] and int(acc["members"]) == 3
    den = distances.pair_counts(acc)
    assert den[0, 0] == 1 + 3 + 1 and den[3, 3] == 3 * 3 and den[0, 3] == 6 + 9 + 6 and den[0, 1] == 2 + 0 + 2
    assert den[1, 1] == 0 and den[2, 2] == 0
    dist = {}
    for p in range(4):
        for q in range(4):
            dist[p, q] = [np.linalg.norm(x[i] - x[j]) for x, bins in zip(xs, layouts) for i in range(6)
                          for j in range(6) if i < j and sorted((bins[i], bins[j])) == sorted((p, q))]
    mean, rms, std = distances.mean_distance(acc), distances.rms_distance(acc), distances.std_distance(acc)
    for (p, q), v in dist.items():
        if not v:
            assert np.isnan(mean[p, q]) and np.isnan(rms[p, q]) and np.isnan(std[p, q]), (p, q)
            continue
        v = np.asarray(v)
        assert len(v) == den[p, q]
        assert abs(mean[p, q] - v.mean()) < 1e-6 and abs(rms[p, q] - np.sqrt((v * v).mean())) < 1e-6
        assert abs(std[p, q] - v.std()) < 1e-5
    rmean, rstd = distances.radial_profile(acc)
    assert np.isnan(rmean[2]) and np.isnan(rstd[2])
    for p in (0, 1, 3):
        r = np.concatenate([np.linalg.norm(x[bins == p] - center, axis=1) for x, bins in zip(xs, layouts)])
        assert abs(rmean[p] - r.mean()) < 1e-6 and abs(rstd[p] - r.std()) < 1e-5


def test_radial_sums_exact():
    rng = np.random.default_rng(5)
    x = rng.normal(size=(500, 3)) * 3.0
    c = np.array([0.1, 0.2, -0.3])
    bins = rng.integers(-1, 9, size=500)
    rs, r2s = distances.radial_sums(x, c, bins, 9)
    for p in range(9):
        d = x[bins == p] - c
        r2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        assert int(rs[p]) == sum(int(round(float(v) * 2**24)) for v in np.sqrt(r2))
        assert int(r2s[p]) == sum(int(round(float(v) * 2**24)) for v in r2)
