"""The loop readout on the host: the loop table and each member's rows against the loader's own bonds
(genome-wide with shuffling, chromosome, region, down-sampling; rows on unmodelled chromosomes and
inter-chromosomal rows), the numpy restatement of the device add (tests/loops_ref.py) against a brute-force
loop, the loops files (round trip, exact order-independent aggregation, mismatch and overflow refusals), the
readers (contact_frequency, mean/std distance, apa, apa_score) on hand-built files, and the settings."""
import os

import numpy as np
import pytest

import loops_ref as LR
from multimm_b200 import loaders, loops, synthetic
from multimm_b200.distances import quantise

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


# ---- the table against the loader -------------------------------------------------------------------------
def _with_extra_rows(tmp_path, src, seed, name="extra.bedpe"):
    """src plus rows the synthetic files lack: chrX / chrY anchors (not modelled by default), inter-chromosomal
    rows in both orders, a duplicate, a short loop, and an anchor beyond the chromosome's end."""
    rng = np.random.default_rng(seed)
    lines = open(src).read().splitlines()
    extra = [
        ("chrX", 5_000_000, 5_010_000, "chrX", 7_000_000, 7_010_000, 80.0),
        ("chr1", 30_000_000, 30_010_000, "chrY", 2_000_000, 2_010_000, 80.0),
        ("chr3", 50_000_000, 50_010_000, "chr2", 40_000_000, 40_010_000, 90.0),
        ("chr2", 40_000_000, 40_010_000, "chr3", 50_000_000, 50_010_000, 90.0),
        ("chr1", 20_000_000, 20_010_000, "chr5", 90_000_000, 90_010_000, 12.0),
        ("chr1", 25_000_000, 25_010_000, "chr7", 40_000_000, 40_010_000, 60.0),
        ("chr1", 30_000_000, 30_010_000, "chr1", 30_020_000, 30_030_000, 70.0),
    ]
    for _ in range(20):
        c = int(rng.integers(0, 22))
        a = int(rng.integers(1, loaders.CHROM_LENGTHS[c] - 3_000_000))
        extra.append((loaders.CHROM_NAMES[c], a, a + 10_000, loaders.CHROM_NAMES[int(rng.integers(0, 22))],
                      a + 1_000_000, a + 1_010_000, float(rng.integers(13, 200))))
    lines += ["\t".join(str(v) for v in r) for r in extra]
    lines.insert(len(lines) // 2, lines[3])  # a duplicate row
    path = tmp_path / name
    path.write_text("\n".join(lines) + "\n")
    return str(path)


def _check_member(bedpe, n, chrom=None, coords=None, shuffle=False, seed=0, down=1.0, threshold=0):
    lay = {}
    ms, ns, _, chr_ends, idxs = loaders.import_mns_from_bedpe(bedpe, N_beads=n, coords=coords, chrom=chrom,
                                                               path=None, shuffle=shuffle, seed=seed,
                                                               down_prob=down, threshold=threshold, layout=lay)
    tab = loops.table(bedpe, chrom, coords)
    mr = loops.member_rows(tab, lay, n, ms, ns, chrom)
    # the loader's own anchors of every row, from its own arithmetic, clamped as it clamps
    import pandas as pd

    df = loaders.loop_rows(pd.read_csv(bedpe, header=None, sep="\t"), chrom, coords)
    assert np.array_equal(tab["row"], df.index.to_numpy())
    m, nn, _, _ = loaders.loop_anchor_beads(df.reset_index(drop=True), lay["chrom_idxs"], lay["ends"], n, chrom, coords)
    m, nn = np.minimum(m, n - 1), np.minimum(nn, n - 1)
    names = {chrom} if chrom else {loaders.CHROM_NAMES[int(c)] for c in idxs}
    modelled = np.isin(tab["chrom1"], list(names)) & np.isin(tab["chrom2"], list(names))
    bonds = set(zip(ms.tolist(), ns.tolist()))
    produced = set(zip(m[modelled].tolist(), nn[modelled].tolist()))
    v, g = mr["valid"], mr["group"]
    enforced = set(zip(mr["lo"][v & (g == 0)].tolist(), mr["hi"][v & (g == 0)].tolist()))
    held = set(zip(mr["lo"][v & (g == 1)].tolist(), mr["hi"][v & (g == 1)].tolist()))
    assert (bonds & produced) <= enforced          # every bond a modelled row produces is an enforced row
    assert enforced <= bonds and not held & bonds  # ... and no held-out row is a bond
    assert not v[~modelled].any()                  # rows on unmodelled chromosomes are never measured
    assert np.all(mr["hi"][v] > mr["lo"][v] + 2)
    for s in ("lo", "hi"):                         # every anchor lies in its block
        assert np.all((mr[f"first_{s}"][v] <= mr[s][v]) & (mr[s][v] < mr[f"end_{s}"][v]))
    assert np.all((mr["first_lo"][v] >= 0) & (mr["end_hi"][v] <= n))
    return tab, mr, lay, (ms, ns)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_genome_wide_shuffled_rows_match_the_loader(tmp_path, seed):
    bedpe = _with_extra_rows(tmp_path, BEDPE, seed)
    for n, down in ((20_000, 1.0), (7_919, 0.5), (3_000, 1.0)):
        tab, mr, _, _ = _check_member(bedpe, n, shuffle=True, seed=seed, down=down)
        assert len(tab["row"]) == sum(1 for _ in open(bedpe))
        assert mr["valid"].any()  # most synthetic loops fall under min_loop_dist at these resolutions, as in the loader
        if down < 1.0:
            assert (mr["group"][mr["valid"]] == 1).sum() > 0.3 * mr["valid"].sum()


def test_shuffling_changes_the_anchors_not_the_table(tmp_path):
    bedpe = _with_extra_rows(tmp_path, BEDPE, 5)
    t0, m0, _, _ = _check_member(bedpe, 10_000, shuffle=True, seed=0)
    t1, m1, _, _ = _check_member(bedpe, 10_000, shuffle=True, seed=1)
    for k in loops.TABLE_KEYS:
        assert np.array_equal(t0[k], t1[k])
    assert not np.array_equal(m0["lo"], m1["lo"])
    # an inter-chromosomal row is measured in both members but enforced only where it points downstream
    inter = (t0["chrom1"] != t0["chrom2"]) & m0["valid"]
    assert inter.any() and np.all(m0["group"][inter & (m0["lo"] != m0["hi"])] >= 0)


def test_chromosome_region_and_downsampled_runs(tmp_path):
    bedpe = _with_extra_rows(tmp_path, BEDPE, 9)
    _check_member(bedpe, 5_000, chrom="chr1", coords=[0, loaders.CHROM_SIZES["chr1"]])
    tab, mr, _, _ = _check_member(bedpe, 2_000, chrom="chr1", coords=[10_000_000, 60_000_000])
    inter = tab["chrom2"] != "chr1"
    assert inter.any() and not mr["valid"][inter].any()  # inter-chromosomal rows pass the filter, not the table
    _check_member(bedpe, 2_000, chrom="chr1", coords=[10_000_000, 60_000_000], down=0.5, seed=4)
    _check_member(bedpe, 2_000, chrom="chr1", coords=[10_000_000, 60_000_000], threshold=100)
    p = tmp_path / "region.bedpe"
    synthetic.write_bedpe(str(p), 300, seed=3, chrom="chr2", region=(20_000_000, 80_000_000))
    _, mr, _, (ms, _) = _check_member(str(p), 1_500, chrom="chr2", coords=[20_000_000, 80_000_000], down=0.5, seed=2)
    assert (mr["group"][mr["valid"]] == 0).sum() >= len(ms)


def test_synthetic_genome_wide_file(tmp_path):
    p = tmp_path / "gw.bedpe"
    synthetic.write_bedpe(str(p), 4_000, seed=11)
    for seed in (0, 3):
        _check_member(str(p), 50_000, shuffle=True, seed=seed, down=0.7)


# ---- the restatement against brute force ------------------------------------------------------------------
def _brute(x, rows, rc, w):
    r = len(rows["bead_lo"])
    span = 2 * w + 1
    out = dict(contacts=np.zeros(r, np.uint64), dist_sum=np.zeros(r, np.uint64), dist2_sum=np.zeros(r, np.uint64),
               apa_contacts=np.zeros((2, span, span), np.uint64), apa_dist_sum=np.zeros((2, span, span), np.uint64))

    def pair(i, j):
        dx, dy, dz = x[i, 0] - x[j, 0], x[i, 1] - x[j, 1], x[i, 2] - x[j, 2]
        d2 = (dx * dx + dy * dy) + dz * dz
        return int(d2 < rc * rc), int(quantise(np.sqrt(d2))), int(quantise(d2))

    for k in range(r):
        lo, hi, g = int(rows["bead_lo"][k]), int(rows["bead_hi"][k]), int(rows["group"][k])
        c, q, q2 = pair(lo, hi)
        out["contacts"][k], out["dist_sum"][k], out["dist2_sum"][k] = c, q, q2
        for a in range(-w, w + 1):
            for b in range(-w, w + 1):
                i, j = lo + a, hi + b
                if not (rows["first_lo"][k] <= i < rows["end_lo"][k] and rows["first_hi"][k] <= j < rows["end_hi"][k]
                        and i < j):
                    continue
                c, q, _ = pair(i, j)
                out["apa_contacts"][g, a + w, b + w] += np.uint64(c)
                out["apa_dist_sum"][g, a + w, b + w] += np.uint64(q)
    return out


def _small_rows(n, chr_ends, rng, r):
    """Rows with anchors at chain and chromosome ends, inter-chromosomal rows and random ones."""
    ce = np.asarray(chr_ends)
    rows = []
    for k in range(len(ce) - 1):
        a, b = int(ce[k]), int(ce[k + 1])
        rows += [(a, b - 1), (a, a + 3), (b - 4, b - 1), (a + 1, (a + b) // 2)]
    rows += [(int(ce[1]) - 1, int(ce[2]) - 1), (0, n - 1), (int(ce[1]) - 2, int(ce[1]) + 1)]
    while len(rows) < r:
        i, j = sorted(rng.integers(0, n, size=2).tolist())
        if j > i + 2:
            rows.append((i, j))
    lo, hi = np.array([p[0] for p in rows]), np.array([p[1] for p in rows])
    blk = lambda b: np.searchsorted(ce, b, side="right") - 1  # noqa: E731
    return dict(bead_lo=lo, bead_hi=hi, first_lo=ce[blk(lo)], end_lo=ce[blk(lo) + 1], first_hi=ce[blk(hi)],
                end_hi=ce[blk(hi) + 1], group=rng.integers(0, 2, size=len(rows)))


@pytest.mark.parametrize("w", [0, 1, 3, 25])
def test_restatement_equals_brute_force(w):
    rng = np.random.default_rng(w)
    n = 90
    chr_ends = [0, 30, 31, 64, 90]  # a one-bead chromosome too
    x = rng.normal(scale=0.3, size=(n, 3))
    rows = _small_rows(n, chr_ends, rng, 40)
    rows = {k: v[rows["bead_hi"] - rows["bead_lo"] > 0] for k, v in rows.items()}
    for rc in (0.2, 0.35):
        got, want = LR.loop_sums(x, rows, rc, w), _brute(x, rows, rc, w)
        for k in want:
            assert got[k].dtype == np.uint64 and np.array_equal(got[k], want[k]), k
    assert want["apa_contacts"].sum() > 0


def test_window_pairs_equal_the_brute_force_count():
    rng = np.random.default_rng(7)
    n, chr_ends = 90, [0, 30, 31, 64, 90]
    rows = _small_rows(n, chr_ends, rng, 30)
    mr = dict(lo=rows["bead_lo"], hi=rows["bead_hi"], first_lo=rows["first_lo"], end_lo=rows["end_lo"],
              first_hi=rows["first_hi"], end_hi=rows["end_hi"], group=rows["group"],
              valid=rows["bead_hi"] > rows["bead_lo"] + 2)
    for w in (0, 2, 25):
        want = np.zeros((2, 2 * w + 1, 2 * w + 1), np.uint64)
        for k in np.flatnonzero(mr["valid"]):
            for a in range(-w, w + 1):
                for b in range(-w, w + 1):
                    i, j = mr["lo"][k] + a, mr["hi"][k] + b
                    if mr["first_lo"][k] <= i < mr["end_lo"][k] and mr["first_hi"][k] <= j < mr["end_hi"][k] and i < j:
                        want[mr["group"][k], a + w, b + w] += np.uint64(1)
        assert np.array_equal(loops.window_pairs(mr, w), want)


# ---- files ------------------------------------------------------------------------------------------------
def _member_file(tmp_path, name, seed, samples=1, window=3, n=4_000, bedpe=BEDPE):
    lay = {}
    ms, ns, *_ = loaders.import_mns_from_bedpe(bedpe, N_beads=n, path=None, shuffle=True, seed=seed, layout=lay,
                                               down_prob=0.6)
    tab = loops.table(bedpe)
    mr = loops.member_rows(tab, lay, n, ms, ns)
    rows = loops.device_rows(mr)
    rng = np.random.default_rng(seed)
    sums = None
    for _ in range(samples):
        s = LR.loop_sums(rng.normal(scale=2.0, size=(n, 3)), rows, 0.5, window)
        sums = s if sums is None else {k: sums[k] + s[k] for k in s}
    d = loops.result(tab, mr, sums, 0.5, window, samples)
    path = str(tmp_path / name)
    loops.save(path, d)
    return path, d


def test_round_trip_and_exact_order_independent_aggregate(tmp_path):
    paths, ds = zip(*[_member_file(tmp_path, f"m{i}.npz", i, samples=1 + i % 2) for i in range(3)])
    back = loops.load(paths[0])
    assert set(back) == set(loops.KEYS)
    for k in loops.KEYS:
        assert np.array_equal(back[k], ds[0][k]) and back[k].dtype == np.asarray(ds[0][k]).dtype, k
    a, b = loops.aggregate(paths), loops.aggregate(paths[::-1])
    for k in loops.KEYS:
        assert np.array_equal(a[k], b[k]), k
    for k in loops.ROW_SUMS + loops.APA_SUMS:
        assert np.array_equal(a[k], sum(d[k] for d in ds)), k
    assert int(a["members"]) == 4
    assert int(a["bead_bp_min"]) == min(int(d["bead_bp_min"]) for d in ds)
    assert int(a["bead_bp_max"]) == max(int(d["bead_bp_max"]) for d in ds)
    assert np.all(a["contacts"] <= a["measured"]) and np.all(a["enforced"] <= a["measured"])
    out = str(tmp_path / "agg.npz")
    loops.save(out, a)
    assert np.array_equal(loops.load(out)["apa_pairs"], a["apa_pairs"])


def test_aggregate_refuses_mismatches_and_overflow(tmp_path):
    p0, d0 = _member_file(tmp_path, "a.npz", 0)
    for key, val in (("radius_nm", np.float64(0.3)), ("apa_window", np.int64(4)), ("quantum_log2", np.int64(-20)),
                     ("start1", d0["start1"] + 1), ("chrom2", d0["chrom2"][::-1]), ("row", d0["row"][:-1])):
        bad = dict(d0, **{key: val})
        p = str(tmp_path / f"bad_{key}.npz")
        loops.save(p, bad)
        with pytest.raises(ValueError, match=f"bad_{key}.npz: {key} differs"):
            loops.aggregate([p0, p])
    big = dict(d0, dist_sum=np.where(d0["dist_sum"] > 0, np.uint64(2**64 - 5), np.uint64(0)))
    p = str(tmp_path / "big.npz")
    loops.save(p, big)
    with pytest.raises(ValueError, match="big.npz: dist_sum would overflow"):
        loops.aggregate([p0, p])
    with pytest.raises(ValueError, match="not a loops file"):
        np.savez(str(tmp_path / "other.npz"), counts=np.zeros(3))
        loops.load(str(tmp_path / "other.npz"))


# ---- readers on hand-built files --------------------------------------------------------------------------
def _hand(w=1):
    span = 2 * w + 1
    q = 2.0 ** 24
    d = dict(measured=np.array([4, 0, 2], np.uint64), contacts=np.array([3, 0, 0], np.uint64),
             dist_sum=np.array([4 * q, 0, 2 * 3 * q], np.uint64),
             dist2_sum=np.array([(1 + 1 + 1 + 1) * q, 0, (4 + 16) * q], np.uint64),
             apa_window=np.int64(w), quantum_log2=np.int64(-24))
    pairs = np.full((2, span, span), 10, np.uint64)
    pairs[1, 0, 0] = 0
    cont = np.zeros((2, span, span), np.uint64)
    cont[:, w, w] = [8, 5]
    cont[:, 2 * w - max(1, w // 3) + 1:, :max(1, w // 3)] = 2
    d.update(apa_pairs=pairs, apa_contacts=cont, apa_dist_sum=(pairs * np.uint64(q)).astype(np.uint64))
    return d


def test_readers_on_a_hand_built_file():
    d = _hand(1)
    f = loops.contact_frequency(d)
    assert f[0] == 0.75 and np.isnan(f[1]) and f[2] == 0.0
    m = loops.mean_distance(d)
    assert m[0] == 1.0 and np.isnan(m[1]) and m[2] == 3.0
    s = loops.std_distance(d)
    assert s[0] == 0.0 and s[2] == 1.0  # distances 2 and 4: mean 3, rms^2 10
    freq, dist = loops.apa(d, 0)
    assert freq[1, 1] == 0.8 and freq[2, 0] == 0.2 and freq[0, 2] == 0.0 and np.all(dist == 1.0)
    freq1, dist1 = loops.apa(d, 1)
    assert np.isnan(freq1[0, 0]) and np.isnan(dist1[0, 0]) and freq1[1, 1] == 0.5
    assert loops.apa_score(d, 0) == pytest.approx(4.0) and loops.apa_score(d, 1) == pytest.approx(2.5)


def test_apa_score_corner_is_juicers_at_w10():
    d = _hand(10)
    freq, _ = loops.apa(d, 0)
    assert np.all(freq[18:, :3] == 0.2) and freq[17, 0] == 0.0 and freq[18, 3] == 0.0
    assert loops.apa_score(d, 0) == pytest.approx(0.8 / 0.2)
    d0 = _hand(0)
    assert loops.apa_score(d0, 0) == pytest.approx(1.0)  # k = 1 at W = 0: the corner is the centre
    d["apa_contacts"][0, 18:, :3] = 0
    assert np.isnan(loops.apa_score(d, 0))


# ---- settings ---------------------------------------------------------------------------------------------
def _cfg(tmp_path, **kw):
    from multimm_b200.config import SimulationConfig

    base = dict(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    base.update(kw)
    return SimulationConfig(**base)


def test_settings_are_extras_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import EXTRA_FIELDS, LOOP_FIELDS, SimulationConfig, contact_setting

    assert set(LOOP_FIELDS) == {"SAVE_LOOPS", "LOOP_APA_WINDOW"} and set(LOOP_FIELDS) <= set(EXTRA_FIELDS)
    plain = _cfg(tmp_path)
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert contact_setting(plain, "SAVE_LOOPS") is False and contact_setting(plain, "LOOP_APA_WINDOW") == 10
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\nSAVE_LOOPS = True\n")
    args, _ = run.get_config(["-c", str(ini), "--loop_apa_window", "5"])
    assert contact_setting(args, "SAVE_LOOPS") is True and contact_setting(args, "LOOP_APA_WINDOW") == 5


@pytest.mark.parametrize("w", [-1, 26])
def test_bad_window_refused_before_any_output(tmp_path, w):
    from multimm_b200 import run

    with pytest.raises(ValueError, match="LOOP_APA_WINDOW"):
        run.args_tests(_cfg(tmp_path, SAVE_LOOPS=True, LOOP_APA_WINDOW=w))
    assert not (tmp_path / "o").exists()


def test_md_sampling_accepts_the_loop_readout_alone(tmp_path):
    from multimm_b200 import run

    for w in (0, 25):
        run.args_tests(_cfg(tmp_path, SAVE_LOOPS=True, LOOP_APA_WINDOW=w, SIM_RUN_MD=True, SIM_N_STEPS=1000,
                            SIM_SAMPLING_STEP=100, MD_SAMPLE_STEP=200))
    with pytest.raises(ValueError, match="SAVE_CONTACTS or SAVE_DISTANCES"):
        run.args_tests(_cfg(tmp_path, SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100, MD_SAMPLE_STEP=200))
