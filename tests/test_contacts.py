"""Contact maps on the host: the numpy restatement against brute force, canonical genomic bins (unshuffled,
shuffled, chromosome and region layouts), the SAVE_CONTACTS config checks, and the file format and its
aggregation over ensemble members."""
import os

import numpy as np
import pytest

import contacts_ref as R
from multimm_b200 import contacts, loaders

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


def _layout(n=4000, shuffle=False, seed=0, chrom=None, coords=None):
    lay = {}
    loaders.import_mns_from_bedpe(BEDPE, N_beads=n, chrom=chrom, coords=coords, path=None, shuffle=shuffle,
                                  seed=seed, layout=lay)
    return lay


# ---- the numpy restatement ----------------------------------------------------------------------------
@pytest.mark.parametrize("n,scale,rc", [(300, 1.0, 0.2), (517, 0.6, 0.15), (800, 2.0, 0.5)])
def test_reference_matches_brute_force(n, scale, rc):
    x = np.random.default_rng(n).uniform(-scale, scale, size=(n, 3))
    i, j = R.contact_pairs(x, rc)
    bi, bj = R.brute_pairs(x, rc)
    assert len(i) > 0
    order = np.lexsort((j, i)), np.lexsort((bj, bi))
    assert np.array_equal(i[order[0]], bi[order[1]]) and np.array_equal(j[order[0]], bj[order[1]])


def test_reference_lattice_boundary():
    """On a 0.1 nm lattice the neighbours sit at the threshold: the exact test decides, and both
    enumerations decide the same."""
    g = np.stack(np.meshgrid(*[np.arange(6)] * 3, indexing="ij"), -1).reshape(-1, 3) * 0.1
    for rc in (0.1, 0.1 * (1 + 1e-12), 0.1 * (1 - 1e-12)):
        i, j = R.contact_pairs(g, rc)
        bi, bj = R.brute_pairs(g, rc)
        assert len(i) == len(bi)
    assert len(R.brute_pairs(g, 0.1 * (1 + 1e-9))[0]) > len(R.brute_pairs(g, 0.1 * (1 - 1e-9))[0])


def test_reference_counts_symmetric_and_sep():
    rng = np.random.default_rng(5)
    x = rng.uniform(0, 1.2, size=(600, 3))
    bins = rng.integers(-1, 7, size=600)
    chrom = np.repeat([0, 1, 2], 200)
    cmap, sep, pairs = R.contact_counts(x, 0.2, bins, 7, chrom)
    i, j = R.brute_pairs(x, 0.2)
    assert np.array_equal(cmap, cmap.T) and pairs == len(i)
    ok = (bins[i] >= 0) & (bins[j] >= 0)
    assert int(np.trace(cmap)) + int(np.triu(cmap, 1).sum()) == int(ok.sum())
    assert int(sep.sum()) == int(np.count_nonzero(chrom[i] == chrom[j])) and sep[0] == 0


# ---- genomic bins ------------------------------------------------------------------------------------
def test_genome_wide_unshuffled_bins():
    lay = _layout()
    gb = contacts.genome_bins(lay)
    assert gb.n_bins <= contacts.AUTO_BINS
    assert np.all(np.diff(gb.bins) >= 0)  # chromosomes in CHROM_NAMES order, positions increasing
    assert list(np.unique(gb.bin_chrom)) == list(range(22))
    chrom, bp = contacts.bead_loci(lay, 4000)
    assert np.array_equal(gb.bin_chrom[gb.bins], chrom)
    assert np.all(gb.bin_start_bp[gb.bins] <= bp) and np.all(bp < gb.bin_start_bp[gb.bins] + gb.resolution_bp)
    # no bin straddles a chromosome
    for c in range(22):
        starts = gb.bin_start_bp[gb.bin_chrom == c]
        assert starts[0] == 0 and starts[-1] < loaders.CHROM_LENGTHS[c] <= starts[-1] + gb.resolution_bp


@pytest.mark.parametrize("chrom,coords", [("chr1", [0, loaders.CHROM_SIZES["chr1"]]), ("chr2", [10_000_000, 60_000_000])])
def test_chromosome_and_region_bins(chrom, coords):
    lay = _layout(n=2000, chrom=chrom, coords=coords)
    gb = contacts.genome_bins(lay)
    assert gb.n_bins <= contacts.AUTO_BINS
    assert np.all(gb.bin_chrom == loaders._chrom_index(chrom))
    assert gb.bin_start_bp[0] == coords[0] and gb.bin_start_bp[-1] < coords[1] <= gb.bin_start_bp[-1] + gb.resolution_bp
    assert gb.bins[0] == 0 and np.all(np.diff(gb.bins) >= 0)
    _, bp = contacts.bead_loci(lay, 2000)
    assert bp.min() >= coords[0] and bp.max() < coords[1]
    # an explicit resolution
    gb2 = contacts.genome_bins(lay, 1_000_000)
    assert gb2.resolution_bp == 1_000_000 and gb2.n_bins == -(-(coords[1] - coords[0]) // 1_000_000)


@pytest.mark.parametrize("seed", [1, 4])
def test_shuffled_member_maps_to_the_same_loci(seed):
    """Bead i is a different locus in every shuffled member; its canonical (chromosome, bp) is still where the
    unshuffled layout puts the same stretch of genome, to within one bead width."""
    n = 4000
    lu, ls = _layout(n), _layout(n, shuffle=True, seed=seed)
    assert not np.array_equal(ls["chrom_idxs"], lu["chrom_idxs"])
    cu, bu = contacts.bead_loci(lu, n)
    cs, bs = contacts.bead_loci(ls, n)
    width = max(lu["resolution"], ls["resolution"])
    for c in range(22):
        ref = np.sort(bu[cu == c])
        q = bs[cs == c]
        k = np.clip(np.searchsorted(ref, q), 1, len(ref) - 1)
        near = np.minimum(np.abs(q - ref[k - 1]), np.abs(q - ref[k]))
        assert near.max() <= width, (c, near.max(), width)
    # one bin table for both: bin p is the same locus in every member
    gu = contacts.genome_bins(lu, 5_000_000)
    gs = contacts.genome_bins(ls, 5_000_000)
    assert np.array_equal(gu.bin_chrom, gs.bin_chrom) and np.array_equal(gu.bin_start_bp, gs.bin_start_bp)
    assert np.array_equal(gs.bin_chrom[gs.bins], cs)


@pytest.mark.parametrize("shuffle,seed", [(False, 0), (True, 2)])
def test_loop_anchors_fall_in_their_midpoint_bins(shuffle, seed):
    import pandas as pd

    n = 40000
    lay = {}
    ms, ns, _, _, _ = loaders.import_mns_from_bedpe(BEDPE, N_beads=n, path=None, shuffle=shuffle, seed=seed, layout=lay)
    gb = contacts.genome_bins(lay, 2_000_000)
    chrom, bp = contacts.bead_loci(lay, n)
    res = lay["resolution"]
    df = pd.read_csv(BEDPE, header=None, sep="\t")
    pos = {int(c): k for k, c in enumerate(lay["chrom_idxs"])}
    got = crossed = 0
    anchors = set(map(tuple, np.stack([ms, ns], 1)))
    for row in df.itertuples(index=False):
        c = loaders._chrom_index(row[0])
        if c not in pos:
            continue
        off = int(lay["ends"][pos[c]])
        m = ((row[1] + off) // res + (row[2] + off) // res) // 2
        nn = ((row[4] + off) // res + (row[5] + off) // res) // 2
        if (m, nn) not in anchors:
            continue
        for bead, mid in ((m, (row[1] + row[2]) // 2), (nn, (row[4] + row[5]) // 2)):
            if chrom[bead] != c:  # the loader puts a locus within one bead of a chromosome's end into the next block
                assert mid + 2 * res >= loaders.CHROM_LENGTHS[c]
                crossed += 1
                continue
            assert abs(bp[bead] - mid) <= res
            b_mid = int(np.searchsorted(gb.bin_start_bp[gb.bin_chrom == c], mid, side="right") - 1
                        + np.flatnonzero(gb.bin_chrom == c)[0])
            edge = min(abs(mid - gb.bin_start_bp[b_mid]), abs(gb.bin_start_bp[b_mid] + gb.resolution_bp - mid))
            assert gb.bins[bead] == b_mid or edge <= res
            got += 1
    assert got > 500 and crossed <= got // 50


def test_automatic_resolution_stays_within_1000_bins():
    for lay in (_layout(), _layout(shuffle=True, seed=3), _layout(n=2000, chrom="chr21", coords=[0, loaders.CHROM_SIZES["chr21"]]),
                _layout(n=2000, chrom="chr1", coords=[5_000_000, 60_000_000 + 123])):
        gb = contacts.genome_bins(lay)
        assert 900 <= gb.n_bins <= 1000


def test_too_many_bins_refused():
    with pytest.raises(ValueError, match="4096"):
        contacts.genome_bins(_layout(), 100_000)


# ---- config --------------------------------------------------------------------------------------------
def test_contact_settings_are_extras_present_only_when_given(tmp_path):
    """SAVE_CONTACTS / CONTACT_RADIUS / CONTACT_RESOLUTION are validated like fields, but a config without
    them has the same fields and dumps as before; given, they survive a dump and reload (the ensemble
    driver rebuilds every member's config from the dump) and reach the command line."""
    from multimm_b200 import run
    from multimm_b200.config import CONTACT_FIELDS, SimulationConfig, contact_setting

    plain = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), NOT_A_FIELD=1)
    assert not set(CONTACT_FIELDS) & set(SimulationConfig.model_fields)
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert [contact_setting(plain, k) for k in CONTACT_FIELDS] == [False, 0.2, 0]
    given = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), SAVE_CONTACTS="yes",
                             CONTACT_RADIUS="0.25", CONTACT_RESOLUTION="2000000")
    again = SimulationConfig(**given.model_dump())
    assert [contact_setting(again, k) for k in CONTACT_FIELDS] == [True, 0.25, 2_000_000]
    with pytest.raises(ValueError):
        SimulationConfig(LOOPS_PATH=BEDPE, CONTACT_RESOLUTION="many")
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\nSAVE_CONTACTS = true\n")
    args, _ = run.get_config(["-c", str(ini), "--contact_radius", "0.3"])
    assert contact_setting(args, "SAVE_CONTACTS") is True and contact_setting(args, "CONTACT_RADIUS") == 0.3
    assert "save_contacts = True" in (tmp_path / "cli" / "metadata" / "config_auto.ini").read_text()


@pytest.mark.parametrize("fields", [dict(CONTACT_RADIUS=0.0), dict(CONTACT_RADIUS=-0.2), dict(CONTACT_RADIUS="nan"),
                                    dict(CONTACT_RADIUS="inf"), dict(CONTACT_RESOLUTION=-5),
                                    dict(CONTACT_RESOLUTION=100_000),
                                    dict(CONTACT_RESOLUTION=10_000, CHROM="chr1", LOC_START=0, LOC_END=50_000_000)])
def test_bad_contact_fields_refused_before_any_output(tmp_path, fields):
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    out = tmp_path / "out"
    args = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(out), SAVE_CONTACTS=True, **fields)
    with pytest.raises(ValueError, match="CONTACT_"):
        run.args_tests(args)
    assert not out.exists()


def test_contact_fields_defaults_and_valid_values(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    args = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    run.args_tests(args)
    run.args_tests(SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), SAVE_CONTACTS="yes",
                                    CONTACT_RESOLUTION=1_000_000))


# ---- files and aggregation -------------------------------------------------------------------------------
def _member(rng, b=9, n=50):
    m = rng.integers(0, 5, size=(b, b)).astype(np.uint64)
    m = np.triu(m) + np.triu(m, 1).T
    gb = contacts.GenomeBins(np.zeros(n, np.int32), np.arange(b, dtype=np.int32) // 3, np.arange(b, dtype=np.int64) * 7, 7)
    chrom = np.repeat([0, 1, 2], [20, 17, 13])
    return contacts.result(m, rng.integers(0, 9, size=n).astype(np.uint64), int(rng.integers(0, 999)), 0.2, gb,
                           contacts.sep_pairs(chrom))


def test_member_files_sum_to_the_dense_ensemble_file(tmp_path):
    rng = np.random.default_rng(0)
    members = [_member(rng) for _ in range(4)]
    paths = []
    for k, d in enumerate(members):
        p = str(tmp_path / "contacts" / f"member_{k}.npz")
        contacts.save_member(p, d)
        paths.append(p)
        back = contacts.load(p)
        assert np.array_equal(back["counts"], d["counts"]) and back["counts"].dtype == np.uint64
    agg = contacts.aggregate(paths[::-1])
    assert int(agg["members"]) == 4
    assert np.array_equal(agg["counts"], sum(d["counts"] for d in members))
    assert np.array_equal(agg["sep_contacts"], sum(d["sep_contacts"] for d in members))
    assert np.array_equal(agg["sep_pairs"], sum(d["sep_pairs"] for d in members))
    assert int(agg["pairs"]) == sum(int(d["pairs"]) for d in members)
    contacts.save_dense(str(tmp_path / "ensemble_contacts.npz"), agg)
    back = contacts.load(str(tmp_path / "ensemble_contacts.npz"))
    for k in ("counts", "members", "radius_nm", "resolution_bp", "bin_chrom", "bin_start_bp", "sep_contacts",
              "sep_pairs", "pairs"):
        assert np.array_equal(back[k], agg[k]), k


def test_aggregate_refuses_mismatched_bins(tmp_path):
    rng = np.random.default_rng(1)
    a, b = _member(rng), _member(rng)
    b["resolution_bp"] = np.int64(8)
    contacts.save_member(str(tmp_path / "a.npz"), a)
    contacts.save_member(str(tmp_path / "b.npz"), b)
    with pytest.raises(ValueError, match="resolution_bp"):
        contacts.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])


@pytest.mark.parametrize("lengths", [[40], [7, 30, 1, 12], [25, 25]])
def test_sep_pairs_denominator_brute_force(lengths):
    chrom = np.repeat(np.arange(len(lengths)) * 3 % 5, lengths)
    n = len(chrom)
    i, j = np.triu_indices(n, k=1)
    same = chrom[i] == chrom[j]
    brute = np.bincount(j[same] - i[same], minlength=n)[:n]
    assert np.array_equal(contacts.sep_pairs(chrom), brute.astype(np.uint64))
    d = dict(sep_contacts=brute // 2, sep_pairs=contacts.sep_pairs(chrom))
    p = contacts.contact_probability(d)
    assert np.isnan(p[0]) and np.all(p[1:max(lengths)] <= 1.0)
