"""The fine (sparse) contact map on the host: the CONTACT_FINE_RESOLUTION setting and its checks, genomic
bins beyond the dense cap, the fine file format, its exact aggregation, and the coarsen / fine_block views."""
import os

import numpy as np
import pytest

from multimm_b200 import contacts, loaders

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


def _layout(n=4000, shuffle=False, seed=0, chrom=None, coords=None):
    lay = {}
    loaders.import_mns_from_bedpe(BEDPE, N_beads=n, chrom=chrom, coords=coords, path=None, shuffle=shuffle,
                                  seed=seed, layout=lay)
    return lay


# ---- config --------------------------------------------------------------------------------------------
def test_fine_setting_is_an_extra_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import CONTACT_FINE_FIELDS, CONTACT_FIELDS, SimulationConfig, contact_setting

    assert "CONTACT_FINE_RESOLUTION" not in CONTACT_FIELDS
    assert not set(CONTACT_FINE_FIELDS) & set(SimulationConfig.model_fields)
    plain = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert contact_setting(plain, "CONTACT_FINE_RESOLUTION") == 0
    given = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), SAVE_CONTACTS="yes",
                             CONTACT_FINE_RESOLUTION="5000")
    again = SimulationConfig(**given.model_dump())
    assert contact_setting(again, "CONTACT_FINE_RESOLUTION") == 5000
    with pytest.raises(ValueError):
        SimulationConfig(LOOPS_PATH=BEDPE, CONTACT_FINE_RESOLUTION="fine")

    # the same dumps as without the extension when it is not given, and the CLI reaches it
    def dumps(name, *extra):
        ini = tmp_path / f"{name}.ini"
        ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / name}\n")
        args, _ = run.get_config(["-c", str(ini), *extra])
        return args, (tmp_path / name / "metadata" / "config_auto.ini").read_text()

    _, plain_ini = dumps("a")
    _, plain_ini2 = dumps("b")
    assert "contact_fine" not in plain_ini and plain_ini.replace(str(tmp_path / "a"), "") == \
        plain_ini2.replace(str(tmp_path / "b"), "")
    args, ini = dumps("c", "--contact_fine_resolution", "10000", "--save_contacts", "true")
    assert contact_setting(args, "CONTACT_FINE_RESOLUTION") == 10_000 and "contact_fine_resolution = 10000" in ini
    run.args_tests(args)


@pytest.mark.parametrize("fields", [dict(CONTACT_FINE_RESOLUTION=-1), dict(CONTACT_FINE_RESOLUTION=1),
                                    dict(CONTACT_FINE_RESOLUTION=1, CHROM="chr1", LOC_START=0,
                                         LOC_END=3_000_000_000)])
def test_bad_fine_resolution_refused_before_any_output(tmp_path, fields):
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    out = tmp_path / "out"
    args = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(out), SAVE_CONTACTS=True, **fields)
    with pytest.raises(ValueError, match="CONTACT_FINE_RESOLUTION"):
        run.args_tests(args)
    assert not out.exists()


def test_fine_resolution_valid_values(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    for res in (0, 5000, 2):  # 2 bp genome-wide: 1.4e9 bins, still int32
        run.args_tests(SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), SAVE_CONTACTS=True,
                                        CONTACT_FINE_RESOLUTION=res))


# ---- bins ----------------------------------------------------------------------------------------------
def test_genome_bins_beyond_the_dense_cap():
    lay = _layout()
    with pytest.raises(ValueError, match="4096"):
        contacts.genome_bins(lay, 50_000)
    gb = contacts.genome_bins(lay, 50_000, max_bins=contacts.MAX_FINE_BINS)
    assert gb.n_bins == contacts.bin_count(contacts.spans(range(22)), 50_000) > contacts.MAX_BINS
    coarse = contacts.genome_bins(lay, 5_000_000)
    # both grids start at every chromosome's lo: coarse bin = first coarse bin of the chromosome + fine offset // k
    first_f = {c: int(np.flatnonzero(gb.bin_chrom == c)[0]) for c in range(22)}
    first_c = {c: int(np.flatnonzero(coarse.bin_chrom == c)[0]) for c in range(22)}
    ch = gb.bin_chrom[gb.bins]
    want = np.array([first_c[c] for c in ch]) + (gb.bins - np.array([first_f[c] for c in ch])) // 100
    assert np.array_equal(coarse.bins, want)


# ---- files ---------------------------------------------------------------------------------------------
def _fine_member(rng, gb, nnz=300, members=1):
    """A random sparse upper triangle over gb's bins, as Engine.contacts_sparse returns it."""
    nb = gb.n_bins
    p, q = rng.integers(0, nb, size=(2, nnz))
    keys = np.unique(np.minimum(p, q).astype(np.int64) * nb + np.maximum(p, q))
    vals = rng.integers(1, 2**40, size=len(keys)).astype(np.uint64)
    return contacts.fine_result((keys // nb).astype(np.int32), (keys % nb).astype(np.int32), vals,
                                int(rng.integers(0, 10**6)), 0.2, gb, members)


def _dense(d):
    nb = int(d["n_bins"])
    out = np.zeros((nb, nb), np.uint64)
    out[d["rows"], d["cols"]] = d["vals"]
    out[d["cols"], d["rows"]] = d["vals"]
    return out


def _small_bins():
    """Fine bins over three short chromosomes: 7, 10 and 3 bins of 1000 bp."""
    chrom = np.repeat(np.array([0, 4, 9], np.int32), [7, 10, 3])
    start = np.concatenate([np.arange(7), np.arange(10), np.arange(3)]).astype(np.int64) * 1000
    return contacts.GenomeBins(np.zeros(10, np.int32), chrom, start, 1000)


def test_fine_file_round_trip_and_load_refuses_it(tmp_path):
    rng = np.random.default_rng(0)
    d = _fine_member(rng, _small_bins())
    p = str(tmp_path / "contacts_fine.npz")
    contacts.save_fine(p, d)
    with np.load(p) as z:
        assert set(z.files) == set(contacts.FINE_KEYS) and "counts" not in z.files
    back = contacts.load_fine(p)
    for k in contacts.FINE_KEYS:
        assert back[k].dtype == np.asarray(d[k]).dtype and np.array_equal(back[k], d[k]), k
    with pytest.raises(ValueError, match="load_fine"):
        contacts.load(p)


def test_aggregate_fine_exact_and_order_independent(tmp_path):
    rng = np.random.default_rng(1)
    gb = _small_bins()
    members = [_fine_member(rng, gb, nnz=int(n)) for n in (0, 40, 150, 300, 5)]
    paths = []
    for k, d in enumerate(members):
        paths.append(str(tmp_path / f"member_{k}_fine.npz"))
        contacts.save_fine(paths[-1], d)
    agg = contacts.aggregate_fine(paths)
    assert np.array_equal(_dense(agg), sum(_dense(d) for d in members))
    keys = agg["rows"].astype(np.int64) * int(agg["n_bins"]) + agg["cols"]
    assert np.all(np.diff(keys) > 0) and np.all(agg["rows"] <= agg["cols"]) and np.all(agg["vals"] > 0)
    assert int(agg["members"]) == 5 and int(agg["pairs"]) == sum(int(d["pairs"]) for d in members)
    for order in ([4, 3, 2, 1, 0], [2, 0, 4, 1, 3]):
        other = contacts.aggregate_fine([paths[k] for k in order])
        for k in contacts.FINE_KEYS:
            assert agg[k].dtype == other[k].dtype and agg[k].tobytes() == other[k].tobytes(), k


@pytest.mark.parametrize("key,value", [("resolution_bp", np.int64(500)), ("radius_nm", np.float64(0.3)),
                                       ("bin_start_bp", None)])
def test_aggregate_fine_refuses_mismatches(tmp_path, key, value):
    rng = np.random.default_rng(2)
    a, b = _fine_member(rng, _small_bins()), _fine_member(rng, _small_bins())
    b[key] = value if value is not None else b[key] + 1
    contacts.save_fine(str(tmp_path / "a.npz"), a)
    contacts.save_fine(str(tmp_path / "b.npz"), b)
    with pytest.raises(ValueError, match=key):
        contacts.aggregate_fine([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])
    with pytest.raises(ValueError):
        contacts.aggregate_fine([])


def test_coarsen_equals_numpy_sum():
    rng = np.random.default_rng(3)
    gb = _small_bins()
    d = _fine_member(rng, gb, nnz=200)
    dense = _dense(d)
    for k in (1, 2, 3, 7):
        # coarse bin = the chromosome's first coarse bin + fine offset // k, as a 0/1 matrix P
        chrom = gb.bin_chrom
        cmap, nb = [], 0
        for c in (0, 4, 9):
            m = int(np.count_nonzero(chrom == c))
            cmap.extend(nb + np.arange(m) // k)
            nb += -(-m // k)
        P = np.zeros((len(chrom), nb), np.uint64)
        P[np.arange(len(chrom)), cmap] = 1
        up = P.T @ np.triu(dense) @ P  # each contact once; a pair inside one coarse bin adds 1 to (a, a) once
        assert np.array_equal(contacts.coarsen(d, 1000 * k), up + up.T - np.diag(np.diag(up))), k
    with pytest.raises(ValueError, match="multiple"):
        contacts.coarsen(d, 1500)


def test_coarsen_matches_genome_bins_of_a_real_layout():
    rng = np.random.default_rng(4)
    lay = _layout()
    fine = contacts.genome_bins(lay, 100_000, max_bins=contacts.MAX_FINE_BINS)
    coarse = contacts.genome_bins(lay, 5_000_000)
    i, j = rng.integers(0, 4000, size=(2, 20_000))
    p, q = np.minimum(fine.bins[i], fine.bins[j]).astype(np.int64), np.maximum(fine.bins[i], fine.bins[j])
    keys, vals = np.unique(p * fine.n_bins + q, return_counts=True)
    d = contacts.fine_result(keys // fine.n_bins, keys % fine.n_bins, vals, len(i), 0.2, fine)
    want = np.zeros((coarse.n_bins, coarse.n_bins), np.uint64)
    np.add.at(want, (coarse.bins[i], coarse.bins[j]), np.uint64(1))
    off = coarse.bins[i] != coarse.bins[j]
    np.add.at(want, (coarse.bins[j][off], coarse.bins[i][off]), np.uint64(1))
    assert np.array_equal(contacts.coarsen(d, 5_000_000), want)


def test_fine_block_equals_the_dense_block():
    rng = np.random.default_rng(5)
    gb = _small_bins()
    d = _fine_member(rng, gb, nnz=200)
    dense = _dense(d)
    block, starts = contacts.fine_block(d, loaders.CHROM_NAMES[4], 2500, 6000)  # bins 2..5 of the 2nd chromosome
    assert np.array_equal(starts, [2000, 3000, 4000, 5000])
    assert np.array_equal(block, dense[9:13, 9:13])
    block, starts = contacts.fine_block(d, 9, 0, 10**9)
    assert np.array_equal(block, dense[17:20, 17:20]) and len(starts) == 3
    assert contacts.fine_block(d, 1, 0, 10**9)[0].shape == (0, 0)
