"""Host loaders against golden outputs of the REFERENCE's own functions
(tests/golden/loaders_golden.npz, produced by tests/golden/make_golden.py importing
$MULTIMM_REFERENCE/src/multimm/utils.py).  Integer arrays must match exactly."""
import os

import numpy as np
import pytest

from common import NO_REFERENCE, reference_file
from multimm_b200 import loaders

GOLD = os.path.join(os.path.dirname(__file__), "golden")
G = np.load(os.path.join(GOLD, "loaders_golden.npz"))
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")
BED = os.path.join(GOLD, "synthetic_subcompartments.bed")
REF_FIXTURE = reference_file("tests/fixtures/ENCFF045MJY_simple.bedpe")

CASES = {
    "gw_20k": dict(N_beads=20000, chrom=None, coords=None, shuffle=False, seed=0),
    "gw_20k_shuffle3": dict(N_beads=20000, chrom=None, coords=None, shuffle=True, seed=3),
    "gw_5k_down": dict(N_beads=5000, chrom=None, coords=None, shuffle=True, seed=1, down_prob=0.8),
    "chr1_region": dict(N_beads=2000, chrom="chr1", coords=[10_000_000, 110_000_000], shuffle=False, seed=0),
    "chr6_whole": dict(N_beads=3000, chrom="chr6", coords=[0, 172126628], shuffle=False, seed=2),
}
BED_EXTRA = {"gw_5k_down": dict(flip_prob=0.2, noise_strength=0.5), "chr1_region": dict(flip_prob=0.1)}


@pytest.mark.parametrize("name", list(CASES))
def test_bedpe_matches_reference(name):
    kw = dict(CASES[name])
    ms, ns, ds, ce, ci = loaders.import_mns_from_bedpe(BEDPE, path=None, **kw)
    assert np.array_equal(ms, G[f"{name}.ms"])
    assert np.array_equal(ns, G[f"{name}.ns"])
    assert np.array_equal(ce, G[f"{name}.loop_chr_ends"])
    assert np.array_equal(ci, G[f"{name}.loop_chrom_idxs"])
    assert np.allclose(ds, G[f"{name}.ds"], rtol=1e-13, atol=0)
    assert ds.min() >= 0.1 - 1e-12 and ds.max() <= 0.2 + 1e-12
    assert np.all(ns > ms + 2)


@pytest.mark.parametrize("name", list(CASES))
def test_bed_matches_reference(name):
    kw = {k: v for k, v in CASES[name].items() if k != "down_prob"}
    cs, ce, ci = loaders.import_bed(BED, save_path=None, **kw, **BED_EXTRA.get(name, {}))
    assert np.array_equal(cs, G[f"{name}.Cs"])
    assert np.array_equal(ce, G[f"{name}.bed_chr_ends"])
    assert np.array_equal(ci, G[f"{name}.bed_chrom_idxs"])
    assert set(np.unique(cs)) <= {-2, -1, 0, 1, 2}


def test_resolutions_differ_between_loaders():
    """Appendix A, Q4: the bed loader divides the genome length, the bedpe loader the largest loop
    coordinate, so the two chr_ends are slightly different; the model keeps the bedpe one."""
    a = G["gw_20k.loop_chr_ends"]
    b = G["gw_20k.bed_chr_ends"]
    assert a[0] == b[0] == 0 and a[-1] == b[-1] == 20000
    assert len(a) == len(b) == 23


def test_chrom_strength_table():
    assert np.allclose(loaders.CHROM_STRENGTH, G["chrom_strength"], rtol=0, atol=0)
    assert loaders.CHROM_STRENGTH[0] == 0.0 and loaders.CHROM_STRENGTH[20] == 1.0  # chr1, chr21


@pytest.mark.skipif(REF_FIXTURE is None, reason=NO_REFERENCE)
@pytest.mark.parametrize("n_beads,chrom,coords", [(1000, None, None), (200000, None, None),
                                                  (10000, "chr1", [0, 248387328])])
def test_reference_fixture(n_beads, chrom, coords):
    """The one data fixture the reference ships (tests/fixtures/ENCFF045MJY_simple.bedpe)."""
    key = f"fixture_{n_beads}_{chrom or 'gw'}"
    ms, ns, ds, ce, _ = loaders.import_mns_from_bedpe(REF_FIXTURE, N_beads=n_beads, chrom=chrom, coords=coords,
                                                      path=None)
    assert np.array_equal(ms, G[f"{key}.ms"]) and np.array_equal(ns, G[f"{key}.ns"])
    assert np.array_equal(ce, G[f"{key}.chr_ends"])
    assert np.allclose(ds, G[f"{key}.ds"], rtol=1e-13, atol=0)


def test_empty_region_raises(tmp_path):
    with pytest.raises(ValueError, match="does not include loops"):
        loaders.import_mns_from_bedpe(BEDPE, N_beads=100, chrom="chr1", coords=[5, 6], path=None)


def test_equal_counts_give_unit_distances(tmp_path):
    # utils.py:520: all counts equal -> ds = 1.0 everywhere
    p = tmp_path / "eq.bedpe"
    rows = [f"chr1\t{a}\t{a + 10000}\tchr1\t{a + 900000}\t{a + 910000}\t5.0" for a in range(100000, 5000000, 400000)]
    p.write_text("\n".join(rows) + "\n")
    ms, ns, ds, _, _ = loaders.import_mns_from_bedpe(str(p), N_beads=1000, chrom="chr1", coords=[0, 10_000_000],
                                                    path=None)
    assert len(ms) > 0 and np.all(ds == 1.0)
