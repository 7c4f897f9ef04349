"""Randomised differential test of the host loaders against the REFERENCE's own functions, run live
($MULTIMM_REFERENCE/src/multimm/utils.py: import_mns_from_bedpe :425, import_bed :220).  Only where the
reference checkout exists (MULTIMM_REFERENCE); the frozen cases of test_loaders.py run
everywhere.  Integer outputs must be identical, distances equal to the last bit or two."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from common import NO_REFERENCE, reference_file
from multimm_b200 import loaders, synthetic

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.skipif(reference_file("src/multimm/utils.py") is None, reason=NO_REFERENCE)


@pytest.fixture(scope="module")
def ref():
    """The reference's utils.py; the stand-in modules planted for its imports are removed afterwards."""
    before = set(sys.modules)
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    yield mg.load_reference_utils()
    for name in set(sys.modules) - before:
        del sys.modules[name]


def draw_case(seed):
    rng = np.random.default_rng(1000 + seed)
    kind = seed % 3
    if kind == 0:  # genome-wide
        n_chroms = int(rng.integers(2, 23))
        return dict(n_chroms=n_chroms, chrom=None, coords=None, N_beads=int(rng.integers(6000, 40000)),
                    n_loops=int(rng.integers(80, 900)), shuffle=bool(rng.integers(0, 2)), seed=int(rng.integers(0, 50)),
                    down_prob=float(rng.choice([1.0, 1.0, 0.7, 0.35])))
    chrom = loaders.CHROM_NAMES[int(rng.integers(0, 22))]
    size = loaders.CHROM_SIZES[chrom]
    if kind == 1:  # whole chromosome
        coords = [0, int(size)]
    else:  # region
        a = int(rng.integers(0, size // 2))
        coords = [a, int(a + rng.integers(size // 8, size // 2))]
    return dict(n_chroms=22, chrom=chrom, coords=coords, N_beads=int(rng.integers(200, 3000)),
                n_loops=int(rng.integers(40, 500)), shuffle=False, seed=0,
                down_prob=float(rng.choice([1.0, 0.6])))


@pytest.mark.parametrize("seed", range(18))
def test_bedpe_loader_equals_the_reference(ref, tmp_path, seed):
    c = draw_case(seed)
    bedpe = str(tmp_path / "loops.bedpe")
    synthetic.write_bedpe(bedpe, n_loops=c["n_loops"], seed=seed, chrom=c["chrom"],
                          region=c["coords"] if seed % 3 == 2 else None, n_chroms=c["n_chroms"])
    kw = dict(N_beads=c["N_beads"], chrom=c["chrom"], coords=c["coords"], shuffle=c["shuffle"], seed=c["seed"],
              down_prob=c["down_prob"])
    os.makedirs(tmp_path / "metadata", exist_ok=True)
    np.random.seed(seed)  # the down-sampling draw is unseeded in the reference (utils.py:466-470)
    try:
        want = ref.import_mns_from_bedpe(bedpe_file=bedpe, path=str(tmp_path) + "/", **kw)
    except Exception as e:  # whatever the reference rejects, the mirror must reject too
        np.random.seed(seed)
        with pytest.raises(Exception):
            loaders.import_mns_from_bedpe(bedpe, path=None, **kw)
        pytest.skip(f"reference rejects this input ({type(e).__name__})")
    np.random.seed(seed)
    got = loaders.import_mns_from_bedpe(bedpe, path=None, **kw)
    for g, w, name in zip(got, want, ("ms", "ns", "ds", "chr_ends", "chrom_idxs")):
        if name == "ds":
            assert np.allclose(g, w, rtol=1e-13, atol=0), (c, name)
        else:
            assert np.array_equal(np.asarray(g), np.asarray(w)), (c, name)


@pytest.mark.parametrize("seed", range(12))
def test_bed_loader_equals_the_reference(ref, tmp_path, seed):
    c = draw_case(seed)
    rng = np.random.default_rng(seed)
    bed = str(tmp_path / "sub.bed")
    synthetic.write_bed(bed, seed=seed, chrom=c["chrom"], n_chroms=c["n_chroms"],
                        bin_size=int(rng.choice([50_000, 100_000, 250_000])))
    extra = dict(flip_prob=float(rng.choice([0.0, 0.15])), noise_strength=float(rng.choice([0.0, 0.4])))
    kw = dict(N_beads=c["N_beads"], chrom=c["chrom"], coords=c["coords"], shuffle=c["shuffle"], seed=c["seed"], **extra)
    os.makedirs(tmp_path / "metadata", exist_ok=True)
    np.random.seed(seed)
    want = ref.import_bed(bed_file=bed, save_path=str(tmp_path) + "/", **kw)
    np.random.seed(seed)
    got = loaders.import_bed(bed, save_path=None, **kw)
    for g, w, name in zip(got, want, ("Cs", "chr_ends", "chrom_idxs")):
        assert np.array_equal(np.asarray(g), np.asarray(w)), (c, name)
