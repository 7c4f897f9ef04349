"""Randomised differential test of MultiMM.__init__ (input ingestion, chromosome ends / ids /
spins / strengths, gene window; $MULTIMM_REFERENCE/src/multimm/model.py:24-162) against the
REFERENCE's own __init__, run live on freshly drawn synthetic inputs.  Only where the reference
checkout exists (MULTIMM_REFERENCE); the frozen cases of test_model_init_golden.py run everywhere."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from common import NO_REFERENCE, reference_file
from multimm_b200 import loaders, model, synthetic
from multimm_b200.config import SimulationConfig

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.skipif(reference_file("src/multimm/model.py") is None, reason=NO_REFERENCE)
GENES = ("gene_id\tgene_name\tchromosome\tstart\tend\nENSG01\tAAA\tchr1\t30000000\t30600000\n"
         "ENSG02\tBBB\tchr2\t50000000\t50090000\nENSG03\tCCC\tchr17\t7000000\t7020000\n")
ATTRS = ("ms", "ns", "chr_ends", "chrom_idxs", "Cs", "chrom_spin", "gene_start", "gene_end")


@pytest.fixture(scope="module")
def ref_model():
    before = set(sys.modules)
    spec = importlib.util.spec_from_file_location("make_golden_forcefield",
                                                  os.path.join(HERE, "golden", "make_golden_forcefield.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    yield mg.load_reference_model()
    for name in set(sys.modules) - before:
        del sys.modules[name]


def draw(seed, bed):
    rng = np.random.default_rng(500 + seed)
    kind = seed % 4
    kw = dict(SHUFFLING_SEED=int(rng.integers(0, 100)))
    if rng.random() < 0.7:
        kw.update(COMPARTMENT_PATH=bed, COMPARTMENT_FLIP_PROB=float(rng.choice([0.0, 0.25])),
                  COMPARTMENT_NOISE_STD=float(rng.choice([0.0, 0.3])))
    if rng.random() < 0.4:
        kw["DOWNSAMPLING_PROB"] = float(rng.uniform(0.4, 0.95))
    if kind == 0:  # genome-wide
        kw.update(N_BEADS=int(rng.integers(6000, 30000)), SHUFFLE_CHROMS=bool(rng.integers(0, 2)))
    elif kind == 1:  # whole chromosome
        chrom = loaders.CHROM_NAMES[int(rng.integers(0, 22))]
        kw.update(N_BEADS=int(rng.integers(500, 4000)), CHROM=chrom, LOC_START=0, LOC_END=int(loaders.CHROM_SIZES[chrom]))
    elif kind == 2:  # region
        chrom = loaders.CHROM_NAMES[int(rng.integers(0, 12))]
        size = int(loaders.CHROM_SIZES[chrom])
        a = int(rng.integers(0, size // 2))
        kw.update(N_BEADS=int(rng.integers(500, 3000)), CHROM=chrom, LOC_START=a, LOC_END=a + int(rng.integers(size // 6, size // 2)))
    else:  # gene
        by_name = bool(rng.integers(0, 2))
        kw.update(N_BEADS=int(rng.integers(600, 2000)), MODELLING_LEVEL="gene",
                  GENE_WINDOW=int(rng.integers(15_000_000, 40_000_000)),
                  **(dict(GENE_NAME=str(rng.choice(["AAA", "BBB"]))) if by_name else dict(GENE_ID=str(rng.choice(["ENSG01", "ENSG02"])))))
    return kw


@pytest.mark.parametrize("seed", range(16))
def test_init_equals_the_reference(ref_model, tmp_path, seed):
    bedpe, bed, tsv = str(tmp_path / "l.bedpe"), str(tmp_path / "c.bed"), str(tmp_path / "genes.tsv")
    synthetic.write_bedpe(bedpe, n_loops=int(800 + 150 * seed), seed=seed)
    synthetic.write_bed(bed, seed=seed, bin_size=int([50_000, 100_000, 250_000][seed % 3]))
    with open(tsv, "w") as fh:
        fh.write(GENES)
    kw = draw(seed, bed)
    outs = []
    for who, cls, extra in (("ref", ref_model.MultiMM, {}), ("our", model.MultiMM, dict(PLATFORM="B200"))):
        args = SimulationConfig(LOOPS_PATH=bedpe, OUT_PATH=str(tmp_path / who), GENE_TSV=tsv, **kw, **extra)
        np.random.seed(seed)  # unseeded draws (down-sampling) must see the same stream on both sides
        try:
            outs.append(cls(args))
        except Exception as e:  # noqa: BLE001
            outs.append(e)
    want, got = outs
    if isinstance(want, Exception):
        assert isinstance(got, Exception), (kw, want)
        pytest.skip(f"reference rejects this input ({type(want).__name__})")
    assert not isinstance(got, Exception), (kw, got)
    for attr in ATTRS:
        w, g = getattr(want, attr, None), getattr(got, attr, None)
        if w is None:
            assert g is None, (attr, kw)
        else:
            assert np.array_equal(np.asarray(g), np.asarray(w)), (attr, kw)
    assert np.allclose(got.ds, want.ds, rtol=1e-13, atol=0)
    assert np.array_equal(np.asarray(got.chrom_strength), np.asarray(want.chrom_strength))
