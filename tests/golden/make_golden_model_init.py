"""Generates tests/golden/model_init_golden.npz by running the REFERENCE's own MultiMM.__init__
($MULTIMM_REFERENCE/src/multimm/model.py:24-162: input ingestion, chromosome spins and strengths, gene
window) with its own loaders on the synthetic inputs of tests/golden.  Absent modules are stand-ins
(see make_golden_forcefield.py); nothing in __init__ touches OpenMM.  Needs MULTIMM_REFERENCE.

    python tests/golden/make_golden_model_init.py
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from make_golden_forcefield import load_reference_model  # noqa: E402
from multimm_b200.config import SimulationConfig  # noqa: E402

BEDPE = os.path.join(HERE, "synthetic_loops.bedpe")
BED = os.path.join(HERE, "synthetic_subcompartments.bed")
GENES = "gene_id\tgene_name\tchromosome\tstart\tend\nENSG01\tAAA\tchr1\t30000000\t30600000\nENSG02\tBBB\tchr2\t50000000\t50090000\n"

CASES = {
    "gw_shuffle": dict(N_BEADS=20000, COMPARTMENT_PATH=BED, SHUFFLE_CHROMS=True, SHUFFLING_SEED=3),
    "gw_plain_downsampled": dict(N_BEADS=8000, COMPARTMENT_PATH=BED, SHUFFLING_SEED=1, DOWNSAMPLING_PROB=0.8,
                                 COMPARTMENT_FLIP_PROB=0.2),
    "chr1_region": dict(N_BEADS=2000, CHROM="chr1", LOC_START=10_000_000, LOC_END=110_000_000, COMPARTMENT_PATH=BED),
    "chr6_no_comps": dict(N_BEADS=3000, CHROM="chr6", LOC_START=0, LOC_END=172126628),
    "gene_by_name": dict(N_BEADS=1000, MODELLING_LEVEL="gene", GENE_NAME="AAA", GENE_WINDOW=20_000_000),
    "gene_by_id": dict(N_BEADS=1000, MODELLING_LEVEL="gene", GENE_ID="ENSG02", GENE_WINDOW=30_000_000),
}


def main():
    model = load_reference_model()
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        tsv = os.path.join(tmp, "genes.tsv")
        with open(tsv, "w") as fh:
            fh.write(GENES)
        for name, kw in CASES.items():
            args = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=os.path.join(tmp, name), GENE_TSV=tsv, **kw)
            m = model.MultiMM(args)
            for attr in ("ms", "ns", "ds", "chr_ends", "chrom_idxs", "Cs", "chrom_spin", "chrom_strength"):
                v = getattr(m, attr, None)
                if v is not None:
                    out[f"{name}.{attr}"] = np.asarray(v)
            for attr in ("gene_start", "gene_end"):
                if hasattr(m, attr):
                    out[f"{name}.{attr}"] = np.asarray(getattr(m, attr))
            print(name, {k.split(".")[1]: v.shape for k, v in out.items() if k.startswith(name + ".")})
    np.savez_compressed(os.path.join(HERE, "model_init_golden.npz"), **out)


if __name__ == "__main__":
    main()
