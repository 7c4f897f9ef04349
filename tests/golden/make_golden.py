"""Generates tests/golden/*.npz by running the REFERENCE's own loaders
($MULTIMM_REFERENCE/src/multimm/utils.py: import_bed, import_mns_from_bedpe) on synthetic input
files written by multimm_b200.synthetic.  Run only with MULTIMM_REFERENCE set; the inputs and
outputs are committed.

    python tests/golden/make_golden.py

utils.py imports matplotlib, pyBigWig and openmm.unit at module level; none is installed here and
none is used by the two loaders, so they are stubbed in sys.modules before the file is loaded.
"""
import importlib.util
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REFERENCE = os.environ["MULTIMM_REFERENCE"]  # a checkout of the original MultiMM
REF_UTILS = os.path.join(REFERENCE, "src", "multimm", "utils.py")
REF_FIXTURE = os.path.join(REFERENCE, "tests", "fixtures", "ENCFF045MJY_simple.bedpe")


def load_reference_utils():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.colors", "pyBigWig", "openmm", "openmm.unit"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib.colors"].to_hex = lambda c: "#000000"
    sys.modules["matplotlib.pyplot"].figure = lambda *a, **k: None
    sys.modules["openmm.unit"].Quantity = type("Quantity", (), {})
    spec = importlib.util.spec_from_file_location("ref_utils", REF_UTILS)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


CASES = {
    # name: (kind, kwargs)
    "gw_20k": dict(N_beads=20000, chrom=None, coords=None, shuffle=False, seed=0),
    "gw_20k_shuffle3": dict(N_beads=20000, chrom=None, coords=None, shuffle=True, seed=3),
    "gw_5k_down": dict(N_beads=5000, chrom=None, coords=None, shuffle=True, seed=1, down_prob=0.8),
    "chr1_region": dict(N_beads=2000, chrom="chr1", coords=[10_000_000, 110_000_000], shuffle=False, seed=0),
    "chr6_whole": dict(N_beads=3000, chrom="chr6", coords=[0, 172126628], shuffle=False, seed=2),
}
BED_EXTRA = {
    "gw_5k_down": dict(flip_prob=0.2, noise_strength=0.5),
    "chr1_region": dict(flip_prob=0.1),
}


def main():
    from multimm_b200 import synthetic

    ref = load_reference_utils()
    bedpe = os.path.join(HERE, "synthetic_loops.bedpe")
    bed = os.path.join(HERE, "synthetic_subcompartments.bed")
    synthetic.write_bedpe(bedpe, n_loops=1500, seed=11)
    synthetic.write_bed(bed, seed=11, bin_size=250_000)
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "metadata"))
        for name, kw in CASES.items():
            kw = dict(kw)
            down = kw.pop("down_prob", 1.0)
            ms, ns, ds, ce, ci = ref.import_mns_from_bedpe(bedpe_file=bedpe, path=tmp + "/", down_prob=down, **kw)
            out[f"{name}.ms"], out[f"{name}.ns"], out[f"{name}.ds"] = ms, ns, ds
            out[f"{name}.loop_chr_ends"], out[f"{name}.loop_chrom_idxs"] = ce, ci
            cs, ce2, ci2 = ref.import_bed(bed_file=bed, save_path=tmp + "/", **kw, **BED_EXTRA.get(name, {}))
            out[f"{name}.Cs"], out[f"{name}.bed_chr_ends"], out[f"{name}.bed_chrom_idxs"] = cs, ce2, ci2
        # the reference's own shipped loop fixture (the one data file its tests use)
        for n_beads, chrom, coords in ((1000, None, None), (200000, None, None), (10000, "chr1", [0, 248387328])):
            key = f"fixture_{n_beads}_{chrom or 'gw'}"
            ms, ns, ds, ce, ci = ref.import_mns_from_bedpe(bedpe_file=REF_FIXTURE, N_beads=n_beads, chrom=chrom,
                                                           coords=coords, path=tmp + "/")
            out[f"{key}.ms"], out[f"{key}.ns"], out[f"{key}.ds"], out[f"{key}.chr_ends"] = ms, ns, ds, ce
    out["chrom_strength"] = np.asarray(ref.chrom_strength)
    np.savez_compressed(os.path.join(HERE, "loaders_golden.npz"), **out)
    print("wrote", len(out), "arrays;", {k: v.shape for k, v in list(out.items())[:6]})


if __name__ == "__main__":
    main()
