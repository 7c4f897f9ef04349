"""Generates tests/golden/structures_golden.npz and tests/golden/cif_*.txt by running the
REFERENCE's own structure generators and file writers
($MULTIMM_REFERENCE/src/multimm/initial_structure_tools.py: polymer_circle, helix_structure,
spiral_structure, sphere_surface_structure, trefoil_knot_structure, build_init_mmcif, write_mmcif,
write_mmcif_chrom, generate_psf; utils.get_coordinates_cif).  Needs MULTIMM_REFERENCE; outputs are
committed.  The module imports matplotlib, hilbertcurve, scipy.interpolate, tqdm and (through
.utils) pyBigWig / openmm.unit at the top; none is used by the functions called here, the absent
ones are stubbed.  The Hilbert curve itself cannot be generated (hilbertcurve is not installed):
it stays pinned by the invariants in tests/test_oracle.py.

    python tests/golden/make_golden_structures.py
"""
import importlib.util
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.environ["MULTIMM_REFERENCE"], "src", "multimm")  # a checkout of the original MultiMM


def load_reference():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.colors", "pyBigWig", "openmm", "openmm.unit",
                 "hilbertcurve", "hilbertcurve.hilbertcurve", "tqdm"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib.colors"].to_hex = lambda c: "#000000"
    sys.modules["matplotlib.pyplot"].figure = lambda *a, **k: None
    sys.modules["openmm.unit"].Quantity = type("Quantity", (), {})
    sys.modules["hilbertcurve.hilbertcurve"].HilbertCurve = type("HilbertCurve", (), {})
    sys.modules["tqdm"].tqdm = lambda it, *a, **k: it
    pkg = types.ModuleType("multimm")
    pkg.__path__ = [REF]
    sys.modules["multimm"] = pkg
    mods = {}
    for name in ("enums", "utils", "initial_structure_tools"):
        spec = importlib.util.spec_from_file_location(f"multimm.{name}", os.path.join(REF, f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[f"multimm.{name}"] = mod
        spec.loader.exec_module(mod)
        mods[name] = mod
    return mods["initial_structure_tools"], mods["utils"]


def main():
    ist, utils = load_reference()
    out = {}
    for n in (7, 60, 500):
        out[f"circle_{n}"] = ist.compute_init_struct(n, "circle")
        out[f"helix_{n}"] = ist.compute_init_struct(n, "helix")
        out[f"spiral_{n}"] = ist.compute_init_struct(n, "spiral")
        out[f"knot_{n}"] = ist.compute_init_struct(n, "knot")
        # the random curves draw from the global numpy stream (seeded by the loaders in a real run,
        # utils.py:233/439): seed it here so that the draw sequence itself is pinned
        for mode in ("sphere", "rw", "confined_rw") + (("self_avoiding_rw",) if n <= 60 else ()):
            np.random.seed(1000 + n)
            out[f"{mode}_{n}"] = ist.compute_init_struct(n, mode)
    np.savez_compressed(os.path.join(HERE, "structures_golden.npz"), **out)

    n, chrom_ends = 60, np.array([0, 25, 41, 60])
    with tempfile.TemporaryDirectory() as tmp:
        ist.build_init_mmcif(n, chrom_ends, psf=True, path=tmp + "/", curve="helix")
        for src, dst in (("MultiMM_init.cif", "cif_init_helix60.txt"), ("MultiMM.psf", "psf_60.txt")):
            with open(os.path.join(tmp, src)) as f, open(os.path.join(HERE, dst), "w") as g:
                g.write(f.read())
        coords = ist.compute_init_struct(n, "spiral") * 3.7 + 0.12345
        ist.write_mmcif(coords, chrom_ends, tmp + "/w.cif")
        ist.write_mmcif_chrom(coords[:25], tmp + "/c.cif")
        for src, dst in (("w.cif", "cif_write_spiral60.txt"), ("c.cif", "cif_chrom_spiral25.txt")):
            with open(os.path.join(tmp, src)) as f, open(os.path.join(HERE, dst), "w") as g:
                g.write(f.read())
        # the reference's reader: ATOM lines only, whitespace columns 10-12 (utils.py:168-205)
        np.save(os.path.join(HERE, "cif_read_back_init_helix60.npy"), utils.get_coordinates_cif(tmp + "/MultiMM_init.cif"))
    print("written", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    main()
