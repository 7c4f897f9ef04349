"""Generates tests/golden/analysis_*_report.txt by running the REFERENCE's own analyze_structure
($MULTIMM_REFERENCE/src/multimm/plots.py:630-829) on two small structures.  Needs MULTIMM_REFERENCE.
plots.py imports matplotlib, pyvista, seaborn, mpl_toolkits at the top and draws figures at the
end of analyze_structure; those modules are absent here and are replaced by MagicMock objects — the
numeric report (the part re-hosted in multimm_b200/analysis.py) does not depend on them.

    python tests/golden/make_golden_analysis.py
"""
import importlib.util
import os
import shutil
import sys
import tempfile
import types
from unittest.mock import MagicMock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.path.join(os.environ["MULTIMM_REFERENCE"], "src", "multimm")  # a checkout of the original MultiMM


def load_plots():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.lines", "matplotlib.colors", "pyvista", "seaborn",
                 "mpl_toolkits", "mpl_toolkits.mplot3d", "pyBigWig", "openmm", "openmm.unit"):
        sys.modules[name] = MagicMock()
    sys.modules["matplotlib.pyplot"].subplots = lambda *a, **k: (MagicMock(), MagicMock())
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]  # `import matplotlib.pyplot as plt`
    pkg = types.ModuleType("multimm")
    pkg.__path__ = [REF]
    sys.modules["multimm"] = pkg
    mods = {}
    for name in ("utils", "plots"):
        spec = importlib.util.spec_from_file_location(f"multimm.{name}", os.path.join(REF, f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[f"multimm.{name}"] = mod
        spec.loader.exec_module(mod)
        mods[name] = mod
    return mods["plots"]


def structures_for_golden():
    from multimm_b200 import structures

    rng = np.random.default_rng(7)
    walk = np.cumsum(rng.normal(0, 1.0, size=(400, 3)), axis=0)
    return {"walk400": walk, "helix250": structures.compute_init_struct(250, "helix") * 1.3}


def main():
    plots = load_plots()
    for name, V in structures_for_golden().items():
        tmp = tempfile.mkdtemp()
        plots.analyze_structure(V, tmp, name=name)
        shutil.copy(os.path.join(tmp, "analysis", f"{name}_report.txt"), os.path.join(HERE, f"analysis_{name}_report.txt"))
        np.save(os.path.join(HERE, f"analysis_{name}_input.npy"), V)
    print(open(os.path.join(HERE, "analysis_walk400_report.txt")).read())


if __name__ == "__main__":
    main()
