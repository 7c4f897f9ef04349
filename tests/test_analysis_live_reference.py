"""Randomised differential test of the structure report against the REFERENCE's own
analyze_structure ($MULTIMM_REFERENCE/src/multimm/plots.py:630-829), run live: the report text must be
identical.  Only where the reference checkout exists (MULTIMM_REFERENCE)."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from common import NO_REFERENCE, reference_file
from multimm_b200 import analysis, structures

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.skipif(reference_file("src/multimm/plots.py") is None, reason=NO_REFERENCE)


@pytest.fixture(scope="module")
def plots():
    before = set(sys.modules)
    spec = importlib.util.spec_from_file_location("make_golden_analysis",
                                                  os.path.join(HERE, "golden", "make_golden_analysis.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    yield mg.load_plots()
    for name in set(sys.modules) - before:
        del sys.modules[name]


def draw(seed):
    rng = np.random.default_rng(40 + seed)
    n = int(rng.integers(30, 900))
    kind = seed % 4
    if kind == 0:
        return np.cumsum(rng.normal(0, rng.uniform(0.05, 3.0), size=(n, 3)), axis=0)
    if kind == 1:
        return structures.compute_init_struct(n, str(rng.choice(["helix", "spiral", "circle", "knot"]))) * rng.uniform(0.3, 4.0)
    if kind == 2:  # compact globule
        return rng.normal(0, 1.0, size=(n, 3)) * rng.uniform(0.5, 20.0) + rng.normal(0, 50, size=3)
    return np.cumsum(rng.normal(0, 1.0, size=(n, 3)), axis=0) * np.array([1.0, 0.2, 5.0])  # anisotropic


@pytest.mark.parametrize("seed", range(12))
def test_report_text_equals_the_reference(plots, tmp_path, seed):
    V = draw(seed)
    name = f"s{seed}"
    plots.analyze_structure(V.copy(), str(tmp_path / "ref"), name=name)
    analysis.analyze_structure(V.copy(), str(tmp_path / "our"), name=name)
    want = (tmp_path / "ref" / "analysis" / f"{name}_report.txt").read_text()
    got = (tmp_path / "our" / "analysis" / f"{name}_report.txt").read_text()
    assert got == want


@pytest.mark.parametrize("seed", range(6))
def test_contact_map_equals_the_reference_heatmap(plots, tmp_path, seed):
    """get_heatmap (plots.py:504-596) reads a CIF and returns the matrix it draws."""
    from multimm_b200 import cif

    V = draw(seed)[:300]
    ends = np.array([0, len(V) // 3, len(V)])
    path = str(tmp_path / "s.cif")
    cif.write_mmcif(V, ends, path, hetatm_ends=bool(seed % 2), connections=False, decimals=4)
    kw = dict(log_scale=bool(seed % 3), reorder_by_diagonal=bool(seed % 2 == 0))
    want = plots.get_heatmap(path, viz=False, save=False, save_path=str(tmp_path / "plots"), **kw)
    got = analysis.contact_map(cif.read_cif_coordinates(path, include_hetatm=False), **kw)
    assert got.shape == want.shape and np.allclose(got, want, rtol=1e-12, atol=1e-14)
