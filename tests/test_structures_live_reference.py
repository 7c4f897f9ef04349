"""Randomised differential test of the structure files and start curves against the REFERENCE's
own writers and generators, run live ($MULTIMM_REFERENCE/src/multimm/initial_structure_tools.py:
build_init_mmcif, write_mmcif, write_mmcif_chrom, generate_psf, compute_init_struct;
utils.get_coordinates_cif).  Text must match byte for byte.  Only where the reference checkout
exists (MULTIMM_REFERENCE); the frozen files of test_structures_io.py run everywhere."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from common import NO_REFERENCE, reference_file
from multimm_b200 import cif, structures

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.skipif(reference_file("src/multimm/initial_structure_tools.py") is None, reason=NO_REFERENCE)


@pytest.fixture(scope="module")
def ref():
    before = set(sys.modules)
    spec = importlib.util.spec_from_file_location("make_golden_structures",
                                                  os.path.join(HERE, "golden", "make_golden_structures.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    yield mg.load_reference()
    for name in set(sys.modules) - before:
        del sys.modules[name]


def draw(seed):
    rng = np.random.default_rng(300 + seed)
    n = int(rng.choice([2, 3, 9, 40, 333, 1200, 10500]))
    n_chr = int(rng.integers(1, min(24, max(2, n // 3)))) if n > 4 else 1
    cuts = np.sort(rng.choice(np.arange(2, n - 1), size=n_chr - 1, replace=False)) if n_chr > 1 else np.array([], int)
    ends = np.concatenate([[0], cuts, [n]]).astype(int)
    scale = float(rng.choice([0.01, 1.0, 37.0, 2500.0]))
    xyz = rng.normal(0, scale, size=(n, 3))
    xyz[rng.integers(0, n)] = [0.0005, -0.0005, 1e-9]  # rounding ties and a negative zero candidate
    return n, ends, xyz


@pytest.mark.parametrize("seed", range(14))
def test_whole_model_and_chromosome_cif_equal_the_reference_writers(ref, tmp_path, seed):
    ist, utils = ref
    n, ends, xyz = draw(seed)
    ist.write_mmcif(xyz, ends, str(tmp_path / "ref.cif"))
    cif.write_mmcif(xyz, ends, str(tmp_path / "our.cif"), hetatm_ends=False, connections=False, decimals=3)
    assert (tmp_path / "our.cif").read_text() == (tmp_path / "ref.cif").read_text()
    a, b = int(ends[0]), int(ends[1])
    ist.write_mmcif_chrom(xyz[a:b], str(tmp_path / "refc.cif"))
    cif.write_mmcif_chrom(xyz[a:b], str(tmp_path / "ourc.cif"))
    assert (tmp_path / "ourc.cif").read_text() == (tmp_path / "refc.cif").read_text()
    got = cif.read_cif_coordinates(str(tmp_path / "ref.cif"), include_hetatm=False)
    want = utils.get_coordinates_cif(str(tmp_path / "ref.cif"))
    assert got.shape == np.shape(want) and np.array_equal(got, want)


@pytest.mark.parametrize("seed", range(8))
@pytest.mark.parametrize("curve", ["helix", "circle", "spiral", "knot"])
def test_initial_cif_and_psf_equal_the_reference(ref, tmp_path, seed, curve):
    ist, _ = ref
    n, ends, _ = draw(seed)
    if n > 2000:
        n, ends = 2000, np.concatenate([ends[ends < 1990], [2000]])
    (tmp_path / "r").mkdir()
    ist.build_init_mmcif(n, ends, psf=True, path=str(tmp_path / "r") + "/", curve=curve)
    pts = structures.compute_init_struct(n, curve)
    cif.write_mmcif(pts, ends, str(tmp_path / "i.cif"), hetatm_ends=True, connections=True, decimals=3)
    cif.write_psf(n, str(tmp_path / "m.psf"))
    assert (tmp_path / "i.cif").read_text() == (tmp_path / "r" / "MultiMM_init.cif").read_text()
    assert (tmp_path / "m.psf").read_text() == (tmp_path / "r" / "MultiMM.psf").read_text()


@pytest.mark.parametrize("mode", ["sphere", "rw", "confined_rw", "self_avoiding_rw"])
@pytest.mark.parametrize("seed", range(5))
def test_random_start_curves_consume_the_stream_like_the_reference(ref, mode, seed):
    ist, _ = ref
    n = int(np.random.default_rng(seed).integers(2, 90 if mode == "self_avoiding_rw" else 700))
    np.random.seed(seed)
    want = ist.compute_init_struct(n, mode)
    after_ref = np.random.random()
    np.random.seed(seed)
    got = structures.compute_init_struct(n, mode)
    after_ours = np.random.random()
    assert np.allclose(got, want, rtol=1e-12, atol=1e-12)
    assert after_ours == after_ref  # same number of draws taken from the global stream
