"""Structure generators and structure files against golden outputs of the REFERENCE's own code
(tests/golden/make_golden_structures.py ran initial_structure_tools.py / utils.py from
$MULTIMM_REFERENCE): the .cif / .psf files are part of the contract (north star: "keeps ... structure
outputs"), so the text must match byte for byte."""
import os

import numpy as np
import pytest

from multimm_b200 import cif, structures

GOLD = os.path.join(os.path.dirname(__file__), "golden")
G = np.load(os.path.join(GOLD, "structures_golden.npz"))
CHROM_ENDS = np.array([0, 25, 41, 60])


def gold_text(name):
    with open(os.path.join(GOLD, name)) as f:
        return f.read()


@pytest.mark.parametrize("mode", ["circle", "helix", "spiral", "knot"])
@pytest.mark.parametrize("n", [7, 60, 500])
def test_deterministic_start_curves(mode, n):
    ours = structures.compute_init_struct(n, mode)
    assert ours.shape == (n, 3)
    assert np.allclose(ours, G[f"{mode}_{n}"], rtol=1e-13, atol=1e-13)


@pytest.mark.parametrize("mode", ["sphere", "rw", "confined_rw", "self_avoiding_rw"])
@pytest.mark.parametrize("n", [7, 60, 500])
def test_random_start_curves_draw_the_same_sequence(mode, n):
    """The random curves use the global numpy stream; with the same seed ours must consume it exactly
    as the reference does."""
    if f"{mode}_{n}" not in G:
        pytest.skip("not generated at this size")
    np.random.seed(1000 + n)
    ours = structures.compute_init_struct(n, mode)
    assert np.allclose(ours, G[f"{mode}_{n}"], rtol=1e-12, atol=1e-12)


def test_unknown_curve_raises():
    with pytest.raises(ValueError, match="Invalid option for initial structure"):
        structures.compute_init_struct(10, "zigzag")


def test_init_cif_and_psf_are_byte_identical(tmp_path):
    pts = structures.compute_init_struct(60, "helix")
    cif.write_mmcif(pts, CHROM_ENDS, str(tmp_path / "i.cif"), hetatm_ends=True, connections=True, decimals=3)
    assert (tmp_path / "i.cif").read_text() == gold_text("cif_init_helix60.txt")
    cif.write_psf(60, str(tmp_path / "m.psf"))
    assert (tmp_path / "m.psf").read_text() == gold_text("psf_60.txt")


def test_chromosome_cif_is_byte_identical(tmp_path):
    coords = structures.compute_init_struct(60, "spiral") * 3.7 + 0.12345
    cif.write_mmcif_chrom(coords[:25], str(tmp_path / "c.cif"))
    assert (tmp_path / "c.cif").read_text() == gold_text("cif_chrom_spiral25.txt")


def test_whole_model_cif_matches_reference_writer(tmp_path):
    """initial_structure_tools.write_mmcif (ATOM for every bead, 3 decimals, no connection block)."""
    coords = structures.compute_init_struct(60, "spiral") * 3.7 + 0.12345
    cif.write_mmcif(coords, CHROM_ENDS, str(tmp_path / "w.cif"), hetatm_ends=False, connections=False, decimals=3)
    assert (tmp_path / "w.cif").read_text() == gold_text("cif_write_spiral60.txt")


def test_reader_matches_the_reference_reader():
    """utils.get_coordinates_cif keeps ATOM lines only (HETATM chromosome ends are dropped)."""
    ref = np.load(os.path.join(GOLD, "cif_read_back_init_helix60.npy"))
    ours = cif.read_cif_coordinates(os.path.join(GOLD, "cif_init_helix60.txt"), include_hetatm=False)
    assert ours.shape == ref.shape and np.array_equal(ours, ref)
    full = cif.read_cif_coordinates(os.path.join(GOLD, "cif_init_helix60.txt"), include_hetatm=True)
    assert full.shape == (60, 3)


def test_large_write_read_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    xyz = rng.normal(0, 50, size=(20000, 3))
    ends = np.array([0, 5000, 12000, 20000])
    cif.write_mmcif(xyz, ends, str(tmp_path / "big.cif"), hetatm_ends=True, connections=False, decimals=4)
    back = cif.read_cif_coordinates(str(tmp_path / "big.cif"), include_hetatm=True)
    assert back.shape == xyz.shape and np.abs(back - xyz).max() <= 0.5e-4 + 1e-12


def test_dcd_round_trip(tmp_path):
    w = cif.DCDWriter(str(tmp_path / "t.dcd"), 11, 0.001, 10)
    frames = [np.arange(33, dtype=float).reshape(11, 3) * (k + 1) for k in range(4)]
    for f in frames:
        w.write(f)
    w.close()
    back = cif.read_dcd(str(tmp_path / "t.dcd"))
    assert back.shape == (4, 11, 3) and np.allclose(back, np.array(frames), rtol=1e-6)
