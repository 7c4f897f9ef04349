"""Randomised differential test of the config model against the REFERENCE's own
($MULTIMM_REFERENCE/src/multimm/config.py: SimulationConfig; run.py: ArgumentChanger, args_tests), run
live: random subsets of fields given as the strings an ini file would hold (booleans in every
accepted spelling, numbers, quantities with units, enum values, chromosome names, the occasional
malformed value).  Same accept / reject decision at each stage, same field values before and after
the MODELLING_LEVEL presets.  Only where the reference checkout exists (MULTIMM_REFERENCE)."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from common import NO_REFERENCE, reference_file
from multimm_b200 import run
from multimm_b200.config import SimulationConfig
from test_config_golden import DIFFERENT, plain, same

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.skipif(reference_file("src/multimm/config.py") is None, reason=NO_REFERENCE)
BEDPE = "tests/golden/synthetic_loops.bedpe"
BED = "tests/golden/synthetic_subcompartments.bed"

BOOLS = ("true", "True", "1", "y", "yes", "false", "False", "0", "n", "no", "", "none", "maybe")
BOOL_FIELDS = ("SHUFFLE_CHROMS", "SAVE_PLOTS", "POL_USE_HARMONIC_BOND", "POL_USE_HARMONIC_ANGLE", "LE_USE_HARMONIC_BOND",
               "LE_FIXED_DISTANCES", "EV_USE_EXCLUDED_VOLUME", "SC_USE_SPHERICAL_CONTAINER", "CHB_USE_CHROMOSOMAL_BLOCKS",
               "COB_USE_COMPARTMENT_BLOCKS", "SCB_USE_SUBCOMPARTMENT_BLOCKS", "IBL_USE_B_LAMINA_INTERACTION",
               "CF_USE_CENTRAL_FORCE", "SIM_RUN_MD", "GENERATE_ENSEMBLE", "BUILD_INITIAL_STRUCTURE")
FLOAT_FIELDS = ("EV_EPSILON", "EV_R_SMALL", "EV_POWER", "SC_SCALE", "CHB_KC", "CHB_DE", "COB_EA", "COB_EB", "SCB_EA1",
                "SCB_EB2", "IBL_SCALE", "CF_STRENGTH", "DOWNSAMPLING_PROB", "COMPARTMENT_FLIP_PROB")
QUANTITIES = {
    "POL_HARMONIC_BOND_R0": ("0.1 nanometer", "1.5 angstrom", "120 picometer", "fast", "0.1"),
    "POL_HARMONIC_BOND_K": ("3e5 kilojoules_per_mole/nanometer**2", "700 kilocalories_per_mole/angstrom**2"),
    "POL_HARMONIC_ANGLE_R0": ("3.14 radian", "175 degrees"),
    "LE_HARMONIC_BOND_R0": ("0.12 nanometers", "1 angstrom"),
    "SC_RADIUS1": ("0.3 nanometer", "", "none"), "SC_RADIUS2": ("12 angstrom", ""),
    "COB_DISTANCE": ("0.4 nanometer", ""), "SCB_DISTANCE": ("3 angstrom", "none"),
    "SIM_TEMPERATURE": ("300 kelvin", "310.5 kelvin"), "SIM_INTEGRATOR_STEP": ("2 femtoseconds", "0.001 picosecond"),
}
LEVELS = ("gene", "GENE", "region", "loc", "chrom", "chromosome", "GW", "genome", "gw", "", "nonsense")
CHROMS = ("chr1", "1", "chrX", "X", "chr22", "22", "", "none", "chr7")
CURVES = ("hilbert", "helix", "rw", "circle", "zigzag")


@pytest.fixture(scope="module")
def ref():
    before = set(sys.modules)
    spec = importlib.util.spec_from_file_location("make_golden_config", os.path.join(ROOT, "tests", "golden", "make_golden_config.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    config, rrun, utils = mg.load_reference()
    yield mg, config, rrun, utils
    for name in set(sys.modules) - before:
        del sys.modules[name]


def draw(seed):
    rng = np.random.default_rng(900 + seed)
    pick = lambda seq: str(seq[int(rng.integers(0, len(seq)))])  # noqa: E731
    kw = dict(LOOPS_PATH=BEDPE if rng.random() < 0.96 else pick(("", "/nonexistent/x.bedpe")), OUT_PATH="/tmp/o")
    if rng.random() < 0.6:
        kw["COMPARTMENT_PATH"] = BED if rng.random() < 0.85 else ""
    if rng.random() < 0.7:
        kw["MODELLING_LEVEL"] = pick(LEVELS)
    if rng.random() < 0.5:
        kw["CHROM"] = pick(CHROMS)
    if rng.random() < 0.3:
        kw["LOC_START"], kw["LOC_END"] = str(int(rng.integers(0, 10**7))), str(int(rng.integers(10**7, 10**8)))
    if rng.random() < 0.4:
        kw["N_BEADS"] = pick(("777", "20000", "3000")) if rng.random() < 0.9 else pick(("12.5", "many"))
    if rng.random() < 0.3:
        kw["INITIAL_STRUCTURE_TYPE"] = pick(CURVES[:-1]) if rng.random() < 0.9 else CURVES[-1]
    for f in rng.choice(BOOL_FIELDS, size=int(rng.integers(0, 7)), replace=False):
        kw[str(f)] = pick(BOOLS[:-1]) if rng.random() < 0.93 else BOOLS[-1]
    for f in rng.choice(FLOAT_FIELDS, size=int(rng.integers(0, 5)), replace=False):
        kw[str(f)] = pick(("3.0", "0.25", "1e-3", "7")) if rng.random() < 0.95 else "x7"
    for f in rng.choice(list(QUANTITIES), size=int(rng.integers(0, 4)), replace=False):
        good = [q for q in QUANTITIES[str(f)] if q not in ("fast", "0.1")]
        kw[str(f)] = pick(good) if rng.random() < 0.93 else pick(("fast", "0.1"))
    return kw


@pytest.mark.parametrize("seed", range(80))
def test_same_outcome_as_the_reference_config(ref, monkeypatch, seed):
    mg, config, rrun, utils = ref
    monkeypatch.chdir(ROOT)
    kw = draw(seed)
    want = mg.outcome(config.SimulationConfig, rrun.ArgumentChanger, rrun.args_tests, utils.chrom_sizes, dict(kw))
    got = mg.outcome(SimulationConfig, lambda args, _sizes: run.ArgumentChanger(args), run.args_tests, None, dict(kw))
    assert got["construct"] == want["construct"], (kw, got["construct"], want["construct"])
    if want["construct"] != "ok":
        return
    for stage in ("fields", "after_preset"):
        for field, w in want[stage].items():
            if field not in DIFFERENT:
                assert same(w, got[stage][field]), (kw, stage, field, w, got[stage][field])
    assert got["preset"] == want["preset"], (kw, got["preset"], want["preset"])
    assert got["checks"] == want["checks"], (kw, got["checks"], want["checks"])


@pytest.mark.parametrize("name", ["config_gw.ini", "config_specific_region.ini", "config_single_cell.ini"])
def test_reference_example_inis_load_unmodified(name, tmp_path):
    """The ini files the reference ships (examples/*.ini, all PLATFORM = OpenCL) load here as they
    are: same field values, and the platform name is accepted as the preference it is upstream.  Only
    the authors' absolute data paths are pointed at this repo's fixtures (they do not exist anywhere)."""
    from multimm_b200.model import resolve_platform

    path = reference_file(f"examples/{name}")
    if path is None:
        pytest.skip("example not shipped in this checkout")
    raw = run.read_ini(path)
    assert raw["PLATFORM"] == "OpenCL"
    raw["LOOPS_PATH"] = BEDPE
    if raw.get("COMPARTMENT_PATH"):
        raw["COMPARTMENT_PATH"] = BED
    raw["ATACSEQ_PATH"] = ""
    raw["OUT_PATH"] = str(tmp_path / "out")
    if name == "config_single_cell.ini":
        # broken upstream as shipped: SC_RADIUS1 = 1 has no unit, which the reference's own
        # parse_quantity (config.py:23-30) rejects with the same message
        with pytest.raises(Exception, match="Can't recognise Quantity format"):
            SimulationConfig(**raw)
        raw["SC_RADIUS1"], raw["SC_RADIUS2"] = "1 nanometer", "2 nanometer"
    args = SimulationConfig(**raw)
    assert args.PLATFORM == "OpenCL" and resolve_platform(args.PLATFORM) == "B200"
    run.ArgumentChanger(args).convenient_argument_changer()
    run.args_tests(args)  # accepted: nothing about the platform, the integrator or the files is refused
