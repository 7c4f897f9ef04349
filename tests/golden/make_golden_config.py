"""Generates tests/golden/config_golden.json by running the REFERENCE's own config model, MODELLING_LEVEL
presets and cross-field checks ($MULTIMM_REFERENCE/src/multimm/config.py: SimulationConfig;
run.py: ArgumentChanger.convenient_argument_changer, args_tests) on a matrix of inputs.
`openmm.unit` (absent) is replaced by this repo's units module, which is what the reference's
parse_quantity evaluates unit expressions against; every other absent import is a MagicMock.
Needs MULTIMM_REFERENCE.     python tests/golden/make_golden_config.py
"""
import importlib.util
import json
import os
import sys
import types
from enum import Enum
from unittest.mock import MagicMock

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.path.join(os.environ["MULTIMM_REFERENCE"], "src", "multimm")  # a checkout of the original MultiMM

from multimm_b200 import units  # noqa: E402

BEDPE = "tests/golden/synthetic_loops.bedpe"          # relative to the repo root (tests run from there)
BED = "tests/golden/synthetic_subcompartments.bed"

CASES = {
    "defaults": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o"),
    "gene": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", MODELLING_LEVEL="GENE", COMPARTMENT_PATH=BED, SHUFFLE_CHROMS=True),
    "region": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", MODELLING_LEVEL="region", COMPARTMENT_PATH=BED, CHROM="chr3"),
    "loc_no_comps": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", MODELLING_LEVEL="loc", CHROM="3"),
    "chrom": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", MODELLING_LEVEL="chrom", CHROM="chrX", CF_USE_CENTRAL_FORCE=True),
    "gw_comps": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", MODELLING_LEVEL="GW", COMPARTMENT_PATH=BED,
                     CHB_USE_CHROMOSOMAL_BLOCKS=True, SCB_USE_SUBCOMPARTMENT_BLOCKS=True, N_BEADS=123),
    "gw_no_comps": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", MODELLING_LEVEL="genome", SIM_RUN_MD=True),
    "strings_from_ini": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", N_BEADS="777", EV_POWER="3.0", SHUFFLE_CHROMS="yes",
                             SAVE_PLOTS="0", CHROM="chr7", LOC_START="1000", LOC_END="9000000",
                             POL_HARMONIC_BOND_R0="1.5 angstrom", SIM_INTEGRATOR_STEP="2 femtoseconds",
                             SIM_TEMPERATURE="300 kelvin", COMPARTMENT_PATH="", INITIAL_STRUCTURE_TYPE="helix"),
    "cob_without_bed": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", COB_USE_COMPARTMENT_BLOCKS=True),
    "scb_without_bed": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", SCB_USE_SUBCOMPARTMENT_BLOCKS=True),
    "lamina_without_bed": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", IBL_USE_B_LAMINA_INTERACTION=True),
    "lamina_without_block_force": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", IBL_USE_B_LAMINA_INTERACTION=True,
                                       COMPARTMENT_PATH=BED),
    "lamina_ok": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", IBL_USE_B_LAMINA_INTERACTION=True, COMPARTMENT_PATH=BED,
                      COB_USE_COMPARTMENT_BLOCKS=True),
    "cf_single_chrom": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", CF_USE_CENTRAL_FORCE=True, CHROM="chr1"),
    "chb_single_chrom": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", CHB_USE_CHROMOSOMAL_BLOCKS=True, CHROM="chr1"),
    "missing_file": dict(LOOPS_PATH="/nonexistent/x.bedpe", OUT_PATH="/tmp/o"),
    "no_loops": dict(LOOPS_PATH="", OUT_PATH="/tmp/o"),
    "bad_quantity": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", POL_HARMONIC_BOND_R0="fast"),
    "bad_bool": dict(LOOPS_PATH=BEDPE, OUT_PATH="/tmp/o", SHUFFLE_CHROMS="maybe"),
}


def plain(v):
    if isinstance(v, units.Quantity):
        return {"quantity_md": v.md}
    if isinstance(v, Enum):
        return v.value
    return v


def load_reference():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.lines", "matplotlib.colors", "pyvista", "seaborn",
                 "mpl_toolkits", "mpl_toolkits.mplot3d", "pyBigWig", "hilbertcurve", "hilbertcurve.hilbertcurve",
                 "openmm", "openmm.app"):
        sys.modules[name] = MagicMock()
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    unit = types.ModuleType("openmm.unit")
    for name, u in units.UNITS.items():
        setattr(unit, name, u)
    unit.Quantity, unit.Unit, unit.BaseUnit = units.Quantity, units.Unit, units.Unit
    sys.modules["openmm.unit"] = unit
    sys.modules["openmm"].unit = unit
    pkg = types.ModuleType("multimm")
    pkg.__path__ = [REF]
    sys.modules["multimm"] = pkg
    for name in ("enums", "config", "utils", "logger", "initial_structure_tools", "nucleosome_interpolation", "plots",
                 "model", "run"):
        spec = importlib.util.spec_from_file_location(f"multimm.{name}", os.path.join(REF, f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[f"multimm.{name}"] = mod
        spec.loader.exec_module(mod)
    return sys.modules["multimm.config"], sys.modules["multimm.run"], sys.modules["multimm.utils"]


def outcome(config_cls, changer_cls, args_tests, chrom_sizes, kw):
    res = {}
    try:
        args = config_cls(**kw)
    except Exception as e:
        return {"construct": type(e).__name__}
    res["construct"] = "ok"
    res["fields"] = {k: plain(v) for k, v in args.model_dump().items()}
    try:
        changer_cls(args, chrom_sizes).convenient_argument_changer()
        res["preset"] = "ok"
    except Exception as e:
        res["preset"] = type(e).__name__
    res["after_preset"] = {k: plain(v) for k, v in args.model_dump().items()}
    try:
        args_tests(args)
        res["checks"] = "ok"
    except Exception as e:
        res["checks"] = type(e).__name__
    return res


def main():
    os.chdir(ROOT)
    config, run, utils = load_reference()
    out = {name: outcome(config.SimulationConfig, run.ArgumentChanger, run.args_tests, utils.chrom_sizes, kw)
           for name, kw in CASES.items()}
    # precedence defaults < ini < CLI through the reference's own get_config (run.py:349-395)
    argv = ["-c", "tests/golden/sample_config.ini", "--n_beads", "4321", "--sc_use_spherical_container", "True",
            "--modelling_level", "region", "--chrom", "chr2"]
    old = sys.argv
    sys.argv = ["MultiMM"] + argv
    try:
        cli = run.get_config()
    finally:
        sys.argv = old
    with open(os.path.join(HERE, "config_golden.json"), "w") as fh:
        json.dump({"cases": CASES, "reference": out, "cli_argv": argv,
                   "cli_reference": {k: plain(v) for k, v in cli.model_dump().items()}}, fh, indent=1, sort_keys=True)
    for k, v in out.items():
        print(k, v["construct"], v.get("preset"), v.get("checks"))


if __name__ == "__main__":
    main()
