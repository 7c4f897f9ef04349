"""config.ini semantics against the REFERENCE's own config model, presets and cross-field checks
(tests/golden/make_golden_config.py ran $MULTIMM_REFERENCE/src/multimm/config.py and run.py): same
coercions, same defaults for every field the two models share, same MODELLING_LEVEL overrides,
same accept / reject decisions."""
import json
import os
from enum import Enum

import pytest

from multimm_b200 import run, units
from multimm_b200.config import SimulationConfig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "config_golden.json")))

# fields whose meaning deliberately differs here (DESIGN.md 1): the platform is the B200, defaults of
# paths into the package differ, and the engine adds its own knobs
DIFFERENT = {"PLATFORM", "FORCEFIELD_PATH", "GENE_TSV"}


def plain(v):
    if isinstance(v, units.Quantity):
        return {"quantity_md": v.md}
    if isinstance(v, Enum):
        return v.value
    return v


def same(a, b):
    if isinstance(a, dict) and "quantity_md" in a:
        return isinstance(b, dict) and b["quantity_md"] == pytest.approx(a["quantity_md"], rel=1e-12)
    return a == b


@pytest.fixture(autouse=True)
def from_repo_root(monkeypatch):
    monkeypatch.chdir(ROOT)  # the golden cases name their input files relative to the repo root


@pytest.mark.parametrize("name", sorted(GOLD["cases"]))
def test_same_outcome_as_the_reference(name):
    kw, ref = GOLD["cases"][name], GOLD["reference"][name]
    try:
        args = SimulationConfig(**kw)
    except Exception as e:
        assert ref["construct"] == type(e).__name__, (name, e)
        return
    assert ref["construct"] == "ok"
    ours = {k: plain(v) for k, v in args.model_dump().items()}
    for field, want in ref["fields"].items():
        if field in DIFFERENT:
            continue
        assert field in ours, f"field {field} of the reference's config is missing here"
        assert same(want, ours[field]), (name, field, want, ours[field])
    run.ArgumentChanger(args).convenient_argument_changer()
    after = {k: plain(v) for k, v in args.model_dump().items()}
    for field, want in ref["after_preset"].items():
        if field not in DIFFERENT:
            assert same(want, after[field]), (name, "after preset", field, want, after[field])
    try:
        run.args_tests(args)
        got = "ok"
    except Exception as e:
        got = type(e).__name__
    assert got == ref["checks"], (name, got, ref["checks"])


def test_cli_precedence_matches_the_reference_get_config(tmp_path):
    """defaults < ini (all sections, keys case-folded) < CLI, then the presets: run.py:349-395.
    get_config writes metadata/config_auto.ini under OUT_PATH, so the ini is run from a copy whose
    OUT_PATH points into tmp_path; the reference kept the ini's OUT_PATH as written."""
    ref_out = GOLD["cli_reference"]["OUT_PATH"]
    text = open(os.path.join(ROOT, "tests", "golden", "sample_config.ini")).read()
    assert f"OUT_PATH = {ref_out}\n" in text
    ini = tmp_path / "sample_config.ini"
    out = str(tmp_path / "out")
    ini.write_text(text.replace(f"OUT_PATH = {ref_out}\n", f"OUT_PATH = {out}\n"))
    argv = [str(ini) if a.endswith("sample_config.ini") else a for a in GOLD["cli_argv"]]
    args, _ = run.get_config(argv)
    ours = {k: plain(v) for k, v in args.model_dump().items()}
    assert os.path.exists(os.path.join(out, "metadata", "config_auto.ini"))
    for field, want in dict(GOLD["cli_reference"], OUT_PATH=out).items():
        if field not in DIFFERENT:
            assert same(want, ours[field]), (field, want, ours[field])
    assert ours["N_BEADS"] == 5000 and ours["EV_POWER"] == 5.0  # the region preset wins over the CLI's n_beads


def test_only_documented_extra_fields():
    """Fields this repo adds to the reference's set: the engine's own knobs, nothing else."""
    ref_fields = set(GOLD["reference"]["defaults"]["fields"])
    ours = set(SimulationConfig.model_fields)
    assert ref_fields <= ours
    assert ours - ref_fields == {"PAIR_CUTOFF", "MIN_TOLERANCE", "MIN_MAX_ITERATIONS", "MIN_COARSE_CUTOFF",
                                 "MIN_COARSE_MAX_ITERATIONS", "MIN_COARSE_FAR_FIELD", "MIN_COARSE_TOLERANCE", "MIN_COARSE_ROUNDS",
                                 "MIN_EXACT_PROBE_ITERATIONS"}
