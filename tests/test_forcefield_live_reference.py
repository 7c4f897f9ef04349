"""Randomised differential test of the force-field builder against the REFERENCE's own add_*
methods, run live ($MULTIMM_REFERENCE/src/multimm/model.py:164-720 executed unmodified against the
recording `openmm` stand-in of tests/golden/make_golden_forcefield.py, their Lepton strings
evaluated in FP64).  Every numeric config field that feeds a term is drawn at random, together with
the functional forms, the geometry, the chromosome layout and the loops; this repo's chain (host
mirror -> the calls it makes on the C-ABI -> CPU oracle) must give the same ten energies.  Only
where the reference checkout exists (MULTIMM_REFERENCE); the frozen cases of
test_forcefield_golden.py run everywhere."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from common import NO_REFERENCE, O, reference_file
from multimm_b200 import model
from multimm_b200.config import SimulationConfig

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.skipif(reference_file("src/multimm/model.py") is None, reason=NO_REFERENCE)

FORMS = dict(EV_FORCE_TYPE=("powerlaw", "gaussian_core"), COB_FORCE_TYPE=("gaussian", "yukawa", "theta"),
             SCB_FORCE_TYPE=("gaussian", "yukawa", "theta"), CHB_FORCE_TYPE=("polynomial", "gaussian", "saturating"),
             BLAMINA_FORCE_TYPE=("sin", "gaussian_shell", "harmonic_shell", "logistic_shell"),
             CENTRAL_FORCE_TYPE=("harmonic", "gaussian", "logistic"),
             LE_LOOP_FORCE_TYPE=("harmonic", "fene_soft", "gaussian_tether"))
# numeric fields: (default, unit string or None)
NUMERIC = dict(EV_EPSILON=(100.0, None), EV_R_SMALL=(0.05, None), SC_SCALE=(1000.0, None), CHB_KC=(0.3, None),
               CHB_DE=(1e-4, None), COB_EA=(1.0, None), COB_EB=(2.0, None), SCB_EA1=(1.0, None), SCB_EA2=(1.33, None),
               SCB_EB1=(1.66, None), SCB_EB2=(2.0, None), IBL_SCALE=(400.0, None), CF_STRENGTH=(20.0, None),
               POL_HARMONIC_BOND_R0=(0.1, "nanometer"), POL_HARMONIC_BOND_K=(3e5, "kilojoules_per_mole/nanometer**2"),
               POL_HARMONIC_ANGLE_R0=(np.pi, "radian"), POL_HARMONIC_ANGLE_CONSTANT_K=(100.0, "kilojoules_per_mole/radian**2"),
               LE_HARMONIC_BOND_R0=(0.1, "nanometer"), LE_HARMONIC_BOND_K=(3e4, "kilojoules_per_mole/nanometer**2"))
OPTIONAL_Q = dict(SC_RADIUS1=(0.2, 0.6), SC_RADIUS2=(0.8, 1.6), COB_DISTANCE=(0.15, 0.6), SCB_DISTANCE=(0.15, 0.6))
USE = ("EV_USE_EXCLUDED_VOLUME", "COB_USE_COMPARTMENT_BLOCKS", "SCB_USE_SUBCOMPARTMENT_BLOCKS",
       "CHB_USE_CHROMOSOMAL_BLOCKS", "SC_USE_SPHERICAL_CONTAINER", "IBL_USE_B_LAMINA_INTERACTION",
       "CF_USE_CENTRAL_FORCE", "POL_USE_HARMONIC_BOND", "LE_USE_HARMONIC_BOND", "POL_USE_HARMONIC_ANGLE")


@pytest.fixture(scope="module")
def ref():
    """The generator module with the reference's model.py loaded; the stand-in modules it plants
    in sys.modules (openmm, matplotlib, ...) are removed again afterwards."""
    before = set(sys.modules)
    spec = importlib.util.spec_from_file_location("make_golden_forcefield",
                                                  os.path.join(HERE, "golden", "make_golden_forcefield.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    mg.ref_model = mg.load_reference_model()
    yield mg
    for name in set(sys.modules) - before:
        del sys.modules[name]


def draw(seed):
    rng = np.random.default_rng(7000 + seed)
    n = int(rng.integers(24, 80))
    x = np.cumsum(rng.normal(0, 0.08, size=(n, 3)), axis=0) + rng.normal(0, 0.02, size=(n, 3))
    n_chr = int(rng.integers(1, 5))
    cuts = np.sort(rng.choice(np.arange(4, n - 4), size=n_chr - 1, replace=False)) if n_chr > 1 else np.array([], int)
    chr_ends = np.concatenate([[0], cuts, [n]]).astype(int)
    chrom_idxs = rng.permutation(n_chr)
    strength = rng.random(n_chr)
    spin, cstr = np.zeros(n), np.zeros(n)
    for k in range(n_chr):
        spin[chr_ends[k]:chr_ends[k + 1]] = chrom_idxs[k]
        cstr[chr_ends[k]:chr_ends[k + 1]] = strength[k]
    n_loops = int(rng.integers(1, 9))
    ms = rng.integers(0, n - 4, size=n_loops)
    ns = np.minimum(ms + rng.integers(3, 20, size=n_loops), n - 1)
    geo = dict(x=x, chr_ends=chr_ends, Cs=rng.choice([-2, -1, 0, 1, 2], size=n), ms=ms, ns=ns,
               ds=0.1 + 0.1 * rng.random(n_loops), chrom_spin=spin, chrom_strength=cstr)
    over = {k: str(rng.choice(v)) for k, v in FORMS.items()}
    for k, (default, unit) in NUMERIC.items():
        v = float(default * rng.uniform(0.5, 2.0))
        if k == "POL_HARMONIC_ANGLE_R0":
            v = float(rng.uniform(2.0, np.pi))
        over[k] = f"{v!r} {unit}" if unit else v
    for k, (lo, hi) in OPTIONAL_Q.items():
        if rng.random() < 0.6:
            over[k] = f"{float(rng.uniform(lo, hi))!r} nanometer"
    over["EV_POWER"] = float(rng.choice([3.0, 4.0, 6.0, 4.5, 2.5]))
    over["LE_FIXED_DISTANCES"] = bool(rng.integers(0, 2))
    for k in USE:  # mostly on, so that a seed exercises many terms at once
        over[k] = bool(rng.random() < 0.85)
    return n, geo, over


class Recorder:
    def __init__(self):
        self.calls = {}

    def __getattr__(self, name):
        def rec(*a, **k):
            self.calls.setdefault(name, []).append((a, k))
        return rec


def reference_energies(mg, n, geo, args):
    obj = mg.ref_model.MultiMM.__new__(mg.ref_model.MultiMM)
    obj.args, obj.system = args, mg.System(n)
    for k in ("chr_ends", "Cs", "ms", "ns", "ds", "chrom_spin", "chrom_strength"):
        setattr(obj, k, geo[k])
    obj.set_radiuses()
    obj.mass_center = np.average(geo["x"], axis=0)
    obj.add_forcefield()
    # which term a recorded force is: the order add_forcefield builds the enabled ones in (model.py:722-745)
    enabled = [name for flag, name in zip(USE, ("EV", "COB", "SCB", "CHB", "SC", "LAM", "CF", "BOND", "LOOP", "ANGLE"))
               if getattr(args, flag)]
    assert len(obj.system.forces) == len(enabled)
    e = dict.fromkeys(O.TERM_NAMES, 0.0)
    for name, f in zip(enabled, obj.system.forces):
        e[name] = mg.energy(f, geo["x"])
    return np.array([e[t] for t in O.TERM_NAMES]), obj


def our_energies(n, geo, args):
    m = model.MultiMM.__new__(model.MultiMM)
    m.args, m.engine, m.timings = args, Recorder(), {}
    for k in ("chr_ends", "Cs", "ms", "ns", "ds", "chrom_spin", "chrom_strength"):
        setattr(m, k, geo[k])
    m.set_radiuses()
    m.mass_center = np.average(geo["x"], axis=0)
    m.add_forcefield()
    c = m.engine.calls
    pair = {a[0]: (a[1], list(a[2])) for a, _ in c.get("set_pair_term", [])}
    ext = {a[0]: (a[1], list(a[2])) for a, _ in c.get("set_external_term", [])}
    full = lambda v, ref: np.broadcast_to(np.asarray(v, dtype=float), np.shape(ref)).copy()  # noqa: E731
    kw = dict(n=n, ev=pair.get("EV"), cob=pair.get("COB"), scb=pair.get("SCB"), chb=pair.get("CHB"),
              sc=ext.get("SC"), lam=ext.get("LAM"), cf=ext.get("CF"), cutoff=0.0)
    if "set_bead_params" in c:
        (s, chrom, cstr), _ = c["set_bead_params"][0]
        kw.update(s=np.asarray(s, dtype=np.int8), chrom=np.asarray(chrom, dtype=np.int32), cstr=np.asarray(cstr, float))
    if "set_bonds" in c:
        (bi, bj, br0, bk), _ = c["set_bonds"][0]
        kw["bonds"] = (np.asarray(bi, np.int32), np.asarray(bj, np.int32), full(br0, bi), full(bk, bi))
    if "set_loops" in c:
        (li, lj, lr0, lk), lkw = c["set_loops"][0]
        kw["loops"] = (np.asarray(li, np.int32), np.asarray(lj, np.int32), full(lr0, li), full(lk, li))
        kw["loop_form"] = lkw["form"]
    if "set_angles" in c:
        (ai, aj, ak, at0, akt), _ = c["set_angles"][0]
        kw["angles"] = (np.asarray(ai, np.int32), np.asarray(aj, np.int32), np.asarray(ak, np.int32), full(at0, ai),
                        full(akt, ai))
    e, _ = O.energy_forces(O.System(**kw), geo["x"])
    return np.asarray(e), m


@pytest.mark.parametrize("seed", range(24))
def test_random_force_field_equals_the_reference_builder(ref, seed):
    n, geo, over = draw(seed)
    args = SimulationConfig(LOOPS_PATH="unused.bedpe", OUT_PATH="/tmp/unused", N_BEADS=n, **over)
    want, robj = reference_energies(ref, n, geo, args)
    got, m = our_energies(n, geo, args)
    for t, name in enumerate(O.TERM_NAMES):
        assert got[t] == pytest.approx(want[t], rel=1e-9, abs=1e-11), (seed, name, got[t], want[t], over)
    assert np.allclose([m.radius1, m.radius2, m.r_comp], [robj.radius1, robj.radius2, robj.r_comp], rtol=1e-15)
