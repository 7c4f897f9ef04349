"""Generates tests/golden/forcefield_golden.npz / .json by executing the REFERENCE's own force-field
builder ($MULTIMM_REFERENCE/src/multimm/model.py: set_radiuses and the ten add_* methods, unmodified)
against a RECORDING stand-in for the `openmm` module, and then evaluating the energy expressions
the reference handed to it — its own Lepton strings, global and per-particle parameters, bond /
angle / loop lists — with a small Lepton-to-numpy evaluator in FP64.

What this pins (the reference's tests pin nothing on this path): every functional form the
reference can select, which config field feeds which parameter, the per-particle parameter
plumbing (Cs, chrom_spin, chrom_strength), the topology rules, the radii.  What it cannot pin:
OpenMM's own evaluation of those expressions (OpenMM is not installable here); its conventions used
by the evaluator are the documented ones: HarmonicBondForce 1/2 k (r-r0)^2, HarmonicAngleForce
1/2 k (theta-theta0)^2, CustomNonbondedForce NoCutoff = sum over i<j with particle 1 = lower index,
delta(x) = [x == 0], step(x) = [x >= 0].

Needs MULTIMM_REFERENCE.   python tests/golden/make_golden_forcefield.py
"""
import importlib.util
import json
import os
import re
import sys
import types
from unittest.mock import MagicMock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.path.join(os.environ["MULTIMM_REFERENCE"], "src", "multimm")  # a checkout of the original MultiMM

from multimm_b200 import units  # noqa: E402
from multimm_b200.config import SimulationConfig  # noqa: E402


def md(v):
    return v.md if isinstance(v, units.Quantity) else float(v)


# ------------------------------------------------------------------------------------------------
# recording stand-in for the openmm module
# ------------------------------------------------------------------------------------------------
class _Force:
    kind = "?"

    def __init__(self, expr=None):
        self.expr, self.globals, self.per_names, self.rows, self.group = expr, {}, [], [], None

    def setEnergyFunction(self, e):
        self.expr = e

    def setForceGroup(self, g):
        self.group = g

    def addGlobalParameter(self, name, defaultValue=None):
        self.globals[name] = md(defaultValue)

    def addPerParticleParameter(self, name):
        self.per_names.append(name)

    addPerBondParameter = addPerParticleParameter


class CustomNonbondedForce(_Force):
    kind = "nonbonded"

    def addParticle(self, params=()):
        self.rows.append([md(p) for p in params])


class CustomExternalForce(_Force):
    kind = "external"

    def addParticle(self, index, params=()):
        self.rows.append((int(index), [md(p) for p in params]))


class CustomBondForce(_Force):
    kind = "custombond"

    def addBond(self, i, j, params=()):
        self.rows.append((int(i), int(j), [md(p) for p in params]))


class HarmonicBondForce(_Force):
    kind = "harmonicbond"

    def addBond(self, i, j, r0, k):
        self.rows.append((int(i), int(j), md(r0), md(k)))


class HarmonicAngleForce(_Force):
    kind = "harmonicangle"

    def addAngle(self, i, j, k, t0, kt):
        self.rows.append((int(i), int(j), int(k), md(t0), md(kt)))


class System:
    def __init__(self, n):
        self.n, self.forces = n, []

    def getNumParticles(self):
        return self.n

    def addForce(self, f):
        self.forces.append(f)


def load_reference_model():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.lines", "matplotlib.colors", "pyvista", "seaborn",
                 "mpl_toolkits", "mpl_toolkits.mplot3d", "pyBigWig", "hilbertcurve", "hilbertcurve.hilbertcurve",
                 "openmm.app"):
        sys.modules[name] = MagicMock()
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    mm = types.ModuleType("openmm")
    for cls in (CustomNonbondedForce, CustomExternalForce, CustomBondForce, HarmonicBondForce, HarmonicAngleForce):
        setattr(mm, cls.__name__, cls)
    unit = types.ModuleType("openmm.unit")
    unit.Quantity, unit.nanometers = units.Quantity, units.nanometers
    mm.unit = unit
    sys.modules["openmm"], sys.modules["openmm.unit"] = mm, unit
    pkg = types.ModuleType("multimm")
    pkg.__path__ = [REF]
    sys.modules["multimm"] = pkg
    for name in ("enums", "utils", "initial_structure_tools", "nucleosome_interpolation", "plots", "model"):
        spec = importlib.util.spec_from_file_location(f"multimm.{name}", os.path.join(REF, f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[f"multimm.{name}"] = mod
        spec.loader.exec_module(mod)
    return sys.modules["multimm.model"]


# ------------------------------------------------------------------------------------------------
# Lepton -> numpy
# ------------------------------------------------------------------------------------------------
FUNCS = dict(exp=np.exp, sin=np.sin, cos=np.cos, sqrt=np.sqrt, log=np.log, abs=np.abs,
             delta=lambda x: (np.asarray(x) == 0).astype(float), step=lambda x: (np.asarray(x) >= 0).astype(float),
             max=np.maximum, min=np.minimum)


def lepton(expr: str, env: dict):
    """Value of a Lepton expression "main; name = expr; ..." (later definitions may be used by earlier ones)."""
    fix = lambda t: re.sub(r"\blambda\b", "lambda_", t).replace("^", "**")  # noqa: E731
    parts = [p.strip() for p in expr.split(";") if p.strip()]
    ns = dict(FUNCS)
    ns.update({("lambda_" if k == "lambda" else k): v for k, v in env.items()})
    for part in reversed(parts[1:]):
        name, rhs = part.split("=", 1)
        ns[fix(name.strip())] = eval(fix(rhs), {"__builtins__": {}}, ns)  # noqa: S307 (trusted: the reference's own strings)
    return eval(fix(parts[0]), {"__builtins__": {}}, ns)  # noqa: S307


def energy(force, x):
    n = len(x)
    if force.kind == "nonbonded":
        i, j = np.triu_indices(n, k=1)
        d = x[i] - x[j]
        env = dict(force.globals, r=np.sqrt((d * d).sum(axis=1)))
        rows = np.asarray(force.rows, dtype=float).reshape(n, -1)
        for c, name in enumerate(force.per_names):
            env[name + "1"], env[name + "2"] = rows[i, c], rows[j, c]
        return float(np.sum(lepton(force.expr, env) * np.ones(len(i))))
    if force.kind == "external":
        idx = np.array([r[0] for r in force.rows])
        env = dict(force.globals, x=x[idx, 0], y=x[idx, 1], z=x[idx, 2])
        for c, name in enumerate(force.per_names):
            env[name] = np.array([r[1][c] for r in force.rows])
        return float(np.sum(lepton(force.expr, env) * np.ones(len(idx))))
    if force.kind == "harmonicbond":
        i, j = np.array([r[0] for r in force.rows]), np.array([r[1] for r in force.rows])
        r0, k = np.array([r[2] for r in force.rows]), np.array([r[3] for r in force.rows])
        r = np.linalg.norm(x[i] - x[j], axis=1)
        return float(np.sum(0.5 * k * (r - r0) ** 2))
    if force.kind == "custombond":
        i, j = np.array([r[0] for r in force.rows]), np.array([r[1] for r in force.rows])
        env = dict(force.globals, r=np.linalg.norm(x[i] - x[j], axis=1))
        for c, name in enumerate(force.per_names):
            env[name] = np.array([r[2][c] for r in force.rows])
        return float(np.sum(lepton(force.expr, env)))
    if force.kind == "harmonicangle":
        e = 0.0
        for i, j, k, t0, kt in force.rows:
            u, v = x[i] - x[j], x[k] - x[j]
            th = np.arccos(np.clip(np.dot(u, v) / (np.linalg.norm(u) * np.linalg.norm(v)), -1.0, 1.0))
            e += 0.5 * kt * (th - t0) ** 2
        return float(e)
    raise ValueError(force.kind)


# ------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------
ALL_ON = dict(EV_USE_EXCLUDED_VOLUME=True, COB_USE_COMPARTMENT_BLOCKS=True, SCB_USE_SUBCOMPARTMENT_BLOCKS=True,
              CHB_USE_CHROMOSOMAL_BLOCKS=True, SC_USE_SPHERICAL_CONTAINER=True, IBL_USE_B_LAMINA_INTERACTION=True,
              CF_USE_CENTRAL_FORCE=True, POL_USE_HARMONIC_BOND=True, LE_USE_HARMONIC_BOND=True, POL_USE_HARMONIC_ANGLE=True)
CASES = {
    "default_forms": dict(),
    "fixed_loop_distances": dict(LE_FIXED_DISTANCES=True, EV_POWER=3.0),
    "alt1": dict(EV_FORCE_TYPE="gaussian_core", COB_FORCE_TYPE="yukawa", SCB_FORCE_TYPE="yukawa", CHB_FORCE_TYPE="gaussian",
                 BLAMINA_FORCE_TYPE="gaussian_shell", CENTRAL_FORCE_TYPE="gaussian", LE_LOOP_FORCE_TYPE="fene_soft"),
    "alt2": dict(COB_FORCE_TYPE="theta", SCB_FORCE_TYPE="theta", CHB_FORCE_TYPE="saturating",
                 BLAMINA_FORCE_TYPE="harmonic_shell", CENTRAL_FORCE_TYPE="logistic", LE_LOOP_FORCE_TYPE="gaussian_tether"),
    "alt3": dict(BLAMINA_FORCE_TYPE="logistic_shell", EV_POWER=4.5, COB_EA=1.7, SCB_EB2=2.6, CHB_DE=0.01, CF_STRENGTH=3.0),
}
TERM_OF_ATTR = [("ev_force", "EV"), ("comp_force", "COB"), ("scomp_force", "SCB"), ("chrom_block_force", "CHB"),
                ("container_force", "SC"), ("Blamina_force", "LAM"), ("central_force", "CF"), ("bond_force", "BOND"),
                ("loop_force", "LOOP"), ("angle_force", "ANGLE")]


def geometry(seed=5, n=60):
    rng = np.random.default_rng(seed)
    x = np.cumsum(rng.normal(0, 0.08, size=(n, 3)), axis=0) + rng.normal(0, 0.02, size=(n, 3))
    chr_ends = np.array([0, 25, 41, n])
    chrom_idxs = np.array([2, 0, 1])  # a shuffled order
    Cs = rng.choice([-2, -1, 0, 1, 2], size=n)
    ms = np.array([1, 5, 12, 30, 44])
    ns = np.array([9, 20, 19, 38, 57])
    ds = np.array([0.1, 0.13, 0.2, 0.17, 0.11])
    strength = np.array([0.0, 0.35, 1.0])  # by POSITION in the shuffled order (model.py:162)
    spin, cstr = np.zeros(n), np.zeros(n)
    for k in range(3):
        spin[chr_ends[k]:chr_ends[k + 1]] = chrom_idxs[k]
        cstr[chr_ends[k]:chr_ends[k + 1]] = strength[k]
    return dict(x=x, chr_ends=chr_ends, chrom_idxs=chrom_idxs, Cs=Cs, ms=ms, ns=ns, ds=ds, chrom_spin=spin,
                chrom_strength=cstr)


def main():
    model = load_reference_model()
    geo = geometry()
    n = len(geo["x"])
    out, audit = {k: np.asarray(v) for k, v in geo.items()}, {}
    for name, over in CASES.items():
        args = SimulationConfig(LOOPS_PATH="unused.bedpe", OUT_PATH="/tmp/unused", N_BEADS=n, **ALL_ON, **over)
        obj = model.MultiMM.__new__(model.MultiMM)
        obj.args, obj.system = args, System(n)
        for k in ("chr_ends", "Cs", "ms", "ns", "ds", "chrom_spin", "chrom_strength"):
            setattr(obj, k, geo[k])
        obj.set_radiuses()
        obj.mass_center = np.average(geo["x"], axis=0)
        obj.add_forcefield()
        assert len(obj.system.forces) == 10, [type(f).__name__ for f in obj.system.forces]
        energies = np.zeros(10)
        audit[name] = dict(overrides={k: v for k, v in over.items()}, radius1=obj.radius1, radius2=obj.radius2,
                           r_comp=obj.r_comp, forces={})
        # attribute names differ between terms; take the forces in the order add_forcefield built them
        for t, f in enumerate(obj.system.forces):
            energies[t] = energy(f, geo["x"])
            audit[name]["forces"][TERM_OF_ATTR[t][1]] = dict(kind=f.kind, expr=f.expr, globals=f.globals,
                                                             per=f.per_names, n_rows=len(f.rows))
        out[f"{name}.energies"] = energies
        out[f"{name}.radii"] = np.array([obj.radius1, obj.radius2, obj.r_comp])
        bond = obj.system.forces[7]
        out[f"{name}.bonds"] = np.array([(r[0], r[1]) for r in bond.rows])
        ang = obj.system.forces[9]
        out[f"{name}.angles"] = np.array([(r[0], r[1], r[2]) for r in ang.rows])
        print(name, np.array2string(energies, precision=6))
    np.savez_compressed(os.path.join(HERE, "forcefield_golden.npz"), **out)
    with open(os.path.join(HERE, "forcefield_golden_expressions.json"), "w") as fh:
        json.dump(audit, fh, indent=1, default=float)


if __name__ == "__main__":
    main()
