"""The force field against the REFERENCE's own builder.

tests/golden/make_golden_forcefield.py executed the unmodified add_* methods of
$MULTIMM_REFERENCE/src/multimm/model.py against a recording stand-in for `openmm` and evaluated the
Lepton strings, parameters and bond/angle lists they produced (FP64).  Here the same inputs go
through THIS repo's chain — host mirror (multimm_b200/model.py) -> the calls it would make on the
C-ABI -> CPU oracle — and every per-term energy must agree.  This pins, for every functional form:
the expressions, which config field feeds which parameter, the per-bead parameter plumbing, the
topology rules and the radii."""
import json
import os

import numpy as np
import pytest

from common import O
from multimm_b200 import model
from multimm_b200.config import SimulationConfig

GOLD = os.path.join(os.path.dirname(__file__), "golden")
G = np.load(os.path.join(GOLD, "forcefield_golden.npz"))
AUDIT = json.load(open(os.path.join(GOLD, "forcefield_golden_expressions.json")))

ALL_ON = dict(EV_USE_EXCLUDED_VOLUME=True, COB_USE_COMPARTMENT_BLOCKS=True, SCB_USE_SUBCOMPARTMENT_BLOCKS=True,
              CHB_USE_CHROMOSOMAL_BLOCKS=True, SC_USE_SPHERICAL_CONTAINER=True, IBL_USE_B_LAMINA_INTERACTION=True,
              CF_USE_CENTRAL_FORCE=True, POL_USE_HARMONIC_BOND=True, LE_USE_HARMONIC_BOND=True, POL_USE_HARMONIC_ANGLE=True)


class Recorder:
    def __init__(self):
        self.calls = {}

    def __getattr__(self, name):
        def rec(*a, **k):
            self.calls.setdefault(name, []).append((a, k))
        return rec


def our_chain(case):
    """Host mirror -> recorded C-ABI calls -> oracle System."""
    n = len(G["x"])
    args = SimulationConfig(LOOPS_PATH="unused.bedpe", OUT_PATH="/tmp/unused", N_BEADS=n, **ALL_ON, **AUDIT[case]["overrides"])
    m = model.MultiMM.__new__(model.MultiMM)
    m.args, m.engine, m.timings = args, Recorder(), {}
    m.chr_ends, m.Cs, m.ms, m.ns, m.ds = G["chr_ends"], G["Cs"], G["ms"], G["ns"], G["ds"]
    m.chrom_spin, m.chrom_strength = G["chrom_spin"], G["chrom_strength"]
    m.set_radiuses()
    m.mass_center = np.average(G["x"], axis=0)
    m.add_forcefield()
    c = m.engine.calls
    pair = {a[0]: (a[1], list(a[2])) for a, _ in c["set_pair_term"]}
    ext = {a[0]: (a[1], list(a[2])) for a, _ in c["set_external_term"]}
    (s, chrom, cstr), _ = c["set_bead_params"][0]
    (bi, bj, br0, bk), _ = c["set_bonds"][0]
    (li, lj, lr0, lk), lkw = c["set_loops"][0]
    (ai, aj, ak, at0, akt), _ = c["set_angles"][0]
    full = lambda v, ref: np.broadcast_to(np.asarray(v, dtype=float), np.shape(ref)).copy()  # noqa: E731
    sysd = O.System(n=n, ev=pair.get("EV"), cob=pair.get("COB"), scb=pair.get("SCB"), chb=pair.get("CHB"),
                    sc=ext.get("SC"), lam=ext.get("LAM"), cf=ext.get("CF"), loop_form=lkw["form"], cutoff=0.0,
                    s=np.asarray(s, dtype=np.int8), chrom=np.asarray(chrom, dtype=np.int32), cstr=np.asarray(cstr, float),
                    bonds=(np.asarray(bi, np.int32), np.asarray(bj, np.int32), full(br0, bi), full(bk, bi)),
                    loops=(np.asarray(li, np.int32), np.asarray(lj, np.int32), full(lr0, li), full(lk, li)),
                    angles=(np.asarray(ai, np.int32), np.asarray(aj, np.int32), np.asarray(ak, np.int32), full(at0, ai),
                            full(akt, ai)))
    return m, sysd, (bi, bj), (ai, aj, ak)


@pytest.mark.parametrize("case", list(AUDIT))
def test_per_term_energies_match_the_reference_builder(case):
    m, sysd, bonds, angles = our_chain(case)
    e, _ = O.energy_forces(sysd, G["x"])
    want = G[f"{case}.energies"]
    for t, name in enumerate(O.TERM_NAMES):
        assert e[t] == pytest.approx(want[t], rel=1e-10, abs=1e-12), (case, name, e[t], want[t])
    # radii and topology are the reference's
    assert np.allclose([m.radius1, m.radius2, m.r_comp], G[f"{case}.radii"], rtol=1e-15)
    assert np.array_equal(np.stack(bonds, axis=1), G[f"{case}.bonds"])
    assert np.array_equal(np.stack(angles, axis=1), G[f"{case}.angles"])


def test_the_golden_set_exercises_every_form():
    forms = {k: set() for k in ("EV", "COB", "SCB", "CHB", "LAM", "CF", "LOOP")}
    for case in AUDIT.values():
        for term in forms:
            forms[term].add(case["forces"][term]["expr"] or case["forces"][term]["kind"])
    assert len(forms["EV"]) == 2 and len(forms["COB"]) == 3 and len(forms["SCB"]) == 3 and len(forms["CHB"]) == 3
    assert len(forms["LAM"]) == 4 and len(forms["CF"]) == 3 and len(forms["LOOP"]) == 3
