"""Shared builders for the tests: one description of a MultiMM system, handed both to the CPU
oracle (oracle/oracle.py) and to the engine through the C-ABI (multimm_b200.Engine)."""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import oracle as O  # noqa: E402

# Root of a checkout of the original MultiMM (github.com/SFGLab/MultiMM).  The tests that run its code
# live need one and skip without it; the outputs it gave are frozen under tests/golden and run everywhere.
REFERENCE = os.environ.get("MULTIMM_REFERENCE", "")
NO_REFERENCE = "no checkout of the original MultiMM named by MULTIMM_REFERENCE"


def reference_file(rel: str) -> str | None:
    """Path of `rel` inside the MULTIMM_REFERENCE checkout, None where there is no such file."""
    path = os.path.join(REFERENCE, rel) if REFERENCE else None
    return path if path and os.path.exists(path) else None

# reference defaults (config.py:188-246)
DEF = dict(
    bond_r0=0.1, bond_k=3.0e5, angle_t0=np.pi, angle_k=100.0, loop_r0=0.1, loop_k=3.0e4,
    ev_eps=100.0, ev_rs=0.05, ev_power=6.0, sc_scale=1000.0, chb_kc=0.3, chb_de=1e-4,
    cob_ea=1.0, cob_eb=2.0, scb=(1.0, 1.33, 1.66, 2.0), ibl_scale=400.0, cf_strength=20.0,
)


def radii(n, b0=0.1):
    """set_radiuses, model.py:1016-1067."""
    r2 = b0 * float(n) ** (1.0 / 3.0)
    r1 = r2 * 0.20 ** (1.0 / 3.0)
    return r1, r2, 1.5 * b0


def backbone(n, chr_ends):
    """Bond and angle start indices with the reference's quirks (model.py:628-635, 711-719)."""
    ce = np.asarray(chr_ends)
    i = np.arange(n - 1)
    bi = i[~np.isin(i, ce)]
    a = np.arange(n - 2)
    ai = a[~np.isin(a, ce) & ~np.isin(a, ce - 1)]
    return bi.astype(np.int32), ai.astype(np.int32)


def hilbert_positions(n, noise=0.0, seed=0):
    pts = O.hilbert_points(n, 8).astype(np.float64) * 0.1
    if noise > 0:
        pts = pts + np.random.default_rng(seed).normal(0.0, noise, size=pts.shape)
    return pts


def make_case(n, n_chrom=1, seed=0, terms=("EV", "SCB", "CHB", "SC", "LAM", "CF", "BOND", "LOOP", "ANGLE"),
              forms=None, n_loops=None, noise=0.01, ev_power=6.0, chb_de=None):
    """A synthetic system shaped like the reference builds it: contiguous chromosomes, 4-state
    compartments in runs, loops with r0 in [0.1, 0.2], Hilbert start with a little noise."""
    rng = np.random.default_rng(seed)
    forms = dict(forms or {})
    r1, r2, r_comp = radii(n)
    # chromosome boundaries (chr_ends = [0, e1, ..., N])
    if n_chrom > 1:
        cuts = np.sort(rng.choice(np.arange(3, n - 3), size=n_chrom - 1, replace=False))
        chr_ends = np.concatenate([[0], cuts, [n]])
    else:
        chr_ends = np.array([0, n])
    ids = rng.permutation(n_chrom)
    chrom = np.zeros(n, dtype=np.int32)
    cstr = np.zeros(n)
    strength = rng.random(max(n_chrom, 1))
    for c in range(n_chrom):
        chrom[chr_ends[c]:chr_ends[c + 1]] = ids[c]
        cstr[chr_ends[c]:chr_ends[c + 1]] = strength[c]
    # compartments in runs of geometric length
    s = np.zeros(n, dtype=np.int8)
    pos = 0
    while pos < n:
        run = int(rng.geometric(1.0 / 12.0))
        s[pos:pos + run] = rng.choice([-2, -1, 0, 1, 2])
        pos += run
    x = hilbert_positions(n, noise=noise, seed=seed + 1)
    center = x.mean(axis=0)
    bi, ai = backbone(n, chr_ends)
    nl = n_loops if n_loops is not None else max(1, n // 25)
    if n > 8:
        lm = rng.integers(0, n - 4, size=nl)
        ln = np.minimum(lm + 3 + rng.geometric(1.0 / 30.0, size=nl), n - 1)
        keep = ln > lm + 2
        lm, ln = lm[keep].astype(np.int32), ln[keep].astype(np.int32)
    else:
        lm = ln = np.zeros(0, dtype=np.int32)
    lr0 = 0.1 + 0.1 * rng.random(len(lm))
    case = dict(n=n, x=x, s=s, chrom=chrom, cstr=cstr, chr_ends=chr_ends, center=center,
                r1=r1, r2=r2, r_comp=r_comp, terms=tuple(terms), forms=forms)
    de = DEF["chb_de"] if chb_de is None else chb_de
    case["ev"] = (forms.get("EV", 0), [DEF["ev_eps"], DEF["ev_rs"], DEF["loop_r0"], ev_power]) if "EV" in terms else None
    case["cob"] = (forms.get("COB", 0), [r_comp, DEF["cob_ea"], DEF["cob_eb"]]) if "COB" in terms else None
    case["scb"] = (forms.get("SCB", 0), [r_comp, *DEF["scb"]]) if "SCB" in terms else None
    case["chb"] = (forms.get("CHB", 0), [DEF["chb_kc"], de]) if "CHB" in terms else None
    case["sc"] = (0, [DEF["sc_scale"], r1, r2, *center]) if "SC" in terms else None
    case["lam"] = (forms.get("LAM", 0), [DEF["ibl_scale"], r1, r2, *center]) if "LAM" in terms else None
    case["cf"] = (forms.get("CF", 0), [DEF["cf_strength"], r1, *center]) if "CF" in terms else None
    case["bonds"] = (bi, bi + 1, np.full(len(bi), DEF["bond_r0"]), np.full(len(bi), DEF["bond_k"])) if "BOND" in terms else None
    case["loops"] = (lm, ln, lr0, np.full(len(lm), DEF["loop_k"])) if "LOOP" in terms else None
    case["loop_form"] = forms.get("LOOP", 0)
    case["angles"] = (ai, ai + 1, ai + 2, np.full(len(ai), DEF["angle_t0"]), np.full(len(ai), DEF["angle_k"])) if "ANGLE" in terms else None
    return case


def to_oracle(case, cutoff=0.0) -> O.System:
    return O.System(n=case["n"], ev=case["ev"], cob=case["cob"], scb=case["scb"], chb=case["chb"], sc=case["sc"],
                    lam=case["lam"], cf=case["cf"], loop_form=case["loop_form"], cutoff=cutoff, s=case["s"],
                    chrom=case["chrom"], cstr=case["cstr"], bonds=case["bonds"], loops=case["loops"],
                    angles=case["angles"])


def to_engine(case, device=0, cutoff=0.0):
    from multimm_b200.engine import Engine

    eng = Engine(case["n"], device=device)
    eng.set_bead_params(case["s"], case["chrom"], case["cstr"])
    for name in ("ev", "cob", "scb", "chb"):
        if case[name] is not None:
            eng.set_pair_term(name.upper(), case[name][0], case[name][1])
    for name in ("sc", "lam", "cf"):
        if case[name] is not None:
            eng.set_external_term(name.upper(), case[name][0], case[name][1])
    if case["bonds"] is not None:
        eng.set_bonds(*case["bonds"])
    if case["loops"] is not None:
        eng.set_loops(*case["loops"], form=case["loop_form"])
    if case["angles"] is not None:
        eng.set_angles(*case["angles"])
    if cutoff > 0:
        eng.set_cutoff(cutoff)
    eng.set_positions(case["x"])
    return eng


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def force_rel_err(f, f_ref):
    """Per-bead force error relative to max(|F_ref_i|, RMS |F_ref|): the 1e-4 bar of the north star."""
    f, f_ref = np.asarray(f), np.asarray(f_ref)
    mag = np.linalg.norm(f_ref, axis=1)
    rms = float(np.sqrt((mag ** 2).mean()))
    den = np.maximum(mag, max(rms, 1e-300))
    return float((np.linalg.norm(f - f_ref, axis=1) / den).max())
