"""FP64 numpy restatement of the coarse stage's far field on cluster centroids (mmm_chb_clusters.cu).

Clusters: a new one starts at every bead i with i % 32 == 0 and wherever the chromosome id changes
(mmm_chb_clusters_build).  With c_T the centroid and n_T the size of cluster T, R = |c_T - c_U|,

    E_far = sum_{T < U} n_T n_U [ same_chromosome(T, U) dE (kC R^4 - R^3 + R^2)
                                  + S(R) eps (sigma / (R + r_s))^p ],

S = 0 for R <= 0.7 rc, the smoothstep t^2 (3 - 2 t), t = (R - 0.7 rc) / (0.6 rc), inside the band, and
1 for R >= 1.3 rc.  The EV tail is energy slot 0, CHB slot 3.  Every bead of T feels -dE_far/dc_T / n_T."""
from __future__ import annotations

import numpy as np

TILE = 32


def clusters(chrom):
    """(start[ncl + 1], chromosome id per cluster) as mmm_chb_clusters_build forms them."""
    chrom = np.asarray(chrom)
    n = len(chrom)
    i = np.arange(n)
    new = (i % TILE == 0)
    new[1:] |= chrom[1:] != chrom[:-1]
    start = np.flatnonzero(new)
    return np.append(start, n), chrom[start]


def centroids(x, start):
    """(c[ncl, 3], n[ncl]) in FP64."""
    x = np.asarray(x, dtype=np.float64)
    sizes = np.diff(start).astype(np.float64)
    sums = np.add.reduceat(x, start[:-1], axis=0)
    return sums / sizes[:, None], sizes


def _pair_terms(r, same, rc, ev, chb):
    """Per cluster pair (unit sizes): EV-tail energy, CHB energy, and -dphi/dR / R."""
    r_lo, r_hi = 0.7 * rc, 1.3 * rc
    e_ev = np.zeros_like(r)
    e_chb = np.zeros_like(r)
    g = np.zeros_like(r)
    if chb is not None:
        kc, de = chb
        e_chb = np.where(same, de * (kc * r ** 4 - r ** 3 + r ** 2), 0.0)
        g -= np.where(same, de * (4.0 * kc * r ** 2 - 3.0 * r + 2.0), 0.0)
    if ev is not None:
        eps, rs, sigma, p = ev
        u = eps * (sigma / (r + rs)) ** p
        du = -p * u / (r + rs)
        t = np.clip((r - r_lo) / (r_hi - r_lo), 0.0, 1.0)
        s = t * t * (3.0 - 2.0 * t)
        ds = np.where((r > r_lo) & (r < r_hi), 6.0 * t * (1.0 - t) / (r_hi - r_lo), 0.0)
        s = np.where(r > r_lo, s, 0.0)
        e_ev = u * s
        g -= (du * s + u * ds) / r
    return e_ev, e_chb, g


def far_field(x, chrom, rc, ev=None, chb=None):
    """E_far and its force.  ev = (eps, r_s, sigma, p) or None, chb = (kC, dE) or None.

    Returns dict: e_ev (slot 0), e_chb (slot 3), force (N, 3) per bead, and n_below / n_band / n_above,
    the numbers of unordered cluster pairs with R <= 0.7 rc, inside the band, and R >= 1.3 rc."""
    start, cchrom = clusters(chrom)
    c, nc = centroids(x, start)
    ncl = len(nc)
    d = c[:, None, :] - c[None, :, :]
    r = np.sqrt((d * d).sum(axis=2))
    off = ~np.eye(ncl, dtype=bool)
    r_safe = np.where(off, r, 1.0)
    same = (cchrom[:, None] == cchrom[None, :]) & off
    e_ev, e_chb, g = _pair_terms(r_safe, same, rc, ev, chb)
    w = nc[:, None] * nc[None, :] * off
    fcl = ((g * nc[None, :] * off)[:, :, None] * d).sum(axis=1)  # force per bead of cluster T
    iu = np.triu_indices(ncl, k=1)
    ru = r[iu]
    return dict(
        e_ev=0.5 * float((w * e_ev).sum()), e_chb=0.5 * float((w * e_chb).sum()),
        force=np.repeat(fcl, np.diff(start), axis=0), start=start, n_clusters=ncl,
        n_below=int((ru <= 0.7 * rc).sum()), n_band=int(((ru > 0.7 * rc) & (ru < 1.3 * rc)).sum()),
        n_above=int((ru >= 1.3 * rc).sum()))


def far_field_loop(x, chrom, rc, ev=None, chb=None):
    """(e_ev, e_chb) by a plain double loop over cluster pairs T < U (small cases only)."""
    start, cchrom = clusters(chrom)
    c, nc = centroids(x, start)
    e_ev = e_chb = 0.0
    r_lo, r_hi = 0.7 * rc, 1.3 * rc
    for t in range(len(nc)):
        for u in range(t + 1, len(nc)):
            r = float(np.sqrt(((c[t] - c[u]) ** 2).sum()))
            w = nc[t] * nc[u]
            if chb is not None and cchrom[t] == cchrom[u]:
                kc, de = chb
                e_chb += w * de * (kc * r ** 4 - r ** 3 + r ** 2)
            if ev is not None and r > r_lo:
                eps, rs, sigma, p = ev
                s = 1.0
                if r < r_hi:
                    q = (r - r_lo) / (r_hi - r_lo)
                    s = q * q * (3.0 - 2.0 * q)
                e_ev += w * s * eps * (sigma / (r + rs)) ** p
    return e_ev, e_chb
