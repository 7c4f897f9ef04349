"""numpy restatement of mmm_loops_add: the per-row sums and the APA sums of one structure, with the FP64
expression of mmm_contacts (d2 = (dx*dx + dy*dy) + dz*dz, operation by operation) and distances.quantise."""
import numpy as np

from multimm_b200.distances import quantise


def d2(x, i, j):
    d = x[i] - x[j]
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def loop_sums(x, rows: dict, rc_nm: float, window: int) -> dict:
    """What Engine.loops_read returns after one add at positions x (N, 3), for the device rows ``rows``
    (loops.device_rows): contacts, dist_sum, dist2_sum uint64[R]; apa_contacts, apa_dist_sum uint64
    [2][2W+1][2W+1]."""
    x = np.asarray(x, np.float64)
    lo, hi = np.asarray(rows["bead_lo"], np.int64), np.asarray(rows["bead_hi"], np.int64)
    f_lo, e_lo = np.asarray(rows["first_lo"], np.int64), np.asarray(rows["end_lo"], np.int64)
    f_hi, e_hi = np.asarray(rows["first_hi"], np.int64), np.asarray(rows["end_hi"], np.int64)
    g = np.asarray(rows["group"], np.int64)
    rc2 = float(rc_nm) * float(rc_nm)
    w = int(window)
    span = 2 * w + 1
    dd = d2(x, lo, hi)
    out = dict(contacts=(dd < rc2).astype(np.uint64), dist_sum=quantise(np.sqrt(dd)), dist2_sum=quantise(dd),
               apa_contacts=np.zeros((2, span, span), np.uint64), apa_dist_sum=np.zeros((2, span, span), np.uint64))
    for ia in range(span):
        pl = lo + ia - w
        for ib in range(span):
            ph = hi + ib - w
            ok = (pl >= f_lo) & (pl < e_lo) & (ph >= f_hi) & (ph < e_hi) & (pl < ph)
            if not ok.any():
                continue
            dd = d2(x, pl[ok], ph[ok])
            hit, q = (dd < rc2).astype(np.uint64), quantise(np.sqrt(dd))
            for grp in (0, 1):
                sel = g[ok] == grp
                out["apa_contacts"][grp, ia, ib] = hit[sel].sum(dtype=np.uint64)
                out["apa_dist_sum"][grp, ia, ib] = q[sel].sum(dtype=np.uint64)
    return out
