"""CPU checks of the two restatements the cut-off GPU tests compare against (tests/cells_ref.py,
tests/far_field_ref.py): each against an independent computation, so that a wrong reference cannot
make a wrong kernel pass."""
import numpy as np
import pytest

import cells_ref as CR
import far_field_ref as FR
from common import O, hilbert_positions


def lattice(side=24, spacing=0.1, offset=(0.013, -0.4, 2.0)):
    g = np.arange(side) * spacing
    return np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) + np.asarray(offset)


def _spread3(v):
    v = v.astype(np.uint32) & 0x3FF
    v = (v | (v << 16)) & 0x030000FF
    v = (v | (v << 8)) & 0x0300F00F
    v = (v | (v << 4)) & 0x030C30C3
    v = (v | (v << 2)) & 0x09249249
    return v


def _count_system(n, rc):
    return O.System(n=n, ev=(0, [100.0, 0.05, 0.1, 6.0]), cutoff=rc)


@pytest.mark.parametrize("rc,outlier", [(0.25, False), (0.45, False), (0.1, True)])
def test_grid_restatement_orders_like_the_oracle(rc, outlier):
    """Keys and (key, id) order of the restated grid equal a numpy Morton sort of the restated cell
    coordinates; the coarse branch (more than 64 cells per axis) gives 64 cells of extent / 63."""
    x = hilbert_positions(3000, noise=0.02, seed=4)
    if outlier:
        x[1717] += np.array([100.0, -60.0, 30.0])
    xc = CR.centred(x)
    keys, order, (cell, dim, origin) = CR.cell_list(xc, rc)
    c = CR.cell_coords(xc, cell, dim, origin)
    k = _spread3(c[:, 0]) | (_spread3(c[:, 1]) << 1) | (_spread3(c[:, 2]) << 2)
    ref_order = np.lexsort((np.arange(len(k)), k))
    assert np.array_equal(order, ref_order) and np.array_equal(keys, k[ref_order])
    extent = np.float32(xc.max()) - np.float32(xc.min())
    if outlier:
        assert dim == 64 and cell == np.float32(extent / np.float32(63)) and cell > rc
    else:
        assert cell == np.float32(np.float32(rc) * np.float32(1 + 2.0 ** -12)) and dim <= 64
        assert (dim - 1) * cell <= extent < dim * cell


def test_centre_is_the_index_order_mean():
    x = hilbert_positions(5000, noise=0.05, seed=9) * 37.0 + 11.0
    c = np.zeros(3)
    for row in x:
        c += row
    assert np.array_equal(CR.centred(x), (x - c / len(x)).astype(np.float32))


@pytest.mark.parametrize("rc", [0.2, 0.25, 0.3, 0.45])
def test_fp32_pair_test_counts_like_the_oracle(rc):
    """The emulated fmaf test accepts exactly the pairs the oracle's pair_in_cut accepts."""
    for x in (lattice(), hilbert_positions(6000, noise=0.01, seed=2)):
        i, _ = CR.in_cut_pairs(CR.centred(x), rc)
        assert len(i) == O.count_pairs(_count_system(len(x), rc), x)


def test_fma32_is_correctly_rounded():
    rng = np.random.default_rng(5)
    a = rng.normal(size=20000).astype(np.float32)
    b = rng.normal(size=20000).astype(np.float32)
    c = rng.normal(size=20000).astype(np.float32)
    # a * b + c = 1 + 3 * 2^-24 - 2^-64: FP64 rounds it onto the midpoint between two FP32 values, and
    # rounding that to even would go the wrong way (and its mirror image with every sign flipped)
    a[:100] = np.float32(2.0 ** -12 * (1 + 2.0 ** -20))
    b[:100] = np.float32(2.0 ** -12 * (1 - 2.0 ** -20))
    c[:100] = np.float32(1 + 2.0 ** -23)
    a[50:100], c[50:100] = -a[50:100], -c[50:100]
    got = CR._fma32(a, b, c)
    from fractions import Fraction

    for q in list(range(100)) + list(range(100, 20000, 97)):
        exact = Fraction(float(a[q])) * Fraction(float(b[q])) + Fraction(float(c[q]))
        lo = np.float32(float(exact))
        cands = [np.nextafter(lo, np.float32(-np.inf)), lo, np.nextafter(lo, np.float32(np.inf))]
        best = min(cands, key=lambda v: (abs(Fraction(float(v)) - exact), int(np.float32(v).view(np.uint32)) & 1))
        assert got[q] == best, (q, got[q], best)


@pytest.mark.parametrize("rc,expected", [(0.2, 3456), (0.3, 1728)])
def test_stencil_misses_on_the_lattice(rc, expected):
    """A grid of edge exactly rc loses in-cut pairs of a 0.1 nm lattice to the 27-cell stencil; the
    kernel's edge rc * (1 + 2^-12) loses none."""
    xc = CR.centred(lattice())
    i, j = CR.stencil_misses(xc, rc)
    assert len(i) == expected
    cc = CR.cell_coords(xc, *CR.grid(xc, rc, 0.0))
    assert (np.abs(cc[i] - cc[j]).max(axis=1) == 2).all()
    assert len(CR.stencil_misses(xc, rc, CR.CELL_MARGIN)[0]) == 0


def _far_layout(n, seed):
    rng = np.random.default_rng(seed)
    chrom = np.zeros(n, np.int32)
    pos, cid = 0, 0
    while pos < n:
        ln = int(rng.integers(1, 70))
        chrom[pos:pos + ln] = cid
        pos += ln
        cid += 1
    x = hilbert_positions(n, noise=0.02, seed=seed)
    return x, chrom


def test_far_field_clusters_split_at_tiles_and_chromosomes():
    chrom = np.array([0] * 31 + [1] * 2 + [2] * 40 + [3])
    start, cc = FR.clusters(chrom)
    assert start.tolist() == [0, 31, 32, 33, 64, 73, 74]
    assert cc.tolist() == [0, 1, 1, 2, 2, 3]


def test_far_field_sum_equals_the_double_loop():
    x, chrom = _far_layout(700, 3)
    for ev, chb in (((100.0, 0.05, 0.1, 6.0), (0.3, 5.0)), ((100.0, 0.05, 0.1, 3.0), None), (None, (0.3, 5.0))):
        r = FR.far_field(x, chrom, 0.4, ev, chb)
        e_ev, e_chb = FR.far_field_loop(x, chrom, 0.4, ev, chb)
        assert abs(r["e_ev"] - e_ev) <= 1e-12 * max(abs(e_ev), 1e-300)
        assert abs(r["e_chb"] - e_chb) <= 1e-12 * max(abs(e_chb), 1e-300)
        assert r["n_below"] > 0 and r["n_band"] > 0 and r["n_above"] > 0


@pytest.mark.parametrize("power", [6.0, 3.0])
def test_far_field_force_is_minus_the_gradient(power):
    """Per-bead force against central differences of the reference's own energy, bead by bead along
    random directions (the band's smoothstep derivative included: most pairs here sit inside it)."""
    x, chrom = _far_layout(400, 7)
    ev, chb, rc = (100.0, 0.05, 0.1, power), (0.3, 5.0), 0.5
    r = FR.far_field(x, chrom, rc, ev, chb)
    assert r["n_band"] > 100

    def energy(y):
        q = FR.far_field(y, chrom, rc, ev, chb)
        return q["e_ev"] + q["e_chb"]

    rng = np.random.default_rng(1)
    h = 1e-5
    for i in rng.choice(len(x), size=12, replace=False):
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        xp, xm = x.copy(), x.copy()
        xp[i] += h * d
        xm[i] -= h * d
        slope = -(energy(xp) - energy(xm)) / (2 * h)
        got = float(r["force"][i] @ d)
        assert abs(slope - got) <= 1e-6 * max(np.abs(r["force"]).max(), 1.0), (i, slope, got)
