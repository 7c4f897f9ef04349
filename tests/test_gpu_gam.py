"""Genome architecture mapping on the device (mmm_gam_configure / mmm_gam_add / mmm_gam_read): the counts, `empty`
and `slices` equal the numpy restatement (tests/gam_ref.py) bit for bit for N from 50 to 2e5 (not all multiples of
32), canonical, holed and scattered bin tables, S = 1, 31, 32, 33, 1024 and 65536 slices, planes of
gam.slice_planes and axis-aligned planes whose boundaries beads hit exactly; the largest table; K adds equal the sum
of K single adds; refusals change nothing; no side effects on evaluations, MD or the other readouts; buffers freed
with the handle; the SAVE_GAM driver against a reproduction through Engine calls, its other outputs unchanged, and
an ensemble's sums.

The cumulative guard (the running slice total must stay below 2^63) cannot be reached in a test: it takes more
than 2^63 / 65536 = 1.4e14 adds."""
import os

import numpy as np
import pytest

import gam_ref as GR
from common import make_case, to_engine
from test_gpu_contacts_fine import BEDPE
from test_gpu_md_sampling import _files
from triplets_ref import globule

pytestmark = pytest.mark.gpu

MMM_ERR_ARG, MMM_ERR_STATE = -1, -3  # include/multimm_b200.h


def _table(kind, n, seed=0):
    rng = np.random.default_rng(seed)
    canon = (np.arange(n, dtype=np.int64) * min(n, 1000) // n).astype(np.int32)
    nb = int(canon[-1]) + 1
    if kind == "canonical":
        return canon, nb
    if kind == "holes":
        return np.where(rng.random(n) < 0.1, -1, canon).astype(np.int32), nb
    nb = 37  # scattered: any bead in any bin, some left out
    return rng.integers(-1, nb, size=n).astype(np.int32), nb


def _planes(x, bins, count, seed, fraction=0.025):
    from multimm_b200 import gam

    return gam.slice_planes(x, np.zeros(3), bins, count, fraction, np.random.default_rng(seed))


def _gam(eng, bins, nb, max_slices, xs_planes):
    eng.gam_configure(bins, nb, max_slices)
    for x, (planes, h) in xs_planes:
        eng.set_positions(x)
        eng.gam_add(planes, h)
    return eng.gam_read()


def _check(r, x, bins, nb, planes, h):
    want, empty = GR.gam_add(x, bins, nb, planes, h)
    assert r["counts"].dtype == np.uint64 and r["counts"].shape == want.shape
    assert np.array_equal(r["counts"], want)
    assert r["empty"] == empty and r["slices"] == len(planes) and r["structures"] == 1
    return want


CASES = [(50, "canonical", 1), (50, "scattered", 31), (50, "holes", 65536),
         (2000, "canonical", 32), (2000, "holes", 33), (2000, "scattered", 1024),
         (20_000, "canonical", 1024), (20_000, "holes", 33), (20_000, "scattered", 32),
         (200_000, "canonical", 1024)]


@pytest.mark.parametrize("n,kind,s", CASES)
def test_counts_equal_reference(built_lib, n, kind, s):
    from multimm_b200.engine import Engine

    x = globule(n, 680, n)
    bins, nb = _table(kind, n, n)
    planes, h = _planes(x, bins, s, n + s, fraction=0.025 if s >= 1024 else 0.1)
    with Engine(n) as eng:
        r = _gam(eng, bins, nb, s, [(x, (planes, h))])
    want = _check(r, x, bins, nb, planes, h)
    assert r["device_ms"] > 0.0
    if s >= 32:
        assert int(want.sum()) > 0


def test_beads_exactly_on_the_slab_boundaries(built_lib):
    """A lattice of spacing 0.5 nm and axis-aligned planes at multiples of 0.25 nm with h = 0.5 nm (and normals of
    length 2): every s is exact, and many beads lie exactly at |s| = h, which counts as inside."""
    from multimm_b200.engine import Engine

    n = 3001
    side = 15
    g = np.stack(np.meshgrid(*(np.arange(side),) * 3, indexing="ij"), -1).reshape(-1, 3)
    x = 0.5 * g[np.random.default_rng(1).permutation(len(g))[:n]].astype(np.float64)
    bins = (np.arange(n) * 40 // n).astype(np.int32)
    rng = np.random.default_rng(2)
    s = 97
    planes = np.zeros((s, 4))
    planes[np.arange(s), rng.integers(0, 3, s)] = rng.choice([1.0, -1.0, 2.0], s)
    planes[:, 3] = 0.25 * rng.integers(-8, 60, s)
    h = 0.5
    proj = ((planes[:, None, 0] * x[None, :, 0] + planes[:, None, 1] * x[None, :, 1]) + planes[:, None, 2] * x[None, :, 2]) \
        - planes[:, None, 3]
    assert np.count_nonzero(np.abs(proj) == h) > 1000
    with Engine(n) as eng:
        r = _gam(eng, bins, 40, s, [(x, (planes, h))])
        _check(r, x, bins, 40, planes, h)
        r2 = _gam(eng, bins, 40, s, [(x, (planes, np.nextafter(h, 0.0)))])
    _check(r2, x, bins, 40, planes, np.nextafter(h, 0.0))
    assert not np.array_equal(r["counts"], r2["counts"])


def test_the_largest_table(built_lib):
    """16383 bins (B (B + 1) / 2 just below 2^27): the beads sit in bins spread over every tile, the last one
    included; the rows of the bins in use equal the restatement and every other row is zero."""
    from multimm_b200 import gam
    from multimm_b200.engine import Engine

    n, nb = 500, gam.MAX_BINS
    x = globule(n, 680, 3)
    bins = ((np.arange(n) * 4099) % nb).astype(np.int32)
    bins[-1] = nb - 1
    planes, h = _planes(x, bins, 300, 4, fraction=0.2)
    with Engine(n) as eng:
        r = _gam(eng, bins, nb, 300, [(x, (planes, h))])
    det = GR.detection(x, bins, nb, planes, h)
    used = np.unique(bins)
    d = det[:, used].astype(np.int64)
    gram = d.T @ d
    i, j = np.triu_indices(len(used))
    p, q = used[i], used[j]
    rows = p * nb - p * (p - 1) // 2 + (q - p)
    assert r["counts"].shape == (nb * (nb + 1) // 2,)
    assert np.array_equal(r["counts"][rows], gram[i, j].astype(np.uint64))
    assert int(r["counts"].sum()) == int(gram[i, j].sum()) > 0
    assert r["empty"] == np.count_nonzero(~det.any(axis=1))


def test_k_adds_equal_the_sum_of_single_adds_and_configure_clears(built_lib):
    from multimm_b200.engine import Engine

    n = 3000
    bins, nb = _table("holes", n)
    runs = [(globule(n, 680, s), _planes(globule(n, 680, s), bins, cnt, s)) for s, cnt in enumerate((1024, 33, 500, 1))]
    with Engine(n) as eng:
        singles = [_gam(eng, bins, nb, 1024, [xp]) for xp in runs]
        r = _gam(eng, bins, nb, 1024, runs)
        assert r["structures"] == 4 and r["slices"] == 1024 + 33 + 500 + 1
        assert np.array_equal(r["counts"], sum(s["counts"] for s in singles))
        assert r["empty"] == sum(s["empty"] for s in singles)
        again = eng.gam_read()  # a read changes nothing
        assert np.array_equal(again["counts"], r["counts"]) and again["structures"] == 4
        eng.gam_configure(bins, nb, 1024)
        z = eng.gam_read()
        assert z["structures"] == z["slices"] == z["empty"] == 0 and not z["counts"].any()


def test_refusals_leave_the_state_unchanged(built_lib):
    from multimm_b200._lib import Error
    from multimm_b200.engine import Engine

    n = 100
    bins = (np.arange(n) % 5).astype(np.int32)
    x = globule(n, 680, 1)
    planes, h = _planes(x, bins, 64, 1, fraction=0.2)
    with Engine(n) as eng:
        for call in (lambda: eng.gam_add(planes, h), eng.gam_read):
            with pytest.raises(Error) as ei:
                call()
            assert ei.value.code == MMM_ERR_STATE
        eng.gam_configure(bins, 5, 64)  # configuring needs no positions; adding does
        with pytest.raises(Error) as ei:
            eng.gam_add(planes, h)
        assert ei.value.code == MMM_ERR_STATE
        eng.set_positions(x)
        bad = [dict(n_bins=0), dict(bin_of_bead=None), dict(bin_of_bead=np.full(n, -2, np.int32)),
               dict(bin_of_bead=np.full(n, 5, np.int32)), dict(max_slices=0), dict(max_slices=65537),
               dict(n_bins=16384, bin_of_bead=np.zeros(n, np.int32))]  # 1.34e8 + 16384 sums > 2^27
        for kw in bad:
            args = dict(bin_of_bead=bins, n_bins=5, max_slices=64)
            args.update(kw)
            with pytest.raises(ValueError):
                eng.gam_configure(**args)
            with pytest.raises(Error) as ei:  # a refused configuration leaves the accumulator unconfigured
                eng.gam_add(planes, h)
            assert ei.value.code == MMM_ERR_STATE
        with pytest.raises(ValueError):
            eng.gam_configure(bins[:-1], 5, 64)
        eng.gam_configure(bins, 5, 64)
        eng.gam_add(planes, h)
        before = eng.gam_read()
        assert before["structures"] == 1
        bad_adds = [(planes[:0], h), (np.concatenate([planes, planes[:1]]), h), (planes, np.nan), (planes, np.inf),
                    (planes, -1.0), (planes, -0.0 - 1e-300)]
        for v in (np.nan, np.inf, -np.inf):
            for col in (0, 3):
                p = planes.copy()
                p[17, col] = v
                bad_adds.append((p, h))
        for p, hh in bad_adds:
            with pytest.raises(ValueError):
                eng.gam_add(p, hh)
            after = eng.gam_read()
            for k in ("structures", "slices", "empty"):
                assert after[k] == before[k], k
            assert np.array_equal(after["counts"], before["counts"])
        with pytest.raises(ValueError):
            eng.gam_add(planes[:, :3], h)
        # non-finite positions never reach the counts (set_positions refuses them and leaves the handle without
        # positions; the add checks them again): the sums stay as they were
        for bad_x in (np.nan, np.inf):
            y = x.copy()
            y[17, 1] = bad_x
            with pytest.raises(Error, match="non-finite"):
                eng.set_positions(y)
            with pytest.raises(Error) as ei:
                eng.gam_add(planes, h)
            assert ei.value.code == MMM_ERR_STATE
            eng.set_positions(x)
            after = eng.gam_read()
            assert after["structures"] == 1 and np.array_equal(after["counts"], before["counts"])
        eng.gam_add(planes, h)  # still configured: the refusals changed nothing
        r = eng.gam_read()
        assert r["structures"] == 2 and np.array_equal(r["counts"], 2 * before["counts"])
        assert r["slices"] == 128 and r["empty"] == 2 * before["empty"]
        eng.gam_add(planes, 0.0)  # h = 0 is a plane of zero thickness: allowed
        assert eng.gam_read()["structures"] == 3


def test_add_leaves_evaluations_md_and_other_readouts_unchanged(built_lib):
    n = 3000
    case = make_case(n, n_chrom=2, seed=3)
    bins = (np.arange(n) * 100 // n).astype(np.int32)
    eng = to_engine(case)
    e0, f0 = eng.energy_forces()
    last0 = eng.last_result()
    eng.gam_configure(bins, 100, 1024)
    eng.gam_add(*_planes(eng.get_positions(), bins, 1024, 0))
    last1 = eng.last_result()
    for a, b in zip(last0, last1):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
    e1, f1 = eng.energy_forces()
    assert np.array_equal(e0, e1) and np.array_equal(f0, f1)
    eng.close()
    out = []
    for added in (False, True):
        eng = to_engine(case)
        eng.minimize(tol=10.0, max_iter=30)
        eng.md_configure("langevin", dt_ps=0.001, seed=7)
        eng.set_velocities_to_temperature(310.0, seed=8)
        eng.sampler_configure(0.3, bins, 100, np.arange(n, dtype=np.int32), n, bins, 100)
        eng.triplets_configure(0.3, bins, 100)
        eng.disthist_configure(bins, 100, [0.2, 0.5, 1.0])
        if added:
            eng.gam_configure(bins, 100, 512)
        reps = []
        for k in range(6):
            reps.append(eng.md_run(5, want_report=True))
            eng.sample()
            eng.triplets_add()
            eng.disthist_add()
            if added:
                eng.gam_add(*_planes(eng.get_positions(), bins, 512, k))
        s, t, dh = eng.sampler_read(), eng.triplets_read(), eng.disthist_read()
        out.append((reps, eng.get_positions(), eng.get_velocities(), eng.energy_forces(), s, t, dh))
        if added:
            assert eng.gam_read()["structures"] == 6
        eng.close()
    (r0, x0, v0, ef0, s0, t0, d0), (r1, x1, v1, ef1, s1, t1, d1) = out
    assert r0 == r1
    assert np.array_equal(x0, x1) and np.array_equal(v0, v1)
    assert np.array_equal(ef0[0], ef1[0]) and np.array_equal(ef0[1], ef1[1])
    for k in ("counts", "sep", "rows", "cols", "vals", "dist_sum", "dist2_sum"):
        assert np.array_equal(s0[k], s1[k]), k
    for k in ("p", "q", "r", "vals"):
        assert np.array_equal(t0[k], t1[k]), k
    assert s0["samples"] == s1["samples"] == 6 and t0["triples"] == t1["triples"]
    assert np.array_equal(d0["counts"], d1["counts"]) and d0["samples"] == d1["samples"] == 6


# ---- driver -------------------------------------------------------------------------------------------
def _ini(path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=1500, LOOPS_PATH=BEDPE, OUT_PATH=str(path / "out"), SAVE_PLOTS=False,
                CHROM="chr1", LOC_START=10_000_000, LOC_END=60_000_000, MIN_MAX_ITERATIONS=150, SIM_RUN_MD=True,
                SIM_N_STEPS=650, SIM_SAMPLING_STEP=100, TRJ_FRAMES=4, DOWNSAMPLING_PROB=0.5, SAVE_GAM=True,
                GAM_RESOLUTION=100_000, GAM_SLICES=700, GAM_SLICE_FRACTION=0.05)
    base.update(fields)
    path.mkdir(parents=True, exist_ok=True)
    ini = path / "config.ini"
    ini.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items() if v is not None))
    return str(ini), base["OUT_PATH"]


def test_driver_files_equal_reproduction(built_lib, tmp_path):
    from multimm_b200 import contacts, gam, loaders, run
    from multimm_b200.model import MultiMM, _f

    step = 150
    ini, out = _ini(tmp_path / "s", MD_SAMPLE_STEP=step)
    assert run.main(["-c", ini]) == 0
    ini0, out0 = _ini(tmp_path / "p", SAVE_GAM=None, GAM_RESOLUTION=None, GAM_SLICES=None, GAM_SLICE_FRACTION=None)
    assert run.main(["-c", ini0]) == 0
    got, plain = _files(out), _files(out0)
    assert set(got) - set(plain) == {"analysis/gam.npz", "analysis/gam_md.npz"}
    assert set(plain) <= set(got)
    for k in plain:
        if isinstance(plain[k], dict):
            assert plain[k].keys() == got[k].keys() and all(np.array_equal(plain[k][a], got[k][a]) for a in plain[k]), k
        else:
            assert plain[k] == got[k], k

    args, _ = run.get_config(["-c", ini, "--out_path", str(tmp_path / "r")])
    m = MultiMM(args)
    m.prepare()
    m.min_energy(write_files=False)
    e, a = m.engine, args
    seed = int(a.SHUFFLING_SEED)
    gb = contacts.genome_bins(m.layout, 100_000, n_beads=1500, max_bins=gam.MAX_BINS)
    assert gb.n_bins == 500

    def add(k):
        planes, h = gam.slice_planes(e.get_positions(), m.mass_center, gb.bins, 700, 0.05,
                                     np.random.default_rng([seed, k]))
        e.gam_add(planes, h)

    e.gam_configure(gb.bins, gb.n_bins, 700)
    add(0)
    one = gam.result(e.gam_read(), gb, 0.05)
    e.md_configure(str(a.SIM_INTEGRATOR_TYPE).lower(), _f(a.SIM_INTEGRATOR_STEP), _f(a.SIM_TEMPERATURE),
                   float(a.SIM_FRICTION_COEFF), loaders.BEAD_MASS, int(a.SHUFFLING_SEED), amd_alpha=_f(a.SIM_AMD_ALPHA),
                   amd_e=_f(a.SIM_AMD_E))
    e.set_velocities_to_temperature(_f(a.SIM_TEMPERATURE), int(a.SHUFFLING_SEED))
    e.gam_configure(gb.bins, gb.n_bins, 700)
    done = 0
    while done < 600:
        e.md_run(50, want_report=False)
        done += 50
        if done % step == 0:
            add(done // step)
    md = gam.result(e.gam_read(), gb, 0.05)
    m.close()
    assert int(one["slices"]) == 700 and int(md["slices"]) == 4 * 700 and int(md["structures"]) == 4
    for name, want in (("gam.npz", one), ("gam_md.npz", md)):
        d = gam.load(os.path.join(out, "analysis", name))
        for k in gam.KEYS:
            assert np.array_equal(d[k], want[k]) and d[k].dtype == np.asarray(want[k]).dtype, (name, k)
        f = gam.detection_frequency(d)
        seen = f > 0
        assert seen.sum() > 0.9 * len(f)
        v = gam.npmi(d)[np.ix_(seen, seen)]
        assert np.all(np.isfinite(v)) and np.all(np.abs(v) <= 1.0 + 1e-12)


def test_ensemble_gam_is_the_sum_of_the_members(built_lib, tmp_path):
    from multimm_b200 import gam, run

    ini, out = _ini(tmp_path, N_BEADS=1000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=2, MD_SAMPLE_STEP=200,
                    SIM_N_STEPS=400, MIN_MAX_ITERATIONS=80)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=[0])
    for name in (lambda p: p, lambda p: p[:-4] + "_md.npz"):
        paths = [name(run.member_gam_path(out, i)) for i in range(2)]
        parts = [gam.load(p) for p in paths]
        got = gam.load(name(os.path.join(out, "ensemble_gam.npz")))
        for k in gam.KEYS:
            assert np.array_equal(got[k], gam.aggregate(paths)[k]), k
        assert np.array_equal(got["counts"], parts[0]["counts"] + parts[1]["counts"])
        for k in ("structures", "slices", "empty"):
            assert int(got[k]) == sum(int(p[k]) for p in parts), k
        assert int(got["counts"].sum()) > 0
        assert not np.array_equal(parts[0]["counts"], parts[1]["counts"])


MEMORY_CHILD = r"""
import json, os, subprocess, sys
import numpy as np
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from triplets_ref import globule
from multimm_b200 import gam
from multimm_b200.engine import Engine

def used_mib():
    out = subprocess.run(["nvidia-smi", "--query-compute-apps=pid,used_memory", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout
    for line in out.splitlines():
        pid, mem = [f.strip() for f in line.split(",")]
        if int(pid) == os.getpid():
            return float(mem.split()[0])
    return None

n = 50_000
x = globule(n, 680, 1)
used = []
for cycle in range(3):
    eng = Engine(n)
    eng.set_positions(x)
    for nb, s in ((1000, 1024), (4096, 16384), (500, 65536)):
        bins = (np.arange(n) * nb // n).astype(np.int32)
        eng.gam_configure(bins, nb, s)
        eng.gam_add(*gam.slice_planes(x, np.zeros(3), bins, s, 0.025, np.random.default_rng(cycle)))
        eng.gam_read()
    eng.close()
    used.append(used_mib())
print(json.dumps(used))
"""


def test_gam_buffers_freed_with_the_handle(built_lib):
    import json
    import shutil
    import subprocess
    import sys

    if shutil.which("nvidia-smi") is None:
        pytest.skip("nvidia-smi is not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = MEMORY_CHILD.replace("ROOT", repr(root))
    res = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stderr[-3000:]
    used = json.loads(res.stdout.strip().splitlines()[-1])
    if used[0] is None:
        pytest.skip("nvidia-smi does not list this process (separate PID namespace)")
    assert used[2] - used[0] <= 2.0, f"device memory after cycles 1, 2, 3: {used} MiB"
