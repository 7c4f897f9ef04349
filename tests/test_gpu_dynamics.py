"""Locus dynamics on the device (mmm_dynamics_configure / _add / _read / _read_runs): the sums and run statistics
equal the numpy restatement (tests/dynamics_ref.py) bit for bit for N from 50 to 2e5, several lag sets (lags
beyond S, a ring that wraps), three kinds of bin table, bins off and rows off; scripted anchor sequences pin the
histogram buckets and the censoring; the closed time per group equals the loop readout's contacts; reads change
nothing and configuring clears; a refusal (arguments, state, the cumulative guard, non-finite positions, a ring
that does not fit) leaves everything as it was; MD, evaluations, the sampler, the loop readout and the three-way
map are unchanged by adds; buffers are freed with the handle; the SAVE_DYNAMICS driver equals a reproduction
through Engine calls, its other outputs are unchanged, and an ensemble's sums are the sums of its members."""
import os

import numpy as np
import pytest

import dynamics_ref as DR
from common import make_case, to_engine
from test_gpu_contacts_fine import BEDPE, _engine
from test_gpu_md_sampling import _files

pytestmark = pytest.mark.gpu

MMM_ERR_ARG, MMM_ERR_STATE, MMM_ERR_NOMEM = -1, -3, -5  # include/multimm_b200.h


def _walk(n, s, seed, step=0.05):
    """s structures of a diffusing chain: anchors a few beads apart open and close at rc = 0.3 nm."""
    rng = np.random.default_rng(seed)
    x = np.cumsum(rng.normal(scale=0.08, size=(n, 3)), axis=0)
    out = []
    for _ in range(s):
        x = x + rng.normal(scale=step, size=(n, 3))
        out.append(x.copy())
    return out


def _bins(n, kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "runs":  # canonical: runs of beads in chain order, the chain ends left out
        b = (np.arange(n) * 97 // n).astype(np.int32)
        b[: n // 20] = -1
        b[-3:] = -1
        return b, 97
    if kind == "scattered":
        return rng.integers(-1, 300, size=n).astype(np.int32), 300
    return None, 0


def _rows(n, r, seed):
    rng = np.random.default_rng(seed)
    lo = rng.integers(0, n - 8, size=r)
    hi = np.minimum(lo + 2 + rng.geometric(0.3, size=r), n - 1)
    far = rng.random(r) < 0.1
    hi = np.where(far, rng.integers(0, n, size=r), hi)
    lo, hi = np.minimum(lo, hi), np.maximum(lo, hi)
    ok = hi > lo
    return dict(bead_lo=lo[ok], bead_hi=hi[ok], group=rng.integers(0, 2, size=ok.sum()).astype(np.int8))


def _read(eng, xs, lags, rc=0.3, bins=None, nb=0, rows=None):
    rows = rows or {}
    eng.dynamics_configure(rc, lags, bins, nb, rows.get("bead_lo"), rows.get("bead_hi"), rows.get("group"))
    for x in xs:
        eng.set_positions(x)
        eng.dynamics_add()
    return eng.dynamics_read()


def _ref(xs, lags, rc=0.3, bins=None, nb=0, rows=None):
    rows = rows or {}
    return DR.dynamics(xs, lags, rc, bins, nb, rows.get("bead_lo"), rows.get("bead_hi"), rows.get("group"))


def _assert_same(got, want, keys=DR.KEYS):
    for k in keys:
        if want[k] is None:
            assert got[k] is None, k
        else:
            assert np.asarray(got[k]).dtype == np.asarray(want[k]).dtype and np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("n,s,lags,kind,r", [
    (50, 5, [1], "runs", 30),
    (1000, 20, [1, 2, 4, 8], "scattered", 300),     # S > 2L: the ring wraps
    (3001, 12, [1, 3, 5, 7], "runs", 0),            # a lag set that is not powers of two; rows off
    (20_000, 10, [2, 16, 64], None, 5000),          # lags beyond S; bins off
    (20_000, 9, [1, 2, 4, 8, 16, 32, 64], "runs", 2000),
    (200_000, 6, [1, 2, 4], "runs", 100_000),
])
def test_sums_equal_reference(built_lib, n, s, lags, kind, r):
    xs = _walk(n, s, seed=n + s)
    bins, nb = _bins(n, kind, seed=n)
    rows = _rows(n, r, seed=r + 1) if r else None
    with _engine(xs[0]) as eng:
        got = _read(eng, xs, lags, bins=bins, nb=nb, rows=rows)
    want = _ref(xs, lags, bins=bins, nb=nb, rows=rows)
    _assert_same(got, want)
    assert got["samples"] == s and got["device_ms"] > 0.0
    if bins is not None:
        assert got["msd_sum"][0].sum() > 0
    if r >= 300:  # rows open and close
        assert got["hist"].sum() > 0 and got["left_runs"].sum() > 0 and 0 < got["closed"].sum() < len(rows["bead_lo"])


def test_scripted_runs_pin_buckets_and_censoring(built_lib):
    from multimm_b200 import contacts, dynamics

    C, O = 1, 0
    a = [C, C, O, O, O, C, O, O, O, O] + [C] * 9  # left closed 2, open 3, closed 1, open 4, closed 9 in progress
    b = [O] * 19                                   # never changes: one whole-window run
    c = [O] + [C] * 18                             # left open 1, closed 18 in progress
    n = 12
    xs = []
    for s in range(19):
        x = np.zeros((n, 3))
        x[:, 1] = np.arange(n) * 10.0  # the rows' pairs are far from each other
        for row, pat in enumerate((a, b, c)):
            x[2 * row + 1, 0] = 0.1 if pat[s] else 1.0  # bead 2 row + 1 against bead 2 row at rc = 0.3 nm
            x[2 * row + 1, 1] = x[2 * row, 1]
        xs.append(x)
    rows = dict(bead_lo=np.array([0, 2, 4]), bead_hi=np.array([1, 3, 5]), group=np.array([0, 1, 1], np.int8))
    with _engine(xs[0]) as eng:
        got = _read(eng, xs, [1, 2], rows=rows)
    _assert_same(got, _ref(xs, [1, 2], rows=rows))
    assert got["closed_runs"].tolist() == [1, 0, 0] and got["closed_len"].tolist() == [1, 0, 0]
    assert got["open_runs"].tolist() == [2, 0, 0] and got["open_len"].tolist() == [7, 0, 0]
    want_hist = np.zeros((2, 2, 64), np.uint64)
    want_hist[0, 0, 0] = 1  # closed, length 1
    want_hist[0, 1, 1] = 1  # open, length 3
    want_hist[0, 1, 2] = 1  # open, length 4
    assert np.array_equal(got["hist"], want_hist)
    assert got["hist_len"].tolist() == [[1, 7], [0, 0]]
    assert got["left_runs"].tolist() == [[1, 0], [0, 1]] and got["left_len"].tolist() == [[2, 0], [0, 1]]
    assert got["closed"].tolist() == [True, False, True] and got["length"].tolist() == [9, 19, 18]
    assert got["from_transition"].tolist() == [True, False, True]
    # the host folds the runs in progress: right-censored (began at a change) or whole-window
    mr = dict(valid=np.ones(3, bool), group=rows["group"].astype(np.int64), resolution=1)
    tab = {k: np.zeros(3, np.int64) for k in ("row", "chrom1", "start1", "end1", "chrom2", "start2", "end2")}
    gb = contacts.GenomeBins(np.zeros(n, np.int32), np.zeros(1, np.int32), np.zeros(1, np.int64), 1)
    got["msd_sum"] = np.zeros((2, 1), np.uint64)
    d = dynamics.result(got, [1, 2], gb, tab, mr, 0.3, 100, 0.001)
    assert d["right_runs"].tolist() == [[1, 0, 1], [0, 0, 0]] and d["right_len"].tolist() == [[9, 0, 18], [0, 0, 0]]
    assert d["whole_runs"].tolist() == [[0, 0, 0], [0, 1, 0]] and d["whole_len"].tolist() == [[0, 0, 0], [0, 19, 0]]
    lt = dynamics.lifetimes(d)
    assert np.allclose(lt["mean_ps"][0], [0.1, 3.5 * 0.1]) and np.isnan(lt["mean_ps"][1]).all()
    assert lt["right"].tolist() == [[1, 0], [1, 0]] and lt["whole"].tolist() == [[0, 0], [0, 1]]


def test_closed_time_equals_the_loop_readout(built_lib):
    n, s = 5000, 15
    xs = _walk(n, s, 3)
    rows = _rows(n, 1500, 4)
    lrows = dict(rows, first_lo=np.zeros_like(rows["bead_lo"]), end_lo=np.full_like(rows["bead_lo"], n),
                 first_hi=np.zeros_like(rows["bead_lo"]), end_hi=np.full_like(rows["bead_lo"], n))
    with _engine(xs[0]) as eng:
        got = _read(eng, xs, [1, 2, 4], rows=rows)
        eng.loops_configure(0.3, 0, **lrows)
        for x in xs:
            eng.set_positions(x)
            eng.loops_add()
        lp = eng.loops_read()
    grp = rows["group"]
    for g in (0, 1):
        m = grp == g
        now = np.where(got["closed"][m], got["length"][m], 0).sum()
        closed_time = int(got["closed_len"][m].sum() + got["left_len"][g, 0] + now)
        assert closed_time == int(lp["contacts"][m].sum()) and closed_time > 0


def test_reads_change_nothing_and_configure_clears(built_lib):
    n = 4000
    xs = _walk(n, 11, 5)
    bins, nb = _bins(n, "runs", 1)
    rows = _rows(n, 800, 6)
    with _engine(xs[0]) as eng:
        once = _read(eng, xs, [1, 2, 4], bins=bins, nb=nb, rows=rows)
        eng.dynamics_configure(0.3, [1, 2, 4], bins, nb, **rows)
        for x in xs:
            eng.set_positions(x)
            eng.dynamics_add()
            eng.dynamics_read()
            eng.dynamics_read()
        _assert_same(eng.dynamics_read(), once)
        eng.dynamics_configure(0.3, [1, 2, 4], bins, nb, **rows)
        r = eng.dynamics_read()
        assert r["samples"] == 0 and r["device_ms"] == 0.0
        assert not any(np.asarray(r[k]).any() for k in DR.KEYS)
        _assert_same(_read(eng, xs, [1, 2, 4], bins=bins, nb=nb, rows=rows), once)


def test_argument_and_state_errors(built_lib):
    from multimm_b200._lib import Error
    from multimm_b200.engine import Engine

    n = 100
    bins = np.zeros(n, np.int32)
    rows = dict(bead_lo=np.array([10]), bead_hi=np.array([20]), group=np.array([0], np.int8))
    with Engine(n) as eng:
        for call in (eng.dynamics_add, eng.dynamics_read):
            with pytest.raises(Error) as ei:
                call()
            assert ei.value.code == MMM_ERR_STATE
        eng.dynamics_configure(0.3, [1], bins, 1)  # configuring needs no positions; adding does
        with pytest.raises(Error) as ei:
            eng.dynamics_add()
        assert ei.value.code == MMM_ERR_STATE
        eng.set_positions(_walk(n, 1, 1)[0])
        bad = [dict(rc_nm=0.0), dict(rc_nm=float("nan")), dict(lags=[]), dict(lags=[0]), dict(lags=[4097]),
               dict(lags=[2, 2]), dict(lags=[4, 2]), dict(n_bins=0), dict(n_bins=2**22 + 1),
               dict(bin_of_bead=np.full(n, 1, np.int32)), dict(bin_of_bead=np.full(n, -2, np.int32)),
               dict(bead_lo=np.array([-1])), dict(bead_hi=np.array([100])), dict(bead_lo=np.array([20])),
               dict(group=np.array([2], np.int8)), dict(bin_of_bead=None, bead_lo=None, bead_hi=None, group=None)]
        for kw in bad:
            args = dict(rc_nm=0.3, lags=[1, 2], bin_of_bead=bins, n_bins=1, **rows)
            args.update(kw)
            with pytest.raises(ValueError):
                eng.dynamics_configure(**args)
            with pytest.raises(Error) as ei:  # a refused configuration leaves the accumulator unconfigured
                eng.dynamics_add()
            assert ei.value.code == MMM_ERR_STATE
        with pytest.raises(ValueError):
            eng.dynamics_configure(0.3, [1], None, 0, rows["bead_lo"], rows["bead_hi"], np.array([0, 1], np.int8))
        eng.dynamics_configure(0.3, [1, 4096], None, 0, **rows)  # rows only
        eng.dynamics_add()
        assert eng.dynamics_read()["samples"] == 1


def test_a_ring_that_does_not_fit_fails_cleanly(built_lib):
    from multimm_b200._lib import Error
    from multimm_b200.engine import Engine

    n = 2_000_000  # L = 4096 needs 197 GB of ring
    x = np.zeros((n, 3))  # a point: the guard allows any number of beads in one bin
    with Engine(n) as eng:
        eng.set_positions(x)
        with pytest.raises(Error) as ei:
            eng.dynamics_configure(0.3, [1, 4096], np.zeros(n, np.int32), 1)
        assert ei.value.code == MMM_ERR_NOMEM
        with pytest.raises(Error) as ei:
            eng.dynamics_add()
        assert ei.value.code == MMM_ERR_STATE
        eng.dynamics_configure(0.3, [1, 2], np.zeros(n, np.int32), 1)
        eng.dynamics_add()
        eng.dynamics_add()
        r = eng.dynamics_read()
        assert r["samples"] == 2 and r["msd_sum"].tolist() == [[0], [0]]


def test_refused_adds_leave_sums_ring_and_states_unchanged(built_lib):
    n = 64
    D = np.sqrt(0.6 * 2.0**32)  # one bin of 64 beads: an add over a union box of diagonal D bounds 0.6 x 2^62
    a = np.zeros((n, 3))
    a[:, 0] = np.arange(n) * (D / 2 / (n - 1))
    a[1::2, 0] = a[0::2, 0]
    a[1::2, 1] = 0.1  # the rows' anchors in contact at rc = 0.3 nm
    b = a.copy()
    b[:, 0] += D / 2  # the union of a and b spans D
    b[1::4, 1] = 5.0  # some anchors open
    far = a.copy()
    far[:, 0] += 2 * D
    bins = np.zeros(n, np.int32)
    rows = dict(bead_lo=np.arange(0, n - 1, 2), bead_hi=np.arange(1, n, 2), group=(np.arange(n // 2) % 2).astype(np.int8))
    with _engine(a) as eng:
        eng.dynamics_configure(0.3, [1, 2], bins, 1, **rows)
        for x in (a, b):
            eng.set_positions(x)
            eng.dynamics_add()
        before = eng.dynamics_read()
        eng.set_positions(far)  # the union would grow to 2.5 D: 3.75 x 2^62 more
        with pytest.raises(ValueError, match="overflow"):
            eng.dynamics_add()
        # set_positions refuses NaN and infinities itself; finite positions whose extent is not (+-1e308) reach
        # the guard, whose bounding box then has no finite diagonal
        huge = b.copy()
        huge[7, 2], huge[9, 2] = 1e308, -1e308
        eng.set_positions(huge)
        with pytest.raises(ValueError, match="overflow"):
            eng.dynamics_add()
        after = eng.dynamics_read()
        _assert_same(after, before)
        assert after["samples"] == 2 and after["device_ms"] == before["device_ms"]
        eng.set_positions(b)  # 0.75 + 0.6 < 2: accepted, and its lag-1 partner is b itself, not far
        eng.dynamics_add()
        _assert_same(eng.dynamics_read(), _ref([a, b, b], [1, 2], bins=bins, nb=1, rows=rows))


def test_add_leaves_md_evaluations_and_other_readouts_unchanged(built_lib):
    n = 3000
    case = make_case(n, n_chrom=2, seed=3)
    bins = (np.arange(n) * 100 // n).astype(np.int32)
    rows = _rows(n, 400, 2)
    lrows = dict(rows, first_lo=np.zeros_like(rows["bead_lo"]), end_lo=np.full_like(rows["bead_lo"], n),
                 first_hi=np.zeros_like(rows["bead_lo"]), end_hi=np.full_like(rows["bead_lo"], n))
    eng = to_engine(case)
    e0, f0 = eng.energy_forces()
    last0 = eng.last_result()
    eng.dynamics_configure(0.3, [1, 2], bins, 100, **rows)
    eng.dynamics_add()
    eng.dynamics_add()
    last1 = eng.last_result()
    for u, v in zip(last0, last1):
        assert np.array_equal(u, v)
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
        eng.loops_configure(0.3, 3, **lrows)
        eng.triplets_configure(0.3, bins, 100)
        if added:
            eng.dynamics_configure(0.3, [1, 2, 4], bins, 100, **rows)
        reps = []
        for _ in range(6):
            reps.append(eng.md_run(5, want_report=True))
            eng.sample()
            eng.loops_add()
            eng.triplets_add()
            if added:
                eng.dynamics_add()
        reads = (eng.sampler_read(), eng.loops_read(), eng.triplets_read())
        out.append((reps, eng.get_positions(), eng.get_velocities(), eng.energy_forces(), reads))
        if added:
            assert eng.dynamics_read()["samples"] == 6
        eng.close()
    (r0, x0, v0, ef0, rd0), (r1, x1, v1, ef1, rd1) = out
    assert r0 == r1 and np.array_equal(x0, x1) and np.array_equal(v0, v1)
    assert np.array_equal(ef0[0], ef1[0]) and np.array_equal(ef0[1], ef1[1])
    for u, v in zip(rd0, rd1):
        for k in u:
            if k == "device_ms":
                continue
            assert (u[k] is None and v[k] is None) or np.array_equal(u[k], v[k]), k


# ---- driver -------------------------------------------------------------------------------------------
def _ini(path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=1500, LOOPS_PATH=BEDPE, OUT_PATH=str(path / "out"), SAVE_PLOTS=False,
                CHROM="chr1", LOC_START=10_000_000, LOC_END=60_000_000, MIN_MAX_ITERATIONS=150, SIM_RUN_MD=True,
                SIM_N_STEPS=650, SIM_SAMPLING_STEP=100, TRJ_FRAMES=4, DOWNSAMPLING_PROB=0.5, SAVE_DYNAMICS=True,
                DYNAMICS_MAX_LAG=2, DYNAMICS_RESOLUTION=500_000, CONTACT_RADIUS=0.25, MD_SAMPLE_STEP=150)
    base.update(fields)
    path.mkdir(parents=True, exist_ok=True)
    ini = path / "config.ini"
    ini.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items() if v is not None))
    return str(ini), base["OUT_PATH"]


def test_driver_file_equals_reproduction(built_lib, tmp_path):
    from multimm_b200 import contacts, dynamics, loaders, loops, run
    from multimm_b200.model import MultiMM, _f

    step = 150
    ini, out = _ini(tmp_path / "s")
    assert run.main(["-c", ini]) == 0
    ini0, out0 = _ini(tmp_path / "p", SAVE_DYNAMICS=None, DYNAMICS_MAX_LAG=None, DYNAMICS_RESOLUTION=None,
                      MD_SAMPLE_STEP=None)
    assert run.main(["-c", ini0]) == 0
    got, plain = _files(out), _files(out0)
    assert set(got) - set(plain) == {"analysis/dynamics.npz"} and set(plain) <= set(got)
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
    gb = contacts.genome_bins(m.layout, 500_000, n_beads=1500, max_bins=dynamics.MAX_BINS)
    rows = loops.device_rows(m.loop_rows)
    assert len(rows["bead_lo"]) > 0
    e.md_configure(str(a.SIM_INTEGRATOR_TYPE).lower(), _f(a.SIM_INTEGRATOR_STEP), _f(a.SIM_TEMPERATURE),
                   float(a.SIM_FRICTION_COEFF), loaders.BEAD_MASS, int(a.SHUFFLING_SEED), amd_alpha=_f(a.SIM_AMD_ALPHA),
                   amd_e=_f(a.SIM_AMD_E))
    e.set_velocities_to_temperature(_f(a.SIM_TEMPERATURE), int(a.SHUFFLING_SEED))
    e.dynamics_configure(0.25, [1, 2], gb.bins, gb.n_bins, rows["bead_lo"], rows["bead_hi"], rows["group"])
    done = 0
    while done < 600:
        e.md_run(50, want_report=False)
        done += 50
        if done % step == 0:
            e.dynamics_add()
    want = dynamics.result(e.dynamics_read(), [1, 2], gb, m.loop_table, m.loop_rows, 0.25, step,
                           _f(a.SIM_INTEGRATOR_STEP))
    m.close()
    d = dynamics.load(os.path.join(out, "analysis", "dynamics.npz"))
    for k in dynamics.KEYS:
        assert np.array_equal(d[k], want[k]) and d[k].dtype == np.asarray(want[k]).dtype, k
    assert int(d["samples"]) == 4 and d["msd_sum"].sum() > 0 and np.array_equal(d["lags"], [1, 2])


def test_ensemble_dynamics_are_the_sum_of_the_members(built_lib, tmp_path):
    from multimm_b200 import dynamics, run

    ini, out = _ini(tmp_path, N_BEADS=1000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=2, MD_SAMPLE_STEP=100,
                    SIM_N_STEPS=400, MIN_MAX_ITERATIONS=80)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=[0])
    parts = [dynamics.load(run.member_dynamics_path(out, i)) for i in range(2)]
    got = dynamics.load(os.path.join(out, "ensemble_dynamics.npz"))
    for k in dynamics.SUMS:
        assert got[k].dtype == np.uint64 and np.array_equal(got[k], parts[0][k] + parts[1][k]), k
    assert int(got["members"]) == 2 and int(got["samples"]) == 8


MEMORY_CHILD = r"""
import json, os, subprocess, sys
import numpy as np
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from test_gpu_dynamics import _rows, _walk
from multimm_b200.engine import Engine

def used_mib():
    out = subprocess.run(["nvidia-smi", "--query-compute-apps=pid,used_memory", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout
    for line in out.splitlines():
        pid, mem = [f.strip() for f in line.split(",")]
        if int(pid) == os.getpid():
            return float(mem.split()[0])
    return None

n = 200_000
xs = _walk(n, 3, 1)
bins = (np.arange(n) * 1000 // n).astype(np.int32)
used = []
for cycle in range(3):
    eng = Engine(n)
    eng.set_positions(xs[0])
    for lags, r in (([1, 2], 1000), ([1, 64], 50_000), ([1, 2, 4, 8, 16, 32, 64, 128, 256], 5000)):  # grow, then stay
        eng.dynamics_configure(0.3, lags, bins, 1000, **_rows(n, r, r))
        for x in xs:
            eng.set_positions(x)
            eng.dynamics_add()
        eng.dynamics_read()
    eng.close()
    used.append(used_mib())
print(json.dumps(used))
"""


def test_dynamics_buffers_freed_with_the_handle(built_lib):
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
