"""The loop readout on the device (mmm_loops_configure / mmm_loops_add / mmm_loops_read): its sums equal the
numpy restatement (tests/loops_ref.py) exactly, for several N, W and R (R = 0 and R = 1e5 included), and the
existing device paths (mmm_contacts_sparse, mmm_distance_map) where they measure the same pairs; K adds equal
the sum of K single reads and configuring clears; no side effects on evaluations or MD; argument, state and
cumulative-overflow refusals; buffers freed with the handle; the SAVE_LOOPS driver against a reproduction
through Engine calls, its other outputs unchanged, and an ensemble's sums."""
import os

import numpy as np
import pytest

import loops_ref as LR
from common import make_case, to_engine
from test_gpu_contacts_fine import BEDPE, _engine
from test_gpu_md_sampling import _files

pytestmark = pytest.mark.gpu

MMM_ERR_ARG, MMM_ERR_STATE = -1, -3  # include/multimm_b200.h


def _chain(n, seed, step=0.08):
    """A compact random walk: near-diagonal bead pairs are in contact at rc ~ 0.3 nm, far ones mostly not."""
    rng = np.random.default_rng(seed)
    return np.cumsum(rng.normal(scale=step, size=(n, 3)), axis=0)


def _rows(n, r, seed, n_chrom=4):
    """r rows on n beads in n_chrom blocks: intra- and inter-block, anchors at block and chain ends."""
    rng = np.random.default_rng(seed)
    ce = np.unique(np.concatenate([[0, n], np.sort(rng.integers(1, n, size=n_chrom - 1))]))
    lo = rng.integers(0, n - 3, size=r)
    span = np.minimum(3 + rng.geometric(1.0 / 40.0, size=r), n - 1 - lo)
    far = rng.random(r) < 0.2
    hi = np.where(far, rng.integers(0, n, size=r), lo + span)
    lo, hi = np.minimum(lo, hi), np.maximum(lo, hi)
    if r >= 4:
        lo[:4], hi[:4] = [0, ce[1] - 1, 0, n - 4], [n - 1, ce[1] + 3, 3, n - 1]
    ok = hi > lo
    lo, hi = lo[ok], hi[ok]
    blk = lambda b: np.searchsorted(ce, b, side="right") - 1  # noqa: E731
    return dict(bead_lo=lo, bead_hi=hi, first_lo=ce[blk(lo)], end_lo=ce[blk(lo) + 1], first_hi=ce[blk(hi)],
                end_hi=ce[blk(hi) + 1], group=rng.integers(0, 2, size=len(lo)).astype(np.int8))


def _read(eng, rows, rc, w, xs):
    eng.loops_configure(rc, w, **rows)
    for x in xs:
        eng.set_positions(x)
        eng.loops_add()
    return eng.loops_read()


KEYS = ("contacts", "dist_sum", "dist2_sum", "apa_contacts", "apa_dist_sum")


def _assert_same(got, want, keys=KEYS):
    for k in keys:
        assert got[k].dtype == np.uint64 and np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("n,r,w", [(50, 0, 10), (50, 30, 0), (1000, 300, 1), (3001, 2000, 10), (20_000, 5000, 25),
                                   (200_000, 100_000, 10)])
def test_sums_equal_reference(built_lib, n, r, w):
    x = _chain(n, seed=n)
    rows = _rows(n, r, seed=r + w)
    rc = 0.3
    with _engine(x) as eng:
        got = _read(eng, rows, rc, w, [x])
        want = LR.loop_sums(x, rows, rc, w)
        _assert_same(got, want)
        assert got["samples"] == 1 and got["apa_contacts"].shape == (2, 2 * w + 1, 2 * w + 1)
        if r:
            assert got["device_ms"] > 0.0
        if r >= 2000:  # both groups and both verdicts occur
            assert 0 < got["contacts"].sum() < len(rows["bead_lo"])
            assert got["apa_contacts"][0].sum() > 0 and got["apa_contacts"][1].sum() > 0


def test_per_row_sums_match_the_sparse_map_and_the_distance_map(built_lib):
    n = 3000
    x = _chain(n, seed=2)
    rows = _rows(n, 400, seed=3)
    rc = 0.3
    with _engine(x) as eng:
        got = _read(eng, rows, rc, 2, [x])
        r, c, _, _ = eng.contacts_sparse(rc, np.arange(n, dtype=np.int32), n)
        keys = set((r.astype(np.int64) * n + c).tolist())
        lo, hi = rows["bead_lo"].astype(np.int64), rows["bead_hi"].astype(np.int64)
        want = np.array([(a * n + b) in keys for a, b in zip(lo, hi)], np.uint64)
        assert np.array_equal(got["contacts"], want) and want.sum() > 0
        for k in range(0, len(lo), 25):
            bins = np.full(n, -1, np.int32)
            bins[lo[k]], bins[hi[k]] = 0, 1
            ds, d2s = eng.distance_map(bins, 2)
            assert ds[0, 1] == got["dist_sum"][k] and d2s[0, 1] == got["dist2_sum"][k]


def test_k_adds_equal_the_sum_of_single_reads_and_configure_clears(built_lib):
    n = 5000
    xs = [_chain(n, seed=s) for s in range(5)]
    rows = _rows(n, 1500, seed=9)
    with _engine(xs[0]) as eng:
        singles = [_read(eng, rows, 0.3, 7, [x]) for x in xs]
        many = _read(eng, rows, 0.3, 7, xs)
        assert many["samples"] == 5
        _assert_same(many, {k: sum(s[k] for s in singles) for k in KEYS})
        eng.loops_configure(0.3, 7, **rows)
        r = eng.loops_read()
        assert r["samples"] == 0 and r["device_ms"] == 0.0 and not any(r[k].any() for k in KEYS)
        eng.loops_configure(0.3, 7, **{k: v[:0] for k, v in rows.items()})  # no rows: adds still count
        eng.loops_add()
        r = eng.loops_read()
        assert r["samples"] == 1 and len(r["contacts"]) == 0 and not r["apa_contacts"].any()


def test_add_leaves_evaluations_and_md_unchanged(built_lib):
    case = make_case(3000, n_chrom=2, seed=3)
    rows = _rows(3000, 500, seed=4)
    eng = to_engine(case)
    e0, f0 = eng.energy_forces()
    last0 = eng.last_result()
    eng.loops_configure(0.2, 10, **rows)
    eng.loops_add()
    last1 = eng.last_result()
    for a, b in zip(last0, last1):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
    e1, f1 = eng.energy_forces()
    assert np.array_equal(e0, e1) and np.array_equal(f0, f1)
    eng.close()
    out = []
    for sampled in (False, True):
        eng = to_engine(case)
        eng.minimize(tol=10.0, max_iter=30)
        eng.md_configure("langevin", dt_ps=0.001, seed=7)
        eng.set_velocities_to_temperature(310.0, seed=8)
        if sampled:
            eng.loops_configure(0.2, 10, **rows)
        reps = []
        for _ in range(6):
            reps.append(eng.md_run(5, want_report=True))
            if sampled:
                eng.loops_add()
        out.append((reps, eng.get_positions(), eng.get_velocities(), eng.energy_forces()))
        if sampled:
            assert eng.loops_read()["samples"] == 6
        eng.close()
    (r0, x0, v0, ef0), (r1, x1, v1, ef1) = out
    assert r0 == r1
    assert np.array_equal(x0, x1) and np.array_equal(v0, v1)
    assert np.array_equal(ef0[0], ef1[0]) and np.array_equal(ef0[1], ef1[1])


def test_argument_and_state_errors(built_lib):
    from multimm_b200._lib import Error
    from multimm_b200.engine import Engine

    n = 100
    rows = _rows(n, 20, seed=1)
    with Engine(n) as eng:
        for call in (eng.loops_add, eng.loops_read):
            with pytest.raises(Error) as ei:
                call()
            assert ei.value.code == MMM_ERR_STATE
        eng.loops_configure(0.2, 3, **rows)  # configuring needs no positions; adding does
        with pytest.raises(Error) as ei:
            eng.loops_add()
        assert ei.value.code == MMM_ERR_STATE
        eng.set_positions(_chain(n, 1))
        one = {k: v[:1].copy() for k, v in rows.items()}
        one.update(bead_lo=np.array([10]), bead_hi=np.array([20]), first_lo=np.array([0]), end_lo=np.array([50]),
                   first_hi=np.array([0]), end_hi=np.array([50]), group=np.array([0], np.int8))
        bad = [dict(rc_nm=0.0), dict(rc_nm=float("inf")), dict(window=-1), dict(window=26),
               dict(bead_lo=np.array([60])), dict(bead_hi=np.array([50])), dict(bead_lo=np.array([20])),
               dict(bead_lo=np.array([30]), bead_hi=np.array([20])), dict(first_lo=np.array([-1])),
               dict(end_hi=np.array([101])), dict(first_hi=np.array([50])), dict(group=np.array([2], np.int8)),
               dict(group=np.array([-1], np.int8))]
        for kw in bad:
            args = dict(rc_nm=0.2, window=3, **one)
            args.update(kw)
            with pytest.raises(ValueError):
                eng.loops_configure(**args)
            with pytest.raises(Error) as ei:  # a refused configuration leaves the accumulator unconfigured
                eng.loops_add()
            assert ei.value.code == MMM_ERR_STATE
        with pytest.raises(ValueError):
            eng.loops_configure(0.2, 3, **dict(one, group=np.array([0, 1], np.int8)))
        eng.loops_configure(0.2, 25, **one)
        eng.loops_add()
        assert eng.loops_read()["samples"] == 1


def test_cumulative_guard_leaves_the_sums_unchanged(built_lib):
    n, r = 64, 40
    rows = _rows(n, r, seed=5)
    r = len(rows["bead_lo"])
    D = np.sqrt(0.99 * 2.0**62 / r / 2.0**24)  # one structure's bound just under 2^62
    x = np.zeros((n, 3))
    x[:, 0] = np.arange(n) * (D / (n - 1))
    with _engine(x) as eng:
        eng.loops_configure(0.2, 2, **rows)
        eng.loops_add()
        eng.loops_add()
        before = eng.loops_read()
        with pytest.raises(ValueError, match="overflow"):
            eng.loops_add()
        after = eng.loops_read()
        _assert_same(after, before)
        assert after["samples"] == 2 and after["device_ms"] == before["device_ms"]
        one = _read(eng, rows, 0.2, 2, [x])
        _assert_same(after, {k: 2 * one[k] for k in KEYS})


# ---- driver -------------------------------------------------------------------------------------------
def _ini(path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=1500, LOOPS_PATH=BEDPE, OUT_PATH=str(path / "out"), SAVE_PLOTS=False,
                CHROM="chr1", LOC_START=10_000_000, LOC_END=60_000_000, MIN_MAX_ITERATIONS=150, SIM_RUN_MD=True,
                SIM_N_STEPS=650, SIM_SAMPLING_STEP=100, TRJ_FRAMES=4, DOWNSAMPLING_PROB=0.5, SAVE_LOOPS=True,
                LOOP_APA_WINDOW=6, CONTACT_RADIUS=0.25)
    base.update(fields)
    path.mkdir(parents=True, exist_ok=True)
    ini = path / "config.ini"
    ini.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items() if v is not None))
    return str(ini), base["OUT_PATH"]


def test_driver_files_equal_reproduction(built_lib, tmp_path):
    from multimm_b200 import contacts, loaders, loops, run
    from multimm_b200.model import MultiMM, _f

    step = 150
    ini, out = _ini(tmp_path / "s", MD_SAMPLE_STEP=step)
    assert run.main(["-c", ini]) == 0
    ini0, out0 = _ini(tmp_path / "p", SAVE_LOOPS=None, LOOP_APA_WINDOW=None)
    assert run.main(["-c", ini0]) == 0
    got, plain = _files(out), _files(out0)
    new = {"analysis/loops.npz", "analysis/loops_md.npz"}
    assert set(got) - set(plain) == new and set(plain) <= set(got)
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
    mr = m.loop_rows
    assert (mr["valid"] & (mr["group"] == 0)).any() and (mr["valid"] & (mr["group"] == 1)).any()
    rows = loops.device_rows(mr)
    e.loops_configure(0.25, 6, **rows)
    e.loops_add()
    one = loops.result(m.loop_table, mr, e.loops_read(), 0.25, 6)
    e.md_configure(str(a.SIM_INTEGRATOR_TYPE).lower(), _f(a.SIM_INTEGRATOR_STEP), _f(a.SIM_TEMPERATURE),
                   float(a.SIM_FRICTION_COEFF), loaders.BEAD_MASS, int(a.SHUFFLING_SEED), amd_alpha=_f(a.SIM_AMD_ALPHA),
                   amd_e=_f(a.SIM_AMD_E))
    e.set_velocities_to_temperature(_f(a.SIM_TEMPERATURE), int(a.SHUFFLING_SEED))
    e.loops_configure(0.25, 6, **rows)
    done = 0
    while done < 600:
        e.md_run(50, want_report=False)
        done += 50
        if done % step == 0:
            e.loops_add()
    md = loops.result(m.loop_table, mr, e.loops_read(), 0.25, 6, 600 // step)
    m.close()
    for name, want in (("loops.npz", one), ("loops_md.npz", md)):
        d = loops.load(os.path.join(out, "analysis", name))
        for k in loops.KEYS:
            assert np.array_equal(d[k], want[k]) and d[k].dtype == np.asarray(want[k]).dtype, (name, k)
    d = loops.load(os.path.join(out, "analysis", "loops_md.npz"))
    assert int(d["members"]) == 4 and np.array_equal(d["measured"], 4 * loops.load(
        os.path.join(out, "analysis", "loops.npz"))["measured"])
    assert contacts.md_path(os.path.join(out, "analysis", "loops.npz")).endswith("loops_md.npz")


def test_ensemble_loops_are_the_aggregate_of_the_members(built_lib, tmp_path):
    from multimm_b200 import loops, run

    ini, out = _ini(tmp_path, N_BEADS=1000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=2, MD_SAMPLE_STEP=200,
                    SIM_N_STEPS=400, MIN_MAX_ITERATIONS=80)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=[0])
    for name in (lambda p: p, lambda p: p[:-4] + "_md.npz"):
        paths = [name(run.member_loops_path(out, i)) for i in range(2)]
        want = loops.aggregate(paths)
        got = loops.load(name(os.path.join(out, "ensemble_loops.npz")))
        for k in loops.KEYS:
            assert np.array_equal(got[k], want[k]) and got[k].dtype == want[k].dtype, k
        parts = [loops.load(p) for p in paths]
        assert int(got["members"]) == sum(int(p["members"]) for p in parts)
        assert not np.array_equal(parts[0]["enforced"], parts[1]["enforced"])  # down-sampling differs per member


MEMORY_CHILD = r"""
import json, os, subprocess, sys
import numpy as np
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from test_gpu_loops import _chain, _rows
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
x = _chain(n, 1)
used = []
for cycle in range(3):
    eng = Engine(n)
    eng.set_positions(x)
    for r, w in ((1000, 3), (300_000, 25), (50_000, 10)):  # the buffers grow, then stay
        eng.loops_configure(0.3, w, **_rows(n, r, seed=r))
        eng.loops_add()
        eng.loops_read()
    eng.close()
    used.append(used_mib())
print(json.dumps(used))
"""


def test_loop_buffers_freed_with_the_handle(built_lib):
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
