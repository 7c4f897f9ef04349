"""Locus dynamics on the host: the numpy restatement (tests/dynamics_ref.py) against a brute-force loop, the
conservation of run lengths and transitions, the dynamics file format and its exact aggregation, the readers
(msd, relative_msd, exponent, lifetimes) and the SAVE_DYNAMICS / DYNAMICS_RESOLUTION / DYNAMICS_MAX_LAG settings
and their checks."""
import math
import os

import numpy as np
import pytest

import dynamics_ref as DR
from multimm_b200 import contacts, dynamics, loaders, loops

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


def _walk(n, s, seed, step=0.05):
    """s structures of n beads: a chain that diffuses, so anchors open and close at rc ~ 0.3 nm."""
    rng = np.random.default_rng(seed)
    x = np.cumsum(rng.normal(scale=0.08, size=(n, 3)), axis=0)
    out = []
    for _ in range(s):
        x = x + rng.normal(scale=step, size=(n, 3))
        out.append(x.copy())
    return out


def _rows(n, r, seed):
    rng = np.random.default_rng(seed)
    lo = rng.integers(0, n - 4, size=r)
    hi = np.minimum(lo + 2 + rng.integers(1, 6, size=r), n - 1)
    return lo, hi, rng.integers(0, 2, size=r)


# ---- the restatement -------------------------------------------------------------------------------------
def _brute(xs, lags, rc, bins, n_bins, lo, hi, group):
    """The definitions, element by element: per-sample states give the runs of every row directly."""
    S, n = len(xs), len(xs[0])
    q = lambda v: int(round(v * 2.0**24)) if v * 2.0**24 % 1 != 0.5 else int(math.floor(v * 2.0**24) + (math.floor(v * 2.0**24) % 2))  # noqa: E731
    d2 = lambda a, b: (((a[0] - b[0]) * (a[0] - b[0]) + (a[1] - b[1]) * (a[1] - b[1])) + (a[2] - b[2]) * (a[2] - b[2]))  # noqa: E731
    msd = np.zeros((len(lags), n_bins), np.uint64)
    rel = np.zeros((len(lags), len(lo)), np.uint64)
    for k, tau in enumerate(lags):
        for s in range(tau, S):
            for i in range(n):
                if bins[i] >= 0:
                    msd[k, bins[i]] += np.uint64(q(d2(xs[s][i], xs[s - tau][i])))
            for r in range(len(lo)):
                e = [(xs[s][hi[r]][c] - xs[s][lo[r]][c]) - (xs[s - tau][hi[r]][c] - xs[s - tau][lo[r]][c]) for c in range(3)]
                rel[k, r] += np.uint64(q((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2]))
    out = dict(msd_sum=msd, rel_msd_sum=rel, hist=np.zeros((2, 2, 64), np.uint64))
    for key in ("closed_runs", "closed_len", "open_runs", "open_len"):
        out[key] = np.zeros(len(lo), np.uint64)
    for key in ("hist_len", "left_runs", "left_len"):
        out[key] = np.zeros((2, 2), np.uint64)
    out.update(closed=np.zeros(len(lo), bool), length=np.zeros(len(lo), np.int64),
               from_transition=np.zeros(len(lo), bool))
    for r in range(len(lo)):
        states = [d2(x[lo[r]], x[hi[r]]) < rc * rc for x in xs]
        runs = []  # (state, length)
        for st in states:
            if runs and runs[-1][0] == st:
                runs[-1][1] += 1
            else:
                runs.append([st, 1])
        g = group[r]
        for j, (st, ln) in enumerate(runs[:-1]):
            k = 0 if st else 1
            if j == 0:
                out["left_runs"][g, k] += np.uint64(1)
                out["left_len"][g, k] += np.uint64(ln)
            else:
                out["closed_runs" if st else "open_runs"][r] += np.uint64(1)
                out["closed_len" if st else "open_len"][r] += np.uint64(ln)
                out["hist"][g, k, ln.bit_length() - 1] += np.uint64(1)
                out["hist_len"][g, k] += np.uint64(ln)
        if runs:
            out["closed"][r], out["length"][r], out["from_transition"][r] = runs[-1][0], runs[-1][1], len(runs) > 1
    return out


@pytest.mark.parametrize("n,s,lags,seed", [(40, 9, [1], 0), (60, 12, [1, 2, 4, 8], 1), (50, 15, [1, 3, 5, 11], 2),
                                           (30, 4, [2, 8, 64], 3)])
def test_restatement_equals_brute_force(n, s, lags, seed):
    xs = _walk(n, s, seed)
    rng = np.random.default_rng(seed)
    bins = rng.integers(-1, 7, size=n)
    lo, hi, grp = _rows(n, 25, seed)
    got = DR.dynamics(xs, lags, 0.3, bins, 7, lo, hi, grp)
    want = _brute(xs, lags, 0.3, bins, 7, lo, hi, grp)
    for k in DR.KEYS:
        assert np.array_equal(got[k], want[k]), k
    assert got["samples"] == s
    if s > 8:  # the walk does open and close loops
        assert got["hist"].sum() > 0 and got["left_runs"].sum() > 0


def test_run_lengths_and_transitions_are_conserved():
    n, s = 200, 40
    xs = _walk(n, s, 7)
    lo, hi, grp = _rows(n, 150, 8)
    d = DR.dynamics(xs, [1, 2, 4], 0.3, None, 0, lo, hi, grp)
    assert d["msd_sum"] is None
    for g in (0, 1):
        m = grp == g
        complete = d["closed_len"][m].sum() + d["open_len"][m].sum()
        assert complete + d["left_len"][g].sum() + d["length"][m].sum() == s * m.sum()
        states = np.array([[DR._pair_d2(x[lo], x[hi])[r] < 0.09 for x in xs] for r in np.flatnonzero(m)])
        transitions = int((states[:, 1:] != states[:, :-1]).sum())
        assert transitions == int(d["closed_runs"][m].sum() + d["open_runs"][m].sum() + d["left_runs"][g].sum())
        assert int(d["hist"][g].sum()) == int(d["closed_runs"][m].sum() + d["open_runs"][m].sum())
    assert d["hist"].sum() > 0


# ---- files -----------------------------------------------------------------------------------------------
def _member(seed, samples=6, n=4_000, lags=(1, 2, 4), sample_step=100, dt_ps=0.001, radius=0.3, down=1.0):
    lay = {}
    ms, ns, _, _, _ = loaders.import_mns_from_bedpe(BEDPE, N_beads=n, chrom=None, coords=None, path=None,
                                                    shuffle=False, seed=seed, down_prob=down, layout=lay)
    tab = loops.table(BEDPE)
    mr = loops.member_rows(tab, lay, n, ms, ns)
    gb = contacts.genome_bins(lay, 5_000_000, n_beads=n, max_bins=dynamics.MAX_BINS)
    rows = loops.device_rows(mr)
    xs = _walk(n, samples, seed, step=0.1)
    read = DR.dynamics(xs, lags, radius, gb.bins, gb.n_bins, rows["bead_lo"], rows["bead_hi"], rows["group"])
    return dynamics.result(read, lags, gb, tab, mr, radius, sample_step, dt_ps), read, mr, gb


def test_result_folds_the_runs_in_progress_and_stores_the_denominators():
    d, read, mr, gb = _member(0)
    v = mr["valid"]
    s = 6
    assert int(d["samples"]) == s and int(d["members"]) == 1 and v.sum() > 0
    beads = np.bincount(gb.bins[gb.bins >= 0], minlength=gb.n_bins)
    assert np.array_equal(d["msd_pairs"], np.outer(s - np.array([1, 2, 4]), beads).astype(np.uint64))
    assert np.array_equal(d["rel_pairs"][:, v], np.repeat((s - np.array([1, 2, 4]))[:, None], v.sum(), 1))
    assert not d["rel_pairs"][:, ~v].any() and not d["measured"][~v].any() and (d["measured"][v] == s).all()
    # every valid row has exactly one run in progress: right-censored or whole-window, by its state
    per_row = d["right_runs"].sum(0) + d["whole_runs"].sum(0)
    assert np.array_equal(per_row, v.astype(np.uint64))
    total = (d["closed_len"] + d["open_len"] + d["right_len"].sum(0) + d["whole_len"].sum(0))[v]
    left = read["left_len"].sum()
    assert int(total.sum() + left) == s * int(v.sum())
    for key, g in (("group_right_runs", "right_runs"), ("group_whole_len", "whole_len")):
        assert int(d[key].sum()) == int(d[g].sum())


def test_file_round_trip(tmp_path):
    d, *_ = _member(1)
    p = str(tmp_path / "dynamics" / "m.npz")
    dynamics.save(p, d)
    got = dynamics.load(p)
    assert set(got) == set(dynamics.KEYS)
    for k in dynamics.KEYS:
        assert np.array_equal(got[k], d[k]) and got[k].dtype == np.asarray(d[k]).dtype, k
    np.savez(str(tmp_path / "other.npz"), a=np.zeros(1))
    with pytest.raises(ValueError, match="not a dynamics file"):
        dynamics.load(str(tmp_path / "other.npz"))


def test_aggregate_exact_and_order_independent(tmp_path):
    parts = [_member(seed, down=0.6)[0] for seed in range(3)]
    paths = []
    for i, d in enumerate(parts):
        paths.append(str(tmp_path / f"m{i}.npz"))
        dynamics.save(paths[-1], d)
    a, b = dynamics.aggregate(paths), dynamics.aggregate(paths[::-1])
    for k in dynamics.KEYS:
        assert np.array_equal(a[k], b[k]), k
    for k in dynamics.SUMS:
        assert a[k].dtype == np.uint64 and np.array_equal(a[k], sum(p[k] for p in parts)), k
    assert int(a["members"]) == 3 and int(a["samples"]) == 18
    with pytest.raises(ValueError, match="no dynamics files"):
        dynamics.aggregate([])


@pytest.mark.parametrize("kw", [dict(lags=(1, 2, 8)), dict(sample_step=50), dict(dt_ps=0.002), dict(radius=0.25)])
def test_aggregate_refuses_mismatches(tmp_path, kw):
    a, b = _member(0)[0], _member(1, **kw)[0]
    dynamics.save(str(tmp_path / "a.npz"), a)
    dynamics.save(str(tmp_path / "b.npz"), b)
    with pytest.raises(ValueError, match="differs from the other members"):
        dynamics.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])


@pytest.mark.parametrize("key", ["bin_start_bp", "resolution_bp", "start1", "chrom2", "quantum_log2"])
def test_aggregate_refuses_a_different_bin_or_loop_table(tmp_path, key):
    a = _member(0)[0]
    b = dict(a)
    b[key] = np.asarray(a[key]) + (1 if a[key].dtype.kind in "iu" else "x")
    dynamics.save(str(tmp_path / "a.npz"), a)
    dynamics.save(str(tmp_path / "b.npz"), b)
    with pytest.raises(ValueError, match=f"{key} differs"):
        dynamics.aggregate([str(tmp_path / "a.npz"), str(tmp_path / "b.npz")])


# ---- readers ---------------------------------------------------------------------------------------------
def test_readers_on_hand_built_sums():
    q = 2.0**24
    d = dict(quantum_log2=np.int64(-24), lags=np.array([1, 2, 4]), sample_step=np.int64(200), dt_ps=np.float64(0.01),
             msd_sum=np.array([[3 * q, 0], [8 * q, 0], [12 * q, 0]], np.uint64),
             msd_pairs=np.array([[3, 0], [2, 0], [1, 0]], np.uint64),
             rel_msd_sum=np.array([[2 * q], [4 * q], [8 * q]], np.uint64), rel_pairs=np.array([[2], [2], [2]], np.uint64),
             rel_group_sum=np.array([[2 * q, 4 * q, 8 * q], [0, 0, 0]], np.uint64),
             rel_group_pairs=np.array([[2, 2, 2], [0, 0, 0]], np.uint64),
             hist=np.zeros((2, 2, 64), np.uint64), hist_len=np.array([[12, 0], [3, 5]], np.uint64),
             left_runs=np.array([[1, 0], [0, 2]], np.uint64), group_right_runs=np.array([[0, 1], [1, 0]], np.uint64),
             group_whole_runs=np.array([[0, 0], [4, 0]], np.uint64))
    d["hist"][0, 0, 1], d["hist"][0, 0, 2] = 2, 1  # 3 complete closed runs, 12 samples in all
    d["hist"][1, 0, 1], d["hist"][1, 1, 2] = 1, 1
    m = dynamics.msd(d)
    assert np.array_equal(m[:, 0], [1.0, 4.0, 12.0]) and np.isnan(m[:, 1]).all()
    per_row, per_group = dynamics.relative_msd(d)
    assert np.array_equal(per_row[:, 0], [1.0, 2.0, 4.0]) and np.array_equal(per_group[0], [1.0, 2.0, 4.0])
    assert np.isnan(per_group[1]).all()
    ex = dynamics.exponent(d["lags"], m)
    assert ex.shape == (2, 2) and np.allclose(ex[:, 0], [2.0, math.log(3) / math.log(2)]) and np.isnan(ex[:, 1]).all()
    assert np.allclose(dynamics.exponent(d["lags"], per_row)[:, 0], 1.0)
    lt = dynamics.lifetimes(d)
    step_ps = 200 * 0.01  # a run of one sample lasts MD_SAMPLE_STEP x SIM_INTEGRATOR_STEP
    assert np.allclose(lt["mean_ps"][0, 0], 4.0 * step_ps) and np.isnan(lt["mean_ps"][0, 1])
    assert np.allclose(lt["mean_ps"][1], [3.0 * step_ps, 5.0 * step_ps])
    assert np.array_equal(lt["complete"], [[3, 0], [1, 1]]) and np.array_equal(lt["left"], d["left_runs"])
    assert np.array_equal(lt["right"], d["group_right_runs"]) and np.array_equal(lt["whole"], d["group_whole_runs"])


def test_lag_set():
    assert dynamics.lag_set(1).tolist() == [1] and dynamics.lag_set(64).tolist() == [1, 2, 4, 8, 16, 32, 64]
    assert dynamics.lag_set(4096)[-1] == 4096 and dynamics.lag_set(8).dtype == np.int32
    for bad in (0, 3, 48, 8192, -2):
        with pytest.raises(ValueError, match="DYNAMICS_MAX_LAG"):
            dynamics.lag_set(bad)


# ---- settings --------------------------------------------------------------------------------------------
def _cfg(tmp_path, **kw):
    from multimm_b200.config import SimulationConfig

    base = dict(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    base.update(kw)
    return SimulationConfig(**base)


MD = dict(SIM_RUN_MD=True, SIM_N_STEPS=1000, SIM_SAMPLING_STEP=100, MD_SAMPLE_STEP=200)


def test_settings_are_extras_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import DYNAMICS_FIELDS, EXTRA_FIELDS, SimulationConfig, contact_setting

    assert set(DYNAMICS_FIELDS) == {"SAVE_DYNAMICS", "DYNAMICS_RESOLUTION", "DYNAMICS_MAX_LAG"}
    assert set(DYNAMICS_FIELDS) <= set(EXTRA_FIELDS) and not set(DYNAMICS_FIELDS) & set(SimulationConfig.model_fields)
    plain = _cfg(tmp_path)
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert contact_setting(plain, "SAVE_DYNAMICS") is False and contact_setting(plain, "DYNAMICS_RESOLUTION") == 0
    assert contact_setting(plain, "DYNAMICS_MAX_LAG") == 64
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\nSAVE_DYNAMICS = True\n")
    args, _ = run.get_config(["-c", str(ini), "--dynamics_resolution", "5000", "--dynamics_max_lag", "16"])
    assert contact_setting(args, "SAVE_DYNAMICS") is True and contact_setting(args, "DYNAMICS_RESOLUTION") == 5000
    assert contact_setting(args, "DYNAMICS_MAX_LAG") == 16


def _dumps(tmp_path, name):
    """(config_auto.ini, parameters.txt) bytes of a config without the dynamics settings."""
    import types

    from multimm_b200 import run
    from multimm_b200.model import MultiMM

    ini = tmp_path / f"{name}.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / name}\nSAVE_LOOPS = true\n")
    args, _ = run.get_config(["-c", str(ini)])
    params = tmp_path / f"{name}_parameters.txt"
    MultiMM.save_args_to_txt(types.SimpleNamespace(args=args), str(params))
    auto = (tmp_path / name / "metadata" / "config_auto.ini").read_bytes()
    return auto.replace(str(tmp_path / name).encode(), b"OUT"), params.read_bytes().replace(str(tmp_path / name).encode(), b"OUT")


def test_dumps_without_the_settings_are_unchanged(tmp_path, monkeypatch):
    from multimm_b200 import config

    with_fields = _dumps(tmp_path, "a")
    for word in (b"save_dynamics", b"dynamics_resolution", b"dynamics_max_lag"):
        assert word not in with_fields[0].lower() + with_fields[1].lower()
    for k in config.DYNAMICS_FIELDS:
        monkeypatch.delitem(config.EXTRA_FIELDS, k)
    assert _dumps(tmp_path, "b") == with_fields


@pytest.mark.parametrize("fields,match", [
    (dict(MD_SAMPLE_STEP=None), "SAVE_DYNAMICS"),
    (dict(SIM_RUN_MD=False, MD_SAMPLE_STEP=None), "SAVE_DYNAMICS"),
    (dict(MD_SAMPLE_STEP=600), "at least two MD samples"),
    (dict(MD_SAMPLE_STEP=1000), "at least two MD samples"),
    (dict(DYNAMICS_MAX_LAG=0), "DYNAMICS_MAX_LAG"),
    (dict(DYNAMICS_MAX_LAG=24), "DYNAMICS_MAX_LAG"),
    (dict(DYNAMICS_MAX_LAG=8192), "DYNAMICS_MAX_LAG"),
    (dict(DYNAMICS_RESOLUTION=-1), "DYNAMICS_RESOLUTION"),
    (dict(DYNAMICS_RESOLUTION=500), "DYNAMICS_RESOLUTION"),  # 6.2e6 bins genome-wide
    (dict(DYNAMICS_RESOLUTION=10, CHROM="chr1", LOC_START=0, LOC_END=50_000_000), "DYNAMICS_RESOLUTION"),
])
def test_bad_dynamics_fields_refused_before_any_output(tmp_path, fields, match):
    from multimm_b200 import run

    kw = dict(MD, SAVE_DYNAMICS=True)
    kw.update(fields)
    with pytest.raises(ValueError, match=match):
        run.args_tests(_cfg(tmp_path, **{k: v for k, v in kw.items() if v is not None}))
    assert not (tmp_path / "o").exists()


def test_dynamics_fields_valid_values(tmp_path):
    from multimm_b200 import run

    for res, lag in ((0, 64), (1_000, 1), (5_000, 4096)):  # 1 kb: about 3.1e6 bins genome-wide
        run.args_tests(_cfg(tmp_path, SAVE_DYNAMICS=True, DYNAMICS_RESOLUTION=res, DYNAMICS_MAX_LAG=lag, **MD))
    run.args_tests(_cfg(tmp_path, **dict(MD, MD_SAMPLE_STEP=500), SAVE_DYNAMICS=True))  # exactly two samples
    run.args_tests(_cfg(tmp_path, DYNAMICS_MAX_LAG=32))  # off: no MD needed
    assert not (tmp_path / "o").exists()


def test_md_sampling_accepts_the_dynamics_alone(tmp_path):
    from multimm_b200 import run

    run.args_tests(_cfg(tmp_path, SAVE_DYNAMICS=True, **MD))
    with pytest.raises(ValueError, match="SAVE_CONTACTS or SAVE_DISTANCES"):
        run.args_tests(_cfg(tmp_path, **MD))
