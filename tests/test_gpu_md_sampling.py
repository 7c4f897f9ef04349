"""The trajectory sampler on the device (mmm_sampler_configure / mmm_sample / mmm_sampler_read[_fine]): its sums
equal, exactly, the sums of the one-shot calls (mmm_contacts, mmm_contacts_sparse, mmm_distance_map) at the
same positions and the numpy restatements; the fine map's merge at its edges (every key colliding, disjoint
keys, nothing binned, growth); no side effects on MD, one-shot results or mmm_contacts_sparse_read; argument,
state and cumulative-overflow refusals; the MD_SAMPLE_STEP driver against a reproduction through Engine calls,
its other outputs unchanged, and an ensemble's *_md sums."""
import os

import numpy as np
import pytest

import contacts_ref as CR
import distances_ref as DR
from common import make_case, to_engine
from test_gpu_contacts_fine import BEDPE, _bin_sets, _engine, _globule

pytestmark = pytest.mark.gpu

MMM_ERR_ARG, MMM_ERR_STATE = -1, -3  # include/multimm_b200.h
RC = 0.2


def _structures(n, k, seed):
    """k structures of one globule moved a little each: keys partly shared, partly new."""
    x = _globule(n, seed=seed)
    rng = np.random.default_rng(seed + 1)
    return [x + rng.normal(scale=0.02, size=x.shape) * s for s in range(k)]


def _coarse(bins, nb, limit=4096):
    """bins usable by the dense maps (<= 4096): the set itself, or its ids folded."""
    if nb <= limit:
        return bins, nb
    return np.where(bins >= 0, bins % 997, -1).astype(np.int32), 997


def _one_shot_sums(eng, xs, cb, nc, fb, nf, db, nd):
    counts = np.zeros((nc, nc), np.uint64)
    sep = np.zeros(len(cb), np.uint64)
    dsum, d2sum = np.zeros((nd, nd), np.uint64), np.zeros((nd, nd), np.uint64)
    pairs, keys, vals = 0, [], []
    for x in xs:
        eng.set_positions(x)
        m, s, p = eng.contacts(RC, cb, nc)
        counts += m
        sep += s
        pairs += p
        r, c, v, _ = eng.contacts_sparse(RC, fb, nf)
        keys.append(r.astype(np.int64) * nf + c)
        vals.append(v)
        a, b = eng.distance_map(db, nd)
        dsum += a
        d2sum += b
    u, inv = np.unique(np.concatenate(keys), return_inverse=True)
    fv = np.zeros(len(u), np.uint64)
    np.add.at(fv, inv, np.concatenate(vals))
    return dict(counts=counts, sep=sep, pairs=pairs, rows=(u // nf).astype(np.int32), cols=(u % nf).astype(np.int32),
                vals=fv, dist_sum=dsum, dist2_sum=d2sum, samples=len(xs))


def _sampled(eng, xs, cb, nc, fb, nf, db, nd):
    eng.sampler_configure(RC, cb, nc, fb, nf, db, nd)
    for x in xs:
        eng.set_positions(x)
        eng.sample()
    return eng.sampler_read()


def _assert_same(got, want, keys=("counts", "sep", "pairs", "rows", "cols", "vals", "dist_sum", "dist2_sum", "samples")):
    for k in keys:
        g, w = got[k], want[k]
        if isinstance(w, np.ndarray):
            assert g.dtype == w.dtype and np.array_equal(g, w), k
        else:
            assert g == w, k


@pytest.mark.parametrize("n,k,left_out", [(33, 40, False), (1000 + 7, 7, True), (3000, 2, False), (3000, 40, True),
                                          (12_345, 1, True), (12_345, 7, False)])
def test_sums_equal_one_shot_calls_and_reference(built_lib, n, k, left_out):
    rng = np.random.default_rng(n + k)
    xs = _structures(n, k, seed=n)
    with _engine(xs[0]) as eng:
        for fb, nf in _bin_sets(n, rng):
            if left_out:
                fb = np.where(rng.random(n) < 0.1, -1, fb).astype(np.int32)
            cb, nc = _coarse(fb, nf)
            db, nd = _coarse(fb, nf, 300)
            got = _sampled(eng, xs, cb, nc, fb, nf, db, nd)
            want = _one_shot_sums(eng, xs, cb, nc, fb, nf, db, nd)
            _assert_same(got, want)
            assert got["device_ms"] > 0.0
            if n * n * k > 4e8:
                continue
            # the numpy restatements, summed over the structures
            ref_counts = sum(CR.contact_counts(x, RC, cb, nc)[0] for x in xs)
            ref_sep = sum(CR.contact_counts(x, RC)[1] for x in xs)
            assert np.array_equal(got["counts"], ref_counts) and np.array_equal(got["sep"], ref_sep)
            keys = []
            for x in xs:
                i, j = CR.contact_pairs(x, RC)
                bi, bj = fb.astype(np.int64)[i], fb.astype(np.int64)[j]
                ok = (bi >= 0) & (bj >= 0)
                keys.append(np.minimum(bi[ok], bj[ok]) * nf + np.maximum(bi[ok], bj[ok]))
            u, c = np.unique(np.concatenate(keys), return_counts=True)
            assert np.array_equal(got["rows"].astype(np.int64) * nf + got["cols"], u)
            assert np.array_equal(got["vals"], c.astype(np.uint64))
            if n <= 3000:
                ds = [DR.distance_sums(x, db, nd) for x in xs[:2]]
                one = _sampled(eng, xs[:2], cb, nc, fb, nf, db, nd)
                assert np.array_equal(one["dist_sum"], sum(d[0] for d in ds))
                assert np.array_equal(one["dist2_sum"], sum(d[1] for d in ds))


def _spread(n, spacing=1.0):
    """Beads on a line 1 nm apart: no contact at rc = 0.2 nm."""
    x = np.zeros((n, 3))
    x[:, 0] = np.arange(n) * spacing
    return x


def test_merge_edge_cases(built_lib):
    n = 2000
    x = _globule(n, seed=5)
    fb = np.arange(n, dtype=np.int32)
    cb = (np.arange(n) * 64 // n).astype(np.int32)
    half = n // 2
    a, b = x.copy(), x.copy()
    a[half:] = _spread(n - half) + 1000.0          # contacts among the first half only
    b[:half] = _spread(half) + 1000.0              # ... and the second half only: disjoint keys
    with _engine(x) as eng:
        one = _sampled(eng, [x], cb, 64, fb, n, None, 0)
        twice = _sampled(eng, [x, x], cb, 64, fb, n, None, 0)  # every key collides: counts double
        assert np.array_equal(twice["rows"], one["rows"]) and np.array_equal(twice["cols"], one["cols"])
        assert np.array_equal(twice["vals"], 2 * one["vals"]) and twice["pairs"] == 2 * one["pairs"]
        for xs in ([a, b], [b, a], [_spread(n)], [_spread(n), x, _spread(n)], [a, x, b, x]):
            _assert_same(_sampled(eng, xs, cb, 64, fb, n, None, 0),
                         _one_shot_sums(eng, xs, cb, 64, fb, n, cb, 64), keys=("counts", "rows", "cols", "vals", "pairs"))
        empty = _sampled(eng, [_spread(n)], cb, 64, fb, n, None, 0)
        assert empty["samples"] == 1 and len(empty["vals"]) == 0 and empty["pairs"] == 0
        # an accumulator that grows across samples: sparse first, dense later
        dense = _globule(n, seed=6, radius=0.6)
        xs = [_spread(n), a, x, dense, dense * 0.9]
        got = _sampled(eng, xs, cb, 64, fb, n, None, 0)
        _assert_same(got, _one_shot_sums(eng, xs, cb, 64, fb, n, cb, 64), keys=("counts", "rows", "cols", "vals", "pairs"))


@pytest.mark.parametrize("integrator", ["langevin", "brownian"])
def test_md_run_sampled_is_bit_identical(built_lib, integrator):
    case = make_case(3000, n_chrom=2, seed=3)
    bins = (np.arange(3000) * 50 // 3000).astype(np.int32)
    out = []
    for sampled in (False, True):
        eng = to_engine(case)
        eng.minimize(tol=10.0, max_iter=30)
        eng.md_configure(integrator, dt_ps=0.001, seed=7)
        eng.set_velocities_to_temperature(310.0, seed=8)
        if sampled:
            eng.sampler_configure(RC, bins, 50, np.arange(3000, dtype=np.int32), 3000, bins, 50)
        reps = []
        for _ in range(6):
            reps.append(eng.md_run(5, want_report=True))
            if sampled:
                eng.sample()
        out.append((reps, eng.get_positions(), eng.get_velocities(), eng.energy_forces()))
        if sampled:
            assert eng.sampler_read()["samples"] == 6
        eng.close()
    (r0, x0, v0, ef0), (r1, x1, v1, ef1) = out
    assert r0 == r1
    assert np.array_equal(x0, x1) and np.array_equal(v0, v1)
    assert np.array_equal(ef0[0], ef1[0]) and np.array_equal(ef0[1], ef1[1])


def test_one_shot_results_unchanged_and_reconfigure_clears(built_lib):
    n = 3000
    xs = _structures(n, 3, seed=9)
    fb = np.arange(n, dtype=np.int32)
    cb = (np.arange(n) * 100 // n).astype(np.int32)
    with _engine(xs[0]) as eng:
        want = eng.contacts_sparse(RC, fb, n)
        dense = eng.contacts(RC, cb, 100)
        dist = eng.distance_map(cb, 100)
        stats = eng.contacts_stats()
        eng.sampler_configure(RC, cb, 100, fb, n, cb, 100)
        for x in xs:
            eng.set_positions(x)
            eng.sample()
        lib = eng._lib
        import ctypes as C
        e = len(want[0])
        rows, cols, vals = np.empty(e, np.int32), np.empty(e, np.int32), np.empty(e, np.uint64)
        assert lib.mmm_contacts_sparse_read(eng._h, rows.ctypes.data_as(C.c_void_p), cols.ctypes.data_as(C.c_void_p),
                                            vals.ctypes.data_as(C.c_void_p)) == 0
        for g, w in zip((rows, cols, vals), want[:3]):
            assert np.array_equal(g, w)
        assert eng.contacts_stats()["candidates"] == stats["candidates"]
        eng.set_positions(xs[0])
        for g, w in zip(eng.contacts(RC, cb, 100), dense):
            assert np.array_equal(g, w) if isinstance(w, np.ndarray) else g == w
        for g, w in zip(eng.distance_map(cb, 100), dist):
            assert np.array_equal(g, w)
        eng.sampler_configure(RC, cb, 100, fb, n, cb, 100)
        r = eng.sampler_read()
        assert r["samples"] == 0 and r["pairs"] == 0 and len(r["vals"]) == 0 and r["device_ms"] == 0.0
        assert not r["counts"].any() and not r["sep"].any() and not r["dist_sum"].any() and not r["dist2_sum"].any()
        eng.sample()
        _assert_same(eng.sampler_read(), _one_shot_sums(eng, [xs[0]], cb, 100, fb, n, cb, 100))


def test_argument_and_state_errors(built_lib):
    from multimm_b200._lib import Error
    from multimm_b200.engine import Engine

    n = 100
    bins = np.zeros(n, np.int32)
    with Engine(n) as eng:
        for call in (eng.sample, eng.sampler_read):
            with pytest.raises(Error) as ei:
                call()
            assert ei.value.code == MMM_ERR_STATE
        eng.sampler_configure(RC, bins, 1)  # configuring needs no positions; sampling does
        with pytest.raises(Error) as ei:
            eng.sample()
        assert ei.value.code == MMM_ERR_STATE
        eng.set_positions(_globule(n))
        bad = [dict(), dict(rc_nm=0.0, contact_bins=bins, n_contact_bins=1),
               dict(rc_nm=float("nan"), contact_bins=bins, n_contact_bins=1),
               dict(contact_bins=bins, n_contact_bins=0), dict(contact_bins=bins, n_contact_bins=4097),
               dict(contact_bins=bins + 1, n_contact_bins=1), dict(contact_bins=bins - 2, n_contact_bins=1),
               dict(fine_bins=bins, n_fine_bins=1, distance_bins=bins, n_distance_bins=1),
               dict(contact_bins=bins, n_contact_bins=1, fine_bins=bins, n_fine_bins=0),
               dict(distance_bins=bins, n_distance_bins=4097), dict(distance_bins=bins + 5, n_distance_bins=5)]
        for kw in bad:
            with pytest.raises(ValueError):
                eng.sampler_configure(**kw)
            with pytest.raises(Error) as ei:  # a refused configuration leaves the sampler unconfigured
                eng.sample()
            assert ei.value.code == MMM_ERR_STATE
        with pytest.raises(ValueError):
            eng.sampler_configure(RC, bins[:-1], 1)
        eng.sampler_configure(RC, None, 0, None, 0, bins, 1)
        eng.sample()
        assert eng.sampler_read()["counts"] is None and eng.sampler_read()["samples"] == 1


def test_cumulative_distance_guard(built_lib):
    n = 33
    pmax = n * (n - 1) / 2
    D = np.sqrt(0.99 * 2.0**62 / pmax / 2.0**24)  # one structure's bound just under 2^62
    x = _spread(n, D / (n - 1))
    bins = np.zeros(n, np.int32)
    fb = np.arange(n, dtype=np.int32)
    with _engine(x) as eng:
        eng.distance_map(bins, 1)  # one structure alone passes
        eng.sampler_configure(RC, bins, 1, fb, n, bins, 1)
        eng.sample()
        eng.sample()
        before = eng.sampler_read()
        with pytest.raises(ValueError, match="overflow"):
            eng.sample()
        after = eng.sampler_read()
        _assert_same(after, before)
        assert after["samples"] == 2 and after["device_ms"] == before["device_ms"]
        ds = eng.distance_map(bins, 1)
        assert np.array_equal(after["dist_sum"], 2 * ds[0]) and np.array_equal(after["dist2_sum"], 2 * ds[1])


# ---- driver -------------------------------------------------------------------------------------------
def _ini(path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=1500, LOOPS_PATH=BEDPE, OUT_PATH=str(path / "out"), SAVE_PLOTS=False,
                CHROM="chr1", LOC_START=10_000_000, LOC_END=60_000_000, MIN_MAX_ITERATIONS=150, SIM_RUN_MD=True,
                SIM_N_STEPS=650, SIM_SAMPLING_STEP=100, TRJ_FRAMES=4, SAVE_CONTACTS=True,
                CONTACT_RESOLUTION=500_000, CONTACT_FINE_RESOLUTION=100_000, SAVE_DISTANCES=True,
                DISTANCE_RESOLUTION=1_000_000)
    base.update(fields)
    path.mkdir(parents=True, exist_ok=True)
    ini = path / "config.ini"
    ini.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items() if v is not None))
    return str(ini), base["OUT_PATH"]


def _files(out):
    res = {}
    for root, _, names in os.walk(out):
        for f in names:
            rel = os.path.relpath(os.path.join(root, f), out)
            if rel.endswith(".npz"):
                with np.load(os.path.join(root, f)) as z:
                    res[rel] = {k: z[k] for k in z.files}
            elif rel not in ("metadata/config_auto.ini", "metadata/parameters.txt") and not rel.endswith(".log"):
                with open(os.path.join(root, f), "rb") as fh:
                    res[rel] = fh.read()
    return res


def test_driver_md_files_equal_reproduction(built_lib, tmp_path):
    from multimm_b200 import contacts, distances, loaders, run
    from multimm_b200.config import contact_setting
    from multimm_b200.model import MultiMM, _f

    step = 150
    ini, out = _ini(tmp_path / "s", MD_SAMPLE_STEP=step)
    assert run.main(["-c", ini]) == 0
    ini0, out0 = _ini(tmp_path / "p", MD_SAMPLE_STEP=None)
    assert run.main(["-c", ini0]) == 0
    got, plain = _files(out), _files(out0)
    md = {k for k in got if k.endswith("_md.npz")}
    assert md == {"analysis/contacts_md.npz", "analysis/contacts_fine_md.npz", "analysis/distances_md.npz"}
    assert set(got) - md == set(plain)
    for k in plain:
        if isinstance(plain[k], dict):
            assert plain[k].keys() == got[k].keys() and all(np.array_equal(plain[k][a], got[k][a]) for a in plain[k]), k
        else:
            assert plain[k] == got[k], k

    # the reproduction: the same run through Engine calls, one-shot passes at the sampled steps, summed
    args, _ = run.get_config(["-c", ini0, "--out_path", str(tmp_path / "r")])
    m = MultiMM(args)
    m.prepare()
    m.min_energy(write_files=False)
    e, a = m.engine, args
    temp = _f(a.SIM_TEMPERATURE)
    e.md_configure(str(a.SIM_INTEGRATOR_TYPE).lower(), _f(a.SIM_INTEGRATOR_STEP), temp, float(a.SIM_FRICTION_COEFF),
                   loaders.BEAD_MASS, int(a.SHUFFLING_SEED), amd_alpha=_f(a.SIM_AMD_ALPHA), amd_e=_f(a.SIM_AMD_E))
    e.set_velocities_to_temperature(temp, int(a.SHUFFLING_SEED))
    gb, fb, db = m._contact_bins(), m._contact_bins(fine=True), m._distance_bins()
    rc = float(contact_setting(a, "CONTACT_RADIUS"))
    done, sums = 0, None
    while done < 600:
        e.md_run(50, want_report=False)
        done += 50
        if done % step:
            continue
        cm, sep, pairs = e.contacts(rc, gb.bins, gb.n_bins)
        r, c, v, _ = e.contacts_sparse(rc, fb.bins, fb.n_bins)
        ds, d2 = e.distance_map(db.bins, db.n_bins)
        rs, r2s = distances.radial_sums(e.get_positions(), m.mass_center, db.bins, db.n_bins)
        fine = contacts.fine_result(r, c, v, pairs, rc, fb)
        if sums is None:
            sums = [cm, sep, pairs, fine, ds, d2, rs, r2s]
        else:
            sums = [sums[0] + cm, sums[1] + sep, sums[2] + pairs,
                    dict(sums[3], **dict(zip(("rows", "cols", "vals"), contacts._merge(
                        sums[3]["rows"], sums[3]["cols"], sums[3]["vals"], r, c, v, fb.n_bins)))),
                    sums[4] + ds, sums[5] + d2, sums[6] + rs, sums[7] + r2s]
    m.close()
    S = 600 // step
    c = contacts.load(os.path.join(out, "analysis", "contacts_md.npz"))
    assert int(c["members"]) == S and int(c["pairs"]) == sums[2]
    assert np.array_equal(c["counts"], sums[0]) and np.array_equal(c["sep_contacts"], sums[1])
    assert np.array_equal(c["sep_pairs"], np.uint64(S) * contacts.sep_pairs(m.chrom_spin))
    f = contacts.load_fine(os.path.join(out, "analysis", "contacts_fine_md.npz"))
    assert int(f["members"]) == S
    for k in ("rows", "cols", "vals"):
        assert np.array_equal(f[k], sums[3][k]), k
    d = distances.load(os.path.join(out, "analysis", "distances_md.npz"))
    assert int(d["members"]) == S
    for k, w in (("dist_sum", sums[4]), ("dist2_sum", sums[5]), ("radial_sum", sums[6]), ("radial2_sum", sums[7])):
        assert np.array_equal(d[k], w), k
    one = distances.load(os.path.join(out, "analysis", "distances.npz"))
    assert np.array_equal(d["pair_count"], np.uint64(S) * one["pair_count"])


def test_ensemble_md_files_sum_the_members(built_lib, tmp_path):
    from multimm_b200 import contacts, distances, run

    ini, out = _ini(tmp_path, N_BEADS=1000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=2,
                    MD_SAMPLE_STEP=200, SIM_N_STEPS=400, MIN_MAX_ITERATIONS=80)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=[0])
    parts = [contacts.load(contacts.md_path(run.member_contacts_path(out, i))) for i in range(2)]
    agg = contacts.load(os.path.join(out, "ensemble_contacts_md.npz"))
    assert int(agg["members"]) == 4 and all(int(p["members"]) == 2 for p in parts)
    assert np.array_equal(agg["counts"], parts[0]["counts"] + parts[1]["counts"])
    fp = [contacts.load_fine(contacts.md_path(run.member_contacts_fine_path(out, i))) for i in range(2)]
    fa = contacts.load_fine(os.path.join(out, "ensemble_contacts_fine_md.npz"))
    want = contacts._merge(fp[0]["rows"], fp[0]["cols"], fp[0]["vals"], fp[1]["rows"], fp[1]["cols"], fp[1]["vals"],
                           int(fa["n_bins"]))
    for g, w in zip((fa["rows"], fa["cols"], fa["vals"]), want):
        assert np.array_equal(g, w)
    dp = [distances.load(contacts.md_path(run.member_distances_path(out, i))) for i in range(2)]
    da = distances.load(os.path.join(out, "ensemble_distances_md.npz"))
    for k in ("dist_sum", "dist2_sum", "pair_count", "bin_beads", "radial_sum"):
        assert np.array_equal(da[k], dp[0][k] + dp[1][k]), k


MEMORY_CHILD = r"""
import json, os, subprocess, sys
import numpy as np
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from test_gpu_contacts_fine import _globule
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
x = _globule(n, seed=1)
bins = (np.arange(n) * 4096 // n).astype(np.int32)
used = []
for cycle in range(3):
    eng = Engine(n)
    eng.set_positions(x)
    eng.sampler_configure(0.2, bins, 4096, np.arange(n, dtype=np.int32), n, bins, 4096)
    for s in range(4):
        eng.set_positions(x * (1.0 - 0.05 * s))  # denser each time: the fine map grows
        eng.sample()
    eng.sampler_read()
    eng.close()
    used.append(used_mib())
print(json.dumps(used))
"""


def test_sampler_buffers_freed_with_the_handle(built_lib):
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
