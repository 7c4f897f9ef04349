"""Distance distributions on the device (mmm_disthist_configure / mmm_disthist_add / mmm_disthist_read): the counts
equal the numpy restatement (tests/disthist_ref.py) exactly for several N (not all multiples of 32), canonical,
holed and scattered bin tables, 1, 19 and 63 edges, and edges that real pairs hit exactly; at canonical bins they sum
to the distance map's pair counts and their cumulative counts equal the contact map at every edge (up to N = 2e5);
K adds equal the sum of K single reads; refusals change nothing; no side effects on evaluations, MD or the other
readouts; buffers freed with the handle; the SAVE_DISTANCE_HIST driver against a reproduction through Engine calls,
its other outputs unchanged, and an ensemble's sums.

The cumulative overflow guard (the running total of one add's bound, the pairs of the fullest bin pair, must stay
below 2^63) cannot be reached in a test: it takes more than 2^63 / (N^2 / 2) adds, 2.3e8 at N = 2e5."""
import os

import numpy as np
import pytest

import disthist_ref as HR
from common import make_case, to_engine
from test_gpu_contacts_fine import BEDPE
from test_gpu_md_sampling import _files
from triplets_ref import globule

pytestmark = pytest.mark.gpu

MMM_ERR_ARG, MMM_ERR_STATE = -1, -3  # include/multimm_b200.h
DEFAULT = [0.1, 0.15, 0.2, 0.3, 0.5, 0.7, 1, 1.5, 2, 3, 5, 7, 10, 15, 20, 30, 50, 70, 100]
EDGE_SETS = {"default": DEFAULT, "one": [0.3], "63": list(np.geomspace(0.02, 8.0, 63))}


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


def _hist(eng, bins, nb, edges, xs):
    eng.disthist_configure(bins, nb, edges)
    for x in xs:
        eng.set_positions(x)
        eng.disthist_add()
    return eng.disthist_read()


CASES = [(50, "canonical", "default"), (50, "scattered", "63"), (1000, "holes", "one"), (1000, "scattered", "default"),
         (4133, "canonical", "63"), (4133, "holes", "default"), (4133, "scattered", "one"),
         (20_000, "canonical", "default"), (20_000, "holes", "63")]


@pytest.mark.parametrize("n,kind,edges", CASES)
def test_counts_equal_reference(built_lib, n, kind, edges):
    from multimm_b200.engine import Engine

    x = globule(n, 680, n)
    bins, nb = _table(kind, n, n)
    e = EDGE_SETS[edges]
    with Engine(n) as eng:
        r = _hist(eng, bins, nb, e, [x])
    want = HR.hist_counts(x, bins, nb, e)
    assert r["samples"] == 1 and r["counts"].dtype == np.uint64 and r["counts"].shape == want.shape
    assert np.array_equal(r["counts"], want)
    assert int(want.sum()) > 0 and r["device_ms"] > 0.0


def test_pairs_exactly_on_the_edges(built_lib):
    """Lattice pairs at exactly 0.5, 1, 1.5, 2 nm, and edges taken from real pairs of a globule whose squares give
    back the pair's d2: both belong to the upper cell."""
    from multimm_b200.engine import Engine

    n = 3001
    side = 15
    g = np.stack(np.meshgrid(*(np.arange(side),) * 3, indexing="ij"), -1).reshape(-1, 3)
    x = 0.5 * g[np.random.default_rng(1).permutation(len(g))[:n]].astype(np.float64)
    bins = (np.arange(n) * 40 // n).astype(np.int32)
    with Engine(n) as eng:
        got = _hist(eng, bins, 40, [0.5, 1.0, 1.5, 2.0], [x])["counts"]
    assert np.array_equal(got, HR.hist_counts(x, bins, 40, [0.5, 1.0, 1.5, 2.0]))
    y = globule(2000, 680, 2)
    i, j = np.triu_indices(2000, 1)
    pick = np.random.default_rng(3).choice(len(i), 4000, replace=False)
    d = y[i[pick]] - y[j[pick]]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    e = np.sqrt(d2)
    hit = np.unique(e[(e * e == d2) & (e < 1.5)])[:: 64][:63]
    assert len(hit) >= 20
    b = (np.arange(2000) * 10 // 2000).astype(np.int32)
    with Engine(2000) as eng:
        got = _hist(eng, b, 10, hit, [y])["counts"]
    assert np.array_equal(got, HR.hist_counts(y, b, 10, hit))


@pytest.mark.parametrize("n", [20_000, 200_000])
def test_canonical_counts_sum_to_pair_counts_and_contact_maps(built_lib, n):
    from multimm_b200 import contacts, distances
    from multimm_b200.engine import Engine

    x = globule(n, 680, 5)
    bins, nb = _table("canonical", n)
    nb = min(nb, 1000)
    iu = np.triu_indices(nb)
    with Engine(n) as eng:
        r = _hist(eng, bins, nb, DEFAULT, [x])
        gb = contacts.GenomeBins(bins, np.zeros(nb, np.int32), np.arange(nb, dtype=np.int64), 1)
        pairs, _ = distances._counts(gb)
        assert np.array_equal(r["counts"].sum(axis=1, dtype=np.uint64), pairs[iu])
        cum = np.cumsum(r["counts"], axis=1, dtype=np.uint64)
        for k, e in enumerate(DEFAULT):
            if e > 2:
                break
            cmap, _, _ = eng.contacts(float(e), bins, nb, want_sep=False)
            assert np.array_equal(cum[:, k], cmap[iu]), e


def test_k_adds_equal_the_sum_of_single_reads_and_configure_clears(built_lib):
    from multimm_b200.engine import Engine

    n = 3000
    xs = [globule(n, 680, s) for s in range(4)]
    bins, nb = _table("holes", n)
    with Engine(n) as eng:
        singles = [_hist(eng, bins, nb, DEFAULT, [x])["counts"] for x in xs]
        r = _hist(eng, bins, nb, DEFAULT, xs)
        assert r["samples"] == 4 and np.array_equal(r["counts"], sum(singles))
        again = eng.disthist_read()  # a read changes nothing
        assert np.array_equal(again["counts"], r["counts"]) and again["samples"] == 4
        eng.disthist_configure(bins, nb, DEFAULT)
        z = eng.disthist_read()
        assert z["samples"] == 0 and not z["counts"].any()


def test_refusals_leave_the_state_unchanged(built_lib):
    from multimm_b200._lib import Error
    from multimm_b200.engine import Engine

    n = 100
    bins = np.zeros(n, np.int32)
    with Engine(n) as eng:
        for call in (eng.disthist_add, eng.disthist_read):
            with pytest.raises(Error) as ei:
                call()
            assert ei.value.code == MMM_ERR_STATE
        eng.disthist_configure(bins, 1, [0.3])  # configuring needs no positions; adding does
        with pytest.raises(Error) as ei:
            eng.disthist_add()
        assert ei.value.code == MMM_ERR_STATE
        x = globule(n, 680, 1)
        eng.set_positions(x)
        bad = [dict(n_bins=0), dict(bin_of_bead=None), dict(bin_of_bead=np.full(n, -2, np.int32)),
               dict(bin_of_bead=np.full(n, 1, np.int32)), dict(edges_nm=None), dict(edges_nm=[]),
               dict(edges_nm=list(np.linspace(0.1, 7.0, 64))), dict(edges_nm=[0.2, 0.1]), dict(edges_nm=[0.2, 0.2]),
               dict(edges_nm=[0.0, 0.2]), dict(edges_nm=[-0.2]), dict(edges_nm=[0.1, np.inf]),
               dict(edges_nm=[np.nan]), dict(edges_nm=[1e200]), dict(edges_nm=[1e-170]),
               dict(n_bins=5000, bin_of_bead=np.zeros(n, np.int32), edges_nm=DEFAULT)]  # 2.5e8 counters > 2^27
        for kw in bad:
            args = dict(bin_of_bead=bins, n_bins=1, edges_nm=[0.3])
            args.update(kw)
            with pytest.raises(ValueError):
                eng.disthist_configure(**args)
            with pytest.raises(Error) as ei:  # a refused configuration leaves the accumulator unconfigured
                eng.disthist_add()
            assert ei.value.code == MMM_ERR_STATE
        with pytest.raises(ValueError):
            eng.disthist_configure(bins[:-1], 1, [0.3])
        # the largest table: 3663 bins with the 19 default edges, 1.34e8 counters
        eng.disthist_configure(np.arange(n, dtype=np.int32) % 3663, 3663, DEFAULT)
        eng.disthist_add()
        assert eng.disthist_read()["counts"].sum() == n * (n - 1) // 2
        # non-finite positions never reach the counts (set_positions refuses them and leaves the handle without
        # positions; the add checks them again): the counts and samples stay as they were
        eng.disthist_configure(bins, 1, DEFAULT)
        eng.disthist_add()
        before = eng.disthist_read()
        for bad_x in (np.nan, np.inf):
            y = x.copy()
            y[17, 1] = bad_x
            with pytest.raises(Error, match="non-finite"):
                eng.set_positions(y)
            with pytest.raises(Error) as ei:
                eng.disthist_add()
            assert ei.value.code == MMM_ERR_STATE
            eng.set_positions(x)
            after = eng.disthist_read()
            assert after["samples"] == before["samples"] == 1 and np.array_equal(after["counts"], before["counts"])
        eng.disthist_add()  # still configured: the refusals changed nothing
        r = eng.disthist_read()
        assert r["samples"] == 2 and np.array_equal(r["counts"], 2 * before["counts"])


def test_add_leaves_evaluations_md_and_other_readouts_unchanged(built_lib):
    n = 3000
    case = make_case(n, n_chrom=2, seed=3)
    bins = (np.arange(n) * 100 // n).astype(np.int32)
    eng = to_engine(case)
    e0, f0 = eng.energy_forces()
    last0 = eng.last_result()
    eng.disthist_configure(bins, 100, DEFAULT)
    eng.disthist_add()
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
        if added:
            eng.disthist_configure(bins, 100, DEFAULT)
        reps = []
        for _ in range(6):
            reps.append(eng.md_run(5, want_report=True))
            eng.sample()
            eng.triplets_add()
            if added:
                eng.disthist_add()
        s, t = eng.sampler_read(), eng.triplets_read()
        out.append((reps, eng.get_positions(), eng.get_velocities(), eng.energy_forces(), s, t))
        if added:
            assert eng.disthist_read()["samples"] == 6
        eng.close()
    (r0, x0, v0, ef0, s0, t0), (r1, x1, v1, ef1, s1, t1) = out
    assert r0 == r1
    assert np.array_equal(x0, x1) and np.array_equal(v0, v1)
    assert np.array_equal(ef0[0], ef1[0]) and np.array_equal(ef0[1], ef1[1])
    for k in ("counts", "sep", "rows", "cols", "vals", "dist_sum", "dist2_sum"):
        assert np.array_equal(s0[k], s1[k]), k
    for k in ("p", "q", "r", "vals"):
        assert np.array_equal(t0[k], t1[k]), k
    assert s0["samples"] == s1["samples"] == 6 and t0["triples"] == t1["triples"]


def test_distance_histogram_sums_helper(built_lib):
    from multimm_b200 import disthist

    x = globule(777, 680, 9)
    bins, nb = _table("scattered", 777, 9)
    assert np.array_equal(disthist.distance_histogram_sums(x, bins, nb, DEFAULT), HR.hist_counts(x, bins, nb, DEFAULT))


# ---- driver -------------------------------------------------------------------------------------------
def _ini(path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=1500, LOOPS_PATH=BEDPE, OUT_PATH=str(path / "out"), SAVE_PLOTS=False,
                CHROM="chr1", LOC_START=10_000_000, LOC_END=60_000_000, MIN_MAX_ITERATIONS=150, SIM_RUN_MD=True,
                SIM_N_STEPS=650, SIM_SAMPLING_STEP=100, TRJ_FRAMES=4, DOWNSAMPLING_PROB=0.5, SAVE_DISTANCE_HIST=True,
                DISTANCE_HIST_RESOLUTION=100_000, DISTANCE_HIST_EDGES="0.1,0.2,0.3,0.5,1")
    base.update(fields)
    path.mkdir(parents=True, exist_ok=True)
    ini = path / "config.ini"
    ini.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items() if v is not None))
    return str(ini), base["OUT_PATH"]


def test_driver_files_equal_reproduction(built_lib, tmp_path):
    from multimm_b200 import contacts, disthist, loaders, run
    from multimm_b200.model import MultiMM, _f

    step = 150
    edges = [0.1, 0.2, 0.3, 0.5, 1.0]
    ini, out = _ini(tmp_path / "s", MD_SAMPLE_STEP=step)
    assert run.main(["-c", ini]) == 0
    ini0, out0 = _ini(tmp_path / "p", SAVE_DISTANCE_HIST=None, DISTANCE_HIST_RESOLUTION=None, DISTANCE_HIST_EDGES=None)
    assert run.main(["-c", ini0]) == 0
    got, plain = _files(out), _files(out0)
    assert set(got) - set(plain) == {"analysis/distance_hist.npz", "analysis/distance_hist_md.npz"}
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
    gb = contacts.genome_bins(m.layout, 100_000, n_beads=1500, max_bins=disthist.max_bins(len(edges)))
    assert gb.n_bins == 500
    e.disthist_configure(gb.bins, gb.n_bins, edges)
    e.disthist_add()
    one = disthist.result(e.disthist_read()["counts"], edges, gb)
    e.md_configure(str(a.SIM_INTEGRATOR_TYPE).lower(), _f(a.SIM_INTEGRATOR_STEP), _f(a.SIM_TEMPERATURE),
                   float(a.SIM_FRICTION_COEFF), loaders.BEAD_MASS, int(a.SHUFFLING_SEED), amd_alpha=_f(a.SIM_AMD_ALPHA),
                   amd_e=_f(a.SIM_AMD_E))
    e.set_velocities_to_temperature(_f(a.SIM_TEMPERATURE), int(a.SHUFFLING_SEED))
    e.disthist_configure(gb.bins, gb.n_bins, edges)
    done = 0
    while done < 600:
        e.md_run(50, want_report=False)
        done += 50
        if done % step == 0:
            e.disthist_add()
    md = disthist.result(e.disthist_read()["counts"], edges, gb, 600 // step)
    m.close()
    assert int(one["counts"].sum()) == 1500 * 1499 // 2
    for name, want in (("distance_hist.npz", one), ("distance_hist_md.npz", md)):
        d = disthist.load(os.path.join(out, "analysis", name))
        for k in disthist.KEYS:
            assert np.array_equal(d[k], want[k]) and d[k].dtype == np.asarray(want[k]).dtype, (name, k)
    assert int(disthist.load(os.path.join(out, "analysis", "distance_hist_md.npz"))["members"]) == 4


def test_ensemble_distance_hist_is_the_sum_of_the_members(built_lib, tmp_path):
    from multimm_b200 import disthist, run

    ini, out = _ini(tmp_path, N_BEADS=1000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=2, MD_SAMPLE_STEP=200,
                    SIM_N_STEPS=400, MIN_MAX_ITERATIONS=80)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=[0])
    for name in (lambda p: p, lambda p: p[:-4] + "_md.npz"):
        paths = [name(run.member_distance_hist_path(out, i)) for i in range(2)]
        parts = [disthist.load(p) for p in paths]
        got = disthist.load(name(os.path.join(out, "ensemble_distance_hist.npz")))
        for k in disthist.KEYS:
            assert np.array_equal(got[k], disthist.aggregate(paths)[k]), k
        assert np.array_equal(got["counts"], parts[0]["counts"] + parts[1]["counts"])
        assert int(got["members"]) == sum(int(p["members"]) for p in parts)
        assert int(got["counts"].sum()) > 0


MEMORY_CHILD = r"""
import json, os, subprocess, sys
import numpy as np
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from triplets_ref import globule
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
    for nb, ne in ((1000, 19), (1500, 63), (500, 1)):
        eng.disthist_configure((np.arange(n) * nb // n).astype(np.int32), nb, np.geomspace(0.05, 50.0, ne))
        eng.disthist_add()
        eng.disthist_read()
    eng.close()
    used.append(used_mib())
print(json.dumps(used))
"""


def test_disthist_buffers_freed_with_the_handle(built_lib):
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
