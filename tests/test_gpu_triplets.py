"""The three-way contact map on the device (mmm_triplets_configure / mmm_triplets_add / mmm_triplets_read[_entries]):
its entries and total equal the numpy restatement (tests/triplets_ref.py) exactly, for N from 50 to 2e5, two
radii and three kinds of bin table; any chunk cap gives the same bits; K adds equal the sum of K single reads and
configuring clears; every bead-level triple is a triangle of the device's own sparse contact map; no side effects
on evaluations, MD, the one-shot sparse map or the sampler; argument and state refusals; buffers freed with the
handle; the SAVE_TRIPLETS driver against a reproduction through Engine calls, its other outputs unchanged, and an
ensemble's sums."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

import contacts_ref as CR
import triplets_ref as TR
from common import make_case, to_engine
from test_gpu_contacts_fine import BEDPE, _engine
from test_gpu_md_sampling import _files

pytestmark = pytest.mark.gpu

MMM_ERR_ARG, MMM_ERR_STATE = -1, -3  # include/multimm_b200.h
ENTRY_KEYS = ("p", "q", "r", "vals")


def _tables(n, seed):
    """Identity bins, about 1000 contiguous bins (as genome_bins makes them), and the same with beads left out."""
    rng = np.random.default_rng(seed)
    canon = (np.arange(n, dtype=np.int64) * 1000 // n).astype(np.int32)
    holes = np.where(rng.random(n) < 0.1, -1, canon).astype(np.int32)
    return [("identity", np.arange(n, dtype=np.int32), n), ("canonical", canon, int(canon[-1]) + 1),
            ("holes", holes, int(canon[-1]) + 1)]


def _read(eng, rc, bins, nb, xs, cap=0):
    eng.triplets_configure(rc, bins, nb, cap)
    for x in xs:
        eng.set_positions(x)
        eng.triplets_add()
    return eng.triplets_read()


def _assert_same(got, want):
    for k in ENTRY_KEYS:
        assert got[k].dtype == np.asarray(want[k]).dtype and np.array_equal(got[k], want[k]), k
    assert got["triples"] == want["triples"]


@pytest.mark.parametrize("n,rc,density", [(50, 0.2, 680), (50, 0.3, 680), (1000, 0.2, 680), (1000, 0.3, 680),
                                          (20_000, 0.2, 680), (20_000, 0.3, 680), (200_000, 0.2, 680),
                                          (200_000, 0.3, 250)])
def test_entries_equal_reference(built_lib, n, rc, density):
    x = TR.globule(n, density, seed=n)
    tri = TR.triangles_from_pairs(n, *CR.contact_pairs(x, rc))
    with _engine(x) as eng:
        for name, bins, nb in _tables(n, seed=n + 1):
            got = _read(eng, rc, bins, nb, [x])
            p, q, r, vals = TR.binned(*tri, bins, nb)
            _assert_same(got, dict(p=p, q=q, r=r, vals=vals, triples=len(tri[0])))
            assert got["samples"] == 1 and got["triples"] > 0, name
            assert got["chunks"] == (1 if len(vals) else 0) and got["device_ms"] > 0.0, name
            if name == "holes":
                assert vals.sum() < len(tri[0])


def test_chunk_cap_gives_identical_bits(built_lib):
    n = 20_000
    x = TR.globule(n, 680, seed=3)
    with _engine(x) as eng:
        for _, bins, nb in _tables(n, seed=4):
            ref = _read(eng, 0.3, bins, nb, [x])
            assert ref["chunks"] == 1
            for cap in (1, 1000, 123_457):
                got = _read(eng, 0.3, bins, nb, [x], cap=cap)
                _assert_same(got, ref)
                assert got["chunks"] > 1
            one = _read(eng, 0.3, bins, nb, [x], cap=1)
            assert one["chunks"] == np.count_nonzero(np.diff(_bead_offsets(x, 0.3, bins)))  # one bead per chunk


def _bead_offsets(x, rc, bins):
    """Exclusive prefix of the binned triples per lowest bead i."""
    ti, tj, tk = TR.triangles_from_pairs(len(x), *CR.contact_pairs(x, rc))
    keep = (bins[ti] >= 0) & (bins[tj] >= 0) & (bins[tk] >= 0)
    return np.concatenate([[0], np.cumsum(np.bincount(ti[keep], minlength=len(x)))])


def test_k_adds_equal_the_sum_of_single_reads_and_configure_clears(built_lib):
    from multimm_b200 import triplets

    n = 5000
    xs = [TR.globule(n, 680, seed=s) for s in range(4)]
    bins, nb = _tables(n, seed=1)[2][1:]
    with _engine(xs[0]) as eng:
        singles = [_read(eng, 0.3, bins, nb, [x]) for x in xs]
        many = _read(eng, 0.3, bins, nb, xs, cap=5000)
        keys = np.concatenate([(s["p"].astype(np.int64) * nb + s["q"]) * nb + s["r"] for s in singles])
        p, q, r, vals = triplets._reduce(keys, np.concatenate([s["vals"] for s in singles]), nb)
        _assert_same(many, dict(p=p, q=q, r=r, vals=vals, triples=sum(s["triples"] for s in singles)))
        assert many["samples"] == 4 and many["chunks"] > 4
        eng.triplets_configure(0.3, bins, nb)
        r0 = eng.triplets_read()
        assert (r0["samples"], r0["triples"], r0["chunks"], r0["device_ms"], len(r0["vals"])) == (0, 0, 0, 0.0, 0)


def test_bead_triples_are_triangles_of_the_sparse_contact_map(built_lib):
    n = 3000
    x = TR.globule(n, 680, seed=9)
    ident = np.arange(n, dtype=np.int32)
    with _engine(x) as eng:
        got = _read(eng, 0.3, ident, n, [x])
        rows, cols, vals, pairs = eng.contacts_sparse(0.3, ident, n)
    assert np.all(vals == 1) and got["triples"] == int(got["vals"].sum()) and np.all(got["vals"] == 1)
    keys = rows.astype(np.int64) * n + cols
    p, q, r = (got[k].astype(np.int64) for k in ("p", "q", "r"))
    assert np.all((p < q) & (q < r))
    for a, b in ((p, q), (p, r), (q, r)):
        assert np.isin(a * n + b, keys).all()
    a = sp.csr_matrix((np.ones(len(rows), np.int64), (rows, cols)), shape=(n, n))
    a = a + a.T
    assert got["triples"] == int((a @ a).multiply(a).sum()) // 6 > n


def test_add_leaves_evaluations_md_sparse_map_and_sampler_unchanged(built_lib):
    import ctypes as C

    n = 3000
    case = make_case(n, n_chrom=2, seed=3)
    bins = (np.arange(n) * 100 // n).astype(np.int32)
    eng = to_engine(case)
    e0, f0 = eng.energy_forces()
    last0 = eng.last_result()
    sparse0 = eng.contacts_sparse(0.3, bins, 100)
    eng.triplets_configure(0.3, bins, 100, 700)
    eng.triplets_add()
    e = len(sparse0[0])
    rows, cols, vals = np.empty(e, np.int32), np.empty(e, np.int32), np.empty(e, np.uint64)
    eng._ck(eng._lib.mmm_contacts_sparse_read(eng._h, rows.ctypes.data_as(C.c_void_p), cols.ctypes.data_as(C.c_void_p),
                                              vals.ctypes.data_as(C.c_void_p)))
    assert all(np.array_equal(a, b) for a, b in zip((rows, cols, vals), sparse0[:3]))
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
        if added:
            eng.triplets_configure(0.3, bins, 100)
        reps = []
        for _ in range(6):
            reps.append(eng.md_run(5, want_report=True))
            eng.sample()
            if added:
                eng.triplets_add()
        s = eng.sampler_read()
        out.append((reps, eng.get_positions(), eng.get_velocities(), eng.energy_forces(), s))
        if added:
            assert eng.triplets_read()["samples"] == 6
        eng.close()
    (r0, x0, v0, ef0, s0), (r1, x1, v1, ef1, s1) = out
    assert r0 == r1
    assert np.array_equal(x0, x1) and np.array_equal(v0, v1)
    assert np.array_equal(ef0[0], ef1[0]) and np.array_equal(ef0[1], ef1[1])
    for k in ("counts", "sep", "rows", "cols", "vals", "dist_sum", "dist2_sum"):
        assert np.array_equal(s0[k], s1[k]), k
    assert s0["pairs"] == s1["pairs"] and s0["samples"] == s1["samples"] == 6


def test_argument_and_state_errors(built_lib):
    from multimm_b200._lib import Error
    from multimm_b200.engine import Engine

    n = 100
    bins = np.zeros(n, np.int32)
    with Engine(n) as eng:
        for call in (eng.triplets_add, eng.triplets_read):
            with pytest.raises(Error) as ei:
                call()
            assert ei.value.code == MMM_ERR_STATE
        eng.triplets_configure(0.2, bins, 1)  # configuring needs no positions; adding does
        with pytest.raises(Error) as ei:
            eng.triplets_add()
        assert ei.value.code == MMM_ERR_STATE
        eng.set_positions(TR.globule(n, 680, 1))
        bad = [dict(rc_nm=0.0), dict(rc_nm=-0.2), dict(rc_nm=float("inf")), dict(rc_nm=float("nan")), dict(n_bins=0),
               dict(n_bins=2**20 + 1), dict(bin_of_bead=None), dict(bin_of_bead=np.full(n, -2, np.int32)),
               dict(bin_of_bead=np.full(n, 1, np.int32)), dict(max_chunk_keys=-1)]
        for kw in bad:
            args = dict(rc_nm=0.2, bin_of_bead=bins, n_bins=1, max_chunk_keys=0)
            args.update(kw)
            with pytest.raises(ValueError):
                eng.triplets_configure(**args)
            with pytest.raises(Error) as ei:  # a refused configuration leaves the accumulator unconfigured
                eng.triplets_add()
            assert ei.value.code == MMM_ERR_STATE
        with pytest.raises(ValueError):
            eng.triplets_configure(0.2, bins[:-1], 1)
        eng.triplets_configure(0.3, np.full(n, 2**20 - 1, np.int32), 2**20)  # the largest key: (B^3 - 1) < 2^60
        eng.triplets_add()
        r = eng.triplets_read()
        assert r["samples"] == 1 and r["triples"] > 0 and len(r["vals"]) == 1
        assert (int(r["p"][0]), int(r["q"][0]), int(r["r"][0])) == (2**20 - 1,) * 3 and int(r["vals"][0]) == r["triples"]


# ---- driver -------------------------------------------------------------------------------------------
def _ini(path, **fields):
    base = dict(PLATFORM="B200", N_BEADS=1500, LOOPS_PATH=BEDPE, OUT_PATH=str(path / "out"), SAVE_PLOTS=False,
                CHROM="chr1", LOC_START=10_000_000, LOC_END=60_000_000, MIN_MAX_ITERATIONS=150, SIM_RUN_MD=True,
                SIM_N_STEPS=650, SIM_SAMPLING_STEP=100, TRJ_FRAMES=4, DOWNSAMPLING_PROB=0.5, SAVE_TRIPLETS=True,
                TRIPLET_RESOLUTION=100_000, CONTACT_RADIUS=0.3)
    base.update(fields)
    path.mkdir(parents=True, exist_ok=True)
    ini = path / "config.ini"
    ini.write_text("[Main]\n" + "".join(f"{k} = {v}\n" for k, v in base.items() if v is not None))
    return str(ini), base["OUT_PATH"]


def test_driver_files_equal_reproduction(built_lib, tmp_path):
    from multimm_b200 import contacts, loaders, run, triplets
    from multimm_b200.model import MultiMM, _f

    step = 150
    ini, out = _ini(tmp_path / "s", MD_SAMPLE_STEP=step)
    assert run.main(["-c", ini]) == 0
    ini0, out0 = _ini(tmp_path / "p", SAVE_TRIPLETS=None, TRIPLET_RESOLUTION=None, CONTACT_RADIUS=None)
    assert run.main(["-c", ini0]) == 0
    got, plain = _files(out), _files(out0)
    new = {"analysis/triplets.npz", "analysis/triplets_md.npz"}
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
    gb = contacts.genome_bins(m.layout, 100_000, n_beads=1500, max_bins=triplets.MAX_BINS)
    assert gb.n_bins == 500
    e.triplets_configure(0.3, gb.bins, gb.n_bins)
    e.triplets_add()
    one = triplets.result(e.triplets_read(), 0.3, gb)
    e.md_configure(str(a.SIM_INTEGRATOR_TYPE).lower(), _f(a.SIM_INTEGRATOR_STEP), _f(a.SIM_TEMPERATURE),
                   float(a.SIM_FRICTION_COEFF), loaders.BEAD_MASS, int(a.SHUFFLING_SEED), amd_alpha=_f(a.SIM_AMD_ALPHA),
                   amd_e=_f(a.SIM_AMD_E))
    e.set_velocities_to_temperature(_f(a.SIM_TEMPERATURE), int(a.SHUFFLING_SEED))
    e.triplets_configure(0.3, gb.bins, gb.n_bins)
    done = 0
    while done < 600:
        e.md_run(50, want_report=False)
        done += 50
        if done % step == 0:
            e.triplets_add()
    md = triplets.result(e.triplets_read(), 0.3, gb, 600 // step)
    m.close()
    assert int(one["triples"]) > 0 and len(one["vals"]) > 0
    for name, want in (("triplets.npz", one), ("triplets_md.npz", md)):
        d = triplets.load(os.path.join(out, "analysis", name))
        for k in triplets.KEYS:
            assert np.array_equal(d[k], want[k]) and d[k].dtype == np.asarray(want[k]).dtype, (name, k)
    assert int(triplets.load(os.path.join(out, "analysis", "triplets_md.npz"))["members"]) == 4


def test_ensemble_triplets_are_the_aggregate_of_the_members(built_lib, tmp_path):
    from multimm_b200 import run, triplets

    ini, out = _ini(tmp_path, N_BEADS=1000, GENERATE_ENSEMBLE=True, N_ENSEMBLE=2, MD_SAMPLE_STEP=200,
                    SIM_N_STEPS=400, MIN_MAX_ITERATIONS=80)
    args, _ = run.get_config(["-c", ini])
    run.run_ensemble(args, devices=[0])
    for name in (lambda p: p, lambda p: p[:-4] + "_md.npz"):
        paths = [name(run.member_triplets_path(out, i)) for i in range(2)]
        parts = [triplets.load(p) for p in paths]
        got = triplets.load(name(os.path.join(out, "ensemble_triplets.npz")))
        want = triplets.aggregate(paths)
        for k in triplets.KEYS:
            assert np.array_equal(got[k], want[k]) and got[k].dtype == want[k].dtype, k
        assert int(got["members"]) == sum(int(p["members"]) for p in parts)
        assert int(got["triples"]) == sum(int(p["triples"]) for p in parts) > 0
        assert int(got["vals"].sum()) == sum(int(p["vals"].sum()) for p in parts)


MEMORY_CHILD = r"""
import json, os, subprocess, sys
import numpy as np
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import triplets_ref as TR
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
x = TR.globule(n, 680, 1)
canon = (np.arange(n) * 1000 // n).astype(np.int32)
used = []
for cycle in range(3):
    eng = Engine(n)
    eng.set_positions(x)
    for rc, bins, nb, cap in ((0.2, canon, 1000, 0), (0.3, np.arange(n, dtype=np.int32), n, 10**6), (0.25, canon, 1000, 0)):
        eng.triplets_configure(rc, bins, nb, cap)
        eng.triplets_add()
        eng.triplets_read()
    eng.close()
    used.append(used_mib())
print(json.dumps(used))
"""


def test_triplet_buffers_freed_with_the_handle(built_lib):
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
