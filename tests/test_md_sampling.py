"""Trajectory maps on the host: the MD_SAMPLE_STEP setting and its refusals, the sampling schedule of
MultiMM.run_md on a stand-in engine (which steps are sampled; the trajectory, DCD and frames unchanged), the
*_md files built from S sampled structures and their ensemble sums, and a numpy restatement of the device's
merge-path merge (k_merge_part, k_merge, k_rle<kKeyVals>) against contacts._merge."""
import os

import numpy as np
import pytest

from multimm_b200 import contacts, distances

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BEDPE = os.path.join(GOLD, "synthetic_loops.bedpe")


def _cfg(tmp_path, **kw):
    from multimm_b200.config import SimulationConfig

    base = dict(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"), SIM_RUN_MD=True, SIM_N_STEPS=1000,
                SIM_SAMPLING_STEP=100, SAVE_CONTACTS=True, MD_SAMPLE_STEP=250)
    base.update(kw)
    return SimulationConfig(**base)


# ---- settings ------------------------------------------------------------------------------------------
def test_setting_is_an_extra_present_only_when_given(tmp_path):
    from multimm_b200 import run
    from multimm_b200.config import EXTRA_FIELDS, MD_SAMPLE_FIELDS, SimulationConfig, contact_setting

    assert MD_SAMPLE_FIELDS == {"MD_SAMPLE_STEP": (int, 0)}
    assert set(MD_SAMPLE_FIELDS) <= set(EXTRA_FIELDS) and not set(MD_SAMPLE_FIELDS) & set(SimulationConfig.model_fields)
    plain = SimulationConfig(LOOPS_PATH=BEDPE, OUT_PATH=str(tmp_path / "o"))
    assert set(plain.model_dump()) == set(SimulationConfig.model_fields)
    assert contact_setting(plain, "MD_SAMPLE_STEP") == 0
    again = SimulationConfig(**SimulationConfig(LOOPS_PATH=BEDPE, MD_SAMPLE_STEP="50").model_dump())
    assert contact_setting(again, "MD_SAMPLE_STEP") == 50
    with pytest.raises(ValueError):
        SimulationConfig(LOOPS_PATH=BEDPE, MD_SAMPLE_STEP="often")
    ini = tmp_path / "c.ini"
    ini.write_text(f"[Main]\nLOOPS_PATH = {BEDPE}\nOUT_PATH = {tmp_path / 'cli'}\n")
    args, _ = run.get_config(["-c", str(ini), "--md_sample_step", "200"])
    assert contact_setting(args, "MD_SAMPLE_STEP") == 200
    assert "md_sample_step = 200" in (tmp_path / "cli" / "metadata" / "config_auto.ini").read_text()
    args, _ = run.get_config(["-c", str(ini)])
    assert "md_sample_step" not in (tmp_path / "cli" / "metadata" / "config_auto.ini").read_text()


@pytest.mark.parametrize("fields,match", [
    (dict(MD_SAMPLE_STEP=-1), ">= 0"),
    (dict(SIM_RUN_MD=False), "SIM_RUN_MD"),
    (dict(SAVE_CONTACTS=False), "SAVE_CONTACTS or SAVE_DISTANCES"),
    (dict(MD_SAMPLE_STEP=1001), "no structure would be sampled"),
    (dict(SIM_N_STEPS=1050, MD_SAMPLE_STEP=1010), "no structure would be sampled"),  # the loop runs 1000 steps
    (dict(SIM_N_STEPS=99, MD_SAMPLE_STEP=50), "no structure would be sampled"),     # ... and here none
])
def test_bad_sample_step_refused_before_any_output(tmp_path, fields, match):
    from multimm_b200 import run

    args = _cfg(tmp_path, **fields)
    with pytest.raises(ValueError, match=match):
        run.args_tests(args)
    assert not (tmp_path / "o").exists()


def test_valid_sample_steps(tmp_path):
    from multimm_b200 import run

    for kw in (dict(MD_SAMPLE_STEP=0, SIM_RUN_MD=False, SAVE_CONTACTS=False), dict(MD_SAMPLE_STEP=1000),
               dict(MD_SAMPLE_STEP=7), dict(SAVE_CONTACTS=False, SAVE_DISTANCES=True),
               dict(SIM_N_STEPS=1050, MD_SAMPLE_STEP=1000)):
        run.args_tests(_cfg(tmp_path, **kw))
    assert not (tmp_path / "o").exists()


# ---- run_md on a stand-in engine ----------------------------------------------------------------------------
N = 40


def _positions(step):
    return np.random.default_rng(1000 + step).normal(scale=0.3, size=(N, 3))


def _one_shot(step, nc, nf, nd):
    """Stand-in maps of the structure at `step` (what the one-shot calls would return there)."""
    rng = np.random.default_rng(step)
    keys = np.unique(rng.integers(0, nf * nf, size=12)) if nf else np.zeros(0, np.int64)
    keys = np.unique(np.minimum(keys // nf, keys % nf) * nf + np.maximum(keys // nf, keys % nf)) if nf else keys
    return dict(counts=rng.integers(0, 5, size=(nc, nc)).astype(np.uint64) if nc else None,
                sep=rng.integers(0, 5, size=N).astype(np.uint64) if nc else None, pairs=int(rng.integers(0, 99)),
                keys=keys, vals=rng.integers(1, 4, size=len(keys)).astype(np.uint64),
                dist_sum=rng.integers(0, 2**40, size=(nd, nd)).astype(np.uint64) if nd else None,
                dist2_sum=rng.integers(0, 2**40, size=(nd, nd)).astype(np.uint64) if nd else None)


class FakeEngine:
    """Records the MD chunks and the samples; positions are a function of the step, as the real trajectory
    (its noise is keyed by step) does not depend on how the run is cut into chunks."""

    def __init__(self):
        self.step, self.runs, self.samples, self.cfg = 0, [], [], None

    def md_configure(self, *a, **k):
        pass

    def set_velocities_to_temperature(self, *a):
        pass

    def md_run(self, n, want_report=True):
        self.runs.append((self.step, n, want_report))
        self.step += n
        return dict(step=self.step, potential=float(self.step), kinetic=0.5, temperature=310.0) if want_report else None

    def get_positions(self):
        return _positions(self.step)

    def sampler_configure(self, rc, cb, nc, fb, nf, db, nd):
        self.cfg = (rc, nc if cb is not None else 0, nf if fb is not None else 0, nd if db is not None else 0)

    def sample(self):
        self.samples.append(self.step)

    def sampler_read(self):
        _, nc, nf, nd = self.cfg
        parts = [_one_shot(s, nc, nf, nd) for s in self.samples]
        out = dict(samples=len(parts), device_ms=1.0, rows=None, cols=None, vals=None)
        for k in ("counts", "sep", "dist_sum", "dist2_sum"):
            out[k] = sum(p[k] for p in parts) if parts and parts[0][k] is not None else None
        out["pairs"] = sum(p["pairs"] for p in parts)
        if nf:
            keys = np.concatenate([p["keys"] for p in parts])
            u, inv = np.unique(keys, return_inverse=True)
            vals = np.zeros(len(u), np.uint64)
            np.add.at(vals, inv, np.concatenate([p["vals"] for p in parts]))
            out["rows"], out["cols"], out["vals"] = (u // nf).astype(np.int32), (u % nf).astype(np.int32), vals
        return out


def _model(tmp_path, name, **kw):
    from multimm_b200.model import MultiMM

    cfg = _cfg(tmp_path, OUT_PATH=str(tmp_path / name), N_BEADS=N, SIM_SAMPLING_STEP=kw.pop("every", 100),
               TRJ_FRAMES=kw.pop("frames", 4), CONTACT_RESOLUTION=20_000, CONTACT_FINE_RESOLUTION=5_000,
               SAVE_DISTANCES=True, DISTANCE_RESOLUTION=30_000, **kw)
    m = MultiMM.__new__(MultiMM)
    m.args, m.save_path, m.timings = cfg, str(tmp_path / name) + "/", {}
    for sub in ("md_frames", "metadata", "model", "analysis"):
        os.makedirs(os.path.join(m.save_path, sub), exist_ok=True)
    m.engine, m.chr_ends = FakeEngine(), np.array([0, N])
    m.chrom_spin = np.zeros(N)
    m.mass_center = np.array([0.1, -0.2, 0.05])
    m.layout = dict(resolution=5_000, ends=[0], chr_ends=[0, N], chrom_idxs=[0], start_bp=1_000_000,
                    stop_bp=1_000_000 + 5_000 * N)
    m.contacts = m.contacts_fine = m.distances = None
    m.contacts_md = m.contacts_fine_md = m.distances_md = None
    m.contacts_file = m.contacts_fine_file = m.distances_file = None
    m.positions_minimized = _positions(0)
    m.report = None
    return m


def _tree(path):
    out = {}
    for sub in ("md_frames", "metadata", "model"):
        for f in sorted(os.listdir(os.path.join(path, sub))):
            with open(os.path.join(path, sub, f), "rb") as fh:
                out[f"{sub}/{f}"] = fh.read()
    return out


@pytest.mark.parametrize("n_steps,every,frames,sample", [(1000, 100, 4, 250), (1000, 100, 4, 30), (950, 100, 10, 100),
                                                         (600, 50, 600, 7), (1000, 1000, 1, 1000)])
def test_schedule_samples_and_leaves_the_trajectory_alone(tmp_path, n_steps, every, frames, sample, capsys):
    plain = _model(tmp_path, "plain", SIM_N_STEPS=n_steps, every=every, frames=frames, MD_SAMPLE_STEP=0,
                   SAVE_CONTACTS=False)
    plain.run_md()
    sampled = _model(tmp_path, "sampled", SIM_N_STEPS=n_steps, every=every, frames=frames, MD_SAMPLE_STEP=sample)
    sampled.run_md()
    ran = (n_steps // every) * every
    assert plain.engine.step == sampled.engine.step == ran
    assert sampled.engine.samples == list(range(sample, ran + 1, sample)) and plain.engine.samples == []
    # every chunk boundary of the unsampled run is one of the sampled run's; reports at the same steps
    bounds = lambda e: {s + n for s, n, _ in e.runs}
    assert bounds(plain.engine) <= bounds(sampled.engine)
    reports = lambda e: [s + n for s, n, r in e.runs if r]
    assert reports(plain.engine) == reports(sampled.engine)
    assert _tree(plain.save_path) == _tree(sampled.save_path)  # DCD, frames, thermodynamics, afterMD
    assert plain.contacts_md is None and sampled.contacts_md is not None


def test_files_from_sampled_structures(tmp_path):
    m = _model(tmp_path, "run", SIM_N_STEPS=1000, MD_SAMPLE_STEP=200)
    m.run_md()
    steps = m.engine.samples
    S = len(steps)
    assert S == 5
    rc, nc, nf, nd = m.engine.cfg
    parts = [_one_shot(s, nc, nf, nd) for s in steps]
    m.write_minimized = lambda: None
    m._whole, m.args.SAVE_PLOTS = False, False
    m.finish()
    c = contacts.load(os.path.join(m.save_path, "analysis", "contacts_md.npz"))
    assert int(c["members"]) == S and int(c["pairs"]) == sum(p["pairs"] for p in parts)
    assert np.array_equal(c["counts"], sum(p["counts"] for p in parts))
    assert np.array_equal(c["sep_pairs"], np.uint64(S) * contacts.sep_pairs(m.chrom_spin))
    f = contacts.load_fine(os.path.join(m.save_path, "analysis", "contacts_fine_md.npz"))
    assert int(f["members"]) == S and int(f["n_bins"]) == nf
    d = distances.load(os.path.join(m.save_path, "analysis", "distances_md.npz"))
    gb = m._distance_bins()
    one = distances.result(parts[0]["dist_sum"], parts[0]["dist2_sum"], gb, _positions(steps[0]), m.mass_center)
    assert int(d["members"]) == S
    assert np.array_equal(d["pair_count"], np.uint64(S) * one["pair_count"])
    assert np.array_equal(d["bin_beads"], np.uint64(S) * one["bin_beads"])
    rs = sum(distances.radial_sums(_positions(s), m.mass_center, gb.bins, gb.n_bins)[0] for s in steps)
    assert np.array_equal(d["radial_sum"], rs)
    iu = np.triu_indices(gb.n_bins)  # the file keeps the upper triangle (the stand-in maps are not symmetric)
    assert np.array_equal(d["dist_sum"][iu], sum(p["dist_sum"] for p in parts)[iu])
    assert not os.path.exists(os.path.join(m.save_path, "analysis", "contacts.npz"))  # no minimised-structure map here


def test_means_of_identical_structures_equal_one_structures(tmp_path):
    rng = np.random.default_rng(3)
    gb = contacts.GenomeBins(np.repeat(np.arange(5), 8).astype(np.int32), np.zeros(5, np.int32),
                             np.arange(5, dtype=np.int64) * 1000, 1000)
    x = rng.normal(size=(40, 3))
    ds, d2 = rng.integers(0, 2**40, size=(5, 5)).astype(np.uint64), rng.integers(0, 2**40, size=(5, 5)).astype(np.uint64)
    one = distances.result(ds, d2, gb, x, np.zeros(3))
    S = 37
    many = distances.sampled_result(ds * np.uint64(S), d2 * np.uint64(S), gb, one["radial_sum"] * np.uint64(S),
                                    one["radial2_sum"] * np.uint64(S), S)
    for fn in (distances.mean_distance, distances.rms_distance, distances.std_distance):
        assert np.array_equal(fn(one), fn(many), equal_nan=True)
    for a, b in zip(distances.radial_profile(one), distances.radial_profile(many)):
        assert np.array_equal(a, b, equal_nan=True)
    cmap = rng.integers(0, 9, size=(5, 5)).astype(np.uint64)
    sep = rng.integers(0, 9, size=40).astype(np.uint64)
    den = contacts.sep_pairs(np.zeros(40))
    c1 = contacts.result(cmap, sep, 3, 0.2, gb, den)
    cS = contacts.result(cmap * np.uint64(S), sep * np.uint64(S), 3 * S, 0.2, gb, den * np.uint64(S), members=S)
    assert np.array_equal(contacts.contact_probability(c1), contacts.contact_probability(cS), equal_nan=True)


def test_ensemble_md_files_are_the_sums_of_the_members(tmp_path):
    from multimm_b200 import run

    out = tmp_path / "ens"
    results = []
    for i in range(2):
        m = _model(tmp_path, f"run_{i}", SIM_N_STEPS=1000, MD_SAMPLE_STEP=100 * (i + 2))
        m.args.OUT_PATH = str(out)
        m.engine.samples = []
        m.run_md()
        m.contacts_file = run.member_contacts_path(str(out), i)
        m.contacts_fine_file = run.member_contacts_fine_path(str(out), i)
        m.distances_file = run.member_distances_path(str(out), i)
        m.write_minimized = lambda: None
        m._whole, m.args.SAVE_PLOTS = False, False
        m.save_args_to_txt = lambda path: None
        # the minimised-structure maps, as a member writes them beside the trajectory maps
        m.contacts = dict(m.contacts_md, members=np.int64(1))
        m.contacts_fine = dict(m.contacts_fine_md, members=np.int64(1))
        m.distances = dict(m.distances_md, members=np.int64(1))
        m.finish()
        results.append(dict(replica=i))
    args = _cfg(tmp_path, OUT_PATH=str(out), SAVE_DISTANCES=True, CONTACT_FINE_RESOLUTION=5_000)
    run.write_ensemble_contacts(args, results)
    run.write_ensemble_distances(args, results)
    parts = [contacts.load(contacts.md_path(run.member_contacts_path(str(out), i))) for i in range(2)]
    agg = contacts.load(str(out / "ensemble_contacts_md.npz"))
    assert int(agg["members"]) == 5 + 3
    assert np.array_equal(agg["counts"], parts[0]["counts"] + parts[1]["counts"])
    assert np.array_equal(agg["sep_pairs"], parts[0]["sep_pairs"] + parts[1]["sep_pairs"])
    fine = [contacts.load_fine(contacts.md_path(run.member_contacts_fine_path(str(out), i))) for i in range(2)]
    fagg = contacts.load_fine(str(out / "ensemble_contacts_fine_md.npz"))
    want = contacts._merge(fine[0]["rows"], fine[0]["cols"], fine[0]["vals"], fine[1]["rows"], fine[1]["cols"],
                           fine[1]["vals"], int(fine[0]["n_bins"]))
    for g, w in zip((fagg["rows"], fagg["cols"], fagg["vals"]), want):
        assert np.array_equal(g, w)
    dparts = [distances.load(contacts.md_path(run.member_distances_path(str(out), i))) for i in range(2)]
    dagg = distances.load(str(out / "ensemble_distances_md.npz"))
    for k in ("dist_sum", "pair_count", "bin_beads", "radial_sum"):
        assert np.array_equal(dagg[k], dparts[0][k] + dparts[1][k])
    assert os.path.exists(out / "ensemble_contacts.npz") and os.path.exists(out / "ensemble_distances.npz")


# ---- the device merge, restated ---------------------------------------------------------------------------
def _diag(a, b, d):
    """mg_diag: keys taken from a among the first d outputs (a first among equal keys)."""
    lo, hi = max(0, d - len(b)), min(d, len(a))
    while lo < hi:
        mid = (lo + hi) // 2
        if a[mid] <= b[d - 1 - mid]:
            lo = mid + 1
        else:
            hi = mid
    return lo


def device_merge(ak, av, bk, bv, threads=4, per=2):
    """k_merge_part + k_merge (CTA tiles of threads * per outputs, one diagonal search per CTA, then per
    thread inside the CTA's slices) + k_rle<kKeyVals> (equal neighbours added)."""
    tile, total = threads * per, len(ak) + len(bk)
    part = [_diag(ak, bk, min(p * tile, total)) for p in range(-(-total // tile) + 1)]
    ok, ov = np.zeros(total, np.uint64), np.zeros(total, np.uint64)
    for c in range(len(part) - 1):
        d0, d1 = c * tile, min(c * tile + tile, total)
        sa, sb = ak[part[c]:part[c + 1]], bk[d0 - part[c]:d1 - part[c + 1]]
        va, vb = av[part[c]:part[c + 1]], bv[d0 - part[c]:d1 - part[c + 1]]
        for t in range(threads):
            d = min(t * per, len(sa) + len(sb))
            i = _diag(sa, sb, d)
            j = d - i
            for q in range(per):
                if d + q >= len(sa) + len(sb):
                    break
                if i < len(sa) and (j >= len(sb) or sa[i] <= sb[j]):
                    ok[d0 + d + q], ov[d0 + d + q] = sa[i], va[i]
                    i += 1
                else:
                    ok[d0 + d + q], ov[d0 + d + q] = sb[j], vb[j]
                    j += 1
    assert np.all(ok[1:] >= ok[:-1])
    head = np.ones(total, bool)
    head[1:] = ok[1:] != ok[:-1]
    e = np.cumsum(head) - 1
    keys, vals = ok[head], np.zeros(int(head.sum()), np.uint64)
    np.add.at(vals, e, ov)
    return keys, vals


def _lists(kind, rng):
    if kind == "empty_a":
        return np.zeros(0, np.uint64), rng.choice(50, 9, replace=False)
    if kind == "empty_b":
        return rng.choice(50, 9, replace=False), np.zeros(0, np.uint64)
    if kind == "both_empty":
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
    if kind == "all_equal":
        k = rng.choice(10**6, 23, replace=False)
        return k, k.copy()
    if kind == "disjoint":
        return rng.choice(100, 17, replace=False), 1000 + rng.choice(100, 13, replace=False)
    if kind == "disjoint_reversed":
        return 1000 + rng.choice(100, 13, replace=False), rng.choice(100, 17, replace=False)
    if kind == "interleaved":
        k = rng.choice(10**4, 60, replace=False)
        return k[:31], k[31:]
    # runs of equal keys across partition boundaries: half the keys shared, long lists
    k = rng.choice(2**62, 200, replace=False)
    return np.concatenate([k[:120], k[150:170]]), np.concatenate([k[60:150], k[170:]])


@pytest.mark.parametrize("kind", ["empty_a", "empty_b", "both_empty", "all_equal", "disjoint", "disjoint_reversed",
                                  "interleaved", "runs_across_tiles"])
@pytest.mark.parametrize("threads,per", [(4, 2), (3, 3), (256, 8)])
def test_merge_restatement_matches_host_merge(kind, threads, per):
    rng = np.random.default_rng(hash(kind) % 2**32)
    a, b = _lists(kind, rng)
    ak, bk = np.sort(np.asarray(a, np.uint64)), np.sort(np.asarray(b, np.uint64))
    av = rng.integers(1, 2**40, size=len(ak)).astype(np.uint64)
    bv = rng.integers(1, 2**40, size=len(bk)).astype(np.uint64)
    nb = 2**31 - 1
    got_k, got_v = device_merge(ak, av, bk, bv, threads, per)
    rows, cols, vals = contacts._merge((ak // nb).astype(np.int32), (ak % nb).astype(np.int32), av,
                                       (bk // nb).astype(np.int32), (bk % nb).astype(np.int32), bv, nb)
    assert np.array_equal(got_k, rows.astype(np.uint64) * np.uint64(nb) + cols.astype(np.uint64))
    assert np.array_equal(got_v, vals)
    # tiles of an odd number of outputs cut the merged list between the two copies of a shared key
    merged = np.sort(np.concatenate([ak, bk]))
    tile = threads * per
    cuts = [p * tile for p in range(1, -(-len(merged) // tile)) if merged[p * tile - 1] == merged[p * tile]]
    if kind in ("all_equal", "runs_across_tiles") and tile % 2:
        assert cuts
