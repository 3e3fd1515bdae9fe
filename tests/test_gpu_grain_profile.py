"""GPU: per-plane grain profiles (cet_grain_profile_group / cetkmc.grain_profile_group) against the NumPy reference
of tests/profileref.py over the label volume of Context.grains(labels=True), after each kind of labelling
(Context.grains: arrival-order gid, metrics_group: site-order gid, the theta_only criterion), for groups of 1, 4 and
18 in either order; identities with the metrics row; edge lattices; non-interference with the cadence and sweeps;
rejections; and the drivers' profile files, solo against grouped."""
import csv
import ctypes as C
import filecmp
import os

import numpy as np
import pytest

import profileref

pytestmark = pytest.mark.gpu

THR = 3.0
EVERY, SEED = 10, 77


def _half_grown(cet, L, q):
    """A half-grown lattice of its own NU_DEP and substrate temperature, a few sweeps in (test_gpu_metrics_group)."""
    from cetkmc import _synth
    from cetkmc._config import rate_params, thermal_params
    packed, th, ph, T = _synth.half_grown(L, seed=40 + q, grain=4)
    ctx = cet.Context(L=L)
    ctx.set_rate_params(rate_params(0.1, overrides={"NU_DEP": 2e13 * (1 + q % 5)}))
    st, df = _synth.unpack(packed)
    ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
    sp = cet._lib.SweepParams()
    sp.seed, sp.events_per_sweep, sp.p_max = 300 + q, 0.005 * L ** 3, 0.1
    sp.defect_fraction, sp.thermal_every = 0.01, 5
    tp = thermal_params(1e-6, nan_to_num=True, t_floor=2600.0 + 50.0 * (q % 5))
    ctx.sweep_run(7 + q % 3, sp, tp)
    return ctx, sp, tp


def _driver(cet, L, q, n_sweeps):
    """The G-R driver's lattice (initialize_lattice, nuclei on k = 0, T rising with k) after n_sweeps sweeps."""
    from cetkmc import campaign
    from cetkmc import kmc_simulation as ks
    from cetkmc._config import rate_params
    temp, nu_dep = (2600.0, 2800.0, 3000.0)[q % 3], (1e12, 2e13, 1e14)[q % 3]
    np.random.seed(11 + q)
    ctx = cet.Context(L=L)
    ctx.set_rate_params(rate_params(0.1, 1, 2, 3, overrides={"NU_DEP": nu_dep}))
    campaign._upload_initial(ctx, L, 20, temp, 0.1, None, 0, L)
    sp, tp = campaign._sweep_setup(L, 11 + q, temp, None, 0.1, 3e-3, ks.THERMAL_EVERY)
    ctx.sweep_run(n_sweeps, sp, tp)
    return ctx


def _params(cet, ctxs):
    from cetkmc import metrics
    from cetkmc._config import constants
    out = []
    n_sites = int(np.prod(ctxs[0].owned_shape))
    for _ in ctxs:
        p = cet._lib.MetricsParams()
        p.theta_threshold, p.ar_threshold = 0.5, THR
        p.pct_pos[:] = metrics.percentile_positions(n_sites)
        p.refresh, p.carbon_id, p.epoch, p.seed = 0, 3, 4, SEED
        p.prob_base, p.e_mig, p.kT, p.T_default = 0.12, 0.3, constants.K_T, constants.T_SUB
        out.append(p)
    return out


def _label(cet, ctxs, kind):
    """Label every context of ctxs with one kind of labelling; returns the metrics rows for kind 'metrics'."""
    if kind == "metrics":
        return cet.metrics_group(ctxs, _params(cet, ctxs))
    for c in ctxs:
        c.grains(0.5, theta_only=kind == "theta")
    return None


def _reference(c, kind):
    """Label volume and reference grain data of the labelling `kind` (relabels: call after the device profiles)."""
    g = c.grains(0.5, labels=True, theta_only=kind == "theta")
    return g


def _check_group(cet, ctxs, kind):
    rows = _label(cet, ctxs, kind)
    got = {ax: cet.grain_profile_group(ctxs, ax, THR) for ax in range(3)}
    rev = {ax: cet.grain_profile_group(ctxs[::-1], ax, THR)[::-1] for ax in range(3)}
    solo = {ax: np.stack([cet.grain_profile_group([c], ax, THR)[0] for c in ctxs]) for ax in range(3)}
    L = ctxs[0].shape[0]
    for ax in range(3):
        assert got[ax].shape == (len(ctxs), 4, L) and got[ax].dtype == np.int64
        assert np.array_equal(got[ax], rev[ax]) and np.array_equal(got[ax], solo[ax])
    for q, c in enumerate(ctxs):
        g = _reference(c, kind)
        lab = g["labels"]
        _sizes, lo, hi = profileref.grain_boxes(lab, g["n"])
        assert np.array_equal(lo, g["box_lo"]) and np.array_equal(hi, g["box_hi"])
        eq = profileref.aspect_ratios(lo, hi) < THR
        for ax in range(3):
            want = profileref.grain_profile(lab, ax, THR, g["n"])
            assert np.array_equal(got[ax][q], want), (kind, q, ax)
            # identities with the labelling's statistics and, for metrics_group, its row
            assert got[ax][q, 0].sum() == g["size"].sum()
            assert got[ax][q, 1].sum() == g["size"][eq].sum()
            assert got[ax][q, 2].sum() == (g["box_hi"][:, ax] - g["box_lo"][:, ax] + 1).sum()
            if rows is not None:
                assert got[ax][q, 0].sum() == rows[q]["size_sum"]
                assert int(eq.sum()) == rows[q]["n_equiaxed"] and g["n"] == rows[q]["n_grains"]
    return got


@pytest.mark.parametrize("L", [24, 30, 64, 96])
@pytest.mark.parametrize("kind", ["grains", "metrics", "theta"])
def test_profile_equals_reference(cet, L, kind):
    ctxs = [_half_grown(cet, L, 0)[0], _driver(cet, L, 0, 40), _half_grown(cet, L, 1)[0], _driver(cet, L, 1, 120)]
    try:
        got = _check_group(cet, ctxs, kind)
        assert all(got[ax][:, 0].sum() > 0 for ax in range(3))
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("kind", ["grains", "metrics"])
def test_profile_group_of_18(cet, kind):
    ctxs = [_half_grown(cet, 30, q)[0] for q in range(14)] + [_driver(cet, 30, q, 30 + 20 * q) for q in range(4)]
    try:
        _check_group(cet, ctxs, kind)
    finally:
        for c in ctxs:
            c.close()


def test_profile_driver_lattices_after_300_sweeps(cet):
    ctxs = [_driver(cet, 64, q, 300) for q in range(3)]
    try:
        _check_group(cet, ctxs, "metrics")
    finally:
        for c in ctxs:
            c.close()


# -- edge lattices --------------------------------------------------------------------------------------------------

def _upload(cet, state, theta, phi):
    L = state.shape[0]
    ctx = cet.Context(L=L)
    ctx.upload(state=state.astype(np.int64), theta=theta, phi=phi, T=np.full(state.shape, 2900.0),
               defects=np.zeros(state.shape, np.int64))
    return ctx


def _even(L):
    i = np.arange(L)
    return ((i[:, None, None] + i[None, :, None] + i[None, None, :]) % 2 == 0).astype(np.int64)


def _edge(name):
    rng = np.random.default_rng(5)
    if name == "empty":
        return np.zeros((24,) * 3, np.int64), np.zeros((24,) * 3), np.zeros((24,) * 3), 0
    if name == "one":
        return _even(24), np.full((24,) * 3, 0.3), np.full((24,) * 3, 1.1), 1
    if name == "filling":                      # every site one orientation: the two parity classes, each filling the box
        return np.ones((25,) * 3, np.int64), np.full((25,) * 3, 0.3), np.full((25,) * 3, 1.1), 2
    if name == "single_site":
        st = np.zeros((25,) * 3, np.int64)
        st[24, 0, 13] = 2
        return st, np.full((25,) * 3, 0.3), np.full((25,) * 3, 1.1), 1
    L = 64                                     # pepper: random orientations, > 10^5 grains
    return rng.integers(1, 4, (L, L, L)), rng.uniform(0, np.pi, (L, L, L)), rng.uniform(0, 2 * np.pi, (L, L, L)), None


@pytest.mark.parametrize("name", ["empty", "one", "filling", "single_site", "pepper"])
@pytest.mark.parametrize("kind", ["grains", "metrics"])
def test_profile_edge_lattices(cet, name, kind):
    st, th, ph, n_expected = _edge(name)
    ctxs = [_upload(cet, st, th, ph), _upload(cet, st, th, ph)]
    try:
        got = _check_group(cet, ctxs, kind)
        n = ctxs[0].grains(0.5)["n"]
        if n_expected is None:
            assert n > 10 ** 5
        else:
            assert n == n_expected
        L = st.shape[0]
        if name == "pepper":                                                               # both classes occur
            assert all(0 < got[ax][0, 1].sum() < got[ax][0, 0].sum() for ax in range(3))
        if name == "empty":
            assert not got[0].any() and not got[1].any() and not got[2].any()
        if name == "filling":
            for ax in range(3):
                assert np.array_equal(got[ax][0, 0], np.full(L, L * L)) and np.array_equal(got[ax][0, 2], np.full(L, 2))
                assert np.array_equal(got[ax][0, 1], got[ax][0, 0])                      # AR 1: equiaxed
    finally:
        for c in ctxs:
            c.close()


# -- non-interference ----------------------------------------------------------------------------------------------

def _run(ctx, q):
    np.random.seed(1000 + q)
    return dict(ctx=ctx, rng=np.random.get_state(), consts=(1.0e6 * (q + 1), 2.0, 3.0e-9, 4.0), rows=[], profiles=[],
                total_time=1e-3 * q, nucleation_count=5 * q, cet_detected=False)


def _labels(cet, ctx):
    lab = np.empty(ctx.owned_shape, np.int32)
    L = cet._lib
    L.check(L.lib().cet_grains_download_labels(ctx._h, L._ptr(lab)), "labels")
    return lab


def _snapshot(cet, ctx, rates=True, labels=True):
    s = dict(packed=ctx.download_packed(), clock=ctx.sweep_state(), theta=ctx.download(theta=True)["theta"])
    if rates:
        s["site_rate"], s["dep_rate"] = ctx.rates_download()
    if labels:
        s["labels"] = _labels(cet, ctx)
    return s


def _same_snapshots(cet, xs, ys, rates=True):
    for x, y in zip(xs, ys):
        sx, sy = _snapshot(cet, x, rates), _snapshot(cet, y, rates)
        for k in sx:
            assert (sx[k] == sy[k]) if k == "clock" else np.array_equal(sx[k], sy[k], equal_nan=True), k


@pytest.mark.parametrize("philox", [False, True])
def test_profile_calls_change_nothing(cet, philox):
    from cetkmc import campaign
    a = [_half_grown(cet, 24, q) for q in range(4)]
    b = [_half_grown(cet, 24, q) for q in range(4)]
    ra = [_run(c, q) for q, (c, _, _) in enumerate(a)]
    rb = [_run(c, q) for q, (c, _, _) in enumerate(b)]
    try:
        for last in (EVERY, EVERY + 3, 2 * EVERY):
            campaign._cadence_group(ra, last, EVERY, philox, SEED, profile_axis=last % 3)
            cet.grain_profile_group([r["ctx"] for r in ra][::-1], 1, THR)                    # extra calls in between
            campaign._cadence_group(rb, last, EVERY, philox, SEED)
            for x, y in zip(ra, rb):
                assert x["rows"][-1] == y["rows"][-1] and x["cet_detected"] == y["cet_detected"]
                assert x["rng"][0] == y["rng"][0] and np.array_equal(x["rng"][1], y["rng"][1]) and x["rng"][2:] == y["rng"][2:]
                assert x["profiles"][-1][0] == last and x["profiles"][-1][1].shape == (4, 24)
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b], rates=False)    # a refresh left them stale
            ga = cet.sweep_run_group([c for c, _, _ in a], 6, [s for _, s, _ in a], [t for _, _, t in a])
            gb = cet.sweep_run_group([c for c, _, _ in b], 6, [s for _, s, _ in b], [t for _, _, t in b])
            assert ga == gb
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b])
    finally:
        for c, _, _ in a + b:
            c.close()


# -- rejections ----------------------------------------------------------------------------------------------------

def _raw(cet, ctxs, axis, out, n=None):
    """cet_grain_profile_group called directly (the binding's own checks bypassed): its return code."""
    h = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
    ptr = None if out is None else out.ctypes.data_as(C.POINTER(C.c_int64))
    return cet._lib.lib().cet_grain_profile_group(h, len(ctxs) if n is None else n, axis, THR, ptr)


def test_rejections_leave_everything_untouched(cet):
    a, sa, ta = _half_grown(cet, 24, 0)
    b, sb, tb = _half_grown(cet, 24, 1)
    a2, sa2, ta2 = _half_grown(cet, 24, 0)
    b2, sb2, tb2 = _half_grown(cet, 24, 1)
    fresh = _upload(cet, *_edge("one")[:3])                                      # never labelled
    other = _upload(cet, *_edge("filling")[:3])
    slab = cet.Context(L=24, i_begin=0, i_end=12)
    try:
        cet.metrics_group([a, b], _params(cet, [a, b]))
        cet.metrics_group([a2, b2], _params(cet, [a2, b2]))
        other.grains(0.5)
        before = [_snapshot(cet, x, rates=False, labels=x is not fresh) for x in (a, b, fresh)]
        out = np.full((70, 4, 24), -7, np.int64)
        sentinel = out.copy()
        for ctxs, axis, o, n, match in (([a, fresh], 2, out, None, "labell"),
                                        ([a, slab], 2, out, None, "slab"),
                                        ([a, other], 2, out, None, "L ="),
                                        ([a, b, a], 2, out, None, "repeats"),
                                        ([a] * 65, 2, out, None, "n_ctx"),
                                        ([a, b], 3, out, None, "axis"),
                                        ([a, b], -1, out, None, "axis"),
                                        ([a, b], 2, None, None, "NULL"),
                                        ([a, b], 2, out, 0, "n_ctx")):
            assert _raw(cet, ctxs, axis, o, n) != 0
            assert match in cet._lib.lib().cet_last_error().decode()
            assert np.array_equal(out, sentinel)
        with pytest.raises(RuntimeError, match="labell"):
            cet.grain_profile_group([fresh], 0, THR)
        for x, s in zip((a, b, fresh), before):
            t = _snapshot(cet, x, rates=False, labels=x is not fresh)
            for k in s:
                assert (s[k] == t[k]) if k == "clock" else np.array_equal(s[k], t[k], equal_nan=True), k
        # both still work and match their twins, and so do the sweeps that follow
        for ax in range(3):
            assert np.array_equal(cet.grain_profile_group([a, b], ax, THR), cet.grain_profile_group([a2, b2], ax, THR))
        assert cet.sweep_run_group([a, b], 5, [sa, sb], [ta, tb]) == cet.sweep_run_group([a2, b2], 5, [sa2, sb2], [ta2, tb2])
        _same_snapshots(cet, [a, b], [a2, b2])
    finally:
        for x in (a, b, a2, b2, fresh, other, slab):
            x.close()


# -- the drivers -----------------------------------------------------------------------------------------------------

def _tree_files(root):
    out = []
    for d, _, fs in os.walk(root):
        out += [os.path.relpath(os.path.join(d, f), root) for f in fs]
    return sorted(out)


def _same_tree(a, b):
    files = _tree_files(a)
    assert files == _tree_files(b)
    for f in files:
        assert filecmp.cmp(os.path.join(a, f), os.path.join(b, f), shallow=False), f
    return files


def _read(path):
    with open(path) as fh:
        return list(csv.DictReader(fh))


def _same_subset(plain, other):
    """Every file of the run without profile_axis, byte-identical in the run with it; returns the extra files."""
    files = _tree_files(plain)
    for f in files:
        assert filecmp.cmp(os.path.join(plain, f), os.path.join(other, f), shallow=False), f
    return sorted(set(_tree_files(other)) - set(files))


def _terminating_replica(monkeypatch, campaign, temp):
    """Replica 1 (init_seed 43) of the cases at T_sub = temp starts from a W lattice with three empty sites: it
    terminates early, inside an interval (test_gpu_init_group)."""
    upload = campaign._upload_initial

    def upload_initial(ctx, L, n_seeds, t, impurity_c, lattice, i_begin, i_end):
        if t == temp and getattr(ctx, "init_seed", None) == 43:
            st = np.ones((L, L, L), np.int64)
            th, ph = np.full((L, L, L), 0.5), np.full((L, L, L), 1.0)
            for j, k in ((3, 4), (11, 17), (20, 9)):
                st[L - 1, j, k] = 0
                th[L - 1, j, k] = ph[L - 1, j, k] = 0.0
            lattice = (st, th, ph, np.full((L, L, L), 2900.0), np.zeros((L, L, L), np.int64))
        return upload(ctx, L, n_seeds, t, impurity_c, lattice, i_begin, i_end)
    monkeypatch.setattr(campaign, "_upload_initial", upload_initial)


def _check_case_profiles(root, files):
    """Every metrics row of every case has its L planes in cet_profile.csv, and the final profile's Solid column sums
    to the sites the grains hold."""
    prof = [f for f in files if f.endswith("/cet_profile.csv")]
    assert len(prof) == sum(f.endswith("/metrics.csv") for f in files if not f.startswith("plot_cet/"))
    for f in prof:
        rows = _read(os.path.join(root, f))
        steps = [int(r["Step"]) for r in _read(os.path.join(root, f.replace("cet_profile.csv", "metrics.csv")))]
        assert sorted({int(r["Step"]) for r in rows}) == sorted(steps)
        assert len(rows) == 24 * len(steps)
    return prof


GR = dict(L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3, seed=7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_gr_sweep_profiles(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign, metrics
    monkeypatch.chdir(tmp_path)
    kw = dict(GR, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    temps, nu_deps = [2700.0, 3000.0], [2e13, 1e14]
    _terminating_replica(monkeypatch, campaign, 3000.0)
    base, ens = campaign.run_gr_sweep(temps, nu_deps, output_root="plain", replicas=3, **kw)
    a, ens_a = campaign.run_gr_sweep(temps, nu_deps, output_root="solo", replicas=3, profile_axis=2, **kw)
    b, ens_b = campaign.run_gr_sweep(temps, nu_deps, output_root="grouped", replicas=3, batch=4, profile_axis=2, **kw)
    assert a == base and b == base and ens_a == ens and ens_b == ens
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    prof = _check_case_profiles("outputs/solo", files)
    assert len(prof) == 12 and extra == sorted(prof + ["cet_map_profile_rank0.csv"])
    for root in ("plain", "solo", "grouped"):
        campaign.merge_cet_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    rows = _read("outputs/solo/cet_map_profile.csv")
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP", "CET_Height", "Front_Height"]
    assert [(int(r["case"]), int(r["replica"])) for r in rows] == [(q, r) for q in range(4) for r in range(3)]
    for r in rows:
        p = f"outputs/solo/T{float(r['T_sub']):g}_R{float(r['NU_DEP']):g}" + ("" if r["replica"] == "0" else f"/rep{r['replica']}")
        _step, prof_last = campaign.read_profile_csv(f"{p}/cet_profile.csv")
        s = metrics.cet_profile_summary(prof_last, 24 * 24)
        assert (int(r["CET_Height"]), int(r["Front_Height"])) == (s["CET_Height"], s["Front_Height"])
    # the profile ensemble: statistics recomputed from the per-replica rows
    ens_rows = _read("outputs/solo/cet_map_profile_ensemble.csv")
    assert len(ens_rows) == 4
    for q, e in enumerate(ens_rows):
        h = np.array([int(r["CET_Height"]) for r in rows if int(r["case"]) == q])
        v = h[h >= 0].astype(np.float64)
        assert int(e["replicas"]) == 3 and float(e["p_cet_height"]) == float(np.mean(h >= 0))
        assert e["CET_Height_mean"] == (str(float(np.mean(v))) if v.size else "")
        assert e["CET_Height_se"] == (str(float(np.std(v, ddof=1) / np.sqrt(v.size))) if v.size > 1 else "")


MAP = dict(L=24, n_sweeps=61, metrics_every=30, thermal_every=5, n_seeds=6, defect_fraction=3e-3, start=(12.0, 2.0),
           dt=1e-7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_melt_pool_map_profiles(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    kw = dict(MAP, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    powers, speeds = [150.0, 300.0], [1.0]
    _terminating_replica(monkeypatch, campaign, 2900.0)
    base = campaign.run_melt_pool_map(powers, speeds, output_root="plain", temp=2900.0, replicas=2, **kw)
    a = campaign.run_melt_pool_map(powers, speeds, output_root="solo", temp=2900.0, replicas=2, profile_axis=0, **kw)
    b = campaign.run_melt_pool_map(powers, speeds, output_root="grouped", temp=2900.0, replicas=2, batch=4, profile_axis=0,
                                   **kw)
    assert a == base and b == base
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    prof = _check_case_profiles("outputs/solo", files)
    assert extra == sorted(prof + ["melt_pool_map_profile_rank0.csv"])
    reps = _read("outputs/solo/melt_pool_map_replicas_rank0.csv")
    assert [int(r["Step"]) < 60 for r in reps if r["replica"] == "1"] == [True, True]           # terminated early
    for root in ("plain", "solo", "grouped"):
        campaign.merge_melt_pool_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    assert len(_read("outputs/solo/melt_pool_map_profile.csv")) == 4
    assert len(_read("outputs/solo/melt_pool_map_profile_ensemble.csv")) == 2


def test_run_cet_sublattice_profile_rows(cet, tmp_path, monkeypatch):
    """The solo driver's cet_profile.csv: the profile of each row's labelling, as grain_profile_group reports it."""
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="p", verbose=False,
                                profile_axis=1, seed=3)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="q", verbose=False, seed=3)
    assert filecmp.cmp("outputs/p/metrics.csv", "outputs/q/metrics.csv", shallow=False)
    assert not os.path.exists("outputs/q/cet_profile.csv")
    rows = _read("outputs/p/cet_profile.csv")
    m = _read("outputs/p/metrics.csv")
    steps = [int(r["Step"]) for r in m]
    assert len(steps) >= 2 and [int(r["Step"]) for r in rows] == [s for s in steps for _ in range(24)]
    assert [int(r["Plane"]) for r in rows] == list(range(24)) * len(steps)
    for step, mr in zip(steps, m):
        sl = [r for r in rows if int(r["Step"]) == step]
        n_occ = int(mr["W_Count"]) + int(mr["Re_Count"]) + int(mr["C_Count"])
        assert sum(int(r["Solid"]) for r in sl) >= n_occ
