"""GPU: the front conditions (cet_front_group / cetkmc.front_group) against the NumPy reference of tests/frontref.py
over download(state=True, T=True), exactly (integers equal, doubles bit-equal with their NaN positions): at L = 24, 25,
30, 64 and 96 on every axis, on lattices built by upload and by init_group, after grouped sweeps with thermal steps,
after laser steps, on the wavy-front lattice, on empty and full lattices; groups of 1, 4 and 18 in either order and
solo; non-interference with sweeps, rows, profiles and shapes; rejections; the gradient of a fresh linear-T lattice;
and the drivers' front files, solo against grouped."""
import ctypes as C
import filecmp
import os

import numpy as np
import pytest

import frontref
from test_gpu_grain_profile import (EVERY, SEED, _driver, _half_grown, _read, _run, _same_snapshots, _same_subset,
                                    _same_tree, _snapshot, _terminating_replica, _upload)

pytestmark = pytest.mark.gpu


def _check(cet, ctxs):
    """front_group of the group, reversed and solo against the reference on every axis; returns the group's dicts."""
    snaps = [c.download(state=True, T=True) for c in ctxs]
    out = {}
    for ax in range(3):
        got = cet.front_group(ctxs, ax)
        rev = cet.front_group(ctxs[::-1], ax)
        solo = [cet.front_group([c], ax) for c in ctxs]
        n, L = len(ctxs), ctxs[0].shape[2]
        for k in ("front", "top", "T_front", "dT_front"):
            assert got[k].shape == (n, L, L)
            assert got[k].dtype == (np.int32 if k in ("front", "top") else np.float64)
        for q, s in enumerate(snaps):
            want = frontref.front(s["state"], s["T"], ax)
            for i, k in enumerate(("front", "top")):
                assert np.array_equal(got[k][q], want[i]), (q, ax, k)
                assert np.array_equal(rev[k][n - 1 - q], want[i]) and np.array_equal(solo[q][k][0], want[i])
            for i, k in ((2, "T_front"), (3, "dT_front")):
                b = frontref.bits(want[i])
                assert np.array_equal(frontref.bits(got[k][q]), b), (q, ax, k)
                assert np.array_equal(frontref.bits(rev[k][n - 1 - q]), b) and np.array_equal(frontref.bits(solo[q][k][0]), b)
        out[ax] = got
    return out


def _close(ctxs):
    for c in ctxs:
        c.close()


def _grouped_sweeps(cet, cases, n=6):
    """Grouped sweeps with thermal steps (thermal_every 5) of the (ctx, sp, tp) triples."""
    cet.sweep_run_group([c for c, _, _ in cases], n, [s for _, s, _ in cases], [t for _, _, t in cases])


@pytest.mark.parametrize("L", [24, 25, 30, 64, 96])
def test_front_equals_reference(cet, L):
    cases = [_half_grown(cet, L, q) for q in range(2)]
    ctxs = [c for c, _, _ in cases] + [_driver(cet, L, 0, 40), _driver(cet, L, 1, 120)]
    try:
        _check(cet, ctxs)
        _grouped_sweeps(cet, cases, 11)                                   # two thermal steps inside
        got = _check(cet, ctxs)
        assert got[2]["front"][2:].any() and (got[2]["top"] >= got[2]["front"]).all()
    finally:
        _close(ctxs)


def test_front_group_of_18(cet):
    cases = [_half_grown(cet, 30, q) for q in range(14)]
    ctxs = [c for c, _, _ in cases] + [_driver(cet, 30, q, 30 + 20 * q) for q in range(4)]
    try:
        _grouped_sweeps(cet, cases)
        _check(cet, ctxs)
        _check(cet, ctxs[:1])
        _check(cet, ctxs[5:9])
    finally:
        _close(ctxs)


def test_front_init_group_lattices(cet):
    """Generated lattices built on the device by init_group, fresh and after grouped sweeps."""
    from cetkmc import _host, campaign
    from cetkmc import kmc_simulation as ks
    from cetkmc._config import rate_params
    L = 32
    ctxs = [cet.Context(L=L) for _ in range(4)]
    try:
        for q, c in enumerate(ctxs):
            c.set_rate_params(rate_params(0.1, 1, 2, 3))
        cet.init_group(ctxs, [_host.initial_nuclei(L, 20, 2700.0 + 100 * q, 42 + q, 0.1) for q in range(4)])
        _check(cet, ctxs)
        sps, tps = zip(*[campaign._sweep_setup(L, 5 + q, 2700.0 + 100 * q, None, 0.1, 3e-3, ks.THERMAL_EVERY)
                         for q in range(4)])
        cet.sweep_run_group(ctxs, 60, list(sps), list(tps))
        _check(cet, ctxs)
    finally:
        _close(ctxs)


def test_front_after_laser_steps(cet):
    """After thermal_full_group laser steps T is no longer the initial linear profile."""
    from cetkmc._config import thermal_full_params
    from cetkmc.thermal_solver import laser_source_top
    cases = [_half_grown(cet, 48, q) for q in range(3)]
    ctxs = [c for c, _, _ in cases]
    try:
        T0 = ctxs[0].download(T=True)["T"]
        for c, sp, _ in cases:
            c.snapshot_state()
            sp.thermal_every = 0                                 # the laser step replaces the sweeps' thermal step
        for step in range(3):
            qs = [laser_source_top(48, (24.0, 6.0 * step), 150.0 + 100.0 * q, 1e-5, 0.4) for q in range(3)]
            cet.thermal_full_group(ctxs, [thermal_full_params(1e-7)] * 3, qs)
            for c, sp, _ in cases:
                c.sweep_run(4, sp, None)
        assert not np.array_equal(ctxs[0].download(T=True)["T"], T0)
        _check(cet, ctxs)
    finally:
        _close(ctxs)


def test_front_wavy_and_edge_lattices(cet):
    from cetkmc import _synth
    L = 40
    ctxs = []
    try:
        for fill in (1.0, 0.5):                         # the wavy front k < L/2 + 8 sin(2 pi i / L), dense and sparse
            packed, th, ph, T = _synth.half_grown(L, seed=9, grain=4, fill=fill)
            st, df = _synth.unpack(packed)
            c = cet.Context(L=L)
            c.upload(state=st, theta=th, phi=ph, T=T, defects=df)
            ctxs.append(c)
        zero = np.zeros((L,) * 3)
        ctxs.append(_upload(cet, np.zeros((L,) * 3, np.int64), zero, zero))
        ctxs.append(_upload(cet, np.ones((L,) * 3, np.int64), np.full((L,) * 3, 0.3), np.full((L,) * 3, 1.1)))
        got = _check(cet, ctxs)
        i = np.arange(L)
        assert np.array_equal(got[2]["front"][0], np.broadcast_to(np.ceil(L / 2 + 8 * np.sin(2 * np.pi * i / L))[:, None],
                                                                  (L, L)).astype(np.int32))
        for ax in range(3):
            assert not got[ax]["front"][2].any() and not got[ax]["top"][2].any()
            assert (got[ax]["front"][3] == L).all() and np.isnan(got[ax]["T_front"][3]).all()
            assert np.isnan(got[ax]["dT_front"][2]).all() and (got[ax]["T_front"][2] == 2900.0).all()
    finally:
        _close(ctxs)


def test_front_gradient_of_a_fresh_linear_lattice(cet):
    """On the generated lattice before any sweep, T is linear along k: G_Front is the nominal G."""
    from cetkmc import campaign, metrics
    from cetkmc._config import constants, rate_params
    L = 64
    for temp in (2600.0, 3000.0):
        np.random.seed(3)
        ctx = cet.Context(L=L)
        try:
            ctx.set_rate_params(rate_params(0.1, 1, 2, 3))
            campaign._upload_initial(ctx, L, 20, temp, 0.1, None, 0, L)
            f = cet.front_group([ctx], 2)
            s = metrics.front_summary(f["front"][0], f["top"][0], f["T_front"][0], f["dT_front"][0])
            G = campaign._gr(L, temp, 1e13)[0]
            assert s["GradColumns"] > 0 and s["G_Front"] == pytest.approx(G, rel=1e-12)
            assert s["FrontColumns"] == L * L and s["Undercooling"] > 0
            assert s["Undercooling"] == constants.T_MELT - s["T_Front"]
        finally:
            ctx.close()


# -- non-interference ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("philox", [False, True])
def test_front_calls_change_nothing(cet, philox):
    from cetkmc import campaign
    a = [_half_grown(cet, 24, q) for q in range(4)]
    b = [_half_grown(cet, 24, q) for q in range(4)]
    ra = [dict(_run(c, q), shapes=[], fronts=[]) for q, (c, _, _) in enumerate(a)]
    rb = [dict(_run(c, q), shapes=[]) for q, (c, _, _) in enumerate(b)]
    try:
        for last in (EVERY, EVERY + 3, 2 * EVERY):
            cet.front_group([r["ctx"] for r in ra][::-1], 0)                                  # extra calls in between
            campaign._cadence_group(ra, last, EVERY, philox, SEED, profile_axis=1, shape_axis=2, front_axis=last % 3)
            cet.front_group([r["ctx"] for r in ra], 1)
            campaign._cadence_group(rb, last, EVERY, philox, SEED, profile_axis=1, shape_axis=2)
            for x, y in zip(ra, rb):
                assert x["rows"][-1] == y["rows"][-1] and x["cet_detected"] == y["cet_detected"]
                assert np.array_equal(x["profiles"][-1][1], y["profiles"][-1][1])
                assert np.array_equal(x["shapes"][-1][1], y["shapes"][-1][1])
                assert x["rng"][0] == y["rng"][0] and np.array_equal(x["rng"][1], y["rng"][1]) and x["rng"][2:] == y["rng"][2:]
                assert x["fronts"][-1][0] == last and x["fronts"][-1][1] == x["total_time"]
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b], rates=False)
            for x, y in zip(a, b):
                assert np.array_equal(x[0].download(T=True)["T"], y[0].download(T=True)["T"], equal_nan=True)
            ga = cet.sweep_run_group([c for c, _, _ in a], 6, [s for _, s, _ in a], [t for _, _, t in a])
            gb = cet.sweep_run_group([c for c, _, _ in b], 6, [s for _, s, _ in b], [t for _, _, t in b])
            assert ga == gb
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b])
    finally:
        for c, _, _ in a + b:
            c.close()


# -- rejections ----------------------------------------------------------------------------------------------------

def _raw(cet, ctxs, axis, fr, tm, n=None):
    """cet_front_group called directly (the binding's own checks bypassed): its return code."""
    h = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
    return cet._lib.lib().cet_front_group(h, len(ctxs) if n is None else n, axis,
                                          None if fr is None else fr.ctypes.data_as(C.POINTER(C.c_int32)),
                                          None if tm is None else tm.ctypes.data_as(C.POINTER(C.c_double)))


def test_rejections_leave_everything_untouched(cet):
    a, sa, ta = _half_grown(cet, 24, 0)
    b, sb, tb = _half_grown(cet, 24, 1)
    a2, sa2, ta2 = _half_grown(cet, 24, 0)
    b2, sb2, tb2 = _half_grown(cet, 24, 1)
    other = _upload(cet, np.ones((25,) * 3, np.int64), np.full((25,) * 3, 0.3), np.full((25,) * 3, 1.1))
    slab = cet.Context(L=24, i_begin=0, i_end=12)
    try:
        before = [_snapshot(cet, x, rates=False, labels=False) for x in (a, b)]
        fr = np.full(70 * 2 * 24 * 24, -7, np.int32)
        tm = np.full(70 * 2 * 24 * 24, -7.0)
        f0, t0 = fr.copy(), tm.copy()
        for ctxs, axis, f, t, kw, match in (([a, slab], 2, fr, tm, {}, "slab"),
                                            ([a, other], 2, fr, tm, {}, "L ="),
                                            ([a, b, a], 2, fr, tm, {}, "repeats"),
                                            ([a] * 65, 2, fr, tm, {}, "n_ctx"),
                                            ([a, b], 2, fr, tm, dict(n=0), "n_ctx"),
                                            ([a, b], 3, fr, tm, {}, "axis"),
                                            ([a, b], -1, fr, tm, {}, "axis"),
                                            ([a, b], 2, None, tm, {}, "NULL"),
                                            ([a, b], 2, fr, None, {}, "NULL")):
            assert _raw(cet, ctxs, axis, f, t, **kw) != 0
            assert match in cet._lib.lib().cet_last_error().decode()
            assert np.array_equal(fr, f0) and np.array_equal(tm, t0)
        with pytest.raises(RuntimeError, match="slab"):
            cet.front_group([slab], 0)
        with pytest.raises(RuntimeError, match="n_ctx"):
            cet.front_group([], 0)
        for x, s in zip((a, b), before):
            t = _snapshot(cet, x, rates=False, labels=False)
            for k in s:
                assert (s[k] == t[k]) if k == "clock" else np.array_equal(s[k], t[k], equal_nan=True), k
        assert cet.sweep_run_group([a, b], 5, [sa, sb], [ta, tb]) == cet.sweep_run_group([a2, b2], 5, [sa2, sb2], [ta2, tb2])
        for x, y in ((a, a2), (b, b2)):                                 # never labelled: no label volume to compare
            sx, sy = _snapshot(cet, x, labels=False), _snapshot(cet, y, labels=False)
            for k in sx:
                assert (sx[k] == sy[k]) if k == "clock" else np.array_equal(sx[k], sy[k], equal_nan=True), k
    finally:
        for x in (a, b, a2, b2, other, slab):
            x.close()


# -- the drivers -----------------------------------------------------------------------------------------------------

def _check_case_fronts(root, files):
    """Every metrics row of every case has its row in front.csv, with the same Step and Time."""
    from cetkmc import campaign
    fr = [f for f in files if f.endswith("/front.csv")]
    assert len(fr) == sum(f.endswith("/metrics.csv") for f in files if not f.startswith("plot_cet/"))
    for f in fr:
        rows = campaign.read_front_csv(os.path.join(root, f))
        m = _read(os.path.join(root, f.replace("front.csv", "metrics.csv")))
        assert [(r["Step"], r["Time"]) for r in rows] == [(int(r["Step"]), float(r["Time"])) for r in m]
        assert rows[0]["V_Front"] == ""
    return fr


GR = dict(L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3, seed=7)


def test_gr_sweep_fronts(cet, tmp_path, monkeypatch):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    temps, nu_deps = [2700.0, 3000.0], [2e13, 1e14]
    _terminating_replica(monkeypatch, campaign, 3000.0)
    base, ens = campaign.run_gr_sweep(temps, nu_deps, output_root="plain", replicas=3, shape_axis=2, **GR)
    a, ens_a = campaign.run_gr_sweep(temps, nu_deps, output_root="solo", replicas=3, shape_axis=2, front_axis=2, **GR)
    b, ens_b = campaign.run_gr_sweep(temps, nu_deps, output_root="grouped", replicas=3, batch=4, shape_axis=2,
                                     front_axis=2, **GR)
    assert a == base and b == base and ens_a == ens and ens_b == ens
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    fr = _check_case_fronts("outputs/solo", files)
    assert len(fr) == 12 and extra == sorted(fr + ["cet_map_front_rank0.csv"])
    for root in ("plain", "solo", "grouped"):
        campaign.merge_cet_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    rows = _read("outputs/solo/cet_map_front.csv")
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP", "G", "R", "G_Front", "V_Front", "G_over_V",
                                    "Undercooling", "FrontMean", "FrontRMS"]
    assert [(int(r["case"]), int(r["replica"])) for r in rows] == [(q, r) for q in range(4) for r in range(3)]
    maps = _read("outputs/solo/cet_map.csv")
    for r in rows:
        m = maps[int(r["case"])]
        assert (r["G"], r["R"]) == (m["G"], m["R"])
        p = f"outputs/solo/T{float(r['T_sub']):g}_R{float(r['NU_DEP']):g}" + ("" if r["replica"] == "0" else f"/rep{r['replica']}")
        fc = campaign.read_front_csv(f"{p}/front.csv")
        assert r["G_Front"] == ("" if fc[-1]["G_Front"] == "" else repr(fc[-1]["G_Front"]))
    assert len(_read("outputs/solo/cet_map_front_ensemble.csv")) == 4


MAP = dict(L=24, n_sweeps=61, metrics_every=30, thermal_every=5, n_seeds=6, defect_fraction=3e-3, start=(12.0, 2.0),
           dt=1e-7)


def test_melt_pool_map_fronts(cet, tmp_path, monkeypatch):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    kw = dict(MAP, mask_stream="philox")
    powers, speeds = [150.0, 300.0], [1.0]
    _terminating_replica(monkeypatch, campaign, 2900.0)
    base = campaign.run_melt_pool_map(powers, speeds, output_root="plain", temp=2900.0, replicas=2, **kw)
    a = campaign.run_melt_pool_map(powers, speeds, output_root="solo", temp=2900.0, replicas=2, front_axis=2, **kw)
    b = campaign.run_melt_pool_map(powers, speeds, output_root="grouped", temp=2900.0, replicas=2, batch=4, front_axis=2,
                                   **kw)
    assert a == base and b == base
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    fr = _check_case_fronts("outputs/solo", files)
    assert extra == sorted(fr + ["melt_pool_map_front_rank0.csv"])
    for root in ("plain", "solo", "grouped"):
        campaign.merge_melt_pool_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    assert len(_read("outputs/solo/melt_pool_map_front.csv")) == 4
    assert len(_read("outputs/solo/melt_pool_map_front_ensemble.csv")) == 2


def test_run_cet_sublattice_front_rows(cet, tmp_path, monkeypatch):
    """The solo driver's front.csv: one row per metrics row; metrics.csv unchanged."""
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="p", verbose=False,
                                front_axis=2, seed=3)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="q", verbose=False, seed=3)
    assert filecmp.cmp("outputs/p/metrics.csv", "outputs/q/metrics.csv", shallow=False)
    assert not os.path.exists("outputs/q/front.csv")
    rows = campaign.read_front_csv("outputs/p/front.csv")
    m = _read("outputs/p/metrics.csv")
    assert [(r["Step"], r["Time"]) for r in rows] == [(int(r["Step"]), float(r["Time"])) for r in m]
    assert len(rows) >= 2 and rows[0]["V_Front"] == "" and all(r["V_Front"] != "" for r in rows[1:])
