"""GPU: the per-plane bond counts and boundary misorientation (cet_boundary_group / cetkmc.boundary_group) against the
NumPy reference of tests/boundaryref.py over the label volume of the last labelling and the resident orientation
vectors read through device_ptr(5), exactly: at L = 24, 25, 30, 64 and 96 on every axis with the default edges and
with 31 edges, after each kind of labelling (Context.grains, metrics_group), on lattices built by upload and by
init_group, after grouped sweeps and a relabel; groups of 1, 4 and 18 in either order and solo; no boundary bond below
the labelling's threshold; non-interference with sweeps, rows, profiles, shapes, fronts and texture; rejections; and
the drivers' boundary files, solo against grouped."""
import ctypes as C
import filecmp
import os

import numpy as np
import pytest

import boundaryref
import textureref
from test_gpu_grain_profile import (EVERY, SEED, _driver, _half_grown, _label, _labels, _read, _run, _same_snapshots,
                                    _same_subset, _same_tree, _snapshot, _terminating_replica)
from test_gpu_init_group import _dev_bytes
from test_gpu_texture import EDGES_31

pytestmark = pytest.mark.gpu


def _check(cet, ctxs, edges_deg=None):
    """boundary_group of the group, reversed and solo against the reference on every axis over each context's last
    labelling; returns the group's results per axis."""
    from cetkmc import _lib
    kw = {} if edges_deg is None else dict(edges_deg=edges_deg)
    c_edges = _lib._texture_edges("t", _lib.BOUNDARY_EDGES_DEG if edges_deg is None else edges_deg)
    L, n = ctxs[0].shape[2], len(ctxs)
    snaps = [(_labels(cet, c), textureref.vectors(_dev_bytes(*c.device_ptr(5)), L)) for c in ctxs]
    out = {}
    for ax in range(3):
        got = cet.boundary_group(ctxs, ax, **kw)
        rev = cet.boundary_group(ctxs[::-1], ax, **kw)
        solo = [cet.boundary_group([c], ax, **kw) for c in ctxs]
        assert got[0].shape == (n, L, 7, 3) and got[1].shape == (n, L, c_edges.size + 1) and got[2].shape == (n, L)
        for q, (lab, v) in enumerate(snaps):
            want = boundaryref.split(boundaryref.table(lab, v, ax, c_edges))
            for i in range(3):
                assert np.array_equal(got[i][q], want[i]), (q, ax, i)
                assert np.array_equal(rev[i][n - 1 - q], want[i]) and np.array_equal(solo[q][i][0], want[i])
        out[ax] = got
    return out


def _close(ctxs):
    for c in ctxs:
        c.close()


def _no_boundary_below_threshold(got):
    """With the default edges (10-degree bins) the bins 0-10 and 10-20 lie wholly below 0.5 rad (28.6 degrees)."""
    for ax in range(3):
        assert not got[ax][1][:, :, :2].any()


@pytest.mark.parametrize("L", [24, 25, 30, 64, 96])
def test_boundary_equals_reference(cet, L):
    cases = [_half_grown(cet, L, q) for q in range(2)]
    ctxs = [c for c, _, _ in cases] + [_driver(cet, L, 0, 40), _driver(cet, L, 1, 120)]
    try:
        _label(cet, ctxs, "metrics")
        got = _check(cet, ctxs)
        _no_boundary_below_threshold(got)
        _check(cet, ctxs, EDGES_31)
        _label(cet, ctxs, "grains")
        _check(cet, ctxs)
        cet.sweep_run_group([c for c, _, _ in cases], 11, [s for _, s, _ in cases], [t for _, _, t in cases])
        _label(cet, ctxs, "metrics")                                      # relabel after the sweeps
        got = _check(cet, ctxs)
        _check(cet, ctxs, EDGES_31)
        _no_boundary_below_threshold(got)
        for ax in range(3):
            b = got[ax][0]
            assert b[..., 1].sum() > 0 and (b.sum(axis=(1, 2, 3)) == got[0][0].sum(axis=(1, 2, 3))).all()
            assert (got[ax][1].sum(axis=(1, 2)) == b[..., 1].sum(axis=(1, 2))).all()
    finally:
        _close(ctxs)


def test_boundary_group_of_18(cet):
    cases = [_half_grown(cet, 30, q) for q in range(14)]
    ctxs = [c for c, _, _ in cases] + [_driver(cet, 30, q, 30 + 20 * q) for q in range(4)]
    try:
        _label(cet, ctxs, "metrics")
        _check(cet, ctxs)
        _check(cet, ctxs, EDGES_31)
        _check(cet, ctxs[5:9])
        _check(cet, ctxs[:1], EDGES_31)
    finally:
        _close(ctxs)


def test_boundary_init_group_lattices(cet):
    """Generated lattices built on the device by init_group, fresh and after grouped sweeps."""
    from cetkmc import _host, campaign
    from cetkmc import kmc_simulation as ks
    from cetkmc._config import rate_params
    L = 32
    ctxs = [cet.Context(L=L) for _ in range(4)]
    try:
        for c in ctxs:
            c.set_rate_params(rate_params(0.1, 1, 2, 3))
        cet.init_group(ctxs, [_host.initial_nuclei(L, 20, 2700.0 + 100 * q, 42 + q, 0.1) for q in range(4)])
        _label(cet, ctxs, "metrics")
        _check(cet, ctxs)
        sps, tps = zip(*[campaign._sweep_setup(L, 5 + q, 2700.0 + 100 * q, None, 0.1, 3e-3, ks.THERMAL_EVERY)
                         for q in range(4)])
        cet.sweep_run_group(ctxs, 60, list(sps), list(tps))
        _label(cet, ctxs, "grains")
        _check(cet, ctxs, EDGES_31)
    finally:
        _close(ctxs)


# -- non-interference ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("philox", [False, True])
def test_boundary_calls_change_nothing(cet, philox):
    from cetkmc import campaign
    a = [_half_grown(cet, 24, q) for q in range(4)]
    b = [_half_grown(cet, 24, q) for q in range(4)]
    ra = [dict(_run(c, q), shapes=[], fronts=[], textures=[], boundaries=[]) for q, (c, _, _) in enumerate(a)]
    rb = [dict(_run(c, q), shapes=[], fronts=[], textures=[]) for q, (c, _, _) in enumerate(b)]
    try:
        for last in (EVERY, EVERY + 3, 2 * EVERY):
            campaign._cadence_group(ra, last, EVERY, philox, SEED, profile_axis=1, shape_axis=2, front_axis=2,
                                    texture_axis=2, boundary_axis=last % 3)
            cet.boundary_group([r["ctx"] for r in ra][::-1], 0, EDGES_31)                 # extra calls in between
            campaign._cadence_group(rb, last, EVERY, philox, SEED, profile_axis=1, shape_axis=2, front_axis=2,
                                    texture_axis=2)
            for x, y in zip(ra, rb):
                assert x["rows"][-1] == y["rows"][-1] and x["cet_detected"] == y["cet_detected"]
                assert np.array_equal(x["profiles"][-1][1], y["profiles"][-1][1])
                assert np.array_equal(x["shapes"][-1][1], y["shapes"][-1][1])
                assert x["fronts"][-1] == y["fronts"][-1]
                assert all(np.array_equal(u, w) for u, w in zip(x["textures"][-1][1:], y["textures"][-1][1:]))
                assert x["rng"][0] == y["rng"][0] and np.array_equal(x["rng"][1], y["rng"][1]) and x["rng"][2:] == y["rng"][2:]
                assert x["boundaries"][-1][0] == last and x["boundaries"][-1][2].shape == (24, 18)
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b], rates=False)
            for x, y in zip(a, b):
                assert np.array_equal(_dev_bytes(*x[0].device_ptr(5)), _dev_bytes(*y[0].device_ptr(5)))
                assert np.array_equal(x[0].download(T=True)["T"], y[0].download(T=True)["T"], equal_nan=True)
            ga = cet.sweep_run_group([c for c, _, _ in a], 6, [s for _, s, _ in a], [t for _, _, t in a])
            gb = cet.sweep_run_group([c for c, _, _ in b], 6, [s for _, s, _ in b], [t for _, _, t in b])
            assert ga == gb
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b])
    finally:
        for c, _, _ in a + b:
            c.close()


# -- rejections ----------------------------------------------------------------------------------------------------

def _raw(cet, ctxs, axis, edges, out, n=None, m=None):
    """cet_boundary_group called directly (the binding's own checks bypassed): its return code."""
    h = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
    e = None if edges is None else np.ascontiguousarray(edges, np.float64)
    return cet._lib.lib().cet_boundary_group(h, len(ctxs) if n is None else n, axis,
                                             None if e is None else e.ctypes.data_as(C.POINTER(C.c_double)),
                                             (0 if e is None else e.size) if m is None else m,
                                             None if out is None else out.ctypes.data_as(C.POINTER(C.c_int64)))


def test_rejections_leave_everything_untouched(cet):
    a, sa, ta = _half_grown(cet, 24, 0)
    b, sb, tb = _half_grown(cet, 24, 1)
    a2, sa2, ta2 = _half_grown(cet, 24, 0)
    b2, sb2, tb2 = _half_grown(cet, 24, 1)
    fresh, _, _ = _half_grown(cet, 24, 2)                                   # never labelled
    slab = cet.Context(L=24, i_begin=0, i_end=12)
    good = np.array([-0.5, 0.0, 0.5])
    try:
        for x in (a, b, a2, b2):
            x.grains(0.5)
        before = [_snapshot(cet, x, rates=False) for x in (a, b)]
        out = np.full(70 * 24 * 60, -7, np.int64)
        o0 = out.copy()
        for ctxs, axis, e, kw, match in (([a, slab], 2, good, {}, "slab"),
                                         ([a, b, a], 2, good, {}, "repeats"),
                                         ([a] * 65, 2, good, {}, "n_ctx"),
                                         ([a, b], 2, good, dict(n=0), "n_ctx"),
                                         ([a, b], 3, good, {}, "axis"),
                                         ([a, b], -1, good, {}, "axis"),
                                         ([a, b], 2, None, {}, "NULL"),
                                         ([a, b], 2, np.zeros(0), dict(m=0), "n_edges"),
                                         ([a, b], 2, np.linspace(-0.9, 0.9, 32), {}, "n_edges"),
                                         ([a, b], 2, np.array([0.5, 0.0]), {}, "ascend"),
                                         ([a, b], 2, np.array([0.0, 0.0]), {}, "ascend"),
                                         ([a, b], 2, np.array([0.0, np.nan]), {}, "finite"),
                                         ([a, b], 2, np.array([-1.5, 0.0]), {}, "[-1, 1]"),
                                         ([a, b], 2, np.array([0.0, np.inf]), {}, "finite"),
                                         ([a, fresh], 2, good, {}, "context 1 has no labelling")):
            assert _raw(cet, ctxs, axis, e, out, **kw) != 0
            assert match in cet._lib.lib().cet_last_error().decode()
            assert np.array_equal(out, o0)
        assert _raw(cet, [a, b], 2, good, None) != 0 and "NULL" in cet._lib.lib().cet_last_error().decode()
        with pytest.raises(RuntimeError, match="slab"):
            cet.boundary_group([slab], 0)
        with pytest.raises(RuntimeError, match="no labelling"):
            cet.boundary_group([fresh], 0)
        for x, s in zip((a, b), before):
            t = _snapshot(cet, x, rates=False)
            for k in s:
                assert (s[k] == t[k]) if k == "clock" else np.array_equal(s[k], t[k], equal_nan=True), k
        assert cet.sweep_run_group([a, b], 5, [sa, sb], [ta, tb]) == cet.sweep_run_group([a2, b2], 5, [sa2, sb2], [ta2, tb2])
        for x, y in ((a, a2), (b, b2)):
            sx, sy = _snapshot(cet, x), _snapshot(cet, y)
            for k in sx:
                assert (sx[k] == sy[k]) if k == "clock" else np.array_equal(sx[k], sy[k], equal_nan=True), k
    finally:
        for x in (a, b, a2, b2, fresh, slab):
            x.close()


def test_rejects_a_table_over_the_shared_memory_limit(cet):
    """L = 1056 with 31 edges: a table of 1056 (8 + 4 * 53) + 248 bytes = 232 568 bytes, over the B200's 232 448-byte
    opt-in; the context is never labelled, so the table check comes first.  Needs about 90 GB of free device memory."""
    import torch
    L = 1056
    if torch.cuda.mem_get_info()[0] < 100 * 2 ** 30:
        pytest.skip("needs about 90 GB of free device memory")
    ctx = cet.Context(L=L)
    try:
        out = np.full(16, -7, np.int64)
        assert _raw(cet, [ctx], 2, np.linspace(-0.9, 0.9, 31), out) != 0
        msg = cet._lib.lib().cet_last_error().decode()
        assert "L = 1056" in msg and "m = 31" in msg and "232568 bytes" in msg
        assert (out == -7).all()
    finally:
        ctx.close()


# -- the drivers -----------------------------------------------------------------------------------------------------

def _check_case_boundaries(root, files, L=24):
    """Every metrics row of every case has its L planes in boundaries.csv, and each plane's bins hold its boundary bonds."""
    from cetkmc import campaign
    bx = [f for f in files if f.endswith("/boundaries.csv")]
    assert len(bx) == sum(f.endswith("/metrics.csv") for f in files if not f.startswith("plot_cet/"))
    for f in bx:
        _edges, recs = campaign.read_boundary_csv(os.path.join(root, f))
        m = _read(os.path.join(root, f.replace("boundaries.csv", "metrics.csv")))
        assert [r[0] for r in recs] == [int(r["Step"]) for r in m]
        assert all(r[1].shape == (L, 7, 3) and r[2].shape == (L, 18) for r in recs)
        assert all((r[2].sum(1) == r[1][:, :, 1].sum(1)).all() for r in recs)
        assert all(not r[2][:, :2].any() for r in recs)
    return bx


GR = dict(L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3, seed=7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_gr_sweep_boundaries(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign, metrics
    monkeypatch.chdir(tmp_path)
    kw = dict(GR, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    temps, nu_deps = [2700.0, 3000.0], [2e13, 1e14]
    _terminating_replica(monkeypatch, campaign, 3000.0)
    base, ens = campaign.run_gr_sweep(temps, nu_deps, output_root="plain", replicas=3, texture_axis=2, **kw)
    a, ens_a = campaign.run_gr_sweep(temps, nu_deps, output_root="solo", replicas=3, texture_axis=2, boundary_axis=2, **kw)
    b, ens_b = campaign.run_gr_sweep(temps, nu_deps, output_root="grouped", replicas=3, batch=4, texture_axis=2,
                                     boundary_axis=2, **kw)
    assert a == base and b == base and ens_a == ens and ens_b == ens
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    bx = _check_case_boundaries("outputs/solo", files)
    assert len(bx) == 12 and extra == sorted(bx + ["cet_map_boundary_rank0.csv"])
    reps = _read("outputs/solo/cet_map_replicas_rank0.csv")
    assert any(int(r["Step"]) < 60 for r in reps if r["replica"] == "1")                        # terminated early
    for root in ("plain", "solo", "grouped"):
        campaign.merge_cet_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    rows = _read("outputs/solo/cet_map_boundary.csv")
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP"] + list(metrics.BOUNDARY_COLUMNS)
    assert [(int(r["case"]), int(r["replica"])) for r in rows] == [(q, r) for q in range(4) for r in range(3)]
    for r in rows:
        p = f"outputs/solo/T{float(r['T_sub']):g}_R{float(r['NU_DEP']):g}" + ("" if r["replica"] == "0" else f"/rep{r['replica']}")
        edges, recs = campaign.read_boundary_csv(f"{p}/boundaries.csv")
        s = metrics.boundary_summary(*recs[-1][1:], 2, edges)
        assert int(r["BoundaryBonds"]) == s["BoundaryBonds"] and r["InterceptAlong"] == repr(s["InterceptAlong"])
    assert len(_read("outputs/solo/cet_map_boundary_ensemble.csv")) == 4


MAP = dict(L=24, n_sweeps=61, metrics_every=30, thermal_every=5, n_seeds=6, defect_fraction=3e-3, start=(12.0, 2.0),
           dt=1e-7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_melt_pool_map_boundaries(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    kw = dict(MAP, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    powers, speeds = [150.0, 300.0], [1.0]
    _terminating_replica(monkeypatch, campaign, 2900.0)
    base = campaign.run_melt_pool_map(powers, speeds, output_root="plain", temp=2900.0, replicas=2, **kw)
    a = campaign.run_melt_pool_map(powers, speeds, output_root="solo", temp=2900.0, replicas=2, boundary_axis=2, **kw)
    b = campaign.run_melt_pool_map(powers, speeds, output_root="grouped", temp=2900.0, replicas=2, batch=4,
                                   boundary_axis=2, **kw)
    assert a == base and b == base
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    bx = _check_case_boundaries("outputs/solo", files)
    assert extra == sorted(bx + ["melt_pool_map_boundary_rank0.csv"])
    reps = _read("outputs/solo/melt_pool_map_replicas_rank0.csv")
    assert [int(r["Step"]) < 60 for r in reps if r["replica"] == "1"] == [True, True]           # terminated early
    for root in ("plain", "solo", "grouped"):
        campaign.merge_melt_pool_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    assert len(_read("outputs/solo/melt_pool_map_boundary.csv")) == 4
    assert len(_read("outputs/solo/melt_pool_map_boundary_ensemble.csv")) == 2


def test_run_cet_sublattice_boundary_rows(cet, tmp_path, monkeypatch):
    """The solo driver's boundaries.csv: one record per metrics row; metrics.csv unchanged; every record's solid bonds
    join sites the row's labelling counted."""
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="p", verbose=False,
                                boundary_axis=1, seed=3)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="q", verbose=False, seed=3)
    assert filecmp.cmp("outputs/p/metrics.csv", "outputs/q/metrics.csv", shallow=False)
    assert not os.path.exists("outputs/q/boundaries.csv")
    edges, recs = campaign.read_boundary_csv("outputs/p/boundaries.csv")
    m = _read("outputs/p/metrics.csv")
    assert edges == tuple(float(x) for x in cet._lib.BOUNDARY_EDGES_DEG)
    assert [r[0] for r in recs] == [int(r["Step"]) for r in m] and len(recs) >= 2
    assert all(r[1][:, :, 0].sum() > 0 and r[1][:, :, 1].sum() > 0 for r in recs)
