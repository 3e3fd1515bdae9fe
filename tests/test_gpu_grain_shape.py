"""GPU: grain-shape histograms (cet_grain_shape_group / cetkmc.grain_shape_group) against the NumPy reference of
tests/shaperef.py over the label volume of Context.grains(labels=True), after each kind of labelling (Context.grains:
arrival-order gid, metrics_group: site-order gid, the theta_only criterion), for groups of 1, 4 and 18 in either order,
with the default edges and with edges at elongations the reference attains; identities with the metrics row and the
profile; edge lattices, up to grains whose Q passes 2^64; non-interference with the cadence and sweeps; rejections;
and the drivers' shape files, solo against grouped."""
import ctypes as C
import filecmp
import os

import numpy as np
import pytest

import shaperef
from test_gpu_grain_profile import (EVERY, SEED, THR, _driver, _edge, _even, _half_grown, _label, _params, _read,
                                    _reference, _run, _same_snapshots, _same_subset, _same_tree, _snapshot,
                                    _terminating_replica, _upload)

pytestmark = pytest.mark.gpu


def _attained_edges(labels, n, axis):
    """Up to 62 edges placed at elongations the reference attains (shaperef, min_size 1): a grain whose A differed by
    one ulp from the reference's would change bin at one of them."""
    _sizes, a = shaperef.elongations(labels, axis, n)
    u = np.unique(a)
    if u.size == 0:
        return (1.0,)
    return tuple(float(x) for x in u[np.linspace(0, u.size - 1, min(62, u.size)).round().astype(int)].tolist())


def _check_group(cet, ctxs, kind):
    rows = _label(cet, ctxs, kind)
    nb = len(cet._lib.SHAPE_EDGES) + 2
    got = {ax: cet.grain_shape_group(ctxs, ax) for ax in range(3)}
    rev = {ax: cet.grain_shape_group(ctxs[::-1], ax)[::-1] for ax in range(3)}
    solo = {ax: np.stack([cet.grain_shape_group([c], ax)[0] for c in ctxs]) for ax in range(3)}
    prof = cet.grain_profile_group(ctxs, 2, THR)
    refs = [_reference(c, kind) for c in ctxs]                    # relabels (the same labelling): after the device calls
    for ax in range(3):
        assert got[ax].shape == (len(ctxs), 2, nb) and got[ax].dtype == np.int64
        assert np.array_equal(got[ax], rev[ax]) and np.array_equal(got[ax], solo[ax])
    for q, g in enumerate(refs):
        for ax in range(3):
            want = shaperef.grain_shape(g["labels"], ax, cet._lib.SHAPE_EDGES, cet._lib.SHAPE_MIN_SIZE, g["n"])
            assert np.array_equal(got[ax][q], want), (kind, q, ax)
            assert got[ax][q, 1].sum() == g["size"].sum() == prof[q, 0].sum()
            assert got[ax][q, 0].sum() == g["n"]
            if rows is not None:
                assert got[ax][q, 0].sum() == rows[q]["n_grains"] and got[ax][q, 1].sum() == rows[q]["size_sum"]
    # edges at attained elongations, min_size 1: every grain binned by its exact A
    _label(cet, ctxs, kind)
    for ax in range(3):
        edges = _attained_edges(refs[0]["labels"], refs[0]["n"], ax)
        h = cet.grain_shape_group(ctxs, ax, edges, 1)
        for q, g in enumerate(refs):
            assert np.array_equal(h[q], shaperef.grain_shape(g["labels"], ax, edges, 1, g["n"])), (kind, q, ax)
    return got


@pytest.mark.parametrize("L", [24, 30, 64, 96])
@pytest.mark.parametrize("kind", ["grains", "metrics", "theta"])
def test_shape_equals_reference(cet, L, kind):
    ctxs = [_half_grown(cet, L, 0)[0], _driver(cet, L, 0, 40), _half_grown(cet, L, 1)[0], _driver(cet, L, 1, 120)]
    try:
        got = _check_group(cet, ctxs, kind)
        assert got[2][:, 0, :-1].sum() > 0
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("kind", ["grains", "metrics"])
def test_shape_group_of_18(cet, kind):
    ctxs = [_half_grown(cet, 30, q)[0] for q in range(14)] + [_driver(cet, 30, q, 30 + 20 * q) for q in range(4)]
    try:
        _check_group(cet, ctxs, kind)
    finally:
        for c in ctxs:
            c.close()


def test_shape_driver_lattices_after_300_sweeps(cet):
    ctxs = [_driver(cet, 64, q, 300) for q in range(3)]
    try:
        got = _check_group(cet, ctxs, "metrics")
        assert (got[2][:, 0, 4:-1].sum(axis=1) > 0).all()                  # columnar grains (A >= 3) along the growth axis
    finally:
        for c in ctxs:
            c.close()


# -- edge lattices --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["empty", "one", "filling", "single_site", "pepper"])
@pytest.mark.parametrize("kind", ["grains", "metrics"])
def test_shape_edge_lattices(cet, name, kind):
    st, th, ph, n_expected = _edge(name)
    ctxs = [_upload(cet, st, th, ph), _upload(cet, st, th, ph)]
    try:
        got = _check_group(cet, ctxs, kind)
        n = ctxs[0].grains(0.5)["n"]
        assert n > 10 ** 5 if n_expected is None else n == n_expected
        if name == "empty":
            assert not any(got[ax].any() for ax in range(3))
        if name in ("one", "filling"):                                      # cubes of one parity: A = 1, bin 1
            for ax in range(3):
                assert got[ax][0, 0].tolist() == [0, n_expected] + [0] * 10
    finally:
        for c in ctxs:
            c.close()


def _uniform_moments(n, extents):
    """Moments of a grain whose marginal along each axis x is uniform over 0..extents[x]-1."""
    s = [n // e * (e * (e - 1) // 2) for e in extents]
    ss = [n // e * ((e - 1) * e * (2 * e - 1) // 6) for e in extents]
    return n, s, ss


@pytest.mark.parametrize("L, half", [(256, False), (400, True)])
def test_shape_large_grains(cet, L, half):
    """One grain, the even sites of a full 256^3 lattice (Q = 2^62 along every axis; with the 14-offset neighbourhood
    no grain holds both parities, so none reaches 2^64 at 256^3), and two grains, the even and the odd sites of the
    lower half (j < L / 2) of a 400^3 lattice (1.6e7 sites each, Q above 2^64): moments known in closed form."""
    st = _even(L) if not half else np.ones((L, L, L), np.int64)
    if half:
        st[:, L // 2:, :] = 0
    ctx = _upload(cet, st, np.full(st.shape, 0.3), np.full(st.shape, 1.1))
    del st
    try:
        g = ctx.grains(0.5)
        ext = (L, L // 2 if half else L, L)
        n = L * ext[1] * L // 2
        assert g["n"] == (2 if half else 1) and g["size"].tolist() == [n] * g["n"]
        mom = _uniform_moments(n, ext)
        qs = [shaperef.q_moment(mom[0], mom[1][x], mom[2][x]) for x in range(3)]
        assert max(qs) > (2 ** 64 if half else 2 ** 61)
        for ax in range(3):
            a = shaperef.elongation_of(*mom, ax)
            edges = (np.nextafter(a, 0.0), a, np.nextafter(a, np.inf))
            h = cet.grain_shape_group([ctx], ax, edges, 1)[0]
            assert h.tolist() == [[0, 0, g["n"], 0, 0], [0, 0, g["n"] * n, 0, 0]], (L, ax, a)
    finally:
        ctx.close()


# -- non-interference ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("philox", [False, True])
def test_shape_calls_change_nothing(cet, philox):
    from cetkmc import campaign
    a = [_half_grown(cet, 24, q) for q in range(4)]
    b = [_half_grown(cet, 24, q) for q in range(4)]
    ra = [dict(_run(c, q), shapes=[]) for q, (c, _, _) in enumerate(a)]
    rb = [_run(c, q) for q, (c, _, _) in enumerate(b)]
    try:
        for last in (EVERY, EVERY + 3, 2 * EVERY):
            campaign._cadence_group(ra, last, EVERY, philox, SEED, profile_axis=1, shape_axis=last % 3)
            cet.grain_shape_group([r["ctx"] for r in ra][::-1], 1, (1.0, 2.0), 1)             # extra calls in between
            campaign._cadence_group(rb, last, EVERY, philox, SEED, profile_axis=1)
            for x, y in zip(ra, rb):
                assert x["rows"][-1] == y["rows"][-1] and x["cet_detected"] == y["cet_detected"]
                assert np.array_equal(x["profiles"][-1][1], y["profiles"][-1][1])
                assert x["rng"][0] == y["rng"][0] and np.array_equal(x["rng"][1], y["rng"][1]) and x["rng"][2:] == y["rng"][2:]
                assert x["shapes"][-1][0] == last and x["shapes"][-1][1].shape == (2, 12)
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b], rates=False)
            ga = cet.sweep_run_group([c for c, _, _ in a], 6, [s for _, s, _ in a], [t for _, _, t in a])
            gb = cet.sweep_run_group([c for c, _, _ in b], 6, [s for _, s, _ in b], [t for _, _, t in b])
            assert ga == gb
            _same_snapshots(cet, [c for c, _, _ in a], [c for c, _, _ in b])
    finally:
        for c, _, _ in a + b:
            c.close()


# -- rejections ----------------------------------------------------------------------------------------------------

def _raw(cet, ctxs, axis, out, n=None, edges=(1.0, 2.0, 3.0), n_edges=None, min_size=8):
    """cet_grain_shape_group called directly (the binding's own checks bypassed): its return code."""
    h = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
    e = None if edges is None else np.ascontiguousarray(edges, np.float64)
    ptr = None if out is None else out.ctypes.data_as(C.POINTER(C.c_int64))
    return cet._lib.lib().cet_grain_shape_group(h, len(ctxs) if n is None else n, axis,
                                                None if e is None else e.ctypes.data_as(C.POINTER(C.c_double)),
                                                (0 if e is None else e.size) if n_edges is None else n_edges, min_size, ptr)


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
        out = np.full((70, 2, 64), -7, np.int64)
        sentinel = out.copy()
        for ctxs, axis, o, kw, match in (([a, fresh], 2, out, {}, "labell"),
                                         ([a, slab], 2, out, {}, "slab"),
                                         ([a, other], 2, out, {}, "L ="),
                                         ([a, b, a], 2, out, {}, "repeats"),
                                         ([a] * 65, 2, out, {}, "n_ctx"),
                                         ([a, b], 2, out, dict(n=0), "n_ctx"),
                                         ([a, b], 3, out, {}, "axis"),
                                         ([a, b], -1, out, {}, "axis"),
                                         ([a, b], 2, None, {}, "NULL"),
                                         ([a, b], 2, out, dict(edges=None, n_edges=3), "NULL"),
                                         ([a, b], 2, out, dict(n_edges=0), "n_edges"),
                                         ([a, b], 2, out, dict(edges=np.arange(1.0, 64.0)), "n_edges"),
                                         ([a, b], 2, out, dict(edges=(1.0, np.nan)), "finite"),
                                         ([a, b], 2, out, dict(edges=(1.0, np.inf)), "finite"),
                                         ([a, b], 2, out, dict(edges=(0.0, 1.0)), "finite"),
                                         ([a, b], 2, out, dict(edges=(2.0, 2.0)), "ascend"),
                                         ([a, b], 2, out, dict(edges=(3.0, 2.0)), "ascend"),
                                         ([a, b], 2, out, dict(min_size=0), "min_size")):
            assert _raw(cet, ctxs, axis, o, **kw) != 0
            assert match in cet._lib.lib().cet_last_error().decode()
            assert np.array_equal(out, sentinel)
        with pytest.raises(RuntimeError, match="labell"):
            cet.grain_shape_group([fresh], 0)
        for x, s in zip((a, b, fresh), before):
            t = _snapshot(cet, x, rates=False, labels=x is not fresh)
            for k in s:
                assert (s[k] == t[k]) if k == "clock" else np.array_equal(s[k], t[k], equal_nan=True), k
        for ax in range(3):
            assert np.array_equal(cet.grain_shape_group([a, b], ax), cet.grain_shape_group([a2, b2], ax))
        assert cet.sweep_run_group([a, b], 5, [sa, sb], [ta, tb]) == cet.sweep_run_group([a2, b2], 5, [sa2, sb2], [ta2, tb2])
        _same_snapshots(cet, [a, b], [a2, b2])
    finally:
        for x in (a, b, a2, b2, fresh, other, slab):
            x.close()


# -- the drivers -----------------------------------------------------------------------------------------------------

def _check_case_shapes(root, files):
    """Every metrics row of every case has its bins in grain_shape.csv, and the final histogram's sites sum to the
    occupied sites of the final profile."""
    from cetkmc import campaign
    shp = [f for f in files if f.endswith("/grain_shape.csv")]
    assert len(shp) == sum(f.endswith("/metrics.csv") for f in files if not f.startswith("plot_cet/"))
    for f in shp:
        rows = _read(os.path.join(root, f))
        steps = [int(r["Step"]) for r in _read(os.path.join(root, f.replace("grain_shape.csv", "metrics.csv")))]
        assert [int(r["Step"]) for r in rows] == [s for s in steps for _ in range(12)]
        _step, hist, edges = campaign.read_shape_csv(os.path.join(root, f))
        assert edges == campaign._lib.SHAPE_EDGES
        pf = os.path.join(root, f.replace("grain_shape.csv", "cet_profile.csv"))
        if os.path.exists(pf):
            assert hist[1].sum() == campaign.read_profile_csv(pf)[1][0].sum()
    return shp


GR = dict(L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3, seed=7)


def test_gr_sweep_shapes(cet, tmp_path, monkeypatch):
    from cetkmc import campaign, metrics
    monkeypatch.chdir(tmp_path)
    temps, nu_deps = [2700.0, 3000.0], [2e13, 1e14]
    _terminating_replica(monkeypatch, campaign, 3000.0)
    base, ens = campaign.run_gr_sweep(temps, nu_deps, output_root="plain", replicas=3, profile_axis=2, **GR)
    a, ens_a = campaign.run_gr_sweep(temps, nu_deps, output_root="solo", replicas=3, profile_axis=2, shape_axis=2, **GR)
    b, ens_b = campaign.run_gr_sweep(temps, nu_deps, output_root="grouped", replicas=3, batch=4, profile_axis=2,
                                     shape_axis=2, **GR)
    assert a == base and b == base and ens_a == ens and ens_b == ens
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    shp = _check_case_shapes("outputs/solo", files)
    assert len(shp) == 12 and extra == sorted(shp + ["cet_map_shape_rank0.csv"])
    for root in ("plain", "solo", "grouped"):
        campaign.merge_cet_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    rows = _read("outputs/solo/cet_map_shape.csv")
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP", "ColumnarVolumeFraction",
                                    "ColumnarGrainFraction", "ShapedGrains"]
    assert [(int(r["case"]), int(r["replica"])) for r in rows] == [(q, r) for q in range(4) for r in range(3)]
    for r in rows:
        p = f"outputs/solo/T{float(r['T_sub']):g}_R{float(r['NU_DEP']):g}" + ("" if r["replica"] == "0" else f"/rep{r['replica']}")
        _step, hist, edges = campaign.read_shape_csv(f"{p}/grain_shape.csv")
        s = metrics.grain_shape_summary(hist, edges)
        assert float(r["ColumnarVolumeFraction"]) == s["ColumnarVolumeFraction"] and int(r["ShapedGrains"]) == s["ShapedGrains"]
    ens_rows = _read("outputs/solo/cet_map_shape_ensemble.csv")
    assert len(ens_rows) == 4
    for q, e in enumerate(ens_rows):
        v = np.array([float(r["ColumnarVolumeFraction"]) for r in rows if int(r["case"]) == q])
        assert int(e["replicas"]) == 3 and float(e["ColumnarVolumeFraction_mean"]) == pytest.approx(np.mean(v), rel=1e-15)
        assert float(e["ColumnarVolumeFraction_se"]) == pytest.approx(np.std(v, ddof=1) / np.sqrt(3), rel=1e-12, abs=1e-300)


MAP = dict(L=24, n_sweeps=61, metrics_every=30, thermal_every=5, n_seeds=6, defect_fraction=3e-3, start=(12.0, 2.0),
           dt=1e-7)


def test_melt_pool_map_shapes(cet, tmp_path, monkeypatch):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    kw = dict(MAP, mask_stream="philox")
    powers, speeds = [150.0, 300.0], [1.0]
    _terminating_replica(monkeypatch, campaign, 2900.0)
    base = campaign.run_melt_pool_map(powers, speeds, output_root="plain", temp=2900.0, replicas=2, **kw)
    a = campaign.run_melt_pool_map(powers, speeds, output_root="solo", temp=2900.0, replicas=2, shape_axis=0, **kw)
    b = campaign.run_melt_pool_map(powers, speeds, output_root="grouped", temp=2900.0, replicas=2, batch=4, shape_axis=0,
                                   **kw)
    assert a == base and b == base
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    shp = _check_case_shapes("outputs/solo", files)
    assert extra == sorted(shp + ["melt_pool_map_shape_rank0.csv"])
    for root in ("plain", "solo", "grouped"):
        campaign.merge_melt_pool_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    assert len(_read("outputs/solo/melt_pool_map_shape.csv")) == 4
    assert len(_read("outputs/solo/melt_pool_map_shape_ensemble.csv")) == 2


def test_run_cet_sublattice_shape_rows(cet, tmp_path, monkeypatch):
    """The solo driver's grain_shape.csv: the histogram of each row's labelling; metrics.csv unchanged."""
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="p", verbose=False,
                                shape_axis=2, seed=3)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="q", verbose=False, seed=3)
    assert filecmp.cmp("outputs/p/metrics.csv", "outputs/q/metrics.csv", shallow=False)
    assert not os.path.exists("outputs/q/grain_shape.csv")
    rows = _read("outputs/p/grain_shape.csv")
    m = _read("outputs/p/metrics.csv")
    steps = [int(r["Step"]) for r in m]
    assert len(steps) >= 2 and [int(r["Step"]) for r in rows] == [s for s in steps for _ in range(12)]
    for step, mr in zip(steps, m):
        sl = [r for r in rows if int(r["Step"]) == step]
        assert sum(int(r["Grains"]) for r in sl) == int(float(mr["GrainCount"]))
