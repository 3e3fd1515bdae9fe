"""GPU: the per-plane orientation histograms (cet_texture_group / cetkmc.texture_group) against the NumPy reference of
tests/textureref.py over download_packed() and the resident orientation vectors read through device_ptr(5), exactly:
at L = 24, 25, 30, 64 and 96 on every axis with the default edges and with 31 edges, at L = 512 (a table past 48 KB
of shared memory), on lattices built by upload and by init_group, after grouped sweeps with thermal steps and after
laser steps; groups of 1, 4 and 18 in either order and solo; non-interference with sweeps, rows, profiles, shapes and
fronts; rejections; and the drivers' texture files, solo against grouped."""
import ctypes as C
import filecmp
import os

import numpy as np
import pytest

import textureref
from test_gpu_grain_profile import (EVERY, SEED, _driver, _half_grown, _read, _run, _same_snapshots, _same_subset,
                                    _same_tree, _snapshot, _terminating_replica, _upload)
from test_gpu_init_group import _dev_bytes

pytestmark = pytest.mark.gpu

EDGES_31 = tuple(5.0 * np.arange(1, 32) + 1.25)                  # 31 edges, 6.25 .. 156.25 degrees


def _check(cet, ctxs, edges_deg=None):
    """texture_group of the group, reversed and solo against the reference on every axis; returns the group's
    results per axis."""
    from cetkmc import _lib
    kw = {} if edges_deg is None else dict(edges_deg=edges_deg)
    c_edges = _lib._texture_edges("t", _lib.TEXTURE_EDGES_DEG if edges_deg is None else edges_deg)
    L, n = ctxs[0].shape[2], len(ctxs)
    snaps = [(c.download_packed(), textureref.vectors(_dev_bytes(*c.device_ptr(5)), L)) for c in ctxs]
    out = {}
    for ax in range(3):
        got = cet.texture_group(ctxs, ax, **kw)
        rev = cet.texture_group(ctxs[::-1], ax, **kw)
        solo = [cet.texture_group([c], ax, **kw) for c in ctxs]
        assert got[0].shape == (n, L, c_edges.size + 1) and got[1].shape == got[2].shape == (n, L)
        for q, (packed, v) in enumerate(snaps):
            want = textureref.split(textureref.table(packed, v, ax, c_edges))
            for i in range(3):
                assert np.array_equal(got[i][q], want[i]), (q, ax, i)
                assert np.array_equal(rev[i][n - 1 - q], want[i]) and np.array_equal(solo[q][i][0], want[i])
        out[ax] = got
    return out


def _close(ctxs):
    for c in ctxs:
        c.close()


def _grouped_sweeps(cet, cases, n=6):
    """Grouped sweeps with thermal steps (thermal_every 5) of the (ctx, sp, tp) triples."""
    cet.sweep_run_group([c for c, _, _ in cases], n, [s for _, s, _ in cases], [t for _, _, t in cases])


@pytest.mark.parametrize("L", [24, 25, 30, 64, 96])
def test_texture_equals_reference(cet, L):
    cases = [_half_grown(cet, L, q) for q in range(2)]
    ctxs = [c for c, _, _ in cases] + [_driver(cet, L, 0, 40), _driver(cet, L, 1, 120)]
    try:
        _check(cet, ctxs)
        _check(cet, ctxs, EDGES_31)
        _grouped_sweeps(cet, cases, 11)                                   # two thermal steps inside
        got = _check(cet, ctxs)
        _check(cet, ctxs, EDGES_31)
        for ax in range(3):
            assert got[ax][0].sum() > 0 and (got[ax][0].sum(axis=(1, 2)) == got[0][0].sum(axis=(1, 2))).all()
    finally:
        _close(ctxs)


def test_texture_past_48KB_of_table(cet):
    """L = 512 with 31 edges: a table of 512 (32 * 4 + 16) bytes = 72 KB of shared memory.  vox and v are written on
    the device (random states with some defect bits, random unit vectors); only the texture reads them."""
    import torch
    L = 512
    ctx = cet.Context(L=L)
    try:
        g = torch.Generator(device="cuda").manual_seed(5)
        n = L ** 3

        class Dev:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
        vox = torch.as_tensor(Dev(ctx.device_ptr(0)[0], (n,), "|u1"), device="cuda")
        v = torch.as_tensor(Dev(ctx.device_ptr(5)[0], (n, 4), "<f8"), device="cuda")
        k = torch.arange(n, device="cuda") % L
        occ = torch.rand(n, generator=g, device="cuda", dtype=torch.float64) < (1.0 - k.double() / L)   # thinning along k
        st = torch.randint(1, 4, (n,), generator=g, device="cuda", dtype=torch.uint8)
        vox.copy_(torch.where(occ, st, torch.zeros_like(st)) | (torch.rand(n, generator=g, device="cuda") < 0.05).to(torch.uint8) * 16)
        th = torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * np.pi
        ph = torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * 2 * np.pi
        v.copy_(torch.stack([th.sin() * ph.cos(), th.sin() * ph.sin(), th.cos(), torch.zeros_like(th)], 1))
        v[:1000, 2] = torch.tensor(np.cos(np.radians(EDGES_31[7])), device="cuda", dtype=torch.float64)   # on an edge
        torch.cuda.synchronize()
        packed = ctx.download_packed()
        c_edges = cet._lib._texture_edges("t", EDGES_31)
        for ax in range(3):
            comp = v[:, ax].contiguous().cpu().numpy().reshape(L, L, L)
            want = textureref.split(textureref.table_c(packed, comp, ax, c_edges))
            got = cet.texture_group([ctx], ax, EDGES_31)
            for i in range(3):
                assert np.array_equal(got[i][0], want[i]), (ax, i)
            assert got[0][0].sum() == int(((packed & 0x0F) != 0).sum())
        del vox, v
    finally:
        ctx.close()


def test_texture_group_of_18(cet):
    cases = [_half_grown(cet, 30, q) for q in range(14)]
    ctxs = [c for c, _, _ in cases] + [_driver(cet, 30, q, 30 + 20 * q) for q in range(4)]
    try:
        _grouped_sweeps(cet, cases)
        _check(cet, ctxs)
        _check(cet, ctxs[:1], EDGES_31)
        _check(cet, ctxs[5:9])
    finally:
        _close(ctxs)


def test_texture_init_group_lattices(cet):
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
        _check(cet, ctxs, EDGES_31)
    finally:
        _close(ctxs)


def test_texture_after_laser_steps(cet):
    from cetkmc._config import thermal_full_params
    from cetkmc.thermal_solver import laser_source_top
    cases = [_half_grown(cet, 48, q) for q in range(3)]
    ctxs = [c for c, _, _ in cases]
    try:
        before = ctxs[0].download_packed()
        for c, sp, _ in cases:
            c.snapshot_state()
            sp.thermal_every = 0                                 # the laser step replaces the sweeps' thermal step
        for step in range(3):
            qs = [laser_source_top(48, (24.0, 6.0 * step), 150.0 + 100.0 * q, 1e-5, 0.4) for q in range(3)]
            cet.thermal_full_group(ctxs, [thermal_full_params(1e-7)] * 3, qs)
            for c, sp, _ in cases:
                c.sweep_run(4, sp, None)
        assert not np.array_equal(ctxs[0].download_packed(), before)
        _check(cet, ctxs)
    finally:
        _close(ctxs)


def test_texture_edge_lattices(cet):
    """Empty and full lattices, one orientation along +k: every site in the first angle bin along axis 2."""
    L = 40
    zero = np.zeros((L,) * 3)
    ctxs = [_upload(cet, np.zeros((L,) * 3, np.int64), zero, zero),
            _upload(cet, np.ones((L,) * 3, np.int64), zero, zero)]
    try:
        got = _check(cet, ctxs)
        for ax in range(3):
            assert not got[ax][0][0].any() and not got[ax][1][0].any()
            assert (got[ax][0][1].sum(1) == L * L).all()
        assert (got[2][0][1][:, 0] == L * L).all() and (got[2][1][1] == L * L * 2 ** 32).all()
    finally:
        _close(ctxs)


# -- non-interference ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("philox", [False, True])
def test_texture_calls_change_nothing(cet, philox):
    from cetkmc import campaign
    a = [_half_grown(cet, 24, q) for q in range(4)]
    b = [_half_grown(cet, 24, q) for q in range(4)]
    ra = [dict(_run(c, q), shapes=[], fronts=[], textures=[]) for q, (c, _, _) in enumerate(a)]
    rb = [dict(_run(c, q), shapes=[], fronts=[]) for q, (c, _, _) in enumerate(b)]
    try:
        for last in (EVERY, EVERY + 3, 2 * EVERY):
            cet.texture_group([r["ctx"] for r in ra][::-1], 0)                                # extra calls in between
            campaign._cadence_group(ra, last, EVERY, philox, SEED, profile_axis=1, shape_axis=2, front_axis=2,
                                    texture_axis=last % 3)
            cet.texture_group([r["ctx"] for r in ra], 1, EDGES_31)
            campaign._cadence_group(rb, last, EVERY, philox, SEED, profile_axis=1, shape_axis=2, front_axis=2)
            for x, y in zip(ra, rb):
                assert x["rows"][-1] == y["rows"][-1] and x["cet_detected"] == y["cet_detected"]
                assert np.array_equal(x["profiles"][-1][1], y["profiles"][-1][1])
                assert np.array_equal(x["shapes"][-1][1], y["shapes"][-1][1])
                assert x["fronts"][-1] == y["fronts"][-1]
                assert x["rng"][0] == y["rng"][0] and np.array_equal(x["rng"][1], y["rng"][1]) and x["rng"][2:] == y["rng"][2:]
                assert x["textures"][-1][0] == last and x["textures"][-1][1].shape == (24, 12)
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
    """cet_texture_group called directly (the binding's own checks bypassed): its return code."""
    h = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
    e = None if edges is None else np.ascontiguousarray(edges, np.float64)
    return cet._lib.lib().cet_texture_group(h, len(ctxs) if n is None else n, axis,
                                            None if e is None else e.ctypes.data_as(C.POINTER(C.c_double)),
                                            (0 if e is None else e.size) if m is None else m,
                                            None if out is None else out.ctypes.data_as(C.POINTER(C.c_int64)))


def test_rejections_leave_everything_untouched(cet):
    a, sa, ta = _half_grown(cet, 24, 0)
    b, sb, tb = _half_grown(cet, 24, 1)
    a2, sa2, ta2 = _half_grown(cet, 24, 0)
    b2, sb2, tb2 = _half_grown(cet, 24, 1)
    other = _upload(cet, np.ones((25,) * 3, np.int64), np.full((25,) * 3, 0.3), np.full((25,) * 3, 1.1))
    slab = cet.Context(L=24, i_begin=0, i_end=12)
    good = np.array([-0.5, 0.0, 0.5])
    try:
        before = [_snapshot(cet, x, rates=False, labels=False) for x in (a, b)]
        out = np.full(70 * 24 * 40, -7, np.int64)
        o0 = out.copy()
        for ctxs, axis, e, kw, match in (([a, slab], 2, good, {}, "slab"),
                                         ([a, other], 2, good, {}, "L ="),
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
                                         ([a, b], 2, np.array([0.0, np.inf]), {}, "finite")):
            assert _raw(cet, ctxs, axis, e, out, **kw) != 0
            assert match in cet._lib.lib().cet_last_error().decode()
            assert np.array_equal(out, o0)
        assert _raw(cet, [a, b], 2, good, None) != 0 and "NULL" in cet._lib.lib().cet_last_error().decode()
        with pytest.raises(RuntimeError, match="slab"):
            cet.texture_group([slab], 0)
        with pytest.raises(RuntimeError, match="n_ctx"):
            cet.texture_group([], 0)
        for x, s in zip((a, b), before):
            t = _snapshot(cet, x, rates=False, labels=False)
            for k in s:
                assert (s[k] == t[k]) if k == "clock" else np.array_equal(s[k], t[k], equal_nan=True), k
        assert cet.sweep_run_group([a, b], 5, [sa, sb], [ta, tb]) == cet.sweep_run_group([a2, b2], 5, [sa2, sb2], [ta2, tb2])
        for x, y in ((a, a2), (b, b2)):
            sx, sy = _snapshot(cet, x, labels=False), _snapshot(cet, y, labels=False)
            for k in sx:
                assert (sx[k] == sy[k]) if k == "clock" else np.array_equal(sx[k], sy[k], equal_nan=True), k
    finally:
        for x in (a, b, a2, b2, other, slab):
            x.close()


# -- the drivers -----------------------------------------------------------------------------------------------------

def _check_case_textures(root, files, L=24):
    """Every metrics row of every case has its L planes in texture.csv, and each plane's Solid is its bins' sum."""
    from cetkmc import campaign
    tx = [f for f in files if f.endswith("/texture.csv")]
    assert len(tx) == sum(f.endswith("/metrics.csv") for f in files if not f.startswith("plot_cet/"))
    for f in tx:
        _edges, recs = campaign.read_texture_csv(os.path.join(root, f))
        m = _read(os.path.join(root, f.replace("texture.csv", "metrics.csv")))
        assert [r[0] for r in recs] == [int(r["Step"]) for r in m]
        assert all(r[1].shape == (L, 12) for r in recs)
        rows = _read(os.path.join(root, f))
        assert all(int(r["Solid"]) == sum(int(v) for v in list(r.values())[5:]) for r in rows)
    return tx


GR = dict(L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3, seed=7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_gr_sweep_textures(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign, metrics
    monkeypatch.chdir(tmp_path)
    kw = dict(GR, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    temps, nu_deps = [2700.0, 3000.0], [2e13, 1e14]
    _terminating_replica(monkeypatch, campaign, 3000.0)
    base, ens = campaign.run_gr_sweep(temps, nu_deps, output_root="plain", replicas=3, front_axis=2, **kw)
    a, ens_a = campaign.run_gr_sweep(temps, nu_deps, output_root="solo", replicas=3, front_axis=2, texture_axis=2, **kw)
    b, ens_b = campaign.run_gr_sweep(temps, nu_deps, output_root="grouped", replicas=3, batch=4, front_axis=2,
                                     texture_axis=2, **kw)
    assert a == base and b == base and ens_a == ens and ens_b == ens
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    tx = _check_case_textures("outputs/solo", files)
    assert len(tx) == 12 and extra == sorted(tx + ["cet_map_texture_rank0.csv"])
    reps = _read("outputs/solo/cet_map_replicas_rank0.csv")
    assert any(int(r["Step"]) < 60 for r in reps if r["replica"] == "1")                        # terminated early
    for root in ("plain", "solo", "grouped"):
        campaign.merge_cet_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    rows = _read("outputs/solo/cet_map_texture.csv")
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP"] + list(metrics.TEXTURE_COLUMNS)
    assert [(int(r["case"]), int(r["replica"])) for r in rows] == [(q, r) for q in range(4) for r in range(3)]
    for r in rows:
        p = f"outputs/solo/T{float(r['T_sub']):g}_R{float(r['NU_DEP']):g}" + ("" if r["replica"] == "0" else f"/rep{r['replica']}")
        edges, recs = campaign.read_texture_csv(f"{p}/texture.csv")
        s = metrics.texture_summary(*recs[-1][1:], edges)
        assert int(r["TexturedSolid"]) == s["TexturedSolid"] and r["Hermans"] == repr(s["Hermans"])
    assert len(_read("outputs/solo/cet_map_texture_ensemble.csv")) == 4


MAP = dict(L=24, n_sweeps=61, metrics_every=30, thermal_every=5, n_seeds=6, defect_fraction=3e-3, start=(12.0, 2.0),
           dt=1e-7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_melt_pool_map_textures(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    kw = dict(MAP, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    powers, speeds = [150.0, 300.0], [1.0]
    _terminating_replica(monkeypatch, campaign, 2900.0)
    base = campaign.run_melt_pool_map(powers, speeds, output_root="plain", temp=2900.0, replicas=2, **kw)
    a = campaign.run_melt_pool_map(powers, speeds, output_root="solo", temp=2900.0, replicas=2, texture_axis=2, **kw)
    b = campaign.run_melt_pool_map(powers, speeds, output_root="grouped", temp=2900.0, replicas=2, batch=4,
                                   texture_axis=2, **kw)
    assert a == base and b == base
    files = _same_tree("outputs/solo", "outputs/grouped")
    extra = _same_subset("outputs/plain", "outputs/solo")
    tx = _check_case_textures("outputs/solo", files)
    assert extra == sorted(tx + ["melt_pool_map_texture_rank0.csv"])
    reps = _read("outputs/solo/melt_pool_map_replicas_rank0.csv")
    assert [int(r["Step"]) < 60 for r in reps if r["replica"] == "1"] == [True, True]           # terminated early
    for root in ("plain", "solo", "grouped"):
        campaign.merge_melt_pool_map(root)
    _same_subset("outputs/plain", "outputs/grouped")
    _same_tree("outputs/solo", "outputs/grouped")
    assert len(_read("outputs/solo/melt_pool_map_texture.csv")) == 4
    assert len(_read("outputs/solo/melt_pool_map_texture_ensemble.csv")) == 2


def test_run_cet_sublattice_texture_rows(cet, tmp_path, monkeypatch):
    """The solo driver's texture.csv: one record per metrics row; metrics.csv unchanged; the final record equals a
    texture_group call on the final lattice."""
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="p", verbose=False,
                                texture_axis=1, seed=3)
    campaign.run_cet_sublattice(L=24, n_sweeps=41, metrics_every=20, n_seeds=6, output_prefix="q", verbose=False, seed=3)
    assert filecmp.cmp("outputs/p/metrics.csv", "outputs/q/metrics.csv", shallow=False)
    assert not os.path.exists("outputs/q/texture.csv")
    edges, recs = campaign.read_texture_csv("outputs/p/texture.csv")
    m = _read("outputs/p/metrics.csv")
    assert edges == tuple(float(x) for x in cet._lib.TEXTURE_EDGES_DEG)
    assert [r[0] for r in recs] == [int(r["Step"]) for r in m] and len(recs) >= 2
    n_occ = int(m[-1]["W_Count"]) + int(m[-1]["Re_Count"]) + int(m[-1]["C_Count"])
    assert recs[-1][1].sum() >= n_occ
