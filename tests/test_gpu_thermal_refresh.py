"""GPU: the rates after a thermal step of cet_sweep_run.  On a whole-lattice context with L % 32 == 0 whose rates were
current before the step, the stencil marks the sites whose temperature changed and only the rates that read one of
them are refreshed (csrc/sweep.cu, thermal_refresh); every other case, and debug flag FORCE_DENSE, runs the dense
rebuild.  Both sides must leave the same lattice, counters and resident rates, bit for bit, and the rates must equal
a rebuild from the lattice."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FORCE_DENSE = 524288


def _sp(cet, L, seed=17, thermal_every=3, eps=0.01):
    sp = cet._lib.SweepParams()
    sp.seed, sp.events_per_sweep, sp.p_max = seed, eps * L ** 3, 0.2
    sp.defect_fraction, sp.thermal_every = 0.01, thermal_every
    return sp


def _ctx(cet, L, T, flags):
    from cetkmc import _synth
    from cetkmc._config import rate_params
    packed, th, ph, _ = _synth.half_grown(L, seed=5, grain=4)
    st, df = _synth.unpack(packed)
    ctx = cet.Context(L=L)
    ctx.debug_flags(flags)
    ctx.set_rate_params(rate_params(0.1))
    ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
    return ctx


def _profile(L, kind):
    """Temperature fields: 'k' the dyadic gradient along k of the benchmark, 'i' one along i, 'bump' the i gradient
    with a parabola on its lowest planes (every plane of it changes), 'random' noise (every site changes)."""
    i = np.arange(L, dtype=np.float64)[:, None, None]
    k = np.arange(L, dtype=np.float64)[None, None, :]
    if kind == "k":
        T = 2800.0 + 895.0 * k / 512 + 0.0 * i
    elif kind == "i":
        T = 2800.0 + 2.0 * i + 0.0 * k
    elif kind == "bump":
        T = 2800.0 + 2.0 * i + np.where(i < 12, 0.5 * (12 - i) ** 2, 0.0) + 0.0 * k
    else:
        T = 2800.0 + 400.0 * np.random.default_rng(3).random((L, L, L))
    return np.ascontiguousarray(np.broadcast_to(T, (L, L, L)))


def _run(cet, L, T, flags, n, tp, thermal_every=3, seed=17):
    ctx = _ctx(cet, L, T, flags)
    ctx.profile_enable(True)
    res = ctx.sweep_run(n, _sp(cet, L, seed, thermal_every), tp)
    prof = {k: ctx.profile_read(k) for k in ("rates", "refresh", "thermal")}
    ctx.profile_enable(False)
    lat = ctx.download(state=True, theta=True, phi=True, T=True)
    sr, dr = ctx.rates_download()
    ctx.rates_build()
    sr2, dr2 = ctx.rates_download()
    np.testing.assert_array_equal(sr, sr2)            # the resident rates equal a rebuild from the lattice
    np.testing.assert_array_equal(dr, dr2)
    return ctx, res, lat, (sr, dr), prof


def _same(a, b):
    _, ra, la, (sa, da), _ = a
    _, rb, lb, (sb, db), _ = b
    assert ra == rb
    for k in la:
        np.testing.assert_array_equal(la[k], lb[k])
    np.testing.assert_array_equal(sa, sb)
    np.testing.assert_array_equal(da, db)


# side: "refresh" (few stale sites), "over" (every site stale: the thermal refresh counts them and rebuilds densely),
# "dense" (L % 32 != 0: no bitmap, the dense rebuild)
@pytest.mark.parametrize("L,kind,side", [(64, "k", "refresh"), (96, "k", "refresh"), (128, "i", "refresh"),
                                         (128, "bump", "refresh"), (80, "k", "dense"), (64, "random", "over")])
def test_thermal_refresh_equals_dense(cet, L, kind, side):
    from cetkmc._config import thermal_params
    tp = thermal_params(1e-6, nan_to_num=True)
    n = 13                                              # thermal steps at sweeps 0, 3, 6, 9, 12
    a = _run(cet, L, _profile(L, kind), 0, n, tp)
    b = _run(cet, L, _profile(L, kind), FORCE_DENSE, n, tp)
    _same(a, b)
    assert a[1]["events_applied"] > 100 and not a[1]["terminated"]
    # the first step follows the upload: dense on both sides; the forced side rebuilds after every step
    assert b[4]["rates"][1] == 5 and a[4]["thermal"][1] == 5
    assert a[4]["rates"][1] == (1 if side == "refresh" else 5)
    assert a[4]["refresh"][1] == n + 1 + (0 if side == "dense" else 4)
    for r in (a, b):
        r[0].close()


def test_thermal_refresh_keeps_tile_state(cet):
    """Sweeps continued on the tile state the incremental steps left equal sweeps continued on a rebuilt one."""
    from cetkmc._config import thermal_params
    tp = thermal_params(1e-6, nan_to_num=True)
    L = 64
    outs = []
    for rebuild in (False, True):
        ctx = _ctx(cet, L, _profile(L, "k"), 0)
        ctx.sweep_run(8, _sp(cet, L), tp)
        if rebuild:
            ctx.upload(T=ctx.download(T=True)["T"])    # drops the tile state and the rates (same values)
        res = ctx.sweep_run(7, _sp(cet, L), tp)
        outs.append((res, ctx.download(state=True, theta=True, phi=True, T=True), ctx.rates_download()))
        ctx.close()
    (r1, l1, s1), (r2, l2, s2) = outs
    assert r1 == r2
    for k in l1:
        np.testing.assert_array_equal(l1[k], l2[k])
    for x, y in zip(s1, s2):
        np.testing.assert_array_equal(x, y)


def _bump(L, m):
    i = np.arange(L, dtype=np.float64)[:, None, None]
    T = 2800.0 + 2.0 * i + np.where(i < m, 0.5 * (m - i) ** 2, 0.0) + 0.0 * np.arange(L)[None, None, :]
    return np.ascontiguousarray(np.broadcast_to(T, (L, L, L)))


def _stale_planes(oracle, T):
    """Planes whose rates the second thermal step makes stale: T depends on i only, so whole planes change, and a
    changed plane makes stale the planes within two of it."""
    T1 = oracle.thermal_cet(T, nan_to_num=True)
    T2 = oracle.thermal_cet(T1, nan_to_num=True)
    changed = np.flatnonzero(np.any(T1.view(np.int64) != T2.view(np.int64), axis=(1, 2)))
    return len({q for p in changed for q in range(p - 2, p + 3) if 0 <= q < T.shape[0]})


@pytest.mark.parametrize("planes,incremental", [(24, True), (25, False)])
def test_thermal_refresh_threshold(cet, oracle, planes, incremental):
    """Up to three eighths of the sites stale: the refresh; one plane more: the dense rebuild.  The bump's height is
    chosen on the host (the oracle's stencil is the device's, bit for bit) so that the second thermal step makes
    exactly `planes` of the 64 planes stale."""
    from cetkmc._config import thermal_params
    tp = thermal_params(1e-6, nan_to_num=True)
    L = 64
    m = next(m for m in range(L // 2) if _stale_planes(oracle, _bump(L, m)) == planes)
    ctx = _ctx(cet, L, _bump(L, m), 0)
    sp = _sp(cet, L, thermal_every=1, eps=1e-9)
    ctx.sweep_run(1, sp, tp)                           # priming pass + sweep 0: the first step, dense after the upload
    ctx.profile_enable(True)
    res = ctx.sweep_run(1, sp, tp)                     # the second step
    prof = {k: ctx.profile_read(k) for k in ("rates", "refresh")}
    ctx.profile_enable(False)
    assert res["sweeps_done"] == 1 and res["events_applied"] == 0
    # the thermal step's refresh span is there on both sides (stale sites counted), the sweep's refresh follows
    assert prof["refresh"][1] == 2 and prof["rates"][1] == (0 if incremental else 1)
    np.testing.assert_array_equal(ctx.download(T=True)["T"],
                                  oracle.thermal_cet(oracle.thermal_cet(_bump(L, m), nan_to_num=True), nan_to_num=True))
    sr, dr = ctx.rates_download()
    ctx.rates_build()
    sr2, dr2 = ctx.rates_download()
    ctx.close()
    np.testing.assert_array_equal(sr, sr2)
    np.testing.assert_array_equal(dr, dr2)


def test_thermal_refresh_terminated(cet, oracle):
    """A lattice without events (every site W): the priming pass terminates the run, so every later stencil pass is
    the identity; the refresh side finds no changed site and keeps the rates, the forced side rebuilds them."""
    from cetkmc._config import rate_params, thermal_params
    tp = thermal_params(1e-6, nan_to_num=True)
    L = 64
    T0 = _profile(L, "k")
    outs = []
    for flags in (0, FORCE_DENSE):
        ctx = cet.Context(L=L)
        ctx.debug_flags(flags)
        ctx.set_rate_params(rate_params(0.1))
        ctx.upload(state=np.ones((L, L, L), np.int64), theta=np.full((L, L, L), 0.5), phi=np.full((L, L, L), 1.0),
                   T=T0, defects=np.zeros((L, L, L), np.int64))
        ctx.profile_enable(True)
        res = ctx.sweep_run(6, _sp(cet, L, thermal_every=2), tp)
        prof = {k: ctx.profile_read(k) for k in ("rates", "refresh", "thermal")}
        ctx.profile_enable(False)
        outs.append((res, prof, ctx.download(state=True, T=True), ctx.rates_download()))
        ctx.close()
    (ra, pa, la, sa), (rb, pb, lb, sb) = outs
    assert ra["terminated"] and ra == rb
    assert pa["thermal"][1] == 3 and pa["rates"][1] == 1 and pa["refresh"][1] == 7 + 2
    assert pb["thermal"][1] == 3 and pb["rates"][1] == 3 and pb["refresh"][1] == 7
    np.testing.assert_array_equal(la["T"], oracle.thermal_cet(T0, nan_to_num=True))    # only the first pass changed T
    for k in la:
        np.testing.assert_array_equal(la[k], lb[k])
    for x, y in zip(sa, sb):
        np.testing.assert_array_equal(x, y)
