"""GPU: the grouped metrics cadence (cet_metrics_group / cetkmc.metrics_group, campaign._cadence_group) against
twin contexts that run the per-context cadence (campaign._cadence): identical metrics rows and NumPy stream
positions, identical lattices (mask refresh included) that then sweep identically, the grain state the call leaves
behind, grain counts at the edges of the pairwise AR sum, order independence and rejections."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EVERY, SEED = 10, 77


def _case(cet, L, q):
    """Context q of a test group: its own half-grown lattice, NU_DEP and substrate temperature, a few sweeps in."""
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


def _run(ctx, q):
    np.random.seed(1000 + q)
    return dict(ctx=ctx, rng=np.random.get_state(), consts=(1.0e6 * (q + 1), 2.0, 3.0e-9, 4.0), rows=[],
                total_time=1e-3 * q, nucleation_count=5 * q, cet_detected=False)


def _twin_cadence(runs, last, philox):
    from cetkmc import campaign
    for r in runs:
        np.random.set_state(r["rng"])
        row, r["cet_detected"] = campaign._cadence(r["ctx"], last, EVERY, philox, SEED, 1, r["total_time"],
                                                   r["nucleation_count"], r["cet_detected"], r["consts"], verbose=False)
        r["rng"] = np.random.get_state()
        r["rows"].append(row)


def _same_rows(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert type(a[k]) is type(b[k]) and repr(a[k]) == repr(b[k]), (k, a[k], b[k])


def _same_rng(a, b):
    assert a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


def _grain_state(cet, ctx):
    """The last labelling of ctx as cet_grains_stats and cet_grains_download_labels report it (no relabelling)."""
    L = cet._lib
    n = ctx._last_n
    root, size = np.empty(n, np.int32), np.empty(n, np.int32)
    lo, hi = np.empty((n, 3), np.int32), np.empty((n, 3), np.int32)
    if n:
        L.check(L.lib().cet_grains_stats(ctx._h, n, L._ptr(root), L._ptr(size), L._ptr(lo), L._ptr(hi)), "stats")
    o = np.argsort(root)
    lab = np.empty(ctx.owned_shape, np.int32)
    L.check(L.lib().cet_grains_download_labels(ctx._h, L._ptr(lab)), "labels")
    return root[o], size[o], lo[o], hi[o], lab


def _snapshot(ctx):
    sr, dr = ctx.rates_download()
    return dict(packed=ctx.download_packed(), site_rate=sr, dep_rate=dr, clock=ctx.sweep_state(),
                theta=ctx.download(theta=True)["theta"])


@pytest.mark.parametrize("L,B", [(24, 4), (30, 4), (64, 4), (24, 18), (64, 1)])
@pytest.mark.parametrize("philox", [False, True])
@pytest.mark.parametrize("last", [EVERY, EVERY + 3])            # a refresh row and a row without refresh
def test_group_cadence_equals_per_context_cadence(cet, L, B, philox, last):
    from cetkmc import campaign
    a = [_case(cet, L, q) for q in range(B)]
    b = [_case(cet, L, q) for q in range(B)]
    ra = [_run(c, q) for q, (c, _, _) in enumerate(a)]
    rb = [_run(c, q) for q, (c, _, _) in enumerate(b)]
    campaign._cadence_group(ra, last, EVERY, philox, SEED)
    _twin_cadence(rb, last, philox)
    for x, y in zip(ra, rb):
        _same_rows(x["rows"][-1], y["rows"][-1])
        assert x["cet_detected"] == y["cet_detected"]
        _same_rng(x["rng"], y["rng"])
        assert np.array_equal(x["ctx"].download_packed(), y["ctx"].download_packed())
    assert any(x["rows"][-1]["GrainCount"] > 0 for x in ra)
    # the grain state the call leaves behind is the twin's labelling
    for x, y in zip(ra, rb):
        x["ctx"]._last_n = y["ctx"]._last_n = int(x["rows"][-1]["GrainCount"])
        for u, v in zip(_grain_state(cet, x["ctx"]), _grain_state(cet, y["ctx"])):
            assert np.array_equal(u, v)
    # the sweeps that follow see the same lattice (a refresh marks the rates stale on both sides)
    ga = cet.sweep_run_group([c for c, _, _ in a], 6, [s for _, s, _ in a], [t for _, _, t in a])
    gb = cet.sweep_run_group([c for c, _, _ in b], 6, [s for _, s, _ in b], [t for _, _, t in b])
    assert ga == gb
    for (x, _, _), (y, _, _) in zip(a, b):
        sx, sy = _snapshot(x), _snapshot(y)
        for k in sx:
            assert (sx[k] == sy[k]) if k == "clock" else np.array_equal(sx[k], sy[k], equal_nan=True), k
    for c, _, _ in a + b:
        c.close()


def _upload(cet, state, theta, phi):
    L = state.shape[0]
    ctx = cet.Context(L=L)
    ctx.upload(state=state.astype(np.int64), theta=theta, phi=phi, T=np.full(state.shape, 2900.0),
               defects=np.zeros(state.shape, np.int64))
    return ctx


def _even(L):
    """Sites with i + j + k even occupied: every neighbour offset keeps that parity, so a fully occupied lattice of
    one orientation is two grains, and this half of it one."""
    i = np.arange(L)
    return ((i[:, None, None] + i[None, :, None] + i[None, None, :]) % 2 == 0).astype(np.int64)


def _blocks(L, nb_i, nb_j):
    """Blocks of nb_i ranges along axis 0 and nb_j along axis 1 (each at least 2 sites wide), 4 orientations at
    right angles so that no two touching blocks join, on the even sites: nb_i * nb_j grains."""
    bi = np.minimum(np.arange(L) * nb_i // L, nb_i - 1)
    bj = np.minimum(np.arange(L) * nb_j // L, nb_j - 1)
    colour = (bi[:, None, None] % 2) * 2 + (bj[None, :, None] % 2) + np.zeros((1, 1, L), np.int64)
    theta = np.array([0.0, np.pi / 2, np.pi / 2, np.pi])[colour]
    phi = np.array([0.0, 0.0, np.pi / 2, 0.0])[colour]
    return _even(L), theta, phi


def _edge_lattices():
    rng = np.random.default_rng(5)
    L = 64
    pepper = (rng.integers(1, 4, (L, L, L)), rng.uniform(0, np.pi, (L, L, L)), rng.uniform(0, 2 * np.pi, (L, L, L)))
    return dict(empty=(np.zeros((24,) * 3, np.int64), np.zeros((24,) * 3), np.zeros((24,) * 3)),
                one=(_even(24), np.full((24,) * 3, 0.3), np.full((24,) * 3, 1.1)),
                five=_blocks(24, 5, 1), hundred=_blocks(30, 10, 10), b129=_blocks(86, 3, 43), pepper=pepper)


@pytest.mark.parametrize("name,n_expected", [("empty", 0), ("one", 1), ("five", 5), ("hundred", 100), ("b129", 129),
                                              ("pepper", None)])
def test_grain_counts_at_the_edges(cet, name, n_expected):
    from cetkmc import kmc_simulation as ks
    st, th, ph = _edge_lattices()[name]
    a, b = _upload(cet, st, th, ph), _upload(cet, st, th, ph)
    ra, rb = _run(a, 0), _run(b, 0)
    from cetkmc import campaign
    campaign._cadence_group([ra], EVERY + 1, EVERY, False, SEED)
    row, _ = ks._metrics_row(EVERY + 1, rb["total_time"], rb["nucleation_count"], False, rb["consts"], b, verbose=False)
    _same_rows(ra["rows"][-1], row)
    n = row["GrainCount"]
    if n_expected is None:
        assert n >= 10 ** 5
    else:
        assert n == n_expected
    a._last_n = b._last_n = n
    for u, v in zip(_grain_state(cet, a), _grain_state(cet, b)):
        assert np.array_equal(u, v)
    a.close(); b.close()


def _params(cet, ctxs, refresh=True):
    from cetkmc import metrics
    from cetkmc._config import constants
    out = []
    n_sites = int(np.prod(ctxs[0].owned_shape))
    for _ in ctxs:
        p = cet._lib.MetricsParams()
        p.theta_threshold, p.ar_threshold = 0.5, constants.CET_AR_THRESHOLD
        p.pct_pos[:] = metrics.percentile_positions(n_sites)
        p.refresh, p.carbon_id, p.epoch, p.seed = int(refresh), 3, 4, SEED
        p.prob_base, p.e_mig, p.kT, p.T_default = 0.12, 0.3, constants.K_T, constants.T_SUB
        out.append(p)
    return out


def test_group_order_does_not_matter(cet):
    fwd = [_case(cet, 24, q)[0] for q in range(4)]
    rev = [_case(cet, 24, q)[0] for q in range(4)][::-1]
    ra = cet.metrics_group(fwd, _params(cet, fwd))
    rb = cet.metrics_group(rev, _params(cet, rev))[::-1]
    for x, y in zip(ra, rb):
        assert x.keys() == y.keys()
        for k in x:
            assert np.array_equal(x[k], y[k]), k
    for x, y in zip(fwd, rev[::-1]):
        assert np.array_equal(x.download_packed(), y.download_packed())
    assert np.array_equal(cet.counts_group(fwd), np.stack([c.counts() for c in fwd]))
    for c in fwd + rev:
        c.close()


def test_group_rejections_leave_contexts_untouched(cet):
    a, _, _ = _case(cet, 24, 0)
    b, _, _ = _case(cet, 24, 1)
    before = [x.download_packed() for x in (a, b)]
    n_c = [int(x.counts()[3]) for x in (a, b)]
    assert min(n_c) > 0
    u = np.random.default_rng(3)
    few = [u.random(n_c[0]), u.random(n_c[1] - 1)]                  # too few draws for the second context
    np.random.seed(3)
    rng = np.random.get_state()

    def rejected(ctxs, params=None, draws=None, match=None):
        with pytest.raises(RuntimeError, match=match):
            cet.metrics_group(ctxs, _params(cet, ctxs) if params is None else params, draws)

    rejected([a, a])                                                # a repeated context
    closed = cet.Context(L=24)
    closed.close()
    rejected([a, closed])                                           # a NULL context
    with pytest.raises(RuntimeError, match="n_ctx"):
        cet.metrics_group([a] * 65, _params(cet, [a] * 65))          # 65 contexts
    other = cet.Context(L=30)
    rejected([a, other])                                            # mixed L
    other.close()
    slab = cet.Context(L=24, i_begin=0, i_end=12)
    rejected([a, slab])                                             # a slab
    slab.close()
    rejected([a, b], draws=few, match="draws")
    with pytest.raises(RuntimeError):
        cet.counts_group([a, a])
    for x, p in zip((a, b), before):
        assert np.array_equal(x.download_packed(), p)
    _same_rng(np.random.get_state(), rng)
    # after all that, both still work and match their twins
    ra = cet.metrics_group([a, b], _params(cet, [a, b]))
    a2, _, _ = _case(cet, 24, 0)
    b2, _, _ = _case(cet, 24, 1)
    rb = cet.metrics_group([a2, b2], _params(cet, [a2, b2]))
    for x, y in zip(ra, rb):
        for k in x:
            assert np.array_equal(x[k], y[k]), k
    for x, y in zip((a, b), (a2, b2)):
        assert np.array_equal(x.download_packed(), y.download_packed())
    for x in (a, b, a2, b2):
        x.close()
