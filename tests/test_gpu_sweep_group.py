"""GPU: grouped sweeps (cet_sweep_run_group / cetkmc.sweep_run_group) — every lattice of a group ends bit for
bit where a solo sweep_run of the same inputs leaves it, whatever else is in the group and in whatever order;
and the batched G-R sweep driver writes the same files as the unbatched one."""
import filecmp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

THERMAL_EVERY = 5


def _case(cet, L, q):
    """Context q of a test group: its own lattice, seed, NU_DEP and substrate temperature."""
    from cetkmc import _synth
    from cetkmc._config import rate_params, thermal_params
    packed, th, ph, T = _synth.half_grown(L, seed=20 + q, grain=4)
    ctx = cet.Context(L=L)
    ctx.set_rate_params(rate_params(0.1, overrides={"NU_DEP": 2e13 * (1 + q)}))
    st, df = _synth.unpack(packed)
    ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
    sp = cet._lib.SweepParams()
    sp.seed, sp.events_per_sweep, sp.p_max = 100 + q, 0.005 * L ** 3, 0.1 + 0.02 * q
    sp.defect_fraction, sp.thermal_every = 0.01, THERMAL_EVERY
    tp = thermal_params(1e-6, nan_to_num=True, t_floor=2600.0 + 50.0 * q)
    return ctx, sp, tp


def _snapshot(ctx):
    f = ctx.download(state=True, theta=True, phi=True, T=True)
    sr, dr = ctx.rates_download()
    return dict(f, packed=ctx.download_packed(), site_rate=sr, dep_rate=dr, clock=ctx.sweep_state())


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if k == "clock":
            assert a[k] == b[k]
        else:
            assert np.array_equal(a[k], b[k], equal_nan=True), k


def _solo(cet, L, qs, n, pre=None):
    """Snapshot and result of each case q run alone: optional solo `pre` sweeps, then n."""
    out = []
    for q in qs:
        ctx, sp, tp = _case(cet, L, q)
        if pre:
            ctx.sweep_run(pre[q] if isinstance(pre, dict) else pre, sp, tp)
        res = ctx.sweep_run(n, sp, tp)
        out.append((res, _snapshot(ctx)))
        ctx.close()
    return out


def _grouped(cet, L, qs, n, pre=None):
    cases = [_case(cet, L, q) for q in qs]
    if pre:
        for q, (ctx, sp, tp) in zip(qs, cases):
            if (pre[q] if isinstance(pre, dict) else pre):
                ctx.sweep_run(pre[q] if isinstance(pre, dict) else pre, sp, tp)
    res = cet.sweep_run_group([c for c, _, _ in cases], n, [s for _, s, _ in cases], [t for _, _, t in cases])
    out = [(r, _snapshot(c)) for r, (c, _, _) in zip(res, cases)]
    for c, _, _ in cases:
        c.close()
    return out


@pytest.mark.parametrize("L", [64, 24])              # 64: the TMA dense rebuild; 24: the compact gather rebuild
def test_group_equals_solo(cet, L):
    qs = [0, 1, 2, 3]
    solo = _solo(cet, L, qs, 45)
    grp = _grouped(cet, L, qs, 45)
    for (rs, ss), (rg, sg) in zip(solo, grp):
        assert rs == rg
        _same(ss, sg)
    assert all(r["events_applied"] > 0 and not r["overflow"] for r, _ in grp)


def test_group_above_sixteen_equals_solo(cet):
    """18 lattices: the 64-entry argument tables of the grouped kernels."""
    qs = list(range(18))
    solo = _solo(cet, 24, qs, 12)
    grp = _grouped(cet, 24, qs, 12)
    for (rs, ss), (rg, sg) in zip(solo, grp):
        assert rs == rg
        _same(ss, sg)


def test_group_order_does_not_matter(cet):
    L, qs = 24, [0, 1, 2, 3]
    fwd = _grouped(cet, L, qs, 23)
    rev = _grouped(cet, L, qs[::-1], 23)[::-1]
    for (ra, sa), (rb, sb) in zip(fwd, rev):
        assert ra == rb
        _same(sa, sb)


def _terminated_case(cet, L):
    """A lattice with no event at all (every site W, no empty neighbour): its first sweep terminates it."""
    from cetkmc._config import rate_params, thermal_params
    ctx = cet.Context(L=L)
    ctx.set_rate_params(rate_params(0.1))
    ctx.upload(state=np.ones((L, L, L), np.int64), theta=np.full((L, L, L), 0.5), phi=np.full((L, L, L), 1.0),
               T=np.full((L, L, L), 2900.0), defects=np.zeros((L, L, L), np.int64))
    sp = cet._lib.SweepParams()
    sp.seed, sp.events_per_sweep, sp.p_max, sp.defect_fraction, sp.thermal_every = 9, 0.005 * L ** 3, 0.1, 0.0, THERMAL_EVERY
    return ctx, sp, thermal_params(1e-6, nan_to_num=True)


def test_group_of_mixed_states(cet):
    """One context 7 sweeps into its run, one fresh (primed by the call), one already terminated."""
    L, n = 24, 17
    a, sa, ta = _case(cet, L, 0)
    a.sweep_run(7, sa, ta)
    b, sb, tb = _case(cet, L, 1)
    c, sc, tc = _terminated_case(cet, L)
    assert c.sweep_run(3, sc, tc)["terminated"]
    res = cet.sweep_run_group([a, b, c], n, [sa, sb, sc], [ta, tb, tc])
    got = [_snapshot(x) for x in (a, b, c)]
    for x in (a, b, c):
        x.close()
    a, sa, ta = _case(cet, L, 0)
    a.sweep_run(7, sa, ta)
    b, sb, tb = _case(cet, L, 1)
    c, sc, tc = _terminated_case(cet, L)
    c.sweep_run(3, sc, tc)
    want = [x.sweep_run(n, s, t) for x, s, t in ((a, sa, ta), (b, sb, tb), (c, sc, tc))]
    for r, w, g, x in zip(res, want, got, (a, b, c)):
        assert r == w
        _same(g, _snapshot(x))
        x.close()
    assert res[0]["sweep_index"] == 7 + n and res[1]["sweep_index"] == n and res[2]["terminated"]


def test_group_continues_solo_runs(cet):
    """Grouped N then solo M, and solo N then grouped M, both equal solo N + M."""
    L, qs, N, M = 24, [0, 1, 2], 11, 9
    ref = _solo(cet, L, qs, N + M)
    cases = [_case(cet, L, q) for q in qs]
    cet.sweep_run_group([c for c, _, _ in cases], N, [s for _, s, _ in cases], [t for _, _, t in cases])
    first = [(c.sweep_run(M, s, t), _snapshot(c)) for c, s, t in cases]
    for c, _, _ in cases:
        c.close()
    second = _grouped(cet, L, qs, M, pre=N)
    for (rr, sr), (r1, s1), (r2, s2) in zip(ref, first, second):
        _same(sr, s1)
        _same(sr, s2)
        assert rr["sweep_index"] == r1["sweep_index"] == r2["sweep_index"] == N + M
        assert r1 == r2


def test_group_of_one_equals_sweep_run(cet):
    (rs, ss), = _solo(cet, 64, [2], 12)
    (rg, sg), = _grouped(cet, 64, [2], 12)
    assert rs == rg
    _same(ss, sg)


def test_group_rejections_leave_contexts_untouched(cet):
    L = 24
    a, sa, ta = _case(cet, L, 0)
    b, sb, tb = _case(cet, L, 1)
    for x, s, t in ((a, sa, ta), (b, sb, tb)):
        x.sweep_run(2, s, t)                                       # resident rates and a running clock to compare
    before = [_snapshot(x) for x in (a, b)]

    def rejected(ctxs, sps, tps=None, n=3):
        with pytest.raises(RuntimeError):
            cet.sweep_run_group(ctxs, n, sps, tps)

    rejected([a, a], [sa, sa], [ta, ta])                           # a repeated context
    closed = cet.Context(L=L)
    closed.close()
    rejected([a, closed], [sa, sb], [ta, tb])                      # a NULL context
    other_L, so, to = _case(cet, 32, 2)
    rejected([a, other_L], [sa, so], [ta, to])                     # different L
    other_L.close()
    slab = cet.Context(L=L, i_begin=0, i_end=L // 2)
    rejected([a, slab], [sa, sb], [ta, tb])                        # a partial plane range
    slab.close()
    norp = cet.Context(L=L)
    rejected([a, norp], [sa, sb], [ta, tb])                        # no rate params
    norp.close()
    b.debug_flags(2)
    rejected([a, b], [sa, sb], [ta, tb])                           # debug flags
    b.debug_flags(0)
    oriented, so, to = _case(cet, L, 2)                            # an empty site with an orientation: gather path
    st, th = oriented.download(state=True)["state"], oriented.download(theta=True)["theta"]
    z = np.argwhere(st == 0)[0]
    th[tuple(z)] = 0.7
    oriented.upload(theta=th)
    rejected([a, oriented], [sa, so], [ta, to])
    oriented.close()
    bad = cet._lib.SweepParams()
    bad.seed, bad.events_per_sweep, bad.p_max, bad.thermal_every = 1, 10.0, 1.5, 0
    rejected([a, b], [sa, bad], [ta, tb])                          # an argument cet_sweep_run rejects
    rejected([a, b], [sa, sb], None)                               # thermal_every without thermal params
    rejected([], [], None)                                         # n_ctx < 1
    with pytest.raises(RuntimeError, match="n_ctx"):                # n_ctx above the maximum (checked first)
        cet.sweep_run_group([a] * 65, 3, [sa] * 65, [ta] * 65)
    for x, s in zip((a, b), before):
        _same(_snapshot(x), s)
        assert x.sweep_state()[0] == 2
    # after all that, both still run and match their solo runs
    res = cet.sweep_run_group([a, b], 6, [sa, sb], [ta, tb])
    got = [_snapshot(x) for x in (a, b)]
    a.close(); b.close()
    for (rs, ss), r, g in zip(_solo(cet, L, [0, 1], 6, pre=2), res, got):
        assert rs == r
        _same(ss, g)


def _tree_files(root):
    out = []
    for d, _, fs in os.walk(root):
        out += [os.path.relpath(os.path.join(d, f), root) for f in fs]
    return sorted(out)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_batched_gr_sweep_writes_the_same_files(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    # the case T_sub = 3100, NU_DEP = 1e14 starts from a lattice without events (every site W): it terminates in its
    # first interval, writes one row and leaves its group while the others go on
    upload = campaign._upload_initial

    def upload_initial(ctx, L, n_seeds, temp, impurity_c, lattice, i_begin, i_end):
        if temp == 3100.0 and ctx is not None and getattr(ctx, "_nu_dep", None) == 1e14:
            ones = np.ones((L, L, L), np.int64)
            lattice = (ones, np.full((L, L, L), 0.5), np.full((L, L, L), 1.0), np.full((L, L, L), 2900.0), ones)
        return upload(ctx, L, n_seeds, temp, impurity_c, lattice, i_begin, i_end)
    set_rp = cet.Context.set_rate_params

    def set_rate_params(ctx, rp):
        ctx._nu_dep = rp.nu_dep
        return set_rp(ctx, rp)
    monkeypatch.setattr(campaign, "_upload_initial", upload_initial)
    monkeypatch.setattr(cet.Context, "set_rate_params", set_rate_params)
    kw = {} if mask_stream is None else dict(mask_stream=mask_stream)
    temps, nu_deps = [2700.0, 3100.0], [2e13, 1e14]
    a = campaign.run_gr_sweep(temps, nu_deps, L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3,
                              output_root="plain", **kw)
    b = campaign.run_gr_sweep(temps, nu_deps, L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3,
                              output_root="grouped", batch=3, **kw)
    assert len(a) == 4 and a == b
    files = _tree_files("outputs/plain")
    assert files == _tree_files("outputs/grouped") and "cet_map_rank0.csv" in files
    assert sum(f.endswith("metrics.csv") for f in files) == 4
    n_rows = {f: len(open(os.path.join("outputs/grouped", f)).read().strip().splitlines()) - 1
              for f in files if f.endswith("/metrics.csv")}
    assert n_rows.pop("T3100_R1e+14/metrics.csv") == 1 and set(n_rows.values()) == {4}
    assert a[3]["CET_Detected"] is not None and str(a[3]["Step"]) == "0"
    for f in files:
        assert filecmp.cmp(os.path.join("outputs/plain", f), os.path.join("outputs/grouped", f), shallow=False), f
