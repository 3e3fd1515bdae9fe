"""GPU: the grouped laser step (cet_thermal_full_group / cetkmc.thermal_full_group) — every lattice of a group ends
bit for bit where thermal_full + snapshot_state leave it alone, including what the fused snapshot and pair operands
do to the sweeps and steps that follow; rejected calls change nothing; and the melt-pool map writes the same files
with and without batch."""
import ctypes as C
import filecmp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _case(cet, L, q):
    """Context q of a test group: its own lattice and seed, a previous state in which some of today's solid sites were
    empty (a non-zero latent-heat term), and its own laser: power, position, speed and dt."""
    from cetkmc import _synth
    from cetkmc._config import rate_params, thermal_full_params
    from cetkmc.thermal_solver import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS
    packed, th, ph, T = _synth.half_grown(L, seed=40 + q, grain=4)
    st, df = _synth.unpack(packed)
    ctx = cet.Context(L=L)
    ctx.set_rate_params(rate_params(0.1, overrides={"NU_DEP": 2e13 * (1 + q % 5)}))
    ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
    prev = st.copy()
    rng = np.random.default_rng(q)
    prev[(st != 0) & (rng.random(st.shape) < 0.2)] = 0
    assert np.any((prev == 0) & (st != 0))
    ctx.upload_prev_state(prev)
    sp = cet._lib.SweepParams()
    sp.seed, sp.events_per_sweep, sp.p_max = 300 + q, 0.005 * L ** 3, 0.1 + 0.01 * (q % 8)
    sp.defect_fraction, sp.thermal_every = 0.01, 0
    laser = dict(power=150.0 + 37.0 * q, pos=[1.0 + 0.5 * q, (3.0 * q) % L], speed=0.5 + 0.25 * (q % 4),
                 dt=1e-7 * (1 + q % 3))
    laser["tfp"] = thermal_full_params(laser["dt"])
    laser["q_top"] = lambda: _lib_source(L, laser, DEFAULT_BEAM_RADIUS, DEFAULT_ABSORPTIVITY)
    return ctx, sp, laser


def _lib_source(L, laser, radius, absorptivity):
    from cetkmc.thermal_solver import laser_source_top
    return laser_source_top(L, tuple(laser["pos"]), laser["power"], radius, absorptivity)


def _snapshot(ctx, rates=True):
    f = ctx.download(state=True, theta=True, phi=True, T=True)
    out = dict(f, packed=ctx.download_packed(), clock=ctx.sweep_state())
    if rates:
        out["site_rate"], out["dep_rate"] = ctx.rates_download()
    return out


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if k == "clock":
            assert a[k] == b[k]
        else:
            assert np.array_equal(a[k], b[k], equal_nan=True), k


def _solo_step(ctx, laser):
    ctx.thermal_full(laser["tfp"], laser["q_top"]())
    ctx.snapshot_state()


def _group_step(cet, cases):
    cet.thermal_full_group([c for c, _, _ in cases], [l["tfp"] for _, _, l in cases], [l["q_top"]() for _, _, l in cases],
                           snapshot=True)


def _close(cases):
    for c, _, _ in cases:
        c.close()


@pytest.mark.parametrize("n", [1, 4, 18])              # 18: the 64-entry argument table
@pytest.mark.parametrize("L", [64, 30, 25])            # the V = 4, V = 2 and scalar stencils
def test_group_step_equals_thermal_full_and_snapshot(cet, L, n):
    solo = [_case(cet, L, q) for q in range(n)]
    for c, _, l in solo:
        _solo_step(c, l)
    grp = [_case(cet, L, q) for q in range(n)]
    _group_step(cet, grp)
    for (a, _, _), (b, _, _) in zip(solo, grp):
        _same(_snapshot(a, rates=False), _snapshot(b, rates=False))
    # the snapshot: a second step sees no solidified site on either side
    for c, _, l in solo:
        _solo_step(c, l)
    _group_step(cet, grp)
    for (a, _, _), (b, _, _) in zip(solo, grp):
        _same(_snapshot(a, rates=False), _snapshot(b, rates=False))
    _close(solo)
    _close(grp)


BLOCKS = (5, 7, 4, 6)


def _run_blocks(cet, L, qs, grouped, stale=()):
    """The laser driver's loop on the cases qs: snapshot_state, then per block one laser step (the melt pool moving on)
    and the block's sweeps; `stale`: cases whose tile state is dropped (a T upload) before the third step."""
    cases = [_case(cet, L, q) for q in qs]
    for c, _, _ in cases:
        c.snapshot_state()
    out = []
    for b, blk in enumerate(BLOCKS):
        if b == 2:
            for q, (c, _, _) in zip(qs, cases):
                if q in stale:
                    c.upload(T=c.download(T=True)["T"])
        if grouped:
            _group_step(cet, cases)
            res = cet.sweep_run_group([c for c, _, _ in cases], blk, [s for _, s, _ in cases])
        else:
            res = []
            for c, s, l in cases:
                _solo_step(c, l)
                res.append(c.sweep_run(blk, s, None))
        for _, _, l in cases:
            l["pos"][1] += l["speed"]
        out.append([(r, _snapshot(c)) for r, (c, _, _) in zip(res, cases)])
    _close(cases)
    return out


def _same_runs(a, b):
    for blk_a, blk_b in zip(a, b):
        for (ra, sa), (rb, sb) in zip(blk_a, blk_b):
            assert ra == rb
            _same(sa, sb)


@pytest.mark.parametrize("L", [64, 24])                # 64: the TMA dense rebuild; 24: the compact rebuild
def test_later_steps_and_sweeps_equal_the_solo_driver(cet, L):
    qs = [0, 1, 2, 3]
    solo = _run_blocks(cet, L, qs, False)
    grp = _run_blocks(cet, L, qs, True)
    _same_runs(solo, grp)
    assert all(sum(blk[i][0]["events_applied"] for blk in grp) > 0 for i in range(len(qs)))


def test_group_order_does_not_matter(cet):
    qs = [0, 1, 2, 3]
    fwd = _run_blocks(cet, 24, qs, True)
    rev = [blk[::-1] for blk in _run_blocks(cet, 24, qs[::-1], True)]
    _same_runs(fwd, rev)


def test_stale_tile_state_stays_stale_and_matches(cet):
    """Cases 1 and 2 have their tile state dropped before the third step: it is rebuilt by the next sweeps, as alone."""
    qs = [0, 1, 2]
    solo = _run_blocks(cet, 24, qs, False, stale={1, 2})
    grp = _run_blocks(cet, 24, qs, True, stale={1, 2})
    _same_runs(solo, grp)


def test_rejections_leave_contexts_untouched(cet):
    L = 24
    cases = [_case(cet, L, q) for q in range(2)]
    (a, sa, la), (b, sb, lb) = cases
    for c, s, _ in cases:
        c.snapshot_state()
        c.sweep_run(3, s, None)                                     # a valid tile state and resident rates
    before = [_snapshot(c) for c, _, _ in cases]
    p, qt = la["tfp"], la["q_top"]()

    def rejected(ctxs):
        with pytest.raises(RuntimeError):
            cet.thermal_full_group(ctxs, [p] * len(ctxs), [qt] * len(ctxs))

    rejected([a, a])                                                # a repeated context
    closed = cet.Context(L=L)
    closed.close()
    rejected([a, closed])                                           # a NULL context
    other, _, _ = _case(cet, 32, 2)
    with pytest.raises(RuntimeError):                               # mixed L
        cet.thermal_full_group([a, other], [p, p], [qt, np.zeros((32, 32))])
    other.close()
    slab = cet.Context(L=L, i_begin=0, i_end=L // 2)
    slab.snapshot_state()
    rejected([a, slab])                                             # a slab
    slab.close()
    box = cet.Context(shape=(L + 2, L, L))                          # not cubic
    box.snapshot_state()
    rejected([b, box])
    box.close()
    fresh = cet.Context(L=L)                                        # no previous state
    with pytest.raises(RuntimeError, match="no previous state"):
        cet.thermal_full_group([a, fresh], [p, p], [qt, qt])
    fresh.close()
    with pytest.raises(RuntimeError, match="n_ctx"):
        cet.thermal_full_group([], [], [])
    with pytest.raises(RuntimeError, match="n_ctx"):
        cet.thermal_full_group([a] * 65, [p] * 65, [qt] * 65)
    lib = cet._lib.lib()
    handles = (C.c_void_p * 2)(a._h.value, b._h.value)
    tfp = (cet._lib.ThermalFullParams * 2)(p, p)
    planes = (C.c_void_p * 2)(qt.ctypes.data, None)
    assert lib.cet_thermal_full_group(handles, 2, tfp, planes, 1) != 0            # q_top[1] NULL
    planes = (C.c_void_p * 2)(qt.ctypes.data, qt.ctypes.data)
    assert lib.cet_thermal_full_group(handles, 2, None, planes, 1) != 0           # NULL params
    assert lib.cet_thermal_full_group(handles, 2, tfp, None, 1) != 0              # NULL planes
    for (c, _, _), s in zip(cases, before):
        _same(_snapshot(c), s)
    # after all that, both continue exactly as twins that saw no rejection
    _group_step(cet, cases)
    got = [(r, _snapshot(c)) for r, (c, _, _) in
           zip(cet.sweep_run_group([a, b], 5, [sa, sb]), cases)]
    _close(cases)
    twins = [_case(cet, L, q) for q in range(2)]
    for c, s, _ in twins:
        c.snapshot_state()
        c.sweep_run(3, s, None)
        _snapshot(c)                                                # as the rejected pair was read
    want = []
    for c, s, l in twins:
        _solo_step(c, l)
        want.append((c.sweep_run(5, s, None), _snapshot(c)))
    _close(twins)
    for (rg, sg), (rw, sw) in zip(got, want):
        assert rg == rw
        _same(sg, sw)


def test_mixed_devices_are_rejected(cet):
    if cet.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = 24
    (a, _, la), = [_case(cet, L, 0)]
    a.snapshot_state()
    far = cet.Context(L=L, device=1)
    far.snapshot_state()
    before = _snapshot(a, rates=False)
    with pytest.raises(RuntimeError, match="another device"):
        cet.thermal_full_group([a, far], [la["tfp"]] * 2, [la["q_top"]()] * 2)
    _same(_snapshot(a, rates=False), before)
    far.close()
    a.close()


def _tree_files(root):
    out = []
    for d, _, fs in os.walk(root):
        out += [os.path.relpath(os.path.join(d, f), root) for f in fs]
    return sorted(out)


MAP = dict(L=24, n_sweeps=61, metrics_every=30, thermal_every=5, n_seeds=6, defect_fraction=3e-3, start=(12.0, 2.0),
           dt=1e-7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_batched_map_writes_the_same_files(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    # the cases of power 300 W start from a W lattice with three empty top-plane sites: they terminate once those fill,
    # inside a metrics interval, and leave their group there (both drivers set up their cases in case order, one
    # _upload_initial call per case)
    powers, speeds = [150.0, 300.0], [0.5, 1.0, 2.0]
    order = [p for p in powers for _ in speeds]
    upload = campaign._upload_initial
    made = [0]

    def upload_initial(ctx, L, n_seeds, temp, impurity_c, lattice, i_begin, i_end):
        power = order[made[0] % len(order)]
        made[0] += 1
        if power == 300.0:
            st = np.ones((L, L, L), np.int64)
            th, ph = np.full((L, L, L), 0.5), np.full((L, L, L), 1.0)
            for j, k in ((3, 4), (11, 17), (20, 9)):
                st[L - 1, j, k] = 0
                th[L - 1, j, k] = ph[L - 1, j, k] = 0.0
            lattice = (st, th, ph, np.full((L, L, L), 2900.0), np.zeros((L, L, L), np.int64))
        return upload(ctx, L, n_seeds, temp, impurity_c, lattice, i_begin, i_end)
    monkeypatch.setattr(campaign, "_upload_initial", upload_initial)
    kw = {} if mask_stream is None else dict(mask_stream=mask_stream)
    a = campaign.run_melt_pool_map(powers, speeds, output_root="plain", **MAP, **kw)
    made[0] = 0
    b = campaign.run_melt_pool_map(powers, speeds, output_root="grouped", batch=4, **MAP, **kw)
    assert len(a) == 6 and a == b
    files = _tree_files("outputs/plain")
    assert files == _tree_files("outputs/grouped") and "melt_pool_map_rank0.csv" in files
    for f in files:
        assert filecmp.cmp(os.path.join("outputs/plain", f), os.path.join("outputs/grouped", f), shallow=False), f
    steps = [int(r["Step"]) for r in a]
    assert steps[:3] == [60, 60, 60]
    assert all(s < 60 for s in steps[3:])                           # the 300 W cases terminated
    assert any(s % 30 != 0 for s in steps[3:])                      # ... inside an interval


def test_unbatched_map_case_is_run_cet_sublattice(cet, tmp_path, monkeypatch):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    campaign.run_melt_pool_map([220.0], [0.75], output_root="map", temp=2750.0, nu_dep=3e13, **MAP)
    m = dict(MAP)
    L, n_sweeps, start, dt = m.pop("L"), m.pop("n_sweeps"), m.pop("start"), m.pop("dt")
    from cetkmc._config import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS
    campaign.run_cet_sublattice(L=L, n_sweeps=n_sweeps, temp=2750.0, nu_dep=3e13, output_prefix="direct", verbose=False,
                                laser=dict(power=220.0, speed=0.75, start=start, dt=dt, beam_radius=DEFAULT_BEAM_RADIUS,
                                           absorptivity=DEFAULT_ABSORPTIVITY), **m)
    assert filecmp.cmp("outputs/map/P220_V0.75/metrics.csv", "outputs/direct/metrics.csv", shallow=False)
