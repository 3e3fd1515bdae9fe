"""GPU: initial lattices built on the device (cet_init_group / cetkmc.init_group) against twin contexts given the
dense arrays by Context.upload: every field has the same bits, and so do the sweeps and laser steps that follow;
rejected calls change nothing.  And the map drivers with replicas: batched and solo runs write the same trees, replica
0 writes what a run without replicas writes, replica r is run_cet_sublattice(seed=seed + r, init_seed=42 + r), and the
ensemble file holds the statistics of the replica files."""
import csv
import filecmp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from cetkmc import _host  # noqa: E402
from cetkmc._config import constants as K  # noqa: E402


def _dev_bytes(ptr, nbytes):
    """A copy of nbytes of device memory at ptr (the context's device is device 0)."""
    import torch

    class Raw:
        __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}
    return torch.as_tensor(Raw(), device="cuda").cpu().numpy()


def _fields(ctx):
    f = ctx.download(state=True, theta=True, phi=True, T=True)
    f["packed"] = ctx.download_packed()
    f["v"] = _dev_bytes(*ctx.device_ptr(5))
    f["T_dev"] = _dev_bytes(*ctx.device_ptr(3))
    f["clock"] = ctx.sweep_state()
    return f


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if k == "clock":
            assert a[k] == b[k]
        else:
            assert np.array_equal(a[k], b[k], equal_nan=True), k


def _spec(L, q):
    """Initial lattice q of a test group: (n_seeds, T_sub, random_seed, impurity_c), with no nuclei, one, a full
    k = 0 plane and carbon-rich lattices among them."""
    n = (20, 0, 1, L * L, 20, 7)[q % 6]
    c = (0.1, 0.5, 1.0 - K.IMPURITY_RE)[q % 3]
    return n, 2650.0 + 25.0 * q, 42 + q, c


def _rp(q):
    from cetkmc._config import rate_params
    return rate_params(0.1, overrides={"NU_DEP": 2e13 * (1 + q % 5)})


def _dense(cet, L, q, snapshot=False):
    n, T_sub, seed, c = _spec(L, q)
    ctx = cet.Context(L=L)
    ctx.set_rate_params(_rp(q))
    st, th, ph, T, at = _host.initialize_lattice(L, n, T_sub, random_seed=seed, impurity_c=c)
    mask, _ = _host.introduce_defects(st, at, T)
    ctx.upload(state=st, theta=th, phi=ph, T=T, defects=mask)
    if snapshot:
        ctx.snapshot_state()
    return ctx


def _grouped(cet, L, qs, snapshot=False):
    """Contexts that held another lattice before (every field must be overwritten), built by one init_group call with
    the group in the order of qs."""
    from cetkmc import _synth
    ctxs = []
    for q in qs:
        ctx = cet.Context(L=L)
        ctx.set_rate_params(_rp(q))
        packed, th, ph, T = _synth.half_grown(L, seed=70 + q, grain=4)
        st, df = _synth.unpack(packed)
        ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
        ctx.snapshot_state()
        ctxs.append(ctx)
    nuclei = []
    for q in qs:
        n, T_sub, seed, c = _spec(L, q)
        nuclei.append(_host.initial_nuclei(L, n, T_sub, seed, c))
    cet.init_group(ctxs, nuclei, snapshot=snapshot)
    return ctxs


def _close(*groups):
    for g in groups:
        for c in g:
            c.close()


@pytest.mark.parametrize("snapshot", [False, True])
@pytest.mark.parametrize("n", [1, 4, 18])              # 18: the 64-entry argument table
@pytest.mark.parametrize("L", [64, 30, 25, 24])
def test_init_group_equals_the_dense_upload(cet, L, n, snapshot):
    qs = list(range(n))[::-1]
    g = _grouped(cet, L, qs, snapshot)
    d = [_dense(cet, L, q, snapshot) for q in qs]
    try:
        for a, b in zip(g, d):
            _same(_fields(a), _fields(b))
    finally:
        _close(g, d)


@pytest.mark.parametrize("L", [64, 30, 25, 24])        # 64: the TMA rebuild; 30, 25, 24: the compact one
def test_sweeps_after_init_group_stay_identical(cet, L):
    from cetkmc._config import thermal_params
    qs = [3, 0, 5, 2]
    g = _grouped(cet, L, qs)
    d = [_dense(cet, L, q) for q in qs]
    try:
        sps, tps = [], []
        for q in qs:
            sp = cet._lib.SweepParams()
            sp.seed, sp.events_per_sweep, sp.p_max = 500 + q, 0.005 * L ** 3, 0.1
            sp.defect_fraction, sp.thermal_every = 3e-3, 10
            sps.append(sp)
            tps.append(thermal_params(1e-6, nan_to_num=True, t_floor=2650.0))
        ra = cet.sweep_run_group(g, 50, sps, tps)
        rb = cet.sweep_run_group(d, 50, sps, tps)
        assert ra == rb and sum(r["events_applied"] for r in ra) > 0
        for a, b in zip(g, d):
            fa, fb = _fields(a), _fields(b)
            fa["site_rate"], fa["dep_rate"] = a.rates_download()
            fb["site_rate"], fb["dep_rate"] = b.rates_download()
            _same(fa, fb)
            assert a.grains()["n"] == b.grains()["n"]
    finally:
        _close(g, d)


@pytest.mark.parametrize("L", [64, 25])
def test_snapshot_feeds_the_laser_step(cet, L):
    """init_group(snapshot=True) leaves the previous state that cet_snapshot_state leaves: the latent-heat term of the
    next laser steps, with sweeps between them, gives the same bits."""
    from cetkmc._config import thermal_full_params
    from cetkmc.thermal_solver import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS, laser_source_top
    qs = [1, 4]
    g = _grouped(cet, L, qs, snapshot=True)
    d = [_dense(cet, L, q, snapshot=True) for q in qs]
    try:
        tfp = [thermal_full_params(1e-7) for _ in qs]
        sps = []
        for q in qs:
            sp = cet._lib.SweepParams()
            sp.seed, sp.events_per_sweep, sp.p_max, sp.defect_fraction, sp.thermal_every = 9 + q, 0.005 * L ** 3, 0.1, 0.0, 0
            sps.append(sp)
        for step in range(3):
            q_tops = [laser_source_top(L, (L / 2, 2.0 * step), 250.0, DEFAULT_BEAM_RADIUS, DEFAULT_ABSORPTIVITY) for _ in qs]
            cet.thermal_full_group(g, tfp, q_tops, snapshot=True)
            cet.thermal_full_group(d, tfp, q_tops, snapshot=True)
            assert cet.sweep_run_group(g, 5, sps) == cet.sweep_run_group(d, 5, sps)
        for a, b in zip(g, d):
            _same(_fields(a), _fields(b))
    finally:
        _close(g, d)


def test_rejected_calls_change_nothing(cet):
    import ctypes as C
    L = 24
    qs = [0, 1, 2]                                      # 20, 0 and 1 nuclei
    g = _grouped(cet, L, qs)
    other = cet.Context(L=30)
    slab = cet.Context(L=L, i_begin=0, i_end=L // 2)
    try:
        before = [_fields(c) for c in g]
        good = [_host.initial_nuclei(L, *_spec(L, q)) for q in qs]

        def edit(q, i, f):
            nu = [list(x) for x in good]
            nu[q][i] = f(nu[q][i].copy())
            return [tuple(x) for x in nu]
        bad_calls = [
            ("outside the k = 0 plane", g, edit(2, 0, lambda s: s + 1)),
            ("outside the k = 0 plane", g, edit(0, 0, lambda s: np.where(np.arange(len(s)) == 3, L ** 3, s))),
            ("outside the k = 0 plane", g, edit(0, 0, lambda s: np.where(np.arange(len(s)) == 0, -L, s))),
            ("repeats site", g, edit(0, 0, lambda s: np.where(np.arange(len(s)) == 1, s[0], s))),
            ("byte", g, edit(0, 1, lambda b: np.where(np.arange(len(b)) == 0, 4, b).astype(np.uint8))),
            ("byte", g, edit(0, 1, lambda b: np.where(np.arange(len(b)) == 0, 0, b).astype(np.uint8))),
            ("byte", g, edit(2, 1, lambda b: (b | 0x20).astype(np.uint8))),
            ("repeats context", [g[0], g[1], g[0]], good),
            ("L = 30", [g[0], other, g[2]], [good[0], _host.initial_nuclei(30, *_spec(30, 1)), good[2]]),
            ("slab", [g[0], g[1], slab], good),
            ("n_ctx", g * 22, good * 22),
        ]
        for msg, ctxs, nuclei in bad_calls:
            with pytest.raises(RuntimeError, match=msg):
                cet.init_group(ctxs, nuclei)
        # a NULL nucleus array with a non-zero count, through the C-ABI
        descs = (cet._lib.InitDesc * 3)(*[cet._lib.InitDesc(len(nu[0]), *[a.ctypes.data for a in nu]) for nu in good])
        descs[0].theta = None                                       # context 0 has 20 nuclei
        handles = (C.c_void_p * 3)(*[c._h.value for c in g])
        assert cet._lib.lib().cet_init_group(handles, 3, descs, 0) != 0
        assert b"NULL" in cet._lib.lib().cet_last_error()
        for c, f in zip(g, before):
            _same(_fields(c), f)
    finally:
        _close(g, [other, slab])


# -- the map drivers with replicas ------------------------------------------------------------------------------------

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


def _terminating_replica(monkeypatch, campaign, temp):
    """Replica 1 of the cases at T_sub = temp starts from a W lattice with three empty top-plane sites: it terminates
    early, inside an interval, in solo and grouped runs alike."""
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


GR = dict(L=24, n_sweeps=61, metrics_every=20, n_seeds=6, defect_fraction=3e-3, seed=7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_gr_sweep_replicas(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign
    monkeypatch.chdir(tmp_path)
    kw = dict(GR, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    temps, nu_deps = [2700.0, 3000.0], [2e13, 1e14]
    base = campaign.run_gr_sweep(temps, nu_deps, output_root="base", **kw)
    _terminating_replica(monkeypatch, campaign, 3000.0)
    a, ens_a = campaign.run_gr_sweep(temps, nu_deps, output_root="solo", replicas=3, **kw)
    b, ens_b = campaign.run_gr_sweep(temps, nu_deps, output_root="grouped", replicas=3, batch=4, **kw)
    assert a == base and b == base and ens_a == ens_b
    files = _same_tree("outputs/solo", "outputs/grouped")
    assert sum(f.endswith("/metrics.csv") for f in files) == 4 * 3
    assert sum(f.startswith("plot_cet/") for f in files) == 4                 # replica 0 of each case
    # replica 0 and the map files are those of the run without replicas
    for f in _tree_files("outputs/base"):
        assert filecmp.cmp(os.path.join("outputs/base", f), os.path.join("outputs/solo", f), shallow=False), f
    reps = _read("outputs/solo/cet_map_replicas_rank0.csv")
    assert [(int(r["case"]), int(r["replica"])) for r in reps] == [(q, r) for q in range(4) for r in range(3)]
    stopped = [int(r["Step"]) for r in reps if r["T_sub"] == "3000.0" and r["replica"] == "1"]
    assert stopped and all(s < 60 for s in stopped)
    # replica 2 of case 1 is run_cet_sublattice with seed + 2 and init_seed 44
    campaign.run_cet_sublattice(temp=2700.0, nu_dep=1e14, output_prefix="direct", verbose=False, init_seed=44,
                                **dict(kw, seed=9))
    assert filecmp.cmp("outputs/direct/metrics.csv", "outputs/solo/T2700_R1e+14/rep2/metrics.csv", shallow=False)
    # the ensemble: statistics of the replica files
    campaign.merge_cet_map("solo")
    stats = campaign.ensemble_stats(reps, ("T_sub", "NU_DEP"))
    assert _read("outputs/solo/cet_map_ensemble.csv") == [{k: str(v) for k, v in e.items()} for e in stats]
    assert [{k: str(v) for k, v in e.items()} for e in ens_a] == [{k: str(v) for k, v in e.items()} for e in stats]
    for e, q in zip(stats, range(4)):
        ar = [float(r["AspectRatio"]) for r in reps if int(r["case"]) == q]
        assert e["replicas"] == 3 and e["AspectRatio_mean"] == float(np.mean(ar))
        assert e["AspectRatio_se"] == float(np.std(ar, ddof=1) / np.sqrt(3))


MAP = dict(L=24, n_sweeps=61, metrics_every=30, thermal_every=5, n_seeds=6, defect_fraction=3e-3, start=(12.0, 2.0),
           dt=1e-7)


@pytest.mark.parametrize("mask_stream", [None, "philox"])
def test_melt_pool_map_replicas(cet, tmp_path, monkeypatch, mask_stream):
    from cetkmc import campaign
    from cetkmc._config import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS
    monkeypatch.chdir(tmp_path)
    kw = dict(MAP, **({} if mask_stream is None else dict(mask_stream=mask_stream)))
    powers, speeds = [150.0, 300.0], [1.0]
    _terminating_replica(monkeypatch, campaign, 2900.0)
    a, ens_a = campaign.run_melt_pool_map(powers, speeds, output_root="solo", temp=2900.0, replicas=3, **kw)
    b, ens_b = campaign.run_melt_pool_map(powers, speeds, output_root="grouped", temp=2900.0, replicas=3, batch=4, **kw)
    assert a == b and ens_a == ens_b
    _same_tree("outputs/solo", "outputs/grouped")
    reps = _read("outputs/solo/melt_pool_map_replicas_rank0.csv")
    assert [int(r["Step"]) < 60 for r in reps if r["replica"] == "1"] == [True, True]
    # replica r of case 1 against run_cet_sublattice(seed=42 + r, init_seed=42 + r); replica 0 against a run without
    # replicas
    m = dict(kw)
    L, n_sweeps, start, dt = m.pop("L"), m.pop("n_sweeps"), m.pop("start"), m.pop("dt")
    laser = dict(power=300.0, speed=1.0, start=start, dt=dt, beam_radius=DEFAULT_BEAM_RADIUS,
                 absorptivity=DEFAULT_ABSORPTIVITY)
    campaign.run_cet_sublattice(L=L, n_sweeps=n_sweeps, temp=2900.0, output_prefix="direct", verbose=False, laser=laser,
                                seed=K.RANDOM_SEED + 2, init_seed=44, **m)
    assert filecmp.cmp("outputs/direct/metrics.csv", "outputs/solo/P300_V1/rep2/metrics.csv", shallow=False)
    campaign.run_melt_pool_map(powers, speeds, output_root="plain", temp=2900.0, **kw)
    for f in _tree_files("outputs/plain"):
        assert filecmp.cmp(os.path.join("outputs/plain", f), os.path.join("outputs/solo", f), shallow=False), f
    campaign.merge_melt_pool_map("solo")
    stats = campaign.ensemble_stats(reps, ("power", "speed", "T_sub", "NU_DEP"))
    assert _read("outputs/solo/melt_pool_map_ensemble.csv") == [{k: str(v) for k, v in e.items()} for e in stats]
