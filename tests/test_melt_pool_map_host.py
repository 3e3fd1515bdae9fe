"""Host logic of the melt-pool map that needs no device: the argument checks of cetkmc.thermal_full_group that run
before the library is called, the arguments run_melt_pool_map refuses, and which run each case of the map is."""
import csv
import ctypes as C
import os

import numpy as np
import pytest

from cetkmc import _lib, campaign


@pytest.fixture
def no_library(monkeypatch):
    def lib():
        raise AssertionError("the library must not be reached")
    monkeypatch.setattr(_lib, "lib", lib)


@pytest.fixture
def fake_ctxs():
    """Context objects of an 8^3 lattice with a dummy handle and no library behind them."""
    made = []

    def make(n, L=8):
        for _ in range(n):
            c = object.__new__(_lib.Context)
            c._h, c.shape = C.c_void_p(1), (L, L, L)
            made.append(c)
        return made[-n:]
    yield make
    for c in made:
        c._h = C.c_void_p(None)                  # nothing to destroy


def _planes(n, L=8):
    return [np.zeros((L, L), np.float64) for _ in range(n)]


def test_thermal_full_group_checks_lists_before_the_library(no_library, fake_ctxs):
    p = _lib.ThermalFullParams()
    a, b = fake_ctxs(2)
    with pytest.raises(ValueError, match="params"):
        _lib.thermal_full_group([a, b], [p], _planes(2))
    with pytest.raises(ValueError, match="source planes"):
        _lib.thermal_full_group([a, b], [p, p], _planes(1))
    with pytest.raises(TypeError):
        _lib.thermal_full_group([a], [_lib.ThermalParams()], _planes(1))
    with pytest.raises(TypeError):
        _lib.thermal_full_group([object()], [p], _planes(1))


def test_thermal_full_group_checks_the_source_planes_before_the_library(no_library, fake_ctxs):
    p = _lib.ThermalFullParams()
    a, b = fake_ctxs(2)
    good = _planes(1)[0]
    with pytest.raises(TypeError):                                   # float32
        _lib.thermal_full_group([a, b], [p, p], [good, good.astype(np.float32)])
    with pytest.raises(TypeError):                                   # not C-contiguous
        _lib.thermal_full_group([a, b], [p, p], [good, np.zeros((8, 16))[:, ::2]])
    with pytest.raises(TypeError):                                   # not an array
        _lib.thermal_full_group([a], [p], [good.tolist()])
    with pytest.raises(ValueError):                                  # wrong shape
        _lib.thermal_full_group([a, b], [p, p], [good, np.zeros((8, 9))])
    with pytest.raises(ValueError):
        _lib.thermal_full_group([a], [p], [np.zeros(64)])


def test_thermal_full_group_is_bound_and_exported():
    import cetkmc
    assert cetkmc.thermal_full_group is _lib.thermal_full_group
    assert "cet_thermal_full_group" in _lib.SIGNATURES
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "cetkmc.h")).read()
    assert "int cet_thermal_full_group(" in header


@pytest.mark.parametrize("args, kw", [(([], [1.0]), {}), (([100.0], []), {}), (([100.0], [1.0]), dict(thermal_every=0)),
                                      (([100.0], [1.0]), dict(thermal_every=-3))])
def test_map_refuses_empty_axes_and_no_laser_step(args, kw, tmp_path, monkeypatch, no_library):
    monkeypatch.chdir(tmp_path)
    for batch in (None, 2):
        with pytest.raises(ValueError):
            campaign.run_melt_pool_map(*args, L=8, n_sweeps=3, batch=batch, **kw)


@pytest.mark.parametrize("kw", [dict(checkpoint_every=1), dict(resume_from="x"), dict(lattice=(1, 2, 3, 4, 5)),
                                dict(batch=0), dict(batch=_lib.GROUP_MAX + 1)])
def test_batched_map_refuses_single_lattice_features(kw, tmp_path, monkeypatch, no_library):
    monkeypatch.chdir(tmp_path)
    kw = dict(dict(batch=2), **kw)
    with pytest.raises(ValueError):
        campaign.run_melt_pool_map([100.0], [1.0], L=8, n_sweeps=3, **kw)


_ROW = dict(Step=7, Time=1.5e-9, AspectRatio=1.25, EquiaxedFraction=0.5, GrainCount=3, AvgGrainSize=4.0,
            NucleationCount=2, CET_Class="columnar", CET_Detected=False)


def _fake_metrics(prefix, extra=None):
    os.makedirs(f"outputs/{prefix}", exist_ok=True)
    row = dict(_ROW, **(extra or {}))
    with open(f"outputs/{prefix}/metrics.csv", "w", newline="") as fh:
        w = csv.DictWriter(fh, fieldnames=list(row))
        w.writeheader()
        w.writerow(row)


def test_map_cases_run_powers_by_speeds_with_their_prefixes(tmp_path, monkeypatch, no_library):
    monkeypatch.chdir(tmp_path)
    calls = []

    def solo(**kw):
        calls.append(kw)
        _fake_metrics(kw["output_prefix"], dict(Step=len(calls)))
    monkeypatch.setattr(campaign, "run_cet_sublattice", solo)
    rows = campaign.run_melt_pool_map([100, 250.5], [0.5, 2], L=8, n_sweeps=5, temp=2700.0, nu_dep=3e13,
                                      start=(4.0, 1.0), dt=2e-7, beam_radius=4e-5, absorptivity=0.3, n_seeds=3,
                                      output_root="mp", metrics_every=2, thermal_every=3, seed=11)
    want = [(100.0, 0.5), (100.0, 2.0), (250.5, 0.5), (250.5, 2.0)]
    assert [c["output_prefix"] for c in calls] == ["mp/P100_V0.5", "mp/P100_V2", "mp/P250.5_V0.5", "mp/P250.5_V2"]
    for c, (P, V) in zip(calls, want):
        assert c["laser"] == dict(power=P, speed=V, start=(4.0, 1.0), dt=2e-7, beam_radius=4e-5, absorptivity=0.3)
        assert (c["temp"], c["nu_dep"], c["L"], c["n_sweeps"], c["n_seeds"]) == (2700.0, 3e13, 8, 5, 3)
        assert (c["metrics_every"], c["thermal_every"], c["seed"], c["device"], c["verbose"]) == (2, 3, 11, 0, False)
    G, R, _rp, _ = campaign._gr(8, 2700.0, 3e13)
    assert [(r["case"], r["power"], r["speed"]) for r in rows] == [(q,) + pv for q, pv in enumerate(want)]
    with open("outputs/mp/melt_pool_map_rank0.csv") as fh:
        got = list(csv.DictReader(fh))
    assert list(got[0]) == ["case", "power", "speed", "T_sub", "NU_DEP", "G", "R", "G_over_R", "Step", "Time", "AspectRatio",
                            "EquiaxedFraction", "GrainCount", "AvgGrainSize", "NucleationCount", "CET_Class", "CET_Detected"]
    assert [int(r["Step"]) for r in got] == [1, 2, 3, 4]
    assert float(got[0]["G"]) == G and float(got[0]["R"]) == R and float(got[0]["G_over_R"]) == G / R
    for q in range(4):
        assert os.path.exists(f"outputs/mp/plot_cet/outputs/impurity_c_{q}/metrics_{q}.csv")
    merged = campaign.merge_melt_pool_map("mp")
    assert [int(r["case"]) for r in merged] == [0, 1, 2, 3] and os.path.exists("outputs/mp/melt_pool_map.csv")


def test_map_defaults_and_ranks(tmp_path, monkeypatch, no_library):
    from cetkmc import kmc_simulation as ks
    from cetkmc._config import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS, constants
    monkeypatch.chdir(tmp_path)
    calls = []

    def solo(**kw):
        calls.append(kw)
        _fake_metrics(kw["output_prefix"])
    monkeypatch.setattr(campaign, "run_cet_sublattice", solo)
    rows = campaign.run_melt_pool_map([1.0, 2.0, 3.0], [4.0], L=8, n_sweeps=5, rank=1, world=2, devices=[0, 1])
    assert [r["case"] for r in rows] == [1]
    (c,) = calls
    assert c["laser"] == dict(power=2.0, speed=4.0, start=(0.0, 0.0), dt=ks.THERMAL_DT, beam_radius=DEFAULT_BEAM_RADIUS,
                              absorptivity=DEFAULT_ABSORPTIVITY)
    assert (c["temp"], c["nu_dep"], c["device"]) == (constants.T_SUB, constants.NU_DEP, 0)
    assert os.path.exists("outputs/melt_pool_map/melt_pool_map_rank1.csv")


def test_batched_map_passes_groups_with_their_lasers(tmp_path, monkeypatch, no_library):
    monkeypatch.chdir(tmp_path)
    groups = []

    def grouped(cases, **kw):
        groups.append((cases, kw))
        for prefix, _t, _r in cases:
            _fake_metrics(prefix)
    monkeypatch.setattr(campaign, "_run_cases_grouped", grouped)
    rows = campaign.run_melt_pool_map([10.0, 20.0, 30.0], [1.0, 2.0], L=8, n_sweeps=5, temp=2900.0, nu_dep=1e13, batch=4,
                                      metrics_every=2, mask_stream="philox")
    assert [r["case"] for r in rows] == list(range(6))
    assert [[p for p, _t, _r in cases] for cases, _kw in groups] == [
        ["melt_pool_map/P10_V1", "melt_pool_map/P10_V2", "melt_pool_map/P20_V1", "melt_pool_map/P20_V2"],
        ["melt_pool_map/P30_V1", "melt_pool_map/P30_V2"]]
    cases, kw = groups[1]
    assert all((t, r) == (2900.0, 1e13) for _p, t, r in cases)
    assert [(d["power"], d["speed"]) for d in kw["lasers"]] == [(30.0, 1.0), (30.0, 2.0)]
    assert kw["metrics_every"] == 2 and kw["mask_stream"] == "philox" and kw["device"] == 0


def test_grouped_driver_refuses_a_laser_without_thermal_steps(no_library):
    with pytest.raises(ValueError):
        campaign._run_cases_grouped([("x", 2800.0, 2e13)], L=8, n_sweeps=3, impurity_c=0.0, n_seeds=2, defect_fraction=0.0,
                                    device=0, thermal_every=0, lasers=[dict(power=1.0)])
