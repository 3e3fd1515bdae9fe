"""CPU: the drop-in keeps the reference's public surface.  Signature comparison against the live
reference runs in the build container only; the shim resolution test needs the reference too."""
import inspect
import os
import subprocess
import sys

import pytest

import refharness
from conftest import ROOT, golden

PKG = os.path.join(ROOT, "cet-driven-simulation-for-3d-printing-am-kmc-approach_b200")
need_ref = pytest.mark.skipif(not refharness.available(), reason="reference tree not present")

PUBLIC = {
    "kmc_event_rates": ["compute_misorientation", "get_bcc_neighbors", "compute_row_events", "get_event_rates"],
    "kmc_simulation": ["run_kmc"],
    "thermal_solver": ["build_temperature_field", "update_temperature", "update_temperature_cet"],
}


def test_public_names_exist():
    import cetkmc  # noqa: F401
    import importlib
    for mod, names in PUBLIC.items():
        m = importlib.import_module(f"cetkmc.{mod}")
        for n in names:
            assert callable(getattr(m, n)), (mod, n)
    ts = importlib.import_module("cetkmc.thermal_solver")
    assert (ts.K, ts.RHO, ts.CP, ts.DEFAULT_BEAM_RADIUS, ts.DEFAULT_ABSORPTIVITY) == (173.0, 19300.0, 132.0, 50e-6, 0.35)
    assert ts.ALPHA == 173.0 / (19300.0 * 132.0)


@need_ref
def test_signatures_match_reference():
    import importlib
    ref = refharness.load()
    for mod, names in PUBLIC.items():
        ours = importlib.import_module(f"cetkmc.{mod}")
        for n in names:
            theirs = getattr(ref[mod], n)
            theirs = getattr(theirs, "py_func", theirs)              # numba dispatcher -> python function
            want = list(inspect.signature(theirs).parameters.items())
            got = list(inspect.signature(getattr(ours, n)).parameters.items())
            assert [k for k, _ in got[:len(want)]] == [k for k, _ in want], (mod, n)
            for (k, a), (_, b) in zip(got, want):
                assert a.default == b.default or (a.default is inspect.Parameter.empty) == (b.default is inspect.Parameter.empty), (mod, n, k)
            # anything we add beyond the reference's parameters must be optional
            assert all(p.default is not inspect.Parameter.empty for _, p in got[len(want):]), (mod, n)


@need_ref
def test_shims_resolve_in_front_of_reference(tmp_path):
    code = r'''
import sys, types
for n in ("matplotlib", "matplotlib.pyplot", "mpl_toolkits", "mpl_toolkits.mplot3d"):
    sys.modules[n] = types.ModuleType(n)
sys.modules["mpl_toolkits.mplot3d"].Axes3D = object
import kmc_simulation, kmc_event_rates, thermal_solver, utils, metrics
assert kmc_simulation.run_kmc.__module__ == "cetkmc.kmc_simulation"
assert kmc_simulation.initialize_lattice.__module__ == "lattice_init"
assert kmc_simulation.compute_metrics.__module__ == "cetkmc.metrics"
assert metrics.compute_CET.__module__ == "cetkmc.metrics" and metrics.detect_CET_transition.__module__ == "cetkmc.metrics"
assert utils.get_bcc_neighbors.__module__ == "cetkmc.kmc_event_rates"
assert thermal_solver.update_temperature_cet.__module__ == "cetkmc.thermal_solver"
from cetkmc._config import constants
assert constants.source.endswith("constants.py")
print("ok")
'''
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(PKG, "dropin"), refharness.REF_DIR]),
               NUMBA_CACHE_DIR=str(tmp_path / "nbc"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=str(tmp_path))
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_host_metrics_match_reference():
    """hostref.compute_metrics (graph connected components) == the reference's DFS clustering, on the
    reference's own outputs stored by oracle/gen_golden.py (metrics.compute_metrics, utils.get_clusters)."""
    import numpy as np
    import hostref as _host
    for name in ("grains_grown12.npz", "grains_grown16.npz", "grains_half14.npz"):
        g = golden(name)
        st, th, ph, df = g["state"].astype(np.int64), g["theta"], g["phi"], g["defects"].astype(np.int64)
        b = _host.compute_metrics(st, th, ph, defects=df)
        for k in ("AspectRatio", "EquiaxedFraction", "NucleationDensity", "AvgGrainSize", "GrainCount", "DefectDensity",
                  "Grain_d50_um", "Grain_d90_um"):
            a = float(g[f"m_{k}"])
            assert np.isclose(a, b[k], rtol=1e-13, atol=0), (name, k, a, b[k])
        labels, n = _host.label_grains(st, th, ph, 0.5)
        assert n == len(g["sizes"]) and np.array_equal(labels, g["visited"]), name
