"""Front conditions (cetkmc.front_group): one grouped call over B lattices against B back-to-back groups of one, the same
lattices' grouped metrics row (cetkmc.metrics_group) for scale, the launches and copies of one call with its kernel
time and achieved bytes/s, and the maps: the 16-case 96^3 G-R map and a small melt-pool map, each without and with
front_axis=2.  Writes one JSON file.

    python scripts/bench_front_group.py --out profiles/front_group.json [--quick]

Lattices are half-grown: _synth.half_grown with fill = 1, a dense solid below the wavy front k < L/2 + 8 sin(2 pi i / L)
and the linear T of the benchmark, one seed per lattice.  Each timing point: one warm-up call per path, then REPS calls
per path, the paths alternated, host clock around calls that end in a device synchronise; the median is reported.
The vox bytes of 64 x 128^3 lattices (134 MB) exceed the 126 MB L2, those of the smaller groups fit; no cache flush is
done between repetitions, as in the driver's cadence, which reads the same lattices just before.
"""
import argparse
import filecmp
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import cetkmc  # noqa: E402
from cetkmc import _lib, _synth, campaign  # noqa: E402
from cetkmc import metrics as _metrics  # noqa: E402
from cetkmc._config import constants, rate_params  # noqa: E402
from bench_sweep_group import gpu_info  # noqa: E402

REPS, AXIS = 9, 2


def lattices(L, B):
    ctxs = []
    for q in range(B):
        packed, th, ph, T = _synth.half_grown(L, seed=500 + q, grain=4, fill=1.0)
        st, df = _synth.unpack(packed)
        ctx = cetkmc.Context(L=L)
        ctx.set_rate_params(rate_params(0.1, 1, 2, 3))
        ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
        ctxs.append(ctx)
    return ctxs


def metrics_params(ctxs):
    n_sites = int(np.prod(ctxs[0].owned_shape))
    out = []
    for _ in ctxs:
        p = _lib.MetricsParams()
        p.theta_threshold, p.ar_threshold = 0.5, constants.CET_AR_THRESHOLD
        p.pct_pos[:] = _metrics.percentile_positions(n_sites)
        p.refresh = 0
        out.append(p)
    return out


def clock(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def algorithmic_bytes(L, B):
    """n L^3 vox bytes, at most two T reads per column, and the output (two int32 and two float64 per column)."""
    return B * L ** 3 + B * L * L * 2 * 8 + B * L * L * 2 * (4 + 8)


def time_point(ctxs, L, B):
    group = ctxs[:B]
    mp = metrics_params(group)
    paths = dict(grouped=lambda: cetkmc.front_group(group, AXIS),
                 b2b=lambda: [cetkmc.front_group([c], AXIS) for c in group])
    got = cetkmc.front_group(group, AXIS)
    solo = [cetkmc.front_group([c], AXIS) for c in group]
    assert all(np.array_equal(got["front"][q], solo[q]["front"][0]) for q in range(B))
    t = {k: [] for k in paths}
    for _ in range(REPS):
        for k, fn in paths.items():
            t[k].append(clock(fn))
    tm = [clock(lambda: cetkmc.metrics_group(group, mp)) for _ in range(REPS)]
    g, s, m = (float(np.median(v)) for v in (t["grouped"], t["b2b"], tm))
    return dict(L=L, B=B, axis=AXIS, ms_grouped=g, ms_grouped_reps=t["grouped"], ms_b2b=s, ms_b2b_reps=t["b2b"],
                b2b_over_grouped=s / g, ms_metrics_group_row=m, ms_metrics_group_row_reps=tm, front_over_metrics_row=g / m,
                front_mean=float(np.mean(got["front"])))


def launches(ctxs, L, B):
    """Kernel launches and copies of one grouped call on every axis, counted by torch.profiler, with the kernel's
    device time and the achieved bytes/s over algorithmic_bytes."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    group = ctxs[:B]
    out = []
    for axis in range(3):
        cetkmc.front_group(group, axis)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(REPS):
                cetkmc.front_group(group, axis)
            torch.cuda.synchronize()
        k = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        copies = [e for e in k if "memcpy" in e.name.lower()]
        memsets = [e for e in k if "memset" in e.name.lower()]
        kernels = [e for e in k if e not in copies and e not in memsets]
        us = float(np.median([e.device_time for e in kernels])) if kernels else None
        nb = algorithmic_bytes(L, B)
        out.append(dict(L=L, B=B, axis=axis, kernel_launches_per_call=len(kernels) / REPS,
                        copies_per_call=len(copies) / REPS, memsets_per_call=len(memsets) / REPS,
                        kernels=sorted({e.name.split("(")[0] for e in kernels}), kernel_us_median=us,
                        algorithmic_bytes=nb, achieved_GB_s=(nb / (us * 1e-6) / 1e9) if us else None))
        print(json.dumps(out[-1]), flush=True)
    return out


def _tree_files(root):
    out = []
    for d, _, fs in os.walk(root):
        out += [os.path.relpath(os.path.join(d, f), root) for f in fs]
    return sorted(out)


def maps(quick=False):
    """scripts/run_gr_sweep.py's 16-case 96^3 grid (batch=16) and a small melt-pool map (2 powers x 2 speeds, 64^3,
    batch=4; the melt-pool script's settings otherwise), each without and with front_axis=2.  Every file of the run
    without front_axis must be byte-identical in the run with it; the map front files are kept."""
    gr = dict(temps=[2600.0, 2800.0, 3000.0, 3200.0], nu_deps=[1e12, 5e12, 2e13, 1e14], L=96, n_sweeps=401, batch=16)
    mp = dict(powers=[100.0, 400.0], speeds=[0.5, 2.0], L=64, n_sweeps=401, batch=4)
    if quick:
        gr.update(temps=gr["temps"][:2], nu_deps=gr["nu_deps"][:2], L=32, n_sweeps=41, batch=4)
        mp.update(L=32, n_sweeps=41)
    out = {}
    with tempfile.TemporaryDirectory() as d:
        cwd = os.getcwd()
        os.chdir(d)
        try:
            for name, fn, merge in (("gr", lambda root, kw: campaign.run_gr_sweep(
                                        gr["temps"], gr["nu_deps"], L=gr["L"], n_sweeps=gr["n_sweeps"], n_seeds=20,
                                        defect_fraction=3e-3, impurity_c=0.1, output_root=root, metrics_every=100,
                                        batch=gr["batch"], **kw), campaign.merge_cet_map),
                                    ("melt_pool", lambda root, kw: campaign.run_melt_pool_map(
                                        mp["powers"], mp["speeds"], L=mp["L"], n_sweeps=mp["n_sweeps"],
                                        start=(mp["L"] / 2, 0.0), n_seeds=20, defect_fraction=3e-3, impurity_c=0.1,
                                        output_root=root, metrics_every=100, batch=mp["batch"], **kw),
                                     campaign.merge_melt_pool_map)):
                runs = []
                for axis in (None, AXIS):
                    root = f"{name}_{axis}"
                    t0 = time.perf_counter()
                    fn(root, {} if axis is None else dict(front_axis=axis))
                    merge(root)
                    runs.append(dict(front_axis=axis, wall_s=time.perf_counter() - t0))
                plain = _tree_files(f"outputs/{name}_None")
                runs[1]["preexisting_files_identical"] = all(
                    filecmp.cmp(os.path.join(f"outputs/{name}_None", f), os.path.join(f"outputs/{name}_{AXIS}", f),
                                shallow=False) for f in plain)
                mname = "cet_map" if name == "gr" else "melt_pool_map"
                for f in (f"{mname}.csv", f"{mname}_front.csv"):
                    with open(f"outputs/{name}_{AXIS}/{f}") as fh:
                        runs[1][f] = fh.read()
                out[name] = dict(settings=gr if name == "gr" else mp, runs=runs)
                print(json.dumps({k: v for k, v in runs[1].items()}), flush=True)
        finally:
            os.chdir(cwd)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="front_group.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    _lib.require_gpu()
    res = dict(gpu=gpu_info(), settings=dict(reps=REPS, axis=AXIS, lattices="_synth.half_grown(fill=1.0)"))
    res["time"], res["launches"] = [], []
    Bs = (1, 2) if args.quick else (1, 4, 16, 64)
    for L in ((32,) if args.quick else (64, 96, 128)):
        ctxs = lattices(L, max(Bs))
        try:
            for B in Bs:
                res["time"].append(time_point(ctxs, L, B))
                print(json.dumps({k: v for k, v in res["time"][-1].items() if not k.endswith("_reps")}), flush=True)
            if L == (32 if args.quick else 128):
                res["launches"] += launches(ctxs, L, max(Bs))
        finally:
            for c in ctxs:
                c.close()
    res["maps"] = maps(args.quick)
    res["gpu_after"] = gpu_info()
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
