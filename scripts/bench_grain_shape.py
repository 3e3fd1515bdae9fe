"""Grain-shape histograms (cetkmc.grain_shape_group): one grouped call over B lattices against B back-to-back groups of
one, the same lattices' grouped metrics row (cetkmc.metrics_group) for scale, the launches, memsets and copies of one
call, and the 16-case 96^3 G-R driver with batch=16 without and with shape_axis=2, with the call's default min_size (8)
and with min_size 1.  Writes one JSON file.

    python scripts/bench_grain_shape.py --out profiles/grain_shape.json [--quick]

Lattices are the driver's own (run_gr_sweep's set-up: initialize_lattice with 20 seeds, impurity_c = 0.1, its sweep
parameters) advanced by ADVANCE sweeps and labelled by one metrics_group row.  Each timing point: one warm-up call per
path, then REPS calls per path, the paths alternated, host clock around calls that end in a device synchronise; the
median is reported.  Labels and moment buffers of up to 64 x 128^3 lattices partly fit in the 126 MB L2; that is the
regime the driver runs in, so no cache flush is done between repetitions.
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
from cetkmc import _lib, campaign  # noqa: E402
from cetkmc import metrics as _metrics  # noqa: E402
from cetkmc._config import constants, rate_params  # noqa: E402
from bench_sweep_group import gpu_info  # noqa: E402

ADVANCE, REPS, AXIS = 300, 7, 2
TEMPS, NU_DEPS = (2600.0, 2800.0, 3000.0, 3200.0), (1e12, 5e12, 2e13, 1e14)


def lattices(L, B, seed=42):
    """B of the driver's cases (its T_sub x NU_DEP grid, repeated) advanced by ADVANCE sweeps together."""
    ctxs, sps, tps = [], [], []
    for q in range(B):
        temp, nu_dep = TEMPS[(q // 4) % 4], NU_DEPS[q % 4]
        np.random.seed(seed)
        ctx = cetkmc.Context(L=L)
        ctx.set_rate_params(rate_params(0.1, 1, 2, 3, overrides={"NU_DEP": nu_dep}))
        campaign._upload_initial(ctx, L, 20, temp, 0.1, None, 0, L)
        sp, tp = campaign._sweep_setup(L, seed + q, temp, None, 0.1, 3e-3, 20)
        ctxs.append(ctx); sps.append(sp); tps.append(tp)
    cetkmc.sweep_run_group(ctxs, ADVANCE, sps, tps)
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


def time_point(L, B):
    ctxs = lattices(L, B)
    mp = metrics_params(ctxs)
    rows = cetkmc.metrics_group(ctxs, mp)
    paths = dict(grouped=lambda: cetkmc.grain_shape_group(ctxs, AXIS),
                 b2b=lambda: [cetkmc.grain_shape_group([c], AXIS) for c in ctxs])
    got = cetkmc.grain_shape_group(ctxs, AXIS)
    assert np.array_equal(got, np.concatenate([cetkmc.grain_shape_group([c], AXIS) for c in ctxs]))
    assert all(int(got[q, 1].sum()) == rows[q]["size_sum"] and int(got[q, 0].sum()) == rows[q]["n_grains"]
               for q in range(B))
    t = {k: [] for k in paths}
    for _ in range(REPS):
        for k, fn in paths.items():
            t[k].append(clock(fn))
    # the metrics row the histogram follows in the driver's cadence (it relabels; the histogram of its labelling is
    # the same)
    tm = [clock(lambda: cetkmc.metrics_group(ctxs, mp)) for _ in range(REPS)]
    n_grains = [r["n_grains"] for r in rows]
    for c in ctxs:
        c.close()
    g, s, m = (float(np.median(v)) for v in (t["grouped"], t["b2b"], tm))
    return dict(L=L, B=B, axis=AXIS, ms_grouped=g, ms_grouped_reps=t["grouped"], ms_b2b=s, ms_b2b_reps=t["b2b"],
                b2b_over_grouped=s / g, ms_metrics_group_row=m, ms_metrics_group_row_reps=tm,
                shape_over_metrics_row=g / m, grains_min=min(n_grains), grains_max=max(n_grains))


def launches(L, B):
    """Kernel launches, memsets and copies of one grouped call, counted by torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctxs = lattices(L, B)
    cetkmc.metrics_group(ctxs, metrics_params(ctxs))
    cetkmc.grain_shape_group(ctxs, AXIS)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        cetkmc.grain_shape_group(ctxs, AXIS)
        torch.cuda.synchronize()
    k = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    memsets = [e for e in k if "memset" in e.name.lower()]
    copies = [e for e in k if "memcpy" in e.name.lower()]
    kernels = [e for e in k if e not in memsets and e not in copies]
    names = {}
    for e in kernels:
        nm = e.name.split("(")[0].split("<")[0]
        names[nm] = names.get(nm, 0) + 1
    for c in ctxs:
        c.close()
    return dict(L=L, B=B, kernel_launches=len(kernels), memsets=len(memsets), copies=len(copies),
                copy_names=sorted({e.name for e in copies}), kernels=names)


def _tree_files(root):
    out = []
    for d, _, fs in os.walk(root):
        out += [os.path.relpath(os.path.join(d, f), root) for f in fs]
    return sorted(out)


def driver(n_side=4, L=96, n_sweeps=401, batch=16):
    """run_gr_sweep over scripts/run_gr_sweep.py's 16-case grid on one GPU with batch=16: without shape_axis, with
    shape_axis=2, and with shape_axis=2 and the call's min_size set to 1 (the binding wrapped for that run only), then
    again without.  Every file of a run without shape_axis must be byte-identical in the runs with it; per case the
    final row's ColumnarVolumeFraction at min_size 8 and 1."""
    temps, nu_deps = list(TEMPS[:n_side]), list(NU_DEPS[:n_side])
    order = ((None, 8), (AXIS, 8), (AXIS, 1), (None, 8))
    out = []
    orig = _lib.grain_shape_group
    with tempfile.TemporaryDirectory() as d:
        cwd = os.getcwd()
        os.chdir(d)
        try:
            for rep, (axis, min_size) in enumerate(order):
                root = f"run{rep}"
                kw = {} if axis is None else dict(shape_axis=axis)
                _lib.grain_shape_group = orig if min_size == 8 else (
                    lambda ctxs, ax, edges=_lib.SHAPE_EDGES, min_size=8: orig(ctxs, ax, edges, 1))
                t0 = time.perf_counter()
                try:
                    campaign.run_gr_sweep(temps, nu_deps, L=L, n_sweeps=n_sweeps, n_seeds=20, defect_fraction=3e-3,
                                          impurity_c=0.1, output_root=root, metrics_every=100, batch=batch, **kw)
                finally:
                    _lib.grain_shape_group = orig
                campaign.merge_cet_map(root)
                wall = time.perf_counter() - t0
                out.append(dict(shape_axis=axis, min_size=min_size, wall_s=wall, files=len(_tree_files(f"outputs/{root}"))))
                print(json.dumps(out[-1]), flush=True)
            files = _tree_files("outputs/run0")
            for i, (axis, min_size) in enumerate(order):
                out[i]["preexisting_files_identical_to_run0"] = all(
                    filecmp.cmp(os.path.join("outputs/run0", f), os.path.join(f"outputs/run{i}", f), shallow=False)
                    for f in files)
                if axis is not None:
                    with open(f"outputs/run{i}/cet_map_shape.csv") as fh:
                        out[i]["cet_map_shape"] = fh.read()
                    with open(f"outputs/run{i}/cet_map.csv") as fh:
                        out[i]["cet_map"] = fh.read()
        finally:
            os.chdir(cwd)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="grain_shape.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    _lib.require_gpu()
    res = dict(gpu=gpu_info(), settings=dict(advance_sweeps=ADVANCE, reps=REPS, axis=AXIS, edges=_lib.SHAPE_EDGES,
                                             min_size=_lib.SHAPE_MIN_SIZE))
    res["time"] = []
    for L in ((32,) if args.quick else (64, 96, 128)):
        for B in ((1, 2) if args.quick else (1, 4, 16, 64)):
            res["time"].append(time_point(L, B))
            print(json.dumps({k: v for k, v in res["time"][-1].items() if not k.endswith("_reps")}), flush=True)
    res["launches"] = []
    for L, B in (((32, 1), (32, 2)) if args.quick else ((64, 1), (64, 4), (96, 16), (128, 64))):
        res["launches"].append(launches(L, B))
        print(json.dumps(res["launches"][-1]), flush=True)
    res["driver"] = driver(2, 32, 41, 4) if args.quick else driver()
    res["gpu_after"] = gpu_info()
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
