"""Per-plane grain profiles (cetkmc.grain_profile_group): one grouped call over B lattices against B back-to-back groups
of one, the same lattices' grouped metrics row (cetkmc.metrics_group) for scale, the launches and copies of one call,
and the 16-case 96^3 G-R driver with batch=16 with and without profile_axis=2.  Writes one JSON file.

    python scripts/bench_grain_profile.py --out profiles/grain_profile.json [--quick]

Lattices are the driver's own (run_gr_sweep's set-up: initialize_lattice with 20 seeds, impurity_c = 0.1, its sweep
parameters) advanced by ADVANCE sweeps and labelled by one metrics_group row.  Each timing point: one warm-up call per
path, then REPS calls per path, the paths alternated, host clock around calls that end in a device synchronise; the
median is reported.  Labels and grain buffers of up to 64 x 128^3 lattices partly fit in the 126 MB L2; that is the
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
    thr = constants.CET_AR_THRESHOLD
    paths = dict(grouped=lambda: cetkmc.grain_profile_group(ctxs, AXIS, thr),
                 b2b=lambda: [cetkmc.grain_profile_group([c], AXIS, thr) for c in ctxs])
    got = cetkmc.grain_profile_group(ctxs, AXIS, thr)
    assert np.array_equal(got, np.concatenate([cetkmc.grain_profile_group([c], AXIS, thr) for c in ctxs]))
    assert all(int(got[q, 0].sum()) == rows[q]["size_sum"] for q in range(B))
    t = {k: [] for k in paths}
    for _ in range(REPS):
        for k, fn in paths.items():
            t[k].append(clock(fn))
    # the metrics row the profile follows in the driver's cadence (it relabels; the profile of its labelling is the same)
    tm = [clock(lambda: cetkmc.metrics_group(ctxs, mp)) for _ in range(REPS)]
    n_grains = [r["n_grains"] for r in rows]
    for c in ctxs:
        c.close()
    g, s, m = (float(np.median(v)) for v in (t["grouped"], t["b2b"], tm))
    return dict(L=L, B=B, axis=AXIS, ms_grouped=g, ms_grouped_reps=t["grouped"], ms_b2b=s, ms_b2b_reps=t["b2b"],
                b2b_over_grouped=s / g, ms_metrics_group_row=m, ms_metrics_group_row_reps=tm,
                profile_over_metrics_row=g / m, grains_min=min(n_grains), grains_max=max(n_grains))


def launches(L, B):
    """Kernel launches, memsets and copies of one grouped call, counted by torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctxs = lattices(L, B)
    cetkmc.metrics_group(ctxs, metrics_params(ctxs))
    cetkmc.grain_profile_group(ctxs, AXIS, constants.CET_AR_THRESHOLD)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        cetkmc.grain_profile_group(ctxs, AXIS, constants.CET_AR_THRESHOLD)
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


def driver(n_side=4, L=96, n_sweeps=401, order=(None, 2, None, 2), batch=16):
    """run_gr_sweep over scripts/run_gr_sweep.py's 16-case grid on one GPU with batch=16, without and with
    profile_axis (alternated); every file of the run without it must be byte-identical in the run with it."""
    temps, nu_deps = list(TEMPS[:n_side]), list(NU_DEPS[:n_side])
    out = []
    with tempfile.TemporaryDirectory() as d:
        cwd = os.getcwd()
        os.chdir(d)
        try:
            for rep, axis in enumerate(order):
                root = f"run{rep}"
                kw = {} if axis is None else dict(profile_axis=axis)
                t0 = time.perf_counter()
                campaign.run_gr_sweep(temps, nu_deps, L=L, n_sweeps=n_sweeps, n_seeds=20, defect_fraction=3e-3,
                                      impurity_c=0.1, output_root=root, metrics_every=100, batch=batch, **kw)
                campaign.merge_cet_map(root)
                wall = time.perf_counter() - t0
                out.append(dict(profile_axis=axis, wall_s=wall, files=len(_tree_files(f"outputs/{root}"))))
                print(json.dumps(out[-1]), flush=True)
            plain = [i for i, a in enumerate(order) if a is None]
            for i, a in enumerate(order):
                ref = f"outputs/run{plain[0]}"
                files = _tree_files(ref)
                same = all(filecmp.cmp(os.path.join(ref, f), os.path.join(f"outputs/run{i}", f), shallow=False)
                           for f in files)
                out[i]["preexisting_files_identical_to_run0"] = same
                if a is not None:
                    with open(f"outputs/run{i}/cet_map_profile.csv") as fh:
                        out[i]["cet_map_profile"] = fh.read()
        finally:
            os.chdir(cwd)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="grain_profile.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    _lib.require_gpu()
    res = dict(gpu=gpu_info(), settings=dict(advance_sweeps=ADVANCE, reps=REPS, axis=AXIS))
    res["time"] = []
    for L in ((32,) if args.quick else (64, 96, 128)):
        for B in ((1, 2) if args.quick else (1, 4, 16, 64)):
            res["time"].append(time_point(L, B))
            print(json.dumps({k: v for k, v in res["time"][-1].items() if not k.endswith("_reps")}), flush=True)
    res["launches"] = []
    for L, B in (((32, 1), (32, 2)) if args.quick else ((64, 1), (64, 4), (96, 16), (128, 64))):
        res["launches"].append(launches(L, B))
        print(json.dumps(res["launches"][-1]), flush=True)
    res["driver"] = driver(2, 32, 41, (None, 2), 4) if args.quick else driver()
    res["gpu_after"] = gpu_info()
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
