"""The laser step of the melt-pool driver: the grouped step (cetkmc.thermal_full_group, snapshot fused) against the
same lattices stepped back to back (Context.thermal_full + snapshot_state), with and without what the next sweep call
then does first (sweep_run(0) / sweep_run_group(0): the solo path rebuilds its tile state there); the kernel launches
and copies of one step; and the 16-case 96^3 melt-pool map with batch=None and batch=16.  Writes one JSON file.

    python scripts/bench_melt_pool_group.py --out profiles/melt_pool_group.json [--quick]

Lattices: bench_sweep_group's half-grown lattices, advanced by one laser block (step + ADVANCE sweeps) so that their
tile state is current, as in the driver.  Each timing point: one warm-up step, then REPS repetitions of STEPS steps
per path, the two paths alternated, host clock around steps that end in a device synchronise (every laser step
synchronises); the median per step is reported.  The lattices (<= 32 x 128^3 x ~50 B touched per step) partly fit
in the 126 MB L2; that is the regime the driver runs in, so no cache flush is done between repetitions.
"""
import argparse
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
from cetkmc._config import thermal_full_params  # noqa: E402
from cetkmc.thermal_solver import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS, laser_source_top  # noqa: E402
from bench_sweep_group import gpu_info, make  # noqa: E402

ADVANCE, STEPS, REPS = 19, 10, 5


def cases(L, B):
    runs = []
    for q, (ctx, sp, _tp) in enumerate(make(L, B)):
        sp.thermal_every = 0
        ctx.snapshot_state()
        runs.append(dict(ctx=ctx, sp=sp, tfp=thermal_full_params(1e-7),
                         q_top=laser_source_top(L, (L / 2, 2.0 + q), 200.0 + 10.0 * q, DEFAULT_BEAM_RADIUS,
                                                DEFAULT_ABSORPTIVITY)))
    step_grouped(runs)
    cetkmc.sweep_run_group([r["ctx"] for r in runs], ADVANCE, [r["sp"] for r in runs])
    return runs


def step_grouped(runs):
    cetkmc.thermal_full_group([r["ctx"] for r in runs], [r["tfp"] for r in runs], [r["q_top"] for r in runs])


def step_b2b(runs):
    for r in runs:
        r["ctx"].thermal_full(r["tfp"], r["q_top"])
        r["ctx"].snapshot_state()


def prime_grouped(runs):
    cetkmc.sweep_run_group([r["ctx"] for r in runs], 0, [r["sp"] for r in runs])


def prime_b2b(runs):
    for r in runs:
        r["ctx"].sweep_run(0, r["sp"], None)


def close(runs):
    for r in runs:
        r["ctx"].close()


def timed(fn):
    t0 = time.perf_counter()
    for _ in range(STEPS):
        fn()
    return (time.perf_counter() - t0) * 1e3 / STEPS


def grouped_vs_b2b(L, B):
    runs = cases(L, B)
    paths = dict(grouped=lambda: step_grouped(runs), b2b=lambda: step_b2b(runs),
                 grouped_then_sweep0=lambda: (step_grouped(runs), prime_grouped(runs)),
                 b2b_then_sweep0=lambda: (step_b2b(runs), prime_b2b(runs)))
    for fn in paths.values():
        fn()
    reps = {k: [] for k in paths}
    for _ in range(REPS):
        for k, fn in paths.items():
            reps[k].append(timed(fn))
    close(runs)
    med = {k: float(np.median(v)) for k, v in reps.items()}
    return dict(L=L, B=B, ms_per_step_grouped=med["grouped"], ms_per_step_b2b=med["b2b"],
                b2b_over_grouped=med["b2b"] / med["grouped"],
                ms_per_step_grouped_then_sweep0=med["grouped_then_sweep0"],
                ms_per_step_b2b_then_sweep0=med["b2b_then_sweep0"],
                b2b_over_grouped_then_sweep0=med["b2b_then_sweep0"] / med["grouped_then_sweep0"], reps_ms=reps)


def launches(L, B):
    """Kernel launches and copies of one laser step (+ the next sweep call's preparation), counted by torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    runs = cases(L, B)
    out = dict(L=L, B=B)
    for name, fn in (("grouped", lambda: step_grouped(runs)), ("b2b", lambda: step_b2b(runs)),
                     ("grouped_then_sweep0", lambda: (step_grouped(runs), prime_grouped(runs))),
                     ("b2b_then_sweep0", lambda: (step_b2b(runs), prime_b2b(runs)))):
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        k = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        kernels = [e for e in k if "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]
        names = {}
        for e in kernels:
            nm = e.name.split("(")[0].split("<")[0]
            names[nm] = names.get(nm, 0) + 1
        out[name] = dict(kernel_launches=len(kernels), copies_and_memsets=len(k) - len(kernels), kernels=names)
    close(runs)
    return out


def driver(n_side=4, L=96, n_sweeps=401, order=(None, 16, None, 16)):
    """run_melt_pool_map over 16 cases (scripts/run_melt_pool_map.py's grid and settings) on one GPU, batch=None and
    batch=16 alternated; the map files of every run are compared with the first one's."""
    powers = [100.0, 200.0, 300.0, 400.0][:n_side]
    speeds = [0.25, 0.5, 1.0, 2.0][:n_side]
    out, ref = [], None
    with tempfile.TemporaryDirectory() as d:
        cwd = os.getcwd()
        os.chdir(d)
        try:
            for rep, batch in enumerate(order):
                t0 = time.perf_counter()
                rows = campaign.run_melt_pool_map(powers, speeds, L=L, n_sweeps=n_sweeps, start=(L / 2, 0.0), n_seeds=20,
                                                  defect_fraction=3e-3, impurity_c=0.1, output_root=f"run{rep}",
                                                  metrics_every=100, batch=batch)
                wall = time.perf_counter() - t0
                key = [{k: v for k, v in r.items()} for r in rows]
                ref = key if ref is None else ref
                out.append(dict(batch=batch, wall_s=wall, same_map_as_first=key == ref,
                                classes=sorted(set(r["CET_Class"] for r in rows)), steps=[int(r["Step"]) for r in rows]))
                print(json.dumps(out[-1]), flush=True)
        finally:
            os.chdir(cwd)
    return dict(cases=len(powers) * len(speeds), L=L, n_sweeps=n_sweeps, runs=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="melt_pool_group.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    _lib.require_gpu()
    res = dict(gpu=gpu_info(), settings=dict(advance_sweeps=ADVANCE, steps_per_rep=STEPS, reps=REPS))
    res["grouped_vs_b2b"] = []
    for L in ((64,) if args.quick else (64, 96, 128)):
        for B in ((1, 4) if args.quick else (1, 4, 16, 32)):
            res["grouped_vs_b2b"].append(grouped_vs_b2b(L, B))
            print(json.dumps({k: v for k, v in res["grouped_vs_b2b"][-1].items() if k != "reps_ms"}), flush=True)
    res["launches"] = []
    for L, B in (((64, 1), (64, 4)) if args.quick else ((96, 1), (96, 4), (96, 16), (96, 32))):
        res["launches"].append(launches(L, B))
        print(json.dumps(res["launches"][-1]), flush=True)
    res["driver"] = driver(2, 32, 41, (None, 2)) if args.quick else driver()
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
