"""Grouped sweeps (cetkmc.sweep_run_group) against the same lattices run one after another with sweep_run, the
launches per grouped sweep, and the G-R sweep driver with and without batching.  Writes one JSON file.

    python scripts/bench_sweep_group.py --out profiles/sweep_group.json [--quick]

Workload of every point: B half-grown lattices of L^3 sites (bench.py's generator, one seed and NU_DEP per
lattice), events_per_sweep = 0.5 % of the sites, p_max = 0.1, defect_fraction = 3e-3, an update_temperature_cet
step every 20 sweeps (bench.py's settings).  Each point: 20 warm-up sweeps, then REPS repetitions of TIMED sweeps
in one call, timed by the host clock around calls that end in a device synchronise.  At these sizes the
lattices of a point (<= 32 x 128^3 x ~100 B) partly fit in the 126 MB L2 for the small L; that is the regime a G-R
study runs in, so no cache flush is done between repetitions.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cetkmc  # noqa: E402
from cetkmc import _synth  # noqa: E402
from cetkmc._config import rate_params, thermal_params  # noqa: E402

THERMAL_EVERY, EVENTS_FRACTION, P_MAX = 20, 0.005, 0.1
WARMUP, TIMED, REPS = 20, 200, 3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


_lattices = {}


def lattice(L, q):
    if (L, q) not in _lattices:
        _lattices[(L, q)] = _synth.half_grown(L, seed=1234 + q)
    return _lattices[(L, q)]


def make(L, B):
    out = []
    for q in range(B):
        packed, th, ph, T = lattice(L, q)
        ctx = cetkmc.Context(L=L)
        ctx.set_rate_params(rate_params(0.1, overrides={"NU_DEP": 2e13 * (1 + q % 8)}))
        ctx.upload_packed(packed)
        ctx.upload(theta=th, phi=ph, T=T)
        sp = cetkmc._lib.SweepParams()
        sp.seed, sp.events_per_sweep, sp.p_max = 42 + q, EVENTS_FRACTION * L ** 3, P_MAX
        sp.defect_fraction, sp.thermal_every = 3e-3, THERMAL_EVERY
        out.append((ctx, sp, thermal_params(1e-6, nan_to_num=True, t_floor=2600.0 + 25.0 * (q % 8))))
    return out


def close(cs):
    for c, _, _ in cs:
        c.close()


def time_point(L, B):
    grp = make(L, B)
    ctxs, sps, tps = [c for c, _, _ in grp], [s for _, s, _ in grp], [t for _, _, t in grp]
    cetkmc.sweep_run_group(ctxs, WARMUP, sps, tps)
    t_grp = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        res = cetkmc.sweep_run_group(ctxs, TIMED, sps, tps)
        t_grp.append((time.perf_counter() - t0) * 1e3 / TIMED)
    assert not any(r["overflow"] or r["terminated"] for r in res)
    close(grp)
    solo = make(L, B)
    for c, s, t in solo:
        c.sweep_run(WARMUP, s, t)
    t_solo = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        for c, s, t in solo:
            c.sweep_run(TIMED, s, t)
        t_solo.append((time.perf_counter() - t0) * 1e3 / TIMED)
    close(solo)
    g, s = float(np.median(t_grp)), float(np.median(t_solo))
    return dict(L=L, B=B, ms_per_grouped_sweep=g, ms_grouped_reps=t_grp, ms_per_b2b_sweeps=s, ms_b2b_reps=t_solo,
                spread_grouped=(max(t_grp) - min(t_grp)) / g, spread_b2b=(max(t_solo) - min(t_solo)) / s,
                b2b_over_grouped=s / g, site_updates_per_s_grouped=B * L ** 3 / (g * 1e-3),
                site_updates_per_s_b2b=B * L ** 3 / (s * 1e-3))


def launches(L, B, n=THERMAL_EVERY):
    """Kernel launches per sweep over `n` sweeps (one thermal step among them), grouped and back to back, counted
    by torch.profiler (CUDA activities) in a run of its own."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    def count(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        k = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
             and "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]
        names = {}
        for e in k:
            names[e.name.split("(")[0].split("<")[0]] = names.get(e.name.split("(")[0].split("<")[0], 0) + 1
        return len(k), names

    grp = make(L, B)
    ctxs, sps, tps = [c for c, _, _ in grp], [s for _, s, _ in grp], [t for _, _, t in grp]
    cetkmc.sweep_run_group(ctxs, WARMUP, sps, tps)        # sweep index 20: the next window starts with a thermal step
    ng, names_g = count(lambda: cetkmc.sweep_run_group(ctxs, n, sps, tps))
    close(grp)
    solo = make(L, B)
    for c, s, t in solo:
        c.sweep_run(WARMUP, s, t)
    ns, _ = count(lambda: [c.sweep_run(n, s, t) for c, s, t in solo])
    close(solo)
    return dict(L=L, B=B, sweeps=n, launches_per_grouped_sweep=ng / n, launches_per_b2b_sweeps=ns / n,
                grouped_kernels=names_g)


def driver(n_cases_side=4, L=96, n_sweeps=401, order=(None, 16, None, 16)):
    """run_gr_sweep over 16 cases (scripts/run_gr_sweep.py's grid and settings) on one GPU, batch=None and
    batch=16 alternated (the first run of the process pays one-time costs), with the wall time split into set-up
    (context, rate params, initial lattice and upload), sweeps, the metrics cadence (defect-mask refresh and metrics
    row), the final download of run_cet_sublattice, closing the contexts, the CSV writes, and the rest."""
    from cetkmc import _lib, campaign
    from cetkmc import kmc_simulation as ks
    temps = [2600.0, 2800.0, 3000.0, 3200.0][:n_cases_side]
    nu_deps = [1e12, 5e12, 2e13, 1e14][:n_cases_side]
    acc, depth = {}, [0]

    def timed(key, fn):
        def w(*a, **k):                      # only the outermost timed call counts (the cadence downloads too)
            depth[0] += 1
            t0 = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                depth[0] -= 1
                if depth[0] == 0:
                    acc[key] = acc.get(key, 0.0) + time.perf_counter() - t0
        return w

    targets = [(campaign, "_upload_initial", "setup"), (_lib.Context, "__init__", "setup"),
               (_lib.Context, "set_rate_params", "setup"), (_lib.Context, "sweep_run", "sweeps"),
               (_lib, "sweep_run_group", "sweeps"), (campaign, "_cadence", "cadence"), (campaign, "_cadence_group", "cadence"),
               (_lib.Context, "download", "final_download"), (_lib.Context, "close", "close"),
               (ks, "_write_csv", "csv")]
    saved = [(obj, name, getattr(obj, name)) for obj, name, _k in targets]
    for (obj, name, key), (_o, _n, fn) in zip(targets, saved):
        setattr(obj, name, timed(key, fn))
    out = []
    try:
        with tempfile.TemporaryDirectory() as d:
            cwd = os.getcwd()
            os.chdir(d)
            try:
                for rep, batch in enumerate(order):
                    acc.clear()
                    t0 = time.perf_counter()
                    rows = campaign.run_gr_sweep(temps, nu_deps, L=L, n_sweeps=n_sweeps, n_seeds=20, defect_fraction=3e-3,
                                                 impurity_c=0.1, output_root=f"r{rep}", metrics_every=100, batch=batch)
                    wall = time.perf_counter() - t0
                    split = {f"{k}_s": acc.get(k, 0.0) for k in ("setup", "sweeps", "cadence", "final_download", "close", "csv")}
                    out.append(dict(run=rep, batch=batch, cases=len(rows), L=L, sweeps=n_sweeps, wall_s=wall, **split,
                                    other_s=wall - sum(acc.values()),
                                    site_updates_per_s=len(rows) * L ** 3 * n_sweeps / wall,
                                    sweep_site_updates_per_s=len(rows) * L ** 3 * n_sweeps / acc["sweeps"]))
                    print(json.dumps(out[-1]), flush=True)
                maps = [open(f"outputs/r{rep}/cet_map_rank0.csv", "rb").read() for rep in range(len(order))]
                out.append(dict(cet_map_identical=all(m == maps[0] for m in maps)))
            finally:
                os.chdir(cwd)
    finally:
        for obj, name, fn in saved:
            setattr(obj, name, fn)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="sweep_group.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    cetkmc._lib.require_gpu()
    points = [(64, 2), (32, 2)] if args.quick else [(L, B) for L in (64, 96, 128) for B in (1, 4, 16, 32)] + [(64, 64)]
    res = dict(gpu=gpu_info(), settings=dict(warmup=WARMUP, timed_sweeps=TIMED, reps=REPS, thermal_every=THERMAL_EVERY,
                                             events_fraction=EVENTS_FRACTION, p_max=P_MAX, defect_fraction=3e-3))
    res["grouped_vs_b2b"] = []
    for L, B in points:
        r = time_point(L, B)
        print(json.dumps(r), flush=True)
        res["grouped_vs_b2b"].append(r)
    res["launches"] = []
    for L, B in ([(64, 1), (64, 4)] if args.quick else [(64, 1), (64, 4), (64, 16), (96, 16), (24, 1), (24, 16)]):
        r = launches(L, B)
        print(json.dumps(r), flush=True)
        res["launches"].append(r)
    res["driver"] = driver(2, 32, 41, (None, 2)) if args.quick else driver()
    print(json.dumps(res["driver"]), flush=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
