"""The metrics cadence of the G-R sweep driver: where the per-context cadence (campaign._cadence) spends its time,
the grouped cadence (campaign._cadence_group, one cetkmc.metrics_group call) against back-to-back per-context
cadences, the kernel launches of one grouped call, and the 16-case 96^3 driver with batch=None and batch=16.
Writes one JSON file.

    python scripts/bench_cadence_group.py --out profiles/cadence_group.json [--quick]

Lattices are the driver's own (run_gr_sweep's set-up: initialize_lattice with 20 seeds, impurity_c = 0.1, its
sweep parameters) advanced by ADVANCE sweeps, i.e. to the driver's later rows.  Each timing point: one warm-up
call, then REPS calls per path, the two paths alternated, host clock around calls that end in a device
synchronise; the median is reported.  The lattices (<= 32 x 128^3 x ~100 B) partly fit in the 126 MB L2; that is
the regime the driver runs in, so no cache flush is done between repetitions.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import cetkmc  # noqa: E402
from cetkmc import _lib, campaign  # noqa: E402
from cetkmc import defects as _defects  # noqa: E402
from cetkmc import metrics as _metrics  # noqa: E402
from cetkmc._config import constants, rate_params  # noqa: E402
from bench_sweep_group import driver, gpu_info  # noqa: E402

EVERY, ADVANCE, REPS = 100, 300, 5
TEMPS, NU_DEPS = (2600.0, 2800.0, 3000.0, 3200.0), (1e12, 5e12, 2e13, 1e14)


def cases(L, B, seed=42):
    """B of the driver's cases (its T_sub x NU_DEP grid, repeated) advanced by ADVANCE sweeps together."""
    runs = []
    for q in range(B):
        temp, nu_dep = TEMPS[(q // 4) % 4], NU_DEPS[q % 4]
        np.random.seed(seed)
        ctx = cetkmc.Context(L=L)
        ctx.set_rate_params(rate_params(0.1, 1, 2, 3, overrides={"NU_DEP": nu_dep}))
        campaign._upload_initial(ctx, L, 20, temp, 0.1, None, 0, L)
        sp, tp = campaign._sweep_setup(L, seed, temp, None, 0.1, 3e-3, 20)
        runs.append(dict(ctx=ctx, sp=sp, tp=tp, rng=np.random.get_state(), consts=campaign._gr(L, temp, nu_dep), rows=[],
                         total_time=0.0, nucleation_count=0, cet_detected=False))
    cetkmc.sweep_run_group([r["ctx"] for r in runs], ADVANCE, [r["sp"] for r in runs], [r["tp"] for r in runs])
    return runs


def close(runs):
    for r in runs:
        r["ctx"].close()


def clock(fn):
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def split(L):
    """One per-context cadence with a refresh (NumPy stream), part by part."""
    r, = cases(L, 1)
    ctx = r["ctx"]
    h = ctx._h
    parts = {k: [] for k in ("counts", "numpy_draws", "defects_refresh", "labelling", "grains_stats", "host_metrics",
                             "cadence_total")}
    n_grains = 0
    n_sites = L ** 3
    for rep in range(REPS + 1):
        t = {}
        t["counts"] = clock(lambda: ctx.counts())
        n_c = int(ctx.counts()[_defects.CARBON_ID])
        box = {}
        t["numpy_draws"] = clock(lambda: box.setdefault("d", np.random.random(n_c)))
        t["defects_refresh"] = clock(lambda: ctx.defects_refresh(draws=box["d"], prob_base=constants.DEFECT_PROB_BASE,
                                                                 e_mig=_defects.E_MIGRATION, kT=constants.K_T,
                                                                 T_default=constants.T_SUB, carbon_id=3, defect_id=4))
        n = _lib.C.c_int64(0)
        t["labelling"] = clock(lambda: _lib.check(_lib.lib().cet_grains_label_ex(h, 0.5, 0, _lib.C.byref(n)), "label"))
        n_grains = n.value
        g = dict(n=n_grains, root=np.empty(n_grains, np.int32), size=np.empty(n_grains, np.int32),
                 box_lo=np.empty((n_grains, 3), np.int32), box_hi=np.empty((n_grains, 3), np.int32))
        P = _lib._ptr
        t["grains_stats"] = clock(lambda: _lib.check(_lib.lib().cet_grains_stats(h, n_grains, P(g["root"]), P(g["size"]),
                                                                                  P(g["box_lo"]), P(g["box_hi"])), "stats"))

        def host():
            o = np.argsort(g["root"], kind="stable")
            _metrics.metrics_from_grains(dict(n=n_grains, root=g["root"][o], size=g["size"][o], box_lo=g["box_lo"][o],
                                              box_hi=g["box_hi"][o]), n_sites)
        t["host_metrics"] = clock(host)
        t["cadence_total"] = clock(lambda: campaign._cadence(ctx, EVERY * (rep + 4), EVERY, False, 42, 1, 0.0, 0, False,
                                                             r["consts"], verbose=False))
        if rep:
            for k in parts:
                parts[k].append(t[k] * 1e3)
    close([r])
    med = {k + "_ms": float(np.median(v)) for k, v in parts.items()}
    return dict(L=L, n_grains=n_grains, carbon_sites=n_c, **med, reps_ms=parts)


def grouped_vs_b2b(L, B, philox):
    runs = cases(L, B)
    rep_state = {"last": EVERY * 4}

    def solo():
        last = rep_state["last"]
        for r in runs:
            np.random.set_state(r["rng"])
            row, r["cet_detected"] = campaign._cadence(r["ctx"], last, EVERY, philox, 42, 1, r["total_time"],
                                                       r["nucleation_count"], r["cet_detected"], r["consts"], verbose=False)
            r["rng"] = np.random.get_state()
        rep_state["last"] += EVERY

    def grouped():
        campaign._cadence_group(runs, rep_state["last"], EVERY, philox, 42)
        rep_state["last"] += EVERY
    grouped(); solo()
    tg, ts = [], []
    for _ in range(REPS):
        tg.append(clock(grouped) * 1e3)
        ts.append(clock(solo) * 1e3)
    n_grains = [int(r["rows"][-1]["GrainCount"]) for r in runs]
    close(runs)
    g, s = float(np.median(tg)), float(np.median(ts))
    return dict(L=L, B=B, mask_stream="philox" if philox else "numpy", ms_grouped=g, ms_grouped_reps=tg, ms_b2b=s,
                ms_b2b_reps=ts, b2b_over_grouped=s / g, grains_min=min(n_grains), grains_max=max(n_grains))


def launches(L, B):
    """Kernel launches of one grouped cadence call with a refresh (NumPy stream), counted by torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    runs = cases(L, B)
    campaign._cadence_group(runs, EVERY, EVERY, False, 42)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        campaign._cadence_group(runs, 2 * EVERY, EVERY, False, 42)
        torch.cuda.synchronize()
    k = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels = [e for e in k if "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]
    names = {}
    for e in kernels:
        nm = e.name.split("(")[0].split("<")[0]
        names[nm] = names.get(nm, 0) + 1
    close(runs)
    return dict(L=L, B=B, kernel_launches=len(kernels), copies_and_memsets=len(k) - len(kernels), kernels=names)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="cadence_group.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    _lib.require_gpu()
    res = dict(gpu=gpu_info(), settings=dict(metrics_every=EVERY, advance_sweeps=ADVANCE, reps=REPS))
    res["split"] = []
    for L in ((32,) if args.quick else (64, 96, 128)):
        res["split"].append(split(L))
        print(json.dumps(res["split"][-1]), flush=True)
    res["grouped_vs_b2b"] = []
    for L, B in (((32, 2),) if args.quick else ((96, 1), (96, 4), (96, 16), (96, 32), (64, 16), (128, 16))):
        for philox in (False, True):
            res["grouped_vs_b2b"].append(grouped_vs_b2b(L, B, philox))
            print(json.dumps(res["grouped_vs_b2b"][-1]), flush=True)
    res["launches"] = []
    for L, B in (((32, 1), (32, 2)) if args.quick else ((64, 1), (64, 4), (64, 16), (96, 32))):
        res["launches"].append(launches(L, B))
        print(json.dumps(res["launches"][-1]), flush=True)
    res["driver"] = driver(2, 32, 41, (None, 2)) if args.quick else driver()
    print(json.dumps(res["driver"]), flush=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
