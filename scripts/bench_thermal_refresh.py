#!/usr/bin/env python
"""The two sides of the rates after a thermal step of cet_sweep_run, timed at 512^3: the refresh of the sites whose
rates read a changed temperature (dilation of the changed bitmap, one host read of the counts, stamp scan, refresh)
against the dense rebuild (debug flag 524288).  The threshold in csrc/sweep.cu (thermal_refresh_max) is the
crossover this measures.

A case is the half-grown lattice with T depending on i only: the linear gradient 2800 + 2 i plus a parabola on the
planes i < m.  The first thermal step follows the upload (dense on both sides); the second one changes the planes
[0, m + 2) and two at the top, whole planes, so m sets the stale fraction.  Per case and side: one sweep with that
second step, as the PROF_STEP span (the sweep's own kernels are the same bits on both sides) and the refresh / rates
spans.  The benchmark's own profile (the k gradient of bench.py, its second thermal step) is timed the same way,
and a torch.profiler trace of its refresh side gives the gap the host read leaves between the dilation kernel and
the next launch (the GPU waits that long per thermal step).

    python scripts/bench_thermal_refresh.py [--L 512] [--reps 3] [--out profiles/thermal_refresh.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FORCE_DENSE = 524288
FRACTIONS = (0.01, 0.02, 0.05, 0.10, 0.20, 0.30, 0.40, 0.60, 0.80)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def make_T(L, kind, m=0):
    i = np.arange(L, dtype=np.float64)[:, None, None]
    k = np.arange(L, dtype=np.float64)[None, None, :]
    if kind == "bench":
        T = 2800.0 + 895.0 * k / L + 0.0 * i
    else:
        T = 2800.0 + 2.0 * i + np.where(i < m, 200.0 * ((m - i) / max(m, 1)) ** 2, 0.0) + 0.0 * k   # below the clip
    return np.ascontiguousarray(np.broadcast_to(T, (L, L, L)))


def one(cet, L, T, flags, lattice, thermal_every, trace=None):
    """Time the sweep that holds the second thermal step; returns spans (ms) and the stale fraction."""
    from cetkmc._config import rate_params, thermal_params
    st, th, ph, df = lattice
    ctx = cet.Context(L=L)
    ctx.debug_flags(flags)
    ctx.set_rate_params(rate_params(0.1))
    ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
    sp = cet._lib.SweepParams()
    sp.seed, sp.events_per_sweep, sp.p_max, sp.defect_fraction, sp.thermal_every = 42, 0.005 * L ** 3, 0.1, 3e-3, thermal_every
    tp = thermal_params(1e-6, nan_to_num=True)
    ctx.sweep_run(thermal_every, sp, tp)            # priming + the first step (dense after the upload), then sweeps
    ctx.sync()
    T1 = ctx.download(T=True)["T"]
    ctx.profile_enable(True)
    if trace is not None:
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.sweep_run(1, sp, tp)
            ctx.sync()
        torch.cuda.synchronize()
        trace.extend((e.name, e.time_range.start, e.time_range.end) for e in prof.events() if e.device_type.name == "CUDA")
    else:
        ctx.sweep_run(1, sp, tp)                    # the second step + one sweep
    ctx.sync()
    spans = {k: ctx.profile_read(k) for k in ("step", "refresh", "rates", "thermal")}
    ctx.profile_enable(False)
    T2 = ctx.download(T=True)["T"]
    ctx.close()
    chg = (T1.view(np.int64) != T2.view(np.int64))
    del T1, T2
    out = {k: v[0] for k, v in spans.items()}
    out["launches"] = {k: int(v[1]) for k, v in spans.items()}
    out["changed_fraction"] = float(chg.mean())
    if thermal_every == 1:                          # whole planes change: the stale planes are those within two
        pl = np.flatnonzero(chg.any(axis=(1, 2)))
        out["stale_fraction"] = len({q for p in pl for q in range(p - 2, p + 3) if 0 <= q < L}) / L
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, default=512)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "thermal_refresh.json"))
    args = ap.parse_args()
    import cetkmc as cet
    from cetkmc import _synth
    cet._lib.require_gpu()
    L = args.L
    packed, th, ph, _ = _synth.half_grown(L, seed=1234)
    st, df = _synth.unpack(packed)
    lattice = (st, th, ph, df)
    rows = []
    for f in FRACTIONS:
        m = max(int(round(f * L)) - 8, 0)           # stale planes: m + 8 (faces included)
        res = {"refresh": [], "dense": []}
        for _ in range(args.reps):                  # the two sides alternate
            for side, flags in (("refresh", 0), ("dense", FORCE_DENSE)):
                res[side].append(one(cet, L, make_T(L, "bump", m), flags, lattice, 1))
        row = {"m": m, "stale_fraction": res["refresh"][0]["stale_fraction"],
               "changed_fraction": res["refresh"][0]["changed_fraction"]}
        for side in res:
            row[side] = {k: float(np.median([r[k] for r in res[side]])) for k in ("step", "refresh", "rates", "thermal")}
            row[side]["step_all"] = [r["step"] for r in res[side]]
            row[side]["launches"] = res[side][0]["launches"]
        rows.append(row)
        print(json.dumps(row), flush=True)
    # the benchmark's profile: its second thermal step (thermal_every 20 as bench.py)
    bench = {"refresh": [], "dense": []}
    for _ in range(args.reps):
        for side, flags in (("refresh", 0), ("dense", FORCE_DENSE)):
            bench[side].append(one(cet, L, make_T(L, "bench"), flags, lattice, 20))
    bench_row = {"changed_fraction": bench["refresh"][0]["changed_fraction"]}
    for side in bench:
        bench_row[side] = {k: float(np.median([r[k] for r in bench[side]])) for k in ("step", "refresh", "rates", "thermal")}
        bench_row[side]["step_all"] = [r["step"] for r in bench[side]]
        bench_row[side]["launches"] = bench[side][0]["launches"]
    print(json.dumps(bench_row), flush=True)
    gap = None
    try:
        trace = []
        one(cet, L, make_T(L, "bench"), 0, lattice, 20, trace=trace)
        trace.sort(key=lambda e: e[1])
        ks = [q for q, e in enumerate(trace) if "thermal_stale_kernel" in e[0]]
        # the host read: the counts' copy after the dilation kernel, then the first launch issued after the host saw them
        if ks and ks[0] + 2 < len(trace):
            a, cp, b = trace[ks[0]], trace[ks[0] + 1], trace[ks[0] + 2]
            gap = {"after": cp[0], "next": b[0], "gap_us": b[1] - cp[2], "copy_us": cp[2] - cp[1], "kernel_to_copy_us": cp[1] - a[2]}
    except Exception as e:                           # the trace is a side measurement
        gap = {"error": repr(e)}
    print(json.dumps({"host_read_gap": gap}), flush=True)
    # crossover: the smallest measured stale fraction at which the dense side is the faster
    cross = next((r["stale_fraction"] for r in rows if r["dense"]["step"] < r["refresh"]["step"]), None)
    out = {"what": "ms of the sweep holding the second thermal step (PROF_STEP span, median of the reps), refresh side "
                   "vs dense side (debug flag 524288), 512^3 half-grown lattice, T = 2800 + 2 i + parabola on i < m",
           "gpu": gpu_info(), "L": L, "reps": args.reps, "rows": rows, "bench_profile": bench_row,
           "host_read_gap": gap, "first_fraction_where_dense_wins": cross}
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"crossover": cross, "gpu": out["gpu"]}), flush=True)


if __name__ == "__main__":
    main()
