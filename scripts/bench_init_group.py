"""Initial lattices built on the device (cetkmc.init_group) against the per-lattice dense set-up of the map drivers
(campaign._upload_initial: initialize_lattice + introduce_defects on the host, then Context.upload), and the G-R
driver with replicas.  Writes one JSON file.

    python scripts/bench_init_group.py --out profiles/init_group.json [--quick]

1. split: where the per-lattice set-up of the batched driver goes (Context(), set_rate_params, initialize_lattice,
   introduce_defects, Context.upload), summed over B lattices of L^3, host clock (upload ends in a synchronise).
2. init_vs_upload: B lattices set up by _upload_initial one after another, against initial_nuclei for each plus one
   init_group call (and the init_group call alone); median of REPS after one warm-up, host clock, every timed call
   ends in a device synchronise.  Contexts are created once per point and not timed.
3. launches: kernels and copies of one init_group call, counted by torch.profiler in a run of its own.
4. driver: run_gr_sweep over 16 cases x 4 replicas at 96^3, batch=None and batch=64 alternated twice, with the
   wall-time split of scripts/bench_sweep_group.py and whether the ensemble files are identical.
Set-up work of 20 nuclei per lattice, impurity_c = 0.1, as the map scripts use.
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
from cetkmc import _host, _lib, campaign  # noqa: E402
from cetkmc import kmc_simulation as ks  # noqa: E402
from cetkmc._config import rate_params  # noqa: E402

N_SEEDS, IMPURITY_C, REPS = 20, 0.1, 5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _temp(q):
    return 2600.0 + 37.5 * (q % 16)


def split(L, B):
    acc = dict(context=0.0, rate_params=0.0, initialize_lattice=0.0, introduce_defects=0.0, upload=0.0)
    ctxs = []

    def tick(key, fn):
        t0 = time.perf_counter()
        out = fn()
        acc[key] += time.perf_counter() - t0
        return out
    t_all = time.perf_counter()
    for q in range(B):
        ctx = tick("context", lambda: _lib.Context(L=L))
        ctxs.append(ctx)
        tick("rate_params", lambda: ctx.set_rate_params(rate_params(IMPURITY_C, 1, 2, 3, overrides={"NU_DEP": 2e13})))
        st, th, ph, T, at = tick("initialize_lattice", lambda: ks.initialize_lattice(
            lattice_size=L, n_seeds=N_SEEDS, T_sub=_temp(q), impurity_c=IMPURITY_C))
        mask, _ = tick("introduce_defects", lambda: ks.introduce_defects(st, at, T, apply_to_state=False))
        tick("upload", lambda: ctx.upload(state=np.ascontiguousarray(st, dtype=np.int64), theta=th, phi=ph, T=T,
                                          defects=mask))
    total = time.perf_counter() - t_all
    # what the device path replaces of it, on the same contexts
    t0 = time.perf_counter()
    nuc = [_host.initial_nuclei(L, N_SEEDS, _temp(q), 42, IMPURITY_C) for q in range(B)]
    t_nuc = time.perf_counter() - t0
    t0 = time.perf_counter()
    cetkmc.init_group(ctxs, nuc)
    t_ig = time.perf_counter() - t0
    for c in ctxs:
        c.close()
    host_init = acc["initialize_lattice"] + acc["introduce_defects"]
    return dict(L=L, B=B, total_s=total, **{f"{k}_s": v for k, v in acc.items()},
                share=dict(context=acc["context"] / total, host_init=host_init / total, upload=acc["upload"] / total),
                replaced_s=host_init + acc["upload"], initial_nuclei_s=t_nuc, init_group_s=t_ig)


def compare(L, B):
    ctxs = [_lib.Context(L=L) for _ in range(B)]
    for c in ctxs:
        c.set_rate_params(rate_params(IMPURITY_C, 1, 2, 3, overrides={"NU_DEP": 2e13}))

    def dense():
        for q, c in enumerate(ctxs):
            campaign._upload_initial(c, L, N_SEEDS, _temp(q), IMPURITY_C, None, 0, L)

    def sparse():
        cetkmc.init_group(ctxs, [_host.initial_nuclei(L, N_SEEDS, _temp(q), 42, IMPURITY_C) for q in range(B)])
    nuc = [_host.initial_nuclei(L, N_SEEDS, _temp(q), 42, IMPURITY_C) for q in range(B)]

    def call():
        cetkmc.init_group(ctxs, nuc)
    res = dict(L=L, B=B)
    for name, fn in (("upload_initial", dense), ("init_group_with_host", sparse), ("init_group_call", call)):
        fn()
        ts = []
        for _ in range(REPS):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        res[f"{name}_ms"] = 1e3 * float(np.median(ts))
        res[f"{name}_ms_per_lattice"] = res[f"{name}_ms"] / B
    res["speedup_with_host"] = res["upload_initial_ms"] / res["init_group_with_host_ms"]
    # the device part moves 58 B/site (vox, theta, phi, v, T, no snapshot: 57 B) plus the nuclei
    res["init_group_call_GBps"] = B * L ** 3 * 57 / (res["init_group_call_ms"] * 1e-3) / 1e9
    for c in ctxs:
        c.close()
    return res


def launches(L, B):
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctxs = [_lib.Context(L=L) for _ in range(B)]
    nuc = [_host.initial_nuclei(L, N_SEEDS, _temp(q), 42, IMPURITY_C) for q in range(B)]
    cetkmc.init_group(ctxs, nuc)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        cetkmc.init_group(ctxs, nuc, snapshot=True)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    copies = [e.name for e in ev if "memcpy" in e.name.lower()]
    kernels = [e.name.split("(")[0].split("<")[0] for e in ev if "memcpy" not in e.name.lower()
               and "memset" not in e.name.lower()]
    for c in ctxs:
        c.close()
    return dict(L=L, B=B, kernels=len(kernels), kernel_names=sorted(set(kernels)), copies=len(copies))


def driver(temps=(2600.0, 2800.0, 3000.0, 3200.0), nu_deps=(1e12, 5e12, 2e13, 1e14), L=96, n_sweeps=401, replicas=4,
           order=(None, 64, None, 64)):
    acc, depth = {}, [0]

    def timed(key, fn):
        def w(*a, **k):
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
               (_lib.Context, "set_rate_params", "setup"), (_lib, "init_group", "setup"),
               (_lib.Context, "sweep_run", "sweeps"), (_lib, "sweep_run_group", "sweeps"),
               (campaign, "_cadence", "cadence"), (campaign, "_cadence_group", "cadence"),
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
                    rows, ens = campaign.run_gr_sweep(list(temps), list(nu_deps), L=L, n_sweeps=n_sweeps, n_seeds=N_SEEDS,
                                                      defect_fraction=3e-3, impurity_c=IMPURITY_C, output_root=f"r{rep}",
                                                      metrics_every=100, batch=batch, replicas=replicas)
                    wall = time.perf_counter() - t0
                    campaign.merge_cet_map(f"r{rep}")
                    split_s = {f"{k}_s": acc.get(k, 0.0) for k in ("setup", "sweeps", "cadence", "final_download", "close",
                                                                   "csv")}
                    n_lat = len(rows) * replicas
                    out.append(dict(run=rep, batch=batch, cases=len(rows), replicas=replicas, L=L, sweeps=n_sweeps,
                                    wall_s=wall, **split_s, other_s=wall - sum(acc.values()),
                                    site_updates_per_s=n_lat * L ** 3 * n_sweeps / wall,
                                    classes=sorted(set(r["CET_Class"] for r in rows)),
                                    p_equiaxed=[e["p_equiaxed"] for e in ens]))
                    print(json.dumps(out[-1]), flush=True)
                files = ("cet_map.csv", "cet_map_replicas.csv", "cet_map_ensemble.csv")
                same = {f: len({open(f"outputs/r{rep}/{f}", "rb").read() for rep in range(len(order))}) == 1 for f in files}
                out.append(dict(identical_across_runs=same))
            finally:
                os.chdir(cwd)
    finally:
        for obj, name, fn in saved:
            setattr(obj, name, fn)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="init_group.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    _lib.require_gpu()
    _lib.Context(L=8).close()                  # device start-up is not set-up work
    res = dict(gpu=gpu_info(), settings=dict(n_seeds=N_SEEDS, impurity_c=IMPURITY_C, reps=REPS))
    res["split"] = [split(L, B) for L, B in ([(32, 4)] if args.quick else [(96, 16), (64, 64)])]
    print(json.dumps(res["split"]), flush=True)
    res["init_vs_upload"] = []
    for L in ((32,) if args.quick else (64, 96, 128)):
        for B in ((1, 4) if args.quick else (1, 4, 16, 64)):
            r = compare(L, B)
            print(json.dumps(r), flush=True)
            res["init_vs_upload"].append(r)
    res["launches"] = [launches(L, B) for L, B in ([(32, 2)] if args.quick else [(96, 1), (96, 16), (64, 64)])]
    print(json.dumps(res["launches"]), flush=True)
    res["driver"] = (driver((2700.0, 2900.0), (2e13,), 32, 41, 2, (None, 4)) if args.quick else driver())
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
