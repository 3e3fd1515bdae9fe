"""Grain boundaries along the growth axis (cetkmc.boundary_group): one grouped call over B lattices against B
back-to-back groups of one, the same lattices' grouped metrics row (cetkmc.metrics_group) for scale, the launches,
memsets and copies of one call with its kernel time and achieved bytes/s on every axis, and the maps: the 16-case 96^3
G-R map and a small melt-pool map, each without and with boundary_axis=2, with the boundary network of every case
(linear intercepts along and across the axis, boundary fraction, misorientation against the truncated nucleation
null).  Writes one JSON file.

    python scripts/bench_boundary_group.py --out profiles/boundary_group.json [--quick]

Lattices are half-grown: _synth.half_grown with fill = 1, a dense solid below the wavy front k < L/2 + 8 sin(2 pi i / L)
with orientations constant over 4^3 blocks, one seed per lattice, labelled once by a grouped metrics row.  Each timing
point: one warm-up call per path, then REPS calls per path, the paths alternated, host clock around calls that end in
a device synchronise; the median and the extremes are reported.  The labels of 64 x 128^3 lattices (537 MB) exceed the
126 MB L2; no cache flush is done between repetitions, as in the driver's cadence, which labels the same lattices just
before.  Bytes: algorithmic = 4 n L^3 (the labels, once) + 2 x 24 B per boundary bond (x, y, z of both ends); the
neighbour labels are counted once, as they come from L1 / L2.
"""
import argparse
import csv
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
# metrics.boundary_summary's truncated nucleation null (misorientation > 0.5 rad), ascending 10-degree bins
NULL = dict(MeanMisorientationCos=-0.0847, shares=[0, 0, 0.0072, 0.0593, 0.0679, 0.0746, 0.0794, 0.0825, 0.0841, 0.0841,
                                                    0.0825, 0.0794, 0.0746, 0.0679, 0.0593, 0.0483, 0.0342, 0.0145])


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


def stats(v):
    return dict(median=float(np.median(v)), min=float(np.min(v)), max=float(np.max(v)))


def time_point(ctxs, L, B):
    group = ctxs[:B]
    mp = metrics_params(group)
    cetkmc.metrics_group(group, mp)                                 # the labelling the calls read
    paths = dict(grouped=lambda: cetkmc.boundary_group(group, AXIS),
                 b2b=lambda: [cetkmc.boundary_group([c], AXIS) for c in group])
    got = cetkmc.boundary_group(group, AXIS)
    solo = [cetkmc.boundary_group([c], AXIS) for c in group]
    assert all(np.array_equal(got[i][q], solo[q][i][0]) for q in range(B) for i in range(3))
    t = {k: [] for k in paths}
    for _ in range(REPS):
        for k, fn in paths.items():
            t[k].append(clock(fn))
    tm = [clock(lambda: cetkmc.metrics_group(group, mp)) for _ in range(REPS)]
    g, s, m = (stats(v) for v in (t["grouped"], t["b2b"], tm))
    return dict(L=L, B=B, axis=AXIS, ms_grouped=g, ms_grouped_reps=t["grouped"], ms_b2b=s, ms_b2b_reps=t["b2b"],
                b2b_over_grouped=s["median"] / g["median"], ms_metrics_group_row=m, ms_metrics_group_row_reps=tm,
                boundary_over_metrics_row=g["median"] / m["median"], solid_bonds=int(got[0][..., 0].sum()),
                boundary_bonds=int(got[0][..., 1].sum()))


def launches(ctxs, L, B):
    """Kernel launches, memsets and copies of one grouped call on every axis, counted by torch.profiler, with the
    kernel's device time and the achieved bytes/s over the algorithmic and the sector bytes."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    group = ctxs[:B]
    cetkmc.metrics_group(group, metrics_params(group))
    bnd = int(cetkmc.boundary_group(group, AXIS)[0][..., 1].sum())
    out = []
    for axis in range(3):
        cetkmc.boundary_group(group, axis)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(REPS):
                cetkmc.boundary_group(group, axis)
            torch.cuda.synchronize()
        k = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        copies = [e for e in k if "memcpy" in e.name.lower()]
        memsets = [e for e in k if "memset" in e.name.lower()]
        kernels = [e for e in k if e not in copies and e not in memsets]
        us = float(np.median([e.device_time for e in kernels])) if kernels else None
        alg = 4 * B * L ** 3 + 48 * bnd
        out.append(dict(L=L, B=B, axis=axis, kernel_launches_per_call=len(kernels) / REPS,
                        copies_per_call=len(copies) / REPS, memsets_per_call=len(memsets) / REPS,
                        copy_kinds=sorted({e.name for e in copies}),
                        kernels=sorted({e.name.split("(")[0] for e in kernels}), kernel_us_median=us,
                        boundary_bonds=bnd, algorithmic_bytes=alg,
                        achieved_algorithmic_GB_s=(alg / (us * 1e-6) / 1e9) if us else None))
        print(json.dumps(out[-1]), flush=True)
    return out


def _tree_files(root):
    out = []
    for d, _, fs in os.walk(root):
        out += [os.path.relpath(os.path.join(d, f), root) for f in fs]
    return sorted(out)


def case_network(path):
    """The boundary network of a case's final row: the misorientation shares per bin (ascending angle) over all
    planes, and per plane the solid, boundary and interface bonds (the last the solid-liquid surface)."""
    _edges, recs = campaign.read_boundary_csv(path)
    _step, bonds, hist, _f = recs[-1]
    tot = hist.sum(0)
    return dict(shares=[float(x) for x in tot / max(int(tot.sum()), 1)],
                planes=dict(solid=bonds[:, :, 0].sum(1).tolist(), boundary=bonds[:, :, 1].sum(1).tolist(),
                            interface=bonds[:, :, 2].sum(1).tolist()))


def maps(quick=False):
    """scripts/run_gr_sweep.py's 16-case 96^3 grid (batch=16) and a small melt-pool map (2 powers x 2 speeds, 64^3,
    batch=4; the melt-pool script's settings otherwise), each without and with boundary_axis=2.  Every file of the run
    without boundary_axis must be byte-identical in the run with it; every case's row of the map boundary file is kept
    with its misorientation shares and per-plane bonds."""
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
            for name, fn, merge, L in (("gr", lambda root, kw: campaign.run_gr_sweep(
                                           gr["temps"], gr["nu_deps"], L=gr["L"], n_sweeps=gr["n_sweeps"], n_seeds=20,
                                           defect_fraction=3e-3, impurity_c=0.1, output_root=root, metrics_every=100,
                                           batch=gr["batch"], **kw), campaign.merge_cet_map, gr["L"]),
                                       ("melt_pool", lambda root, kw: campaign.run_melt_pool_map(
                                           mp["powers"], mp["speeds"], L=mp["L"], n_sweeps=mp["n_sweeps"],
                                           start=(mp["L"] / 2, 0.0), n_seeds=20, defect_fraction=3e-3, impurity_c=0.1,
                                           output_root=root, metrics_every=100, batch=mp["batch"], **kw),
                                        campaign.merge_melt_pool_map, mp["L"])):
                runs = []
                for axis in (None, AXIS):
                    root = f"{name}_{axis}"
                    t0 = time.perf_counter()
                    fn(root, {} if axis is None else dict(boundary_axis=axis))
                    merge(root)
                    runs.append(dict(boundary_axis=axis, wall_s=time.perf_counter() - t0))
                plain = _tree_files(f"outputs/{name}_None")
                runs[1]["preexisting_files_identical"] = all(
                    filecmp.cmp(os.path.join(f"outputs/{name}_None", f), os.path.join(f"outputs/{name}_{AXIS}", f),
                                shallow=False) for f in plain)
                mname = "cet_map" if name == "gr" else "melt_pool_map"
                cases = []
                with open(f"outputs/{name}_{AXIS}/{mname}_boundary.csv") as fh:
                    for r in csv.DictReader(fh):
                        prefix = (f"T{float(r['T_sub']):g}_R{float(r['NU_DEP']):g}" if name == "gr"
                                  else f"P{float(r['power']):g}_V{float(r['speed']):g}")
                        nw = case_network(f"outputs/{name}_{AXIS}/{prefix}/boundaries.csv")
                        cases.append(dict(r, null=NULL, shares=nw["shares"], planes=nw["planes"]))
                        print(json.dumps({k: v for k, v in cases[-1].items() if k != "planes"}), flush=True)
                runs[1]["cases"] = cases
                out[name] = dict(settings=gr if name == "gr" else mp, runs=runs)
                print(json.dumps({k: v for k, v in runs[1].items() if k != "cases"}), flush=True)
        finally:
            os.chdir(cwd)
    return out


def compact_json(o, ind=0):
    """JSON with one line per leaf: a dict or list of scalars (or of dicts and lists of scalars only) on one line."""
    def leaf(x):
        return not isinstance(x, (dict, list)) or all(not isinstance(v, (dict, list)) for v in (x.values() if isinstance(x, dict) else x))
    if leaf(o):
        return json.dumps(o)
    pad = " " * (ind + 1)
    if isinstance(o, dict):
        body = ",\n".join(f"{pad}{json.dumps(k)}: {compact_json(v, ind + 1)}" for k, v in o.items())
        return "{\n" + body + "\n" + " " * ind + "}"
    return "[\n" + ",\n".join(pad + compact_json(v, ind + 1) for v in o) + "\n" + " " * ind + "]"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="boundary_group.json")
    ap.add_argument("--quick", action="store_true", help="a small subset (rehearsal)")
    args = ap.parse_args()
    _lib.require_gpu()
    res = dict(gpu=gpu_info(), settings=dict(reps=REPS, axis=AXIS, lattices="_synth.half_grown(fill=1.0)",
                                             edges_deg=list(_lib.BOUNDARY_EDGES_DEG)))
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
        fh.write(compact_json(res) + "\n")


if __name__ == "__main__":
    main()
