"""BASELINE configs[4]: the G-R parameter sweep (batched independent lattices, replicas only) over the
GPUs of one box, producing cet_map.csv and the tree the reference's plot_cet.py reads.

    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29541 \
        scripts/run_gr_sweep.py [--L 64] [--sweeps 400] [--out gr_sweep] [--batch 16] [--replicas 4]

--batch k: the cases of a GPU advance in groups of up to k lattices (one kernel launch per group and kernel);
the outputs are the same as without it.
--replicas n: every case runs n times (replica r with seed + r and initial-lattice seed 42 + r); rank 0 also writes
cet_map_ensemble.csv (mean, standard error and equiaxed fraction over the replicas of each case) and prints it.
--profile-axis a: every case also records per-plane grain profiles along axis a (0, 1 or 2; the generated lattices
grow along 2) in <case>/cet_profile.csv; rank 0 writes cet_map_profile.csv (CET height and front height of every
lattice) and prints it, and with --replicas also cet_map_profile_ensemble.csv.
--shape-axis a: every case also records the growth-axis elongation histogram of its grains along axis a in
<case>/grain_shape.csv; rank 0 writes cet_map_shape.csv (columnar volume and grain fractions of every lattice) and
prints it, and with --replicas also cet_map_shape_ensemble.csv.
--front-axis a: every case also records the solidification conditions at its front along growth axis a (front height
and roughness, gradient, undercooling, velocity) in <case>/front.csv; rank 0 writes cet_map_front.csv (the measured
G_Front and V_Front of every lattice beside the nominal G and R) and prints it, and with --replicas also
cet_map_front_ensemble.csv.
--texture-axis a: every case also records the per-plane orientation histograms of its occupied sites along growth
axis a in <case>/texture.csv; rank 0 writes cet_map_texture.csv (mean cosine, Hermans factor and aligned fraction of every
lattice) and prints it, and with --replicas also cet_map_texture_ensemble.csv.
--boundary-axis a: every case also records the per-plane bond counts and boundary misorientation histograms of its
labelling along growth axis a in <case>/boundaries.csv; rank 0 writes cet_map_boundary.csv (linear intercepts along and
across the axis, their ratio, boundary fraction and mean misorientation of every lattice) and prints it, and with
--replicas also cet_map_boundary_ensemble.csv.
"""
import argparse
import csv
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

from cetkmc import campaign


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, default=64)
    ap.add_argument("--sweeps", type=int, default=401)
    ap.add_argument("--out", default="gr_sweep")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--replicas", type=int, default=None)
    ap.add_argument("--profile-axis", type=int, default=None, choices=(0, 1, 2))
    ap.add_argument("--shape-axis", type=int, default=None, choices=(0, 1, 2))
    ap.add_argument("--front-axis", type=int, default=None, choices=(0, 1, 2))
    ap.add_argument("--texture-axis", type=int, default=None, choices=(0, 1, 2))
    ap.add_argument("--boundary-axis", type=int, default=None, choices=(0, 1, 2))
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    temps = [2600.0, 2800.0, 3000.0, 3200.0]                      # T_sub -> G = (T_MELT - T_sub) / (L dx)
    nu_deps = [1e12, 5e12, 2e13, 1e14]                            # NU_DEP -> R
    t0 = time.perf_counter()
    rows = campaign.run_gr_sweep(temps, nu_deps, L=args.L, n_sweeps=args.sweeps, n_seeds=20, defect_fraction=3e-3,
                                 impurity_c=0.1, output_root=args.out, metrics_every=100, batch=args.batch, replicas=args.replicas,
                                 **({} if args.profile_axis is None else {"profile_axis": args.profile_axis}),
                                 **({} if args.shape_axis is None else {"shape_axis": args.shape_axis}),
                                 **({} if args.front_axis is None else {"front_axis": args.front_axis}),
                                 **({} if args.texture_axis is None else {"texture_axis": args.texture_axis}),
                                 **({} if args.boundary_axis is None else {"boundary_axis": args.boundary_axis}))
    dt = time.perf_counter() - t0
    # replicas only: the one rendezvous is "everybody is done" before rank 0 merges the per-rank files
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
        dist.barrier()
    if rank == 0:
        merged = campaign.merge_cet_map(args.out)
        wall = time.perf_counter() - t0
        sites = len(temps) * len(nu_deps) * (args.replicas or 1) * args.L ** 3 * args.sweeps
        print(json.dumps({"cases": len(merged), "world": world, "L": args.L, "sweeps": args.sweeps, "batch": args.batch, "replicas": args.replicas, "wall_s": wall,
                          "rank0_s": dt, "site_updates_per_s": sites / wall,
                          "classes": sorted(set(r["CET_Class"] for r in merged))}))
        for r in merged:
            print(f"case {int(r['case']):2d} T_sub {float(r['T_sub']):6.0f} NU_DEP {float(r['NU_DEP']):8.1e} G/R {float(r['G_over_R']):9.3e} "
                  f"AR {float(r['AspectRatio']):.3f} eq {float(r['EquiaxedFraction']):.3f} grains {int(float(r['GrainCount']))} {r['CET_Class']}")
        if args.boundary_axis is not None:
            for fn in ("cet_map_boundary.csv",) + (("cet_map_boundary_ensemble.csv",) if args.replicas is not None else ()):
                with open(f"outputs/{args.out}/{fn}") as fh:
                    for e in csv.DictReader(fh):
                        print(json.dumps(e))
        if args.texture_axis is not None:
            for fn in ("cet_map_texture.csv",) + (("cet_map_texture_ensemble.csv",) if args.replicas is not None else ()):
                with open(f"outputs/{args.out}/{fn}") as fh:
                    for e in csv.DictReader(fh):
                        print(json.dumps(e))
        if args.front_axis is not None:
            for fn in ("cet_map_front.csv",) + (("cet_map_front_ensemble.csv",) if args.replicas is not None else ()):
                with open(f"outputs/{args.out}/{fn}") as fh:
                    for e in csv.DictReader(fh):
                        print(json.dumps(e))
        if args.shape_axis is not None:
            for fn in ("cet_map_shape.csv",) + (("cet_map_shape_ensemble.csv",) if args.replicas is not None else ()):
                with open(f"outputs/{args.out}/{fn}") as fh:
                    for e in csv.DictReader(fh):
                        print(json.dumps(e))
        if args.profile_axis is not None:
            for fn in ("cet_map_profile.csv",) + (("cet_map_profile_ensemble.csv",) if args.replicas is not None else ()):
                with open(f"outputs/{args.out}/{fn}") as fh:
                    for e in csv.DictReader(fh):
                        print(json.dumps(e))
        if args.replicas is not None:
            with open(f"outputs/{args.out}/cet_map_ensemble.csv") as fh:
                for e in csv.DictReader(fh):
                    print(json.dumps(e))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
