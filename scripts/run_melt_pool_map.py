"""A melt-pool CET map: one laser-driven lattice per (beam power, scan speed) point (replicas only) over the GPUs of
one box, producing melt_pool_map.csv and the tree the reference's plot_cet.py reads.

    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29542 \
        scripts/run_melt_pool_map.py [--L 64] [--sweeps 401] [--out melt_pool_map] [--batch 16] [--replicas 4]

--batch k: the cases of a GPU advance in groups of up to k lattices (one kernel launch per group and kernel for the
sweeps and for the laser step); the outputs are the same as without it.
--replicas n: every case runs n times (replica r with seed + r and initial-lattice seed 42 + r); rank 0 also writes
melt_pool_map_ensemble.csv (mean, standard error and equiaxed fraction over the replicas of each case) and prints it.
--profile-axis a: every case also records per-plane grain profiles along axis a (0, 1 or 2; the generated lattices
grow along 2) in <case>/cet_profile.csv; rank 0 writes melt_pool_map_profile.csv (CET height and front height of every
lattice) and prints it, and with --replicas also melt_pool_map_profile_ensemble.csv.
"""
import argparse
import csv
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cetkmc import campaign


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, default=64)
    ap.add_argument("--sweeps", type=int, default=401)
    ap.add_argument("--out", default="melt_pool_map")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--replicas", type=int, default=None)
    ap.add_argument("--profile-axis", type=int, default=None, choices=(0, 1, 2))
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    powers = [100.0, 200.0, 300.0, 400.0]                         # W
    speeds = [0.25, 0.5, 1.0, 2.0]                                # voxels per thermal step along axis 1
    t0 = time.perf_counter()
    campaign.run_melt_pool_map(powers, speeds, L=args.L, n_sweeps=args.sweeps, start=(args.L / 2, 0.0),
                               n_seeds=20, defect_fraction=3e-3, impurity_c=0.1, output_root=args.out,
                               metrics_every=100, batch=args.batch, replicas=args.replicas,
                               **({} if args.profile_axis is None else {"profile_axis": args.profile_axis}))
    dt = time.perf_counter() - t0
    # replicas only: the one rendezvous is "everybody is done" before rank 0 merges the per-rank files
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
        dist.barrier()
    if rank == 0:
        merged = campaign.merge_melt_pool_map(args.out)
        wall = time.perf_counter() - t0
        sites = len(powers) * len(speeds) * (args.replicas or 1) * args.L ** 3 * args.sweeps
        print(json.dumps({"cases": len(merged), "world": world, "L": args.L, "sweeps": args.sweeps, "batch": args.batch, "replicas": args.replicas,
                          "wall_s": wall, "rank0_s": dt, "site_updates_per_s": sites / wall,
                          "classes": sorted(set(r["CET_Class"] for r in merged))}))
        for r in merged:
            print(f"case {int(r['case']):2d} P {float(r['power']):6.1f} W V {float(r['speed']):5.2f} "
                  f"AR {float(r['AspectRatio']):.3f} eq {float(r['EquiaxedFraction']):.3f} grains {int(float(r['GrainCount']))} "
                  f"step {r['Step']} {r['CET_Class']}")
        if args.profile_axis is not None:
            for fn in ("melt_pool_map_profile.csv",) + (("melt_pool_map_profile_ensemble.csv",) if args.replicas is not None else ()):
                with open(f"outputs/{args.out}/{fn}") as fh:
                    for e in csv.DictReader(fh):
                        print(json.dumps(e))
        if args.replicas is not None:
            with open(f"outputs/{args.out}/melt_pool_map_ensemble.csv") as fh:
                for e in csv.DictReader(fh):
                    print(json.dumps(e))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
