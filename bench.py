#!/usr/bin/env python
"""bench.py — KMC site-updates/s of the sublattice sweep on the 512^3 lattice (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl cetkmc|reference]
                    [--scaling strong|weak] [--L 512] [--thermal cet|laser] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One step = one synchronous-sublattice sweep over the whole lattice (csrc/sweep.cu): thermal stencil
+ dense rate rebuild when due (every 20 sweeps, kmc_simulation.py:248), one fire decision per site
against its resident rate sum, event pick + conflict resolution + apply for the fired sites,
neighbour-rate refresh of the sites the events touched, totals for the next time increment, and
(N > 1) the halo exchange.
Workload: the 'half-grown' synthetic lattice of SURVEY §8(d)(ii), 512^3 at N = 1 (the lattice the
metric names).
    default / --scaling weak   : N GPUs hold (512 N) x 512 x 512 split into z-slabs, 512 planes each
    --scaling strong           : the same L^3 lattice split into z-slabs over the N GPUs: --L 512 is the
                                 metric's lattice at 2/4/8 GPUs, --L 1024 is BASELINE configs[3]
    --thermal laser            : BASELINE configs[2] — the thermal step is thermal_solver.update_temperature
                                 (laser source + latent heat, thermal_solver.py:36-105) with the melt pool
                                 moving along axis 1, driven between 20-sweep blocks (N = 1)

Prints ONE JSON line (rank 0).  Keys beyond the base contract: roofline (dominant kernel, live
CUDA-event timing), roofline_all, cpu_baseline (the oracle port on the host cores, bounded sample),
e2e (the sweep API call with host buffers, copies inside the timed region), api_e2e (the reference-
signature calls run_kmc / update_temperature_cet / get_event_rates, host arrays in, host arrays out),
clocks, gpu_launches.

--dump-outputs DIR (N = 1) writes, after the timed sweeps, what they left on the device as DIR/<name>.npy:
the lattice a caller of the sweep receives (state, defects, theta, phi, T) and the resident site rate sums
at a fixed seeded sample of sites (site_index), the deposition rates of the top plane (dep_rate, 0 where a
site offers no deposition), and the counters the timed sweep call returned (sweep_<name>).
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L_BENCH = 512
THERMAL_EVERY = 20
EVENTS_FRACTION = 0.005         # events_per_sweep = 0.5 % of the sites (fidelity at this setting: tests/test_gpu_sweep.py, level 3)
P_MAX = 0.1
# Algorithmic bytes per unit (SURVEY §8d; DESIGN.md §4).  The contract figure of the rate evaluation is
# 33 B/site (1 B state + 8 B theta + 8 B phi + 8 B T read, 8 B rate sum written); the resident layout the
# kernels read is listed beside it as bytes_layout.
BYTES_STREAM = 8                # resident rate sum read once per site
BYTES_RATES = 33
BYTES_RATES_LAYOUT = 25         # compact tile state: 1 B class code + 8 B pair operand + 8 B T read, 8 B written
BYTES_STAMP = 1.0 / 8.0         # refresh scan: one stamp BIT per site
BYTES_THERMAL = 16              # T read + T written
CPU_SAMPLE_L = 160              # cpu_baseline leg of the GPU arm: one 160^3 block of the same workload (~10 s)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _oracle(threads):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    os.environ["OMP_NUM_THREADS"] = str(threads)
    O.build()
    return O


def cpu_rate_sample(threads):
    """The oracle port (oracle/oracle.c, OpenMP over planes) evaluating every event rate of a
    CPU_SAMPLE_L^3 block of the benchmark workload — the reference's get_event_rates sweep, which
    is what one 'site-update' costs on the CPU path (kmc_simulation.py:253)."""
    O = _oracle(threads)
    from cetkmc import _synth
    Ls = CPU_SAMPLE_L
    packed, th, ph, T = _synth.half_grown(Ls, seed=1234)
    st, df = _synth.unpack(packed)
    p = O.make_params(0.1)
    t0 = time.perf_counter()
    reps = 0
    while True:
        O.site_rates(st, th, ph, T, df, Ls, p)
        reps += 1
        dt = time.perf_counter() - t0
        if dt > 10.0 or reps >= 400:                 # ~10 s of host work (bounded sample)
            break
    return Ls ** 3 * reps / dt, dt, reps


def workload_name(args, world):
    L = args.L
    if args.scaling == "weak":
        shape = f"{L * world}x{L}x{L} ({L} planes per GPU)"
    else:
        shape = f"{L}x{L}x{L}" + (f" split into {world} z-slabs" if world > 1 else "")
    therm = ("update_temperature_cet" if args.thermal == "cet" else "update_temperature with a moving laser source")
    return (f"half-grown lattice {shape} (SURVEY 8d-ii: 25% solid, salt-and-pepper below a wavy front, linear G), "
            f"synchronous-sublattice sweeps with resident rates + neighbour-rate refresh, {therm} and dense rate "
            f"rebuild every {THERMAL_EVERY} sweeps, events_per_sweep={EVENTS_FRACTION}N, p_max={P_MAX}, defect_fraction=3e-3")


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm for this path on all host threads.  The
    reference is pure Python / Numba and cannot travel to the GPU box (the tier forbids shipping its
    sources), so this arm times its C restatement (oracle/oracle.c, OpenMP, pinned bit-exact to the
    reference by tests/) on the SAME lattice the GPU arm sweeps at N = 1: one step = one full
    get_event_rates evaluation of the half-grown L^3 lattice — what every executed event of the
    reference's loop costs (kmc_simulation.py:253).  For scale: the reference's own single-thread
    Numba path measured 3.4e5 sites/s in the build container (BASELINE.md §2), ~200x below this port."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    O = _oracle(threads)
    from cetkmc import _synth
    Ls = args.L
    packed, th, ph, T = _synth.half_grown(Ls, seed=1234)
    st, df = _synth.unpack(packed)
    del packed
    p = O.make_params(0.1)
    for _ in range(max(min(args.warmup, 3), 1)):
        O.site_rates(st, th, ph, T, df, Ls, p)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.site_rates(st, th, ph, T, df, Ls, p)        # one full rate sweep = one visit of every site
    dt = time.perf_counter() - t0
    value = Ls ** 3 * args.steps / dt
    sample = f"the whole half-grown {Ls}^3 lattice, one full event-rate evaluation per step (oracle.c, OpenMP, {threads} threads)"
    print(json.dumps({
        "impl": "reference", "metric": "kmc_site_updates_per_s", "value": value, "unit": "site-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, 1)},
        "cpu_baseline": {"value": value, "unit": "site-updates/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "site-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def pinned(shape, dtype):
    """Page-locked host array (torch allocator) — falls back to pageable memory."""
    try:
        import torch
        t = torch.empty(tuple(shape), dtype={np.float64: torch.float64, np.uint8: torch.uint8, np.int64: torch.int64}[dtype],
                        pin_memory=True)
        return t.numpy(), t
    except Exception:
        return np.empty(shape, dtype=dtype), None


DUMP_SITES = 1 << 20            # sampled sites: 48 B each over 7 arrays, ~50 MB in all with dep_rate at 512^2


def dump_outputs(ctx, res, out_dir):
    """--dump-outputs: the resident lattice and rate sums at a fixed seeded sample of DUMP_SITES sites
    (all of them on a smaller lattice), the deposition rates of the top plane, and the sweep counters.
    Every value written is finite; a non-finite one is an error."""
    os.makedirs(out_dir, exist_ok=True)
    n = int(np.prod(ctx.owned_shape))
    idx = np.arange(n) if n <= DUMP_SITES else np.unique(np.random.default_rng(0).integers(0, n, DUMP_SITES))
    packed = ctx.download_packed().reshape(-1)[idx]
    out = {"site_index": idx.astype(np.float64), "state": (packed & 15).astype(np.float32),
           "defects": (packed >> 4).astype(np.float32)}
    for name in ("theta", "phi", "T"):
        out[name] = ctx.download(**{name: True})[name].reshape(-1)[idx]
    sr, dr = ctx.rates_download()
    # the device marks a top-plane site without a deposition event (occupied, or rate at or below the
    # threshold) with NaN; such a site offers rate 0, as kmc_exact.cu reads it
    out["site_rate_sum"], out["dep_rate"] = sr.reshape(-1)[idx], np.where(np.isnan(dr), 0.0, dr)
    for k, v in res.items():
        out["sweep_" + k] = np.float64(v)
    bad = [name for name, a in out.items() if not np.all(np.isfinite(a))]
    if bad:
        raise RuntimeError(f"--dump-outputs: non-finite values in {bad}")
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def api_e2e():
    """The reference-signature calls (host NumPy arrays in, host NumPy arrays out), wall clock around
    the call as a user makes it: run_kmc at the main.py default lattice, update_temperature_cet at
    512^3, get_event_rates at 128^3 (BASELINE configs[0..1])."""
    import io
    import tempfile
    from cetkmc import _synth, kmc_event_rates, kmc_simulation, thermal_solver
    out = {}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        stdout, sys.stdout = sys.stdout, io.StringIO()
        try:
            kw = dict(L=30, temp=2800, defect_fraction=3e-3, n_seeds=20, impurity_c=0.1, output_prefix="bench")
            kmc_simulation.run_kmc(n_steps=201, **kw)                   # warm-up (library load, first launches)
            dt = float("inf")
            for _ in range(2):                                          # host-side Python dominates: best of two
                t0 = time.perf_counter()
                kmc_simulation.run_kmc(n_steps=4001, **kw)
                dt = min(dt, time.perf_counter() - t0)
        finally:
            sys.stdout = stdout
            os.chdir(cwd)
    out["run_kmc_L30"] = {"value": 4001 / dt, "unit": "KMC steps/s",
                          "what": "run_kmc(L=30, n_steps=4001, defect_fraction=3e-3, n_seeds=20, impurity_c=0.1) incl. lattice "
                                  "set-up, metrics rows and CSV; reference: 11.7 steps/s (BASELINE.md)"}
    T = np.ascontiguousarray(np.broadcast_to(2800.0 + 895.0 * np.arange(512) / 512, (512, 512, 512)))
    thermal_solver.update_temperature_cet(T[:64], None, dt=1e-6)
    dt = float("inf")
    for _ in range(2):
        t0 = time.perf_counter()
        T2 = thermal_solver.update_temperature_cet(T, None, dt=1e-6)
        dt = min(dt, time.perf_counter() - t0)
    out["update_temperature_cet_512"] = {"value": T.size / dt, "unit": "sites/s", "h2d_bytes": T.nbytes, "d2h_bytes": T2.nbytes,
                                         "what": "one call, (512,512,512) float64 host array in, new host array out (pageable "
                                                 "memory, as a caller of the reference holds it); reference: 1.6e7 sites/s"}
    del T, T2
    packed, th, ph, Tt = _synth.half_grown(128, seed=1234)
    st, df = _synth.unpack(packed)
    t0 = time.perf_counter()
    ev = kmc_event_rates.get_event_rates(st, th, ph, Tt, st, df, 128, 1, 2, 3, impurity_c=0.1)
    dt = time.perf_counter() - t0
    out["get_event_rates_128"] = {"value": 128 ** 3 / dt, "unit": "sites/s", "events": len(ev),
                                  "what": "one call on the half-grown 128^3 lattice returning the reference's Python list of "
                                          "tuples (building the list dominates); reference: 3.4e5 sites/s"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cetkmc", choices=["cetkmc", "reference"])
    ap.add_argument("--L", type=int, default=L_BENCH, help="edge length (strong) / sites per edge in a plane and planes per GPU (weak)")
    ap.add_argument("--scaling", default="weak", choices=["strong", "weak"])
    ap.add_argument("--thermal", default="cet", choices=["cet", "laser"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-api-e2e", action="store_true")
    ap.add_argument("--debug-flags", type=int, default=0, help="refresh variant for A/B runs (cet_debug_flags)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed sweeps computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    if args.thermal == "laser" and world > 1:
        raise SystemExit("--thermal laser is the single-GPU configuration (BASELINE configs[2])")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs is the single-GPU configuration")
    warm = max(args.warmup, 3)

    import cetkmc
    from cetkmc import _synth
    from cetkmc._config import rate_params, thermal_full_params, thermal_params
    from cetkmc.kmc_simulation import slab_bounds
    cetkmc._lib.require_gpu()                       # no CPU fallback
    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"       # keep NCCL's version banner out of the one-JSON-line stdout
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    L = args.L
    if args.scaling == "weak":
        n0 = L * world
        i_begin, i_end = rank * L, (rank + 1) * L
    else:
        n0 = L
        i_begin, i_end = slab_bounds(L, world, rank)
    halo = 6 if world > 1 else 0
    packed, th, ph, T = _synth.half_grown(L, seed=1234, planes=(i_begin, i_end), n0=n0)
    own_planes = i_end - i_begin
    sites_total = n0 * L * L

    ctx = cetkmc.Context(L=L, n0=n0, device=local_rank, i_begin=i_begin, i_end=i_end, halo=halo)
    ctx.debug_flags(args.debug_flags)
    ctx.set_rate_params(rate_params(0.1))
    ctx.upload_packed(packed)
    ctx.upload(theta=th, phi=ph, T=T)
    if world > 1:
        import torch
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(cetkmc._lib.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        ctx.comm_init(bytes(uid.cpu().numpy().tobytes()), rank, world)
        ctx.halo_exchange(7)
    sp = cetkmc._lib.SweepParams()
    sp.seed, sp.events_per_sweep, sp.p_max = 42, EVENTS_FRACTION * sites_total, P_MAX
    sp.defect_fraction = 3e-3
    laser = args.thermal == "laser"
    sp.thermal_every = 0 if laser else THERMAL_EVERY
    tp = None if laser else thermal_params(1e-6, nan_to_num=True)
    if laser:
        from cetkmc.thermal_solver import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS, laser_source_top
        tfp = thermal_full_params(1e-6)
        pool = {"j": 0.25 * L}
        ctx.snapshot_state()

        def laser_step():
            # thermal_solver.update_temperature (:36-105) on the resident lattice: the top-plane source (L^2 values,
            # formed on the host with the reference's expression) follows the melt pool along axis 1
            ctx.thermal_full(tfp, laser_source_top(L, (0.0, pool["j"]), 200.0, DEFAULT_BEAM_RADIUS, DEFAULT_ABSORPTIVITY))
            ctx.snapshot_state()
            pool["j"] += 4.0

    def run_block(n):
        """n sweeps; with the laser the thermal step is driven from here before every 20-sweep block."""
        tot = None
        done = 0
        while done < n:
            blk = min(n - done, THERMAL_EVERY) if laser else n - done
            if laser:
                laser_step()
            r = ctx.sweep_run(blk, sp, tp)
            if tot is not None:                     # counts add up over the blocks; the clock is the last block's
                for k in ("events_applied", "events_fired", "sites_refreshed", "sweeps_done"):
                    r[k] += tot[k]
            tot = r
            done += blk
        return tot

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    # warm-up (a fresh clock is primed inside the first call).  Its first dense rebuild runs on the synthetic lattice
    # as generated (SURVEY 8d-ii) — the rebuild inside the timed window sees the lattice the sweeps have since evolved —
    # and is timed on the side for roofline_all
    ctx.profile_enable(True)
    run_block(warm)
    ctx.sync()
    fresh_rates = ctx.profile_read("rates")
    for k in ("decide", "pick", "apply", "refresh", "thermal", "halo", "allreduce", "boundary", "step"):
        ctx.profile_read(k)                         # drop the warm-up's spans of the other kinds
    ctx.profile_enable(False)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    ctx.profile_enable(True)
    ctx.timer_begin()
    res = run_block(args.steps)
    ms = ctx.timer_end_ms()
    clocks = sampler.stop()
    ctx.profile_enable(False)
    barrier()
    if args.dump_outputs:
        dump_outputs(ctx, res, args.dump_outputs)
    if dist is not None:
        import torch
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        ev = torch.tensor([res["events_applied"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(ev)
        events = float(ev.item())
    else:
        events = float(res["events_applied"])
    KINDS = ("decide", "pick", "apply", "refresh", "thermal", "rates", "halo", "allreduce", "boundary", "step")
    prof = {k: ctx.profile_read(k) for k in KINDS}
    value = sites_total * args.steps / (ms * 1e-3)
    peak, peak_kind = peaks()
    # planes a dense kernel processes: the owned planes plus the ghost planes it must evaluate (N > 1)
    ghost_eval = 0 if world == 1 else (4 if rank in (0, world - 1) else 8)
    eval_sites = (own_planes + ghost_eval) * L * L

    def roof(kind, nbytes, layout_bytes=None):
        t_ms, n = prof[kind]
        if n == 0 or t_ms <= 0:
            return None
        ach = nbytes / (t_ms / n * 1e-3) / 1e9
        r = {"achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "launches": int(n),
             "ms_per_launch": t_ms / n, "bytes_per_launch": nbytes}
        if layout_bytes is not None:
            r["bytes_layout_per_launch"] = layout_bytes
            r["frac_layout"] = layout_bytes / (t_ms / n * 1e-3) / 1e9 / peak
        return r

    refreshed = res["sites_refreshed"] / max(args.steps, 1)
    # the dense rebuild runs the TMA tile kernel when the rows can be described by a tensor map (sweep_tile.cu:tile_tma_ok)
    dense_k = "rates_dense_kernel" if (L % 16 == 0 and L >= 64) else "rates_compact_kernel"
    refresh_name = "dirty_scan + rates_refresh_kernel (neighbour-rate refresh)"
    dense_name = dense_k + " (dense rebuild after the thermal step)"
    rl = {
        "sweep_stream_kernel": roof("decide", BYTES_STREAM * eval_sites),
        refresh_name:
            roof("refresh", BYTES_RATES * refreshed + BYTES_STAMP * eval_sites, BYTES_RATES_LAYOUT * refreshed + BYTES_STAMP * eval_sites),
        dense_name:
            roof("rates", BYTES_RATES * eval_sites, BYTES_RATES_LAYOUT * eval_sites),
        "thermal_kernel": roof("thermal", BYTES_THERMAL * own_planes * L * L),
    }
    if fresh_rates[1] > 0 and fresh_rates[0] > 0:           # the warm-up's rebuild(s): the lattice as generated
        t_ms = fresh_rates[0] / fresh_rates[1]
        ach = BYTES_RATES * eval_sites / (t_ms * 1e-3) / 1e9
        rl[dense_k + " (same kernel on the lattice as generated, during warm-up)"] = {
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "launches": int(fresh_rates[1]),
            "ms_per_launch": t_ms, "bytes_per_launch": BYTES_RATES * eval_sites,
            "bytes_layout_per_launch": BYTES_RATES_LAYOUT * eval_sites,
            "frac_layout": BYTES_RATES_LAYOUT * eval_sites / (t_ms * 1e-3) / 1e9 / peak}
    share = {k: prof[k][0] for k in ("decide", "pick", "apply", "refresh", "thermal", "rates", "halo", "allreduce", "boundary")}
    dominant = max(share, key=share.get)
    dom_name = {"decide": "sweep_stream_kernel", "refresh": refresh_name, "rates": dense_name, "thermal": "thermal_kernel"}.get(dominant)
    traffic = None                   # dram__bytes_read+write per launch of the dominant kernel, from this round's ncu capture
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            per = json.load(f)["per_kernel"]
        pick_k = {"decide": ["sweep_stream_kernel"], "refresh": ["dirty_scan_kernel", "rates_refresh_kernel"],
                  "rates": [dense_k], "thermal": ["thermal_kernel_v2"]}.get(dominant, [])
        vals = [v for n in pick_k for k, v in per.items() if n in k]
        traffic = sum(vals) if len(vals) == len(pick_k) and vals else None
    except Exception:
        pass
    main_roof = dict(rl[dom_name]) if dom_name and rl.get(dom_name) else {"achieved": None, "peak": peak, "unit": "GB/s", "frac": None}
    main_roof.update({"bound": "hbm", "kernel": dom_name or dominant, "traffic": traffic, "peak_kind": peak_kind,
                      "share_of_step": share[dominant] / max(sum(share.values()), 1e-9)})
    n_thermal = int(prof["thermal"][1])
    out = {
        "metric": "kmc_site_updates_per_s", "value": value, "unit": "site-updates/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, world),
                   "l2": "fields swept per step (>= 1 GB rate sums per sweep at 512^3) exceed the 126 MB L2; no flush needed",
                   "thermal_in_window": f"{n_thermal} thermal step(s) + dense rebuild(s) fall inside the {args.steps} timed sweeps "
                                        f"(cadence {THERMAL_EVERY})",
                   "parallelism": f"zslab{world}"},
        "executed_events_per_s": events / (ms * 1e-3),
        "kernel_ms_per_step": {k: v / args.steps for k, v in share.items()},
        "step_span_ms": prof["step"][0] / args.steps,
        "roofline": main_roof,
        "roofline_all": rl,
        # per sweep: reset, stream, plane-reduce, pick, apply, stamp scan, refresh, finalize; per thermal step: stencil,
        # pair-operand update, dense rebuild; N > 1 adds 2 tile-state kernels + 2 stamp fills per cut face
        "gpu_launches": int(8 * args.steps + 3 * n_thermal + (0 if world == 1 else 4 * args.steps)),
        "clocks": clocks,
    }

    # ---- e2e: the sweep API call with host buffers (copies inside the timed region) ------------
    if not args.no_e2e and not laser:
        from cetkmc.kmc_simulation import run_kmc_sublattice_slab
        hp, _k1 = pinned(packed.shape, np.uint8); hp[...] = packed
        hth, _k2 = pinned(th.shape, np.float64); hth[...] = th
        hph, _k3 = pinned(ph.shape, np.float64); hph[...] = ph
        hT, _k4 = pinned(T.shape, np.float64); hT[...] = T
        res_buf = {"packed": pinned(packed.shape, np.uint8), "theta": pinned(th.shape, np.float64),
                   "phi": pinned(ph.shape, np.float64)}
        res_keep = {k: v[1] for k, v in res_buf.items()}            # the torch owners of the pinned pages
        res_out = {k: v[0] for k, v in res_buf.items()}
        for v in res_out.values():
            v[...] = 0                                                # touch the pages outside the timed region
        barrier()
        t0 = time.perf_counter()
        r = run_kmc_sublattice_slab(ctx, hp, hth, hph, hT, args.steps, sp, tp, out=res_out)
        barrier()
        dt = time.perf_counter() - t0
        if dist is not None:
            import torch
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        h2d = hp.nbytes + hth.nbytes + hph.nbytes + hT.nbytes
        d2h = r["packed"].nbytes + r["theta"].nbytes + r["phi"].nbytes
        out["e2e"] = {"value": sites_total * args.steps / dt, "unit": "site-updates/s",
                      "h2d_bytes_per_step": h2d / args.steps, "d2h_bytes_per_step": d2h / args.steps,
                      "what": f"run_kmc_sublattice_slab: upload packed state+theta+phi+T from pinned host memory, {args.steps} "
                              "sweeps, download packed state+theta+phi into pinned host memory; one call.  The sweep has no "
                              "reference-signature counterpart; the reference-signature calls are timed under api_e2e"}
        # the same call over one metrics interval of the reference (METRIC_UPDATE_STEP = 200, kmc_simulation.py:335: the
        # cadence at which its loop hands the lattice to the host code): the copies are paid once per 200 sweeps
        n_long = 200
        barrier()
        t0 = time.perf_counter()
        r = run_kmc_sublattice_slab(ctx, hp, hth, hph, hT, n_long, sp, tp, out=res_out)
        barrier()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        out["e2e"]["per_metrics_interval"] = {"value": sites_total * n_long / dt, "unit": "site-updates/s", "sweeps_per_call": n_long,
                                              "h2d_bytes_per_step": h2d / n_long, "d2h_bytes_per_step": d2h / n_long}
        del res_keep
    ctx.close()
    del packed, th, ph, T

    if rank == 0 and world == 1 and not args.no_api_e2e and not laser:
        out["api_e2e"] = api_e2e()
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, dt, reps = cpu_rate_sample(threads)
        out["cpu_baseline"] = {"value": v, "unit": "site-updates/s", "cores": threads, "kind": "port",
                               "sample": f"{reps} full event-rate sweeps of a {CPU_SAMPLE_L}^3 block of the same "
                                         f"workload ({dt:.1f} s, oracle.c with OpenMP over planes)"}
    if rank == 0:
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
