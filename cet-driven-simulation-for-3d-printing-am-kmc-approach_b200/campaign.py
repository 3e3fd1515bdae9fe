"""Large-lattice drivers and on-disk contracts around the hot path (SURVEY §8f rows N2 and N4).

    save_lattice / load_lattice      the reference's five-file .npy snapshot (lattice_init.py:98-105)
    checkpoint / resume              the same set plus the defect mask and the run counters: a
                                     run can be stopped and continued (the reference cannot)
    run_cet_sublattice               the large-lattice analogue of run_kmc (kmc_simulation.py:203-398):
                                     synchronous-sublattice sweeps on the resident lattice, the
                                     200-step cadence (defect-mask refresh, clustering, metrics row)
                                     on the device, outputs/<prefix>/metrics.csv with the reference's
                                     18 columns; optionally the laser / latent-heat thermal step
                                     (thermal_solver.update_temperature, :36-105) with a melt pool
                                     moving along axis 1 at a fixed speed — SURVEY §8d config 3
    run_melt_pool_map                a CET map over laser power x scan speed: one laser-driven
                                     run_cet_sublattice per point, optionally advanced in groups
                                     (cetkmc.thermal_full_group + sweep_run_group)
    run_gr_sweep                     config 5: independent lattices over a grid of (G, R), one per
                                     GPU (replicas only, no communication), one cet_map.csv and a tree
                                     the unmodified plot_cet.py reads (write_plot_cet_tree)
    ensemble_stats                   mean, standard error and equiaxed fraction over the replicas of
                                     each point of a map (run_gr_sweep / run_melt_pool_map, replicas=n)
    profile_axis=0|1|2               (run_cet_sublattice and the map drivers) per-plane grain profiles of
                                     every metrics row in outputs/<prefix>/cet_profile.csv
                                     (cetkmc.grain_profile_group), and per map the CET height of every
                                     lattice (metrics.cet_profile_summary) in <map>_profile.csv
"""
from __future__ import annotations

import json
import os

import numpy as np

from . import _host, _lib
from . import defects as _defects
from . import kmc_simulation as _ks
from . import metrics as _metrics
from ._config import constants, rate_params, thermal_full_params, thermal_params
from .thermal_solver import DEFAULT_ABSORPTIVITY, DEFAULT_BEAM_RADIUS, laser_source_top

_FILES = ("state", "orientation_theta", "orientation_phi", "temperature", "atom_type")


def save_lattice(state, orientation_theta, orientation_phi, T, atom_type, prefix="init"):
    """lattice_init.py:98-105 — `<prefix>_{state,orientation_theta,orientation_phi,temperature,atom_type}.npy`."""
    for name, a in zip(_FILES, (state, orientation_theta, orientation_phi, T, atom_type)):
        np.save(f"{prefix}_{name}.npy", a)


def load_lattice(prefix="init"):
    """Inverse of save_lattice: (state, theta, phi, T, atom_type) in the reference's dtypes."""
    st, th, ph, T, at = (np.load(f"{prefix}_{name}.npy") for name in _FILES)
    return (np.ascontiguousarray(st, dtype=np.int64), np.ascontiguousarray(th, dtype=np.float64),
            np.ascontiguousarray(ph, dtype=np.float64), np.ascontiguousarray(T, dtype=np.float64),
            np.ascontiguousarray(at, dtype=np.int64))


def checkpoint(ctx, prefix, **meta):
    """Write the resident lattice as the reference's snapshot set plus `<prefix>_defects.npy` and
    `<prefix>_meta.json` (run counters)."""
    f = ctx.download(state=True, atom_type=True, theta=True, phi=True, T=True)
    save_lattice(f["state"], f["theta"], f["phi"], f["T"], f["atom_type"], prefix=prefix)
    np.save(f"{prefix}_defects.npy", (ctx.download_packed() >> 4).astype(np.int64))
    idx, tau, t = ctx.sweep_state()
    meta = dict(meta, sweep_clock=[idx, float.hex(tau), float.hex(t)], numpy_rng=_rng_to_json(np.random.get_state()))
    with open(f"{prefix}_meta.json", "w") as fh:
        json.dump(meta, fh)


def resume(ctx, prefix):
    """Load a checkpoint into `ctx`; returns the meta dict."""
    st, th, ph, T, _at = load_lattice(prefix)
    df = np.load(f"{prefix}_defects.npy") if os.path.exists(f"{prefix}_defects.npy") else None
    ctx.upload(state=st, theta=th, phi=ph, T=T, defects=df)
    meta = {}
    if os.path.exists(f"{prefix}_meta.json"):
        with open(f"{prefix}_meta.json") as fh:
            meta = json.load(fh)
    if "sweep_clock" in meta:
        idx, tau, t = meta["sweep_clock"]
        ctx.sweep_set_state(int(idx), float.fromhex(tau), float.fromhex(t))
    if "numpy_rng" in meta:
        np.random.set_state(_rng_from_json(meta["numpy_rng"]))
    return meta


def _rng_to_json(st):
    return [st[0], np.asarray(st[1]).tolist(), int(st[2]), int(st[3]), float(st[4])]


def _rng_from_json(j):
    return (j[0], np.array(j[1], dtype=np.uint32), int(j[2]), int(j[3]), float(j[4]))


def _gr(L, temp, nu_dep):
    """kmc_simulation.py:236-239 with the run's own T_sub / NU_DEP."""
    G = (constants.T_MELT - temp) / (L * constants.VOXEL_SIZE)
    R = nu_dep * 2.74e-10 / constants.VOXEL_SIZE
    R_phys = nu_dep * constants.ATOMIC_SPACING_W
    return G, R, R_phys, (G / R_phys if R_phys > 0 else np.inf)


def _slab_comm(world):
    """Rendezvous helpers of a multi-GPU run (one process per GPU under torch.distributed.run): the
    process group is only plumbing — NCCL unique id broadcast and the small host-side gathers of the
    metrics cadence; the lattice exchange itself is libcetkmc's (comm.cu)."""
    import torch
    import torch.distributed as dist
    if not dist.is_initialized():
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo")

    def all_gather(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    def bcast_bytes(b):
        box = [b]
        dist.broadcast_object_list(box, src=0)
        return box[0]
    return all_gather, bcast_bytes


def _upload_initial(ctx, L, n_seeds, temp, impurity_c, lattice, i_begin, i_end):
    """The run's initial lattice on the device: initialize_lattice + introduce_defects (NumPy's global stream,
    seeded with ctx.init_seed when the driver set one, else with initialize_lattice's default 42), or the given
    `lattice`.  A context whose driver set ctx.init_nuclei to a list (the grouped driver) gets a generated lattice
    appended there in sparse form instead (_host.initial_nuclei, the same draws); the driver then builds the
    lattices of its whole group with one cetkmc.init_group call."""
    init_seed = getattr(ctx, "init_seed", None)
    if lattice is None and getattr(ctx, "init_nuclei", None) is not None:
        ctx.init_nuclei.append(_host.initial_nuclei(L, n_seeds, temp, 42 if init_seed is None else init_seed,
                                                    impurity_c))
        return
    if lattice is None:
        state, theta, phi, T, atom_type = _ks.initialize_lattice(
            lattice_size=L, n_seeds=n_seeds, T_sub=temp, impurity_c=impurity_c,
            **({} if init_seed is None else {"random_seed": init_seed}))
        defects_mask, _ = _ks.introduce_defects(state, atom_type, T, apply_to_state=False)
    else:
        state, theta, phi, T, atom_type = lattice[:5]
        defects_mask = lattice[5] if len(lattice) > 5 else None
    own = slice(i_begin, i_end)
    ctx.upload(state=np.ascontiguousarray(state[own], dtype=np.int64), theta=theta[own], phi=phi[own], T=T[own],
               defects=None if defects_mask is None else defects_mask[own])


def _sweep_setup(L, seed, temp, events_per_sweep, p_max, defect_fraction, thermal_every):
    """Sweep and thermal parameters of a run (thermal_every 0: no update_temperature_cet in the sweeps)."""
    sp = _lib.SweepParams()
    sp.seed = seed
    sp.events_per_sweep = float(events_per_sweep if events_per_sweep is not None else 0.005 * L ** 3)
    sp.p_max, sp.defect_fraction = float(p_max), float(defect_fraction)
    sp.thermal_every = int(thermal_every)
    tp = None if not thermal_every else thermal_params(_ks.THERMAL_DT, nan_to_num=True, t_floor=temp)
    return sp, tp


def _stop_at(sweep, every, n_sweeps):
    """The last sweep of the next metrics interval (run_kmc's cadence)."""
    return min(((sweep + every - 1) // every) * every, n_sweeps - 1)


def _cadence(ctx, last, every, philox_mask, seed, world, total_time, nucleation_count, cet_detected, consts,
             verbose, all_gather=None):
    """What follows the sweeps of a metrics interval that ended at sweep `last`: the defect-mask refresh on
    multiples of `every` (kmc_simulation.py:335-338) and the metrics row.  Returns (row, cet_detected)."""
    if last % every == 0:
        if not philox_mask:
            _defects.refresh_resident(ctx)
        else:
            ctx.defects_refresh(draws=None, seed=seed, epoch=last // every, prob_base=constants.DEFECT_PROB_BASE,
                                e_mig=_defects.E_MIGRATION, kT=constants.K_T, T_default=constants.T_SUB,
                                carbon_id=_defects.CARBON_ID, defect_id=constants.DEFECT_ID)
            if world > 1:
                ctx.halo_exchange(1)                                          # the ghost copies of the mask nibble
    return _ks._metrics_row(last, total_time, nucleation_count, cet_detected, consts, ctx, verbose=verbose,
                            all_gather=all_gather)


def _cadence_group(runs, last, every, philox_mask, seed, profile_axis=None):
    """_cadence for every case of a group at once (cetkmc.metrics_group, one launch per kernel for the group): the
    defect-mask refresh on multiples of `every` and each case's metrics row, appended to r["rows"].  The Philox
    stream is keyed by r["seed"] where a case has one, else by `seed`.  With NumPy's
    stream each case draws its mask from its own saved position (r["rng"]), in group order, as refresh_resident
    draws it.  profile_axis: one cetkmc.grain_profile_group call over the labelling the rows used appends each
    case's (step, profile) to r["profiles"]."""
    ctxs = [r["ctx"] for r in runs]
    refresh = last % every == 0
    draws = None
    if refresh and not philox_mask:
        draws = []
        for r, n_c in zip(runs, _lib.counts_group(ctxs)[:, _defects.CARBON_ID]):
            np.random.set_state(r["rng"])
            draws.append(np.random.random(int(n_c)) if n_c > 0 else np.zeros(0))      # defects.py:9,18
            r["rng"] = np.random.get_state()
    n_sites = int(np.prod(ctxs[0].owned_shape))
    params = []
    for run in runs:
        p = _lib.MetricsParams()
        p.theta_threshold, p.ar_threshold = 0.5, constants.CET_AR_THRESHOLD
        p.pct_pos[:] = _metrics.percentile_positions(n_sites)
        p.refresh, p.carbon_id, p.epoch, p.seed = int(refresh), _defects.CARBON_ID, last // every, run.get("seed", seed)
        p.prob_base, p.e_mig, p.kT, p.T_default = constants.DEFECT_PROB_BASE, _defects.E_MIGRATION, constants.K_T, constants.T_SUB
        params.append(p)
    for r, res in zip(runs, _lib.metrics_group(ctxs, params, draws)):
        m = _metrics.metrics_from_summary(res, n_sites, voxel_size=constants.VOXEL_SIZE)
        row, r["cet_detected"] = _ks._row_from_metrics(last, r["total_time"], r["nucleation_count"], r["cet_detected"],
                                                       r["consts"], res["counts"], m, n_sites, verbose=False)
        r["rows"].append(row)
    if profile_axis is not None:
        for r, prof in zip(runs, _lib.grain_profile_group(ctxs, profile_axis, constants.CET_AR_THRESHOLD)):
            r["profiles"].append((last, prof))


PROFILE_CSV = "cet_profile.csv"


def _check_profile_axis(fn, profile_axis, world=1, checkpoint_every=0, resume_from=None):
    """Refuse what a run with per-plane grain profiles does not take: an axis outside {0, 1, 2}, a lattice split into
    slabs (their labels are slab-local) and checkpoints (they do not carry the profile history)."""
    if profile_axis is None:
        return
    if isinstance(profile_axis, bool) or not isinstance(profile_axis, (int, np.integer)) or int(profile_axis) not in (0, 1, 2):
        raise ValueError(f"{fn}: profile_axis must be None, 0, 1 or 2, got {profile_axis!r}")
    if world > 1:
        raise ValueError(f"{fn}: profile_axis needs a whole lattice on one GPU (world = 1)")
    if checkpoint_every or resume_from:
        raise ValueError(f"{fn}: profile_axis does not take checkpoint_every or resume_from")


def _check_mask_and_laser(fn, mask_stream, laser, thermal_every):
    """Refuse a defect-mask stream other than "numpy" or "philox", and a laser run (`laser` true) without a thermal
    step (thermal_every < 1)."""
    if mask_stream not in ("numpy", "philox"):
        raise ValueError("mask_stream must be 'numpy' or 'philox'")
    if laser and int(thermal_every) < 1:
        raise ValueError(f"{fn}: the laser variant needs thermal_every >= 1")


def _write_profile_csv(profiles, output_dir):
    """outputs/<prefix>/cet_profile.csv: one row per (metrics row, plane) of the (step, (4, L) profile) pairs."""
    import csv
    if not profiles:
        return
    with open(os.path.join(output_dir, PROFILE_CSV), "w", newline="") as fh:
        w = csv.writer(fh)
        w.writerow(("Step", "Plane") + _lib.PROFILE_COLUMNS)
        for step, prof in profiles:
            for z in range(prof.shape[1]):
                w.writerow([int(step), z] + [int(v) for v in prof[:, z]])


def read_profile_csv(path):
    """The last metrics row's profile of a cet_profile.csv: (step, (4, L) int64 array)."""
    import csv
    with open(path) as fh:
        rows = list(csv.DictReader(fh))
    step = rows[-1]["Step"]
    last = [r for r in rows if r["Step"] == step]
    prof = np.array([[int(r[c]) for r in last] for c in _lib.PROFILE_COLUMNS], np.int64)
    return int(step), prof


def run_cet_sublattice(L=None, n_sweeps=2000, temp=None, defect_fraction=0.0, n_seeds=5, impurity_c=0.0,
                       output_prefix="cet_sublattice", metrics_every=None, events_per_sweep=None, p_max=0.1,
                       nu_dep=None, laser=None, thermal_every=_ks.THERMAL_EVERY, device=0, seed=None,
                       checkpoint_every=0, resume_from=None, lattice=None, verbose=True, rank=0, world=1,
                       mask_stream="numpy", init_seed=None, profile_axis=None):
    """run_kmc's large-lattice sibling.  Same set-up (initialize_lattice + introduce_defects with the
    run's seed), same cadence and CSV; the steps are synchronous-sublattice sweeps (csrc/sweep.cu), so
    `Step` counts sweeps and `Time` is the accumulated sweep interval.

    laser: None -> update_temperature_cet every `thermal_every` sweeps (the reference's driver);
           dict(power=W, speed=voxels per thermal step along axis 1, start=(i0, j0), dt=s,
           beam_radius=m, absorptivity=) -> thermal_solver.update_temperature with the moving source.
    lattice: optional (state, theta, phi, T, atom_type[, defects]) to start from instead of
           initialize_lattice.  Returns (state, atom_type, total_time, theta, phi) like run_kmc.
    init_seed: the random_seed of initialize_lattice (None: its default, 42).  `seed` keys the sweeps and the
           defect-mask stream; init_seed picks the initial nuclei.
    profile_axis: None, or 0, 1 or 2: every metrics row also takes the per-plane grain profile of the labelling it
           used along that axis (cetkmc.grain_profile_group), written to outputs/<prefix>/cet_profile.csv with the
           columns Step, Plane, Solid, EquiaxedSolid, GrainsSpanning, EquiaxedGrainsSpanning, one row per (metrics
           row, plane).  Every other output is the same as without it.  Not with world > 1, checkpoint_every or
           resume_from.
    world > 1: the lattice is split into z-slabs, one per rank / GPU (launch every rank with the same
           arguments plus its rank; torch.distributed.run provides the rendezvous).  The trajectory and
           the CSV do not depend on the number of slabs.  Rank 0 writes the CSV; every rank returns its
           own planes.  The laser variant and checkpoints are single-GPU.
    mask_stream: "numpy" — the 200-step defect-mask refresh consumes NumPy's global stream in C order
           like defects.py:18 (single GPU only); "philox" — the device's counter-based stream keyed by
           (seed, refresh number, global site), which a slab run always uses (an ordered host stream
           cannot be split over slabs); a single-GPU run with "philox" equals the slab run bit for bit.
    `Time` is the accumulated sweep interval (a physical clock); run_kmc's CSV carries the reference's
    clock, which its 1e-12 s floor makes a step counter (Time = 1e-12 s x steps, SURVEY 3.3) — the two
    columns are not comparable and level-3 parity is therefore matched by executed events (tests).
    """
    L = constants.LATTICE_SIZE if L is None else int(L)
    temp = constants.T_SUB if temp is None else temp
    nu_dep = constants.NU_DEP if nu_dep is None else nu_dep
    seed = constants.RANDOM_SEED if seed is None else int(seed)
    every = constants.METRIC_UPDATE_STEP if metrics_every is None else int(metrics_every)
    _check_profile_axis("run_cet_sublattice", profile_axis, world, checkpoint_every, resume_from)
    np.random.seed(seed)                                    # a resumed run restores the stream position below
    output_dir = f"outputs/{output_prefix}"
    os.makedirs(output_dir, exist_ok=True)
    consts = _gr(L, temp, nu_dep)

    if world > 1 and (laser or checkpoint_every or resume_from):
        raise ValueError("run_cet_sublattice: the laser variant and checkpoint / resume are single-GPU")
    _check_mask_and_laser("run_cet_sublattice", mask_stream, laser, thermal_every)
    philox_mask = world > 1 or mask_stream == "philox"
    all_gather = None
    i_begin, i_end = _ks.slab_bounds(L, world, rank)
    ctx = _lib.Context(L=L, device=device, i_begin=i_begin, i_end=i_end, halo=_ks.SWEEP_HALO if world > 1 else 0)
    ctx.init_seed = init_seed
    try:
        ctx.set_rate_params(rate_params(impurity_c, 1, 2, 3, overrides={"NU_DEP": nu_dep}))
        sweep0, total_time, nucleation_count, cet_detected, rows, profiles = 0, 0.0, 0, False, [], []
        if resume_from:
            meta = resume(ctx, resume_from)
            sweep0, total_time = int(meta.get("sweep", 0)), float(meta.get("time", 0.0))
            nucleation_count, cet_detected = int(meta.get("nucleation_count", 0)), bool(meta.get("cet_detected", False))
            rows = list(meta.get("rows", []))
        else:
            _upload_initial(ctx, L, n_seeds, temp, impurity_c, lattice, i_begin, i_end)
        if world > 1:
            all_gather, bcast_bytes = _slab_comm(world)
            ctx.comm_init(bcast_bytes(_lib.comm_unique_id() if rank == 0 else None), rank, world)
            ctx.halo_exchange(7)
        sp, tp = _sweep_setup(L, seed, temp, events_per_sweep, p_max, defect_fraction, 0 if laser else thermal_every)
        if laser:
            l_dt = float(laser.get("dt", _ks.THERMAL_DT))
            l_pos = [float(x) for x in laser.get("start", (0.0, 0.0))]
            tfp = thermal_full_params(l_dt)

        def advance(n):
            """n sweeps; with a laser the thermal step is driven from here every `thermal_every` sweeps."""
            nonlocal total_time, nucleation_count
            done, terminated = 0, False
            while done < n and not terminated:
                blk = n - done if not laser else min(n - done, thermal_every - ((sweep + done) % thermal_every))
                if laser and (sweep + done) % thermal_every == 0:
                    ctx.thermal_full(tfp, laser_source_top(L, tuple(l_pos), float(laser["power"]),
                                                           float(laser.get("beam_radius", DEFAULT_BEAM_RADIUS)),
                                                           float(laser.get("absorptivity", DEFAULT_ABSORPTIVITY))))
                    ctx.snapshot_state()                     # prev_state of the next latent-heat term
                    l_pos[1] += float(laser.get("speed", 0.0))
                res = ctx.sweep_run(blk, sp, tp)
                total_time += res["time"]
                nucleation_count += res["nucleation_count"] if world == 1 else int(np.sum(all_gather(res["nucleation_count"])))
                done += res["sweeps_done"]
                terminated = bool(res["terminated"]) or res["sweeps_done"] == 0
                if res["overflow"]:
                    raise RuntimeError("fired-event list overflowed: lower events_per_sweep")
            return done, terminated

        sweep = sweep0
        if laser:
            ctx.snapshot_state()
        terminated = False
        while sweep < n_sweeps and not terminated:
            done, terminated = advance(_stop_at(sweep, every, n_sweeps) - sweep + 1)
            sweep += done
            row, cet_detected = _cadence(ctx, sweep - 1, every, philox_mask, seed, world, total_time, nucleation_count,
                                         cet_detected, consts, verbose=verbose and rank == 0, all_gather=all_gather)
            rows.append(row)
            if profile_axis is not None:
                profiles.append((sweep - 1, _lib.grain_profile_group([ctx], profile_axis, constants.CET_AR_THRESHOLD)[0]))
            if checkpoint_every and (len(rows) % checkpoint_every == 0):
                checkpoint(ctx, os.path.join(output_dir, "checkpoint"), sweep=sweep, time=total_time,
                           nucleation_count=nucleation_count, cet_detected=cet_detected,
                           rows=[{k: (v if not isinstance(v, (np.generic,)) else v.item()) for k, v in r.items()} for r in rows])
        if rank == 0:
            _ks._write_csv(rows, output_dir)
            _write_profile_csv(profiles, output_dir)
        f = ctx.download(state=True, atom_type=True, theta=True, phi=True)
    finally:
        ctx.close()
    return f["state"], f["atom_type"], total_time, f["theta"], f["phi"]


def gr_partition(n_cases, rank, world, devices, batch=None):
    """Which cases of a G-R sweep this rank runs, where, and together with which: a list of
    (device, [case numbers]).  Case q belongs to rank q % world and runs on devices[(q // world) % len(devices)];
    batch=None runs every case on its own, batch=k the cases of one device in groups of up to k lattices
    (in case order)."""
    mine = [q for q in range(n_cases) if q % world == rank]
    if batch is None:
        return [(devices[(q // world) % len(devices)], [q]) for q in mine]
    if int(batch) < 1 or int(batch) > _lib.GROUP_MAX:
        raise ValueError(f"run_gr_sweep: batch must be 1 to {_lib.GROUP_MAX}, got {batch}")
    by_dev = {}
    for q in mine:
        by_dev.setdefault(devices[(q // world) % len(devices)], []).append(q)
    return [(d, qs[i:i + int(batch)]) for d, qs in by_dev.items() for i in range(0, len(qs), int(batch))]


def run_gr_sweep(temps, nu_deps, L=64, n_sweeps=400, impurity_c=0.0, n_seeds=20, defect_fraction=0.0,
                 output_root="gr_sweep", rank=None, world=None, devices=None, batch=None, replicas=None, **kw):
    """SURVEY §8d config 5: one independent lattice per (T_sub, NU_DEP) grid point — T_sub sets the
    thermal gradient G = (T_MELT - T_sub) / (L dx), NU_DEP the growth velocity R (kmc_simulation.py:
    236-239).  Replicas only: case q runs on rank q % world (torchrun: RANK / WORLD_SIZE / LOCAL_RANK)
    or, in a single process, on device q % len(devices).  Every case writes its own metrics.csv; the
    rank that owns a case appends its final row to outputs/<output_root>/cet_map_rank<r>.csv, and
    merge_cet_map() joins them into cet_map.csv (columns G, R, G_over_R, AspectRatio,
    EquiaxedFraction, GrainCount, CET_Class, ...).
    batch=k: the cases of one device advance in groups of up to k lattices, one kernel launch per group
    and kernel (cetkmc.sweep_run_group) instead of one per lattice; every output file is the same as
    with batch=None.  Not with `laser`, `checkpoint_every`, `resume_from` or `lattice`.
    replicas=n: every case runs n times, replica r as run_cet_sublattice(seed=seed + r, init_seed=42 + r) writing
    outputs/<prefix>/metrics.csv for r = 0 and outputs/<prefix>/rep<r>/metrics.csv for r >= 1; the (case, replica)
    lattices are partitioned and grouped as cases are.  cet_map_rank<r>.csv and the plot_cet tree come from
    replica 0, so they equal those of a run without replicas; each rank also writes cet_map_replicas_rank<r>.csv
    (one row per (case, replica), the map's columns).  Returns (map rows, ensemble_stats rows; None when
    world > 1) instead of the map rows.  Not with `checkpoint_every`, `resume_from` or `lattice`.
    profile_axis=a (through **kw): every case writes outputs/<prefix>/cet_profile.csv (run_cet_sublattice), and each
    rank writes cet_map_profile_rank<r>.csv (_map_profile_rows); every other file is the same as without it."""
    cases = [(float(t), float(r)) for t in temps for r in nu_deps]

    def case_row(q):
        temp, nu_dep = cases[q]
        G, R, _rp, _gr_phys = _gr(L, temp, nu_dep)
        return {"T_sub": temp, "NU_DEP": nu_dep, "G": G, "R": R, "G_over_R": G / R if R > 0 else np.inf}
    return _run_map("run_gr_sweep", "cet_map", ("T_sub", "NU_DEP"), case_row, output_root,
                    [(f"{output_root}/T{temp:g}_R{nu_dep:g}", temp, nu_dep) for temp, nu_dep in cases], None,
                    ("laser", "checkpoint_every", "resume_from", "lattice"), rank, world, devices, batch, replicas,
                    dict(kw, L=L, n_sweeps=n_sweeps, impurity_c=impurity_c, n_seeds=n_seeds,
                         defect_fraction=defect_fraction))


def _run_map(fn, name, axes, case_row, output_root, cases, lasers, batch_refuses, rank, world, devices, batch,
             replicas, kw):
    """The body of the map driver `fn` (run_gr_sweep, run_melt_pool_map): every replica of case q of `cases` (output
    prefix, temp, nu_dep) is run_cet_sublattice(output_prefix=..., temp=..., nu_dep=..., laser=lasers[q] unless
    lasers is None, **kw), partitioned over ranks and devices by gr_partition; batch=k advances them in groups
    (_run_cases_grouped) and refuses the keywords `batch_refuses`.  Writes and returns the map `name` (_map_outputs)."""
    rank = int(os.environ.get("RANK", 0)) if rank is None else rank
    world = int(os.environ.get("WORLD_SIZE", 1)) if world is None else world
    devices = [int(os.environ.get("LOCAL_RANK", 0))] if devices is None else list(devices)
    n_rep = _check_replicas(fn, replicas, kw)
    _check_profile_axis(fn, kw.get("profile_axis"), 1, kw.get("checkpoint_every"), kw.get("resume_from"))
    _check_mask_and_laser(fn, kw.get("mask_stream", "numpy"), lasers is not None or kw.get("laser"),
                          kw.get("thermal_every", _ks.THERMAL_EVERY))
    if batch is not None:
        bad = [k for k in batch_refuses if kw.get(k)]
        if bad:
            raise ValueError(f"{fn}: batch does not take {', '.join(bad)}")
    os.makedirs(f"outputs/{output_root}", exist_ok=True)
    lats = _map_lattices([p for p, _t, _r in cases], n_rep)
    parts = gr_partition(len(lats), rank, world, devices, batch)
    for device, ls in parts:
        if batch is None:
            q, r, p = lats[ls[0]]
            run_cet_sublattice(output_prefix=p, temp=cases[q][1], nu_dep=cases[q][2], device=device, verbose=False,
                               **({} if lasers is None else {"laser": lasers[q]}), **_replica_kw(kw, replicas, r))
        else:
            _run_cases_grouped([(lats[l][2],) + cases[lats[l][0]][1:] for l in ls], device=device,
                               lasers=None if lasers is None else [lasers[lats[l][0]] for l in ls],
                               replicas=None if replicas is None else [lats[l][1] for l in ls], **kw)
    return _map_outputs(output_root, name, lats, [l for _d, ls in parts for l in ls], case_row, axes, replicas, rank,
                        world, kw.get("profile_axis"))


_MAP_FINAL = ("Step", "Time", "AspectRatio", "EquiaxedFraction", "GrainCount", "AvgGrainSize", "NucleationCount",
              "CET_Class", "CET_Detected")
ENSEMBLE_COLUMNS = ("AspectRatio", "EquiaxedFraction", "GrainCount", "AvgGrainSize", "NucleationCount", "Step")


def _check_replicas(fn, replicas, kw):
    """Replicas per case of a map driver (1 for replicas=None), refusing what a replica run does not take."""
    if replicas is None:
        return 1
    if int(replicas) < 1:
        raise ValueError(f"{fn}: replicas must be >= 1, got {replicas}")
    bad = [k for k in ("lattice", "resume_from", "checkpoint_every") if kw.get(k)]
    if bad:
        raise ValueError(f"{fn}: replicas does not take {', '.join(bad)}")
    return int(replicas)


def _map_lattices(prefix, n_rep):
    """The lattices of a map, case by case: (case, replica, output prefix).  Replica 0 of case q writes to prefix[q],
    replica r >= 1 to <prefix[q]>/rep<r>."""
    return [(q, r, p if r == 0 else f"{p}/rep{r}") for q, p in enumerate(prefix) for r in range(n_rep)]


def _replica_kw(kw, replicas, r):
    """run_cet_sublattice's keywords for replica r of a case: seed + r and init_seed = 42 + r (kw itself without
    replicas)."""
    if replicas is None:
        return kw
    seed = kw.get("seed")
    return dict(kw, seed=(constants.RANDOM_SEED if seed is None else int(seed)) + r, init_seed=42 + r)


def _map_outputs(output_root, name, lats, mine, case_row, axes, replicas, rank, world, profile_axis=None):
    """The per-rank files of a map driver over the lattices `mine` (indices into `lats`) this rank ran:
    <name>_rank<rank>.csv (case, case_row(case), the final row's _MAP_FINAL columns) and the plot_cet tree from
    replica 0 of each case, with replicas <name>_replicas_rank<rank>.csv, one row per (case, replica), and with
    profile_axis <name>_profile_rank<rank>.csv (_map_profile_rows).  Returns the map rows; with replicas (map rows,
    ensemble_stats of the replica rows), the latter None when world > 1 (merge_* joins the ranks)."""
    import csv
    rows, rep_rows = [], []
    for l in sorted(mine):
        q, r, p = lats[l]
        with open(f"outputs/{p}/metrics.csv") as fh:
            last = list(csv.DictReader(fh))[-1]
        row = {"case": q, **case_row(q), **{k: last[k] for k in _MAP_FINAL}}
        rep_rows.append({"case": q, "replica": r, **{k: v for k, v in row.items() if k != "case"}})
        if r == 0:
            rows.append(row)
    out_dir = f"outputs/{output_root}"
    _write_rows(rows, os.path.join(out_dir, f"{name}_rank{rank}.csv"))
    if profile_axis is not None:
        _write_rows(_map_profile_rows(lats, sorted(mine), case_row, axes),
                    os.path.join(out_dir, f"{name}_profile_rank{rank}.csv"))
    write_plot_cet_tree([(row["case"], f"outputs/{lats[l][2]}/metrics.csv")
                         for row, l in zip(rows, sorted(l for l in mine if lats[l][1] == 0))],
                        os.path.join(out_dir, "plot_cet"))
    if replicas is None:
        return rows
    _write_rows(rep_rows, os.path.join(out_dir, f"{name}_replicas_rank{rank}.csv"))
    return rows, (ensemble_stats(rep_rows, axes) if world == 1 else None)


def _map_profile_rows(lats, mine, case_row, axes):
    """One row per lattice of `mine` (case, replica, the map's axis columns, CET_Height and Front_Height of
    metrics.cet_profile_summary over the final row's profile in outputs/<prefix>/cet_profile.csv)."""
    out = []
    for l in mine:
        q, r, p = lats[l]
        _step, prof = read_profile_csv(f"outputs/{p}/{PROFILE_CSV}")
        s = _metrics.cet_profile_summary(prof, prof.shape[1] ** 2)
        c = case_row(q)
        out.append({"case": q, "replica": r, **{k: c[k] for k in axes}, "CET_Height": s["CET_Height"],
                    "Front_Height": s["Front_Height"]})
    return out


def profile_ensemble_stats(rows, axes):
    """One row per case over the rows of a <map>_profile.csv (dicts with case, replica, the axis columns `axes`,
    CET_Height; numbers or the strings a CSV gives back), in case order: case, the axes, replicas (n), p_cet_height
    (the fraction of replicas with a CET height >= 0) and CET_Height_mean / CET_Height_se over those replicas (the
    standard error is the sample standard deviation, ddof=1, over the square root of their number; empty below 2,
    the mean empty when no replica has a CET height)."""
    by_case = {}
    for r in rows:
        by_case.setdefault(int(r["case"]), []).append(r)
    out = []
    for case in sorted(by_case):
        rs = by_case[case]
        h = np.array([int(r["CET_Height"]) for r in rs])
        v = h[h >= 0].astype(np.float64)
        out.append({"case": case, **{k: rs[0][k] for k in axes}, "replicas": len(rs),
                    "p_cet_height": float(np.mean(h >= 0)),
                    "CET_Height_mean": float(np.mean(v)) if v.size else "",
                    "CET_Height_se": float(np.std(v, ddof=1) / np.sqrt(v.size)) if v.size > 1 else ""})
    return out


def ensemble_stats(rows, axes):
    """One row per case over the replica rows `rows` of a map (dicts with case, the axis columns `axes`, G, R,
    G_over_R, ENSEMBLE_COLUMNS, CET_Class and CET_Detected; numbers, or the strings a CSV gives back), in case order:
    case, the axes, G, R, G_over_R, replicas (n), <col>_mean and <col>_se for every column of ENSEMBLE_COLUMNS (the
    standard error is the sample standard deviation, ddof=1, over sqrt(n); empty for n = 1), p_equiaxed (the
    fraction of replicas whose final CET_Class is Equiaxed) with its binomial standard error sqrt(p (1 - p) / n)
    as p_equiaxed_se, and p_cet_detected (the fraction with CET_Detected)."""
    by_case = {}
    for r in rows:
        by_case.setdefault(int(r["case"]), []).append(r)
    out = []
    for case in sorted(by_case):
        rs = by_case[case]
        n = len(rs)
        e = {"case": case, **{k: rs[0][k] for k in tuple(axes) + ("G", "R", "G_over_R")}, "replicas": n}
        for col in ENSEMBLE_COLUMNS:
            v = np.array([float(r[col]) for r in rs])
            e[f"{col}_mean"] = float(np.mean(v))
            e[f"{col}_se"] = float(np.std(v, ddof=1) / np.sqrt(n)) if n > 1 else ""
        p = float(np.mean([r["CET_Class"] == "Equiaxed" for r in rs]))
        e["p_equiaxed"], e["p_equiaxed_se"] = p, float(np.sqrt(p * (1.0 - p) / n))
        e["p_cet_detected"] = float(np.mean([str(r["CET_Detected"]) == "True" for r in rs]))
        out.append(e)
    return out


def _run_cases_grouped(cases, L, n_sweeps, impurity_c, n_seeds, defect_fraction, device, metrics_every=None,
                       events_per_sweep=None, p_max=0.1, thermal_every=_ks.THERMAL_EVERY, seed=None, mask_stream="numpy",
                       lasers=None, replicas=None, profile_axis=None):
    """run_cet_sublattice(output_prefix=p, temp=t, nu_dep=r, ...) for every (p, t, r) of `cases` on one device, the
    lattices advancing together by sweep_run_group.  Each case has its own set-up, cadence and metrics.csv exactly as
    alone; with mask_stream="numpy" each case keeps its own position in NumPy's global stream (saved and restored
    around its host draws).  The metrics cadence of the group is one cetkmc.metrics_group call per row
    (_cadence_group).  A case that terminates leaves the group after the block of sweeps it terminated in, with its
    row at that block's last sweep, as run_cet_sublattice stops it; a block is a metrics interval, or with lasers the
    part of one between two thermal steps.
    lasers: None, or one laser dict per case (run_cet_sublattice(laser=...)): every `thermal_every` sweeps one
    cetkmc.thermal_full_group over the cases still running replaces their thermal_full + snapshot_state.
    replicas: None, or the replica number r of each case: the case then runs as run_cet_sublattice(seed=seed + r,
    init_seed=42 + r).  The generated initial lattices of the group are built on the device by one cetkmc.init_group
    call (_upload_initial).
    profile_axis: every metrics row also takes its cases' grain profiles with one cetkmc.grain_profile_group call
    (_cadence_group), and each case writes the cet_profile.csv run_cet_sublattice(profile_axis=...) writes."""
    _check_mask_and_laser("_run_cases_grouped", mask_stream, lasers is not None, thermal_every)
    _check_profile_axis("_run_cases_grouped", profile_axis)
    seed = constants.RANDOM_SEED if seed is None else int(seed)
    every = constants.METRIC_UPDATE_STEP if metrics_every is None else int(metrics_every)
    philox_mask = mask_stream == "philox"
    reps = [0] * len(cases) if replicas is None else [int(r) for r in replicas]
    runs = []
    try:
        for q, (prefix, temp, nu_dep) in enumerate(cases):
            seed_q = seed + reps[q]
            np.random.seed(seed_q)
            os.makedirs(f"outputs/{prefix}", exist_ok=True)
            ctx = _lib.Context(L=L, device=device)
            ctx.init_seed = None if replicas is None else 42 + reps[q]
            ctx.init_nuclei = []
            r = dict(ctx=ctx, prefix=prefix, seed=seed_q, consts=_gr(L, temp, nu_dep), rows=[], profiles=[], total_time=0.0,
                     nucleation_count=0, cet_detected=False, terminated=False)
            runs.append(r)
            ctx.set_rate_params(rate_params(impurity_c, 1, 2, 3, overrides={"NU_DEP": nu_dep}))
            _upload_initial(ctx, L, n_seeds, temp, impurity_c, None, 0, L)
            r["sp"], r["tp"] = _sweep_setup(L, seed_q, temp, events_per_sweep, p_max, defect_fraction,
                                            0 if lasers is not None else thermal_every)
            r["rng"] = np.random.get_state()
            if lasers is not None:
                r["laser"] = lasers[q]
                r["tfp"] = thermal_full_params(float(lasers[q].get("dt", _ks.THERMAL_DT)))
                r["pos"] = [float(x) for x in lasers[q].get("start", (0.0, 0.0))]
        gen = [r["ctx"] for r in runs if r["ctx"].init_nuclei]
        if gen:
            _lib.init_group(gen, [c.init_nuclei[0] for c in gen], snapshot=lasers is not None)
        if lasers is not None:
            for r in runs:
                if not r["ctx"].init_nuclei:                         # uploaded dense: a given lattice
                    r["ctx"].snapshot_state()
        sweep = 0
        active = runs
        while sweep < n_sweeps and active:
            end = _stop_at(sweep, every, n_sweeps) + 1
            while sweep < end and active:
                blk = end - sweep if lasers is None else min(end - sweep, thermal_every - sweep % thermal_every)
                if lasers is not None and sweep % thermal_every == 0:
                    _laser_step_group(active, L)
                tps = None if active[0]["tp"] is None else [r["tp"] for r in active]     # one thermal_every for all cases
                _absorb(active, _lib.sweep_run_group([r["ctx"] for r in active], blk, [r["sp"] for r in active], tps))
                sweep += blk
                stopped = [r for r in active if r["terminated"]]
                if stopped:
                    _cadence_group(stopped, sweep - 1, every, philox_mask, seed, profile_axis)
                    active = [r for r in active if not r["terminated"]]
            if active:
                _cadence_group(active, sweep - 1, every, philox_mask, seed, profile_axis)
        for r in runs:
            _ks._write_csv(r["rows"], f"outputs/{r['prefix']}")
            _write_profile_csv(r["profiles"], f"outputs/{r['prefix']}")
    finally:
        for r in runs:
            r["ctx"].close()


def _absorb(runs, results):
    """Add the sweep results of a group to its cases' running totals."""
    for r, res in zip(runs, results):
        if res["overflow"]:
            raise RuntimeError("fired-event list overflowed: lower events_per_sweep")
        r["total_time"] += res["time"]
        r["nucleation_count"] += res["nucleation_count"]
        r["terminated"] = bool(res["terminated"]) or res["sweeps_done"] == 0


def _laser_step_group(runs, L):
    """The laser driver's thermal step of run_cet_sublattice (thermal_full, snapshot_state, the melt pool moves on)
    for every case of `runs`, one cetkmc.thermal_full_group call."""
    q_tops = []
    for r in runs:
        las = r["laser"]
        q_tops.append(laser_source_top(L, tuple(r["pos"]), float(las["power"]),
                                       float(las.get("beam_radius", DEFAULT_BEAM_RADIUS)),
                                       float(las.get("absorptivity", DEFAULT_ABSORPTIVITY))))
    _lib.thermal_full_group([r["ctx"] for r in runs], [r["tfp"] for r in runs], q_tops, snapshot=True)
    for r in runs:
        r["pos"][1] += float(r["laser"].get("speed", 0.0))


def run_melt_pool_map(powers, speeds, L=64, n_sweeps=400, temp=None, nu_dep=None, start=(0.0, 0.0), dt=None,
                      beam_radius=DEFAULT_BEAM_RADIUS, absorptivity=DEFAULT_ABSORPTIVITY, impurity_c=0.0, n_seeds=20,
                      defect_fraction=0.0, output_root="melt_pool_map", rank=None, world=None, devices=None,
                      batch=None, replicas=None, **kw):
    """A CET map over the two quantities of the moving melt pool a user sets: beam power (W) and scan speed (voxels
    per thermal step along axis 1).  Case q of powers x speeds (in that order) is run_cet_sublattice(laser=dict(
    power=P, speed=V, start=start, dt=dt, beam_radius=..., absorptivity=...), output_prefix=
    "<output_root>/P<P>_V<V>"), every case with the same temp, nu_dep, seed and cadence.  Cases are partitioned over
    ranks and devices as in run_gr_sweep (gr_partition).  Every case writes its own metrics.csv; each rank writes
    outputs/<output_root>/melt_pool_map_rank<r>.csv (case, power, speed, T_sub, NU_DEP, G, R, G_over_R and the final
    row's Step, Time, AspectRatio, EquiaxedFraction, GrainCount, AvgGrainSize, NucleationCount, CET_Class,
    CET_Detected) and adds its cases to the plot_cet tree; merge_melt_pool_map() joins the rank files.
    batch=k: the cases of one device advance in groups of up to k lattices (cetkmc.sweep_run_group for the sweeps,
    cetkmc.thermal_full_group for the laser steps); every output file is the same as with batch=None.  Not with
    `checkpoint_every`, `resume_from` or `lattice`.
    replicas=n: every case runs n times, replica r as run_cet_sublattice(seed=seed + r, init_seed=42 + r) writing
    outputs/<prefix>/metrics.csv for r = 0 and outputs/<prefix>/rep<r>/metrics.csv for r >= 1; the (case, replica)
    lattices are partitioned and grouped as cases are.  The map file and the plot_cet tree come from replica 0, so
    they equal those of a run without replicas; each rank also writes melt_pool_map_replicas_rank<r>.csv (one row
    per (case, replica), the map's columns).  Returns (map rows, ensemble_stats rows; None when world > 1).
    Not with `checkpoint_every`, `resume_from` or `lattice`.
    profile_axis=a (through **kw): every case writes outputs/<prefix>/cet_profile.csv (run_cet_sublattice), and each
    rank writes melt_pool_map_profile_rank<r>.csv (_map_profile_rows); every other file is the same as without it."""
    powers, speeds = [float(p) for p in powers], [float(v) for v in speeds]
    if not powers or not speeds:
        raise ValueError("run_melt_pool_map: needs at least one power and one speed")
    temp = constants.T_SUB if temp is None else float(temp)
    nu_dep = constants.NU_DEP if nu_dep is None else float(nu_dep)
    dt = _ks.THERMAL_DT if dt is None else float(dt)
    cases = [(p, v) for p in powers for v in speeds]
    lasers = [dict(power=p, speed=v, start=tuple(start), dt=dt, beam_radius=beam_radius, absorptivity=absorptivity)
              for p, v in cases]
    G, R, _rp, _gr_phys = _gr(L, temp, nu_dep)

    def case_row(q):
        return {"power": cases[q][0], "speed": cases[q][1], "T_sub": temp, "NU_DEP": nu_dep, "G": G, "R": R,
                "G_over_R": G / R if R > 0 else np.inf}
    return _run_map("run_melt_pool_map", "melt_pool_map", ("power", "speed", "T_sub", "NU_DEP"), case_row, output_root,
                    [(f"{output_root}/P{p:g}_V{v:g}", temp, nu_dep) for p, v in cases], lasers,
                    ("checkpoint_every", "resume_from", "lattice"), rank, world, devices, batch, replicas,
                    dict(kw, L=L, n_sweeps=n_sweeps, impurity_c=impurity_c, n_seeds=n_seeds,
                         defect_fraction=defect_fraction))


def write_plot_cet_tree(cases, root):
    """Lay per-case metrics files out the way the reference's plot_cet.py discovers them
    (plot_cet.py:26: `outputs/impurity_c_<id>/metrics_<id>.csv` below the working directory; it
    labels a series "<id>% C", reads Step / AspectRatio / DefectDensity / EquiaxedFraction, :49-71):
    `<root>/outputs/impurity_c_<id>/metrics_<id>.csv` for every (id, path of a metrics.csv) in `cases`.
    Run the unmodified script from `<root>`: `cd <root> && python /path/to/plot_cet.py`; for a G-R
    sweep the id is the case number of cet_map.csv (which holds its T_sub, NU_DEP, G and R).  Every
    rank of a sweep adds its own cases."""
    import shutil
    for cid, path in cases:
        d = os.path.join(root, "outputs", f"impurity_c_{int(cid)}")
        os.makedirs(d, exist_ok=True)
        shutil.copyfile(path, os.path.join(d, f"metrics_{int(cid)}.csv"))
    return root


def _write_rows(rows, path):
    import csv
    if not rows:
        return
    with open(path, "w", newline="") as fh:
        w = csv.DictWriter(fh, fieldnames=list(rows[0].keys()))
        w.writeheader()
        w.writerows(rows)


def _merge_rank_files(output_root, name):
    """Join outputs/<output_root>/<name>_rank*.csv into outputs/<output_root>/<name>.csv (sorted by case and
    replica)."""
    import csv
    import glob
    rows = []
    for p in sorted(glob.glob(f"outputs/{output_root}/{name}_rank*.csv")):
        with open(p) as fh:
            rows += list(csv.DictReader(fh))
    rows.sort(key=lambda r: (int(r["case"]), int(r.get("replica", 0))))
    _write_rows(rows, f"outputs/{output_root}/{name}.csv")
    return rows


def _merge_map(output_root, name, axes):
    rows = _merge_rank_files(output_root, name)
    reps = _merge_rank_files(output_root, f"{name}_replicas")
    if reps:
        _write_rows(ensemble_stats(reps, axes), f"outputs/{output_root}/{name}_ensemble.csv")
    prof = _merge_rank_files(output_root, f"{name}_profile")
    if prof and reps:
        _write_rows(profile_ensemble_stats(prof, axes), f"outputs/{output_root}/{name}_profile_ensemble.csv")
    return rows


def merge_cet_map(output_root="gr_sweep"):
    """Join the per-rank files of run_gr_sweep into outputs/<output_root>/cet_map.csv (sorted by case); after a run
    with replicas also cet_map_replicas.csv and cet_map_ensemble.csv (ensemble_stats, one row per case); after a run
    with profile_axis also cet_map_profile.csv (sorted by case and replica), and with replicas
    cet_map_profile_ensemble.csv (profile_ensemble_stats)."""
    return _merge_map(output_root, "cet_map", ("T_sub", "NU_DEP"))


def merge_melt_pool_map(output_root="melt_pool_map"):
    """Join the per-rank files of run_melt_pool_map into outputs/<output_root>/melt_pool_map.csv (sorted by case);
    after a run with replicas also melt_pool_map_replicas.csv and melt_pool_map_ensemble.csv (ensemble_stats); after
    a run with profile_axis also melt_pool_map_profile.csv and, with replicas, melt_pool_map_profile_ensemble.csv."""
    return _merge_map(output_root, "melt_pool_map", ("power", "speed", "T_sub", "NU_DEP"))
