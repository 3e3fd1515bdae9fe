"""Drop-in for the reference's kmc_simulation.py (run_kmc, kmc_simulation.py:203-398).

`run_kmc` keeps the reference's signature, return value `(state, atom_type, total_time, theta,
phi)`, RNG streams and `outputs/<prefix>/metrics.csv`.  The lattice lives in HBM for the whole
run; the per-step body (thermal update every 20 steps, rates, BKL selection, apply, defect
injection, time increment — kmc_simulation.py:246-332) executes on the GPU in runs of up to
METRIC_UPDATE_STEP steps with the random draws of those steps injected:

    Python `random` (seeded RANDOM_SEED)   u1 select, [u2 defect], u3 time        (:265,:323,:331)
    NumPy global stream (seeded RANDOM_SEED)  theta, phi of dep/nuc events; the defect masks
    species stream                          one draw per deposition event per step
                                            (kmc_event_rates.py:65; see kmc_event_rates.seed_species)

After each run the host streams are rewound to exactly the number of draws the steps consumed,
so the streams stay in lock-step with a reference run.  Only the 200-step metrics cadence
(:335-389) comes back to the host.

`run_kmc_sublattice` is the large-lattice path (synchronous-sublattice sweeps, optionally one
slab per GPU); it has no reference counterpart.
"""
from __future__ import annotations

import os
import random

import numpy as np

from . import _host, _lib
from . import kmc_event_rates as _rates
from ._config import constants, rate_params, thermal_params

try:                                                      # the user's own modules, when present
    from lattice_init import initialize_lattice           # type: ignore
except Exception:                                         # noqa: BLE001
    initialize_lattice = _host.initialize_lattice
try:
    from defects import introduce_defects                 # type: ignore
except Exception:                                         # noqa: BLE001
    introduce_defects = _host.introduce_defects
from . import defects as _gpu_defects                     # the 200-step mask refresh runs on the resident lattice
# Observables: grains are clustered on the GPU from the resident lattice (csrc/grains.cu).
from . import metrics as _gpu_metrics
compute_metrics, compute_CET, detect_CET_transition = (_gpu_metrics.compute_metrics, _gpu_metrics.compute_CET,
                                                       _gpu_metrics.detect_CET_transition)   # kmc_simulation.py:194

LATTICE_SIZE = constants.LATTICE_SIZE
N_STEPS = constants.N_STEPS
T_SUB = constants.T_SUB

THERMAL_EVERY = 20          # kmc_simulation.py:248
THERMAL_DT = 1e-6           # kmc_simulation.py:250


def _replay(stream_state_setter, state, draw, n):
    """Rewind a host stream to `state` and consume exactly n draws."""
    stream_state_setter(state)
    draw(n)


def _metrics_row(step, total_time, nucleation_count, cet_detected, consts, ctx, verbose=True, all_gather=None):
    """kmc_simulation.py:341-378 — one metrics.csv row, from the lattice resident in `ctx`; with
    `all_gather` (a lattice split into z-slabs, one context per rank) from all slabs, identical on every rank."""
    counts = ctx.counts()
    if all_gather is None:
        n_sites = int(np.prod(ctx.owned_shape))
        grains = ctx.grains(0.5)
    else:
        counts = np.sum(all_gather(counts), axis=0)
        n_sites = int(ctx.n0 * ctx.owned_shape[1] * ctx.owned_shape[2])
        grains = _gpu_metrics.grains_distributed(ctx, all_gather, 0.5)
    m = _gpu_metrics.metrics_from_grains(grains, n_sites, voxel_size=constants.VOXEL_SIZE)
    return _row_from_metrics(step, total_time, nucleation_count, cet_detected, consts, counts, m, n_sites, verbose)


def _row_from_metrics(step, total_time, nucleation_count, cet_detected, consts, counts, m, n_sites, verbose):
    """The metrics.csv row of _metrics_row from the state histogram `counts`, the grain metrics `m`
    (metrics_from_grains or metrics_from_summary; updated in place) and the number of sites."""
    G, R, R_phys, G_over_R_phys = consts
    n_w, n_re, n_c = int(counts[1]), int(counts[2]), int(counts[3])
    defect_voxels = int(counts[constants.DEFECT_ID])
    m["Defect_voxel_count"] = defect_voxels
    m["DefectDensity"] = float(defect_voxels / n_sites)
    newly = (not cet_detected) and detect_CET_transition(m)
    if newly:
        cet_detected = True
        if verbose:
            print(f"CET detected at step {step} (G/R={G / R:.2e})")
    # compute_CET(state, theta, phi) re-clusters the same lattice and applies the same two
    # thresholds to AspectRatio / EquiaxedFraction (metrics.py:99-105); reuse m instead.
    cet_cls = "Equiaxed" if detect_CET_transition(m) else "Columnar"
    row = {
        "Step": step, "Time": total_time,
        "AspectRatio": m["AspectRatio"], "EquiaxedFraction": m["EquiaxedFraction"],
        "NucleationDensity": m["NucleationDensity"], "DefectDensity": m["DefectDensity"],
        "AvgGrainSize": m["AvgGrainSize"], "GrainCount": m["GrainCount"],
        "W_Count": n_w, "Re_Count": n_re, "C_Count": n_c, "NucleationCount": nucleation_count,
        "G_over_R": (G / R) if R > 0 else np.inf, "G_phys": G, "R_phys": R_phys,
        "G_over_R_phys": G_over_R_phys, "CET_Class": cet_cls, "CET_Detected": cet_detected,
    }
    if verbose:
        print(f"Step {step}: AR={row['AspectRatio']:.2f}, EqFrac={row['EquiaxedFraction']:.2f}, "
              f"NucDens={row['NucleationDensity']:.3e}, DefectDens={row['DefectDensity']:.3e}, "
              f"CET={row['CET_Class']}, Detected={row['CET_Detected']}, Time={row['Time']:.2e}s")
    return row, cet_detected


def _write_csv(rows, output_dir):
    if not rows:
        return None
    path = os.path.join(output_dir, "metrics.csv")
    try:
        import pandas as pd
        pd.DataFrame(rows).to_csv(path, index=False)
    except ImportError:
        import csv
        with open(path, "w", newline="") as f:
            w = csv.DictWriter(f, fieldnames=list(rows[0].keys()))
            w.writeheader()
            w.writerows(rows)
    # plot_cet.py:26 globs outputs/impurity_c_*/metrics_*.csv while the driver writes metrics.csv
    # (kmc_simulation.py:393): for main.py's `impurity_c_<pct>` prefixes the file is also written
    # under the name the plotting script looks for
    base = os.path.basename(os.path.normpath(output_dir))
    if base.startswith("impurity_c_") and base.rsplit("_", 1)[-1].isdigit():
        import shutil
        shutil.copyfile(path, os.path.join(output_dir, f"metrics_{base.rsplit('_', 1)[-1]}.csv"))
    print(f"Metrics saved to {path}")
    return path


def run_kmc(L: int = LATTICE_SIZE, n_steps: int = N_STEPS, temp: float = T_SUB,
            defect_fraction: float = 0.0, n_seeds: int = 5, impurity_c: float = 0.0,
            output_prefix: str = "cet_run", device: int = 0, event_log: list = None):
    """kmc_simulation.py:203-398 on the GPU.  Extra keyword arguments (`device`, `event_log`)
    have defaults that keep the reference's call sites unchanged; when `event_log` is a list the
    chosen event of every step is appended to it as (type, pos, target, atom, rate, total)."""
    seed = constants.RANDOM_SEED
    np.random.seed(seed)                                   # :219
    random.seed(seed)                                      # :220
    _rates.seed_species(seed)
    output_dir = f"outputs/{output_prefix}"
    os.makedirs(output_dir, exist_ok=True)

    state, theta, phi, T, atom_type = initialize_lattice(
        lattice_size=L, n_seeds=n_seeds, T_sub=temp, impurity_c=impurity_c)           # :226
    defects_mask, _ = introduce_defects(state, atom_type, T, apply_to_state=False)    # :231

    G = (constants.T_MELT - constants.T_SUB) / (L * constants.VOXEL_SIZE)             # :236-239
    R = constants.NU_DEP * 2.74e-10 / constants.VOXEL_SIZE
    R_phys = constants.NU_DEP * constants.ATOMIC_SPACING_W
    consts = (G, R, R_phys, G / R_phys)

    state = np.ascontiguousarray(state, dtype=np.int64)
    atom_type = np.ascontiguousarray(atom_type, dtype=np.int64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    phi = np.ascontiguousarray(phi, dtype=np.float64)
    T = np.ascontiguousarray(T, dtype=np.float64)

    ctx = _lib.Context(L=L, device=device)
    try:
        ctx.set_rate_params(rate_params(impurity_c, 1, 2, 3))                         # :255
        ctx.upload(state=state, theta=theta, phi=phi, T=T, defects=defects_mask)
        tp = thermal_params(THERMAL_DT, nan_to_num=True)                              # :249-250
        per_step = 3 if defect_fraction > 0.0 else 2
        every = constants.METRIC_UPDATE_STEP
        sp_rng = _rates.species_rng()
        total_time, nucleation_count, cet_detected = 0.0, 0, False
        rows = []
        step, terminated = 0, False
        last_step = -1
        while step < n_steps and not terminated:
            # run up to and including the next metrics step (multiples of `every`, and n_steps-1)
            stop_at = min(((step + every - 1) // every) * every, n_steps - 1)
            nb = stop_at - step + 1
            py_state, np_state, sp_state = random.getstate(), np.random.get_state(), sp_rng.get_state()
            py = np.fromiter((random.random() for _ in range(per_step * nb)), dtype=np.float64,
                             count=per_step * nb)
            npd = np.random.random_sample(2 * nb)
            sp_budget = nb * L * L
            spd = sp_rng.random_sample(sp_budget)
            res = ctx.kmc_run(step, nb, defect_fraction, tp, THERMAL_EVERY, py, npd, spd,
                              total_time0=total_time, log=event_log is not None)
            if res["starved"]:
                raise RuntimeError("cet_kmc_run ran out of injected draws (internal sizing error)")
            random.setstate(py_state)
            for _ in range(res["py_used"]):
                random.random()
            np.random.set_state(np_state)
            np.random.random_sample(res["np_used"])
            sp_rng.set_state(sp_state)
            sp_rng.random_sample(res["sp_used"])
            total_time = res["total_time"]
            nucleation_count += res["nucleation_count"]
            if event_log is not None:
                event_log.extend(zip(res["log_type"].tolist(), res["log_pos"].tolist(),
                                     res["log_target"].tolist(), res["log_atom"].tolist(),
                                     res["log_rate"].tolist(), res["log_total"].tolist()))
            step += res["steps_done"]
            if res["terminated"]:
                print(f"Terminating at step {step}: no valid events (rate={res['last_total_rate']:.2e})")
                terminated = True
                break
            last_step = step - 1
            # resident cadence (kmc_simulation.py:335-389): the mask refresh, the clustering and the
            # species counts all run on the device; nothing but the row's scalars crosses PCIe
            if last_step % every == 0:                                                # :335-338
                _gpu_defects.refresh_resident(ctx)
            row, cet_detected = _metrics_row(last_step, total_time, nucleation_count, cet_detected, consts, ctx)
            rows.append(row)
        ctx.download(out=dict(state=state, atom_type=atom_type, theta=theta, phi=phi, T=T))
        if terminated:
            last_step = step
        _write_csv(rows, output_dir)
        print(f"Completed {last_step + 1} steps in {total_time:.2e} s")
    finally:
        ctx.close()
    return state, atom_type, total_time, theta, phi


def slab_bounds(L: int, world: int, rank: int):
    """Planes [i_begin, i_end) of axis 0 owned by `rank`: contiguous, sizes differ by at most one."""
    base, extra = divmod(L, world)
    i_begin = rank * base + min(rank, extra)
    return i_begin, i_begin + base + (1 if rank < extra else 0)


SWEEP_HALO = 6       # ghost planes per side a slab needs for one communication per sweep


def run_kmc_sublattice_slab(ctx, packed, theta, phi, T, n_sweeps, sweep_params, thermal=None, out=None):
    """One call = upload this rank's planes from host memory (packed uint8 state | defects << 4,
    float64 theta / phi / T), refresh the ghost planes, run n_sweeps synchronous-sublattice
    sweeps, and read the lattice back.  `ctx` is an existing cetkmc.Context (already bound to its
    communicator when the lattice spans several GPUs).  `out` (optional): dict with preallocated
    `packed` / `theta` / `phi` arrays of the owned shape that receive the result — with page-locked
    buffers on both sides the copies run at PCIe speed instead of the pageable-memory rate."""
    ctx.upload_packed(packed)
    ctx.upload(theta=theta, phi=phi, T=T)
    ctx.halo_exchange(7)
    res = ctx.sweep_run(n_sweeps, sweep_params, thermal)
    if out is None:
        res["packed"] = ctx.download_packed()
        res.update(ctx.download(theta=True, phi=True))
    else:
        res["packed"] = ctx.download_packed(out=out["packed"])
        res.update(ctx.download(out=dict(theta=out["theta"], phi=out["phi"])))
    return res


def run_kmc_sublattice(state, theta, phi, T, defects_mask=None, n_sweeps=100, impurity_c=0.0,
                       defect_fraction=0.0, seed=None, events_per_sweep=None, p_max=0.1,
                       thermal_every=THERMAL_EVERY, device=0, rank=0, world=1, unique_id=None,
                       return_fields=True, packed=False):
    """Synchronous-sublattice KMC on a lattice resident in HBM (see csrc/sweep.cu).

    state/theta/phi/T/defects_mask are the FULL (L,L,L) arrays in the reference layout (or, when
    world > 1, may be the rank's own planes `slab_bounds(L, world, rank)` with 6 ghost planes
    taken from the neighbours — pass full arrays and the slicing is done here).  Every rank of a
    multi-GPU run calls this with the same arguments plus its rank and the shared NCCL
    `unique_id` (cetkmc._lib.comm_unique_id() created on rank 0).

    packed=True: `state` is the one-byte-per-voxel form (uint8, state | defects_mask << 4) and the
    result carries `packed` instead of the int64 state / atom_type arrays — 1 B instead of 24 B per
    voxel across PCIe.

    events_per_sweep (default 0.005 L^3) and p_max (default 0.1) set the sweep interval
    tau = min(events_per_sweep / R_total, -ln(1 - p_max) / R_max).  The defaults are the validated
    envelope: level-3 parity against the serial reference (tests/test_gpu_sweep.py) is established
    for <= 0.6 % of the sites firing per sweep; larger values trade fidelity (more dropped claim
    conflicts, staler synchronous reads) for fewer sweeps.  Raises RuntimeError if the fired-site
    list overflows (events would be dropped): lower events_per_sweep.

    Returns a dict: counters of the run and, if return_fields, the rank's owned planes of
    state / atom_type / theta / phi / T.
    """
    L = state.shape[0]
    seed = constants.RANDOM_SEED if seed is None else seed
    i_begin, i_end = slab_bounds(L, world, rank)
    halo = SWEEP_HALO if world > 1 else 0
    ctx = _lib.Context(L=L, device=device, i_begin=i_begin, i_end=i_end, halo=halo)
    try:
        ctx.set_rate_params(rate_params(impurity_c, 1, 2, 3))
        own = slice(i_begin, i_end)
        if packed:
            ctx.upload_packed(state[own])
            ctx.upload(theta=theta[own], phi=phi[own], T=T[own])
        else:
            ctx.upload(state=state[own], theta=theta[own], phi=phi[own], T=T[own],
                       defects=None if defects_mask is None else defects_mask[own])
        if world > 1:
            if unique_id is None:
                raise ValueError("world > 1 needs the NCCL unique id created on rank 0")
            ctx.comm_init(unique_id, rank, world)
            ctx.halo_exchange(7)
        sp = _lib.SweepParams()
        sp.seed = int(seed)
        sp.events_per_sweep = float(events_per_sweep if events_per_sweep is not None else 0.005 * L ** 3)
        sp.p_max = float(p_max)
        sp.defect_fraction = float(defect_fraction)
        sp.thermal_every = int(thermal_every)
        tp = thermal_params(THERMAL_DT, nan_to_num=True) if thermal_every > 0 else None
        out = ctx.sweep_run(n_sweeps, sp, tp)
        if out["overflow"]:
            raise RuntimeError("run_kmc_sublattice: the fired-site list overflowed (events were dropped); "
                               "lower events_per_sweep")
        out["i_begin"], out["i_end"] = i_begin, i_end
        if return_fields and packed:
            out["packed"] = ctx.download_packed()
            out.update(ctx.download(theta=True, phi=True, T=True))
        elif return_fields:
            out.update(ctx.download(state=True, atom_type=True, theta=True, phi=True, T=True))
        return out
    finally:
        ctx.close()
