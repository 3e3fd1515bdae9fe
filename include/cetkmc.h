/*
 * cetkmc.h — C-ABI of the B200-native KMC / thermal hot path (libcetkmc.so).
 *
 * This is the drop-in boundary.  The reference is pure Python, so its "FFI" for
 * this path is the Python module surface (main.py:6, kmc_simulation.py:192-193,
 * utils.py:7).  Each entry point below names the reference interface it replaces;
 * the ctypes stubs a maintainer adds are shown in INTEGRATION.md and live in
 * cet-driven-simulation-for-3d-printing-am-kmc-approach_b200/_lib.py.
 *
 * Conventions
 *   - every function returns int: 0 = ok, non-zero = error; cet_last_error()
 *     returns a thread-local message (Python wrappers raise RuntimeError);
 *   - plain pointers and sizes only; host pointers are borrowed for the call;
 *   - reference array layouts at the boundary: state / atom_type / defects_mask
 *     are int64, theta / phi / T are float64, C-contiguous (L, L, L), k fastest
 *     (lattice_init.py:23-32);
 *   - all work of a context is ordered on one CUDA stream owned by the context;
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef CETKMC_H
#define CETKMC_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define CET_ABI_VERSION 1

typedef struct cet_ctx cet_ctx; /* opaque: one lattice (or one z-slab of it) resident in HBM */

/* Event type codes (kmc_event_rates.py:72,109,132,158: b'dep', b'diff', b'nuc', b'att'). */
enum { CET_EV_DEP = 0, CET_EV_DIFF = 1, CET_EV_NUC = 2, CET_EV_ATT = 3 };

/* Values of constants.py consumed by kmc_event_rates.py:3-7,164-173; filled from the
 * caller's `constants` module at call time so edits to constants.py keep working. */
typedef struct cet_rate_params {
    double nu, nu_dep;            /* NU, NU_DEP */
    double E_b[3], E_diff[3];     /* E_B_{W,RE,C}, E_DIFF_{W,RE,C} */
    double kT, T_melt, i0, delta_T_c;
    double k_nuc, beta_imp_nuc, max_imp_fraction;
    double rate_threshold, anisotropy, impurity_re, impurity_c;
    int32_t states_w, states_re, states_c, defect_id;
} cet_rate_params;

/* thermal_solver.py:107-117 (+ kmc_simulation.py:249 when nan_to_num != 0).
 * dt_alpha = dt*ALPHA, inv_dx2 = 1/VOXEL_SIZE**2, lo = T_SUB, hi = T_MELT*1.1 are formed
 * in Python so they carry Python's exact doubles. */
typedef struct cet_thermal_params {
    double dt_alpha, inv_dx2, lo, hi, nan_value;
    int32_t nan_to_num, pad_;
} cet_thermal_params;

/* thermal_solver.py:36-105 */
typedef struct cet_thermal_full_params {
    double dt, alpha, inv_dx2, rho_cp, latent_over_cp, lo, hi;
} cet_thermal_full_params;

/* Result block of cet_kmc_run (kmc_simulation.py:246-332). */
typedef struct cet_kmc_result {
    int64_t steps_done;        /* steps executed (a terminating step is not counted) */
    int64_t py_used;           /* draws consumed from the Python `random` stream */
    int64_t np_used;           /* draws consumed from the NumPy global stream */
    int64_t sp_used;           /* draws consumed from the species (Numba) stream */
    int64_t nucleation_count;  /* kmc_simulation.py:310 */
    int64_t fallback_last;     /* steps that took the events[-1] fallback (:273-274) */
    double total_time;         /* kmc_simulation.py:332 */
    double last_total_rate;
    int32_t terminated;        /* kmc_simulation.py:260-262 */
    int32_t starved;           /* stopped early because a draw buffer ran out: refill and call again */
} cet_kmc_result;

/* Synchronous-sublattice sweep (large-lattice path; no reference counterpart). */
typedef struct cet_sweep_params {
    uint64_t seed;             /* Philox key; draws are keyed by (seed, sweep, global site) */
    double events_per_sweep;   /* tau = events_per_sweep / R_total(previous sweep) ... */
    double p_max;              /* ... capped so that 1-exp(-R_max*tau) <= p_max */
    double defect_fraction;    /* kmc_simulation.py:323 */
    int32_t thermal_every;     /* sweeps between update_temperature_cet calls (0 = never) */
    int32_t pad_;
} cet_sweep_params;

typedef struct cet_sweep_result {
    int64_t sweeps_done;
    int64_t events_fired;      /* sites whose draw fired */
    int64_t events_applied;    /* fired events that won their claim and were applied */
    int64_t nucleation_count;
    int64_t sweep_index;       /* running sweep counter of the context after the call */
    double time;               /* sum of tau over the sweeps of this call */
    double last_total_rate, last_max_rate, last_tau;
    int32_t terminated;
    int32_t overflow;          /* the fired-event list overflowed (events dropped): lower events_per_sweep */
    int64_t sites_refreshed;   /* sites whose rates the neighbour-rate updates re-evaluated */
} cet_sweep_result;

/* Per-context arguments of cet_metrics_group. */
typedef struct cet_metrics_params {
    double theta_threshold;    /* grain misorientation threshold in rad (metrics.py:43 passes 0.5) */
    double ar_threshold;       /* n_equiaxed counts the grains with aspect ratio < ar_threshold */
    int64_t pct_pos[4];        /* positions x whose searchsorted(cum, x, side="right") pct_index returns */
    int32_t refresh;           /* != 0: redraw the defect mask first, as cet_defects_refresh(apply_to_state = 0) */
    int32_t carbon_id;         /* the refresh's arguments (1..15) ... */
    uint32_t epoch;
    int32_t pad_;
    uint64_t seed;
    double prob_base, e_mig, kT, T_default;
} cet_metrics_params;

/* What one metrics row (metrics.py:41-96) needs of a lattice, from cet_metrics_group. */
typedef struct cet_metrics_result {
    int64_t counts[16];        /* histogram of the owned states (cet_counts) */
    int64_t n_carbon;          /* the refresh's carbon sites and sites with the mask set (0 without a refresh) */
    int64_t n_defects;
    int64_t n_grains;
    int64_t size_sum;          /* voxels over all grains */
    int64_t n_equiaxed;        /* grains with aspect ratio < ar_threshold */
    int64_t pct_index[4];      /* searchsorted(cum, pct_pos[k], side="right"), cum = cumsum([n_sites - size_sum, sizes...]) */
    double ar_sum;             /* sum of the grains' aspect ratios in cluster order, in NumPy's pairwise order */
} cet_metrics_result;

/* ---- library ---- */
const char *cet_last_error(void);
int cet_abi_version(void);
int cet_device_count(int *n);
int cet_device_name(int device, char *buf, int buflen);

/* ---- context ----
 * A context holds planes [i_begin, i_end) of a global L^3 lattice plus `halo` ghost planes
 * on each side (single GPU: i_begin=0, i_end=L, halo=0).  For thermal-only use the lattice
 * may be non-cubic: cet_create_shape(n0, n1, n2). */
int cet_create(cet_ctx **ctx, int device, int64_t L, int64_t i_begin, int64_t i_end, int32_t halo);
/* Same with n0 planes along axis 0 and L x L sites per plane (n0 == L is the reference's cubic
 * lattice; n0 > L stacks slabs for weak scaling over several GPUs). */
int cet_create_slab(cet_ctx **ctx, int device, int64_t n0, int64_t L, int64_t i_begin, int64_t i_end,
                    int32_t halo);
int cet_create_shape(cet_ctx **ctx, int device, int64_t n0, int64_t n1, int64_t n2);
int cet_destroy(cet_ctx *ctx);
int cet_sync(cet_ctx *ctx);
int cet_set_rate_params(cet_ctx *ctx, const cet_rate_params *p);

/* ---- fields: host (reference layout) <-> packed device layout ----
 * Owned planes only.  NULL pointers are skipped.  state values must be 0..15 and defects
 * 0..15 (they share one byte per voxel in HBM). */
int cet_upload(cet_ctx *ctx, const int64_t *state, const double *theta, const double *phi,
               const double *T, const int64_t *defects);
int cet_download(cet_ctx *ctx, int64_t *state, int64_t *atom_type, double *theta, double *phi,
                 double *T);
int cet_upload_prev_state(cet_ctx *ctx, const int64_t *prev_state);
int cet_snapshot_state(cet_ctx *ctx); /* prev_state := state, on device */
/* Packed fast path: one byte per voxel (state | defects<<4). */
int cet_upload_packed(cet_ctx *ctx, const uint8_t *packed);
int cet_download_packed(cet_ctx *ctx, uint8_t *packed);
/* Raw device pointers for tensor hand-off (torch.distributed halo exchange, tests).
 * which: 0 packed state, 1 theta, 2 phi, 3 T, 4 site_rate, 5 orientation unit vectors (32-byte records x,y,z,pad).  Pointer addresses local plane 0
 * (ghost planes included); nbytes is the full extent. */
int cet_device_ptr(cet_ctx *ctx, int which, void **ptr, int64_t *nbytes);
int cet_counts(cet_ctx *ctx, int64_t counts[16]); /* histogram of state values, owned planes */

/* ---- thermal_solver.py ---- */
/* update_temperature_cet (thermal_solver.py:107): T <- clip(T + dt*ALPHA*laplace(T)/dx^2) in HBM. */
int cet_thermal_cet(cet_ctx *ctx, const cet_thermal_params *p);
/* update_temperature (thermal_solver.py:36): q_top[n1*n2] = I_surface/VOXEL_SIZE (host pointer). */
int cet_thermal_full(cet_ctx *ctx, const cet_thermal_full_params *p, const double *q_top);
/* update_temperature for n_ctx whole-lattice contexts of one L in one stencil launch: context q takes p[q] and the
 * host source plane q_top[q] (L*L doubles, borrowed for the call).  Each context ends exactly as
 * cet_thermal_full(ctxs[q], &p[q], q_top[q]) followed, when snapshot != 0, by cet_snapshot_state(ctxs[q]) would
 * leave it; the snapshot is written by the stencil pass itself.  A context whose sweep tile state is current also
 * gets the new temperature of its empty sites' pair operands in that pass and keeps its tile state (a solo call
 * drops it and the next sweep rebuilds it, with the same bits); a stale tile state stays stale.
 * The contexts must be distinct whole-lattice contexts (no slabs) of one cubic L on one device, each with a
 * previous state (cet_upload_prev_state / cet_snapshot_state); 1 <= n_ctx <= 64.  Everything is checked before
 * anything is copied or launched, so a rejected call leaves every context as it was.  The work is ordered on the
 * stream of ctxs[0] after the work already queued on every context's stream: one H2D copy per context, one launch,
 * one host synchronisation.  When profiling is enabled on ctxs[0], the launch is recorded there as a thermal span. */
int cet_thermal_full_group(cet_ctx *const *ctxs, int32_t n_ctx, const cet_thermal_full_params *p,
                           const double *const *q_top, int32_t snapshot);
/* build_temperature_field (thermal_solver.py:15): T[i,:,:] = t0 + g*i. */
int cet_thermal_fill_gradient(cet_ctx *ctx, double t0, double g);

/* ---- kmc_event_rates.py ---- */
/* get_event_rates (kmc_event_rates.py:162): rebuild every per-site rate total, the top-plane
 * deposition rates and the per-row / per-plane-segment sums used by the BKL search. */
int cet_rates_build(cet_ctx *ctx);
int cet_rates_total(cet_ctx *ctx, double *total, int64_t *n_dep);
int cet_rates_download(cet_ctx *ctx, double *site_rate, double *dep_rate);
/* The legacy event list in the reference's order (parity level 1 / compat).  species_draws
 * (may be NULL -> atom = W) is the stream of kmc_event_rates.py:65, one per dep event. */
int cet_events_count(cet_ctx *ctx, int64_t *n_events, int64_t *n_dep);
int cet_events_export(cet_ctx *ctx, const double *species_draws, int64_t n_draws, int64_t cap,
                      uint8_t *type, int64_t *pos, double *rate, int64_t *target, int32_t *atom,
                      int64_t *n_written);

/* ---- kmc_simulation.py:246-332: exact rejection-free BKL steps with injected draws ----
 * py_draws: u1, [u2 iff defect_fraction > 0], u3 per step; np_draws: theta, phi per dep/nuc
 * event; sp_draws: species stream (advanced by the number of dep events every step).
 * thermal_every (20 in the reference) <= 0 disables the in-loop thermal update.
 * log_* (host, may be NULL, capacity n_steps): the chosen event of every step. */
int cet_kmc_run(cet_ctx *ctx, int64_t step0, int64_t n_steps, double defect_fraction,
                const cet_thermal_params *tp, int32_t thermal_every,
                const double *py_draws, int64_t n_py, const double *np_draws, int64_t n_np,
                const double *sp_draws, int64_t n_sp, double total_time0, cet_kmc_result *res,
                uint8_t *log_type, int64_t *log_pos, int64_t *log_target, int32_t *log_atom,
                double *log_rate, double *log_total);

/* ---- synchronous-sublattice sweeps (large lattices) ----
 * A context whose clock is fresh (tau == 0) first runs one priming pass that only measures the total
 * rate, so that every counted sweep is a real one. */
int cet_sweep_run(cet_ctx *ctx, int64_t n_sweeps, const cet_sweep_params *sp,
                  const cet_thermal_params *tp, cet_sweep_result *res);
/* Advance n_ctx independent lattices by n_sweeps sweeps each, with one launch per kernel for the whole group.
 * sp, tp, res are arrays of n_ctx (tp may be NULL when no sp[q].thermal_every > 0).  Every context ends exactly
 * as cet_sweep_run(ctxs[q], n_sweeps, &sp[q], &tp[q], &res[q]) would leave it, bit for bit, whatever else is in
 * the group and in whatever order.  The contexts must be distinct whole-lattice contexts (no slabs) of one L on
 * one device, with rate params, no debug flags and no empty site carrying an orientation; 1 <= n_ctx <= 64.
 * Everything is checked before any sweep buffer is allocated or any sweep runs (the check of the last condition
 * derives each examined context's compact tile state, which no caller can read).  The work is ordered on the
 * stream of ctxs[0]; the call returns when it is done.  The thermal step, tile_pairop_T and the dense rate rebuild
 * are grouped too, except the rebuild on L that a tensor map cannot describe (L % 16 != 0 or L < 64), which runs
 * per context.  When profiling is enabled on ctxs[0], the spans of the grouped kernels are recorded there. */
int cet_sweep_run_group(cet_ctx *const *ctxs, int32_t n_ctx, int64_t n_sweeps, const cet_sweep_params *sp,
                        const cet_thermal_params *tp, cet_sweep_result *res);
int cet_sweep_reset(cet_ctx *ctx); /* zero the sweep counter, clock, tau and event counters */
/* Checkpoint / resume of the sweep clock: running sweep counter (the Philox key of the next sweep),
 * the interval tau the next sweep will use, the accumulated time. */
int cet_sweep_get_state(cet_ctx *ctx, int64_t *sweep_index, double *tau, double *time);
int cet_sweep_set_state(cet_ctx *ctx, int64_t sweep_index, double tau, double time);

/* ---- z-slab decomposition over the GPUs of one box (NCCL over NVLink) ---- */
int cet_comm_unique_id(void *id128);
int cet_comm_init(cet_ctx *ctx, const void *id128, int rank, int world);
int cet_comm_destroy(cet_ctx *ctx);
/* fields bitmask: 1 state, 2 theta+phi, 4 T */
int cet_halo_exchange(cet_ctx *ctx, int fields);
int cet_allreduce_f64(cet_ctx *ctx, double *inout_host, int n, int op /* 0 sum, 1 max */);

/* ---- defects.py:4-31 track_defects / introduce_defects on the resident lattice ----
 * Rewrites the defect mask (high nibble of the voxel byte): 0 everywhere, and on carbon sites
 * u < clip(prob_base * exp(-e_mig / (kT * T')), 0, 1) with T' = T if T > 0 else T_default.
 * draws != NULL: the q-th carbon site in C order takes draws[q] (the reference's NumPy stream,
 * defects.py:18; n_draws >= number of carbon sites, whole-lattice contexts only); draws == NULL:
 * Philox keyed by (seed, epoch, global site).  apply_to_state != 0 also turns the masked sites into
 * defect_id (defects.py:28-29).  n_carbon = draws consumed, n_defects = sites with the mask set. */
int cet_defects_refresh(cet_ctx *ctx, const double *draws, int64_t n_draws, uint64_t seed, uint32_t epoch,
                        double prob_base, double e_mig, double kT, double T_default, int32_t carbon_id,
                        int32_t defect_id, int32_t apply_to_state, int64_t *n_carbon, int64_t *n_defects);

/* ---- utils.get_clusters / metrics.compute_metrics (utils.py:28-84,104-111; metrics.py:41-96) ----
 * Grains = connected components of occupied sites (state != 0) joined by the 14-offset
 * neighbourhood with misorientation < theta_threshold.  On a slab (ghost planes current) the labels are
 * local components of the owned planes + 2 ghost planes per cut face, roots are GLOBAL site indices and
 * the statistics count owned voxels; metrics.grains_distributed joins them across slabs. */
int cet_grains_label(cet_ctx *ctx, double theta_threshold, int64_t *n_grains);
/* criterion 0: misorientation of the orientation vectors < threshold (utils.py:51-56; cet_grains_label);
 * criterion 1: |theta1 - theta2| < threshold (utils.py:49-50, get_clusters(..., orientation_phi=None)). */
int cet_grains_label_ex(cet_ctx *ctx, double theta_threshold, int criterion, int64_t *n_grains);
/* Per grain (arbitrary order; sort by root for the reference's cluster order): root = smallest
 * C-order site index (the grain's first voxel), voxel count, bounding box lo/hi [3*g + axis]. */
int cet_grains_stats(cet_ctx *ctx, int64_t cap, int32_t *root, int32_t *size, int32_t *box_lo,
                     int32_t *box_hi);
/* Label volume: root site index per occupied site, -1 for empty sites (owned planes). */
int cet_grains_download_labels(cet_ctx *ctx, int32_t *labels);

/* ---- initial lattices of a group (lattice_init.py:10-59 + defects.py:4-31, in sparse form) ----
 * One context's initial lattice: n_nuclei nuclei, each at a C-order flat site of the k = 0 plane with its voxel byte
 * (state 1..3 | defect 0..1 << 4), theta and phi; every other site is empty with theta = phi = 0; T[i, j, k] =
 * T_row[k].  Host pointers, borrowed for the call. */
typedef struct cet_init_desc {
    int64_t n_nuclei;
    const int64_t *site;
    const uint8_t *byte;
    const double *theta, *phi;
    const double *T_row;          /* L values */
} cet_init_desc;
/* Context q ends exactly as cet_upload(ctxs[q], state, theta, phi, T, defects) of the dense arrays of d[q] would
 * leave it, followed, when snapshot != 0, by cet_snapshot_state(ctxs[q]).  The contexts must be distinct
 * whole-lattice contexts (no slabs) of one cubic L on one device; 1 <= n_ctx <= 64; no two nuclei of a context share
 * a site.  Everything is checked before anything is copied or launched, so a rejected call leaves every context as it
 * was.  The work is ordered on the stream of ctxs[0] after the work already queued on every context's stream: one
 * H2D copy of a packed table for the group, one fill launch over every site of the group, one scatter launch of the
 * nuclei (none when the group has no nuclei), one host synchronisation. */
int cet_init_group(cet_ctx *const *ctxs, int32_t n_ctx, const cet_init_desc *d, int32_t snapshot);

/* ---- grouped metrics cadence (kmc_simulation.py:335-378 for many lattices at once) ----
 * The contexts must be distinct whole-lattice contexts (no slabs) of one cubic L on one device; 1 <= n_ctx <= 64.
 * The work is ordered on the stream of ctxs[0] after the work already queued on every context's stream, each
 * kernel is one launch for the whole group, and the call returns when the work is done.
 * cet_counts_group: counts[16 * q + s] = cet_counts(ctxs[q])[s]; one host synchronisation. */
int cet_counts_group(cet_ctx *const *ctxs, int32_t n_ctx, int64_t *counts);
/* Per context q: if mp[q].refresh, the defect mask is redrawn exactly as cet_defects_refresh(ctxs[q], draws[q],
 * n_draws[q], mp[q].seed, mp[q].epoch, ..., apply_to_state = 0) redraws it (draws == NULL or draws[q] == NULL: the
 * Philox stream; else n_draws[q] must cover the lattice's carbon sites); then the grains are labelled as
 * cet_grains_label_ex(ctxs[q], mp[q].theta_threshold, 0, ...) labels them, and cet_grains_stats /
 * cet_grains_download_labels report that labelling afterwards; res[q] receives the histogram, the refresh's counts
 * and the grain reductions of a metrics row.  Everything but the carbon-site count is checked before the device
 * is used; that count is checked before any mask byte is written: a rejected call leaves every context as it was.
 * Three host synchronisations per call whatever n_ctx (carbon counts, grain counts, results); no device
 * allocation once the per-context buffers have grown to the lattice's needs. */
int cet_metrics_group(cet_ctx *const *ctxs, int32_t n_ctx, const cet_metrics_params *mp, const double *const *draws,
                      const int64_t *n_draws, cet_metrics_result *res);
/* ---- per-plane grain profile of a group (where along a growth axis the grains turn equiaxed) ----
 * Per-plane profile of the last grain labelling (cet_grains_label[_ex] or cet_metrics_group) of each context, along
 * `axis` (0, 1 or 2).  out[(q * 4 + f) * L + z], int64, for context q and plane z:
 *   f = 0  Solid                    occupied sites (label >= 0) with coordinate z
 *   f = 1  EquiaxedSolid            of those, sites whose grain has aspect ratio < ar_threshold
 *   f = 2  GrainsSpanning           grains whose bounding box along `axis` contains z
 *   f = 3  EquiaxedGrainsSpanning   of those, grains with aspect ratio < ar_threshold
 * The aspect ratio is metrics.grain_aspect_ratios' (utils.py:104-111), evaluated exactly as cet_metrics_group
 * evaluates it, so a grain's class is the one its EquiaxedFraction counts.  Grains are joined through the 14-offset
 * neighbourhood, which steps +-2 along each axis, so a grain can hold sites on planes z and z + 2 and none on
 * z + 1: the spanning columns count the grains whose bounding box (what the aspect ratio measures) covers z, not
 * the grains with a site on z.
 * The contexts must be distinct whole-lattice contexts (no slabs) of one cubic L on one device, 1 <= n_ctx <= 64,
 * each with a labelling of the whole lattice (a context never labelled is rejected).  The call reports that
 * labelling as cet_grains_stats does and does not relabel; it is read-only on the lattice, the labels and the mask,
 * so the next metrics row and the next sweeps are what they would have been without it.  Everything, `out`
 * included, is checked before anything is launched or written: a rejected call leaves every context and `out` as
 * they were.  The work is ordered on the stream of ctxs[0] after the work already queued on every context's
 * stream: one memset, five launches for the whole group, one D2H copy of the table, one host synchronisation. */
int cet_grain_profile_group(cet_ctx *const *ctxs, int32_t n_ctx, int32_t axis, double ar_threshold, int64_t *out);
/* The same for global planes [i_lo, i_hi) within the labelled planes of a slab (owned + 2 ghost planes per
 * cut face): what two neighbouring slabs compare to join the grains that cross their cut. */
int cet_grains_download_planes(cet_ctx *ctx, int64_t i_lo, int64_t i_hi, int32_t *labels);

/* Test hook: number of sites whose cached neighbour-state word differs from a fresh gather
 * (-1 when the cache is declared stale). */
int cet_debug_nst_mismatches(cet_ctx *ctx, int64_t *n_bad);
/* Test / profiling hook: which kernels keep the rate sums current in cet_sweep_run (all variants give
 * the same bits).  Default: stamped sites are refreshed by the class-sorted list kernel on the compact tile
 * state (class codes + pair operands; rates_refresh.cu); the dense rebuild after a thermal step runs the
 * class-sorted tile kernel staged by 3-D TMA boxes (rates_dense.cu) when L % 16 == 0 and L >= 64, the dense
 * gather kernel on the compact state otherwise.
 * 262144: refresh by the pair-compacting list kernel (rates.cu); 131072: the dense tile kernel walks its sites by
 * class only, without the sort by pair count; 65536: dense rebuilds by the compact gather kernel;
 * 2: the gather refresh + dense kernel of the first design (neighbour-class cache + unit vectors);
 * 32: the shared-memory tile kernel of sweep_tile.cu for the refresh and the rebuild; 1: that kernel staged by
 * scalar loads, 16: by 16-byte vector loads; 4: it walks the 14 neighbour slots per lane instead of compacting
 * the pairs across the warp; 8: dense rebuilds by the first design's gather kernel;
 * 64 / 128: timing probes of the apply kernel (stamps / field writes skipped: results invalid);
 * bits 8-15: stamped sites per warp and queue entry of the pair-compacting refresh, in units of 32 (0 = default 64). */
int cet_debug_flags(cet_ctx *ctx, int flags);

/* ---- per-kernel device timing: CUDA event pairs recorded on the context stream around every
 * launch of a kind while enabled.  kind: 0 sweep stream (fire decision), 1 sweep apply,
 * 2 thermal stencil, 3 dense rate kernel, 4 halo exchange, 5 whole sweep, 6 sweep pick,
 * 7 neighbour-rate refresh, 8 totals all-reduce, 9 ghost-zone cache + rate rebuild after the exchange. */
int cet_profile_enable(cet_ctx *ctx, int on);
int cet_profile_read(cet_ctx *ctx, int kind, double *ms_total, int64_t *launches, int reset);

/* ---- timing helper: elapsed ms of the last N kernels of a kind (CUDA events on the ctx stream) */
int cet_timer_begin(cet_ctx *ctx);
int cet_timer_end_ms(cet_ctx *ctx, float *ms);

#ifdef __cplusplus
}
#endif
#endif /* CETKMC_H */
