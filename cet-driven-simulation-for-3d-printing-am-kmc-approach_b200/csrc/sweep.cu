// sweep.cu — synchronous-sublattice KMC sweeps for large lattices (no reference counterpart:
// the reference executes ONE event per O(L^3) rate rebuild, kmc_simulation.py:246-332).
//
// The per-site rate sums stay resident in HBM (site_rate, dep_rate — the same arrays the exact
// BKL path uses) and are kept current by neighbour-rate updates, so one sweep is
//   stream  (dense, HBM-bound, 8 B/site): every site reads its rate sum R, draws one uniform and
//           fires with p = 1-exp(-R*tau); fired sites go to a compact list; per-plane totals of R
//           are accumulated in a fixed order for the next time increment.  Draws come from a
//           counter-based Philox4x32-10 keyed by (seed, sweep, GLOBAL site), so a site's decision
//           does not depend on which GPU evaluates it;
//   pick    (sparse): a fired site re-enumerates its <= 15 events (site_events, the same code
//           that produced R) and picks one with probability rate/R, then claims the sites the
//           event writes (itself; a diffusion event also its target);
//   apply   (sparse): conflicts are resolved by sublattice order — the 5x5x5 checkerboard colour
//           of the source site, rotated every sweep, is the claim priority.  Two sites of one
//           colour differ by multiples of 5 per axis, while two events can only collide when
//           their sources differ by a neighbour offset or a difference of two offsets (every
//           coordinate <= 4), so a colour never conflicts with itself and the outcome is
//           deterministic.  Winners are applied exactly as kmc_simulation.py:280-327 and mark the
//           sites whose rates they invalidate (the changed sites and their 14 neighbours);
//   refresh : the dense row pass of rates.cu restricted to the marked sites (coalesced, same
//           arithmetic, so the resident rates stay bit-identical to a full rebuild);
//   tau     for the next sweep from the totals of this one:
//           tau = min(events_per_sweep / R_total, -ln(1-p_max) / R_max).
// A thermal step (every thermal_every sweeps) is followed by a refresh of the rates that read a
// changed temperature (thermal_refresh) or, when those are many, by a dense rebuild.
// Slabs: a context with halo H >= 6 evaluates ghost sites to depth 4 and resolves claims to
// depth 2, which is everything that can write an owned site; after the one halo exchange per
// sweep (comm.cu) the rates of the evaluated ghost planes and of the two outermost owned planes
// are rebuilt densely (6 planes per cut face).  Plane sums are combined in a fixed order so the trajectory is independent of the
// number of slabs.
#include <algorithm>
#include <memory>
#include "ctx.cuh"
#include "rate_tile.cuh"
#include "reduce.cuh"
#include "philox.cuh"
#include "tile_state.cuh"

namespace cet {

int thermal_cet_step(cet_ctx *c, const cet_thermal_params *p, const int32_t *stop_flag);
int thermal_cet_step_tracked(cet_ctx *c, const cet_thermal_params *p, const int32_t *stop_flag, uint32_t *changed,
                             unsigned int *n_changed);
int rates_rows(cet_ctx *c, int p_lo, int p_hi);                                  // rates.cu
int rates_rows_dirty(cet_ctx *c, int p_lo, int p_hi, const uint32_t *stamp, int32_t *list, unsigned int *counter);
int comm_sweep_reduce(cet_ctx *c, double *plane_sum, int n, double *max_inout);   // comm.cu
int comm_halo_exchange(cet_ctx *c, int fields);
int comm_delta_alloc(cet_ctx *c);
int comm_delta_exchange(cet_ctx *c);
// sweep_tile.cu — the fused tile kernel (refresh + stream) and the arrays it stages
int tile_state_ensure(cet_ctx *c);
int tile_state_build(cet_ctx *c, int p_lo, int p_hi);
int tile_pairop_T_update(cet_ctx *c);
int tile_pass(cet_ctx *c, int p_lo, int p_hi, bool all);
bool tile_tma_ok(const cet_ctx *c);
int stamp_fill(cet_ctx *c, int p_lo, int p_hi);
int rates_rows_dirty_compact(cet_ctx *c, int p_lo, int p_hi, const uint32_t *stamp, int32_t *list, unsigned int *counter);
int rates_rows_compact(cet_ctx *c, int p_lo, int p_hi);
int comm_sweep_reduce_join(cet_ctx *c);                                           // comm.cu
int rates_rows_dense(cet_ctx *c, int p_lo, int p_hi);                            // rates_dense.cu
int rate_tables_ensure(cet_ctx *c);
int rates_rows_dirty_compact_group(cet_ctx *const *cs, int n, int p_lo, int p_hi, int *refresh_blocks);  // rates.cu
int rates_rows_dense_group(cet_ctx *const *cs, int n, int *blocks_per_sm);          // rates_dense.cu
unsigned int *dense_queue(cet_ctx *c);
int thermal_cet_step_group(cet_ctx *const *cs, const cet_thermal_params *const *tps, int n);   // thermal.cu
int tile_pairop_T_update_group(cet_ctx *const *cs, int n);                          // sweep_tile.cu

struct Record {          // one fired event
    int32_t src;         // local linear index of the source site
    int32_t info;        // type | (slot+1) << 4 | atom << 12 | colour rank << 20   (-1: no event)
    double theta, phi;   // orientation the written site receives (att: neighbour's; dep/nuc: drawn)
};

__device__ __forceinline__ int colour_rank(int i, int j, int k, uint32_t sweep)
{
    const int c = ((i % 5) * 5 + (j % 5)) * 5 + (k % 5);
    return (int)((c + 37u * sweep) % 125u);     // rotate the sublattice order every sweep
}
__device__ __forceinline__ unsigned long long claim_key(int rank, long long gsite)
{
    return ((unsigned long long)(125 - rank) << 48) | (unsigned long long)(gsite + 1);
}

// ---- stream: one fire test per site against the resident rate sum --------------------------------
// HBM-bound by design: 8 B/site.  A thread owns 8 sites of a 2048-site tile of one plane (four
// coalesced 16-byte loads) and one Philox4x32-10 block (128 bits) = one 16-bit digit per site, the
// leading digit of the site's uniform in base 65536: with x = R*tau and p = 1-exp(-x) <= x the site
// can only fire if digit <= floor(65536 x), which rejects all but ~p of the sites after three fp64
// instructions; the survivors evaluate p exactly and, when digit == floor(65536 p), draw the
// remaining digits from a second Philox block.  P(fire) = floor(65536 p)/65536 + P(u' < frac)/65536 = p.
// Fired sites are staged in 2 KB of shared memory and appended with one list reservation per CTA;
// 6 CTAs per SM stay resident (96 KB of loads in flight per SM).
constexpr int ST_THREADS = 256, ST_PER_THREAD = 8, ST_TILE = ST_THREADS * ST_PER_THREAD, ST_STAGE = 512, ST_CAND = 512;

struct StreamArgs {
    const double *site_rate, *dep_rate;   // dep_rate: plane of the global top (NaN = no event)
    SweepState *ss;
    int32_t *fired;
    unsigned int cap_fired;
    double *blk_sum, *blk_max;
    int p_lo;                // first evaluated local plane
    int top_plane;           // local index of the global top plane, or -1
    int plane_sites;         // L*L
    int tiles_per_plane;
    int i_off;
    uint64_t seed;
    uint32_t sweep;
};

// The rare exact test of a site that survived the digit pre-filter (kept out of line: it holds an
// expm1 and a second Philox block, and inlining it costs the streaming loop its occupancy).
__device__ __noinline__ bool stream_fire_exact(double x, double d, uint64_t seed, uint64_t gsite, uint32_t sweep)
{
    const double p16 = -expm1(-x) * 65536.0;
    const double f = floor(p16);
    if (d != f) return d < f;
    double u_rest, unused;                              // leading digit ties: the rest of the uniform decides
    philox_u2(seed, gsite, sweep, STREAM_FIRE_REST, &u_rest, &unused);
    return u_rest < p16 - f;
}

// a fired site: staged per CTA, or appended to the global list directly once the staging area is full
__device__ __forceinline__ void stream_append(const StreamArgs &a, int *s_list, unsigned int *s_cnt, int32_t site)
{
    const unsigned int q = atomicAdd(s_cnt, 1u);
    if (q < ST_STAGE) { s_list[q] = site; return; }
    const unsigned int g = atomicAdd(&a.ss->n_fired, 1u);
    if (g < a.cap_fired) a.fired[g] = site;
    else a.ss->overflow = 1;
}

// The kernel bodies below take their arguments by reference: the solo kernels pass their own parameter, the
// grouped kernels (cet_sweep_run_group) the table entry of their lattice, so both run the same instructions.
__device__ __forceinline__ void sweep_stream_body(const StreamArgs &a)
{
    __shared__ double s_sum[ST_THREADS / 32], s_max[ST_THREADS / 32];
    __shared__ int s_list[ST_STAGE];
    __shared__ double c_R[ST_CAND];                 // staged survivors of the digit pre-filter: rate sum ...
    __shared__ uint32_t c_sd[ST_CAND];              // ... site within the tile << 16 | leading digit
    __shared__ unsigned int s_cnt, s_base, s_ncand;
    if (threadIdx.x == 0) { s_cnt = 0; s_ncand = 0; }
    __syncthreads();
    const int pl = blockIdx.y, tile = blockIdx.x;                   // grid: (tiles per plane, evaluated planes)
    const int blk = pl * a.tiles_per_plane + tile;
    const int p = a.p_lo + pl;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const double tau = a.ss->terminated ? 0.0 : a.ss->tau;
    const int64_t base = (int64_t)p * a.plane_sites;
    // site e of this thread: pairs interleaved across the warp so that every load is a coalesced
    // 512-byte warp access: q(e) = tile*ST_TILE + w*256 + (e/2)*64 + lane*2 + (e&1)
    const int qw = tile * ST_TILE + w * (32 * ST_PER_THREAD) + lane * 2;
    double R[ST_PER_THREAD];
    const bool vec = (a.plane_sites & 1) == 0;                       // every plane then starts 16-byte aligned
#pragma unroll
    for (int m = 0; m < ST_PER_THREAD / 2; ++m) {
        const int q = qw + m * 64;
        if (vec && q + 1 < a.plane_sites) {
            const double2 v = __ldcs(reinterpret_cast<const double2 *>(a.site_rate + base + q));
            R[2 * m] = v.x; R[2 * m + 1] = v.y;
        } else {
            R[2 * m] = q < a.plane_sites ? a.site_rate[base + q] : 0.0;
            R[2 * m + 1] = q + 1 < a.plane_sites ? a.site_rate[base + q + 1] : 0.0;
        }
    }
    if (p == a.top_plane) {
#pragma unroll
        for (int e = 0; e < ST_PER_THREAD; ++e) {
            const int q = qw + (e >> 1) * 64 + (e & 1);
            if (q < a.plane_sites) {
                const double d = a.dep_rate[q];
                if (d == d) R[e] = d + R[e];
            }
        }
    }
    double rsum = 0.0, rmax = 0.0;
#pragma unroll
    for (int e = 0; e < ST_PER_THREAD; ++e) { rsum += R[e]; rmax = fmax(rmax, R[e]); }
    if (tau > 0.0 && rmax > 0.0) {
        const uint32_t tid_in_plane = (uint32_t)(tile * ST_THREADS + threadIdx.x);
        const u32x4 r = philox4x32_10(u32x4{tid_in_plane, (uint32_t)(a.i_off + p), a.sweep, (uint32_t)STREAM_FIRE},
                                      (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
        const uint32_t words[4] = {r.x, r.y, r.z, r.w};
        const double tau16 = tau * 65536.0;
        // pre-filter: else digit > floor(65536 x) >= floor(65536 p): cannot fire
        unsigned cand = 0;
#pragma unroll
        for (int e = 0; e < ST_PER_THREAD; ++e) {
            const uint32_t digit = (words[e >> 1] >> (16 * (e & 1))) & 0xFFFFu;
            const double d = __hiloint2double(0x43300000, (int)digit) - 4503599627370496.0;   // (double)digit
            if (d <= R[e] * tau16) cand |= 1u << e;
        }
        // the survivors (~0.5 % of the sites, about one per warp) are staged for the CTA: evaluated where they
        // arise, each exact test (an expm1, ~140 instructions) would run with one lane of its warp
        while (cand) {
            const int e = __ffs(cand) - 1;
            cand &= cand - 1;
            double Re = R[0];
            uint32_t wd = words[0];
#pragma unroll
            for (int q = 1; q < ST_PER_THREAD; ++q) if (e == q) Re = R[q];
#pragma unroll
            for (int q = 1; q < 4; ++q) if ((e >> 1) == q) wd = words[q];
            const uint32_t digit = (wd >> (16 * (e & 1))) & 0xFFFFu;
            const uint32_t st = (uint32_t)(qw - tile * ST_TILE + (e >> 1) * 64 + (e & 1));      // site within the tile
            const unsigned int pos = atomicAdd(&s_ncand, 1u);
            if (pos < ST_CAND) {
                c_R[pos] = Re; c_sd[pos] = st << 16 | digit;
            } else {                                            // staging full (only at high firing probabilities): test it here
                const double d = __hiloint2double(0x43300000, (int)digit) - 4503599627370496.0;
                const uint64_t gsite = (uint64_t)(a.i_off + p) * (uint64_t)a.plane_sites + (uint64_t)(tile * ST_TILE) + st;
                if (stream_fire_exact(Re * tau, d, a.seed, gsite, a.sweep)) stream_append(a, s_list, &s_cnt, (int32_t)(base + tile * ST_TILE + (int)st));
            }
        }
    }
    rsum = warp_sum(rsum);
    rmax = warp_max_nonneg(rmax);                 // rate sums are >= +0 and never NaN (keep_rate)
    if (lane == 0) { s_sum[w] = rsum; s_max[w] = rmax; }
    __syncthreads();
    // exact tests of the staged survivors, one per thread; fired sites are staged per CTA (one global list
    // reservation per CTA: a reservation per warp would put ~4e5 atomics per sweep on one address); a CTA with
    // more than ST_STAGE of them appends the rest directly
    const unsigned int ncand = min(s_ncand, (unsigned)ST_CAND);
    for (unsigned int q = threadIdx.x; q < ncand; q += ST_THREADS) {
        const double Re = c_R[q];
        const uint32_t sd = c_sd[q], st = sd >> 16;
        const double d = __hiloint2double(0x43300000, (int)(sd & 0xFFFFu)) - 4503599627370496.0;   // (double)digit
        const uint64_t gsite = (uint64_t)(a.i_off + p) * (uint64_t)a.plane_sites + (uint64_t)(tile * ST_TILE) + st;
        if (stream_fire_exact(Re * tau, d, a.seed, gsite, a.sweep)) stream_append(a, s_list, &s_cnt, (int32_t)(base + tile * ST_TILE + (int)st));
    }
    if (threadIdx.x == ST_THREADS - 1) {          // the tile's totals, meanwhile
        double t = 0.0, m = 0.0;
        for (int q = 0; q < ST_THREADS / 32; ++q) { t += s_sum[q]; m = fmax(m, s_max[q]); }
        a.blk_sum[blk] = t;
        a.blk_max[blk] = m;
    }
    if (ncand == 0 && s_ncand == 0) return;       // nothing could fire in this tile (uniform: s_ncand is final after the barrier)
    __syncthreads();
    const unsigned int n_staged = min(s_cnt, (unsigned)ST_STAGE);
    if (n_staged == 0) return;
    if (threadIdx.x == 0) s_base = atomicAdd(&a.ss->n_fired, n_staged);
    __syncthreads();
    for (unsigned int q = threadIdx.x; q < n_staged; q += ST_THREADS) {
        if (s_base + q < a.cap_fired) a.fired[s_base + q] = s_list[q];
        else a.ss->overflow = 1;
    }
}
__global__ void __launch_bounds__(ST_THREADS, 6) sweep_stream_kernel(const __grid_constant__ StreamArgs a) { sweep_stream_body(a); }
template <int CAP>
__global__ void __launch_bounds__(ST_THREADS, 6) sweep_stream_group_kernel(const __grid_constant__ GroupArgs<StreamArgs, CAP> g)
{
    sweep_stream_body(g.a[blockIdx.z]);
}

// ---- pick: choose the event of every fired site, record it and claim its write set --------------
struct PickArgs {
    Lat g;
    const double *theta, *phi, *site_rate, *dep_rate;
    cet_rate_params P;
    SweepState *ss;
    const int32_t *fired;
    unsigned int cap_fired;
    Record *records;
    unsigned long long *claim;
    uint64_t seed;
    uint32_t sweep;
    // compact tile state (NULL: enumerate with site_events from vox / v / T)
    const uint8_t *cvox;
    const double *pairop, *tab;
};

// The events of site s in the reference's list order from the compact tile state — the arithmetic of
// the refresh kernels (tile_site_prep / tile_pair_rate), so the rates add up to the resident sum bit for
// bit.  All 14 class codes and then all pair operands are requested before any is used: two memory
// round trips per site instead of one per neighbour.  emit(type, slot, rate, atom) as site_events.
template <class F>
__device__ __forceinline__ void site_events_compact(const PickArgs &a, int s, int i, int j, int k, F &&emit)
{
    const int L = a.g.L;
    const unsigned inb = inbounds_mask(i, j, k, a.g.n0, L);
    const unsigned c = a.cvox[s];
    unsigned b[14];
#pragma unroll
    for (int o = 0; o < 14; ++o)
        b[o] = (inb >> o & 1u) ? (unsigned)a.cvox[s + (CET_NB_DI(o) * L + CET_NB_DJ(o)) * L + CET_NB_DK(o)] & 15u : 0u;
    const unsigned code = c & 15u;
    double T_self = 1.0, T_m = 1.0, T_p = 1.0;
    if (code == TC_EMPTY) {
        T_self = a.pairop[s];
        T_m = k > 0 ? a.g.T[s - 1] : T_self;
        T_p = k < L - 1 ? a.g.T[s + 1] : T_self;
    } else {
        T_self = a.g.T[s];
    }
    uint64_t w = 0;
#pragma unroll
    for (int o = 0; o < 14; ++o) w |= (uint64_t)b[o] << (4 * o);
    const TilePrep q = tile_site_prep(a.P, a.tab, w, c, T_self, T_m, T_p);
    double op[14];
#pragma unroll
    for (int o = 0; o < 14; ++o)
        op[o] = (q.pm >> (4 * o) & 1u) ? a.pairop[s + (CET_NB_DI(o) * L + CET_NB_DJ(o)) * L + CET_NB_DK(o)] : 0.0;
    if (q.sum0 != 0.0) emit((int)CET_EV_NUC, -1, q.sum0, a.P.states_w);
    const int self_state = a.g.vox[s] & 0x0F;
#pragma unroll
    for (int o = 0; o < 14; ++o) {
        if (!(q.pm >> (4 * o) & 1u)) continue;
        const double rate = tile_pair_rate(a.P, a.tab, q.is_emp, q.A, q.B, op[o]);
        if (rate == 0.0) continue;
        if (q.is_emp) emit((int)CET_EV_ATT, o, rate, b[o] == TC_W ? a.P.states_w : b[o] == TC_RE ? a.P.states_re : a.P.states_c);
        else emit((int)CET_EV_DIFF, o, rate, self_state);
    }
}

__device__ __forceinline__ void sweep_pick_body(const PickArgs &a)
{
    const unsigned int n = min(a.ss->n_fired, a.cap_fired);
    const int L = a.g.L;
    const int64_t LL = (int64_t)L * L;
    for (unsigned int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const int s = a.fired[q];
        const int p = (int)(s / LL), j = (int)((s / L) % L), k = s % L;
        const int i = a.g.i_off + p;
        const long long gsite = (long long)i * LL + (long long)j * L + k;
        double R = a.site_rate[s], dep = 0.0;
        bool has_dep = false;
        if (i == a.g.n0 - 1) {
            dep = a.dep_rate[(int64_t)j * L + k];
            has_dep = dep == dep;
            if (has_dep) R = dep + R;
        }
        double u_pick, unused;
        philox_u2(a.seed, (uint64_t)gsite, a.sweep, STREAM_PICK, &u_pick, &unused);
        // pick one event with probability rate / R (list order: dep, then the site's events)
        const double x = u_pick * R;
        double cum = 0.0;
        int ety = -1, eslot = -1, eatom = 0;
        bool found = false;
        if (has_dep) {
            cum = dep; ety = CET_EV_DEP; eatom = a.P.states_w;
            if (cum >= x) found = true;
        }
        auto take = [&](int ty, int slot, double rate, int atom) {
            if (found) return;
            cum += rate; ety = ty; eslot = slot; eatom = atom;
            if (cum >= x) found = true;
        };
        if (!found) {
            if (a.cvox) site_events_compact(a, s, i, j, k, take);
            else site_events(a.g, a.P, i, j, k, take);
        }
        Record rec;
        rec.src = s;
        rec.theta = 0.0; rec.phi = 0.0;
        rec.info = -1;
        if (ety >= 0) {
            int64_t tgt = -1;
            if (ety == CET_EV_DEP || ety == CET_EV_NUC) {
                double ut, up;
                philox_u2(a.seed, (uint64_t)gsite, a.sweep, STREAM_ANGLES, &ut, &up);
                rec.theta = __dmul_rn(3.141592653589793, ut);          // np.random.uniform(0, pi)
                rec.phi = __dmul_rn(2 * 3.141592653589793, up);        // np.random.uniform(0, 2pi)
                if (ety == CET_EV_DEP) {                               // kmc_event_rates.py:65-71
                    double us;
                    philox_u2(a.seed, (uint64_t)gsite, a.sweep, STREAM_SPECIES, &us, &unused);
                    eatom = dep_species(a.P, us);
                }
            } else {
                tgt = a.g.nb(s, eslot);
                if (ety == CET_EV_ATT) { rec.theta = a.theta[tgt]; rec.phi = a.phi[tgt]; }
                else { rec.theta = a.theta[s]; rec.phi = a.phi[s]; }
            }
            const int rank = colour_rank(i, j, k, a.sweep);
            rec.info = ety | ((eslot + 1) << 4) | (eatom << 12) | (rank << 20);
            const unsigned long long key = claim_key(rank, gsite);
            atomicMax(&a.claim[s], key);
            if (ety == CET_EV_DIFF) atomicMax(&a.claim[tgt], key);
        }
        a.records[q] = rec;
    }
}
__global__ void __launch_bounds__(128) sweep_pick_kernel(const __grid_constant__ PickArgs a) { sweep_pick_body(a); }
template <int CAP>
__global__ void __launch_bounds__(128) sweep_pick_group_kernel(const __grid_constant__ GroupArgs<PickArgs, CAP> g)
{
    sweep_pick_body(g.a[blockIdx.z]);
}

// One warp per evaluated plane: fixed-order sum of the plane's tile partials.  plane_sum is
// indexed by GLOBAL plane so that every slab count produces the same numbers.
__device__ __forceinline__ void sweep_plane_reduce_body(const double *blk_sum, const double *blk_max, int blks_per_plane,
                                                        int n_planes, int first_global, int own_lo, int own_hi,
                                                        double *plane_sum, double *max_out)
{
    const int pl = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pl >= n_planes) return;
    const int lane = threadIdx.x & 31;
    const int gi = first_global + pl;
    double s = 0.0, m = 0.0;
    for (int q = lane; q < blks_per_plane; q += 32) {
        s += blk_sum[(int64_t)pl * blks_per_plane + q];
        m = fmax(m, blk_max[(int64_t)pl * blks_per_plane + q]);
    }
    s = warp_sum(s);
    m = warp_max(m);
    if (lane == 0 && gi >= own_lo && gi < own_hi) {   // ghost planes are another slab's to report
        plane_sum[gi] = s;
        atomicMax((unsigned long long *)max_out, (unsigned long long)__double_as_longlong(m));   // m >= 0
    }
}
__global__ void sweep_plane_reduce_kernel(const double *blk_sum, const double *blk_max, int blks_per_plane,
                                          int n_planes, int first_global, int own_lo, int own_hi,
                                          double *plane_sum, double *max_out)
{
    sweep_plane_reduce_body(blk_sum, blk_max, blks_per_plane, n_planes, first_global, own_lo, own_hi, plane_sum, max_out);
}

// What differs between the lattices of a group in the small kernels (reset, plane reduce, finalize).
struct CloseArgs {
    SweepState *ss;
    const double *blk_sum, *blk_max;
    double *plane_sum;         // [n0] holds the running max
    uint32_t *stamp;
    unsigned int *refresh_queue, *dense_queue;
    double events_per_sweep, p_max;
};

// Single CTA: total in fixed plane order, tau for the next sweep, time bookkeeping.
__device__ __forceinline__ void sweep_finalize_body(SweepState *ss, const double *plane_sum, int L, const double *max_in,
                                                    double events_per_sweep, double p_max)
{
    __shared__ double sm[40];
    const double total = block_sum(plane_sum, L, sm);
    if (threadIdx.x == 0 && !ss->terminated) {
        const double rmax = *max_in;
        ss->time += ss->tau;                       // the sweep that just ran advanced time by its tau
        ss->n_refreshed_total += (unsigned long long)ss->n_dirty + ss->n_dirty_emp;
        ss->sum_rate = total; ss->max_rate = rmax;
        if (total < 1e-25 || !finite_f64(total)) { // kmc_simulation.py:260-262
            ss->terminated = 1; ss->tau = 0.0;
        } else {
            double tau = events_per_sweep / total;
            const double cap = -log1p(-p_max) / rmax;
            if (cap < tau) tau = cap;
            ss->tau = tau;
        }
    }
}
__global__ void sweep_finalize_kernel(SweepState *ss, const double *plane_sum, int L, const double *max_in,
                                      double events_per_sweep, double p_max)
{
    sweep_finalize_body(ss, plane_sum, L, max_in, events_per_sweep, p_max);
}

// Grouped small kernels.  reset: the stamp bitmap, the plane sums, the list counters and the refresh queue of
// every lattice (what sweep_once clears with two memsets, sweep_reset_kernel and rates_refresh_list's memset), and
// the dense rebuild's queue for the next sweep's rebuild (rates_rows_dense clears it before its launch);
// grid (CTAs per lattice, lattices).
template <int CAP>
__global__ void __launch_bounds__(256) sweep_reset_group_kernel(const __grid_constant__ GroupArgs<CloseArgs, CAP> g, int stamp_words, int n0)
{
    const CloseArgs &a = g.a[blockIdx.y];
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < stamp_words; q += gridDim.x * blockDim.x) a.stamp[q] = 0u;
    if (blockIdx.x == 0) {
        for (int q = threadIdx.x; q <= n0; q += blockDim.x) a.plane_sum[q] = 0.0;
        if (threadIdx.x == 0) { a.ss->n_fired = 0; a.ss->n_dirty = 0; a.ss->n_dirty_emp = 0; *a.refresh_queue = 0u; *a.dense_queue = 0u; }
    }
}
// grid (plane blocks, lattices); single-slab lattices: every evaluated plane is owned
template <int CAP>
__global__ void sweep_plane_reduce_group_kernel(const __grid_constant__ GroupArgs<CloseArgs, CAP> g, int blks_per_plane, int n_planes)
{
    const CloseArgs &a = g.a[blockIdx.y];
    sweep_plane_reduce_body(a.blk_sum, a.blk_max, blks_per_plane, n_planes, 0, 0, n_planes, a.plane_sum, a.plane_sum + n_planes);
}
// one CTA per lattice
template <int CAP>
__global__ void sweep_finalize_group_kernel(const __grid_constant__ GroupArgs<CloseArgs, CAP> g, int L)
{
    const CloseArgs &a = g.a[blockIdx.x];
    sweep_finalize_body(a.ss, a.plane_sum, L, a.plane_sum + L, a.events_per_sweep, a.p_max);
}

// ---- apply ---------------------------------------------------------------------------------------
struct ApplyArgs {
    uint8_t *vox;
    double *theta, *phi;
    Vec4 *v;
    SweepState *ss;
    const Record *records;
    unsigned int cap_fired;
    unsigned long long *claim;
    uint32_t *stamp;       // refresh requests, one bit per local site
    unsigned long long *nst;
    cet_rate_params P;
    int L, n0, i_off, np;
    int c_lo, c_hi;        // local planes with complete claims
    int own_lo, own_hi;    // local planes owned by this slab (for the counters)
    uint64_t seed;
    uint32_t sweep;
    double defect_fraction;
    // tile state of sweep_tile.cu, kept in step with the lattice (NULL: the gather kernels run instead)
    uint8_t *cvox;
    double *pairop;
    const double *T;
    uint64_t tlut;
    // delta halo exchange: owned sites changed within DELTA_ZONE planes of a cut face are appended to the
    // face's send buffer (NULL: no neighbour on that side)
    unsigned char *delta_lo, *delta_hi;
    unsigned int delta_cap;
    int probe;             // timing probes (cet_debug_flags 64 / 128): 1 = skip the stamps, 2 = skip the field writes — results invalid
};

// the owner of `site` tells the neighbouring slab(s) what the site holds now
__device__ __forceinline__ void delta_emit(const ApplyArgs &a, int site, uint8_t vox, double theta, double phi)
{
    const int LL = a.L * a.L;
    const int p = site / LL;
    if (p < a.own_lo || p >= a.own_hi) return;
#pragma unroll
    for (int face = 0; face < 2; ++face) {
        unsigned char *buf = face == 0 ? a.delta_lo : a.delta_hi;
        const int z0 = face == 0 ? a.own_lo : a.own_hi - DELTA_ZONE;
        if (!buf || p < z0 || p >= z0 + DELTA_ZONE) continue;
        const unsigned int q = atomicAdd(reinterpret_cast<unsigned int *>(buf), 1u);
        if (q >= a.delta_cap) { a.ss->overflow = 1; continue; }
        DeltaEntry e;
        e.theta = theta; e.phi = phi;
        e.zidx = site - z0 * LL; e.vox = vox;
        reinterpret_cast<DeltaEntry *>(buf + DELTA_HEADER)[q] = e;
    }
}

// cvox / pairop of a site whose voxel byte is now `vox` (orientation z component z, temperature T)
__device__ __forceinline__ void tile_put(const ApplyArgs &a, int site, uint8_t vox, double z, double T)
{
    if (!a.cvox) return;
    const unsigned code = (unsigned)(a.tlut >> (4 * (vox & 0x0F))) & 15u;
    a.cvox[site] = (uint8_t)((vox & 0xF0) | code);
    a.pairop[site] = code == TC_EMPTY ? T : tile_pairop(a.P, code, 0.0, z);
}
// one site's new content: lattice, orientation vector, tile state
__device__ __forceinline__ void site_write(const ApplyArgs &a, int site, uint8_t vox, double theta, double phi, const Vec4 &uv, double T)
{
    if (a.probe & 2) return;
    a.vox[site] = vox;
    a.theta[site] = theta; a.phi[site] = phi;
    a.v[site] = uv;
    tile_put(a, site, vox, uv.z, T);
}

// A site changed state: request a refresh of the site and of its neighbours.  The refresh pass
// (rates.cu) re-evaluates every site whose stamp bit is set and rewrites its cached neighbour-class
// word from a fresh gather — exactly the sites whose neighbourhood changed.  The stamps are a
// bitmap (16.8 MB at 512^3: the ~1e7 scattered requests of a sweep are atomic ORs that meet in L2,
// where one-byte stamps cost a 32-byte DRAM sector fill each).
// (Maintaining the words here with one 64-bit atomic add per neighbour was measured: it removes the
// gather from the refresh, -0.13 ms, but costs the apply kernel +0.52 ms per sweep at 6.6e5 events.)
__device__ __forceinline__ void site_changed(const ApplyArgs &a, int site, int, int)
{
    if (a.probe & 1) return;
    const int LL = a.L * a.L;
    const int p = site / LL, j = (site / a.L) % a.L, k = site % a.L;
    atomicOr(&a.stamp[site >> 5], 1u << (site & 31));
    const unsigned inb = inbounds_mask(a.i_off + p, j, k, a.n0, a.L);    // inside the GLOBAL lattice ...
#pragma unroll
    for (int o = 0; o < 14; ++o) {                                       // unrolled: the offsets are immediates
        const int pn = p + CET_NB_DI(o);
        if (!(inb >> o & 1u) || pn < 0 || pn >= a.np) continue;          // ... and inside the local planes
        const int n = site + (CET_NB_DI(o) * a.L + CET_NB_DJ(o)) * a.L + CET_NB_DK(o);
        atomicOr(&a.stamp[n >> 5], 1u << (n & 31));
    }
}

__device__ __forceinline__ void sweep_apply_body(const ApplyArgs &a)
{
    const unsigned int n = min(a.ss->n_fired, a.cap_fired);
    const int LL = a.L * a.L;
    int fired = 0, applied = 0, nuc = 0;
    for (unsigned int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const Record rec = a.records[q];
        if (rec.info < 0) continue;
        const int ety = rec.info & 15, eslot = ((rec.info >> 4) & 255) - 1, eatom = (rec.info >> 12) & 255;
        const int rank = rec.info >> 20;
        const int s = rec.src;
        const int p = s / LL, j = (s / a.L) % a.L, k = s % a.L;
        const long long gsite = (long long)(a.i_off + p) * LL + (long long)j * a.L + k;
        const unsigned long long key = claim_key(rank, gsite);
        int tgt = -1, pt = p;
        if (ety == CET_EV_DIFF || ety == CET_EV_ATT) {
            tgt = s + (c_nb_off[eslot][0] * a.L + c_nb_off[eslot][1]) * a.L + c_nb_off[eslot][2];
            if (ety == CET_EV_DIFF) pt = p + c_nb_off[eslot][0];
        }
        const bool owned = p >= a.own_lo && p < a.own_hi;
        if (owned) ++fired;
        const bool complete = p >= a.c_lo && p < a.c_hi && pt >= a.c_lo && pt < a.c_hi;
        // Everything the event reads — both claims, both voxel bytes, the source's temperature — is requested
        // here in one batch; the write phase below works from registers (the kernel is a latency chain per
        // event: every dependent global read costs a DRAM round trip under ~1e6 scattered accesses).
        const bool two = ety == CET_EV_DIFF;
        const unsigned long long cs = a.claim[s];
        const unsigned long long ct = two ? a.claim[tgt] : key;
        const uint8_t vox_s = a.vox[s];
        const uint8_t vox_t = two ? a.vox[tgt] : (uint8_t)0;
        const double T_s = (two && a.cvox) ? a.T[s] : 0.0;              // a vacated site's pair operand is its temperature
        const bool win = complete && cs == key && ct == key;
        if (win) {
            const int src_state = vox_s & 0x0F;                         // before the event
            Vec4 uv = unit_vec4(rec.theta, rec.phi);                    // same bits as the source's resident vector
            const Vec4 none = Vec4{0.0, 0.0, 1.0, 0.0};
            double th = rec.theta, ph = rec.phi;
            // the site that receives the atom: the target of a diffusion event, the source otherwise
            const int upd = two ? tgt : s;
            uint8_t vox_u = two ? (uint8_t)((vox_t & 0xF0) | src_state) : (uint8_t)((vox_s & 0xF0) | eatom);
            int upd_state = two ? src_state : eatom;
            if (ety == CET_EV_NUC && owned) ++nuc;
            if (a.defect_fraction > 0.0) {                               // :323-327
                double u2, unused;
                philox_u2(a.seed, (uint64_t)gsite, a.sweep, STREAM_DEFECT, &u2, &unused);
                if (u2 < a.defect_fraction) {
                    vox_u = (uint8_t)((vox_u & 0xF0) | a.P.defect_id);
                    th = 0.0; ph = 0.0; uv = none;
                    upd_state = a.P.defect_id;
                }
            }
            site_write(a, upd, vox_u, th, ph, uv, 0.0);                  // dep / nuc / att / diff target (:280-317)
            if (two) site_write(a, s, (uint8_t)(vox_s & 0xF0), 0.0, 0.0, none, T_s);     // :299-301
            if (owned) ++applied;
            if (two) {
                site_changed(a, s, src_state, 0);
                site_changed(a, tgt, 0, upd_state);
                delta_emit(a, s, (uint8_t)(vox_s & 0xF0), 0.0, 0.0);
                delta_emit(a, tgt, vox_u, th, ph);
            } else {
                site_changed(a, s, 0, upd_state);
                delta_emit(a, s, vox_u, th, ph);
            }
        }
        // release the claims this event holds (only the top claimant of a site clears it)
        if (cs == key) a.claim[s] = 0ull;
        if (ety == CET_EV_DIFF && ct == key) a.claim[tgt] = 0ull;
    }
    // one set of atomics per CTA
    __shared__ int cta_cnt[3];
    if (threadIdx.x < 3) cta_cnt[threadIdx.x] = 0;
    __syncthreads();
    fired = warp_sum_i(fired); applied = warp_sum_i(applied); nuc = warp_sum_i(nuc);
    if ((threadIdx.x & 31) == 0) {
        if (fired) atomicAdd(&cta_cnt[0], fired);
        if (applied) atomicAdd(&cta_cnt[1], applied);
        if (nuc) atomicAdd(&cta_cnt[2], nuc);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (cta_cnt[0]) atomicAdd(&a.ss->n_fired_total, (unsigned long long)cta_cnt[0]);
        if (cta_cnt[1]) atomicAdd(&a.ss->n_applied, (unsigned long long)cta_cnt[1]);
        if (cta_cnt[2]) atomicAdd(&a.ss->n_nuc, (unsigned long long)cta_cnt[2]);
    }
}
__global__ void __launch_bounds__(128) sweep_apply_kernel(const __grid_constant__ ApplyArgs a) { sweep_apply_body(a); }
template <int CAP>
__global__ void __launch_bounds__(128) sweep_apply_group_kernel(const __grid_constant__ GroupArgs<ApplyArgs, CAP> g)
{
    sweep_apply_body(g.a[blockIdx.z]);
}

// Receiver side of the delta exchange: the neighbour's changed sites are written into the ghost planes
// [g0, g0 + DELTA_ZONE) — lattice, orientation vector, tile state — and stamped (with their neighbours)
// for the refresh pass.
__global__ void __launch_bounds__(128) delta_scatter_kernel(const __grid_constant__ ApplyArgs a, const unsigned char *buf, int g0)
{
    const unsigned int n = min(*reinterpret_cast<const unsigned int *>(buf), a.delta_cap);
    const DeltaEntry *ent = reinterpret_cast<const DeltaEntry *>(buf + DELTA_HEADER);
    const int LL = a.L * a.L;
    for (unsigned int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const DeltaEntry e = ent[q];
        const int site = g0 * LL + e.zidx;
        const int old_state = a.vox[site] & 0x0F, new_state = (int)(e.vox & 0x0Fu);
        site_write(a, site, (uint8_t)e.vox, e.theta, e.phi, unit_vec4(e.theta, e.phi), a.T[site]);
        site_changed(a, site, old_state, new_state);
    }
}

__global__ void sweep_reset_kernel(SweepState *ss, double *max_slot)
{
    ss->n_fired = 0; ss->n_dirty = 0; ss->n_dirty_emp = 0;
    *max_slot = 0.0;
}

static int sweep_alloc(cet_ctx *c)
{
    if (!c->sweep) {
        CET_CUDA(cudaMalloc(&c->sweep, sizeof(SweepState)));
        CET_CUDA(cudaMemsetAsync(c->sweep, 0, sizeof(SweepState), c->stream));
    }
    if (!c->claim) {
        CET_CUDA(cudaMalloc(&c->claim, (size_t)c->nloc * sizeof(unsigned long long)));
        CET_CUDA(cudaMemsetAsync(c->claim, 0, (size_t)c->nloc * sizeof(unsigned long long), c->stream));
    }
    if (!c->stamp) {
        CET_CUDA(cudaMalloc(&c->stamp, (size_t)c->nloc / 8 + 64));
        CET_CUDA(cudaMemsetAsync(c->stamp, 0, (size_t)c->nloc / 8 + 64, c->stream));
    }
    if (!c->dirty) {
        c->cap_dirty = (size_t)c->nloc;               // occupied list + empty list, one entry per site each
        CET_CUDA(cudaMalloc(&c->dirty, 2 * c->cap_dirty * sizeof(int32_t)));
    }
    if (!c->fired) {
        c->cap_fired = (size_t)c->nloc / 8 + 4096;
        CET_CUDA(cudaMalloc(&c->fired, c->cap_fired * sizeof(int32_t)));
        CET_CUDA(cudaMalloc(&c->records, c->cap_fired * sizeof(Record)));
        c->cap_records = c->cap_fired;
    }
    const int tpp = (int)((c->plane + ST_TILE - 1) / ST_TILE);
    if (!c->blk_sum) {
        c->n_blk = (int64_t)tpp * c->np;
        CET_CUDA(cudaMalloc(&c->blk_sum, (size_t)c->n_blk * sizeof(double)));
        CET_CUDA(cudaMalloc(&c->blk_max, (size_t)c->n_blk * sizeof(double)));
        CET_CUDA(cudaMalloc(&c->plane_sum, (size_t)(c->n0 + 2) * sizeof(double)));
    }
    return 0;
}

// Local plane ranges of a slab (see the header comment).
struct SlabRanges { int eval_lo, eval_hi, claim_lo, claim_hi, own_lo, own_hi; };
static SlabRanges slab_ranges(const cet_ctx *c)
{
    SlabRanges r;
    const int i_off = (int)(c->i_begin - c->halo), np = (int)c->np;
    const int dom_lo = i_off < 0 ? -i_off : 0;                         // first local plane inside the domain
    const int dom_hi = (i_off + np > c->n0) ? (int)(c->n0 - i_off) : np;
    const bool cut_lo = i_off > 0, cut_hi = i_off + np < c->n0;        // slab face with missing neighbours beyond
    r.eval_lo = cut_lo ? 2 : dom_lo;  r.eval_hi = cut_hi ? np - 2 : dom_hi;
    r.claim_lo = cut_lo ? 4 : dom_lo; r.claim_hi = cut_hi ? np - 4 : dom_hi;
    r.own_lo = c->halo; r.own_hi = np - c->halo;
    return r;
}

}  // namespace cet

using namespace cet;

extern "C" int cet_sweep_reset(cet_ctx *c)
{
    CET_REQUIRE(c, "cet_sweep_reset: NULL ctx");
    cet::DeviceGuard dg(c->device);
    if (c->sweep) CET_CUDA(cudaMemsetAsync(c->sweep, 0, sizeof(SweepState), c->stream));
    c->sweep_index = 0;
    c->last_thermal_index = -1;
    c->T_finite = false;          // a terminated run skips its stencil passes: re-check T next time
    return 0;
}

// Checkpoint / resume of the sweep clock: the running sweep counter (the Philox key of the next
// sweep), the interval tau the next sweep will use and the accumulated time.  With the lattice
// restored and these three values set, a resumed run continues bit for bit (the resident rates are
// rebuilt densely, which equals the refreshed rates bit for bit).
extern "C" int cet_sweep_get_state(cet_ctx *c, int64_t *sweep_index, double *tau, double *time)
{
    CET_REQUIRE(c, "cet_sweep_get_state: NULL ctx");
    cet::DeviceGuard dg(c->device);
    SweepState h;
    memset(&h, 0, sizeof(h));
    if (c->sweep) {
        CET_CUDA(cudaMemcpyAsync(&h, c->sweep, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
        CET_CUDA(cudaStreamSynchronize(c->stream));
    }
    if (sweep_index) *sweep_index = c->sweep_index;
    if (tau) *tau = h.tau;
    if (time) *time = h.time;
    return 0;
}

extern "C" int cet_sweep_set_state(cet_ctx *c, int64_t sweep_index, double tau, double time)
{
    CET_REQUIRE(c && sweep_index >= 0, "cet_sweep_set_state: bad argument");
    cet::DeviceGuard dg(c->device);
    if (int rc = sweep_alloc(c)) return rc;
    SweepState h;
    CET_CUDA(cudaMemcpyAsync(&h, c->sweep, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    h.tau = tau; h.time = time; h.terminated = 0;
    CET_CUDA(cudaMemcpyAsync(c->sweep, &h, sizeof(h), cudaMemcpyHostToDevice, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    c->sweep_index = sweep_index;
    c->last_thermal_index = -1;
    c->sweep_rates_valid = false;
    return 0;
}

namespace cet {

// Refresh of the stamped sites on the compact tile state: list-driven gathers from cvox / pairop, or
// (debug flag 32) the shared-memory tile kernel, which wins when a sweep stamps a large part of the lattice.
static int refresh_tiled(cet_ctx *c, const SlabRanges &R)
{
    if (c->debug_flags & 32) return tile_pass(c, R.eval_lo, R.eval_hi, false);
    return rates_rows_dirty_compact(c, R.eval_lo, R.eval_hi, c->stamp, c->dirty, &c->sweep->n_dirty);
}

// ---- after a thermal step: refresh only the rates whose temperatures changed -------------------------
// A site's rates read T at the site itself, at its k +- 1 neighbours (grad_z of an empty site) and at its empty
// neighbours among the 14 (the diffusion / attachment pair operand is then pairop = T).  The offsets are symmetric,
// so a changed site x makes stale x, x +- 1 and x +- 2 in k, x + (0, +-1, +-1) and x + (+-1, +-1, 0), x + (+-2, 0, 0)
// and x + (0, +-2, 0).  One thread per stamp word: the OR of the changed bitmap's words at those row offsets, shifted
// by dk within the row (rows start on word boundaries: L % 32 == 0; rows outside the lattice contribute nothing).
// Every word of the stamp bitmap is written; the stale sites are counted.
__device__ __forceinline__ uint32_t kshift1(uint32_t w, uint32_t l, uint32_t r) { return (w >> 1 | r << 31) | (w << 1 | l >> 31); }
__device__ __forceinline__ uint32_t kshift2(uint32_t w, uint32_t l, uint32_t r) { return (w >> 2 | r << 30) | (w << 2 | l >> 30); }

__global__ void __launch_bounds__(256) thermal_stale_kernel(const uint32_t *__restrict__ chg, uint32_t *__restrict__ stamp, int L,
                                                            int n0, int n_words, unsigned int *n_stale)
{
    const int wpr = L >> 5;                                       // words per row
    unsigned cnt = 0;
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += gridDim.x * blockDim.x) {
        const int r = w / wpr, kw = w - r * wpr;                  // row (plane * L + j), word within the row
        const int p = r / L, j = r - p * L;
        auto at = [&](int dp, int dj, int dw) -> uint32_t {
            const int pp = p + dp, jj = j + dj, ww = kw + dw;
            if (pp < 0 || pp >= n0 || jj < 0 || jj >= L || ww < 0 || ww >= wpr) return 0u;
            return chg[((int64_t)pp * L + jj) * wpr + ww];
        };
        const uint32_t c = at(0, 0, 0);
        uint32_t s = c | kshift1(c, at(0, 0, -1), at(0, 0, 1)) | kshift2(c, at(0, 0, -1), at(0, 0, 1));
#pragma unroll
        for (int dj = -1; dj <= 1; dj += 2) s |= kshift1(at(0, dj, 0), at(0, dj, -1), at(0, dj, 1));
        s |= at(1, 1, 0) | at(1, -1, 0) | at(-1, 1, 0) | at(-1, -1, 0) | at(2, 0, 0) | at(-2, 0, 0) | at(0, 2, 0) | at(0, -2, 0);
        stamp[w] = s;
        cnt += __popc(s);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);                   // one counter update per warp
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(n_stale, cnt);
}

// Above this many stale sites the dense rebuild is the faster side.  Measured at 512^3 on a B200 (1000 W, 1965 MHz;
// scripts/bench_thermal_refresh.py, profiles/thermal_refresh.json): the sweep holding the thermal step took 1.02 /
// 1.21 / 1.49 / 2.06 / 2.63 ms on the refresh side at 1.6 / 5 / 10 / 20 / 30 % of the sites stale, about 5.8 ms
// per unit of stale fraction, against 3.07-3.19 ms on the dense side, so the two meet near 40 %.  Both sides give
// the same bits: the choice only costs time.
static int64_t thermal_refresh_max(const cet_ctx *c) { return c->nloc / 8 * 3; }

// The rates after a thermal step of the solo tiled path: the stencil has kept pairop (ThermalTrack); when the rates
// were valid before it and L % 32 == 0 it has also marked its changed sites, and only the rates that read a changed
// temperature are refreshed.  One host read of the counts per thermal step.  *done: the rates are current.
static int thermal_refresh(cet_ctx *c, const SlabRanges &R, bool *done)
{
    *done = false;
    ProfScope ps(c, PROF_REFRESH);
    const int n_words = (int)(c->nloc >> 5);
    thermal_stale_kernel<<<(int)std::min<int64_t>((n_words + 255) / 256, (int64_t)sm_count(c) * 8), 256, 0, c->stream>>>(
        c->t_changed, c->stamp, (int)c->n1, (int)c->n0, n_words, &c->sweep->n_t_stale);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(c->t_count_host, &c->sweep->n_t_changed, 2 * sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    if (c->t_count_host[0] == 0) { *done = true; return 0; }      // no temperature changed: every rate still holds
    if ((int64_t)c->t_count_host[1] > thermal_refresh_max(c)) return 0;
    CET_CUDA(cudaMemsetAsync(&c->sweep->n_dirty, 0, sizeof(unsigned int), c->stream));   // sweep_reset_kernel clears it again
    if (int rc = rates_rows_dirty_compact(c, R.eval_lo, R.eval_hi, c->stamp, c->dirty, &c->sweep->n_dirty)) return rc;
    *done = true;
    return 0;
}

// One sweep.  tiled: the rate sums are kept current by the TMA tile kernel (sweep_tile.cu), which needs
// the orientation invariant of tile_state.cuh; otherwise by the gather kernels of the first design
// (stamp scan + list-driven re-evaluation, rates.cu).  Stream, pick and apply are the same either
// way, so both variants run the same trajectory bit for bit.
// count == false is the priming pass of a fresh clock: tau is still 0, nothing can fire, and the pass
// only measures the totals that give the first real sweep its interval.
// The start of a sweep: the thermal step when one is due, and the dense rebuild when the resident rates are stale.
static int sweep_prepare(cet_ctx *c, const cet_sweep_params *sp, const cet_thermal_params *tp, const SlabRanges &R, bool tiled)
{
    if (sp->thermal_every > 0 && c->sweep_index % sp->thermal_every == 0 && c->last_thermal_index != c->sweep_index) {
        // solo tiled path: the stencil keeps pairop itself (ThermalTrack); slabs run tile_pairop_T after the exchange
        const bool solo = tiled && c->world == 1 && c->halo == 0 && c->tile_valid;
        // the incremental refresh needs rates that were current before the stencil, the bitmap (L % 32 == 0), and the
        // default rebuild (debug flags 8 / 32 / 65536 / 131072 select another rebuild kernel; 524288 forces the dense side)
        const bool incremental = solo && c->sweep_rates_valid && c->t_changed && c->t_count_host &&
                                 !(c->debug_flags & (8 | 32 | 65536 | 131072 | 524288));
        if (solo) {
            if (incremental) CET_CUDA(cudaMemsetAsync(&c->sweep->n_t_changed, 0, 2 * sizeof(unsigned int), c->stream));
            if (int rc = thermal_cet_step_tracked(c, tp, &c->sweep->terminated, incremental ? c->t_changed : nullptr,
                                                  &c->sweep->n_t_changed)) return rc;    // clears sweep_rates_valid
        } else {
            if (int rc = thermal_cet_step(c, tp, &c->sweep->terminated)) return rc;      // clears sweep_rates_valid
            if (c->world > 1) if (int rc = comm_halo_exchange(c, 4)) return rc;
            if (tiled) if (int rc = tile_pairop_T_update(c)) return rc;
        }
        c->last_thermal_index = c->sweep_index;
        if (incremental) {
            bool done = false;
            if (int rc = thermal_refresh(c, R, &done)) return rc;
            c->sweep_rates_valid = done;
        }
    }
    if (!c->sweep_rates_valid) {                     // new lattice, new T or new parameters: dense rebuild
        if (tiled && !(c->debug_flags & 8)) {
            ProfScope ps(c, PROF_RATES);
            // dense rebuild: the class-sorted TMA tile kernel (rates_dense.cu) where the rows allow TMA; the dense
            // gather kernel on the compact state serves every other L (flag 65536 forces it), and flag 32 runs the
            // refresh's tile kernel over every site instead (the three agree bit for bit)
            const bool tma = tile_tma_ok(c) && !(c->debug_flags & 65536);
            if (c->debug_flags & 32) { if (int rc = tile_pass(c, R.eval_lo, R.eval_hi, true)) return rc; }
            else if (tma) { if (int rc = rates_rows_dense(c, R.eval_lo, R.eval_hi)) return rc; }
            else if (int rc = rates_rows_compact(c, R.eval_lo, R.eval_hi)) return rc;
        } else {
            if (tiled) c->nst_valid = false;         // nobody maintains the neighbour cache on the tile path
            if (int rc = nst_ensure(c)) return rc;
            if (int rc = rates_rows(c, R.eval_lo, R.eval_hi)) return rc;
        }
        c->sweep_rates_valid = true;
    }
    return 0;
}

// Kernel arguments of one sweep of context c.
static StreamArgs stream_args(const cet_ctx *c, const cet_sweep_params *sp, const SlabRanges &R)
{
    const int i_off = (int)(c->i_begin - c->halo);
    const int top_plane = (int)(c->n0 - 1 - i_off);
    StreamArgs a;
    a.site_rate = c->site_rate; a.dep_rate = c->dep_rate; a.ss = c->sweep;
    a.fired = c->fired; a.cap_fired = (unsigned int)c->cap_fired;
    a.blk_sum = c->blk_sum; a.blk_max = c->blk_max;
    a.p_lo = R.eval_lo;
    a.top_plane = (top_plane >= R.eval_lo && top_plane < R.eval_hi) ? top_plane : -1;
    a.plane_sites = (int)c->plane; a.tiles_per_plane = (int)((c->plane + ST_TILE - 1) / ST_TILE); a.i_off = i_off;
    a.seed = sp->seed; a.sweep = (uint32_t)c->sweep_index;
    return a;
}
static PickArgs pick_args(const cet_ctx *c, const cet_sweep_params *sp, bool tiled)
{
    PickArgs a;
    a.g = c->lat(); a.theta = c->theta; a.phi = c->phi; a.site_rate = c->site_rate; a.dep_rate = c->dep_rate;
    a.P = c->rp; a.ss = c->sweep; a.fired = c->fired; a.cap_fired = (unsigned int)c->cap_fired;
    a.records = (Record *)c->records; a.claim = c->claim;
    a.seed = sp->seed; a.sweep = (uint32_t)c->sweep_index;
    a.cvox = tiled ? c->cvox : nullptr; a.pairop = c->pairop; a.tab = c->rate_tab;
    return a;
}
static ApplyArgs apply_args_of(const cet_ctx *c, const cet_sweep_params *sp, const SlabRanges &R, bool tiled, bool count)
{
    ApplyArgs b;
    b.vox = c->vox; b.theta = c->theta; b.phi = c->phi; b.v = c->v;
    b.ss = c->sweep; b.records = (const Record *)c->records; b.cap_fired = (unsigned int)c->cap_fired;
    b.claim = c->claim; b.stamp = c->stamp; b.nst = (unsigned long long *)c->nst;
    b.P = c->rp; b.L = (int)c->n1; b.n0 = (int)c->n0; b.i_off = (int)(c->i_begin - c->halo); b.np = (int)c->np;
    b.c_lo = R.claim_lo; b.c_hi = R.claim_hi; b.own_lo = R.own_lo; b.own_hi = R.own_hi;
    b.seed = sp->seed; b.sweep = (uint32_t)c->sweep_index;
    b.defect_fraction = sp->defect_fraction;
    b.cvox = tiled ? c->cvox : nullptr; b.pairop = c->pairop; b.T = c->T; b.tlut = tile_code_lut(c->rp);
    const bool deltas = tiled && c->world > 1 && count;
    b.delta_lo = (deltas && c->rank > 0) ? (unsigned char *)c->delta_send[0] : nullptr;
    b.delta_hi = (deltas && c->rank < c->world - 1) ? (unsigned char *)c->delta_send[1] : nullptr;
    b.delta_cap = (unsigned int)c->delta_cap;
    b.probe = (c->debug_flags >> 6) & 3;
    return b;
}

static int sweep_once(cet_ctx *c, const cet_sweep_params *sp, const cet_thermal_params *tp, const SlabRanges &R, bool tiled,
                      bool count)
{
    const int n_eval = R.eval_hi - R.eval_lo;
    const int i_off = (int)(c->i_begin - c->halo);
    const int tpp = (int)((c->plane + ST_TILE - 1) / ST_TILE);
    double *max_slot = c->plane_sum + c->n0;      // plane_sum[n0] holds the running max
    ProfScope step_scope(c, PROF_STEP);
    if (int rc = sweep_prepare(c, sp, tp, R, tiled)) return rc;
    CET_CUDA(cudaMemsetAsync(c->stamp, 0, (size_t)c->nloc / 8 + 8, c->stream));      // stamp bitmap of this sweep
    sweep_reset_kernel<<<1, 1, 0, c->stream>>>(c->sweep, max_slot);
    CET_CUDA(cudaMemsetAsync(c->plane_sum, 0, (size_t)c->n0 * sizeof(double), c->stream));
    {
        const StreamArgs a = stream_args(c, sp, R);
        ProfScope ps(c, PROF_DECIDE);
        sweep_stream_kernel<<<dim3((unsigned)tpp, (unsigned)n_eval), ST_THREADS, 0, c->stream>>>(a);
    }
    CET_CUDA(cudaGetLastError());
    sweep_plane_reduce_kernel<<<(n_eval + 3) / 4, 128, 0, c->stream>>>(
        c->blk_sum, c->blk_max, tpp, n_eval, i_off + R.eval_lo, (int)c->i_begin, (int)c->i_end,
        c->plane_sum, max_slot);
    CET_CUDA(cudaGetLastError());
    // the totals are only needed for the next tau (sweep_finalize_kernel, last kernel of the sweep): the reduction
    // over the slabs starts here — on a side stream when the context has a second communicator — and is joined there
    if (c->world > 1) if (int rc = comm_sweep_reduce(c, c->plane_sum, (int)c->n0, max_slot)) return rc;
    const int sparse_grid = sm_count(c) * 32;
    ApplyArgs apply_args;
    {
        const PickArgs a = pick_args(c, sp, tiled);
        ProfScope ps(c, PROF_PICK);
        sweep_pick_kernel<<<sparse_grid, 128, 0, c->stream>>>(a);
    }
    CET_CUDA(cudaGetLastError());
    {
        const ApplyArgs b = apply_args_of(c, sp, R, tiled, count);
        if (b.delta_lo) CET_CUDA(cudaMemsetAsync(b.delta_lo, 0, DELTA_HEADER, c->stream));
        if (b.delta_hi) CET_CUDA(cudaMemsetAsync(b.delta_hi, 0, DELTA_HEADER, c->stream));
        apply_args = b;
        ProfScope ps(c, PROF_APPLY);
        sweep_apply_kernel<<<sparse_grid, 128, 0, c->stream>>>(b);
    }
    CET_CUDA(cudaGetLastError());
    if (!tiled) {
        ProfScope ps(c, PROF_REFRESH);
        if (int rc = rates_rows_dirty(c, R.eval_lo, R.eval_hi, c->stamp, c->dirty, &c->sweep->n_dirty)) return rc;
    } else if (c->world == 1) {
        ProfScope ps(c, PROF_REFRESH);
        if (int rc = refresh_tiled(c, R)) return rc;
    }
    if (c->world > 1 && count) {
        if (tiled) {
            // Delta exchange: every slab sends the owned sites it changed within DELTA_ZONE planes of a cut
            // face (one fixed-capacity message per neighbour, ~24 B per site) and writes what it receives
            // into its ghost planes, stamping those sites and their neighbours; the one refresh pass of the
            // sweep then covers the slab's own events and the ghost updates alike.  Ghost planes 4-5 were
            // already updated by the locally resolved events with the owner's outcome (same inputs, same
            // deterministic claims), planes 0-3 only by the deltas.
            {
                ProfScope ps(c, PROF_HALO);
                if (int rc = comm_delta_exchange(c)) return rc;
            }
            {
                ProfScope pb(c, PROF_BOUNDARY);
                ApplyArgs d = apply_args;
                d.delta_lo = d.delta_hi = nullptr;
                if (c->rank > 0)
                    delta_scatter_kernel<<<sm_count(c) * 4, 128, 0, c->stream>>>(d, (const unsigned char *)c->delta_recv[0], 0);
                if (c->rank < c->world - 1)
                    delta_scatter_kernel<<<sm_count(c) * 4, 128, 0, c->stream>>>(d, (const unsigned char *)c->delta_recv[1],
                                                                                 (int)c->np - DELTA_ZONE);
                CET_CUDA(cudaGetLastError());
            }
            ProfScope ps(c, PROF_REFRESH);
            if (int rc = refresh_tiled(c, R)) return rc;
        } else {
            {
                ProfScope ps(c, PROF_HALO);
                if (int rc = comm_halo_exchange(c, 1 | 2)) return rc;
            }
            // The ghost planes now hold the owners' lattice.  Events this slab could not resolve
            // (write set reaching beyond ghost depth 2) may have changed ghost planes that the two
            // outermost owned planes read, so the evaluated ghost planes and those two owned planes on
            // each cut face are rebuilt densely.
            ProfScope pb(c, PROF_BOUNDARY);
            c->nst_valid = true;       // the exchange marked the whole cache stale; only the planes rebuilt below are
            if (R.own_lo > R.eval_lo) {
                if (int rc = nst_build(c, R.eval_lo, R.own_lo + 2)) return rc;
                if (int rc = rates_rows(c, R.eval_lo, R.own_lo + 2)) return rc;
            }
            if (R.eval_hi > R.own_hi) {
                if (int rc = nst_build(c, R.own_hi - 2, R.eval_hi)) return rc;
                if (int rc = rates_rows(c, R.own_hi - 2, R.eval_hi)) return rc;
            }
        }
    }
    if (c->world > 1) {
        ProfScope ps(c, PROF_ALLREDUCE);          // what the main stream still waits for the reduction
        if (int rc = comm_sweep_reduce_join(c)) return rc;
    }
    sweep_finalize_kernel<<<1, 256, 0, c->stream>>>(c->sweep, c->plane_sum, (int)c->n0, max_slot,
                                                    sp->events_per_sweep, sp->p_max);
    CET_CUDA(cudaGetLastError());
    if (count) c->sweep_index++;
    return 0;
}

// The result block of a call from the sweep state before and after it.
static int sweep_finish(cet_ctx *c, const SweepState &before, const SweepState &after, int64_t n_sweeps, cet_sweep_result *res)
{
    if (after.dirty_overflow) {      // refresh list overflowed: the resident rates are stale
        c->sweep_rates_valid = false;
        CET_CUDA(cudaMemsetAsync(&c->sweep->dirty_overflow, 0, sizeof(unsigned int), c->stream));
    }
    res->sweeps_done = n_sweeps;
    res->events_fired = (int64_t)(after.n_fired_total - before.n_fired_total);
    res->events_applied = (int64_t)(after.n_applied - before.n_applied);
    res->nucleation_count = (int64_t)(after.n_nuc - before.n_nuc);
    res->sweep_index = c->sweep_index;
    res->time = after.time - before.time;
    res->last_total_rate = after.sum_rate; res->last_max_rate = after.max_rate; res->last_tau = after.tau;
    res->sites_refreshed = (int64_t)(after.n_refreshed_total - before.n_refreshed_total);
    res->terminated = after.terminated;
    res->overflow = (int32_t)(after.overflow | (after.dirty_overflow << 1));
    return 0;
}

}  // namespace cet

extern "C" int cet_sweep_run(cet_ctx *c, int64_t n_sweeps, const cet_sweep_params *sp,
                             const cet_thermal_params *tp, cet_sweep_result *res)
{
    CET_REQUIRE(c && sp && res, "cet_sweep_run: NULL argument");
    CET_REQUIRE(c->cubic && c->have_rp, "cet_sweep_run: needs a cubic context with rate params");
    CET_REQUIRE(sp->p_max > 0.0 && sp->p_max < 1.0 && sp->events_per_sweep > 0.0,
                "cet_sweep_run: need 0 < p_max < 1 and events_per_sweep > 0");
    CET_REQUIRE(sp->thermal_every <= 0 || tp != nullptr, "cet_sweep_run: thermal_every needs thermal params");
    CET_REQUIRE(c->world == 1 || c->halo >= 6, "cet_sweep_run: slabs need halo >= 6");
    CET_REQUIRE(c->world > 1 || (c->i_begin == 0 && c->i_end == c->n0),
                "cet_sweep_run: a partial slab needs cet_comm_init");
    CET_REQUIRE(c->nloc < (1ll << 31), "cet_sweep_run: the local lattice must have fewer than 2^31 sites");
    cet::DeviceGuard dg(c->device);
    if (int rc = sweep_alloc(c)) return rc;
    const SlabRanges R = slab_ranges(c);

    SweepState before;
    CET_CUDA(cudaMemcpyAsync(&before, c->sweep, sizeof(before), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));

    // Which refresh: the TMA tile kernel when no empty site carries an orientation (the reference's
    // invariant, checked here on the device), the gather kernels otherwise.  A change of variant
    // drops the state only the other one maintains.
    bool tiled = !(c->debug_flags & 2);
    if (tiled) {
        if (int rc = tile_state_ensure(c)) return rc;
        tiled = c->emp_canonical;
    }
    if (c->world > 1) {                      // every slab must take the same path
        double f = tiled ? 0.0 : 1.0;
        if (int rc = cet_allreduce_f64(c, &f, 1, 1)) return rc;
        tiled = f == 0.0;
    }
    if (tiled) {
        if (int rc = rate_tables_ensure(c)) return rc;      // the pick kernel reads the K_eff / E_tot tables
        c->nst_valid = false;                // the tile path keeps no neighbour cache
        if (c->world > 1) if (int rc = comm_delta_alloc(c)) return rc;
        // the changed-site bitmap and the count buffer of the thermal refresh (sweep_prepare), outside the sweep loop
        if (c->world == 1 && c->halo == 0 && c->n1 % 32 == 0 && sp->thermal_every > 0 && n_sweeps > 0) {
            if (!c->t_changed) CET_CUDA(cudaMalloc(&c->t_changed, (size_t)c->nloc / 8));
            if (!c->t_count_host) CET_CUDA(cudaMallocHost(&c->t_count_host, 2 * sizeof(unsigned int)));
        }
    } else {
        c->tile_valid = false;               // the gather path's apply does not maintain cvox / pairop
        if (int rc = nst_ensure(c)) return rc;
    }
    if (n_sweeps > 0 && before.tau == 0.0 && !before.terminated)
        if (int rc = sweep_once(c, sp, tp, R, tiled, false)) return rc;
    for (int64_t n = 0; n < n_sweeps; ++n)
        if (int rc = sweep_once(c, sp, tp, R, tiled, true)) return rc;
    c->rates_valid = false;          // the BKL sum hierarchy is not maintained by the sweeps
    SweepState after;
    CET_CUDA(cudaMemcpyAsync(&after, c->sweep, sizeof(after), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return sweep_finish(c, before, after, n_sweeps, res);
}

// ---- grouped sweeps -------------------------------------------------------------------------------
// A group of independent whole-lattice contexts of one L advances with one launch per kernel for all of them.
// Per sweep: the thermal stencil and tile_pairop_T of the contexts whose step is due, the dense rebuild of the
// contexts whose rates are stale, then reset, stream, plane reduce, pick, apply, dirty scan, refresh and finalize,
// each one grouped launch whose CTAs find their lattice's arguments in the launch's table (the stencil: one launch
// per variant in use, with and without the nan_to_num pass).  On L that a tensor map cannot describe (tile_tma_ok)
// the dense rebuild is the compact gather kernel, issued per context.  Every lattice runs the solo kernel bodies
// on its own data, so it ends bit for bit where cet_sweep_run would leave it.
namespace cet {

struct GroupMember {
    cet_ctx *c;
    const cet_sweep_params *sp;
    const cet_thermal_params *tp;
};

template <int CAP>
struct GroupTables {
    GroupArgs<CloseArgs, CAP> close;
    GroupArgs<StreamArgs, CAP> stream;
    GroupArgs<PickArgs, CAP> pick;
    GroupArgs<ApplyArgs, CAP> apply;
};
static_assert(group_fits<StreamArgs>() && group_fits<PickArgs>() && group_fits<ApplyArgs>() && group_fits<CloseArgs>(),
              "a table of GROUP_MAX entries must fit the kernel parameter space");

// occupancy of the persistent grouped kernels, queried on their first launch in a call
struct GroupBlocks {
    int refresh = 0, dense = 0;
};

// sweep_prepare for a group: the due thermal steps, then the rebuild of every context whose rates are stale
static int sweep_group_prepare(const std::vector<GroupMember> &m, const SlabRanges &R, GroupBlocks &blocks)
{
    std::vector<cet_ctx *> due, stale;
    std::vector<const cet_thermal_params *> due_tp;
    for (const GroupMember &g : m) {
        cet_ctx *c = g.c;
        if (g.sp->thermal_every > 0 && c->sweep_index % g.sp->thermal_every == 0 && c->last_thermal_index != c->sweep_index) {
            due.push_back(c);
            due_tp.push_back(g.tp);
        }
    }
    if (!due.empty()) {
        if (int rc = thermal_cet_step_group(due.data(), due_tp.data(), (int)due.size())) return rc;   // clears sweep_rates_valid
        if (int rc = tile_pairop_T_update_group(due.data(), (int)due.size())) return rc;
        for (cet_ctx *c : due) c->last_thermal_index = c->sweep_index;
    }
    for (const GroupMember &g : m)
        if (!g.c->sweep_rates_valid) stale.push_back(g.c);
    if (stale.empty()) return 0;
    {
        ProfScope ps(m[0].c, PROF_RATES);
        if (tile_tma_ok(m[0].c)) {
            if (int rc = rates_rows_dense_group(stale.data(), (int)stale.size(), &blocks.dense)) return rc;
        } else {
            for (cet_ctx *c : stale)
                if (int rc = rates_rows_compact(c, R.eval_lo, R.eval_hi)) return rc;
        }
    }
    for (cet_ctx *c : stale) c->sweep_rates_valid = true;
    return 0;
}

template <int CAP>
static int sweep_group_once(const std::vector<GroupMember> &m, GroupTables<CAP> &t, GroupBlocks &blocks, bool count)
{
    const int n = (int)m.size();
    cet_ctx *c0 = m[0].c;
    cudaStream_t st = c0->stream;
    const SlabRanges R = slab_ranges(c0);             // single-slab contexts of one L: the same for all
    const int n_eval = R.eval_hi - R.eval_lo;
    const int tpp = (int)((c0->plane + ST_TILE - 1) / ST_TILE);
    ProfScope step_scope(c0, PROF_STEP);
    if (int rc = sweep_group_prepare(m, R, blocks)) return rc;
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = m[q].c;
        CloseArgs &a = t.close.a[q];
        a.ss = c->sweep; a.blk_sum = c->blk_sum; a.blk_max = c->blk_max; a.plane_sum = c->plane_sum; a.stamp = c->stamp;
        a.refresh_queue = (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES) + 3;
        a.dense_queue = dense_queue(c);
        a.events_per_sweep = m[q].sp->events_per_sweep; a.p_max = m[q].sp->p_max;
        t.stream.a[q] = stream_args(c, m[q].sp, R);
        t.pick.a[q] = pick_args(c, m[q].sp, true);
        t.apply.a[q] = apply_args_of(c, m[q].sp, R, true, count);
    }
    const int stamp_words = (int)(((size_t)c0->nloc / 8 + 8 + 3) / 4);
    sweep_reset_group_kernel<CAP><<<dim3((unsigned)std::min((stamp_words + 255) / 256, 64), (unsigned)n), 256, 0, st>>>(
        t.close, stamp_words, (int)c0->n0);
    CET_CUDA(cudaGetLastError());
    {
        ProfScope ps(c0, PROF_DECIDE);
        sweep_stream_group_kernel<CAP><<<dim3((unsigned)tpp, (unsigned)n_eval, (unsigned)n), ST_THREADS, 0, st>>>(t.stream);
    }
    CET_CUDA(cudaGetLastError());
    sweep_plane_reduce_group_kernel<CAP><<<dim3((unsigned)((n_eval + 3) / 4), (unsigned)n), 128, 0, st>>>(t.close, tpp, n_eval);
    CET_CUDA(cudaGetLastError());
    // pick / apply stride over each lattice's fired list; the split of a list over CTAs does not change the outcome
    // (claims are resolved by atomicMax of fixed keys, counters by integer atomics)
    const unsigned sparse_x = (unsigned)std::max(1, (sm_count(c0) * 32 + n - 1) / n);
    {
        ProfScope ps(c0, PROF_PICK);
        sweep_pick_group_kernel<CAP><<<dim3(sparse_x, 1, (unsigned)n), 128, 0, st>>>(t.pick);
    }
    CET_CUDA(cudaGetLastError());
    {
        ProfScope ps(c0, PROF_APPLY);
        sweep_apply_group_kernel<CAP><<<dim3(sparse_x, 1, (unsigned)n), 128, 0, st>>>(t.apply);
    }
    CET_CUDA(cudaGetLastError());
    {
        ProfScope ps(c0, PROF_REFRESH);
        std::vector<cet_ctx *> cs(n);
        for (int q = 0; q < n; ++q) cs[q] = m[q].c;
        if (int rc = rates_rows_dirty_compact_group(cs.data(), n, R.eval_lo, R.eval_hi, &blocks.refresh)) return rc;
    }
    sweep_finalize_group_kernel<CAP><<<n, 256, 0, st>>>(t.close, (int)c0->n0);
    CET_CUDA(cudaGetLastError());
    if (count)
        for (const GroupMember &g : m) g.c->sweep_index++;
    return 0;
}

template <int CAP>
static int sweep_group_run(const std::vector<GroupMember> &all, const std::vector<GroupMember> &priming, int64_t n_sweeps)
{
    std::unique_ptr<GroupTables<CAP>> t(new GroupTables<CAP>());
    GroupBlocks blocks;
    if (!priming.empty())
        if (int rc = sweep_group_once<CAP>(priming, *t, blocks, false)) return rc;
    for (int64_t s = 0; s < n_sweeps; ++s)
        if (int rc = sweep_group_once<CAP>(all, *t, blocks, true)) return rc;
    return 0;
}

// The group's work runs on the first context's stream: every context's stream is pointed at it for the call
// (so that the per-context compact rebuild of non-TMA L launches there too) and restored after it.  The call synchronises every context before and after, so no events are needed to order the work.
struct StreamSwap {
    std::vector<cet_ctx *> cs;
    std::vector<cudaStream_t> own;
    StreamSwap(cet_ctx *const *ctxs, int n) : cs(ctxs, ctxs + n)
    {
        for (cet_ctx *c : cs) { own.push_back(c->stream); c->stream = cs[0]->stream; }
    }
    ~StreamSwap() { for (size_t q = 0; q < cs.size(); ++q) cs[q]->stream = own[q]; }
};

}  // namespace cet

extern "C" int cet_sweep_run_group(cet_ctx *const *ctxs, int32_t n_ctx, int64_t n_sweeps, const cet_sweep_params *sp,
                                   const cet_thermal_params *tp, cet_sweep_result *res)
{
    CET_REQUIRE(ctxs && sp && res, "cet_sweep_run_group: NULL argument");
    CET_REQUIRE(n_ctx >= 1 && n_ctx <= GROUP_MAX, "cet_sweep_run_group: need 1 <= n_ctx <= %d, got %d", GROUP_MAX, (int)n_ctx);
    CET_REQUIRE(n_sweeps >= 0, "cet_sweep_run_group: n_sweeps < 0");
    for (int q = 0; q < n_ctx; ++q) {
        const cet_ctx *c = ctxs[q];
        CET_REQUIRE(c, "cet_sweep_run_group: context %d is NULL", q);
        for (int r = 0; r < q; ++r) CET_REQUIRE(ctxs[r] != c, "cet_sweep_run_group: context %d repeats context %d", q, r);
        CET_REQUIRE(c->device == ctxs[0]->device, "cet_sweep_run_group: context %d is on another device", q);
        CET_REQUIRE(c->world == 1 && c->halo == 0 && c->i_begin == 0 && c->i_end == c->n0,
                    "cet_sweep_run_group: context %d is a slab; groups take whole-lattice contexts", q);
        CET_REQUIRE(c->cubic && c->have_rp, "cet_sweep_run_group: context %d needs a cubic lattice with rate params", q);
        CET_REQUIRE(c->n1 == ctxs[0]->n1, "cet_sweep_run_group: context %d has L = %lld, context 0 L = %lld", q,
                    (long long)c->n1, (long long)ctxs[0]->n1);
        CET_REQUIRE(c->debug_flags == 0, "cet_sweep_run_group: context %d has debug flags set", q);
        CET_REQUIRE(c->nloc < (1ll << 31), "cet_sweep_run_group: the lattice must have fewer than 2^31 sites");
        CET_REQUIRE(sp[q].p_max > 0.0 && sp[q].p_max < 1.0 && sp[q].events_per_sweep > 0.0,
                    "cet_sweep_run_group: context %d: need 0 < p_max < 1 and events_per_sweep > 0", q);
        CET_REQUIRE(sp[q].thermal_every <= 0 || tp != nullptr, "cet_sweep_run_group: context %d: thermal_every needs thermal params", q);
    }
    cet::DeviceGuard dg(ctxs[0]->device);
    // the tile path's state and its condition (no empty site carries an orientation), checked on every context
    // before anything else is allocated or launched: a lattice that fails it needs the gather kernels, which are not
    // grouped.  The check derives the compact tile state (cvox / pairop) of the contexts it examines; nothing a
    // caller can read changes.
    for (int q = 0; q < n_ctx; ++q) {
        cet_ctx *c = ctxs[q];
        if (int rc = tile_state_ensure(c)) return rc;
        CET_REQUIRE(c->emp_canonical, "cet_sweep_run_group: context %d has empty sites with an orientation (gather path)", q);
    }
    for (int q = 0; q < n_ctx; ++q)
        if (int rc = sweep_alloc(ctxs[q])) return rc;
    std::vector<SweepState> before(n_ctx), after(n_ctx);
    std::vector<GroupMember> all, priming;
    for (int q = 0; q < n_ctx; ++q) {
        cet_ctx *c = ctxs[q];
        if (int rc = rate_tables_ensure(c)) return rc;
        c->nst_valid = false;
        CET_CUDA(cudaMemsetAsync(dense_queue(c), 0, sizeof(unsigned int), c->stream));    // the grouped rebuild's queue
        CET_CUDA(cudaMemcpyAsync(&before[q], c->sweep, sizeof(SweepState), cudaMemcpyDeviceToHost, c->stream));
        CET_CUDA(cudaStreamSynchronize(c->stream));
        const GroupMember g{c, &sp[q], tp ? &tp[q] : nullptr};
        all.push_back(g);
        if (n_sweeps > 0 && before[q].tau == 0.0 && !before[q].terminated) priming.push_back(g);
    }
    {
        StreamSwap swap(ctxs, n_ctx);
        const int rc = n_ctx <= 16 ? sweep_group_run<16>(all, priming, n_sweeps) : sweep_group_run<GROUP_MAX>(all, priming, n_sweeps);
        if (rc) return rc;
        for (int q = 0; q < n_ctx; ++q) {
            ctxs[q]->rates_valid = false;
            CET_CUDA(cudaMemcpyAsync(&after[q], ctxs[q]->sweep, sizeof(SweepState), cudaMemcpyDeviceToHost, ctxs[q]->stream));
        }
        CET_CUDA(cudaStreamSynchronize(ctxs[0]->stream));
    }
    for (int q = 0; q < n_ctx; ++q)
        if (int rc = sweep_finish(ctxs[q], before[q], after[q], n_sweeps, &res[q])) return rc;
    return 0;
}
