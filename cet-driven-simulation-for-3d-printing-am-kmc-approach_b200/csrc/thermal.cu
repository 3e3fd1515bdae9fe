// thermal.cu — explicit finite-difference heat stencil (thermal_solver.py).
//
// update_temperature_cet (thermal_solver.py:107-117) and update_temperature (:36-105) are
// 7-point fp64 stencils with edge-replicate boundaries (scipy.ndimage.laplace mode='reflect')
// followed by a clip.  HBM-bound: 8 B read + 8 B written per voxel (16 B/site algorithmic).
//
// Bit-exactness: the reference runs the stencil 16x past its stability limit, round-off is
// amplified every call, so the scipy operation order is reproduced exactly with explicit
// round-to-nearest intrinsics (no FMA contraction):
//     t_a = c*(-2) + (l_a + r_a)   for axis a = 0,1,2
//     lap = ((t_0 + t_1) + t_2) * inv_dx2
//     new = clip(c + (dt*ALPHA) * lap, lo, hi)
//
// Kernel shape: one thread per voxel column segment; a CTA covers a (TJ x TK) tile of one
// plane and marches over PLANES_PER_CTA consecutive planes keeping the i-1 / i / i+1 values
// in registers, so each T value is fetched from L2/HBM once along i; the j and k neighbours
// come from L1 (same CTA touches the adjacent rows) and warp shuffles.
#include "ctx.cuh"
#include "tile_state.cuh"

namespace cet {

__device__ __forceinline__ double fix_nan(double v, int nan_to_num, double nan_value)
{
    if (nan_to_num) {
        if (v != v) return nan_value;                                // np.nan_to_num(nan=T_SUB)
        if (v == INFINITY) return 1.7976931348623157e308;
        if (v == -INFINITY) return -1.7976931348623157e308;
    }
    return v;
}

struct ThermalArgs {
    const double *Tin;
    double *Tout;
    const uint8_t *vox, *vox_prev;   // full variant only
    const double *q_top;             // full variant only (n1*n2)
    int n0, n1, n2;                  // global extents
    int i_off;                       // global i of local plane 0
    int p_lo, p_hi;                  // local planes to update
    int np;
    double dt_alpha, inv_dx2, lo, hi, nan_value;
    int nan_to_num;
    const int32_t *stop;             // device flag: when set the step is the identity (run terminated)
    // full variant
    double dt, alpha, rho_cp, latent_over_cp, inv_dt_latent;
};

constexpr int TH_TK = 128;   // threads along k
constexpr int TH_TJ = 4;     // rows per CTA
constexpr int TH_PLANES = 8; // planes marched per CTA

// What cet_thermal_full_group fuses into the full stencil pass of a lattice: the thread that reads vox_prev[s] and
// vox[s] for its centre site s then writes vox_prev[s] = vox[s] (cet_snapshot_state), and, while the lattice's tile
// state is valid, an empty site's pair operand takes its new temperature (tile_pairop_T).  Kept out of ThermalArgs,
// which the solo kernels take by value.
struct ThermalFuse {
    uint8_t *vox_prev;               // snapshot target (NULL: no snapshot)
    const uint8_t *cvox;             // NULL: the tile state is stale and stays so
    double *pairop;
};
__device__ __forceinline__ void thermal_fuse_site(const ThermalArgs &a, const ThermalFuse *x, int64_t s, double v)
{
    if (x->vox_prev) x->vox_prev[s] = a.vox[s];
    if (x->cvox && (x->cvox[s] & 15u) == TC_EMPTY) x->pairop[s] = v;
}

// What cet_sweep_run fuses into update_temperature_cet on a whole-lattice context whose tile state is valid: a site
// is *changed* when its new temperature differs in bit pattern from the value read (a NaN that nan_to_num replaced
// counts).  A changed empty site's pair operand takes its new temperature: pairop == T held on every empty site
// before the step, so pairop ends as tile_pairop_T would leave it.  With a bitmap (n2 % 32 == 0, the vector kernel
// only) every word of it is written, one bit per local site, and the changed sites are counted.
struct ThermalTrack {
    const uint8_t *cvox;
    double *pairop;
    uint32_t *changed;               // NULL: no bitmap, no count
    unsigned int *n_changed;
};

// The kernel bodies take their arguments by reference and the plane block `zb` (blockIdx.z of a solo launch): the
// grouped launches of cet_sweep_run_group and cet_thermal_full_group run them for the table entry of their lattice.
// FUSE (full variant, whole-lattice contexts, no stop flag): x holds the fused writes of ThermalFuse.
// TRACK (CET variant): t holds the pair-operand writes of ThermalTrack (the scalar kernel keeps no bitmap).
template <bool FULL, bool FUSE = false, bool TRACK = false>
__device__ __forceinline__ void thermal_body(const ThermalArgs &a, int zb, const ThermalFuse *x = nullptr,
                                             const ThermalTrack *t = nullptr)
{
    const int k = blockIdx.x * TH_TK + threadIdx.x;
    const int j = blockIdx.y * TH_TJ + threadIdx.y;
    const int p0 = a.p_lo + zb * TH_PLANES;
    if (k >= a.n2 || j >= a.n1) return;
    const int64_t plane = (int64_t)a.n1 * a.n2;
    const int jm = j > 0 ? j - 1 : 0, jp = j < a.n1 - 1 ? j + 1 : a.n1 - 1;
    const int km = k > 0 ? k - 1 : 0, kp = k < a.n2 - 1 ? k + 1 : a.n2 - 1;
    const int p1 = min(p0 + TH_PLANES, a.p_hi);
    if (a.stop != nullptr && *a.stop != 0) {       // kmc_simulation.py:260-262: no update after termination
        for (int p = p0; p < p1; ++p) {
            const int64_t s = (int64_t)p * plane + (int64_t)j * a.n2 + k;
            a.Tout[s] = a.Tin[s];
        }
        return;
    }

    auto ld = [&](int p, int jj, int kk) {
        return fix_nan(a.Tin[(int64_t)p * plane + (int64_t)jj * a.n2 + kk], a.nan_to_num, a.nan_value);
    };
    // plane below p0 (replicate at the global bottom)
    int gi = a.i_off + p0;
    double below = ld(gi > 0 ? p0 - 1 : p0, j, k);
    double centre = ld(p0, j, k);
    for (int p = p0; p < p1; ++p, ++gi) {
        const double above = ld(gi < a.n0 - 1 ? p + 1 : p, j, k);
        const double l1 = ld(p, jm, k), r1 = ld(p, jp, k);
        const double l2 = ld(p, j, km), r2 = ld(p, j, kp);
        const double m2c = __dmul_rn(centre, -2.0);
        const double t0 = __dadd_rn(m2c, __dadd_rn(below, above));
        const double t1 = __dadd_rn(m2c, __dadd_rn(l1, r1));
        const double t2 = __dadd_rn(m2c, __dadd_rn(l2, r2));
        double lap = __dadd_rn(__dadd_rn(t0, t1), t2);
        lap = __dmul_rn(lap, a.inv_dx2);
        double v;
        if (!FULL) {
            v = __dadd_rn(centre, __dmul_rn(a.dt_alpha, lap));
        } else {
            const int64_t s = (int64_t)p * plane + (int64_t)j * a.n2 + k;
            const double q = (gi == a.n0 - 1) ? a.q_top[(int64_t)j * a.n2 + k] : 0.0;
            const bool solidified = (a.vox_prev[s] & 0x0F) == 0 && (a.vox[s] & 0x0F) != 0;
            const double dFdt = solidified ? a.inv_dt_latent : 0.0;
            const double dTdt = __dadd_rn(__dadd_rn(__dmul_rn(a.alpha, lap), __ddiv_rn(q, a.rho_cp)),
                                          __dmul_rn(a.latent_over_cp, dFdt));
            v = __dadd_rn(centre, __dmul_rn(a.dt, dTdt));
        }
        if (v < a.lo) v = a.lo;       // np.clip: NaN stays NaN
        if (v > a.hi) v = a.hi;
        a.Tout[(int64_t)p * plane + (int64_t)j * a.n2 + k] = v;
        if constexpr (FUSE) thermal_fuse_site(a, x, (int64_t)p * plane + (int64_t)j * a.n2 + k, v);
        if constexpr (TRACK) {
            const int64_t s = (int64_t)p * plane + (int64_t)j * a.n2 + k;
            if (__double_as_longlong(v) != __double_as_longlong(a.Tin[s]) && (t->cvox[s] & 15u) == TC_EMPTY) t->pairop[s] = v;
        }
        below = centre;
        centre = above;
    }
}
template <bool FULL>
__global__ void __launch_bounds__(TH_TK *TH_TJ) thermal_kernel(ThermalArgs a) { thermal_body<FULL>(a, blockIdx.z); }
__global__ void __launch_bounds__(TH_TK *TH_TJ) thermal_track_kernel(ThermalArgs a, const ThermalTrack t)
{
    thermal_body<false, false, true>(a, blockIdx.z, nullptr, &t);
}

// Fast path (n2 a multiple of V = 2 or 4): V consecutive k per thread with 16-byte loads/stores,
// the k-neighbours exchanged by warp shuffles, the i-neighbours kept in a register queue while
// the CTA marches over TH2_PLANES planes; only the j-neighbour rows are re-read (from L1/L2: the
// same CTA loaded them as centre rows one thread-row away).  Per V outputs: 3*V/2 vector loads,
// V/2 vector stores, 2 shuffles.
constexpr int TH2_TJ = 8, TH2_PLANES = 16;

template <int V, bool NANFIX>
struct RowVec {
    double v[V];
    __device__ __forceinline__ void load(const double *p, double nan_value)
    {
#pragma unroll
        for (int e = 0; e < V; e += 2) {
            const double2 t = *reinterpret_cast<const double2 *>(p + e);
            v[e] = t.x; v[e + 1] = t.y;
        }
        if (NANFIX) {
#pragma unroll
            for (int e = 0; e < V; ++e)      // one compare in the common case: NaN and +-inf fail |v| <= DBL_MAX
                if (!(fabs(v[e]) <= 1.7976931348623157e308)) v[e] = fix_nan(v[e], 1, nan_value);
        }
    }
};

template <bool FULL, bool NANFIX, int V, bool FUSE = false, bool TRACK = false>
__device__ __forceinline__ void thermal_v2_body(const ThermalArgs a, int zb, const ThermalFuse *x = nullptr,
                                                const ThermalTrack *t = nullptr)
{
    const int lane = threadIdx.x;
    const int k0 = (blockIdx.x * 32 + lane) * V;
    const int j = blockIdx.y * TH2_TJ + threadIdx.y;
    const int p0 = a.p_lo + zb * TH2_PLANES;
    if (j >= a.n1) return;                                   // whole warp (threadIdx.y is per warp)
    const bool in = k0 < a.n2;                               // n2 % V == 0: the whole vector is inside
    const int64_t plane = (int64_t)a.n1 * a.n2;
    const int jm = j > 0 ? j - 1 : 0, jp = j < a.n1 - 1 ? j + 1 : a.n1 - 1;
    const int p1 = min(p0 + TH2_PLANES, a.p_hi);
    const int kc = in ? k0 : 0;                              // inactive lanes read a valid address
    const bool stop = a.stop != nullptr && *a.stop != 0;
    // row pointers of plane p0, bumped by one plane per iteration
    const double *pc = a.Tin + (int64_t)p0 * plane + (int64_t)j * a.n2 + kc;
    const double *pm = a.Tin + (int64_t)p0 * plane + (int64_t)jm * a.n2 + kc;
    const double *pp = a.Tin + (int64_t)p0 * plane + (int64_t)jp * a.n2 + kc;
    double *po = a.Tout + (int64_t)p0 * plane + (int64_t)j * a.n2 + kc;
    int gi = a.i_off + p0;
    RowVec<V, NANFIX> below, centre, above, l1, r1;
    unsigned n_chg = 0;                                      // TRACK: changed sites seen by this lane
    below.load(gi > 0 ? pc - plane : pc, a.nan_value);
    centre.load(pc, a.nan_value);
    for (int p = p0; p < p1; ++p, ++gi) {
        above.load(gi < a.n0 - 1 ? pc + plane : pc, a.nan_value);
        l1.load(pm, a.nan_value);
        r1.load(pp, a.nan_value);
        // k neighbours: left of v[0] and right of v[V-1] come from the adjacent lanes
        double left = __shfl_up_sync(0xffffffffu, centre.v[V - 1], 1);
        double right = __shfl_down_sync(0xffffffffu, centre.v[0], 1);
        if (lane == 0) {
            left = centre.v[0];
            if (k0 > 0) { left = pc[-1]; if (NANFIX) left = fix_nan(left, 1, a.nan_value); }
        }
        if (lane == 31 || k0 + V >= a.n2) {
            right = centre.v[V - 1];
            if (in && k0 + V < a.n2) { right = pc[V]; if (NANFIX) right = fix_nan(right, 1, a.nan_value); }
        }
        double out[V];
#pragma unroll
        for (int e = 0; e < V; ++e) {
            const double c = centre.v[e];
            const double kl = e == 0 ? left : centre.v[e > 0 ? e - 1 : 0];
            const double kr = e == V - 1 ? right : centre.v[e < V - 1 ? e + 1 : V - 1];
            const double m2c = __dmul_rn(c, -2.0);
            const double t0 = __dadd_rn(m2c, __dadd_rn(below.v[e], above.v[e]));
            const double t1 = __dadd_rn(m2c, __dadd_rn(l1.v[e], r1.v[e]));
            const double t2 = __dadd_rn(m2c, __dadd_rn(kl, kr));
            double lap = __dadd_rn(__dadd_rn(t0, t1), t2);
            lap = __dmul_rn(lap, a.inv_dx2);
            double v;
            if (!FULL) {
                v = __dadd_rn(c, __dmul_rn(a.dt_alpha, lap));
            } else {
                const int64_t s = (int64_t)p * plane + (int64_t)j * a.n2 + kc + e;
                const double q = (gi == a.n0 - 1) ? a.q_top[(int64_t)j * a.n2 + kc + e] : 0.0;
                const bool solidified = (a.vox_prev[s] & 0x0F) == 0 && (a.vox[s] & 0x0F) != 0;
                const double dFdt = solidified ? a.inv_dt_latent : 0.0;
                const double dTdt = __dadd_rn(__dadd_rn(__dmul_rn(a.alpha, lap), __ddiv_rn(q, a.rho_cp)),
                                              __dmul_rn(a.latent_over_cp, dFdt));
                v = __dadd_rn(c, __dmul_rn(a.dt, dTdt));
            }
            if (v < a.lo) v = a.lo;       // np.clip: NaN stays NaN
            if (v > a.hi) v = a.hi;
            out[e] = v;
        }
        if (in) {
#pragma unroll
            for (int e = 0; e < V; e += 2) {
                double2 o;
                if (stop) o = *reinterpret_cast<const double2 *>(pc + e);
                else { o.x = out[e]; o.y = out[e + 1]; }
                *reinterpret_cast<double2 *>(po + e) = o;
            }
            if constexpr (FUSE) {                             // lanes past n2 read a borrowed address: they write nothing
#pragma unroll
                for (int e = 0; e < V; ++e) thermal_fuse_site(a, x, (int64_t)p * plane + (int64_t)j * a.n2 + kc + e, out[e]);
            }
        }
        if constexpr (TRACK) {
            unsigned nib = 0;                                 // bit e: site kc + e changed (never on the stop path)
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const double raw = NANFIX ? pc[e] : centre.v[e];
                if (__double_as_longlong(out[e]) != __double_as_longlong(raw)) nib |= 1u << e;
            }
            if (!in || stop) nib = 0;
            if (nib) {
                const int64_t s = (int64_t)p * plane + (int64_t)j * a.n2 + kc;
#pragma unroll
                for (int e = 0; e < V; ++e)
                    if ((nib >> e & 1u) && (t->cvox[s + e] & 15u) == TC_EMPTY) t->pairop[s + e] = out[e];
            }
            if constexpr (V == 4) {
                if (t->changed) {                             // n2 % 32 == 0: 8 lanes make one word of one row
                    uint32_t word = nib << (4 * (lane & 7));
                    word |= __shfl_xor_sync(0xffffffffu, word, 1);
                    word |= __shfl_xor_sync(0xffffffffu, word, 2);
                    word |= __shfl_xor_sync(0xffffffffu, word, 4);
                    if (in && (lane & 7) == 0) t->changed[((int64_t)p * plane + (int64_t)j * a.n2 + k0) >> 5] = word;
                    n_chg += __popc(nib);
                }
            }
        }
        below = centre;
        centre = above;
        pc += plane; pm += plane; pp += plane; po += plane;
    }
    if constexpr (TRACK && V == 4) {
        if (t->changed) {                                     // one counter update per warp
            n_chg = __reduce_add_sync(0xffffffffu, n_chg);
            if (lane == 0 && n_chg) atomicAdd(t->n_changed, n_chg);
        }
    }
}
template <bool FULL, bool NANFIX, int V>
__global__ void __launch_bounds__(32 * TH2_TJ) thermal_kernel_v2(const ThermalArgs a) { thermal_v2_body<FULL, NANFIX, V>(a, blockIdx.z); }
template <bool NANFIX, int V>
__global__ void __launch_bounds__(32 * TH2_TJ) thermal_track_kernel_v2(const ThermalArgs a, const ThermalTrack t)
{
    thermal_v2_body<false, NANFIX, V, false, true>(a, blockIdx.z, nullptr, &t);
}

// Grouped update_temperature_cet (cet_sweep_run_group): blockIdx.z = lattice * nzb + plane block.  V = 0: the
// scalar kernel (odd n2).
template <bool NANFIX, int V, int CAP>
__global__ void __launch_bounds__(V ? 32 * TH2_TJ : TH_TK * TH_TJ) thermal_group_kernel(const __grid_constant__ GroupArgs<ThermalArgs, CAP> g, int nzb)
{
    const ThermalArgs &a = g.a[blockIdx.z / nzb];
    if constexpr (V == 0) thermal_body<false>(a, blockIdx.z % nzb);
    else thermal_v2_body<false, NANFIX, V>(a, blockIdx.z % nzb);
}

__global__ void fill_gradient_kernel(double *T, int64_t plane, int np, int i_off, int n0, double t0, double g)
{
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < plane * np;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int gi = i_off + (int)(q / plane);
        if (gi >= 0 && gi < n0) T[q] = __dadd_rn(t0, __dmul_rn(g, (double)gi));   // T_SUB + G*i
    }
}

static void thermal_range(const cet_ctx *c, int *p_lo, int *p_hi)
{
    // every local plane inside the global domain whose i-neighbours are available locally
    const int i_off = (int)(c->i_begin - c->halo);
    int lo = 0, hi = (int)c->np;
    while (lo < hi && i_off + lo < 0) ++lo;
    while (hi > lo && i_off + hi - 1 > c->n0 - 1) --hi;
    if (i_off + lo > 0 && lo == 0) lo = 1;                    // needs plane lo-1
    if (i_off + hi - 1 < c->n0 - 1 && hi == (int)c->np) hi -= 1;   // needs plane hi
    *p_lo = lo; *p_hi = hi;
}

static void thermal_geometry(const cet_ctx *c, ThermalArgs &a)
{
    a.Tin = c->T; a.Tout = c->T2;
    a.n0 = (int)c->n0; a.n1 = (int)c->n1; a.n2 = (int)c->n2;
    a.i_off = (int)(c->i_begin - c->halo);
    a.np = (int)c->np;
    thermal_range(c, &a.p_lo, &a.p_hi);
}
// the host side of a finished step: T2 becomes T, and what the new temperatures invalidate
static void thermal_done(cet_ctx *c, const ThermalArgs &a, bool full)
{
    double *t = c->T; c->T = c->T2; c->T2 = t;
    if (a.nan_to_num) c->T_finite = true;   // a pass skipped by the stop flag cannot be the first of a run
    if (full) c->T_finite = false;          // the laser source term is caller data
    c->rates_valid = false; c->sweep_rates_valid = false;
}

// track (CET variant only): the stencil's ThermalTrack writes (NULL: none)
template <bool FULL>
static int launch_thermal(cet_ctx *c, ThermalArgs &a, const ThermalTrack *track = nullptr)
{
    thermal_geometry(c, a);
    if (a.p_hi <= a.p_lo) return 0;
    // np.nan_to_num is the identity on a finite field, and a finite field stays finite under the
    // clipped update: once a fixing pass has run (or the field is known finite) skip the checks.
    const bool nanfix = a.nan_to_num && !c->T_finite;
    if (c->n2 % 2 == 0) {
        const int V = (c->n2 % 4 == 0) ? 4 : 2;
        dim3 block(32, TH2_TJ);
        dim3 grid((unsigned)((c->n2 / V + 31) / 32), (unsigned)((c->n1 + TH2_TJ - 1) / TH2_TJ),
                  (unsigned)((a.p_hi - a.p_lo + TH2_PLANES - 1) / TH2_PLANES));
        ProfScope ps(c, PROF_THERMAL);
        if (!FULL && track) {
            if (V == 4) {
                if (nanfix) thermal_track_kernel_v2<true, 4><<<grid, block, 0, c->stream>>>(a, *track);
                else thermal_track_kernel_v2<false, 4><<<grid, block, 0, c->stream>>>(a, *track);
            } else {
                if (nanfix) thermal_track_kernel_v2<true, 2><<<grid, block, 0, c->stream>>>(a, *track);
                else thermal_track_kernel_v2<false, 2><<<grid, block, 0, c->stream>>>(a, *track);
            }
        } else if (V == 4) {
            if (nanfix) thermal_kernel_v2<FULL, true, 4><<<grid, block, 0, c->stream>>>(a);
            else thermal_kernel_v2<FULL, false, 4><<<grid, block, 0, c->stream>>>(a);
        } else {
            if (nanfix) thermal_kernel_v2<FULL, true, 2><<<grid, block, 0, c->stream>>>(a);
            else thermal_kernel_v2<FULL, false, 2><<<grid, block, 0, c->stream>>>(a);
        }
    } else {
        dim3 block(TH_TK, TH_TJ);
        dim3 grid((unsigned)((c->n2 + TH_TK - 1) / TH_TK), (unsigned)((c->n1 + TH_TJ - 1) / TH_TJ),
                  (unsigned)((a.p_hi - a.p_lo + TH_PLANES - 1) / TH_PLANES));
        ProfScope ps(c, PROF_THERMAL);
        if (!FULL && track) thermal_track_kernel<<<grid, block, 0, c->stream>>>(a, *track);
        else thermal_kernel<FULL><<<grid, block, 0, c->stream>>>(a);
    }
    CET_CUDA(cudaGetLastError());
    // planes outside [p_lo, p_hi) keep their previous contents: copy them so that the swap
    // below does not resurrect values from two steps ago in ghost planes.
    const int64_t plane = c->plane;
    if (a.p_lo > 0)
        CET_CUDA(cudaMemcpyAsync(c->T2, c->T, (size_t)a.p_lo * plane * 8, cudaMemcpyDeviceToDevice, c->stream));
    if (a.p_hi < c->np)
        CET_CUDA(cudaMemcpyAsync(c->T2 + (int64_t)a.p_hi * plane, c->T + (int64_t)a.p_hi * plane,
                                 (size_t)(c->np - a.p_hi) * plane * 8, cudaMemcpyDeviceToDevice, c->stream));
    thermal_done(c, a, FULL);
    return 0;
}

static ThermalArgs cet_step_args(const cet_thermal_params *p, const int32_t *stop_flag)
{
    ThermalArgs a;
    memset(&a, 0, sizeof(a));
    a.dt_alpha = p->dt_alpha; a.inv_dx2 = p->inv_dx2; a.lo = p->lo; a.hi = p->hi;
    a.nan_value = p->nan_value; a.nan_to_num = p->nan_to_num;
    a.stop = stop_flag;
    return a;
}

// Used by the KMC drivers (kmc_exact.cu, sweep.cu): one update_temperature_cet on the ctx stream.
int thermal_cet_step(cet_ctx *c, const cet_thermal_params *p, const int32_t *stop_flag)
{
    ThermalArgs a = cet_step_args(p, stop_flag);
    return launch_thermal<false>(c, a);
}

// thermal_cet_step of a whole-lattice context with a valid tile state (cet_sweep_run): the stencil also keeps
// pairop == T on the empty sites (ThermalTrack), so tile_pairop_T_update is not needed.  changed (n2 % 32 == 0, else
// NULL): the bitmap of the changed sites, every word written; n_changed, which the caller has zeroed, gains their
// number.
int thermal_cet_step_tracked(cet_ctx *c, const cet_thermal_params *p, const int32_t *stop_flag, uint32_t *changed,
                             unsigned int *n_changed)
{
    CET_REQUIRE(c->world == 1 && c->halo == 0 && c->tile_valid, "thermal_cet_step_tracked: whole-lattice context with a valid tile state");
    CET_REQUIRE(!changed || c->n2 % 32 == 0, "thermal_cet_step_tracked: the changed bitmap needs n2 %% 32 == 0");
    ThermalArgs a = cet_step_args(p, stop_flag);
    const ThermalTrack t{c->cvox, c->pairop, changed, n_changed};
    return launch_thermal<false>(c, a, &t);
}

template <bool NANFIX, int V, int CAP>
static int thermal_group_launch(cet_ctx *const *cs, const ThermalArgs *args, int n)
{
    GroupArgs<ThermalArgs, CAP> g;
    for (int q = 0; q < n; ++q) g.a[q] = args[q];
    const cet_ctx *c = cs[0];
    const int planes = args[0].p_hi - args[0].p_lo;
    dim3 block, grid;
    int nzb;
    if (V) {
        nzb = (planes + TH2_PLANES - 1) / TH2_PLANES;
        block = dim3(32, TH2_TJ);
        grid = dim3((unsigned)((c->n2 / V + 31) / 32), (unsigned)((c->n1 + TH2_TJ - 1) / TH2_TJ), (unsigned)(nzb * n));
    } else {
        nzb = (planes + TH_PLANES - 1) / TH_PLANES;
        block = dim3(TH_TK, TH_TJ);
        grid = dim3((unsigned)((c->n2 + TH_TK - 1) / TH_TK), (unsigned)((c->n1 + TH_TJ - 1) / TH_TJ), (unsigned)(nzb * n));
    }
    thermal_group_kernel<NANFIX, V, CAP><<<grid, block, 0, c->stream>>>(g, nzb);
    CET_CUDA(cudaGetLastError());
    return 0;
}
template <bool NANFIX, int V>
static int thermal_group_launch(cet_ctx *const *cs, const ThermalArgs *args, int n)
{
    return n <= 16 ? thermal_group_launch<NANFIX, V, 16>(cs, args, n) : thermal_group_launch<NANFIX, V, GROUP_MAX>(cs, args, n);
}

// thermal_cet_step for a group of whole-lattice contexts of one L (cet_sweep_run_group), on the stream of cs[0]: one
// launch per kernel variant in use — the contexts whose T is not yet known to be finite take the nan_to_num pass.
int thermal_cet_step_group(cet_ctx *const *cs, const cet_thermal_params *const *tps, int n)
{
    if (n <= 0) return 0;
    ThermalArgs fix[GROUP_MAX], plain[GROUP_MAX];
    cet_ctx *fix_c[GROUP_MAX], *plain_c[GROUP_MAX];
    int n_fix = 0, n_plain = 0;
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = cs[q];
        ThermalArgs a = cet_step_args(tps[q], &c->sweep->terminated);
        thermal_geometry(c, a);
        CET_REQUIRE(a.p_lo == 0 && a.p_hi == (int)c->np, "thermal_cet_step_group: whole-lattice contexts only");
        if (a.nan_to_num && !c->T_finite) { fix_c[n_fix] = c; fix[n_fix++] = a; }
        else { plain_c[n_plain] = c; plain[n_plain++] = a; }
    }
    const int V = cs[0]->n2 % 4 == 0 ? 4 : cs[0]->n2 % 2 == 0 ? 2 : 0;
    {
        ProfScope ps(cs[0], PROF_THERMAL);
        for (int f = 0; f < 2; ++f) {
            cet_ctx *const *gc = f ? fix_c : plain_c;
            const ThermalArgs *ga = f ? fix : plain;
            const int m = f ? n_fix : n_plain;
            if (m == 0) continue;
            int rc;
            if (V == 4) rc = f ? thermal_group_launch<true, 4>(gc, ga, m) : thermal_group_launch<false, 4>(gc, ga, m);
            else if (V == 2) rc = f ? thermal_group_launch<true, 2>(gc, ga, m) : thermal_group_launch<false, 2>(gc, ga, m);
            else rc = thermal_group_launch<false, 0>(gc, ga, m);      // the scalar kernel applies nan_to_num per value
            if (rc) return rc;
        }
    }
    for (int q = 0; q < n_fix; ++q) thermal_done(fix_c[q], fix[q], false);
    for (int q = 0; q < n_plain; ++q) thermal_done(plain_c[q], plain[q], false);
    return 0;
}

// Grouped update_temperature (cet_thermal_full_group): blockIdx.z = lattice * nzb + plane block, the full stencil
// with the fused snapshot / pair-operand writes.  V = 0: the scalar kernel (odd n2).
struct ThermalFullGroupArgs {
    ThermalArgs t;
    ThermalFuse x;
};
static_assert(group_fits<ThermalFullGroupArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

template <int V, int CAP>
__global__ void __launch_bounds__(V ? 32 * TH2_TJ : TH_TK * TH_TJ)
thermal_full_group_kernel(const __grid_constant__ GroupArgs<ThermalFullGroupArgs, CAP> g, int nzb)
{
    const ThermalFullGroupArgs &a = g.a[blockIdx.z / nzb];
    if constexpr (V == 0) thermal_body<true, true>(a.t, blockIdx.z % nzb, &a.x);
    else thermal_v2_body<true, false, V, true>(a.t, blockIdx.z % nzb, &a.x);
}

template <int V, int CAP>
static int thermal_full_group_launch(cet_ctx *c0, const ThermalFullGroupArgs *args, int n)
{
    GroupArgs<ThermalFullGroupArgs, CAP> g;
    for (int q = 0; q < n; ++q) g.a[q] = args[q];
    const int planes = args[0].t.p_hi - args[0].t.p_lo;
    dim3 block, grid;
    int nzb;
    if (V) {
        nzb = (planes + TH2_PLANES - 1) / TH2_PLANES;
        block = dim3(32, TH2_TJ);
        grid = dim3((unsigned)((c0->n2 / V + 31) / 32), (unsigned)((c0->n1 + TH2_TJ - 1) / TH2_TJ), (unsigned)(nzb * n));
    } else {
        nzb = (planes + TH_PLANES - 1) / TH_PLANES;
        block = dim3(TH_TK, TH_TJ);
        grid = dim3((unsigned)((c0->n2 + TH_TK - 1) / TH_TK), (unsigned)((c0->n1 + TH_TJ - 1) / TH_TJ), (unsigned)(nzb * n));
    }
    thermal_full_group_kernel<V, CAP><<<grid, block, 0, c0->stream>>>(g, nzb);
    CET_CUDA(cudaGetLastError());
    return 0;
}
template <int V>
static int thermal_full_group_launch(cet_ctx *c0, const ThermalFullGroupArgs *args, int n)
{
    return n <= 16 ? thermal_full_group_launch<V, 16>(c0, args, n) : thermal_full_group_launch<V, GROUP_MAX>(c0, args, n);
}

}  // namespace cet

using namespace cet;

extern "C" {

int cet_thermal_cet(cet_ctx *c, const cet_thermal_params *p)
{
    CET_REQUIRE(c && p, "cet_thermal_cet: NULL argument");
    cet::DeviceGuard dg(c->device);
    c->tile_valid = false;
    return thermal_cet_step(c, p, nullptr);
}

int cet_thermal_full(cet_ctx *c, const cet_thermal_full_params *p, const double *q_top)
{
    CET_REQUIRE(c && p && q_top, "cet_thermal_full: NULL argument");
    CET_REQUIRE(c->vox_prev != nullptr,
                "cet_thermal_full: no previous state (call cet_upload_prev_state or cet_snapshot_state)");
    cet::DeviceGuard dg(c->device);
    if (!c->q_top) CET_CUDA(cudaMalloc(&c->q_top, c->plane * sizeof(double)));
    CET_CUDA(cudaMemcpyAsync(c->q_top, q_top, c->plane * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    ThermalArgs a;
    memset(&a, 0, sizeof(a));
    a.vox = c->vox; a.vox_prev = c->vox_prev; a.q_top = c->q_top;
    a.inv_dx2 = p->inv_dx2; a.lo = p->lo; a.hi = p->hi;
    a.dt = p->dt; a.alpha = p->alpha; a.rho_cp = p->rho_cp; a.latent_over_cp = p->latent_over_cp;
    a.inv_dt_latent = 1.0 / (p->dt > 1e-12 ? p->dt : 1e-12);   // mask / max(dt, 1e-12), thermal_solver.py:98
    int rc = launch_thermal<true>(c, a);
    c->tile_valid = false;
    if (rc) return rc;
    CET_CUDA(cudaStreamSynchronize(c->stream));   // q_top host pointer is borrowed for the call only
    return 0;
}

// cet_thermal_full (+ cet_snapshot_state) for a group of whole-lattice contexts of one L: one stencil launch for the
// group, on the stream of ctxs[0] after the work queued on every context's stream, one host synchronisation.
int cet_thermal_full_group(cet_ctx *const *ctxs, int32_t n_ctx, const cet_thermal_full_params *p,
                           const double *const *q_top, int32_t snapshot)
{
    CET_REQUIRE(ctxs && p && q_top, "cet_thermal_full_group: NULL argument");
    CET_REQUIRE(n_ctx >= 1 && n_ctx <= GROUP_MAX, "cet_thermal_full_group: need 1 <= n_ctx <= %d, got %d", GROUP_MAX,
                (int)n_ctx);
    for (int q = 0; q < n_ctx; ++q) {
        const cet_ctx *c = ctxs[q];
        CET_REQUIRE(c, "cet_thermal_full_group: context %d is NULL", q);
        for (int r = 0; r < q; ++r) CET_REQUIRE(ctxs[r] != c, "cet_thermal_full_group: context %d repeats context %d", q, r);
        CET_REQUIRE(c->device == ctxs[0]->device, "cet_thermal_full_group: context %d is on another device", q);
        CET_REQUIRE(c->world == 1 && c->halo == 0 && c->i_begin == 0 && c->i_end == c->n0,
                    "cet_thermal_full_group: context %d is a slab; groups take whole-lattice contexts", q);
        CET_REQUIRE(c->cubic, "cet_thermal_full_group: context %d is not a cubic lattice", q);
        CET_REQUIRE(c->n1 == ctxs[0]->n1, "cet_thermal_full_group: context %d has L = %lld, context 0 L = %lld", q,
                    (long long)c->n1, (long long)ctxs[0]->n1);
        CET_REQUIRE(q_top[q], "cet_thermal_full_group: q_top[%d] is NULL", q);
        CET_REQUIRE(c->vox_prev != nullptr,
                    "cet_thermal_full_group: context %d: no previous state (call cet_upload_prev_state or cet_snapshot_state)", q);
    }
    cet::DeviceGuard dg(ctxs[0]->device);
    cet_ctx *c0 = ctxs[0];
    ThermalFullGroupArgs args[GROUP_MAX];
    for (int q = 0; q < n_ctx; ++q) {
        cet_ctx *c = ctxs[q];
        ThermalFullGroupArgs &g = args[q];
        memset(&g, 0, sizeof(g));
        ThermalArgs &a = g.t;
        a.vox = c->vox; a.vox_prev = c->vox_prev;
        a.inv_dx2 = p[q].inv_dx2; a.lo = p[q].lo; a.hi = p[q].hi;
        a.dt = p[q].dt; a.alpha = p[q].alpha; a.rho_cp = p[q].rho_cp; a.latent_over_cp = p[q].latent_over_cp;
        a.inv_dt_latent = 1.0 / (p[q].dt > 1e-12 ? p[q].dt : 1e-12);   // as cet_thermal_full
        thermal_geometry(c, a);
        CET_REQUIRE(a.p_lo == 0 && a.p_hi == (int)c->np, "cet_thermal_full_group: whole-lattice contexts only");
        g.x.vox_prev = snapshot ? c->vox_prev : nullptr;
        if (c->tile_valid) { g.x.cvox = c->cvox; g.x.pairop = c->pairop; }
    }
    for (int q = 0; q < n_ctx; ++q) {
        cet_ctx *c = ctxs[q];
        if (!c->q_top) CET_CUDA(cudaMalloc(&c->q_top, c->plane * sizeof(double)));
        args[q].t.q_top = c->q_top;
        if (c != c0) {
            if (!c->ev_group) CET_CUDA(cudaEventCreateWithFlags(&c->ev_group, cudaEventDisableTiming));
            CET_CUDA(cudaEventRecord(c->ev_group, c->stream));
            CET_CUDA(cudaStreamWaitEvent(c0->stream, c->ev_group, 0));
        }
    }
    for (int q = 0; q < n_ctx; ++q)
        CET_CUDA(cudaMemcpyAsync(ctxs[q]->q_top, q_top[q], c0->plane * sizeof(double), cudaMemcpyHostToDevice, c0->stream));
    {
        ProfScope ps(c0, PROF_THERMAL);
        const int V = c0->n2 % 4 == 0 ? 4 : c0->n2 % 2 == 0 ? 2 : 0;
        const int rc = V == 4 ? thermal_full_group_launch<4>(c0, args, n_ctx)
                     : V == 2 ? thermal_full_group_launch<2>(c0, args, n_ctx) : thermal_full_group_launch<0>(c0, args, n_ctx);
        if (rc) return rc;
    }
    CET_CUDA(cudaStreamSynchronize(c0->stream));   // the q_top host pointers are borrowed for the call only
    for (int q = 0; q < n_ctx; ++q) thermal_done(ctxs[q], args[q].t, true);   // tile_valid as it was: see ThermalFuse
    return 0;
}

int cet_thermal_fill_gradient(cet_ctx *c, double t0, double g)
{
    CET_REQUIRE(c, "cet_thermal_fill_gradient: NULL ctx");
    cet::DeviceGuard dg(c->device);
    fill_gradient_kernel<<<sm_count(c) * 8, 256, 0, c->stream>>>(c->T, c->plane, (int)c->np,
                                                         (int)(c->i_begin - c->halo), (int)c->n0, t0, g);
    CET_CUDA(cudaGetLastError());
    lattice_changed(c);
    return 0;
}

}  // extern "C"
