// rates.cu — dense per-voxel event-rate evaluation (kmc_event_rates.py:43-176) and the sum
// hierarchy the BKL search walks, plus the legacy event-list export.
//
// What is stored per site is the SUM of the site's event rates in reference list order
// (diff events of an occupied site, nuc+att events of an empty one); individual events are
// re-enumerated on demand by `site_events` (site_rates.cuh).  On the top plane (global
// i == L-1) empty sites additionally own one deposition event each (kmc_event_rates.py:55-72)
// kept in dep_rate (NaN = no event).
//
// Hierarchy, all in the reference's canonical list order
//   plane i -> [dep segment | occupied-site segment | empty-site segment] -> row j -> site k
//   row_occ/row_emp[p*n1+j] : warp_row_sums over k
//   seg[3p+{0,1,2}]         : warp_strided_sum over j
//   total                   : block_sum over seg
//
// Dense kernel shape: one CTA per 256 consecutive sites — see rate_tile.cuh.
#include "ctx.cuh"
#include "rate_tile.cuh"
#include "tile_state.cuh"
#include <algorithm>
#include "reduce.cuh"

namespace cet {

constexpr int RB_WARPS = 8;

// K_eff / E_tot tables of rate_tile.cuh, from the per-event inline functions themselves.
__global__ void rate_tables_kernel(const cet_rate_params P, double *tab)
{
    const int t = threadIdx.x;
    if (t < 256) tab[RT_KEFF + t] = nuc_K_eff(P, t >> 4, t & 15);
    if (t < 48) tab[RT_ETOT + t] = occ_E_tot(P, t >> 4, t & 15);
    if (t < 32) tab[RT_EXP2 + t] = d_exp2_tab[t];
    if (t < 4) tab[RT_HE + t] = 0.5 * P.E_b[t == 3 ? 1 : t];
}

struct RateTileArgs;
template <int MINB>
__global__ void rates_tile_kernel(const __grid_constant__ RateTileArgs a, int s_lo, int s_hi, unsigned int *queue);
__global__ void dirty_eval_kernel(const __grid_constant__ RateTileArgs a, const int32_t *list, const unsigned int *n_list,
                                  unsigned int *queue);

int rates_refresh_list(cet_ctx *c, const int32_t *list, const unsigned int *counter, int64_t nsite_hint);     // rates_refresh.cu
int rates_refresh_list_group(cet_ctx *const *cs, int n, int64_t nsite_hint, int *blocks_per_sm);

int rate_tables_ensure(cet_ctx *c)
{
    if (!c->rate_attr_set) {                 // per device; a context lives on one device
        CET_CUDA(cudaFuncSetAttribute(rates_tile_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RateSmem)));
        CET_CUDA(cudaFuncSetAttribute(dirty_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RateSmem)));
        c->rate_attr_set = true;
    }
    if (c->rate_tab_valid) return 0;
    if (!c->rate_tab) CET_CUDA(cudaMalloc(&c->rate_tab, RT_TABLE_DOUBLES * sizeof(double) + 64));
    rate_tables_kernel<<<1, 256, 0, c->stream>>>(c->rp, c->rate_tab);
    CET_CUDA(cudaGetLastError());
    c->rate_tab_valid = true;
    return 0;
}

static RateTileArgs tile_args(cet_ctx *c)
{
    RateTileArgs a;
    a.g = c->lat();
    a.P = c->rp;
    a.tab = c->rate_tab;
    a.site_rate = c->site_rate; a.dep_rate = c->dep_rate; a.nst_out = c->nst;
    const int64_t top = c->n0 - 1 - (c->i_begin - c->halo);          // local plane of the global top
    if (top >= 0 && top < c->np) { a.top_lo = (int)(top * c->plane); a.top_hi = (int)((top + 1) * c->plane); }
    else { a.top_lo = 0; a.top_hi = 0; }
    a.nloc = (int)c->nloc;
    a.lut = nb_code_lut(c->rp);
    return a;
}

// Dense rate kernel: persistent CTAs, warps pull 256-site chunks of [s_lo, s_hi) from the queue.
template <int MINB>
__global__ void __launch_bounds__(RT_THREADS, MINB) rates_tile_kernel(const __grid_constant__ RateTileArgs a, int s_lo, int s_hi,
                                                                      unsigned int *queue)
{
    extern __shared__ __align__(16) unsigned char rate_dyn_smem[];
    RateSmem &sm = *reinterpret_cast<RateSmem *>(rate_dyn_smem);
    rate_smem_init(sm, a);
    rate_cta_loop<false>(a, sm, s_lo, s_hi - s_lo, nullptr, queue);
}

// BKL hierarchy level 1 (exact mode only): per-row sums split by occupancy class, one warp per row.
struct RowSumArgs {
    const uint8_t *vox;
    const double *site_rate, *dep_rate;
    double *row_occ, *row_emp, *row_dep;
    int32_t *row_depcnt;
    int L, p_lo, p_hi, top_plane;     // top_plane: local plane of the global top or -1
};
__global__ void __launch_bounds__(RB_WARPS * 32) row_sums_kernel(const RowSumArgs a)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int row = blockIdx.x * RB_WARPS + wid;
    if (row >= (a.p_hi - a.p_lo) * a.L) return;
    const int p = a.p_lo + row / a.L, j = row % a.L;
    const int64_t rbase = ((int64_t)p * a.L + j) * a.L;
    double occ, emp;
    warp_row_sums(a.vox + rbase, a.site_rate + rbase, a.L, &occ, &emp);
    if (lane == 0) { a.row_occ[p * a.L + j] = occ; a.row_emp[p * a.L + j] = emp; }
    if (p == a.top_plane) {
        double ds; int dc;
        warp_dep_row(a.dep_rate + j * a.L, a.L, &ds, &dc);
        if (lane == 0) { a.row_dep[j] = ds; a.row_depcnt[j] = dc; }
    }
}

// Neighbour-rate refresh (sweep.cu): the sites stamped in this sweep are re-evaluated with the same
// tile code as the dense pass.  Two kernels:
//   scan  streams the stamp bitmap (1 bit/site) and compacts the stamped sites into one global list
//         (one atomic per 8192-site CTA, so the list stays roughly in lattice order: a tile of 32
//         entries comes from one or two adjacent rows and its neighbour gathers coalesce;
//         emitting the list in 8 x 8 x L blocks instead was measured and is slower, 1.43 vs 1.39 ms
//         at 0.5 % N events per sweep and 6.2 vs 3.2 ms at 2 % N);
//   eval  evaluates the list with the tile code of the dense pass; the cached neighbour-class
//         word of every evaluated site is rewritten from a fresh gather (exactly the sites whose
//         neighbourhood changed), so the apply kernel needs no atomics to maintain the cache.
// Results go straight to site_rate / dep_rate; the BKL row sums are not maintained.
struct DirtyArgs {
    const uint32_t *stamp;            // one bit per local site
    int s_lo, s_hi;                   // local linear site range to scan
    int32_t *list;                    // capacity: one entry per local site
    unsigned int *n_list;             // list length (device counter)
};

constexpr int DS_STAGE = 2048;     // staged list entries per CTA (256 words = 8192 sites)

__device__ __forceinline__ void dirty_scan_body(const DirtyArgs &a)
{
    __shared__ int s_list[DS_STAGE];                                // staging; spills are appended directly
    __shared__ unsigned int c_list, b_list, s_first_spill;
    if (threadIdx.x == 0) { c_list = 0; s_first_spill = 0xffffffffu; }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int wi = (a.s_lo >> 5) + blockIdx.x * (RB_WARPS * 32) + threadIdx.x;      // this thread's 32 sites
    const int b0 = wi << 5;
    uint32_t match = b0 < a.s_hi ? a.stamp[wi] : 0u;
    if (b0 < a.s_lo) match &= 0xffffffffu << (a.s_lo - b0);                       // range ends inside a word
    if (b0 + 32 > a.s_hi && b0 < a.s_hi) match &= 0xffffffffu >> (b0 + 32 - a.s_hi);
    // ordered compaction of the warp's 1024 sites: warp scan of the match counts, one counter update per warp
    const int nm = __popc(match);
    int inc = nm;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    const int tot = __shfl_sync(0xffffffffu, inc, 31);
    if (tot) {
        unsigned int q0 = 0;
        int spill = 0;
        if (lane == 0) {
            q0 = atomicAdd(&c_list, (unsigned)tot);
            if (q0 + tot > DS_STAGE) {                                  // staging full: append directly
                atomicMin(&s_first_spill, q0);
                q0 = atomicAdd(a.n_list, (unsigned)tot);
                spill = 1;
            }
        }
        q0 = __shfl_sync(0xffffffffu, q0, 0);
        spill = __shfl_sync(0xffffffffu, spill, 0);
        int *dst = (spill ? a.list : s_list) + q0 + (inc - nm);
        while (match) {
            const int e = __ffs(match) - 1;
            match &= match - 1;
            *dst++ = b0 + e;
        }
    }
    __syncthreads();
    // the staged prefix is contiguous up to the first warp that did not fit
    const unsigned int n = min(c_list, s_first_spill);
    if (threadIdx.x == 0) b_list = n ? atomicAdd(a.n_list, n) : 0u;
    __syncthreads();
    for (unsigned int q = threadIdx.x; q < n; q += RB_WARPS * 32) a.list[b_list + q] = s_list[q];
}
__global__ void __launch_bounds__(RB_WARPS * 32) dirty_scan_kernel(const __grid_constant__ DirtyArgs a) { dirty_scan_body(a); }
// grouped sweeps: grid (CTAs per lattice, 1, lattices)
template <int CAP>
__global__ void __launch_bounds__(RB_WARPS * 32) dirty_scan_group_kernel(const __grid_constant__ GroupArgs<DirtyArgs, CAP> g)
{
    dirty_scan_body(g.a[blockIdx.z]);
}

__global__ void __launch_bounds__(RT_THREADS, 5) dirty_eval_kernel(const __grid_constant__ RateTileArgs a, const int32_t *list,
                                                                   const unsigned int *n_list, unsigned int *queue)
{
    extern __shared__ __align__(16) unsigned char rate_dyn_smem[];
    RateSmem &sm = *reinterpret_cast<RateSmem *>(rate_dyn_smem);
    rate_smem_init(sm, a);
    rate_cta_loop<true>(a, sm, 0, (int)*n_list, list, queue);
}

// ---- refresh on the compact tile state (tile_state.cuh) -------------------------------------------
// Same list, same queue-driven persistent CTAs, but a stamped site is re-evaluated from cvox (1 byte
// class code per site) and pairop (one 8-byte pair operand per site) instead of vox + the 8-byte
// neighbour-class cache + 32-byte unit vectors + T: the 14 class-code gathers of a warp fall into a
// handful of 128-byte lines of a 1-byte array, a pair costs one 8-byte gather whatever its class, and
// nothing is written but the rate sum.  DRAM traffic per refreshed site drops from ~660 B to ~190 B.
struct CompactWarpSmem {
    double rate[RT_WARP_PAIRS];
    double A[32], B[32];
    uint32_t idx[RT_WARP_PAIRS];             // local linear index of the pair's neighbour
    uint8_t own[RT_WARP_PAIRS];              // lane that owns the pair
};
struct CompactSmem {
    double tab[RT_TABLE_DOUBLES];
    int lin[16];
    unsigned int chunk[2];
    CompactWarpSmem w[RT_WARPS];
};
struct CompactArgs {
    const uint8_t *cvox;
    const double *pairop, *T;
    double *site_rate, *dep_rate;
    const double *tab;
    cet_rate_params P;
    int L, n0, i_off, nloc;
    int top_lo, top_hi;
    int chunk;               // list mode: stamped sites per warp and queue entry
};

__device__ __forceinline__ void compact_tile(const CompactArgs &a, const CompactSmem &sm, CompactWarpSmem &ws, int s, bool active)
{
    const cet_rate_params &P = a.P;
    const int lane = threadIdx.x & 31;
    const int L = a.L;
    unsigned c = 0;
    uint32_t wlo = 0, whi = 0;
    double T_self = 1.0, T_m = 1.0, T_p = 1.0;
    if (active) {
        const int LL = L * L;
        const int p = s / LL, r = s - p * LL, j = r / L, k = r - j * L;
        const unsigned inb = inbounds_mask(a.i_off + p, j, k, a.n0, L);
        c = a.cvox[s];
        unsigned b[14];
#pragma unroll
        for (int o = 0; o < 14; ++o) b[o] = (inb >> o & 1u) ? (unsigned)a.cvox[s + sm.lin[o]] & 15u : 0u;    // 0 = outside the lattice
#pragma unroll
        for (int o = 0; o < 8; ++o) wlo |= b[o] << (4 * o);
#pragma unroll
        for (int o = 8; o < 14; ++o) whi |= b[o] << (4 * (o - 8));
        const unsigned code = c & 15u;
        if (code == TC_EMPTY) {
            T_self = a.pairop[s];                                    // an empty site's pairop is its temperature
            T_m = T_self; T_p = T_self;
            if ((wlo | whi) & 0x11111111u) {                         // an occupied neighbour: grad_z is needed (:151-153)
                // an empty k neighbour keeps its temperature in pairop, in the sector just read for T_self
                if (k > 0) T_m = (a.cvox[s - 1] & 15u) == TC_EMPTY ? a.pairop[s - 1] : a.T[s - 1];
                if (k < L - 1) T_p = (a.cvox[s + 1] & 15u) == TC_EMPTY ? a.pairop[s + 1] : a.T[s + 1];
            }
        } else if ((code & 1u) && code != TC_DEFECT) {
            T_self = a.T[s];
        }
    }
    const uint64_t w = (uint64_t)wlo | ((uint64_t)whi << 32);
    const TilePrep q = tile_site_prep(P, sm.tab, w, active ? c : 0u, T_self, T_m, T_p);
    const uint64_t pm = q.pm;
    const bool is_emp = q.is_emp;
    if (pm) { ws.A[lane] = q.A; ws.B[lane] = q.B; }
    const int cnt = popc64(pm);
    const unsigned mine = is_emp ? (unsigned)cnt : (unsigned)cnt << 16;
    const unsigned all = __reduce_add_sync(0xffffffffu, mine);
    double sum = q.sum0;
    const int npass = all == 0 ? 0 : (((all & 0xFFFFu) + (all >> 16) > (unsigned)RT_WARP_PAIRS) ? 2 : 1);
    for (int pass = 0; pass < npass; ++pass) {
        const bool part = npass == 1 || (lane >> 4) == pass;
        const unsigned mine_p = part ? mine : 0u;
        unsigned inc = mine_p;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned u = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += u;
        }
        const unsigned total = __shfl_sync(0xffffffffu, inc, 31), excl = inc - mine_p;
        const int n_att = (int)(total & 0xFFFFu), n_diff = (int)(total >> 16);
        const int cnt_p = part ? cnt : 0;
        const int start = is_emp ? (int)(excl & 0xFFFFu) : RT_WARP_PAIRS - (int)(excl >> 16) - cnt_p;
        if (part) {
            int pos = start;
            unsigned lo = (unsigned)pm, hi = (unsigned)(pm >> 32);
            while (lo) {
                const int bb = __ffs(lo) - 1;
                lo &= lo - 1;
                ws.idx[pos] = (uint32_t)(s + sm.lin[bb >> 2]); ws.own[pos] = (uint8_t)lane; ++pos;
            }
            while (hi) {
                const int bb = __ffs(hi) - 1;
                hi &= hi - 1;
                ws.idx[pos] = (uint32_t)(s + sm.lin[8 + (bb >> 2)]); ws.own[pos] = (uint8_t)lane; ++pos;
            }
        }
        __syncwarp();
        // pairs, 32 at a time: attachment from the front, diffusion from the back; the operand gathers of the
        // next trip are issued before the arithmetic of the current one
        const int qd0 = RT_WARP_PAIRS - n_diff;
        const int n_trip = ((n_att > n_diff ? n_att : n_diff) + 31) >> 5;
        double oa = 0.0, od = 1.0;
        if (lane < n_att) oa = a.pairop[ws.idx[lane]];
        if (lane < n_diff) od = a.pairop[ws.idx[qd0 + lane]];
        for (int t = 0; t < n_trip; ++t) {
            const int qq = 32 * t + lane, qn = qq + 32;
            const double oa_c = oa, od_c = od;
            if (qn < n_att) oa = a.pairop[ws.idx[qn]];
            if (qn < n_diff) od = a.pairop[ws.idx[qd0 + qn]];
            if (qq < n_att) {                                        // kmc_event_rates.py:135-158
                const int ts = ws.own[qq];
                ws.rate[qq] = att_pair_rate_E(P, oa_c, ws.A[ts], ws.B[ts], sm.tab + RT_EXP2);
            }
            if (qq < n_diff) {                                       // :100-109
                const int ts = ws.own[qd0 + qq];
                ws.rate[qd0 + qq] = diff_pair_rate(P, ws.A[ts], ws.B[ts], od_c);
            }
        }
        __syncwarp();
        for (int q0 = 0; q0 < cnt_p; ++q0) sum += ws.rate[start + q0];     // slot order: the association order of site_rate_sum
        __syncwarp();
    }
    if (active) {
        a.site_rate[s] = sum;
        if (s >= a.top_lo && s < a.top_hi) {                             // deposition (:55-72): top plane only
            double dep;
            a.dep_rate[s - a.top_lo] = (is_emp && dep_rate(P, T_self, &dep)) ? dep : NAN;
        }
    }
}

// Queue-driven loop of one CTA over n sites (dense: s = s_lo + index; list != nullptr: s = list[index]).
// CHUNK = sites per warp and queue entry.  The list-driven refresh pulls small entries (32 per warp): the
// resident CTAs then work within ~10 planes of each other and the sectors a stamped site gathers are
// still in L2 when the stamped sites of the neighbouring planes need them; with 256 per warp the CTAs
// were spread over ~77 planes (340 MB of cvox + pairop + T against 126 MB of L2).
__device__ __forceinline__ void compact_cta_loop(const CompactArgs &a, CompactSmem &sm, int s_lo, int n, const int32_t *list,
                                                 unsigned int *queue, int CHUNK)
{
    for (int q = threadIdx.x; q < RT_TABLE_DOUBLES; q += blockDim.x) sm.tab[q] = a.tab[q];
    if (threadIdx.x < 14)
        sm.lin[threadIdx.x] = ((int)c_nb_off[threadIdx.x][0] * a.L + c_nb_off[threadIdx.x][1]) * a.L + c_nb_off[threadIdx.x][2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int CTA_CHUNK = CHUNK * RT_WARPS;
    if (threadIdx.x == 0) sm.chunk[0] = atomicAdd(queue, 1u);
    __syncthreads();
    for (int it = 0;; ++it) {
        const int64_t c0 = (int64_t)sm.chunk[it & 1] * CTA_CHUNK;
        if (c0 >= n) break;
        if (threadIdx.x == 0) sm.chunk[(it + 1) & 1] = atomicAdd(queue, 1u);      // the next chunk, popped ahead of need
        const int hi = (int)(c0 + CTA_CHUNK < n ? c0 + CTA_CHUNK : n);
        for (int q0 = (int)c0 + 32 * wid; q0 < hi; q0 += 32 * RT_WARPS) {
            const bool active = q0 + lane < hi;
            const int s = active ? (list ? list[q0 + lane] : s_lo + q0 + lane) : 0;
            compact_tile(a, sm, sm.w[wid], s, active);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(RT_THREADS, 4) dirty_eval_compact_kernel(const __grid_constant__ CompactArgs a, const int32_t *list,
                                                                           const unsigned int *n_list, unsigned int *queue)
{
    extern __shared__ __align__(16) unsigned char rate_dyn_smem[];
    compact_cta_loop(a, *reinterpret_cast<CompactSmem *>(rate_dyn_smem), 0, (int)*n_list, list, queue, a.chunk);
}

// Dense pass over local sites [s_lo, s_hi) on the compact tile state (the rebuild after a thermal step).
__global__ void __launch_bounds__(RT_THREADS, 5) rates_compact_kernel(const __grid_constant__ CompactArgs a, int s_lo, int s_hi,
                                                                      unsigned int *queue)
{
    extern __shared__ __align__(16) unsigned char rate_dyn_smem[];
    compact_cta_loop(a, *reinterpret_cast<CompactSmem *>(rate_dyn_smem), s_lo, s_hi - s_lo, nullptr, queue, RT_CHUNK);
}

static int compact_args(cet_ctx *c, CompactArgs &a)
{
    if (int rc = rate_tables_ensure(c)) return rc;
    if (!c->compact_attr_set) {
        CET_CUDA(cudaFuncSetAttribute(dirty_eval_compact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CompactSmem)));
        CET_CUDA(cudaFuncSetAttribute(rates_compact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CompactSmem)));
        c->compact_attr_set = true;
    }
    a.cvox = c->cvox; a.pairop = c->pairop; a.T = c->T;
    a.site_rate = c->site_rate; a.dep_rate = c->dep_rate; a.tab = c->rate_tab;
    a.P = c->rp;
    a.L = (int)c->n1; a.n0 = (int)c->n0; a.i_off = (int)(c->i_begin - c->halo); a.nloc = (int)c->nloc;
    const int64_t top = c->n0 - 1 - (c->i_begin - c->halo);
    if (top >= 0 && top < c->np) { a.top_lo = (int)(top * c->plane); a.top_hi = (int)((top + 1) * c->plane); }
    else { a.top_lo = 0; a.top_hi = 0; }
    a.chunk = ((c->debug_flags >> 8) & 0xff) ? 32 * ((c->debug_flags >> 8) & 0xff) : 64;      // measured at 512^3: 0.641 / 0.631 / 0.671 / 0.734 ms for 32 / 64 / 128 / 256
    return 0;
}

// Dense evaluation of local planes [p_lo, p_hi) from cvox / pairop.
int rates_rows_compact(cet_ctx *c, int p_lo, int p_hi)
{
    if (p_hi <= p_lo) return 0;
    CompactArgs a;
    if (int rc = compact_args(c, a)) return rc;
    const int s_lo = (int)(p_lo * c->plane), s_hi = (int)(p_hi * c->plane);
    unsigned int *queue = (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES);
    CET_CUDA(cudaMemsetAsync(queue, 0, sizeof(unsigned int), c->stream));
    const int grid = (int)std::min<int64_t>(((int64_t)s_hi - s_lo + RT_CHUNK * RT_WARPS - 1) / (RT_CHUNK * RT_WARPS),
                                            (int64_t)sm_count(c) * 5);
    rates_compact_kernel<<<grid, RT_THREADS, sizeof(CompactSmem), c->stream>>>(a, s_lo, s_hi, queue);
    CET_CUDA(cudaGetLastError());
    return 0;
}

static DirtyArgs dirty_args(const cet_ctx *c, int p_lo, int p_hi, const uint32_t *stamp, int32_t *list, unsigned int *counter)
{
    DirtyArgs d;
    d.stamp = stamp; d.s_lo = (int)(p_lo * c->plane); d.s_hi = (int)(p_hi * c->plane);
    d.list = list; d.n_list = counter;
    return d;
}

// Re-evaluate, on local planes [p_lo, p_hi), the sites whose stamp bit is set — from cvox / pairop.
int rates_rows_dirty_compact(cet_ctx *c, int p_lo, int p_hi, const uint32_t *stamp, int32_t *list, unsigned int *counter)
{
    if (p_hi <= p_lo) return 0;
    CompactArgs a;
    if (int rc = compact_args(c, a)) return rc;
    const DirtyArgs d = dirty_args(c, p_lo, p_hi, stamp, list, counter);
    const int n_words = ((d.s_hi + 31) >> 5) - (d.s_lo >> 5);
    dirty_scan_kernel<<<(n_words + RB_WARPS * 32 - 1) / (RB_WARPS * 32), RB_WARPS * 32, 0, c->stream>>>(d);
    CET_CUDA(cudaGetLastError());
    const int64_t nsite = (int64_t)(p_hi - p_lo) * c->plane;
    // evaluation: the class-sorted kernel of rates_refresh.cu; debug flag 262144 runs the pair-compacting kernel below
    if (!(c->debug_flags & 262144)) return rates_refresh_list(c, list, counter, nsite);
    const int grid = (int)std::min<int64_t>((nsite + RT_CHUNK * RT_WARPS - 1) / (RT_CHUNK * RT_WARPS), (int64_t)sm_count(c) * 4);   // 4 resident CTAs per SM: measured 0.74 ms per sweep at 512^3 against 0.85 (5), 0.81 (3), 1.46 (6) — the gathers live on the L1 the CTAs leave free
    unsigned int *queue = (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES) + 1;
    CET_CUDA(cudaMemsetAsync(queue, 0, sizeof(unsigned int), c->stream));
    dirty_eval_compact_kernel<<<grid, RT_THREADS, sizeof(CompactSmem), c->stream>>>(a, list, counter, queue);
    CET_CUDA(cudaGetLastError());
    return 0;
}

// rates_rows_dirty_compact for a group of contexts of one L (grouped sweeps, sweep.cu): one scan launch, then one
// refresh launch, on the stream of cs[0].  Every context's refresh queue has been cleared by the sweep's reset.
template <int CAP>
static int dirty_scan_group(cet_ctx *const *cs, int n, int p_lo, int p_hi)
{
    GroupArgs<DirtyArgs, CAP> g;
    for (int q = 0; q < n; ++q) g.a[q] = dirty_args(cs[q], p_lo, p_hi, cs[q]->stamp, cs[q]->dirty, &cs[q]->sweep->n_dirty);
    const int n_words = ((g.a[0].s_hi + 31) >> 5) - (g.a[0].s_lo >> 5);
    dirty_scan_group_kernel<CAP><<<dim3((unsigned)((n_words + RB_WARPS * 32 - 1) / (RB_WARPS * 32)), 1, (unsigned)n), RB_WARPS * 32, 0,
                                   cs[0]->stream>>>(g);
    CET_CUDA(cudaGetLastError());
    return 0;
}
int rates_rows_dirty_compact_group(cet_ctx *const *cs, int n, int p_lo, int p_hi, int *refresh_blocks)
{
    if (p_hi <= p_lo) return 0;
    if (int rc = n <= 16 ? dirty_scan_group<16>(cs, n, p_lo, p_hi) : dirty_scan_group<GROUP_MAX>(cs, n, p_lo, p_hi)) return rc;
    return rates_refresh_list_group(cs, n, (int64_t)(p_hi - p_lo) * cs[0]->plane, refresh_blocks);
}

// One warp per local plane: plane-segment sums in list order.
__global__ void seg_kernel(const double *row_occ, const double *row_emp, const double *row_dep,
                           double *seg, int n1, int p_lo, int p_hi, int i_off, int n0)
{
    const int p = p_lo + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= p_hi) return;
    const double so = warp_strided_sum(row_occ + (int64_t)p * n1, n1);
    const double se = warp_strided_sum(row_emp + (int64_t)p * n1, n1);
    const double sd = (i_off + p == n0 - 1) ? warp_strided_sum(row_dep, n1) : 0.0;
    if ((threadIdx.x & 31) == 0) { seg[3 * p + 0] = sd; seg[3 * p + 1] = so; seg[3 * p + 2] = se; }
}

__global__ void total_kernel(const double *seg, const int32_t *row_depcnt, double *total, int p_lo,
                             int p_hi, int n1, int has_top)
{
    __shared__ double sm[40];
    __shared__ long long smi[40];
    const double t = block_sum(seg + 3 * p_lo, 3 * (p_hi - p_lo), sm);
    const long long nd = has_top ? block_sum_i(row_depcnt, n1, smi) : 0;
    if (threadIdx.x == 0) { total[0] = t; ((long long *)total)[1] = nd; }
}

// Dense evaluation of local planes [p_lo, p_hi): site_rate and (on the global top plane) dep_rate.
int rates_rows(cet_ctx *c, int p_lo, int p_hi)
{
    CET_REQUIRE(c->cubic, "rates: context was created with cet_create_shape (thermal only)");
    CET_REQUIRE(c->have_rp, "rates: cet_set_rate_params has not been called");
    if (p_hi <= p_lo) return 0;
    CET_REQUIRE(c->nloc < (1ll << 31), "rates: the local lattice must have fewer than 2^31 sites");
    if (int rc = nst_ensure(c)) return rc;
    if (int rc = rate_tables_ensure(c)) return rc;
    const RateTileArgs a = tile_args(c);
    const int s_lo = (int)(p_lo * c->plane), s_hi = (int)(p_hi * c->plane);
    {
        ProfScope ps(c, PROF_RATES);
        unsigned int *queue = (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES);
        CET_CUDA(cudaMemsetAsync(queue, 0, sizeof(unsigned int), c->stream));
        const int grid = (int)std::min<int64_t>(((int64_t)s_hi - s_lo + RT_CHUNK * RT_WARPS - 1) / (RT_CHUNK * RT_WARPS),
                                                (int64_t)sm_count(c) * 5);
        rates_tile_kernel<5><<<grid, RT_THREADS, sizeof(RateSmem), c->stream>>>(a, s_lo, s_hi, queue);
    }
    CET_CUDA(cudaGetLastError());
    return 0;
}

// Re-evaluate, on local planes [p_lo, p_hi), the sites whose stamp bit is set.
// list: nloc int32; counter: one device unsigned int (zeroed by the caller).
int rates_rows_dirty(cet_ctx *c, int p_lo, int p_hi, const uint32_t *stamp, int32_t *list, unsigned int *counter)
{
    if (p_hi <= p_lo) return 0;
    if (int rc = nst_ensure(c)) return rc;
    if (int rc = rate_tables_ensure(c)) return rc;
    DirtyArgs d;
    d.stamp = stamp; d.s_lo = (int)(p_lo * c->plane); d.s_hi = (int)(p_hi * c->plane);
    d.list = list; d.n_list = counter;
    const int n_words = ((d.s_hi + 31) >> 5) - (d.s_lo >> 5);
    dirty_scan_kernel<<<(n_words + RB_WARPS * 32 - 1) / (RB_WARPS * 32), RB_WARPS * 32, 0, c->stream>>>(d);
    CET_CUDA(cudaGetLastError());
    const int64_t nsite = (int64_t)(p_hi - p_lo) * c->plane;
    const int grid = (int)std::min<int64_t>((nsite + RT_CHUNK * RT_WARPS - 1) / (RT_CHUNK * RT_WARPS), (int64_t)sm_count(c) * 5);
    unsigned int *queue = (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES) + 1;
    CET_CUDA(cudaMemsetAsync(queue, 0, sizeof(unsigned int), c->stream));
    dirty_eval_kernel<<<grid, RT_THREADS, sizeof(RateSmem), c->stream>>>(tile_args(c), list, counter, queue);
    CET_CUDA(cudaGetLastError());
    return 0;
}

int rates_build(cet_ctx *c)
{
    const int p_lo = c->halo, p_hi = (int)(c->np - c->halo);
    if (int rc = rates_rows(c, p_lo, p_hi)) return rc;
    const int i_off = (int)(c->i_begin - c->halo);
    RowSumArgs r;
    r.vox = c->vox; r.site_rate = c->site_rate; r.dep_rate = c->dep_rate;
    r.row_occ = c->row_occ; r.row_emp = c->row_emp; r.row_dep = c->row_dep; r.row_depcnt = c->row_depcnt;
    r.L = (int)c->n1; r.p_lo = p_lo; r.p_hi = p_hi;
    r.top_plane = (c->n0 - 1 - i_off >= p_lo && c->n0 - 1 - i_off < p_hi) ? (int)(c->n0 - 1 - i_off) : -1;
    const int nrows = (p_hi - p_lo) * (int)c->n1;
    row_sums_kernel<<<(nrows + RB_WARPS - 1) / RB_WARPS, RB_WARPS * 32, 0, c->stream>>>(r);
    CET_CUDA(cudaGetLastError());
    const int npl = p_hi - p_lo;
    seg_kernel<<<(npl + 3) / 4, 128, 0, c->stream>>>(c->row_occ, c->row_emp, c->row_dep, c->seg, (int)c->n1,
                                                     p_lo, p_hi, i_off, (int)c->n0);
    CET_CUDA(cudaGetLastError());
    total_kernel<<<1, 256, 0, c->stream>>>(c->seg, c->row_depcnt, c->total, p_lo, p_hi, (int)c->n1,
                                           c->i_end == c->n0 ? 1 : 0);
    CET_CUDA(cudaGetLastError());
    c->rates_valid = true;
    if (c->halo == 0) c->sweep_rates_valid = true;
    return 0;
}

// ---------------------------------------------------------------------------------------
// Legacy event list (kmc_event_rates.py:162-176 return value) as SoA, reference order.
// ---------------------------------------------------------------------------------------
struct ExportArgs {
    Lat g;
    cet_rate_params P;
    int p_lo;
    long long *plane_counts;      // [3 * planes]: dep, occ, emp event counts
    const long long *plane_base;  // [3 * planes]: first list index of each segment
    const double *species;        // device copy of the species draws (may be NULL)
    long long n_species;
    long long cap;
    uint8_t *type; long long *pos; double *rate; long long *target; int32_t *atom;
};

__device__ __forceinline__ int block_excl_scan_i(int v, int *smem, int *total)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) smem[w] = inc;
    __syncthreads();
    if (w == 0) {
        int t = lane < nw ? smem[lane] : 0, ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += u;
        }
        if (lane < nw) smem[lane] = ti - t;
        if (lane == 31) smem[32] = ti;
    }
    __syncthreads();
    *total = smem[32];
    return smem[w] + inc - v;
}

// One CTA per plane.  WRITE=false counts the events of the three segments; WRITE=true writes
// them at plane_base + rank-in-segment.
template <bool WRITE>
__global__ void __launch_bounds__(256) export_kernel(const ExportArgs a)
{
    __shared__ int sm[40];
    const int L = a.g.L;
    const int pl = blockIdx.x, p = a.p_lo + pl, i = a.g.i_off + p;
    const int64_t LL = (int64_t)L * L;
    const int nsite = L * L;
    for (int segm = 0; segm < 3; ++segm) {
        if (segm == 0 && i != a.g.n0 - 1) {
            if (!WRITE && threadIdx.x == 0) a.plane_counts[3 * pl] = 0;
            continue;
        }
        long long run = 0;
        for (int c0 = 0; c0 < nsite; c0 += blockDim.x) {
            const int q = c0 + threadIdx.x;
            const int j = q / L, k = q % L;
            int cnt = 0;
            double drate = 0.0;
            bool mine = false;
            if (q < nsite) {
                const int st = vox_state(a.g.vox[a.g.idx(i, j, k)]);
                if (segm == 0) {
                    if (st == 0 && dep_rate(a.P, a.g.T[a.g.idx(i, j, k)], &drate)) cnt = 1;
                } else {
                    mine = (segm == 1) ? (st != 0) : (st == 0);
                    if (mine) site_rate_sum(a.g, a.P, i, j, k, &cnt);
                }
            }
            int tot;
            const int off = block_excl_scan_i(cnt, sm, &tot);
            if (WRITE && cnt > 0) {
                long long e = a.plane_base[3 * pl + segm] + run + off;
                const long long self = (long long)i * LL + (long long)j * L + k;
                if (segm == 0) {
                    if (e < a.cap) {
                        const long long di = run + off;   // index into the species stream
                        int atom = a.P.states_w;
                        if (a.species && di < a.n_species) atom = dep_species(a.P, a.species[di]);
                        a.type[e] = CET_EV_DEP; a.pos[e] = self; a.rate[e] = drate; a.target[e] = -1;
                        a.atom[e] = atom;
                    }
                } else {
                    site_events(a.g, a.P, i, j, k, [&](int ty, int slot, double r, int atom) {
                        if (e < a.cap) {
                            a.type[e] = (uint8_t)ty; a.pos[e] = self; a.rate[e] = r;
                            a.target[e] = slot < 0 ? -1
                                                   : self + CET_NB_DI(slot) * LL + CET_NB_DJ(slot) * L + CET_NB_DK(slot);
                            a.atom[e] = atom;
                        }
                        ++e;
                    });
                }
            }
            run += tot;
        }
        if (!WRITE && threadIdx.x == 0) a.plane_counts[3 * pl + segm] = run;
    }
}

}  // namespace cet

using namespace cet;

extern "C" {

int cet_rates_build(cet_ctx *c)
{
    CET_REQUIRE(c, "cet_rates_build: NULL ctx");
    cet::DeviceGuard dg(c->device);
    return rates_build(c);
}

int cet_rates_total(cet_ctx *c, double *total, int64_t *n_dep)
{
    CET_REQUIRE(c, "cet_rates_total: NULL ctx");
    CET_REQUIRE(c->rates_valid, "cet_rates_total: rates are stale (call cet_rates_build)");
    cet::DeviceGuard dg(c->device);
    double h[2];
    CET_CUDA(cudaMemcpyAsync(h, c->total, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    if (total) *total = h[0];
    if (n_dep) memcpy(n_dep, &h[1], 8);
    return 0;
}

int cet_rates_download(cet_ctx *c, double *site_rate, double *dep_rate)
{
    CET_REQUIRE(c, "cet_rates_download: NULL ctx");
    CET_REQUIRE(c->rates_valid || c->sweep_rates_valid, "cet_rates_download: rates are stale (call cet_rates_build)");
    cet::DeviceGuard dg(c->device);
    if (site_rate)
        CET_CUDA(cudaMemcpyAsync(site_rate, c->site_rate + c->owned_offset(), (size_t)c->owned_sites() * 8,
                                 cudaMemcpyDeviceToHost, c->stream));
    if (dep_rate) {
        CET_REQUIRE(c->i_end == c->n0, "cet_rates_download: this slab does not own the top plane");
        CET_CUDA(cudaMemcpyAsync(dep_rate, c->dep_rate, (size_t)c->plane * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

static int export_counts(cet_ctx *c, ExportArgs &a, long long *h_counts, int npl)
{
    a.g = c->lat(); a.P = c->rp; a.p_lo = c->halo;
    if (int rc = ensure_stage(c, (size_t)npl * 6 * sizeof(long long))) return rc;
    a.plane_counts = (long long *)c->stage;
    a.plane_base = a.plane_counts + 3 * npl;
    export_kernel<false><<<npl, 256, 0, c->stream>>>(a);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(h_counts, a.plane_counts, (size_t)npl * 3 * sizeof(long long),
                             cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

int cet_events_count(cet_ctx *c, int64_t *n_events, int64_t *n_dep)
{
    CET_REQUIRE(c && c->cubic && c->have_rp, "cet_events_count: needs a cubic context with rate params");
    cet::DeviceGuard dg(c->device);
    const int npl = (int)(c->i_end - c->i_begin);
    long long *h = new long long[3 * npl];
    ExportArgs a;
    memset(&a, 0, sizeof(a));
    int rc = export_counts(c, a, h, npl);
    long long tot = 0, nd = 0;
    for (int q = 0; q < 3 * npl; ++q) { tot += h[q]; if (q % 3 == 0) nd += h[q]; }
    delete[] h;
    if (rc) return rc;
    if (n_events) *n_events = tot;
    if (n_dep) *n_dep = nd;
    return 0;
}

int cet_events_export(cet_ctx *c, const double *species_draws, int64_t n_draws, int64_t cap,
                      uint8_t *type, int64_t *pos, double *rate, int64_t *target, int32_t *atom,
                      int64_t *n_written)
{
    CET_REQUIRE(c && c->cubic && c->have_rp, "cet_events_export: needs a cubic context with rate params");
    CET_REQUIRE(cap >= 0, "cet_events_export: negative capacity");
    cet::DeviceGuard dg(c->device);
    const int npl = (int)(c->i_end - c->i_begin);
    long long *h = new long long[6 * npl];
    ExportArgs a;
    memset(&a, 0, sizeof(a));
    int rc = export_counts(c, a, h, npl);
    if (rc) { delete[] h; return rc; }
    long long run = 0;
    for (int q = 0; q < 3 * npl; ++q) { h[3 * npl + q] = run; run += h[q]; }
    const long long n = run < cap ? run : cap;
    if (n_written) *n_written = run;
    void *dbuf = nullptr, *dsp = nullptr;
    rc = 0;
    do {
        if (n == 0) break;
        if (cudaMemcpyAsync((void *)a.plane_base, h + 3 * npl, (size_t)npl * 3 * sizeof(long long),
                            cudaMemcpyHostToDevice, c->stream) != cudaSuccess) { rc = 1; break; }
        const size_t per = 1 + 8 + 8 + 8 + 4;
        if (cudaMalloc(&dbuf, (size_t)n * per + 64) != cudaSuccess) { rc = 1; break; }
        char *q = (char *)dbuf;
        a.pos = (long long *)q; q += (size_t)n * 8;
        a.rate = (double *)q; q += (size_t)n * 8;
        a.target = (long long *)q; q += (size_t)n * 8;
        a.atom = (int32_t *)q; q += (size_t)n * 4;
        a.type = (uint8_t *)q;
        a.cap = n;
        if (species_draws && n_draws > 0) {
            if (cudaMalloc(&dsp, (size_t)n_draws * 8) != cudaSuccess) { rc = 1; break; }
            if (cudaMemcpyAsync(dsp, species_draws, (size_t)n_draws * 8, cudaMemcpyHostToDevice, c->stream) !=
                cudaSuccess) { rc = 1; break; }
            a.species = (const double *)dsp; a.n_species = n_draws;
        }
        export_kernel<true><<<npl, 256, 0, c->stream>>>(a);
        if (cudaGetLastError() != cudaSuccess) { rc = 1; break; }
        cudaError_t e = cudaSuccess;
        if (pos) e = cudaMemcpyAsync(pos, a.pos, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream);
        if (!e && rate) e = cudaMemcpyAsync(rate, a.rate, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream);
        if (!e && target) e = cudaMemcpyAsync(target, a.target, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream);
        if (!e && atom) e = cudaMemcpyAsync(atom, a.atom, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream);
        if (!e && type) e = cudaMemcpyAsync(type, a.type, (size_t)n, cudaMemcpyDeviceToHost, c->stream);
        if (!e) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { rc = 1; break; }
    } while (0);
    if (rc) set_error("cet_events_export: CUDA failure: %s", cudaGetErrorString(cudaGetLastError()));
    if (dbuf) cudaFree(dbuf);
    if (dsp) cudaFree(dsp);
    delete[] h;
    return rc;
}

}  // extern "C"
