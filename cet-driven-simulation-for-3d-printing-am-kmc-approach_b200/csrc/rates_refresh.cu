// rates_refresh.cu — neighbour-rate refresh: re-evaluation of the stamped sites of a sweep (the sites an event
// changed, and their neighbours) from the compact tile state, list-driven.
//
// The list comes from dirty_scan_kernel (rates.cu) in lattice order.  The first compact refresh
// (dirty_eval_compact_kernel, kept as a tested variant) compacted the (site, slot) PAIRS of 32 sites across the
// warp through shared memory; ncu on the 512^3 benchmark: 1 550 warp instructions per 32 stamped sites, issue
// slots 56 % busy, L1 wavefronts 61 %, DRAM only 36 % — bound by what surrounds the arithmetic.  This kernel
// applies the structure of the dense kernel (rates_dense.cu) to gathered sites:
//   pass A  a lane reads the 15 class codes of its site straight from cvox (1-byte array: a warp's gathers fall
//           into a few 128-byte lines; in-bounds mask only when a lane of the warp sits within 2 sites of a lattice
//           face), packs them and classifies; sites without events store 0, the others go to the CTA's list of their
//           class (empty sites from the front, occupied sites from the back);
//   pass B  32 sites of ONE class per warp and trip: the pair operands of a lane's site are fetched by cp.async
//           (8 bytes each, no register staging) into the lane's column of the warp's shared-memory slab while the
//           per-site half (tile_prep_emp / tile_prep_occ) is computed; then the lane walks its operands in slot
//           order with the sum in a register (pair_walk.cuh).
// Same inline arithmetic as every other rate kernel: the result equals a dense rebuild bit for bit (tested).
#include <algorithm>
#include <memory>
#include "ctx.cuh"
#include "pair_walk.cuh"
#include "tile_state.cuh"

namespace cet {

int rate_tables_ensure(cet_ctx *c);      // rates.cu
int sm_count(cet_ctx *c);

constexpr int RF_THREADS = 256, RF_WARPS = RF_THREADS / 32;
// ROWS = 32-site rows per warp and chunk in pass A; a chunk (RF_WARPS * ROWS * 32 stamped sites) is what a CTA pops from
// the queue: small, so that the resident CTAs stay within a few planes of each other and share their sectors in L2
enum { RF_KM_EMPTY = 1u << 8, RF_KP_EMPTY = 1u << 9, RF_K_GT0 = 1u << 10, RF_K_LTL = 1u << 11 };

template <int ROWS>
struct RefreshSmem {
    static constexpr int RF_CHUNK = RF_WARPS * ROWS * 32;
    double op[RF_WARPS][14][32];                         // pair operands of the trip a warp is evaluating: [rank][lane]
    double tab[RT_TABLE_DOUBLES];
    uint64_t lw[RF_CHUNK];                               // class codes of the 14 neighbours, 4 bits per slot
    int32_t ls[RF_CHUNK];                                // local linear site index
    uint32_t lc[RF_CHUNK];                               // own cvox byte | RF_* flags
    int n_list[2][2];                                    // [chunk parity][att, diff] list lengths
    unsigned int chunk[2];
};

struct RefreshArgs {
    const uint8_t *cvox;
    const double *pairop, *T;
    double *site_rate, *dep_rate;
    const double *tab;
    const int32_t *list;
    const unsigned int *n_list;
    unsigned int *queue;
    cet_rate_params P;
    int L, n0, i_off;
    int top_lo, top_hi;
    unsigned int mLL, mL;                                // floor(2^32 / d) + 1: quotient estimates, one correction step
    int lin[14];
};

// n / d for 0 <= n < 2^31 with m = floor(2^32 / d) + 1: the estimate is the quotient or one above it
__device__ __forceinline__ int fast_div(int n, int d, unsigned int m, int *rem)
{
    int q = (int)__umulhi((unsigned int)n, m);
    int r = n - q * d;
    if (r < 0) { --q; r += d; }
    *rem = r;
    return q;
}
__device__ __forceinline__ void cp_async8(uint32_t dst, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

// The pairs of one site in slot order from the lane's operand column (rank r at opaddr + 256 r), out of line for the
// rare sites with an Arrhenius argument outside fast_exp's range.
template <bool ATT>
__device__ __noinline__ double rf_pairs_slow(const cet_rate_params &P, const double *tab, int cnt, uint32_t opaddr, double A, double B, double sum)
{
    for (int r = 0; r < cnt; ++r) {
        const double op = lds_f64(opaddr + 256u * (uint32_t)r);
        sum += ATT ? att_pair_rate_E(P, op, A, B, tab) : diff_pair_rate(P, A, B, op);
    }
    return sum;
}
template <bool ATT>
__device__ __forceinline__ double rf_pairs(const cet_rate_params &P, const double *exp_tab, int cnt, uint32_t opaddr, double A, double B,
                                           const double sum0)
{
    double sum = sum0;
    int xmax = 0;
    uint32_t addr = opaddr;
    for (int r = 0; r < cnt; r += 2, addr += 512u) {                    // two pairs in flight per trip
        const bool two = r + 1 < cnt;
        const double op0 = lds_f64(addr);
        double op1 = 0.0;
        if (two) op1 = lds_f64(addr + 256u);
        const double r0 = pair_rate_raw<ATT>(P, exp_tab, op0, A, B, xmax);
        const double r1 = pair_rate_raw<ATT>(P, exp_tab, op1, A, B, xmax);
        add_kept(P, sum, r0);
        if (two) add_kept(P, sum, r1);
    }
    if (ATT && xmax >= EXP_RANGE_HI) sum = rf_pairs_slow<ATT>(P, exp_tab, cnt, opaddr, A, B, sum0);
    return sum;
}

template <int ROWS>
__device__ __forceinline__ void rates_refresh_body(const RefreshArgs &a)
{
    constexpr int RF_CHUNK = RF_WARPS * ROWS * 32, RF_ROWS = ROWS;
    extern __shared__ __align__(16) unsigned char refresh_dyn_smem[];
    RefreshSmem<ROWS> &sm = *reinterpret_cast<RefreshSmem<ROWS> *>(refresh_dyn_smem);
    const cet_rate_params &P = a.P;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int L = a.L, LL = L * L;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int n = (int)*a.n_list;

    for (int q = tid; q < RT_TABLE_DOUBLES; q += RF_THREADS) sm.tab[q] = a.tab[q];
    if (tid == 0) {
        sm.chunk[0] = atomicAdd(a.queue, 1u);
        sm.n_list[0][0] = 0; sm.n_list[0][1] = 0;
    }
    __syncthreads();
    const uint32_t op0 = (uint32_t)__cvta_generic_to_shared(&sm.op[wid][0][lane]);

    for (unsigned it = 0;; ++it) {
        const int64_t c0 = (int64_t)sm.chunk[it & 1u] * RF_CHUNK;
        if (c0 >= n) break;
        int *n_list = sm.n_list[it & 1u];
        if (tid == 0) {
            sm.chunk[(it + 1u) & 1u] = atomicAdd(a.queue, 1u);            // the next chunk, popped ahead of need
            sm.n_list[(it + 1u) & 1u][0] = 0; sm.n_list[(it + 1u) & 1u][1] = 0;
        }
        const int hi = (int)(c0 + RF_CHUNK < n ? c0 + RF_CHUNK : n);

        // ---- pass A: gather the class codes, classify ---------------------------------------------------------
#pragma unroll
        for (int r = 0; r < RF_ROWS; ++r) {
            const int q = (int)c0 + 32 * (wid * RF_ROWS + r) + lane;
            const bool active = q < hi;
            const int s = active ? a.list[q] : 0;
            int rem, k;
            const int p = fast_div(s, LL, a.mLL, &rem), j = fast_div(rem, L, a.mL, &k);
            const int gi = a.i_off + p;
            const bool interior = (unsigned)(gi - 2) < (unsigned)(a.n0 - 4) && (unsigned)(j - 2) < (unsigned)(L - 4) &&
                                  (unsigned)(k - 2) < (unsigned)(L - 4);
            unsigned inb = 0x3FFFu;
            if (!__all_sync(0xffffffffu, interior || !active)) inb = inbounds_mask(gi, j, k, a.n0, L);
            const uint8_t *cs = a.cvox + s;
            unsigned c = 0, b[14], km = 0, kp = 0;
#pragma unroll
            for (int o = 0; o < 14; ++o) b[o] = 0;
            if (active) {
                c = cs[0];
                if (k > 0) km = cs[-1];
                if (k < L - 1) kp = cs[1];
#pragma unroll
                for (int o = 0; o < 14; ++o)
                    if (inb >> o & 1u) b[o] = cs[a.lin[o]];
            }
            uint32_t wlo = 0, whi = 0;
#pragma unroll
            for (int o = 0; o < 8; ++o) wlo += (b[o] & 15u) << (4 * o);
#pragma unroll
            for (int o = 8; o < 14; ++o) whi += (b[o] & 15u) << (4 * (o - 8));
            const unsigned code = c & 15u;
            const bool is_emp = active && code == TC_EMPTY;
            const bool is_occ = active && (code & 1u) && code != TC_DEFECT;
            const uint32_t emp = (~wlo & (wlo >> 3) & 0x11111111u) | (~whi & (whi >> 3) & 0x00111111u);
            const bool to_att = is_emp, to_diff = is_occ && emp != 0u;
            if (active && !to_att && !to_diff) {
                a.site_rate[s] = 0.0;
                if (s >= a.top_lo && s < a.top_hi) a.dep_rate[s - a.top_lo] = NAN;      // deposition needs an empty site (:55-72)
            }
            const unsigned b_att = __ballot_sync(0xffffffffu, to_att), b_diff = __ballot_sync(0xffffffffu, to_diff);
            if (b_att | b_diff) {
                int base_a = 0, base_d = 0;
                if (lane == 0) {
                    if (b_att) base_a = atomicAdd(&n_list[0], __popc(b_att));
                    if (b_diff) base_d = atomicAdd(&n_list[1], __popc(b_diff));
                }
                base_a = __shfl_sync(0xffffffffu, base_a, 0); base_d = __shfl_sync(0xffffffffu, base_d, 0);
                const uint32_t ent = c | ((km & 15u) == TC_EMPTY ? RF_KM_EMPTY : 0u) | ((kp & 15u) == TC_EMPTY ? RF_KP_EMPTY : 0u) |
                                     (k > 0 ? RF_K_GT0 : 0u) | (k < L - 1 ? RF_K_LTL : 0u);
                const uint64_t w = (uint64_t)wlo | ((uint64_t)whi << 32);
                int pos = -1;
                if (to_att) pos = base_a + __popc(b_att & lt_mask);
                if (to_diff) pos = RF_CHUNK - 1 - base_d - __popc(b_diff & lt_mask);
                if (pos >= 0) { sm.lw[pos] = w; sm.ls[pos] = s; sm.lc[pos] = ent; }
            }
        }
        __syncthreads();

        // ---- pass B: the lists, 32 sites per warp and trip; a trip runs one class ---------------------------------
        const int n_att = n_list[0], n_diff = n_list[1];
        const int nb_att = (n_att + 31) >> 5, nb_all = nb_att + ((n_diff + 31) >> 5);
#pragma unroll 1
        for (int bt = wid; bt < nb_all; bt += RF_WARPS) {
            const bool att = bt < nb_att;
            const int q = att ? 32 * bt + lane : 32 * (bt - nb_att) + lane;
            const bool on = q < (att ? n_att : n_diff);
            const int pos = att ? q : RF_CHUNK - 1 - q;
            uint64_t w = 0;
            uint32_t e = 0;
            int s = 0;
            if (on) { w = sm.lw[pos]; s = sm.ls[pos]; e = sm.lc[pos]; }
            // the site's pair mask and the operand gathers, issued before anything waits
            const uint64_t pm = !on ? 0ull : att ? (w & (w >> 3) & CET_NIB_LSB) : (~w & (w >> 3) & CET_NIB_LSB);
            // slot-major, so that the lanes of a warp — consecutive stamped sites, mostly neighbours along k — ask for
            // neighbouring addresses in the same instruction (a lane-major walk of the masks scatters them)
            const uint32_t pm_lo = (uint32_t)pm, pm_hi = (uint32_t)(pm >> 32);
            const int cnt = __popc(pm_lo) + __popc(pm_hi);
            {
                const double *src = a.pairop + s;
                uint32_t dst = op0;
#pragma unroll
                for (int o = 0; o < 14; ++o) {
                    if ((o < 8 ? pm_lo >> (4 * o) : pm_hi >> (4 * (o - 8))) & 1u) {
                        cp_async8(dst, src + a.lin[o]);
                        dst += 256u;
                    }
                }
            }
            if (att) {                                                   // empty sites: nucleation + attachment (kmc_event_rates.py:116-158)
                double T_self = 1.0, T_m = 1.0, T_p = 1.0;
                if (on) {
                    T_self = a.pairop[s];                                // an empty site's pairop is its temperature
                    T_m = T_self; T_p = T_self;
                    if (pm) {                                            // grad_z (:151-153); an empty k neighbour keeps its temperature in pairop
                        if (e & RF_K_GT0) T_m = (e & RF_KM_EMPTY) ? a.pairop[s - 1] : a.T[s - 1];
                        if (e & RF_K_LTL) T_p = (e & RF_KP_EMPTY) ? a.pairop[s + 1] : a.T[s + 1];
                    }
                }
                const TilePrep pr = tile_prep_emp(P, sm.tab, w, T_self, T_m, T_p);
                cp_async_wait_all();
                if (on) {
                    a.site_rate[s] = cnt ? rf_pairs<true>(P, sm.tab + RT_EXP2, cnt, op0, pr.A, pr.B, pr.sum0) : pr.sum0;
                    if (s >= a.top_lo && s < a.top_hi) {                 // deposition (:55-72): top plane only
                        double dep;
                        a.dep_rate[s - a.top_lo] = dep_rate(P, T_self, &dep) ? dep : NAN;
                    }
                }
            } else {                                                     // occupied sites: diffusion (:79-109)
                const double T_self = on ? a.T[s] : 1.0;
                const unsigned c = e & 255u;
                const TilePrep pr = tile_prep_occ(P, sm.tab, w, c & 15u, (int)(c >> 4), T_self);
                cp_async_wait_all();
                if (on) {
                    a.site_rate[s] = rf_pairs<false>(P, sm.tab + RT_EXP2, cnt, op0, pr.A, pr.B, 0.0);
                    if (s >= a.top_lo && s < a.top_hi) a.dep_rate[s - a.top_lo] = NAN;
                }
            }
        }
        __syncthreads();                                           // the lists may be overwritten
    }
}
template <int ROWS>
__global__ void __launch_bounds__(RF_THREADS, 4) rates_refresh_kernel(const __grid_constant__ RefreshArgs a) { rates_refresh_body<ROWS>(a); }
// grouped sweeps: grid (CTAs per lattice, 1, lattices); each lattice's CTAs pop chunks of its own list from its own queue
template <int ROWS, int CAP>
__global__ void __launch_bounds__(RF_THREADS, 4) rates_refresh_group_kernel(const __grid_constant__ GroupArgs<RefreshArgs, CAP> g)
{
    rates_refresh_body<ROWS>(g.a[blockIdx.z]);
}

template <int ROWS>
static int refresh_launch(cet_ctx *c, const RefreshArgs &a, int64_t nsite_hint, int *blocks_per_sm)
{
    constexpr int CHUNK = RF_WARPS * ROWS * 32;
    const size_t smem = sizeof(RefreshSmem<ROWS>);
    if (*blocks_per_sm == 0) {
        CET_CUDA(cudaFuncSetAttribute(rates_refresh_kernel<ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int nb = 0;
        CET_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rates_refresh_kernel<ROWS>, RF_THREADS, smem));
        CET_REQUIRE(nb >= 1, "rates_refresh_kernel does not fit an SM");
        *blocks_per_sm = nb;
    }
    const int grid = (int)std::min<int64_t>((nsite_hint + CHUNK - 1) / CHUNK, (int64_t)sm_count(c) * *blocks_per_sm);
    rates_refresh_kernel<ROWS><<<grid, RF_THREADS, smem, c->stream>>>(a);
    CET_CUDA(cudaGetLastError());
    return 0;
}

static RefreshArgs refresh_args(const cet_ctx *c, const int32_t *list, const unsigned int *counter)
{
    RefreshArgs a;
    memset(&a, 0, sizeof(a));
    a.cvox = c->cvox; a.pairop = c->pairop; a.T = c->T;
    a.site_rate = c->site_rate; a.dep_rate = c->dep_rate; a.tab = c->rate_tab;
    a.list = list; a.n_list = counter;
    a.queue = (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES) + 3;
    a.P = c->rp;
    a.L = (int)c->n1; a.n0 = (int)c->n0; a.i_off = (int)(c->i_begin - c->halo);
    const int64_t top = c->n0 - 1 - (c->i_begin - c->halo);
    if (top >= 0 && top < c->np) { a.top_lo = (int)(top * c->plane); a.top_hi = (int)((top + 1) * c->plane); }
    a.mLL = (unsigned int)((1ull << 32) / (uint64_t)c->plane) + 1u;
    a.mL = (unsigned int)((1ull << 32) / (uint64_t)c->n1) + 1u;
    for (int o = 0; o < 14; ++o) a.lin[o] = (h_nb_off[o][0] * a.L + h_nb_off[o][1]) * a.L + h_nb_off[o][2];
    return a;
}

// Re-evaluate the sites listed in `list` (length *counter, produced by dirty_scan_kernel) from cvox / pairop.
int rates_refresh_list(cet_ctx *c, const int32_t *list, const unsigned int *counter, int64_t nsite_hint)
{
    if (int rc = rate_tables_ensure(c)) return rc;
    const RefreshArgs a = refresh_args(c, list, counter);
    CET_CUDA(cudaMemsetAsync(a.queue, 0, sizeof(unsigned int), c->stream));
    // stamped sites per CTA and queue entry: 512 (default), 256 / 1024 by debug flag 1048576 / 2097152
    const int v = (c->debug_flags & 1048576) ? 0 : (c->debug_flags & 2097152) ? 2 : 1;
    if (v == 0) return refresh_launch<1>(c, a, nsite_hint, &c->refresh_blocks[0]);
    if (v == 2) return refresh_launch<4>(c, a, nsite_hint, &c->refresh_blocks[2]);
    return refresh_launch<2>(c, a, nsite_hint, &c->refresh_blocks[1]);
}

// rates_refresh_list for a group of contexts of one L (grouped sweeps): each context's stamped-site list and the
// queue its CTAs pop chunks from (cleared by the sweep's reset kernel); the list lengths are read on the device.
// The CTAs resident on the device are shared out evenly; which CTA evaluates a chunk does not change the result.
template <int CAP>
static int refresh_group_launch(cet_ctx *const *cs, int n, int64_t nsite_hint, int *blocks_per_sm)
{
    constexpr int ROWS = 2, CHUNK = RF_WARPS * ROWS * 32;
    const size_t smem = sizeof(RefreshSmem<ROWS>);
    static_assert(group_fits<RefreshArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");
    cet_ctx *c0 = cs[0];
    if (*blocks_per_sm == 0) {
        CET_CUDA(cudaFuncSetAttribute(rates_refresh_group_kernel<ROWS, CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int nb = 0;
        CET_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rates_refresh_group_kernel<ROWS, CAP>, RF_THREADS, smem));
        CET_REQUIRE(nb >= 1, "rates_refresh_group_kernel does not fit an SM");
        *blocks_per_sm = nb;
    }
    GroupArgs<RefreshArgs, CAP> g;
    for (int q = 0; q < n; ++q) g.a[q] = refresh_args(cs[q], cs[q]->dirty, &cs[q]->sweep->n_dirty);
    const int64_t per_ctx = std::max<int64_t>(1, ((int64_t)sm_count(c0) * *blocks_per_sm + n - 1) / n);
    const int grid = (int)std::min<int64_t>((nsite_hint + CHUNK - 1) / CHUNK, per_ctx);
    rates_refresh_group_kernel<ROWS, CAP><<<dim3((unsigned)grid, 1, (unsigned)n), RF_THREADS, smem, c0->stream>>>(g);
    CET_CUDA(cudaGetLastError());
    return 0;
}
// blocks_per_sm: the grouped kernel's occupancy, queried on first use (a group call keeps it for all its sweeps)
int rates_refresh_list_group(cet_ctx *const *cs, int n, int64_t nsite_hint, int *blocks_per_sm)
{
    return n <= 16 ? refresh_group_launch<16>(cs, n, nsite_hint, blocks_per_sm)
                   : refresh_group_launch<GROUP_MAX>(cs, n, nsite_hint, blocks_per_sm);
}

}  // namespace cet
