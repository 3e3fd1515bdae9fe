// rates_dense.cuh — the dense rate kernel's shared-memory layout, arguments and body (rates_dense.cu), shared by
// the solo kernel (rates_dense.cu) and the grouped kernel of cet_sweep_run_group (rates_dense_group.cu).  The two
// live in separate translation units so that the solo kernel's code generation is that of a module of its own.
#pragma once
#include <cuda.h>
#include <algorithm>
#include <utility>
#include "ctx.cuh"
#include "tile_state.cuh"
#include "tma.cuh"
#include "pair_walk.cuh"

namespace cet {

int rate_tables_ensure(cet_ctx *c);      // rates.cu
int tile_maps_ensure(cet_ctx *c);        // sweep_tile.cu
int sm_count(cet_ctx *c);

constexpr int DN_ROWS = TL_I * TL_J;                     // 32 rows of 32 sites per tile
constexpr int DN_WROWS = DN_ROWS / TL_WARPS;             // rows per warp in pass A
constexpr uint32_t DN_LISTED = 1u << 23;
constexpr int DN_INLINE_MIN = 12;                        // pass A evaluates pairless empty sites itself from this many per row on

struct DenseSmem {
    double po[TL_HI * TL_HJ * TL_PK];                    // 128-byte aligned TMA destinations first
    uint8_t vx[TL_VBYTES];
    double tab[RT_TABLE_DOUBLES];
    // the tile's sites as pass A staged them (index = tile-local site index li << 8 | lj << 5 | lk) ...
    uint64_t lw[TL_SITES];                               // class codes of the 14 neighbours, 4 bits per slot
    uint32_t lc[TL_SITES];                               // own cvox byte | sort key << 8 | rank within the key << 13 | DN_LISTED
    // ... and the order pass B walks them in: by class, then (SORT) by pair count — a trip costs its longest lane,
    // and unsorted only 17 of 32 lanes were busy in the pair loops
    uint16_t perm[TL_SITES + 32];
    int key_cnt[32], key_start[32];                      // sort key: class << 4 | pair count
    int n_slots;                                         // slots of perm in use (the first class padded to whole trips)
    int16_t dpb[16];                                     // [15 - o]: byte offset of neighbour slot o's pairop from the site's own
    unsigned long long bar;
    int4 tile[2];                                        // {tile index, p0, j0, k0} of this / the next iteration (popped ahead of need)
};

struct DenseArgs {
    const double *T;
    double *site_rate, *dep_rate;
    const double *tab;
    unsigned int *queue;
    cet_rate_params P;
    int L, p_lo, p_hi, top_plane;
    int njb, nkb, n_tiles;
};

template <int O>
__device__ __forceinline__ unsigned dn_code(uint32_t vaddr)
{
    return lds_u8<(CET_NB_DI(O) * TL_HJ + CET_NB_DJ(O)) * TL_VK + CET_NB_DK(O)>(vaddr) & 15u;
}
template <int... O>
__device__ __forceinline__ uint32_t dn_pack(uint32_t vaddr, int base, std::integer_sequence<int, O...>)
{
    return ((dn_code<O>(vaddr) << (4 * (O - base))) + ...);            // disjoint nibbles: + is |, and one LEA per slot
}
// The pairs of one site in slot order, out of line: the rare sites with an Arrhenius argument outside fast_exp's range.
template <bool ATT>
__device__ __noinline__ double dn_pairs_slow(const cet_rate_params &P, const double *tab, const int16_t *dpb, uint32_t m, uint32_t base, double A,
                                             double B, double sum)
{
    while (m) {
        const int h = 31 - __clz(m);
        m ^= 1u << h;
        const double op = lds_f64(base + (uint32_t)(int)dpb[h >> 1]);
        sum += ATT ? att_pair_rate_E(P, op, A, B, tab) : diff_pair_rate(P, A, B, op);
    }
    return sum;
}

// The pairs of one site in slot order.  m: pair_walk_mask; base: shared address of the site's own pairop;
// dpb: shared address of the offset table.  ILP pairs are in flight per trip.
template <bool ATT, int ILP>
__device__ __forceinline__ double dn_pairs(const cet_rate_params &P, const DenseSmem &sm, const uint32_t m0, uint32_t base, uint32_t dpb, double A,
                                           double B, const double sum0)
{
    uint32_t m = m0;
    double sum = sum0;
    int xmax = 0;                                                        // largest |Arrhenius argument| (high word) of the site
    do {
        double rate[ILP];
        bool on[ILP];
#pragma unroll
        for (int u = 0; u < ILP; ++u) {
            on[u] = u == 0 || m != 0u;
            const int h = (u == 0 || on[u]) ? 31 - __clz(m) : 0;         // FLO: position of the leading bit
            m &= (1u << h) - 1u;
            double op = 0.0;
            if (on[u]) op = lds_f64(base + (uint32_t)lds_s16(dpb + (uint32_t)h));
            rate[u] = pair_rate_raw<ATT>(P, sm.tab + RT_EXP2, op, A, B, xmax);
        }
#pragma unroll
        for (int u = 0; u < ILP; ++u)
            if (on[u]) add_kept(P, sum, rate[u]);
    } while (m);
    const bool bad = xmax >= EXP_RANGE_HI;                               // outside fast_exp's range
    if (ATT && bad) sum = dn_pairs_slow<ATT>(P, sm.tab + RT_EXP2, sm.dpb, m0, base, A, B, sum0);
    return sum;
}

// The kernel body takes its arguments and tensor maps by reference: the solo kernel passes its own parameters, the
// grouped kernel of cet_sweep_run_group the table entries of its lattice.
template <bool SORT>
__device__ __forceinline__ void rates_dense_body(const DenseArgs &a, const CUtensorMap &tm_vox, const CUtensorMap &tm_po)
{
    extern __shared__ unsigned char dense_dyn_smem[];
    DenseSmem &sm = *reinterpret_cast<DenseSmem *>(dense_dyn_smem + ((1024u - (smem_u32(dense_dyn_smem) & 1023u)) & 1023u));
    const cet_rate_params &P = a.P;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int L = a.L;
    const unsigned lt_mask = (1u << lane) - 1u;

    for (int q = tid; q < RT_TABLE_DOUBLES; q += TL_THREADS) sm.tab[q] = a.tab[q];
    if (tid < 14) sm.dpb[15 - tid] = (int16_t)((((int)c_nb_off[tid][0] * TL_HJ + c_nb_off[tid][1]) * TL_PK + c_nb_off[tid][2]) * 8);
    const int tiles_per_iblock = a.njb * a.nkb;
    // thread 0 pops a tile and works out its origin for everybody
    auto pop_tile = [&](int slot) {
        const int t = (int)atomicAdd(a.queue, 1u);
        const int ib = t / tiles_per_iblock, r = t - ib * tiles_per_iblock, jb = r / a.nkb, kb = r - jb * a.nkb;
        sm.tile[slot] = make_int4(t, a.p_lo + TL_I * ib, TL_J * jb, TL_K * kb);
    };
    if (tid == 0) {
        mbar_init(&sm.bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        pop_tile(0);
    }
    if (tid < 32) sm.key_cnt[tid] = 0;
    __syncthreads();
    const uint32_t vx0 = smem_u32(sm.vx), po0 = smem_u32(sm.po), dpb0 = smem_u32(sm.dpb);

    for (unsigned it = 0;; ++it) {
        const int4 ti = sm.tile[it & 1u];
        if (ti.x >= a.n_tiles) break;
        const int p0 = ti.y, j0 = ti.z, k0 = ti.w;
        if (tid == 0) {
            mbar_expect_tx(&sm.bar, (unsigned)(TL_VBYTES + TL_PBYTES));
            tma_load_3d(sm.vx, &tm_vox, &sm.bar, k0 - TL_VK0, j0 - 2, p0 - 2);
            tma_load_3d(sm.po, &tm_po, &sm.bar, k0 - TL_PK0, j0 - 2, p0 - 2);
            pop_tile((it + 1u) & 1u);                                    // read after the barrier that ends this tile
        }
        mbar_wait(&sm.bar, it & 1u);

        // ---- pass A: classify the warp's rows ------------------------------------------------------------
#pragma unroll 1
        for (int r = 0; r < DN_WROWS; ++r) {
            const int row = wid * DN_WROWS + r, li = row >> 3, lj = row & 7;
            const int p = p0 + li, j = j0 + lj, k = k0 + lane;
            const bool active = p < a.p_hi && j < L && k < L;
            const int rowbase = (li + 2) * TL_HJ + lj + 2;
            const uint32_t vaddr = vx0 + (uint32_t)(rowbase * TL_VK + TL_VK0 + lane);
            const unsigned c = lds_u8<0>(vaddr);
            const uint32_t wlo = dn_pack(vaddr, 0, std::integer_sequence<int, 0, 1, 2, 3, 4, 5, 6, 7>{});
            const uint32_t whi = dn_pack(vaddr, 8, std::integer_sequence<int, 8, 9, 10, 11, 12, 13>{});
            const unsigned code = c & 15u;
            const bool is_emp = active && code == TC_EMPTY;
            const bool is_occ = active && (code & 1u) && code != TC_DEFECT;
            const uint32_t att = (wlo & (wlo >> 3) & 0x11111111u) | (whi & (whi >> 3) & 0x00111111u);
            const uint32_t emp = (~wlo & (wlo >> 3) & 0x11111111u) | (~whi & (whi >> 3) & 0x00111111u);
            const bool to_diff = is_occ && emp != 0u;
            const int s = (p * L + j) * L + k;
            const uint64_t w = (uint64_t)wlo | ((uint64_t)whi << 32);
            // pairless empty sites: nucleation only.  Where they are most of the row they are evaluated here.
            const bool lone = is_emp && att == 0u;
            const bool inl = __popc(__ballot_sync(0xffffffffu, lone)) >= DN_INLINE_MIN;
            double T_self = 1.0;
            if (is_emp && (inl || p == a.top_plane)) T_self = lds_f64(po0 + (uint32_t)((rowbase * TL_PK + TL_PK0 + lane) * 8));
            const bool to_att = is_emp && !(lone && inl);
            if (active && !to_att && !to_diff) {
                double sum = 0.0;
                if (lone) {
                    const double local_T = pymax(T_self, 1.0);
                    sum = tile_nuc_rate(P, sm.tab, w, 0ull, local_T, rcp(P.kT * local_T));
                }
                a.site_rate[s] = sum;
            }
            if (p == a.top_plane && active) {                            // deposition (:55-72): top plane only
                double dep;
                a.dep_rate[j * L + k] = (is_emp && dep_rate(P, T_self, &dep)) ? dep : NAN;
            }
            // stage the site with its sort key and its rank within the key (one shared-memory atomic per distinct key of the warp)
            const bool listed = to_att || to_diff;
            const int np = to_att ? __popc(att) : __popc(emp);
            const int key = (to_att ? 0 : 16) + (SORT ? np : 0);
            const unsigned peers = __match_any_sync(0xffffffffu, listed ? key : -1);
            int rank = 0;
            if (listed) {
                const int leader = __ffs(peers) - 1;
                if (lane == leader) rank = atomicAdd(&sm.key_cnt[key], __popc(peers));
                rank = __shfl_sync(peers, rank, leader) + __popc(peers & lt_mask);
            }
            const int slot = row * 32 + lane;
            sm.lw[slot] = w;
            sm.lc[slot] = listed ? (c | ((uint32_t)key << 8) | ((uint32_t)rank << 13) | DN_LISTED) : 0u;
        }
        __syncthreads();
        // ---- counting sort: start of every key (the occupied class starts on a whole trip) ---------------------------
        if (wid == 0) {
            const int cnt = sm.key_cnt[lane];
            int inc = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += u;
            }
            const int n_emp_cls = __shfl_sync(0xffffffffu, inc, 15), pad = (32 - (n_emp_cls & 31)) & 31;
            sm.key_start[lane] = inc - cnt + (lane >= 16 ? pad : 0);
            sm.key_cnt[lane] = 0;                                        // for the next tile
            if (lane < pad) sm.perm[n_emp_cls + lane] = 0xFFFFu;
            if (lane == 31) sm.n_slots = inc + pad;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < DN_WROWS; ++r) {
            const int slot = (wid * DN_WROWS + r) * 32 + lane;
            const uint32_t e = sm.lc[slot];
            if (e & DN_LISTED) sm.perm[sm.key_start[(e >> 8) & 31u] + (int)((e >> 13) & 1023u)] = (uint16_t)slot;
        }
        __syncthreads();

        // ---- pass B: 32 sites per warp and trip; a trip runs one class and (SORT) mostly one pair count ------------------
        const int n_slots = sm.n_slots, nb_all = (n_slots + 31) >> 5;
#pragma unroll 1
        for (int b = wid; b < nb_all; b += TL_WARPS) {
            const int q = 32 * b + lane;
            unsigned slot = 0xFFFFu;
            if (q < n_slots) slot = sm.perm[q];
            const bool on = slot != 0xFFFFu;
            uint32_t e = 0;
            if (on) e = sm.lc[slot];
            const bool att_trip = __any_sync(0xffffffffu, on && !(e & (16u << 8)));       // a trip holds one class
            if (on) {
                const uint64_t w = sm.lw[slot];
                const int li = (slot >> 8) & 3, lj = (slot >> 5) & 7, lk = slot & 31;
                const int rowbase = (li + 2) * TL_HJ + lj + 2;
                const uint32_t base = po0 + (uint32_t)((rowbase * TL_PK + TL_PK0 + lk) * 8);
                const int k = k0 + lk;
                const int s = ((p0 + li) * L + j0 + lj) * L + k;
                if (att_trip) {                                          // empty sites: nucleation + attachment (kmc_event_rates.py:116-158)
                    const double T_self = lds_f64(base);                 // an empty site's pairop is its temperature
                    double T_m = T_self, T_p = T_self;
                    if ((uint32_t)w & 0x11111111u || (uint32_t)(w >> 32) & 0x00111111u) {     // an occupied neighbour: grad_z (:151-153)
                        const uint32_t vaddr = vx0 + (uint32_t)(rowbase * TL_VK + TL_VK0 + lk);
                        // an empty k neighbour keeps its temperature in pairop
                        if (k > 0) T_m = (lds_u8<-1>(vaddr) & 15u) == TC_EMPTY ? lds_f64(base - 8u) : a.T[s - 1];
                        if (k < L - 1) T_p = (lds_u8<1>(vaddr) & 15u) == TC_EMPTY ? lds_f64(base + 8u) : a.T[s + 1];
                    }
                    const TilePrep pr = tile_prep_emp(P, sm.tab, w, T_self, T_m, T_p);
                    a.site_rate[s] = pr.pm ? dn_pairs<true, 2>(P, sm, pair_walk_mask(pr.pm), base, dpb0, pr.A, pr.B, pr.sum0) : pr.sum0;
                } else {                                                 // occupied sites: diffusion (:79-109)
                    const unsigned c = e & 255u;
                    const TilePrep pr = tile_prep_occ(P, sm.tab, w, c & 15u, (int)(c >> 4), a.T[s]);
                    a.site_rate[s] = dn_pairs<false, 2>(P, sm, pair_walk_mask(pr.pm), base, dpb0, pr.A, pr.B, 0.0);
                }
            }
        }
        __syncthreads();                                           // the tile and the lists may be overwritten
    }
}
static inline DenseArgs dense_args(const cet_ctx *c, int p_lo, int p_hi)
{
    DenseArgs a;
    memset(&a, 0, sizeof(a));
    a.T = c->T; a.site_rate = c->site_rate; a.dep_rate = c->dep_rate; a.tab = c->rate_tab;
    a.queue = (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES) + 2;
    a.P = c->rp;
    a.L = (int)c->n1; a.p_lo = p_lo; a.p_hi = p_hi;
    const int top = (int)(c->n0 - 1 - (c->i_begin - c->halo));
    a.top_plane = (top >= p_lo && top < p_hi) ? top : -1;
    a.njb = (int)((c->n1 + TL_J - 1) / TL_J); a.nkb = (int)((c->n2 + TL_K - 1) / TL_K);
    a.n_tiles = ((p_hi - p_lo + TL_I - 1) / TL_I) * a.njb * a.nkb;
    return a;
}

}  // namespace cet
