// sweep_tile.cu — the tile kernel that keeps the resident rate sums current: neighbour-rate refresh
// after a sweep's events, and the dense rebuild after a thermal step.
//
// Per 4 x 8 x 32 tile of sites a CTA stages cvox + pairop (tile_state.cuh) with their halo of 2 in
// shared memory by two 3-D TMA loads (cp.async.bulk.tensor, completion on an mbarrier) and then
// re-evaluates the rate sum of every site whose stamp bit is set (the sites an event changed, and
// their neighbours) — or of every site — reading neighbour classes and pair operands from the tile.
// While the loads are in flight one warp turns the tile's stamp words into a list of its stamped
// sites.  Several CTAs share an SM, so one tile's loads run under another tile's arithmetic.
//
// This replaces the list-driven gather refresh of the first design (stamp scan + re-evaluation that
// touched ~15 DRAM sectors per refreshed site, 5.3 GB per sweep at 512^3 for 0.35 GB of information,
// plus an 8-byte neighbour-class cache per site that the gathers maintained): DRAM now sees one
// streaming read of cvox (1 B) and pairop (8 B) per site and the halo re-reads stay in L2.
//
// The pair arithmetic is the per-event code of site_rates.cuh (att_pair_rate_E / diff_pair_rate),
// the per-site half is tile_site_prep (tile_state.cuh), and a site adds its pairs in slot order, so
// the result equals site_rate_sum — and the dense kernel of rates.cu — bit for bit (tested).
#include <cuda.h>
#include <algorithm>
#include "ctx.cuh"
#include "reduce.cuh"
#include "tile_state.cuh"
#include "tma.cuh"

namespace cet {

int rate_tables_ensure(cet_ctx *c);      // rates.cu

constexpr int TL_PAIRS = 256;            // pair slots per warp (16 sites x 14 pairs fit: a fuller tile runs as two halves)

struct TileWarpSmem {
    double rate[TL_PAIRS];
    double A[32], B[32];
    uint32_t desc[TL_PAIRS];             // staged pairop index of the neighbour | owner lane << 14
};
// EVAL 0: pairs compacted across the warp (TileWarpSmem scratch); EVAL 1: every lane walks its own 14 slots
template <int EVAL>
struct TileSmem {
    double po[TL_HI * TL_HJ * TL_PK];            // 128-byte aligned TMA destinations first
    uint8_t vx[TL_VBYTES];
    double tab[RT_TABLE_DOUBLES];
    TileWarpSmem w[EVAL == 0 ? TL_WARPS : 1];
    uint16_t dlist[TL_SITES];
    int dp[16];                                  // staged pairop offset of neighbour slot o
    unsigned long long bar;
    unsigned int n_dirty;
};
static_assert((TL_PBYTES % 128) == 0 && (TL_VBYTES % 128) == 0, "TMA destinations must stay 128-byte aligned");

enum { TM_ALL = 1 };

struct TileArgs {
    const uint8_t *cvox;
    const double *pairop, *T;
    double *site_rate, *dep_rate;
    const uint32_t *stamp;
    SweepState *ss;
    const double *tab;
    cet_rate_params P;
    int L, n0, np, i_off;
    int p_lo, p_hi;              // evaluated local planes
    int top_plane;               // local plane of the global top plane, or -1
    int njb, nkb, n_tiles;
    int mode;
};

// What a lane knows about its site before the pair phase.
struct TileSite {
    TilePrep q;
    double T_self;
    int pidx, s;
};

// Per-site half: class codes of the 14 neighbours from the staged tile, temperatures, tile_site_prep.
// Tpre != nullptr: T[s-1], T[s], T[s+1] were loaded before the tile arrived (the trip's only global reads).
__device__ __forceinline__ TileSite tile_site(const TileArgs &a, const double *tab, const uint8_t *sv, const double *sp, int li,
                                              int lj, int lk, int p, int j, int k, bool active, const double *Tpre)
{
    TileSite r;
    const int vidx = ((li + 2) * TL_HJ + (lj + 2)) * TL_VK + lk + TL_VK0;
    r.pidx = ((li + 2) * TL_HJ + (lj + 2)) * TL_PK + lk + TL_PK0;
    r.s = (p * a.L + j) * a.L + k;
    unsigned c = 0;
    uint32_t wlo = 0, whi = 0;
    double T_self = 1.0, T_m = 1.0, T_p = 1.0;
    if (active) {
        c = sv[vidx];
#pragma unroll
        for (int o = 0; o < 8; ++o)
            wlo |= ((unsigned)sv[vidx + (CET_NB_DI(o) * TL_HJ + CET_NB_DJ(o)) * TL_VK + CET_NB_DK(o)] & 15u) << (4 * o);
#pragma unroll
        for (int o = 8; o < 14; ++o)
            whi |= ((unsigned)sv[vidx + (CET_NB_DI(o) * TL_HJ + CET_NB_DJ(o)) * TL_VK + CET_NB_DK(o)] & 15u) << (4 * (o - 8));
        const unsigned code = c & 15u;
        if (code == TC_EMPTY) {
            T_self = sp[r.pidx];                                     // an empty site's pairop is its temperature
            T_m = T_self; T_p = T_self;
            if ((wlo | whi) & 0x11111111u) {                         // an occupied neighbour: grad_z is needed (:151-153)
                if (k > 0) T_m = (sv[vidx - 1] & 15u) == TC_EMPTY ? sp[r.pidx - 1] : (Tpre ? Tpre[0] : a.T[r.s - 1]);
                if (k < a.L - 1) T_p = (sv[vidx + 1] & 15u) == TC_EMPTY ? sp[r.pidx + 1] : (Tpre ? Tpre[2] : a.T[r.s + 1]);
            }
        } else if ((code & 1u) && code != TC_DEFECT) {
            T_self = Tpre ? Tpre[1] : a.T[r.s];
        }
    }
    const uint64_t w = (uint64_t)wlo | ((uint64_t)whi << 32);
    r.q = tile_site_prep(a.P, tab, w, active ? c : 0u, T_self, T_m, T_p);
    r.T_self = T_self;
    return r;
}

__device__ __forceinline__ void tile_store(const TileArgs &a, const TileSite &t, double sum, int p, int j, int k)
{
    a.site_rate[t.s] = sum;
    if (p == a.top_plane) {                                          // deposition (:55-72)
        double dep;
        a.dep_rate[j * a.L + k] = (t.q.is_emp && dep_rate(a.P, t.T_self, &dep)) ? dep : NAN;
    }
}

// EVAL 0 — 32 sites per warp, their pairs compacted across the warp (all 32 lanes call).
__device__ __forceinline__ void tile_eval_packed(const TileArgs &a, const double *tab, const int *dp, TileWarpSmem &ws,
                                                 const uint8_t *sv, const double *sp, int li, int lj, int lk, int p, int j,
                                                 int k, bool active, const double *Tpre)
{
    const cet_rate_params &P = a.P;
    const int lane = threadIdx.x & 31;
    const TileSite t = tile_site(a, tab, sv, sp, li, lj, lk, p, j, k, active, Tpre);
    const uint64_t pm = t.q.pm;
    const bool is_emp = t.q.is_emp;
    if (pm) { ws.A[lane] = t.q.A; ws.B[lane] = t.q.B; }
    const int cnt = popc64(pm);
    // ---- packed counts: attachment pairs in the low half, diffusion pairs in the high half
    const unsigned mine = is_emp ? (unsigned)cnt : (unsigned)cnt << 16;
    const unsigned all = __reduce_add_sync(0xffffffffu, mine);
    double sum = t.q.sum0;
    const int npass = all == 0 ? 0 : (((all & 0xFFFFu) + (all >> 16) > (unsigned)TL_PAIRS) ? 2 : 1);
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
        const int start = is_emp ? (int)(excl & 0xFFFFu) : TL_PAIRS - (int)(excl >> 16) - cnt_p;
        if (part) {
            int pos = start;
            unsigned lo = (unsigned)pm, hi = (unsigned)(pm >> 32);
            const unsigned base = ((unsigned)lane << 14) + (unsigned)t.pidx;
            while (lo) {
                const int b = __ffs(lo) - 1;
                lo &= lo - 1;
                ws.desc[pos++] = base + (unsigned)dp[b >> 2];
            }
            while (hi) {
                const int b = __ffs(hi) - 1;
                hi &= hi - 1;
                ws.desc[pos++] = base + (unsigned)dp[8 + (b >> 2)];
            }
        }
        __syncwarp();
        // ---- pairs, 32 at a time: attachment from the front, diffusion from the back
        const int qd0 = TL_PAIRS - n_diff;
        for (int q0 = lane; q0 < n_att; q0 += 32) {                   // kmc_event_rates.py:135-158
            const unsigned d = ws.desc[q0];
            const int ts = d >> 14;
            ws.rate[q0] = att_pair_rate_E(P, sp[d & 0x3FFFu], ws.A[ts], ws.B[ts], tab + RT_EXP2);
        }
        for (int q0 = lane; q0 < n_diff; q0 += 32) {                  // :100-109
            const unsigned d = ws.desc[qd0 + q0];
            const int ts = d >> 14;
            ws.rate[qd0 + q0] = diff_pair_rate(P, ws.A[ts], ws.B[ts], sp[d & 0x3FFFu]);
        }
        __syncwarp();
        // ---- per-site sums in slot order (the association order of site_rate_sum)
        for (int q0 = 0; q0 < cnt_p; ++q0) sum += ws.rate[start + q0];
        __syncwarp();
    }
    if (active) tile_store(a, t, sum, p, j, k);
}

// EVAL 1 — every lane walks the 14 slots of its own site; neighbour offsets are immediates.
__device__ __forceinline__ void tile_eval_serial(const TileArgs &a, const double *tab, const uint8_t *sv, const double *sp, int li,
                                                 int lj, int lk, int p, int j, int k, bool active, const double *Tpre)
{
    const cet_rate_params &P = a.P;
    const TileSite t = tile_site(a, tab, sv, sp, li, lj, lk, p, j, k, active, Tpre);
    double sum = t.q.sum0;
    if (__any_sync(0xffffffffu, t.q.pm != 0)) {
        const bool is_emp = t.q.is_emp;
        const double A = t.q.A, B = t.q.B;
        const unsigned lo = (unsigned)t.q.pm, hi = (unsigned)(t.q.pm >> 32);
#pragma unroll
        for (int o = 0; o < 14; ++o) {
            const bool on = ((o < 8 ? lo >> (4 * o) : hi >> (4 * (o - 8))) & 1u) != 0;
            if (on) {
                const double op = sp[t.pidx + (CET_NB_DI(o) * TL_HJ + CET_NB_DJ(o)) * TL_PK + CET_NB_DK(o)];
                sum += is_emp ? att_pair_rate_E(P, op, A, B, tab + RT_EXP2) : diff_pair_rate(P, A, B, op);
            }
        }
    }
    if (active) tile_store(a, t, sum, p, j, k);
}

template <int STAGE, int EVAL>
__global__ void __launch_bounds__(TL_THREADS, EVAL == 0 ? 3 : 4)
    rates_tile3d_kernel(const __grid_constant__ TileArgs a, const __grid_constant__ CUtensorMap tm_vox,
                        const __grid_constant__ CUtensorMap tm_po)
{
    extern __shared__ unsigned char tile_dyn_smem[];
    TileSmem<EVAL> &sm = *reinterpret_cast<TileSmem<EVAL> *>(tile_dyn_smem + ((1024u - (smem_u32(tile_dyn_smem) & 1023u)) & 1023u));
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int L = a.L;

    for (int q = tid; q < RT_TABLE_DOUBLES; q += TL_THREADS) sm.tab[q] = a.tab[q];
    if (tid < 14) sm.dp[tid] = ((int)c_nb_off[tid][0] * TL_HJ + c_nb_off[tid][1]) * TL_PK + c_nb_off[tid][2];
    constexpr bool TMA = STAGE == 0;
    if (TMA && tid == 0) {
        mbar_init(&sm.bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int tiles_per_iblock = a.njb * a.nkb;
    const bool all = (a.mode & TM_ALL) != 0;
    constexpr int NH = (TL_I * TL_J + 31) / 32;
    // stamp words of a tile's rows (warp 0, one row per lane and h): loaded one tile ahead
    auto load_stamps = [&](int t, unsigned *bits) {
        const int kb = t % a.nkb, jb = (t / a.nkb) % a.njb, ib = t / tiles_per_iblock;
        const int p0 = a.p_lo + TL_I * ib, j0 = TL_J * jb, k0 = TL_K * kb;
#pragma unroll
        for (int h = 0; h < NH; ++h) {
            const int row = lane + 32 * h, p = p0 + (row >> 3), j = j0 + (row & 7);
            unsigned b = 0;
            if (t < a.n_tiles && row < TL_I * TL_J && p < a.p_hi && j < L && k0 < L) {
                const int s0 = (p * L + j) * L + k0;
                const unsigned w0 = a.stamp[s0 >> 5], w1 = a.stamp[(s0 >> 5) + 1];
                b = __funnelshift_r(w0, w1, s0 & 31);
                if (L - k0 < 32) b &= (1u << (L - k0)) - 1u;
            }
            bits[h] = b;
        }
    };
    unsigned next_bits[NH];
    if (!all && wid == 0) load_stamps((int)blockIdx.x, next_bits);
    unsigned int n_staged = 0;                  // tiles staged so far: the mbarrier's phase parity
    unsigned int n_refreshed = 0;
    for (int t = (int)blockIdx.x; t < a.n_tiles; t += (int)gridDim.x) {
        const int kb = t % a.nkb, jb = (t / a.nkb) % a.njb, ib = t / tiles_per_iblock;
        const int p0 = a.p_lo + TL_I * ib, j0 = TL_J * jb, k0 = TL_K * kb;
        if (TMA && tid == 0) {                                        // both boxes of the tile; one completion barrier
            mbar_expect_tx(&sm.bar, (unsigned)(TL_VBYTES + TL_PBYTES));
            tma_load_3d(sm.vx, &tm_vox, &sm.bar, k0 - TL_VK0, j0 - 2, p0 - 2);
            tma_load_3d(sm.po, &tm_po, &sm.bar, k0 - TL_PK0, j0 - 2, p0 - 2);
        }
        // ---- the tile's stamped sites, listed by warp 0 while the loads are in flight
        int spt = 32, e0 = 0;
        bool act0 = false;
        double Tpre[3] = {1.0, 1.0, 1.0};
        if (!all) {
            if (wid == 0) {
                unsigned bits[NH];
                int mine = 0;
#pragma unroll
                for (int h = 0; h < NH; ++h) { bits[h] = next_bits[h]; mine += __popc(bits[h]); }
                load_stamps(t + (int)gridDim.x, next_bits);           // the next tile's, used one iteration on
                int inc = mine;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int u = __shfl_up_sync(0xffffffffu, inc, d);
                    if (lane >= d) inc += u;
                }
                int pos = inc - mine;
#pragma unroll
                for (int h = 0; h < NH; ++h) {
                    unsigned b = bits[h];
                    const int row = lane + 32 * h;
                    while (b) {
                        const int e = __ffs(b) - 1;
                        b &= b - 1;
                        sm.dlist[pos++] = (uint16_t)(row * TL_K + e);
                    }
                }
                if (lane == 31) sm.n_dirty = (unsigned)inc;
            }
            __syncthreads();
            // a short list is dealt to all warps (fewer sites per trip: the trips are latency chains), and the
            // temperatures of the first trip are requested before the tile arrives
            const int n_d = (int)sm.n_dirty;
            if (n_d < 32 * TL_WARPS) {
                const int per = (n_d + TL_WARPS - 1) / TL_WARPS;
                spt = per <= 8 ? 8 : per <= 16 ? 16 : 32;
            }
            const int q = spt * wid + lane;
            act0 = lane < spt && q < n_d;
            if (act0) {
                e0 = (int)sm.dlist[q];
                const int p = p0 + (e0 >> 8), j = j0 + ((e0 >> 5) & 7), k = k0 + (e0 & 31);
                const int s = (p * L + j) * L + k;
                Tpre[1] = a.T[s];
                Tpre[0] = k > 0 ? a.T[s - 1] : Tpre[1];
                Tpre[2] = k < L - 1 ? a.T[s + 1] : Tpre[1];
            }
        }
        if (TMA) {
            mbar_wait(&sm.bar, n_staged & 1u);
        } else if (STAGE == 1) {
            // vector loads (L % 16 == 0): a warp copies whole rows of the tile, 16 bytes per lane; rows and
            // 16-byte chunks outside the lattice become zeros (class code 0 = outside)
            constexpr int ROWS = TL_HI * TL_HJ, PCH = TL_PK / 2, VCH = TL_VK / 16, VR = 32 / VCH;
#pragma unroll 4
            for (int row = wid; row < ROWS; row += TL_WARPS) {
                const int aa = row / TL_HJ, b = row - aa * TL_HJ;
                const int gp = p0 - 2 + aa, gj = j0 - 2 + b, gk = k0 - TL_PK0 + 2 * lane;
                if (lane < PCH) {
                    double2 val = make_double2(0.0, 0.0);
                    if (gp >= 0 && gp < a.np && gj >= 0 && gj < L && gk >= 0 && gk + 1 < L)
                        val = __ldg(reinterpret_cast<const double2 *>(a.pairop + ((int64_t)gp * L + gj) * L + gk));
                    *reinterpret_cast<double2 *>(sm.po + row * TL_PK + 2 * lane) = val;
                }
            }
#pragma unroll 2
            for (int r0 = wid * VR; r0 < ROWS; r0 += TL_WARPS * VR) {
                const int row = r0 + lane / VCH, ch = lane % VCH;
                const int aa = row / TL_HJ, b = row - aa * TL_HJ;
                const int gp = p0 - 2 + aa, gj = j0 - 2 + b, gk = k0 - TL_VK0 + 16 * ch;
                if (row < ROWS) {
                    uint4 val = make_uint4(0u, 0u, 0u, 0u);
                    if (gp >= 0 && gp < a.np && gj >= 0 && gj < L && gk >= 0 && gk + 15 < L)
                        val = __ldg(reinterpret_cast<const uint4 *>(a.cvox + ((int64_t)gp * L + gj) * L + gk));
                    *reinterpret_cast<uint4 *>(sm.vx + row * TL_VK + 16 * ch) = val;
                }
            }
        } else {
            // scalar loads (any L): zero outside the local array
            for (int q = tid; q < TL_VBYTES; q += TL_THREADS) {
                const int x = q % TL_VK, b = (q / TL_VK) % TL_HJ, aa = q / (TL_VK * TL_HJ);
                const int gp = p0 - 2 + aa, gj = j0 - 2 + b, gk = k0 - TL_VK0 + x;
                const bool in = gp >= 0 && gp < a.np && gj >= 0 && gj < L && gk >= 0 && gk < L;
                sm.vx[q] = in ? a.cvox[((int64_t)gp * L + gj) * L + gk] : (uint8_t)0;
            }
            for (int q = tid; q < TL_HI * TL_HJ * TL_PK; q += TL_THREADS) {
                const int x = q % TL_PK, b = (q / TL_PK) % TL_HJ, aa = q / (TL_PK * TL_HJ);
                const int gp = p0 - 2 + aa, gj = j0 - 2 + b, gk = k0 - TL_PK0 + x;
                const bool in = gp >= 0 && gp < a.np && gj >= 0 && gj < L && gk >= 0 && gk < L;
                sm.po[q] = in ? a.pairop[((int64_t)gp * L + gj) * L + gk] : 0.0;
            }
        }
        __syncthreads();
        const int n_eval = all ? TL_SITES : (int)sm.n_dirty;
        ++n_staged;
        // ---- up to 32 sites per warp and trip
        bool first = !all;
        for (int q0 = spt * wid; q0 < n_eval; q0 += spt * TL_WARPS) {
            const int q = q0 + lane;
            bool active = lane < spt && q < n_eval;
            const int e = active ? (all ? q : (first ? e0 : (int)sm.dlist[q])) : 0;
            const int li = e >> 8, lj = (e >> 5) & 7, lk = e & 31;
            const int p = p0 + li, j = j0 + lj, k = k0 + lk;
            if (all) active = active && p < a.p_hi && j < L && k < L;
            const double *tp = first ? Tpre : nullptr;
            if (EVAL == 0) tile_eval_packed(a, sm.tab, sm.dp, sm.w[wid], sm.vx, sm.po, li, lj, lk, p, j, k, active, tp);
            else tile_eval_serial(a, sm.tab, sm.vx, sm.po, li, lj, lk, p, j, k, active, tp);
            first = false;
        }
        if (!all) n_refreshed += (unsigned)n_eval;
        __syncthreads();                                       // the tile (and the list) may be overwritten
    }
    if (tid == 0 && n_refreshed) atomicAdd(&a.ss->n_dirty, n_refreshed);
}

// ---- resident tile state -----------------------------------------------------------------------
// cvox / pairop of local sites [s_lo, s_hi) from vox, T and the orientation vectors; planes outside the
// global lattice keep cvox = 0.  flag[0] is set when an empty site carries an orientation.
__global__ void tile_state_build_kernel(const uint8_t *__restrict__ vox, const Vec4 *__restrict__ v, const double *__restrict__ T,
                                        uint8_t *cvox, double *pairop, const cet_rate_params P, uint64_t lut, int64_t s_lo,
                                        int64_t s_hi, int *flag)
{
    for (int64_t s = s_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < s_hi; s += (int64_t)gridDim.x * blockDim.x) {
        const unsigned b = vox[s];
        const unsigned code = (unsigned)(lut >> (4 * (b & 15u))) & 15u;
        cvox[s] = (uint8_t)((b & 0xF0u) | code);
        double po = 0.0;
        if (code == TC_EMPTY) {
            const Vec4 u = v[s];
            if (!(u.x == 0.0 && u.y == 0.0 && u.z == 1.0)) *flag = 1;
            po = T[s];
        } else if ((code & 9u) == 9u) {
            po = tile_pairop(P, code, 0.0, v[s].z);
        }
        pairop[s] = po;
    }
}
// after a thermal step: the temperature half of pairop
__device__ __forceinline__ void tile_pairop_T_body(const uint8_t *__restrict__ cvox, const double *__restrict__ T, double *pairop,
                                                   int64_t s_lo, int64_t s_hi)
{
    for (int64_t s = s_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < s_hi; s += (int64_t)gridDim.x * blockDim.x)
        if ((cvox[s] & 15u) == TC_EMPTY) pairop[s] = T[s];
}
__global__ void tile_pairop_T_kernel(const uint8_t *__restrict__ cvox, const double *__restrict__ T, double *pairop, int64_t s_lo,
                                     int64_t s_hi)
{
    tile_pairop_T_body(cvox, T, pairop, s_lo, s_hi);
}
// grouped sweeps: grid (CTAs per lattice, lattices), whole-lattice contexts of one size
struct PairopTArgs {
    const uint8_t *cvox;
    const double *T;
    double *pairop;
};
template <int CAP>
__global__ void tile_pairop_T_group_kernel(const __grid_constant__ GroupArgs<PairopTArgs, CAP> g, int64_t n_sites)
{
    const PairopTArgs &a = g.a[blockIdx.y];
    tile_pairop_T_body(a.cvox, a.T, a.pairop, 0, n_sites);
}
// set the stamp bits of local sites [s_lo, s_hi)
__global__ void stamp_fill_kernel(uint32_t *stamp, int64_t s_lo, int64_t s_hi)
{
    const int64_t w_lo = s_lo >> 5, w_hi = (s_hi + 31) >> 5;
    for (int64_t w = w_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < w_hi; w += (int64_t)gridDim.x * blockDim.x) {
        uint32_t m = 0xffffffffu;
        if (w == w_lo) m &= 0xffffffffu << (s_lo & 31);
        if (w == w_hi - 1 && (s_hi & 31)) m &= 0xffffffffu >> (32 - (s_hi & 31));
        if (m == 0xffffffffu) stamp[w] = m;
        else atomicOr(&stamp[w], m);
    }
}

int sm_count(cet_ctx *c)
{
    if (c->n_sm <= 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, c->device) != cudaSuccess || n <= 0) n = 148;
        c->n_sm = n;
    }
    return c->n_sm;
}

// local planes that lie inside the global lattice
static void domain_planes(const cet_ctx *c, int *lo, int *hi)
{
    const int i_off = (int)(c->i_begin - c->halo), np = (int)c->np;
    *lo = i_off < 0 ? -i_off : 0;
    *hi = (i_off + np > c->n0) ? (int)(c->n0 - i_off) : np;
}

int tile_state_alloc(cet_ctx *c)
{
    if (!c->cvox) {
        CET_CUDA(cudaMalloc(&c->cvox, (size_t)c->nloc + 64));
        CET_CUDA(cudaMemsetAsync(c->cvox, 0, (size_t)c->nloc + 64, c->stream));
    }
    if (!c->pairop) {
        CET_CUDA(cudaMalloc(&c->pairop, (size_t)c->nloc * sizeof(double)));
        CET_CUDA(cudaMemsetAsync(c->pairop, 0, (size_t)c->nloc * sizeof(double), c->stream));
    }
    if (!c->tile_flag) CET_CUDA(cudaMalloc(&c->tile_flag, 64));
    return 0;
}

// Rebuild cvox / pairop on local planes [p_lo, p_hi) (clipped to the global lattice).
int tile_state_build(cet_ctx *c, int p_lo, int p_hi)
{
    if (int rc = tile_state_alloc(c)) return rc;
    int d_lo, d_hi;
    domain_planes(c, &d_lo, &d_hi);
    if (p_lo < d_lo) p_lo = d_lo;
    if (p_hi > d_hi) p_hi = d_hi;
    if (p_hi <= p_lo) return 0;
    const int64_t s_lo = (int64_t)p_lo * c->plane, s_hi = (int64_t)p_hi * c->plane;
    const int grid = (int)std::min<int64_t>((s_hi - s_lo + 255) / 256, (int64_t)sm_count(c) * 16);
    tile_state_build_kernel<<<grid, 256, 0, c->stream>>>(c->vox, c->v, c->T, c->cvox, c->pairop, c->rp, tile_code_lut(c->rp), s_lo,
                                                         s_hi, c->tile_flag);
    CET_CUDA(cudaGetLastError());
    return 0;
}

// Full rebuild + the check of the orientation invariant (one host read).
int tile_state_ensure(cet_ctx *c)
{
    if (c->tile_valid) return 0;
    if (int rc = tile_state_alloc(c)) return rc;
    CET_CUDA(cudaMemsetAsync(c->tile_flag, 0, sizeof(int), c->stream));
    if (int rc = tile_state_build(c, 0, (int)c->np)) return rc;
    int h = 0;
    CET_CUDA(cudaMemcpyAsync(&h, c->tile_flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    c->emp_canonical = h == 0;
    c->tile_valid = true;
    return 0;
}

int tile_pairop_T_update(cet_ctx *c)
{
    int d_lo, d_hi;
    domain_planes(c, &d_lo, &d_hi);
    const int64_t s_lo = (int64_t)d_lo * c->plane, s_hi = (int64_t)d_hi * c->plane;
    const int grid = (int)std::min<int64_t>((s_hi - s_lo + 255) / 256, (int64_t)sm_count(c) * 16);
    tile_pairop_T_kernel<<<grid, 256, 0, c->stream>>>(c->cvox, c->T, c->pairop, s_lo, s_hi);
    CET_CUDA(cudaGetLastError());
    return 0;
}

template <int CAP>
static int tile_pairop_T_group_launch(cet_ctx *const *cs, int n)
{
    GroupArgs<PairopTArgs, CAP> g;
    for (int q = 0; q < n; ++q) g.a[q] = PairopTArgs{cs[q]->cvox, cs[q]->T, cs[q]->pairop};
    const int64_t n_sites = cs[0]->nloc;
    const int per = (int)std::max<int64_t>(1, std::min<int64_t>((n_sites + 255) / 256, ((int64_t)sm_count(cs[0]) * 16 + n - 1) / n));
    tile_pairop_T_group_kernel<CAP><<<dim3((unsigned)per, (unsigned)n), 256, 0, cs[0]->stream>>>(g, n_sites);
    CET_CUDA(cudaGetLastError());
    return 0;
}
// tile_pairop_T_update for a group of whole-lattice contexts of one L (cet_sweep_run_group), on the stream of cs[0]
int tile_pairop_T_update_group(cet_ctx *const *cs, int n)
{
    if (n <= 0) return 0;
    return n <= 16 ? tile_pairop_T_group_launch<16>(cs, n) : tile_pairop_T_group_launch<GROUP_MAX>(cs, n);
}

int stamp_fill(cet_ctx *c, int p_lo, int p_hi)
{
    if (p_hi <= p_lo) return 0;
    const int64_t s_lo = (int64_t)p_lo * c->plane, s_hi = (int64_t)p_hi * c->plane;
    const int64_t nw = ((s_hi + 31) >> 5) - (s_lo >> 5);
    stamp_fill_kernel<<<(int)std::min<int64_t>((nw + 255) / 256, (int64_t)sm_count(c) * 8), 256, 0, c->stream>>>(c->stamp, s_lo,
                                                                                                                   s_hi);
    CET_CUDA(cudaGetLastError());
    return 0;
}

// ---- TMA descriptors -----------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
        (void)cudaGetLastError();
    }
    return fn;
}


// Tensor maps over the local arrays (k fastest, then j, then plane); rebuilt when a pointer changed.
int tile_maps_ensure(cet_ctx *c)
{
    if (c->tmap_vox_ptr == c->cvox && c->tmap_po_ptr == c->pairop) return 0;
    EncodeTiledFn enc = encode_tiled_fn();
    CET_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[3] = {(cuuint64_t)c->n2, (cuuint64_t)c->n1, (cuuint64_t)c->np};
    const cuuint32_t estr[3] = {1, 1, 1};
    {
        const cuuint64_t strides[2] = {(cuuint64_t)c->n2, (cuuint64_t)c->plane};
        const cuuint32_t box[3] = {TL_VK, TL_HJ, TL_HI};
        CUresult r = enc((CUtensorMap *)c->tmap_vox, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, c->cvox, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        CET_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(cvox) failed with CUresult %d", (int)r);
    }
    {
        const cuuint64_t strides[2] = {(cuuint64_t)c->n2 * 8, (cuuint64_t)c->plane * 8};
        const cuuint32_t box[3] = {TL_PK, TL_HJ, TL_HI};
        CUresult r = enc((CUtensorMap *)c->tmap_po, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, c->pairop, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        CET_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(pairop) failed with CUresult %d", (int)r);
    }
    c->tmap_vox_ptr = c->cvox; c->tmap_po_ptr = c->pairop;
    return 0;
}

// rows that a tensor map can describe (16-byte strides for the 1-byte array) and that fill a box
bool tile_tma_ok(const cet_ctx *c) { return c->n1 % 16 == 0 && c->n1 >= 64; }

template <int STAGE, int EVAL>
static int tile_launch(cet_ctx *c, const TileArgs &a, int *blocks_per_sm)
{
    const size_t smem = sizeof(TileSmem<EVAL>) + 1024;
    if (*blocks_per_sm == 0) {
        CET_CUDA(cudaFuncSetAttribute(rates_tile3d_kernel<STAGE, EVAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int nb = 0;
        CET_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rates_tile3d_kernel<STAGE, EVAL>, TL_THREADS, smem));
        CET_REQUIRE(nb >= 1, "rates_tile3d_kernel does not fit an SM");
        *blocks_per_sm = nb;
    }
    const int grid = std::min(a.n_tiles, sm_count(c) * *blocks_per_sm);
    if (STAGE == 0) {
        rates_tile3d_kernel<STAGE, EVAL><<<grid, TL_THREADS, smem, c->stream>>>(a, *(const CUtensorMap *)c->tmap_vox,
                                                                              *(const CUtensorMap *)c->tmap_po);
    } else {
        CUtensorMap dummy;
        memset(&dummy, 0, sizeof(dummy));
        rates_tile3d_kernel<STAGE, EVAL><<<grid, TL_THREADS, smem, c->stream>>>(a, dummy, dummy);
    }
    CET_CUDA(cudaGetLastError());
    return 0;
}

// One pass of the tile kernel over local planes [p_lo, p_hi): every site (all) or the stamped ones.
int tile_pass(cet_ctx *c, int p_lo, int p_hi, bool all)
{
    if (p_hi <= p_lo) return 0;
    if (int rc = rate_tables_ensure(c)) return rc;
    TileArgs a;
    memset(&a, 0, sizeof(a));
    a.cvox = c->cvox; a.pairop = c->pairop; a.T = c->T;
    a.site_rate = c->site_rate; a.dep_rate = c->dep_rate; a.stamp = c->stamp;
    a.ss = c->sweep; a.tab = c->rate_tab;
    a.P = c->rp;
    a.L = (int)c->n1; a.n0 = (int)c->n0; a.np = (int)c->np; a.i_off = (int)(c->i_begin - c->halo);
    a.p_lo = p_lo; a.p_hi = p_hi;
    const int top = (int)(c->n0 - 1 - (c->i_begin - c->halo));
    a.top_plane = (top >= p_lo && top < p_hi) ? top : -1;
    a.njb = (int)((c->n1 + TL_J - 1) / TL_J); a.nkb = (int)((c->n2 + TL_K - 1) / TL_K);
    a.n_tiles = ((p_hi - p_lo + TL_I - 1) / TL_I) * a.njb * a.nkb;
    a.mode = all ? TM_ALL : 0;
    // staging: 3-D TMA boxes when the rows allow it (L % 16 == 0), scalar loads otherwise; 16-byte vector
    // loads on request (debug flag 16; measured 2.7x slower than TMA for the same bytes, profiles/)
    const bool aligned = tile_tma_ok(c);
    const int stage = !aligned || (c->debug_flags & 1) ? 2 : (c->debug_flags & 16) ? 1 : 0;
    const bool serial = (c->debug_flags & 4) != 0;
    if (stage == 0) if (int rc = tile_maps_ensure(c)) return rc;
    int *bps = &c->tile_blocks[stage * 2 + (serial ? 1 : 0)];
    switch (stage * 2 + (serial ? 1 : 0)) {
        case 0: return tile_launch<0, 0>(c, a, bps);
        case 1: return tile_launch<0, 1>(c, a, bps);
        case 2: return tile_launch<1, 0>(c, a, bps);
        case 3: return tile_launch<1, 1>(c, a, bps);
        case 4: return tile_launch<2, 0>(c, a, bps);
        default: return tile_launch<2, 1>(c, a, bps);
    }
}

}  // namespace cet
