// cadence.cuh — device bodies of the metrics cadence: the defect-mask refresh (defects.cu), the state
// histogram (api_ctx.cu) and the grain labelling and statistics (grains.cu).  The solo kernels and the
// grouped kernels of cet_metrics_group (metrics_group.cu) run these bodies, so a mask, a histogram or a label
// has the same bits whichever path computed it.  A body takes its CTA's place from blockIdx.x / gridDim.x;
// a grouped kernel selects the lattice with another grid axis.
#pragma once
#include "ctx.cuh"
#include "reduce.cuh"

namespace cet {

// ---- defect mask (defects.py:4-31) ----

constexpr int DF_THREADS = 256, DF_PER_THREAD = 4, DF_TILE = DF_THREADS * DF_PER_THREAD;

__device__ __forceinline__ void philox_round10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

struct DefectArgs {
    uint8_t *vox;              // owned planes
    const double *T;
    int64_t n;                 // owned sites
    int64_t g_off;             // global linear index of the first owned site
    const double *draws;
    uint64_t seed;
    uint32_t epoch;
    int carbon_id, defect_id, apply_to_state;
    double base, e_mig, kT, T_default;
    unsigned int *tile_count;      // [n_tiles + 1]: counts, then exclusive offsets
    unsigned long long *totals;    // [0] carbon sites, [1] defects set
};

// pass 1: carbon sites per tile
__device__ __forceinline__ void defects_count_body(const DefectArgs &a)
{
    __shared__ int sm[DF_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * DF_TILE;
    int c = 0;
#pragma unroll
    for (int e = 0; e < DF_PER_THREAD; ++e) {
        const int64_t s = base + e * DF_THREADS + threadIdx.x;
        if (s < a.n && (a.vox[s] & 15) == a.carbon_id) ++c;
    }
    c = warp_sum_i(c);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < DF_THREADS / 32; ++w) t += sm[w];
        a.tile_count[blockIdx.x] = (unsigned)t;
    }
}

// pass 2: exclusive scan of the tile counts (one CTA of 1024 threads, sequential over 1024-entry strips);
// totals[0] receives the sum
__device__ __forceinline__ void tile_scan_body(unsigned int *tile_count, int n_tiles, unsigned long long *totals)
{
    __shared__ unsigned int sm[33];
    __shared__ unsigned long long run;
    if (threadIdx.x == 0) run = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int t0 = 0; t0 < n_tiles; t0 += 1024) {
        const int q = t0 + threadIdx.x;
        const unsigned v = q < n_tiles ? tile_count[q] : 0u;
        unsigned inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) sm[w] = inc;
        __syncthreads();
        if (w == 0) {
            unsigned x = sm[lane], xi = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, xi, d);
                if (lane >= d) xi += t;
            }
            sm[lane] = xi - x;
            if (lane == 31) sm[32] = xi;
        }
        __syncthreads();
        const unsigned long long r0 = run;
        if (q < n_tiles) tile_count[q] = (unsigned)(r0 + sm[w] + inc - v);      // < 2^32: fewer than 2^31 sites per context
        __syncthreads();
        if (threadIdx.x == 0) run = r0 + sm[32];
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[0] = run;
}

// pass 3: rewrite the mask nibble of every site
__device__ __forceinline__ void defects_assign_body(const DefectArgs &a)
{
    __shared__ int sm[DF_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * DF_TILE;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned run = a.draws ? a.tile_count[blockIdx.x] : 0u;     // C-order rank of the tile's first carbon site
    int set = 0;
    for (int e = 0; e < DF_PER_THREAD; ++e) {                   // strips of 256 consecutive sites keep C order
        const int64_t s = base + e * DF_THREADS + threadIdx.x;
        const uint8_t vb = s < a.n ? a.vox[s] : 0;
        const bool carbon = s < a.n && (vb & 15) == a.carbon_id;
        unsigned rank = 0;
        if (a.draws) {                                          // ordered rank inside the strip (uniform branch)
            const unsigned m = __ballot_sync(0xffffffffu, carbon);
            if (lane == 0) sm[w] = __popc(m);
            __syncthreads();
            unsigned before = 0, total = 0;
#pragma unroll
            for (int q = 0; q < DF_THREADS / 32; ++q) { if (q < w) before += sm[q]; total += sm[q]; }
            rank = run + before + __popc(m & ((1u << lane) - 1u));
            run += total;
            __syncthreads();
        }
        if (s >= a.n) continue;
        uint8_t mask = 0;
        if (carbon) {
            double u;
            if (a.draws) u = a.draws[rank];
            else {
                const uint64_t g = (uint64_t)(a.g_off + s);
                uint32_t c[4] = {(uint32_t)g, (uint32_t)(g >> 32), a.epoch, 0x44454643u};
                philox_round10(c, (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
                u = (double)((((uint64_t)c[0] << 32) | c[1]) >> 11) * 1.1102230246251565e-16;
            }
            const double Tv = a.T[s];
            const double valid_T = Tv > 0.0 ? Tv : a.T_default;                       // defects.py:13
            double prob = a.base * exp(-a.e_mig / (a.kT * valid_T));                 // :14
            prob = prob < 0.0 ? 0.0 : (prob > 1.0 ? 1.0 : prob);                      // :17 (NaN stays NaN: u < NaN is false)
            mask = u < prob ? 1 : 0;                                                  // :18
        }
        uint8_t st = vb & 15;
        if (mask && a.apply_to_state) st = (uint8_t)a.defect_id;                      // :28-29
        a.vox[s] = (uint8_t)(st | (mask << 4));
        set += mask;
    }
    set = warp_sum_i(set);
    if (lane == 0 && set) atomicAdd(&a.totals[1], (unsigned long long)set);
}

// ---- state histogram ----

__device__ __forceinline__ void counts_body(const uint8_t *__restrict__ vox, int64_t n, unsigned long long *out)
{
    __shared__ unsigned int h[16];
    if (threadIdx.x < 16) h[threadIdx.x] = 0;
    __syncthreads();
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n;
         q += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&h[vox[q] & 0x0F], 1u);
    __syncthreads();
    if (threadIdx.x < 16 && h[threadIdx.x]) atomicAdd(&out[threadIdx.x], (unsigned long long)h[threadIdx.x]);
}

// ---- grains (utils.py:28-84, 104-111; see grains.cu) ----

__device__ __forceinline__ int uf_find(int *label, int x)
{
    int p = label[x];
    while (p != x) {                      // path halving
        const int gp = label[p];
        if (gp != p) label[x] = gp;
        x = p; p = gp;
    }
    return x;
}
__device__ __forceinline__ void uf_union(int *label, int a, int b)
{
    while (true) {
        a = uf_find(label, a); b = uf_find(label, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }          // a < b: hook b under a
        const int old = atomicMin(&label[b], a);
        if (old == b) return;
        b = old;                                                // someone re-hooked b meanwhile: retry from there
    }
}

__device__ __forceinline__ void grains_init_body(const uint8_t *__restrict__ vox, int *label, int64_t lo, int64_t hi)
{
    for (int64_t s = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < hi; s += (int64_t)gridDim.x * blockDim.x)
        label[s] = (vox[s] & 0x0F) != 0 ? (int)s : -1;
}

// offsets 0,1,4,5,8,10,12 are one of each +/- pair of the neighbour table
// theta == nullptr: edge iff clamp(v1.v2) > thr (thr = cos of the misorientation threshold);
// theta != nullptr: the |theta1 - theta2| < thr criterion of utils.py:49-50 (orientation_phi=None).
__device__ __forceinline__ void grains_union_body(const uint8_t *__restrict__ vox, const Vec4 *__restrict__ v,
                                                  const double *__restrict__ theta, int *label, int L, int p_lo, int p_hi,
                                                  double thr)
{
    const int LL = L * L;
    const int64_t lo = (int64_t)p_lo * LL, hi = (int64_t)p_hi * LL;
    for (int64_t s = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < hi; s += (int64_t)gridDim.x * blockDim.x) {
        if ((vox[s] & 0x0F) == 0) continue;
        const int p = (int)(s / LL), j = (int)((s / L) % L), k = (int)(s % L);
        Vec4 a = Vec4{0.0, 0.0, 0.0, 0.0};
        double ta = 0.0;
        if (theta) ta = theta[s]; else a = v[s];
        const int pos[7] = {0, 1, 4, 5, 8, 10, 12};
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            const int o = pos[q];
            const int pi = p + CET_NB_DI(o), nj = j + CET_NB_DJ(o), nk = k + CET_NB_DK(o);
            if (pi < p_lo || pi >= p_hi || nj < 0 || nj >= L || nk < 0 || nk >= L) continue;
            const int64_t t = s + ((int64_t)CET_NB_DI(o) * L + CET_NB_DJ(o)) * L + CET_NB_DK(o);
            if ((vox[t] & 0x0F) == 0) continue;
            bool edge;
            if (theta) {
                edge = fabs(ta - theta[t]) < thr;
            } else {
                const Vec4 b = v[t];
                double dot = a.x * b.x + a.y * b.y + a.z * b.z;
                dot = pymax(pymin(dot, 1.0), -1.0);
                edge = dot > thr;
            }
            if (edge) uf_union(label, (int)s, (int)t);
        }
    }
}

struct GrainStat { int root, size, lo[3], hi[3]; };

// label[s] := root of s.  GID: roots are counted and given dense ids in order of arrival (the grouped path
// numbers them in site order afterwards instead).
template <bool GID>
__device__ __forceinline__ void grains_flatten_body(int *label, int *gid, int64_t lo, int64_t hi, unsigned int *n_roots)
{
    for (int64_t s = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < hi; s += (int64_t)gridDim.x * blockDim.x) {
        int r = label[s];
        if (r < 0) continue;
        // read-only walk (no path halving here: a halving store by another thread could overwrite
        // the final label of a site its owner has already flattened); owners only shorten chains
        for (int x = (int)s; r != x;) { x = r; r = label[x]; }
        if (r == (int)s) { if (GID) gid[s] = (int)atomicAdd(n_roots, 1u); }
        else label[s] = r;       // a root's own entry never changes, so concurrent walks stay valid
    }
}

__device__ __forceinline__ void grain_stat_init(GrainStat *g, int root)
{
    GrainStat t;
    t.root = root; t.size = 0;
    t.lo[0] = t.lo[1] = t.lo[2] = 0x7fffffff;
    t.hi[0] = t.hi[1] = t.hi[2] = -1;
    *g = t;
}

// utils.py:104-111 as metrics.grain_aspect_ratios evaluates it; a grain is equiaxed when this is below the
// AR threshold (metrics_reduce_group_kernel's n_equiaxed, cet_grain_profile_group's class)
__device__ __forceinline__ double grain_ar(const GrainStat &s)
{
    const int d0 = s.hi[0] - s.lo[0] + 1, d1 = s.hi[1] - s.lo[1] + 1, d2 = s.hi[2] - s.lo[2] + 1;
    const int mx = max(d0, max(d1, d2)), mn = min(d0, min(d1, d2));
    return __ddiv_rn((double)mx, (double)max(mn, 1));
}

// One atomic set per (warp, grain): lanes holding voxels of the same grain elect a leader.
__device__ __forceinline__ void grains_stats_body(const int *__restrict__ label, const int *__restrict__ gid, int64_t lo,
                                                  int64_t hi, GrainStat *st, int L, int i_off)
{
    const int LL = L * L;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    for (int64_t s0 = lo + (int64_t)blockIdx.x * blockDim.x; s0 < hi; s0 += stride) {
        const int64_t s = s0 + threadIdx.x;
        const int r = s < hi ? label[s] : -1;
        const unsigned live = __ballot_sync(0xffffffffu, r >= 0);
        if (r < 0) continue;
        const unsigned peers = __match_any_sync(live, r);
        const int c0 = i_off + (int)(s / LL), c1 = (int)((s / L) % L), c2 = (int)(s % L);
        const int mn0 = __reduce_min_sync(peers, c0), mx0 = __reduce_max_sync(peers, c0);
        const int mn1 = __reduce_min_sync(peers, c1), mx1 = __reduce_max_sync(peers, c1);
        const int mn2 = __reduce_min_sync(peers, c2), mx2 = __reduce_max_sync(peers, c2);
        if (lane == __ffs(peers) - 1) {
            GrainStat *g = st + gid[r];
            atomicAdd(&g->size, __popc(peers));
            atomicMin(&g->lo[0], mn0); atomicMax(&g->hi[0], mx0);
            atomicMin(&g->lo[1], mn1); atomicMax(&g->hi[1], mx1);
            atomicMin(&g->lo[2], mn2); atomicMax(&g->hi[2], mx2);
        }
    }
}

}  // namespace cet
