// metrics_group.cu — the metrics cadence of a group of whole-lattice contexts (cet_counts_group,
// cet_metrics_group): defect-mask refresh, state histogram, grain labelling, per-grain statistics and the
// reductions of a metrics row, each kernel one launch for the whole group.  As in the grouped sweeps, a CTA takes
// its lattice's arguments from a table passed by value in kernel parameter space (blockIdx.y, or blockIdx.x for
// the one-CTA-per-lattice kernels), and a group of up to 16 launches the small table.
//
// The refresh, the histogram and the labelling run the bodies of the solo kernels (cadence.cuh), so masks and
// labels have the same bits as after cet_defects_refresh / cet_grains_label_ex.  Then, per lattice:
//   - root ranks: a two-level ordered count of the roots (label[s] == s) in site order numbers every grain in the
//     reference's cluster order (raster order of its first voxel); gid[root] := that number;
//   - statistics: voxel count and bounding box of each grain, at its number (grains_stats_body);
//   - reduction (one CTA per lattice): size sum, grains with AR < threshold, the four searchsorted indices of
//     metrics_from_grains' percentiles over cumsum([n_sites - size_sum, sizes...]), and the AR sum in NumPy's
//     pairwise order (np.mean(ar.tolist()) = pw(ar, 0, n) / n): the leaves (<= 128 elements) of that recursion
//     start at multiples of 8 and are summed in parallel with NumPy's 8-accumulator loop; one thread combines them
//     along the recursion.  Every add is __dadd_rn (the build also passes -fmad=false).
#include <algorithm>
#include <vector>
#include "cadence.cuh"

namespace cet {

// One lattice's entry of the result table in device memory (group_tab of ctxs[0]).
struct MgEntry {
    unsigned long long totals[2];   // [0] carbon sites, [1] sites with the mask set (DefectArgs::totals)
    unsigned long long n_grains;
    unsigned long long size_sum, n_equiaxed;
    unsigned long long counts[16];
    long long pct_index[4];
    double ar_sum;
};

struct MgArgs {
    const uint8_t *vox;
    const Vec4 *v;
    int *label, *gid;
    unsigned int *root_tiles;       // [n_tiles + 1]: roots per DF_TILE sites, then exclusive offsets
    GrainStat *st;                  // [n_grains], in cluster order
    double *leaf;                   // pairwise leaf sums, at (first element of the leaf) / 8
    MgEntry *out;
    long long pct_pos[4];
    double ar_threshold;
    double cos_thr;                 // cos of the misorientation threshold (cet_grains_label_ex's criterion 0)
    int n_grains;
};
static_assert(group_fits<MgArgs>() && group_fits<DefectArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

constexpr int PW_LEAF = 128;        // NumPy's PW_BLOCKSIZE: pairwise_sum adds at most this many elements in one loop

template <int CAP>
__global__ void __launch_bounds__(DF_THREADS) metrics_defects_count_group_kernel(const __grid_constant__ GroupArgs<DefectArgs, CAP> g)
{
    defects_count_body(g.a[blockIdx.y]);
}

template <int CAP>
__global__ void __launch_bounds__(1024) metrics_defects_scan_group_kernel(const __grid_constant__ GroupArgs<DefectArgs, CAP> g, int n_tiles)
{
    tile_scan_body(g.a[blockIdx.x].tile_count, n_tiles, g.a[blockIdx.x].totals);
}

template <int CAP>
__global__ void __launch_bounds__(DF_THREADS) metrics_defects_assign_group_kernel(const __grid_constant__ GroupArgs<DefectArgs, CAP> g)
{
    defects_assign_body(g.a[blockIdx.y]);
}

template <int CAP>
__global__ void metrics_counts_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int64_t n)
{
    counts_body(g.a[blockIdx.y].vox, n, g.a[blockIdx.y].out->counts);
}

template <int CAP>
__global__ void metrics_grains_init_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int64_t n)
{
    grains_init_body(g.a[blockIdx.y].vox, g.a[blockIdx.y].label, 0, n);
}

template <int CAP>
__global__ void metrics_grains_union_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int L)
{
    const MgArgs &a = g.a[blockIdx.y];
    grains_union_body(a.vox, a.v, nullptr, a.label, L, 0, L, a.cos_thr);
}

template <int CAP>
__global__ void metrics_grains_flatten_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int64_t n)
{
    grains_flatten_body<false>(g.a[blockIdx.y].label, nullptr, 0, n, nullptr);
}

// roots per DF_TILE sites
template <int CAP>
__global__ void __launch_bounds__(DF_THREADS) metrics_roots_count_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int64_t n)
{
    const MgArgs &a = g.a[blockIdx.y];
    __shared__ int sm[DF_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * DF_TILE;
    int c = 0;
#pragma unroll
    for (int e = 0; e < DF_PER_THREAD; ++e) {
        const int64_t s = base + e * DF_THREADS + threadIdx.x;
        if (s < n && a.label[s] == (int)s) ++c;
    }
    c = warp_sum_i(c);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < DF_THREADS / 32; ++w) t += sm[w];
        a.root_tiles[blockIdx.x] = (unsigned)t;
    }
}

template <int CAP>
__global__ void __launch_bounds__(1024) metrics_roots_scan_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int n_tiles)
{
    tile_scan_body(g.a[blockIdx.x].root_tiles, n_tiles, &g.a[blockIdx.x].out->n_grains);
}

// gid[root] := rank of the root in site order; the grain's statistics entry starts empty
template <int CAP>
__global__ void __launch_bounds__(DF_THREADS) metrics_roots_assign_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int64_t n)
{
    const MgArgs &a = g.a[blockIdx.y];
    __shared__ int sm[DF_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * DF_TILE;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned run = a.root_tiles[blockIdx.x];
    for (int e = 0; e < DF_PER_THREAD; ++e) {                   // strips of 256 consecutive sites keep site order
        const int64_t s = base + e * DF_THREADS + threadIdx.x;
        const bool root = s < n && a.label[s] == (int)s;
        const unsigned m = __ballot_sync(0xffffffffu, root);
        if (lane == 0) sm[w] = __popc(m);
        __syncthreads();
        unsigned before = 0, total = 0;
#pragma unroll
        for (int q = 0; q < DF_THREADS / 32; ++q) { if (q < w) before += sm[q]; total += sm[q]; }
        const unsigned rank = run + before + __popc(m & ((1u << lane) - 1u));
        run += total;
        __syncthreads();
        if (root) {
            a.gid[s] = (int)rank;
            grain_stat_init(a.st + rank, (int)s);
        }
    }
}

template <int CAP>
__global__ void metrics_stats_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int64_t n, int L)
{
    const MgArgs &a = g.a[blockIdx.y];
    grains_stats_body(a.label, a.gid, 0, n, a.st, L, 0);
}

// NumPy's pairwise_sum of a[lo, lo + m) for m <= PW_LEAF
__device__ double pw_leaf(const GrainStat *st, int lo, int m)
{
    if (m < 8) {
        double r = -0.0;
        for (int i = 0; i < m; ++i) r = __dadd_rn(r, grain_ar(st[lo + i]));
        return r;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = grain_ar(st[lo + j]);
    int i = 8;
    for (; i < m - m % 8; i += 8)
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], grain_ar(st[lo + i + j]));
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < m; ++i) res = __dadd_rn(res, grain_ar(st[lo + i]));
    return res;
}

__device__ __forceinline__ int pw_split(int m) { const int h = m / 2; return h - h % 8; }

__device__ __forceinline__ long long block_sum_ll(long long v, long long *sm)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    long long t = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm[w];
    return t;
}

// one CTA of 1024 threads per lattice
template <int CAP>
__global__ void __launch_bounds__(1024) metrics_reduce_group_kernel(const __grid_constant__ GroupArgs<MgArgs, CAP> g, int64_t n_sites)
{
    const MgArgs &a = g.a[blockIdx.x];
    const int n = a.n_grains, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    __shared__ long long sm[32];
    __shared__ long long carry;
    long long ssum = 0, neq = 0;
    for (int i = tid; i < n; i += blockDim.x) {
        const GrainStat s = a.st[i];
        ssum += s.size;
        neq += grain_ar(s) < a.ar_threshold ? 1 : 0;
    }
    const long long size_sum = block_sum_ll(ssum, sm);
    const long long n_eq = block_sum_ll(neq, sm);
    // searchsorted(cum, x, side="right") = #{i : cum[i] <= x}, cum[0] = n_sites - size_sum, cum[g + 1] = cum[0] + sizes[0..g]
    const long long cum0 = n_sites - size_sum;
    long long cnt[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) cnt[k] = (tid == 0 && cum0 <= a.pct_pos[k]) ? 1 : 0;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + tid;
        long long inc = i < n ? a.st[i].size : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) sm[w] = inc;
        __syncthreads();
        long long before = carry;
        for (int q = 0; q < w; ++q) before += sm[q];
        if (i < n) {
            const long long c = cum0 + before + inc;
#pragma unroll
            for (int k = 0; k < 4; ++k) cnt[k] += c <= a.pct_pos[k] ? 1 : 0;
        }
        __syncthreads();
        if (tid == blockDim.x - 1) carry = before + inc;
        __syncthreads();
    }
    long long idx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) idx[k] = block_sum_ll(cnt[k], sm);
    // leaves of pw(ar, 0, n): descend the recursion to the leaf that holds element p = 8k
    for (int k = tid; 8 * k < n; k += blockDim.x) {
        const int p = 8 * k;
        int lo = 0, m = n;
        while (m > PW_LEAF) {
            const int n2 = pw_split(m);
            if (p < lo + n2) m = n2;
            else { lo += n2; m -= n2; }
        }
        if (lo == p) a.leaf[p >> 3] = pw_leaf(a.st, lo, m);
    }
    __syncthreads();
    if (tid != 0) return;
    // pw(lo, m) = m <= 128 ? leaf(lo) : pw(lo, n2) + pw(lo + n2, m - n2), post-order on an explicit stack
    double ar_sum = 0.0;
    if (n > 0) {
        struct Frame { int lo, m, stage; double left; };
        Frame stk[40];
        int sp = 0;
        stk[0] = Frame{0, n, 0, 0.0};
        while (sp >= 0) {
            Frame &f = stk[sp];
            if (f.m <= PW_LEAF) { ar_sum = a.leaf[f.lo >> 3]; --sp; continue; }
            const int n2 = pw_split(f.m);
            if (f.stage == 0) { f.stage = 1; stk[sp + 1] = Frame{f.lo, n2, 0, 0.0}; ++sp; }
            else if (f.stage == 1) { f.left = ar_sum; f.stage = 2; stk[sp + 1] = Frame{f.lo + n2, f.m - n2, 0, 0.0}; ++sp; }
            else { ar_sum = __dadd_rn(f.left, ar_sum); --sp; }
        }
    }
    MgEntry *o = a.out;
    o->size_sum = (unsigned long long)size_sum;
    o->n_equiaxed = (unsigned long long)n_eq;
#pragma unroll
    for (int k = 0; k < 4; ++k) o->pct_index[k] = idx[k];
    o->ar_sum = ar_sum;
}

// ---- host side ----

int group_check(const char *fn, cet_ctx *const *ctxs, int32_t n_ctx)
{
    CET_REQUIRE(ctxs, "%s: NULL argument", fn);
    CET_REQUIRE(n_ctx >= 1 && n_ctx <= GROUP_MAX, "%s: need 1 <= n_ctx <= %d, got %d", fn, GROUP_MAX, (int)n_ctx);
    for (int q = 0; q < n_ctx; ++q) {
        const cet_ctx *c = ctxs[q];
        CET_REQUIRE(c, "%s: context %d is NULL", fn, q);
        for (int r = 0; r < q; ++r) CET_REQUIRE(ctxs[r] != c, "%s: context %d repeats context %d", fn, q, r);
        CET_REQUIRE(c->device == ctxs[0]->device, "%s: context %d is on another device", fn, q);
        CET_REQUIRE(c->world == 1 && c->halo == 0 && c->i_begin == 0 && c->i_end == c->n0,
                    "%s: context %d is a slab; groups take whole-lattice contexts", fn, q);
        CET_REQUIRE(c->cubic && c->n0 == c->n1, "%s: context %d is not a cubic lattice", fn, q);
        CET_REQUIRE(c->n1 == ctxs[0]->n1, "%s: context %d has L = %lld, context 0 L = %lld", fn, q, (long long)c->n1,
                    (long long)ctxs[0]->n1);
        CET_REQUIRE(c->nloc < (1ll << 31), "%s: the lattice must have fewer than 2^31 sites", fn);
    }
    return 0;
}

// the group's work goes to ctxs[0]'s stream, after the work already queued on every member's stream
int group_order(cet_ctx *const *ctxs, int n)
{
    cet_ctx *c0 = ctxs[0];
    for (int q = 1; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        if (!c->ev_group) CET_CUDA(cudaEventCreateWithFlags(&c->ev_group, cudaEventDisableTiming));
        CET_CUDA(cudaEventRecord(c->ev_group, c->stream));
        CET_CUDA(cudaStreamWaitEvent(c0->stream, c->ev_group, 0));
    }
    return 0;
}

// group_order, and the result table (in ctxs[0]) zeroed
static int mg_begin(cet_ctx *const *ctxs, int n)
{
    cet_ctx *c0 = ctxs[0];
    if (!c0->group_tab) CET_CUDA(cudaMalloc(&c0->group_tab, GROUP_MAX * sizeof(MgEntry)));
    if (int rc = group_order(ctxs, n)) return rc;
    CET_CUDA(cudaMemsetAsync(c0->group_tab, 0, (size_t)n * sizeof(MgEntry), c0->stream));
    return 0;
}

static int mg_read(cet_ctx *c0, int n, std::vector<MgEntry> &h)
{
    h.resize(n);
    CET_CUDA(cudaMemcpyAsync(h.data(), c0->group_tab, (size_t)n * sizeof(MgEntry), cudaMemcpyDeviceToHost, c0->stream));
    CET_CUDA(cudaStreamSynchronize(c0->stream));
    return 0;
}

static size_t align64(size_t b) { return (b + 63) & ~(size_t)63; }

template <int CAP>
static int counts_group_run(cet_ctx *const *ctxs, int n, int64_t *counts)
{
    cet_ctx *c0 = ctxs[0];
    GroupArgs<MgArgs, CAP> t{};
    for (int q = 0; q < n; ++q) {
        t.a[q].vox = ctxs[q]->vox;
        t.a[q].out = (MgEntry *)c0->group_tab + q;
    }
    const int64_t ns = c0->nloc;
    const int gx = (int)std::min<int64_t>((ns + 255) / 256, std::max(1, (sm_count(c0) * 16 + n - 1) / n));
    metrics_counts_group_kernel<CAP><<<dim3(gx, n), 256, 0, c0->stream>>>(t, ns);
    CET_CUDA(cudaGetLastError());
    std::vector<MgEntry> h;
    if (int rc = mg_read(c0, n, h)) return rc;
    for (int q = 0; q < n; ++q)
        for (int s = 0; s < 16; ++s) counts[16 * q + s] = (int64_t)h[q].counts[s];
    return 0;
}

template <int CAP>
static int metrics_group_run(cet_ctx *const *ctxs, int n, const cet_metrics_params *mp, const double *const *draws,
                             const int64_t *n_draws, cet_metrics_result *res)
{
    cet_ctx *c0 = ctxs[0];
    cudaStream_t st = c0->stream;
    const int L = (int)c0->n1;
    const int64_t ns = c0->nloc;
    const int n_tiles = (int)((ns + DF_TILE - 1) / DF_TILE);
    const size_t tiles_bytes = align64((size_t)(n_tiles + 1) * sizeof(unsigned int));
    auto host_draws = [&](int q) { return mp[q].refresh && draws && draws[q]; };
    // per-context buffers: labels, and in the stage the tile counts of the refresh and of the roots, then the draws
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        if (!c->grain_label) CET_CUDA(cudaMalloc(&c->grain_label, (size_t)c->nloc * sizeof(int)));
        if (!c->grain_gid) CET_CUDA(cudaMalloc(&c->grain_gid, (size_t)c->nloc * sizeof(int)));
        if (int rc = ensure_stage(c, 2 * tiles_bytes + (host_draws(q) ? (size_t)n_draws[q] * sizeof(double) : 0))) return rc;
    }
    if (int rc = mg_begin(ctxs, n)) return rc;
    MgEntry *tab = (MgEntry *)c0->group_tab;
    GroupArgs<DefectArgs, CAP> dt{};
    GroupArgs<MgArgs, CAP> gt{};
    std::vector<int> ref;                        // the refreshing contexts, in group order: entries of dt
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        MgArgs &m = gt.a[q];
        m.vox = c->vox; m.v = c->v; m.label = c->grain_label; m.gid = c->grain_gid;
        m.root_tiles = (unsigned int *)((char *)c->stage + tiles_bytes);
        m.out = tab + q;
        for (int k = 0; k < 4; ++k) m.pct_pos[k] = mp[q].pct_pos[k];
        m.ar_threshold = mp[q].ar_threshold;
        m.cos_thr = cos(mp[q].theta_threshold);
        if (!mp[q].refresh) continue;
        DefectArgs &d = dt.a[ref.size()];
        d.vox = c->vox; d.T = c->T; d.n = ns; d.g_off = 0;
        d.draws = host_draws(q) ? (const double *)((char *)c->stage + 2 * tiles_bytes) : nullptr;
        d.seed = mp[q].seed; d.epoch = mp[q].epoch;
        d.carbon_id = mp[q].carbon_id; d.defect_id = 0; d.apply_to_state = 0;
        d.base = mp[q].prob_base; d.e_mig = mp[q].e_mig; d.kT = mp[q].kT; d.T_default = mp[q].T_default;
        d.tile_count = (unsigned int *)c->stage;
        d.totals = tab[q].totals;
        ref.push_back(q);
    }
    const int n_ref = (int)ref.size();
    std::vector<MgEntry> h;
    // 1. mask refresh: count, scan; with host draws, the carbon counts are checked before any mask byte is written
    if (n_ref) {
        metrics_defects_count_group_kernel<CAP><<<dim3(n_tiles, n_ref), DF_THREADS, 0, st>>>(dt);
        metrics_defects_scan_group_kernel<CAP><<<n_ref, 1024, 0, st>>>(dt, n_tiles);
        CET_CUDA(cudaGetLastError());
        bool any_host = false;
        for (int q : ref) any_host = any_host || host_draws(q);
        if (any_host) {
            if (int rc = mg_read(c0, n, h)) return rc;
            for (int q : ref)
                if (host_draws(q))
                    CET_REQUIRE((int64_t)h[q].totals[0] <= n_draws[q], "cet_metrics_group: context %d has %lld carbon sites but only %lld draws",
                                q, (long long)h[q].totals[0], (long long)n_draws[q]);
            for (int r = 0; r < n_ref; ++r)
                if (host_draws(ref[r]))
                    CET_CUDA(cudaMemcpyAsync((void *)dt.a[r].draws, draws[ref[r]], (size_t)h[ref[r]].totals[0] * sizeof(double),
                                             cudaMemcpyHostToDevice, st));
        }
        metrics_defects_assign_group_kernel<CAP><<<dim3(n_tiles, n_ref), DF_THREADS, 0, st>>>(dt);
        CET_CUDA(cudaGetLastError());
    }
    // 2. histogram; 3. labelling; 4. root counts
    const int gx = (int)std::min<int64_t>((ns + 255) / 256, std::max(1, (sm_count(c0) * 16 + n - 1) / n));
    metrics_counts_group_kernel<CAP><<<dim3(gx, n), 256, 0, st>>>(gt, ns);
    metrics_grains_init_group_kernel<CAP><<<dim3(gx, n), 256, 0, st>>>(gt, ns);
    metrics_grains_union_group_kernel<CAP><<<dim3(gx, n), 256, 0, st>>>(gt, L);
    metrics_grains_flatten_group_kernel<CAP><<<dim3(gx, n), 256, 0, st>>>(gt, ns);
    metrics_roots_count_group_kernel<CAP><<<dim3(n_tiles, n), DF_THREADS, 0, st>>>(gt, ns);
    metrics_roots_scan_group_kernel<CAP><<<n, 1024, 0, st>>>(gt, n_tiles);
    CET_CUDA(cudaGetLastError());
    if (int rc = mg_read(c0, n, h)) return rc;
    // 5. per-grain buffers (grow-only), ranks and statistics; 6. reductions
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        const size_t ng = (size_t)h[q].n_grains;
        const size_t need = align64(ng * sizeof(GrainStat)) + (ng / 8 + 1) * sizeof(double);
        if (c->cap_grain_st < need) {
            if (c->grain_st) { cudaFree(c->grain_st); c->grain_st = nullptr; c->cap_grain_st = 0; }
            CET_CUDA(cudaMalloc(&c->grain_st, need + need / 4));
            c->cap_grain_st = need + need / 4;
        }
        gt.a[q].st = (GrainStat *)c->grain_st;
        gt.a[q].leaf = (double *)((char *)c->grain_st + align64(ng * sizeof(GrainStat)));
        gt.a[q].n_grains = (int)ng;
    }
    metrics_roots_assign_group_kernel<CAP><<<dim3(n_tiles, n), DF_THREADS, 0, st>>>(gt, ns);
    metrics_stats_group_kernel<CAP><<<dim3(gx, n), 256, 0, st>>>(gt, ns, L);
    metrics_reduce_group_kernel<CAP><<<n, 1024, 0, st>>>(gt, ns);
    CET_CUDA(cudaGetLastError());
    if (int rc = mg_read(c0, n, h)) return rc;
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        c->n_grains = (int64_t)h[q].n_grains;
        c->grain_p_lo = 0; c->grain_p_hi = (int)c->np;
        if (mp[q].refresh) lattice_changed(c);             // defect factors changed (kmc_event_rates.py:94)
        cet_metrics_result &r = res[q];
        for (int s = 0; s < 16; ++s) r.counts[s] = (int64_t)h[q].counts[s];
        r.n_carbon = (int64_t)h[q].totals[0]; r.n_defects = (int64_t)h[q].totals[1];
        r.n_grains = (int64_t)h[q].n_grains; r.size_sum = (int64_t)h[q].size_sum; r.n_equiaxed = (int64_t)h[q].n_equiaxed;
        for (int k = 0; k < 4; ++k) r.pct_index[k] = h[q].pct_index[k];
        r.ar_sum = h[q].ar_sum;
    }
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" int cet_counts_group(cet_ctx *const *ctxs, int32_t n_ctx, int64_t *counts)
{
    if (int rc = group_check("cet_counts_group", ctxs, n_ctx)) return rc;
    CET_REQUIRE(counts, "cet_counts_group: NULL argument");
    cet::DeviceGuard dg(ctxs[0]->device);
    if (int rc = mg_begin(ctxs, n_ctx)) return rc;
    return n_ctx <= 16 ? counts_group_run<16>(ctxs, n_ctx, counts) : counts_group_run<GROUP_MAX>(ctxs, n_ctx, counts);
}

extern "C" int cet_metrics_group(cet_ctx *const *ctxs, int32_t n_ctx, const cet_metrics_params *mp, const double *const *draws,
                                 const int64_t *n_draws, cet_metrics_result *res)
{
    if (int rc = group_check("cet_metrics_group", ctxs, n_ctx)) return rc;
    CET_REQUIRE(mp && res, "cet_metrics_group: NULL argument");
    for (int q = 0; q < n_ctx; ++q) {
        if (!mp[q].refresh) continue;
        CET_REQUIRE(mp[q].carbon_id >= 1 && mp[q].carbon_id <= 15, "cet_metrics_group: context %d: carbon state id must be in 1..15", q);
        CET_REQUIRE(!(draws && draws[q]) || (n_draws && n_draws[q] >= 0), "cet_metrics_group: context %d: draws without a count", q);
    }
    cet::DeviceGuard dg(ctxs[0]->device);
    return n_ctx <= 16 ? metrics_group_run<16>(ctxs, n_ctx, mp, draws, n_draws, res)
                       : metrics_group_run<GROUP_MAX>(ctxs, n_ctx, mp, draws, n_draws, res);
}
