// grain_shape_group.cu — growth-axis elongation histograms of a group of whole-lattice contexts
// (cet_grain_shape_group): per lattice, the grains and their sites binned by A (grain_shape.cuh), grains below
// min_size in a bucket of their own.  The call reads the last labelling of each context (label, gid, n_grains) and
// writes nothing a sweep, a metrics row or a profile reads.  As in profile_group.cu a CTA takes its lattice's
// arguments from a table in kernel parameter space (blockIdx.y); a group of up to 16 launches the small table.
// Three launches for the whole group:
//   1. zero: every grain's moment slot (SHAPE_WORDS words at gid) starts at zero;
//   2. moments: per site, label -> gid, the sums n, S_x, S_xx of every grain, aggregated per warp over the lanes of
//      one grain (32-bit partials: 32 c^2 < 2^26) and added with one set of 64-bit atomics per (warp, grain);
//   3. per grain: the bin (shape_bin), aggregated per warp, privatised in shared memory, flushed with global atomics.
// One memset zeroes the group's table beforehand; one D2H copy returns it.
#include <algorithm>
#include "cadence.cuh"
#include "grain_shape.cuh"

namespace cet {

struct GsArgs {
    const int *label, *gid;
    unsigned long long *mom;        // [n_grains][SHAPE_WORDS], at gid
    unsigned long long *tab;        // [2][n_edges + 2]: the lattice's part of the result table
    int n_grains;
};
static_assert(group_fits<GsArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

struct GsEdges {
    double e[SHAPE_EDGES_MAX];
};

constexpr int GS_THREADS = 256;

template <int CAP>
__global__ void __launch_bounds__(GS_THREADS) shape_zero_group_kernel(const __grid_constant__ GroupArgs<GsArgs, CAP> g)
{
    const GsArgs &a = g.a[blockIdx.y];
    const int64_t n = (int64_t)a.n_grains * SHAPE_WORDS;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        a.mom[i] = 0ull;
}

template <int CAP>
__global__ void __launch_bounds__(GS_THREADS) shape_moments_group_kernel(const __grid_constant__ GroupArgs<GsArgs, CAP> g, int64_t n,
                                                                        int L)
{
    const GsArgs &a = g.a[blockIdx.y];
    const int LL = L * L, lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t s0 = (int64_t)blockIdx.x * blockDim.x; s0 < n; s0 += stride) {      // warp-uniform trip count
        const int64_t s = s0 + threadIdx.x;
        const int r = s < n ? a.label[s] : -1;
        const unsigned live = __ballot_sync(0xffffffffu, r >= 0);
        if (r < 0) continue;
        const unsigned peers = __match_any_sync(live, r);
        const unsigned c0 = (unsigned)(s / LL), c1 = (unsigned)((s / L) % L), c2 = (unsigned)(s % L);
        const unsigned s_0 = __reduce_add_sync(peers, c0), s_1 = __reduce_add_sync(peers, c1), s_2 = __reduce_add_sync(peers, c2);
        const unsigned q_0 = __reduce_add_sync(peers, c0 * c0), q_1 = __reduce_add_sync(peers, c1 * c1),
                       q_2 = __reduce_add_sync(peers, c2 * c2);
        if (lane == __ffs(peers) - 1) {
            unsigned long long *m = a.mom + (size_t)a.gid[r] * SHAPE_WORDS;
            atomicAdd(m + SHAPE_N, (unsigned long long)__popc(peers));
            atomicAdd(m + SHAPE_S + 0, (unsigned long long)s_0);
            atomicAdd(m + SHAPE_S + 1, (unsigned long long)s_1);
            atomicAdd(m + SHAPE_S + 2, (unsigned long long)s_2);
            atomicAdd(m + SHAPE_SS + 0, (unsigned long long)q_0);
            atomicAdd(m + SHAPE_SS + 1, (unsigned long long)q_1);
            atomicAdd(m + SHAPE_SS + 2, (unsigned long long)q_2);
        }
    }
}

// dynamic shared memory: double e[n_edges], then unsigned h[2][n_edges + 2] = grains, sites of the CTA's grains
// (a lattice has fewer than 2^31 sites, so neither count wraps)
template <int CAP>
__global__ void __launch_bounds__(GS_THREADS) shape_bins_group_kernel(const __grid_constant__ GroupArgs<GsArgs, CAP> g,
                                                                     const __grid_constant__ GsEdges ed, int n_edges, int axis,
                                                                     int64_t min_size)
{
    extern __shared__ double e[];
    unsigned *h = (unsigned *)(e + n_edges);
    const GsArgs &a = g.a[blockIdx.y];
    const int nb = n_edges + 2, lane = threadIdx.x & 31;
    for (int b = threadIdx.x; b < n_edges; b += blockDim.x) e[b] = ed.e[b];
    for (int b = threadIdx.x; b < 2 * nb; b += blockDim.x) h[b] = 0;
    __syncthreads();
    const int stride = gridDim.x * blockDim.x;
    for (int i0 = blockIdx.x * blockDim.x; i0 < a.n_grains; i0 += stride) {      // warp-uniform trip count
        const int i = i0 + threadIdx.x;
        const bool live = i < a.n_grains;
        int bin = -1;
        unsigned size = 0;
        if (live) {
            const ulonglong2 *p = (const ulonglong2 *)(a.mom + (size_t)i * SHAPE_WORDS);
            uint64_t m[SHAPE_WORDS];
#pragma unroll
            for (int w = 0; w < SHAPE_WORDS / 2; ++w) {
                const ulonglong2 v = p[w];
                m[2 * w] = v.x; m[2 * w + 1] = v.y;
            }
            bin = shape_bin(m, axis, e, n_edges, min_size);
            size = (unsigned)m[SHAPE_N];
        }
        const unsigned act = __ballot_sync(0xffffffffu, live);
        if (!live) continue;
        const unsigned peers = __match_any_sync(act, bin);
        const unsigned sites = __reduce_add_sync(peers, size);
        if (lane == __ffs(peers) - 1) {
            atomicAdd(&h[bin], (unsigned)__popc(peers));
            atomicAdd(&h[nb + bin], sites);
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < 2 * nb; b += blockDim.x)
        if (h[b]) atomicAdd(&a.tab[b], (unsigned long long)h[b]);
}

static size_t align64(size_t b) { return (b + 63) & ~(size_t)63; }

template <int CAP>
static int shape_group_run(cet_ctx *const *ctxs, int n, int axis, const double *edges, int n_edges, int64_t min_size,
                           int64_t *out)
{
    cet_ctx *c0 = ctxs[0];
    cudaStream_t st = c0->stream;
    const int L = (int)c0->n1;
    const int64_t ns = c0->nloc;
    const int nb = n_edges + 2;
    const size_t tab_bytes = align64((size_t)n * 2 * nb * sizeof(unsigned long long));
    // per-context moment buffers (grow-only); n_grains is known since the labelling
    GroupArgs<GsArgs, CAP> t{};
    int max_ng = 0;
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        const size_t need = (size_t)c->n_grains * SHAPE_WORDS * sizeof(unsigned long long);
        if (c->cap_grain_mom < need) {
            if (c->grain_mom) { cudaFree(c->grain_mom); c->grain_mom = nullptr; c->cap_grain_mom = 0; }
            CET_CUDA(cudaMalloc(&c->grain_mom, need + need / 4));
            c->cap_grain_mom = need + need / 4;
        }
        max_ng = std::max(max_ng, (int)c->n_grains);
    }
    if (c0->cap_shape_tab < tab_bytes) {
        if (c0->shape_tab) { cudaFree(c0->shape_tab); c0->shape_tab = nullptr; c0->cap_shape_tab = 0; }
        CET_CUDA(cudaMalloc(&c0->shape_tab, tab_bytes));
        c0->cap_shape_tab = tab_bytes;
    }
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        GsArgs &p = t.a[q];
        p.label = c->grain_label; p.gid = c->grain_gid;
        p.mom = (unsigned long long *)c->grain_mom;
        p.tab = (unsigned long long *)c0->shape_tab + (size_t)q * 2 * nb;
        p.n_grains = (int)c->n_grains;
    }
    GsEdges ed{};
    for (int b = 0; b < n_edges; ++b) ed.e[b] = edges[b];
    if (int rc = group_order(ctxs, n)) return rc;
    CET_CUDA(cudaMemsetAsync(c0->shape_tab, 0, tab_bytes, st));
    const int per = std::max(1, (sm_count(c0) * 8 + n - 1) / n);
    const int gz = (int)std::max<int64_t>(1, std::min<int64_t>(((int64_t)max_ng * SHAPE_WORDS + GS_THREADS - 1) / GS_THREADS, per));
    const int gx = (int)std::min<int64_t>((ns + GS_THREADS - 1) / GS_THREADS, std::max(1, (sm_count(c0) * 16 + n - 1) / n));
    const int gg = (int)std::max<int64_t>(1, std::min<int64_t>((max_ng + 8 * GS_THREADS - 1) / (8 * GS_THREADS), per));
    shape_zero_group_kernel<CAP><<<dim3(gz, n), GS_THREADS, 0, st>>>(t);
    shape_moments_group_kernel<CAP><<<dim3(gx, n), GS_THREADS, 0, st>>>(t, ns, L);
    shape_bins_group_kernel<CAP><<<dim3(gg, n), GS_THREADS, n_edges * sizeof(double) + 2 * nb * sizeof(unsigned), st>>>(
        t, ed, n_edges, axis, min_size);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(out, c0->shape_tab, (size_t)n * 2 * nb * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CET_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" int cet_grain_shape_group(cet_ctx *const *ctxs, int32_t n_ctx, int32_t axis, const double *edges,
                                     int32_t n_edges, int64_t min_size, int64_t *out)
{
    if (int rc = group_check("cet_grain_shape_group", ctxs, n_ctx)) return rc;
    CET_REQUIRE(edges && out, "cet_grain_shape_group: NULL argument");
    CET_REQUIRE(axis >= 0 && axis <= 2, "cet_grain_shape_group: axis must be 0, 1 or 2, got %d", (int)axis);
    CET_REQUIRE(n_edges >= 1 && n_edges <= SHAPE_EDGES_MAX, "cet_grain_shape_group: need 1 <= n_edges <= %d, got %d",
                SHAPE_EDGES_MAX, (int)n_edges);
    for (int b = 0; b < n_edges; ++b) {
        CET_REQUIRE(finite_f64(edges[b]) && edges[b] > 0.0, "cet_grain_shape_group: edge %d is not finite and > 0", b);
        CET_REQUIRE(b == 0 || edges[b] > edges[b - 1], "cet_grain_shape_group: edges must ascend strictly (edge %d)", b);
    }
    CET_REQUIRE(min_size >= 1, "cet_grain_shape_group: min_size must be >= 1, got %lld", (long long)min_size);
    for (int q = 0; q < n_ctx; ++q) {
        const cet_ctx *c = ctxs[q];
        CET_REQUIRE(c->grain_label && c->grain_p_lo == 0 && c->grain_p_hi == c->np,
                    "cet_grain_shape_group: context %d has no labelling of the whole lattice (label its grains first)", q);
    }
    cet::DeviceGuard dg(ctxs[0]->device);
    return n_ctx <= 16 ? shape_group_run<16>(ctxs, n_ctx, axis, edges, n_edges, min_size, out)
                       : shape_group_run<GROUP_MAX>(ctxs, n_ctx, axis, edges, n_edges, min_size, out);
}
