// profile_group.cu — per-plane grain profiles of a group of whole-lattice contexts (cet_grain_profile_group): along
// one axis, per plane z, the occupied sites, those of equiaxed grains, the grains whose bounding box spans z, and the
// equiaxed ones among them.  The call reads the last labelling of each context (label, gid, n_grains) and writes
// nothing a sweep or a metrics row reads.  As in metrics_group.cu a CTA takes its lattice's arguments from a table in
// kernel parameter space (blockIdx.y, or blockIdx.x for the one-CTA-per-lattice kernel); a group of up to 16
// launches the small table.  Five launches for the whole group:
//   1. stats init: every root's GrainStat at gid[root] starts empty (grain_stat_init);
//   2. stats: voxel count and bounding box of every grain (grains_stats_body).  gid numbers the grains in arrival
//      order after cet_grains_label_ex and in site order after cet_metrics_group; either serves;
//   3. per grain: the class byte (grain_ar < threshold, metrics_reduce_group_kernel's test) and +1 / -1 entries of the
//      span differences at lo[axis] and hi[axis] + 1, aggregated per warp and privatised in shared memory;
//   4. per site: site -> label -> gid -> class, binned by the plane coordinate in shared memory (aggregated per warp
//      across lanes of one plane along axes 0 and 1), flushed with global atomics;
//   5. finalize (one CTA per lattice): prefix sums of the span differences into the table.
// One memset zeroes the group's table and differences beforehand; one D2H copy returns the table.
#include <algorithm>
#include "cadence.cuh"

namespace cet {

struct PgArgs {
    const int *label, *gid;
    GrainStat *st;                  // [n_grains], at gid
    uint8_t *cls;                   // [n_grains]: 1 = equiaxed
    unsigned long long *tab;        // [4][L]: the lattice's part of the result table
    int *span;                      // [2][L + 1]: differences of GrainsSpanning, EquiaxedGrainsSpanning
    int n_grains;
};
static_assert(group_fits<PgArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

constexpr int PG_THREADS = 256, PG_SITES_PER_THREAD = 16, PG_TILE = PG_THREADS * PG_SITES_PER_THREAD;

__device__ __forceinline__ int plane_of(int s, int L, int axis)
{
    return axis == 0 ? s / (L * L) : axis == 1 ? (s / L) % L : s % L;
}

template <int CAP>
__global__ void __launch_bounds__(PG_THREADS) profile_stats_init_group_kernel(const __grid_constant__ GroupArgs<PgArgs, CAP> g, int64_t n)
{
    const PgArgs &a = g.a[blockIdx.y];
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x)
        if (a.label[s] == (int)s) grain_stat_init(a.st + a.gid[s], (int)s);
}

template <int CAP>
__global__ void __launch_bounds__(PG_THREADS) profile_stats_group_kernel(const __grid_constant__ GroupArgs<PgArgs, CAP> g, int64_t n, int L)
{
    const PgArgs &a = g.a[blockIdx.y];
    grains_stats_body(a.label, a.gid, 0, n, a.st, L, 0);
}

// dynamic shared memory: int d[4][L + 1] = span differences of all grains at lo, at hi + 1, then of the equiaxed ones
template <int CAP>
__global__ void __launch_bounds__(PG_THREADS) profile_grains_group_kernel(const __grid_constant__ GroupArgs<PgArgs, CAP> g, int L, int axis,
                                                                         double ar_threshold)
{
    extern __shared__ int d[];
    const PgArgs &a = g.a[blockIdx.y];
    const int W = L + 1, lane = threadIdx.x & 31;
    for (int z = threadIdx.x; z < 4 * W; z += blockDim.x) d[z] = 0;
    __syncthreads();
    const int stride = gridDim.x * blockDim.x;
    for (int i0 = blockIdx.x * blockDim.x; i0 < a.n_grains; i0 += stride) {      // warp-uniform trip count
        const int i = i0 + threadIdx.x;
        const bool live = i < a.n_grains;
        int lo = 0, hi = 0;
        bool eq = false;
        if (live) {
            const GrainStat s = a.st[i];
            eq = grain_ar(s) < ar_threshold;
            a.cls[i] = eq ? 1 : 0;
            lo = s.lo[axis]; hi = s.hi[axis] + 1;
        }
        const unsigned act = __ballot_sync(0xffffffffu, live), eqm = __ballot_sync(0xffffffffu, eq);
        if (!live) continue;
        const unsigned pl = __match_any_sync(act, lo), ph = __match_any_sync(act, hi);
        if (lane == __ffs(pl) - 1) {
            atomicAdd(&d[lo], __popc(pl));
            if (pl & eqm) atomicAdd(&d[2 * W + lo], __popc(pl & eqm));
        }
        if (lane == __ffs(ph) - 1) {
            atomicAdd(&d[W + hi], __popc(ph));
            if (ph & eqm) atomicAdd(&d[3 * W + hi], __popc(ph & eqm));
        }
    }
    __syncthreads();
    for (int z = threadIdx.x; z < W; z += blockDim.x) {
        const int all = d[z] - d[W + z], eqd = d[2 * W + z] - d[3 * W + z];
        if (all) atomicAdd(&a.span[z], all);
        if (eqd) atomicAdd(&a.span[W + z], eqd);
    }
}

// dynamic shared memory: unsigned h[2][L] = Solid, EquiaxedSolid of the CTA's PG_TILE consecutive sites
template <int CAP>
__global__ void __launch_bounds__(PG_THREADS) profile_sites_group_kernel(const __grid_constant__ GroupArgs<PgArgs, CAP> g, int64_t n, int L,
                                                                        int axis)
{
    extern __shared__ unsigned int h[];
    const PgArgs &a = g.a[blockIdx.y];
    const int lane = threadIdx.x & 31;
    for (int z = threadIdx.x; z < 2 * L; z += blockDim.x) h[z] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * PG_TILE;
    constexpr int U = 4;                                        // sites per thread in flight
    for (int e0 = 0; e0 < PG_SITES_PER_THREAD; e0 += U) {
        int r[U], c[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t s = base + (e0 + u) * PG_THREADS + threadIdx.x;
            r[u] = s < n ? a.label[s] : -1;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) c[u] = r[u] >= 0 ? a.gid[r[u]] : -1;
#pragma unroll
        for (int u = 0; u < U; ++u) c[u] = c[u] >= 0 ? (int)a.cls[c[u]] : -1;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int s = (int)(base + (e0 + u) * PG_THREADS + threadIdx.x);
            const bool occ = c[u] >= 0;
            const int z = occ ? plane_of(s, L, axis) : 0;
            if (axis == 2) {                                    // consecutive sites: distinct planes
                if (occ) {
                    atomicAdd(&h[z], 1u);
                    if (c[u]) atomicAdd(&h[L + z], 1u);
                }
            } else {                                            // consecutive sites: one or two planes per warp
                const unsigned act = __ballot_sync(0xffffffffu, occ), eqm = __ballot_sync(0xffffffffu, c[u] == 1);
                if (!occ) continue;
                const unsigned peers = __match_any_sync(act, z);
                if (lane == __ffs(peers) - 1) {
                    atomicAdd(&h[z], (unsigned)__popc(peers));
                    if (peers & eqm) atomicAdd(&h[L + z], (unsigned)__popc(peers & eqm));
                }
            }
        }
    }
    __syncthreads();
    for (int z = threadIdx.x; z < 2 * L; z += blockDim.x)
        if (h[z]) atomicAdd(&a.tab[z], (unsigned long long)h[z]);
}

// one CTA of 64 threads per lattice: warp w scans the span differences of column 2 + w
template <int CAP>
__global__ void __launch_bounds__(64) profile_finalize_group_kernel(const __grid_constant__ GroupArgs<PgArgs, CAP> g, int L)
{
    const PgArgs &a = g.a[blockIdx.x];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int *d = a.span + w * (L + 1);
    unsigned long long *o = a.tab + (2 + w) * L;
    int carry = 0;
    for (int z0 = 0; z0 < L; z0 += 32) {
        const int z = z0 + lane;
        int v = z < L ? d[z] : 0;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, k);
            if (lane >= k) v += t;
        }
        if (z < L) o[z] = (unsigned long long)(carry + v);
        carry += __shfl_sync(0xffffffffu, v, 31);
    }
}

static size_t align64(size_t b) { return (b + 63) & ~(size_t)63; }

template <int CAP>
static int profile_group_run(cet_ctx *const *ctxs, int n, int axis, double ar_threshold, int64_t *out)
{
    cet_ctx *c0 = ctxs[0];
    cudaStream_t st = c0->stream;
    const int L = (int)c0->n1;
    const int64_t ns = c0->nloc;
    const size_t tab_bytes = align64((size_t)n * 4 * L * sizeof(unsigned long long));
    const size_t all_bytes = tab_bytes + (size_t)n * 2 * (L + 1) * sizeof(int);
    // per-context grain buffers (grow-only, shared with cet_metrics_group); n_grains is known since the labelling
    GroupArgs<PgArgs, CAP> t{};
    int max_ng = 0;
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        const size_t ng = (size_t)c->n_grains;
        const size_t need = align64(ng * sizeof(GrainStat)) + ng;
        if (c->cap_grain_st < need) {
            if (c->grain_st) { cudaFree(c->grain_st); c->grain_st = nullptr; c->cap_grain_st = 0; }
            CET_CUDA(cudaMalloc(&c->grain_st, need + need / 4));
            c->cap_grain_st = need + need / 4;
        }
        max_ng = std::max(max_ng, (int)ng);
    }
    if (c0->cap_profile_tab < all_bytes) {
        if (c0->profile_tab) { cudaFree(c0->profile_tab); c0->profile_tab = nullptr; c0->cap_profile_tab = 0; }
        CET_CUDA(cudaMalloc(&c0->profile_tab, all_bytes));
        c0->cap_profile_tab = all_bytes;
    }
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = ctxs[q];
        PgArgs &p = t.a[q];
        p.label = c->grain_label; p.gid = c->grain_gid;
        p.st = (GrainStat *)c->grain_st;
        p.cls = (uint8_t *)c->grain_st + align64((size_t)c->n_grains * sizeof(GrainStat));
        p.tab = (unsigned long long *)c0->profile_tab + (size_t)q * 4 * L;
        p.span = (int *)((char *)c0->profile_tab + tab_bytes) + (size_t)q * 2 * (L + 1);
        p.n_grains = (int)c->n_grains;
    }
    if (int rc = group_order(ctxs, n)) return rc;
    CET_CUDA(cudaMemsetAsync(c0->profile_tab, 0, all_bytes, st));
    const int gx = (int)std::min<int64_t>((ns + PG_THREADS - 1) / PG_THREADS, std::max(1, (sm_count(c0) * 16 + n - 1) / n));
    const int gg = (int)std::max<int64_t>(1, std::min<int64_t>((max_ng + 8 * PG_THREADS - 1) / (8 * PG_THREADS),
                                                               std::max(1, (sm_count(c0) * 8 + n - 1) / n)));
    const int gs = (int)((ns + PG_TILE - 1) / PG_TILE);
    profile_stats_init_group_kernel<CAP><<<dim3(gx, n), PG_THREADS, 0, st>>>(t, ns);
    profile_stats_group_kernel<CAP><<<dim3(gx, n), PG_THREADS, 0, st>>>(t, ns, L);
    profile_grains_group_kernel<CAP><<<dim3(gg, n), PG_THREADS, 4 * (L + 1) * sizeof(int), st>>>(t, L, axis, ar_threshold);
    profile_sites_group_kernel<CAP><<<dim3(gs, n), PG_THREADS, 2 * L * sizeof(unsigned int), st>>>(t, ns, L, axis);
    profile_finalize_group_kernel<CAP><<<n, 64, 0, st>>>(t, L);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(out, c0->profile_tab, (size_t)n * 4 * L * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CET_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" int cet_grain_profile_group(cet_ctx *const *ctxs, int32_t n_ctx, int32_t axis, double ar_threshold, int64_t *out)
{
    if (int rc = group_check("cet_grain_profile_group", ctxs, n_ctx)) return rc;
    CET_REQUIRE(out, "cet_grain_profile_group: NULL argument");
    CET_REQUIRE(axis >= 0 && axis <= 2, "cet_grain_profile_group: axis must be 0, 1 or 2, got %d", (int)axis);
    for (int q = 0; q < n_ctx; ++q) {
        const cet_ctx *c = ctxs[q];
        CET_REQUIRE(c->grain_label && c->grain_p_lo == 0 && c->grain_p_hi == c->np,
                    "cet_grain_profile_group: context %d has no labelling of the whole lattice (label its grains first)", q);
    }
    cet::DeviceGuard dg(ctxs[0]->device);
    return n_ctx <= 16 ? profile_group_run<16>(ctxs, n_ctx, axis, ar_threshold, out)
                       : profile_group_run<GROUP_MAX>(ctxs, n_ctx, axis, ar_threshold, out);
}
