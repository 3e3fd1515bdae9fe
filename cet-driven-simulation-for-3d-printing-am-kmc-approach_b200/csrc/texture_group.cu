// texture_group.cu — per-plane orientation histograms of a group of whole-lattice contexts (cet_texture_group): along
// one axis a, per plane z, the occupied sites binned by c = v[a] (the cosine between the resident orientation and +a)
// over caller-given edges, and the exact fixed-point sums F1 = sum llrint(c 2^32), F2 = sum llrint(fl(c c) 2^32).
// The call needs no labelling; it reads vox and v and writes nothing a sweep, a metrics row, a profile, a shape
// histogram or a front reads.  As in profile_group.cu a CTA takes its lattice's arguments from a table in kernel
// parameter space (blockIdx.y); a group of up to 16 launches the small table.
// One launch for the whole group: each CTA walks tiles of consecutive sites of its lattice, streams vox once (one
// byte per site) and loads the one component v[s][a] of occupied sites only.  Its table of the L planes lives in
// shared memory: u32 bin counts and u64 sums (two's complement, so the signed F1 adds as unsigned).  Along axes 0 and
// 1 a warp's sites lie in a few planes: lanes of one plane add their sums with one 32-bit reduction per 17-bit half
// (below) and lanes of one (plane, bin) their count, so a warp makes one shared atomic per distinct key; along axis 2
// consecutive sites lie in distinct planes and every lane adds its own.  The CTA flushes its non-zero entries with
// 64-bit global atomics.  The table takes 16 L + 4 L (n_edges + 1) bytes plus the edges: past the 48 KB default
// (L >= 342 with 31 edges) the launch opts in to more dynamic shared memory, which covers every whole-lattice L.
// One memset zeroes the group's table beforehand; one D2H copy returns it.
#include <algorithm>
#include "cadence.cuh"

namespace cet {

constexpr int TEXTURE_EDGES_MAX = 31;

struct TgArgs {
    const uint8_t *vox;
    const double *c;                // &v[0].x + axis: the component along the axis, 4 doubles per site
    unsigned long long *tab;        // [L][n_edges + 3]: the lattice's part of the result table
};
static_assert(group_fits<TgArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

struct TgEdges {
    double e[TEXTURE_EDGES_MAX];
};

constexpr int TG_THREADS = 256, TG_SITES_PER_THREAD = 16, TG_TILE = TG_THREADS * TG_SITES_PER_THREAD;
constexpr double TG_SCALE = 4294967296.0;     // 2^32

__device__ __forceinline__ int tg_plane(int s, int L, int axis)
{
    return axis == 0 ? s / (L * L) : axis == 1 ? (s / L) % L : s % L;
}

// dynamic shared memory: unsigned long long f[L][2] (F1, F2), double e[n_edges], unsigned h[L][n_edges + 1]
template <int CAP>
__global__ void __launch_bounds__(TG_THREADS) texture_group_kernel(const __grid_constant__ GroupArgs<TgArgs, CAP> g,
                                                                  const __grid_constant__ TgEdges ed, int64_t n, int L,
                                                                  int axis, int n_edges)
{
    extern __shared__ unsigned long long f[];
    double *e = (double *)(f + 2 * L);
    unsigned *h = (unsigned *)(e + n_edges);
    const TgArgs &a = g.a[blockIdx.y];
    const int nb = n_edges + 1, W = n_edges + 3, lane = threadIdx.x & 31;
    for (int z = threadIdx.x; z < 2 * L; z += blockDim.x) f[z] = 0ull;
    for (int b = threadIdx.x; b < n_edges; b += blockDim.x) e[b] = ed.e[b];
    for (int z = threadIdx.x; z < L * nb; z += blockDim.x) h[z] = 0u;
    __syncthreads();
    constexpr int U = 4;                                        // sites per thread in flight
    for (int64_t base = (int64_t)blockIdx.x * TG_TILE; base < n; base += (int64_t)gridDim.x * TG_TILE) {
        for (int e0 = 0; e0 < TG_SITES_PER_THREAD; e0 += U) {
            uint8_t b8[U];
            double c[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t s = base + (e0 + u) * TG_THREADS + threadIdx.x;
                b8[u] = s < n ? __ldg(a.vox + s) : (uint8_t)0;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t s = base + (e0 + u) * TG_THREADS + threadIdx.x;
                c[u] = (b8[u] & 0x0F) ? __ldg(a.c + 4 * s) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int s = (int)(base + (e0 + u) * TG_THREADS + threadIdx.x);
                const bool occ = (b8[u] & 0x0F) != 0;
                const int z = occ ? tg_plane(s, L, axis) : 0;
                const int bin = occ ? tg_bin(e, n_edges, c[u]) : 0;
                const long long f1 = __double2ll_rn(__dmul_rn(c[u], TG_SCALE));                      // in [-2^32, 2^32]
                const long long f2 = __double2ll_rn(__dmul_rn(__dmul_rn(c[u], c[u]), TG_SCALE));     // in [0, 2^32]
                if (axis == 2) {                                        // consecutive sites: distinct planes
                    if (occ) {
                        atomicAdd(&h[z * nb + bin], 1u);
                        atomicAdd(&f[2 * z], (unsigned long long)f1);
                        atomicAdd(&f[2 * z + 1], (unsigned long long)f2);
                    }
                } else {                                                // consecutive sites: few planes per warp
                    const unsigned act = __ballot_sync(0xffffffffu, occ);
                    if (!occ) continue;
                    const unsigned key = __match_any_sync(act, z * nb + bin);
                    if (lane == __ffs(key) - 1) atomicAdd(&h[z * nb + bin], (unsigned)__popc(key));
                    // f1 + 2^32 and f2 fit 34 bits: 17-bit halves sum over 32 lanes without wrapping a u32
                    const unsigned peers = __match_any_sync(act, z);
                    const unsigned long long u1 = (unsigned long long)(f1 + (1ll << 32)), u2 = (unsigned long long)f2;
                    const unsigned h1 = __reduce_add_sync(peers, (unsigned)(u1 >> 17)), l1 = __reduce_add_sync(peers, (unsigned)(u1 & 0x1FFFFu));
                    const unsigned h2 = __reduce_add_sync(peers, (unsigned)(u2 >> 17)), l2 = __reduce_add_sync(peers, (unsigned)(u2 & 0x1FFFFu));
                    if (lane == __ffs(peers) - 1) {
                        atomicAdd(&f[2 * z], ((unsigned long long)h1 << 17) + l1 - ((unsigned long long)__popc(peers) << 32));
                        atomicAdd(&f[2 * z + 1], ((unsigned long long)h2 << 17) + l2);
                    }
                }
            }
        }
    }
    __syncthreads();
    for (int z = threadIdx.x; z < L * nb; z += blockDim.x)
        if (h[z]) atomicAdd(&a.tab[(z / nb) * W + z % nb], (unsigned long long)h[z]);
    for (int z = threadIdx.x; z < 2 * L; z += blockDim.x)
        if (f[z]) atomicAdd(&a.tab[(z >> 1) * W + nb + (z & 1)], f[z]);
}

template <int CAP>
static int texture_group_run(cet_ctx *const *ctxs, int n, int axis, const double *edges, int n_edges, int64_t *out,
                             size_t smem)
{
    cet_ctx *c0 = ctxs[0];
    cudaStream_t st = c0->stream;
    const int L = (int)c0->n1, W = n_edges + 3;
    const int64_t ns = c0->nloc;
    const size_t tab_bytes = (size_t)n * L * W * sizeof(unsigned long long);
    if (c0->cap_texture_tab < tab_bytes) {
        if (c0->texture_tab) { cudaFree(c0->texture_tab); c0->texture_tab = nullptr; c0->cap_texture_tab = 0; }
        CET_CUDA(cudaMalloc(&c0->texture_tab, tab_bytes));
        c0->cap_texture_tab = tab_bytes;
    }
    GroupArgs<TgArgs, CAP> t{};
    for (int q = 0; q < n; ++q) {
        TgArgs &p = t.a[q];
        p.vox = ctxs[q]->vox;
        p.c = &ctxs[q]->v[0].x + axis;
        p.tab = (unsigned long long *)c0->texture_tab + (size_t)q * L * W;
    }
    TgEdges ed{};
    for (int b = 0; b < n_edges; ++b) ed.e[b] = edges[b];
    if (smem > 48 * 1024)
        CET_CUDA(cudaFuncSetAttribute(texture_group_kernel<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CET_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, texture_group_kernel<CAP>, TG_THREADS, smem));
    // one wave over the group: every CTA zeroes and flushes a whole table, so more CTAs only add flushes
    const int gx = (int)std::min<int64_t>((ns + TG_TILE - 1) / TG_TILE, std::max(1, (sm_count(c0) * std::max(per_sm, 1) + n - 1) / n));
    if (int rc = group_order(ctxs, n)) return rc;
    CET_CUDA(cudaMemsetAsync(c0->texture_tab, 0, tab_bytes, st));
    texture_group_kernel<CAP><<<dim3(gx, n), TG_THREADS, smem, st>>>(t, ed, ns, L, axis, n_edges);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(out, c0->texture_tab, tab_bytes, cudaMemcpyDeviceToHost, st));
    CET_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" int cet_texture_group(cet_ctx *const *ctxs, int32_t n_ctx, int32_t axis, const double *edges,
                                 int32_t n_edges, int64_t *out)
{
    if (int rc = group_check("cet_texture_group", ctxs, n_ctx)) return rc;
    CET_REQUIRE(edges && out, "cet_texture_group: NULL argument");
    CET_REQUIRE(axis >= 0 && axis <= 2, "cet_texture_group: axis must be 0, 1 or 2, got %d", (int)axis);
    CET_REQUIRE(n_edges >= 1 && n_edges <= TEXTURE_EDGES_MAX, "cet_texture_group: need 1 <= n_edges <= %d, got %d",
                TEXTURE_EDGES_MAX, (int)n_edges);
    for (int b = 0; b < n_edges; ++b) {
        CET_REQUIRE(finite_f64(edges[b]) && edges[b] >= -1.0 && edges[b] <= 1.0,
                    "cet_texture_group: edge %d is not finite and within [-1, 1]", b);
        CET_REQUIRE(b == 0 || edges[b] > edges[b - 1], "cet_texture_group: edges must ascend strictly (edge %d)", b);
    }
    for (int q = 0; q < n_ctx; ++q)
        CET_REQUIRE(ctxs[q]->v, "cet_texture_group: context %d has no orientation vectors", q);
    const int L = (int)ctxs[0]->n1;
    const size_t smem = (size_t)L * 2 * sizeof(unsigned long long) + (size_t)n_edges * sizeof(double) +
                        (size_t)L * (n_edges + 1) * sizeof(unsigned);
    cet::DeviceGuard dg(ctxs[0]->device);
    int optin = 0;
    CET_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctxs[0]->device));
    CET_REQUIRE(smem <= (size_t)optin, "cet_texture_group: a table of L = %d planes and %d bins needs %zu bytes of shared "
                "memory, the device allows %d", L, (int)n_edges + 1, smem, optin);
    return n_ctx <= 16 ? texture_group_run<16>(ctxs, n_ctx, axis, edges, n_edges, out, smem)
                       : texture_group_run<GROUP_MAX>(ctxs, n_ctx, axis, edges, n_edges, out, smem);
}
