// boundary_group.cu — per-plane bond counts and boundary misorientation of a group of whole-lattice contexts
// (cet_boundary_group): along one axis a, per plane z, the bonds of the model's neighbourhood graph (the 7 positive
// offsets of the labelling's union pass) counted by class (solid, boundary, interface) per offset, and the boundary
// bonds binned by the cosine d of the misorientation of their ends' orientations over caller-given edges, with the
// exact fixed-point sum F = sum llrint(d 2^32).  Occupancy and grains are those of the last labelling (label >= 0,
// equal labels); the call writes nothing a sweep, a metrics row, a profile, a shape, a front or a texture reads.  As
// in texture_group.cu a CTA takes its lattice's arguments from a table in kernel parameter space (blockIdx.y); a
// group of up to 16 launches the small table.
// One launch for the whole group: each CTA walks tiles of consecutive sites of its lattice and streams label (4 bytes
// per site); the 7 neighbour labels of a site come mostly from L1 / L2.  The orientations v[s] and v[t] are loaded for
// boundary bonds only, so a site with no bond class set costs its label loads alone.  The CTA's table of the L planes
// lives in shared memory: u32 counts and u64 sums F (two's complement, so the signed terms add as unsigned).  Along
// axes 0 and 1 a warp's sites lie in one or two planes: lanes of one plane add each count once (__match_any_sync on
// the site's plane, one ballot per bond class present in the warp), lanes of one (plane, bin) their bin count, and
// their F with one 32-bit reduction per 17-bit half; along axis 2 consecutive sites lie in distinct planes and every
// lane adds its own.  The CTA flushes its non-zero entries with 64-bit global atomics.  The table takes
// 8 L + 4 L (22 + n_edges) bytes plus the edges: past the 48 KB default the launch opts in to more dynamic shared
// memory.  One memset zeroes the group's table beforehand; one D2H copy returns it.
#include <algorithm>
#include "cadence.cuh"

namespace cet {

constexpr int BOUNDARY_EDGES_MAX = 31;
constexpr int BG_CLASSES = 21;      // 7 offsets x (solid, boundary, interface)

struct BgArgs {
    const int *label;
    const Vec4 *v;
    unsigned long long *tab;        // [L][n_edges + 23]: the lattice's part of the result table
};
static_assert(group_fits<BgArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

struct BgEdges {
    double e[BOUNDARY_EDGES_MAX];
};

constexpr int BG_THREADS = 256, BG_SITES_PER_THREAD = 16, BG_TILE = BG_THREADS * BG_SITES_PER_THREAD;
constexpr double BG_SCALE = 4294967296.0;     // 2^32

// the 7 positive offsets {0, 1, 4, 5, 8, 10, 12} of CET_NB_TABLE_INIT, in that order
__device__ constexpr int BG_OFF[7][3] = {{1, 1, 0}, {1, -1, 0}, {0, 1, 1}, {0, 1, -1}, {2, 0, 0}, {0, 2, 0}, {0, 0, 2}};

// dynamic shared memory: unsigned long long f[L] (F), double e[n_edges], unsigned h[L][22 + n_edges] (the 21 bond
// classes, then the boundary bonds per bin)
template <int CAP>
__global__ void __launch_bounds__(BG_THREADS) boundary_group_kernel(const __grid_constant__ GroupArgs<BgArgs, CAP> g,
                                                                   const __grid_constant__ BgEdges ed, int64_t n, int L,
                                                                   int axis, int n_edges)
{
    extern __shared__ unsigned long long f[];
    double *e = (double *)(f + L);
    unsigned *h = (unsigned *)(e + n_edges);
    const BgArgs &a = g.a[blockIdx.y];
    const int NC = BG_CLASSES + n_edges + 1, W = NC + 1, lane = threadIdx.x & 31, LL = L * L;
    // the offset whose bond lies in the plane below the site's along the axis (its component along the axis is -1)
    const int r_low = axis == 1 ? 1 : axis == 2 ? 3 : -1;
    for (int z = threadIdx.x; z < L; z += blockDim.x) f[z] = 0ull;
    for (int b = threadIdx.x; b < n_edges; b += blockDim.x) e[b] = ed.e[b];
    for (int z = threadIdx.x; z < L * NC; z += blockDim.x) h[z] = 0u;
    __syncthreads();
    for (int64_t base = (int64_t)blockIdx.x * BG_TILE; base < n; base += (int64_t)gridDim.x * BG_TILE) {
        for (int e0 = 0; e0 < BG_SITES_PER_THREAD; ++e0) {
            const int64_t s64 = base + e0 * BG_THREADS + threadIdx.x;
            const bool valid = s64 < n;
            const int s = valid ? (int)s64 : 0;
            const int i = s / LL, j = (s / L) % L, k = s % L;
            const int c = axis == 0 ? i : axis == 1 ? j : k;
            const int own = valid ? __ldg(a.label + s) : -1;
            int nl[7];
#pragma unroll
            for (int r = 0; r < 7; ++r) {
                const int ni = i + BG_OFF[r][0], nj = j + BG_OFF[r][1], nk = k + BG_OFF[r][2];
                const bool in = valid && ni < L && nj >= 0 && nj < L && nk >= 0 && nk < L;
                nl[r] = in ? __ldg(a.label + s + (BG_OFF[r][0] * L + BG_OFF[r][1]) * L + BG_OFF[r][2]) : -2;
            }
            unsigned sol = 0, bnd = 0, itf = 0;
#pragma unroll
            for (int r = 0; r < 7; ++r) {
                if (nl[r] == -2) continue;                              // outside the lattice: no bond
                const bool os = own >= 0, ot = nl[r] >= 0;
                if (os && ot) {
                    sol |= 1u << r;
                    if (own != nl[r]) bnd |= 1u << r;
                } else if (os != ot) {
                    itf |= 1u << r;
                }
            }
            // boundary bonds: bin and fixed-point term of d = clamp(fl(fl(fl(x x') + fl(y y')) + fl(z z')), -1, 1)
            unsigned long long bins = 0ull;                             // 5 bits per offset
            long long f_here = 0, f_low = 0;                            // F of the bonds in plane c and in plane c - 1
            if (bnd) {
                const Vec4 p = a.v[s];
#pragma unroll
                for (int r = 0; r < 7; ++r) {
                    if (!(bnd >> r & 1u)) continue;
                    const Vec4 q = a.v[s + (BG_OFF[r][0] * L + BG_OFF[r][1]) * L + BG_OFF[r][2]];
                    double d = __dadd_rn(__dadd_rn(__dmul_rn(p.x, q.x), __dmul_rn(p.y, q.y)), __dmul_rn(p.z, q.z));
                    d = pymax(pymin(d, 1.0), -1.0);
                    bins |= (unsigned long long)tg_bin(e, n_edges, d) << (5 * r);
                    const long long t = __double2ll_rn(__dmul_rn(d, BG_SCALE));              // in [-2^32, 2^32]
                    if (r == r_low) f_low = t;
                    else f_here += t;
                }
            }
            if (axis == 2) {                                            // consecutive sites: distinct planes
                const unsigned flags = sol | bnd << 7 | itf << 14;
                for (unsigned rem = flags; rem; rem &= rem - 1) {
                    const int bit = __ffs(rem) - 1, r = bit % 7, cls = bit / 7;
                    atomicAdd(&h[(c - (r == r_low)) * NC + 3 * r + cls], 1u);
                }
                for (unsigned rem = bnd; rem; rem &= rem - 1) {
                    const int r = __ffs(rem) - 1;
                    atomicAdd(&h[(c - (r == r_low)) * NC + BG_CLASSES + (int)(bins >> (5 * r) & 31u)], 1u);
                }
                if (bnd & ~(1u << 3)) atomicAdd(&f[c], (unsigned long long)f_here);
                if (bnd & (1u << 3)) atomicAdd(&f[c - 1], (unsigned long long)f_low);
            } else {                                                    // consecutive sites: one or two planes per warp
                const unsigned flags = sol | bnd << 7 | itf << 14;
                const unsigned peers = __match_any_sync(0xffffffffu, c);
                const bool leader = lane == __ffs(peers) - 1;
                const unsigned any = __reduce_or_sync(0xffffffffu, flags);
                for (unsigned rem = any; rem; rem &= rem - 1) {         // warp-uniform
                    const int bit = __ffs(rem) - 1, r = bit % 7, cls = bit / 7;
                    const unsigned m = __ballot_sync(0xffffffffu, flags >> bit & 1u) & peers;
                    if (leader && m) atomicAdd(&h[(c - (r == r_low)) * NC + 3 * r + cls], (unsigned)__popc(m));
                }
                for (unsigned rem = any >> 7 & 0x7Fu; rem; rem &= rem - 1) {
                    const int r = __ffs(rem) - 1;
                    const bool has = bnd >> r & 1u;
                    const unsigned act = __ballot_sync(0xffffffffu, has);
                    if (has) {
                        const int z = c - (r == r_low), b = (int)(bins >> (5 * r) & 31u);
                        const unsigned key = __match_any_sync(act, z * 32 + b);
                        if (lane == __ffs(key) - 1) atomicAdd(&h[z * NC + BG_CLASSES + b], (unsigned)__popc(key));
                    }
                }
                if (any >> 7) {
                    // F + 2^32 per bond is in [0, 2^33]; a lane's sum of at most 7 fits 36 bits, so 17-bit halves sum over
                    // 32 lanes without wrapping a u32
                    const unsigned n_here = __popc(bnd & ~(r_low >= 0 ? 1u << r_low : 0u)), n_low = r_low >= 0 ? (bnd >> r_low & 1u) : 0u;
                    const unsigned long long u0 = (unsigned long long)(f_here + ((long long)n_here << 32));
                    const unsigned long long u1 = (unsigned long long)(f_low + ((long long)n_low << 32));
                    const unsigned h0 = __reduce_add_sync(peers, (unsigned)(u0 >> 17)), l0 = __reduce_add_sync(peers, (unsigned)(u0 & 0x1FFFFu));
                    const unsigned c0 = __reduce_add_sync(peers, n_here);
                    const unsigned h1 = __reduce_add_sync(peers, (unsigned)(u1 >> 17)), l1 = __reduce_add_sync(peers, (unsigned)(u1 & 0x1FFFFu));
                    const unsigned c1 = __reduce_add_sync(peers, n_low);
                    if (leader && c0) atomicAdd(&f[c], ((unsigned long long)h0 << 17) + l0 - ((unsigned long long)c0 << 32));
                    if (leader && c1) atomicAdd(&f[c - 1], ((unsigned long long)h1 << 17) + l1 - ((unsigned long long)c1 << 32));
                }
            }
        }
    }
    __syncthreads();
    for (int z = threadIdx.x; z < L * NC; z += blockDim.x)
        if (h[z]) atomicAdd(&a.tab[(z / NC) * W + z % NC], (unsigned long long)h[z]);
    for (int z = threadIdx.x; z < L; z += blockDim.x)
        if (f[z]) atomicAdd(&a.tab[z * W + NC], f[z]);
}

template <int CAP>
static int boundary_group_run(cet_ctx *const *ctxs, int n, int axis, const double *edges, int n_edges, int64_t *out,
                              size_t smem)
{
    cet_ctx *c0 = ctxs[0];
    cudaStream_t st = c0->stream;
    const int L = (int)c0->n1, W = BG_CLASSES + n_edges + 2;
    const int64_t ns = c0->nloc;
    const size_t tab_bytes = (size_t)n * L * W * sizeof(unsigned long long);
    if (c0->cap_boundary_tab < tab_bytes) {
        if (c0->boundary_tab) { cudaFree(c0->boundary_tab); c0->boundary_tab = nullptr; c0->cap_boundary_tab = 0; }
        CET_CUDA(cudaMalloc(&c0->boundary_tab, tab_bytes));
        c0->cap_boundary_tab = tab_bytes;
    }
    GroupArgs<BgArgs, CAP> t{};
    for (int q = 0; q < n; ++q) {
        BgArgs &p = t.a[q];
        p.label = ctxs[q]->grain_label;
        p.v = ctxs[q]->v;
        p.tab = (unsigned long long *)c0->boundary_tab + (size_t)q * L * W;
    }
    BgEdges ed{};
    for (int b = 0; b < n_edges; ++b) ed.e[b] = edges[b];
    if (smem > 48 * 1024)
        CET_CUDA(cudaFuncSetAttribute(boundary_group_kernel<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CET_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, boundary_group_kernel<CAP>, BG_THREADS, smem));
    // one wave over the group: every CTA zeroes and flushes a whole table, so more CTAs only add flushes
    const int gx = (int)std::min<int64_t>((ns + BG_TILE - 1) / BG_TILE, std::max(1, (sm_count(c0) * std::max(per_sm, 1) + n - 1) / n));
    if (int rc = group_order(ctxs, n)) return rc;
    CET_CUDA(cudaMemsetAsync(c0->boundary_tab, 0, tab_bytes, st));
    boundary_group_kernel<CAP><<<dim3(gx, n), BG_THREADS, smem, st>>>(t, ed, ns, L, axis, n_edges);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(out, c0->boundary_tab, tab_bytes, cudaMemcpyDeviceToHost, st));
    CET_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" int cet_boundary_group(cet_ctx *const *ctxs, int32_t n_ctx, int32_t axis, const double *edges,
                                  int32_t n_edges, int64_t *out)
{
    if (int rc = group_check("cet_boundary_group", ctxs, n_ctx)) return rc;
    CET_REQUIRE(edges && out, "cet_boundary_group: NULL argument");
    CET_REQUIRE(axis >= 0 && axis <= 2, "cet_boundary_group: axis must be 0, 1 or 2, got %d", (int)axis);
    CET_REQUIRE(n_edges >= 1 && n_edges <= BOUNDARY_EDGES_MAX, "cet_boundary_group: need 1 <= n_edges <= %d, got %d",
                BOUNDARY_EDGES_MAX, (int)n_edges);
    for (int b = 0; b < n_edges; ++b) {
        CET_REQUIRE(finite_f64(edges[b]) && edges[b] >= -1.0 && edges[b] <= 1.0,
                    "cet_boundary_group: edge %d is not finite and within [-1, 1]", b);
        CET_REQUIRE(b == 0 || edges[b] > edges[b - 1], "cet_boundary_group: edges must ascend strictly (edge %d)", b);
    }
    const int L = (int)ctxs[0]->n1;
    const size_t smem = (size_t)L * sizeof(unsigned long long) + (size_t)n_edges * sizeof(double) +
                        (size_t)L * (BG_CLASSES + n_edges + 1) * sizeof(unsigned);
    cet::DeviceGuard dg(ctxs[0]->device);
    int optin = 0;
    CET_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctxs[0]->device));
    CET_REQUIRE(smem <= (size_t)optin, "cet_boundary_group: a table of L = %d planes and m = %d edges needs %zu bytes of "
                "shared memory, the device allows %d", L, (int)n_edges, smem, optin);
    for (int q = 0; q < n_ctx; ++q) {
        const cet_ctx *c = ctxs[q];
        CET_REQUIRE(c->v, "cet_boundary_group: context %d has no orientation vectors", q);
        CET_REQUIRE(c->grain_label && c->grain_p_lo == 0 && c->grain_p_hi == c->np,
                    "cet_boundary_group: context %d has no labelling of the whole lattice (label its grains first)", q);
    }
    return n_ctx <= 16 ? boundary_group_run<16>(ctxs, n_ctx, axis, edges, n_edges, out, smem)
                       : boundary_group_run<GROUP_MAX>(ctxs, n_ctx, axis, edges, n_edges, out, smem);
}
