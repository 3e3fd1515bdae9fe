// grains.cu — grain clustering and per-grain statistics on the device (SURVEY §8f row N1).
//
// The reference grows grains with a pure-Python DFS (utils.py:28-84): a grain is a connected
// component of the graph whose edges join occupied sites (state != 0, defects included) that are
// neighbours (the 14-offset set, kmc_event_rates.py:29-36) with misorientation < theta_threshold
// (metrics.py:43 passes 0.5 rad).  A DFS started at an unvisited site visits exactly that site's
// component, and the edge relation is symmetric, so the components do not depend on the visiting
// order: a lock-free union-find over the 7 "positive" offsets reproduces them exactly.  The
// reference numbers grains in raster order of their first voxel = the smallest site index of the
// component = the root chosen by union-by-minimum, so sorting the roots gives its cluster order.
// Per grain: voxel count and bounding box (utils.py:104-111 aspect ratio).
//
// misorientation < t  <=>  arccos(clamp(v1.v2)) < t  <=>  clamp(v1.v2) > cos t, evaluated on the
// resident unit vectors (kmc_event_rates.py:11-23).
#include <algorithm>
#include "cadence.cuh"

namespace cet {

__global__ void grains_init_kernel(const uint8_t *__restrict__ vox, int *label, int64_t lo, int64_t hi)
{
    grains_init_body(vox, label, lo, hi);
}

__global__ void grains_union_kernel(const uint8_t *__restrict__ vox, const Vec4 *__restrict__ v, const double *__restrict__ theta,
                                    int *label, int L, int p_lo, int p_hi, double thr)
{
    grains_union_body(vox, v, theta, label, L, p_lo, p_hi, thr);
}

// label[s] := root of s; roots counted and given dense ids in order of arrival (the host orders
// the grains by root index afterwards)
__global__ void grains_flatten_kernel(int *label, int *gid, int64_t lo, int64_t hi, unsigned int *n_roots)
{
    grains_flatten_body<true>(label, gid, lo, hi, n_roots);
}

__global__ void grains_stats_init_kernel(const int *__restrict__ label, const int *__restrict__ gid, int64_t lo,
                                         int64_t hi, GrainStat *st)
{
    for (int64_t s = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < hi; s += (int64_t)gridDim.x * blockDim.x) {
        if (label[s] != (int)s) continue;
        grain_stat_init(st + gid[s], (int)s);
    }
}

__global__ void grains_stats_kernel(const int *__restrict__ label, const int *__restrict__ gid, int64_t lo, int64_t hi,
                                    GrainStat *st, int L, int i_off)
{
    grains_stats_body(label, gid, lo, hi, st, L, i_off);
}

}  // namespace cet

using namespace cet;

extern "C" {

// utils.get_clusters (utils.py:69-84) on the resident lattice: label the grains of the owned
// planes.  n_grains receives the number of components.
int cet_grains_label_ex(cet_ctx *c, double theta_threshold, int criterion, int64_t *n_grains);
int cet_grains_download_planes(cet_ctx *c, int64_t i_lo, int64_t i_hi, int32_t *labels);
int cet_grains_label(cet_ctx *c, double theta_threshold, int64_t *n_grains)
{
    return cet_grains_label_ex(c, theta_threshold, 0, n_grains);
}

// criterion 0: misorientation of the orientation vectors < threshold (utils.py:51-56, what metrics.py uses);
// criterion 1: |theta1 - theta2| < threshold (utils.py:49-50, get_clusters(..., orientation_phi=None)).
int cet_grains_label_ex(cet_ctx *c, double theta_threshold, int criterion, int64_t *n_grains)
{
    CET_REQUIRE(c && n_grains && c->cubic, "cet_grains_label: bad argument");
    CET_REQUIRE(criterion == 0 || criterion == 1, "cet_grains_label: unknown criterion %d", criterion);
    CET_REQUIRE(c->nloc < (1ll << 31) && c->n0 * c->plane < (1ll << 31),
                "cet_grains_label: the lattice must have fewer than 2^31 sites");
    CET_REQUIRE(c->halo == 0 || c->halo >= 2, "cet_grains_label: a slab needs at least 2 ghost planes");
    cet::DeviceGuard dg(c->device);
    if (!c->grain_label) CET_CUDA(cudaMalloc(&c->grain_label, (size_t)c->nloc * sizeof(int)));
    if (!c->grain_gid) CET_CUDA(cudaMalloc(&c->grain_gid, (size_t)c->nloc * sizeof(int)));
    if (int rc = ensure_stage(c, 64)) return rc;
    unsigned int *cnt = (unsigned int *)c->stage;
    CET_CUDA(cudaMemsetAsync(cnt, 0, 64, c->stream));
    // A slab labels its owned planes plus 2 ghost planes per cut face (the reach of the neighbourhood
    // along axis 0): a grain that crosses the cut is then a local component on both sides, joined by
    // the host through the labels both slabs give the shared planes (metrics.grains_distributed).
    const int i_off = (int)(c->i_begin - c->halo);
    int p_lo = c->halo >= 2 ? c->halo - 2 : 0, p_hi = (int)c->np - (c->halo >= 2 ? c->halo - 2 : 0);
    if (i_off + p_lo < 0) p_lo = -i_off;
    if (i_off + p_hi > c->n0) p_hi = (int)(c->n0 - i_off);
    c->grain_p_lo = p_lo; c->grain_p_hi = p_hi;
    const int64_t lo = (int64_t)p_lo * c->plane, hi = (int64_t)p_hi * c->plane;
    const int grid = (int)std::min<int64_t>((hi - lo + 255) / 256, (int64_t)sm_count(c) * 16);
    grains_init_kernel<<<grid, 256, 0, c->stream>>>(c->vox, c->grain_label, lo, hi);
    grains_union_kernel<<<grid, 256, 0, c->stream>>>(c->vox, c->v, criterion == 1 ? c->theta : nullptr, c->grain_label, (int)c->n1,
                                                     p_lo, p_hi, criterion == 1 ? theta_threshold : cos(theta_threshold));
    grains_flatten_kernel<<<grid, 256, 0, c->stream>>>(c->grain_label, c->grain_gid, lo, hi, cnt);
    CET_CUDA(cudaGetLastError());
    unsigned int h = 0;
    CET_CUDA(cudaMemcpyAsync(&h, cnt, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    c->n_grains = h;
    *n_grains = (int64_t)h;
    return 0;
}

// Per-grain statistics of the last cet_grains_label call, in arbitrary order (the caller sorts
// by root to obtain the reference's cluster order): root[g] = smallest site index of the grain
// (its first voxel in raster order), size[g] = voxel count (len(cluster)), box_lo / box_hi
// [3*g + axis] = bounding box (utils.py:104-111).  cap >= n_grains.
int cet_grains_stats(cet_ctx *c, int64_t cap, int32_t *root, int32_t *size, int32_t *box_lo, int32_t *box_hi)
{
    CET_REQUIRE(c && c->grain_label, "cet_grains_stats: call cet_grains_label first");
    CET_REQUIRE(cap >= (int64_t)c->n_grains, "cet_grains_stats: capacity %lld < %lld grains", (long long)cap,
                (long long)c->n_grains);
    cet::DeviceGuard dg(c->device);
    const unsigned int n = (unsigned int)c->n_grains;
    if (n == 0) return 0;
    GrainStat *st = nullptr;
    CET_CUDA(cudaMalloc(&st, (size_t)n * sizeof(GrainStat)));
    // roots anywhere in the labelled planes; voxels counted on the OWNED planes only, so that the
    // statistics of a grain that spans several slabs add up (a local component without owned voxels
    // reports size 0)
    const int64_t lo = (int64_t)c->grain_p_lo * c->plane, hi = (int64_t)c->grain_p_hi * c->plane;
    const int64_t o_lo = c->owned_offset(), o_hi = o_lo + c->owned_sites();
    const int grid = (int)std::min<int64_t>((hi - lo + 255) / 256, (int64_t)sm_count(c) * 16);
    grains_stats_init_kernel<<<grid, 256, 0, c->stream>>>(c->grain_label, c->grain_gid, lo, hi, st);
    grains_stats_kernel<<<grid, 256, 0, c->stream>>>(c->grain_label, c->grain_gid, o_lo, o_hi, st, (int)c->n1,
                                                     (int)(c->i_begin - c->halo));
    std::vector<GrainStat> h(n);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), st, (size_t)n * sizeof(GrainStat), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(st);
    if (e != cudaSuccess) { set_error("cet_grains_stats: %s", cudaGetErrorString(e)); return 1000 + (int)e; }
    const int root_off = (int)((c->i_begin - c->halo) * c->plane);       // local -> global site index
    for (unsigned int g = 0; g < n; ++g) {
        if (root) root[g] = h[g].root + root_off;
        if (size) size[g] = h[g].size;
        for (int ax = 0; ax < 3; ++ax) {
            if (box_lo) box_lo[3 * g + ax] = h[g].lo[ax];
            if (box_hi) box_hi[3 * g + ax] = h[g].hi[ax];
        }
    }
    return 0;
}

// Label volume: root site index per occupied site (the grain's first voxel in raster order),
// -1 for empty sites.  The reference's `visited` volume (utils.py:75-84) is rank-of-root + 1.
int cet_grains_download_labels(cet_ctx *c, int32_t *labels)
{
    CET_REQUIRE(c, "cet_grains_download_labels: NULL ctx");
    return cet_grains_download_planes(c, c->i_begin, c->i_end, labels);
}

// Labels (GLOBAL site index of the local root, -1 for empty sites) of global planes [i_lo, i_hi), which
// must lie within the planes the last cet_grains_label call labelled (owned + 2 ghost planes per cut face).
int cet_grains_download_planes(cet_ctx *c, int64_t i_lo, int64_t i_hi, int32_t *labels)
{
    CET_REQUIRE(c && labels && c->grain_label, "cet_grains_download_planes: call cet_grains_label first");
    const int64_t i_off = c->i_begin - c->halo;
    CET_REQUIRE(i_lo < i_hi && i_lo - i_off >= c->grain_p_lo && i_hi - i_off <= c->grain_p_hi,
                "cet_grains_download_planes: planes [%lld, %lld) were not labelled", (long long)i_lo, (long long)i_hi);
    cet::DeviceGuard dg(c->device);
    const int64_t n = (i_hi - i_lo) * c->plane;
    CET_CUDA(cudaMemcpyAsync(labels, c->grain_label + (i_lo - i_off) * c->plane, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost,
                             c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    const int off = (int)(i_off * c->plane);
    if (off)
        for (int64_t q = 0; q < n; ++q)
            if (labels[q] >= 0) labels[q] += off;
    return 0;
}

}  // extern "C"
