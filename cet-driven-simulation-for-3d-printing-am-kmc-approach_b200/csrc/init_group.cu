// init_group.cu — cet_init_group: the initial lattices of a group of whole-lattice contexts built on the device.
// An initial lattice (lattice_init.py:10-59 + defects.py:4-31) is empty but for a few nuclei on the k = 0 plane,
// and its temperature depends on k only.  So the caller sends the nuclei and one temperature row per lattice, one
// launch writes the empty-site record of every site of the group, and a second one writes the nuclei over it: the
// same fields, with the same bits, as cet_upload of the dense arrays.
#include <algorithm>
#include "ctx.cuh"

namespace cet {

struct InitGroupArgs {
    uint8_t *vox, *vox_prev;         // vox_prev NULL: no snapshot
    double *theta, *phi, *T;
    Vec4 *v;
    const double *row;               // T along k (device copy)
    const int64_t *site;             // nuclei (device copies)
    const uint8_t *byte;
    const double *th, *ph;
    int64_t n_nuc;
};
static_assert(group_fits<InitGroupArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

constexpr int INIT_BLOCK = 256;

// blockIdx.y = lattice; every site of it takes the empty-site record
template <int CAP>
__global__ void __launch_bounds__(INIT_BLOCK)
init_fill_kernel(const __grid_constant__ GroupArgs<InitGroupArgs, CAP> g, int L, int64_t n)
{
    const InitGroupArgs &a = g.a[blockIdx.y];
    const Vec4 v0 = unit_vec4(0.0, 0.0);                   // orient_kernel's value of an empty site
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
        a.vox[s] = 0;
        a.theta[s] = 0.0;
        a.phi[s] = 0.0;
        a.v[s] = v0;
        a.T[s] = a.row[s % L];
        if (a.vox_prev) a.vox_prev[s] = 0;
    }
}

// blockIdx.y = lattice; its nuclei, after the fill (same stream)
template <int CAP>
__global__ void __launch_bounds__(INIT_BLOCK)
init_scatter_kernel(const __grid_constant__ GroupArgs<InitGroupArgs, CAP> g)
{
    const InitGroupArgs &a = g.a[blockIdx.y];
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < a.n_nuc; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = a.site[q];
        const uint8_t b = a.byte[q];
        const double th = a.th[q], ph = a.ph[q];
        a.vox[s] = b;
        a.theta[s] = th;
        a.phi[s] = ph;
        a.v[s] = unit_vec4(th, ph);
        if (a.vox_prev) a.vox_prev[s] = b;
    }
}

template <int CAP>
static int init_group_launch(cet_ctx *c0, const InitGroupArgs *args, int n, int64_t max_nuc)
{
    GroupArgs<InitGroupArgs, CAP> g;
    for (int q = 0; q < n; ++q) g.a[q] = args[q];
    const int64_t sites = c0->nloc;
    // enough CTAs to fill the device once over the whole group; each thread then strides over its lattice
    const int64_t want = std::max<int64_t>(1, (int64_t)sm_count(c0) * 16 / n);
    const int64_t gx = std::min<int64_t>((sites + INIT_BLOCK - 1) / INIT_BLOCK, want);
    init_fill_kernel<CAP><<<dim3((unsigned)gx, (unsigned)n), INIT_BLOCK, 0, c0->stream>>>(g, (int)c0->n2, sites);
    CET_CUDA(cudaGetLastError());
    if (max_nuc > 0) {
        init_scatter_kernel<CAP><<<dim3((unsigned)((max_nuc + INIT_BLOCK - 1) / INIT_BLOCK), (unsigned)n), INIT_BLOCK, 0,
                                   c0->stream>>>(g);
        CET_CUDA(cudaGetLastError());
    }
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" {

int cet_init_group(cet_ctx *const *ctxs, int32_t n_ctx, const cet_init_desc *d, int32_t snapshot)
{
    CET_REQUIRE(ctxs && d, "cet_init_group: NULL argument");
    CET_REQUIRE(n_ctx >= 1 && n_ctx <= GROUP_MAX, "cet_init_group: need 1 <= n_ctx <= %d, got %d", GROUP_MAX, (int)n_ctx);
    int64_t n_total = 0, max_nuc = 0;
    for (int q = 0; q < n_ctx; ++q) {
        const cet_ctx *c = ctxs[q];
        CET_REQUIRE(c, "cet_init_group: context %d is NULL", q);
        for (int r = 0; r < q; ++r) CET_REQUIRE(ctxs[r] != c, "cet_init_group: context %d repeats context %d", q, r);
        CET_REQUIRE(c->device == ctxs[0]->device, "cet_init_group: context %d is on another device", q);
        CET_REQUIRE(c->world == 1 && c->halo == 0 && c->i_begin == 0 && c->i_end == c->n0,
                    "cet_init_group: context %d is a slab; groups take whole-lattice contexts", q);
        CET_REQUIRE(c->cubic && c->n0 == c->n1 && c->n1 == c->n2, "cet_init_group: context %d is not a cubic lattice", q);
        CET_REQUIRE(c->n1 == ctxs[0]->n1, "cet_init_group: context %d has L = %lld, context 0 L = %lld", q,
                    (long long)c->n1, (long long)ctxs[0]->n1);
        const cet_init_desc &e = d[q];
        CET_REQUIRE(e.T_row, "cet_init_group: context %d: T_row is NULL", q);
        CET_REQUIRE(e.n_nuclei >= 0 && e.n_nuclei <= c->plane, "cet_init_group: context %d: %lld nuclei for %lld sites of "
                    "the k = 0 plane", q, (long long)e.n_nuclei, (long long)c->plane);
        CET_REQUIRE(e.n_nuclei == 0 || (e.site && e.byte && e.theta && e.phi),
                    "cet_init_group: context %d: NULL nucleus array with %lld nuclei", q, (long long)e.n_nuclei);
        n_total += e.n_nuclei;
        max_nuc = std::max(max_nuc, e.n_nuclei);
    }
    {
        const int64_t L = ctxs[0]->n1, plane = ctxs[0]->plane;
        std::vector<uint8_t> seen((size_t)plane);
        for (int q = 0; q < n_ctx; ++q) {
            const cet_init_desc &e = d[q];
            std::fill(seen.begin(), seen.end(), 0);
            for (int64_t i = 0; i < e.n_nuclei; ++i) {
                const int64_t s = e.site[i];
                CET_REQUIRE(s >= 0 && s < plane * L && s % L == 0,
                            "cet_init_group: context %d: nucleus %lld at site %lld, outside the k = 0 plane of the lattice",
                            q, (long long)i, (long long)s);
                CET_REQUIRE(!seen[s / L], "cet_init_group: context %d: nucleus %lld repeats site %lld", q, (long long)i,
                            (long long)s);
                seen[s / L] = 1;
                const int st = e.byte[i] & 15, df = e.byte[i] >> 4;
                CET_REQUIRE(st >= 1 && st <= 3 && df <= 1,
                            "cet_init_group: context %d: nucleus %lld has byte 0x%02x (state 1..3, defect 0..1)", q,
                            (long long)i, (unsigned)e.byte[i]);
            }
        }
    }
    cet::DeviceGuard dg(ctxs[0]->device);
    cet_ctx *c0 = ctxs[0];
    const int64_t L = c0->n1;
    // packed table: rows (n_ctx * L doubles) | theta | phi | site | byte, every section 8-byte aligned
    const size_t b_rows = (size_t)n_ctx * L * 8, b_th = (size_t)n_total * 8, b_site = (size_t)n_total * 8;
    const size_t o_th = b_rows, o_ph = o_th + b_th, o_site = o_ph + b_th, o_byte = o_site + b_site;
    const size_t bytes = o_byte + (size_t)n_total;
    std::vector<unsigned char> h(bytes);
    InitGroupArgs args[GROUP_MAX];
    if (int rc = ensure_stage(c0, bytes)) return rc;
    unsigned char *dev = (unsigned char *)c0->stage;
    int64_t off = 0;
    for (int q = 0; q < n_ctx; ++q) {
        cet_ctx *c = ctxs[q];
        const cet_init_desc &e = d[q];
        const size_t nb = (size_t)e.n_nuclei;
        memcpy(h.data() + (size_t)q * L * 8, e.T_row, (size_t)L * 8);
        if (nb) {
            memcpy(h.data() + o_th + off * 8, e.theta, nb * 8);
            memcpy(h.data() + o_ph + off * 8, e.phi, nb * 8);
            memcpy(h.data() + o_site + off * 8, e.site, nb * 8);
            memcpy(h.data() + o_byte + off, e.byte, nb);
        }
        if (snapshot && !c->vox_prev) CET_CUDA(cudaMalloc(&c->vox_prev, c->nloc));
        InitGroupArgs &a = args[q];
        a.vox = c->vox; a.vox_prev = snapshot ? c->vox_prev : nullptr;
        a.theta = c->theta; a.phi = c->phi; a.T = c->T; a.v = c->v;
        a.row = (const double *)(dev + (size_t)q * L * 8);
        a.th = (const double *)(dev + o_th + off * 8);
        a.ph = (const double *)(dev + o_ph + off * 8);
        a.site = (const int64_t *)(dev + o_site + off * 8);
        a.byte = dev + o_byte + off;
        a.n_nuc = e.n_nuclei;
        off += e.n_nuclei;
        if (c != c0) {
            if (!c->ev_group) CET_CUDA(cudaEventCreateWithFlags(&c->ev_group, cudaEventDisableTiming));
            CET_CUDA(cudaEventRecord(c->ev_group, c->stream));
            CET_CUDA(cudaStreamWaitEvent(c0->stream, c->ev_group, 0));
        }
    }
    // as cet_upload: everything derived from the lattice is stale from here on, also when the call fails half way
    for (int q = 0; q < n_ctx; ++q) {
        lattice_changed(ctxs[q]);
        ctxs[q]->nst_valid = false;
        ctxs[q]->T_finite = false;
    }
    CET_CUDA(cudaMemcpyAsync(dev, h.data(), bytes, cudaMemcpyHostToDevice, c0->stream));
    const int rc = n_ctx <= 16 ? init_group_launch<16>(c0, args, n_ctx, max_nuc)
                               : init_group_launch<GROUP_MAX>(c0, args, n_ctx, max_nuc);
    if (rc) return rc;
    CET_CUDA(cudaStreamSynchronize(c0->stream));
    return 0;
}

}  // extern "C"
