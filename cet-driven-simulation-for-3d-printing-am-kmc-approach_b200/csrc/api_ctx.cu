// api_ctx.cu — library/context entry points of include/cetkmc.h: error reporting, context
// life cycle, and conversion between the reference's host layouts (int64 / float64 arrays,
// lattice_init.py:23-32) and the packed HBM layout (1 byte per voxel + float64 fields).
#include <stdarg.h>
#include "cadence.cuh"
#include "rate_tile.cuh"

namespace cet {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int ensure_stage(cet_ctx *c, size_t bytes)
{
    if (c->stage_bytes >= bytes) return 0;
    if (c->stage) { cudaFree(c->stage); c->stage = nullptr; c->stage_bytes = 0; }
    CET_CUDA(cudaMalloc(&c->stage, bytes));
    c->stage_bytes = bytes;
    return 0;
}

// state/defects (int64, host layout) -> packed byte.  A NULL source keeps that nibble.
// bad[0] is set when a value does not fit its nibble.
__global__ void pack_kernel(const int64_t *__restrict__ state, const int64_t *__restrict__ defects,
                            uint8_t *vox, int64_t n, int *bad)
{
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n;
         q += (int64_t)gridDim.x * blockDim.x) {
        uint8_t v = vox[q];
        if (state) {
            const int64_t s = state[q];
            if (s < 0 || s > 15) *bad = 1;
            v = (uint8_t)((v & 0xF0) | (uint8_t)(s & 15));
        }
        if (defects) {
            const int64_t d = defects[q];
            if (d < 0 || d > 15) *bad = 2;
            v = (uint8_t)((v & 0x0F) | (uint8_t)((d & 15) << 4));
        }
        vox[q] = v;
    }
}

__global__ void unpack_kernel(const uint8_t *__restrict__ vox, int64_t *state, int64_t n)
{
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n;
         q += (int64_t)gridDim.x * blockDim.x)
        state[q] = vox[q] & 0x0F;
}

__global__ void counts_kernel(const uint8_t *__restrict__ vox, int64_t n, unsigned long long *out)
{
    counts_body(vox, n, out);
}

__global__ void orient_kernel(const double *__restrict__ theta, const double *__restrict__ phi, Vec4 *v, int64_t n)
{
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n;
         q += (int64_t)gridDim.x * blockDim.x)
        v[q] = unit_vec4(theta[q], phi[q]);
}

// nst[s] = cached neighbour-state word of s (rate_tile.cuh: nst_word)
__global__ void nst_build_kernel(const uint64_t lut, const uint8_t *__restrict__ vox, uint64_t *nst, int L, int n0,
                                 int i_off, int p_lo, int p_hi)
{
    const int64_t LL = (int64_t)L * L;
    const int64_t n = (int64_t)(p_hi - p_lo) * LL;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = (int64_t)p_lo * LL + q;
        const int p = (int)(s / LL), j = (int)((s / L) % L), k = (int)(s % L);
        nst[s] = nst_word(lut, vox, s, i_off + p, j, k, n0, L);
    }
}

__global__ void nst_check_kernel(const uint64_t lut, const uint8_t *__restrict__ vox, const uint64_t *__restrict__ nst,
                                 int L, int n0, int i_off, int p_lo, int p_hi, unsigned long long *bad)
{
    const int64_t LL = (int64_t)L * L;
    const int64_t n = (int64_t)(p_hi - p_lo) * LL;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = (int64_t)p_lo * LL + q;
        const int p = (int)(s / LL), j = (int)((s / L) % L), k = (int)(s % L);
        if (nst[s] != nst_word(lut, vox, s, i_off + p, j, k, n0, L)) atomicAdd(bad, 1ull);
    }
}

static int grid_for(cet_ctx *c, int64_t n, int block)
{
    int64_t g = (n + block - 1) / block;
    const int64_t cap = (int64_t)sm_count(c) * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

int nst_build(cet_ctx *c, int p_lo, int p_hi)
{
    if (p_hi <= p_lo) return 0;
    const int64_t n = (int64_t)(p_hi - p_lo) * c->plane;
    nst_build_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(nb_code_lut(c->rp), c->vox, c->nst, (int)c->n1, (int)c->n0,
                                                               (int)(c->i_begin - c->halo), p_lo, p_hi);
    CET_CUDA(cudaGetLastError());
    return 0;
}

int nst_ensure(cet_ctx *c)
{
    if (c->nst_valid) return 0;
    // planes whose i +- 2 neighbours are stored locally or lie outside the global lattice
    const int i_off = (int)(c->i_begin - c->halo), np = (int)c->np;
    const int lo = i_off > 0 ? 2 : (i_off < 0 ? -i_off : 0);
    const int hi = (i_off + np < c->n0) ? np - 2 : (int)(c->n0 - i_off < np ? c->n0 - i_off : np);
    if (int rc = nst_build(c, lo, hi)) return rc;
    c->nst_valid = true;
    return 0;
}

int orient_update(cet_ctx *c, int64_t p_lo, int64_t p_hi)
{
    if (p_hi <= p_lo) return 0;
    const int64_t off = p_lo * c->plane, n = (p_hi - p_lo) * c->plane;
    orient_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(c->theta + off, c->phi + off, c->v + off, n);
    CET_CUDA(cudaGetLastError());
    return 0;
}

static int create_common(cet_ctx **out, int device, int64_t n0, int64_t n1, int64_t n2,
                         int64_t i_begin, int64_t i_end, int halo, bool cubic)
{
    CET_REQUIRE(out != nullptr, "cet_create: ctx pointer is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_error("cet_create: no CUDA device available (%s); libcetkmc has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return 2;
    }
    CET_REQUIRE(device >= 0 && device < ndev, "cet_create: device %d out of range (have %d)", device, ndev);
    CET_REQUIRE(n0 > 0 && n1 > 0 && n2 > 0, "cet_create: extents must be positive");
    CET_REQUIRE(n0 < 32768 && n1 < 32768 && n2 < 32768, "cet_create: extent too large");
    CET_REQUIRE(0 <= i_begin && i_begin < i_end && i_end <= n0, "cet_create: bad slab [%lld,%lld) of %lld",
                (long long)i_begin, (long long)i_end, (long long)n0);
    CET_REQUIRE(halo >= 0 && halo <= 8, "cet_create: halo must be in 0..8");
    cet::DeviceGuard dg(device);
    CET_REQUIRE(dg.ok, "cet_create: cudaSetDevice(%d) failed", device);
    cet_ctx *c = new cet_ctx();
    c->device = device;
    c->n0 = n0; c->n1 = n1; c->n2 = n2;
    c->i_begin = i_begin; c->i_end = i_end; c->halo = halo;
    c->np = (i_end - i_begin) + 2 * halo;
    c->plane = n1 * n2;
    c->nloc = c->np * c->plane;
    c->cubic = cubic;
    *out = c;
    CET_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CET_CUDA(cudaEventCreate(&c->ev0));
    CET_CUDA(cudaEventCreate(&c->ev1));
    CET_CUDA(cudaMalloc(&c->vox, c->nloc));
    CET_CUDA(cudaMemsetAsync(c->vox, 0, c->nloc, c->stream));
    CET_CUDA(cudaMalloc(&c->T, c->nloc * sizeof(double)));
    CET_CUDA(cudaMalloc(&c->T2, c->nloc * sizeof(double)));
    CET_CUDA(cudaMemsetAsync(c->T, 0, c->nloc * sizeof(double), c->stream));
    CET_CUDA(cudaMemsetAsync(c->T2, 0, c->nloc * sizeof(double), c->stream));
    if (cubic) {
        CET_CUDA(cudaMalloc(&c->theta, c->nloc * sizeof(double)));
        CET_CUDA(cudaMalloc(&c->phi, c->nloc * sizeof(double)));
        CET_CUDA(cudaMemsetAsync(c->theta, 0, c->nloc * sizeof(double), c->stream));
        CET_CUDA(cudaMemsetAsync(c->phi, 0, c->nloc * sizeof(double), c->stream));
        CET_CUDA(cudaMalloc(&c->v, c->nloc * sizeof(Vec4)));
        CET_CUDA(cudaMalloc(&c->nst, c->nloc * sizeof(uint64_t)));
        CET_CUDA(cudaMemsetAsync(c->nst, 0, c->nloc * sizeof(uint64_t), c->stream));
        if (int rc = orient_update(c, 0, c->np)) return rc;
        CET_CUDA(cudaMalloc(&c->site_rate, c->nloc * sizeof(double)));
        CET_CUDA(cudaMemsetAsync(c->site_rate, 0, c->nloc * sizeof(double), c->stream));
        CET_CUDA(cudaMalloc(&c->dep_rate, c->plane * sizeof(double)));
        CET_CUDA(cudaMemsetAsync(c->dep_rate, 0xFF, c->plane * sizeof(double), c->stream));  // NaN
        CET_CUDA(cudaMalloc(&c->row_occ, c->np * n1 * sizeof(double)));
        CET_CUDA(cudaMalloc(&c->row_emp, c->np * n1 * sizeof(double)));
        CET_CUDA(cudaMalloc(&c->row_dep, n1 * sizeof(double)));
        CET_CUDA(cudaMalloc(&c->row_depcnt, n1 * sizeof(int32_t)));
        CET_CUDA(cudaMalloc(&c->seg, 3 * c->np * sizeof(double)));
        CET_CUDA(cudaMalloc(&c->total, 4 * sizeof(double)));
        CET_CUDA(cudaMemsetAsync(c->row_occ, 0, c->np * n1 * sizeof(double), c->stream));
        CET_CUDA(cudaMemsetAsync(c->row_emp, 0, c->np * n1 * sizeof(double), c->stream));
        CET_CUDA(cudaMemsetAsync(c->row_dep, 0, n1 * sizeof(double), c->stream));
        CET_CUDA(cudaMemsetAsync(c->row_depcnt, 0, n1 * sizeof(int32_t), c->stream));
        CET_CUDA(cudaMemsetAsync(c->seg, 0, 3 * c->np * sizeof(double), c->stream));
        CET_CUDA(cudaMemsetAsync(c->total, 0, 4 * sizeof(double), c->stream));
        CET_CUDA(cudaMalloc(&c->kmc, sizeof(cet::KmcState)));
        CET_CUDA(cudaMemsetAsync(c->kmc, 0, sizeof(cet::KmcState), c->stream));
    }
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" {

const char *cet_last_error(void) { return cet::g_err; }
int cet_abi_version(void) { return CET_ABI_VERSION; }

int cet_device_count(int *n)
{
    CET_REQUIRE(n != nullptr, "cet_device_count: NULL");
    int nd = 0;
    cudaError_t e = cudaGetDeviceCount(&nd);
    if (e != cudaSuccess) { nd = 0; (void)cudaGetLastError(); }
    *n = nd;
    return 0;
}

int cet_device_name(int device, char *buf, int buflen)
{
    CET_REQUIRE(buf && buflen > 0, "cet_device_name: bad buffer");
    cudaDeviceProp p;
    CET_CUDA(cudaGetDeviceProperties(&p, device));
    snprintf(buf, buflen, "%s (sm_%d%d, %d SMs)", p.name, p.major, p.minor, p.multiProcessorCount);
    return 0;
}

int cet_create(cet_ctx **ctx, int device, int64_t L, int64_t i_begin, int64_t i_end, int32_t halo)
{
    return create_common(ctx, device, L, L, L, i_begin, i_end, halo, true);
}

int cet_create_slab(cet_ctx **ctx, int device, int64_t n0, int64_t L, int64_t i_begin, int64_t i_end, int32_t halo)
{
    return create_common(ctx, device, n0, L, L, i_begin, i_end, halo, true);
}

int cet_create_shape(cet_ctx **ctx, int device, int64_t n0, int64_t n1, int64_t n2)
{
    return create_common(ctx, device, n0, n1, n2, 0, n0, 0, false);
}

int cet_comm_destroy(cet_ctx *ctx);

int cet_destroy(cet_ctx *c)
{
    if (!c) return 0;
    cet::DeviceGuard dg(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    cet_comm_destroy(c);
    void *ptrs[] = {c->vox, c->vox_prev, c->theta, c->phi, c->v, c->nst, c->T, c->T2, c->site_rate, c->dep_rate,
                    c->row_occ, c->row_emp, c->row_dep, c->row_depcnt, c->seg, c->total, c->q_top,
                    c->stage, c->kmc, c->d_py, c->d_np, c->d_sp, c->d_log, c->sweep, c->claim,
                    c->records, c->blk_sum, c->blk_max, c->plane_sum, c->stamp, c->dirty, c->fired,
                    c->grain_label, c->grain_gid, c->grain_st, c->group_tab, c->profile_tab, c->rate_tab, c->cvox, c->pairop, c->tile_flag,
                    c->delta_send[0], c->delta_send[1], c->delta_recv[0], c->delta_recv[1]};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (auto &sp : c->prof_spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    for (auto e : c->prof_pool) cudaEventDestroy(e);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev_group) cudaEventDestroy(c->ev_group);
    if (c->ev_reduce_ready) cudaEventDestroy(c->ev_reduce_ready);
    if (c->ev_reduce_done) cudaEventDestroy(c->ev_reduce_done);
    if (c->stream2) cudaStreamDestroy(c->stream2);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}

int cet_sync(cet_ctx *c)
{
    CET_REQUIRE(c, "cet_sync: NULL ctx");
    cet::DeviceGuard dg(c->device);
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

int cet_set_rate_params(cet_ctx *c, const cet_rate_params *p)
{
    CET_REQUIRE(c && p, "cet_set_rate_params: NULL argument");
    CET_REQUIRE(p->states_w >= 1 && p->states_w <= 15 && p->states_re >= 1 && p->states_re <= 15 &&
                    p->states_c >= 1 && p->states_c <= 15,
                "cet_set_rate_params: species ids must be in 1..15");
    CET_REQUIRE(p->states_w != p->states_re && p->states_w != p->states_c && p->states_re != p->states_c &&
                    p->defect_id != p->states_w && p->defect_id != p->states_re && p->defect_id != p->states_c,
                "cet_set_rate_params: the W / Re / C / defect state ids must be distinct");
    c->rp = *p;
    c->have_rp = true;
    c->rate_tab_valid = false;
    c->nst_valid = false;             // the cached neighbour classes depend on the state ids
    lattice_changed(c);
    return 0;
}

int cet_upload(cet_ctx *c, const int64_t *state, const double *theta, const double *phi,
               const double *T, const int64_t *defects)
{
    CET_REQUIRE(c, "cet_upload: NULL ctx");
    cet::DeviceGuard dg(c->device);
    const int64_t n = c->owned_sites();
    const int64_t off = c->owned_offset();
    const size_t fb = (size_t)n * sizeof(double);
    if ((theta || phi) && !c->cubic) { set_error("cet_upload: theta/phi need a cubic context"); return 1; }
    // everything derived from the lattice is stale from here on, also when the call fails half way
    lattice_changed(c);
    if (state) c->nst_valid = false;
    if (theta) CET_CUDA(cudaMemcpyAsync(c->theta + off, theta, fb, cudaMemcpyHostToDevice, c->stream));
    if (phi) CET_CUDA(cudaMemcpyAsync(c->phi + off, phi, fb, cudaMemcpyHostToDevice, c->stream));
    if (T) { CET_CUDA(cudaMemcpyAsync(c->T + off, T, fb, cudaMemcpyHostToDevice, c->stream)); c->T_finite = false; }
    if (state || defects) {
        const size_t need = (size_t)n * sizeof(int64_t) * ((state ? 1 : 0) + (defects ? 1 : 0)) + 256;
        if (int rc = ensure_stage(c, need)) return rc;
        int64_t *ds = nullptr, *dd = nullptr;
        char *p = (char *)c->stage;
        int *bad = (int *)p; p += 256;
        CET_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), c->stream));
        if (state) { ds = (int64_t *)p; p += (size_t)n * 8; CET_CUDA(cudaMemcpyAsync(ds, state, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream)); }
        if (defects) { dd = (int64_t *)p; CET_CUDA(cudaMemcpyAsync(dd, defects, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream)); }
        pack_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(ds, dd, c->vox + off, n, bad);
        CET_CUDA(cudaGetLastError());
        if (state) c->nst_valid = false;
        int hbad = 0;
        CET_CUDA(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CET_CUDA(cudaStreamSynchronize(c->stream));
        CET_REQUIRE(hbad == 0, "cet_upload: %s value outside 0..15 (one byte per voxel holds state | defects<<4)",
                    hbad == 1 ? "state" : "defects_mask");
    }
    if (theta || phi) if (int rc = orient_update(c, c->halo, c->np - c->halo)) return rc;
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

int cet_download(cet_ctx *c, int64_t *state, int64_t *atom_type, double *theta, double *phi, double *T)
{
    CET_REQUIRE(c, "cet_download: NULL ctx");
    cet::DeviceGuard dg(c->device);
    const int64_t n = c->owned_sites();
    const int64_t off = c->owned_offset();
    const size_t fb = (size_t)n * sizeof(double);
    if ((theta || phi) && !c->cubic) { set_error("cet_download: theta/phi need a cubic context"); return 1; }
    if (theta) CET_CUDA(cudaMemcpyAsync(theta, c->theta + off, fb, cudaMemcpyDeviceToHost, c->stream));
    if (phi) CET_CUDA(cudaMemcpyAsync(phi, c->phi + off, fb, cudaMemcpyDeviceToHost, c->stream));
    if (T) CET_CUDA(cudaMemcpyAsync(T, c->T + off, fb, cudaMemcpyDeviceToHost, c->stream));
    if (state || atom_type) {
        if (int rc = ensure_stage(c, (size_t)n * 8)) return rc;
        unpack_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(c->vox + off, (int64_t *)c->stage, n);
        CET_CUDA(cudaGetLastError());
        // kmc_simulation.py:281-282,293-294,306-307,314-315,324-325: atom_type is written with
        // the same value as state at every update, so one unpack serves both arrays.
        if (state) CET_CUDA(cudaMemcpyAsync(state, c->stage, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
        if (atom_type) CET_CUDA(cudaMemcpyAsync(atom_type, c->stage, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

int cet_upload_prev_state(cet_ctx *c, const int64_t *prev_state)
{
    CET_REQUIRE(c && prev_state, "cet_upload_prev_state: NULL argument");
    cet::DeviceGuard dg(c->device);
    const int64_t n = c->owned_sites();
    const int64_t off = c->owned_offset();
    if (!c->vox_prev) {
        CET_CUDA(cudaMalloc(&c->vox_prev, c->nloc));
        CET_CUDA(cudaMemsetAsync(c->vox_prev, 0, c->nloc, c->stream));
    }
    if (int rc = ensure_stage(c, (size_t)n * 8 + 256)) return rc;
    int *bad = (int *)c->stage;
    int64_t *ds = (int64_t *)((char *)c->stage + 256);
    CET_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), c->stream));
    CET_CUDA(cudaMemcpyAsync(ds, prev_state, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
    pack_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(ds, nullptr, c->vox_prev + off, n, bad);
    CET_CUDA(cudaGetLastError());
    int hbad = 0;
    CET_CUDA(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    CET_REQUIRE(hbad == 0, "cet_upload_prev_state: state value outside 0..15");
    return 0;
}

int cet_snapshot_state(cet_ctx *c)
{
    CET_REQUIRE(c, "cet_snapshot_state: NULL ctx");
    cet::DeviceGuard dg(c->device);
    if (!c->vox_prev) CET_CUDA(cudaMalloc(&c->vox_prev, c->nloc));
    CET_CUDA(cudaMemcpyAsync(c->vox_prev, c->vox, c->nloc, cudaMemcpyDeviceToDevice, c->stream));
    return 0;
}

int cet_upload_packed(cet_ctx *c, const uint8_t *packed)
{
    CET_REQUIRE(c && packed, "cet_upload_packed: NULL argument");
    cet::DeviceGuard dg(c->device);
    CET_CUDA(cudaMemcpyAsync(c->vox + c->owned_offset(), packed, (size_t)c->owned_sites(),
                             cudaMemcpyHostToDevice, c->stream));
    c->nst_valid = false;
    lattice_changed(c);
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

int cet_download_packed(cet_ctx *c, uint8_t *packed)
{
    CET_REQUIRE(c && packed, "cet_download_packed: NULL argument");
    cet::DeviceGuard dg(c->device);
    CET_CUDA(cudaMemcpyAsync(packed, c->vox + c->owned_offset(), (size_t)c->owned_sites(),
                             cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

int cet_device_ptr(cet_ctx *c, int which, void **ptr, int64_t *nbytes)
{
    CET_REQUIRE(c && ptr, "cet_device_ptr: NULL argument");
    void *p = nullptr;
    int64_t nb = 0;
    switch (which) {
        case 0: p = c->vox; nb = c->nloc; break;
        case 1: p = c->theta; nb = c->nloc * 8; break;
        case 2: p = c->phi; nb = c->nloc * 8; break;
        case 3: p = c->T; nb = c->nloc * 8; break;
        case 4: p = c->site_rate; nb = c->nloc * 8; break;
        case 5: p = c->v; nb = c->nloc * 32; break;
        default: set_error("cet_device_ptr: unknown field %d", which); return 1;
    }
    CET_REQUIRE(p != nullptr, "cet_device_ptr: field %d not allocated for this context", which);
    *ptr = p;
    if (nbytes) *nbytes = nb;
    return 0;
}

int cet_counts(cet_ctx *c, int64_t counts[16])
{
    CET_REQUIRE(c && counts, "cet_counts: NULL argument");
    cet::DeviceGuard dg(c->device);
    if (int rc = ensure_stage(c, 16 * sizeof(unsigned long long))) return rc;
    CET_CUDA(cudaMemsetAsync(c->stage, 0, 16 * sizeof(unsigned long long), c->stream));
    const int64_t n = c->owned_sites();
    counts_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(c->vox + c->owned_offset(), n,
                                                           (unsigned long long *)c->stage);
    CET_CUDA(cudaGetLastError());
    unsigned long long h[16];
    CET_CUDA(cudaMemcpyAsync(h, c->stage, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    for (int q = 0; q < 16; ++q) counts[q] = (int64_t)h[q];
    return 0;
}

int cet_debug_nst_mismatches(cet_ctx *c, int64_t *n_bad)
{
    CET_REQUIRE(c && n_bad && c->cubic, "cet_debug_nst_mismatches: bad argument");
    cet::DeviceGuard dg(c->device);
    if (!c->nst_valid) { *n_bad = -1; return 0; }           // stale by declaration: nothing to check
    const int i_off = (int)(c->i_begin - c->halo), np = (int)c->np;
    const int lo = i_off > 0 ? 2 : (i_off < 0 ? -i_off : 0);
    const int hi = (i_off + np < c->n0) ? np - 2 : (int)(c->n0 - i_off < np ? c->n0 - i_off : np);
    if (int rc = ensure_stage(c, 8)) return rc;
    CET_CUDA(cudaMemsetAsync(c->stage, 0, 8, c->stream));
    const int64_t n = (int64_t)(hi - lo) * c->plane;
    nst_check_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(nb_code_lut(c->rp), c->vox, c->nst, (int)c->n1, (int)c->n0, i_off, lo, hi,
                                                               (unsigned long long *)c->stage);
    CET_CUDA(cudaGetLastError());
    unsigned long long h = 0;
    CET_CUDA(cudaMemcpyAsync(&h, c->stage, 8, cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    *n_bad = (int64_t)h;
    return 0;
}

int cet_debug_flags(cet_ctx *c, int flags)
{
    CET_REQUIRE(c, "cet_debug_flags: NULL ctx");
    c->debug_flags = flags;
    return 0;
}

int cet_profile_enable(cet_ctx *c, int on)
{
    CET_REQUIRE(c, "cet_profile_enable: NULL ctx");
    c->profile = on != 0;
    return 0;
}

int cet_profile_read(cet_ctx *c, int kind, double *ms_total, int64_t *launches, int reset)
{
    CET_REQUIRE(c && kind >= 0 && kind < cet::PROF_KINDS, "cet_profile_read: bad argument");
    cet::DeviceGuard dg(c->device);
    CET_CUDA(cudaStreamSynchronize(c->stream));
    double tot = 0.0;
    int64_t n = 0;
    std::vector<cet_ctx::ProfSpan> keep;
    for (auto &sp : c->prof_spans) {
        if (sp.kind == kind) {
            float ms = 0.f;
            CET_CUDA(cudaEventElapsedTime(&ms, sp.a, sp.b));
            tot += ms; ++n;
            if (reset) { c->prof_pool.push_back(sp.a); c->prof_pool.push_back(sp.b); continue; }
        }
        keep.push_back(sp);
    }
    c->prof_spans.swap(keep);
    if (ms_total) *ms_total = tot;
    if (launches) *launches = n;
    return 0;
}

int cet_timer_begin(cet_ctx *c)
{
    CET_REQUIRE(c, "cet_timer_begin: NULL ctx");
    cet::DeviceGuard dg(c->device);
    CET_CUDA(cudaEventRecord(c->ev0, c->stream));
    return 0;
}

int cet_timer_end_ms(cet_ctx *c, float *ms)
{
    CET_REQUIRE(c && ms, "cet_timer_end_ms: NULL argument");
    cet::DeviceGuard dg(c->device);
    CET_CUDA(cudaEventRecord(c->ev1, c->stream));
    CET_CUDA(cudaEventSynchronize(c->ev1));
    CET_CUDA(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return 0;
}

}  // extern "C"
