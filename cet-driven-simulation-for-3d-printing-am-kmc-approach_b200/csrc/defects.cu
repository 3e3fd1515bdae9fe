// defects.cu — track_defects / introduce_defects (defects.py:4-31) on the resident lattice
// (SURVEY §8f row N3).
//
// The reference rebuilds the defect mask every METRIC_UPDATE_STEP steps on the host
// (kmc_simulation.py:335-338): mask = 0 everywhere, and on carbon sites (atom_type == 3)
//     mask = u < clip(DEFECT_PROB_BASE * exp(-0.3 / (K_T * T')), 0, 1),   T' = T if T > 0 else T_SUB,
// with one draw u of NumPy's global stream per carbon site in C order (defects.py:18).  That costs a
// download of atom_type and T and an upload of the mask; here the mask (the high nibble of the voxel
// byte) is rewritten in place.  Two draw sources:
//   draws != NULL  the caller's stream: the q-th carbon site in C order takes draws[q], so a run
//                  stays in lock-step with the reference's NumPy stream (the rank of a carbon site
//                  comes from a two-level ordered count: per-tile counts, a scan of the tile counts,
//                  in-tile ranks by ballot);
//   draws == NULL  Philox4x32-10 keyed by (seed, epoch, global site): the large-lattice path.
#include "cadence.cuh"

namespace cet {

__global__ void __launch_bounds__(DF_THREADS) defects_count_kernel(const DefectArgs a)
{
    defects_count_body(a);
}

__global__ void __launch_bounds__(1024) defects_scan_kernel(unsigned int *tile_count, int n_tiles, unsigned long long *totals)
{
    tile_scan_body(tile_count, n_tiles, totals);
}

// pass 3.  The body of defects_assign_body (cadence.cuh), kept here as the kernel's own code: called through the
// shared body, this kernel is allocated one register fewer.
__global__ void __launch_bounds__(DF_THREADS) defects_assign_kernel(const DefectArgs a)
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

}  // namespace cet

using namespace cet;

extern "C" int cet_defects_refresh(cet_ctx *c, const double *draws, int64_t n_draws, uint64_t seed, uint32_t epoch,
                                   double prob_base, double e_mig, double kT, double T_default, int32_t carbon_id,
                                   int32_t defect_id, int32_t apply_to_state, int64_t *n_carbon, int64_t *n_defects)
{
    CET_REQUIRE(c, "cet_defects_refresh: NULL ctx");
    CET_REQUIRE(carbon_id >= 1 && carbon_id <= 15, "cet_defects_refresh: carbon state id must be in 1..15");
    CET_REQUIRE(c->nloc < (1ll << 31), "cet_defects_refresh: the local lattice must have fewer than 2^31 sites");
    CET_REQUIRE(!draws || c->world == 1, "cet_defects_refresh: an injected draw stream needs the whole lattice in one context");
    cet::DeviceGuard dg(c->device);
    const int64_t n = c->owned_sites();
    const int n_tiles = (int)((n + DF_TILE - 1) / DF_TILE);
    const size_t need = (size_t)(n_tiles + 1) * sizeof(unsigned int) + 64 + (draws ? (size_t)n_draws * sizeof(double) : 0);
    if (int rc = ensure_stage(c, need)) return rc;
    DefectArgs a;
    a.totals = (unsigned long long *)c->stage;
    a.tile_count = (unsigned int *)((char *)c->stage + 64);
    double *d_draws = (double *)((char *)c->stage + 64 + (((size_t)(n_tiles + 1) * sizeof(unsigned int) + 63) & ~(size_t)63));
    if (int rc = ensure_stage(c, (size_t)((char *)d_draws - (char *)c->stage) + (draws ? (size_t)n_draws * sizeof(double) : 0))) return rc;
    a.totals = (unsigned long long *)c->stage;                       // ensure_stage may have moved the buffer
    a.tile_count = (unsigned int *)((char *)c->stage + 64);
    d_draws = (double *)((char *)c->stage + 64 + (((size_t)(n_tiles + 1) * sizeof(unsigned int) + 63) & ~(size_t)63));
    a.vox = c->vox + c->owned_offset(); a.T = c->T + c->owned_offset();
    a.n = n; a.g_off = c->i_begin * c->plane;
    a.draws = draws ? d_draws : nullptr;
    a.seed = seed; a.epoch = epoch;
    a.carbon_id = carbon_id; a.defect_id = defect_id; a.apply_to_state = apply_to_state;
    a.base = prob_base; a.e_mig = e_mig; a.kT = kT; a.T_default = T_default;
    CET_CUDA(cudaMemsetAsync(a.totals, 0, 64, c->stream));
    defects_count_kernel<<<n_tiles, DF_THREADS, 0, c->stream>>>(a);
    defects_scan_kernel<<<1, 1024, 0, c->stream>>>(a.tile_count, n_tiles, a.totals);
    CET_CUDA(cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    CET_CUDA(cudaMemcpyAsync(h, a.totals, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    if (n_carbon) *n_carbon = (int64_t)h[0];
    if (draws) {
        CET_REQUIRE((int64_t)h[0] <= n_draws, "cet_defects_refresh: %lld carbon sites but only %lld draws", (long long)h[0],
                    (long long)n_draws);
        CET_CUDA(cudaMemcpyAsync(d_draws, draws, (size_t)h[0] * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    }
    defects_assign_kernel<<<n_tiles, DF_THREADS, 0, c->stream>>>(a);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(h, a.totals, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CET_CUDA(cudaStreamSynchronize(c->stream));
    if (n_defects) *n_defects = (int64_t)h[1];
    lattice_changed(c);                                              // defect factors changed (kmc_event_rates.py:94)
    if (apply_to_state && h[1]) c->nst_valid = false;
    return 0;
}
