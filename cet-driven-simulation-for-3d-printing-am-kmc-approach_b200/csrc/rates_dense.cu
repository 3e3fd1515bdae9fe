// rates_dense.cu — dense evaluation of every site's rate sum (the rebuild after a thermal step, an upload or a
// parameter change) from the compact tile state: the rate kernel of kmc_event_rates.py:43-160 for the sweep path.
//
// The pass is bound by instruction issue and the FP64 pipe, not by HBM (DESIGN.md §4.2): an attachment pair
// costs one fp64 exp (15 FP64 instructions = 30 pipe cycles per warp), a diffusion pair one reciprocal, and a
// site next to a solid/empty interface owns up to 14 of them.  What the counters of the earlier kernels said
// (997 warp instructions per 32 sites, only 110 of them FP64) is that everything AROUND the arithmetic has to
// go, so this kernel is built to execute little else (477 per 32 sites):
//   * persistent CTAs pop 4 x 8 x 32 tiles from a queue; one thread stages cvox + pairop with their halo of 2 by
//     two 3-D TMA boxes (zero fill outside the lattice = class code 0 = "outside": no bounds logic anywhere);
//     neighbour classes and pair operands are LDS with immediate offsets from one base register per site;
//   * pass A (4 rows per warp) reads the 15 class codes of a site, packs them 4 bits per slot, and only
//     CLASSIFIES: sites without events store 0, empty sites without an occupied neighbour evaluate their
//     nucleation rate on the spot when they are the bulk of the row (the melt above the front), everything else
//     is staged with the key (class, number of pairs) and counting-sorted over the tile;
//   * pass B deals trips of 32 sorted sites to the warps, so a trip runs ONE class — the per-site half
//     (tile_prep_emp / tile_prep_occ: one exp each) without the other class's lanes idling beside it — and
//     almost always ONE pair count; then every lane walks its own pair mask in slot order with the running sum
//     in a register: no descriptors, no shared-memory round trip for operands or rates, and the association
//     order of site_rate_sum for free.  (The sort costs nothing in locality here: the whole neighbourhood is in
//     shared memory.  The list-driven refresh, rates_refresh.cu, gathers from global memory and must not sort.)
// The arithmetic is the shared inline code of site_rates.cuh / tile_state.cuh / pair_walk.cuh, so the result
// equals the per-event code, the refresh kernels and the other dense kernels bit for bit (tests/test_gpu_sweep.py).
#include "rates_dense.cuh"

namespace cet {

template <bool SORT>
__global__ void __launch_bounds__(TL_THREADS, 4)
    rates_dense_kernel(const __grid_constant__ DenseArgs a, const __grid_constant__ CUtensorMap tm_vox, const __grid_constant__ CUtensorMap tm_po)
{
    rates_dense_body<SORT>(a, tm_vox, tm_po);
}
template <bool SORT>
static int dense_launch(cet_ctx *c, const DenseArgs &a, int *blocks_per_sm)
{
    const size_t smem = sizeof(DenseSmem) + 1024;
    if (*blocks_per_sm == 0) {
        CET_CUDA(cudaFuncSetAttribute(rates_dense_kernel<SORT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int nb = 0;
        CET_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rates_dense_kernel<SORT>, TL_THREADS, smem));
        CET_REQUIRE(nb >= 1, "rates_dense_kernel does not fit an SM");
        *blocks_per_sm = nb;
    }
    const int grid = std::min(a.n_tiles, sm_count(c) * *blocks_per_sm);
    rates_dense_kernel<SORT><<<grid, TL_THREADS, smem, c->stream>>>(a, *(const CUtensorMap *)c->tmap_vox, *(const CUtensorMap *)c->tmap_po);
    CET_CUDA(cudaGetLastError());
    return 0;
}

// Dense evaluation of local planes [p_lo, p_hi) from cvox / pairop (rows a tensor map can describe: tile_tma_ok).
int rates_rows_dense(cet_ctx *c, int p_lo, int p_hi)
{
    if (p_hi <= p_lo) return 0;
    if (int rc = rate_tables_ensure(c)) return rc;
    if (int rc = tile_maps_ensure(c)) return rc;
    const DenseArgs a = dense_args(c, p_lo, p_hi);
    CET_CUDA(cudaMemsetAsync(a.queue, 0, sizeof(unsigned int), c->stream));
    // pass B walks the tile's sites sorted by class and pair count (default) or by class only (debug flag 131072); the same bits
    if (c->debug_flags & 131072) { if (int rc = dense_launch<false>(c, a, &c->dense_blocks[0])) return rc; }
    else if (int rc = dense_launch<true>(c, a, &c->dense_blocks[1])) return rc;
    CET_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace cet
