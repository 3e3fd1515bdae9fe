// rates_dense_group.cu — the dense rate kernel (rates_dense.cu) for the lattices of a grouped sweep
// (cet_sweep_run_group): one launch rebuilds the rates of every lattice whose rates are stale.
#include "rates_dense.cuh"

namespace cet {

// Grouped sweeps: grid (CTAs per lattice, 1, lattices); each lattice's CTAs pop the tiles of that lattice from its own
// queue.  The tensor maps are separate arrays so that 64 entries fit the 32 KB of kernel parameter space.
template <int CAP>
struct DenseGroup {
    CUtensorMap vox[CAP], po[CAP];
    DenseArgs a[CAP];
};
static_assert(sizeof(DenseGroup<GROUP_MAX>) <= 32764, "a table of GROUP_MAX entries must fit the kernel parameter space");
template <int CAP>
__global__ void __launch_bounds__(TL_THREADS, 4) rates_dense_group_kernel(const __grid_constant__ DenseGroup<CAP> g)
{
    rates_dense_body<true>(g.a[blockIdx.z], g.vox[blockIdx.z], g.po[blockIdx.z]);
}

// The queue of the dense kernel (zero before a launch: rates_rows_dense clears it, grouped sweeps clear it in their
// reset kernel and before their first sweep).
unsigned int *dense_queue(cet_ctx *c) { return (unsigned int *)(c->rate_tab + RT_TABLE_DOUBLES) + 2; }

// rates_rows_dense over all planes of a group of whole-lattice contexts of one TMA-capable L (cet_sweep_run_group), one
// launch on the stream of cs[0].  blocks_per_sm: the grouped kernel's occupancy, queried on first use.
template <int CAP>
static int dense_group_launch(cet_ctx *const *cs, int n, int *blocks_per_sm)
{
    const size_t smem = sizeof(DenseSmem) + 1024;
    if (*blocks_per_sm == 0) {
        CET_CUDA(cudaFuncSetAttribute(rates_dense_group_kernel<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int nb = 0;
        CET_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rates_dense_group_kernel<CAP>, TL_THREADS, smem));
        CET_REQUIRE(nb >= 1, "rates_dense_group_kernel does not fit an SM");
        *blocks_per_sm = nb;
    }
    DenseGroup<CAP> g;
    for (int q = 0; q < n; ++q) {
        cet_ctx *c = cs[q];
        if (int rc = tile_maps_ensure(c)) return rc;
        memcpy(&g.vox[q], c->tmap_vox, sizeof(CUtensorMap));
        memcpy(&g.po[q], c->tmap_po, sizeof(CUtensorMap));
        g.a[q] = dense_args(c, 0, (int)c->np);
    }
    const int per = std::max(1, std::min(g.a[0].n_tiles, (sm_count(cs[0]) * *blocks_per_sm + n - 1) / n));
    rates_dense_group_kernel<CAP><<<dim3((unsigned)per, 1, (unsigned)n), TL_THREADS, smem, cs[0]->stream>>>(g);
    CET_CUDA(cudaGetLastError());
    return 0;
}
int rates_rows_dense_group(cet_ctx *const *cs, int n, int *blocks_per_sm)
{
    if (n <= 0) return 0;
    return n <= 16 ? dense_group_launch<16>(cs, n, blocks_per_sm) : dense_group_launch<GROUP_MAX>(cs, n, blocks_per_sm);
}

}  // namespace cet
