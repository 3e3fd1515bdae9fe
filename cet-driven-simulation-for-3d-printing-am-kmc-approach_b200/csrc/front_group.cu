// front_group.cu — the solidification front of a group of whole-lattice contexts (cet_front_group): per column along
// a growth axis, the front height h (consecutive occupied sites from plane 0), the top (1 + the highest occupied
// plane), and T at the front and its step T[h] - T[h - 1].  The call reads vox and T and writes nothing a sweep, a
// metrics row, a profile or a shape histogram reads.  As in profile_group.cu a CTA takes its lattice's arguments
// from a table in kernel parameter space (blockIdx.y); a group of up to 16 launches the small table.
// One launch for the whole group, each lattice's vox streamed once:
//   axes 0, 1: one thread per column, adjacent threads on adjacent k, so every plane's loads coalesce;
//   axis 2:    one warp per column (contiguous along k), 32 sites per ballot: __ffs of the first non-occupied lane
//              gives h, __clz of the occupied lanes the top; lanes k >= L of the last chunk count as neither.
// Every column's four values are written (no memset); two D2H copies return them.
#include <algorithm>
#include "cadence.cuh"

namespace cet {

constexpr unsigned long long FRONT_NAN = 0x7ff8000000000000ull;   // the one quiet NaN of T_front / dT_front

struct FgArgs {
    const uint8_t *vox;
    const double *T;
    int32_t *front;                 // [2][L * L]: front, top
    double *temp;                   // [2][L * L]: T_front, dT_front
};
static_assert(group_fits<FgArgs>(), "a table of GROUP_MAX entries must fit the kernel parameter space");

constexpr int FG_THREADS = 256;

// T at the front site (plane h of the column whose plane-0 site is s0, planes `step` sites apart) and the step
// T[h] - T[h - 1]; FRONT_NAN where the plane does not exist, and for a difference that is NaN (inf - inf, a NaN T)
__device__ __forceinline__ void front_write(const FgArgs &a, int LL, int c, int64_t s0, int64_t step, int h, int top, int L)
{
    const double nan = __longlong_as_double((long long)FRONT_NAN);
    double tf = nan, dt = nan;
    if (h < L) {
        tf = a.T[s0 + h * step];
        if (h > 0) {
            const double d = tf - a.T[s0 + (h - 1) * step];
            dt = d != d ? nan : d;
        }
    }
    a.front[c] = h; a.front[LL + c] = top;
    a.temp[c] = tf; a.temp[LL + c] = dt;
}

// axes 0 and 1: thread per column c = u * L + w; axis 0 column (j, k) at sites i * L^2 + c, axis 1 column (i, k) at
// sites i * L^2 + j * L + k
template <int CAP>
__global__ void __launch_bounds__(FG_THREADS) front_strided_group_kernel(const __grid_constant__ GroupArgs<FgArgs, CAP> g, int L, int axis)
{
    const FgArgs &a = g.a[blockIdx.y];
    const int LL = L * L;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= LL) return;
    const int64_t s0 = axis == 0 ? (int64_t)c : (int64_t)(c / L) * LL + c % L;
    const int64_t step = axis == 0 ? LL : L;
    const uint8_t *__restrict__ v = a.vox + s0;
    int h = L, top = 0;
#pragma unroll 8
    for (int p = 0; p < L; ++p) {
        const bool occ = (__ldg(v + p * step) & 0x0F) != 0;
        if (occ) top = p + 1;
        else h = min(h, p);
    }
    front_write(a, LL, c, s0, step, h, top, L);
}

// axis 2: warp per column c = i * L + j at sites c * L + k
template <int CAP>
__global__ void __launch_bounds__(FG_THREADS) front_contig_group_kernel(const __grid_constant__ GroupArgs<FgArgs, CAP> g, int L)
{
    const FgArgs &a = g.a[blockIdx.y];
    const int LL = L * L, lane = threadIdx.x & 31;
    const int c = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);      // warp-uniform
    if (c >= LL) return;
    const int64_t s0 = (int64_t)c * L;
    int h = L, top = 0;
    for (int k0 = 0; k0 < L; k0 += 32) {
        const int k = k0 + lane;
        const bool in = k < L;
        const bool occ = in && (__ldg(a.vox + s0 + k) & 0x0F) != 0;
        const unsigned hole = __ballot_sync(0xffffffffu, in && !occ), full = __ballot_sync(0xffffffffu, occ);
        if (h == L && hole) h = k0 + __ffs(hole) - 1;
        if (full) top = k0 + 32 - __clz(full);
    }
    if (lane == 0) front_write(a, LL, c, s0, 1, h, top, L);
}

static size_t align64(size_t b) { return (b + 63) & ~(size_t)63; }

template <int CAP>
static int front_group_run(cet_ctx *const *ctxs, int n, int axis, int32_t *front_out, double *temp_out)
{
    cet_ctx *c0 = ctxs[0];
    cudaStream_t st = c0->stream;
    const int L = (int)c0->n1, LL = L * L;
    const size_t int_bytes = (size_t)n * 2 * LL * sizeof(int32_t), dbl_bytes = (size_t)n * 2 * LL * sizeof(double);
    const size_t all_bytes = align64(int_bytes) + dbl_bytes;
    if (c0->cap_front_tab < all_bytes) {
        if (c0->front_tab) { cudaFree(c0->front_tab); c0->front_tab = nullptr; c0->cap_front_tab = 0; }
        CET_CUDA(cudaMalloc(&c0->front_tab, all_bytes));
        c0->cap_front_tab = all_bytes;
    }
    int32_t *d_front = (int32_t *)c0->front_tab;
    double *d_temp = (double *)((char *)c0->front_tab + align64(int_bytes));
    GroupArgs<FgArgs, CAP> t{};
    for (int q = 0; q < n; ++q) {
        FgArgs &p = t.a[q];
        p.vox = ctxs[q]->vox; p.T = ctxs[q]->T;
        p.front = d_front + (size_t)q * 2 * LL;
        p.temp = d_temp + (size_t)q * 2 * LL;
    }
    if (int rc = group_order(ctxs, n)) return rc;
    if (axis == 2)
        front_contig_group_kernel<CAP><<<dim3((unsigned)(((int64_t)LL * 32 + FG_THREADS - 1) / FG_THREADS), n), FG_THREADS, 0, st>>>(t, L);
    else
        front_strided_group_kernel<CAP><<<dim3((LL + FG_THREADS - 1) / FG_THREADS, n), FG_THREADS, 0, st>>>(t, L, axis);
    CET_CUDA(cudaGetLastError());
    CET_CUDA(cudaMemcpyAsync(front_out, d_front, int_bytes, cudaMemcpyDeviceToHost, st));
    CET_CUDA(cudaMemcpyAsync(temp_out, d_temp, dbl_bytes, cudaMemcpyDeviceToHost, st));
    CET_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace cet

using namespace cet;

extern "C" int cet_front_group(cet_ctx *const *ctxs, int32_t n_ctx, int32_t axis, int32_t *front_out, double *temp_out)
{
    if (int rc = group_check("cet_front_group", ctxs, n_ctx)) return rc;
    CET_REQUIRE(front_out && temp_out, "cet_front_group: NULL argument");
    CET_REQUIRE(axis >= 0 && axis <= 2, "cet_front_group: axis must be 0, 1 or 2, got %d", (int)axis);
    cet::DeviceGuard dg(ctxs[0]->device);
    return n_ctx <= 16 ? front_group_run<16>(ctxs, n_ctx, axis, front_out, temp_out)
                       : front_group_run<GROUP_MAX>(ctxs, n_ctx, axis, front_out, temp_out);
}
