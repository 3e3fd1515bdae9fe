// Test-only host build of csrc/grain_shape.cuh: runs the derivation the grain-shape kernels inline (Q from the exact
// moments, fl(), the elongation A and the histogram bin) on the CPU, so that it can be checked bit for bit against
// Python integers and float() without a GPU.  Not part of the product (nothing in the package links or loads this).
#include <stdint.h>
#include "../../cet-driven-simulation-for-3d-printing-am-kmc-approach_b200/csrc/grain_shape.cuh"

using namespace cet;

// Q_x of count grains (m: count x SHAPE_WORDS moment slots) along axis x, as (low, high) 64-bit halves
extern "C" void hostsim_shape_q(const uint64_t *m, long long count, int x, uint64_t *out)
{
    for (long long g = 0; g < count; ++g) {
        const uint64_t *s = m + g * SHAPE_WORDS;
        const u128 q = shape_q(s[SHAPE_N], s[SHAPE_S + x], s[SHAPE_SS + x]);
        out[2 * g] = (uint64_t)q;
        out[2 * g + 1] = (uint64_t)(q >> 64);
    }
}

// fl() of count integers v < 2^106 given as (low, high) 64-bit halves
extern "C" void hostsim_shape_fl(const uint64_t *v, long long count, double *out)
{
    for (long long g = 0; g < count; ++g) out[g] = shape_fl(((u128)v[2 * g + 1] << 64) | v[2 * g]);
}

// A and the bin of count grains
extern "C" void hostsim_shape_bins(const uint64_t *m, long long count, int axis, const double *edges, int n_edges,
                                   long long min_size, double *a_out, int32_t *bin_out)
{
    for (long long g = 0; g < count; ++g) {
        a_out[g] = shape_elongation(m + g * SHAPE_WORDS, axis);
        bin_out[g] = shape_bin(m + g * SHAPE_WORDS, axis, edges, n_edges, min_size);
    }
}
