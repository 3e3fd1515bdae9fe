// grain_shape.cuh — the growth-axis elongation A of a grain and its histogram bin (cet_grain_shape_group), from the
// grain's exact integer moments.  A grain of n sites at coordinates c = (i, j, k) has, per axis x, S_x = sum c_x and
// S_xx = sum c_x^2, and
//     Q_x = 12 (n S_xx - S_x^2) + n^2          (n^2 times 12 (variance along x + 1/12): each site a unit cube)
//     A   = sqrt(fl(2 Q_a) / fl(Q_b + Q_c))    (a the growth axis, b and c the other two)
// where fl() rounds an unsigned integer to the nearest double (ties to even, as Python's float(int)) and the
// division and square root are IEEE round-to-nearest.  Every step before fl() is exact in unsigned 128-bit
// arithmetic, so A is one fixed sequence of correctly rounded operations on exact integers: a host reference
// reproduces it bit for bit.  A single site has A = 1, a 1 x 1 x h column along a has A = h, an a x b x c box
// sqrt(2 a^2 / (b^2 + c^2)).
// The kernels of grain_shape_group.cu inline these functions; they also compile for the host (g++, tests/hostsim
// only: a checker of this arithmetic that needs no GPU).
#pragma once
#include <math.h>
#include <stdint.h>
#include "site_rates.cuh"

namespace cet {

typedef unsigned __int128 u128;

// One grain's slot of the per-grain moment buffer: n, S_0, S_1, S_2, S_00, S_11, S_22 and a pad word (64 bytes).
// A context has fewer than 2^31 sites and L < 1291, so S_x < 2^42 and S_xx < 2^52.
enum { SHAPE_N = 0, SHAPE_S = 1, SHAPE_SS = 4, SHAPE_WORDS = 8 };
constexpr int SHAPE_EDGES_MAX = 62;

// n S_xx >= S_x^2 (Cauchy-Schwarz), so the difference is exact; Q < 2^84 for any grain of a context
CET_HD u128 shape_q(uint64_t n, uint64_t s, uint64_t ss)
{
    return (u128)12 * ((u128)n * ss - (u128)s * s) + (u128)n * n;
}

// fl(v) for v < 2^106: v = h 2^53 + l with h, l < 2^53 exact in fp64, h 2^53 exact, one rounding of the exact sum
CET_HD double shape_fl(u128 v)
{
    const double h = (double)(uint64_t)(v >> 53), l = (double)((uint64_t)v & ((1ull << 53) - 1));
#if defined(__CUDA_ARCH__)
    return __dadd_rn(__dmul_rn(h, 0x1p53), l);
#else
    return h * 0x1p53 + l;
#endif
}

// A of the grain with moments m[SHAPE_WORDS] along growth axis `axis` (constant indices only, so that a kernel
// keeps m in registers)
CET_HD double shape_elongation(const uint64_t *m, int axis)
{
    const uint64_t n = m[SHAPE_N];
    const u128 q0 = shape_q(n, m[SHAPE_S + 0], m[SHAPE_SS + 0]), q1 = shape_q(n, m[SHAPE_S + 1], m[SHAPE_SS + 1]),
               q2 = shape_q(n, m[SHAPE_S + 2], m[SHAPE_SS + 2]);
    const u128 qa = axis == 0 ? q0 : axis == 1 ? q1 : q2;
    const u128 qbc = axis == 0 ? q1 + q2 : axis == 1 ? q0 + q2 : q0 + q1;
    const double num = shape_fl(2 * qa), den = shape_fl(qbc);
#if defined(__CUDA_ARCH__)
    return __dsqrt_rn(__ddiv_rn(num, den));
#else
    return sqrt(num / den);
#endif
}

// The histogram bin of a grain: n_edges + 1 when it has fewer than min_size sites, else the number of edges
// e_b <= A (bin b holds e_{b-1} <= A < e_b, with e_{-1} = 0 and e_{n_edges} = infinity)
CET_HD int shape_bin(const uint64_t *m, int axis, const double *edges, int n_edges, int64_t min_size)
{
    if ((int64_t)m[SHAPE_N] < min_size) return n_edges + 1;
    const double A = shape_elongation(m, axis);
    int b = 0;
    while (b < n_edges && edges[b] <= A) ++b;
    return b;
}

}  // namespace cet
