"""The sites whose rates read the temperature of a site x, against the oracle.  After a thermal step cet_sweep_run
refreshes only the sites within this set of a changed site (csrc/sweep.cu, thermal_stale_kernel): x itself, x +- 1 and
x +- 2 along k, x + (0, +-1, +-1), x + (+-1, +-1, 0), x + (+-2, 0, 0) and x + (0, +-2, 0).  A perturbation of T at x
must change no other site's rate sum or deposition rate."""
import numpy as np
import pytest


def _stale_set(x, L):
    i, j, k = x
    offs = {(0, 0, 0), (0, 0, 1), (0, 0, -1), (0, 0, 2), (0, 0, -2), (2, 0, 0), (-2, 0, 0), (0, 2, 0), (0, -2, 0)}
    offs |= {(0, a, b) for a in (-1, 1) for b in (-1, 1)} | {(a, b, 0) for a in (-1, 1) for b in (-1, 1)}
    return {(i + a, j + b, k + c) for a, b, c in offs if 0 <= i + a < L and 0 <= j + b < L and 0 <= k + c < L}


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_rates_read_T_only_within_the_stale_set(oracle, seed):
    L = 12
    st, th, ph, T, df = oracle.half_grown_lattice(L, seed=seed, grain=3)
    P = oracle.make_params(0.1)
    sr0, dep0, _, _ = oracle.site_rates(st, th, ph, T, df, L, P)
    rng = np.random.default_rng(seed)
    sites = [(5, 6, 5), (0, 0, 0), (1, L - 1, 1), (L - 1, 4, 7), (L - 1, L - 1, L - 1), (L - 2, 0, L - 2), (6, 1, L - 1)]
    sites += [tuple(int(v) for v in rng.integers(0, L, 3)) for _ in range(6)]
    seen = 0
    for x in sites:
        for dT in (-350.0, 0.125, 900.0):
            T1 = T.copy()
            T1[x] += dT
            sr1, dep1, _, _ = oracle.site_rates(st, th, ph, T1, df, L, P)
            moved = {tuple(int(v) for v in s) for s in np.argwhere(sr1.view(np.int64) != sr0.view(np.int64))}
            moved |= {(L - 1, int(j), int(k)) for j, k in np.argwhere(dep1.view(np.int64) != dep0.view(np.int64))}
            assert moved <= _stale_set(x, L), (x, dT, sorted(moved - _stale_set(x, L)))
            seen += len(moved)
    assert seen > 0
