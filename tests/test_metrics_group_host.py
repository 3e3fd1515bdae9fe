"""CPU: the host side of the grouped metrics cadence (cetkmc.metrics_group).  NumPy's mean over a list of floats
is the pairwise recursion the device restates; a metrics dict built from the per-lattice summary the device
returns equals metrics_from_grains value for value and type for type; the ctypes structs match the header; the
bindings check their lists before the library is reached."""
import ctypes as C

import numpy as np
import pytest

from conftest import golden
import hostref
from cetkmc import _lib, metrics


def pw(a, lo, n):
    """cet_metrics_group's AR sum: NumPy's pairwise_sum over the whole array (leaves of <= 128 elements with 8
    accumulators, splits at multiples of 8)."""
    if n < 8:
        r = -0.0
        for i in range(n):
            r += a[lo + i]
        return r
    if n <= 128:
        r = a[lo:lo + 8]
        i = 8
        while i < n - n % 8:
            r = [r[j] + a[lo + i + j] for j in range(8)]
            i += 8
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        for k in range(i, n):
            res += a[lo + k]
        return res
    n2 = n // 2
    n2 -= n2 % 8
    return pw(a, lo, n2) + pw(a, lo + n2, n - n2)


def ar_like(rng, n):
    hi, lo = rng.integers(1, 97, n), rng.integers(1, 97, n)
    return np.maximum(hi, lo).astype(np.float64) / np.minimum(hi, lo).astype(np.float64)


@pytest.mark.parametrize("n", [1, 2, 7, 8, 9, 127, 128, 129, 255, 8191, 8192, 8193, 10 ** 5, 10 ** 6])
def test_pairwise_recursion_is_numpys_mean(n):
    a = ar_like(np.random.default_rng(n), n)
    a[::7] *= 1.0 + 1e-3 * np.random.default_rng(n + 1).random(len(a[::7]))     # not only ratios of small integers
    lst = a.tolist()
    assert (-0.0 + pw(lst, 0, n)) / n == np.mean(lst)
    assert np.float64(pw(lst, 0, n)) / n == np.mean(lst)


def summary(sizes, ar, n_sites, thr):
    """What cet_metrics_group returns for grains of these sizes and aspect ratios, in cluster order."""
    sizes = np.asarray(sizes, np.int64)
    cum = np.cumsum(np.concatenate(([n_sites - int(sizes.sum())], sizes)))
    pos = metrics.percentile_positions(n_sites)
    return dict(n_grains=len(sizes), size_sum=int(sizes.sum()), n_equiaxed=int(np.sum(ar < thr)),
                ar_sum=pw(ar.tolist(), 0, len(sizes)), pct_index=[int(np.searchsorted(cum, x, side="right")) for x in pos])


def same_dict(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert type(a[k]) is type(b[k]), (k, type(a[k]), type(b[k]))
        assert a[k] == b[k] or (a[k] != a[k] and b[k] != b[k]), (k, a[k], b[k])


def boxes(labels, n):
    lab = labels[labels > 0].astype(np.int64) - 1
    coords = np.nonzero(labels > 0)
    lo = np.full((n, 3), np.iinfo(np.int64).max)
    hi = np.full((n, 3), -1)
    for ax in range(3):
        np.minimum.at(lo[:, ax], lab, coords[ax])
        np.maximum.at(hi[:, ax], lab, coords[ax])
    return lo.astype(np.int32), hi.astype(np.int32)


@pytest.mark.parametrize("name", ["grains_grown12.npz", "grains_grown16.npz", "grains_half14.npz"])
def test_summary_metrics_match_grain_metrics_on_golden_lattices(name):
    d = golden(name)
    labels = d["visited"]
    n = int(labels.max())
    sizes, ar = hostref.grain_statistics(labels, n)
    lo, hi = boxes(labels, n)
    g = dict(n=n, size=sizes.astype(np.int32), box_lo=lo, box_hi=hi)
    assert np.array_equal(metrics.grain_aspect_ratios(g), ar)
    thr = metrics.K.CET_AR_THRESHOLD
    same_dict(metrics.metrics_from_summary(summary(sizes, ar, labels.size, thr), labels.size),
              metrics.metrics_from_grains(g, labels.size))


@pytest.mark.parametrize("n", [0, 1, 5, 100, 129])
def test_summary_metrics_match_grain_metrics_on_synthetic_statistics(n):
    rng = np.random.default_rng(n)
    n_sites = 40 ** 3
    lo = rng.integers(0, 30, (n, 3)).astype(np.int32)
    hi = (lo + rng.integers(0, 10, (n, 3))).astype(np.int32)
    sizes = rng.integers(1, 400, n).astype(np.int32)
    g = dict(n=n, size=sizes, box_lo=lo, box_hi=hi)
    ar = metrics.grain_aspect_ratios(g)
    thr = metrics.K.CET_AR_THRESHOLD
    same_dict(metrics.metrics_from_summary(summary(sizes, ar, n_sites, thr), n_sites),
              metrics.metrics_from_grains(g, n_sites))


def test_struct_sizes_match_header():
    assert C.sizeof(_lib.MetricsParams) == 2 * 8 + 4 * 8 + 4 * 4 + 8 + 4 * 8
    assert C.sizeof(_lib.MetricsResult) == 16 * 8 + 9 * 8 + 8


def test_group_bindings_check_their_lists_before_the_library(monkeypatch):
    def no_library():
        raise AssertionError("the library must not be reached")
    monkeypatch.setattr(_lib, "lib", no_library)
    mp = _lib.MetricsParams()
    with pytest.raises(TypeError):
        _lib.counts_group([object()])
    with pytest.raises(ValueError):
        _lib.metrics_group([object(), object()], [mp])
    with pytest.raises(ValueError):
        _lib.metrics_group([object()], [mp], draws=[None, None])
    with pytest.raises(TypeError):
        _lib.metrics_group([object()], [object()])
    with pytest.raises(TypeError):
        _lib.metrics_group([object()], [mp])
