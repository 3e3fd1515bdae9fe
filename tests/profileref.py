"""Test infrastructure: a NumPy restatement of cet_grain_profile_group (cetkmc.grain_profile_group) from a label
volume, used as the checker of the device profile; nothing in the product imports it."""
import numpy as np


def grain_boxes(labels, n_grains):
    """Per grain (numbered 1..n_grains in `labels`, 0 = empty): voxel count and bounding box lo / hi, (n, 3)."""
    occ = labels > 0
    lab = labels[occ].astype(np.int64) - 1
    sizes = np.bincount(lab, minlength=n_grains)
    coords = np.nonzero(occ)
    lo = np.full((n_grains, 3), np.iinfo(np.int64).max)
    hi = np.full((n_grains, 3), -1)
    for ax in range(3):
        np.minimum.at(lo[:, ax], lab, coords[ax])
        np.maximum.at(hi[:, ax], lab, coords[ax])
    return sizes, lo, hi


def aspect_ratios(lo, hi):
    """utils.py:104-111 per grain: longest / max(shortest, 1) of the bounding-box dimensions."""
    dims = hi - lo + 1
    if dims.shape[0] == 0:
        return np.zeros(0)
    return dims.max(axis=1).astype(np.float64) / np.maximum(dims.min(axis=1), 1).astype(np.float64)


def grain_profile(labels, axis, ar_threshold, n_grains=None):
    """(4, L) int64: per plane z along `axis`, the occupied sites, those of grains with AR < ar_threshold, the grains
    whose bounding box along `axis` contains z, and the equiaxed ones among them."""
    labels = np.asarray(labels)
    n = int(labels.max()) if n_grains is None else int(n_grains)
    L = labels.shape[axis]
    out = np.zeros((4, L), np.int64)
    if n == 0:
        return out
    _sizes, lo, hi = grain_boxes(labels, n)
    eq = aspect_ratios(lo, hi) < ar_threshold
    occ = labels > 0
    eq_site = np.zeros(labels.shape, bool)
    eq_site[occ] = eq[labels[occ] - 1]
    other = tuple(a for a in range(3) if a != axis)
    out[0] = occ.sum(axis=other)
    out[1] = eq_site.sum(axis=other)
    z = np.arange(L)
    span = (lo[:, axis][:, None] <= z[None, :]) & (z[None, :] <= hi[:, axis][:, None])
    out[2] = span.sum(axis=0)
    out[3] = span[eq].sum(axis=0)
    return out
