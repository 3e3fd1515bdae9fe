"""Test infrastructure: a NumPy / Python-integer restatement of cet_grain_shape_group (cetkmc.grain_shape_group) from a
label volume, used as the checker of the device histograms; nothing in the product imports it.  The moments are exact
int64 sums, Q is computed in Python integers, fl() is float(int), and the division and square root are IEEE fp64, so
the elongation of every grain has the bits the device computes."""
import math

import numpy as np


def grain_moments(labels, n_grains=None):
    """Per grain (numbered 1..n_grains in `labels`, 0 = empty): n and, per axis x, S_x and S_xx, as int64 arrays
    (n, (3, n), (3, n))."""
    labels = np.asarray(labels)
    n_grains = int(labels.max(initial=0)) if n_grains is None else int(n_grains)
    occ = labels > 0
    lab = labels[occ].astype(np.int64) - 1
    n = np.bincount(lab, minlength=n_grains).astype(np.int64)
    s = np.zeros((3, n_grains), np.int64)
    ss = np.zeros((3, n_grains), np.int64)
    for ax, c in enumerate(np.nonzero(occ)):
        c = c.astype(np.int64)
        np.add.at(s[ax], lab, c)
        np.add.at(ss[ax], lab, c * c)
    return n, s, ss


def q_moment(n, s, ss):
    """Q = 12 (n S_xx - S_x^2) + n^2, exact (Python integers)."""
    n, s, ss = int(n), int(s), int(ss)
    return 12 * (n * ss - s * s) + n * n


def elongation_of(n, s, ss, axis):
    """A of one grain from its moments (n, [S_0, S_1, S_2], [S_00, S_11, S_22]) along `axis`."""
    q = [q_moment(n, s[x], ss[x]) for x in range(3)]
    b, c = [x for x in range(3) if x != axis]
    return math.sqrt(float(2 * q[axis]) / float(q[b] + q[c]))


def elongations(labels, axis, n_grains=None):
    """(sizes, A) per grain of the label volume."""
    n, s, ss = grain_moments(labels, n_grains)
    no = n.astype(object)
    q = [12 * (no * ss[x].astype(object) - s[x].astype(object) ** 2) + no * no for x in range(3)]
    b, c = [x for x in range(3) if x != axis]
    num = np.array([float(v) for v in 2 * q[axis]], np.float64)
    den = np.array([float(v) for v in q[b] + q[c]], np.float64)
    return n, np.sqrt(num / den)


def grain_shape(labels, axis, edges, min_size, n_grains=None):
    """(2, len(edges) + 2) int64: grains and sites per bin (bin b: size >= min_size and edges[b-1] <= A < edges[b]),
    and in the last bin the grains of fewer than min_size sites."""
    e = np.asarray(edges, np.float64)
    n, a = elongations(labels, axis, n_grains)
    out = np.zeros((2, e.size + 2), np.int64)
    big = n >= int(min_size)
    b = np.where(big, np.searchsorted(e, a, side="right"), e.size + 1)
    np.add.at(out[0], b, 1)
    np.add.at(out[1], b, n)
    return out
