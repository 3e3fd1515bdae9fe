"""NumPy reference of cet_boundary_group: the per-plane table of one lattice along a growth axis, from the label volume of
the last labelling (Context.grains(labels=True), or cet_grains_download_labels) and the raw bytes of the resident
orientation vectors (device_ptr(5): 32-byte records x, y, z, pad), bit for bit.  The misorientation cosine takes the
kernel's operation order, one np.multiply or np.add on float64 per step (no fused multiply-add)."""
import numpy as np

SCALE = 2.0 ** 32
OFFSETS = ((1, 1, 0), (1, -1, 0), (0, 1, 1), (0, 1, -1), (2, 0, 0), (0, 2, 0), (0, 0, 2))


def misorientation_cos(a, b):
    """d = clamp(fl(fl(fl(x x') + fl(y y')) + fl(z z')), -1, 1) of the rows of two (n, >= 3) float64 arrays, the
    clamp pymax(pymin(d, 1), -1)."""
    d = np.add(np.add(np.multiply(a[:, 0], b[:, 0]), np.multiply(a[:, 1], b[:, 1])), np.multiply(a[:, 2], b[:, 2]))
    d = np.where(d > 1.0, 1.0, d)
    return np.where(d < -1.0, -1.0, d)


def table(labels, v, axis, edges):
    """The (L, 21 + len(edges) + 2) int64 rows of the ABI for one lattice: per plane z along `axis`, the bonds of
    offset r and class f at column 3 r + f (f: 0 solid, 1 boundary, 2 interface), the boundary bonds per bin
    b = #{i : edges[i] <= d} at column 21 + b, then F = sum rint(d 2^32)."""
    lab = np.asarray(labels)
    v = np.asarray(v, np.float64)
    e = np.asarray(edges, np.float64)
    L, m = lab.shape[0], e.size
    W = 21 + m + 2
    out = np.zeros((L, W), np.int64)
    coord = np.indices(lab.shape)[axis]
    for r, d in enumerate(OFFSETS):
        src = tuple(slice(max(0, -x), L - max(0, x)) for x in d)
        dst = tuple(slice(max(0, x), L - max(0, -x)) for x in d)
        a, b = lab[src], lab[dst]
        plane = np.minimum(coord[src], coord[dst])
        oa, ob = a >= 0, b >= 0
        sol = oa & ob
        bnd = sol & (a != b)
        for f, mask in enumerate((sol, bnd, oa != ob)):
            out[:, 3 * r + f] += np.bincount(plane[mask], minlength=L)
        dc = misorientation_cos(v[src][bnd], v[dst][bnd])
        pz = plane[bnd]
        np.add.at(out, (pz, 21 + np.searchsorted(e, dc, side="right")), 1)
        np.add.at(out[:, W - 1], pz, np.rint(np.multiply(dc, SCALE)).astype(np.int64))
    return out


def split(tab):
    """The binding's (bonds (L, 7, 3), hist in ascending angle, sum_cos) of one lattice's ABI table."""
    m = tab.shape[1] - 23
    return tab[:, :21].reshape(-1, 7, 3), tab[:, 21 + m:20:-1], tab[:, 21 + m + 1]
