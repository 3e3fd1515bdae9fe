"""NumPy reference of cet_texture_group: the per-plane table of one lattice along a growth axis, from the state
(Context.download(state=True), or the packed vox of download_packed) and the raw bytes of the resident orientation
vectors (device_ptr(5): 32-byte records x, y, z, pad), bit for bit."""
import numpy as np

SCALE = 2.0 ** 32


def vectors(raw, L):
    """The (L, L, L, 4) float64 records of the raw bytes of v."""
    return np.frombuffer(np.ascontiguousarray(raw, np.uint8).tobytes(), np.float64).reshape(L, L, L, 4)


def table(state, v, axis, edges):
    """The (L, n_edges + 3) int64 rows of the ABI for one lattice: per plane z along `axis`, the occupied sites in bin
    j = #{i : edges[i] <= c} (c = v[..., axis]), then F1 = sum rint(c 2^32) and F2 = sum rint(fl(c c) 2^32)."""
    return table_c(state, np.asarray(v, np.float64)[..., axis], axis, edges)


def table_c(state, c, axis, edges):
    """table() from the (L, L, L) component c = v[..., axis] alone."""
    e = np.asarray(edges, np.float64)
    occ = np.moveaxis((np.asarray(state) & 0x0F) != 0, axis, 0)
    c = np.moveaxis(np.asarray(c, np.float64), axis, 0)
    L, m = occ.shape[0], e.size
    out = np.zeros((L, m + 3), np.int64)
    for z in range(L):
        cz = c[z][occ[z]]
        b = np.searchsorted(e, cz, side="right")                 # #{i : e_i <= c}
        out[z, :m + 1] = np.bincount(b, minlength=m + 1)
        out[z, m + 1] = int(np.rint(cz * SCALE).astype(np.int64).sum())
        out[z, m + 2] = int(np.rint((cz * cz) * SCALE).astype(np.int64).sum())
    return out


def split(tab):
    """The binding's (hist in ascending angle, sum_cos, sum_cos2) of one lattice's ABI table."""
    m = tab.shape[1] - 3
    return tab[:, m::-1], tab[:, m + 1], tab[:, m + 2]
