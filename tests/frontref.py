"""NumPy reference of cet_front_group: the four column arrays of one lattice along a growth axis, from the state
(Context.download(state=True)) and T (download(T=True)), bit for bit."""
import numpy as np

NAN = np.uint64(0x7FF8000000000000).view(np.float64)      # the one quiet NaN of T_front / dT_front


def front(state, T, axis):
    """(front, top, T_front, dT_front), each (L, L): column (u, w) is the line along `axis` at the other two
    coordinates, u the lower-numbered axis; plane 0 is where growth starts."""
    occ = np.moveaxis(np.asarray(state) != 0, axis, -1)
    Tm = np.moveaxis(np.asarray(T, np.float64), axis, -1)
    L = occ.shape[-1]
    hole = ~occ
    h = np.where(hole.any(-1), hole.argmax(-1), L).astype(np.int32)
    top = np.where(occ.any(-1), L - occ[..., ::-1].argmax(-1), 0).astype(np.int32)
    at = np.minimum(h, L - 1).astype(np.int64)[..., None]
    t1 = np.take_along_axis(Tm, at, -1)[..., 0]
    t0 = np.take_along_axis(Tm, np.maximum(at - 1, 0), -1)[..., 0]
    with np.errstate(invalid="ignore"):
        d = t1 - t0
    d = np.where(np.isnan(d), NAN, d)
    T_front = np.where(h < L, t1, NAN)
    dT_front = np.where((h > 0) & (h < L), d, NAN)
    return h, top, T_front, dT_front


def bits(a):
    """The bit patterns of a float64 array (NaN payloads included), for exact comparison."""
    return np.ascontiguousarray(a, np.float64).view(np.uint64)
