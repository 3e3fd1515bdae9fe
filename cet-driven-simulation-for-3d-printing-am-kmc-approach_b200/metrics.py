"""Drop-in for the observables the KMC driver takes from the reference's metrics.py / utils.py
(SURVEY §8f row N1): grain clustering runs on the GPU (csrc/grains.cu, a union-find connected-
component labelling over the 14-offset neighbourhood) instead of the pure-Python DFS of
utils.py:28-84, which costs ~1 s at 30^3 and is run twice per metrics row
(kmc_simulation.py:341-377).

    compute_metrics(state, theta, phi, defects=None, ...)   metrics.py:41-96
    compute_CET(state, theta, phi)                          metrics.py:99-101
    detect_CET_transition(metrics_dict)                     metrics.py:103-105
    get_clusters(state, theta, phi, theta_threshold=0.5)    utils.py:69-84
    calculate_aspect_ratio(cluster)                         utils.py:104-111

`compute_metrics(..., ctx=<cetkmc.Context>)` clusters the lattice already resident in HBM (what
`run_kmc` does every METRIC_UPDATE_STEP steps) and needs no upload.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from ._config import constants as K


def _percentile_position(n, q):
    """(pos, lo, hi) of np.percentile's linear method over n values: pos = q/100 * (n - 1), its floor and ceil."""
    pos = (q / 100.0) * (n - 1)
    return pos, int(np.floor(pos)), int(np.ceil(pos))


def _interpolate(values, pos, lo, i_lo, i_hi):
    a = float(values[i_lo])
    b = float(values[i_hi])
    t = pos - lo
    return a + (b - a) * t if t < 0.5 else b - (b - a) * (1 - t)


def _percentile_of_counts(values, counts, q):
    """np.percentile(np.repeat(values, counts), q) (method 'linear') without materialising the
    repeat; values ascending."""
    n = int(np.sum(counts))
    if n == 0:
        return 0.0
    cum = np.cumsum(counts)
    pos, lo, hi = _percentile_position(n, q)
    return _interpolate(values, pos, lo, np.searchsorted(cum, lo, side="right"), np.searchsorted(cum, hi, side="right"))


PERCENTILES = (50.0, 90.0)          # Grain_d50_um, Grain_d90_um


def percentile_positions(n_sites):
    """The lo and hi positions of each of PERCENTILES over n_sites values, in that order: what
    cet_metrics_params.pct_pos takes (metrics_from_summary reads the indices the device returns for them)."""
    out = []
    for q in PERCENTILES:
        _pos, lo, hi = _percentile_position(n_sites, q)
        out += [lo, hi]
    return out


def grain_aspect_ratios(g):
    """utils.py:104-111 per grain: longest / max(shortest, 1) of the bounding-box dimensions."""
    dims = (g["box_hi"].astype(np.int64) - g["box_lo"].astype(np.int64)) + 1
    if dims.shape[0] == 0:
        return np.zeros(0)
    return dims.max(axis=1).astype(np.float64) / np.maximum(dims.min(axis=1), 1).astype(np.float64)


def metrics_from_grains(g, n_sites, defects=None, voxel_size=None, rng_seed=None):
    """metrics.py:41-96 from the per-grain statistics of Context.grains()."""
    voxel_size = K.VOXEL_SIZE if voxel_size is None else voxel_size
    n = int(g["n"])
    if n == 0:
        return _no_grains(voxel_size, rng_seed)
    ar = grain_aspect_ratios(g)
    sizes = g["size"].astype(np.int64)
    volume = n_sites * (voxel_size ** 3)
    def_count = np.sum(defects) if defects is not None else 0
    # metrics.py:43,76 hands the `visited` label volume (not the sizes) to equivalent_diameter_um:
    # value 0 on the empty sites, grain number q (1..n) on the sizes[q-1] voxels of grain q
    vals = np.arange(0, n + 1, dtype=np.float64)
    cnts = np.concatenate(([n_sites - int(sizes.sum())], sizes))
    diam = ((6.0 * (vals * (voxel_size ** 3)) / np.pi) ** (1.0 / 3.0)) * 1e6
    return {
        "AspectRatio": np.mean(ar.tolist()),
        "EquiaxedFraction": np.mean(ar < K.CET_AR_THRESHOLD),
        "NucleationDensity": n / volume if volume > 0 else 0.0,
        "AvgGrainSize": np.mean(sizes.tolist()) * voxel_size * 1e6,
        "GrainCount": n,
        "DefectDensity": def_count / volume if volume > 0 else 0.0,
        "Frac_W": 0.0, "Frac_Re": 0.0, "Frac_C": 0.0,
        "C_boundary_frac": 0.0, "Re_boundary_frac": 0.0,
        "Defect_voxel_count": def_count,
        "Defect_voxel_frac": def_count / n_sites if n_sites > 0 else 0.0,
        "Grain_d50_um": _percentile_of_counts(diam, cnts, 50.0),
        "Grain_d90_um": _percentile_of_counts(diam, cnts, 90.0),
        "VOXEL_SIZE_m": voxel_size, "RANDOM_SEED": rng_seed,
    }


def _no_grains(voxel_size, rng_seed):
    return {"AspectRatio": 0.0, "EquiaxedFraction": 0.0, "NucleationDensity": 0.0,
            "AvgGrainSize": 0.0, "GrainCount": 0, "DefectDensity": 0.0,
            "Frac_W": 0.0, "Frac_Re": 0.0, "Frac_C": 0.0,
            "C_boundary_frac": 0.0, "Re_boundary_frac": 0.0,
            "Defect_voxel_count": 0, "Defect_voxel_frac": 0.0,
            "Grain_d50_um": 0.0, "Grain_d90_um": 0.0,
            "VOXEL_SIZE_m": voxel_size, "RANDOM_SEED": rng_seed}


def metrics_from_summary(res, n_sites, voxel_size=None, rng_seed=None):
    """metrics_from_grains(g, n_sites) from the per-lattice summary of cetkmc.metrics_group (n_grains, size_sum,
    n_equiaxed, ar_sum in NumPy's pairwise order, and the percentile indices for percentile_positions(n_sites)):
    the same dict, value for value and type for type.  np.mean over the AR list is pw(ar) / n, over the bool
    array n_equiaxed / n, and over the int64 sizes size_sum / n, exact below 2^53."""
    voxel_size = K.VOXEL_SIZE if voxel_size is None else voxel_size
    n = int(res["n_grains"])
    if n == 0:
        return _no_grains(voxel_size, rng_seed)
    volume = n_sites * (voxel_size ** 3)
    def_count = 0
    # the diameters of the grain numbers 0..n, as metrics_from_grains evaluates them
    vals = np.arange(0, n + 1, dtype=np.float64)
    diam = ((6.0 * (vals * (voxel_size ** 3)) / np.pi) ** (1.0 / 3.0)) * 1e6
    idx = [int(i) for i in res["pct_index"]]
    d = []
    for k, q in enumerate(PERCENTILES):
        pos, lo, _hi = _percentile_position(n_sites, q)
        d.append(_interpolate(diam, pos, lo, idx[2 * k], idx[2 * k + 1]))
    return {
        "AspectRatio": np.float64(res["ar_sum"]) / n,
        "EquiaxedFraction": np.float64(res["n_equiaxed"]) / n,
        "NucleationDensity": n / volume if volume > 0 else 0.0,
        "AvgGrainSize": np.float64(res["size_sum"]) / n * voxel_size * 1e6,
        "GrainCount": n,
        "DefectDensity": def_count / volume if volume > 0 else 0.0,
        "Frac_W": 0.0, "Frac_Re": 0.0, "Frac_C": 0.0,
        "C_boundary_frac": 0.0, "Re_boundary_frac": 0.0,
        "Defect_voxel_count": def_count,
        "Defect_voxel_frac": def_count / n_sites if n_sites > 0 else 0.0,
        "Grain_d50_um": d[0],
        "Grain_d90_um": d[1],
        "VOXEL_SIZE_m": voxel_size, "RANDOM_SEED": rng_seed,
    }


def cet_profile_summary(profile, plane_sites, eq_threshold=K.CET_EQ_THRESHOLD, min_solid=0.5):
    """Where along the profile's axis a lattice turns equiaxed, from one (4, L) grain profile of
    cetkmc.grain_profile_group (rows Solid, EquiaxedSolid, GrainsSpanning, EquiaxedGrainsSpanning).

    The solidified planes P are the planes z with Solid[z] >= min_solid * plane_sites (plane_sites: the
    sites of one plane, L * L), so melt or vapour planes above the front do not count; a plane without
    solid is never in P.
        Front_Height  the largest z in P; -1 when P is empty.
        CET_Height    with eq[z] = EquiaxedSolid[z] / Solid[z], the smallest z in P such that
                      eq[z'] >= eq_threshold for every z' in P with z' >= z; -1 when P is empty or the
                      top plane of P is below the threshold.
    A lattice equiaxed through every solidified plane gets the lowest plane of P (0 when the substrate
    plane is solidified); a lattice columnar at its front gets -1; an equiaxed plane below a columnar band
    does not count.  Returns {"CET_Height": int, "Front_Height": int}."""
    p = np.asarray(profile)
    if p.ndim != 2 or p.shape[0] != 4:
        raise ValueError(f"cet_profile_summary: need a (4, L) profile, got shape {p.shape}")
    solid, eq_solid = p[0].astype(np.float64), p[1].astype(np.float64)
    planes = np.nonzero(solid >= float(min_solid) * float(plane_sites))[0]
    planes = planes[solid[planes] > 0]
    if planes.size == 0:
        return {"CET_Height": -1, "Front_Height": -1}
    eq = eq_solid[planes] / solid[planes]
    cet = -1
    for k in range(planes.size - 1, -1, -1):            # walk down from the front while the planes stay equiaxed
        if eq[k] < eq_threshold:
            break
        cet = int(planes[k])
    return {"CET_Height": cet, "Front_Height": int(planes[-1])}


def grains_distributed(ctx, all_gather, theta_threshold=0.5):
    """Grains of a lattice that is split into z-slabs over several contexts (one per rank), in the form
    Context.grains() returns for a whole lattice — the reference's clusters (utils.py:28-84) in its
    order — identical on every rank.

    Every slab labels its owned planes plus 2 ghost planes per cut face (cet_grains_label).  A grain
    that crosses a cut is a local component on both sides, and the two slabs give the SAME sites of
    the 2 planes below the cut two labels: the pairs (label below, label above) are the edges that
    join local components into grains.  They are gathered (a few thousand integers per cut), the
    components of that small graph are found on the host, and the per-component statistics (voxel
    counts of owned sites, bounding boxes) are added up per grain.

    ctx: this rank's Context (ghost planes current, i.e. after the sweep's exchange);
    all_gather(obj) -> list of every rank's obj in rank order (e.g. torch.distributed.all_gather_object
    wrapped; see campaign.run_cet_sublattice)."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    loc = ctx.grains_local(theta_threshold)
    i_begin, i_end = ctx.i_begin, ctx.i_end
    n0 = ctx.n0
    # the 2 owned planes below my upper cut, as I label them; and the neighbour's 2 planes below my lower
    # cut (ghosts here), as I label them
    mine_top = ctx.grain_label_planes(i_end - 2, i_end) if i_end < n0 else None
    ghost_below = ctx.grain_label_planes(i_begin - 2, i_begin) if i_begin > 0 else None
    tops = all_gather(mine_top)                         # tops[r] = rank r's labels of its top 2 owned planes
    pairs = np.zeros((0, 2), np.int64)
    if ghost_below is not None:
        theirs = tops[ctx.rank - 1]
        occ = ghost_below >= 0
        pairs = np.unique(np.stack([theirs[occ].astype(np.int64), ghost_below[occ].astype(np.int64)], axis=1), axis=0)
    gathered = all_gather((loc, pairs))
    root = np.concatenate([g[0]["root"] for g in gathered])
    size = np.concatenate([g[0]["size"] for g in gathered])
    lo = np.concatenate([g[0]["box_lo"] for g in gathered]).astype(np.int64)
    hi = np.concatenate([g[0]["box_hi"] for g in gathered]).astype(np.int64)
    edges = np.concatenate([g[1] for g in gathered])
    # local components that share a global root index on two ranks do not exist (a root is the smallest
    # LOCAL site of the component, and each rank reports it as a global index of its own labelling), but a
    # component is reported by every rank that labelled any of its sites: ids = unique (rank, root) pairs
    owner = np.concatenate([np.full(len(g[0]["root"]), r, np.int64) for r, g in enumerate(gathered)])
    key = owner * (np.int64(1) << 40) + root
    order = np.argsort(key)
    key, root, size, lo, hi, owner = key[order], root[order], size[order], lo[order], hi[order], owner[order]

    def node(rank_of, roots):
        return np.searchsorted(key, rank_of * (np.int64(1) << 40) + roots)

    n = len(key)
    if n == 0:
        z = np.zeros((0, 3), np.int32)
        return dict(n=0, root=np.zeros(0, np.int32), size=np.zeros(0, np.int32), box_lo=z, box_hi=z)
    if len(edges):
        e_rank = np.concatenate([np.full(len(g[1]), r, np.int64) for r, g in enumerate(gathered)])
        a = node(e_rank - 1, edges[:, 0])               # the lower slab's component ...
        b = node(e_rank, edges[:, 1])                   # ... is the same grain as the upper slab's
        graph = coo_matrix((np.ones(len(a), np.int8), (a, b)), shape=(n, n))
    else:
        graph = coo_matrix((n, n), dtype=np.int8)
    n_comp, comp = connected_components(graph, directed=False)
    g_size = np.bincount(comp, weights=size, minlength=n_comp).astype(np.int64)
    big = np.iinfo(np.int64).max
    g_lo = np.full((n_comp, 3), big, np.int64); g_hi = np.full((n_comp, 3), -1, np.int64)
    has = size > 0
    np.minimum.at(g_lo, comp[has], lo[has]); np.maximum.at(g_hi, comp[has], hi[has])
    g_root = np.full(n_comp, big, np.int64)
    np.minimum.at(g_root, comp, root)                   # = the grain's smallest site: its owner's component is rooted there
    keep = g_size > 0
    order = np.argsort(g_root[keep], kind="stable")
    return dict(n=int(keep.sum()), root=g_root[keep][order].astype(np.int64), size=g_size[keep][order].astype(np.int32),
                box_lo=g_lo[keep][order].astype(np.int32), box_hi=g_hi[keep][order].astype(np.int32))


def _resident(state, theta, phi, device=0):
    state = np.asarray(state)
    if state.ndim != 3 or len(set(state.shape)) != 1:
        raise ValueError("grain clustering needs a cubic (L, L, L) lattice")
    ctx = _lib.Context(L=state.shape[0], device=device)
    ctx.upload(state=state, theta=theta, phi=np.zeros_like(np.asarray(theta, dtype=np.float64)) if phi is None else phi)
    return ctx


def compute_metrics(state, theta, phi, defects=None, voxel_size=None, W_mask=None, Re_mask=None,
                    C_mask=None, grain_ids=None, rng_seed=None, ctx=None, device=0):
    """metrics.py:41-96.  With `ctx` the lattice resident in that context is clustered (state /
    theta / phi are then only used for `state.size`)."""
    own = ctx is None
    if own:
        ctx = _resident(state, theta, phi, device)
    try:
        g = ctx.grains(0.5)
    finally:
        if own:
            ctx.close()
    n_sites = int(np.prod(ctx.owned_shape)) if state is None else int(np.asarray(state).size)
    m = metrics_from_grains(g, n_sites, defects=defects, voxel_size=voxel_size, rng_seed=rng_seed)
    if m["GrainCount"]:
        for key, mask in (("Frac_W", W_mask), ("Frac_Re", Re_mask), ("Frac_C", C_mask)):
            if mask is not None:
                m[key] = np.count_nonzero(mask) / n_sites if n_sites > 0 else 0.0
    return m


def detect_CET_transition(metrics_dict):
    """metrics.py:103-105"""
    return (metrics_dict["AspectRatio"] < K.CET_AR_THRESHOLD and
            metrics_dict["EquiaxedFraction"] > K.CET_EQ_THRESHOLD)


def compute_CET(state, theta, phi, voxel_size=None, ctx=None):
    """metrics.py:99-101"""
    m = compute_metrics(state, theta, phi, voxel_size=voxel_size, ctx=ctx)
    return "Equiaxed" if detect_CET_transition(m) else "Columnar"


def get_clusters(state, orientation_theta, orientation_phi=None, theta_threshold=0.5, device=0):
    """utils.py:69-84: (clusters, visited).  Clusters come in the reference's order (raster order
    of their first voxel) and `visited` is the reference's label volume; inside a cluster the
    voxels are listed in raster order (the reference lists them in DFS order; its consumers —
    len() and the bounding box — do not depend on it).  orientation_phi=None selects the
    reference's |theta1 - theta2| criterion (utils.py:49-50), which only the unused
    detect_CET_transition of utils.py:117 takes."""
    state = np.asarray(state)
    if state.size == 0:
        return [], np.array([])
    ctx = _resident(state, orientation_theta, orientation_phi, device)
    try:
        g = ctx.grains(theta_threshold, labels=True, theta_only=orientation_phi is None)
    finally:
        ctx.close()
    visited, n = g["labels"], g["n"]
    flat = visited.ravel()
    occ = np.flatnonzero(flat)
    order = np.argsort(flat[occ], kind="stable")
    coords = np.stack(np.unravel_index(occ[order], visited.shape), axis=1)
    bounds = np.searchsorted(flat[occ][order], np.arange(1, n + 2))
    clusters = [[tuple(map(int, v)) for v in coords[bounds[q]:bounds[q + 1]]] for q in range(n)]
    return clusters, visited


def calculate_aspect_ratio(cluster):
    """utils.py:104-111"""
    coords = np.array(cluster)
    dims = coords.max(axis=0) - coords.min(axis=0) + 1
    return float(np.max(dims)) / float(max(np.min(dims), 1))
