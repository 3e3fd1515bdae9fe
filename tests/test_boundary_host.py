"""Host side of the grain-boundary bonds along a growth axis that needs no device: the NumPy reference
(tests/boundaryref.py) on hand-built label volumes along each axis against a brute-force walk over the bonds; the
degree-to-cosine conversion of the edges and the bin order of cetkmc.boundary_group (through a stand-in library that
answers with the reference); metrics.boundary_summary, its empty cases and the truncated nucleation null its docstring
states; the argument checks of the binding before the library is reached; the arguments the drivers refuse before any
Context exists; and the per-case boundaries.csv, the map boundary files, their merge and the boundary ensemble."""
import csv
import ctypes as C
import os

import numpy as np
import pytest

import boundaryref
from cetkmc import _lib, campaign, metrics

L = 6
EDGES = np.cos(np.radians([150.0, 90.0, 45.0, 20.0]))        # ascending cosines: angle bins 0-20-45-90-150-180


def _brute(lab, v, axis, edges):
    """The ABI table by a walk over every site and offset, one bond at a time."""
    n = lab.shape[0]
    m = len(edges)
    out = np.zeros((n, 21 + m + 2), np.int64)
    for s in np.ndindex(lab.shape):
        for r, d in enumerate(_lib.BOUNDARY_OFFSETS):
            t = tuple(x + y for x, y in zip(s, d))
            if not all(0 <= x < n for x in t):
                continue
            z = min(s[axis], t[axis])
            a, b = int(lab[s]), int(lab[t])
            if a >= 0 and b >= 0:
                out[z, 3 * r] += 1
                if a != b:
                    out[z, 3 * r + 1] += 1
                    dc = boundaryref.misorientation_cos(v[s][None], v[t][None])[0]
                    out[z, 21 + int(np.searchsorted(edges, dc, side="right"))] += 1
                    out[z, -1] += int(np.rint(dc * 2.0 ** 32))
            elif (a >= 0) != (b >= 0):
                out[z, 3 * r + 2] += 1
    return out


def _vectors(rng, shape):
    th, ph = rng.uniform(0, np.pi, shape), rng.uniform(0, 2 * np.pi, shape)
    return np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th), np.zeros_like(th)], -1)


def _coord(axis, n=L):
    return np.indices((n,) * 3)[axis]


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_bicrystal_counts_the_crossing_bonds(axis):
    """Two grains split by the plane between coordinates 2 and 3 along the axis; orientations +k and 40 degrees from it."""
    alpha = np.radians(40.0)
    c = _coord(axis)
    lab = np.where(c < 3, 0, 1).astype(np.int32)
    v = np.zeros((L,) * 3 + (4,))
    v[..., 2] = 1.0
    v[c >= 3, 0], v[c >= 3, 2] = np.sin(alpha), np.cos(alpha)
    tab = boundaryref.table(lab, v, axis, EDGES)
    assert np.array_equal(tab, _brute(lab, v, axis, EDGES))
    bonds, hist, f = boundaryref.split(tab)
    crossing = sum(1 for s in np.ndindex(lab.shape) for d in _lib.BOUNDARY_OFFSETS
                   if all(0 <= x + y < L for x, y in zip(s, d)) and (s[axis] < 3) != (s[axis] + d[axis] < 3))
    B = int(bonds[:, :, 1].sum())
    assert B == crossing > 0 and int(bonds[:, :, 2].sum()) == 0
    assert set(np.nonzero(bonds[:, :, 1].sum(1))[0]) <= {1, 2}               # min coordinate of a crossing bond
    assert np.array_equal(hist.sum(0), [0, 1, 0, 0, 0] * np.array(B))         # 40 degrees: the 20-45 bin
    assert int(f.sum()) == B * int(np.rint(np.cos(alpha) * 2.0 ** 32))
    s = metrics.boundary_summary(bonds, hist, f, axis, (20, 45, 90, 150))
    assert s["BoundaryBonds"] == B and s["InterfaceBonds"] == 0 and s["SolidBonds"] == int(bonds[:, :, 0].sum())
    assert s["InterceptAcross"] == "" and s["InterceptAnisotropy"] == ""     # no boundary across the axis
    Sa, Ba = int(bonds[:, 4 + axis, 0].sum()), int(bonds[:, 4 + axis, 1].sum())
    assert Ba == 2 * L * L and s["InterceptAlong"] == 2 * Sa / Ba * metrics.K.VOXEL_SIZE


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_single_grain_has_no_boundary(axis):
    rng = np.random.default_rng(axis)
    lab = np.zeros((L,) * 3, np.int32)
    v = _vectors(rng, (L,) * 3)
    tab = boundaryref.table(lab, v, axis, EDGES)
    assert np.array_equal(tab, _brute(lab, v, axis, EDGES))
    bonds, hist, f = boundaryref.split(tab)
    assert not bonds[:, :, 1:].any() and not hist.any() and not f.any()
    # bonds per offset: both ends inside the lattice, no wrap
    for r, d in enumerate(_lib.BOUNDARY_OFFSETS):
        assert bonds[:, r, 0].sum() == np.prod([L - abs(x) for x in d])
    s = metrics.boundary_summary(bonds, hist, f, axis, (20, 45, 90, 150))
    assert s["BoundaryFraction"] == 0.0 and s["BoundaryBonds"] == 0
    assert s["InterceptAlong"] == s["InterceptAcross"] == s["InterceptAnisotropy"] == s["MeanMisorientationCos"] == ""


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_parity_classes_share_no_bond(axis):
    """One occupied site of each parity of i + j + k, next to each other and in different grains: no bond joins them."""
    lab = np.full((L,) * 3, -1, np.int32)
    lab[2, 2, 2], lab[2, 2, 3] = 5, 9
    v = np.zeros((L,) * 3 + (4,))
    v[..., 2] = 1.0
    tab = boundaryref.table(lab, v, axis, EDGES)
    assert np.array_equal(tab, _brute(lab, v, axis, EDGES))
    bonds, _hist, _f = boundaryref.split(tab)
    assert bonds[:, :, 0].sum() == 0 and bonds[:, :, 1].sum() == 0
    assert bonds[:, :, 2].sum() == 2 * 14                                    # every neighbour of both is empty


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_interface_bonds_of_a_solid_slab(axis):
    c = _coord(axis)
    rng = np.random.default_rng(3 + axis)
    lab = np.where(c < 4, rng.integers(0, 5, (L,) * 3), -1).astype(np.int32)
    v = _vectors(rng, (L,) * 3)
    tab = boundaryref.table(lab, v, axis, EDGES)
    assert np.array_equal(tab, _brute(lab, v, axis, EDGES))
    bonds, _hist, _f = boundaryref.split(tab)
    crossing = sum(1 for s in np.ndindex(lab.shape) for d in _lib.BOUNDARY_OFFSETS
                   if all(0 <= x + y < L for x, y in zip(s, d)) and (s[axis] < 4) != (s[axis] + d[axis] < 4))
    assert bonds[:, :, 2].sum() == crossing and set(np.nonzero(bonds[:, :, 2].sum(1))[0]) == {2, 3}
    assert not bonds[4:].any()


def test_random_labels_against_the_walk():
    rng = np.random.default_rng(11)
    lab = rng.integers(-1, 3, (7, 7, 7)).astype(np.int32)
    v = _vectors(rng, (7, 7, 7))
    v[0, 0, 0, :3] = v[1, 1, 0, :3] = (0.0, 0.0, 1.0)                        # d = 1 exactly: the top bin, F = 2^32
    lab[0, 0, 0], lab[1, 1, 0] = 0, 1
    for axis in range(3):
        tab = boundaryref.table(lab, v, axis, EDGES)
        assert np.array_equal(tab, _brute(lab, v, axis, EDGES))
    assert boundaryref.table(lab, v, 2, EDGES)[0, 21 + 4] >= 1


def test_rounding_half_to_even_and_clamp():
    a = np.array([[1.0, 0.0, 0.0], [1.0, 0.0, 0.0], [1.0 + 2 ** -52, 0.0, 0.0]])
    b = np.array([[2.5 / 2 ** 32, 0.0, 0.0], [3.5 / 2 ** 32, 0.0, 0.0], [1.0 + 2 ** -52, 0.0, 0.0]])
    d = boundaryref.misorientation_cos(a, b)
    assert d[2] == 1.0 and np.rint(np.multiply(d[:2], 2.0 ** 32)).tolist() == [2.0, 4.0]


# -- edge conversion and the binding --------------------------------------------------------------------------------

def test_default_edges():
    assert _lib.BOUNDARY_EDGES_DEG == tuple(range(10, 180, 10)) and _lib.BOUNDARY_SCALE == 2 ** 32
    c = _lib._texture_edges("boundary_group", _lib.BOUNDARY_EDGES_DEG)
    assert c.size == 17 and np.array_equal(c, np.cos(np.radians(np.arange(170, 0, -10, dtype=float))))
    # no edge lies within an ulp of the labelling's threshold of 0.5 rad
    assert np.abs(c - np.cos(0.5)).min() > 1e-3


class _Lib:
    """A stand-in for the library whose cet_boundary_group answers with the reference over given lattices."""

    def __init__(self, lattices, n):
        self.lattices, self.L, self.calls = lattices, n, []

    def cet_boundary_group(self, handles, n, axis, edges, m, out):
        e = np.ctypeslib.as_array(edges, (m,)).copy()
        self.calls.append((n, axis, e))
        o = np.ctypeslib.as_array(out, (n * self.L * (m + 23),)).reshape(n, self.L, m + 23)
        for q in range(n):
            o[q] = boundaryref.table(*self.lattices[q], axis, e)
        return 0


def _contexts(n, Lc):
    made = []
    for _ in range(n):
        c = object.__new__(_lib.Context)
        c._h, c.shape = C.c_void_p(1), (Lc, Lc, Lc)
        made.append(c)
    return made


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_binding_bin_order(monkeypatch, axis):
    rng = np.random.default_rng(axis)
    lats = [(rng.integers(-1, 4, (L,) * 3).astype(np.int32), _vectors(rng, (L,) * 3)) for _ in range(2)]
    fake = _Lib(lats, L)
    monkeypatch.setattr(_lib, "lib", lambda: fake)
    made = _contexts(2, L)
    try:
        deg = (20.0, 45.0, 90.0, 150.0)
        bonds, hist, f = _lib.boundary_group(made, axis, deg)
        assert fake.calls[-1][:2] == (2, axis) and np.array_equal(fake.calls[-1][2], np.cos(np.radians(deg[::-1])))
        assert bonds.shape == (2, L, 7, 3) and hist.shape == (2, L, 5) and f.shape == (2, L)
        assert bonds.dtype == hist.dtype == f.dtype == np.int64
        for q, (lab, v) in enumerate(lats):
            want = boundaryref.split(boundaryref.table(lab, v, axis, np.cos(np.radians(deg[::-1]))))
            assert np.array_equal(bonds[q], want[0]) and np.array_equal(hist[q], want[1]) and np.array_equal(f[q], want[2])
            # ascending angle: bin k holds deg[k - 1] < angle <= deg[k] (no draw lies on an edge)
            ang = []
            for s in np.ndindex(lab.shape):
                for d in _lib.BOUNDARY_OFFSETS:
                    t = tuple(x + y for x, y in zip(s, d))
                    if all(0 <= x < L for x in t) and lab[s] >= 0 and lab[t] >= 0 and lab[s] != lab[t]:
                        ang.append(np.degrees(np.arccos(np.clip(np.dot(v[s][:3], v[t][:3]), -1, 1))))
            assert np.array_equal(hist[q].sum(0), np.histogram(ang, bins=[0.0, *deg, 180.0])[0])
        _b, hist_d, _f = _lib.boundary_group(made[:1], axis)
        assert hist_d.shape == (1, L, 18)
    finally:
        for c in made:
            c._h = C.c_void_p(None)


@pytest.fixture
def no_library(monkeypatch):
    def lib():
        raise AssertionError("the library must not be reached")
    monkeypatch.setattr(_lib, "lib", lib)


def test_binding_checks_before_the_library(no_library):
    made = _contexts(2, 8)
    try:
        for axis in (3, -1, None, True, 1.0, "2"):
            with pytest.raises(ValueError, match="boundary_group: axis"):
                _lib.boundary_group(made, axis)
        for edges in ([], list(range(1, 33)), [30, 15], [15, 15], [15, np.nan], [15, np.inf], [0, 15], [15, 180],
                      [-5, 30], [30, 200], "ab", [[15, 30]]):
            with pytest.raises(ValueError, match="boundary_group: edges_deg"):
                _lib.boundary_group(made, 2, edges)
        with pytest.raises(ValueError, match="do not ascend"):
            _lib.boundary_group(made, 2, [1e-9, 2e-9])
        with pytest.raises(TypeError):
            _lib.boundary_group([made[0], object()], 2)
    finally:
        for c in made:
            c._h = C.c_void_p(None)
    assert "cet_boundary_group" in _lib.SIGNATURES
    import cetkmc
    assert cetkmc.boundary_group is _lib.boundary_group


# -- boundary_summary ------------------------------------------------------------------------------------------------

def test_boundary_summary_definitions():
    deg = (30.0, 90.0)
    bonds = np.zeros((3, 7, 3), np.int64)
    bonds[0, 4] = (10, 2, 1)         # axis 0 offset
    bonds[1, 5] = (7, 3, 0)          # axis 1 offset
    bonds[2, 6] = (9, 1, 4)          # axis 2 offset
    bonds[2, 0] = (5, 4, 2)
    hist = np.array([[0, 1, 1], [1, 2, 0], [0, 3, 2]], np.int64)
    f = np.array([3 * 2 ** 31, -2 ** 32, 7], np.int64)
    s = metrics.boundary_summary(bonds, hist, f, 2, deg, voxel_size=2.0)
    assert list(s) == list(metrics.BOUNDARY_COLUMNS)
    assert (s["SolidBonds"], s["BoundaryBonds"], s["InterfaceBonds"]) == (31, 10, 7)
    assert s["BoundaryFraction"] == 10 / 31
    assert s["InterceptAlong"] == 2 * 9 / 1 * 2.0 and s["InterceptAcross"] == 2 * 17 / 5 * 2.0
    assert s["InterceptAnisotropy"] == 9 * 5 / (1 * 17)
    assert s["MeanMisorientationCos"] == (3 * 2 ** 31 - 2 ** 32 + 7) / (10 * 2 ** 32)
    s0 = metrics.boundary_summary(bonds, hist, f, 0, deg)
    assert s0["InterceptAlong"] == 2 * 10 / 2 * metrics.K.VOXEL_SIZE and s0["InterceptAnisotropy"] == 10 * 4 / (2 * 16)
    empty = metrics.boundary_summary(np.zeros((4, 7, 3), np.int64), np.zeros((4, 3), np.int64), np.zeros(4, np.int64),
                                     1, deg)
    assert empty == {"SolidBonds": 0, "BoundaryBonds": 0, "InterfaceBonds": 0, "BoundaryFraction": "",
                     "InterceptAlong": "", "InterceptAcross": "", "InterceptAnisotropy": "", "MeanMisorientationCos": ""}
    with pytest.raises(ValueError, match="boundary_summary"):
        metrics.boundary_summary(bonds[:, :6], hist, f, 2, deg)
    with pytest.raises(ValueError, match="boundary_summary"):
        metrics.boundary_summary(bonds, hist[:, :2], f, 2, deg)
    with pytest.raises(ValueError, match="boundary_summary: axis"):
        metrics.boundary_summary(bonds, hist, f, 3, deg)
    with pytest.raises(ValueError, match="histogram"):
        metrics.boundary_summary(bonds, hist * 2, f, 2, deg)


def _null_parts(x, n=1000):
    """P(d <= x) and E[d; d <= x] for d = v . v' of two independent nucleation draws (theta ~ U(0, pi), phi ~ U(0, 2 pi)):
    d = A cos(dphi) + B with A = sin t sin t', B = cos t cos t' and dphi uniform, so the phi integral is closed
    (P = 1 - arccos(u) / pi, E[cos dphi; cos dphi <= u] = -sqrt(1 - u^2) / pi at u = (x - B) / A) and theta, theta' take
    n-point Gauss-Legendre quadrature."""
    g, w = np.polynomial.legendre.leggauss(n)
    t, w = (g + 1) * np.pi / 2, w / 2
    A, B = np.outer(np.sin(t), np.sin(t)), np.outer(np.cos(t), np.cos(t))
    W = np.outer(w, w)
    u = np.clip((x - B) / A, -1, 1)
    return (W * (1 - np.arccos(u) / np.pi)).sum(), (W * (B * (1 - np.arccos(u) / np.pi) - A * np.sqrt(1 - u * u) / np.pi)).sum()


def test_truncated_null_stated_in_the_docstring():
    thr = np.cos(0.5)
    p_all, m_all = _null_parts(1.0)
    assert abs(p_all - 1.0) < 1e-9 and abs(m_all) < 1e-9                      # E[v] = 0: mean cosine 0
    p, m = _null_parts(thr)
    assert round(100 * p, 2) == 91.76 and round(m / p, 4) == -0.0847
    deg = _lib.BOUNDARY_EDGES_DEG
    lo, hi = (0,) + deg, deg + (180,)
    shares = []
    for a0, a1 in zip(lo, hi):
        top = p if a0 == 0 else _null_parts(min(np.cos(np.radians(a0)), thr))[0]
        bot = 0.0 if a1 == 180 else _null_parts(np.cos(np.radians(a1)))[0]
        shares.append(max(top - bot, 0.0) / p if np.cos(np.radians(a1)) < thr else 0.0)
    stated = (0, 0, 0.0072, 0.0593, 0.0679, 0.0746, 0.0794, 0.0825, 0.0841, 0.0841, 0.0825, 0.0794, 0.0746, 0.0679,
              0.0593, 0.0483, 0.0342, 0.0145)
    assert abs(sum(shares) - 1) < 1e-9 and all(abs(x - y) < 5e-5 for x, y in zip(shares, stated))
    assert all(("%.4f" % x) in metrics.boundary_summary.__doc__ for x in stated if x)
    assert "91.76 %" in metrics.boundary_summary.__doc__ and "-0.0847" in metrics.boundary_summary.__doc__


# -- driver refusals: before any Context exists ---------------------------------------------------------------------

@pytest.fixture
def no_context(monkeypatch, tmp_path):
    monkeypatch.chdir(tmp_path)

    def ctx(*a, **kw):
        raise AssertionError("a Context was created")
    monkeypatch.setattr(_lib, "Context", ctx)


@pytest.mark.parametrize("bad", [dict(world=2, rank=0), dict(checkpoint_every=2), dict(resume_from="ck"),
                                 dict(boundary_axis=3), dict(boundary_axis=-1), dict(boundary_axis=True),
                                 dict(boundary_axis=2.0)])
def test_run_cet_sublattice_refusals(no_context, bad):
    kw = dict(boundary_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="boundary_axis"):
        campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)


@pytest.mark.parametrize("driver", ["gr", "melt"])
@pytest.mark.parametrize("bad", [dict(checkpoint_every=2), dict(resume_from="ck"), dict(boundary_axis=5)])
def test_map_driver_refusals(no_context, monkeypatch, driver, bad):
    monkeypatch.setattr(campaign, "run_cet_sublattice", lambda **kw: pytest.fail("a lattice ran"))
    monkeypatch.setattr(campaign, "_run_cases_grouped", lambda *a, **kw: pytest.fail("a group ran"))
    kw = dict(boundary_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="boundary_axis"):
        if driver == "gr":
            campaign.run_gr_sweep([2700.0], [1e13], L=8, n_sweeps=5, **kw)
        else:
            campaign.run_melt_pool_map([100.0], [1.0], L=8, n_sweeps=5, **kw)


def test_grouped_driver_refuses_a_bad_axis(no_context):
    with pytest.raises(ValueError, match="boundary_axis"):
        campaign._run_cases_grouped([("x", 2700.0, 1e13)], L=8, n_sweeps=5, impurity_c=0.0, n_seeds=2,
                                    defect_fraction=0.0, device=0, boundary_axis=4)


def test_existing_axis_messages_unchanged(no_context):
    for kw, msg in ((dict(profile_axis=4), "run_cet_sublattice: profile_axis must be None, 0, 1 or 2, got 4"),
                    (dict(shape_axis=1, resume_from="ck"),
                     "run_cet_sublattice: shape_axis does not take checkpoint_every or resume_from"),
                    (dict(front_axis=1, world=2), "run_cet_sublattice: front_axis needs a whole lattice on one GPU (world = 1)"),
                    (dict(texture_axis=4), "run_cet_sublattice: texture_axis must be None, 0, 1 or 2, got 4"),
                    (dict(boundary_axis=4), "run_cet_sublattice: boundary_axis must be None, 0, 1 or 2, got 4"),
                    (dict(texture_axis=1, boundary_axis=4),
                     "run_cet_sublattice: boundary_axis must be None, 0, 1 or 2, got 4")):
        with pytest.raises(ValueError) as ei:
            campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)
        assert str(ei.value) == msg


# -- boundaries CSV, map boundary files, merge and ensemble ---------------------------------------------------------

def _read(path):
    with open(path) as fh:
        return list(csv.DictReader(fh))


def _record(rng, step, Lc=8, empty=False):
    bonds = np.zeros((Lc, 7, 3), np.int64)
    hist = np.zeros((Lc, 18), np.int64)
    f = np.zeros(Lc, np.int64)
    if not empty:
        bonds[..., 0] = rng.integers(5, 60, (Lc, 7))
        bonds[..., 1] = rng.integers(0, 5, (Lc, 7))
        bonds[..., 2] = rng.integers(0, 9, (Lc, 7))
        for z in range(Lc):
            b = int(bonds[z, :, 1].sum())
            hist[z] = np.bincount(rng.integers(2, 18, b), minlength=18)
            f[z] = int(rng.integers(-b, b + 1)) * 2 ** 31
    return step, bonds, hist, f


def test_boundary_csv_round_trip(tmp_path):
    rng = np.random.default_rng(2)
    recs = [_record(rng, 99), _record(rng, 199), _record(rng, 201, empty=True)]
    campaign._write_boundary_csv(recs, str(tmp_path))
    rows = _read(tmp_path / "boundaries.csv")
    head = list(rows[0].keys())
    assert head[:5] == ["Step", "Plane", "Solid0", "Boundary0", "Interface0"] and head[22] == "Interface6"
    assert head[23:25] == ["0-10", "10-20"] and head[-2:] == ["170-180", "SumCos"] and len(head) == 2 + 21 + 18 + 1
    assert len(rows) == 3 * 8 and [int(r["Plane"]) for r in rows[:8]] == list(range(8))
    assert [int(r["Boundary3"]) for r in rows[:8]] == recs[0][1][:, 3, 1].tolist()
    assert all(v.lstrip("-").isdigit() for r in rows for v in r.values())
    edges, back = campaign.read_boundary_csv(str(tmp_path / "boundaries.csv"))
    assert edges == tuple(float(x) for x in _lib.BOUNDARY_EDGES_DEG) and len(back) == 3
    for (step, b, h, f), (bs, bb, bh, bf) in zip(recs, back):
        assert bs == step and np.array_equal(bb, b) and np.array_equal(bh, h) and np.array_equal(bf, f)
        assert bb.dtype == bh.dtype == bf.dtype == np.int64
    odd = (1e-5, 12.5, 0.1 + 0.2 + 20, 170.0)
    campaign._write_boundary_csv([(3, np.ones((2, 7, 3), np.int64), np.ones((2, 5), np.int64), np.zeros(2, np.int64))],
                                 str(tmp_path), odd)
    assert campaign.read_boundary_csv(str(tmp_path / "boundaries.csv"))[0] == odd
    campaign._write_boundary_csv([], str(tmp_path / "none"))
    assert not os.path.exists(tmp_path / "none" / "boundaries.csv")


def _synthetic_map(tmp_path, monkeypatch, n_case, n_rep, seed=3, empty=()):
    monkeypatch.chdir(tmp_path)
    rng = np.random.default_rng(seed)
    lats = campaign._map_lattices([f"m/T{q}" for q in range(n_case)], n_rep)
    for q, r, p in lats:
        os.makedirs(f"outputs/{p}", exist_ok=True)
        campaign._write_boundary_csv([_record(rng, 5), _record(rng, 9), _record(rng, 13, empty=(q, r) in empty)],
                                     f"outputs/{p}")
    return lats


def _case_row(q):
    return {"T_sub": 2600.0 + q, "NU_DEP": 1e12 * (q + 1), "G": 1.0e6 * (q + 1), "R": 2.0, "G_over_R": 0.5}


def test_map_boundary_rows_merge_and_ensemble(tmp_path, monkeypatch):
    n_case, n_rep = 3, 4
    lats = _synthetic_map(tmp_path, monkeypatch, n_case, n_rep, empty={(1, 2)})
    axes = ("T_sub", "NU_DEP")
    rows = campaign._map_boundary_rows(lats, list(range(len(lats))), _case_row, axes, 2)
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP"] + list(metrics.BOUNDARY_COLUMNS)
    for (q, r, p), row in zip(lats, rows):
        edges, recs = campaign.read_boundary_csv(f"outputs/{p}/boundaries.csv")
        assert (row["case"], row["replica"], row["T_sub"]) == (q, r, 2600.0 + q)
        assert {k: row[k] for k in metrics.BOUNDARY_COLUMNS} == metrics.boundary_summary(*recs[-1][1:], 2, edges)
    assert rows[1 * n_rep + 2]["InterceptAlong"] == "" and rows[0]["InterceptAlong"] != ""
    mine = [[l for l in range(len(lats)) if l % 2 == k] for k in range(2)]
    for k in range(2):
        campaign._write_rows(campaign._map_boundary_rows(lats, mine[k], _case_row, axes, 2),
                             f"outputs/m/cet_map_boundary_rank{k}.csv")
        campaign._write_rows([{"case": lats[l][0], "replica": lats[l][1], **_case_row(lats[l][0]),
                               **{c: 1.0 for c in campaign.ENSEMBLE_COLUMNS}, "CET_Class": "Equiaxed",
                               "CET_Detected": True} for l in mine[k]], f"outputs/m/cet_map_replicas_rank{k}.csv")
    campaign.merge_cet_map("m")
    merged = _read("outputs/m/cet_map_boundary.csv")
    assert [(int(r["case"]), int(r["replica"])) for r in merged] == [(q, r) for q, r, _ in lats]
    assert [r["InterceptAnisotropy"] for r in merged] == [repr(r["InterceptAnisotropy"]) if r["InterceptAnisotropy"] != ""
                                                          else "" for r in rows]
    ens = _read("outputs/m/cet_map_boundary_ensemble.csv")
    assert list(ens[0].keys()) == ["case", "T_sub", "NU_DEP", "replicas"] + [
        f"{c}_{s}" for c in campaign.BOUNDARY_ENSEMBLE for s in ("mean", "se")]
    assert campaign.BOUNDARY_ENSEMBLE == ("InterceptAlong", "InterceptAcross", "InterceptAnisotropy", "BoundaryFraction")
    for q, e in enumerate(ens):
        assert int(e["case"]) == q and int(e["replicas"]) == n_rep
        for col in campaign.BOUNDARY_ENSEMBLE:
            v = np.array([r[col] for r in rows[q * n_rep:(q + 1) * n_rep] if r[col] != ""], np.float64)
            assert v.size == (n_rep - 1 if q == 1 else n_rep)
            assert float(e[f"{col}_mean"]) == pytest.approx(np.mean(v), rel=1e-15)
            assert float(e[f"{col}_se"]) == pytest.approx(np.std(v, ddof=1) / np.sqrt(v.size), rel=1e-12)
    assert not os.path.exists("outputs/m/cet_map_texture.csv") and not os.path.exists("outputs/m/cet_map_front.csv")


def test_merge_without_replicas_writes_no_boundary_ensemble(tmp_path, monkeypatch):
    lats = _synthetic_map(tmp_path, monkeypatch, 2, 1)
    campaign._write_rows(campaign._map_boundary_rows(lats, [1, 0], _case_row, ("T_sub", "NU_DEP"), 1),
                         "outputs/m/melt_pool_map_boundary_rank0.csv")
    campaign.merge_melt_pool_map("m")
    assert [int(r["case"]) for r in _read("outputs/m/melt_pool_map_boundary.csv")] == [0, 1]
    assert not os.path.exists("outputs/m/melt_pool_map_boundary_ensemble.csv")
