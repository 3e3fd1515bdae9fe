"""Host side of the texture along a growth axis that needs no device: the NumPy reference (tests/textureref.py) on
hand-built lattices along each axis; the degree-to-cosine conversion of the edges and the bin order of
cetkmc.texture_group (through a stand-in library that answers with the reference); metrics.texture_summary and the
nucleation nulls it documents; the argument checks of the binding before the library is reached; the arguments the
drivers refuse before any Context exists; and the per-case texture.csv, the map texture files, their merge and the
texture ensemble."""
import csv
import ctypes as C
import os

import numpy as np
import pytest

import textureref
from cetkmc import _lib, campaign, metrics

L = 6
EDGES = np.array([-0.5, 0.0, 0.5])


def _lattice(axis, c_of_plane, occupied=None):
    """A lattice whose every site of plane z along `axis` has v[axis] = c_of_plane[z] (the other components 0.25 and
    -0.5, so that a wrong component shows), occupied where `occupied` (default everywhere)."""
    v = np.zeros((L, L, L, 4))
    for k in range(3):
        v[..., k] = (0.25, -0.5, 0.125)[k]
    sh = [1, 1, 1]
    sh[axis] = L
    v[..., axis] = np.asarray(c_of_plane, np.float64).reshape(sh)
    st = np.ones((L,) * 3, np.int64) if occupied is None else occupied.astype(np.int64)
    return st, v


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_reference_edges_and_extremes(axis):
    c = np.array([-1.0, -0.5, 0.0, 0.25, 0.5, 1.0])               # on the edges, between them and at +-1
    st, v = _lattice(axis, c)
    tab = textureref.table(st, v, axis, EDGES)
    assert tab.shape == (L, 6) and tab.dtype == np.int64
    want_bin = [0, 1, 2, 2, 3, 3]                                  # b = #{i : e_i <= c}
    for z in range(L):
        row = np.zeros(4, np.int64)
        row[want_bin[z]] = L * L
        assert np.array_equal(tab[z, :4], row), (axis, z)
        assert tab[z, 4] == L * L * int(c[z] * 2 ** 32) and tab[z, 5] == L * L * int(c[z] * c[z] * 2 ** 32)


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_reference_empty_full_and_a_plane_without_solid(axis):
    st, v = _lattice(axis, np.linspace(-0.9, 0.9, L))
    assert not textureref.table(np.zeros_like(st), v, axis, EDGES).any()
    full = textureref.table(st, v, axis, EDGES)
    assert (full[:, :4].sum(1) == L * L).all()
    occ = np.ones((L,) * 3, bool)
    idx = [slice(None)] * 3
    idx[axis] = 2
    occ[tuple(idx)] = False                                        # plane 2 along the axis: no solid
    occ[(0, 0, 0)] = False
    packed = occ.astype(np.uint8) * 2 | np.uint8(0x10)             # state 2 with the defect bit: the low nibble counts
    tab = textureref.table(packed, v, axis, EDGES)
    assert not tab[2].any() and tab[0, :4].sum() == L * L - 1 and (tab[1:, :4].sum(1)[np.arange(1, L) != 2] == L * L).all()
    defect_only = np.full((L,) * 3, 0x10, np.uint8)                # the mask bit alone is an empty site
    assert not textureref.table(defect_only, v, axis, EDGES).any()


def test_reference_rounding_half_to_even():
    st = np.zeros((L,) * 3, np.int64)
    v = np.zeros((L, L, L, 4))
    st[0, :2, 0] = 1                                               # two sites of plane 0 along axis 2
    v[0, 0, 0, 2] = 2.5 / 2 ** 32                                  # c 2^32 = 2.5 -> 2
    v[0, 1, 0, 2] = 3.5 / 2 ** 32                                  # -> 4
    tab = textureref.table(st, v, 2, EDGES)
    assert tab[0, 4] == 6 and tab[0, 5] == 0


def test_uniform_theta_grid_gives_the_flat_axis2_histogram():
    n = 180 * 48
    theta = (np.arange(n) + 0.5) * np.pi / n                       # midpoints of n equal slices of (0, pi)
    phi = np.linspace(0.0, 2 * np.pi, n, endpoint=False)
    Lg = round(n ** (1 / 3)) + 1
    st = np.zeros(Lg ** 3, np.int64)
    v = np.zeros((Lg ** 3, 4))
    st[:n] = 1
    v[:n, 0], v[:n, 1], v[:n, 2] = np.sin(theta) * np.cos(phi), np.sin(theta) * np.sin(phi), np.cos(theta)
    st, v = st.reshape((Lg,) * 3), v.reshape((Lg,) * 3 + (4,))
    c = _lib._texture_edges("t", _lib.TEXTURE_EDGES_DEG)
    hist, f1, f2 = textureref.split(textureref.table(st, v, 2, c))
    total = hist.sum(0)
    assert total.shape == (12,) and (total == n // 12).all()
    s = metrics.texture_summary(hist, f1, f2, _lib.TEXTURE_EDGES_DEG)
    assert s["TexturedSolid"] == n and abs(s["MeanCos"]) < 1e-12 and s["AlignedFraction"] == 30 / 180
    assert s["Hermans"] == pytest.approx(0.25, abs=1e-6)


# -- edge conversion and the binding --------------------------------------------------------------------------------

def test_degree_to_cosine_conversion():
    assert _lib.TEXTURE_EDGES_DEG == tuple(range(15, 180, 15)) and _lib.TEXTURE_SCALE == 2 ** 32
    c = _lib._texture_edges("t", _lib.TEXTURE_EDGES_DEG)
    assert np.array_equal(c, np.cos(np.radians(np.array(_lib.TEXTURE_EDGES_DEG, float)[::-1])))
    assert (np.diff(c) > 0).all() and c.flags.c_contiguous and c.dtype == np.float64
    assert np.array_equal(_lib._texture_edges("t", [90]), np.cos(np.radians([90.0])))
    assert _lib._texture_edges("t", np.arange(1, 32) * 5.0).size == 31


class _Lib:
    """A stand-in for the library whose cet_texture_group answers with the reference over given lattices."""

    def __init__(self, lattices):
        self.lattices, self.calls = lattices, []

    def cet_texture_group(self, handles, n, axis, edges, m, out):
        e = np.ctypeslib.as_array(edges, (m,)).copy()
        self.calls.append((n, axis, e))
        o = np.ctypeslib.as_array(out, (n * self.L * (m + 3),)).reshape(n, self.L, m + 3)
        for q in range(n):
            o[q] = textureref.table(*self.lattices[q], axis, e)
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
    lats = []
    for q in range(2):
        th, ph = rng.uniform(0, np.pi, (L,) * 3), rng.uniform(0, 2 * np.pi, (L,) * 3)
        v = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th), np.zeros_like(th)], -1)
        lats.append((rng.integers(0, 3, (L,) * 3), v))
    fake = _Lib(lats)
    fake.L = L
    monkeypatch.setattr(_lib, "lib", lambda: fake)
    made = _contexts(2, L)
    try:
        deg = (20.0, 45.0, 90.0, 150.0)
        hist, f1, f2 = _lib.texture_group(made, axis, deg)
        assert fake.calls[-1][:2] == (2, axis) and np.array_equal(fake.calls[-1][2], np.cos(np.radians(deg[::-1])))
        assert hist.shape == (2, L, 5) and f1.shape == f2.shape == (2, L) and hist.dtype == f1.dtype == np.int64
        for q, (st, v) in enumerate(lats):
            moved = np.moveaxis(v[..., axis], axis, 0)
            occ = np.moveaxis(st != 0, axis, 0)
            ang = np.degrees(np.arccos(moved))
            for z in range(L):
                a = ang[z][occ[z]]
                want = np.histogram(a, bins=[0.0, *deg, 180.0])[0]   # no angle of this draw lies on an edge
                assert np.array_equal(hist[q, z], want), (q, z)
            want_h, want_f1, want_f2 = textureref.split(textureref.table(st, v, axis, np.cos(np.radians(deg[::-1]))))
            assert np.array_equal(hist[q], want_h) and np.array_equal(f1[q], want_f1) and np.array_equal(f2[q], want_f2)
        hist_d, _, _ = _lib.texture_group(made[:1], axis)
        assert hist_d.shape == (1, L, 12)
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
            with pytest.raises(ValueError, match="axis"):
                _lib.texture_group(made, axis)
        for edges in ([], list(range(1, 33)), [30, 15], [15, 15], [15, np.nan], [15, np.inf], [0, 15], [15, 180],
                      [-5, 30], [30, 200], "ab", [[15, 30]]):
            with pytest.raises(ValueError, match="edges_deg"):
                _lib.texture_group(made, 2, edges)
        with pytest.raises(ValueError, match="do not ascend"):     # 1e-9 degrees apart: the same cosine
            _lib.texture_group(made, 2, [1e-9, 2e-9])
        with pytest.raises(TypeError):
            _lib.texture_group([made[0], object()], 2)
    finally:
        for c in made:
            c._h = C.c_void_p(None)
    assert "cet_texture_group" in _lib.SIGNATURES
    import cetkmc
    assert cetkmc.texture_group is _lib.texture_group


# -- texture_summary ---------------------------------------------------------------------------------------------

def test_texture_summary_definitions():
    deg = (30.0, 90.0)
    hist = np.array([[3, 1, 0], [1, 0, 4], [0, 0, 0]], np.int64)
    f1 = np.array([5 * 2 ** 32 // 2, -3 * 2 ** 32, 0], np.int64)
    f2 = np.array([3 * 2 ** 32, 2 * 2 ** 32 + 7, 0], np.int64)
    s = metrics.texture_summary(hist, f1, f2, deg)
    assert list(s) == list(metrics.TEXTURE_COLUMNS)
    assert s["TexturedSolid"] == 9 and s["MeanCos"] == (2.5 - 3.0) / 9
    assert s["Hermans"] == (3 * (5 * 2 ** 32 + 7) - 9 * 2 ** 32) / (2 * 9 * 2 ** 32)
    assert s["AlignedFraction"] == 4 / 9
    assert metrics.texture_summary(hist, f1, f2, deg, aligned_deg=90)["AlignedFraction"] == 5 / 9
    empty = metrics.texture_summary(np.zeros((4, 3), np.int64), np.zeros(4, np.int64), np.zeros(4, np.int64), deg)
    assert empty == {"TexturedSolid": 0, "MeanCos": "", "Hermans": "", "AlignedFraction": ""}
    with pytest.raises(ValueError, match="aligned_deg"):
        metrics.texture_summary(hist, f1, f2, deg, aligned_deg=45)
    with pytest.raises(ValueError, match="texture_summary"):
        metrics.texture_summary(hist[:, :2], f1, f2, deg)
    with pytest.raises(ValueError, match="texture_summary"):
        metrics.texture_summary(hist, f1[:2], f2, deg)


def test_texture_summary_extremes():
    deg = _lib.TEXTURE_EDGES_DEG
    n = np.array([10], np.int64)
    up = metrics.texture_summary(np.array([[10] + [0] * 11]), n * 2 ** 32, n * 2 ** 32, deg)
    assert (up["MeanCos"], up["Hermans"], up["AlignedFraction"]) == (1.0, 1.0, 1.0)
    flat = metrics.texture_summary(np.array([[0] * 6 + [10] + [0] * 5]), np.zeros(1, np.int64), np.zeros(1, np.int64), deg)
    assert (flat["MeanCos"], flat["Hermans"], flat["AlignedFraction"]) == (0.0, -0.5, 0.0)


@pytest.mark.parametrize("axis,hermans", [(2, 0.25), (0, -0.125), (1, -0.125)])
def test_texture_summary_nucleation_nulls(axis, hermans):
    """theta ~ U(0, pi), phi ~ U(0, 2 pi) as the nuclei draw them: 64^3 sites, tolerances 5 standard errors (MeanCos
    <= 0.71 / 512, Hermans <= 0.36 / 512, AlignedFraction sqrt(1/6 * 5/6) / 512 per standard error)."""
    rng = np.random.default_rng(17 + axis)
    Lc = 64
    th, ph = rng.uniform(0, np.pi, (Lc,) * 3), rng.uniform(0, 2 * np.pi, (Lc,) * 3)
    v = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th), np.zeros_like(th)], -1)
    c = _lib._texture_edges("t", _lib.TEXTURE_EDGES_DEG)
    hist, f1, f2 = textureref.split(textureref.table(np.ones((Lc,) * 3, np.int64), v, axis, c))
    s = metrics.texture_summary(hist, f1, f2, _lib.TEXTURE_EDGES_DEG)
    assert s["TexturedSolid"] == Lc ** 3
    assert abs(s["MeanCos"]) < 5 * 0.71 / 512 and abs(s["Hermans"] - hermans) < 5 * 0.36 / 512
    if axis == 2:
        assert abs(s["AlignedFraction"] - 30 / 180) < 5 * np.sqrt(5 / 36) / 512
        per_bin = hist.sum(0) / Lc ** 3
        assert np.all(np.abs(per_bin - 15 / 180) < 5 * np.sqrt(1 / 12 * 11 / 12) / 512)


# -- driver refusals: before any Context exists ---------------------------------------------------------------------

@pytest.fixture
def no_context(monkeypatch, tmp_path):
    monkeypatch.chdir(tmp_path)

    def ctx(*a, **kw):
        raise AssertionError("a Context was created")
    monkeypatch.setattr(_lib, "Context", ctx)


@pytest.mark.parametrize("bad", [dict(world=2, rank=0), dict(checkpoint_every=2), dict(resume_from="ck"),
                                 dict(texture_axis=3), dict(texture_axis=-1), dict(texture_axis=True),
                                 dict(texture_axis=2.0)])
def test_run_cet_sublattice_refusals(no_context, bad):
    kw = dict(texture_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="texture_axis"):
        campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)


@pytest.mark.parametrize("driver", ["gr", "melt"])
@pytest.mark.parametrize("bad", [dict(checkpoint_every=2), dict(resume_from="ck"), dict(texture_axis=5)])
def test_map_driver_refusals(no_context, monkeypatch, driver, bad):
    monkeypatch.setattr(campaign, "run_cet_sublattice", lambda **kw: pytest.fail("a lattice ran"))
    monkeypatch.setattr(campaign, "_run_cases_grouped", lambda *a, **kw: pytest.fail("a group ran"))
    kw = dict(texture_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="texture_axis"):
        if driver == "gr":
            campaign.run_gr_sweep([2700.0], [1e13], L=8, n_sweeps=5, **kw)
        else:
            campaign.run_melt_pool_map([100.0], [1.0], L=8, n_sweeps=5, **kw)


def test_grouped_driver_refuses_a_bad_axis(no_context):
    with pytest.raises(ValueError, match="texture_axis"):
        campaign._run_cases_grouped([("x", 2700.0, 1e13)], L=8, n_sweeps=5, impurity_c=0.0, n_seeds=2,
                                    defect_fraction=0.0, device=0, texture_axis=4)


def test_existing_axis_messages_unchanged(no_context):
    for kw, msg in ((dict(profile_axis=4), "run_cet_sublattice: profile_axis must be None, 0, 1 or 2, got 4"),
                    (dict(shape_axis=1, resume_from="ck"),
                     "run_cet_sublattice: shape_axis does not take checkpoint_every or resume_from"),
                    (dict(front_axis=1, world=2), "run_cet_sublattice: front_axis needs a whole lattice on one GPU (world = 1)"),
                    (dict(texture_axis=4), "run_cet_sublattice: texture_axis must be None, 0, 1 or 2, got 4")):
        with pytest.raises(ValueError) as ei:
            campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)
        assert str(ei.value) == msg


# -- texture CSV, map texture files, merge and ensemble ------------------------------------------------------------

def _read(path):
    with open(path) as fh:
        return list(csv.DictReader(fh))


def _record(rng, step, Lc=8, empty=False):
    hist = np.zeros((Lc, 12), np.int64) if empty else rng.integers(0, 40, (Lc, 12))
    n = hist.sum(1)
    f1 = np.array([int(rng.integers(-k, k + 1)) * 2 ** 31 if k else 0 for k in n], np.int64)
    f2 = np.array([int(rng.integers(0, k + 1)) * 2 ** 32 - (k > 0) for k in n], np.int64)
    return step, hist, f1, f2


def test_texture_csv_round_trip(tmp_path):
    rng = np.random.default_rng(2)
    recs = [_record(rng, 99), _record(rng, 199), _record(rng, 201, empty=True)]
    campaign._write_texture_csv(recs, str(tmp_path))
    rows = _read(tmp_path / "texture.csv")
    assert list(rows[0].keys()) == ["Step", "Plane", "Solid", "SumCos", "SumCos2", "0-15", "15-30", "30-45", "45-60",
                                    "60-75", "75-90", "90-105", "105-120", "120-135", "135-150", "150-165", "165-180"]
    assert len(rows) == 3 * 8 and [int(r["Plane"]) for r in rows[:8]] == list(range(8))
    assert [int(r["Solid"]) for r in rows[:8]] == recs[0][1].sum(1).tolist()
    edges, back = campaign.read_texture_csv(str(tmp_path / "texture.csv"))
    assert edges == tuple(float(x) for x in _lib.TEXTURE_EDGES_DEG) and len(back) == 3
    for (step, h, f1, f2), (bs, bh, bf1, bf2) in zip(recs, back):
        assert bs == step and np.array_equal(bh, h) and np.array_equal(bf1, f1) and np.array_equal(bf2, f2)
        assert bh.dtype == np.int64
    odd = (1e-5, 12.5, 0.1 + 0.2 + 20, 170.0)                        # names keep every edge exactly
    campaign._write_texture_csv([(3, np.ones((2, 5), np.int64), np.zeros(2, np.int64), np.zeros(2, np.int64))],
                                str(tmp_path), odd)
    assert campaign.read_texture_csv(str(tmp_path / "texture.csv"))[0] == odd
    campaign._write_texture_csv([], str(tmp_path / "none"))         # no rows: no file
    assert not os.path.exists(tmp_path / "none" / "texture.csv")


def _synthetic_map(tmp_path, monkeypatch, n_case, n_rep, seed=3, empty=()):
    monkeypatch.chdir(tmp_path)
    rng = np.random.default_rng(seed)
    lats = campaign._map_lattices([f"m/T{q}" for q in range(n_case)], n_rep)
    for q, r, p in lats:
        os.makedirs(f"outputs/{p}", exist_ok=True)
        campaign._write_texture_csv([_record(rng, 5), _record(rng, 9), _record(rng, 13, empty=(q, r) in empty)],
                                    f"outputs/{p}")
    return lats


def _case_row(q):
    return {"T_sub": 2600.0 + q, "NU_DEP": 1e12 * (q + 1), "G": 1.0e6 * (q + 1), "R": 2.0, "G_over_R": 0.5}


def test_map_texture_rows_merge_and_ensemble(tmp_path, monkeypatch):
    n_case, n_rep = 3, 4
    lats = _synthetic_map(tmp_path, monkeypatch, n_case, n_rep, empty={(1, 2)})
    axes = ("T_sub", "NU_DEP")
    rows = campaign._map_texture_rows(lats, list(range(len(lats))), _case_row, axes)
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP"] + list(metrics.TEXTURE_COLUMNS)
    for (q, r, p), row in zip(lats, rows):
        edges, recs = campaign.read_texture_csv(f"outputs/{p}/texture.csv")
        assert (row["case"], row["replica"], row["T_sub"]) == (q, r, 2600.0 + q)
        assert {k: row[k] for k in metrics.TEXTURE_COLUMNS} == metrics.texture_summary(*recs[-1][1:], edges)
    assert rows[1 * n_rep + 2]["Hermans"] == "" and rows[0]["Hermans"] != ""
    mine = [[l for l in range(len(lats)) if l % 2 == k] for k in range(2)]
    for k in range(2):
        campaign._write_rows(campaign._map_texture_rows(lats, mine[k], _case_row, axes),
                             f"outputs/m/cet_map_texture_rank{k}.csv")
        campaign._write_rows([{"case": lats[l][0], "replica": lats[l][1], **_case_row(lats[l][0]),
                               **{c: 1.0 for c in campaign.ENSEMBLE_COLUMNS}, "CET_Class": "Equiaxed",
                               "CET_Detected": True} for l in mine[k]], f"outputs/m/cet_map_replicas_rank{k}.csv")
    campaign.merge_cet_map("m")
    merged = _read("outputs/m/cet_map_texture.csv")
    assert [(int(r["case"]), int(r["replica"])) for r in merged] == [(q, r) for q, r, _ in lats]
    assert [r["Hermans"] for r in merged] == [repr(r["Hermans"]) if r["Hermans"] != "" else "" for r in rows]
    ens = _read("outputs/m/cet_map_texture_ensemble.csv")
    assert list(ens[0].keys()) == ["case", "T_sub", "NU_DEP", "replicas"] + [
        f"{c}_{s}" for c in campaign.TEXTURE_ENSEMBLE for s in ("mean", "se")]
    for q, e in enumerate(ens):
        assert int(e["case"]) == q and int(e["replicas"]) == n_rep
        for col in campaign.TEXTURE_ENSEMBLE:
            v = np.array([r[col] for r in rows[q * n_rep:(q + 1) * n_rep] if r[col] != ""], np.float64)
            assert v.size == (n_rep - 1 if q == 1 else n_rep)
            assert float(e[f"{col}_mean"]) == pytest.approx(np.mean(v), rel=1e-15)
            assert float(e[f"{col}_se"]) == pytest.approx(np.std(v, ddof=1) / np.sqrt(v.size), rel=1e-12)
    assert not os.path.exists("outputs/m/cet_map_front.csv") and not os.path.exists("outputs/m/cet_map_shape.csv")


def test_texture_ensemble_undefined_values():
    rows = [{"case": 0, "T_sub": 1, "MeanCos": "", "Hermans": "0.5", "AlignedFraction": 0.25},
            {"case": 0, "T_sub": 1, "MeanCos": "", "Hermans": "", "AlignedFraction": 0.75}]
    e = campaign.texture_ensemble_stats(rows, ("T_sub",))[0]
    assert e["replicas"] == 2 and e["MeanCos_mean"] == "" and e["MeanCos_se"] == ""
    assert e["Hermans_mean"] == 0.5 and e["Hermans_se"] == ""
    assert e["AlignedFraction_mean"] == 0.5 and e["AlignedFraction_se"] == pytest.approx(0.25)


def test_merge_without_replicas_writes_no_texture_ensemble(tmp_path, monkeypatch):
    lats = _synthetic_map(tmp_path, monkeypatch, 2, 1)
    campaign._write_rows(campaign._map_texture_rows(lats, [1, 0], _case_row, ("T_sub", "NU_DEP")),
                         "outputs/m/melt_pool_map_texture_rank0.csv")
    campaign.merge_melt_pool_map("m")
    assert [int(r["case"]) for r in _read("outputs/m/melt_pool_map_texture.csv")] == [0, 1]
    assert not os.path.exists("outputs/m/melt_pool_map_texture_ensemble.csv")
    assert not os.path.exists("outputs/m/melt_pool_map.csv")
