"""Host side of the front conditions that needs no device: the NumPy reference (tests/frontref.py) on hand-built
lattices along each axis; metrics.front_summary and metrics.front_velocity; the argument checks of cetkmc.front_group
before the library is reached; the arguments the drivers refuse before any Context exists; and the per-case
front.csv, the map front files, their merge and the front ensemble."""
import csv
import ctypes as C
import os

import numpy as np
import pytest

import frontref
from cetkmc import _lib, campaign, metrics

L = 6


def _along(axis, col):
    """A lattice whose column (u, w) = (1, 2) along `axis` holds `col` (length L), every other site empty, and
    T = 1000 + 10 * plane + 0.5 * u along the axis."""
    st = np.zeros((L,) * 3, np.int64)
    idx = [1, 2]
    idx.insert(axis, slice(None))
    st[tuple(idx)] = col
    p = np.arange(L, dtype=np.float64)
    sh = [1, 1, 1]
    sh[axis] = L
    u_axis = (1, 0, 0)[axis]                     # the lower-numbered of the other two axes
    su = [1, 1, 1]
    su[u_axis] = L
    T = 1000.0 + 10.0 * p.reshape(sh) + 0.5 * p.reshape(su) + np.zeros((L,) * 3)
    return st, T


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_reference_empty_and_full(axis):
    st, T = _along(axis, np.zeros(L, np.int64))
    h, top, tf, dt = frontref.front(st, T, axis)
    assert not h.any() and not top.any() and np.isnan(dt).all()
    assert np.array_equal(frontref.bits(tf), frontref.bits(np.moveaxis(T, axis, -1)[..., 0]))
    full = np.ones((L,) * 3, np.int64)
    h, top, tf, dt = frontref.front(full, T, axis)
    assert (h == L).all() and (top == L).all() and np.isnan(tf).all() and np.isnan(dt).all()
    assert (frontref.bits(tf) == 0x7FF8000000000000).all() and (frontref.bits(dt) == 0x7FF8000000000000).all()
    assert h.dtype == np.int32 and top.dtype == np.int32 and tf.shape == (L, L)


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_reference_one_column_gap_and_defect(axis):
    for col, want_h, want_top in (([1, 2, 1, 0, 0, 0], 3, 3),          # one solid column, front at plane 3
                                  ([1, 1, 0, 0, 3, 0], 2, 5),          # solid detached above a gap
                                  ([4, 1, 1, 1, 0, 0], 4, 4),          # a defect (state 4) is occupied
                                  ([0, 0, 0, 0, 0, 2], 0, 6)):
        st, T = _along(axis, np.array(col, np.int64))
        h, top, tf, dt = frontref.front(st, T, axis)
        assert h[1, 2] == want_h and top[1, 2] == want_top, (axis, col)
        assert h.sum() == want_h and top.sum() == want_top                  # every other column is empty
        assert tf[1, 2] == 1000.0 + 10.0 * want_h + 0.5
        if want_h > 0:
            assert dt[1, 2] == (1000.0 + 10.0 * want_h + 0.5) - (1000.0 + 10.0 * (want_h - 1) + 0.5)
        else:
            assert np.isnan(dt[1, 2])
        assert np.isnan(dt).sum() == L * L - (want_h > 0)


def test_reference_column_index_and_non_finite_T():
    rng = np.random.default_rng(4)
    st = rng.integers(0, 2, (5, 5, 5))
    T = rng.uniform(2000, 3000, (5, 5, 5))
    T[0, 0, :] = np.inf
    T[1, 1, 0] = np.float64(np.uint64(0x7FF8000000000123).view(np.float64))
    for axis in range(3):
        h, top, tf, dt = frontref.front(st, T, axis)
        for u in range(5):
            for w in range(5):
                idx = [u, w]
                idx.insert(axis, slice(None))
                col, tcol = st[tuple(idx)], T[tuple(idx)]
                zero = np.flatnonzero(col == 0)
                hh = zero[0] if zero.size else 5
                occ = np.flatnonzero(col)
                assert h[u, w] == hh and top[u, w] == (occ[-1] + 1 if occ.size else 0)
                if hh < 5:
                    assert frontref.bits(tf[u, w]) == frontref.bits(tcol[hh])         # copied as it is
                if 0 < hh < 5:
                    d = tcol[hh] - tcol[hh - 1]
                    assert frontref.bits(dt[u, w]) == (0x7FF8000000000000 if np.isnan(d) else frontref.bits(d))


# -- front_summary and front_velocity -------------------------------------------------------------------------------

def test_front_summary_definitions():
    n = frontref.NAN                                    # L = 4: four copies of the columns below
    h = np.array([0, 2, 4, 3] * 4, np.int32).reshape(4, 4)
    top = np.array([0, 3, 4, 3] * 4, np.int32).reshape(4, 4)
    tf = np.array([3000.0, 3100.0, n, 3200.0] * 4).reshape(4, 4)
    dt = np.array([n, 20.0, n, 40.0] * 4).reshape(4, 4)
    s = metrics.front_summary(h, top, tf, dt, t_melt=3500.0, voxel_size=2.0)
    m = np.array([0, 2, 4, 3] * 4, float)
    assert list(s) == list(metrics.FRONT_COLUMNS)
    assert s["FrontMean"] == np.mean(m) and s["FrontRMS"] == np.std(m) and (s["FrontMin"], s["FrontMax"]) == (0, 4)
    assert s["AheadMean"] == 0.25 and s["AheadFraction"] == 0.25
    assert s["FrontColumns"] == 12 and s["T_Front"] == np.mean([3000.0, 3100.0, 3200.0] * 4)
    assert s["Undercooling"] == 3500.0 - s["T_Front"]
    assert s["GradColumns"] == 8 and s["G_Front"] == 30.0 / 2.0
    d = metrics.front_summary(h, top, tf, dt)
    assert d["Undercooling"] == metrics.K.T_MELT - d["T_Front"] and d["G_Front"] == 30.0 / metrics.K.VOXEL_SIZE


def test_front_summary_empty_means():
    full = np.full((3, 3), 3, np.int32)
    n = np.full((3, 3), frontref.NAN)
    s = metrics.front_summary(full, full, n, n)
    assert (s["FrontColumns"], s["T_Front"], s["Undercooling"], s["GradColumns"], s["G_Front"]) == (0, "", "", 0, "")
    zero = np.zeros((3, 3), np.int32)
    s = metrics.front_summary(zero, zero, np.full((3, 3), 2000.0), n)
    assert s["FrontColumns"] == 9 and s["T_Front"] == 2000.0 and (s["GradColumns"], s["G_Front"]) == (0, "")
    assert s["FrontRMS"] == 0.0 and s["AheadFraction"] == 0.0
    with pytest.raises(ValueError, match="front_summary"):
        metrics.front_summary(zero, zero[:2], n, n)
    with pytest.raises(ValueError, match="front_summary"):
        metrics.front_summary(zero[0], zero[0], n[0], n[0])


def test_front_velocity():
    assert metrics.front_velocity(2.0, 1e-3, 5.0, 3e-3, 5e-6) == 3.0 * 5e-6 / 2e-3
    assert metrics.front_velocity(5.0, 1e-3, 2.0, 3e-3, 1.0) == -3.0 / 2e-3
    assert metrics.front_velocity(2.0, 1e-3, 5.0, 1e-3) == ""
    assert metrics.front_velocity(2.0, 2e-3, 5.0, 1e-3) == ""
    assert metrics.front_velocity("2.5", "0", "3.5", "1e-3", 1.0) == 1.0 / 1e-3


# -- the binding ---------------------------------------------------------------------------------------------------

@pytest.fixture
def no_library(monkeypatch):
    def lib():
        raise AssertionError("the library must not be reached")
    monkeypatch.setattr(_lib, "lib", lib)


def test_binding_checks_before_the_library(no_library):
    made = []
    for _ in range(2):
        c = object.__new__(_lib.Context)
        c._h, c.shape = C.c_void_p(1), (8, 8, 8)
        made.append(c)
    try:
        for axis in (3, -1, None, True, 1.0, "2"):
            with pytest.raises(ValueError, match="axis"):
                _lib.front_group(made, axis)
        with pytest.raises(TypeError):
            _lib.front_group([made[0], object()], 2)
    finally:
        for c in made:
            c._h = C.c_void_p(None)
    assert "cet_front_group" in _lib.SIGNATURES
    import cetkmc
    assert cetkmc.front_group is _lib.front_group


# -- driver refusals: before any Context exists ---------------------------------------------------------------------

@pytest.fixture
def no_context(monkeypatch, tmp_path):
    monkeypatch.chdir(tmp_path)

    def ctx(*a, **kw):
        raise AssertionError("a Context was created")
    monkeypatch.setattr(_lib, "Context", ctx)


@pytest.mark.parametrize("bad", [dict(world=2, rank=0), dict(checkpoint_every=2), dict(resume_from="ck"),
                                 dict(front_axis=3), dict(front_axis=-1), dict(front_axis=True), dict(front_axis=2.0)])
def test_run_cet_sublattice_refusals(no_context, bad):
    kw = dict(front_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="front_axis"):
        campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)


@pytest.mark.parametrize("driver", ["gr", "melt"])
@pytest.mark.parametrize("bad", [dict(checkpoint_every=2), dict(resume_from="ck"), dict(front_axis=5)])
def test_map_driver_refusals(no_context, monkeypatch, driver, bad):
    monkeypatch.setattr(campaign, "run_cet_sublattice", lambda **kw: pytest.fail("a lattice ran"))
    monkeypatch.setattr(campaign, "_run_cases_grouped", lambda *a, **kw: pytest.fail("a group ran"))
    kw = dict(front_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="front_axis"):
        if driver == "gr":
            campaign.run_gr_sweep([2700.0], [1e13], L=8, n_sweeps=5, **kw)
        else:
            campaign.run_melt_pool_map([100.0], [1.0], L=8, n_sweeps=5, **kw)


def test_grouped_driver_refuses_a_bad_axis(no_context):
    with pytest.raises(ValueError, match="front_axis"):
        campaign._run_cases_grouped([("x", 2700.0, 1e13)], L=8, n_sweeps=5, impurity_c=0.0, n_seeds=2,
                                    defect_fraction=0.0, device=0, front_axis=4)


def test_existing_axis_messages_unchanged(no_context):
    for kw, msg in ((dict(profile_axis=4), "run_cet_sublattice: profile_axis must be None, 0, 1 or 2, got 4"),
                    (dict(profile_axis=1, world=2), "run_cet_sublattice: profile_axis needs a whole lattice on one GPU (world = 1)"),
                    (dict(profile_axis=1, checkpoint_every=3),
                     "run_cet_sublattice: profile_axis does not take checkpoint_every or resume_from"),
                    (dict(shape_axis=4), "run_cet_sublattice: shape_axis must be None, 0, 1 or 2, got 4"),
                    (dict(shape_axis=1, resume_from="ck"),
                     "run_cet_sublattice: shape_axis does not take checkpoint_every or resume_from"),
                    (dict(front_axis=4), "run_cet_sublattice: front_axis must be None, 0, 1 or 2, got 4")):
        with pytest.raises(ValueError) as ei:
            campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)
        assert str(ei.value) == msg


# -- front CSV, map front files, merge and ensemble ----------------------------------------------------------------

def _read(path):
    with open(path) as fh:
        return list(csv.DictReader(fh))


def _summary(rng, grad=True):
    Lc = 8
    h = rng.integers(1 if grad else Lc, Lc, (Lc, Lc)).astype(np.int32) if grad else np.full((Lc, Lc), Lc, np.int32)
    top = h + rng.integers(0, 2, (Lc, Lc)).astype(np.int32)
    tf = np.where(h < Lc, rng.uniform(3000, 3400, (Lc, Lc)), frontref.NAN)
    dt = np.where((h > 0) & (h < Lc), rng.uniform(5, 50, (Lc, Lc)), frontref.NAN)
    return metrics.front_summary(h, np.minimum(top, Lc), tf, dt)


def test_front_csv_round_trip(tmp_path):
    rng = np.random.default_rng(2)
    fronts = [(99, 1.5e-3, _summary(rng)), (199, 3.25e-3, _summary(rng)), (201, 3.25e-3, _summary(rng, grad=False))]
    campaign._write_front_csv(fronts, str(tmp_path))
    rows = _read(tmp_path / "front.csv")
    assert list(rows[0].keys()) == ["Step", "Time"] + list(metrics.FRONT_COLUMNS) + ["V_Front"]
    assert rows[0]["V_Front"] == "" and rows[2]["V_Front"] == "" and rows[2]["G_Front"] == ""
    back = campaign.read_front_csv(str(tmp_path / "front.csv"))
    for (step, t, s), b in zip(fronts, back):
        assert b["Step"] == step and b["Time"] == t and {k: b[k] for k in s} == s
    assert back[1]["V_Front"] == metrics.front_velocity(fronts[0][2]["FrontMean"], 1.5e-3, fronts[1][2]["FrontMean"], 3.25e-3)
    campaign._write_front_csv([], str(tmp_path / "none"))                # no rows: no file
    assert not os.path.exists(tmp_path / "none" / "front.csv")


def _synthetic_map(tmp_path, monkeypatch, n_case, n_rep, seed=3):
    monkeypatch.chdir(tmp_path)
    rng = np.random.default_rng(seed)
    lats = campaign._map_lattices([f"m/T{q}" for q in range(n_case)], n_rep)
    for q, r, p in lats:
        os.makedirs(f"outputs/{p}", exist_ok=True)
        campaign._write_front_csv([(5, 1e-4, _summary(rng)), (9, 2e-4 + 1e-5 * r, _summary(rng)),
                                   (13, 3e-4 + 1e-5 * r, _summary(rng))], f"outputs/{p}")
    return lats


def _case_row(q):
    return {"T_sub": 2600.0 + q, "NU_DEP": 1e12 * (q + 1), "G": 1.0e6 * (q + 1), "R": 2.0, "G_over_R": 0.5}


def test_map_front_rows_merge_and_ensemble(tmp_path, monkeypatch):
    n_case, n_rep = 3, 4
    lats = _synthetic_map(tmp_path, monkeypatch, n_case, n_rep)
    axes = ("T_sub", "NU_DEP")
    rows = campaign._map_front_rows(lats, list(range(len(lats))), _case_row, axes)
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP", "G", "R", "G_Front", "V_Front", "G_over_V",
                                    "Undercooling", "FrontMean", "FrontRMS"]
    for (q, r, p), row in zip(lats, rows):
        fr = campaign.read_front_csv(f"outputs/{p}/front.csv")
        v = (fr[-1]["FrontMean"] - fr[0]["FrontMean"]) * metrics.K.VOXEL_SIZE / (fr[-1]["Time"] - fr[0]["Time"])
        assert (row["case"], row["replica"], row["G"]) == (q, r, 1.0e6 * (q + 1))
        assert row["V_Front"] == v and row["G_Front"] == fr[-1]["G_Front"] and row["FrontRMS"] == fr[-1]["FrontRMS"]
        assert row["G_over_V"] == (row["G_Front"] / v if v > 0 else "")
    mine = [[l for l in range(len(lats)) if l % 2 == k] for k in range(2)]
    for k in range(2):
        campaign._write_rows(campaign._map_front_rows(lats, mine[k], _case_row, axes), f"outputs/m/cet_map_front_rank{k}.csv")
        campaign._write_rows([{"case": lats[l][0], "replica": lats[l][1], **_case_row(lats[l][0]),
                               **{c: 1.0 for c in campaign.ENSEMBLE_COLUMNS}, "CET_Class": "Equiaxed",
                               "CET_Detected": True} for l in mine[k]], f"outputs/m/cet_map_replicas_rank{k}.csv")
    campaign.merge_cet_map("m")
    merged = _read("outputs/m/cet_map_front.csv")
    assert [(int(r["case"]), int(r["replica"])) for r in merged] == [(q, r) for q, r, _ in lats]
    assert [float(r["V_Front"]) for r in merged] == [r["V_Front"] for r in rows]
    ens = _read("outputs/m/cet_map_front_ensemble.csv")
    assert list(ens[0].keys()) == ["case", "T_sub", "NU_DEP", "G", "R", "replicas"] + [
        f"{c}_{s}" for c in campaign.FRONT_ENSEMBLE for s in ("mean", "se")]
    for q, e in enumerate(ens):
        assert int(e["case"]) == q and int(e["replicas"]) == n_rep
        for col in campaign.FRONT_ENSEMBLE:
            v = np.array([r[col] for r in rows[q * n_rep:(q + 1) * n_rep]], np.float64)
            assert float(e[f"{col}_mean"]) == pytest.approx(np.mean(v), rel=1e-15)
            assert float(e[f"{col}_se"]) == pytest.approx(np.std(v, ddof=1) / np.sqrt(n_rep), rel=1e-12)
    assert not os.path.exists("outputs/m/cet_map_shape.csv") and not os.path.exists("outputs/m/cet_map_profile.csv")


def test_front_ensemble_undefined_values():
    rows = [{"case": 0, "T_sub": 1, "G": 2, "R": 3, "G_Front": "", "V_Front": "4.0", "Undercooling": 5.0, "FrontRMS": 1.0},
            {"case": 0, "T_sub": 1, "G": 2, "R": 3, "G_Front": "", "V_Front": "", "Undercooling": 7.0, "FrontRMS": 3.0}]
    e = campaign.front_ensemble_stats(rows, ("T_sub",))[0]
    assert e["replicas"] == 2 and e["G_Front_mean"] == "" and e["G_Front_se"] == ""
    assert e["V_Front_mean"] == 4.0 and e["V_Front_se"] == ""
    assert e["Undercooling_mean"] == 6.0 and e["Undercooling_se"] == pytest.approx(1.0)


def test_merge_without_replicas_writes_no_front_ensemble(tmp_path, monkeypatch):
    lats = _synthetic_map(tmp_path, monkeypatch, 2, 1)
    campaign._write_rows(campaign._map_front_rows(lats, [1, 0], _case_row, ("T_sub", "NU_DEP")),
                         "outputs/m/melt_pool_map_front_rank0.csv")
    campaign.merge_melt_pool_map("m")
    assert [int(r["case"]) for r in _read("outputs/m/melt_pool_map_front.csv")] == [0, 1]
    assert not os.path.exists("outputs/m/melt_pool_map_front_ensemble.csv")
    assert not os.path.exists("outputs/m/melt_pool_map.csv")
