"""Host side of the per-plane grain profiles that needs no device: metrics.cet_profile_summary on synthetic profiles,
the NumPy reference profile (tests/profileref.py) on hand-counted lattices, the argument checks of
cetkmc.grain_profile_group before the library is reached, the arguments the drivers refuse before any Context exists,
and the map profile files, their merge and the profile ensemble."""
import csv
import ctypes as C
import os

import numpy as np
import pytest

import hostref
import profileref
from cetkmc import _lib, campaign, metrics


# -- metrics.cet_profile_summary ----------------------------------------------------------------------------------

def _prof(solid, eq):
    p = np.zeros((4, len(solid)), np.int64)
    p[0], p[1] = solid, eq
    return p


def _summary(solid, eq, plane_sites=10, **kw):
    return metrics.cet_profile_summary(_prof(solid, eq), plane_sites, **kw)


def test_summary_all_columnar():
    assert _summary([10] * 6, [0] * 6) == {"CET_Height": -1, "Front_Height": 5}


def test_summary_equiaxed_everywhere_gives_lowest_solid_plane():
    assert _summary([10] * 6, [10] * 6) == {"CET_Height": 0, "Front_Height": 5}
    # the substrate plane not solidified: the lowest plane of P
    assert _summary([2, 10, 10, 10], [2, 9, 8, 10]) == {"CET_Height": 1, "Front_Height": 3}


def test_summary_clean_transition():
    assert _summary([10] * 8, [0, 0, 1, 4, 6, 9, 10, 10]) == {"CET_Height": 4, "Front_Height": 7}


def test_summary_isolated_equiaxed_plane_below_a_columnar_band_does_not_count():
    assert _summary([10] * 8, [10, 10, 0, 0, 0, 7, 8, 9]) == {"CET_Height": 5, "Front_Height": 7}
    assert _summary([10] * 5, [10, 10, 0, 0, 0]) == {"CET_Height": -1, "Front_Height": 4}


def test_summary_melt_planes_above_the_front_are_excluded():
    # planes 4..5 hold a few columnar sites only (melt / vapour): below min_solid, so the front is plane 3
    assert _summary([10, 10, 10, 10, 4, 1], [0, 6, 7, 8, 0, 0]) == {"CET_Height": 1, "Front_Height": 3}
    # a lower min_solid lets them in, and the front turns columnar
    assert _summary([10, 10, 10, 10, 4, 1], [0, 6, 7, 8, 0, 0], min_solid=0.1) == {"CET_Height": -1, "Front_Height": 5}


def test_summary_empty_lattice():
    assert _summary([0] * 4, [0] * 4) == {"CET_Height": -1, "Front_Height": -1}
    assert _summary([0] * 4, [0] * 4, min_solid=0.0) == {"CET_Height": -1, "Front_Height": -1}


def test_summary_threshold_is_inclusive():
    assert _summary([10] * 4, [0, 5, 5, 5]) == {"CET_Height": 1, "Front_Height": 3}     # eq = 0.5 = threshold
    assert _summary([10] * 4, [0, 5, 5, 5], eq_threshold=0.51) == {"CET_Height": -1, "Front_Height": 3}
    assert _summary([4] * 3, [2, 2, 2], plane_sites=8) == {"CET_Height": 0, "Front_Height": 2}     # Solid = 0.5 * sites


def test_summary_rejects_a_bad_shape():
    with pytest.raises(ValueError):
        metrics.cet_profile_summary(np.zeros((3, 5)), 25)


# -- the NumPy reference on hand-counted lattices -------------------------------------------------------------------

def _label(state, theta=None):
    theta = np.full(state.shape, 0.3) if theta is None else theta
    return hostref.label_grains(state, theta, np.full(state.shape, 1.1))


def test_reference_single_column_grain():
    L = 6
    st = np.zeros((L, L, L), np.int64)
    st[2, 3, :] = 1                          # joined through (0, 0, +-2) steps: two grains, k even and k odd
    lab, n = _label(st)
    assert n == 2
    p = profileref.grain_profile(lab, 2, 3.0)
    # grain k even spans planes 0..4, grain k odd 1..5; each box is 1 x 1 x 5: AR 5, not equiaxed
    assert p.tolist() == [[1] * 6, [0] * 6, [1, 2, 2, 2, 2, 1], [0] * 6]
    # along axis 0 the whole column sits on plane 2
    assert profileref.grain_profile(lab, 0, 3.0).tolist() == [[0, 0, 6, 0, 0, 0], [0] * 6, [0, 0, 2, 0, 0, 0], [0] * 6]
    # with a threshold above 5 both are equiaxed; at 5 (strict) neither
    assert profileref.grain_profile(lab, 2, 5.5)[1].tolist() == [1] * 6
    assert profileref.grain_profile(lab, 2, 5.0)[1].tolist() == [0] * 6


def test_reference_grain_spans_a_plane_it_has_no_site_on():
    L = 5
    st = np.zeros((L, L, L), np.int64)
    st[1, 1, 0] = st[1, 1, 2] = 1            # linked only through the (0, 0, 2) offset: one grain, nothing on k = 1
    st[3, 3, 4] = 2                          # a second, single-site grain
    th = np.full(st.shape, 0.3)
    th[3, 3, 4] = 2.0
    lab, n = _label(st, th)
    assert n == 2
    p = profileref.grain_profile(lab, 2, 3.0)
    # box of grain 1: 1 x 1 x 3 (AR 3, columnar); grain 2: 1 x 1 x 1 (AR 1, equiaxed)
    assert p[0].tolist() == [1, 0, 1, 0, 1]
    assert p[1].tolist() == [0, 0, 0, 0, 1]
    assert p[2].tolist() == [1, 1, 1, 0, 1]          # plane 1: spanned, but no site of the grain on it
    assert p[3].tolist() == [0, 0, 0, 0, 1]


def test_reference_two_grains_and_classes():
    L = 4
    st = np.zeros((L, L, L), np.int64)
    st[0, 0, 0] = st[0, 1, 1] = st[1, 0, 1] = 1      # (0,1,1) and (1,-1,0) steps: one grain, box 2 x 2 x 2
    th = np.full(st.shape, 0.3)
    st[3, :, 3] = 1                                    # (0, +-2, 0) steps: j even and j odd, two 1 x 3 x 1 boxes
    th[3, :, 3] = 2.0
    lab, n = _label(st, th)
    assert n == 3
    p = profileref.grain_profile(lab, 1, 3.0)
    # along j: the small grain has sites on j = 0 (two) and j = 1 (one), the columns one site per plane
    assert p[0].tolist() == [3, 2, 1, 1]
    assert p[1].tolist() == [2, 1, 0, 0]             # the 2 x 2 x 2 box is equiaxed (AR 1), the columns are not (AR 3)
    assert p[2].tolist() == [2, 3, 2, 1]             # boxes j 0..1, 0..2 and 1..3
    assert p[3].tolist() == [1, 1, 0, 0]
    assert profileref.grain_profile(np.zeros((3, 3, 3), np.int32), 0, 3.0).tolist() == [[0] * 3] * 4


# -- the binding ----------------------------------------------------------------------------------------------------

@pytest.fixture
def no_library(monkeypatch):
    def lib():
        raise AssertionError("the library must not be reached")
    monkeypatch.setattr(_lib, "lib", lib)


@pytest.fixture
def fake_ctxs():
    made = []

    def make(n, L=8):
        for _ in range(n):
            c = object.__new__(_lib.Context)
            c._h, c.shape = C.c_void_p(1), (L, L, L)
            made.append(c)
        return made[-n:]
    yield make
    for c in made:
        c._h = C.c_void_p(None)


def test_binding_checks_before_the_library(no_library, fake_ctxs):
    a = fake_ctxs(2)
    for axis in (3, -1, None, True, 1.0, "2"):
        with pytest.raises(ValueError, match="axis"):
            _lib.grain_profile_group(a, axis, 3.0)
    for thr in (np.nan, np.inf, -np.inf):
        with pytest.raises(ValueError, match="finite"):
            _lib.grain_profile_group(a, 2, thr)
    with pytest.raises(TypeError):
        _lib.grain_profile_group([a[0], object()], 2, 3.0)
    assert _lib.PROFILE_COLUMNS == ("Solid", "EquiaxedSolid", "GrainsSpanning", "EquiaxedGrainsSpanning")
    assert "cet_grain_profile_group" in _lib.SIGNATURES


# -- driver refusals: before any Context exists ---------------------------------------------------------------------

@pytest.fixture
def no_context(monkeypatch, tmp_path):
    monkeypatch.chdir(tmp_path)

    def ctx(*a, **kw):
        raise AssertionError("a Context was created")
    monkeypatch.setattr(_lib, "Context", ctx)


@pytest.mark.parametrize("bad", [dict(world=2, rank=0), dict(checkpoint_every=2), dict(resume_from="ck"),
                                 dict(profile_axis=3), dict(profile_axis=-1), dict(profile_axis=True)])
def test_run_cet_sublattice_refusals(no_context, bad):
    kw = dict(profile_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="profile_axis"):
        campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)


@pytest.mark.parametrize("driver", ["gr", "melt"])
@pytest.mark.parametrize("bad", [dict(checkpoint_every=2), dict(resume_from="ck"), dict(profile_axis=5)])
def test_map_driver_refusals(no_context, monkeypatch, driver, bad):
    monkeypatch.setattr(campaign, "run_cet_sublattice", lambda **kw: pytest.fail("a lattice ran"))
    monkeypatch.setattr(campaign, "_run_cases_grouped", lambda *a, **kw: pytest.fail("a group ran"))
    kw = dict(profile_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="profile_axis"):
        if driver == "gr":
            campaign.run_gr_sweep([2700.0], [1e13], L=8, n_sweeps=5, **kw)
        else:
            campaign.run_melt_pool_map([100.0], [1.0], L=8, n_sweeps=5, **kw)


def test_grouped_driver_refuses_a_bad_axis(no_context):
    with pytest.raises(ValueError, match="profile_axis"):
        campaign._run_cases_grouped([("x", 2700.0, 1e13)], L=8, n_sweeps=5, impurity_c=0.0, n_seeds=2,
                                    defect_fraction=0.0, device=0, profile_axis=4)


# -- profile CSV, map profile files, merge and ensemble -------------------------------------------------------------

def _read(path):
    with open(path) as fh:
        return list(csv.DictReader(fh))


def test_profile_csv_round_trip(tmp_path):
    rng = np.random.default_rng(1)
    profs = [(99, rng.integers(0, 50, (4, 6))), (199, rng.integers(0, 50, (4, 6)))]
    campaign._write_profile_csv(profs, str(tmp_path))
    rows = _read(tmp_path / "cet_profile.csv")
    assert list(rows[0].keys()) == ["Step", "Plane", "Solid", "EquiaxedSolid", "GrainsSpanning", "EquiaxedGrainsSpanning"]
    assert len(rows) == 12 and [int(r["Plane"]) for r in rows[:6]] == list(range(6))
    step, p = campaign.read_profile_csv(str(tmp_path / "cet_profile.csv"))
    assert step == 199 and np.array_equal(p, profs[1][1])
    campaign._write_profile_csv([], str(tmp_path / "none"))           # no rows: no file
    assert not os.path.exists(tmp_path / "none" / "cet_profile.csv")


def _synthetic_map(tmp_path, monkeypatch, n_case, n_rep, L=6, seed=3):
    """cet_profile.csv files of n_case x n_rep lattices and their (case, replica, prefix) list."""
    monkeypatch.chdir(tmp_path)
    rng = np.random.default_rng(seed)
    lats = campaign._map_lattices([f"m/T{q}" for q in range(n_case)], n_rep)
    for q, r, p in lats:
        os.makedirs(f"outputs/{p}", exist_ok=True)
        solid = np.full(L, L * L)
        solid[-1] = rng.integers(0, L * L // 2)                       # a melt plane above the front
        eq = (solid * np.clip(np.linspace(-0.5, 1.5, L) + rng.uniform(-0.6, 0.6), 0, 1)).astype(np.int64)
        if rng.random() < 0.3:
            eq[-2] = 0                                                 # columnar at the front
        prof = np.zeros((4, L), np.int64)
        prof[0], prof[1] = solid, eq
        campaign._write_profile_csv([(5, prof * 0), (9, prof)], f"outputs/{p}")
    return lats


def _case_row(q):
    return {"T_sub": 2600.0 + q, "NU_DEP": 1e12 * (q + 1), "G": 1.0, "R": 2.0, "G_over_R": 0.5}


def test_map_profile_rows_merge_and_ensemble(tmp_path, monkeypatch):
    n_case, n_rep = 3, 4
    lats = _synthetic_map(tmp_path, monkeypatch, n_case, n_rep)
    axes = ("T_sub", "NU_DEP")
    rows = campaign._map_profile_rows(lats, list(range(len(lats))), _case_row, axes)
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP", "CET_Height", "Front_Height"]
    for (q, r, p), row in zip(lats, rows):
        _s, prof = campaign.read_profile_csv(f"outputs/{p}/cet_profile.csv")
        assert (row["case"], row["replica"]) == (q, r)
        s = metrics.cet_profile_summary(prof, 36)
        assert (row["CET_Height"], row["Front_Height"]) == (s["CET_Height"], s["Front_Height"])
        assert row["Front_Height"] == 4
    heights = np.array([r["CET_Height"] for r in rows])
    assert (heights >= 0).any() and (heights < 0).any()
    # two ranks, interleaved; merge sorts by (case, replica)
    mine = [[l for l in range(len(lats)) if l % 2 == k] for k in range(2)]
    for k in range(2):
        campaign._write_rows(campaign._map_profile_rows(lats, mine[k], _case_row, axes),
                             f"outputs/m/cet_map_profile_rank{k}.csv")
        campaign._write_rows([{"case": lats[l][0], "replica": lats[l][1], **_case_row(lats[l][0]),
                               **{c: 1.0 for c in campaign.ENSEMBLE_COLUMNS}, "CET_Class": "Equiaxed",
                               "CET_Detected": True} for l in mine[k]], f"outputs/m/cet_map_replicas_rank{k}.csv")
    campaign.merge_cet_map("m")
    merged = _read("outputs/m/cet_map_profile.csv")
    assert [(int(r["case"]), int(r["replica"])) for r in merged] == [(q, r) for q, r, _ in lats]
    assert [int(r["CET_Height"]) for r in merged] == heights.tolist()
    ens = _read("outputs/m/cet_map_profile_ensemble.csv")
    assert list(ens[0].keys()) == ["case", "T_sub", "NU_DEP", "replicas", "p_cet_height", "CET_Height_mean", "CET_Height_se"]
    for q, e in enumerate(ens):
        h = heights[q * n_rep:(q + 1) * n_rep]
        v = h[h >= 0].astype(np.float64)
        assert int(e["case"]) == q and int(e["replicas"]) == n_rep
        assert float(e["p_cet_height"]) == np.mean(h >= 0)
        if v.size:
            assert float(e["CET_Height_mean"]) == np.mean(v)
        else:
            assert e["CET_Height_mean"] == ""
        if v.size > 1:
            assert float(e["CET_Height_se"]) == pytest.approx(np.std(v, ddof=1) / np.sqrt(v.size), rel=1e-15)
        else:
            assert e["CET_Height_se"] == ""


def test_profile_ensemble_small_counts():
    rows = [{"case": 0, "T_sub": 1, "CET_Height": 3}, {"case": 1, "T_sub": 2, "CET_Height": -1},
            {"case": 1, "T_sub": 2, "CET_Height": 4}, {"case": 2, "T_sub": 3, "CET_Height": "7"},
            {"case": 2, "T_sub": 3, "CET_Height": "2"}]
    e = campaign.profile_ensemble_stats(rows, ("T_sub",))
    assert e[0] == {"case": 0, "T_sub": 1, "replicas": 1, "p_cet_height": 1.0, "CET_Height_mean": 3.0, "CET_Height_se": ""}
    assert e[1]["p_cet_height"] == 0.5 and e[1]["CET_Height_mean"] == 4.0 and e[1]["CET_Height_se"] == ""
    assert e[2]["CET_Height_mean"] == 4.5 and e[2]["CET_Height_se"] == pytest.approx(np.std([7.0, 2.0], ddof=1) / np.sqrt(2))


def test_merge_without_replicas_writes_no_profile_ensemble(tmp_path, monkeypatch):
    lats = _synthetic_map(tmp_path, monkeypatch, 2, 1)
    campaign._write_rows(campaign._map_profile_rows(lats, [1, 0], _case_row, ("T_sub", "NU_DEP")),
                         "outputs/m/cet_map_profile_rank0.csv")
    campaign.merge_cet_map("m")
    assert [int(r["case"]) for r in _read("outputs/m/cet_map_profile.csv")] == [0, 1]
    assert not os.path.exists("outputs/m/cet_map_profile_ensemble.csv")
    assert not os.path.exists("outputs/m/cet_map.csv")        # no map rank files: nothing else appears
