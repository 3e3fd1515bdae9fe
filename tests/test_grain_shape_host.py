"""Host side of the grain-shape histograms that needs no device: the derivation the kernels inline (csrc/grain_shape.cuh,
compiled by g++ as a test-only shim) bit for bit against Python integers and float(); the NumPy reference
(tests/shaperef.py) on hand-built lattices; metrics.grain_shape_summary; the argument checks of
cetkmc.grain_shape_group before the library is reached; the arguments the drivers refuse before any Context exists; and
the per-case CSV, the map shape files, their merge and the shape ensemble."""
import csv
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import hostref
import shaperef
from cetkmc import _lib, campaign, metrics
from conftest import ROOT

SRC = os.path.join(ROOT, "tests", "hostsim", "grain_shape_host.cpp")
OUT = os.path.join(ROOT, "tests", "hostsim", "_build")
L_MAX = 1290                       # the largest L of a context (fewer than 2^31 sites)
N_MAX = 2 ** 31 - 1
WORDS = 8


@pytest.fixture(scope="module")
def shim():
    os.makedirs(OUT, exist_ok=True)
    so = os.path.join(OUT, "libgrainshape.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so, SRC], check=True)
    lib = C.CDLL(so)
    lib.hostsim_shape_q.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]
    lib.hostsim_shape_fl.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p]
    lib.hostsim_shape_bins.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p,
                                       C.c_void_p]
    return lib


def _slots(moms):
    """(count, 8) uint64 moment slots from a list of (n, [S_0, S_1, S_2], [S_00, S_11, S_22])."""
    m = np.zeros((len(moms), WORDS), np.uint64)
    for g, (n, s, ss) in enumerate(moms):
        m[g, 0] = n
        m[g, 1:4] = s
        m[g, 4:7] = ss
    return np.ascontiguousarray(m)


def _q(shim, m, x):
    out = np.zeros((m.shape[0], 2), np.uint64)
    shim.hostsim_shape_q(m.ctypes.data, m.shape[0], x, out.ctypes.data)
    return [int(lo) | (int(hi) << 64) for lo, hi in out]


def _fl(shim, vals):
    v = np.array([[x & (2 ** 64 - 1), x >> 64] for x in vals], np.uint64)
    out = np.zeros(len(vals))
    shim.hostsim_shape_fl(v.ctypes.data, len(vals), out.ctypes.data)
    return out


def _bins(shim, m, axis, edges=_lib.SHAPE_EDGES, min_size=1):
    e = np.ascontiguousarray(edges, dtype=np.float64)
    a, b = np.zeros(m.shape[0]), np.zeros(m.shape[0], np.int32)
    shim.hostsim_shape_bins(m.ctypes.data, m.shape[0], axis, e.ctypes.data, e.size, min_size, a.ctypes.data, b.ctypes.data)
    return a, b


def _random_moments(rng, count, n_max=N_MAX, c_max=L_MAX - 1):
    """Moments of grains whose n sites sit on up to three coordinate values per axis (any valid moment set has
    n S_xx >= S_x^2; these are realisable), n log-uniform up to n_max."""
    out = []
    for _ in range(count):
        n = int(min(n_max, max(1, round(math.exp(rng.uniform(0, math.log(n_max)))))))
        s, ss = [], []
        for _x in range(3):
            k1 = int(rng.integers(0, n + 1))
            k2 = int(rng.integers(0, n - k1 + 1))
            vals = [int(v) for v in rng.integers(0, c_max + 1, 3)]
            ks = [k1, k2, n - k1 - k2]
            s.append(sum(k * v for k, v in zip(ks, vals)))
            ss.append(sum(k * v * v for k, v in zip(ks, vals)))
        out.append((n, s, ss))
    return out


# -- the derivation the kernels inline, bit for bit ----------------------------------------------------------------

def test_derivation_matches_python_on_random_moments(shim):
    rng = np.random.default_rng(12)
    moms = _random_moments(rng, 4000) + _random_moments(rng, 1000, n_max=64, c_max=23)
    m = _slots(moms)
    qs = {x: _q(shim, m, x) for x in range(3)}
    for g, (n, s, ss) in enumerate(moms):
        for x in range(3):
            assert qs[x][g] == shaperef.q_moment(n, s[x], ss[x])
    assert max(max(q) for q in qs.values()) > 2 ** 64                       # the 128-bit range is exercised
    assert any(2 ** 53 < q < 2 ** 64 for q in qs[0])
    edges = (1.0, 1.5, 2.0, 3.0, 4.0, 6.0, 8.0, 12.0, 16.0, 32.0)
    for axis in range(3):
        a, b = _bins(shim, m, axis, edges, min_size=1)
        want = [shaperef.elongation_of(n, s, ss, axis) for n, s, ss in moms]
        assert a.tobytes() == np.array(want).tobytes()
        assert b.tolist() == np.searchsorted(edges, want, side="right").tolist()
        # edges at attained values: a one-ulp difference in A would move a grain to another bin
        at = sorted(set(want))[::max(1, len(set(want)) // 60)][:62]
        _a, b2 = _bins(shim, m, axis, at, min_size=1)
        assert b2.tolist() == np.searchsorted(at, want, side="right").tolist()
        assert (b2 > 0).any() and (np.array(want)[b2 > 0] >= np.array(at)[b2[b2 > 0] - 1]).all()


def test_fl_rounds_like_python_float(shim):
    rng = np.random.default_rng(3)
    vals = [0, 1, 2 ** 53 - 1, 2 ** 53, 2 ** 53 + 1, 2 ** 64 - 1, 2 ** 64, 2 ** 64 + 1, 2 ** 106 - 1]
    vals += [int(rng.integers(0, 2 ** 62)) << int(rng.integers(0, 44)) | int(rng.integers(0, 2 ** 40)) for _ in range(2000)]
    # exactly halfway between two doubles, with an even and an odd lower neighbour (ties go to even)
    for e in (53, 54, 60, 64, 65, 80, 104):
        for mant in (2 ** 52, 2 ** 52 + 1, 2 ** 52 + 2, 2 ** 53 - 1, 2 ** 52 + 12345):
            d = mant << (e - 52)
            vals += [d + (1 << (e - 53)), d + (1 << (e - 53)) - 1, d + (1 << (e - 53)) + 1]
    vals = [v for v in vals if v < 2 ** 106]
    got = _fl(shim, vals)
    assert got.tobytes() == np.array([float(v) for v in vals]).tobytes()


def test_elongation_properties(shim):
    def box(a, b, c, off=(0, 0, 0), axis=2):
        dims = [0, 0, 0]
        dims[axis], dims[(axis + 1) % 3], dims[(axis + 2) % 3] = a, b, c
        g = np.zeros([d + o + 1 for d, o in zip(dims, off)], np.int32)
        g[off[0]:off[0] + dims[0], off[1]:off[1] + dims[1], off[2]:off[2] + dims[2]] = 1
        return g
    for axis in range(3):
        assert shaperef.elongations(box(1, 1, 1, axis=axis), axis)[1].tolist() == [1.0]
        for h in (2, 3, 7, 64, 1289):
            assert shaperef.elongations(box(h, 1, 1, axis=axis), axis)[1].tolist() == [float(h)]
        for a, b, c in ((3, 2, 5), (8, 8, 8), (10, 1, 4)):
            _n, A = shaperef.elongations(box(a, b, c, axis=axis), axis)
            assert A[0] == math.sqrt(float(2 * a * a) / float(b * b + c * c))
            _n, A2 = shaperef.elongations(box(a, b, c, off=(5, 2, 9), axis=axis), axis)
            assert A2.tobytes() == A.tobytes()                                  # translation
        # the derivation of the shim on the same moments
        n, s, ss = shaperef.grain_moments(box(3, 2, 5, off=(1, 4, 2), axis=axis))
        a, _b = _bins(shim, _slots([(n[0], s[:, 0].tolist(), ss[:, 0].tolist())]), axis)
        assert a.tobytes() == shaperef.elongations(box(3, 2, 5, axis=axis), axis)[1].tobytes()
    pair = np.zeros((3, 3, 5), np.int32)
    pair[1, 1, 1] = pair[1, 1, 3] = 1
    assert shaperef.elongations(pair, 2)[1].tolist() == [math.sqrt(13.0)]


# -- the NumPy reference on hand-built lattices --------------------------------------------------------------------

def _label(state, theta=None):
    theta = np.full(state.shape, 0.3) if theta is None else theta
    return hostref.label_grains(state, theta, np.full(state.shape, 1.1))


EDGES = (1.0, 2.0, 3.0, 4.0)


def test_reference_single_voxel_and_columns():
    L = 8
    st = np.zeros((L, L, L), np.int64)
    st[2, 3, :] = 1                          # joined through (0, 0, +-2) steps: k even and k odd, 4 sites each
    st[6, 6, 6] = 1                          # a single voxel
    lab, n = _label(st)
    assert n == 3
    h = shaperef.grain_shape(lab, 2, EDGES, 1)
    # the two columns: sites k = 0, 2, 4, 6 -> var 5, Q_a = 16 (12 * 5 + 1) = 976, Q_b = Q_c = 16: A = sqrt(61) = 7.8
    assert h.tolist() == [[0, 1, 0, 0, 2, 0], [0, 1, 0, 0, 8, 0]]
    # across the column: A = sqrt(2 * 16 / (16 + 976)) < 1
    assert shaperef.grain_shape(lab, 0, EDGES, 1).tolist() == [[2, 1, 0, 0, 0, 0], [8, 1, 0, 0, 0, 0]]
    # min_size 2: the voxel goes to the small bucket
    assert shaperef.grain_shape(lab, 2, EDGES, 2).tolist() == [[0, 0, 0, 0, 2, 1], [0, 0, 0, 0, 8, 1]]


def test_reference_pm2_pair_and_min_size():
    L = 5
    st = np.zeros((L, L, L), np.int64)
    st[1, 1, 0] = st[1, 1, 2] = 1            # linked only through the (0, 0, 2) offset: one grain of two sites
    lab, n = _label(st)
    assert n == 1
    e = _lib.SHAPE_EDGES
    h1 = shaperef.grain_shape(lab, 2, e, 1)
    assert h1[0, 4] == 1 and h1[1, 4] == 2 and h1.sum() == 3                 # sqrt(13) = 3.61: bin 4, 3 <= A < 4
    h8 = shaperef.grain_shape(lab, 2, e, _lib.SHAPE_MIN_SIZE)
    assert h8[:, -1].tolist() == [1, 2] and h8[:, :-1].sum() == 0            # no column at the default min_size


def test_reference_axis_permutation_and_translation():
    rng = np.random.default_rng(7)
    L = 12
    st = (rng.random((L, L, L)) < 0.5).astype(np.int64)
    th = rng.choice([0.3, 1.5, 2.7], (L, L, L))
    lab, n = _label(st, th)
    assert n > 3
    e = _lib.SHAPE_EDGES
    for axis in range(3):
        h = shaperef.grain_shape(lab, axis, e, 2)
        assert h[0].sum() == n and h[1].sum() == st.sum()
        # transposing the lattice moves the growth axis with it
        perm = [axis] + [x for x in range(3) if x != axis]
        assert np.array_equal(shaperef.grain_shape(np.transpose(lab, perm), 0, e, 2), h)
        # shifting the lattice inside a larger one
        big = np.zeros((L + 5,) * 3, lab.dtype)
        big[3:3 + L, 1:1 + L, 4:4 + L] = lab
        assert np.array_equal(shaperef.grain_shape(big, axis, e, 2), h)


def test_reference_empty_lattice():
    lab = np.zeros((6, 6, 6), np.int32)
    assert shaperef.grain_shape(lab, 1, EDGES, 1).tolist() == [[0] * 6, [0] * 6]


# -- metrics.grain_shape_summary -----------------------------------------------------------------------------------

def test_summary_definitions():
    e = (1.0, 2.0, 3.0, 4.0)
    h = np.array([[5, 4, 3, 2, 1, 100], [10, 20, 30, 40, 50, 150]])
    s = metrics.grain_shape_summary(h, e, threshold=3.0)
    assert s == {"ColumnarVolumeFraction": 90 / 300, "ColumnarGrainFraction": 3 / 15, "ShapedGrains": 15}
    s = metrics.grain_shape_summary(h, e, threshold=1.0)
    assert s["ColumnarVolumeFraction"] == 140 / 300 and s["ColumnarGrainFraction"] == 10 / 15
    s = metrics.grain_shape_summary(h, e)                                      # default threshold CET_AR_THRESHOLD = 3
    assert s["ColumnarVolumeFraction"] == 90 / 300
    # nothing shaped / nothing occupied
    assert metrics.grain_shape_summary(np.array([[0] * 5 + [7], [0] * 5 + [9]]), e) == \
        {"ColumnarVolumeFraction": 0.0, "ColumnarGrainFraction": 0.0, "ShapedGrains": 0}
    assert metrics.grain_shape_summary(np.zeros((2, 6), np.int64), e) == \
        {"ColumnarVolumeFraction": 0.0, "ColumnarGrainFraction": 0.0, "ShapedGrains": 0}


def test_summary_refusals():
    e = (1.0, 2.0, 3.0, 4.0)
    with pytest.raises(ValueError, match="edges"):
        metrics.grain_shape_summary(np.zeros((2, 6)), e, threshold=2.5)
    with pytest.raises(ValueError, match="histogram"):
        metrics.grain_shape_summary(np.zeros((2, 5)), e)
    with pytest.raises(ValueError, match="histogram"):
        metrics.grain_shape_summary(np.zeros((3, 6)), e)


# -- the binding ---------------------------------------------------------------------------------------------------

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
            _lib.grain_shape_group(a, axis)
    for edges in ((), tuple(float(x) for x in range(1, 64)), (1.0, np.nan), (1.0, np.inf), (0.0, 1.0), (-1.0, 2.0),
                  (1.0, 1.0), (2.0, 1.0), [[1.0, 2.0]], ("a",)):
        with pytest.raises(ValueError, match="edges"):
            _lib.grain_shape_group(a, 2, edges)
    for ms in (0, -3, 1.5, True, None):
        with pytest.raises(ValueError, match="min_size"):
            _lib.grain_shape_group(a, 2, min_size=ms)
    with pytest.raises(TypeError):
        _lib.grain_shape_group([a[0], object()], 2)
    assert _lib.SHAPE_EDGES == (1.0, 1.5, 2.0, 3.0, 4.0, 6.0, 8.0, 12.0, 16.0, 32.0) and _lib.SHAPE_MIN_SIZE == 8
    assert "cet_grain_shape_group" in _lib.SIGNATURES
    import cetkmc
    assert cetkmc.grain_shape_group is _lib.grain_shape_group


# -- driver refusals: before any Context exists ---------------------------------------------------------------------

@pytest.fixture
def no_context(monkeypatch, tmp_path):
    monkeypatch.chdir(tmp_path)

    def ctx(*a, **kw):
        raise AssertionError("a Context was created")
    monkeypatch.setattr(_lib, "Context", ctx)


@pytest.mark.parametrize("bad", [dict(world=2, rank=0), dict(checkpoint_every=2), dict(resume_from="ck"),
                                 dict(shape_axis=3), dict(shape_axis=-1), dict(shape_axis=True)])
def test_run_cet_sublattice_refusals(no_context, bad):
    kw = dict(shape_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="shape_axis"):
        campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)


@pytest.mark.parametrize("driver", ["gr", "melt"])
@pytest.mark.parametrize("bad", [dict(checkpoint_every=2), dict(resume_from="ck"), dict(shape_axis=5)])
def test_map_driver_refusals(no_context, monkeypatch, driver, bad):
    monkeypatch.setattr(campaign, "run_cet_sublattice", lambda **kw: pytest.fail("a lattice ran"))
    monkeypatch.setattr(campaign, "_run_cases_grouped", lambda *a, **kw: pytest.fail("a group ran"))
    kw = dict(shape_axis=2)
    kw.update(bad)
    with pytest.raises(ValueError, match="shape_axis"):
        if driver == "gr":
            campaign.run_gr_sweep([2700.0], [1e13], L=8, n_sweeps=5, **kw)
        else:
            campaign.run_melt_pool_map([100.0], [1.0], L=8, n_sweeps=5, **kw)


def test_grouped_driver_refuses_a_bad_axis(no_context):
    with pytest.raises(ValueError, match="shape_axis"):
        campaign._run_cases_grouped([("x", 2700.0, 1e13)], L=8, n_sweeps=5, impurity_c=0.0, n_seeds=2,
                                    defect_fraction=0.0, device=0, shape_axis=4)


def test_profile_axis_messages_unchanged(no_context):
    for kw, msg in ((dict(profile_axis=4), "run_cet_sublattice: profile_axis must be None, 0, 1 or 2, got 4"),
                    (dict(profile_axis=1, world=2), "run_cet_sublattice: profile_axis needs a whole lattice on one GPU (world = 1)"),
                    (dict(profile_axis=1, checkpoint_every=3),
                     "run_cet_sublattice: profile_axis does not take checkpoint_every or resume_from")):
        with pytest.raises(ValueError) as ei:
            campaign.run_cet_sublattice(L=8, n_sweeps=5, verbose=False, **kw)
        assert str(ei.value) == msg


# -- shape CSV, map shape files, merge and ensemble ----------------------------------------------------------------

def _read(path):
    with open(path) as fh:
        return list(csv.DictReader(fh))


def _hist(rng, nb=12):
    return rng.integers(0, 50, (2, nb)).astype(np.int64)


def test_shape_csv_round_trip(tmp_path):
    rng = np.random.default_rng(1)
    shapes = [(99, _hist(rng)), (199, _hist(rng))]
    campaign._write_shape_csv(shapes, str(tmp_path))
    rows = _read(tmp_path / "grain_shape.csv")
    assert list(rows[0].keys()) == ["Step", "Bin", "Lo", "Hi", "Grains", "Sites"]
    assert len(rows) == 24 and [int(r["Bin"]) for r in rows[:12]] == list(range(11)) + [-1]
    assert (rows[0]["Lo"], rows[0]["Hi"]) == ("0.0", "1.0") and (rows[10]["Lo"], rows[10]["Hi"]) == ("32.0", "inf")
    assert (rows[11]["Lo"], rows[11]["Hi"]) == ("", "")
    assert [float(r["Lo"]) for r in rows[1:11]] == list(_lib.SHAPE_EDGES)
    step, h, edges = campaign.read_shape_csv(str(tmp_path / "grain_shape.csv"))
    assert step == 199 and np.array_equal(h, shapes[1][1]) and edges == _lib.SHAPE_EDGES
    campaign._write_shape_csv([], str(tmp_path / "none"))               # no rows: no file
    assert not os.path.exists(tmp_path / "none" / "grain_shape.csv")


def _synthetic_map(tmp_path, monkeypatch, n_case, n_rep, seed=3):
    monkeypatch.chdir(tmp_path)
    rng = np.random.default_rng(seed)
    lats = campaign._map_lattices([f"m/T{q}" for q in range(n_case)], n_rep)
    for q, r, p in lats:
        os.makedirs(f"outputs/{p}", exist_ok=True)
        campaign._write_shape_csv([(5, _hist(rng) * 0), (9, _hist(rng))], f"outputs/{p}")
    return lats


def _case_row(q):
    return {"T_sub": 2600.0 + q, "NU_DEP": 1e12 * (q + 1), "G": 1.0, "R": 2.0, "G_over_R": 0.5}


def test_map_shape_rows_merge_and_ensemble(tmp_path, monkeypatch):
    n_case, n_rep = 3, 4
    lats = _synthetic_map(tmp_path, monkeypatch, n_case, n_rep)
    axes = ("T_sub", "NU_DEP")
    rows = campaign._map_shape_rows(lats, list(range(len(lats))), _case_row, axes)
    assert list(rows[0].keys()) == ["case", "replica", "T_sub", "NU_DEP", "ColumnarVolumeFraction",
                                    "ColumnarGrainFraction", "ShapedGrains"]
    for (q, r, p), row in zip(lats, rows):
        _s, h, e = campaign.read_shape_csv(f"outputs/{p}/grain_shape.csv")
        s = metrics.grain_shape_summary(h, e)
        assert (row["case"], row["replica"]) == (q, r) and {k: row[k] for k in s} == s
        assert row["ColumnarVolumeFraction"] == h[1, 4:11].sum() / h[1].sum()
    mine = [[l for l in range(len(lats)) if l % 2 == k] for k in range(2)]
    for k in range(2):
        campaign._write_rows(campaign._map_shape_rows(lats, mine[k], _case_row, axes), f"outputs/m/cet_map_shape_rank{k}.csv")
        campaign._write_rows([{"case": lats[l][0], "replica": lats[l][1], **_case_row(lats[l][0]),
                               **{c: 1.0 for c in campaign.ENSEMBLE_COLUMNS}, "CET_Class": "Equiaxed",
                               "CET_Detected": True} for l in mine[k]], f"outputs/m/cet_map_replicas_rank{k}.csv")
    campaign.merge_cet_map("m")
    merged = _read("outputs/m/cet_map_shape.csv")
    assert [(int(r["case"]), int(r["replica"])) for r in merged] == [(q, r) for q, r, _ in lats]
    assert [float(r["ColumnarVolumeFraction"]) for r in merged] == [r["ColumnarVolumeFraction"] for r in rows]
    ens = _read("outputs/m/cet_map_shape_ensemble.csv")
    assert list(ens[0].keys()) == ["case", "T_sub", "NU_DEP", "replicas", "ColumnarVolumeFraction_mean",
                                   "ColumnarVolumeFraction_se", "ColumnarGrainFraction_mean", "ColumnarGrainFraction_se"]
    for q, e in enumerate(ens):
        assert int(e["case"]) == q and int(e["replicas"]) == n_rep
        for col in campaign.SHAPE_FRACTIONS:
            v = np.array([r[col] for r in rows[q * n_rep:(q + 1) * n_rep]])
            assert float(e[f"{col}_mean"]) == pytest.approx(np.mean(v), rel=1e-15)
            assert float(e[f"{col}_se"]) == pytest.approx(np.std(v, ddof=1) / np.sqrt(n_rep), rel=1e-15)
    assert not os.path.exists("outputs/m/cet_map_profile.csv")


def test_shape_ensemble_single_replica():
    e = campaign.shape_ensemble_stats([{"case": 0, "T_sub": 1, "ColumnarVolumeFraction": "0.25",
                                        "ColumnarGrainFraction": 0.5}], ("T_sub",))
    assert e == [{"case": 0, "T_sub": 1, "replicas": 1, "ColumnarVolumeFraction_mean": 0.25,
                  "ColumnarVolumeFraction_se": "", "ColumnarGrainFraction_mean": 0.5, "ColumnarGrainFraction_se": ""}]


def test_merge_without_replicas_writes_no_shape_ensemble(tmp_path, monkeypatch):
    lats = _synthetic_map(tmp_path, monkeypatch, 2, 1)
    campaign._write_rows(campaign._map_shape_rows(lats, [1, 0], _case_row, ("T_sub", "NU_DEP")),
                         "outputs/m/melt_pool_map_shape_rank0.csv")
    campaign.merge_melt_pool_map("m")
    assert [int(r["case"]) for r in _read("outputs/m/melt_pool_map_shape.csv")] == [0, 1]
    assert not os.path.exists("outputs/m/melt_pool_map_shape_ensemble.csv")
    assert not os.path.exists("outputs/m/melt_pool_map.csv")
