"""Host logic of the replica ensembles that needs no device: the sparse initial lattice (_host.initial_nuclei) against
the dense initialize_lattice + introduce_defects pair and the oracle, the argument checks of cetkmc.init_group that run
before the library is reached, the ensemble statistics, and which lattice every (case, replica) of a map is."""
import csv
import ctypes as C
import os

import numpy as np
import pytest

from cetkmc import _host, _lib, campaign
from cetkmc._config import constants as K


def _densify(nuc, L):
    site, byte, theta, phi, row = nuc
    st, df = np.zeros(L ** 3, np.int64), np.zeros(L ** 3, np.int64)
    th, ph = np.zeros(L ** 3), np.zeros(L ** 3)
    st[site], df[site], th[site], ph[site] = byte & 15, byte >> 4, theta, phi
    T = np.broadcast_to(row, (L, L, L))
    return [a.reshape(L, L, L) for a in (st, th, ph)] + [T, df.reshape(L, L, L)]


def _same_stream(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


CASES = [(L, n, seed, c) for L in (1, 2, 9, 30, 64) for n in (0, 1, 20, L * L) if n <= L * L
         for seed, c in ((42, 0.0), (7, 0.1), (1234, 1.0 - K.IMPURITY_RE), (43, 0.1))]


@pytest.mark.parametrize("L,n_seeds,seed,impurity_c", CASES)
def test_initial_nuclei_is_the_dense_pair_in_sparse_form(L, n_seeds, seed, impurity_c):
    T_sub = 2750.0
    state, theta, phi, T, atom_type = _host.initialize_lattice(L, n_seeds, T_sub, random_seed=seed, impurity_c=impurity_c)
    mask, _ = _host.introduce_defects(state, atom_type, T, apply_to_state=False)
    dense_rng = np.random.get_state()
    np.random.seed(999)                                        # initial_nuclei must reseed
    nuc = _host.initial_nuclei(L, n_seeds, T_sub, seed, impurity_c)
    assert _same_stream(np.random.get_state(), dense_rng)
    site, byte, th, ph, row = nuc
    assert (site.dtype, byte.dtype, th.dtype, ph.dtype, row.dtype) == (np.int64, np.uint8, np.float64, np.float64,
                                                                        np.float64)
    assert len(site) == n_seeds and row.shape == (L,)
    st, th_d, ph_d, T_d, df = _densify(nuc, L)
    np.testing.assert_array_equal(st, state)
    np.testing.assert_array_equal(st, atom_type)
    assert np.array_equal(th_d, theta) and np.array_equal(ph_d, phi)
    assert np.array_equal(T_d, T) and np.array_equal(df, mask)
    assert np.all(site % L == 0) and len(set(site.tolist())) == len(site)


def test_initial_nuclei_draws_defects_in_site_order():
    # every nucleus carbon: the defect draws go to the nuclei in C order, not in draw order
    L, n = 12, 144
    nuc = _host.initial_nuclei(L, n, 3600.0, 5, 1.0 - K.IMPURITY_RE)
    st, _, _, T, at = _host.initialize_lattice(L, n, 3600.0, random_seed=5, impurity_c=1.0 - K.IMPURITY_RE)
    mask, _ = _host.introduce_defects(st, at, T)
    assert not np.all(np.diff(nuc[0]) > 0)                     # draw order is not site order here
    assert 0 < int(mask.sum()) < int((at == 3).sum())
    np.testing.assert_array_equal(_densify(nuc, L)[4], mask)


def test_initial_nuclei_matches_the_oracle(oracle):
    for L, n, seed, c in ((9, 20, 42, 0.1), (30, 20, 3, 0.5), (64, 200, 11, 0.0)):
        o = oracle.initialize_lattice(L, n_seeds=n, T_sub=2800.0, random_seed=seed, impurity_c=c)
        d = _densify(_host.initial_nuclei(L, n, 2800.0, seed, c), L)
        for a, b in zip(d[:4], o[:4]):
            assert np.array_equal(a, b)


def test_initial_nuclei_refuses_more_nuclei_than_plane_sites():
    with pytest.raises(ValueError) as dense:
        _host.initialize_lattice(3, 10, 2800.0)
    with pytest.raises(ValueError) as sparse:
        _host.initial_nuclei(3, 10, 2800.0, 42, 0.0)
    assert str(sparse.value) == str(dense.value)


# -- the binding ------------------------------------------------------------------------------------------------------

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


def test_init_group_checks_its_arguments_before_the_library(no_library, fake_ctxs):
    a, b = fake_ctxs(2)
    good = _host.initial_nuclei(8, 5, 2800.0, 42, 0.1)
    with pytest.raises(ValueError, match="nucleus sets"):
        _lib.init_group([a, b], [good])
    with pytest.raises(TypeError):
        _lib.init_group([object()], [good])
    with pytest.raises(ValueError, match="site, byte, theta, phi, T_row"):
        _lib.init_group([a], [good[:4]])
    for i, bad in ((0, good[0].astype(np.int32)), (1, good[1].astype(np.int64)), (2, good[2].astype(np.float32)),
                   (4, list(good[4])), (3, np.zeros((5, 1)))):
        nu = list(good)
        nu[i] = bad
        with pytest.raises(TypeError):
            _lib.init_group([a], [tuple(nu)])
    nu = list(good)
    nu[3] = good[3][:4].copy()
    with pytest.raises(ValueError, match="differ in length"):
        _lib.init_group([a], [tuple(nu)])
    nu = list(good)
    nu[4] = np.zeros(9)
    with pytest.raises(ValueError, match="T_row"):
        _lib.init_group([a], [tuple(nu)])


def test_init_desc_layout():
    assert C.sizeof(_lib.InitDesc) == 48


# -- ensemble statistics ----------------------------------------------------------------------------------------------

def _rep_row(case, rep, ar, eq, cls, det, **kw):
    r = {"case": case, "replica": rep, "T_sub": 2800.0, "NU_DEP": 1e13, "G": 1.5, "R": 2.5, "G_over_R": 0.6,
         "Step": 400, "Time": 1.0, "AspectRatio": ar, "EquiaxedFraction": eq, "GrainCount": 10 + rep,
         "AvgGrainSize": 3.0 * (rep + 1), "NucleationCount": 7 * rep, "CET_Class": cls, "CET_Detected": det}
    r.update(kw)
    return r


def test_ensemble_stats_against_numpy():
    rng = np.random.default_rng(3)
    ar, eq = rng.uniform(0.5, 3, 5), rng.uniform(0, 1, 5)
    cls = ["Equiaxed", "Columnar", "Equiaxed", "Equiaxed", "Columnar"]
    rows = [_rep_row(1, r, ar[r], eq[r], cls[r], r % 2 == 0, Step=str(400 - r)) for r in range(5)]
    rows = [{k: str(v) for k, v in r.items()} for r in rows[::-1]]          # as read back from a CSV, any order
    (e,) = campaign.ensemble_stats(rows, ("T_sub", "NU_DEP"))
    assert list(e)[:7] == ["case", "T_sub", "NU_DEP", "G", "R", "G_over_R", "replicas"]
    assert e["case"] == 1 and e["replicas"] == 5 and e["T_sub"] == "2800.0"
    for col, v in (("AspectRatio", ar), ("EquiaxedFraction", eq), ("GrainCount", 10 + np.arange(5.0)),
                   ("Step", 400 - np.arange(5.0)), ("NucleationCount", 7 * np.arange(5.0))):
        assert e[f"{col}_mean"] == pytest.approx(np.mean(v), rel=1e-15)
        assert e[f"{col}_se"] == pytest.approx(np.std(v, ddof=1) / np.sqrt(5), rel=1e-13)
    assert e["p_equiaxed"] == 0.6 and e["p_equiaxed_se"] == pytest.approx(np.sqrt(0.6 * 0.4 / 5))
    assert e["p_cet_detected"] == 0.6
    assert list(e)[-3:] == ["p_equiaxed", "p_equiaxed_se", "p_cet_detected"]


def test_ensemble_stats_edge_cases():
    one = campaign.ensemble_stats([_rep_row(0, 0, 1.25, 0.5, "Columnar", False)], ("T_sub", "NU_DEP"))[0]
    assert one["replicas"] == 1 and one["AspectRatio_mean"] == 1.25
    assert all(one[f"{c}_se"] == "" for c in campaign.ENSEMBLE_COLUMNS)
    assert one["p_equiaxed"] == 0.0 and one["p_equiaxed_se"] == 0.0 and one["p_cet_detected"] == 0.0
    same = campaign.ensemble_stats([_rep_row(2, r, 2.0, 0.25, "Equiaxed", True, GrainCount=4, AvgGrainSize=1.0,
                                             NucleationCount=3) for r in range(4)], ("T_sub", "NU_DEP"))[0]
    assert same["AspectRatio_mean"] == 2.0 and same["AspectRatio_se"] == 0.0 and same["GrainCount_se"] == 0.0
    assert same["p_equiaxed"] == 1.0 and same["p_equiaxed_se"] == 0.0 and same["p_cet_detected"] == 1.0
    two = campaign.ensemble_stats([_rep_row(q, r, 1.0, 0.0, "Columnar", False) for q in (3, 0) for r in range(2)],
                                  ("T_sub", "NU_DEP"))
    assert [e["case"] for e in two] == [0, 3] and [e["replicas"] for e in two] == [2, 2]


# -- lattices of a map with replicas ----------------------------------------------------------------------------------

def test_map_lattices_and_replica_keywords():
    lats = campaign._map_lattices(["m/a", "m/b"], 3)
    assert lats == [(0, 0, "m/a"), (0, 1, "m/a/rep1"), (0, 2, "m/a/rep2"), (1, 0, "m/b"), (1, 1, "m/b/rep1"),
                    (1, 2, "m/b/rep2")]
    assert campaign._map_lattices(["m/a"], 1) == [(0, 0, "m/a")]
    kw = dict(metrics_every=5)
    assert campaign._replica_kw(kw, None, 0) is kw
    assert campaign._replica_kw(kw, 3, 2) == dict(metrics_every=5, seed=K.RANDOM_SEED + 2, init_seed=44)
    assert campaign._replica_kw(dict(seed=100), 3, 1) == dict(seed=101, init_seed=43)


def _fake_metrics(prefix, step, cls="Columnar"):
    os.makedirs(f"outputs/{prefix}", exist_ok=True)
    with open(f"outputs/{prefix}/metrics.csv", "w", newline="") as fh:
        w = csv.writer(fh)
        w.writerow(["Step", "Time", "AspectRatio", "EquiaxedFraction", "GrainCount", "AvgGrainSize", "NucleationCount",
                    "CET_Class", "CET_Detected"])
        w.writerow([step, 1e-3, 1.0 + step / 100, 0.5, 3, 2.0, step, cls, cls == "Equiaxed"])


def _fake_sublattice(calls):
    def run(output_prefix=None, seed=None, init_seed=None, **kw):
        calls.append((output_prefix, seed, init_seed, kw.get("device")))
        _fake_metrics(output_prefix, 10 * (0 if seed is None else seed) % 97, "Equiaxed" if (seed or 0) % 2 else "Columnar")
    return run


@pytest.mark.parametrize("driver", ["gr", "melt"])
def test_replica_runs_are_run_cet_sublattice_with_shifted_seeds(tmp_path, monkeypatch, no_library, driver):
    monkeypatch.chdir(tmp_path)
    calls = []
    monkeypatch.setattr(campaign, "run_cet_sublattice", _fake_sublattice(calls))
    if driver == "gr":
        rows, ens = campaign.run_gr_sweep([2700.0, 2900.0], [1e13], L=8, n_sweeps=5, output_root="m", replicas=3, seed=10,
                                          devices=[0, 1])
        name, prefixes, axes = "cet_map", ["m/T2700_R1e+13", "m/T2900_R1e+13"], ("T_sub", "NU_DEP")
    else:
        rows, ens = campaign.run_melt_pool_map([100.0, 200.0], [1.0], L=8, n_sweeps=5, output_root="m", replicas=3,
                                               seed=10, devices=[0, 1])
        name, prefixes, axes = "melt_pool_map", ["m/P100_V1", "m/P200_V1"], ("power", "speed", "T_sub", "NU_DEP")
    want = [(p if r == 0 else f"{p}/rep{r}", 10 + r, 42 + r, l % 2)
            for l, (p, r) in enumerate((p, r) for p in prefixes for r in range(3))]
    assert calls == want
    assert [r["case"] for r in rows] == [0, 1] and [r["Step"] for r in rows] == ["3", "3"]
    with open(f"outputs/m/{name}_replicas_rank0.csv") as fh:
        reps = list(csv.DictReader(fh))
    assert [(int(r["case"]), int(r["replica"])) for r in reps] == [(q, r) for q in range(2) for r in range(3)]
    assert [int(r["Step"]) for r in reps] == [100 % 97, 110 % 97, 120 % 97] * 2
    assert ens[0]["replicas"] == 3 and ens[0]["p_equiaxed"] == pytest.approx(1 / 3)
    merge = campaign.merge_cet_map if driver == "gr" else campaign.merge_melt_pool_map
    merged = merge("m")
    assert [r["case"] for r in merged] == ["0", "1"]
    with open(f"outputs/m/{name}_ensemble.csv") as fh:
        ens_file = list(csv.DictReader(fh))
    assert [{k: str(v) for k, v in e.items()} for e in ens] == ens_file
    assert sorted(os.listdir("outputs/m/plot_cet/outputs")) == ["impurity_c_0", "impurity_c_1"]


def test_replicas_none_writes_no_replica_files(tmp_path, monkeypatch, no_library):
    monkeypatch.chdir(tmp_path)
    calls = []
    monkeypatch.setattr(campaign, "run_cet_sublattice", _fake_sublattice(calls))
    rows = campaign.run_gr_sweep([2700.0], [1e13, 2e13], L=8, n_sweeps=5, output_root="m")
    assert isinstance(rows, list) and [c[1:3] for c in calls] == [(None, None), (None, None)]
    assert sorted(f for f in os.listdir("outputs/m") if f.endswith(".csv")) == ["cet_map_rank0.csv"]
    campaign.merge_cet_map("m")
    assert not os.path.exists("outputs/m/cet_map_ensemble.csv")


def test_batched_replicas_pass_groups_with_their_replica_numbers(tmp_path, monkeypatch, no_library):
    monkeypatch.chdir(tmp_path)
    groups = []

    def grouped(cases, **kw):
        groups.append(([p for p, _t, _r in cases], kw["replicas"], kw.get("lasers")))
        for p, _t, _r in cases:
            _fake_metrics(p, 3)
    monkeypatch.setattr(campaign, "_run_cases_grouped", grouped)
    campaign.run_melt_pool_map([10.0, 20.0], [1.0], L=8, n_sweeps=5, output_root="m", batch=4, replicas=3)
    assert [g[0] for g in groups] == [["m/P10_V1", "m/P10_V1/rep1", "m/P10_V1/rep2", "m/P20_V1"],
                                      ["m/P20_V1/rep1", "m/P20_V1/rep2"]]
    assert [g[1] for g in groups] == [[0, 1, 2, 0], [1, 2]]
    assert [[d["power"] for d in g[2]] for g in groups] == [[10.0, 10.0, 10.0, 20.0], [20.0, 20.0]]
    groups.clear()
    campaign.run_gr_sweep([2700.0], [1e13], L=8, n_sweeps=5, output_root="g", batch=2, replicas=2)
    assert groups == [(["g/T2700_R1e+13", "g/T2700_R1e+13/rep1"], [0, 1], None)]


def test_replica_partition_over_ranks():
    # 3 cases x 2 replicas = 6 lattices; rank 1 of 2 runs lattices 1, 3, 5 = (0, 1), (1, 1), (2, 1)
    assert campaign.gr_partition(6, 1, 2, [0]) == [(0, [1]), (0, [3]), (0, [5])]
    assert campaign.gr_partition(6, 0, 1, [0], batch=4) == [(0, [0, 1, 2, 3]), (0, [4, 5])]


@pytest.mark.parametrize("driver", ["gr", "melt"])
@pytest.mark.parametrize("bad", [dict(replicas=0), dict(replicas=-2), dict(replicas=2, lattice=(1,)),
                                 dict(replicas=2, resume_from="ck"), dict(replicas=2, checkpoint_every=3),
                                 dict(replicas=2, batch=2, checkpoint_every=3)])
def test_replicas_refusals(tmp_path, monkeypatch, no_library, driver, bad):
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(campaign, "run_cet_sublattice", lambda **kw: pytest.fail("a lattice ran"))
    monkeypatch.setattr(campaign, "_run_cases_grouped", lambda *a, **kw: pytest.fail("a group ran"))
    with pytest.raises(ValueError):
        if driver == "gr":
            campaign.run_gr_sweep([2700.0], [1e13], L=8, n_sweeps=5, **bad)
        else:
            campaign.run_melt_pool_map([100.0], [1.0], L=8, n_sweeps=5, **bad)
