"""Host logic of grouped sweeps that needs no device: which cases of a G-R sweep run where and together,
the arguments the batched driver refuses, and the argument checks of cetkmc.sweep_run_group that run before
the library is called."""
import pytest

from cetkmc import _lib, campaign


def test_partition_unbatched_is_one_case_per_entry():
    assert campaign.gr_partition(5, 0, 1, [0]) == [(0, [0]), (0, [1]), (0, [2]), (0, [3]), (0, [4])]
    # rank 1 of 2 runs the odd cases; one process over two devices alternates them
    assert campaign.gr_partition(6, 1, 2, [0]) == [(0, [1]), (0, [3]), (0, [5])]
    assert campaign.gr_partition(4, 0, 1, [0, 1]) == [(0, [0]), (1, [1]), (0, [2]), (1, [3])]


def test_partition_batched_groups_cases_of_one_device_in_order():
    assert campaign.gr_partition(7, 0, 1, [0], batch=3) == [(0, [0, 1, 2]), (0, [3, 4, 5]), (0, [6])]
    assert campaign.gr_partition(8, 0, 1, [0, 1], batch=16) == [(0, [0, 2, 4, 6]), (1, [1, 3, 5, 7])]
    assert campaign.gr_partition(16, 3, 8, [3], batch=16) == [(3, [3, 11])]
    # every case of the rank appears exactly once, whatever the batch
    for batch in (1, 2, 5, 64):
        parts = campaign.gr_partition(37, 2, 3, [0, 1, 2], batch=batch)
        got = sorted(q for _d, qs in parts for q in qs)
        assert got == list(range(2, 37, 3))
        assert all(1 <= len(qs) <= batch for _d, qs in parts)


@pytest.mark.parametrize("batch", [0, -1, _lib.GROUP_MAX + 1])
def test_partition_rejects_a_bad_batch(batch):
    with pytest.raises(ValueError):
        campaign.gr_partition(4, 0, 1, [0], batch=batch)


@pytest.mark.parametrize("kw", [dict(laser=dict(power=100.0)), dict(checkpoint_every=1), dict(resume_from="x"),
                                dict(lattice=(1, 2, 3, 4, 5))])
def test_batched_driver_refuses_single_lattice_features(kw, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    with pytest.raises(ValueError):
        campaign.run_gr_sweep([2800.0], [2e13], L=8, n_sweeps=3, batch=2, **kw)


def test_batched_driver_refuses_an_unknown_mask_stream(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    with pytest.raises(ValueError):
        campaign.run_gr_sweep([2800.0], [2e13], L=8, n_sweeps=3, batch=2, mask_stream="host")


def test_sweep_run_group_checks_list_lengths_before_the_library(monkeypatch):
    def no_library():
        raise AssertionError("the library must not be reached")
    monkeypatch.setattr(_lib, "lib", no_library)
    sp = _lib.SweepParams()
    with pytest.raises(ValueError):
        _lib.sweep_run_group([object(), object()], 3, [sp])
    with pytest.raises(ValueError):
        _lib.sweep_run_group([object()], 3, [sp], [_lib.ThermalParams(), _lib.ThermalParams()])
    with pytest.raises(TypeError):
        _lib.sweep_run_group([object()], 3, [sp], None)
