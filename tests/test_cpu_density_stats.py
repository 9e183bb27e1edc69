"""CPU tests of density statistics (``density_stats=``): argument checks, the per-member device bytes of an ensemble and
the frames a run selects -- all without CUDA."""
import numpy as np
import pytest

from conftest import REPO


@pytest.mark.parametrize("value,want", [(None, None), (False, None), (True, (1, None)), ({}, (1, None)),
                                        ({"every": 10}, (10, None)), ({"every": 7, "threshold": 2}, (7, 2.0)),
                                        ({"threshold": 0.5}, (1, 0.5)), ({"every": np.int64(3)}, (3, None))])
def test_density_stats_argument_is_normalised(value, want):
    from optimal_crowds_b200 import simulations
    got = simulations.density_stats_spec(value)
    assert got == want
    if got is not None:
        assert type(got[0]) is int and (got[1] is None or type(got[1]) is float)


@pytest.mark.parametrize("value", [{"every": 0}, {"every": -1}, {"every": 1.5}, {"every": True}, {"every": "10"},
                                   {"threshold": float("nan")}, {"threshold": float("inf")}, {"threshold": "1"},
                                   {"threshold": True}, {"every": 1, "thresold": 1.0}, 1, "yes", [1]])
def test_bad_density_stats_arguments_raise_before_any_gpu_work(value, monkeypatch):
    import torch
    from optimal_crowds_b200 import ensemble, simulations
    monkeypatch.chdir(REPO)
    with pytest.raises(ValueError, match="density_stats"):
        simulations.density_stats_spec(value)
    with pytest.raises(ValueError, match="density_stats"):
        ensemble.ensemble("room_test", 1.0, [0, 1], density_stats=value)
    with pytest.raises(ValueError, match="density_stats"):
        simulations.simulation("room_test", 1.0, density_stats=value)
    assert not torch.cuda.is_initialized()


@pytest.mark.parametrize("kw", [dict(band=True), dict(shard_keys=True)])
def test_density_stats_are_refused_for_decomposed_runs(kw, monkeypatch):
    import torch
    from optimal_crowds_b200 import simulations
    monkeypatch.chdir(REPO)
    with pytest.raises(ValueError, match="band=True.*shard_keys=True"):
        simulations.simulation("room_test", 1.0, density_stats=True, **kw)
    assert not torch.cuda.is_initialized()


def test_member_bytes_add_the_accumulators_only_with_stats(monkeypatch):
    import torch
    from optimal_crowds_b200 import _lib, ensemble, synthetic
    monkeypatch.chdir(REPO)
    rooms = ["room_test", "metro_station", synthetic.ensemble_room(n=97, agents=12)]
    configs = [{}, {"dt": 0.01}, {"sigma_convolution": 0.3}]
    base = ensemble.ensemble(rooms, 2.0, [0, 1, 2], configs=configs).member_bytes()
    want = []
    for room, ov in zip(rooms, configs):
        r = room if isinstance(room, dict) else ensemble.simulations._load_room(room)
        Ny, Nx = _lib.grid_shape(r["room_length"], r["room_height"], 0.05)
        keys = {" or ".join(b[5:]) for b in r["initial_boxes"].values()}
        want.append((Ny * Nx, ensemble.field_bytes_per_member(Ny, Nx, 2.0, ov.get("dt", 0.02), len(keys))))
    assert base == [b for _, b in want]                     # unchanged without stats: the same wave plans
    for arg in (None, False):
        assert ensemble.ensemble(rooms, 2.0, [0, 1, 2], configs=configs, density_stats=arg).member_bytes() == base
    for arg, per_node in ((True, 16), ({"every": 10}, 16), ({"every": 10, "threshold": 1.5}, 20)):
        got = ensemble.ensemble(rooms, 2.0, [0, 1, 2], configs=configs, density_stats=arg).member_bytes()
        assert got == [b + per_node * n for n, b in want]   # 2 doubles per node (+ 1 int32 with a threshold)
    assert not torch.cuda.is_initialized()


def _plain_run_frames(T, dt, every):
    """run()'s loop (simulations.py:427-441) step by step, nobody leaving: the simu_steps of its history frames that the
    statistics take"""
    out, time, simu_step = [], 0., 0
    while time < T:
        if simu_step % every == 0:
            out.append(simu_step)
        time += dt
        simu_step += 1
    return out


@pytest.mark.parametrize("T,dt", [(1.0, 0.02), (2.3, 0.025), (0.1, 0.03), (4.0, 0.01), (0.02, 0.02), (1e-3, 0.02)])
@pytest.mark.parametrize("every", [1, 7, 10, 1000])
@pytest.mark.parametrize("recompute_step", [None, 1, 30, 50])
def test_frames_of_a_run_are_those_of_the_plain_loop(T, dt, every, recompute_step):
    from optimal_crowds_b200 import simulations
    got = simulations.density_frame_steps(T, dt, every, recompute_step)
    assert got == _plain_run_frames(T, dt, every)
    assert all(s % every == 0 for s in got) and got[:1] == [0]
