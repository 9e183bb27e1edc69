"""GPU parity of ensembles whose members have different rooms: different grid shapes (odd widths included) and numbers of
target sets.  Every member must equal its stand-alone ``simulation(room, T, config=cfg)`` run seeded with
``np.random.seed(seed)`` bit for bit."""
import contextlib
import io
import json

import numpy as np
import pytest

from conftest import REPO

pytestmark = pytest.mark.gpu

T = 1.3   # (recompute: one re-solve per member at step 50, t = 1.0)


@pytest.fixture()
def in_repo_cwd(monkeypatch):
    monkeypatch.chdir(REPO)


def _odd_room():
    """a 97 x 97 synthetic room (odd Nx: the LDGSTS variant of the step kernel) with 12 agents"""
    from optimal_crowds_b200 import synthetic
    room = synthetic.ensemble_room(n=97, agents=12)
    room["initial_boxes"]["box"][0] = 1.6
    room["initial_boxes"]["box"][2:4] = [2.0, 2.0]
    room["initial_boxes"]["box"][4] = 12.5 / 4.0
    return room


def _rooms():
    return ["room_test", "exit_opposite", "metro_station", "slalom", _odd_room()]


SEEDS = [3, 4, 5, 6, 7]
CONFIGS = [{"hjb_params": {"sigma": 0.25}}, {"dt": 0.025}, {}, {"recompute_frequency": 30, "hjb_params": {"g": -0.02}},
           {"v_max": 1.5, "hjb_params": {"mu": 4}}]
_ALONE = {}


def _alone(room, recompute, seed, ov=None, chunk_rows=0):
    key = (json.dumps(room, sort_keys=True) if isinstance(room, dict) else room, recompute, seed,
           json.dumps(ov, sort_keys=True), chunk_rows)
    if key not in _ALONE:
        from optimal_crowds_b200 import simulations
        np.random.seed(seed)
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(room, T, recompute=recompute, record=False, config=ov, chunk_rows=chunk_rows)
            simu.run()
        simu._sync_host()
        _ALONE[key] = simu
    return _ALONE[key]


def _assert_member_is(r, one):
    assert r["steps"] == one.simu_step and r["inside"] == one.inside and r["evac_time"] == one.time
    assert np.array_equal(r["exit_order"], np.array(one._exit_order, dtype=np.int64))
    assert np.array_equal(r["final"], one._h_now)
    assert np.array_equal(r["times"], one._h_timev)
    assert set(r["hjb"]) == set(one.targets)
    for k, o in one.targets.items():
        assert r["hjb"][k]["nfev"] == o.last_stats["nfev"], k


@pytest.mark.parametrize("batched", [True, False], ids=["batched_steps", "member_steps"])
@pytest.mark.parametrize("recompute", [True, False], ids=["recompute", "no_recompute"])
def test_members_of_different_rooms_equal_standalone_runs(recompute, batched, in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    rooms = _rooms()
    ens = ensemble.ensemble(rooms, T, SEEDS, recompute=recompute, batched_steps=batched)
    res = ens.run()
    assert sorted(res) == list(range(len(rooms)))
    shapes = set()
    for i, (room, seed) in enumerate(zip(rooms, SEEDS)):
        one = _alone(room, recompute, seed)
        _assert_member_is(res[i], one)
        shapes.add((one.Ny, one.Nx))
    assert len(shapes) == 4 and any(nx % 2 for _, nx in shapes)
    # one solve call per wave and per re-solve step, over the fields of every member and target set
    assert ens.stats["hjb_calls"] == (2 if recompute else 1)


def test_members_of_different_rooms_with_their_own_config(in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    rooms = _rooms()
    res = ensemble.ensemble(rooms, T, SEEDS, recompute=True, configs=CONFIGS).run()
    for i, (room, seed, ov) in enumerate(zip(rooms, SEEDS, CONFIGS)):
        one = _alone(room, True, seed, ov)
        _assert_member_is(res[i], one)
        assert res[i]["config"] == one._config


def test_sharded_one_member_waves_equal_the_one_batch_run(in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    rooms = _rooms()
    whole = ensemble.ensemble(rooms, T, SEEDS, recompute=True).run()
    parts = {}
    for rank in range(2):
        e = ensemble.ensemble(rooms, T, SEEDS, recompute=True, rank=rank, world=2, max_wave=1)
        parts.update(e.run(gather=False))
        assert e.stats["waves"] == len(e.mine)
    assert sorted(parts) == sorted(whole)
    for i in whole:
        for k in ("steps", "inside", "evac_time"):
            assert parts[i][k] == whole[i][k]
        for k in ("final", "times", "exit_order"):
            assert np.array_equal(parts[i][k], whole[i][k])


def test_wave_chunking_is_planned_per_shape(in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    rooms = _rooms() + ["room_test"]
    seeds = SEEDS + [8]
    ens = ensemble.ensemble(rooms, T, seeds, chunk_rows="wave")
    res = ens.run()
    assert res[0]["chunk_rows"] == res[5]["chunk_rows"] > 0
    for i in (0, 3, 4):
        one = _alone(rooms[i], False, seeds[i], chunk_rows=res[i]["chunk_rows"])
        _assert_member_is(res[i], one)
