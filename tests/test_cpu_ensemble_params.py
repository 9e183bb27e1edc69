"""CPU tests of per-member configurations: the config.json override merge, the ensemble's validation of its members'
configurations (before any GPU work) and wave planning from per-member byte counts."""
import copy
import json
import os

import pytest

from conftest import REPO


@pytest.fixture()
def base():
    with open(os.path.join(REPO, "optimal_crowds_b200", "config.json")) as f:
        return json.load(f)


def test_nested_partial_override_keeps_the_other_keys(base):
    from optimal_crowds_b200.optimals import _merge_config
    m = _merge_config(base, {"dt": 0.01, "hjb_params": {"g": -0.02}})
    assert m["dt"] == 0.01 and m["hjb_params"]["g"] == -0.02
    for k, v in base["hjb_params"].items():
        if k != "g":
            assert m["hjb_params"][k] == v
    for k, v in base.items():
        if k not in ("dt", "hjb_params"):
            assert m[k] == v


def test_merge_does_not_mutate_the_base(base):
    from optimal_crowds_b200.optimals import _merge_config
    before = copy.deepcopy(base)
    m = _merge_config(base, {"v_max": 3, "hjb_params": {"sigma": 0.3, "mu": 2}})
    assert base == before
    m["hjb_params"]["g"] = 1.0
    assert base == before


@pytest.mark.parametrize("ov,name", [({"gird_step": 0.1}, "gird_step"), ({"hjb_params": {"sgima": 0.3}}, "sgima")])
def test_unknown_keys_raise(base, ov, name):
    from optimal_crowds_b200.optimals import _merge_config
    with pytest.raises(KeyError, match=name):
        _merge_config(base, ov)


def test_empty_override_is_the_file(base):
    from optimal_crowds_b200.optimals import _merge_config, _load_config
    assert _merge_config(base, {}) == base
    assert _merge_config(base, None) == base
    assert _load_config() == base


def test_ensemble_rejects_bad_configs_before_any_gpu_work(monkeypatch):
    """wrong number of configurations, unknown keys and mixed grid steps are caught by the constructor"""
    import torch
    from optimal_crowds_b200 import ensemble
    monkeypatch.chdir(REPO)
    with pytest.raises(ValueError, match="one configuration per seed"):
        ensemble.ensemble("room_test", 1.0, [1, 2, 3], configs=[{}, {}])
    with pytest.raises(ValueError, match="grid_step"):
        ensemble.ensemble("room_test", 1.0, [1, 2], configs=[{}, {"grid_step": 0.1}])
    with pytest.raises(KeyError, match="recompute_freq"):
        ensemble.ensemble("room_test", 1.0, [1, 2], configs=[{}, {"recompute_freq": 10}])
    # different values of every other key are accepted, and the effective configurations are kept per member
    e = ensemble.ensemble("room_test", 1.0, [1, 2, 3], configs=[{}, {"dt": 0.01, "recompute_frequency": 20},
                                                                 {"hjb_params": {"g": -0.05}}])
    assert e.configs[1]["dt"] == 0.01 and e.configs[2]["hjb_params"]["g"] == -0.05 and e.configs[0]["dt"] == 0.02
    assert not torch.cuda.is_initialized()


def _old_plan_waves(members, bytes_per_member, budget_bytes, max_wave=256):
    per = max(1, min(max_wave, budget_bytes // max(bytes_per_member, 1)))
    return [members[i:i + per] for i in range(0, len(members), per)]


def test_wave_planning_with_per_member_bytes():
    import numpy as np
    from optimal_crowds_b200.ensemble import plan_waves
    rng = np.random.RandomState(0)
    for trial in range(200):
        n = int(rng.randint(0, 40))
        members = list(rng.permutation(1000)[:n])
        per = [int(b) for b in rng.randint(1, 100, size=n)]
        budget = int(rng.randint(1, 400))
        max_wave = int(rng.randint(1, 12))
        waves = plan_waves(members, per, budget, max_wave)
        assert [m for w in waves for m in w] == members                 # order preserved, every member once
        cost = dict(zip(members, per))
        for w in waves:
            assert 1 <= len(w) <= max_wave
            assert len(w) == 1 or sum(cost[m] for m in w) <= budget
        # greedy: a wave closes only when the next member would not fit
        for w, nxt in zip(waves, waves[1:]):
            assert len(w) == max_wave or sum(cost[m] for m in w) + cost[nxt[0]] > budget
    # a member larger than the budget gets a wave of its own
    assert plan_waves([1, 2, 3], [5, 50, 5], 10) == [[1], [2], [3]]
    assert plan_waves([1, 2, 3], [5, 5, 50], 10) == [[1, 2], [3]]
    with pytest.raises(ValueError):
        plan_waves([1, 2], [5], 10)


def test_wave_planning_integer_form_is_unchanged():
    from optimal_crowds_b200.ensemble import field_bytes_per_member, plan_waves
    cases = [(list(range(128)), field_bytes_per_member(512, 512, 20.0, 0.02), int(140e9), 256),
             ([1, 2, 3], field_bytes_per_member(512, 512, 20.0, 0.02), 10, 256), (list(range(50)), 7, 100, 4),
             (list(range(50)), 0, 3, 256), (list(range(9)), 10, 0, 256), (list(range(9)), 10, -5, 256), ([], 10, 100, 256),
             (list(range(33)), 3, 10 ** 6, 8)]
    for members, b, budget, mw in cases:
        assert plan_waves(members, b, budget, mw) == _old_plan_waves(members, b, budget, mw)
