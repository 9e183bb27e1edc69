"""CPU tests of flow statistics (``density_stats=dict(velocity=True)``, ``lines=``): argument checks and refusals, the
per-member device bytes of an ensemble and the counting rule of the measurement lines -- all without CUDA."""
import numpy as np
import pytest

from conftest import REPO
from flow_oracle import line_crossings, orient, run_line_counts


# --------------------------------------------------------------------------------------------- arguments
@pytest.mark.parametrize("value,want", [(True, (1, None, False)), ({"velocity": True}, (1, None, True)),
                                        ({"every": 5, "threshold": 1, "velocity": np.bool_(True)}, (5, 1.0, True)),
                                        ({"velocity": False}, (1, None, False)), (None, None)])
def test_velocity_flag_is_normalised(value, want):
    from optimal_crowds_b200 import simulations
    assert simulations.density_stats_spec(value, with_velocity=True) == want
    if want is not None:   # the two-value form is unchanged
        assert simulations.density_stats_spec(value) == want[:2]


@pytest.mark.parametrize("value", [{"velocity": 1}, {"velocity": "yes"}, {"velocity": None}, {"velocity": [True]},
                                   {"velocity": True, "velocities": True}])
def test_bad_velocity_flags_raise_before_any_gpu_work(value, monkeypatch):
    import torch
    from optimal_crowds_b200 import ensemble, simulations
    monkeypatch.chdir(REPO)
    with pytest.raises(ValueError, match="density_stats"):
        simulations.density_stats_spec(value, with_velocity=True)
    with pytest.raises(ValueError, match="density_stats"):
        ensemble.ensemble("room_test", 1.0, [0, 1], density_stats=value)
    with pytest.raises(ValueError, match="density_stats"):
        simulations.simulation("room_test", 1.0, density_stats=value)
    assert not torch.cuda.is_initialized()


def test_lines_are_normalised():
    from optimal_crowds_b200 import simulations
    assert simulations.lines_spec(None) is None
    names, arr = simulations.lines_spec({"door": (9.5, 2.0, 9.5, 4.0), "mid": np.array([5, 0, 5.0, 6]),
                                         "diag": [0, 0, 1e-9, 0]})
    assert names == ["door", "mid", "diag"]
    assert arr.dtype == np.float64 and arr.shape == (3, 4) and arr.flags.c_contiguous
    assert arr.tolist() == [[9.5, 2.0, 9.5, 4.0], [5.0, 0.0, 5.0, 6.0], [0.0, 0.0, 1e-9, 0.0]]
    many = {f"l{k}": (0, k, 1, k) for k in range(64)}
    assert len(simulations.lines_spec(many)[0]) == 64


_BAD_LINES = [[(0, 0, 1, 1)], (0, 0, 1, 1), {}, {f"l{k}": (0, k, 1, k) for k in range(65)},
              {"a": (0, 0, 1)}, {"a": (0, 0, 1, 1, 2)}, {"a": "0011"}, {"a": (0, 0, "x", 1)}, {"a": (0, 0, True, 1)},
              {"a": (0, float("nan"), 1, 1)}, {"a": (0, 0, float("inf"), 1)}, {"a": (0, 0, 1, -float("inf"))},
              {"a": (2.5, 1.0, 2.5, 1.0)}, {"ok": (0, 0, 1, 0), "a": (3, 3, 3, 3)}, {"a": None}]


@pytest.mark.parametrize("value", _BAD_LINES)
def test_bad_lines_raise_before_any_gpu_work(value, monkeypatch):
    import torch
    from optimal_crowds_b200 import ensemble, simulations
    monkeypatch.chdir(REPO)
    with pytest.raises(ValueError, match="lines"):
        simulations.lines_spec(value)
    with pytest.raises(ValueError, match="lines"):
        ensemble.ensemble("room_test", 1.0, [0, 1], lines=value)
    with pytest.raises(ValueError, match="lines"):
        simulations.simulation("room_test", 1.0, lines=value)
    assert not torch.cuda.is_initialized()


@pytest.mark.parametrize("kw", [dict(band=True), dict(shard_keys=True)])
@pytest.mark.parametrize("opt", [dict(lines={"a": (1, 0, 1, 6)}), dict(density_stats={"velocity": True})])
def test_flow_statistics_are_refused_for_decomposed_runs(kw, opt, monkeypatch):
    import torch
    from optimal_crowds_b200 import simulations
    monkeypatch.chdir(REPO)
    with pytest.raises(ValueError, match="band=True.*shard_keys=True"):
        simulations.simulation("room_test", 1.0, **opt, **kw)
    assert not torch.cuda.is_initialized()


def test_member_bytes_add_velocity_maps_and_line_accumulators(monkeypatch):
    import torch
    from optimal_crowds_b200 import _lib, ensemble, simulations, synthetic
    monkeypatch.chdir(REPO)
    rooms = ["room_test", "metro_station", synthetic.ensemble_room(n=97, agents=12)]
    configs = [{}, {"dt": 0.01}, {"sigma_convolution": 0.3}]
    T = 2.0
    base = ensemble.ensemble(rooms, T, [0, 1, 2], configs=configs).member_bytes()
    info = []
    for room, ov in zip(rooms, configs):
        r = room if isinstance(room, dict) else simulations._load_room(room)
        Ny, Nx = _lib.grid_shape(r["room_length"], r["room_height"], 0.05)
        N = sum(int(b[4] * b[2] * b[3]) for b in r["initial_boxes"].values())
        steps = len(simulations.density_frame_steps(T, ov.get("dt", 0.02), 1))
        info.append((Ny * Nx, N, steps))
    assert all(N > 0 for _, N, _ in info) and info[1][2] == 200 and info[0][2] == 100
    for ds, per_node in (({"velocity": False}, 16), ({"velocity": True}, 40), ({"velocity": True, "threshold": 1}, 44)):
        got = ensemble.ensemble(rooms, T, [0, 1, 2], configs=configs, density_stats=ds).member_bytes()
        assert got == [b + per_node * n for b, (n, _, _) in zip(base, info)], ds
    lines = {"a": (1, 0, 1, 6), "b": (0, 3, 10, 3), "c": (5, 0, 5, 6)}
    got = ensemble.ensemble(rooms, T, [0, 1, 2], configs=configs, lines=lines).member_bytes()
    assert got == [b + 17 * N + 8 * 3 * steps for b, (_, N, steps) in zip(base, info)]   # 17 B/agent, 2 int32/line/step
    both = ensemble.ensemble(rooms, T, [0, 1, 2], configs=configs, lines=lines,
                             density_stats={"velocity": True}).member_bytes()
    assert both == [g + 40 * n for g, (n, _, _) in zip(got, info)]
    assert not torch.cuda.is_initialized()


# --------------------------------------------------------------------------------------------- counting rule
# the line a = (0, 0) -> b = (1, 0): o(a, b, w) = w.y, so "left" is y > 0 and a point with y == 0 is on the right
A_B = [(0.0, 0.0, 1.0, 0.0)]
_CASES = [  # (p, q, expected (to_left, to_right))
    ((0.5, -1.0), (0.5, 1.0), (1, 0)),      # crossing upwards
    ((0.5, 1.0), (0.5, -1.0), (0, 1)),      # and downwards
    ((0.5, 1.0), (0.5, 0.0), (0, 1)),       # a move that ends on the line leaves the left side
    ((0.5, 0.0), (0.5, 1.0), (1, 0)),       # a move from the line to the left enters it
    ((0.5, -1.0), (0.5, 0.0), (0, 0)),      # from the right onto the line: still on the right
    ((0.5, 0.0), (0.5, -1.0), (0, 0)),
    ((0.2, 0.0), (0.8, 0.0), (0, 0)),       # along the line
    ((0.5, 1.0), (0.5, 1.0), (0, 0)),       # zero-length moves, off and on the line
    ((0.5, 0.0), (0.5, 0.0), (0, 0)),
    ((1.0, -1.0), (1.0, 1.0), (1, 0)),      # through endpoint b: o(p, q, b) == 0 is "not left", o(p, q, a) > 0
    ((0.0, -1.0), (0.0, 1.0), (0, 0)),      # through endpoint a: o(p, q, a) == 0 and o(p, q, b) < 0: no crossing
    ((2.0, -1.0), (2.0, 1.0), (0, 0)),      # past the end of the segment
    ((-0.5, 1.0), (1.5, -1.0), (0, 1)),     # a diagonal through the middle
    ((np.nan, -1.0), (0.5, 1.0), (0, 0)),   # NaN positions never cross
    ((0.5, -1.0), (0.5, np.nan), (0, 0)),
    ((0.5, -1.0), (np.nan, np.nan), (0, 0)),
]


@pytest.mark.parametrize("p,q,want", _CASES)
def test_counting_rule_on_hand_built_moves(p, q, want):
    left, right = line_crossings(A_B, [p], [q], [True])
    assert (int(left[0]), int(right[0])) == want
    # an agent that was not inside at the start of the step never counts
    left, right = line_crossings(A_B, [p], [q], [False])
    assert left[0] == right[0] == 0
    # reversing the line swaps the sides (moves touching the line aside)
    if 0.0 not in (p[1], q[1]) and not (np.isnan(p).any() or np.isnan(q).any()) and p[0] not in (0.0, 1.0):
        l2, r2 = line_crossings([(1.0, 0.0, 0.0, 0.0)], [p], [q], [True])
        assert (int(l2[0]), int(r2[0])) == want[::-1]


def test_orientation_is_the_stated_expression():
    rng = np.random.RandomState(0)
    v = rng.uniform(-5, 5, (6, 1000))
    got = orient(*v)
    want = (v[2] - v[0]) * (v[5] - v[1]) - (v[3] - v[1]) * (v[4] - v[0])
    assert np.array_equal(got, want)


def test_counts_of_a_run_follow_inside_and_exit_steps():
    # 3 agents crossing x = 1 (line pointing up: moving +x goes to the right); agent 1 leaves in step 1 (its move in
    # step 1 counts), agent 2 left in step 0 (its later moves do not)
    lines = [(1.0, -5.0, 1.0, 5.0)]
    rows = [np.array([[0.5, 0.0], [0.8, 0.0], [0.9, 0.0]]),
            np.array([[0.9, 0.0], [0.9, 0.0], [1.1, 0.0]]),
            np.array([[1.2, 0.0], [1.3, 0.0], [0.5, 0.0]]),
            np.array([[0.7, 0.0], [0.5, 0.0], [1.5, 0.0]])]
    exit_step = np.array([-1, 1, 0])
    left, right = run_line_counts(lines, rows, exit_step, 3)
    assert left.dtype == np.int32 and left.shape == (3, 1)
    assert right[:, 0].tolist() == [1, 2, 0] and left[:, 0].tolist() == [0, 0, 1]
