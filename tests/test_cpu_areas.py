"""CPU tests of measurement areas (``areas=``): argument checks, refusals, byte counts and the numpy oracle's own
properties.  None of them initialises CUDA."""
import numpy as np
import pytest

from area_oracle import fixed_order_sum, inside, measure

SQUARE = [(1.0, 1.0), (3.0, 1.0), (3.0, 3.0), (1.0, 3.0)]


@pytest.fixture(autouse=True)
def _no_cuda():
    import torch
    yield
    assert not torch.cuda.is_initialized()


def test_areas_spec_accepts_and_flattens():
    from optimal_crowds_b200 import simulations
    assert simulations.areas_spec(None) is None
    tri = np.array([(0, 0), (2, 0), (0, 2)])
    names, verts, offsets = simulations.areas_spec({"sq": SQUARE, "tri": tri, "np": [(np.float32(4), 4), (5, 4),
                                                                                   (np.int64(5), 5)]})
    assert names == ["sq", "tri", "np"]
    assert verts.dtype == np.float64 and verts.shape == (10, 2) and list(offsets) == [0, 4, 7, 10]
    assert np.array_equal(verts[4:7], tri)
    # a concave polygon of 64 vertices, 64 areas, 1024 vertices in all
    t = np.linspace(0, 2 * np.pi, 64, endpoint=False)
    star = np.stack([5 + (2 + np.cos(5 * t)) * np.cos(t), 5 + (2 + np.cos(5 * t)) * np.sin(t)], axis=1)
    spec = {f"a{k}": star + k for k in range(13)}
    spec.update({f"b{k}": SQUARE for k in range(39)})
    spec.update({f"c{k}": tri for k in range(12)})
    names, verts, offsets = simulations.areas_spec(spec)
    assert len(names) == 64 and offsets[-1] == len(verts) == 1024
    assert np.array_equal(np.diff(offsets), [64] * 13 + [4] * 39 + [3] * 12)


@pytest.mark.parametrize("value, match", [
    ([SQUARE], "non-empty dict"),
    ({}, "non-empty dict"),
    ({f"a{k}": SQUARE for k in range(65)}, "at most 64"),
    ({"a": [(0, 0), (1, 0)]}, "3 to 64"),
    ({"a": [(np.cos(t), np.sin(t)) for t in np.linspace(0, 6, 65)]}, "3 to 64"),
    ({"a": [(0, 0), (1, 0), (0, np.nan)]}, "finite"),
    ({"a": [(0, 0), (1, 0), (np.inf, 1)]}, "finite"),
    ({"a": [(0, 0), (1, 0), (2, 0)]}, "zero area"),
    ({"a": [(0, 0), (2, 2), (2, 0), (0, 1)]}, "simple"),                       # a bow tie
    ({"a": [(0, 0), (2, 0), (2, 2), (1, 0), (0, 2)]}, "simple"),               # a vertex on another edge
    ({"a": [(0, 0), (2, 0), (2, 2), (2, 2), (0, 2)]}, "simple"),               # a repeated vertex
    ({"a": [(0, 0), (2, 0), (1, 0), (1, 2)]}, "simple"),                       # an edge folding back
    ({"a": [(0, 0), (3, 0), (3, 3), (1, 1), (2, 1), (0, 3)]}, "simple"),     # crossing edges
    ({"a": "abc"}, "vertices"),
    ({"a": [(0, 0, 1), (1, 0, 1), (0, 1, 1)]}, "vertices"),
    ({"a": [0, 1, 2]}, "vertices"),
    ({"a": [(0, 0), (1, 0), (True, 1)]}, "vertices"),
    ({"a": [(0, 0), (1, 0), ("1", 1)]}, "vertices"),
    ({"a": [(0, 0), (1, 0), None]}, "vertices"),
    ({"a": 3}, "vertices"),
    ({f"a{k}": [(np.cos(t) + k, np.sin(t)) for t in np.linspace(0, 6, 64)] for k in range(17)}, "1024"),
])
def test_bad_areas_are_refused(value, match):
    from optimal_crowds_b200 import simulations
    with pytest.raises(ValueError, match=match):
        simulations.areas_spec(value)


def test_simulations_and_ensembles_refuse_bad_areas_before_any_gpu_work():
    from optimal_crowds_b200 import ensemble, simulations
    with pytest.raises(ValueError, match="simple"):
        simulations.simulation("room_test", 1.0, areas={"a": [(0, 0), (2, 2), (2, 0), (0, 1)]})
    for kw in (dict(band=True), dict(shard_keys=True)):
        with pytest.raises(ValueError, match="areas are not available"):
            simulations.simulation("room_test", 1.0, areas={"a": SQUARE}, **kw)
    with pytest.raises(ValueError, match="zero area"):
        ensemble.ensemble("room_test", 1.0, [1, 2], areas={"a": [(0, 0), (1, 1), (2, 2)]})


def test_member_bytes_count_the_area_accumulator():
    from optimal_crowds_b200 import _lib, ensemble, optimals, simulations
    areas = {"a": SQUARE, "b": [(0, 0), (2, 0), (0, 2)]}
    plain = ensemble.ensemble("room_test", 2.0, [1, 2], configs=[None, {"dt": 0.02}])
    with_areas = ensemble.ensemble("room_test", 2.0, [1, 2], configs=[None, {"dt": 0.02}], areas=areas)
    room = simulations._load_room("room_test")
    N = sum(int(b[4] * b[2] * b[3]) for b in room["initial_boxes"].values())
    dts = [optimals._load_config()["dt"], 0.02]
    for a, b, dt in zip(with_areas.member_bytes(), plain.member_bytes(), dts):
        steps = len(simulations.density_frame_steps(2.0, dt, 1))
        assert a - b == _lib.AreaStats.nbytes(N, 2, 7, steps) == 16 * 7 + 32 * 2 * -(-N // 256) + 28 * 2 * steps
    assert simulations.areas_spec(with_areas.areas) is with_areas.areas                 # members take it as checked


def test_oracle_unit_square_and_boundaries():
    sq = np.array(SQUARE)
    x = np.array([2.0, 0.5, 1.0, 3.0, 2.0, 2.0, 1.0, 3.0, 1.0, 3.0, np.nan, 2.0])
    y = np.array([2.0, 2.0, 2.0, 2.0, 1.0, 3.0, 1.0, 1.0, 3.0, 3.0, 2.0, np.nan])
    got = inside(sq, x, y)
    # the rule puts the left and bottom edges inside, the right and top edges outside (vertices by the same rule)
    assert list(got) == [True, False, True, False, True, False, True, False, False, False, False, False]
    # orientation does not change membership off the edges
    rev = sq[::-1]
    assert list(inside(rev, x[:2], y[:2])) == [True, False]


def test_oracle_concave_polygon_and_horizontal_edges():
    # a U shape: the notch is outside; horizontal edges never toggle on their own
    u = np.array([(0, 0), (3, 0), (3, 3), (2, 3), (2, 1), (1, 1), (1, 3), (0, 3)], dtype=np.float64)
    x = np.array([0.5, 1.5, 2.5, 1.5, 1.5, 1.5, 0.5, 2.0, 0.0])
    y = np.array([2.0, 2.0, 2.0, 0.5, 1.0, 3.0, 0.0, 2.0, 3.0])
    assert list(inside(u, x, y)) == [True, False, True, True, False, False, True, True, False]


def test_oracle_sums_are_the_fixed_order():
    rng = np.random.RandomState(1)
    v = rng.normal(size=600) * 10.0 ** rng.randint(-8, 8, 600)
    s = fixed_order_sum(v)
    assert s == pytest.approx(np.sum(v), rel=1e-9, abs=1e-6)
    assert fixed_order_sum([]) == 0.0 and fixed_order_sum([2.5]) == 2.5
    # all -0.0: the warp-order sum starts from +0.0
    assert np.signbit(fixed_order_sum([-0.0] * 40)) == False  # noqa: E712
    # one warp's butterfly differs from a sequential sum in general; blocks are independent
    assert fixed_order_sum(np.r_[v[:256], np.zeros(256)]) == fixed_order_sum(v[:256])
    m = measure([SQUARE], [2.0, 2.0, 5.0], [2.0, 2.5, 2.0], [3.0, -1.0, 7.0], [4.0, 0.0, 7.0], [1, 0, 1])
    assert list(m["count"]) == [1] and m["speed_sum"][0] == 5.0 and m["vx_sum"][0] == 3.0 and m["vy_sum"][0] == 4.0
