"""CPU tests of the Voronoi maps (``voronoi_maps=``): argument checks, refusals, byte counts, frame selection and the
Python oracle's own properties.  None of them initialises CUDA."""
import numpy as np
import pytest

from voronoi_oracle import ring
from vormap_oracle import add, empty, frame, owners


@pytest.fixture(autouse=True)
def _no_cuda():
    import torch
    yield
    assert not torch.cuda.is_initialized()


@pytest.mark.parametrize("value, match", [
    ("yes", "expected True"),
    ([1], "expected True"),
    ({"step": 1}, "unknown keys"),
    ({"every": 0}, "every"),
    ({"every": -2}, "every"),
    ({"every": 1.5}, "every"),
    ({"every": 2.0}, "every"),
    ({"every": True}, "every"),
    ({"every": "2"}, "every"),
    ({"cutoff": 0}, "cutoff"),
    ({"cutoff": -1.0}, "cutoff"),
    ({"cutoff": 100.5}, "cutoff"),
    ({"cutoff": float("nan")}, "cutoff"),
    ({"cutoff": float("inf")}, "cutoff"),
    ({"cutoff": True}, "cutoff"),
    ({"cutoff": "1"}, "cutoff"),
    ({"edges": 3}, "edges"),
    ({"edges": 33}, "edges"),
    ({"edges": 12.0}, "edges"),
    ({"edges": False}, "edges"),
])
def test_bad_voronoi_maps_arguments_are_refused(value, match):
    from optimal_crowds_b200 import simulations
    with pytest.raises(ValueError, match="voronoi_maps: .*" + match):
        simulations.voronoi_maps_spec(value)


def test_voronoi_maps_spec_defaults():
    from optimal_crowds_b200 import simulations
    assert simulations.voronoi_maps_spec(None) is None and simulations.voronoi_maps_spec(False) is None
    assert simulations.voronoi_maps_spec(True) == (1, 1.0, 12)
    assert simulations.voronoi_maps_spec({"every": np.int32(3), "cutoff": 100, "edges": np.int64(4)}) == (3, 100.0, 4)
    spec = simulations.voronoi_maps_spec({"edges": 32})
    assert spec == (1, 1.0, 32) and simulations.voronoi_maps_spec(spec) is spec
    # the voronoi option keeps its own messages
    with pytest.raises(ValueError, match="^voronoi: cutoff"):
        simulations.voronoi_spec({"cutoff": 0})


def test_simulations_and_ensembles_refuse_voronoi_maps_before_any_gpu_work():
    from optimal_crowds_b200 import ensemble, simulations
    for kw in (dict(band=True), dict(shard_keys=True)):
        with pytest.raises(ValueError, match="voronoi_maps is not available"):
            simulations.simulation("room_test", 1.0, voronoi_maps=True, **kw)
    with pytest.raises(ValueError, match="every"):
        simulations.simulation("room_test", 1.0, voronoi_maps={"every": 0})
    with pytest.raises(ValueError, match="cutoff"):
        ensemble.ensemble("room_test", 1.0, [1, 2], voronoi_maps={"cutoff": 0})
    with pytest.raises(ValueError, match="edges"):
        ensemble.ensemble("room_test", 1.0, [1, 2], voronoi_maps={"edges": 40})


def test_member_bytes_count_the_map_accumulators():
    from optimal_crowds_b200 import _lib, ensemble, simulations
    rooms = ["room_test", "metro_station"]
    kw = dict(configs=[None, {"dt": 0.025}])
    plain = ensemble.ensemble(rooms, 2.0, [1, 2], **kw)
    with_m = ensemble.ensemble(rooms, 2.0, [1, 2], voronoi_maps=dict(every=4, cutoff=0.5, edges=16), **kw)
    for a, b, name in zip(with_m.member_bytes(), plain.member_bytes(), rooms):
        room = simulations._load_room(name)
        L, H = room["room_length"], room["room_height"]
        Ny, Nx = _lib.grid_shape(L, H, 0.05)
        N = sum(int(b_[4] * b_[2] * b_[3]) for b_ in room["initial_boxes"].values())
        bins = _lib.voronoi_bins(L, 0.5) * _lib.voronoi_bins(H, 0.5)
        assert a - b == _lib.VoronoiMaps.nbytes(Ny, Nx, N, 16, bins) == (
            (5 * 8 + 4) * Ny * Nx + 16 * 16 + 8 * (bins + 1) + 24 * N)
    # without the option nothing changes
    assert plain.member_bytes() == ensemble.ensemble(rooms, 2.0, [1, 2], **kw).member_bytes()


@pytest.mark.parametrize("every", [1, 2, 7])
@pytest.mark.parametrize("recompute", [None, 50])
def test_frames_of_a_run_cut_into_blocks(every, recompute):
    """the frames a run takes block by block (VoronoiMaps.count over run()'s advance() blocks) are the plain loop's
    selection, density_frame_steps"""
    from optimal_crowds_b200 import _lib, simulations
    T, dt = 2.3, 0.02
    acc = _lib.VoronoiMaps.__new__(_lib.VoronoiMaps)
    acc.every = every
    steps = len(simulations.density_frame_steps(T, dt, 1))
    want = simulations.density_frame_steps(T, dt, every, recompute)
    assert want == [k for k in range(steps) if k % every == 0]
    taken, k = 0, 0
    while k < steps:
        n = min(steps - k, recompute - k % recompute) if recompute else steps - k
        taken += acc.count(k, n)
        k += n
    assert taken == len(want) and all(acc.due(s) for s in want)


# --------------------------------------------------------------------------------------------- the oracle itself
def _grid(step, L=4.0, H=3.0):
    nx, ny = int(round(L / step)) + 1, int(round(H / step)) + 1
    return np.linspace(0, L, nx), np.linspace(0, H, ny)


@pytest.mark.parametrize("edges", [4, 12, 31])
def test_isolated_agent_owns_exactly_the_nodes_inside_its_ring(edges):
    X, Y = _grid(0.05)
    cutoff, x0, y0 = 0.8, 1.913, 1.377
    x, y = np.array([x0, 3.9, 0.1]), np.array([y0, 2.9, 0.1])      # two more generators, far away
    t = frame(X, Y, np.zeros((len(Y), len(X))), 4.0, 3.0, cutoff, edges, x, y, np.array([0.3, 0, 0]),
              np.array([-0.4, 0, 0]), np.ones(3, np.uint8))
    ox, oy = ring(cutoff, edges)
    XX, YY = np.meshgrid(X, Y)
    inside = np.ones(XX.shape, dtype=bool)
    for k in range(edges):
        k1 = (k + 1) % edges
        inside &= ((x0 + ox[k1]) - (x0 + ox[k])) * (YY - (y0 + oy[k])) - \
                  ((y0 + oy[k1]) - (y0 + oy[k])) * (XX - (x0 + ox[k])) >= 0
    mine = t["owner"] == 0
    assert inside.sum() > 100 and np.array_equal(mine, inside)
    polygon = 0.5 * edges * cutoff * cutoff * np.sin(2 * np.pi / edges)
    assert np.allclose(t["rho"][mine], 1 / polygon, rtol=1e-12)
    assert np.all(t["s"][mine] == 0.5) and np.all(t["vx"][mine] == 0.3) and np.all(t["vy"][mine] == -0.4)


def test_density_integrates_to_one_per_isolated_agent():
    errs = []
    for step in (0.1, 0.05, 0.025, 0.0125):
        X, Y = _grid(step)
        t = frame(X, Y, np.zeros((len(Y), len(X))), 4.0, 3.0, 1.0, 12, np.array([2.01]), np.array([1.49]),
                  np.zeros(1), np.zeros(1), np.ones(1, np.uint8))
        errs.append(abs(np.sum(t["rho"]) * (X[1] - X[0]) * (Y[1] - Y[0]) - 1.0))
    assert errs[-1] < 0.01 and errs[-1] < errs[0]


def test_ties_go_to_the_lowest_index_and_walls_are_never_covered():
    X, Y = np.array([0.0, 1.0, 2.0]), np.array([0.0, 1.0])
    # agents 0 and 1 equidistant from node (1, 0); 2 and 3 coincide
    x, y = np.array([1.5, 0.5, 1.0, 1.0]), np.array([0.0, 0.0, 1.0, 1.0])
    gen = np.ones(4, dtype=bool)
    own = owners(X, Y, x, y, gen, 0.6)
    assert own[0, 1] == 0 and own[1, 1] == 2 and own[0, 0] == 1 and own[1, 0] == -1
    own = owners(X, Y, x[::-1].copy(), y[::-1].copy(), gen, 0.6)
    assert own[0, 1] == 2 and own[1, 1] == 0
    Vg = np.zeros((2, 3))
    Vg[1, 1] = -100.0
    t = frame(X, Y, Vg, 2.0, 1.0, 0.6, 8, x, y, np.ones(4), np.zeros(4), np.ones(4, np.uint8))
    assert not t["covered"][1, 1] and t["covered"][0, 1]
    acc = add(add(empty((2, 3)), t), t)
    assert acc["frames"] == 2 and acc["covered"][0, 1] == 2 and acc["covered"][1, 1] == 0
    assert acc["density_sum"][0, 1] == 2 * t["rho"][0, 1] and acc["vx_sum"][0, 1] == 2.0
