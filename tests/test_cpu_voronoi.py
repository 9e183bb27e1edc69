"""CPU tests of the Voronoi measures (``voronoi=``): argument checks, refusals, the areas' triangulation, byte counts
and the Python oracle's own properties (against scipy.spatial.Voronoi).  None of them initialises CUDA."""
import numpy as np
import pytest

from area_oracle import inside
from voronoi_oracle import area, cell, generators, measure, ring

SQUARE = [(1.0, 1.0), (3.0, 1.0), (3.0, 3.0), (1.0, 3.0)]


@pytest.fixture(autouse=True)
def _no_cuda():
    import torch
    yield
    assert not torch.cuda.is_initialized()


def _star(cx, cy, n, r0, r1, k=5):
    t = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r = r0 + r1 * np.cos(k * t)
    return np.stack([cx + r * np.cos(t), cy + r * np.sin(t)], axis=1)


# the shipped test polygons: concave stars, U shapes (both orientations), rectangles with collinear vertices
POLYGONS = {
    "star64": _star(5, 5, 64, 2.0, 1.0),
    "star7": _star(2, 3, 14, 1.0, 0.6, k=7),
    "star_cw": _star(4, 4, 40, 1.5, 0.5, k=4)[::-1],
    "u": np.array([(0, 0), (3, 0), (3, 3), (2, 3), (2, 1), (1, 1), (1, 3), (0, 3)], dtype=float),
    "u_cw": np.array([(0, 0), (3, 0), (3, 3), (2, 3), (2, 1), (1, 1), (1, 3), (0, 3)], dtype=float)[::-1],
    "rect_collinear": np.array([(0, 0), (1, 0), (2, 0), (3, 0), (3, 1), (3, 2), (1.5, 2), (0, 2), (0, 1)], dtype=float),
    "comb": np.array([(0, 0), (5, 0), (5, 2), (4, 2), (4, 1), (3, 1), (3, 2), (2, 2), (2, 1), (1, 1), (1, 2), (0, 2)],
                     dtype=float),
    "triangle": np.array([(0.5, 0.5), (2, 0.5), (1, 1.5)]),
}


@pytest.mark.parametrize("name", list(POLYGONS))
def test_triangulation_covers_the_polygon(name):
    from optimal_crowds_b200 import _lib, simulations
    v = POLYGONS[name]
    spec = simulations.areas_spec({name: v})
    tris, toff = simulations.voronoi_triangles(spec)
    assert list(toff) == [0, len(tris)] and len(tris) <= len(v) - 2
    a, b, c = tris[:, 0], tris[:, 1], tris[:, 2]
    signed = (b[:, 0] - a[:, 0]) * (c[:, 1] - a[:, 1]) - (b[:, 1] - a[:, 1]) * (c[:, 0] - a[:, 0])
    assert (signed > 0).all()                                                   # counter-clockwise, non-degenerate
    cen = tris.mean(axis=1)
    assert inside(v, cen[:, 0], cen[:, 1]).all()
    total = float(np.sum(signed)) / 2
    assert total == pytest.approx(_lib.polygon_area(v), rel=1e-12)
    # every triangle vertex is a polygon vertex; the triangulation is cached on the spec and does not change
    assert all(any(np.array_equal(p, q) for q in v) for p in tris.reshape(-1, 2))
    assert simulations.voronoi_triangles(spec)[0] is tris


def test_triangle_budget_of_1024_vertices():
    from optimal_crowds_b200 import simulations
    spec = simulations.areas_spec({f"s{k}": _star(5 + 6 * k, 5, 64, 2.0, 1.0, k=3 + k % 4) for k in range(16)})
    tris, toff = simulations.voronoi_triangles(spec)
    assert len(spec[1]) == 1024 and len(tris) == toff[-1] == 992


@pytest.mark.parametrize("value, match", [
    ("yes", "expected True"),
    (1, "expected True"),
    ({"cutoff": 1.0, "edge": 12}, "unknown keys"),
    ({"cutoff": 0.0}, "cutoff"),
    ({"cutoff": -1.0}, "cutoff"),
    ({"cutoff": 100.5}, "cutoff"),
    ({"cutoff": np.nan}, "cutoff"),
    ({"cutoff": np.inf}, "cutoff"),
    ({"cutoff": True}, "cutoff"),
    ({"cutoff": "1"}, "cutoff"),
    ({"edges": 3}, "edges"),
    ({"edges": 33}, "edges"),
    ({"edges": 12.0}, "edges"),
    ({"edges": True}, "edges"),
])
def test_bad_voronoi_arguments_are_refused(value, match):
    from optimal_crowds_b200 import simulations
    with pytest.raises(ValueError, match=match):
        simulations.voronoi_spec(value)


def test_voronoi_spec_defaults():
    from optimal_crowds_b200 import simulations
    assert simulations.voronoi_spec(None) is None and simulations.voronoi_spec(False) is None
    assert simulations.voronoi_spec(True) == (1.0, 12)
    assert simulations.voronoi_spec({"cutoff": 100, "edges": np.int64(4)}) == (100.0, 4)
    spec = simulations.voronoi_spec({"edges": 32})
    assert spec == (1.0, 32) and simulations.voronoi_spec(spec) is spec


def test_simulations_and_ensembles_refuse_voronoi_before_any_gpu_work():
    from optimal_crowds_b200 import ensemble, simulations
    with pytest.raises(ValueError, match="needs measurement areas"):
        simulations.simulation("room_test", 1.0, voronoi=True)
    with pytest.raises(ValueError, match="needs measurement areas"):
        ensemble.ensemble("room_test", 1.0, [1, 2], voronoi=True)
    for kw in (dict(band=True), dict(shard_keys=True)):
        with pytest.raises(ValueError, match="voronoi is not available"):
            simulations.simulation("room_test", 1.0, areas={"a": SQUARE}, voronoi=True, **kw)
    with pytest.raises(ValueError, match="edges"):
        simulations.simulation("room_test", 1.0, areas={"a": SQUARE}, voronoi={"edges": 2})
    with pytest.raises(ValueError, match="cutoff"):
        ensemble.ensemble("room_test", 1.0, [1, 2], areas={"a": SQUARE}, voronoi={"cutoff": 0})


def test_member_bytes_count_the_voronoi_accumulator():
    from optimal_crowds_b200 import _lib, ensemble, optimals, simulations
    areas = {"a": SQUARE, "u": POLYGONS["u"]}
    kw = dict(configs=[None, {"dt": 0.02}], areas=areas)
    plain = ensemble.ensemble("room_test", 2.0, [1, 2], **kw)
    with_v = ensemble.ensemble("room_test", 2.0, [1, 2], voronoi=dict(cutoff=0.5, edges=16), **kw)
    room = simulations._load_room("room_test")
    L, H = room["room_length"], room["room_height"]
    N = sum(int(b[4] * b[2] * b[3]) for b in room["initial_boxes"].values())
    dts = [optimals._load_config()["dt"], 0.02]
    bins = _lib.voronoi_bins(L, 0.5) * _lib.voronoi_bins(H, 0.5)
    assert _lib.voronoi_bins(L, 0.5) == int(L // (1.0 + 1e-6)) and _lib.voronoi_bins(0.3, 1.0) == 1
    assert _lib.voronoi_bins(1e6, 0.01) == 256
    for a, b, dt in zip(with_v.member_bytes(), plain.member_bytes(), dts):
        steps = len(simulations.density_frame_steps(2.0, dt, 1))
        assert a - b == _lib.VoronoiStats.nbytes(N, 2, 8, 16, bins, steps) == (
            16 * 16 + 80 * 8 + 44 * 2 + 4 + 8 * (bins + 1) + 16 * N + 40 * 2 * -(-N // 256) + 40 * 2 * steps)
    # without voronoi nothing changes
    assert plain.member_bytes() == ensemble.ensemble("room_test", 2.0, [1, 2], **kw).member_bytes()


# --------------------------------------------------------------------------------------------- the oracle itself
def _tris(poly):
    from optimal_crowds_b200 import simulations
    spec = simulations.areas_spec({"a": poly})
    return [simulations.voronoi_triangles(spec)[0]]


def test_oracle_interior_cells_equal_scipy_voronoi():
    from scipy.spatial import Voronoi
    rng = np.random.RandomState(3)
    L, H, N = 10.0, 8.0, 60
    x, y = rng.uniform(0, L, N), rng.uniform(0, H, N)
    gen = generators(x, y, np.ones(N))
    ox, oy = ring(100.0, 32)
    vor = Voronoi(np.stack([x, y], axis=1))
    checked = 0
    for i in range(N):
        reg = vor.regions[vor.point_region[i]]
        if -1 in reg or not reg:
            continue
        verts = vor.vertices[reg]
        if not ((verts[:, 0] > 0).all() and (verts[:, 0] < L).all() and (verts[:, 1] > 0).all() and
                (verts[:, 1] < H).all()):
            continue
        V = cell(i, x, y, gen, L, H, 100.0, ox, oy)
        c = verts - verts.mean(axis=0)
        ref = verts[np.argsort(np.arctan2(c[:, 1], c[:, 0]))]
        ref_area = 0.5 * np.sum(ref[:, 0] * np.roll(ref[:, 1], -1) - np.roll(ref[:, 0], -1) * ref[:, 1])
        assert area(V) == pytest.approx(ref_area, abs=1e-9)
        # the same vertices (the clip may keep near-duplicates of a vertex where three cells meet)
        P = np.array(V)
        assert all(np.min(np.hypot(*(P - q).T)) < 1e-9 for q in ref)
        assert all(np.min(np.hypot(*(ref - p).T)) < 1e-9 for p in P)
        checked += 1
    assert checked >= 10


def test_oracle_whole_room_is_covered_and_counts_every_generator():
    rng = np.random.RandomState(5)
    L, H, N = 6.0, 4.0, 90
    x, y = rng.uniform(0, L, N), rng.uniform(0, H, N)
    st = (rng.uniform(size=N) < 0.8).astype(np.uint8)
    x[0], y[1] = np.nan, np.inf                                                  # not generators
    vx, vy = rng.normal(size=N), rng.normal(size=N)
    room = [(0.0, 0.0), (L, 0.0), (L, H), (0.0, H)]
    m = measure(_tris(room), [L * H], L, H, 50.0, 12, x, y, vx, vy, st)
    G = int(generators(x, y, st).sum())
    assert m["covered"][0] == pytest.approx(1.0, abs=1e-12)
    assert m["density"][0] * L * H == pytest.approx(G, abs=1e-12)
    # with a cut-off that leaves gaps, less is covered
    small = measure(_tris(room), [L * H], L, H, 0.1, 12, x, y, vx, vy, st)
    assert 0 < small["covered"][0] < 0.5


def test_oracle_lattice_cells_have_area_a_squared():
    a = 0.7
    gx, gy = np.meshgrid(np.arange(1, 9) * a, np.arange(1, 7) * a)
    x, y = gx.ravel(), gy.ravel()
    gen = generators(x, y, np.ones(len(x)))
    ox, oy = ring(1.0, 16)
    L, H = 9 * a, 7 * a
    for i in range(len(x)):
        V = cell(i, x, y, gen, L, H, 1.0, ox, oy)
        if 2 * a <= x[i] <= 7 * a and 2 * a <= y[i] <= 5 * a:
            assert area(V) == pytest.approx(a * a, rel=1e-12)
    # a coincident duplicate does not clip, and an overflow is NaN
    V = cell(0, np.r_[x, x[0]], np.r_[y, y[0]], np.r_[gen, True], L, H, 1.0, ox, oy)
    assert area(V) == pytest.approx(area(cell(0, x, y, gen, L, H, 1.0, ox, oy)))
    t = np.linspace(0, 2 * np.pi, 80, endpoint=False)
    rx, ry = np.r_[3.0, 3.0 + 0.5 * np.cos(t)], np.r_[3.0, 3.0 + 0.5 * np.sin(t)]
    assert cell(0, rx, ry, np.ones(81, bool), 6.0, 6.0, 1.0, *ring(1.0, 12)) is None
    assert np.isnan(area(None))
