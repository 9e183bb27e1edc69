"""GPU tests of the Voronoi measures of measurement areas (``voronoi=``; oc_voronoi_measure, oc_voronoi_measure_multi,
oc_gcfm_run_observed): single measurements on adversarial crowds, batched measurements, runs on every step path and
ensembles.  Every comparison is bit for bit; the reference is the Python restatement in tests/voronoi_oracle.py,
applied to chosen crowds and to the trajectory record and exit steps of the run without Voronoi measures."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest

from test_gpu_areas import (CONFIGS, ENS_AREAS, KEYS, SEEDS, T_ENS, T_RUN, _areas, _fit, _polys, _rooms, _run,
                            _run_areas, _star, _state)
from test_gpu_density_stats import _ctx, _same
from voronoi_oracle import measure, run_rows

pytestmark = pytest.mark.gpu

VKEYS = ("density", "speed", "velocity", "covered")


@pytest.fixture()
def in_repo_cwd(monkeypatch):
    from conftest import REPO
    monkeypatch.chdir(REPO)


def _stats(ctx, spec, vspec, N, capacity):
    from optimal_crowds_b200 import _lib, simulations
    return _lib.VoronoiStats(ctx, spec[1], spec[2], *simulations.voronoi_triangles(spec), *vspec, N, capacity)


def _oracle(ctx, spec, vspec, x, y, vx, vy, st):
    from optimal_crowds_b200 import _lib, simulations
    tris, toff = simulations.voronoi_triangles(spec)
    per = [tris[a:b] for a, b in zip(toff[:-1], toff[1:])]
    areas = [_lib.polygon_area(p) for p in _polys(spec)]
    return measure(per, areas, ctx.room_length, ctx.room_height, vspec[0], vspec[1], x, y, vx, vy, st)


def _row(acc, k):
    import torch
    torch.cuda.synchronize()
    r = acc.rows[k].cpu().numpy()
    return dict(density=r[:, 0], speed=r[:, 1], velocity=r[:, 2:4], covered=r[:, 4])


def _assert_row(got, want, tag):
    for k in VKEYS:
        assert _same(got[k], want[k]), (tag, k, got[k], want[k])


def _crowd(rng, spec, N, L, H, r):
    """agents in and around the room; on area vertices, edge midpoints and triangle edges (diagonals included);
    coincident pairs, neighbours at exactly 2r, far outside the room, NaN positions and velocities, status 0"""
    from optimal_crowds_b200 import simulations
    names, verts, offsets = spec
    tris = simulations.voronoi_triangles(spec)[0]
    x, y = rng.uniform(-0.5, L + 0.5, N), rng.uniform(-0.5, H + 0.5, N)
    vx, vy = rng.normal(0, 0.9, N), rng.normal(0, 0.9, N)
    st = (rng.uniform(size=N) < 0.9).astype(np.uint8)
    for j, i in enumerate(rng.permutation(N)[: N // 3]):
        kind = j % 5
        if kind == 0:
            x[i], y[i] = verts[rng.randint(len(verts))]
        elif kind == 1:
            v = rng.randint(len(verts))
            a = int(np.searchsorted(offsets, v, side="right")) - 1
            nxt = offsets[a] if v + 1 == offsets[a + 1] else v + 1
            x[i], y[i] = (verts[v] + verts[nxt]) / 2
        elif kind == 2:
            t = tris[rng.randint(len(tris))]
            x[i], y[i] = (t[0] + t[2]) / 2                                  # on the edge c -> a: often a diagonal
        elif kind == 3 and i > 0:
            x[i], y[i] = x[i - 1], y[i - 1]                                 # coincident with the agent before
        elif kind == 4 and i > 0:
            x[i], y[i] = x[i - 1] + 2 * r, y[i - 1]                         # at about 2r (agents 8-11: exactly)
    if N >= 12:
        x[0], st[0] = np.nan, 1
        y[1], st[1] = np.nan, 1
        vx[2], vy[2] = np.nan, 0.0
        st[3] = 0
        x[4], y[4], st[4] = -0.3, H / 2, 1
        x[5], y[5], st[5] = 1e300, 1.0, 1
        x[6], y[6], st[6] = -1e300, -1e300, 1
        x[7], y[7], st[7] = L + 0.7, H + 0.2, 1
        x[8], y[8], st[8] = 2.0, 2.0, 1
        x[9], y[9], st[9] = 2.0, 2.0 + 2 * r, 1
        x[10], y[10], st[10] = 2.0 + 2 * r, 2.0, 1
        x[11], y[11], st[11] = 2.0, 2.0, 1
    return x, y, vx, vy, st


# --------------------------------------------------------------------------------------------- 1. kernels
@pytest.mark.parametrize("N", [0, 1, 255, 256, 257, 20011])
def test_one_measurement_equals_the_oracle(N):
    from optimal_crowds_b200 import simulations
    rng = np.random.RandomState(N + 11)
    ctx = _ctx(721, 1001) if N > 1000 else _ctx(121, 201)
    L, H = ctx.room_length, ctx.room_height
    spec = simulations.areas_spec(_fit(_areas(rng, L, H)))
    assert len(spec[1]) == 1024 and max(np.diff(spec[2])) == 64
    vspec = simulations.voronoi_spec(dict(cutoff=0.5, edges=12))
    acc = _stats(ctx, spec, vspec, N, 3)
    x, y, vx, vy, st = _crowd(rng, spec, N, L, H, vspec[0])
    d = _state(ctx, x, y, vx, vy, st)
    ctx.voronoi_measure(acc, d, 1)
    want = _oracle(ctx, spec, vspec, x, y, vx, vy, st)
    _assert_row(_row(acc, 1), want, N)
    if N > 250:
        assert (want["covered"] > 0).sum() > 30 and np.isfinite(want["density"]).all()
    assert (_row(acc, 0)["density"] == 0).all()                      # other rows untouched
    ctx.voronoi_measure(acc, d, 1)                                    # measured again: overwritten, not added to
    _assert_row(_row(acc, 1), want, N)
    r = acc.result(2)
    assert r["density"].shape == r["covered"].shape == (2, len(spec[0])) and r["velocity"].shape == (2, len(spec[0]), 2)
    assert r["cutoff"] == vspec[0] and r["edges"] == 12
    ctx.close()


@pytest.mark.parametrize("edges", [4, 7, 32])
def test_cut_off_polygons_and_room_clipping(edges):
    """few agents, cells reaching the room's sides, an area covering the whole room"""
    from optimal_crowds_b200 import simulations
    rng = np.random.RandomState(edges)
    ctx = _ctx(61, 101)
    L, H = ctx.room_length, ctx.room_height
    spec = simulations.areas_spec({"room": [(0, 0), (L, 0), (L, H), (0, H)], "u": [(1, 0.5), (4, 0.5), (4, 2.5),
                                   (3, 2.5), (3, 1.5), (2, 1.5), (2, 2.5), (1, 2.5)], "star": _star(3, 1.5, 40, 0.8, 0.3)})
    for cutoff in (0.25, 1.0, 7.0):
        vspec = simulations.voronoi_spec(dict(cutoff=cutoff, edges=edges))
        acc = _stats(ctx, spec, vspec, 300, 1)
        x, y, vx, vy, st = _crowd(rng, spec, 300, L, H, cutoff)
        ctx.voronoi_measure(acc, _state(ctx, x, y, vx, vy, st), 0)
        _assert_row(_row(acc, 0), _oracle(ctx, spec, vspec, x, y, vx, vy, st), (edges, cutoff))
    ctx.close()


@pytest.mark.parametrize("n_ring, overflow", [(80, True), (40, False)])
def test_an_overflowing_cell_gives_nan_only_where_it_reaches(n_ring, overflow):
    from optimal_crowds_b200 import simulations
    ctx = _ctx(121, 201)
    L, H = ctx.room_length, ctx.room_height
    spec = simulations.areas_spec({"near": [(2.5, 2.5), (3.5, 2.5), (3.5, 3.5), (2.5, 3.5)],
                                   "touch": [(3.8, 2.0), (5.0, 2.0), (5.0, 4.0)],
                                   "far": [(7.0, 0.5), (9.0, 0.5), (9.0, 2.0), (7.0, 2.0)]})
    vspec = simulations.voronoi_spec(True)
    t = np.linspace(0, 2 * np.pi, n_ring, endpoint=False)
    rng = np.random.RandomState(n_ring)
    fx, fy = rng.uniform(6.5, 9.5, 30), rng.uniform(0.2, 2.5, 30)      # a crowd in the far area
    x = np.r_[fx, 3.0, 3.0 + 0.5 * np.cos(t)]
    y = np.r_[fy, 3.0, 3.0 + 0.5 * np.sin(t)]
    N = len(x)
    vx, vy, st = rng.normal(size=N), rng.normal(size=N), np.ones(N, np.uint8)
    acc = _stats(ctx, spec, vspec, N, 1)
    ctx.voronoi_measure(acc, _state(ctx, x, y, vx, vy, st), 0)
    want = _oracle(ctx, spec, vspec, x, y, vx, vy, st)
    got = _row(acc, 0)
    _assert_row(got, want, n_ring)
    nan = np.isnan(got["density"])
    assert list(nan) == ([True, True, False] if overflow else [False, False, False])
    assert np.isfinite(got["covered"][2]) and got["covered"][2] > 0
    ctx.close()


def test_batched_measurements_equal_every_member_alone():
    from optimal_crowds_b200 import _lib, simulations
    rng = np.random.RandomState(5)
    sizes = [(75, 131, 700), (64, 90, 0), (40, 64, 1), (97, 97, 257), (33, 47, 3000), (121, 201, 256)]
    cuts = [(1.0, 12), (0.5, 8), (2.0, 32), (0.25, 4), (0.75, 16), (3.0, 12)]
    ctxs, multi, alone, states, specs = [], [], [], [], []
    for q, ((ny, nx, N), cut) in enumerate(zip(sizes, cuts)):
        c = _ctx(ny, nx)
        out = _areas(rng, c.room_length, c.room_height)
        keep = list(out)[q * 9: q * 9 + 3 + 9 * q]
        spec = simulations.areas_spec({k: out[k] for k in keep})
        vspec = simulations.voronoi_spec(dict(cutoff=cut[0], edges=cut[1]))
        ctxs.append(c)
        multi.append(_stats(c, spec, vspec, N, 4))
        alone.append(_stats(c, spec, vspec, N, 4))
        states.append(_crowd(rng, spec, N, c.room_length, c.room_height, cut[0]))
        specs.append((spec, vspec))
    steps = [3, 0, 2, 1, 3, 0]
    dev = [_state(c, *s) for c, s in zip(ctxs, states)]
    n0 = _lib.launch_count()
    _lib.voronoi_measure_multi(ctxs, multi, dev, steps)
    assert _lib.launch_count() - n0 == 6
    for c, a, d, k in zip(ctxs, alone, dev, steps):
        c.voronoi_measure(a, d, k)
    for q in range(len(sizes)):
        got, ref = _row(multi[q], steps[q]), _row(alone[q], steps[q])
        _assert_row(got, ref, q)
        _assert_row(got, _oracle(ctxs[q], *specs[q], *states[q]), q)
    # the bins are left zeroed: measuring again gives the same rows
    _lib.voronoi_measure_multi(ctxs, multi, dev, steps)
    for q in range(len(sizes)):
        _assert_row(_row(multi[q], steps[q]), _row(alone[q], steps[q]), q)
    for c in ctxs:
        c.close()


# --------------------------------------------------------------------------------------------- 2. runs
def _run_oracle(simu, areas, vspec, ref):
    from optimal_crowds_b200 import _lib, simulations
    spec = simulations.areas_spec(areas)
    tris, toff = simulations.voronoi_triangles(spec)
    per = [tris[a:b] for a, b in zip(toff[:-1], toff[1:])]
    return run_rows(per, [_lib.polygon_area(p) for p in _polys(spec)], simu.room_length, simu.room_height, vspec[0],
                    vspec[1], ref._track, ref._exit_step, ref.simu_step)


@pytest.mark.parametrize("room", ["room_test", "exit_opposite"])
def test_run_voronoi_equals_the_oracle_on_the_record(room, in_repo_cwd, monkeypatch):
    seed = 4
    ref = _run(room, seed, monkeypatch=monkeypatch)
    assert ref.simu_step > 50                                            # the run re-solved at step 50
    areas = _run_areas(ref)
    vspec = (0.75, 10)
    want = _run_oracle(ref, areas, vspec, ref)
    assert (want["covered"] > 0).any() and (want["speed"] > 0).any()
    with_areas = _run(room, seed, monkeypatch=monkeypatch, areas=areas)
    classic = with_areas.area_stats()
    for path in ("block", "steps", "no_record"):
        simu = _run(room, seed, record=path != "no_record", fast=path == "block", monkeypatch=monkeypatch, areas=areas,
                    voronoi=dict(cutoff=vspec[0], edges=vspec[1]))
        r = simu.area_stats()
        v = r.pop("voronoi")
        assert v["cutoff"] == 0.75 and v["edges"] == 10
        _assert_row({k: v[k] for k in VKEYS}, want, path)
        # nothing else changed: the classic keys, trajectories, exits, clocks, the generator's state
        assert set(r) == set(classic) and r["names"] == classic["names"]
        for k in KEYS + ("area", "density", "speed", "velocity"):
            assert _same(r[k], classic[k]), (path, k)
        assert simu.simu_step == ref.simu_step and simu.time == ref.time and simu.inside == ref.inside
        assert simu._exit_order == ref._exit_order and np.array_equal(simu._exit_step, ref._exit_step)
        assert _same(simu._h_now, ref._h_now) and _same(simu._h_timev, ref._h_timev)
        if path != "no_record":
            for ra, rb in zip(simu._track, ref._track):
                assert _same(ra, rb)
        sa, sb = simu._np_random.get_state(), ref._np_random.get_state()
        assert sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]
    assert "voronoi" not in classic


def test_bare_steps_measure_and_capacity_grows(in_repo_cwd):
    from optimal_crowds_b200 import simulations
    areas = {"box": [(1.0, 1.5), (3.0, 1.5), (3.0, 4.5), (1.0, 4.5)], "left": [(0, 0), (2, 0), (2, 6), (0, 6)]}
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 0.1, rng=np.random.RandomState(2), areas=areas, voronoi=True)
        cap = len(simulations.density_frame_steps(0.1, simu.dt, 1))
        assert simu._voronoi.rows.shape[0] == cap < 19
        assert simu.area_stats()["voronoi"]["density"].shape == (0, 2)
        simu._solve_all()
        for _ in range(7):
            simu.step(simu.dt)                                           # bare steps measure too, past the capacity
        simu.advance(12)                                                 # and an advance() past it grows first
    r = simu.area_stats()["voronoi"]
    assert r["density"].shape == (19, 2) and r["velocity"].shape == (19, 2, 2) and simu._voronoi.rows.shape[0] >= 19
    want = _run_oracle(simu, areas, (1.0, 12), simu)
    _assert_row({k: r[k] for k in VKEYS}, want, "bare")
    assert r["covered"][0, 0] > 0


# --------------------------------------------------------------------------------------------- 3. ensembles
_ALONE = {}


def _alone(i):
    if i not in _ALONE:
        from optimal_crowds_b200 import simulations
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(_rooms()[i], T_ENS, recompute=True, rng=np.random.RandomState(SEEDS[i]),
                                          config=CONFIGS[i], areas=ENS_AREAS, voronoi=dict(cutoff=0.8, edges=9))
            simu.run()
        _ALONE[i] = simu.area_stats()
    return _ALONE[i]


@pytest.mark.parametrize("batched", [True, False], ids=["batched_steps", "member_steps"])
def test_ensemble_members_equal_their_standalone_voronoi(batched, in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    from test_gpu_density_stats import _assert_same_results
    res = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, batched_steps=batched,
                            areas=ENS_AREAS, voronoi=dict(cutoff=0.8, edges=9)).run()
    plain = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, batched_steps=batched,
                              areas=ENS_AREAS).run()
    total = 0.0
    for i in range(len(SEEDS)):
        want, got = _alone(i)["voronoi"], res[i]["areas"]["voronoi"]
        assert got["density"].shape == (res[i]["steps"], len(ENS_AREAS))
        _assert_row({k: got[k] for k in VKEYS}, {k: want[k] for k in VKEYS}, i)
        total += np.nansum(got["covered"])
        res[i]["areas"].pop("voronoi")
        for k in res[i]["areas"]:
            if k != "names":
                assert _same(res[i]["areas"][k], plain[i]["areas"][k]), (i, k)
    assert total > 0
    for i in plain:
        res[i].pop("areas"), plain[i].pop("areas")
    _assert_same_results(res, plain)


# --------------------------------------------------------------------------------------------- 4. errors
def test_bad_voronoi_accumulators_are_refused():
    import torch
    from optimal_crowds_b200 import _lib, simulations
    lib = _lib.load()
    rng = np.random.RandomState(2)
    ctx = _ctx(40, 64)
    spec = simulations.areas_spec({"a": [(0.5, 0.5), (2, 0.5), (1, 1.5)], "b": [(0, 0), (1, 0), (1, 1), (0, 1)]})
    acc = _stats(ctx, spec, (0.5, 12), 300, 3)
    d = _state(ctx, *_crowd(rng, spec, 300, ctx.room_length, ctx.room_height, 0.5))
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda k: _lib._dev(d[k])
    keep = []

    def call(a, step=0, N=300, drop=None):
        return lib.oc_voronoi_measure(ctx.h, a, N, *[None if k == drop else P(k) for k in ("x", "y", "vx", "vy",
                                                                                         "status")], step, stream)

    def bad(offsets=None, **kw):
        a = _lib.VoronoiAcc.from_buffer_copy(acc.acc)
        if offsets is not None:
            o = np.ascontiguousarray(offsets, dtype=np.int32)
            keep.append(o)
            a.tri_offsets = o.ctypes.data_as(_lib.ip)
            a.n_areas = len(o) - 1
        for k, v in kw.items():
            setattr(a, k, v)
        return C.byref(a)

    assert call(C.byref(acc.acc)) == 0 and call(C.byref(acc.acc), step=2) == 0
    assert call(None) == -2
    bx = acc.acc.bins_x
    cases = [(C.byref(acc.acc), dict(step=3)), (C.byref(acc.acc), dict(step=-1)), (bad(cutoff=0.0), {}),
             (bad(cutoff=-1.0), {}), (bad(cutoff=100.5), {}), (bad(cutoff=float("nan")), {}),
             (bad(cutoff=float("inf")), {}), (bad(edges=3), {}), (bad(edges=33), {}), (bad(n_areas=0), {}),
             (bad(n_areas=65), {}), (bad(offsets=[0, 0, 3]), {}), (bad(offsets=[1, 2, 3]), {}),
             (bad(offsets=[0, 1, 993]), {}), (bad(bins_x=0), {}), (bad(bins_x=bx + 1), {}),
             (bad(bins_x=257, bin_capacity=1 << 20), {}), (bad(bin_capacity=1), {}), (bad(agent_capacity=299), {}),
             (bad(partial_blocks=1), {}), (bad(d_rows=None), {}), (bad(d_order=None), {}), (bad(d_tris=None), {}),
             (bad(tri_offsets=None), {}), (C.byref(acc.acc), dict(drop="vy")), (C.byref(acc.acc), dict(drop="status"))]
    for a, kw in cases:
        assert call(a, **kw) == -2, kw
        assert "bad argument" in lib.oc_last_error().decode()
    assert call(bad(d_partials=None), N=0) == -2                          # the accumulator is checked whatever N
    assert call(C.byref(acc.acc), N=0, drop="x") == 0                     # nothing to measure: no agent arrays read
    # the batched call checks every member, and refuses members that share bins or scratch
    other = _stats(ctx, spec, (0.5, 12), 300, 3)
    a0, a1 = _lib.VoronoiAcc.from_buffer_copy(acc.acc), _lib.VoronoiAcc.from_buffer_copy(acc.acc)
    hs = (C.c_void_p * 2)(ctx.h.value, ctx.h.value)
    accs = (C.c_void_p * 2)(C.addressof(a0), C.addressof(a1))
    Ns = np.array([300, 300], dtype=np.int32)
    steps = np.array([0, 1], dtype=np.int32)
    ptr = lambda k: (C.c_void_p * 2)(d[k].data_ptr(), d[k].data_ptr())
    multi = lambda: lib.oc_voronoi_measure_multi(2, hs, accs, Ns.ctypes.data_as(_lib.ip), ptr("x"), ptr("y"),
                                                 ptr("vx"), ptr("vy"), ptr("status"), steps.ctypes.data_as(_lib.ip),
                                                 stream)
    assert multi() == -2 and "share" in lib.oc_last_error().decode()
    scratch = ("d_bin_count", "d_bin_start", "d_slot", "d_order", "d_partials")
    for shared in scratch:                                               # each pointer is checked on its own
        for k in scratch:
            setattr(a1, k, getattr((acc if k == shared else other).acc, k))
        assert multi() == -2 and "share" in lib.oc_last_error().decode(), shared
    for k in scratch:
        setattr(a1, k, getattr(other.acc, k))
    a1.edges = 2
    assert multi() == -2
    a1.edges = 12
    assert multi() == 0
    steps[1] = 3
    assert multi() == -2
    torch.cuda.synchronize()
    ctx.close()


def test_runs_with_bad_voronoi_accumulators_are_refused_before_any_step(in_repo_cwd):
    from optimal_crowds_b200 import _lib, simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 1.0, rng=np.random.RandomState(1),
                                      areas={"a": [(1, 1), (3, 1), (3, 4), (1, 4)]}, voronoi=True)
        simu._solve_all()
    before = simu._np_random.get_state()
    simu._voronoi.acc.d_partials = None
    with pytest.raises(_lib.OcError, match="NULL"):
        simu.advance(5)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    simu._voronoi.acc.d_partials = simu._voronoi.partials.data_ptr()
    simu._voronoi.ensure = lambda steps: None                            # a capacity the run goes past
    with pytest.raises(_lib.OcError, match="capacity"):
        simu.advance(60)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    simu._voronoi.acc.edges = 40
    with pytest.raises(_lib.OcError, match="edges"):
        simu.advance(5)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    assert (simu.area_stats()["count"].shape[0], simu._areas.count[0].sum().item()) == (0, 0)


def test_member_context_on_another_device_is_refused():
    import torch
    from optimal_crowds_b200 import _lib, simulations
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.RandomState(3)
    spec = simulations.areas_spec({"a": [(0, 0), (1, 0), (0, 1)]})
    c0 = _ctx(40, 64)
    with torch.cuda.device(1):
        c1 = _lib.Context(c0.room_length, c0.room_height, 0.05, device=1)
        d1 = _state(c1, *_crowd(rng, spec, 20, 3, 2, 1.0))
        a1 = _stats(c1, spec, (1.0, 12), 20, 2)
    d0 = _state(c0, *_crowd(rng, spec, 20, 3, 2, 1.0))
    a0 = _stats(c0, spec, (1.0, 12), 20, 2)
    with pytest.raises(_lib.OcError, match="another device"):
        _lib.voronoi_measure_multi([c0, c1], [a0, a1], [d0, d1], [0, 0])
    c0.close(); c1.close()
