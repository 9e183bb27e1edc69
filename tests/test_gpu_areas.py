"""GPU tests of measurement areas (``areas=``; oc_areas_measure, oc_areas_measure_multi, oc_gcfm_run_obs): single
measurements, batched measurements, runs on every step path and ensembles.  Every comparison is bit for bit; the
reference is the numpy restatement in tests/area_oracle.py, applied to chosen crowds and to the trajectory record and
exit steps of the run without areas."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest

from area_oracle import measure, run_area_rows
from conftest import REPO
from test_gpu_density_stats import _ctx, _same

pytestmark = pytest.mark.gpu

KEYS = ("count", "speed_sum", "vx_sum", "vy_sum")


@pytest.fixture()
def in_repo_cwd(monkeypatch):
    monkeypatch.chdir(REPO)


def _star(cx, cy, n, r0, r1, k=5):
    t = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r = r0 + r1 * np.cos(k * t)
    return np.stack([cx + r * np.cos(t), cy + r * np.sin(t)], axis=1)


def _areas(rng, L, H):
    """64 areas: 64-vertex concave stars, rectangles (horizontal edges), concave U shapes, triangles (1084 vertices)"""
    out = {}
    for k in range(13):
        out[f"star{k}"] = _star(rng.uniform(1, L - 1), rng.uniform(1, H - 1), 64, 0.8, 0.35)
    for k in range(24):
        x0, y0 = rng.uniform(-0.5, L - 1), rng.uniform(-0.5, H - 1)
        out[f"rect{k}"] = np.array([(x0, y0), (x0 + rng.uniform(0.3, 3), y0), (x0 + 1.0, y0 + rng.uniform(0.3, 3)),
                                    (x0, y0 + 1.0)])
        out[f"rect{k}"][2] = (out[f"rect{k}"][1][0], out[f"rect{k}"][2][1])
    for k in range(15):
        x0, y0 = rng.uniform(0, L - 3), rng.uniform(0, H - 3)
        out[f"u{k}"] = np.array([(0, 0), (3, 0), (3, 3), (2, 3), (2, 1), (1, 1), (1, 3), (0, 3)], dtype=float) + (x0, y0)
    for k in range(12):
        out[f"tri{k}"] = rng.uniform(0, 1, (3, 2)) * (L, H)
    return out


def _fit(out):
    """drop whole areas from the end until at most 1024 vertices remain"""
    names = list(out)
    while sum(len(out[n]) for n in names) > 1024:
        names.pop()
    return {n: out[n] for n in names}


def _adversarial(rng, spec, N, L, H):
    """agents: uniform in and around the room, and, cycling through the areas' vertices, on vertices, edge midpoints,
    on the y of horizontal edges; NaN positions, agents that left, at rest and with a subnormal speed"""
    names, verts, offsets = spec
    x, y = rng.uniform(-1, L + 1, N), rng.uniform(-1, H + 1, N)
    vx, vy = rng.normal(0, 0.9, N), rng.normal(0, 0.9, N)
    st = (rng.uniform(size=N) < 0.85).astype(np.uint8)
    idx = rng.permutation(N)[: N // 2]
    for j, i in enumerate(idx):
        v = rng.randint(len(verts))
        a = int(np.searchsorted(offsets, v, side="right")) - 1
        nxt = offsets[a] if v + 1 == offsets[a + 1] else v + 1
        kind = j % 4
        if kind == 0:
            x[i], y[i] = verts[v]
        elif kind == 1:
            x[i], y[i] = (verts[v] + verts[nxt]) / 2
        elif kind == 2:
            x[i], y[i] = rng.uniform(min(verts[v][0], verts[nxt][0]) - 0.1, max(verts[v][0], verts[nxt][0]) + 0.1), verts[v][1]
        else:
            x[i] = verts[v][0]
    if N >= 8:
        x[0], st[0] = np.nan, 1
        y[1], st[1] = np.nan, 1
        vx[2], vy[2] = 0.0, 0.0
        vx[3], vy[3] = -3e-160, 2e-160
        vx[4] = np.nan
        st[5] = 0
        x[6], y[6] = verts[0]
        x[7], y[7], st[7] = verts[1][0], verts[1][1], 1
    return x, y, vx, vy, st


def _state(ctx, x, y, vx, vy, st):
    return dict(x=ctx.to_device(x), y=ctx.to_device(y), vx=ctx.to_device(vx), vy=ctx.to_device(vy),
                status=ctx.to_device(st))


def _polys(spec):
    names, verts, offsets = spec
    return [verts[a:b] for a, b in zip(offsets[:-1], offsets[1:])]


def _row(acc, k):
    import torch
    torch.cuda.synchronize()
    return dict(count=acc.count[k].cpu().numpy(), speed_sum=acc.speed_sum[k].cpu().numpy(),
                vx_sum=acc.vx_sum[k].cpu().numpy(), vy_sum=acc.vy_sum[k].cpu().numpy())


def _assert_row(got, want, tag):
    assert np.array_equal(got["count"], want["count"]), tag
    for k in KEYS[1:]:
        assert _same(got[k], want[k]), (tag, k)


# --------------------------------------------------------------------------------------------- 1. kernel
@pytest.mark.parametrize("N", [0, 1, 255, 256, 257, 20011])
def test_one_measurement_equals_the_oracle(N):
    from optimal_crowds_b200 import _lib, simulations
    rng = np.random.RandomState(N + 3)
    ctx = _ctx(121, 201)
    L, H = ctx.room_length, ctx.room_height
    spec = simulations.areas_spec(_fit(_areas(rng, L, H)))
    assert len(spec[1]) == 1024 and max(np.diff(spec[2])) == 64
    acc = _lib.AreaStats(ctx, *spec, N, capacity=3)
    x, y, vx, vy, st = _adversarial(rng, spec, N, L, H)
    d = _state(ctx, x, y, vx, vy, st)
    ctx.areas_measure(acc, d, 1)
    want = measure(_polys(spec), x, y, vx, vy, st)
    _assert_row(_row(acc, 1), want, N)
    if N > 300:
        assert (want["count"] > 0).sum() > 40
    assert (_row(acc, 0)["count"] == 0).all()                       # other rows untouched
    # the same row measured again is overwritten, not added to
    ctx.areas_measure(acc, d, 1)
    _assert_row(_row(acc, 1), want, N)
    r = acc.result(2)
    assert r["count"].shape == (2, len(spec[0])) and r["velocity"].shape == (2, len(spec[0]), 2)
    c = r["count"][1]
    assert np.array_equal(r["density"][1], c / r["area"])
    with np.errstate(invalid="ignore"):
        assert np.array_equal(r["speed"][1], np.where(c == 0, np.nan, r["speed_sum"][1] / np.maximum(c, 1)),
                              equal_nan=True)
    assert np.isnan(r["speed"][0]).all()
    ctx.close()


def test_64_areas_with_every_vertex_budget():
    """64 areas, 13 of them with 64 vertices"""
    from optimal_crowds_b200 import _lib, simulations
    rng = np.random.RandomState(8)
    ctx = _ctx(121, 201)
    L, H = ctx.room_length, ctx.room_height
    out = {f"s{k}": _star(rng.uniform(1, L - 1), rng.uniform(1, H - 1), 64, 1.0, 0.5, k=3 + k % 4) for k in range(13)}
    out.update({f"t{k}": rng.uniform(0, 1, (3, 2)) * (L, H) for k in range(51)})
    spec = simulations.areas_spec(out)
    assert len(spec[0]) == 64 and len(spec[1]) == 13 * 64 + 51 * 3
    acc = _lib.AreaStats(ctx, *spec, 3000, capacity=1)
    x, y, vx, vy, st = _adversarial(rng, spec, 3000, L, H)
    ctx.areas_measure(acc, _state(ctx, x, y, vx, vy, st), 0)
    _assert_row(_row(acc, 0), measure(_polys(spec), x, y, vx, vy, st), "64 areas")
    ctx.close()


def test_batched_measurements_equal_every_member_alone():
    from optimal_crowds_b200 import _lib, simulations
    rng = np.random.RandomState(5)
    sizes = [(75, 131, 700), (64, 90, 0), (40, 64, 1), (97, 97, 257), (33, 47, 5000)]
    ctxs, multi, alone, states, polys = [], [], [], [], []
    for q, (ny, nx, N) in enumerate(sizes):
        c = _ctx(ny, nx)
        out = _areas(rng, c.room_length, c.room_height)
        keep = list(out)[q * 9: q * 9 + 3 + 11 * q]          # different areas per member
        spec = simulations.areas_spec({k: out[k] for k in keep})
        ctxs.append(c)
        multi.append(_lib.AreaStats(c, *spec, N, capacity=4))
        alone.append(_lib.AreaStats(c, *spec, N, capacity=4))
        states.append(_adversarial(rng, spec, N, c.room_length, c.room_height))
        polys.append(_polys(spec))
    steps = [3, 0, 2, 1, 3]
    dev = [_state(c, *s) for c, s in zip(ctxs, states)]
    n0 = _lib.launch_count()
    _lib.areas_measure_multi(ctxs, multi, dev, steps)
    assert _lib.launch_count() - n0 == 2
    for c, a, d, k in zip(ctxs, alone, dev, steps):
        c.areas_measure(a, d, k)
    for q in range(len(sizes)):
        got, ref = _row(multi[q], steps[q]), _row(alone[q], steps[q])
        _assert_row(got, ref, q)
        _assert_row(got, measure(polys[q], *states[q]), q)
    for c in ctxs:
        c.close()


# --------------------------------------------------------------------------------------------- 2. runs
T_RUN = {"room_test": 1.2, "exit_opposite": 1.2}


def _run_areas(ref):
    """strips and boxes of the room, a concave U, and triangles whose vertices are agents' starting points (at step 0
    those agents stand on a vertex)"""
    a = {f"strip{k}": [(k, 0.0), (k + 1.0, 0.0), (k + 1.0, 6.0), (k, 6.0)] for k in range(10)}
    a["u"] = [(1, 1.5), (5, 1.5), (5, 4.5), (4, 4.5), (4, 2.5), (2, 2.5), (2, 4.5), (1, 4.5)]
    a["box"] = [(1.0, 1.5), (3.0, 1.5), (3.0, 4.5), (1.0, 4.5)]
    p = ref._row0[:, :2]
    for i in range(0, len(p) - 2, 3):
        a[f"tri{i}"] = [tuple(p[i]), tuple(p[i + 1]), tuple(p[i + 2])]
    a["row0_x"] = [(p[0][0], 0.0), (10.0, 0.0), (10.0, 6.0), (p[0][0], 6.0)]   # agent 0 starts on its left edge
    from optimal_crowds_b200 import simulations
    try:
        simulations.areas_spec(a)
    except ValueError:                      # (three collinear start points: drop the degenerate triangles)
        for k in [k for k in a if k.startswith("tri")]:
            try:
                simulations.areas_spec({k: a[k]})
            except ValueError:
                del a[k]
    return a


def _run(room, seed, record=True, fast=True, monkeypatch=None, **kw):
    from optimal_crowds_b200 import simulations
    if monkeypatch is not None:
        monkeypatch.setenv("OC_FAST_RUN", "1" if fast else "0")
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation(room, T_RUN[room], recompute=True, record=record, rng=np.random.RandomState(seed),
                                      **kw)
        simu.run()
    simu._sync_host()
    return simu


@pytest.mark.parametrize("room", ["room_test", "exit_opposite"])
def test_run_areas_equal_the_oracle_on_the_record(room, in_repo_cwd, monkeypatch):
    from optimal_crowds_b200 import simulations
    seed = 4
    ref = _run(room, seed, monkeypatch=monkeypatch)
    assert ref.simu_step > 50                                            # the run re-solved at step 50
    areas = _run_areas(ref)
    polys = _polys(simulations.areas_spec(areas))
    want = run_area_rows(polys, ref._track, ref._exit_step, ref.simu_step)
    assert want["count"].sum() > 0 and (want["speed_sum"] > 0).any()
    for path in ("block", "steps", "no_record"):
        simu = _run(room, seed, record=path != "no_record", fast=path == "block", monkeypatch=monkeypatch, areas=areas)
        r = simu.area_stats()
        assert r["names"] == list(areas)
        for k in KEYS:
            assert r[k].shape == (ref.simu_step, len(areas))
        _assert_row({k: r[k] for k in KEYS}, want, path)
        # nothing else changed: trajectories, exits, clocks, the generator's state
        assert simu.simu_step == ref.simu_step and simu.time == ref.time and simu.inside == ref.inside
        assert simu._exit_order == ref._exit_order and np.array_equal(simu._exit_step, ref._exit_step)
        assert _same(simu._h_now, ref._h_now) and _same(simu._h_timev, ref._h_timev)
        if path != "no_record":
            for ra, rb in zip(simu._track, ref._track):
                assert _same(ra, rb)
        sa, sb = simu._np_random.get_state(), ref._np_random.get_state()
        assert sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


def test_bare_steps_measure_and_capacity_grows(in_repo_cwd):
    from optimal_crowds_b200 import simulations
    areas = {"box": [(1.0, 1.5), (3.0, 1.5), (3.0, 4.5), (1.0, 4.5)], "left": [(0, 0), (2, 0), (2, 6), (0, 6)]}
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 0.1, rng=np.random.RandomState(2), areas=areas)
        cap = len(simulations.density_frame_steps(0.1, simu.dt, 1))
        assert simu._areas.count.shape[0] == cap < 19
        assert simu.area_stats()["count"].shape == (0, 2)
        simu._solve_all()
        for _ in range(7):
            simu.step(simu.dt)                                           # bare steps measure too, past the capacity
        simu.advance(12)                                                 # and an advance() past it grows first
    r = simu.area_stats()
    assert r["count"].shape == (19, 2) and simu._areas.count.shape[0] >= 19
    want = run_area_rows(_polys(simulations.areas_spec(areas)), simu._track, simu._exit_step, 19)
    _assert_row({k: r[k] for k in KEYS}, want, "bare")
    assert r["count"][0, 0] > 0
    with pytest.raises(RuntimeError, match="without areas"):
        with contextlib.redirect_stdout(io.StringIO()):
            simulations.simulation("room_test", 0.1, rng=np.random.RandomState(2)).area_stats()


# --------------------------------------------------------------------------------------------- 3. ensembles
T_ENS = 1.3
ROOMS = ["room_test", "exit_opposite", None]
SEEDS = [3, 4, 7]
CONFIGS = [{"sigma_convolution": 0.3}, {"dt": 0.025}, {"sigma_convolution": 0.4, "dt": 0.015}]
ENS_AREAS = {"left": [(0, 0), (2.5, 0), (2.5, 6), (0, 6)], "mid": [(2.5, 1), (5, 1), (5, 5), (2.5, 5)],
             "u": [(1, 1.5), (5, 1.5), (5, 4.5), (4, 4.5), (4, 2.5), (2, 2.5), (2, 4.5), (1, 4.5)],
             "tri": [(1.5, 0.5), (4.5, 2.5), (1.0, 5.5)]}


def _rooms():
    from test_gpu_density_stats import _odd_room
    return [r if r is not None else _odd_room() for r in ROOMS]


_ALONE = {}


def _alone(i):
    if i not in _ALONE:
        from optimal_crowds_b200 import simulations
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(_rooms()[i], T_ENS, recompute=True, rng=np.random.RandomState(SEEDS[i]),
                                          config=CONFIGS[i], areas=ENS_AREAS)
            simu.run()
        _ALONE[i] = simu.area_stats()
    return _ALONE[i]


@pytest.mark.parametrize("batched", [True, False], ids=["batched_steps", "member_steps"])
def test_ensemble_members_equal_their_standalone_areas(batched, in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    from test_gpu_density_stats import _assert_same_results
    res = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, batched_steps=batched,
                            areas=ENS_AREAS).run()
    plain = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, batched_steps=batched).run()
    total = 0
    for i in range(len(SEEDS)):
        want, got = _alone(i), res[i]["areas"]
        assert got["names"] == want["names"] == list(ENS_AREAS)
        assert got["count"].shape == (res[i]["steps"], len(ENS_AREAS))
        _assert_row({k: got[k] for k in KEYS}, {k: want[k] for k in KEYS}, i)
        assert np.array_equal(got["area"], want["area"])
        total += got["count"].sum()
    assert total > 0
    for i in plain:
        res[i].pop("areas")
    _assert_same_results(res, plain)


# --------------------------------------------------------------------------------------------- 4. errors
def test_bad_area_arguments_are_refused():
    import torch
    from optimal_crowds_b200 import _lib, simulations
    lib = _lib.load()
    rng = np.random.RandomState(2)
    ctx = _ctx(40, 64)
    spec = simulations.areas_spec({"a": [(0.5, 0.5), (2, 0.5), (1, 1.5)], "b": [(0, 0), (1, 0), (1, 1), (0, 1)]})
    acc = _lib.AreaStats(ctx, *spec, 300, capacity=3)
    d = _state(ctx, *_adversarial(rng, spec, 300, ctx.room_length, ctx.room_height))
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda k: _lib._dev(d[k])
    keep = []

    def call(a, step=0, N=300, drop=None):
        return lib.oc_areas_measure(ctx.h, a, N, *[None if k == drop else P(k) for k in ("x", "y", "vx", "vy", "status")],
                                    step, stream)

    def bad(verts=None, offsets=None, **kw):
        a = _lib.AreasAcc.from_buffer_copy(acc.acc)
        if verts is not None:
            v = np.ascontiguousarray(verts, dtype=np.float64)
            keep.append(v)
            a.verts = v.ctypes.data_as(_lib.dp)
        if offsets is not None:
            o = np.ascontiguousarray(offsets, dtype=np.int32)
            keep.append(o)
            a.offsets = o.ctypes.data_as(_lib.ip)
            a.n_areas = len(o) - 1
        for k, v in kw.items():
            setattr(a, k, v)
        return C.byref(a)

    assert call(C.byref(acc.acc)) == 0 and call(C.byref(acc.acc), step=2) == 0
    assert call(None) == -2
    cases = [(C.byref(acc.acc), dict(step=3)), (C.byref(acc.acc), dict(step=-1)), (bad(n_areas=0), {}),
             (bad(n_areas=65), {}), (bad(partial_blocks=1), {}), (bad(d_verts=acc.d_verts.data_ptr() + 8), {}),
             (bad(verts=[(0, 0), (1, 0), (0, np.nan), (0, 0), (1, 0), (1, 1), (0, 1)]), {}),
             (bad(verts=[(0, 0), (1, 0), (2, 0), (0, 0), (1, 0), (1, 1), (0, 1)]), {}),          # zero area
             (bad(offsets=[0, 2, 7]), {}), (bad(offsets=[1, 3, 7]), {}), (bad(offsets=[0, 3, 68]), {}),
             (bad(d_count=None), {}), (bad(d_partials=None), {}), (bad(verts=None, d_verts=None), {}),
             (C.byref(acc.acc), dict(drop="vy")), (C.byref(acc.acc), dict(drop="status"))]
    for a, kw in cases:
        assert call(a, **kw) == -2, kw
        assert "bad argument" in lib.oc_last_error().decode()
    assert call(bad(d_partials=None), N=0) == -2                          # the accumulator is checked whatever N
    assert call(C.byref(acc.acc), N=0, drop="x") == 0                     # nothing to measure: no agent arrays read
    # the batched call checks every member
    a0, a1 = _lib.AreasAcc.from_buffer_copy(acc.acc), _lib.AreasAcc.from_buffer_copy(acc.acc)
    a1.n_areas = 65
    hs = (C.c_void_p * 2)(ctx.h.value, ctx.h.value)
    accs = (C.c_void_p * 2)(C.addressof(a0), C.addressof(a1))
    Ns = np.array([300, 300], dtype=np.int32)
    steps = np.array([0, 1], dtype=np.int32)
    ptr = lambda k: (C.c_void_p * 2)(d[k].data_ptr(), d[k].data_ptr())
    multi = lambda: lib.oc_areas_measure_multi(2, hs, accs, Ns.ctypes.data_as(_lib.ip), ptr("x"), ptr("y"), ptr("vx"),
                                               ptr("vy"), ptr("status"), steps.ctypes.data_as(_lib.ip), stream)
    assert multi() == -2
    a1.n_areas = 2
    assert multi() == 0
    steps[1] = 3
    assert multi() == -2
    torch.cuda.synchronize()
    ctx.close()


def test_runs_with_bad_area_accumulators_are_refused_before_any_step(in_repo_cwd):
    from optimal_crowds_b200 import _lib, simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 1.0, rng=np.random.RandomState(1),
                                      areas={"a": [(1, 1), (3, 1), (3, 4), (1, 4)]})
        simu._solve_all()
    before = simu._np_random.get_state()
    simu._areas.acc.d_partials = None
    with pytest.raises(_lib.OcError, match="NULL"):
        simu.advance(5)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    simu._areas.acc.d_partials = simu._areas.partials.data_ptr()
    simu._areas.ensure = lambda steps: None                              # a capacity the run goes past
    with pytest.raises(_lib.OcError, match="capacity"):
        simu.advance(60)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    verts = np.array([[1, 1], [3, 1], [3, 4], [1, 4]], dtype=np.float64)
    simu._areas.acc.verts = verts.ctypes.data_as(_lib.dp)
    verts[:, 1] = 1.0                                                    # a zero area
    with pytest.raises(_lib.OcError, match="non-zero"):
        simu.advance(5)
    assert simu.simu_step == 0


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
        d1 = _state(c1, *_adversarial(rng, spec, 20, 3, 2))
        a1 = _lib.AreaStats(c1, *spec, 20, 2)
    d0 = _state(c0, *_adversarial(rng, spec, 20, 3, 2))
    a0 = _lib.AreaStats(c0, *spec, 20, 2)
    with pytest.raises(_lib.OcError, match="another device"):
        _lib.areas_measure_multi([c0, c1], [a0, a1], [d0, d1], [0, 0])
    c0.close(); c1.close()
