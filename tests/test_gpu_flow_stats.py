"""GPU tests of flow statistics: the velocity and speed maps of the density frames (``density_stats=dict(velocity=True)``;
oc_density_accum_vel, oc_density_accum_vel_multi) and the pedestrian counts through measurement lines (``lines=``;
oc_lines_count, oc_lines_count_multi), in single frames and steps, runs and ensembles (oc_gcfm_run_flow).  Every
comparison is bit for bit; the references are the single-agent C-oracle frames and the numpy counting rule of
tests/flow_oracle.py, applied to the ``history`` frames and trajectory record of the run without statistics."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest

from conftest import REPO
from flow_oracle import line_crossings, run_line_counts, velocity_frame
from test_gpu_density_stats import _crowd, _ctx, _dev_crowd, _same, _walls

pytestmark = pytest.mark.gpu


@pytest.fixture()
def in_repo_cwd(monkeypatch):
    monkeypatch.chdir(REPO)


def _vel_crowd(ctx, rng, N, nan=False):
    x, y, st = _crowd(ctx, rng, N, nan=nan)
    d = _dev_crowd(ctx, x, y, st)
    vx, vy = rng.normal(0, 0.8, N), rng.normal(0, 0.8, N)
    if N >= 6:
        vx[4], vy[4] = 0.0, 0.0             # at rest
        vx[5], vy[5] = -3e-160, 2e-160      # a speed below the smallest normal's square root
    d.update(vx=ctx.to_device(vx), vy=ctx.to_device(vy))
    return (x, y, vx, vy, st), d


def _stats(ctx, V, sigma, velocity=True, threshold=None):
    from optimal_crowds_b200 import _lib
    return _lib.DensityStats(ctx, ctx.to_device(V), sigma, 1, threshold, velocity)


def _accum(ctx, s, d):
    if d["x"].numel():
        ctx.density_accum(s, d["x"], d["y"], d["status"], vx=d["vx"], vy=d["vy"])
    else:
        ctx.density_accum(s, None, None, None)


def _eq(a, b, nan):
    return np.array_equal(a, b, equal_nan=True) if nan else _same(a, b)


# --------------------------------------------------------------------------------------------- 1. velocity frames
@pytest.mark.parametrize("case", ["finite", "nan_agent", "no_agents"])
def test_one_velocity_frame_equals_the_oracle(case):
    rng = np.random.RandomState(21)
    ctx = _ctx(75, 131)                 # odd width, tail tiles in both directions, wall-heavy
    V = _walls(ctx, rng)
    (x, y, vx, vy, st), d = _vel_crowd(ctx, rng, 0 if case == "no_agents" else 300, nan=case == "nan_agent")
    s, plain = _stats(ctx, V, 0.5, threshold=0.2), _stats(ctx, V, 0.5, velocity=False, threshold=0.2)
    _accum(ctx, s, d)
    _accum(ctx, plain, d)
    r, rp = s.result(), plain.result()
    nan = case == "nan_agent"
    # the density part is what the frame without velocity adds, and oc_density of the crowd
    for k in ("sum", "max", "mean"):
        assert _same(r[k], rp[k]), k
    assert np.array_equal(r["above"], rp["above"])
    frame = ctx.density(d["x"] if len(x) else None, d["y"], d["status"], 0.5, s.Vglobal).cpu().numpy()
    assert _same(r["sum"], frame)
    fu, fv, fs = velocity_frame(ctx.X, ctx.Y, V, x, y, vx, vy, st, 0.5)
    assert _eq(r["vx_sum"], fu, nan) and _eq(r["vy_sum"], fv, nan) and _eq(r["speed_sum"], fs, nan)
    wall = V < 0
    for k in ("vx_sum", "vy_sum", "speed_sum"):
        assert (r[k][wall] == 0).all()
    # derived fields: NaN where the density is 0 (walls, empty rooms)
    assert r["velocity"].shape == (ctx.Ny, ctx.Nx, 2) and r["speed"].shape == (ctx.Ny, ctx.Nx)
    assert np.isnan(r["speed"][r["sum"] == 0]).all() and np.isnan(r["velocity"][r["sum"] == 0]).all()
    pos = r["sum"] > 0
    if case == "finite":
        assert pos.any() and (r["speed_sum"] > 0).any() and (r["vx_sum"] < 0).any() and (r["vx_sum"] > 0).any()
        assert _same(r["speed"][pos], r["speed_sum"][pos] / r["sum"][pos])
        assert _same(r["velocity"][pos, 1], r["vy_sum"][pos] / r["sum"][pos])
        # a density-weighted mean speed is never above the fastest agent nor the mean velocity's norm above it
        assert (r["speed"][pos] <= np.sqrt(vx ** 2 + vy ** 2)[st > 0].max() * (1 + 1e-12)).all()
        assert (np.hypot(r["velocity"][pos, 0], r["velocity"][pos, 1]) <= r["speed"][pos] * (1 + 1e-12)).all()
    if case == "nan_agent":
        assert np.isnan(r["vx_sum"][~wall]).all()
    if case == "no_agents":
        assert (r["sum"] == 0).all() and (r["speed_sum"] == 0).all() and np.isnan(r["speed"]).all()
    ctx.close()


def test_k_velocity_frames_are_numpys_sequential_accumulation():
    rng = np.random.RandomState(6)
    ctx = _ctx(64, 90, 0.1)
    V = _walls(ctx, rng, frac=0.15)
    s = _stats(ctx, V, 0.45)
    acc = [np.zeros((ctx.Ny, ctx.Nx)) for _ in range(3)]
    for k in range(4):
        (x, y, vx, vy, st), d = _vel_crowd(ctx, rng, 120 + 41 * k)
        _accum(ctx, s, d)
        for a, f in zip(acc, velocity_frame(ctx.X, ctx.Y, V, x, y, vx, vy, st, 0.45)):
            a += f
    r = s.result()
    assert r["frames"] == 4
    assert _same(r["vx_sum"], acc[0]) and _same(r["vy_sum"], acc[1]) and _same(r["speed_sum"], acc[2])
    ctx.close()


def test_batched_velocity_frames_equal_every_member_alone():
    from optimal_crowds_b200 import _lib
    rng = np.random.RandomState(9)
    # pairwise different grids and sigma; members with and without velocity maps in one call; one without agents
    spec = [(75, 131, 0.05, 0.5, 260, True), (64, 90, 0.1, 0.3, 180, False), (5, 7, 0.05, 0.8, 9, True),
            (40, 64, 0.05, 0.5, 0, True), (33, 47, 0.05, 0.6, 70, False)]
    ctxs, multi, alone = [], [], []
    for ny, nx, step, sigma, N, vel in spec:
        c = _ctx(ny, nx, step)
        V = _walls(c, rng, frac=0.1)
        ctxs.append(c)
        multi.append(_stats(c, V, sigma, velocity=vel, threshold=0.25))
        alone.append(_stats(c, V, sigma, velocity=vel, threshold=0.25))
    for frame in range(3):
        states = [_vel_crowd(c, rng, sp[4], nan=(q == 0 and frame == 2))[1] for q, (c, sp) in enumerate(zip(ctxs, spec))]
        n0 = _lib.launch_count()
        _lib.density_accum_multi(ctxs, multi, states)
        assert _lib.launch_count() - n0 == 2          # one launch per variant
        for c, s, d in zip(ctxs, alone, states):
            _accum(c, s, d)
    for q, (a, b) in enumerate(zip(multi, alone)):
        ra, rb = a.result(), b.result()
        assert ra["frames"] == rb["frames"] == 3 and set(ra) == set(rb)
        assert ("speed" in ra) == spec[q][5]
        for k in ("sum", "max", "vx_sum", "vy_sum", "speed_sum"):
            if k in ra:
                assert _same(ra[k], rb[k]), (q, k)
        assert np.array_equal(ra["above"], rb["above"])
    assert np.isnan(multi[0].result()["speed_sum"][multi[0].Vglobal.cpu().numpy() >= 0]).all()
    assert (multi[3].result()["speed_sum"] == 0).all()
    for c in ctxs:
        c.close()


# --------------------------------------------------------------------------------------------- 2. line counts
def _adversarial_moves(rng, lines, N):
    """moves from p to q: random, ending on a line or an endpoint, starting on one, along one, zero-length and NaN"""
    p = rng.uniform(-1, 11, (N, 2))
    q = p + rng.normal(0, 0.6, (N, 2))
    L = len(lines)
    for i in range(0, N, 7):
        a, b = lines[i % L, :2], lines[i % L, 2:]
        t = [0.0, 1.0, 0.5, 0.25][(i // 7) % 4]
        on = a + t * (b - a)
        kind = (i // 28) % 5
        if kind == 0:
            q[i] = on
        elif kind == 1:
            p[i] = on
        elif kind == 2:
            p[i], q[i] = a, b
        elif kind == 3:
            q[i] = p[i]
        else:
            p[i], q[i] = on - (b - a) * 0.1, on + (b - a) * 0.1
    p[3, 0] = np.nan
    q[10, 1] = np.nan
    return p, q


def _lines(rng, L):
    lines = rng.uniform(0, 10, (L, 4))
    lines[0] = (5.0, 0.0, 5.0, 6.0)       # axis-parallel lines through node-like coordinates
    lines[1] = (0.0, 3.0, 10.0, 3.0)
    lines[2] = (2.0, 2.0, 4.0, 4.0)
    return lines


def test_lines_kernel_equals_the_numpy_rule():
    import torch
    from optimal_crowds_b200 import _lib
    rng = np.random.RandomState(13)
    ctx = _ctx(40, 64)
    N, L = 3000, 64
    lines = _lines(rng, L)
    p, q = _adversarial_moves(rng, lines, N)
    st0 = (rng.uniform(size=N) < 0.9).astype(np.uint8)
    st1 = st0 & (rng.uniform(size=N) < 0.9).astype(np.uint8)          # some leave in the step
    dev = lambda xy, st: dict(x=ctx.to_device(np.ascontiguousarray(xy[:, 0])),
                              y=ctx.to_device(np.ascontiguousarray(xy[:, 1])), status=ctx.to_device(st))
    lc = _lib.LineCounts(ctx, [f"l{k}" for k in range(L)], lines, dev(p, st0), capacity=6)
    ctx.lines_count(lc, dev(q, st1), 2)
    r2 = q + rng.normal(0, 0.6, (N, 2))
    ctx.lines_count(lc, dev(r2, st1), 4)
    torch.cuda.synchronize()
    got = lc.counts.cpu().numpy()
    left, right = line_crossings(lines, p, q, st0 > 0)
    assert np.array_equal(got[2, :, 0], left) and np.array_equal(got[2, :, 1], right)
    assert left.sum() > 50 and right.sum() > 50
    left, right = line_crossings(lines, q, r2, st1 > 0)
    assert np.array_equal(got[4, :, 0], left) and np.array_equal(got[4, :, 1], right)
    assert (got[[0, 1, 3, 5]] == 0).all()
    # the accumulator now holds the last state
    assert _same(lc.px.cpu().numpy(), r2[:, 0]) and np.array_equal(lc.inside.cpu().numpy(), st1)
    res = lc.result(5)
    assert res["names"][:2] == ["l0", "l1"] and res["to_left"].shape == (5, L) and res["to_left"].dtype == np.int32
    ctx.close()


def test_batched_line_counts_equal_every_member_alone():
    import torch
    from optimal_crowds_b200 import _lib
    rng = np.random.RandomState(14)
    sizes = [(40, 64, 700, 3), (75, 131, 0, 1), (20, 30, 257, 64), (33, 47, 1, 7)]
    ctxs, multi, alone, moves = [], [], [], []
    for ny, nx, N, L in sizes:
        c = _ctx(ny, nx)
        lines = _lines(rng, max(L, 3))[:L] if L >= 3 else rng.uniform(0, 10, (L, 4))
        p, q = _adversarial_moves(rng, lines, N) if N >= 11 else (rng.uniform(0, 10, (N, 2)), rng.uniform(0, 10, (N, 2)))
        st = np.ones(N, dtype=np.uint8)
        d0 = dict(x=c.to_device(p[:, 0].copy()), y=c.to_device(p[:, 1].copy()), status=c.to_device(st))
        ctxs.append(c)
        multi.append(_lib.LineCounts(c, [str(k) for k in range(L)], lines, d0, capacity=4))
        alone.append(_lib.LineCounts(c, [str(k) for k in range(L)], lines, d0, capacity=4))
        moves.append(dict(x=c.to_device(q[:, 0].copy()), y=c.to_device(q[:, 1].copy()), status=c.to_device(st)))
    steps = [1, 3, 0, 2]
    _lib.lines_count_multi(ctxs, multi, moves, steps)
    for c, lc, d, k in zip(ctxs, alone, moves, steps):
        if d["x"].numel():
            c.lines_count(lc, d, k)
    torch.cuda.synchronize()
    for a, b in zip(multi, alone):
        assert np.array_equal(a.counts.cpu().numpy(), b.counts.cpu().numpy())
        assert _same(a.px.cpu().numpy(), b.px.cpu().numpy())
    assert multi[0].counts.sum() > 0 and multi[2].counts.sum() > 0
    for c in ctxs:
        c.close()


# --------------------------------------------------------------------------------------------- 3. runs
T_RUN = {"room_test": 1.2, "exit_opposite": 1.2}
LINES = {   # cross-sections of the crowd boxes ("x2.5_down" is "x2.5" reversed: its sides swap)
    "x1.5": (1.5, 0.0, 1.5, 6.0), "x2.5": (2.5, 0.0, 2.5, 6.0), "x2.5_down": (2.5, 6.0, 2.5, 0.0),
    "x3.5": (3.5, 0.0, 3.5, 6.0), "x7.5": (7.5, 0.0, 7.5, 6.0), "y3": (0.0, 3.0, 10.0, 3.0),
    "diag": (1.0, 1.0, 4.0, 5.0)}


def _lines_through(ref):
    """LINES plus a vertical and a horizontal line through every agent's starting point: within these short horizons the
    crowd mostly jitters in place, and an agent starting on a line (the right side) leaves it to either side"""
    out = dict(LINES)
    for i, (x, y) in enumerate(ref._row0[:, :2]):
        out[f"v{i}"] = (x, 0.0, x, 6.0)
        out[f"h{i}"] = (0.0, y, 10.0, y)
    return out
_REF = {}


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


def _reference(room, seed):
    if (room, seed) not in _REF:
        _REF[(room, seed)] = _run(room, seed)
    return _REF[(room, seed)]


def _expected_velocity(ref, every):
    """numpy's accumulation of the oracle's velocity frames over the history frames of the due steps"""
    rows = ref._track
    acc = [np.zeros((ref.Ny, ref.Nx)) for _ in range(3)]
    n = 0
    for k in range(0, ref.simu_step, every):
        act = (ref._exit_step < 0) | (ref._exit_step >= k)
        r = rows[k]
        for a, f in zip(acc, velocity_frame(ref._ctx.X, ref._ctx.Y, ref.V, r[act, 0], r[act, 1], r[act, 2], r[act, 3],
                                            np.ones(act.sum(), np.uint8), ref.sigma_convolution)):
            a += f
        n += 1
    return n, acc


@pytest.mark.parametrize("room", ["room_test", "exit_opposite"])
def test_run_flow_statistics_equal_the_history(room, in_repo_cwd, monkeypatch):
    seed, every = 4, 7
    ref = _reference(room, seed)
    assert ref.simu_step > 50                                            # the run re-solved at step 50
    n, (wu, wv, ws) = _expected_velocity(ref, every)
    frames = [f[-1] for f in ref.history.values()]
    want_sum = np.zeros_like(frames[0])
    for f in frames[::every]:
        want_sum = want_sum + f
    lines = _lines_through(ref)
    assert len(lines) <= 64
    left, right = run_line_counts(list(lines.values()), ref._track, ref._exit_step, ref.simu_step)
    assert left.sum() > 0 and right.sum() > 0
    ds = dict(every=every, velocity=True)
    for path in ("block", "steps", "no_record"):
        simu = _run(room, seed, record=path != "no_record", fast=path == "block", monkeypatch=monkeypatch,
                    density_stats=ds, lines=lines)
        r = simu.density_stats()
        assert r["frames"] == n and _same(r["sum"], want_sum)
        assert _same(r["vx_sum"], wu) and _same(r["vy_sum"], wv) and _same(r["speed_sum"], ws), path
        c = simu.line_counts()
        assert c["names"] == list(lines)
        assert np.array_equal(c["to_left"], left) and np.array_equal(c["to_right"], right), path
        # nothing else changed: trajectories, exits, clocks, the generator's state
        assert simu.simu_step == ref.simu_step and simu.time == ref.time and simu.inside == ref.inside
        assert simu._exit_order == ref._exit_order and np.array_equal(simu._exit_step, ref._exit_step)
        assert _same(simu._h_now, ref._h_now) and _same(simu._h_timev, ref._h_timev)
        if path != "no_record":
            for ra, rb in zip(simu._track, ref._track):
                assert _same(ra, rb)
        sa, sb = simu._np_random.get_state(), ref._np_random.get_state()
        assert sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


def test_bare_steps_count_and_capacity_grows(in_repo_cwd):
    from optimal_crowds_b200 import simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 0.1, rng=np.random.RandomState(2), lines=LINES)
        cap = len(simulations.density_frame_steps(0.1, simu.dt, 1))        # the steps of a run to T = 0.1
        assert simu._lines.counts.shape[0] == cap < 19
        c = simu.line_counts()
        assert c["to_left"].shape == (0, len(LINES))
        simu._solve_all()
        for _ in range(7):
            simu.step(simu.dt)                                           # bare steps count too, past the capacity
        simu.advance(12)                                                 # and an advance() past it grows first
    c = simu.line_counts()
    assert c["to_left"].shape == (19, len(LINES)) and simu._lines.counts.shape[0] >= 19
    left, right = run_line_counts(list(LINES.values()), simu._track, simu._exit_step, 19)
    assert np.array_equal(c["to_left"], left) and np.array_equal(c["to_right"], right)
    assert left.sum() + right.sum() > 0
    with pytest.raises(RuntimeError, match="without lines"):
        _reference("room_test", 4).line_counts()


# --------------------------------------------------------------------------------------------- 4. ensembles
T_ENS = 1.3
ROOMS = ["room_test", "exit_opposite", None]
SEEDS = [3, 4, 7]
CONFIGS = [{"sigma_convolution": 0.3}, {"dt": 0.025}, {"sigma_convolution": 0.4, "dt": 0.015}]
ENS_LINES = {"x1.5": (1.5, 0.0, 1.5, 6.0), "x2.5": (2.5, 0.0, 2.5, 6.0), "x2.5_down": (2.5, 6.0, 2.5, 0.0),
             "x3.5": (3.5, 0.0, 3.5, 6.0), "y3": (0.0, 3.0, 10.0, 3.0)}
ENS_DS = {"every": 4, "velocity": True}


def _rooms():
    from test_gpu_density_stats import _odd_room
    return [r if r is not None else _odd_room() for r in ROOMS]


_ALONE = {}


def _alone(i):
    if i not in _ALONE:
        from optimal_crowds_b200 import simulations
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(_rooms()[i], T_ENS, recompute=True, rng=np.random.RandomState(SEEDS[i]),
                                          config=CONFIGS[i], density_stats=ENS_DS, lines=ENS_LINES)
            simu.run()
        _ALONE[i] = (simu.density_stats(), simu.line_counts())
    return _ALONE[i]


@pytest.mark.parametrize("batched", [True, False], ids=["batched_steps", "member_steps"])
def test_ensemble_members_equal_their_standalone_flow_statistics(batched, in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    from test_gpu_density_stats import _assert_same_results
    res = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, batched_steps=batched,
                            density_stats=ENS_DS, lines=ENS_LINES).run()
    plain = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, batched_steps=batched).run()
    total = np.zeros(2, dtype=np.int64)
    for i in range(len(SEEDS)):
        d, c = _alone(i)
        got = res[i]["density"]
        assert got["frames"] == d["frames"] > 0
        for k in ("sum", "max", "vx_sum", "vy_sum", "speed_sum"):
            assert _same(got[k], d[k]), (i, k)
        lc = res[i]["lines"]
        assert lc["names"] == c["names"] == list(ENS_LINES)
        assert lc["to_left"].shape == (res[i]["steps"], len(ENS_LINES))
        assert np.array_equal(lc["to_left"], c["to_left"]) and np.array_equal(lc["to_right"], c["to_right"]), i
        total += [lc["to_left"].sum(), lc["to_right"].sum()]
    assert (total > 0).all()
    for i in plain:
        res[i].pop("lines")
    _assert_same_results(res, plain)


# --------------------------------------------------------------------------------------------- 5. errors
def test_bad_flow_arguments_are_refused():
    import torch
    from optimal_crowds_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(2)
    ctx = _ctx(40, 64)
    V = _walls(ctx, rng)
    (x, y, vx, vy, st), d = _vel_crowd(ctx, rng, 50)
    s = _stats(ctx, V, 0.5)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda k: _lib._dev(d[k])

    def vcall(vel, vx_=True, vy_=True):
        return lib.oc_density_accum_vel(ctx.h, C.byref(s.acc), vel, 50, P("x"), P("y"), P("vx") if vx_ else None,
                                        P("vy") if vy_ else None, P("status"), stream)

    assert vcall(C.byref(s.vel)) == 0 and vcall(None, False, False) == 0
    assert vcall(C.byref(s.vel), vx_=False) == -2 and vcall(C.byref(s.vel), vy_=False) == -2
    for f in ("d_vx_sum", "d_vy_sum", "d_speed_sum"):
        v = _lib.VelocityAcc.from_buffer_copy(s.vel)
        setattr(v, f, None)
        assert vcall(C.byref(v)) == -2, f
    # lines
    lc = _lib.LineCounts(ctx, ["a", "b"], [(1, 1, 2, 2), (0, 3, 3, 0)], d, capacity=3)

    def lcall(acc, step=0, N=50):
        return lib.oc_lines_count(ctx.h, acc, N, P("x"), P("y"), P("status"), step, stream)

    def bad(lines=None, **kw):
        a = _lib.LinesAcc.from_buffer_copy(lc.acc)
        if lines is not None:
            arr = np.ascontiguousarray(lines, dtype=np.float64)
            bad.keep.append(arr)
            a.lines = arr.ctypes.data_as(_lib.dp)
            a.n_lines = len(arr)
        for k, v in kw.items():
            setattr(a, k, v)
        return C.byref(a)
    bad.keep = []
    assert lcall(C.byref(lc.acc)) == 0 and lcall(C.byref(lc.acc), step=2) == 0
    assert lcall(None) == -2
    for acc, step in ((C.byref(lc.acc), 3), (C.byref(lc.acc), -1), (bad(n_lines=0), 0), (bad(n_lines=65), 0),
                      (bad(lines=[(0, 0, np.nan, 1)]), 0), (bad(lines=[(0, 0, 1, 1), (0, np.inf, 1, 1)]), 0),
                      (bad(lines=[(2, 2, 2, 2)]), 0), (bad(d_counts=None), 0), (bad(d_px=None), 0),
                      (bad(d_inside=None), 0)):
        assert lcall(acc, step) == -2
        assert "bad argument" in lib.oc_last_error().decode()
    assert lcall(bad(d_px=None), N=0) == 0                               # nothing to count: no per-agent arrays read
    # the batched call checks every member
    hs = (C.c_void_p * 2)(ctx.h.value, ctx.h.value)
    a0, a1 = _lib.LinesAcc.from_buffer_copy(lc.acc), _lib.LinesAcc.from_buffer_copy(lc.acc)
    accs = (C.c_void_p * 2)(C.addressof(a0), C.addressof(a1))
    Ns = np.array([50, 50], dtype=np.int32)
    steps = np.array([0, 3], dtype=np.int32)
    ptr = lambda k: (C.c_void_p * 2)(d[k].data_ptr(), d[k].data_ptr())
    multi = lambda: lib.oc_lines_count_multi(2, hs, accs, Ns.ctypes.data_as(_lib.ip), ptr("x"), ptr("y"), ptr("status"),
                                             steps.ctypes.data_as(_lib.ip), stream)
    assert multi() == -2
    steps[1] = 1
    assert multi() == 0
    a1.n_lines = 0
    assert multi() == -2
    torch.cuda.synchronize()
    ctx.close()


def test_runs_with_bad_flow_accumulators_are_refused_before_any_step(in_repo_cwd):
    from optimal_crowds_b200 import _lib, simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 1.0, rng=np.random.RandomState(1), density_stats={"velocity": True},
                                      lines={"a": (2.5, 0, 2.5, 6)})
        simu._solve_all()
    before = simu._np_random.get_state()
    simu._dstats.vel.d_speed_sum = None
    with pytest.raises(_lib.OcError, match="NULL"):
        simu.advance(5)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    simu._dstats.vel.d_speed_sum = simu._dstats.speed_sum.data_ptr()
    simu._lines.ensure = lambda steps: None                              # a capacity the run goes past
    with pytest.raises(_lib.OcError, match="capacity"):
        simu.advance(60)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    lines = np.array([[0, 0, 1, 1]], dtype=np.float64)
    simu._lines.acc.lines = lines.ctypes.data_as(_lib.dp)
    lines[0, 2:] = 0.0                                                   # a zero-length line
    with pytest.raises(_lib.OcError, match="non-zero length"):
        simu.advance(5)
    assert simu.simu_step == 0


def test_member_context_on_another_device_is_refused():
    import torch
    from optimal_crowds_b200 import _lib
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.RandomState(3)
    c0 = _ctx(40, 64)
    with torch.cuda.device(1):
        c1 = _lib.Context(c0.room_length, c0.room_height, 0.05, device=1)
        d1 = _dev_crowd(c1, *_crowd(c1, rng, 20))
        l1 = _lib.LineCounts(c1, ["a"], [(0, 0, 1, 1)], d1, 2)
    d0 = _dev_crowd(c0, *_crowd(c0, rng, 20))
    l0 = _lib.LineCounts(c0, ["a"], [(0, 0, 1, 1)], d0, 2)
    with pytest.raises(_lib.OcError, match="another device"):
        _lib.lines_count_multi([c0, c1], [l0, l1], [d0, d1], [0, 0])
    c0.close(); c1.close()
