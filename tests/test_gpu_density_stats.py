"""GPU tests of density statistics: the summed, peak and above-threshold maps of a run's density frames, accumulated on
the device (oc_density_accum, oc_density_accum_multi, oc_gcfm_run_acc; ``simulation(..., density_stats=...)``,
``ensemble(..., density_stats=...)``).  A frame is the density the reference stores in ``history`` (simulations.py:579-589);
every comparison is bit for bit unless stated."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest

from conftest import REPO

pytestmark = pytest.mark.gpu


@pytest.fixture()
def in_repo_cwd(monkeypatch):
    monkeypatch.chdir(REPO)


def _same(a, b):
    """bit-identical float arrays (NaN payloads included)"""
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _ctx(ny, nx, step=0.05):
    from optimal_crowds_b200 import _lib, synthetic
    return _lib.Context(synthetic.nodes_to_length(nx, step), synthetic.nodes_to_length(ny, step), step)


def _walls(ctx, rng, frac=0.35):
    """a wall-heavy Vglobal: a frame of walls, a wall block and scattered wall nodes"""
    V = np.zeros((ctx.Ny, ctx.Nx))
    V[rng.uniform(size=V.shape) < frac] = -100.0
    V[0], V[-1], V[:, 0], V[:, -1] = -100.0, -100.0, -100.0, -100.0
    V[ctx.Ny // 3: ctx.Ny // 2, ctx.Nx // 4: ctx.Nx // 2] = -100.0
    return V


def _crowd(ctx, rng, N, nan=False):
    """seeded agents: some outside the room (x < 0, beyond the far walls), some left (status 0), optionally one NaN"""
    L, H = ctx.room_length, ctx.room_height
    x = rng.uniform(-1.5, L + 1.5, N)
    y = rng.uniform(-1.0, H + 1.0, N)
    st = (rng.uniform(size=N) < 0.8).astype(np.uint8)
    if N >= 4:
        x[1], st[1] = -0.4, 1           # x < 0, inside the kernel's reach
        y[2], st[2] = H + 0.7, 1        # above the room
        st[3] = 0                       # left the room
    if nan and N:
        x[0], st[0] = np.nan, 1
    return x, y, st


def _dev_crowd(ctx, x, y, st):
    return dict(x=ctx.to_device(x), y=ctx.to_device(y), status=ctx.to_device(st))


def _stats(ctx, V, sigma, every=1, threshold=None):
    from optimal_crowds_b200 import _lib
    return _lib.DensityStats(ctx, ctx.to_device(V), sigma, every, threshold)


# --------------------------------------------------------------------------------------------- 1. kernel
@pytest.mark.parametrize("nan", [False, True], ids=["finite", "nan_agent"])
def test_one_accumulation_is_the_frame_and_the_oracle(nan):
    from oracle import cpu_oracle as co
    rng = np.random.RandomState(11)
    ctx = _ctx(75, 131)                 # odd width, tail tiles in both directions
    V = _walls(ctx, rng)
    x, y, st = _crowd(ctx, rng, 300, nan=nan)
    d = _dev_crowd(ctx, x, y, st)
    s = _stats(ctx, V, 0.5, threshold=0.2)
    ctx.density_accum(s, d["x"], d["y"], d["status"])
    frame = ctx.density(d["x"], d["y"], d["status"], 0.5, s.Vglobal).cpu().numpy()
    r = s.result()
    assert r["frames"] == 1
    assert _same(r["sum"], frame) and _same(r["max"], frame) and _same(r["mean"], frame)
    assert np.array_equal(r["above"], (frame > 0.2).astype(np.int32))
    oracle = co.density(ctx.X, ctx.Y, V, x, y, st, 0.5)
    assert np.array_equal(frame, oracle, equal_nan=True)
    if nan:
        assert np.isnan(frame[V >= 0]).all() and (frame[V < 0] == 0).all()
    else:
        assert (frame > 0.2).any() and (frame <= 0.2).any() and (frame[V < 0] == 0).all()
    ctx.close()


@pytest.mark.parametrize("thr", [None, 0.3])
def test_k_frames_are_numpys_sequential_accumulation(thr):
    rng = np.random.RandomState(5)
    ctx = _ctx(75, 131)
    V = _walls(ctx, rng, frac=0.2)
    s = _stats(ctx, V, 0.45, threshold=thr)
    acc_s = np.zeros((ctx.Ny, ctx.Nx)); acc_m = np.zeros((ctx.Ny, ctx.Nx)); acc_a = np.zeros((ctx.Ny, ctx.Nx), np.int32)
    K = 6
    for k in range(K):
        # the NaN agent joins in the last two frames: it must reach sum and max as numpy's s + f and np.maximum do
        x, y, st = _crowd(ctx, rng, 200 + 37 * k, nan=k >= K - 2)
        d = _dev_crowd(ctx, x, y, st)
        ctx.density_accum(s, d["x"], d["y"], d["status"])
        f = ctx.density(d["x"], d["y"], d["status"], 0.45, s.Vglobal).cpu().numpy()
        acc_s = acc_s + f
        acc_m = np.maximum(acc_m, f)
        if thr is not None:
            acc_a += f > thr
        r = s.result()
        assert r["frames"] == k + 1
        assert np.array_equal(r["sum"], acc_s, equal_nan=True) and np.array_equal(r["max"], acc_m, equal_nan=True)
        if k < K - 2:
            assert _same(r["sum"], acc_s) and _same(r["max"], acc_m)
            assert _same(r["mean"], acc_s / (k + 1))
        if thr is None:
            assert r["above"] is None
        else:
            assert np.array_equal(r["above"], acc_a)
    if thr is not None:
        assert 0 < acc_a.max() and (acc_a < K).any()
    ctx.close()


# --------------------------------------------------------------------------------------------- 2. batched kernel
def test_batched_accumulation_equals_every_member_alone():
    from optimal_crowds_b200 import _lib
    rng = np.random.RandomState(8)
    # pairwise different grids: odd width, grid step 0.1, a tiny grid (one partial tile), an even grid; different sigma;
    # the last member has no agents
    spec = [(75, 131, 0.05, 0.5, 260), (64, 90, 0.1, 0.3, 180), (5, 7, 0.05, 0.8, 9), (40, 64, 0.05, 0.5, 0)]
    ctxs, Vs, multi, alone = [], [], [], []
    for q, (ny, nx, step, sigma, N) in enumerate(spec):
        c = _ctx(ny, nx, step)
        assert (c.Ny, c.Nx) == (ny, nx)
        V = _walls(c, rng, frac=0.1)
        thr = None if q == 1 else 0.25
        ctxs.append(c); Vs.append(V)
        multi.append(_stats(c, V, sigma, threshold=thr)); alone.append(_stats(c, V, sigma, threshold=thr))
    for frame in range(3):
        states = []
        for q, c in enumerate(ctxs):
            N = spec[q][4]
            x, y, st = _crowd(c, rng, N, nan=(q == 0 and frame == 2))
            states.append(_dev_crowd(c, x, y, st))
        _lib.density_accum_multi(ctxs, multi, states)
        for c, s, d in zip(ctxs, alone, states):
            c.density_accum(s, d["x"], d["y"], d["status"])
        for c, s, d in zip(ctxs, alone, states):
            # every member's frame also equals oc_density of its crowd
            if frame == 0:
                f = c.density(d["x"] if d["x"].numel() else None, d["y"], d["status"], s.acc.sigma, s.Vglobal)
                assert _same(f.cpu().numpy(), s.result()["sum"])
    for q, (a, b) in enumerate(zip(multi, alone)):
        ra, rb = a.result(), b.result()
        assert ra["frames"] == rb["frames"] == 3
        for k in ("sum", "max", "mean"):
            assert _same(ra[k], rb[k]), (q, k)
        assert (ra["above"] is None) == (rb["above"] is None) == (q == 1)
        if ra["above"] is not None:
            assert np.array_equal(ra["above"], rb["above"])
    assert (multi[3].result()["sum"] == 0).all()                      # N = 0: frames of zeros
    assert np.isnan(multi[0].result()["sum"][Vs[0] >= 0]).all()       # the NaN reached member 0 only
    assert not np.isnan(multi[1].result()["sum"]).any()
    for c in ctxs:
        c.close()


# --------------------------------------------------------------------------------------------- 3. runs
_REF = {}
T_RUN = {"room_test": 1.2, "exit_opposite": 1.2}


def _run(room, seed, density_stats=None, record=True, fast=True, monkeypatch=None):
    from optimal_crowds_b200 import simulations
    if monkeypatch is not None:
        monkeypatch.setenv("OC_FAST_RUN", "1" if fast else "0")
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation(room, T_RUN[room], recompute=True, record=record,
                                      rng=np.random.RandomState(seed), density_stats=density_stats)
        simu.run()
    simu._sync_host()
    return simu


def _reference(room, seed):
    """the run without statistics, with its history frames (record=True, block path)"""
    if (room, seed) not in _REF:
        simu = _run(room, seed)
        frames = [f[-1] for f in simu.history.values()]
        _REF[(room, seed)] = (simu, frames)
    return _REF[(room, seed)]


def _expected(frames, every, thr):
    sel = [f for k, f in enumerate(frames) if k % every == 0]
    s = np.zeros_like(frames[0]); m = np.zeros_like(frames[0]); a = np.zeros(frames[0].shape, np.int32)
    for f in sel:
        s = s + f
        m = np.maximum(m, f)
        a += f > thr if thr is not None else 0
    return len(sel), s, m, (a if thr is not None else None)


def _assert_stats(got, want):
    n, s, m, a = want
    assert got["frames"] == n
    assert _same(got["sum"], s) and _same(got["max"], m) and _same(got["mean"], s / n)
    if a is None:
        assert got["above"] is None
    else:
        assert np.array_equal(got["above"], a)


@pytest.mark.parametrize("thr", [None, 0.5], ids=["no_threshold", "threshold"])
@pytest.mark.parametrize("every", [1, 7, 10])
@pytest.mark.parametrize("room", ["room_test", "exit_opposite"])
def test_run_statistics_equal_the_history_frames(room, every, thr, in_repo_cwd, monkeypatch):
    from optimal_crowds_b200 import simulations
    seed = 4
    ref, frames = _reference(room, seed)
    assert len(frames) == ref.simu_step and ref.simu_step > 50          # the run re-solved at step 50
    want = _expected(frames, every, thr)
    sel = simulations.density_frame_steps(ref.T, ref.dt, every, ref.recompute_step)
    assert want[0] == len(sel)
    if thr is not None:
        assert want[3].max() > 0
    ds = dict(every=every, threshold=thr)
    for path in ("block", "steps", "no_record"):
        simu = _run(room, seed, ds, record=path != "no_record", fast=path == "block", monkeypatch=monkeypatch)
        _assert_stats(simu.density_stats(), want)
        # nothing else changed: trajectories, exits, clocks, the generator's state
        assert simu.simu_step == ref.simu_step and simu.time == ref.time and simu.inside == ref.inside
        assert simu._exit_order == ref._exit_order and np.array_equal(simu._exit_step, ref._exit_step)
        assert _same(simu._h_now, ref._h_now) and _same(simu._h_timev, ref._h_timev)
        if path != "no_record":
            for ra, rb in zip(simu._track, ref._track):
                assert _same(ra, rb)
        sa, sb = simu._np_random.get_state(), ref._np_random.get_state()
        assert sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


def test_bare_steps_take_no_frames_and_stats_start_empty(in_repo_cwd):
    from optimal_crowds_b200 import simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 1.0, rng=np.random.RandomState(1), density_stats={"threshold": 1.0})
        r = simu.density_stats()
        assert r["frames"] == 0 and r["mean"] is None and (r["sum"] == 0).all() and (r["above"] == 0).all()
        simu._solve_all()
        simu.step(simu.dt)                 # the reference's bare step() writes no history frame
        assert simu.density_stats()["frames"] == 0
        simu.advance(3)                    # three iterations of run()'s body: three frames
        assert simu.density_stats()["frames"] == 3
    with pytest.raises(RuntimeError, match="without density_stats"):
        _reference("room_test", 4)[0].density_stats()


# --------------------------------------------------------------------------------------------- 4. ensembles
T_ENS = 1.3


def _odd_room():
    """a 97 x 97 synthetic room (odd Nx) with 12 agents"""
    from optimal_crowds_b200 import synthetic
    room = synthetic.ensemble_room(n=97, agents=12)
    room["initial_boxes"]["box"][0] = 1.6
    room["initial_boxes"]["box"][2:4] = [2.0, 2.0]
    room["initial_boxes"]["box"][4] = 12.5 / 4.0
    return room


ROOMS = ["room_test", "exit_opposite", "metro_station", "slalom", None]
SEEDS = [3, 4, 5, 6, 7]
CONFIGS = [{"sigma_convolution": 0.3}, {"dt": 0.025}, {}, {"sigma_convolution": 0.7, "dt": 0.015},
           {"sigma_convolution": 0.4}]
_ALONE = {}


def _rooms():
    return [r if r is not None else _odd_room() for r in ROOMS]


def _alone(i, ds):
    import json
    key = (i, json.dumps(ds, sort_keys=True))
    if key not in _ALONE:
        from optimal_crowds_b200 import simulations
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(_rooms()[i], T_ENS, recompute=True, rng=np.random.RandomState(SEEDS[i]),
                                          config=CONFIGS[i], density_stats=ds)
            simu.run()
        _ALONE[key] = simu.density_stats()
    return _ALONE[key]


_PLAIN = {}


def _plain_ensemble(batched):
    if batched not in _PLAIN:
        from optimal_crowds_b200 import ensemble
        _PLAIN[batched] = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS,
                                            batched_steps=batched).run()
    return _PLAIN[batched]


def _assert_same_results(a, b):
    assert sorted(a) == sorted(b)
    for i in a:
        assert set(a[i]) - {"density"} == set(b[i]) - {"density"}
        for k in ("steps", "inside", "evac_time", "N", "seed", "chunk_rows", "config"):
            assert a[i][k] == b[i][k], (i, k)
        assert set(a[i]["hjb"]) == set(b[i]["hjb"])
        for key in a[i]["hjb"]:
            for k in ("nfev", "n_accepted", "n_rejected", "status", "n_out"):
                assert a[i]["hjb"][key][k] == b[i]["hjb"][key][k], (i, key, k)
        for k in ("exit_order", "exit_step"):
            assert np.array_equal(a[i][k], b[i][k]), (i, k)
        for k in ("final", "times"):
            assert _same(a[i][k], b[i][k]), (i, k)


def _assert_density(got, want):
    assert got["frames"] == want["frames"] > 0
    for k in ("sum", "max", "mean"):
        assert _same(got[k], want[k]), k
    assert (got["above"] is None) == (want["above"] is None)
    if got["above"] is not None:
        assert np.array_equal(got["above"], want["above"])


@pytest.mark.parametrize("ds", [True, {"every": 7, "threshold": 0.5}], ids=["every_1", "every_7_threshold"])
@pytest.mark.parametrize("batched", [True, False], ids=["batched_steps", "member_steps"])
def test_ensemble_members_equal_their_standalone_statistics(batched, ds, in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    ens = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, batched_steps=batched,
                            density_stats=ds)
    res = ens.run()
    for i in range(len(SEEDS)):
        _assert_density(res[i]["density"], _alone(i, ds))
    _assert_same_results(res, _plain_ensemble(batched))
    # the members' grids differ (an odd width among them) and so do their sigma and dt
    shapes = {res[i]["density"]["sum"].shape for i in res}
    assert len(shapes) == 4 and any(nx % 2 for _, nx in shapes)


def test_sharded_one_member_waves(in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    ds = {"every": 10, "threshold": 0.5}
    parts = {}
    for rank in range(2):
        e = ensemble.ensemble(_rooms(), T_ENS, SEEDS, recompute=True, configs=CONFIGS, rank=rank, world=2,
                              memory_budget=1, density_stats=ds)
        parts.update(e.run(gather=False))
        assert e.stats["waves"] == len(e.mine)                          # one member per wave
    for i in range(len(SEEDS)):
        _assert_density(parts[i]["density"], _alone(i, ds))
    _assert_same_results(parts, _plain_ensemble(True))


# --------------------------------------------------------------------------------------------- 5. errors
def test_bad_accumulator_arguments_are_refused():
    import torch
    from optimal_crowds_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(2)
    ctx = _ctx(40, 64)
    V = _walls(ctx, rng)
    x, y, st = _crowd(ctx, rng, 50)
    d = _dev_crowd(ctx, x, y, st)
    s = _stats(ctx, V, 0.5, threshold=1.0)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(acc):
        return lib.oc_density_accum(ctx.h, acc, 50, _lib._dev(d["x"]), _lib._dev(d["y"]), _lib._dev(d["status"]), stream)

    def bad(**kw):
        a = _lib.DensityAcc.from_buffer_copy(s.acc)
        for k, v in kw.items():
            setattr(a, k, v)
        return C.byref(a)

    assert call(C.byref(s.acc)) == 0
    assert call(None) == -2
    for kw in (dict(d_sum=None), dict(d_max=None), dict(d_Vglobal=None), dict(every=0), dict(every=-3),
               dict(sigma=0.0), dict(sigma=-0.5), dict(sigma=float("nan")), dict(sigma=float("inf")), dict(C=0.0),
               dict(C=float("inf")), dict(C=float("nan")), dict(threshold=float("nan")), dict(threshold=float("inf"))):
        assert call(bad(**kw)) == -2, kw
        assert "bad argument" in lib.oc_last_error().decode()
    # without the above-threshold map the threshold is not read
    assert call(bad(d_above=None, threshold=float("nan"))) == 0
    assert lib.oc_density_accum(ctx.h, C.byref(s.acc), 5, None, None, None, stream) == -2     # agents without arrays
    assert lib.oc_density_accum(ctx.h, C.byref(s.acc), 0, None, None, None, stream) == 0      # no agents
    # the batched call checks every member
    n = 2
    hs = (C.c_void_p * n)(ctx.h.value, ctx.h.value)
    a0, a1 = _lib.DensityAcc.from_buffer_copy(s.acc), _lib.DensityAcc.from_buffer_copy(s.acc)
    a1.every = 0
    accs = (C.c_void_p * n)(C.addressof(a0), C.addressof(a1))
    Ns = np.array([50, 50], dtype=np.int32)
    ptr = lambda k: (C.c_void_p * n)(d[k].data_ptr(), d[k].data_ptr())
    multi = lambda: lib.oc_density_accum_multi(n, hs, accs, Ns.ctypes.data_as(_lib.ip), ptr("x"), ptr("y"),
                                               ptr("status"), stream)
    assert multi() == -2
    a1.every = 1
    assert multi() == 0
    hs[1] = None
    assert multi() == -2
    torch.cuda.synchronize()
    ctx.close()


def test_member_context_on_another_device_is_refused():
    import torch
    from optimal_crowds_b200 import _lib
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.RandomState(3)
    c0 = _ctx(40, 64)
    with torch.cuda.device(1):
        c1 = _lib.Context(c0.room_length, c0.room_height, 0.05, device=1)
        s1 = _stats(c1, _walls(c1, rng), 0.5)
        d1 = _dev_crowd(c1, *_crowd(c1, rng, 20))
    s0 = _stats(c0, _walls(c0, rng), 0.5)
    d0 = _dev_crowd(c0, *_crowd(c0, rng, 20))
    with pytest.raises(_lib.OcError, match="another device"):
        _lib.density_accum_multi([c0, c1], [s0, s1], [d0, d1])
    c0.close(); c1.close()


def test_run_with_bad_accumulator_is_refused_before_any_step(in_repo_cwd):
    from optimal_crowds_b200 import _lib, simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 1.0, rng=np.random.RandomState(1), density_stats=True)
        simu._solve_all()
    simu._dstats.acc.every = 0
    before = simu._np_random.get_state()
    with pytest.raises(_lib.OcError, match="every"):
        simu.advance(5)
    assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
    simu._dstats.acc.every = 1
    with pytest.raises(_lib.OcError, match="sigma"):
        simu._dstats.acc.sigma = float("nan")
        simu.advance(5)
