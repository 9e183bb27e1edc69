"""GPU tests of the Voronoi maps (``voronoi_maps=``; oc_vormap_accum, oc_vormap_accum_multi,
oc_gcfm_run_observed_maps): frames of adversarial crowds, batched frames, runs on every step path and ensembles.  Every
comparison is bit for bit; the reference is the Python restatement in tests/vormap_oracle.py (a brute-force owner
search, no bins), applied to chosen crowds and to the trajectory record and exit steps of the run without maps."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest

from test_gpu_areas import _state
from test_gpu_density_stats import _ctx, _same, _walls
from vormap_oracle import add, empty, frame, run_maps

pytestmark = pytest.mark.gpu

ACC = ("density_sum", "density_max", "covered", "speed_sum", "vx_sum", "vy_sum")


@pytest.fixture()
def in_repo_cwd(monkeypatch):
    from conftest import REPO
    monkeypatch.chdir(REPO)


def _maps(ctx, V, cutoff, edges, N, every=1):
    from optimal_crowds_b200 import _lib
    return _lib.VoronoiMaps(ctx, ctx.to_device(V), cutoff, edges, every, N)


def _assert_acc(got, want, tag):
    for k in ACC:
        assert _same(got[k], want[k]), (tag, k, int(np.sum(~(got[k] == want[k]))))
    assert got["frames"] == want["frames"], tag


def _read(maps):
    import torch
    torch.cuda.synchronize()
    return maps.result()


def _crowd(rng, ctx, N, r):
    """agents in and around the room; exactly on nodes; groups around a node at exactly the same distance (ties: the
    offsets are powers of two, so every difference is exact); coincident agents; far outside the room, NaN positions
    and velocities; status 0 and 2"""
    X, Y, L, H = ctx.X, ctx.Y, ctx.room_length, ctx.room_height
    x, y = rng.uniform(-0.5, L + 0.5, N), rng.uniform(-0.5, H + 0.5, N)
    vx, vy = rng.normal(0, 0.9, N), rng.normal(0, 0.9, N)
    st = rng.choice(np.array([0, 1, 1, 1, 1, 1, 1, 1, 1, 2], dtype=np.uint8), N)
    perm = rng.permutation(N)
    j = 0
    while j + 4 <= N // 3:
        kind = (j // 4) % 4
        ix, iy = rng.randint(2, len(X) - 2), rng.randint(2, len(Y) - 2)
        a = perm[j:j + 4]
        if kind == 0:                                                  # on nodes
            x[a], y[a] = X[ix], Y[iy]
            x[a[1:]], y[a[1:]] = X[ix + 1], Y[iy - 1]
        elif kind == 1:                                                # four at exactly 1/32 m from one node
            h = 0.03125
            x[a] = X[ix] + np.array([h, -h, 0.0, 0.0])
            y[a] = Y[iy] + np.array([0.0, 0.0, h, -h])
        elif kind == 2:                                                # two pairs of coincident agents
            x[a], y[a] = x[a[0]], y[a[0]]
            x[a[2:]], y[a[2:]] = x[a[0]] + r, y[a[0]]
        else:                                                          # two at exactly 1/64 m on either side
            x[a[:2]], y[a[:2]] = X[ix] + np.array([0.015625, -0.015625]), Y[iy]
        st[a] = 1
        j += 4
    if N >= 12:
        rest = perm[j:j + 10]
        x[rest[0]] = np.nan
        y[rest[1]] = np.nan
        vx[rest[2]], vy[rest[2]] = np.nan, 0.0
        x[rest[3]], y[rest[3]] = 1e300, 1.0
        x[rest[4]], y[rest[4]] = -1e300, -1e300
        x[rest[5]], y[rest[5]] = -0.3, H / 2
        x[rest[6]], y[rest[6]] = L + 0.2, H + 0.1
        st[rest[:7]] = 1
    return x, y, vx, vy, st


def _frame(ctx, V, cutoff, edges, c):
    return frame(ctx.X, ctx.Y, V, ctx.room_length, ctx.room_height, cutoff, edges, *c)


# --------------------------------------------------------------------------------------------- 1. kernels
@pytest.mark.parametrize("N", [0, 1, 255, 256, 257, 20011])
def test_frames_equal_the_oracle(N):
    rng = np.random.RandomState(N + 3)
    ctx = _ctx(241, 401) if N > 1000 else _ctx(121, 201)             # Nx, Ny not multiples of the 32 x 8 tile
    V = _walls(ctx, rng, frac=0.1)
    cutoff, edges = (0.25, 12) if N > 1000 else (0.6, 10)
    maps = _maps(ctx, V, cutoff, edges, N)
    want = empty((ctx.Ny, ctx.Nx))
    frames = 2 if N > 1000 else 3
    for f in range(frames):
        c = _crowd(rng, ctx, N, cutoff)
        ctx.vormap_accum(maps, _state(ctx, *c))
        t = _frame(ctx, V, cutoff, edges, c)
        add(want, t)
        got = _read(maps)
        _assert_acc(got, want, (N, f))
        if N > 250:
            assert t["covered"].sum() > 1000 and np.isfinite(t["rho"]).all()
        assert not got["covered"][V < 0].any() and (got["density_sum"][V < 0] == 0).all()
    r = _read(maps)
    assert r["frames"] == frames and _same(r["density"], want["density_sum"] / frames)
    cov = want["covered"]
    with np.errstate(invalid="ignore", divide="ignore"):
        assert _same(r["speed"], np.where(cov == 0, np.nan, want["speed_sum"] / np.maximum(cov, 1)))
        assert r["velocity"].shape == (ctx.Ny, ctx.Nx, 2)
        assert _same(r["velocity"][..., 1], np.where(cov == 0, np.nan, want["vy_sum"] / np.maximum(cov, 1)))
    ctx.close()


def test_ties_and_coincident_agents_go_to_the_lowest_index():
    from vormap_oracle import owners
    ctx = _ctx(61, 101)
    V = np.zeros((ctx.Ny, ctx.Nx))
    X, Y = ctx.X, ctx.Y
    h = 0.03125
    # four agents at exactly h from node (30, 20), in index order 3, 1, 0, 2 around it; a coincident pair elsewhere
    x = np.array([X[30], X[30] - h, X[30], X[30] + h, 1.0, 1.0])
    y = np.array([Y[20] + h, Y[20], Y[20] - h, Y[20], 2.0, 2.0])
    vx, vy, st = np.arange(6.0), -np.arange(6.0), np.ones(6, np.uint8)
    own = owners(X, Y, x, y, np.ones(6, bool), 0.5)
    assert own[20, 30] == 0
    near = np.argmin(np.abs(X - 1.0)), np.argmin(np.abs(Y - 2.0))
    assert own[near[1], near[0]] == 4
    maps = _maps(ctx, V, 0.5, 12, 6)
    ctx.vormap_accum(maps, _state(ctx, x, y, vx, vy, st))
    want = add(empty((ctx.Ny, ctx.Nx)), _frame(ctx, V, 0.5, 12, (x, y, vx, vy, st)))
    got = _read(maps)
    _assert_acc(got, want, "ties")
    assert got["vx_sum"][20, 30] == 0.0 and got["vx_sum"][near[1], near[0]] == 4.0
    ctx.close()


@pytest.mark.parametrize("n_ring, overflow", [(80, True), (40, False)])
def test_an_overflowing_cell_is_nan_only_at_its_nodes(n_ring, overflow):
    ctx = _ctx(121, 201)
    V = np.zeros((ctx.Ny, ctx.Nx))
    t = np.linspace(0, 2 * np.pi, n_ring, endpoint=False)
    rng = np.random.RandomState(n_ring)
    fx, fy = rng.uniform(6.5, 9.5, 30), rng.uniform(0.2, 2.5, 30)
    x = np.r_[fx, 3.0, 3.0 + 0.5 * np.cos(t)]
    y = np.r_[fy, 3.0, 3.0 + 0.5 * np.sin(t)]
    N = len(x)
    vx, vy, st = rng.normal(size=N), rng.normal(size=N), np.ones(N, np.uint8)
    maps = _maps(ctx, V, 1.0, 12, N)
    for _ in range(2):
        ctx.vormap_accum(maps, _state(ctx, x, y, vx, vy, st))
    tt = _frame(ctx, V, 1.0, 12, (x, y, vx, vy, st))
    want = add(add(empty((ctx.Ny, ctx.Nx)), tt), tt)
    got = _read(maps)
    _assert_acc(got, want, n_ring)
    nan = np.isnan(got["density_sum"])
    assert np.array_equal(nan, tt["owner"] == 30 if overflow else np.zeros_like(nan))
    assert nan.sum() > 0 if overflow else True
    assert np.array_equal(np.isnan(got["density_max"]), nan) and (got["covered"][nan] == 2).all()
    assert np.isfinite(got["density_sum"][tt["owner"] < 30]).all() and (got["covered"] > 0).sum() > nan.sum()
    ctx.close()


def test_batched_frames_equal_every_member_alone():
    from optimal_crowds_b200 import _lib
    rng = np.random.RandomState(5)
    sizes = [(75, 131, 700), (64, 90, 0), (40, 64, 1), (97, 97, 257), (33, 47, 3000), (121, 201, 256)]
    cuts = [(1.0, 12), (0.5, 8), (2.0, 32), (0.25, 4), (0.75, 16), (3.0, 12)]
    ctxs, multi, alone, states, Vs = [], [], [], [], []
    for (ny, nx, N), (cut, edges) in zip(sizes, cuts):
        c = _ctx(ny, nx)
        V = _walls(c, rng, frac=0.2)
        ctxs.append(c)
        Vs.append(V)
        multi.append(_maps(c, V, cut, edges, N))
        alone.append(_maps(c, V, cut, edges, N))
        states.append(_crowd(rng, c, N, cut))
    dev = [_state(c, *s) for c, s in zip(ctxs, states)]
    for rep in range(2):
        n0 = _lib.launch_count()
        _lib.vormap_accum_multi(ctxs, multi, dev)
        assert _lib.launch_count() - n0 == 6
        for c, a, d in zip(ctxs, alone, dev):
            c.vormap_accum(a, d)
        for q in range(len(sizes)):
            _assert_acc(_read(multi[q]), _read(alone[q]), (rep, q))
    for q in (0, 3, 5):
        t = _frame(ctxs[q], Vs[q], *cuts[q], states[q])
        _assert_acc(_read(multi[q]), add(add(empty(Vs[q].shape), t), t), q)
    for c in ctxs:
        c.close()


# --------------------------------------------------------------------------------------------- 2. runs
T_RUN = {"room_test": 1.2, "metro_station": 1.2, "slalom": 1.2}
SPEC = dict(every=3, cutoff=0.8, edges=10)


def _run(room, seed, record=True, fast=True, monkeypatch=None, **kw):
    from optimal_crowds_b200 import simulations
    monkeypatch.setenv("OC_FAST_RUN", "1" if fast else "0")
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation(room, T_RUN[room], recompute=True, record=record, rng=np.random.RandomState(seed),
                                      **kw)
        simu.run()
    simu._sync_host()
    return simu


@pytest.mark.parametrize("room", ["room_test", "metro_station", "slalom"])
def test_run_maps_equal_the_oracle_on_the_record(room, in_repo_cwd, monkeypatch):
    from optimal_crowds_b200 import _lib, simulations
    seed = 4
    ref = _run(room, seed, monkeypatch=monkeypatch)
    assert ref.simu_step > 50                                            # the run re-solved at step 50
    want = run_maps(ref._ctx.X, ref._ctx.Y, ref.V, ref.room_length, ref.room_height, SPEC["cutoff"], SPEC["edges"],
                    SPEC["every"], ref._track, ref._exit_step, ref.simu_step)
    assert (want["covered"] > 0).sum() > 100 and (want["speed_sum"] > 0).any()
    frames = len(simulations.density_frame_steps(ref.T, ref.dt, SPEC["every"], ref.recompute_step))
    for path in ("block", "steps", "no_record"):
        n0 = _lib.launch_count()
        simu = _run(room, seed, record=path != "no_record", fast=path == "block", monkeypatch=monkeypatch,
                    voronoi_maps=SPEC)
        r = simu.voronoi_maps()
        assert r["cutoff"] == 0.8 and r["edges"] == 10
        _assert_acc(r, want, path)
        if ref.inside > 0:
            assert r["frames"] == frames
        # nothing else changed: trajectories, exits, clocks, the generator's state
        assert simu.simu_step == ref.simu_step and simu.time == ref.time and simu.inside == ref.inside
        assert simu._exit_order == ref._exit_order and np.array_equal(simu._exit_step, ref._exit_step)
        assert _same(simu._h_now, ref._h_now) and _same(simu._h_timev, ref._h_timev)
        if path != "no_record":
            for ra, rb in zip(simu._track, ref._track):
                assert _same(ra, rb)
        sa, sb = simu._np_random.get_state(), ref._np_random.get_state()
        assert sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]
        if path == "block":
            # off means off: the run without maps launches exactly six kernels fewer per frame
            n1 = _lib.launch_count()
            plain = _run(room, seed, monkeypatch=monkeypatch)
            assert (n1 - n0) - (_lib.launch_count() - n1) == 6 * r["frames"]
            with pytest.raises(RuntimeError, match="without voronoi_maps"):
                plain.voronoi_maps()


def test_bare_steps_take_no_frame(in_repo_cwd):
    from optimal_crowds_b200 import simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 0.5, rng=np.random.RandomState(2), voronoi_maps=dict(every=2))
        simu._solve_all()
        for _ in range(5):
            simu.step(simu.dt)
        r = simu.voronoi_maps()
        assert r["frames"] == 0 and r["density"] is None and (r["covered"] == 0).all()
        assert np.isnan(r["speed"]).all() and (r["density_sum"] == 0).all()
        simu.advance(6)                                                  # simu_step 5 .. 10: frames at 6, 8, 10
    r = simu.voronoi_maps()
    assert r["frames"] == 3
    acc = empty((simu.Ny, simu.Nx))
    for k in (6, 8, 10):
        row = simu._track[k]
        st = ((simu._exit_step < 0) | (simu._exit_step >= k)).astype(np.uint8)
        add(acc, frame(simu._ctx.X, simu._ctx.Y, simu.V, simu.room_length, simu.room_height, 1.0, 12, row[:, 0],
                       row[:, 1], row[:, 2], row[:, 3], st))
    _assert_acc(r, acc, "bare")


# --------------------------------------------------------------------------------------------- 3. ensembles
ENS_ROOMS = ["room_test", "exit_opposite", "metro_station", "slalom"]
ENS_SEEDS = [3, 4, 7, 9]
ENS_CONFIGS = [None, {"dt": 0.025}, {"sigma_convolution": 0.4}, None]
ENS_SPEC = dict(every=2, cutoff=0.9, edges=11)
T_ENS = 1.3
_ALONE = {}


def _alone(i):
    if i not in _ALONE:
        from optimal_crowds_b200 import simulations
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(ENS_ROOMS[i], T_ENS, recompute=True, rng=np.random.RandomState(ENS_SEEDS[i]),
                                          config=ENS_CONFIGS[i], voronoi_maps=ENS_SPEC)
            simu.run()
        _ALONE[i] = simu.voronoi_maps()
    return _ALONE[i]


@pytest.mark.parametrize("batched", [True, False], ids=["batched_steps", "member_steps"])
def test_ensemble_members_equal_their_standalone_maps(batched, in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    from test_gpu_density_stats import _assert_same_results
    res = ensemble.ensemble(ENS_ROOMS, T_ENS, ENS_SEEDS, recompute=True, configs=ENS_CONFIGS, batched_steps=batched,
                            voronoi_maps=ENS_SPEC).run()
    plain = ensemble.ensemble(ENS_ROOMS, T_ENS, ENS_SEEDS, recompute=True, configs=ENS_CONFIGS,
                              batched_steps=batched).run()
    for i in range(len(ENS_SEEDS)):
        got, want = res[i].pop("voronoi_maps"), _alone(i)
        _assert_acc(got, want, i)
        assert got["frames"] > 0 and (got["covered"] > 0).any()
        assert "voronoi_maps" not in plain[i]
    _assert_same_results(res, plain)


# --------------------------------------------------------------------------------------------- 4. errors
def test_bad_map_accumulators_are_refused_before_any_launch():
    import torch
    from optimal_crowds_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(2)
    ctx = _ctx(40, 64)
    V = np.zeros((ctx.Ny, ctx.Nx))
    maps = _maps(ctx, V, 0.5, 12, 300)
    d = _state(ctx, *_crowd(rng, ctx, 300, 0.5))
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda k: _lib._dev(d[k])

    def call(a, N=300, drop=None):
        return lib.oc_vormap_accum(ctx.h, a, N, *[None if k == drop else P(k) for k in ("x", "y", "vx", "vy",
                                                                                       "status")], stream)

    def bad(**kw):
        a = _lib.VormapAcc.from_buffer_copy(maps.acc)
        for k, v in kw.items():
            setattr(a, k, v)
        return C.byref(a)

    assert call(C.byref(maps.acc)) == 0
    bx = maps.acc.bins_x
    cases = [(None, {}), (bad(cutoff=0.0), {}), (bad(cutoff=-1.0), {}), (bad(cutoff=100.5), {}),
             (bad(cutoff=float("nan")), {}), (bad(cutoff=float("inf")), {}), (bad(edges=3), {}), (bad(edges=33), {}),
             (bad(every=0), {}), (bad(every=-1), {}), (bad(bins_x=0), {}), (bad(bins_x=bx + 1), {}),
             (bad(bins_x=257, bin_capacity=1 << 20), {}), (bad(bin_capacity=1), {}), (bad(agent_capacity=299), {}),
             (bad(d_vol=None), {}), (bad(d_order=None), {}), (bad(d_covered=None), {}), (bad(d_Vglobal=None), {}),
             (bad(d_ring=None), {}), (bad(d_density_max=None), {}), (C.byref(maps.acc), dict(drop="vy")),
             (C.byref(maps.acc), dict(drop="status"))]
    n0 = _lib.launch_count()
    for a, kw in cases:
        assert call(a, **kw) == -2, kw
        assert "bad argument" in lib.oc_last_error().decode()
    assert call(bad(d_vol=None), N=0) == -2                               # the accumulator is checked whatever N
    assert _lib.launch_count() == n0                                      # nothing was launched
    assert call(C.byref(maps.acc), N=0, drop="x") == 0                    # no agents: no agent arrays read
    # the batched call checks every member, and refuses members that share bins, scratch or accumulators
    other = _maps(ctx, V, 0.5, 12, 300)
    a0, a1 = _lib.VormapAcc.from_buffer_copy(maps.acc), _lib.VormapAcc.from_buffer_copy(other.acc)
    hs = (C.c_void_p * 2)(ctx.h.value, ctx.h.value)
    accs = (C.c_void_p * 2)(C.addressof(a0), C.addressof(a1))
    Ns = np.array([300, 300], dtype=np.int32)
    ptr = lambda k: (C.c_void_p * 2)(d[k].data_ptr(), d[k].data_ptr())
    multi = lambda: lib.oc_vormap_accum_multi(2, hs, accs, Ns.ctypes.data_as(_lib.ip), ptr("x"), ptr("y"), ptr("vx"),
                                              ptr("vy"), ptr("status"), stream)
    n0 = _lib.launch_count()
    for k in ("d_bin_count", "d_bin_start", "d_slot", "d_order", "d_vol", "d_density_sum", "d_density_max",
              "d_covered", "d_speed_sum", "d_vx_sum", "d_vy_sum"):
        setattr(a1, k, getattr(maps.acc, k))
        assert multi() == -2 and "share" in lib.oc_last_error().decode(), k
        setattr(a1, k, getattr(other.acc, k))
    a1.every = 0
    assert multi() == -2
    a1.every = 1
    Ns[1] = 301
    assert multi() == -2
    assert _lib.launch_count() == n0
    Ns[1] = 300
    assert multi() == 0
    torch.cuda.synchronize()
    ctx.close()


def test_runs_with_bad_map_accumulators_are_refused_before_any_step(in_repo_cwd):
    from optimal_crowds_b200 import _lib, simulations
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation("room_test", 1.0, rng=np.random.RandomState(1), voronoi_maps=True)
        simu._solve_all()
    before = simu._np_random.get_state()
    for k, v, match in (("d_vol", None, "NULL"), ("edges", 40, "edges"), ("every", 0, "every"),
                        ("agent_capacity", 1, "capacity")):
        keep = getattr(simu._vmaps.acc, k)
        setattr(simu._vmaps.acc, k, v)
        n0 = _lib.launch_count()
        with pytest.raises(_lib.OcError, match=match):
            simu.advance(5)
        assert _lib.launch_count() == n0
        assert simu.simu_step == 0 and simu._np_random.get_state()[2] == before[2]
        setattr(simu._vmaps.acc, k, keep)
    assert simu.voronoi_maps()["frames"] == 0


def test_member_context_on_another_device_is_refused():
    import torch
    from optimal_crowds_b200 import _lib
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.RandomState(3)
    c0 = _ctx(40, 64)
    V = np.zeros((c0.Ny, c0.Nx))
    with torch.cuda.device(1):
        c1 = _lib.Context(c0.room_length, c0.room_height, 0.05, device=1)
        d1 = _state(c1, *_crowd(rng, c1, 20, 1.0))
        a1 = _maps(c1, V, 1.0, 12, 20)
    d0 = _state(c0, *_crowd(rng, c0, 20, 1.0))
    a0 = _maps(c0, V, 1.0, 12, 20)
    with pytest.raises(_lib.OcError, match="another device"):
        _lib.vormap_accum_multi([c0, c1], [a0, a1], [d0, d1])
    c0.close(); c1.close()
