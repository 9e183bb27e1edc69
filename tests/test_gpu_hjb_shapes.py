"""GPU parity of the batched HJB solve over rooms of different grids (oc_hjb_solve_grids): every room must equal
oc_hjb_solve on its own grid context bit for bit, and the CPU oracle to 1e-10, whatever the shapes it shares the batched
launches with; oc_hjb_solve_multi is the same call with every grid = ctx."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_hjb_sampling import NE_MAX, samples_per_attempt

pytestmark = pytest.mark.gpu

RTOL = 1e-10
OC_ERR_ARG = -2


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    return torch


def _ctx(Ny, Nx, step=0.05):
    from optimal_crowds_b200 import _lib
    return _lib.Context((Nx - 1) * step + step / 2, (Ny - 1) * step + step / 2, step)


def _room_V(Ny, Nx, b):
    """frame walls, an interior wall block and a door on the right edge, placed relative to the grid"""
    V = np.zeros((Ny, Nx)); V[0, :] = V[-1, :] = V[:, 0] = V[:, -1] = -100
    if Ny > 12 and Nx > 12:
        y0, x0 = Ny // 4 + b % 3, Nx // 3
        V[y0:y0 + max(2, Ny // 10), x0:x0 + max(2, Nx // 6)] = -100
    V[Ny // 2 - 2:Ny // 2 + 2, -1] = 1.0
    return V


# (Ny, Nx, grid step, sigma, mu, g, T, nt, density, chunk_rows): pairwise different shapes; 121 x 201 has an odd Nx (LDGSTS
# staging), 8 x 10 is the smallest grid of the fused kernel, 50 x 90 has grid step 0.1, and the 70 x 150 room samples
# densely enough for steps with more than NE_MAX samples (phi output)
ROOMS = [(70, 150, 0.05, 0.22, 5.5, 0.01, 1.0, 101, True, 32),
         (64, 128, 0.05, 0.2, 5.0, -0.005, 0.5, 25, False, 0),
         (121, 201, 0.05, 0.25, 4.0, -0.02, 0.4, 21, True, 16),
         (8, 10, 0.05, 0.15, 6.0, 0.0, 0.6, 19, False, 0),
         (50, 90, 0.1, 0.3, 3.0, -0.05, 0.3, 13, True, 48),
         (96, 64, 0.05, 0.18, 4.5, -0.01, 0.45, 16, False, 0)]


@pytest.mark.parametrize("density", [True, False], ids=["density", "no_density"])
@pytest.mark.parametrize("store", ["phi", "velocity"])
def test_rooms_of_different_grids_equal_their_single_solves_and_the_oracle(store, density, cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    from optimal_crowds_b200.optimals import _merge_config
    from oracle import cpu_oracle as co
    vel = store == "velocity"
    rooms = list(ROOMS)
    if vel:   # velocity-only output: at most NE_MAX samples per step
        rooms[0] = rooms[0][:7] + (21,) + rooms[0][8:]
    rng = np.random.RandomState(11)
    grids, Vs, ms = [], [], []
    for b, (Ny, Nx, step, *_r, dens, _c) in enumerate(rooms):
        grids.append(_ctx(Ny, Nx, step))
        Vs.append(_room_V(Ny, Nx, b))
        ms.append(rng.uniform(0, 1, size=(Ny, Nx)) if density and dens else None)
    solver = _ctx(30, 40)   # owns the workspace; its own grid is none of the rooms'
    dV = [g.to_device(v) for g, v in zip(grids, Vs)]
    dm = [g.to_device(m) if m is not None else None for g, m in zip(grids, ms)]
    prm = _lib.hjb_params(cfg, fused=1)
    spec = [dict(sigma=s, mu=mu, g=g, T=T, nt=nt, chunk_rows=c) for (_, _, _, s, mu, g, T, nt, _, c) in rooms]
    res = solver.hjb_solve_grids(grids, dV, dm if density else None, spec, prm, want_vel=vel)
    for b, (Ny, Nx, step, sigma, mu, g, T, nt, _, chunk) in enumerate(rooms):
        prm_b = _lib.hjb_params(_merge_config(cfg, {"hjb_params": dict(sigma=sigma, mu=mu, g=g)}), fused=1,
                                chunk_rows=chunk)
        one = grids[b].hjb_solve(dV[b], dm[b], prm_b, T, nt, want_phi=not vel, want_vel=vel, trace=True)
        st = res[b]["stats"]
        assert st["status"] == 0 and st["n_out"] == nt
        for k in ("nfev", "n_accepted", "n_rejected"):
            assert st[k] == one["stats"][k], (b, k)
        phi_ref, st_ref, h_ref, e_ref = co.hjb_solve(Vs[b], ms[b], T, nt, sigma=sigma, mu=mu, g=g, dx=step, dy=step)
        assert st_ref["nfev"] == st["nfev"], b
        if b == 0 and not vel:
            assert max(samples_per_attempt(T, nt, h_ref, e_ref)) > NE_MAX
        if vel:
            assert res[b]["vx"].shape == (nt - 1, Ny - 2, Nx - 2)
            assert torch_mod.equal(res[b]["vx"], one["vx"]) and torch_mod.equal(res[b]["vy"], one["vy"]), b
            vx_ref, vy_ref = co.fill_field(phi_ref, Ny, Nx, mu=mu, dx=step, dy=step)
            assert np.abs(res[b]["vx"].cpu().numpy() - vx_ref).max() < RTOL
            assert np.abs(res[b]["vy"].cpu().numpy() - vy_ref).max() < RTOL
        else:
            assert res[b]["phi"].shape == (nt, Ny, Nx)
            assert torch_mod.equal(res[b]["phi"], one["phi"]), b
            np.testing.assert_allclose(res[b]["phi"].cpu().numpy().reshape(nt, -1), phi_ref, rtol=RTOL)


def test_launches_mix_shapes_and_split_at_24(cfg, torch_mod, monkeypatch):
    """30 rooms of 5 shapes: every launch holds up to 24 rooms of any shapes.  Each room equals its solo solve and the
    same call with one launch per room and attempt (OC_BATCH_PER_ROOM); the mixed call issues fewer kernel launches than
    the five single-shape calls together, so rooms of different shapes did share launches"""
    from optimal_crowds_b200 import _lib
    shapes = [(40, 60), (33, 47), (64, 100), (20, 130), (90, 42)]
    order = [q % 5 for q in range(30)]       # interleaved: every launch window holds every shape
    ctxs = [_ctx(*sh) for sh in shapes]
    grids = [ctxs[s] for s in order]
    dV = [g.to_device(_room_V(g.Ny, g.Nx, b)) for b, g in enumerate(grids)]
    spec = [dict(sigma=0.2 + 0.002 * b, mu=5.0, g=-0.005, T=0.3, nt=13) for b in range(30)]
    prm = _lib.hjb_params(cfg, fused=1)
    solver = _ctx(30, 40)
    _lib.launch_count(reset=True)
    mixed = solver.hjb_solve_grids(grids, dV, None, spec, prm)
    n_mixed = _lib.launch_count(reset=True)
    n_single = 0
    for s in range(5):
        idx = [b for b in range(30) if order[b] == s]
        solver.hjb_solve_grids([grids[b] for b in idx], [dV[b] for b in idx], None, [spec[b] for b in idx], prm)
        n_single += _lib.launch_count(reset=True)
    assert n_mixed < n_single, (n_mixed, n_single)
    monkeypatch.setenv("OC_BATCH_PER_ROOM", "1")
    per_room = solver.hjb_solve_grids(grids, dV, None, spec, prm)
    monkeypatch.delenv("OC_BATCH_PER_ROOM")
    for b in range(30):
        r = spec[b]
        prm_b = _lib.hjb_params(cfg, fused=1)
        prm_b.sigma = r["sigma"]
        one = grids[b].hjb_solve(dV[b], None, prm_b, r["T"], r["nt"], want_phi=True, want_vel=False)
        for other in (mixed, per_room):
            assert other[b]["stats"]["nfev"] == one["stats"]["nfev"], b
            assert other[b]["stats"]["n_rejected"] == one["stats"]["n_rejected"], b
            assert torch_mod.equal(other[b]["phi"], one["phi"]), b


def test_launch_table_splits_rooms_it_cannot_describe(cfg, torch_mod, monkeypatch):
    """24 rooms of 71 CTAs each (one tile column, 71 chunks of 16 rows): 1704 CTAs whose first CTAs are not multiples of
    any power of two, more than the launch's CTA-to-room table holds at shift 0, so the launch takes fewer rooms.  Every
    room still equals the same call with one launch per room and attempt"""
    from optimal_crowds_b200 import _lib
    g = _ctx(1136, 60)
    dV = [g.to_device(_room_V(1136, 60, b)) for b in range(24)]
    spec = [dict(sigma=0.2 + 0.001 * b, mu=5.0, g=-0.005, T=0.1, nt=3, chunk_rows=16) for b in range(24)]
    prm = _lib.hjb_params(cfg, fused=1)
    solver = _ctx(30, 40)
    batched = solver.hjb_solve_grids([g] * 24, dV, None, spec, prm)
    monkeypatch.setenv("OC_BATCH_PER_ROOM", "1")
    per_room = solver.hjb_solve_grids([g] * 24, dV, None, spec, prm)
    for b in range(24):
        assert batched[b]["stats"]["nfev"] == per_room[b]["stats"]["nfev"], b
        assert torch_mod.equal(batched[b]["phi"], per_room[b]["phi"]), b


def test_multi_solve_treats_a_negative_chunk_rows_as_the_grid_plan(cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    ctx = _ctx(70, 150)
    dV = [ctx.to_device(_room_V(70, 150, b)) for b in range(2)]
    spec = [dict(sigma=0.2, mu=5.0, g=-0.005, T=0.3, nt=11)] * 2
    neg = ctx.hjb_solve_multi(dV, None, spec, _lib.hjb_params(cfg, fused=1, chunk_rows=-16))
    zero = ctx.hjb_solve_multi(dV, None, spec, _lib.hjb_params(cfg, fused=1))
    for b in range(2):
        assert neg[b]["stats"]["nfev"] == zero[b]["stats"]["nfev"]
        assert torch_mod.equal(neg[b]["phi"], zero[b]["phi"])


def test_multi_solve_is_the_grids_solve_with_every_grid_ctx(cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    ctx = _ctx(70, 150)
    dV = [ctx.to_device(_room_V(70, 150, b)) for b in range(4)]
    rng = np.random.RandomState(3)
    dm = [ctx.to_device(rng.uniform(0, 1, (70, 150))) if b % 2 else None for b in range(4)]
    spec = [dict(sigma=0.2 + 0.02 * b, mu=5.0 - b, g=-0.005 * b, T=0.3 + 0.1 * b, nt=11 + 4 * b) for b in range(4)]
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=32)
    multi = ctx.hjb_solve_multi(dV, dm, spec, prm)
    grids = ctx.hjb_solve_grids([ctx] * 4, dV, dm, spec, prm)
    for b in range(4):
        for k in ("nfev", "n_accepted", "n_rejected"):
            assert multi[b]["stats"][k] == grids[b]["stats"][k]
        assert torch_mod.equal(multi[b]["phi"], grids[b]["phi"])


@pytest.mark.parametrize("bad", ["grids_null", "grid_entry_null", "other_device", "grid_too_small", "room_chunk_neg",
                                 "prm_chunk_neg"])
def test_grids_solve_input_checks(bad, cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    if bad == "other_device" and torch_mod.cuda.device_count() < 2:
        pytest.skip("needs a second GPU for a context on another device")
    ctx = _ctx(40, 60)
    g1 = _ctx(33, 47)
    grids = [ctx, g1]
    if bad == "other_device":
        with torch_mod.cuda.device(1):
            grids[1] = _lib.Context(g1.room_length, g1.room_height, 0.05, device=1)
    if bad == "grid_too_small":
        grids[1] = _ctx(7, 20)
    dV = [ctx.to_device(_room_V(40, 60, 0)), g1.to_device(_room_V(33, 47, 1))]
    phi = [ctx.empty(5, 40, 60), g1.empty(5, 33, 47)]
    prm = _lib.hjb_params(cfg, fused=1)
    t_eval = np.linspace(0.2, 0, 5)
    spec = (_lib.HjbRoom * 2)()
    for b in range(2):
        spec[b] = _lib.HjbRoom(0.2, 5.0, -0.005, 0.2, t_eval.ctypes.data_as(_lib.dp), 5, 0)
    if bad == "room_chunk_neg":
        spec[1].chunk_rows = -16
    if bad == "prm_chunk_neg":
        prm.chunk_rows = -16
    hs = None if bad == "grids_null" else (C.c_void_p * 2)(ctx.h.value, None if bad == "grid_entry_null" else
                                                          grids[1].h.value)
    st = (_lib.HjbStats * 2)()
    lib = _lib.load()
    rc = lib.oc_hjb_solve_grids(ctx.h, 2, hs, _lib._ptrs(dV, 2), None, spec, C.byref(prm), _lib._ptrs(phi, 2), None,
                                None, st, _lib._stream())
    assert rc == OC_ERR_ARG, lib.oc_last_error()
    # the context keeps working
    spec[1].chunk_rows = 0
    ok = lib.oc_hjb_solve_grids(ctx.h, 2, (C.c_void_p * 2)(ctx.h.value, g1.h.value), _lib._ptrs(dV, 2), None, spec,
                                C.byref(_lib.hjb_params(cfg, fused=1)), _lib._ptrs(phi, 2), None, None, st, _lib._stream())
    assert ok == 0 and st[1].n_out == 5
