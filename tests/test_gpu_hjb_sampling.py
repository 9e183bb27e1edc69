"""GPU parity of the stage-fused RK45 step at every number of dense-output samples per step attempt.

One launch of ``hjb_fused_kernel<NE>`` writes the NE = 0..6 samples (``t_eval`` points) that the attempt crosses; an
attempt that crosses more (a step much longer than the sample spacing: small ``dt`` in config.json, or a dense
``t_eval``) is launched again for the remaining samples.  The tests below cover every NE, the attempts above six in the
single, batched and row-band solves, grid tails (a last 112-column tile with one or two valid columns, a last row chunk
of a single row), the host-side error reduction of grids with more row chunks than the in-launch reduction stages, and
ensemble members at ``dt = 0.01`` against stand-alone runs.  Every test checks, from the step trace, that its runs
really contain the sample counts it is about, so that a change of the controller cannot make it vacuous.

Pass bar against the CPU oracle (plain C restatement of scipy's RK45): identical nfev / accepted / rejected counts,
step sizes to 1e-11, phi to 1e-10 relative, velocities to 1e-10 absolute.
"""
import contextlib
import io
import json
import os
from collections import Counter

import numpy as np
import pytest

from conftest import REPO

pytestmark = pytest.mark.gpu

NE_MAX = 6          # fused::NE_MAX, samples per launch
BATCH_MAX = 24      # fused::BATCH_MAX, rooms per batched launch
MAX_FINAL_ROWS = 1552  # fused::MAX_FINAL_ROWS, row chunks the in-launch final reduction can stage
VX = 112            # fused::VX, valid columns per tile
OC_ERR_ARG = -2


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    return torch


def samples_per_attempt(T, nt, trace_h, trace_err):
    """histogram {samples: attempts} of the step trace of a solve with t_eval = linspace(T, 0, nt), rejected attempts
    included: an attempt from t to t+h (h < 0) emits the not yet emitted t_eval points in [t+h, t]; only an accepted
    attempt (error norm < 1) moves t and the emitted count on"""
    t_eval = np.linspace(T, 0, nt)
    hist = Counter()
    t, done = T, 0
    for h, err in zip(trace_h, trace_err):
        t_new = t + h
        j = done
        while j < nt and t_eval[j] >= t_new:
            j += 1
        hist[j - done] += 1
        if err < 1:
            t, done = t_new, j
    assert done == nt, "the trace does not reach t = 0"
    return hist


def _lengths(Ny, Nx):
    from optimal_crowds_b200 import _lib
    L, H = (Nx - 1) * 0.05 + 0.025, (Ny - 1) * 0.05 + 0.025
    assert _lib.grid_shape(L, H, 0.05) == (Ny, Nx)
    return L, H


def _frame(Ny, Nx):
    V = np.zeros((Ny, Nx))
    V[0, :] = V[-1, :] = V[:, 0] = V[:, -1] = -100
    return V


def _ragged_room(Ny, Nx):
    """walls, doors on the right and bottom frame, an interior obstacle, a random density (as the ragged-grid test)"""
    rng = np.random.RandomState(Ny)
    V = _frame(Ny, Nx)
    V[Ny // 3: Ny // 3 + 3, Nx // 4: Nx // 2] = -100
    V[Ny // 2 - 2: Ny // 2 + 2, -1] = 1.0
    V[0, 5:9] = 1.0
    return V, rng.uniform(0, 1, (Ny, Nx))


def _room_b(Ny, Nx, b, rng):
    """room b of a batch: obstacle, door and density (odd b) differ from room to room"""
    V = _frame(Ny, Nx)
    r0 = 10 + (b * 7) % (Ny - 30)
    V[r0:r0 + 4, Nx // 4:Nx // 4 + 10 + (b * 13) % (Nx // 2)] = -100
    d = 3 + (b * 5) % (Ny - 20)
    V[d:d + 6, -1] = 1.0
    if b % 3 == 0:
        V[0, 5 + b % 20:12 + b % 20] = 1.0
    m = rng.uniform(0, 1, (Ny, Nx)) if b % 2 else None
    return V, m


def _assert_matches_oracle(res, ref, Ny, Nx, nt, phi=True, vel=True):
    """res: a solver result dict; ref: co.hjb_solve's (phi, stats, trace_h, trace_err) of the same room"""
    from oracle import cpu_oracle as co
    phi_ref, st_ref, h_ref, _ = ref
    st = res["stats"]
    assert st["status"] == 0 and st["n_out"] == nt
    assert (st["nfev"], st["n_accepted"], st["n_rejected"]) == (st_ref["nfev"], st_ref["n_accepted"], st_ref["n_rejected"])
    if "trace_h" in res:
        np.testing.assert_allclose(res["trace_h"], h_ref, rtol=1e-11, atol=0)
    if phi:
        np.testing.assert_allclose(res["phi"].cpu().numpy().reshape(nt, -1), phi_ref, rtol=1e-10, atol=0)
    if vel and nt > 1:
        vx_ref, vy_ref = co.fill_field(phi_ref, Ny, Nx)
        assert np.abs(res["vx"].cpu().numpy() - vx_ref).max() < 1e-10
        assert np.abs(res["vy"].cpu().numpy() - vy_ref).max() < 1e-10


# ---------------------------------------------------------------------------------------------------------------------
# a. single solve: NE = 0..6 and > 6, TMA (even Nx) and cp.async (odd Nx) staging, one- and two-column last tiles,
#    a one-row last chunk
@pytest.mark.parametrize("chunk_rows", [16, 48])
@pytest.mark.parametrize("shape", [(97, 226), (97, 225), (50, 113)], ids=["tma_2col", "cpasync_1col", "cpasync_small"])
def test_single_solve_every_sample_count_and_grid_tail(shape, chunk_rows, cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    Ny, Nx = shape
    assert Nx % VX in (1, 2) and Ny % chunk_rows in (1, 2)   # last tile / last row chunk
    T = 0.5
    L, H = _lengths(Ny, Nx)
    V, m = _ragged_room(Ny, Nx)
    ctx = _lib.Context(L, H, 0.05)
    Vd, md = ctx.to_device(V), ctx.to_device(m)
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=chunk_rows)
    seen = Counter()
    for nt in (3, 21, 41, 101):
        ref = co.hjb_solve(V, m, T, nt)
        res = ctx.hjb_solve(Vd, md, prm, T, nt, want_phi=True, want_vel=True, trace=True)
        _assert_matches_oracle(res, ref, Ny, Nx, nt)
        seen += samples_per_attempt(T, nt, res["trace_h"], res["trace_err"])
        # velocity-only output: NE_MAX scratch slices, stage-wise attempts above NE_MAX samples
        vel = ctx.hjb_solve(Vd, md, prm, T, nt, want_phi=False, want_vel=True, trace=True)
        assert vel["phi"] is None
        _assert_matches_oracle(vel, ref, Ny, Nx, nt, phi=False)
    assert set(range(NE_MAX + 1)) <= set(seen), sorted(seen)
    assert max(seen) > NE_MAX, sorted(seen)
    ctx.close()


def test_stagewise_solve_at_every_sample_count(cfg, torch_mod):
    """control: the stage-wise kernels (fused=0) on the same room and sample counts"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    Ny, Nx, T = 97, 225, 0.5
    V, m = _ragged_room(Ny, Nx)
    ctx = _lib.Context(*_lengths(Ny, Nx), 0.05)
    seen = Counter()
    for nt in (3, 21, 41, 101):
        ref = co.hjb_solve(V, m, T, nt)
        res = ctx.hjb_solve(ctx.to_device(V), ctx.to_device(m), _lib.hjb_params(cfg, fused=0), T, nt, want_phi=True,
                            trace=True)
        _assert_matches_oracle(res, ref, Ny, Nx, nt)
        seen += samples_per_attempt(T, nt, res["trace_h"], res["trace_err"])
    assert set(range(NE_MAX + 1)) <= set(seen) and max(seen) > NE_MAX, sorted(seen)
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# b. more row chunks than the in-launch final reduction can stage: the error sum is made on the host
@pytest.mark.parametrize("nt", [10, 41])
def test_host_side_error_reduction(nt, cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    Ny, Nx, T, rows = 24850, 12, 0.2, 16
    assert -(-Ny // rows) > MAX_FINAL_ROWS
    V = _frame(Ny, Nx)
    V[Ny // 2:Ny // 2 + 40, -1] = 1.0
    V[5000:5003, 3:8] = -100
    m = np.random.RandomState(1).uniform(0, 1, (Ny, Nx))
    V2 = V.copy()
    V2[100:140, 0] = 1.0
    ctx = _lib.Context(*_lengths(Ny, Nx), 0.05)
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=rows)
    dV, dm = [ctx.to_device(V), ctx.to_device(V2)], [ctx.to_device(m), None]
    ref = co.hjb_solve(V, m, T, nt)
    one = ctx.hjb_solve(dV[0], dm[0], prm, T, nt, want_phi=True, trace=True)
    _assert_matches_oracle(one, ref, Ny, Nx, nt)
    hist = samples_per_attempt(T, nt, one["trace_h"], one["trace_err"])
    assert (max(hist) > NE_MAX) == (nt == 41), sorted(hist)
    # two rooms through the batched solve (per-room host reduction): each equals its single solve bit for bit
    batch = ctx.hjb_solve_batch(dV, dm, prm, T, nt)
    singles = [one, ctx.hjb_solve(dV[1], dm[1], prm, T, nt, want_phi=True)]
    for b in range(2):
        for k in ("nfev", "n_accepted", "n_rejected", "status", "n_out"):
            assert batch[b]["stats"][k] == singles[b]["stats"][k]
        assert torch_mod.equal(batch[b]["phi"], singles[b]["phi"])
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# c. batched solve at dense sampling: more rooms than one batched launch takes, attempts with up to ~25 samples
@pytest.mark.parametrize("nt", [61, 16])
@pytest.mark.parametrize("shape,n_rooms,chunk_rows", [((512, 512), 30, 0), ((97, 225), 26, 16)],
                         ids=["512sq_tma", "97x225_cpasync"])
def test_batched_solve_at_dense_sampling(shape, n_rooms, chunk_rows, nt, cfg, torch_mod, monkeypatch):
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    assert n_rooms > BATCH_MAX
    Ny, Nx = shape
    T = 0.3
    ctx = _lib.Context(*_lengths(Ny, Nx), 0.05)
    rng = np.random.RandomState(5)
    rooms = [_room_b(Ny, Nx, b, rng) for b in range(n_rooms)]
    dV = [ctx.to_device(V) for V, _ in rooms]
    dm = [ctx.to_device(m) if m is not None else None for _, m in rooms]
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=chunk_rows)
    monkeypatch.delenv("OC_BATCH_PER_ROOM", raising=False)
    batch = ctx.hjb_solve_batch(dV, dm, prm, T, nt)
    monkeypatch.setenv("OC_BATCH_PER_ROOM", "1")
    per_room = ctx.hjb_solve_batch(dV, dm, prm, T, nt)
    monkeypatch.delenv("OC_BATCH_PER_ROOM")
    over = 0
    for b in range(n_rooms):
        one = ctx.hjb_solve(dV[b], dm[b], prm, T, nt, want_phi=True, want_vel=False, trace=True)
        hist = samples_per_attempt(T, nt, one["trace_h"], one["trace_err"])
        over += max(hist) > NE_MAX
        for k in ("nfev", "n_accepted", "n_rejected", "status", "n_out"):
            assert batch[b]["stats"][k] == one["stats"][k] == per_room[b]["stats"][k], (b, k)
        assert torch_mod.equal(batch[b]["phi"], one["phi"]), b
        assert torch_mod.equal(batch[b]["phi"], per_room[b]["phi"]), b
        if b < 3:
            V, m = rooms[b]
            _assert_matches_oracle(batch[b], co.hjb_solve(V, m, T, nt), Ny, Nx, nt, vel=False)
        del one
    if nt == 61:
        assert over == n_rooms     # every room has attempts that are launched more than once
    else:
        assert over < n_rooms      # rooms within NE_MAX samples: every attempt waits in an NE bucket
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# d. row-band solve at dense sampling
@pytest.mark.parametrize("Nx", [226, 225], ids=["tma", "cpasync"])
def test_band_solve_at_dense_sampling(Nx, cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    Ny, T, nt = 128, 0.3, 61
    V, m = _ragged_room(Ny, Nx)
    ctx = _lib.Context(*_lengths(Ny, Nx), 0.05)
    Vd, md = ctx.to_device(V), ctx.to_device(m)
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=16)
    ref = co.hjb_solve(V, m, T, nt)
    runs = [ctx.hjb_solve_band(Vd, md, prm, T, nt, n_virtual=nv, want_vel=True, trace=True) for nv in (1, 2, 4)]
    hist = samples_per_attempt(T, nt, runs[0]["trace_h"], runs[0]["trace_err"])
    assert max(hist) > NE_MAX, sorted(hist)
    for r in runs:
        _assert_matches_oracle(r, ref, Ny, Nx, nt)
        assert np.array_equal(r["trace_h"], runs[0]["trace_h"]) and np.array_equal(r["trace_err"], runs[0]["trace_err"])
        assert r["stats"]["nfev"] == runs[0]["stats"]["nfev"]
        for k in ("phi", "vx", "vy"):
            assert torch_mod.equal(r[k], runs[0][k]), k
    # velocity-only output keeps NE_MAX scratch slices: a step with more samples is refused ...
    with pytest.raises(_lib.OcError) as e:
        ctx.hjb_solve_band(Vd, md, prm, T, nt, n_virtual=2, want_phi=False, want_vel=True)
    assert e.value.code == OC_ERR_ARG
    # ... and the context keeps working
    again = ctx.hjb_solve_band(Vd, md, prm, T, nt, n_virtual=2, want_vel=True, trace=True)
    _assert_matches_oracle(again, ref, Ny, Nx, nt)
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# e. batched velocity-only output above NE_MAX samples per step: refused, and the context keeps working
def test_batched_velocity_only_refuses_long_steps(cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    Ny, Nx, T, nt = 97, 226, 0.3, 61
    ctx = _lib.Context(*_lengths(Ny, Nx), 0.05)
    rng = np.random.RandomState(9)
    rooms = [_room_b(Ny, Nx, b, rng) for b in range(3)]
    dV = [ctx.to_device(V) for V, _ in rooms]
    dm = [ctx.to_device(m) if m is not None else None for _, m in rooms]
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=16)
    ref = co.hjb_solve(rooms[1][0], rooms[1][1], T, nt)
    assert max(samples_per_attempt(T, nt, ref[2], ref[3])) > NE_MAX
    with pytest.raises(_lib.OcError) as e:
        ctx.hjb_solve_batch(dV, dm, prm, T, nt, want_vel=True)
    assert e.value.code == OC_ERR_ARG
    res = ctx.hjb_solve_batch(dV, dm, prm, T, nt, want_vel=False)
    _assert_matches_oracle(res[1], ref, Ny, Nx, nt, vel=False)
    # velocity-only output at a sampling that stays within NE_MAX
    nt2 = 11
    refs2 = [co.hjb_solve(V, m, T, nt2) for V, m in rooms]
    assert all(max(samples_per_attempt(T, nt2, r[2], r[3])) <= NE_MAX for r in refs2)
    ref2 = refs2[1]
    vel = ctx.hjb_solve_batch(dV, dm, prm, T, nt2, want_vel=True)
    _assert_matches_oracle(vel[1], ref2, Ny, Nx, nt2, phi=False)
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# f. the drop-in API at dt = 0.01: ensemble members equal stand-alone runs bit for bit
def test_ensemble_members_equal_standalone_runs_at_small_dt(tmp_path, monkeypatch, torch_mod):
    from optimal_crowds_b200 import ensemble, simulations
    from oracle import cpu_oracle as co
    with open(os.path.join(REPO, "optimal_crowds_b200", "config.json")) as f:
        cfg = json.load(f)
    cfg["dt"] = 0.01
    (tmp_path / "optimal_crowds").mkdir()
    (tmp_path / "optimal_crowds" / "config.json").write_text(json.dumps(cfg))
    with open(os.path.join(REPO, "rooms", "room_test.json")) as f:
        room = json.load(f)
    monkeypatch.chdir(tmp_path)
    T, seeds = 1.0, [3, 11, 12]
    # record=True keeps the members, and with them their value-function samples
    ens = ensemble.ensemble(room, T, seeds, record=True)
    res = ens.run()
    assert sorted(res) == [0, 1, 2]
    for i, seed in enumerate(seeds):
        np.random.seed(seed)
        with contextlib.redirect_stdout(io.StringIO()):
            one = simulations.simulation(room, T, record=True, field_storage="phi")
            one.run()
        one._sync_host()
        assert one.dt == 0.01
        r = res[i]
        assert r["steps"] == one.simu_step and r["inside"] == one.inside and r["evac_time"] == one.time
        assert np.array_equal(r["exit_order"], np.array(one._exit_order, dtype=np.int64))
        assert np.array_equal(r["final"], one._h_now)
        assert np.array_equal(r["times"], one._h_timev)
        for k, o in one.targets.items():
            assert r["hjb"][k]["nfev"] == o.last_stats["nfev"]
            assert torch_mod.equal(ens.members[i].targets[k].d_phi, o.d_phi)
    # the first solve of the room (T = 1, nt = 100, no density) has steps that emit more than NE_MAX samples
    o = one.targets["door_1"]
    nt = round(T / 0.01)
    _, st_ref, h_ref, e_ref = co.hjb_solve(o.V_host(), None, T, nt)
    assert st_ref["nfev"] == o.last_stats["nfev"]
    assert max(samples_per_attempt(T, nt, h_ref, e_ref)) > NE_MAX
