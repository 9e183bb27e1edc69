"""GPU parity of per-member configurations: the batched HJB solve with per-room sigma, mu, g and horizons
(oc_hjb_solve_multi), ``simulation(..., config=...)`` and ``ensemble(..., configs=...)``.  Every room / member must be
its stand-alone run with its own configuration, bit for bit; the solves also match the CPU oracle run with the room's
constants, so the constants are shown to reach the kernels."""
import contextlib
import ctypes as C
import io
import json
import os

import numpy as np
import pytest

from conftest import REPO
from test_gpu_hjb_sampling import NE_MAX, samples_per_attempt

pytestmark = pytest.mark.gpu

RTOL = 1e-10
OC_ERR_ARG = -2


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    return torch


@pytest.fixture()
def in_repo_cwd(monkeypatch):
    monkeypatch.chdir(REPO)


def _merged(cfg, ov):
    from optimal_crowds_b200.optimals import _merge_config
    return _merge_config(cfg, ov)


# ---------------------------------------------------------------------------------------------------------------------
# 1. C level: oc_hjb_solve_multi
# (sigma, mu, g, T, nt, density) per room: pairwise different in every field; the last room samples densely enough
# for steps that emit more than NE_MAX samples (phi output)
ROOMS = [(0.2, 5.0, -0.005, 0.5, 25, False), (0.25, 4.0, -0.02, 0.4, 21, True), (0.15, 6.0, 0.0, 0.6, 19, False),
         (0.3, 3.0, -0.05, 0.3, 13, True), (0.22, 5.5, 0.01, 1.0, 101, True)]


def _geometry(B, Ny=70, Nx=150):
    """the rooms of test_gpu_hjb.py::test_batched_solve_is_bitwise_the_single_solves"""
    rng = np.random.RandomState(7)
    Vs, ms = [], []
    for b in range(B):
        V = np.zeros((Ny, Nx)); V[0, :] = V[-1, :] = V[:, 0] = V[:, -1] = -100
        V[10 + 5 * b:14 + 5 * b, 40:44 + 10 * b] = -100
        V[Ny // 2 - 3 + b:Ny // 2 + 3 + b, -1] = 1.0
        Vs.append(V)
        ms.append(rng.uniform(0, 1, size=(Ny, Nx)))
    return Vs, ms


def _ctx(Ny=70, Nx=150):
    from optimal_crowds_b200 import _lib
    return _lib.Context((Nx - 1) * 0.05 + 0.025, (Ny - 1) * 0.05 + 0.025, 0.05)


@pytest.mark.parametrize("store", ["phi", "velocity"])
def test_multi_solve_rooms_equal_their_single_solves_and_the_oracle(store, cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    Ny, Nx = 70, 150
    vel = store == "velocity"
    rooms = list(ROOMS)
    if vel:
        # velocity-only output: at most NE_MAX samples per step, so the dense room samples at 0.05 s instead
        rooms[4] = rooms[4][:4] + (21, True)
    ctx = _ctx(Ny, Nx)
    Vs, ms = _geometry(len(rooms), Ny, Nx)
    ms = [m if r[5] else None for m, r in zip(ms, rooms)]
    dV = [ctx.to_device(v) for v in Vs]
    dm = [ctx.to_device(m) if m is not None else None for m in ms]
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=32)
    spec = [dict(sigma=s, mu=mu, g=g, T=T, nt=nt) for s, mu, g, T, nt, _ in rooms]
    multi = ctx.hjb_solve_multi(dV, dm, spec, prm, want_vel=vel)
    for b, (sigma, mu, g, T, nt, _) in enumerate(rooms):
        prm_b = _lib.hjb_params(_merged(cfg, {"hjb_params": dict(sigma=sigma, mu=mu, g=g)}), fused=1, chunk_rows=32)
        one = ctx.hjb_solve(dV[b], dm[b], prm_b, T, nt, want_phi=not vel, want_vel=vel, trace=True)
        st = multi[b]["stats"]
        assert st["status"] == 0 and st["n_out"] == nt
        for k in ("nfev", "n_accepted", "n_rejected"):
            assert st[k] == one["stats"][k], (b, k)
        phi_ref, st_ref, h_ref, e_ref = co.hjb_solve(Vs[b], ms[b], T, nt, sigma=sigma, mu=mu, g=g)
        assert st_ref["nfev"] == st["nfev"]
        if b == 4 and not vel:
            assert max(samples_per_attempt(T, nt, h_ref, e_ref)) > NE_MAX
        if vel:
            assert multi[b]["vx"].shape[0] == nt - 1
            assert torch_mod.equal(multi[b]["vx"], one["vx"]) and torch_mod.equal(multi[b]["vy"], one["vy"])
            vx_ref, vy_ref = co.fill_field(phi_ref, Ny, Nx, mu=mu)
            assert np.abs(multi[b]["vx"].cpu().numpy() - vx_ref).max() < RTOL
            assert np.abs(multi[b]["vy"].cpu().numpy() - vy_ref).max() < RTOL
        else:
            assert multi[b]["phi"].shape[0] == nt
            assert torch_mod.equal(multi[b]["phi"], one["phi"])
            np.testing.assert_allclose(multi[b]["phi"].cpu().numpy().reshape(nt, -1), phi_ref, rtol=RTOL)
    ctx.close()


def test_multi_solve_with_identical_rooms_is_the_batched_solve(cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    ctx = _ctx()
    Vs, ms = _geometry(5)
    dV = [ctx.to_device(v) for v in Vs]
    dm = [ctx.to_device(m) if b % 2 else None for b, m in enumerate(ms)]
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=32)
    T, nt = 0.5, 25
    h = cfg["hjb_params"]
    batch = ctx.hjb_solve_batch(dV, dm, prm, T, nt)
    multi = ctx.hjb_solve_multi(dV, dm, [dict(sigma=h["sigma"], mu=h["mu"], g=h["g"], T=T, nt=nt)] * 5, prm)
    for b in range(5):
        assert batch[b]["stats"]["nfev"] == multi[b]["stats"]["nfev"]
        assert torch_mod.equal(batch[b]["phi"], multi[b]["phi"])
    ctx.close()


@pytest.mark.parametrize("bad", ["rooms_null", "t_eval_null", "nt_0", "sigma_0", "sigma_neg", "sigma_nan", "sigma_inf",
                                 "mu_0", "mu_neg", "mu_nan", "g_nan", "g_inf"])
def test_multi_solve_input_checks(bad, cfg, torch_mod):
    from optimal_crowds_b200 import _lib
    ctx = _ctx()
    Vs, _ = _geometry(2)
    dV = [ctx.to_device(v) for v in Vs]
    phi = [ctx.empty(5, ctx.Ny, ctx.Nx) for _ in range(2)]
    prm = _lib.hjb_params(cfg, fused=1)
    t_eval = np.linspace(0.2, 0, 5)
    spec = (_lib.HjbRoom * 2)()
    for b in range(2):
        spec[b] = _lib.HjbRoom(0.2, 5.0, -0.005, 0.2, t_eval.ctypes.data_as(_lib.dp), 5, 0)
    field, _, val = bad.partition("_")
    if bad == "t_eval_null":
        spec[1].t_eval = None
    elif bad == "nt_0":
        spec[1].nt = 0
    elif field in ("sigma", "mu", "g"):
        setattr(spec[1], field, {"0": 0.0, "neg": -1.0, "nan": float("nan"), "inf": float("inf")}[val])
    st = (_lib.HjbStats * 2)()
    rc = _lib.load().oc_hjb_solve_multi(ctx.h, 2, _lib._ptrs(dV, 2), None, None if bad == "rooms_null" else spec,
                                        C.byref(prm), _lib._ptrs(phi, 2), None, None, st, _lib._stream())
    assert rc == OC_ERR_ARG
    # the context keeps working
    ok = _lib.load().oc_hjb_solve_multi(ctx.h, 2, _lib._ptrs(dV, 2), None, (_lib.HjbRoom * 2)(spec[0], spec[0]),
                                        C.byref(prm), _lib._ptrs(phi, 2), None, None, st, _lib._stream())
    assert ok == 0 and st[1].n_out == 5
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. ensemble members with their own configuration == stand-alone runs with that configuration
CONFIGS = [{}, {"hjb_params": {"sigma": 0.3, "mu": 4, "g": -0.02}}, {"dt": 0.01}, {"dt": 0.025},
           {"recompute_frequency": 20},
           {"relaxation": 0.2, "v_max": 1.5, "eta": 0.08, "repulsion_cutoff": 3, "sigma_convolution": 0.3},
           {"hjb_params": {"wall_potential": -200, "target_potential": 2}}]
_ALONE = {}


def _alone(room, T, recompute, seed, ov):
    key = (json.dumps(room, sort_keys=True) if isinstance(room, dict) else room, T, recompute, seed,
           json.dumps(ov, sort_keys=True))
    if key not in _ALONE:
        from optimal_crowds_b200 import simulations
        np.random.seed(seed)
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(room, T, recompute=recompute, record=False, config=ov)
            simu.run()
        simu._sync_host()
        _ALONE[key] = simu
    return _ALONE[key]


def _assert_member_is(r, one):
    assert r["steps"] == one.simu_step and r["inside"] == one.inside and r["evac_time"] == one.time
    assert np.array_equal(r["exit_order"], np.array(one._exit_order, dtype=np.int64))
    assert np.array_equal(r["final"], one._h_now)
    assert np.array_equal(r["times"], one._h_timev)
    assert r["config"] == one._config
    for k, o in one.targets.items():
        assert r["hjb"][k]["nfev"] == o.last_stats["nfev"]


@pytest.mark.parametrize("batched", [True, False], ids=["batched_steps", "member_steps"])
# (T = 2.3: every member's re-solves fall inside the horizon; see the test below for one that does not)
@pytest.mark.parametrize("room,T,recompute", [("exit_opposite", 2.3, True), ("room_test", 3.0, False)])
def test_members_equal_standalone_runs_with_their_config(room, T, recompute, batched, in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    seeds = [3 + i for i in range(len(CONFIGS))]
    ens = ensemble.ensemble(room, T, seeds, recompute=recompute, configs=CONFIGS, batched_steps=batched)
    res = ens.run()
    assert sorted(res) == list(range(len(seeds)))
    for i, (seed, ov) in enumerate(zip(seeds, CONFIGS)):
        one = _alone(room, T, recompute, seed, ov)
        _assert_member_is(res[i], one)
    assert res[2]["config"]["dt"] == 0.01 and res[3]["config"]["dt"] == 0.025
    if recompute:
        # members re-solve at their own steps: the re-solve calls do not all hold every member
        assert ens.stats["hjb_calls"] > 2 and ens.stats["hjb_call_rooms"] < ens.stats["hjb_calls"] * len(seeds)


def test_member_whose_last_resolve_has_no_samples_fails_as_its_standalone_run(in_repo_cwd):
    """dt = 0.025, T = 2.5: the re-solve at step 100 comes at t = 2.4999999999999951 (summed steps), still inside the
    horizon, and asks for round((T - t) / dt) = 0 samples.  The stand-alone run raises ValueError there, as the
    reference's solve_ivp does on an empty t_eval; the ensemble member must not run on where the stand-alone run stops."""
    from optimal_crowds_b200 import ensemble, simulations
    ov = {"dt": 0.025}
    np.random.seed(3)
    with contextlib.redirect_stdout(io.StringIO()), pytest.raises(ValueError, match="t_eval"):
        simulations.simulation("exit_opposite", 2.5, recompute=True, record=False, config=ov).run()
    with pytest.raises(ValueError, match="t_eval"):
        ensemble.ensemble("exit_opposite", 2.5, [3, 4], recompute=True, configs=[{}, ov]).run()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the per-member constants change the result (and g alone does not without a re-solve, as in the reference)
def test_member_constants_are_not_vacuous(in_repo_cwd):
    from optimal_crowds_b200 import ensemble
    g_ov = {"hjb_params": {"g": -0.05}}
    a = ensemble.ensemble("exit_opposite", 2.5, [5, 5], recompute=True, configs=[{}, g_ov]).run()
    assert not np.array_equal(a[0]["final"], a[1]["final"])
    b = ensemble.ensemble("exit_opposite", 2.5, [5, 5, 5], recompute=False,
                          configs=[{}, g_ov, {"hjb_params": {"sigma": 0.3}}]).run()
    # without a re-solve the only solve is at step 0, where the density is zero: g has no effect
    assert np.array_equal(b[0]["final"], b[1]["final"]) and np.array_equal(b[0]["times"], b[1]["times"])
    assert all(b[0]["hjb"][k]["nfev"] == b[1]["hjb"][k]["nfev"] for k in b[0]["hjb"])
    assert not np.array_equal(b[0]["final"], b[2]["final"])


# ---------------------------------------------------------------------------------------------------------------------
# 4. config= is config.json
def test_config_argument_is_the_config_file(tmp_path, monkeypatch, in_repo_cwd):
    from optimal_crowds_b200 import simulations
    with open(os.path.join(REPO, "rooms", "exit_opposite.json")) as f:
        room = json.load(f)
    ov = {"dt": 0.025, "v_max": 1.8, "recompute_frequency": 30, "hjb_params": {"g": -0.02, "sigma": 0.25}}
    T = 2.0

    def run(**kw):
        np.random.seed(17)
        with contextlib.redirect_stdout(io.StringIO()):
            s = simulations.simulation(room, T, recompute=True, record=False, **kw)
            s.run()
        s._sync_host()
        return s
    over = run(config=ov)
    plain = run()
    empty = run(config={})
    for s in (plain, empty):
        assert s._config == simulations._load_config()
    with open(os.path.join(REPO, "optimal_crowds_b200", "config.json")) as f:
        cfg = json.load(f)
    cfg.update({k: v for k, v in ov.items() if k != "hjb_params"})
    cfg["hjb_params"].update(ov["hjb_params"])
    (tmp_path / "optimal_crowds").mkdir()
    (tmp_path / "optimal_crowds" / "config.json").write_text(json.dumps(cfg))
    monkeypatch.chdir(tmp_path)
    file_run = run()
    assert file_run._config == cfg == over._config
    for a, b in ((over, file_run), (empty, plain)):
        assert a.simu_step == b.simu_step and a.inside == b.inside and a.time == b.time
        assert a._exit_order == b._exit_order
        assert np.array_equal(a._h_now, b._h_now) and np.array_equal(a._h_timev, b._h_timev)
        for k, o in a.targets.items():
            assert o.last_stats["nfev"] == b.targets[k].last_stats["nfev"]
    assert not np.array_equal(over._h_now, plain._h_now)


# ---------------------------------------------------------------------------------------------------------------------
# 5. sharding and waves with heterogeneous configurations
def test_sharding_and_waves_with_member_configs(in_repo_cwd):
    from optimal_crowds_b200 import ensemble, synthetic
    room = synthetic.ensemble_room(n=96, agents=12)
    room["initial_boxes"]["box"][0] = 1.6
    room["initial_boxes"]["box"][2:4] = [2.0, 2.0]
    room["initial_boxes"]["box"][4] = 12.5 / 4.0
    seeds = list(range(6))
    configs = [{}, {"dt": 0.01, "recompute_frequency": 20}, {"hjb_params": {"g": -0.05, "sigma": 0.3}},
               {"dt": 0.025, "recompute_frequency": 10}, {"v_max": 1.5, "sigma_convolution": 0.3}, {"recompute_frequency": 15}]
    whole = ensemble.ensemble(room, 1.0, seeds, recompute=True, configs=configs).run()
    parts = {}
    for rank in range(2):
        e = ensemble.ensemble(room, 1.0, seeds, recompute=True, configs=configs, rank=rank, world=2, max_wave=1)
        parts.update(e.run(gather=False))
        assert e.stats["waves"] == len(e.mine)
    assert sorted(parts) == sorted(whole) == seeds
    for i in whole:
        for k in ("steps", "inside", "evac_time"):
            assert parts[i][k] == whole[i][k]
        assert np.array_equal(parts[i]["final"], whole[i]["final"])
        assert np.array_equal(parts[i]["times"], whole[i]["times"])
        assert np.array_equal(parts[i]["exit_order"], whole[i]["exit_order"])
        assert parts[i]["config"] == whole[i]["config"]
        assert whole[i]["N"] == 12
