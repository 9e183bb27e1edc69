"""GPU parity of the batched GCFM step (oc_gcfm_step_multi_launch / oc_gcfm_step_multi_finish through _lib.GcfmBatch,
the ensemble path): every member of a wave must equal the sequential CPU sweep O2 (oracle/oc_oracle_gcfm.c) bit for
bit after every step -- positions, velocities, times, status, exit sets and exit ORDER -- and its MT19937 state, which
the C side advances, must equal numpy's after the run.

The waves are heterogeneous on purpose: the members of one launch differ in room and grid, crowd size, target sets,
field storage, knobs, simu_step and displacement margin, and single members take a redo (fast-margin redo, exact slow
path, widened search) or hit a sampler-range error while the others do not.  Every test asserts from the members' redo
and pair counts that the path it claims to cover was taken."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TESTS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(TESTS)


def _cfg():
    with open(os.path.join(REPO, "optimal_crowds_b200", "config.json")) as f:
        return json.load(f)


# ---------------------------------------------------------------------------------------------------- rooms and crowds
def _random_crowd(rng, N, L, H, margin=1.0, min_dist=0.25):
    pts = []
    cell = {}
    while len(pts) < N:
        p = (rng.uniform(margin, L - margin), rng.uniform(margin, H - margin))
        c = (int(p[0] / min_dist), int(p[1] / min_dist))
        ok = True
        for dx in (-1, 0, 1):
            for dy in (-1, 0, 1):
                for q in cell.get((c[0] + dx, c[1] + dy), []):
                    if (q[0] - p[0]) ** 2 + (q[1] - p[1]) ** 2 < min_dist ** 2:
                        ok = False
        if ok:
            pts.append(p); cell.setdefault(c, []).append(p)
    return np.array(pts)


def _one_key_room(ctx, co, L, H, nsl):
    """one target set with a smooth synthetic field pointing at a door on the right wall (device + oracle key)"""
    kd = np.array([[L, H / 2, 0.6, 2.0]])
    V = co.create_potential(ctx.X, ctx.Y, [], [], [[L / 2, H / 2, 0.4]], kd)
    V[V < 0] = -100; V[V > 0] = 1
    Xi, Yi = np.meshgrid(ctx.X[1:-1], ctx.Y[1:-1])
    ux, uy = kd[0, 0] - Xi, kd[0, 1] - Yi
    nrm = np.sqrt(ux ** 2 + uy ** 2) + 1e-9
    vx, vy = np.repeat((ux / nrm)[None], nsl, 0), np.repeat((uy / nrm)[None], nsl, 0)
    Vd = ctx.to_device(V)
    tiles, vmin = ctx.wall_tiles(Vd)
    return (dict(V=Vd, tiles=tiles, v_min=vmin, vx=ctx.to_device(vx), vy=ctx.to_device(vy), nt_opt=nsl + 1, doors=kd),
            co.KeyData(V, vx, vy, nsl + 1, kd))


def _two_key_room(ctx, co, L, H, nsl):
    """two target sets: the door on the right wall, and a multi-door set (top wall + left wall) whose field points at its
    first door; a wall and a pillar inside -> [(device key, oracle key)] * 2"""
    out = []
    for kd in (np.array([[L, H / 2, 0.6, 2.0]]), np.array([[L / 2, H, 3.0, 0.6], [0.0, H / 2, 0.6, 2.0]])):
        V = co.create_potential(ctx.X, ctx.Y, [[L / 3, H / 2, 0.4, H / 2]], [], [[2 * L / 3, H / 3, 0.5]], kd)
        V[V < 0] = -100; V[V > 0] = 1
        Xi, Yi = np.meshgrid(ctx.X[1:-1], ctx.Y[1:-1])
        ux, uy = kd[0, 0] - Xi, kd[0, 1] - Yi
        nrm = np.sqrt(ux ** 2 + uy ** 2) + 1e-9
        vx = np.repeat((ux / nrm)[None], nsl, 0) * np.linspace(1, 0.9, nsl)[:, None, None]
        vy = np.repeat((uy / nrm)[None], nsl, 0)
        Vd = ctx.to_device(V)
        tiles, vmin = ctx.wall_tiles(Vd)
        out.append((dict(V=Vd, tiles=tiles, v_min=vmin, vx=ctx.to_device(vx), vy=ctx.to_device(vy), nt_opt=nsl + 1,
                         doors=kd), co.KeyData(V, vx, vy, nsl + 1, kd)))
    return out


def _phi_room(ctx, co, cfg, L, H, nt):
    """one target set whose device key stores phi slices (the sampler differentiates them on the fly); the oracle key
    holds the velocity slices of the same HJB solve"""
    from optimal_crowds_b200 import _lib
    kd = np.array([[L, H / 2, 0.6, 2.0]])
    V = co.create_potential(ctx.X, ctx.Y, [], [], [[L / 2, H / 2, 0.4]], kd)
    V[V < 0] = -100; V[V > 0] = 1
    Vd = ctx.to_device(V)
    tiles, vmin = ctx.wall_tiles(Vd)
    res = ctx.hjb_solve(Vd, None, _lib.hjb_params(cfg, fused=1), nt * cfg["dt"], nt, want_phi=True, want_vel=True)
    key = dict(V=Vd, tiles=tiles, v_min=vmin, phi=res["phi"], nt_opt=nt, doors=kd, mu=float(cfg["hjb_params"]["mu"]),
               lim=10e-3)
    return key, co.KeyData(V, res["vx"].cpu().numpy(), res["vy"].cpu().numpy(), nt, kd)


def _member(ctx, cfg, keys, pos, vx, vy, vdes, key_id, seed, step0=0):
    """one member of a wave: its device state and GcfmBatch record, and its O2 copy stepped with a second generator of
    the same seed (GcfmBatch reads only the record's keys)"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    N = len(pos)
    L, H = ctx.room_length, ctx.room_height
    vdes = np.ascontiguousarray(vdes, dtype=np.float64)
    key_id = np.ascontiguousarray(key_id, dtype=np.int32)
    cpu = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=np.array(vx, dtype=np.float64),
               vy=np.array(vy, dtype=np.float64), time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
    return dict(ctx=ctx, prm=_lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx),
                state={k: ctx.to_device(v) for k, v in cpu.items()}, vdes=ctx.to_device(vdes),
                key_id=ctx.to_device(key_id), keys=ctx.make_keys([k[0] for k in keys]), rng=np.random.RandomState(seed),
                P=co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx), kcpu=[k[1] for k in keys], cpu=cpu, vdes_h=vdes,
                kid_h=key_id, orng=np.random.RandomState(seed), step0=step0, failed=False)


def _sparse_member(cfg, L, H, N, seed, nsl, two_keys=False, door_agents=0, door_gap=0.01, step0=0, knobs=None):
    """N agents at <= 2.5 ped/m^2 in an L x H room, off the walls and pillars; the first door_agents start next to the
    right door, the first door_gap from the door's 0.3 m exit zone, moving towards it (they leave within a few steps, at
    different steps)"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    rng = np.random.RandomState(seed)
    ctx = _lib.Context(L, H, 0.05)
    for k, v in (knobs or {}).items():
        ctx.set_int(k, v)
    keys = _two_key_room(ctx, co, L, H, nsl) if two_keys else [_one_key_room(ctx, co, L, H, nsl)]
    pos = _random_crowd(rng, N + N // 2 + 8, L, H)
    if two_keys:
        keep = (~((np.abs(pos[:, 0] - L / 3) < 0.6) & (np.abs(pos[:, 1] - H / 2) < H / 4 + 0.4)) &
                (np.hypot(pos[:, 0] - 2 * L / 3, pos[:, 1] - H / 3) > 0.9))
    else:
        keep = np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 0.7
    pos = pos[keep][:N]
    assert len(pos) == N
    vx, vy = rng.normal(0, 0.5, N), rng.normal(0, 0.5, N)
    kid = rng.randint(0, len(keys), N)
    d = min(door_agents, N)
    pos[:d] = np.column_stack([L - 0.3 - door_gap - 0.04 * np.arange(d), H / 2 + np.linspace(-0.5, 0.5, d)])
    vx[:d], vy[:d], kid[:d] = 1.2, 0.0, 0
    return _member(ctx, cfg, keys, pos, vx, vy, rng.normal(1.34, 0.26, N), kid, seed + 1000, step0)


def _dense_member(cfg, wide, seed=8):
    """1000 agents on 10.8 x 10.8 m (8.6 ped/m^2, test_gpu_gcfm.py's dense jam): more agents within the candidate reach of
    one agent than the fast path's 512-slot lists hold.  wide: 1 m margin and no field-of-view culling, which overflows
    the lists on every step"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    L = H = 12.0
    rng = np.random.RandomState(8)
    ctx = _lib.Context(L, H, 0.05)
    if wide:
        ctx.set_int("gcfm_margin_mm", 1000)
        ctx.set_int("gcfm_fov_cull", 0)
    key = _one_key_room(ctx, co, L, H, 6)
    pos = _random_crowd(rng, 1000, L, H, margin=0.6, min_dist=0.2)
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 0.7]  # off the pillar
    N = len(pos)
    assert N > 900
    vx, vy = rng.normal(0, 0.4, N), rng.normal(0, 0.4, N)
    return _member(ctx, cfg, [key], pos, vx, vy, rng.normal(1.34, 0.26, N), np.zeros(N), seed)


def _fast_member(cfg, seed=5, nsl=8):
    """400 agents on 30 x 20 m, 10 of them at 8 .. 14 m/s: 0.16 .. 0.28 m per step exceeds the default 0.25 m margin
    (12.5 cm per axis) but not the full one -- the first step is redone on the fast path with the 1 m margin, which is
    then held for the following steps"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    L, H = 30.0, 20.0
    rng = np.random.RandomState(5)
    ctx = _lib.Context(L, H, 0.05)
    key = _one_key_room(ctx, co, L, H, nsl)
    pos = _random_crowd(rng, 400, L, H, margin=2.0)
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 1.0]
    N = len(pos)
    vx, vy = rng.normal(0, 0.5, N), rng.normal(0, 0.5, N)
    fast = rng.choice(N, 10, replace=False)
    vx[fast] = rng.choice([-1, 1], 10) * rng.uniform(8, 14, 10)
    return _member(ctx, cfg, [key], pos, vx, vy, rng.normal(1.34, 0.26, N), np.zeros(N), seed)


def _leaping_member(cfg, seed=3):
    """300 agents on 30 x 20 m, 12 of them at 30 .. 90 m/s (0.6 .. 1.8 m per step, beyond the 0.5 m per axis the full
    margin covers): the candidate search is widened and the step redone on the exact slow path"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    L, H = 30.0, 20.0
    rng = np.random.RandomState(3)
    ctx = _lib.Context(L, H, 0.05)
    key = _one_key_room(ctx, co, L, H, 8)
    pos = _random_crowd(rng, 300, L, H, margin=2.0)
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 1.0]
    N = len(pos)
    vx, vy = rng.normal(0, 0.5, N), rng.normal(0, 0.5, N)
    fast = rng.choice(N, 12, replace=False)
    vx[fast] = rng.choice([-1, 1], 12) * rng.uniform(30, 90, 12)
    return _member(ctx, cfg, [key], pos, vx, vy, rng.normal(1.34, 0.26, N), np.zeros(N), seed)


# ---------------------------------------------------------------------------------------------------- stepping
def _oracle_step(m, simu_step):
    """O2's step of member m with numpy's draws in the order the C side draws them: permutation, then normal pairs"""
    from oracle import cpu_oracle as co
    cpu = m["cpu"]
    perm = m["orng"].permutation(len(cpu["x"]))
    noise = m["orng"].normal(size=(int(cpu["status"].sum()), 2))
    ex, bad, _ = co.gcfm_step(m["P"], cpu, m["vdes_h"], m["kid_h"], m["kcpu"], m["ctx"].X, m["ctx"].Y, perm, noise,
                              simu_step)
    return ex, bad


def _check_states(members, what):
    for q, m in enumerate(members):
        if m["failed"]:
            continue
        for k in ("x", "y", "vx", "vy", "time", "status"):
            assert np.array_equal(m["state"][k].cpu().numpy(), m["cpu"][k]), f"{what}: member {q}: {k} differs"


def _batched_step(batch, members, live, s):
    """one batched step of the live members and the same step of their O2 copies; then every member's state is compared
    (a member outside `live` must stay untouched).  -> {member: dict(rc, bad, redos, pairs, exits)}"""
    n_act = [int(members[q]["cpu"]["status"].sum()) for q in live]
    steps = [members[q]["step0"] + s for q in live]
    batch.launch(live, n_act, steps)
    got = batch.finish()           # (does not raise on a member's sampler-range error)
    out = {}
    for q, (ex, rc), ss in zip(live, got, steps):
        m = members[q]
        out[q] = dict(rc=rc, redos=m["ctx"].gcfm_last_redos(), pairs=m["ctx"].gcfm_last_pairs())
        ex2, bad = _oracle_step(m, ss)
        out[q].update(bad=bad, exits=len(ex2))
        if bad:
            m["failed"] = True     # (the caller asserts what the device reported)
            continue
        assert rc == 0, f"step {s}: member {q}: rc {rc}"
        assert np.array_equal(ex, ex2), f"step {s}: member {q}: exit log differs"
    _check_states(members, f"batched step {s}")
    return out


def _single_step(m, s):
    """one oc_gcfm_step of member m (draws from its own generator) and O2's; -> redos"""
    ctx, cpu = m["ctx"], m["cpu"]
    perm = m["rng"].permutation(len(cpu["x"]))
    noise = m["rng"].normal(size=(int(cpu["status"].sum()), 2))
    ex, rc = ctx.gcfm_step(m["prm"], m["state"], m["vdes"], m["key_id"], m["keys"], perm, noise, m["step0"] + s)
    redos = ctx.gcfm_last_redos()
    ex2, bad = _oracle_step(m, m["step0"] + s)
    assert rc == 0 and bad == 0
    assert np.array_equal(ex, ex2), f"single step {s}: exit log differs"
    _check_states([m], f"single step {s}")
    return redos


def _still_inside(members, live):
    return [q for q in live if not members[q]["failed"] and members[q]["cpu"]["status"].any()]


def _check_rng(batch, members):
    batch.write_back_rng()
    for q, m in enumerate(members):
        a, b = m["rng"].get_state(), m["orng"].get_state()
        assert np.array_equal(a[1], b[1]) and a[2:] == b[2:], f"member {q}: generator state differs from numpy's"


def _close(members):
    for m in members:
        m["ctx"].close()


def _kick(m, agents, vx):
    """the same velocity change on the device and on the O2 copy (the device buffer keeps its address)"""
    import torch
    m["cpu"]["vx"][agents] = vx
    m["state"]["vx"].copy_(torch.from_numpy(m["cpu"]["vx"]))


# ---------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("sweep_ctas", [1, 3, 8])
def test_heterogeneous_wave_is_exact(sweep_ctas):
    """six members in one launch with different rooms and grids (8 x 5, 16 x 12.5, 30 x 20 m), crowds of 1 .. 700, one
    or two target sets (one with two doors), velocity or phi slices, field-of-view culling off in one member, a later
    simu_step in another; agents next to the doors leave at different steps, the one-agent member empties and leaves the
    wave while the others go on"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    cfg = _cfg()
    steps, nsl = 14, 20
    ms = [_sparse_member(cfg, 8.0, 5.0, 1, 100, nsl, door_agents=1, door_gap=0.05),
          _sparse_member(cfg, 16.0, 12.5, 40, 101, nsl, two_keys=True, door_agents=3, door_gap=0.01),
          None,
          _sparse_member(cfg, 30.0, 20.0, 700, 103, nsl, door_agents=4, door_gap=0.15, knobs=dict(gcfm_fov_cull=0)),
          _sparse_member(cfg, 8.0, 5.0, 40, 104, nsl, two_keys=True, door_agents=2, door_gap=0.08, step0=3),
          _sparse_member(cfg, 30.0, 20.0, 120, 105, nsl, door_agents=5, door_gap=0.01, knobs=dict(gcfm_sweep_ctas=2))]
    # phi-slice member: 300 agents in 16 x 12.5 m, the field of an HJB solve
    L, H = 16.0, 12.5
    rng = np.random.RandomState(102)
    ctx = _lib.Context(L, H, 0.05)
    key = _phi_room(ctx, co, cfg, L, H, nsl + 2)
    pos = _random_crowd(rng, 300, L, H)
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 0.7]
    N = len(pos)
    vx, vy = rng.normal(0, 0.5, N), rng.normal(0, 0.5, N)
    pos[:3] = np.column_stack([L - 0.32 - 0.05 * np.arange(3), H / 2 + np.array([-0.4, 0.0, 0.4])])
    vx[:3], vy[:3] = 1.2, 0.0
    ms[2] = _member(ctx, cfg, [key], pos, vx, vy, rng.normal(1.34, 0.26, N), np.zeros(N), 1102)
    assert [len(m["cpu"]["x"]) for m in ms][:2] == [1, 40] and len(ms[3]["cpu"]["x"]) == 700
    batch = _lib.GcfmBatch(ms, sweep_ctas=sweep_ctas)
    live = list(range(len(ms)))
    left_at, first_exit = {}, {}
    for s in range(steps):
        out = _batched_step(batch, ms, live, s)
        for q, o in out.items():
            assert o["redos"] == 0, f"step {s}: member {q} was redone"
            if o["exits"] and q not in first_exit:
                first_exit[q] = s
        live2 = _still_inside(ms, live)
        for q in set(live) - set(live2):
            left_at[q] = s
        live = live2
    _check_rng(batch, ms)
    # the paths claimed: members left at different steps, the one-agent member emptied while the others went on
    assert 0 in left_at and left_at[0] < steps - 2 and len(live) >= 4, (left_at, live)
    assert len(first_exit) >= 4 and len(set(first_exit.values())) >= 2, first_exit
    _close(ms)


@pytest.mark.parametrize("wide", [False, True])
def test_slow_path_redo_of_one_member_is_exact(wide):
    """a jam of ~950 agents at 8.6 ped/m^2 shares the launch with two sparse members.  Default knobs (0.25 m margin,
    field-of-view culling): the culled lists mostly fit, and the jam is exact whichever path a step takes.  wide: its fast attempt overflows the 512-slot lists on every step and is
    redone alone on the exact slow path (global-memory lists).  The sparse members are never redone"""
    from optimal_crowds_b200 import _lib
    cfg = _cfg()
    ms = [_sparse_member(cfg, 8.0, 5.0, 40, 200, 6), _dense_member(cfg, wide),
          _sparse_member(cfg, 16.0, 12.5, 120, 202, 6, two_keys=True)]
    batch = _lib.GcfmBatch(ms, sweep_ctas=8)
    live = [0, 1, 2]
    dense_redos = []
    for s in range(3):
        out = _batched_step(batch, ms, live, s)
        assert out[0]["redos"] == 0 and out[2]["redos"] == 0, out
        assert out[1]["pairs"] > 100000, out           # the jam: ~400 interacting neighbours per agent
        dense_redos.append(out[1]["redos"])
    if wide:
        assert min(dense_redos) >= 1, dense_redos
    _check_rng(batch, ms)
    _close(ms)


def test_fast_margin_redo_of_one_member_is_exact():
    """one member's agents move 0.16 .. 0.28 m in the first step: that member is redone on the fast path with the 1 m
    margin and keeps it, while the others stay on 0.25 m in the same launches.  Then three agents of that member and
    of a 0.25 m member are kicked to 10 m/s (0.2 m per step): only the 0.25 m member is redone"""
    from optimal_crowds_b200 import _lib
    cfg = _cfg()
    ms = [_sparse_member(cfg, 16.0, 12.5, 120, 300, 8), _fast_member(cfg),
          _sparse_member(cfg, 8.0, 5.0, 40, 302, 8, two_keys=True)]
    batch = _lib.GcfmBatch(ms, sweep_ctas=8)
    live = [0, 1, 2]
    redos = []
    for s in range(4):
        if s == 2:
            for m in ms[:2]:
                inner = np.where((np.abs(m["cpu"]["x"] - m["ctx"].room_length / 2) < 4.0) & (m["cpu"]["vx"] < 1.5))[0]
                _kick(m, inner[:3], 10.0)
        out = _batched_step(batch, ms, live, s)
        redos.append([out[q]["redos"] for q in live])
    assert redos == [[0, 1, 0], [0, 0, 0], [1, 0, 0], [0, 0, 0]], redos
    _check_rng(batch, ms)
    _close(ms)


def test_displacement_beyond_the_margin_in_one_member_is_exact():
    """one member's agents move 0.6 .. 1.8 m per step: its candidate search is widened and the step redone on the exact
    slow path; the other members of the launch are not redone"""
    from optimal_crowds_b200 import _lib
    cfg = _cfg()
    ms = [_leaping_member(cfg), _sparse_member(cfg, 8.0, 5.0, 40, 401, 8),
          _sparse_member(cfg, 30.0, 20.0, 300, 402, 8)]
    batch = _lib.GcfmBatch(ms, sweep_ctas=8)
    live = [0, 1, 2]
    out = _batched_step(batch, ms, live, 0)
    assert out[0]["redos"] >= 1 and out[1]["redos"] == 0 and out[2]["redos"] == 0, out
    _batched_step(batch, ms, live, 1)
    _check_rng(batch, ms)
    _close(ms)


@pytest.mark.parametrize("knob", ["gcfm_split", "gcfm_overlap", "gcfm_ws_pair"])
def test_knob_variants_with_a_redone_member_are_exact(knob):
    """the launch takes split / overlap / ws_pair from member 0's context, a member's redo from its own: the knob is off
    on every context (gcfm_split=0: the one-kernel sweep_multi_kernel, and sweep_kernel with its 56 KB of shared memory
    for the fast-margin redo)"""
    from optimal_crowds_b200 import _lib
    cfg = _cfg()
    ms = [_sparse_member(cfg, 16.0, 12.5, 120, 500, 8, knobs={knob: 0}), _fast_member(cfg),
          _sparse_member(cfg, 8.0, 5.0, 40, 502, 8, two_keys=True, knobs={knob: 0})]
    ms[1]["ctx"].set_int(knob, 0)
    batch = _lib.GcfmBatch(ms, sweep_ctas=4)
    live = [0, 1, 2]
    redos = []
    for s in range(3):
        out = _batched_step(batch, ms, live, s)
        redos.append([out[q]["redos"] for q in live])
    assert redos == [[0, 1, 0], [0, 0, 0], [0, 0, 0]], redos
    _check_rng(batch, ms)
    _close(ms)


def test_sampler_range_error_in_one_member():
    """an agent 12 cm from the right wall (outside a door) makes the reference's sampler index past the field
    (IndexError): that member reports OC_ERR_SAMPLER_RANGE, the batch does not raise, the other members are exact and
    go on without it"""
    from optimal_crowds_b200 import _lib
    cfg = _cfg()
    ms = [_sparse_member(cfg, 8.0, 5.0, 40, 600, 8), _sparse_member(cfg, 8.0, 5.0, 20, 601, 8),
          _sparse_member(cfg, 16.0, 12.5, 120, 602, 8, two_keys=True)]
    bad = ms[1]
    L = bad["ctx"].room_length
    for k, v in (("x", L - 0.12), ("y", 1.0), ("vx", 0.0), ("vy", 0.0)):
        bad["cpu"][k][7] = v
        bad["state"][k][7] = v
    batch = _lib.GcfmBatch(ms, sweep_ctas=8)
    live = [0, 1, 2]
    out = _batched_step(batch, ms, live, 0)
    assert out[1]["bad"] != 0                          # O2 flags the position ...
    assert out[1]["rc"] == _lib.OC_ERR_SAMPLER_RANGE   # ... and so does the device, for that member only
    assert out[0]["rc"] == 0 and out[2]["rc"] == 0 and not out[0]["bad"] and not out[2]["bad"]
    live = _still_inside(ms, live)
    assert live == [0, 2]
    for s in (1, 2):
        _batched_step(batch, ms, live, s)
    _check_rng(batch, ms)
    _close(ms)


def _fresh_process_wave(split):
    """batched steps only, in a process that has taken no single GCFM step: a member redone on the exact slow path every
    step and a member redone on the fast path at its first step (the redo kernels' launch setup must come from the
    batched launch).  Raises on any difference."""
    from optimal_crowds_b200 import _lib
    cfg = _cfg()
    ms = [_dense_member(cfg, True), _fast_member(cfg)]
    for m in ms:
        m["ctx"].set_int("gcfm_split", split)
    batch = _lib.GcfmBatch(ms, sweep_ctas=8)
    redos = []
    for s in range(3):
        out = _batched_step(batch, ms, [0, 1], s)
        redos.append([out[0]["redos"], out[1]["redos"]])
    assert min(r[0] for r in redos) >= 1 and [r[1] for r in redos] == [1, 0, 0], redos
    _check_rng(batch, ms)
    _close(ms)
    return redos


@pytest.mark.parametrize("split", [1, 0])
def test_batched_redo_in_a_fresh_process(split):
    """the redo of a member runs the single-step kernels (cand_kernel and sweep_kernel need more than 48 KB of dynamic
    shared memory): it must work in a process whose only GCFM steps are batched ones -- function attributes are per
    process, so this runs in a child interpreter"""
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_gcfm_batch as t\n"
            "print('redos', t._fresh_process_wave(%d))\n" % (REPO, TESTS, split))
    r = subprocess.run([sys.executable, "-c", code], cwd=REPO, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    assert "redos" in r.stdout


def test_batched_and_single_steps_on_the_same_contexts():
    """batched steps and oc_gcfm_step alternate on the same member contexts (the batched step points the member's
    permutation and noise into the batch arena, its redo may allocate the step staging that the single step's graph
    depends on): batched, single right after the batched redos, batched, single"""
    from optimal_crowds_b200 import _lib
    cfg = _cfg()
    ms = [_fast_member(cfg), _dense_member(cfg, True), _sparse_member(cfg, 8.0, 5.0, 40, 802, 8, two_keys=True)]
    redos = []
    for s in range(4):
        if s % 2 == 0:
            batch = _lib.GcfmBatch(ms, sweep_ctas=8)    # (takes over the generators' states)
            out = _batched_step(batch, ms, [0, 1, 2], s)
            batch.write_back_rng()
            redos.append([out[q]["redos"] for q in range(3)])
        else:
            redos.append([_single_step(m, s) for m in ms])
    assert [r[0] for r in redos] == [1, 0, 0, 0] and [r[2] for r in redos] == [0, 0, 0, 0], redos
    assert min(r[1] for r in redos) >= 1, redos
    for q, m in enumerate(ms):
        a, b = m["rng"].get_state(), m["orng"].get_state()
        assert np.array_equal(a[1], b[1]) and a[2:] == b[2:], f"member {q}: generator state differs from numpy's"
    _close(ms)
