"""GPU parity: GCFM path (K4 wall search, K5 prepare, K6 sweep), density (K7) and rasteriser (K8)
through the C ABI.

Bars: bit-exact against the CPU oracle O2 (oracle/oc_oracle_gcfm.c) -- positions, velocities, exit sets and
exit ORDER over whole runs; bit-exact argmin indices and masks against the reference goldens; <= 1e-12
against the reference goldens (O1) for forces and teacher-forced steps (SURVEY.md section 8c).
"""
import json

import numpy as np
import pytest

from conftest import golden, room_grid

pytestmark = pytest.mark.gpu


def _setup(room, cfg):
    from optimal_crowds_b200 import _lib
    ctx = _lib.Context(room["room_length"], room["room_height"], cfg["grid_step"])
    prm = _lib.gcfm_params(cfg, room["room_length"], room["room_height"], ctx.Ny, ctx.Nx)
    return ctx, prm


def test_pair_force_bitexact_vs_oracle_and_close_to_reference(cfg):
    from oracle import cpu_oracle as co
    u = golden("units")
    room = json.loads(str(u["room"]))
    ctx, prm = _setup(room, cfg)
    P = co.gcfm_params(cfg, room["room_length"], room["room_height"], ctx.Ny, ctx.Nx)
    f = ctx.pair_force(prm, ctx.to_device(u["pair_pi"]), ctx.to_device(u["pair_vi"]), ctx.to_device(u["pair_vdes"]),
                       ctx.to_device(u["pair_pj"]), ctx.to_device(u["pair_vj"])).cpu().numpy()
    o2 = np.array([co.pair_force(P, u["pair_pi"][q], u["pair_vi"][q], u["pair_vdes"][q], u["pair_pj"][q],
                                 u["pair_vj"][q]) for q in range(len(f))])
    assert np.array_equal(f, o2)
    assert np.abs(f - u["pair_out"]).max() < 1e-12
    ctx.close()


def test_wall_force_and_argmin(cfg):
    from oracle import cpu_oracle as co
    u = golden("units")
    room = json.loads(str(u["room"]))
    ctx, prm = _setup(room, cfg)
    P = co.gcfm_params(cfg, room["room_length"], room["room_height"], ctx.Ny, ctx.Nx)
    V = ctx.to_device(u["wall_V"])
    p, v = u["wall_p"], u["wall_v"]
    fx, fy, ind = ctx.wall_force(prm, V, ctx.to_device(p[:, 0].copy()), ctx.to_device(p[:, 1].copy()),
                                 ctx.to_device(v[:, 0].copy()), ctx.to_device(v[:, 1].copy()),
                                 ctx.to_device(u["wall_vdes"]))
    assert np.array_equal(ind.cpu().numpy(), u["wall_ind"])  # bit-exact np.argmin incl. ties
    f = np.column_stack([fx.cpu().numpy(), fy.cpu().numpy()])
    assert np.abs(f - u["wall_out"]).max() < 1e-12
    o2 = np.array([co.wall_force(P, ctx.X, ctx.Y, u["wall_V"], p[q], v[q], u["wall_vdes"][q])[:2] for q in range(len(p))])
    assert np.array_equal(f, o2)
    ctx.close()


def test_wall_argmin_far_from_walls(cfg):
    """big empty room: the search must expand many rings and still return np.argmin's first index."""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    Nx, Ny = 700, 500
    L, H = (Nx - 1) * 0.05 + 0.025, (Ny - 1) * 0.05 + 0.025
    ctx = _lib.Context(L, H, 0.05)
    prm = _lib.gcfm_params(cfg, L, H, Ny, Nx)
    V = np.zeros((Ny, Nx)); V[0, :] = V[-1, :] = V[:, 0] = V[:, -1] = -100
    V[250, 350] = -100  # a single interior wall node
    V[100:104, -1] = 1
    rng = np.random.RandomState(0)
    n = 300
    p = np.column_stack([rng.uniform(0.1, L - 0.1, n), rng.uniform(0.1, H - 0.1, n)])
    p[:40] = np.column_stack([ctx.X[rng.randint(1, Nx - 1, 40)] + 0.025, ctx.Y[rng.randint(1, Ny - 1, 40)] + 0.025])
    p[40:50] = [L / 2, H / 2]  # equidistant-ish from several frame nodes
    z = np.zeros(n)
    _, _, ind = ctx.wall_force(prm, ctx.to_device(V), ctx.to_device(p[:, 0].copy()), ctx.to_device(p[:, 1].copy()),
                               ctx.to_device(z), ctx.to_device(z), ctx.to_device(z + 1.3))
    ref = np.array([co.lib().oco_wall_argmin(co._p(ctx.X), co._p(ctx.Y), co._p(V), Ny, Nx,
                                             co.C.c_double(p[q, 0]), co.C.c_double(p[q, 1])) for q in range(n)])
    assert np.array_equal(ind.cpu().numpy(), ref)
    ctx.close()


def _load_keys(g, room, ctx, Ny, Nx, step_fields=None):
    keys_dev, keys_cpu = [], []
    from oracle import cpu_oracle as co
    for kid in range(int(g["n_keys"])):
        key = str(g[f"k{kid}_key"])
        doors = np.array([room["targets"][t] for t in key.split(" or ")], dtype=np.float64)
        V = g[f"k{kid}_V"]
        nt = int(g[f"k{kid}_nt"])
        if step_fields is not None:
            s = step_fields
            vx = np.zeros((s + 1, Ny - 2, Nx - 2)); vy = np.zeros_like(vx)
            vx[s] = g[f"k{kid}_vx_step{s}"]; vy[s] = g[f"k{kid}_vy_step{s}"]
        else:
            vx = vy = None
        Vd = ctx.to_device(V)
        tiles, vmin = ctx.wall_tiles(Vd)
        keys_dev.append(dict(V=Vd, tiles=tiles, v_min=vmin, vx=None if vx is None else ctx.to_device(vx),
                             vy=None if vy is None else ctx.to_device(vy), nt_opt=nt, doors=doors))
        keys_cpu.append(co.KeyData(V, vx if vx is not None else np.zeros((1, Ny - 2, Nx - 2)),
                                   vy if vy is not None else np.zeros((1, Ny - 2, Nx - 2)), nt, doors))
    return keys_dev, keys_cpu


@pytest.mark.parametrize("name", ["gcfm_dense", "gcfm_small"])
def test_teacher_forced_steps_vs_reference_and_oracle(name, cfg):
    """one step from the reference's recorded state with the reference's perm/noise/field."""
    import torch
    from oracle import cpu_oracle as co
    g = golden(name)
    room = json.loads(str(g["room"]))
    ctx, prm = _setup(room, cfg)
    Ny, Nx = ctx.Ny, ctx.Nx
    P = co.gcfm_params(cfg, room["room_length"], room["room_height"], Ny, Nx)
    n_exit_total = 0
    for s in [int(q) for q in g["field_steps"]]:
        keys_dev, keys_cpu = _load_keys(g, room, ctx, Ny, Nx, step_fields=s)
        b, a = g["before"][s], g["after"][s]
        noise = g["noise"][s]; noise = noise[~np.isnan(noise[:, 0])]
        st = {k: ctx.to_device(b[:, i].copy()) for i, k in enumerate(("x", "y", "vx", "vy"))}
        st["time"] = ctx.to_device(b[:, 5].copy())
        st["status"] = ctx.to_device(b[:, 4].astype(np.uint8))
        ex, rc = ctx.gcfm_step(prm, st, ctx.to_device(g["v_des"]), ctx.to_device(g["agent_key"].astype(np.int32)),
                               keys_dev, g["perm"][s], noise, s)
        assert rc == 0
        out = np.column_stack([st[k].cpu().numpy() for k in ("x", "y", "vx", "vy")] +
                              [st["status"].cpu().numpy().astype(float), st["time"].cpu().numpy()])
        # O1: the unmodified reference
        assert np.abs(out - a).max() < 1e-12
        assert np.array_equal(out[:, 4], a[:, 4])
        # O2: bit-exact
        so = {k: np.ascontiguousarray(b[:, i]) for i, k in enumerate(("x", "y", "vx", "vy"))}
        so["time"] = np.ascontiguousarray(b[:, 5]); so["status"] = b[:, 4].astype(np.uint8)
        ex2, bad, _ = co.gcfm_step(P, so, g["v_des"], g["agent_key"], keys_cpu, ctx.X, ctx.Y, g["perm"][s], noise, s)
        o2 = np.column_stack([so[k] for k in ("x", "y", "vx", "vy")] + [so["status"].astype(float), so["time"]])
        assert np.array_equal(out, o2)
        assert np.array_equal(ex, ex2)
        n_exit_total += len(ex)
    if name == "gcfm_small":
        assert n_exit_total == 2
    ctx.close()


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


@pytest.mark.parametrize("N,L,H,steps", [(40, 8.0, 5.0, 60), (1500, 40.0, 30.0, 12)])
def test_free_running_bitexact_vs_oracle(N, L, H, steps, cfg):
    """whole runs: GPU sweep == sequential CPU sweep bit for bit (positions, velocities, exit order)."""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    rng = np.random.RandomState(N)
    ctx = _lib.Context(L, H, 0.05)
    Ny, Nx = ctx.Ny, ctx.Nx
    prm = _lib.gcfm_params(cfg, L, H, Ny, Nx)
    P = co.gcfm_params(cfg, L, H, Ny, Nx)
    # two keys with different doors; a synthetic smooth velocity field pointing to the door
    doors = [np.array([[L, H / 2, 0.6, 2.0]]), np.array([[L / 2, H, 3.0, 0.6], [0.0, H / 2, 0.6, 2.0]])]
    keys_dev, keys_cpu = [], []
    nsl = steps + 2
    Xi, Yi = np.meshgrid(ctx.X[1:-1], ctx.Y[1:-1])
    for kd in doors:
        V = co.create_potential(ctx.X, ctx.Y, [[L / 3, H / 2, 0.4, H / 2]], [], [[2 * L / 3, H / 3, 0.5]], kd)
        V[V < 0] = -100; V[V > 0] = 1
        ux, uy = kd[0, 0] - Xi, kd[0, 1] - Yi
        nrm = np.sqrt(ux ** 2 + uy ** 2) + 1e-9
        vx = np.repeat((ux / nrm)[None], nsl, 0) * np.linspace(1, 0.9, nsl)[:, None, None]
        vy = np.repeat((uy / nrm)[None], nsl, 0)
        Vd = ctx.to_device(V)
        tiles, vmin = ctx.wall_tiles(Vd)
        keys_dev.append(dict(V=Vd, tiles=tiles, v_min=vmin, vx=ctx.to_device(vx), vy=ctx.to_device(vy), nt_opt=nsl + 1, doors=kd))
        keys_cpu.append(co.KeyData(V, vx, vy, nsl + 1, kd))
    pos = _random_crowd(rng, N, L, H)
    # keep agents off wall nodes
    vdes = rng.normal(1.34, 0.26, N)
    key_id = rng.randint(0, 2, N).astype(np.int32)
    # some agents start next to a door so that exits happen early
    pos[:5] = np.column_stack([np.full(5, L - 0.35), H / 2 + np.linspace(-0.8, 0.8, 5)]); key_id[:5] = 0
    cpu = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=rng.normal(0, 0.5, N), vy=rng.normal(0, 0.5, N),
               time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
    dev = {k: ctx.to_device(v) for k, v in cpu.items()}
    vd_dev, kid_dev = ctx.to_device(vdes), ctx.to_device(key_id)
    order_gpu, order_cpu = [], []
    for s in range(steps):
        perm = rng.permutation(N)
        n_act = int(cpu["status"].sum())
        noise = rng.normal(size=(n_act, 2))
        ex, rc = ctx.gcfm_step(prm, dev, vd_dev, kid_dev, keys_dev, perm, noise, s)
        ex2, bad, _ = co.gcfm_step(P, cpu, vdes, key_id, keys_cpu, ctx.X, ctx.Y, perm, noise, s)
        assert rc == 0 and bad == 0
        assert np.array_equal(ex, ex2), f"exit order differs at step {s}"
        order_gpu += list(ex); order_cpu += list(ex2)
        for k in ("x", "y", "vx", "vy", "time", "status"):
            assert np.array_equal(dev[k].cpu().numpy(), cpu[k]), f"{k} differs at step {s}"
    assert len(order_cpu) >= 3
    ctx.close()


def test_sampler_range_error_is_reported(cfg):
    """App. C #7: positions for which the reference raises IndexError -> OC_ERR_SAMPLER_RANGE."""
    from optimal_crowds_b200 import _lib
    u = golden("units")
    room = json.loads(str(u["room"]))
    ctx, prm = _setup(room, cfg)
    Vd = ctx.to_device(u["wall_V"])
    tiles, vmin = ctx.wall_tiles(Vd)
    bad = np.where(u["samp_ok"] == 0)[0]
    assert len(bad) > 0
    for q in list(bad[:3]) + list(np.where(u["samp_ok"] == 1)[0][:3]):
        p = u["samp_p"][q]; t = int(u["samp_t"][q])
        key = dict(V=Vd, tiles=tiles, v_min=vmin, vx=ctx.to_device(u["samp_vx"]), vy=ctx.to_device(u["samp_vy"]),
                   nt_opt=int(u["samp_nt_opt"]), doors=np.array([[100.0, 100.0, 0.1, 0.1]]))
        st = dict(x=ctx.to_device(np.array([p[0]])), y=ctx.to_device(np.array([p[1]])), vx=ctx.to_device(np.zeros(1)),
                  vy=ctx.to_device(np.zeros(1)), time=ctx.to_device(np.zeros(1)),
                  status=ctx.to_device(np.ones(1, dtype=np.uint8)))
        _, rc = ctx.gcfm_step(prm, st, ctx.to_device(np.array([1.3])), ctx.to_device(np.zeros(1, dtype=np.int32)),
                              [key], np.array([0]), np.zeros((1, 2)), t)
        assert (rc == _lib.OC_ERR_SAMPLER_RANGE) == (u["samp_ok"][q] == 0)
    ctx.close()


@pytest.mark.parametrize("rname", ["room_test", "exit_opposite", "dense", "small"])
def test_rasteriser_and_density_vs_reference(rname, cfg):
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    u = golden("units")
    room = json.loads(str(u[f"rast_{rname}_room"]))
    ctx, _ = _setup(room, cfg)
    kid = 0
    while f"rast_{rname}_k{kid}" in u:
        key = str(u[f"rast_{rname}_k{kid}_key"])
        tg = [room["targets"][t] for t in key.split(" or ")]
        V = ctx.rasterise(list(room["walls"].values()), list(room["holes"].values()), list(room["cylinders"].values()),
                          tg, remap=True, wall_value=-100.0, target_value=1.0)
        assert np.array_equal(V.cpu().numpy(), u[f"rast_{rname}_k{kid}"])  # bit-equal masks
        kid += 1
    xy = u[f"dens_{rname}_xy"]
    st = u[f"dens_{rname}_status"]
    d = ctx.density(ctx.to_device(xy[:, 0].copy()), ctx.to_device(xy[:, 1].copy()), ctx.to_device(st), 0.5,
                    ctx.to_device(u[f"rast_{rname}_Vglobal"])).cpu().numpy()
    assert np.abs(d - u[f"dens_{rname}"]).max() < 1e-13
    d2 = co.density(ctx.X, ctx.Y, u[f"rast_{rname}_Vglobal"], xy[:, 0], xy[:, 1], st, 0.5)
    assert np.array_equal(d, d2)
    ctx.close()


def test_step_with_nobody_inside_and_single_agent(cfg):
    """edge cases: every agent already left (no noise consumed, nothing moves) and a crowd of one."""
    from oracle import cpu_oracle as co
    u = golden("units")
    room = json.loads(str(u["room"]))
    ctx, prm = _setup(room, cfg)
    Ny, Nx = ctx.Ny, ctx.Nx
    P = co.gcfm_params(cfg, room["room_length"], room["room_height"], Ny, Nx)
    Vd = ctx.to_device(u["wall_V"])
    tiles, vmin = ctx.wall_tiles(Vd)
    vx = ctx.to_device(u["samp_vx"]); vy = ctx.to_device(u["samp_vy"])
    doors = np.array([[10.0, 3.0, 0.6, 1.2]])
    key = dict(V=Vd, tiles=tiles, v_min=vmin, vx=vx, vy=vy, nt_opt=5, doors=doors)
    kc = co.KeyData(u["wall_V"], u["samp_vx"], u["samp_vy"], 5, doors)
    # (a) nobody inside
    N = 5
    st = dict(x=np.linspace(1, 3, N), y=np.full(N, 2.0), vx=np.zeros(N), vy=np.zeros(N), time=np.full(N, 1.5),
              status=np.zeros(N, dtype=np.uint8))
    dev = {k: ctx.to_device(v) for k, v in st.items()}
    ex, rc = ctx.gcfm_step(prm, dev, ctx.to_device(np.full(N, 1.3)), ctx.to_device(np.zeros(N, dtype=np.int32)), [key],
                           np.arange(N)[::-1].copy(), np.zeros((0, 2)), 0)
    assert rc == 0 and len(ex) == 0
    for k in st:
        assert np.array_equal(dev[k].cpu().numpy(), st[k])
    # (b) one agent next to the door: leaves within a few steps, bit-exact vs the oracle
    st = dict(x=np.array([9.6]), y=np.array([3.0]), vx=np.array([1.0]), vy=np.array([0.0]), time=np.zeros(1),
              status=np.ones(1, dtype=np.uint8))
    dev = {k: ctx.to_device(v) for k, v in st.items()}
    rng = np.random.RandomState(4)
    left = False
    for s in range(4):
        if not st["status"][0]:
            break
        nz = rng.normal(size=(1, 2)) * 0.01
        ex, rc = ctx.gcfm_step(prm, dev, ctx.to_device(np.array([1.3])), ctx.to_device(np.zeros(1, dtype=np.int32)), [key],
                               np.array([0]), nz, s)
        ex2, bad, _ = co.gcfm_step(P, st, np.array([1.3]), np.zeros(1, dtype=np.int32), [kc], ctx.X, ctx.Y, np.array([0]), nz, s)
        assert rc == 0 and bad == 0 and np.array_equal(ex, ex2)
        for k in st:
            assert np.array_equal(dev[k].cpu().numpy(), st[k])
        left = left or len(ex) == 1
    ctx.close()


def test_row_band_field_storage_and_ownership_change_no_bit(cfg):
    """one band that owns every row: phi slices stored as a row band (phi_row0 = -1, phi_rows = Ny + 3: the grid plus
    one halo row below and two above) and an ownership range [0, Ny) give the single-GPU step's bits over whole runs.
    Bands smaller than the grid, and key shards, are checked in test_gpu_gcfm_band.py."""
    import torch
    from optimal_crowds_b200 import _lib
    L, H, N, steps = 12.0, 9.0, 120, 6
    rng = np.random.RandomState(3)
    ctx = _lib.Context(L, H, 0.05)
    Ny, Nx = ctx.Ny, ctx.Nx
    prm = _lib.gcfm_params(cfg, L, H, Ny, Nx)
    from oracle import cpu_oracle as co
    doors = np.array([[L, H / 2, 0.6, 2.0]])
    V = co.create_potential(ctx.X, ctx.Y, [[L / 3, H / 2, 0.4, H / 2]], [], [[2 * L / 3, H / 3, 0.5]], doors)
    V[V < 0] = -100; V[V > 0] = 1
    Vd = ctx.to_device(V)
    tiles, vmin = ctx.wall_tiles(Vd)
    nt = steps + 3
    phi = ctx.hjb_solve(Vd, None, _lib.hjb_params(cfg, fused=1), nt * 0.02, nt, want_phi=True, want_vel=False)["phi"]
    band = torch.zeros((nt, Ny + 3, Nx), dtype=torch.float64, device=phi.device)
    band[:, 1:Ny + 1] = phi
    full_key = dict(V=Vd, tiles=tiles, v_min=vmin, phi=phi, nt_opt=nt, doors=doors)
    band_key = dict(full_key, phi=band, phi_row0=-1, phi_rows=Ny + 3)
    pos = _random_crowd(rng, N, L, H)
    st0 = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=rng.normal(0, 0.5, N), vy=rng.normal(0, 0.5, N),
               time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
    vd, kid = ctx.to_device(rng.normal(1.34, 0.26, N)), ctx.to_device(np.zeros(N, dtype=np.int32))
    a = {k: ctx.to_device(v) for k, v in st0.items()}
    b = {k: ctx.to_device(v) for k, v in st0.items()}
    prm_own = _lib.gcfm_params(cfg, L, H, Ny, Nx)
    prm_own.own0, prm_own.own1 = 0, Ny          # owns every row: no communicator needed
    for s in range(steps):
        perm = rng.permutation(N)
        noise = rng.normal(size=(int(a["status"].cpu().sum()), 2))
        ex_a, rc_a = ctx.gcfm_step(prm, a, vd, kid, [full_key], perm, noise, s)
        ex_b, rc_b = ctx.gcfm_step(prm_own, b, vd, kid, [band_key], perm, noise, s)
        assert rc_a == 0 and rc_b == 0 and np.array_equal(ex_a, ex_b)
        for k in a:
            assert torch.equal(a[k], b[k]), f"{k} differs at step {s}"
    ctx.close()


def test_sweep_result_is_independent_of_the_schedule(cfg):
    """size-independent property at 20k agents (no CPU oracle in reach): the concurrent sweep must give the same bits
    whatever the number of resident warps -- a grid of 2 CTAs (almost sequential), 37 CTAs and the full GPU -- because
    the dependency protocol, not the schedule, defines the result."""
    import torch
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    L, H, N, steps = 120.0, 90.0, 20000, 4
    rng = np.random.RandomState(8)
    outs = []
    for ctas in (2, 37, 0):
        rng = np.random.RandomState(8)
        ctx = _lib.Context(L, H, 0.05)
        ctx.set_int("gcfm_sweep_ctas", ctas)
        Ny, Nx = ctx.Ny, ctx.Nx
        prm = _lib.gcfm_params(cfg, L, H, Ny, Nx)
        doors = np.array([[L, H / 2, 0.6, 6.0], [0.0, H / 2, 0.6, 6.0]])
        Vd = ctx.rasterise([[L / 2, H / 2, 0.4, H / 2]], [], [[L / 3, H / 3, 1.5], [2 * L / 3, 2 * H / 3, 1.5]], doors,
                           remap=True)
        tiles, vmin = ctx.wall_tiles(Vd)
        nsl = steps + 2
        gx = torch.linspace(-1, 1, Nx - 2, device="cuda", dtype=torch.float64)
        vx = gx[None, None, :].expand(nsl, Ny - 2, Nx - 2).contiguous()
        vy = torch.zeros_like(vx)
        key = dict(V=Vd, tiles=tiles, v_min=vmin, vx=vx, vy=vy, nt_opt=nsl + 1, doors=doors)
        # a dense crowd: 20000 agents on a jittered lattice of 0.55 m pitch (3.3 ped/m^2, long dependency chains)
        side = int(np.ceil(np.sqrt(N)))
        gxp, gyp = np.meshgrid(np.arange(side), np.arange(side))
        pos = np.column_stack([gxp.ravel()[:N] * 0.55 + 10.0, gyp.ravel()[:N] * 0.55 + 5.0]) + rng.uniform(-0.1, 0.1, (N, 2))
        st = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=rng.normal(0, 0.5, N), vy=rng.normal(0, 0.5, N),
                  time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
        dev = {k: ctx.to_device(v) for k, v in st.items()}
        vd, kid = ctx.to_device(rng.normal(1.34, 0.26, N)), ctx.to_device(np.zeros(N, dtype=np.int32))
        exits = []
        for s in range(steps):
            perm = rng.permutation(N)
            noise = rng.normal(size=(int(dev["status"].sum().item()), 2))
            ex, rc = ctx.gcfm_step(prm, dev, vd, kid, [key], perm, noise, s)
            assert rc == 0
            exits.append(ex)
        outs.append(({k: v.clone() for k, v in dev.items()}, exits))
        ctx.close()
    for other, ex in outs[1:]:
        for k in outs[0][0]:
            assert torch.equal(outs[0][0][k], other[k]), k
        assert all(np.array_equal(a, b) for a, b in zip(outs[0][1], ex))
    moved = (outs[0][0]["x"].cpu().numpy() - pos[:, 0])
    assert np.abs(moved).max() > 1e-3


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


def _run_both(ctx, co, prm, P, kdev, kcpu, cpu, vdes, steps, rng):
    N = len(vdes)
    dev = {k: ctx.to_device(v) for k, v in cpu.items()}
    vd_dev, kid = ctx.to_device(vdes), np.zeros(N, dtype=np.int32)
    kid_dev = ctx.to_device(kid)
    redos = 0
    for s in range(steps):
        perm = rng.permutation(N)
        noise = rng.normal(size=(int(cpu["status"].sum()), 2))
        ex, rc = ctx.gcfm_step(prm, dev, vd_dev, kid_dev, [kdev], perm, noise, s)
        redos += ctx.gcfm_last_redos()
        ex2, bad, _ = co.gcfm_step(P, cpu, vdes, kid, [kcpu], ctx.X, ctx.Y, perm, noise, s)
        assert rc == 0 and bad == 0
        assert np.array_equal(ex, ex2), f"exit order differs at step {s}"
        for k in ("x", "y", "vx", "vy", "time", "status"):
            assert np.array_equal(dev[k].cpu().numpy(), cpu[k]), f"{k} differs at step {s}"
    return redos


@pytest.mark.parametrize("wide", [True, False])
def test_dense_jam_more_than_512_candidates_is_exact(cfg, wide):
    """8 ped/m^2: more agents within cutoff + 1 m of one agent than the shared-memory lists hold.  The reference has no
    such limit (simulations.py:285-295 visits all pairs); the step is redone on the exact slow path (global-memory
    candidate lists) and must equal the sequential CPU sweep bit for bit.  wide: the round-1 candidate search (1 m
    displacement margin, no field-of-view culling), which overflows the lists on every step; otherwise the default
    search (0.25 m margin, candidates that cannot enter the field of view dropped), which mostly fits them."""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    L = H = 12.0
    rng = np.random.RandomState(8)
    ctx = _lib.Context(L, H, 0.05)
    if wide:
        ctx.set_int("gcfm_margin_mm", 1000)
        ctx.set_int("gcfm_fov_cull", 0)
    prm = _lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    P = co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    kdev, kcpu = _one_key_room(ctx, co, L, H, 6)
    pos = _random_crowd(rng, 1000, L, H, margin=0.6, min_dist=0.2)   # 1000 agents on 10.8 x 10.8 m = 8.6 ped/m^2
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 0.7]  # off the pillar
    N = len(pos)
    assert N > 900
    cpu = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=rng.normal(0, 0.4, N), vy=rng.normal(0, 0.4, N),
               time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
    redos = _run_both(ctx, co, prm, P, kdev, kcpu, cpu, rng.normal(1.34, 0.26, N), 3, rng)
    if wide:
        assert redos >= 3          # every step overflowed the fast path and was redone
        assert ctx.gcfm_last_pairs() > 100000
    ctx.close()


@pytest.mark.parametrize("knobs", [dict(gcfm_fov_cull=0), dict(gcfm_margin_mm=1000), dict(gcfm_margin_mm=60),
                                   dict(gcfm_overlap=0, gcfm_ws_pair=0)])
def test_candidate_search_variants_are_exact(cfg, knobs):
    """the pruning of the candidate search (small displacement margin with a fast redo on the full one, field-of-view
    culling) and the side-stream overlap change no bit: 700 agents at 3.5 ped/m^2, 6 steps, against the sequential sweep"""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    L, H = 16.0, 12.5
    rng = np.random.RandomState(21)
    ctx = _lib.Context(L, H, 0.05)
    for k, v in knobs.items():
        ctx.set_int(k, v)
    prm = _lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    P = co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    kdev, kcpu = _one_key_room(ctx, co, L, H, 6)
    pos = _random_crowd(rng, 700, L, H, margin=0.6, min_dist=0.25)
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 0.7]
    N = len(pos)
    vx, vy = rng.normal(0, 0.7, N), rng.normal(0, 0.7, N)
    vx[:5] = 0.0
    vy[:5] = 0.0                                   # agents at rest: k = 0 whatever the neighbour does
    cpu = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=vx, vy=vy, time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
    redos = _run_both(ctx, co, prm, P, kdev, kcpu, cpu, rng.normal(1.34, 0.26, N), 6, rng)
    if knobs.get("gcfm_margin_mm") == 60:
        assert redos >= 1                          # 3 cm per axis is exceeded at once: redone on the full margin
    ctx.close()


def test_small_margin_overflow_is_redone_on_the_fast_path(cfg):
    """agents moving 0.16 .. 0.28 m per step exceed the default 0.25 m margin (12.5 cm per axis) but not the full one:
    the step is redone with the 1 m margin, which is then kept for the following steps (no further redo)."""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    L, H = 30.0, 20.0
    rng = np.random.RandomState(5)
    ctx = _lib.Context(L, H, 0.05)
    prm = _lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    P = co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    kdev, kcpu = _one_key_room(ctx, co, L, H, 8)
    pos = _random_crowd(rng, 400, L, H, margin=2.0)
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 1.0]
    N = len(pos)
    vx, vy = rng.normal(0, 0.5, N), rng.normal(0, 0.5, N)
    fast = rng.choice(N, 10, replace=False)
    vx[fast] = rng.choice([-1, 1], 10) * rng.uniform(8, 14, 10)
    cpu = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=vx, vy=vy, time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
    redos = _run_both(ctx, co, prm, P, kdev, kcpu, cpu, rng.normal(1.34, 0.26, N), 4, rng)
    assert 1 <= redos <= 2     # (the speed clip brings the fast agents back to v_max after their first step)
    ctx.close()


def test_displacement_beyond_search_margin_is_exact(cfg):
    """agents that move more than 0.5 m per axis in one step (repulsions add to the velocity unclipped, and the position
    update is not speed-limited: simulations.py:303,312-326): the candidate search is widened and the step redone."""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    L, H = 30.0, 20.0
    rng = np.random.RandomState(3)
    ctx = _lib.Context(L, H, 0.05)
    prm = _lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    P = co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    kdev, kcpu = _one_key_room(ctx, co, L, H, 8)
    N = 300
    pos = _random_crowd(rng, N, L, H, margin=2.0)
    pos = pos[np.hypot(pos[:, 0] - L / 2, pos[:, 1] - H / 2) > 1.0]
    N = len(pos)
    vx, vy = rng.normal(0, 0.5, N), rng.normal(0, 0.5, N)
    fast = rng.choice(N, 12, replace=False)
    vx[fast] = rng.choice([-1, 1], 12) * rng.uniform(30, 90, 12)     # 0.6 .. 1.8 m per step
    cpu = dict(x=pos[:, 0].copy(), y=pos[:, 1].copy(), vx=vx, vy=vy, time=np.zeros(N), status=np.ones(N, dtype=np.uint8))
    redos = _run_both(ctx, co, prm, P, kdev, kcpu, cpu, rng.normal(1.34, 0.26, N), 2, rng)
    assert redos >= 1
    ctx.close()


def test_sampler_wraps_negative_indices_like_numpy(cfg):
    """an agent at x < 0 or y < 0 makes the reference read vx_opt[t][-1, ...]: numpy wraps, no exception (App. C #7)"""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import _lib
    L, H = 6.0, 4.0
    rng = np.random.RandomState(1)
    ctx = _lib.Context(L, H, 0.05)
    prm = _lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    P = co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    kdev, kcpu = _one_key_room(ctx, co, L, H, 4)
    pts = np.array([[-0.02, 1.0], [1.0, -0.07], [-0.3, -0.01], [2.0, 2.0]])
    N = len(pts)
    for storage in ("velocity", "phi"):
        cpu = dict(x=pts[:, 0].copy(), y=pts[:, 1].copy(), vx=np.zeros(N), vy=np.zeros(N), time=np.zeros(N),
                   status=np.ones(N, dtype=np.uint8))
        if storage == "velocity":
            _run_both(ctx, co, prm, P, kdev, kcpu, cpu, np.full(N, 1.3), 1, rng)
        else:
            # same answer when the sampler differentiates phi samples on the fly: only the index rule is exercised
            dev = {k: ctx.to_device(v) for k, v in cpu.items()}
            phi = ctx.to_device(rng.uniform(1.0, 2.0, (6, ctx.Ny, ctx.Nx)))
            k2 = dict(kdev, vx=None, vy=None, phi=phi, nt_opt=5)
            _, rc = ctx.gcfm_step(prm, dev, ctx.to_device(np.full(N, 1.3)), ctx.to_device(np.zeros(N, dtype=np.int32)),
                                  [k2], np.arange(N), np.zeros((N, 2)), 0)
            assert rc == 0
    ctx.close()


def test_fp64_peak_microbenchmark(cfg):
    from optimal_crowds_b200 import _lib
    ctx = _lib.Context(6.0, 4.0, 0.05)
    tf = ctx.fp64_peak()
    assert 5.0 < tf < 80.0, tf   # B200: ~34 TFLOP/s measured (nominal 37-40)
    ctx.close()
