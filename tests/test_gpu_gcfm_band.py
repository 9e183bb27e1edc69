"""GPU parity of the distributed GCFM step's per-agent terms, with one GPU running every rank's share in turn.

In a row-decomposed run (`simulation(..., band=True)`) and in a key-sharded run (`shard_keys=True`) a rank evaluates the
field sample and the wall force only for the agents it owns (`oc_gcfm_params.own0/own1`, `key_mod/key_rem`) and writes
all-zero bits for the others; a bit-wise max-reduction over the ranks then merges the terms.  That reproduces the
single-GPU step only if every agent has exactly one owner, the owner's band-shaped phi slices hold every row the sampler
reads, and the owner computes the single-GPU bits.

Without a communicator a step with an ownership range or a key shard computes only that rank's share of the terms.  The
probe agents of one step stand 6 m apart in x, farther than the repulsion cutoff (4 m) plus a step's displacement, so an
agent's result depends on its own terms only: the owner's result for it must equal the single-GPU step (which is checked
against the sequential CPU sweep O2) bit for bit, the owner's return code must be the single-GPU step's, and no other
rank may raise the sampler-range error for it.  The expected owner is computed here from the reference's index rule
(optimals.py:234-248 with numpy's wrap of negative indices), not from the library.

The phi samples are random, so every node's value differs and a read of a wrong row changes bits.  A band's phi block sits
inside a larger allocation whose rows outside the block, and the block's rows outside the grid, are NaN.
"""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H = 6.36                                # 6.36 // 0.05 == 127: Ny = 128, bands of 64 / 32 / 16 rows for R = 2 / 4 / 8
ROOM_LENGTH = {"even": 96.0, "odd": 96.05}   # Nx = 1920 / 1921
PITCH = 6.0                             # x distance between the probe agents of one step
NT = 6                                  # phi samples per target set (nt_opt)
FIELDS = ("x", "y", "vx", "vy", "time", "status")


def _cfg():
    with open(os.path.join(REPO, "optimal_crowds_b200", "config.json")) as f:
        return json.load(f)


# ----------------------------------------------------------------------------------------- the reference's index rule
def _rows(y, P):
    """(i0, i1): the interior field rows the reference's sampler reads for an agent at y (optimals.py:234-248, a negative
    index wrapped as numpy does; the list has one element then)"""
    if y < P.room_height - P.dy:
        i0 = int(y // P.dy)
        i1 = i0 + 1 if y > P.dy else i0
    else:
        i0 = i1 = P.Ny - 3
    if i0 < 0:
        i0 += P.Ny - 2
        i1 = i0
    return i0, i1


def _in_range(y, P):
    i0, i1 = _rows(y, P)
    return i0 >= 0 and i1 < P.Ny - 2


def _owner_band(y, P, R):
    """the band that holds node row i0 + 1 (an index out of range even after the wrap: clamped into the grid)"""
    from optimal_crowds_b200 import dist
    i0, _ = _rows(y, P)
    return min(max(i0 + 1, 0), P.Ny - 1) // dist.band_rows(P.Ny, R)


def _row_probes(P, Y):
    """y of the probe agents: every owner row around every band edge of R = 2, 4, 8, node rows and cell boundaries of the
    sampler with their neighbouring doubles, both ends of the grid, and negative y (wrapped to the last rows or to the
    middle, or out of range even after the wrap).  Second list: y of the probes at x in (-dx, 0), the column wrap."""
    dy, Ny, Hr = P.dy, P.Ny, P.room_height
    up, down = (lambda v: np.nextafter(v, np.inf)), (lambda v: np.nextafter(v, -np.inf))
    ys = []
    for e in range(16, Ny, 16):
        ys += [(r - 0.5) * dy for r in range(e - 2, e + 2)]          # mid-cell, owner rows e-2 .. e+1
        for v in (Y[e - 1], Y[e], (e - 1) * dy, e * dy):              # on a node row / on a cell boundary of the sampler
            ys += [down(v), v, up(v)]
    ys += [0.0, 0.5 * dy, down(dy), dy, up(dy), 1.5 * dy]                # i1 == i0 up to dy
    ys += [(Ny - 3.5) * dy, (Ny - 3) * dy, (Ny - 2.5) * dy, Hr - dy - 0.005, down(Hr - dy),
           Hr - dy, Hr - 0.5 * dy, Y[-2], Hr]                            # the top: out of range below Hr - dy, then clamped
    ys += [-0.0, -1e-300, -0.5 * dy, up(-dy), -dy, down(-dy), -1.5 * dy, -3.0,    # wrapped to the last rows / the middle
           -(Ny - 2.5) * dy, -(Ny - 2) * dy, -(Ny - 1.5) * dy, -50.0]     # wrapped to row 0, then out of range
    wrap = [(e + d) * dy for e in range(16, Ny, 16) for d in (-0.5, 0.5)] + [-0.5 * dy, Hr - 0.5 * dy, -(Ny - 1.5) * dy]
    return ys, wrap


def _groups(ys, wrap, P, L):
    """(x, y) of the probe agents of each step.  The columns stand PITCH apart, and only column 0 can hold a probe of the
    column wrap.  In-range probes share steps; every out-of-range probe gets a step of its own, so that a sampler-range
    error belongs to one agent."""
    x0 = 3.0123                                   # off every node column, so that no agent stands on a wall node
    xw = -0.5 * P.dx
    cols = int((L - 1.0) // PITCH)
    ok, ok_w = [y for y in ys if _in_range(y, P)], [y for y in wrap if _in_range(y, P)]
    chunks = [ok[q:q + cols - 1] for q in range(0, len(ok), cols - 1)]
    chunks += [[]] * (len(ok_w) - len(chunks))
    groups = []
    for c, chunk in enumerate(chunks):
        pts = [(xw, ok_w[c])] if c < len(ok_w) else []
        groups.append(np.array(pts + [(x0 + PITCH * (q + 1), y) for q, y in enumerate(chunk)]))
    groups += [np.array([(x0, y)]) for y in ys if not _in_range(y, P)]
    groups += [np.array([(xw, y)]) for y in wrap if not _in_range(y, P)]
    return groups


# ----------------------------------------------------------------------------------------------------- rooms and steps
def _room(L, n_keys):
    """context of the single-GPU step, context of the ranks' shares (no CUDA graph, like a distributed step), and per
    target set (device key with full-grid random phi samples, O2 key with the velocity slices of the same samples)"""
    import torch
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    cfg = _cfg()
    ctx = _lib.Context(L, H, cfg["grid_step"])
    share = _lib.Context(L, H, cfg["grid_step"])
    share.set_int("gcfm_graph", 0)
    Ny, Nx, Y = ctx.Ny, ctx.Nx, ctx.Y
    assert Ny == 128
    hp = _lib.hjb_params(cfg)
    rng = np.random.RandomState(Nx + n_keys)
    walls = [[PITCH * 3, Y[64], 0.3, 1.5], [PITCH * 7, Y[32], 0.3, 0.8]]      # across band edges, between probe columns
    cyls = [[PITCH * 5, Y[96], 0.5], [PITCH * 9, Y[16], 0.4]]
    # doors on the right, left, top and bottom walls; the probe columns 11 and 13 (x = 69 m, 81 m) cross two of them
    all_doors = [np.array([[L, H / 2, 0.6, 2.0], [PITCH * 13 + 3.0, H, 2.0, 0.6]]), np.array([[0.0, H / 2, 0.6, 2.0]]),
                 np.array([[L / 2, H, 3.0, 0.6], [PITCH * 11 + 3.0, 0.0, 2.0, 0.6]])]
    keys = []
    for kd in all_doors[:n_keys]:
        V = co.create_potential(ctx.X, Y, walls, [], cyls, kd)
        V[V < 0] = -100; V[V > 0] = 1
        Vd = ctx.to_device(V)
        tiles, vmin = ctx.wall_tiles(Vd)
        phi = ctx.to_device(rng.uniform(1.0, 2.0, (NT, Ny, Nx)))
        vx = np.empty((NT - 1, Ny - 2, Nx - 2)); vy = np.empty_like(vx)
        for s in range(NT - 1):             # vx_opt[s] = vels(phi[nt_opt-1-s]) (optimals.py:200-204)
            a, b = ctx.hjb_vels(phi[NT - 1 - s], hp)
            vx[s], vy[s] = a.cpu().numpy(), b.cpu().numpy()
        keys.append((dict(V=Vd, tiles=tiles, v_min=vmin, phi=phi, nt_opt=NT, doors=kd, mu=hp.mu, lim=hp.lim),
                     co.KeyData(V, vx, vy, NT, kd)))
    torch.cuda.synchronize()
    return cfg, ctx, share, keys


def _band_key(key, own0, own1):
    """the key as the rank of band [own0, own1) holds it: phi rows [own0-1, own1+2), cut out of the full samples, inside
    an allocation that is NaN around the block and on the block's rows outside the grid"""
    import torch
    phi = key["phi"]
    nt, Ny, Nx = phi.shape
    rows = own1 - own0 + 3
    buf = torch.full((nt + 2, rows, Nx), float("nan"), dtype=phi.dtype, device=phi.device)
    blk = buf[1:nt + 1]
    lo, hi = max(own0 - 1, 0), min(own1 + 2, Ny)
    blk[:, lo - (own0 - 1):hi - (own0 - 1)] = phi[:, lo:hi]
    return dict(key, phi=blk, phi_row0=own0 - 1, phi_rows=rows)


def _crowd(pts, n_keys, seed):
    rng = np.random.RandomState(seed)
    N = len(pts)
    st = dict(x=pts[:, 0].copy(), y=pts[:, 1].copy(), vx=rng.normal(0, 0.5, N), vy=rng.normal(0, 0.5, N),
              time=np.full(N, 0.02), status=np.ones(N, dtype=np.uint8))
    return st, rng.normal(1.34, 0.26, N), (np.arange(N) + seed) % n_keys, rng.permutation(N), rng.normal(size=(N, 2))


def _step(ctx, prm, keys, crowd, t):
    """one step from the crowd's initial state -> (state as numpy, exit log, return code)"""
    st, vdes, kid, perm, noise = crowd
    dev = {k: ctx.to_device(v) for k, v in st.items()}
    ex, rc = ctx.gcfm_step(prm, dev, ctx.to_device(vdes), ctx.to_device(kid.astype(np.int32)), keys, perm, noise, t)
    return {k: v.cpu().numpy() for k, v in dev.items()}, ex, rc


def _bits(a):
    return a.view(np.uint8) if a.dtype == np.uint8 else a.view(np.int64)


def _full_step(cfg, ctx, keys, crowd, t):
    """the single-GPU step, checked against O2"""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    L, Ny, Nx = ctx.room_length, ctx.Ny, ctx.Nx
    prm = _lib.gcfm_params(cfg, L, H, Ny, Nx)
    res, ex, rc = _step(ctx, prm, [k[0] for k in keys], crowd, t)
    st, vdes, kid, perm, noise = crowd
    cpu = {k: v.copy() for k, v in st.items()}
    ex2, bad, _ = co.gcfm_step(co.gcfm_params(cfg, L, H, Ny, Nx), cpu, vdes, kid, [k[1] for k in keys], ctx.X, ctx.Y,
                               perm, noise, t)
    assert (rc == _lib.OC_ERR_SAMPLER_RANGE) == bool(bad)
    assert np.array_equal(ex, ex2)
    for k in FIELDS:
        assert np.array_equal(_bits(res[k]), _bits(cpu[k])), k
    return res, ex, rc


def _assert_share(res, ex, rc, full, mine, oor, t, what):
    """the share's result for the agents it owns equals the single-GPU step; it raises the sampler-range error exactly
    when one of them is out of range (then so does the single-GPU step)"""
    from optimal_crowds_b200 import _lib
    f_res, f_ex, f_rc = full
    for k in FIELDS:
        assert np.array_equal(_bits(res[k][mine]), _bits(f_res[k][mine])), f"{what}: {k} of an owned agent differs"
    owned = np.flatnonzero(mine)
    assert np.array_equal(ex[np.isin(ex, owned)], f_ex[np.isin(f_ex, owned)]), f"{what}: exit log differs"
    flag = bool(np.any(mine & oor)) and t < NT - 1
    assert (rc == _lib.OC_ERR_SAMPLER_RANGE) == flag, f"{what}: rc {rc}, owns an agent out of range: {flag}"
    if flag:
        assert rc == f_rc


# ------------------------------------------------------------------------------------------------------------ the tests
@pytest.mark.parametrize("t", [0, NT - 2, NT - 1, NT + 3])
@pytest.mark.parametrize("parity", ["even", "odd"])
def test_row_band_shares_reassemble_the_single_gpu_step(parity, t):
    """R = 2, 4, 8 bands of a 128-row grid: every probe agent is owned by exactly one band, the band that holds node row
    i0 + 1 of the sampler's wrapped row indices, and that band's band-shaped phi gives the single-GPU step's bits."""
    from optimal_crowds_b200 import _lib, dist
    from oracle import cpu_oracle as co
    L = ROOM_LENGTH[parity]
    cfg, ctx, share, keys = _room(L, 1)
    assert ctx.Nx % 2 == (parity == "odd")
    P = co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    groups = _groups(*_row_probes(P, ctx.Y), P, L)
    owners = {R: set() for R in (2, 4, 8)}
    n_wrapped = n_oor = 0
    for g, pts in enumerate(groups):
        crowd = _crowd(pts, 1, 100 * g + t)
        full = _full_step(cfg, ctx, keys, crowd, t)
        oor = np.array([not _in_range(y, P) for y in pts[:, 1]])
        n_oor += int(oor.sum())
        n_wrapped += int(np.sum((pts[:, 1] < 0) & ~oor))
        for R in (2, 4, 8):
            owner = np.array([_owner_band(y, P, R) for y in pts[:, 1]])
            owners[R] |= set(owner.tolist())
            for r in range(R):
                own0, own1 = dist.band_of(r, ctx.Ny, R)
                prm = _lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
                prm.own0, prm.own1 = own0, own1
                res, ex, rc = _step(share, prm, [_band_key(keys[0][0], own0, own1)], crowd, t)
                _assert_share(res, ex, rc, full, owner == r, oor, t, f"group {g} (y = {pts[:, 1].tolist()}), band {r}/{R}")
    for R in (2, 4, 8):
        assert owners[R] == set(range(R))
    assert n_wrapped >= 8 and n_oor >= 5
    ctx.close()
    share.close()


@pytest.mark.parametrize("t", [0, NT - 2, NT - 1])
@pytest.mark.parametrize("key_mod", [2, 3])
def test_key_shards_reassemble_the_single_gpu_step(key_mod, t):
    """3 target sets with different doors dealt to key_mod ranks: the rank k % key_mod owns the agents of key k and holds
    only its keys' fields (the others are passed without phi, as optimals(owned=False) leaves them)."""
    from optimal_crowds_b200 import _lib
    from oracle import cpu_oracle as co
    L = ROOM_LENGTH["odd"]
    cfg, ctx, share, keys = _room(L, 3)
    P = co.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
    groups = _groups(*_row_probes(P, ctx.Y), P, L)
    for g, pts in enumerate(groups):
        crowd = _crowd(pts, 3, 100 * g + t)
        kid = crowd[2]
        full = _full_step(cfg, ctx, keys, crowd, t)
        oor = np.array([not _in_range(y, P) for y in pts[:, 1]])
        for rem in range(key_mod):
            prm = _lib.gcfm_params(cfg, L, H, ctx.Ny, ctx.Nx)
            prm.key_mod, prm.key_rem = key_mod, rem
            held = [k[0] if q % key_mod == rem else dict(k[0], phi=None) for q, k in enumerate(keys)]
            res, ex, rc = _step(share, prm, held, crowd, t)
            _assert_share(res, ex, rc, full, kid % key_mod == rem, oor, t, f"group {g}, shard {rem}/{key_mod}")
    ctx.close()
    share.close()


@pytest.mark.parametrize("remap", [True, False])
@pytest.mark.parametrize("parity", ["even", "odd"])
def test_rasterise_band_equals_the_rows_of_the_full_grid(parity, remap):
    """oc_rasterise_band of every band of R = 2, 4, 8 (and of bands that do not start on a block of 8 rows) equals those
    rows of oc_rasterise, bit for bit; walls, holes, cylinders and targets straddle the band edges.  The full grid equals
    O2's create_potential."""
    import torch
    from optimal_crowds_b200 import _lib, dist
    from oracle import cpu_oracle as co
    L = 20.0 + (parity == "odd") * 0.05
    ctx = _lib.Context(L, H, _cfg()["grid_step"])
    Ny, Y = ctx.Ny, ctx.Y
    assert Ny == 128 and ctx.Nx % 2 == (parity == "odd")
    walls = [[L / 3, Y[64], 2.0, 0.4], [2 * L / 3, Y[32] + 0.01, 0.4, 1.6], [L / 2, Y[16], L / 2, 0.05],
             [L / 5, (Y[95] + Y[96]) / 2, 1.0, Y[96] - Y[95]]]
    holes = [[L / 3, Y[64], 0.5, 1.0], [2 * L / 3, Y[32], 0.4, 0.3]]
    cyls = [[L / 4, Y[48], 0.8], [3 * L / 4, Y[96], 0.3], [L / 5, Y[112], 1.0], [L / 3, Y[64], 0.35]]
    targets = [[L, Y[80], 0.6, 2.0], [0.0, Y[48], 0.6, 1.6], [L / 2, H, 3.0, 0.6], [L / 3, Y[64], 0.2, 0.2]]
    full = ctx.rasterise(walls, holes, cyls, targets, remap=remap)
    ref = co.create_potential(ctx.X, Y, walls, holes, cyls, targets)
    if remap:
        ref[ref < 0] = -100.0; ref[ref > 0] = 1.0
    assert np.array_equal(full.cpu().numpy(), ref)
    assert len(np.unique(ref)) >= 3
    bands = [dist.band_of(r, Ny, R) for R in (2, 4, 8) for r in range(R)] + [(5, 18), (61, 67), (Ny - 7, Ny), (0, 1)]
    for own0, own1 in bands:
        V = ctx.rasterise_band(walls, holes, cyls, targets, own0, own1 - own0, remap=remap)
        assert torch.equal(V, full[own0:own1]), (own0, own1)
    ctx.close()
