"""Simulation driver -- mirror of the reference's ``simulations.simulation`` (simulations.py:18-703).

Same public surface: ``simulation(room, T, recompute=False)``, ``run(verbose, draw, mode)``,
``step(dt, verbose)``, ``draw_history(mode)``, ``draw(mode)``, ``draw_final_trajectories()``,
``evac_times(draw)``, ``initial_positions()``, ``gaussian_density(sigma)``, ``create_potential(var_room,
targets)``, ``write_history(time)`` and the attributes the reference's users read (``agents, targets, Vs, V,
N, inside, time, simu_step, history, ...``).  File formats (rooms/*.json, config.json), CWD-relative paths,
printed messages and the numpy legacy global RNG stream are the reference's.

What runs where: JSON parsing, the RNG, the run loop, history bookkeeping and plotting stay on the host;
rasterisation, the HJB solve, the density splat and the whole GCFM step run in liboc_b200.so on the GPU.
The crowd lives on the device as struct-of-arrays; ``self.agents`` are ``pedestrians.ped`` views.
"""
from __future__ import annotations

import json
import warnings

import os

import numpy as np

from . import _crowd, _lib, _rng, optimals, pedestrians
from .optimals import _load_config, _load_room, _merge_config

warnings.filterwarnings("ignore")  # simulations.py:15


def density_stats_spec(value, with_velocity=False):
    """(every, threshold) of a ``density_stats`` argument -- (every, threshold, velocity) with ``with_velocity`` -- or None
    when the statistics are off: None / False (off), True (every frame, no threshold, no velocity maps) or
    dict(every=1, threshold=None, velocity=False); checked without touching a GPU"""
    if value is None or value is False:
        return None
    if value is True:
        return (1, None, False) if with_velocity else (1, None)
    if not isinstance(value, dict):
        raise ValueError("density_stats: expected None, True or dict(every=..., threshold=..., velocity=...)")
    unknown = set(value) - {"every", "threshold", "velocity"}
    if unknown:
        raise ValueError(f"density_stats: unknown keys {sorted(unknown)}")
    every, thr, vel = value.get("every", 1), value.get("threshold"), value.get("velocity", False)
    if isinstance(every, bool) or not isinstance(every, (int, np.integer)) or every < 1:
        raise ValueError("density_stats: every must be an integer >= 1")
    if thr is not None:
        if isinstance(thr, bool) or not isinstance(thr, (int, float, np.integer, np.floating)) or not np.isfinite(thr):
            raise ValueError("density_stats: threshold must be None or a finite number")
        thr = float(thr)
    if not isinstance(vel, (bool, np.bool_)):
        raise ValueError("density_stats: velocity must be True or False")
    return (int(every), thr, bool(vel)) if with_velocity else (int(every), thr)


MAX_LINES = 64


def lines_spec(value):
    """(names, (n, 4) float64 array) of a ``lines`` argument -- {name: (x0, y0, x1, y1)} in metres, 1 to 64 lines, finite
    coordinates, non-zero length -- or None for None; checked without touching a GPU"""
    if value is None:
        return None
    if not isinstance(value, dict) or not value:
        raise ValueError("lines: expected a non-empty dict {name: (x0, y0, x1, y1)}")
    if len(value) > MAX_LINES:
        raise ValueError(f"lines: at most {MAX_LINES} measurement lines")
    names, rows = [], []
    for name, seg in value.items():
        try:
            c = np.asarray(seg, dtype=np.float64)
        except (TypeError, ValueError):
            raise ValueError(f"lines: {name!r} is not (x0, y0, x1, y1)") from None
        if c.shape != (4,) or isinstance(seg, (str, bytes)) or any(isinstance(v, (bool, np.bool_)) for v in seg):
            raise ValueError(f"lines: {name!r} is not (x0, y0, x1, y1)")
        if not np.isfinite(c).all():
            raise ValueError(f"lines: the coordinates of {name!r} must be finite")
        if c[0] == c[2] and c[1] == c[3]:
            raise ValueError(f"lines: {name!r} has zero length")
        names.append(name)
        rows.append(c)
    return names, np.array(rows, dtype=np.float64)


MAX_AREAS, MAX_AREA_VERTS, MAX_VERTS = 64, 64, 1024


def _polygon_simple(v):
    """True when the closed polygon v ((n, 2) float64, n >= 3) does not touch itself: consecutive edges meet only at
    their common vertex (no zero-length edge, no fold back along the same line) and other edges have no point in common"""
    n = len(v)
    a, b = v, np.roll(v, -1, axis=0)                  # edge k: a[k] -> b[k]
    d = b - a
    if (np.all(d == 0, axis=1)).any():
        return False
    # consecutive edges k, k+1: a fold back is collinear with opposite directions
    dn = np.roll(d, -1, axis=0)
    cross = d[:, 0] * dn[:, 1] - d[:, 1] * dn[:, 0]
    if ((cross == 0) & (np.sum(d * dn, axis=1) < 0)).any():
        return False
    i, j = np.triu_indices(n, 2)
    keep = ~((i == 0) & (j == n - 1))                 # (edges n-1 and 0 are consecutive)
    i, j = i[keep], j[keep]
    if not len(i):
        return True
    p1, p2, p3, p4 = a[i], b[i], a[j], b[j]
    o = lambda u, w, z: (w[:, 0] - u[:, 0]) * (z[:, 1] - u[:, 1]) - (w[:, 1] - u[:, 1]) * (z[:, 0] - u[:, 0])
    d1, d2, d3, d4 = o(p3, p4, p1), o(p3, p4, p2), o(p1, p2, p3), o(p1, p2, p4)
    proper = (np.sign(d1) * np.sign(d2) < 0) & (np.sign(d3) * np.sign(d4) < 0)

    def on(u, w, z, dz):                              # z collinear with u-w and inside its bounding box
        return (dz == 0) & (np.minimum(u[:, 0], w[:, 0]) <= z[:, 0]) & (z[:, 0] <= np.maximum(u[:, 0], w[:, 0])) & \
            (np.minimum(u[:, 1], w[:, 1]) <= z[:, 1]) & (z[:, 1] <= np.maximum(u[:, 1], w[:, 1]))
    touch = on(p3, p4, p1, d1) | on(p3, p4, p2, d2) | on(p1, p2, p3, d3) | on(p1, p2, p4, d4)
    return not (proper | touch).any()


class AreasSpec(tuple):
    """(names, (V, 2) float64 vertices, (A + 1) int32 offsets): a checked ``areas`` argument"""


def areas_spec(value):
    """AreasSpec (names, (V, 2) float64 vertices, (A + 1) int32 offsets) of an ``areas`` argument -- {name: [(x0, y0),
    (x1, y1), ...]} in metres: 1 to 64 simple polygons of 3 to 64 vertices, 1024 vertices in all, finite coordinates,
    non-zero area -- or None for None; checked without touching a GPU.  An AreasSpec is returned as it is (ensemble
    members take the ensemble's checked areas)"""
    if value is None or isinstance(value, AreasSpec):
        return value
    if not isinstance(value, dict) or not value:
        raise ValueError("areas: expected a non-empty dict {name: [(x0, y0), (x1, y1), ...]}")
    if len(value) > MAX_AREAS:
        raise ValueError(f"areas: at most {MAX_AREAS} measurement areas")
    names, polys, total = [], [], 0
    for name, poly in value.items():
        bad = ValueError(f"areas: {name!r} is not a list of (x, y) vertices")
        if isinstance(poly, (str, bytes, dict)):
            raise bad
        try:
            pts = list(poly)
            if any(isinstance(p, (str, bytes, dict)) or any(isinstance(c, (bool, np.bool_, str, bytes)) for c in p)
                   for p in pts):
                raise bad
            v = np.asarray(pts, dtype=np.float64)
        except (TypeError, ValueError):
            raise bad from None
        if v.ndim != 2 or v.shape[1] != 2:
            raise bad
        if not MAX_AREA_VERTS >= len(v) >= 3:
            raise ValueError(f"areas: {name!r} must have 3 to {MAX_AREA_VERTS} vertices")
        if not np.isfinite(v).all():
            raise ValueError(f"areas: the vertices of {name!r} must be finite")
        if _lib.polygon_area(v) == 0:
            raise ValueError(f"areas: {name!r} has zero area")
        if not _polygon_simple(v):
            raise ValueError(f"areas: {name!r} is not a simple polygon (its edges touch or cross)")
        total += len(v)
        if total > MAX_VERTS:
            raise ValueError(f"areas: at most {MAX_VERTS} vertices in all")
        names.append(name)
        polys.append(v)
    offsets = np.concatenate([[0], np.cumsum([len(v) for v in polys])]).astype(np.int32)
    return AreasSpec((names, np.concatenate(polys), offsets))


class VoronoiSpec(tuple):
    """(cutoff, edges): a checked ``voronoi`` argument"""


def voronoi_spec(value):
    """VoronoiSpec (cutoff in metres, edges of the cut-off polygon) of a ``voronoi`` argument -- True (cutoff=1.0,
    edges=12) or dict(cutoff=..., edges=...): cutoff finite in (0, 100], edges an integer in 4..32 -- or None for None
    and False; checked without touching a GPU.  A VoronoiSpec is returned as it is"""
    if value is None or value is False or isinstance(value, VoronoiSpec):
        return value if value is not False else None
    if value is True:
        value = {}
    if not isinstance(value, dict):
        raise ValueError("voronoi: expected True or dict(cutoff=1.0, edges=12)")
    unknown = set(value) - {"cutoff", "edges"}
    if unknown:
        raise ValueError(f"voronoi: unknown keys {sorted(map(str, unknown))}")
    return VoronoiSpec(_cutoff_edges(value, "voronoi"))


def _cutoff_edges(value, name):
    """(cutoff, edges) of a dict argument: cutoff finite in (0, 100] metres (default 1.0), edges an integer in 4..32
    (default 12); ValueError naming the option `name` otherwise"""
    cutoff, edges = value.get("cutoff", 1.0), value.get("edges", 12)
    if isinstance(cutoff, (bool, np.bool_)) or not isinstance(cutoff, (int, float, np.integer, np.floating)) or \
            not (np.isfinite(cutoff) and 0 < cutoff <= 100):
        raise ValueError(f"{name}: cutoff must be a finite number of metres in (0, 100]")
    if isinstance(edges, (bool, np.bool_)) or not isinstance(edges, (int, np.integer)) or not 4 <= edges <= 32:
        raise ValueError(f"{name}: edges must be an integer in 4..32")
    return float(cutoff), int(edges)


class VoronoiMapsSpec(tuple):
    """(every, cutoff, edges): a checked ``voronoi_maps`` argument"""


def voronoi_maps_spec(value):
    """VoronoiMapsSpec (every, cutoff in metres, edges of the cut-off polygon) of a ``voronoi_maps`` argument -- True
    (every=1, cutoff=1.0, edges=12) or dict(every=..., cutoff=..., edges=...): every an integer >= 1, cutoff and edges
    as for ``voronoi`` -- or None for None and False; checked without touching a GPU.  A VoronoiMapsSpec is returned as
    it is"""
    if value is None or value is False or isinstance(value, VoronoiMapsSpec):
        return value if value is not False else None
    if value is True:
        value = {}
    if not isinstance(value, dict):
        raise ValueError("voronoi_maps: expected True or dict(every=1, cutoff=1.0, edges=12)")
    unknown = set(value) - {"every", "cutoff", "edges"}
    if unknown:
        raise ValueError(f"voronoi_maps: unknown keys {sorted(map(str, unknown))}")
    every = value.get("every", 1)
    if isinstance(every, (bool, np.bool_)) or not isinstance(every, (int, np.integer)) or every < 1:
        raise ValueError("voronoi_maps: every must be an integer >= 1")
    return VoronoiMapsSpec((int(every),) + _cutoff_edges(value, "voronoi_maps"))


def _turn(a, b, c):
    """orientation of the corner a -> b -> c: > 0 for a left (counter-clockwise) turn, 0 when collinear"""
    return (b[0] - a[0]) * (c[1] - b[1]) - (b[1] - a[1]) * (c[0] - b[0])


def _drop_straight(pts):
    """drop vertices whose turn is exactly zero, one at a time from the front, until none is left"""
    k = 0
    while len(pts) > 3 and k < len(pts):
        if _turn(pts[k - 1], pts[k], pts[(k + 1) % len(pts)]) == 0:
            del pts[k]
            k = 0
        else:
            k += 1
    return pts


def _triangulate(v):
    """counter-clockwise triangles covering the simple polygon v ((n, 2)), by ear clipping: the polygon turned
    counter-clockwise, vertices with a zero turn dropped (again after every ear); the ear is the first vertex, in the
    current order, with a left turn whose triangle holds no other vertex (closed triangle; if no vertex qualifies, open)"""
    pts = [(float(x), float(y)) for x, y in v]
    if sum(a[0] * b[1] - b[0] * a[1] for a, b in zip(pts, pts[1:] + pts[:1])) < 0:
        pts.reverse()
    pts = _drop_straight(pts)
    tris = []

    def holds(a, b, c, p, closed):
        o = (_turn(a, b, p), _turn(b, c, p), _turn(c, a, p))   # (sign of o(a,b,p) etc. for a counter-clockwise a, b, c)
        return all(t >= 0 for t in o) if closed else all(t > 0 for t in o)

    while len(pts) > 3:
        n, ear = len(pts), None
        for closed in (True, False):
            for k in range(n):
                a, b, c = pts[k - 1], pts[k], pts[(k + 1) % n]
                if _turn(a, b, c) <= 0:
                    continue
                if not any(holds(a, b, c, pts[j], closed) for j in range(n) if j not in ((k - 1) % n, k, (k + 1) % n)):
                    ear = k
                    break
            if ear is not None:
                break
        if ear is None:
            raise ValueError("areas: a polygon could not be triangulated")
        tris.append((pts[ear - 1], pts[ear], pts[(ear + 1) % n]))
        del pts[ear]
        pts = _drop_straight(pts)
    tris.append(tuple(pts))
    return tris


def voronoi_triangles(aspec):
    """(T, 3, 2) float64 counter-clockwise triangles of the areas of an AreasSpec, area after area in a fixed order,
    and (n_areas + 1) int32 offsets into them; computed once per AreasSpec"""
    cached = getattr(aspec, "_triangles", None)
    if cached is None:
        names, verts, offsets = aspec
        per = [_triangulate(verts[a:b]) for a, b in zip(offsets[:-1], offsets[1:])]
        tris = np.array([t for p in per for t in p], dtype=np.float64).reshape(-1, 3, 2)
        toff = np.concatenate([[0], np.cumsum([len(p) for p in per])]).astype(np.int32)
        cached = aspec._triangles = (tris, toff)
    return cached


def density_frame_steps(T, dt, every, recompute_step=None):
    """The simu_steps whose frames run() adds to the density statistics when nobody leaves before T: run()'s loop
    (simulations.py:427-441) as it is cut into blocks here -- one advance() per stretch up to the next re-solve (every
    ``recompute_step`` steps, None = no re-solves) -- each block taking the frames of its steps that are multiples of
    ``every``.  The frames do not depend on the cut: this is the plain loop's selection."""
    out, time, step = [], 0., 0
    while time < T:
        n, t = 0, time
        while t < T:
            t += dt
            n += 1
            if recompute_step and (step + n) % recompute_step == 0:
                break
        for _ in range(n):
            if step % every == 0:
                out.append(step)
            time += dt
            step += 1
    return out


class _Agents:
    """``simulation.agents``: the reference's array of ``ped`` objects (simulations.py:142-151), built on first access.
    A ``ped`` here is a view of row i of the device-resident crowd state, so nothing but the object itself is created;
    constructing 1000 of them costs as much as placing the crowd, 100 k half a second.  Indexing (int, slice, index or
    boolean arrays), iteration, ``len`` and ``np.asarray`` behave like the object array."""

    def __init__(self, n, make):
        self._n, self._make, self._made = int(n), make, {}

    def __len__(self):
        return self._n

    @property
    def shape(self):
        return (self._n,)

    size = property(lambda self: self._n)
    dtype = np.dtype(object)
    ndim = 1

    def _one(self, i):
        i = int(i)
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(f"index {i} is out of bounds for axis 0 with size {self._n}")
        a = self._made.get(i)
        if a is None:
            a = self._made[i] = self._make(i)
        return a

    def __getitem__(self, i):
        if isinstance(i, (int, np.integer)):
            return self._one(i)
        idx = range(*i.indices(self._n)) if isinstance(i, slice) else np.arange(self._n)[i]
        out = np.empty(len(idx), dtype=object)
        for q, j in enumerate(idx):
            out[q] = self._one(j)
        return out

    def __iter__(self):
        return (self._one(i) for i in range(self._n))

    def __array__(self, dtype=None, copy=None):
        return self[:]


class _Frame(list):
    """One history frame ``[[pos, vel, target, v_des] per agent inside ..., density]`` (simulations.py:579-589), built
    on first access: the agents' rows come from the device-resident trajectory record (row k = state before step k)
    and the density -- which the reference splats on every step although only draw_history('density') reads it --
    is computed when the LAST element is read."""

    def __init__(self, agents, density_fn):
        """agents: the rows, or a function that returns them (called on first access)"""
        super().__init__()
        self._agents_fn = agents if callable(agents) else (lambda: agents)
        self._density_fn = density_fn

    def _rows(self):
        if self._agents_fn is not None:
            fn, self._agents_fn = self._agents_fn, None
            list.extend(self, fn())
            list.append(self, None)

    def _fill(self):
        self._rows()
        if self._density_fn is not None:
            fn, self._density_fn = self._density_fn, None
            list.__setitem__(self, list.__len__(self) - 1, fn())

    def __len__(self):
        self._rows()
        return list.__len__(self)

    def __getitem__(self, i):
        self._rows()
        n = list.__len__(self)
        if (len(range(*i.indices(n))[-1:]) and range(*i.indices(n))[-1] == n - 1) if isinstance(i, slice) \
                else (i == -1 or i == n - 1):
            self._fill()
        return list.__getitem__(self, i)

    def __iter__(self):
        self._fill()
        return list.__iter__(self)

    def __repr__(self):
        self._fill()
        return list.__repr__(self)

    def __eq__(self, other):
        self._fill()
        return list.__eq__(self, other)


class simulation:

    TRACK_CHUNK = 64  # steps per block of the device-resident trajectory record

    def __init__(self, room, T, recompute=False, record=True, field_storage="phi", fused=1, lookahead=True,
                 rng=None, chunk_rows=0, band=False, shard_keys=False, config=None, density_stats=None, lines=None,
                 areas=None, voronoi=None, voronoi_maps=None, _ctx=None):
        """``room, T, recompute`` as in the reference (simulations.py:20).  Extras, all defaulting to reference
        behaviour: ``record`` (keep the per-step record behind ped.traj / ped.vels / history; it lives on the device and
        is read back on access), ``field_storage`` ('phi': the value-function samples, from which ``vx_opt`` /
        ``vy_opt`` are produced on access and which the sampler differentiates on the fly, bit-identical and half the
        memory; 'velocity': (vx, vy) slices stored like the reference), ``rng`` (a ``np.random.RandomState``; default = numpy's
        legacy global generator, which the reference uses), ``chunk_rows`` (fixes the HJB reduction order),
        ``band`` (True: this process is one rank of a row-decomposed run under torch.distributed -- it solves and
        stores only its band of rows of every HJB field, evaluates the field samples and wall forces of the agents
        in its band, and runs the (replicated, deterministic) sweep; every rank must use the same seed),
        ``shard_keys`` (True: the target sets -- one HJB field each, simulations.py:113-121 -- are dealt round-robin to the
        ranks of torch.distributed: a rank solves and stores only its keys' fields and evaluates the field samples / wall
        forces of the agents heading for them; merge and sweep as for ``band``), ``config`` (a dict of overrides of
        config.json, e.g. ``{"dt": 0.01, "hjb_params": {"g": -0.01}}``: nested ``hjb_params`` are merged key by key, a
        key config.json does not have raises KeyError; ``_config`` is the effective configuration), ``density_stats`` (True
        or dict(every=1, threshold=None): accumulate on the device, per grid node, the sum and the maximum of the density
        frames the reference stores in ``history`` (simulations.py:579-589) at the steps of run()'s loop whose simu_step
        is a multiple of ``every``, and with a threshold the number of frames above it; read them with
        ``density_stats()``; with ``velocity=True`` also the density-weighted sums of the agents' vx, vy and speed, and
        their means ``velocity`` and ``speed``.  Not available with ``band`` or ``shard_keys``), ``lines`` ({name: (x0, y0,
        x1, y1)} in metres, at most 64: count on the device, per step, the agents crossing each line to its left and to
        its right; read them with ``line_counts()``.  Not available with ``band`` or ``shard_keys``), ``areas`` ({name:
        [(x0, y0), (x1, y1), ...]} in metres, at most 64 simple polygons of 3 to 64 vertices, 1024 in all: measure on
        the device, at the start of every step, the pedestrians inside each polygon and the sums of their speeds and
        velocities; read them with ``area_stats()``.  Not available with ``band`` or ``shard_keys``), ``voronoi`` (True
        = dict(cutoff=1.0, edges=12), needs ``areas``: measure also, at the start of every step, each area's Voronoi
        density, speed and velocity and the fraction of it the cells cover (Steffen & Seyfried's method D; cells are
        bounded by the room rectangle and a polygon of ``edges`` vertices at ``cutoff`` metres from the agent, not by
        internal walls); ``area_stats()["voronoi"]`` returns them.  Not available with ``band`` or ``shard_keys``),
        ``voronoi_maps`` (True = dict(every=1, cutoff=1.0, edges=12): accumulate on the device, per grid node and over
        the frames of ``density_stats`` -- the steps of run()'s loop whose simu_step is a multiple of ``every`` -- the
        Voronoi density 1/|V| and the speed and velocity of the pedestrian whose Voronoi cell holds the node (cells as
        for ``voronoi``); read them with ``voronoi_maps()``.  Independent of ``density_stats``, ``areas`` and
        ``voronoi``.  Not available with ``band`` or ``shard_keys``)."""
        import torch
        dstats = density_stats_spec(density_stats, with_velocity=True)
        lspec = lines_spec(lines)
        aspec = areas_spec(areas)
        vspec = voronoi_spec(voronoi)
        mspec = voronoi_maps_spec(voronoi_maps)
        if mspec is not None and (band or shard_keys):
            raise ValueError("voronoi_maps is not available for row-decomposed (band=True) or key-sharded "
                             "(shard_keys=True) runs")
        if vspec is not None and (band or shard_keys):
            raise ValueError("voronoi is not available for row-decomposed (band=True) or key-sharded "
                             "(shard_keys=True) runs")
        if vspec is not None and aspec is None:
            raise ValueError("voronoi needs measurement areas (areas=...)")
        if aspec is not None and (band or shard_keys):
            raise ValueError("areas are not available for row-decomposed (band=True) or key-sharded "
                             "(shard_keys=True) runs")
        if dstats is not None and (band or shard_keys):
            raise ValueError("density_stats is not available for row-decomposed (band=True) or key-sharded "
                             "(shard_keys=True) runs")
        if lspec is not None and (band or shard_keys):
            raise ValueError("lines are not available for row-decomposed (band=True) or key-sharded "
                             "(shard_keys=True) runs")
        self._np_random = rng if rng is not None else np.random
        self.recompute = recompute
        var_config = _load_config()       # simulations.py:42
        if config is not None:
            var_config = _merge_config(var_config, config)
        var_room = _load_room(room)       # simulations.py:47
        self._config, self._room = var_config, var_room
        self.room_length = var_room['room_length']
        self.room_height = var_room['room_height']
        self.grid_step = var_config['grid_step']
        # (_ctx: a library context of the same room size and grid step to reuse -- ensembles recycle the contexts, and
        # with them the device / page-locked workspaces, of finished members)
        if _ctx is not None and (_ctx.room_length, _ctx.room_height, _ctx.dx) != (self.room_length, self.room_height,
                                                                                 self.grid_step):
            raise ValueError("_ctx was created for another room size / grid step")
        self._ctx = _ctx if _ctx is not None else _lib.Context(self.room_length, self.room_height, self.grid_step)
        self.Ny, self.Nx = self._ctx.Ny, self._ctx.Nx       # simulations.py:63-64
        self.dx = self.dy = self.grid_step
        self.sigma_convolution = var_config['sigma_convolution']
        self.pot = var_config['hjb_params']['wall_potential']
        self.lim = 10e-3
        self.T = T
        self.time = 0.
        self.simu_step = 0
        self.dt = var_config['dt']
        self.relaxation = var_config['relaxation']
        self.noise_intensity = var_config['hjb_params']['sigma']
        self.a_min = var_config['b_min']                    # simulations.py:88
        self.tau_a, self.b_min, self.b_max = var_config['tau_a'], var_config['b_min'], var_config['b_max']
        self.eta, self.eta_walls = var_config['eta'], var_config['eta_walls']
        self.repulsion_cutoff = var_config['repulsion_cutoff']
        self.v_max = var_config['v_max']
        self.recompute_step = var_config['recompute_frequency']
        self.history = {}
        self._record = record
        # host RNG draws of step k+1 overlap the GPU's step k (same stream as the reference, see _rng.py)
        self._rng = _rng.StepRandomness(lookahead, self._np_random)
        self._gcfm_prm = _lib.gcfm_params(var_config, self.room_length, self.room_height, self.Ny, self.Nx)
        self._band = None
        if band:
            from . import dist as _dist
            self._band = _dist.init_context(self._ctx)          # (own0, own1) of this rank
            self._gcfm_prm.own0, self._gcfm_prm.own1 = self._band
            if field_storage != "phi":
                raise ValueError("band=True stores the field as phi samples: pass field_storage='phi'")
        self._cuda_stream = None   # raw CUDA stream handle of this simulation's steps (None: torch's current stream)
        # run() / advance() execute blocks of steps inside one library call (oc_gcfm_run); OC_FAST_RUN=0 keeps the
        # step-by-step Python loop (same results)
        self._fast_run = lookahead and os.environ.get("OC_FAST_RUN", "1") != "0"
        self._key_shard = None
        if shard_keys:
            import torch.distributed as tdist
            from . import dist as _dist
            if band:
                raise ValueError("band and shard_keys are alternative decompositions")
            if tdist.is_available() and tdist.is_initialized() and tdist.get_world_size() > 1:
                _dist.init_comm(self._ctx)
                self._key_shard = (tdist.get_world_size(), tdist.get_rank())
                self._gcfm_prm.key_mod, self._gcfm_prm.key_rem = self._key_shard
        diag = float(np.hypot(self.room_length, self.room_height))
        if abs(self.pot) * 10e3 <= diag:
            raise NotImplementedError("wall search assumes |wall_potential|*10e3 exceeds the room diagonal")

        # crowd initialisation (simulations.py:104-160), same RNG consumption
        N = 0
        self.targets = {}
        self.Vs = {}
        self.V = np.zeros((self.Ny, self.Nx)) + 1
        self.place_ped = np.zeros((self.Ny, self.Nx))
        r_in = 0.2
        xs_all, ys_all, vdes_all, key_all, agents = [], [], [], [], []
        X1, Y1 = self._ctx.X, self._ctx.Y
        box_count = {}
        for box_name in var_room['initial_boxes']:
            box = var_room['initial_boxes'][box_name]
            targets = box[5:]
            key = ' or '.join(targets)
            if key not in self.targets:
                # The reference rebuilds the potential and the optimals object for every box and overwrites
                # the dict entries of a repeated key with identical content (simulations.py:116-120,
                # SURVEY App. C #12); building them once per key gives the same objects and the same RNG stream.
                V = self.create_potential(var_room, targets)
                self.Vs[key] = V
                owned = self._key_shard is None or len(self.targets) % self._key_shard[0] == self._key_shard[1]
                self.targets[key] = optimals.optimals(var_room, V, T, key, _ctx=self._ctx, _config=var_config,
                                                      field_storage=field_storage, fused=fused, band=self._band,
                                                      owned=owned)
                self.targets[key]._prm.chunk_rows = int(chunk_rows)
            box_count[key] = box_count.get(key, 0) + 1
            xs, ys, v_des_all = _crowd.place_box(box, X1, Y1, self.place_ped, r_in, self._np_random)
            loc_N = len(xs)
            N += loc_N
            kid = list(self.targets).index(key)
            agents.append((N - loc_N, key, targets))        # (first agent of the box, its key, its target names)
            xs_all.append(xs); ys_all.append(ys); vdes_all.append(v_des_all)
            key_all.append(np.full(loc_N, kid, dtype=np.int32))
        for key, cnt in box_count.items():
            # simulations.py:121 adds the key's potential once per box; the values are small integers
            # (-100, 0, 1), so cnt * V is exactly the repeated sum
            self.V += cnt * self.Vs[key]
        self.V[self.V > np.min(self.V)] = 0                 # simulations.py:157
        self.N = N
        self.inside = self.N

        cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dtype=dt)
        x0, y0 = cat(xs_all, np.float64), cat(ys_all, np.float64)
        self._h_vdes = cat(vdes_all, np.float64)
        box_first = [b[0] for b in agents]

        def make_agent(i, boxes=agents, x0=x0, y0=y0):
            first, key, tg = boxes[int(np.searchsorted(box_first, i, side="right")) - 1]
            a = pedestrians.ped(None, None, self.grid_step, self.Vs[key], key, var_room['targets'], tg,
                                x0[i], y0[i], 0, 0, self.room_length, self.room_height, self._h_vdes[i],
                                self.a_min, self.tau_a, self.b_min, self.b_max, self.eta, self.eta_walls)
            a._bind(self, i)
            return a
        self.agents = _Agents(N, make_agent)                # simulations.py:142-151, built on access
        self._h_key = cat(key_all, np.int32)
        self._h_status = np.ones(N, dtype=np.uint8)
        self._h_time0 = np.zeros(N)
        ctx = self._ctx
        self._state = dict(x=ctx.to_device(x0), y=ctx.to_device(y0), vx=ctx.to_device(np.zeros(N)),
                           vy=ctx.to_device(np.zeros(N)), time=ctx.to_device(np.zeros(N)),
                           status=ctx.to_device(self._h_status.copy()))
        self._d_vdes = ctx.to_device(self._h_vdes)
        self._d_key = ctx.to_device(self._h_key)
        self._d_Vglobal = ctx.to_device(self.V)
        # density statistics of the run's frames (device accumulators, written by oc_density_accum / oc_gcfm_run_acc)
        self._dstats = None if dstats is None else _lib.DensityStats(ctx, self._d_Vglobal, self.sigma_convolution, *dstats)
        # counts through measurement lines (written after every step by oc_lines_count* / oc_gcfm_run_flow), one row per
        # step of a run that lasts until T, grown on the host when the steps go past that
        self._lines = None if lspec is None else _lib.LineCounts(ctx, *lspec, self._state,
                                                                 len(density_frame_steps(T, self.dt, 1)))
        # measurement areas (written before every step by oc_areas_measure* / oc_gcfm_run_obs), rows sized as the lines'
        self._areas = None if aspec is None else _lib.AreaStats(ctx, *aspec, N, len(density_frame_steps(T, self.dt, 1)))
        # their Voronoi measures (oc_voronoi_measure* / oc_gcfm_run_observed, right after the areas), rows sized alike
        self._voronoi = None if vspec is None else _lib.VoronoiStats(ctx, aspec[1], aspec[2], *voronoi_triangles(aspec),
                                                                     *vspec, N, self._areas.count.shape[0])
        # Voronoi maps of the run's frames (oc_vormap_accum* / oc_gcfm_run_observed_maps, next to the density frame)
        self._vmaps = None if mspec is None else _lib.VoronoiMaps(ctx, self._d_Vglobal, mspec[1], mspec[2], mspec[0], N)
        # per-step record of (x, y, vx, vy); row k = state after k steps (ped.traj / ped.vels / history views).  It
        # lives on the DEVICE in blocks of TRACK_CHUNK steps, written by one small kernel per step (oc_state_pack), and
        # is read back -- once per row -- only when somebody looks at it
        self._row0 = np.column_stack([x0, y0, np.zeros(N), np.zeros(N)])
        self._d_track = []                                  # device blocks (TRACK_CHUNK, N, 4)
        self._n_rows = 1                                    # rows recorded so far (row 0 = initial state)
        self._h_rows = [self._row0]                         # host copies of rows 0 .. len-1 (filled on demand)
        self._exit_step = np.full(N, -1, dtype=np.int64)   # step index at which the agent left
        self._exit_order = []                               # agent ids in exit order over the whole run
        self._h_now_cache = self._row0
        self._h_timev_cache = np.zeros(N)
        self._host_dirty = False                            # device state is ahead of _h_now_cache / _h_timev_cache
        print('ABM simulation room created!')               # simulations.py:162

    # ---- helpers -------------------------------------------------------------------------------------
    @property
    def X_opt(self):
        return np.meshgrid(self._ctx.X, self._ctx.Y)[0]

    @property
    def Y_opt(self):
        return np.meshgrid(self._ctx.X, self._ctx.Y)[1]

    def _sync_host(self):
        st = self._state
        import torch
        packed = torch.stack([st["x"], st["y"], st["vx"], st["vy"], st["time"]], dim=1).cpu().numpy()
        self._h_now_cache = packed[:, :4]
        self._h_timev_cache = packed[:, 4].copy()
        self._host_dirty = False

    @property
    def _h_now(self):
        """(N,4) host copy of the current x, y, vx, vy (refreshed from the device when a step has run since)"""
        if self._host_dirty:
            self._sync_host()
        return self._h_now_cache

    @property
    def _h_timev(self):
        if self._host_dirty:
            self._sync_host()
        return self._h_timev_cache

    @property
    def _track(self):
        """host view of the whole record: list of (N,4) rows, row k = state after k steps"""
        return self._rows_upto(self._n_rows - 1)

    def _record_row(self):
        """append the current device state to the device-resident record"""
        import torch
        k = self._n_rows - 1                                # rows 1.. live in the blocks: row r -> block (r-1)//C
        blk, off = divmod(k, self.TRACK_CHUNK)
        if blk == len(self._d_track):
            self._d_track.append(torch.empty((self.TRACK_CHUNK, max(self.N, 1), 4), dtype=torch.float64,
                                             device=self._ctx.torch_device))
        if self.N:
            self._ctx.state_pack(self._state, self._d_track[blk][off], stream=self._cuda_stream)
        self._n_rows += 1

    def _rows_upto(self, last):
        """host copies of rows 0..last (one device read per block touched, cached)"""
        have = len(self._h_rows)
        while have <= last:
            blk, off = divmod(have - 1, self.TRACK_CHUNK)
            n = min(self.TRACK_CHUNK - off, self._n_rows - have)
            part = self._d_track[blk][off:off + n].cpu().numpy()
            self._h_rows.extend(part[q] for q in range(n))
            have += n
        return self._h_rows

    def _agent_now(self, i):
        r = self._h_now[i]
        return np.array(r[:2], dtype=float), np.array(r[2:], dtype=float)

    def _agent_time(self, i):
        t = self._h_timev[i]
        return 0 if t == 0 and self.simu_step == 0 else float(t)

    def _agent_track(self, i, which):
        """list of per-step positions (which=0) or velocities (which=1) up to the agent's exit (ped.traj/vels)."""
        if not self._record and self._n_rows == 1 and self.simu_step > 0:
            raise RuntimeError("this simulation was created with record=False: no trajectories were kept")
        last = self._exit_step[i] + 1 if self._exit_step[i] >= 0 else self._n_rows - 1
        last = min(last, self._n_rows - 1)
        rows = self._rows_upto(last)
        sl = slice(0, 2) if which == 0 else slice(2, 4)
        return [np.array(rows[k][i, sl], dtype=float) for k in range(last + 1)]

    def _set_status(self, i, v):
        self._h_status[i] = 1 if v else 0
        self._state["status"][i] = int(self._h_status[i])

    def _keys(self):
        """marshalled per-target-set descriptors of oc_gcfm_step, rebuilt only when a field changed (a solve replaces
        nt_opt and possibly the field tensors)"""
        sig = tuple((o.nt_opt, id(o.d_phi), id(o.d_vx), id(o.d_V)) for o in self.targets.values())
        if getattr(self, "_keys_sig", None) != sig:
            self._keys_cache = _lib.Context.make_keys([opt.field_key(self._doors[key]) for key, opt in self.targets.items()])
            self._keys_sig = sig
        return self._keys_cache

    @property
    def _doors(self):
        if not hasattr(self, "_doors_cache"):
            self._doors_cache = {}
            for box in self._room['initial_boxes'].values():
                tg = box[5:]
                self._doors_cache[' or '.join(tg)] = np.array([self._room['targets'][t] for t in tg],
                                                              dtype=np.float64).reshape(-1, 4)
        return self._doors_cache

    # ---- simulations.py:252-342 ----------------------------------------------------------------------
    def step(self, dt, verbose=False):
        """One GCFM step for every agent still inside, with the reference's sequential sweep semantics."""
        self._step_finish(self._step_launch(dt), verbose)

    def _step_launch(self, dt):
        """first half of step(): draw this step's randomness and enqueue the sweep on the current CUDA stream
        (ensembles launch every member before finishing any, so the members' kernels overlap)"""
        if dt != self.dt:
            prm = _lib.gcfm_params(dict(self._config, dt=dt), self.room_length, self.room_height, self.Ny, self.Nx)
            prm.own0, prm.own1 = self._gcfm_prm.own0, self._gcfm_prm.own1
            prm.key_mod, prm.key_rem = self._gcfm_prm.key_mod, self._gcfm_prm.key_rem
        else:
            prm = self._gcfm_prm
        pending = None
        self._measure_areas()
        if self.N > 0:
            n_active = int(self._h_status.sum())
            # np.random.choice(np.arange(N), N, replace=False) (simulations.py:271) and one normal pair per active
            # agent in sweep order == N calls of normal(size=2) (simulations.py:303)
            perm, noise = self._rng.draw(self.N, n_active)
            # next step's draws on the helper thread, while this thread enqueues the step and the GPU sweeps
            self._rng.lookahead(self.N, n_active)
            pending = self._ctx.gcfm_step_launch(prm, self._state, self._d_vdes, self._d_key, self._keys(), perm,
                                                 noise, self.simu_step, stream=self._cuda_stream)
        return dt, pending

    def advance(self, n_steps, verbose=False):
        """Up to n_steps iterations of run()'s loop body -- history frame, step -- stopping when nobody is inside; returns
        the number of steps done.  Plain single-GPU simulations on the legacy MT19937 stream run them inside ONE library
        call (oc_gcfm_run: randomness drawn in C, the next step's draws overlapped with the GPU, no return to Python
        between steps); results, RNG stream, history frames and records are those of the step-by-step loop."""
        n_steps = int(n_steps)
        fast = (n_steps > 1 and self.N > 0 and not verbose and self._record and not self._band and self._key_shard is None
                and self._fast_run)
        st = self._rng.rng.get_state() if fast else None
        if not fast or st[0] != "MT19937":
            done = 0
            while done < n_steps and self.inside > 0:
                self.write_history(self.time)
                self._density_frame()
                self.step(self.dt, verbose=verbose)
                done += 1
            return done
        import torch
        self._rng._spec = None   # (a look-ahead drawn for the step-by-step path is simply not used)
        # rows of the device-resident record for the steps to come
        rows = []
        for k in range(self._n_rows - 1, self._n_rows - 1 + n_steps):
            blk, off = divmod(k, self.TRACK_CHUNK)
            while blk >= len(self._d_track):
                self._d_track.append(torch.empty((self.TRACK_CHUNK, max(self.N, 1), 4), dtype=torch.float64,
                                                 device=self._ctx.torch_device))
            rows.append(self._d_track[blk][off])
        n_active = int(self._h_status.sum())
        for acc in (self._lines, self._areas, self._voronoi):
            if acc is not None:
                acc.ensure(self.simu_step + n_steps)
        res = self._ctx.gcfm_run(self._gcfm_prm, self._state, self._d_vdes, self._d_key, self._keys(), st, n_steps,
                                 self.simu_step, n_active, rows=rows, stream=self._cuda_stream, density=self._dstats,
                                 lines=self._lines, areas=self._areas, voronoi=self._voronoi, maps=self._vmaps)
        self._rng.rng.set_state(res["rng_state"])
        self.last_run_stats = dict(steps=res["steps"], device_ms=res["device_ms"], pairs=res["pairs"])
        ex, exs = res["exits"], res["exit_step"]
        e = 0
        for k in range(res["steps"]):
            self.write_history(self.time)          # lazy frame: a view of record row simu_step
            while e < len(ex) and exs[e] == k:
                a = int(ex[e])
                self._h_status[a] = 0
                self._exit_step[a] = self.simu_step
                self._exit_order.append(a)
                self.inside += -1
                e += 1
            self._n_rows += 1
            self.time += self.dt
            self.simu_step += 1
        self._host_dirty = True
        if res["rc"] == _lib.OC_ERR_SAMPLER_RANGE:
            raise IndexError("agent position outside the velocity field's index range "
                             "(numpy raises IndexError in the reference's sampler too: optimals.py:247)")
        return res["steps"]

    def _density_frame(self):
        """add this iteration's frame to the density statistics and the Voronoi maps when they are on and it is due
        (before the step)"""
        st = self._state
        if self._dstats is not None and self._dstats.due(self.simu_step):
            self._ctx.density_accum(self._dstats, st["x"], st["y"], st["status"], stream=self._cuda_stream, vx=st["vx"],
                                    vy=st["vy"])
        if self._vmaps is not None and self._vmaps.due(self.simu_step):
            self._ctx.vormap_accum(self._vmaps, st, stream=self._cuda_stream)

    def voronoi_maps(self):
        """the Voronoi maps of the frames taken so far (``voronoi_maps=`` of the constructor): dict(cutoff, edges, frames,
        density_sum, density_max, covered, speed_sum, vx_sum, vy_sum, density, speed, velocity) -- (Ny, Nx) numpy
        arrays (velocity (Ny, Nx, 2)); ``density`` = density_sum / frames is None before the first frame, ``speed`` and
        ``velocity`` are means over the covered frames, NaN where a node was never covered (include/optimal_crowds.h,
        oc_vormap_acc)"""
        if self._vmaps is None:
            raise RuntimeError("this simulation was created without voronoi_maps")
        import torch
        torch.cuda.synchronize(self._ctx.torch_device)
        return self._vmaps.result()

    def density_stats(self):
        """the density statistics of the frames taken so far (``density_stats=`` of the constructor): dict(frames, sum,
        max, above, mean) -- (Ny, Nx) numpy arrays; ``above`` (int32 counts of frames with density > threshold) is None
        without a threshold, ``mean`` = sum / frames is None before the first frame"""
        if self._dstats is None:
            raise RuntimeError("this simulation was created without density_stats")
        if self._cuda_stream is not None:
            import torch
            torch.cuda.synchronize(self._ctx.torch_device)
        return self._dstats.result()

    def _count_lines(self):
        """count this step's crossings of the measurement lines (after the step is final, before simu_step advances)"""
        if self._lines is not None:
            self._lines.ensure(self.simu_step + 1)
            self._ctx.lines_count(self._lines, self._state, self.simu_step, stream=self._cuda_stream)

    def line_counts(self):
        """the crossings of the measurement lines (``lines=`` of the constructor) by the steps taken so far:
        dict(names, to_left, to_right) -- int32 (simu_step, n_lines) arrays, row k = the step with simu_step k"""
        if self._lines is None:
            raise RuntimeError("this simulation was created without lines")
        import torch
        torch.cuda.synchronize(self._ctx.torch_device)
        return self._lines.result(self.simu_step)

    def _measure_areas(self):
        """measure the state this step starts from into row simu_step of the measurement areas (before the step's
        randomness; a crowd without agents keeps the zero row), and its Voronoi measures when they are on"""
        if self._areas is not None:
            self._areas.ensure(self.simu_step + 1)
            if self.N > 0:
                self._ctx.areas_measure(self._areas, self._state, self.simu_step, stream=self._cuda_stream)
        if self._voronoi is not None:
            self._voronoi.ensure(self.simu_step + 1)
            if self.N > 0:
                self._ctx.voronoi_measure(self._voronoi, self._state, self.simu_step, stream=self._cuda_stream)

    def area_stats(self):
        """the measurement areas (``areas=`` of the constructor) of the steps taken so far: dict(names, area, count,
        speed_sum, vx_sum, vy_sum, density, speed, velocity) -- (simu_step, n_areas) arrays (velocity: (simu_step,
        n_areas, 2)), row k = the state the step with simu_step k started from; ``speed`` and ``velocity`` are NaN where
        nobody is inside.  With ``voronoi`` also "voronoi": dict(cutoff, edges, density, speed, covered (simu_step,
        n_areas) and velocity (simu_step, n_areas, 2)): per area sum(w/|V|) / area, sum(w*speed) / area, sum(w*(vx, vy))
        / area and sum(w) / area over the agents' Voronoi cells V, w the part of V inside the area
        (include/optimal_crowds.h, oc_voronoi_acc)"""
        if self._areas is None:
            raise RuntimeError("this simulation was created without areas")
        import torch
        torch.cuda.synchronize(self._ctx.torch_device)
        out = self._areas.result(self.simu_step)
        if self._voronoi is not None:
            out["voronoi"] = self._voronoi.result(self.simu_step)
        return out

    def _step_finish(self, launched, verbose=False):
        dt, pending = launched
        if pending is not None:
            # ("batched", exits, rc): the step ran inside a batched launch of an ensemble wave and has finished already
            if pending[0] == "batched":
                exits, rc = pending[1:]
            else:
                exits, rc = self._ctx.gcfm_step_finish(pending)
                self._count_lines()
            if rc == _lib.OC_ERR_SAMPLER_RANGE:
                raise IndexError("agent position outside the velocity field's index range "
                                 "(numpy raises IndexError in the reference's sampler too: optimals.py:247)")
            for a in exits:
                self._h_status[a] = 0
                self._exit_step[a] = self.simu_step
                self._exit_order.append(int(a))
            self.inside += -len(exits)
            self._host_dirty = True
            if self._record:
                self._record_row()
        self.time += dt
        self.simu_step += 1
        if verbose:
            print('t = {:.2f}s exit = {}/{}'.format(self.time, self.N - self.inside, self.N) + 10 * ' ', end='\n')

    # ---- simulations.py:344-399 ----------------------------------------------------------------------
    def evac_times(self, draw=False):
        if self.inside > 0:
            raise ValueError('There are still people inside!')
        times = np.array(self._h_timev, dtype=float)
        if draw:
            import matplotlib.pyplot as plt
            plt.figure(figsize=(self.room_length, self.room_height))
            xs, ys = self.initial_positions()
            plt.scatter(xs, ys, c=times)
            plt.xlim(0, self.room_length)
            plt.ylim(0, self.room_height)
            plt.title('Evacuation time')
            plt.colorbar()
        else:
            return times

    def initial_positions(self):
        return np.array(self._row0[:, 0], dtype=float), np.array(self._row0[:, 1], dtype=float)

    # ---- simulations.py:401-451 ----------------------------------------------------------------------
    def run(self, verbose=False, draw=False, mode='scatter'):
        print(f"Computing trajectories at time {self.time}")
        self._solve_all()
        while (self.inside > 0) & (self.time < self.T):
            if self.recompute and (self.simu_step % self.recompute_step == 0) and self.simu_step > 0:
                print(f"Computing trajectories at time {self.time}")
                self._solve_all()
            # the iterations up to the next re-solve / drawing / the end of the horizon run as one block (advance)
            n, t = 0, self.time
            while t < self.T:
                t += self.dt
                n += 1
                k = self.simu_step + n
                if (self.recompute and k % self.recompute_step == 0) or (draw and k % 10 == 0):
                    break
            self.advance(n, verbose=verbose)
            if draw and (self.simu_step % 10) == 0:
                import matplotlib.pyplot as plt
                self.draw(mode)
                plt.show()
        if self.inside == 0:
            print('Evacuation complete in {:.2f}s!'.format(self.time))
        else:
            print('Evacuation failed!' + 10 * ' ')

    def _solve_all(self):
        # simulations.py:424-425 / :434-435: density * (simu_step > 0); the product with False is all zeros,
        # so at step 0 the splat is skipped and no density is passed (identical input to the solver)
        d_m = self._density_device(self.sigma_convolution) if self.simu_step > 0 else None
        for target in self.targets:
            self.targets[target].compute_optimal_velocity(self.time, d_m)

    # ---- simulations.py:453-487 ----------------------------------------------------------------------
    def _density_device(self, sigma):
        st = self._state
        return self._ctx.density(st["x"], st["y"], st["status"], sigma, self._d_Vglobal)

    def gaussian_density(self, sigma):
        return self._density_device(sigma).cpu().numpy()

    # ---- simulations.py:516-576 ----------------------------------------------------------------------
    def create_potential(self, var_room, targets):
        tg = [var_room['targets'][t] for t in targets]
        V = self._ctx.rasterise(list(var_room['walls'].values()), list(var_room['holes'].values()),
                                list(var_room['cylinders'].values()), tg, remap=False)
        return V.cpu().numpy()

    # ---- simulations.py:579-589 ----------------------------------------------------------------------
    def write_history(self, time):
        """history[time] = [[pos, vel, target, v_des] per agent inside, ..., density] (simulations.py:579-589).
        The frame is a view of the device-resident record: row ``simu_step`` holds the state this frame describes and
        the agents inside are those that have not left before this step; nothing is copied or splatted until the frame
        is read (the reference splats the density, O(N Nx Ny) exps, on every step although only
        draw_history('density') reads it).  With ``record=False`` no record exists: the frame is built right away from
        the current state (one device read), as the reference does."""
        keys = list(self.targets)
        k = self.simu_step

        def rows_of(now, act):
            return [[np.array(now[i, :2], dtype=float), np.array(now[i, 2:], dtype=float), keys[self._h_key[i]],
                     self._h_vdes[i]] for i in act]

        if self._record and k < self._n_rows:
            active = lambda: np.nonzero((self._exit_step < 0) | (self._exit_step >= k))[0]
            agents_fn = lambda: rows_of(self._rows_upto(k)[k], active())
            dens_fn = lambda: self._density_of(np.array(self._rows_upto(k)[k][active(), :2], dtype=np.float64),
                                               self.sigma_convolution)
            self.history[time] = _Frame(agents_fn, dens_fn)
        else:
            now = np.array(self._h_now)
            act = np.nonzero(self._h_status)[0]
            xy = np.array(now[act, :2], dtype=np.float64)
            self.history[time] = _Frame(lambda: rows_of(now, act), lambda: self._density_of(xy, self.sigma_convolution))

    def _density_of(self, xy, sigma):
        """density of the crowd at positions xy (n,2), all inside: same kernel, same summation order (agents inside,
        in index order) as gaussian_density at the time the positions were recorded"""
        import torch
        n = len(xy)
        x = self._ctx.to_device(np.ascontiguousarray(xy[:, 0])) if n else None
        y = self._ctx.to_device(np.ascontiguousarray(xy[:, 1])) if n else None
        st = torch.ones(n, dtype=torch.uint8, device=self._ctx.torch_device) if n else None
        return self._ctx.density(x, y, st, sigma, self._d_Vglobal).cpu().numpy()

    # ---- plotting (visualisation only; needs matplotlib / seaborn) ---------------------------------------
    def _ellipse_axes(self, vel, v_des):
        speed = np.linalg.norm(vel)
        a = self.a_min + self.tau_a * speed
        b = self.b_max - (self.b_max - self.b_min) * np.minimum(speed / v_des, 1)
        return a, b

    def _draw_frame(self, frame, mode, title):
        import matplotlib.pyplot as plt
        from matplotlib.patches import Ellipse
        import seaborn as sns
        keys = list(self.targets)
        colors = sns.color_palette(n_colors=len(keys))
        fig = plt.figure(figsize=(self.room_length, self.room_height))
        ax = plt.gca()
        if mode == 'density':
            plt.imshow(np.flip(frame[-1], axis=0), extent=[0, self.room_length, 0, self.room_height])
        else:
            plt.imshow(np.flip(self.V, axis=0), extent=[0, self.room_length, 0, self.room_height])
            for pos, vel, target, v_des in frame[:-1]:
                c = colors[keys.index(target)]
                if mode == 'arrows':
                    plt.quiver(pos[0], pos[1], vel[0], vel[1], color=c)
                else:
                    a, b = self._ellipse_axes(vel, v_des)
                    ang = np.degrees(np.arctan2(vel[1], vel[0]))
                    ax.add_patch(Ellipse((pos[0], pos[1]), 2 * a, 2 * b, angle=ang, color=c))
        plt.xlim([0, self.room_length])
        plt.ylim([0, self.room_height])
        plt.title(title)
        return fig

    def _current_frame(self):
        now, keys = self._h_now, list(self.targets)
        frame = [[np.array(now[i, :2]), np.array(now[i, 2:]), keys[self._h_key[i]], self._h_vdes[i]]
                 for i in np.nonzero(self._h_status)[0]]
        frame.append(self.gaussian_density(self.sigma_convolution))
        return frame

    def draw(self, mode='scatter'):
        """simulations.py:164-250"""
        import matplotlib.pyplot as plt
        self._draw_frame(self._current_frame(), mode,
                         't = {:.2f}s exit = {}/{}'.format(self.time, self.N - self.inside, self.N))
        plt.show()

    def draw_history(self, mode='scatter'):
        """simulations.py:591-703: every 10th recorded frame, then the current state."""
        import matplotlib.pyplot as plt
        times = list(self.history.keys())
        for j, t in enumerate(times):
            if j % 10 == 0 or j == len(times) - 1:
                self._draw_frame(self.history[t], mode, 't = {:.2f}s'.format(t))
                plt.show()
        self.draw(mode)

    def draw_final_trajectories(self):
        """simulations.py:489-514"""
        import matplotlib.pyplot as plt
        from matplotlib.patches import Patch
        import seaborn as sns
        keys = list(self.targets)
        colors = sns.color_palette(n_colors=len(keys))
        plt.figure(figsize=(self.room_length, self.room_height))
        for i in range(self.N):
            traj = np.array(self.agents[i].traj, dtype=float)
            plt.plot(traj[:, 0], traj[:, 1], color=colors[self._h_key[i]])
        plt.imshow(np.flip(self.V, axis=0), extent=[0, self.room_length, 0, self.room_height])
        plt.xlim([0, self.room_length])
        plt.ylim([0, self.room_height])
        plt.title('{}/{} pedestrians evacuated in {:.2f}s'.format(self.N - self.inside, self.N, self.time))
        plt.legend(handles=[Patch(color=colors[i], label=keys[i]) for i in range(len(keys))], loc='upper right',
                   frameon=False)
        plt.show()
