"""Ensembles of independent rooms / seeds (BASELINE.json configs[4]; SURVEY.md section 8e).

With the reference an ensemble is a Python loop -- ``np.random.seed(s); simulations.simulation(room, T).run()`` once
per member.  Members never interact, so here they are sharded one batch per GPU (member i belongs to rank
i % world, no data-path collective) and, inside a batch, run concurrently on one GPU:

  * every member is an ordinary ``simulations.simulation`` whose randomness comes from its own
    ``np.random.RandomState(seed)`` -- the very stream ``np.random.seed(seed)`` gives the reference, so member i
    reproduces the stand-alone run with that seed bit for bit (tests/test_gpu_ensemble.py);
  * the HJB fields of all members of a wave -- every target set of every member -- are solved by ONE
    ``oc_hjb_solve_grids`` call: one RK45 controller and one CUDA stream per field, the step kernels of fields of
    every grid shape sharing batched launches;
  * the GCFM steps of the members advance in lock-step: every member's sweep is launched on its own stream
    (``oc_gcfm_step_launch``) before any is finished (``oc_gcfm_step_finish``), so the host's per-step work (RNG
    draws, exit bookkeeping) of one member overlaps the other members' kernels;
  * members are processed in waves sized to the GPU's memory (a 512^2 room with T = 20 s holds 2.1 GB of field
    samples), and only the per-member results are kept;
  * ``configs``: every member may bring its own overrides of config.json (model parameters, ``dt``, re-solve
    frequency, ...; one grid step for all).  Its HJB solves then run with its own sigma, mu, g and horizon inside the
    same batched call, its re-solves happen at its own steps, and it still equals the stand-alone
    ``simulation(..., config=...)`` run bit for bit (tests/test_gpu_ensemble_params.py);
  * members may have different rooms: different grid shapes and numbers of target sets (one grid step for all).
    Every member still equals its stand-alone run bit for bit (tests/test_gpu_ensemble_shapes.py);
  * ``density_stats``: every member accumulates the sum, maximum and above-threshold count of its density frames on the
    device (one batched ``oc_density_accum_multi`` launch per step for the due members of a wave) and hands them back
    in ``results[i]["density"]`` -- no frames, trajectories or members are kept (tests/test_gpu_density_stats.py);
    with ``velocity=True`` also the frames' density-weighted velocity and speed maps;
  * ``lines``: every member counts, per step, the agents crossing each measurement line in each direction on the device
    (one batched ``oc_lines_count_multi`` launch per step for a wave) and hands them back in ``results[i]["lines"]``
    (tests/test_gpu_flow_stats.py);
  * ``areas``: every member measures, at the start of every step, the pedestrians inside each measurement area and the
    sums of their speeds and velocities on the device (one batched ``oc_areas_measure_multi`` call per step for a wave)
    and hands them back in ``results[i]["areas"]`` (tests/test_gpu_areas.py);
  * ``voronoi``: with ``areas``, every member also measures each area's Voronoi density, speed, velocity and covered
    fraction (one batched ``oc_voronoi_measure_multi`` call per step for a wave, next to the areas' call), handed back in
    ``results[i]["areas"]["voronoi"]`` (tests/test_gpu_voronoi.py);
  * ``voronoi_maps``: every member accumulates Voronoi density, speed and velocity maps of its density frames on the
    device (one batched ``oc_vormap_accum_multi`` call per step for the members due), handed back in
    ``results[i]["voronoi_maps"]`` (tests/test_gpu_voronoi_maps.py).
"""
from __future__ import annotations

import contextlib
import copy
import os
import io

import numpy as np

from . import _lib, optimals, simulations


def shard(n_members: int, rank: int, world: int):
    """member indices owned by `rank`: round-robin, so that every rank gets members of every cost class"""
    if not (0 <= rank < world):
        raise ValueError("rank outside the world")
    return list(range(rank, n_members, world))


def field_bytes_per_member(Ny: int, Nx: int, T: float, dt: float, n_keys: int = 1, field_storage: str = "phi") -> int:
    """device bytes one member holds: field samples (optimals.py:80-81 sizes them by round(T/dt)) + solver workspace
    (the fields of all target sets are solved in one call)"""
    nt = round(T / dt)
    n = Ny * Nx
    field = nt * n * 8 if field_storage == "phi" else 2 * max(nt - 1, 0) * (Ny - 2) * (Nx - 2) * 8
    return n_keys * (field + 2 * n * 8 + 6 * n * 8)


_SOLVER_CTX = {}   # device -> Context owning the batched-solve workspace
_CTX_POOL = {}     # (device, room size, grid step) -> library contexts of finished members, ready for reuse


def _ctx_key(room_length, room_height, step):
    import torch
    return (torch.cuda.current_device(), float(room_length), float(room_height), float(step))


def plan_waves(members, bytes_per_member, budget_bytes: int, max_wave: int = 256):
    """split the member list, in order, into waves that fit `budget_bytes` of device memory and hold at most `max_wave`
    members; a member that does not fit on its own gets a wave of its own.  bytes_per_member: one count for all
    members, or one count per member"""
    if isinstance(bytes_per_member, (int, np.integer)):
        bytes_per_member = [bytes_per_member] * len(members)
    if len(bytes_per_member) != len(members):
        raise ValueError("one byte count per member expected")
    waves, cur, used = [], [], 0
    for m, b in zip(members, bytes_per_member):
        b = max(int(b), 1)
        if cur and (len(cur) == max_wave or used + b > budget_bytes):
            waves.append(cur)
            cur, used = [], 0
        cur.append(m)
        used += b
    if cur:
        waves.append(cur)
    return waves


def gather_results(local: dict, group=None) -> dict:
    """merge the per-rank {member index: result} dicts on every rank (the only exchange of an ensemble run)"""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return dict(local)
    parts = [None] * dist.get_world_size(group)
    dist.all_gather_object(parts, local, group=group)
    merged = {}
    for p in parts:
        merged.update(p)
    return dict(sorted(merged.items()))


class ensemble:
    """``ensemble(room, T, seeds)``: one member per seed of the same room; ``ensemble([room0, room1, ...], T, seeds)``:
    one room per member (rooms of any size and number of target sets).  ``run()`` returns {member index: result} with
    ``evac_time`` (simulation time when the run stopped), ``steps``, ``inside`` (agents left inside: 0 = evacuation
    complete), ``exit_order`` (agent ids in exit order), ``exit_step`` (per agent, -1 = still inside),
    ``times`` (per-agent clocks, as evac_times() returns them), ``final`` (N,4: x, y, vx, vy) and ``hjb`` (solver
    statistics per target set) and ``config`` (the member's effective configuration).

    ``density_stats``: None, True or dict(every=1, threshold=None, velocity=False) for every member, as ``simulation(...,
    density_stats=...)`` takes it (each member with its own ``sigma_convolution``); ``results[i]["density"]`` is then the
    member's ``density_stats()`` dict.

    ``lines``: None or {name: (x0, y0, x1, y1)} in metres (at most 64), the same measurement lines for every member, as
    ``simulation(..., lines=...)`` takes them; ``results[i]["lines"]`` is then the member's ``line_counts()`` dict.

    ``areas``: None or {name: [(x0, y0), (x1, y1), ...]} in metres, the same measurement areas for every member, as
    ``simulation(..., areas=...)`` takes them; ``results[i]["areas"]`` is then the member's ``area_stats()`` dict.

    ``voronoi``: None, True or dict(cutoff=1.0, edges=12), as ``simulation(..., voronoi=...)`` takes it (needs ``areas``);
    ``results[i]["areas"]["voronoi"]`` then holds the member's Voronoi measures.

    ``voronoi_maps``: None, True or dict(every=1, cutoff=1.0, edges=12), as ``simulation(..., voronoi_maps=...)`` takes
    it; ``results[i]["voronoi_maps"]`` is then the member's ``voronoi_maps()`` dict.

    ``configs``: None (every member runs config.json) or one dict of overrides per member, merged onto config.json as
    ``simulation(..., config=...)`` merges them (unknown keys raise KeyError).  All members must share ``grid_step``;
    their rooms may differ in size and number of target sets.

    ``chunk_rows``: 0 (every room chunked as if it were alone: members are bit-identical to stand-alone runs with
    default settings), n > 0 (fixed) or "wave" (planned per grid shape for the number of members of that shape in the
    solve; ``results[i]["chunk_rows"]`` is the value member i was solved with, and ``chunk_rows_used`` the value of a
    single-shape ensemble)."""

    def __init__(self, rooms, T, seeds, recompute=False, field_storage="phi", chunk_rows=0, rank=0, world=1,
                 memory_budget=None, max_wave=256, record=False, verbose=False, batched_steps=True, configs=None,
                 density_stats=None, lines=None, areas=None, voronoi=None, voronoi_maps=None):
        self.chunk_plan_for_wave = chunk_rows == "wave"
        self.T, self.recompute, self.field_storage = T, recompute, field_storage
        self.chunk_rows = 0 if self.chunk_plan_for_wave else int(chunk_rows)
        self.seeds = list(seeds)
        if isinstance(rooms, (list, tuple)):
            if len(rooms) != len(self.seeds):
                raise ValueError("one seed per room expected")
            self.rooms = list(rooms)
        else:
            self.rooms = [rooms] * len(self.seeds)
        # the members' configurations, merged and checked before anything touches a GPU
        base = optimals._load_config()
        if configs is None:
            self.overrides = [None] * len(self.seeds)
        else:
            self.overrides = list(configs)
            if len(self.overrides) != len(self.seeds):
                raise ValueError("one configuration per seed expected")
        self.configs = [optimals._merge_config(base, o) if o is not None else base for o in self.overrides]
        if len({c["grid_step"] for c in self.configs}) > 1:
            raise ValueError("ensemble members must share grid_step (one grid for the batched solves)")
        self.density_stats = simulations.density_stats_spec(density_stats, with_velocity=True)  # (every, thr, vel) / None
        self.lines = simulations.lines_spec(lines)                            # (names, (n, 4) array) or None
        self._lines_arg = None if self.lines is None else dict(zip(self.lines[0], map(tuple, self.lines[1])))
        self.areas = simulations.areas_spec(areas)                            # (names, vertices, offsets) or None
        self.voronoi = simulations.voronoi_spec(voronoi)                      # (cutoff, edges) or None
        if self.voronoi is not None and self.areas is None:
            raise ValueError("voronoi needs measurement areas (areas=...)")
        self.voronoi_maps = simulations.voronoi_maps_spec(voronoi_maps)      # (every, cutoff, edges) or None
        self.rank, self.world = rank, world
        self.mine = shard(len(self.seeds), rank, world)
        self.memory_budget, self.max_wave = memory_budget, max_wave
        self.record, self.verbose = record, verbose
        # True: the GCFM steps of a wave run as batched launches with the randomness drawn in C (oc_gcfm_step_multi_*);
        # False: member by member on their own streams with numpy draws.  Identical results (tests/test_gpu_ensemble.py).
        self.batched_steps = bool(batched_steps)
        self.min_sweep_ctas, self.sweep_ctas = 8, 0   # sweep grid per member: automatic share of the GPU, or fixed
        self.chunk_rows_used = self.chunk_rows
        self.member_chunk_rows = {}   # member index -> chunk_rows of its last solve
        self._rooms_loaded = {}       # room name -> parsed room file (read once, whatever the number of members)
        self.results = {}
        self.members = {}          # member index -> simulation (kept only when record=True)
        self.stats = dict(hjb_ms=0.0, gcfm_ms=0.0, build_ms=0.0, agent_steps=0, cell_updates=0, waves=0, launch_ms=0.0,
                          finish_ms=0.0)

    # ---------------------------------------------------------------------------------------------
    def _room(self, idx):
        room = self.rooms[idx]
        if isinstance(room, dict):
            return room
        if room not in self._rooms_loaded:
            self._rooms_loaded[room] = simulations._load_room(room)
        return self._rooms_loaded[room]

    def member_bytes(self, members=None):
        """device bytes of each member (field_bytes_per_member of its own grid, dt and number of target sets, plus the
        density accumulators when density_stats is on, the line accumulator with lines, the area accumulator with
        areas, the Voronoi accumulator with voronoi and the map accumulators with voronoi_maps); no CUDA"""
        out = []
        for i in (self.mine if members is None else members):
            room, cfg = self._room(i), self.configs[i]
            Ny, Nx = _lib.grid_shape(room["room_length"], room["room_height"], cfg["grid_step"])
            n_keys = len({' or '.join(b[5:]) for b in room["initial_boxes"].values()})
            b = field_bytes_per_member(Ny, Nx, self.T, cfg["dt"], n_keys, self.field_storage)
            if self.density_stats is not None:
                b += _lib.DensityStats.nbytes(Ny, Nx, self.density_stats[1], self.density_stats[2])
            N = sum(int(box[4] * box[2] * box[3]) for box in room["initial_boxes"].values())   # simulations.py:122
            steps = len(simulations.density_frame_steps(self.T, cfg["dt"], 1))
            if self.lines is not None:
                b += _lib.LineCounts.nbytes(N, len(self.lines[0]), steps)
            if self.areas is not None:
                b += _lib.AreaStats.nbytes(N, len(self.areas[0]), len(self.areas[1]), steps)
            if self.voronoi is not None:
                cut, edges = self.voronoi
                bins = _lib.voronoi_bins(room["room_length"], cut) * _lib.voronoi_bins(room["room_height"], cut)
                n_tris = len(simulations.voronoi_triangles(self.areas)[0])
                b += _lib.VoronoiStats.nbytes(N, len(self.areas[0]), n_tris, edges, bins, steps)
            if self.voronoi_maps is not None:
                _, cut, edges = self.voronoi_maps
                bins = _lib.voronoi_bins(room["room_length"], cut) * _lib.voronoi_bins(room["room_height"], cut)
                b += _lib.VoronoiMaps.nbytes(Ny, Nx, N, edges, bins)
            out.append(b)
        return out

    def _build(self, idx):
        # a finished member's library context (device workspace, page-locked buffers, streams) serves the next member
        # of the same room size: a wave of 128 members otherwise pays 128 x (cudaMalloc + cudaMallocHost + frees) per pass
        room = self._room(idx)
        step = self.configs[idx]["grid_step"]
        free = _CTX_POOL.get(_ctx_key(room["room_length"], room["room_height"], step))
        ctx = free.pop() if free else None
        # (the parsed room, not its name: one file read per room, whatever the number of members; a copy per member)
        return simulations.simulation(copy.deepcopy(room), self.T, recompute=self.recompute, record=self.record,
                                      field_storage=self.field_storage, fused=1, lookahead=False,
                                      rng=np.random.RandomState(self.seeds[idx]), chunk_rows=self.chunk_rows,
                                      config=self.overrides[idx], _ctx=ctx,
                                      density_stats=None if self.density_stats is None else
                                      dict(every=self.density_stats[0], threshold=self.density_stats[1],
                                           velocity=self.density_stats[2]), lines=self._lines_arg,
                                      areas=self.areas, voronoi=self.voronoi, voronoi_maps=self.voronoi_maps)

    def _build_wave(self, wave):
        """the members of a wave, constructed by a few host threads: a member's crowd placement (oc_place_box: sequential
        rejection sampling on the member's own RandomState, ~5 ms per 1000 agents), rasterisation and allocations are
        independent of the other members', and the C calls release the GIL"""
        # (measured on the 16-core B200 box, 128 members: 0.52 s on one thread, 0.22 s on 8)
        n_thr = int(os.environ.get("OC_ENSEMBLE_BUILD_THREADS", "8"))
        with contextlib.redirect_stdout(io.StringIO()):   # (one redirection around the pool: sys.stdout is process-wide)
            if n_thr <= 1 or len(wave) < 4:
                return [self._build(i) for i in wave]
            from concurrent.futures import ThreadPoolExecutor
            import torch
            dev = torch.cuda.current_device()

            def build(i):
                torch.cuda.set_device(dev)
                return self._build(i)
            with ThreadPoolExecutor(max_workers=n_thr, thread_name_prefix="oc-build") as ex:
                return list(ex.map(build, wave))

    def _solver_ctx(self, first):
        """the context whose batch workspace (5 arrays per field, 32 streams, one event and one result slot per field)
        the batched solves of this process use, one per device: kept across waves and ensembles, so that a wave does not
        pay ~50 ms of allocations in front of a ~40 ms solve.  Its own grid plays no part: every field is solved on the
        grid of its member's context."""
        import torch
        key = torch.cuda.current_device()
        ctx = _SOLVER_CTX.get(key)
        if ctx is None or not getattr(ctx, "h", None):
            ctx = _SOLVER_CTX[key] = _lib.Context(first.room_length, first.room_height, first._ctx.dx)
        return ctx

    def _solve_wave(self, sims, idx):
        """simulation._solve_all for the given members (wave indices idx) in one batched call over the fields of all
        their target sets, each member with its own grid, sigma, mu, g, horizon and density"""
        import torch
        sctx = self._solver_ctx(sims[0])
        # simulations.py:424-425: density * (simu_step > 0), per member
        d_ms = [s._density_device(s.sigma_convolution) if s.simu_step > 0 else None for s in sims]
        nts = [round((self.T - s.time) / s.dt) for s in sims]                  # optimals.py:140
        if min(nts) < 1:
            raise ValueError("Values in `t_eval` are not within `t_span`.")
        chunk = [self.chunk_rows] * len(sims)
        if self.chunk_plan_for_wave:
            # chunk height planned per grid shape for the members of that shape in this call (a 512^2 room alone would
            # be cut into 16-row chunks to fill the GPU; 64 rooms side by side fill it with 64-row chunks and recompute
            # far fewer halo rows).  The chunking fixes the error-norm summation order: a stand-alone run reproduces a
            # member bit for bit when it is given the same chunk_rows (results[i]["chunk_rows"]).
            count = {}
            for s in sims:
                count[(s.Ny, s.Nx)] = count.get((s.Ny, s.Nx), 0) + 1
            plan = {sh: next(s for s in sims if (s.Ny, s.Nx) == sh)._ctx.plan_chunk_rows(c) for sh, c in count.items()}
            chunk = [plan[(s.Ny, s.Nx)] for s in sims]
            if len(plan) == 1:
                self.chunk_rows_used = chunk[0]
        for i, c in zip(idx, chunk):
            self.member_chunk_rows[i] = c
        # one room per (member, target set)
        opts, grids, Vs, ms, rooms = [], [], [], [], []
        for s, d_m, nt, c in zip(sims, d_ms, nts, chunk):
            for o in s.targets.values():
                if nt - 1 > o._n_slices:
                    raise IndexError("re-solve asks for more slices than the field was allocated for")
                opts.append(o); grids.append(s._ctx); Vs.append(o.d_V); ms.append(d_m)
                rooms.append(dict(sigma=o.sigma, mu=o.mu, g=o.g, T=self.T, nt=nt, chunk_rows=c))
        if all(m is None for m in ms):
            ms = None
        prm = opts[0]._prm   # (rtol, atol, lim: the same for every member; chunk_rows per room above)
        vel = self.field_storage == "velocity"
        import time as _t
        _t0 = _t.perf_counter()
        res = sctx.hjb_solve_grids(grids, Vs, ms, rooms, prm,
                                   out_phi=None if vel else [o.d_phi for o in opts],
                                   out_vx=[o.d_vx for o in opts] if vel else None,
                                   out_vy=[o.d_vy for o in opts] if vel else None)
        self.stats["hjb_call_ms"] = self.stats.get("hjb_call_ms", 0.0) + (_t.perf_counter() - _t0) * 1e3
        self.stats["hjb_calls"] = self.stats.get("hjb_calls", 0) + 1
        self.stats["hjb_call_rooms"] = self.stats.get("hjb_call_rooms", 0) + len(sims)   # (members per call)
        cells = 0
        k = 0
        for s, nt in zip(sims, nts):
            for o in s.targets.values():
                r = res[k]
                k += 1
                o.t, o.nt_opt, o.last_stats = s.time, nt, r["stats"]
                o._h_vx = o._h_vy = None
                if r["stats"]["status"] == -1:
                    raise IndexError("RK45 stopped early (required step size is less than spacing between numbers)")
                cells += r["stats"]["nfev"] * o.Ny * o.Nx
        torch.cuda.synchronize()
        return cells

    def _run_wave(self, wave):
        import time
        import torch
        t0 = time.perf_counter()
        sims = self._build_wave(wave)
        streams = [torch.cuda.Stream() for _ in range(min(len(sims), 128))]
        # the members' sweeps run concurrently: each gets its share of the GPU's resident-CTA slots
        n_sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
        ctas = self.sweep_ctas or max(self.min_sweep_ctas, (n_sm * 4) // len(streams))
        for q, s in enumerate(sims):
            s._ctx.set_int("gcfm_sweep_ctas", ctas)
            s._cuda_stream = streams[q % len(streams)].cuda_stream   # the member's steps run on its own stream
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        self.stats["cell_updates"] += self._solve_wave(sims, wave)
        t2 = time.perf_counter()
        live = list(range(len(sims)))
        batch = None
        if self.batched_steps:
            # one launch per kernel for the whole wave (blockIdx.y = member) and the members' randomness drawn in C from
            # their own MT19937 states: same kernels and same streams of random numbers as the member-by-member path
            main = torch.cuda.current_stream().cuda_stream
            for s in sims:
                s._cuda_stream = main
            # a room's sweep is a dependency chain with ~5 agents runnable at a time (1000 agents, depth ~200): a few warps per
            # room suffice, and every CTA slot given to one room is a slot another room of the wave cannot use
            ctas_b = self.sweep_ctas or int(os.environ.get("OC_ENSEMBLE_CTAS", "0")) or max(2, min(8, (n_sm * 4) // len(sims)))
            batch = _lib.GcfmBatch([dict(ctx=s._ctx, prm=s._gcfm_prm, state=s._state, vdes=s._d_vdes, key_id=s._d_key,
                                         keys=s._keys(), rng=s._np_random) for s in sims], sweep_ctas=ctas_b)
        while live:
            # simulations.py:421: the members due for a re-solve at their own step (their own dt and recompute
            # frequency), solved together; the others keep their fields
            due = [q for q in live if self.recompute and sims[q].simu_step % sims[q].recompute_step == 0
                   and sims[q].simu_step > 0]
            rebind = bool(due)
            if due:
                self.stats["cell_updates"] += self._solve_wave([sims[q] for q in due], [wave[q] for q in due])
            tl0 = time.perf_counter()
            if batch is not None:
                if rebind:
                    for q in due:
                        batch.members[q]["keys"] = sims[q]._keys()
                for q in live:
                    s = sims[q]
                    if self.record:
                        s.write_history(s.time)
                    self.stats["agent_steps"] += s.inside
                if self.density_stats is not None:
                    # this iteration's frames of the members due at their own step, one launch for all of them
                    dd = [q for q in live if sims[q]._dstats.due(sims[q].simu_step)]
                    if dd:
                        _lib.density_accum_multi([sims[q]._ctx for q in dd], [sims[q]._dstats for q in dd],
                                                 [sims[q]._state for q in dd], stream=main)
                if self.voronoi_maps is not None:
                    # the Voronoi map frames of the same members, in one call for all of them
                    dm = [q for q in live if sims[q]._vmaps.due(sims[q].simu_step)]
                    if dm:
                        _lib.vormap_accum_multi([sims[q]._ctx for q in dm], [sims[q]._vmaps for q in dm],
                                                [sims[q]._state for q in dm], stream=main)
                if self.areas is not None:
                    # the state this step starts from, measured for the whole wave in one call
                    for q in live:
                        sims[q]._areas.ensure(sims[q].simu_step + 1)
                    am = [q for q in live if sims[q].N > 0]
                    if am:
                        _lib.areas_measure_multi([sims[q]._ctx for q in am], [sims[q]._areas for q in am],
                                                 [sims[q]._state for q in am], [sims[q].simu_step for q in am],
                                                 stream=main)
                    if self.voronoi is not None:
                        for q in live:
                            sims[q]._voronoi.ensure(sims[q].simu_step + 1)
                        if am:
                            _lib.voronoi_measure_multi([sims[q]._ctx for q in am], [sims[q]._voronoi for q in am],
                                                       [sims[q]._state for q in am],
                                                       [sims[q].simu_step for q in am], stream=main)
                batch.launch(live, [sims[q].inside for q in live], [sims[q].simu_step for q in live], stream=main,
                             rebind=rebind)
                tl1 = time.perf_counter()
                finished = batch.finish()
                if self.lines is not None:
                    # the crossings of this step (final once finish() returns), one launch for the wave
                    lc = [q for q in live if sims[q].N > 0]
                    for q in lc:
                        sims[q]._lines.ensure(sims[q].simu_step + 1)
                    if lc:
                        _lib.lines_count_multi([sims[q]._ctx for q in lc], [sims[q]._lines for q in lc],
                                               [sims[q]._state for q in lc], [sims[q].simu_step for q in lc], stream=main)
                for q, (exits, rc) in zip(live, finished):
                    sims[q]._step_finish((sims[q].dt, ("batched", exits, rc)))
            else:
                launched = []
                for q in live:
                    s = sims[q]
                    if self.record:
                        s.write_history(s.time)
                    self.stats["agent_steps"] += s.inside
                    s._density_frame()
                    launched.append(s._step_launch(s.dt))
                tl1 = time.perf_counter()
                for q, l in zip(live, launched):
                    sims[q]._step_finish(l)
            self.stats["launch_ms"] += (tl1 - tl0) * 1e3
            self.stats["finish_ms"] += (time.perf_counter() - tl1) * 1e3
            live = [q for q in live if (sims[q].inside > 0) and (sims[q].time < sims[q].T)]   # simulations.py:427
        if batch is not None:
            batch.write_back_rng()
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        for i, s in zip(wave, sims):
            s._sync_host()
            self.results[i] = dict(seed=self.seeds[i], evac_time=s.time, steps=s.simu_step, inside=int(s.inside), N=s.N,
                                   exit_order=np.array(s._exit_order, dtype=np.int64), exit_step=s._exit_step.copy(),
                                   times=np.array(s._h_timev, dtype=float), final=np.array(s._h_now, dtype=float),
                                   hjb={k: o.last_stats for k, o in s.targets.items()}, config=self.configs[i],
                                   chunk_rows=self.member_chunk_rows[i])
            if self.density_stats is not None:
                self.results[i]["density"] = s._dstats.result()
            if self.voronoi_maps is not None:
                self.results[i]["voronoi_maps"] = s._vmaps.result()
            if self.lines is not None:
                self.results[i]["lines"] = s._lines.result(s.simu_step)
            if self.areas is not None:
                self.results[i]["areas"] = s._areas.result(s.simu_step)
                if self.voronoi is not None:
                    self.results[i]["areas"]["voronoi"] = s._voronoi.result(s.simu_step)
            if self.record:
                self.members[i] = s
        self.stats["build_ms"] += (t1 - t0) * 1e3
        self.stats["hjb_ms"] += (t2 - t1) * 1e3
        self.stats["gcfm_ms"] += (t3 - t2) * 1e3
        self.stats["waves"] += 1
        if not self.record:
            for s in sims:
                for o in s.targets.values():
                    o.d_phi = o.d_vx = o.d_vy = None
                if len(_CTX_POOL.setdefault(_ctx_key(s.room_length, s.room_height, s.grid_step), [])) < 512:
                    _CTX_POOL[_ctx_key(s.room_length, s.room_height, s.grid_step)].append(s._ctx)
                else:
                    s._ctx.close()
                s.__dict__.clear()   # marshalled key descriptors, state tensors, agents <-> simulation reference cycles
            del sims
            import gc
            gc.collect()             # (a wave holds tens of GB of field samples: do not wait for the cyclic collector)
            # the freed field tensors stay in torch's caching allocator for the next wave (same sizes); they are only
            # handed back to the driver when the device runs short for the library's own allocations
            free, total = torch.cuda.mem_get_info()
            if free < 0.1 * total:
                torch.cuda.empty_cache()

    def run(self, gather=True):
        """run this rank's members wave by wave; with torch.distributed initialised and gather=True every rank
        returns the merged results of all ranks"""
        import torch
        if not self.mine:
            return gather_results({}) if gather else {}
        per = self.member_bytes()
        budget = self.memory_budget
        if budget is None:
            free, _total = torch.cuda.mem_get_info()
            # (blocks cached by torch's allocator are available to the next wave's tensors)
            free += torch.cuda.memory_reserved() - torch.cuda.memory_allocated()
            budget = int(free * 0.8)
        for wave in plan_waves(self.mine, per, budget, self.max_wave):
            self._run_wave(wave)
            if self.verbose:
                print(f"[ensemble rank {self.rank}] wave of {len(wave)} members done "
                      f"({len(self.results)}/{len(self.mine)})", flush=True)
        return gather_results(self.results) if gather else dict(self.results)
