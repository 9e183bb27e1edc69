"""Voronoi maps on the device: what a frame costs.

Arm (a): bench.py's one-GPU slalom room (16384 x 2048 nodes, 12 500 agents) after a few steps: one Voronoi map frame
  (cutoff 1 m, 12 edges; ``oc_vormap_accum``, six launches), one Gaussian ``density_stats`` frame of the same crowd
  (``oc_density_accum``) and one ``advance()`` step without observers, the three alternating pass by pass; CUDA events
  around every frame, wall clock around the steps (medians per call).
Arm (b): one 128-member wave of the configs[4] room (``synthetic.ensemble_room(512, 1000)``), each member its own grid
  context and a crowd moved from the room's start positions: one batched Voronoi map frame (``oc_vormap_accum_multi``)
  against one batched Gaussian frame (``oc_density_accum_multi``), alternating; CUDA events around every call.
One JSON line per arm, with the card's name and power limit read in the same run.

    python scripts/bench_voronoi_maps.py [--frames 10] [--passes 3] [--members 128] [--arms a,b] [--out FILE]
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def _events(fn, n):
    """milliseconds of each of n calls of fn, from CUDA events on the current stream"""
    import torch
    out = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        out.append((e0, e1))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in out]


def arm_a(args):
    import torch
    from optimal_crowds_b200 import _lib, simulations, synthetic
    room = synthetic.slalom_room(16384, 2048, agents=12500)
    np.random.seed(1000)
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation(room, 2.0)
        simu._solve_all()
    simu.advance(5)                               # a crowd in motion: non-zero velocities
    ctx = simu._ctx
    maps = _lib.VoronoiMaps(ctx, simu._d_Vglobal, 1.0, 12, 1, simu.N)
    dens = _lib.DensityStats(ctx, simu._d_Vglobal, simu.sigma_convolution)
    st = simu._state
    modes = {"voronoi_map_frame": lambda: ctx.vormap_accum(maps, st),
             "gaussian_frame": lambda: ctx.density_accum(dens, st["x"], st["y"], st["status"])}
    for fn in modes.values():                     # warm-up
        _events(fn, 2)
    simu.advance(2)
    ms = {k: [] for k in list(modes) + ["advance_step"]}
    for _ in range(args.passes):
        for k, fn in modes.items():
            ms[k] += _events(fn, args.frames if k != "gaussian_frame" else max(args.frames // 4, 2))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        done = simu.advance(args.frames)
        torch.cuda.synchronize()
        ms["advance_step"].append((time.perf_counter() - t0) / max(done, 1) * 1e3)
    torch.cuda.synchronize()
    r = maps.result()
    med = {k: float(np.median(v)) for k, v in ms.items()}
    nodes = simu.Ny * simu.Nx
    return {"arm": "a_slalom_16384x2048", "grid": [simu.Ny, simu.Nx], "agents": int(simu.N),
            "agents_inside": int(simu.inside), "cutoff": 1.0, "edges": 12, "passes": args.passes,
            "ms_median": med, "voronoi_vs_gaussian": med["voronoi_map_frame"] / med["gaussian_frame"],
            "voronoi_vs_step": med["voronoi_map_frame"] / med["advance_step"],
            "covered_node_fraction": float((r["covered"] > 0).mean()),
            "accumulator_bytes_per_frame_lower_bound": 16 * nodes, "all_ms": ms}


def arm_b(args):
    import torch
    from optimal_crowds_b200 import _lib, simulations, synthetic
    n = args.members
    room = synthetic.ensemble_room(512, 1000)
    with contextlib.redirect_stdout(io.StringIO()):
        probe = simulations.simulation(room, 1.0, rng=np.random.RandomState(0))
    x0, y0 = probe._row0[:, 0], probe._row0[:, 1]
    N = probe.N
    ctxs, maps, dens, states = [], [], [], []
    for q in range(n):
        rng = np.random.RandomState(q)
        c = _lib.Context(probe.room_length, probe.room_height, probe.grid_step)
        Vg = c.to_device(probe.V)
        ctxs.append(c)
        maps.append(_lib.VoronoiMaps(c, Vg, 1.0, 12, 1, N))
        dens.append(_lib.DensityStats(c, Vg, probe.sigma_convolution))
        states.append(dict(x=c.to_device(x0 + rng.uniform(-0.2, 0.2, N)), y=c.to_device(y0 + rng.uniform(-0.2, 0.2, N)),
                           vx=c.to_device(rng.normal(0, 1, N)), vy=c.to_device(rng.normal(0, 1, N)),
                           status=c.to_device(np.ones(N, dtype=np.uint8))))
    modes = {"voronoi_map_wave_frame": lambda: _lib.vormap_accum_multi(ctxs, maps, states),
             "gaussian_wave_frame": lambda: _lib.density_accum_multi(ctxs, dens, states)}
    for fn in modes.values():
        _events(fn, 2)
    ms = {k: [] for k in modes}
    for _ in range(args.passes):
        for k, fn in modes.items():
            ms[k] += _events(fn, args.frames)
    med = {k: float(np.median(v)) for k, v in ms.items()}
    out = {"arm": "b_wave_512sq_x%d" % n, "members": n, "grid": [probe.Ny, probe.Nx], "agents": int(N),
           "cutoff": 1.0, "edges": 12, "passes": args.passes, "ms_median": med,
           "voronoi_vs_gaussian": med["voronoi_map_wave_frame"] / med["gaussian_wave_frame"],
           "voronoi_ms_per_member_frame": med["voronoi_map_wave_frame"] / n, "all_ms": ms}
    for c in ctxs:
        c.close()
    probe._ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--frames", type=int, default=10, help="timed calls of every mode per pass")
    ap.add_argument("--passes", type=int, default=3, help="timed passes of every mode (alternating)")
    ap.add_argument("--members", type=int, default=128)
    ap.add_argument("--arms", default="a,b")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    from scripts.bench_sweep import card
    if not torch.cuda.is_available():
        raise SystemExit("bench_voronoi_maps.py measures the GPU: no CUDA device")
    torch.cuda.set_device(0)
    os.chdir(REPO)                 # config.json resolves as for the library's users
    info = card()
    lines = []
    for arm in args.arms.split(","):
        row = (arm_a if arm == "a" else arm_b)(args)
        row["card"] = info
        lines.append(json.dumps(row))
        print(lines[-1], flush=True)
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
