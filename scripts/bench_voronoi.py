"""Voronoi measures of measurement areas on the device: what they cost per step.

Arm (a): bench.py's one-GPU slalom room (16384 x 2048 nodes, 12 500 agents) after a few steps: the ``advance()`` step
  with 16 areas of 16 vertices, classic measures only against classic plus Voronoi measures (cutoff 1 m, 12 edges),
  and classic plus Voronoi with one area covering the whole room (wall clock around K steps of each, the modes
  alternating pass by pass, medians).
Arm (b): one 128-member wave of the configs[4] room (``synthetic.ensemble_room(512, 1000)``): whole ensembles of 128
  members, T = 1 s, batched steps, with 16 areas, without and with Voronoi measures (alternating after a warm-up pass of
  each): wall clock of ``run()`` per pass, its stepping part -- ``ensemble.stats["gcfm_ms"]``, after the HJB solve --
  per wave step, and CUDA events around every ``oc_voronoi_measure_multi`` call (its six launches).
One JSON line per arm, with the card's name and power limit read in the same run.

    python scripts/bench_voronoi.py [--steps 20] [--passes 3] [--members 128] [--arms a,b] [--out FILE]
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

from scripts.bench_areas import areas  # noqa: E402


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
    L, H = simu.room_length, simu.room_height
    cap = simu.simu_step + 8 * args.passes * args.steps + 8
    vspec = simulations.voronoi_spec(True)
    spec16 = simulations.areas_spec(areas(16, L, H, np.random.RandomState(7)))
    room_spec = simulations.areas_spec({"room": [(0.0, 0.0), (L, 0.0), (L, H), (0.0, H)]})
    vor = lambda s: _lib.VoronoiStats(ctx, s[1], s[2], *simulations.voronoi_triangles(s), *vspec, simu.N, cap)
    a16 = _lib.AreaStats(ctx, *spec16, simu.N, cap)
    modes = {"areas_16": (a16, None), "areas_16_voronoi": (a16, vor(spec16)),
             "room_voronoi": (_lib.AreaStats(ctx, *room_spec, simu.N, cap), vor(room_spec))}
    for a, v in modes.values():                   # warm-up of the measuring kernels
        simu._areas, simu._voronoi = a, v
        simu.advance(2)
    walls = {k: [] for k in modes}
    for _ in range(args.passes):
        for mode in walls:
            simu._areas, simu._voronoi = modes[mode]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            done = simu.advance(args.steps)
            torch.cuda.synchronize()
            walls[mode].append((time.perf_counter() - t0) / max(done, 1) * 1e3)
    simu._areas = simu._voronoi = None
    med = {k: float(np.median(v)) for k, v in walls.items()}
    covered = float(modes["room_voronoi"][1].rows[simu.simu_step - 1, 0, 4])
    return {"arm": "a_slalom_16384x2048", "grid": [simu.Ny, simu.Nx], "agents": int(simu.N),
            "agents_inside": int(simu.inside), "voronoi": list(vspec), "passes": args.passes,
            "steps_per_pass": args.steps, "ms_per_step": med,
            "overhead_vs_areas_16": {k: med[k] / med["areas_16"] - 1 for k in med if k != "areas_16"},
            "room_covered_last_step": covered, "all_steps_ms": walls}


def arm_b(args):
    import torch
    from optimal_crowds_b200 import _lib, ensemble, simulations, synthetic
    n = args.members
    room = synthetic.ensemble_room(512, 1000)
    with contextlib.redirect_stdout(io.StringIO()):
        probe = simulations.simulation(room, args.T, rng=np.random.RandomState(0))
    spec16 = areas(16, probe.room_length, probe.room_height, np.random.RandomState(8))
    seeds = list(range(n))
    timed = []
    real = _lib.voronoi_measure_multi

    def timed_multi(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()          # (the ensemble's batched steps run on torch's current stream)
        real(*a, **k)
        e1.record()
        timed.append((e0, e1))
    _lib.voronoi_measure_multi = timed_multi
    modes = {"areas_16": None, "areas_16_voronoi": True}
    acc = {m: dict(wall=0.0, gcfm_ms=0.0, steps=0, passes=0, kernel_ms=0.0, launches=0) for m in modes}
    try:
        for p in range(args.warmup + args.passes):
            for mode, vo in modes.items():
                timed.clear()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ens = ensemble.ensemble([room] * n, args.T, seeds, max_wave=n, areas=spec16, voronoi=vo)
                res = ens.run(gather=False)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                if p < args.warmup:
                    continue
                a = acc[mode]
                a["wall"] += wall
                a["gcfm_ms"] += ens.stats["gcfm_ms"]
                a["passes"] += 1
                a["steps"] += max(r["steps"] for r in res.values())
                a["launches"] += len(timed)
                a["kernel_ms"] += sum(e0.elapsed_time(e1) for e0, e1 in timed)
    finally:
        _lib.voronoi_measure_multi = real
    out = {"arm": "b_ensemble_512sq_x%d" % n, "members": n, "T": args.T, "grid": [probe.Ny, probe.Nx],
           "agents": int(probe.N)}
    for mode, a in acc.items():
        row = {"s_per_pass": a["wall"] / a["passes"], "ms_per_wave_step": a["gcfm_ms"] / a["steps"]}
        if a["launches"]:
            row.update(voronoi_ms_per_wave_step=a["kernel_ms"] / a["launches"])
        out[mode] = row
    out["voronoi_overhead"] = out["areas_16_voronoi"]["ms_per_wave_step"] / out["areas_16"]["ms_per_wave_step"] - 1
    probe._ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=20, help="arm (a): steps per timed advance()")
    ap.add_argument("--passes", type=int, default=3, help="timed passes of every mode (alternating)")
    ap.add_argument("--warmup", type=int, default=1, help="arm (b): untimed ensemble passes of every mode first")
    ap.add_argument("--members", type=int, default=128)
    ap.add_argument("--T", type=float, default=1.0)
    ap.add_argument("--arms", default="a,b")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    from scripts.bench_sweep import card
    if not torch.cuda.is_available():
        raise SystemExit("bench_voronoi.py measures the GPU: no CUDA device")
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
