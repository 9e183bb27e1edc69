"""Measurement areas on the device: what they cost per step.

Arm (a): bench.py's one-GPU slalom room (16384 x 2048 nodes, 12 500 agents) after a few steps: the ``advance()`` step
  with 0, 16 and 64 areas of 16 vertices (wall clock around K steps of each, the modes alternating pass by pass, medians).
Arm (b): one 128-member wave of the configs[4] room (``synthetic.ensemble_room(512, 1000)``): whole ensembles of 128
  members, T = 1 s, batched steps, with 0 and 16 areas (alternating after a warm-up pass of each): wall clock of ``run()``
  per pass, its stepping part -- ``ensemble.stats["gcfm_ms"]``, after the HJB solve -- per wave step, and CUDA events
  around every ``oc_areas_measure_multi`` call (its two launches).
One JSON line per arm, with the card's name and power limit read in the same run.

    python scripts/bench_areas.py [--steps 20] [--passes 3] [--members 128] [--arms a,b] [--out FILE]
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


def areas(n, L, H, rng):
    """n star-shaped (concave) polygons of 16 vertices, radii 2-30 m (at most a fifth of the room's height), anywhere
    in the room"""
    t = np.linspace(0, 2 * np.pi, 16, endpoint=False)
    out = {}
    for k in range(n):
        r = rng.uniform(2, min(30, H / 5))
        cx, cy = rng.uniform(r, L - r), rng.uniform(r, H - r)
        rad = r * (1 + 0.3 * np.cos(4 * t))
        out[f"a{k}"] = np.stack([cx + rad * np.cos(t), cy + rad * np.sin(t)], axis=1)
    return out


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
    rng = np.random.RandomState(7)
    accs = {"off": None}
    for n in (16, 64):
        spec = simulations.areas_spec(areas(n, simu.room_length, simu.room_height, rng))
        accs[f"areas_{n}"] = _lib.AreaStats(ctx, *spec, simu.N, simu.simu_step + 8 * args.passes * args.steps + 8)
    for acc in accs.values():                     # warm-up of the measuring kernels
        simu._areas = acc
        simu.advance(2)
    walls = {k: [] for k in accs}
    for _ in range(args.passes):
        for mode in walls:
            simu._areas = accs[mode]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            done = simu.advance(args.steps)
            torch.cuda.synchronize()
            walls[mode].append((time.perf_counter() - t0) / max(done, 1) * 1e3)
    simu._areas = None
    med = {k: float(np.median(v)) for k, v in walls.items()}
    inside = {k: int(a.count[: simu.simu_step].sum()) for k, a in accs.items() if a is not None}
    return {"arm": "a_slalom_16384x2048", "grid": [simu.Ny, simu.Nx], "agents": int(simu.N),
            "agents_inside": int(simu.inside), "passes": args.passes, "steps_per_pass": args.steps,
            "ms_per_step": med, "overhead": {k: med[k] / med["off"] - 1 for k in med if k != "off"},
            "agent_rows_inside_areas": inside, "all_steps_ms": walls}


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
    real = _lib.areas_measure_multi

    def timed_multi(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()          # (the ensemble's batched steps run on torch's current stream)
        real(*a, **k)
        e1.record()
        timed.append((e0, e1))
    _lib.areas_measure_multi = timed_multi
    modes = {"off": None, "areas_16": spec16}
    acc = {m: dict(wall=0.0, gcfm_ms=0.0, steps=0, passes=0, kernel_ms=0.0, launches=0) for m in modes}
    inside = 0
    try:
        for p in range(args.warmup + args.passes):
            for mode, ar in modes.items():
                timed.clear()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ens = ensemble.ensemble([room] * n, args.T, seeds, max_wave=n, areas=ar)
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
                if ar is not None:
                    inside = int(sum(r["areas"]["count"].sum() for r in res.values()))
    finally:
        _lib.areas_measure_multi = real
    out = {"arm": "b_ensemble_512sq_x%d" % n, "members": n, "T": args.T, "grid": [probe.Ny, probe.Nx],
           "agents": int(probe.N)}
    for mode, a in acc.items():
        row = {"s_per_pass": a["wall"] / a["passes"], "ms_per_wave_step": a["gcfm_ms"] / a["steps"]}
        if a["launches"]:
            row.update(measure_ms_per_wave_step=a["kernel_ms"] / a["launches"], agent_rows_inside_per_pass=inside)
        out[mode] = row
    out["areas_overhead"] = out["areas_16"]["ms_per_wave_step"] / out["off"]["ms_per_wave_step"] - 1
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
        raise SystemExit("bench_areas.py measures the GPU: no CUDA device")
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
