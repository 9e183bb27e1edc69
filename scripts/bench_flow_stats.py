"""Flow statistics on the device: what the velocity maps and the measurement lines cost.

Arm (a): bench.py's one-GPU slalom room (16384 x 2048 nodes, 12 500 agents) after a few steps.  The density frame with and
  without velocity maps (CUDA events around R ``oc_density_accum_vel`` launches of each, alternating), then the
  ``advance()`` step with 0 and 16 measurement lines (wall clock around K steps of each, alternating, medians).
Arm (b): one 128-member wave of the configs[4] room (``synthetic.ensemble_room(512, 1000)``): the batched frame with and
  without velocity maps (CUDA events around R ``oc_density_accum_vel_multi`` launches of each, alternating; the members'
  crowds are one placed crowd jittered per member, their velocities drawn), then whole ensembles of 128 members, T = 1 s,
  batched steps, with 0 and 16 lines (alternating after a warm-up pass of each: wall clock of ``run()`` per pass, its
  stepping part -- ``ensemble.stats["gcfm_ms"]``, after the HJB solve -- per wave step, and CUDA events around every
  ``oc_lines_count_multi`` launch).
One JSON line per arm, with the card's name and power limit read in the same run.

    python scripts/bench_flow_stats.py [--reps 5] [--steps 20] [--passes 2] [--members 128] [--arms a,b] [--out FILE]
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


def sixteen_lines(L, H, rng):
    """16 measurement lines across the room: 8 vertical cross-sections and 8 random segments of 5-50 m"""
    out = {f"x{k}": (L * (k + 0.5) / 8, 0.0, L * (k + 0.5) / 8, H) for k in range(8)}
    for k in range(8):
        x0, y0 = rng.uniform(0, L), rng.uniform(0, H)
        a, r = rng.uniform(0, 2 * np.pi), rng.uniform(5, 50)
        out[f"seg{k}"] = (x0, y0, x0 + r * np.cos(a), y0 + r * np.sin(a))
    return out


def _time_alternating(fns, reps, passes):
    """CUDA-event milliseconds per call of each fn, reps calls per pass, the fns alternating pass by pass"""
    import torch
    ms = {k: [] for k in fns}
    for _ in range(passes):
        for k, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / reps)
    return {k: float(np.median(v)) for k, v in ms.items()}


def arm_a(args):
    import torch
    from optimal_crowds_b200 import _lib, simulations, synthetic
    room = synthetic.slalom_room(16384, 2048, agents=12500)
    np.random.seed(1000)
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation(room, 2.0)
        simu._solve_all()
    simu.advance(5)                               # a crowd in motion: non-zero velocities
    ctx, st = simu._ctx, simu._state
    plain = _lib.DensityStats(ctx, simu._d_Vglobal, simu.sigma_convolution, 1)
    vel = _lib.DensityStats(ctx, simu._d_Vglobal, simu.sigma_convolution, 1, velocity=True)
    acc = lambda s: ctx.density_accum(s, st["x"], st["y"], st["status"], vx=st["vx"], vy=st["vy"])
    acc(plain); acc(vel)                          # warm-up of both kernels
    frame = _time_alternating({"off": lambda: acc(plain), "velocity": lambda: acc(vel)}, args.reps, args.passes)
    assert torch.equal(plain.sum, vel.sum)        # the density part is unchanged by the velocity maps
    names, arr = simulations.lines_spec(sixteen_lines(simu.room_length, simu.room_height, np.random.RandomState(7)))
    lines = _lib.LineCounts(ctx, names, arr, st, simu.simu_step + 2 * args.passes * args.steps + 8)
    simu._lines = lines
    simu.advance(2)                               # warm-up of the counting kernel
    walls = {"off": [], "lines_16": []}
    for _ in range(args.passes):
        for mode in walls:
            simu._lines = lines if mode == "lines_16" else None
            if mode == "lines_16":   # (the kept positions follow the steps taken without lines)
                lines.px.copy_(st["x"]); lines.py.copy_(st["y"]); lines.inside.copy_(st["status"])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            done = simu.advance(args.steps)
            torch.cuda.synchronize()
            walls[mode].append((time.perf_counter() - t0) / max(done, 1) * 1e3)
    simu._lines = lines
    crossings = int(lines.counts.sum())
    off, on = float(np.median(walls["off"])), float(np.median(walls["lines_16"]))
    return {"arm": "a_slalom_16384x2048", "grid": [simu.Ny, simu.Nx], "agents": int(simu.N),
            "agents_inside": int(simu.inside), "reps": args.reps, "passes": args.passes,
            "frame": {"ms_off": frame["off"], "ms_velocity": frame["velocity"],
                      "velocity_overhead": frame["velocity"] / frame["off"] - 1},
            "advance": {"steps_per_pass": args.steps, "ms_per_step_off": off, "ms_per_step_16_lines": on,
                        "lines_overhead": on / off - 1, "crossings_counted": crossings,
                        "all_steps_ms": {k: v for k, v in walls.items()}}}


def arm_b(args):
    import torch
    from optimal_crowds_b200 import _lib, ensemble, simulations, synthetic
    n = args.members
    room = synthetic.ensemble_room(512, 1000)
    with contextlib.redirect_stdout(io.StringIO()):
        probe = simulations.simulation(room, args.T, rng=np.random.RandomState(0))
    ctx = probe._ctx
    rng = np.random.RandomState(5)
    x0, y0 = probe._h_now[:, 0], probe._h_now[:, 1]
    states, plain, vel = [], [], []
    for _ in range(n):
        states.append(dict(x=ctx.to_device(x0 + rng.normal(0, 0.05, probe.N)),
                           y=ctx.to_device(y0 + rng.normal(0, 0.05, probe.N)),
                           vx=ctx.to_device(rng.normal(1.0, 0.3, probe.N)), vy=ctx.to_device(rng.normal(0, 0.3, probe.N)),
                           status=ctx.to_device(np.ones(probe.N, dtype=np.uint8))))
        plain.append(_lib.DensityStats(ctx, probe._d_Vglobal, probe.sigma_convolution, 1))
        vel.append(_lib.DensityStats(ctx, probe._d_Vglobal, probe.sigma_convolution, 1, velocity=True))
    ctxs = [ctx] * n
    run = lambda s: _lib.density_accum_multi(ctxs, s, states)
    run(plain); run(vel)
    frame = _time_alternating({"off": lambda: run(plain), "velocity": lambda: run(vel)}, args.reps, args.passes)
    del states, plain, vel
    # whole ensembles with 0 and 16 lines
    seeds = list(range(n))
    lines = sixteen_lines(probe.room_length, probe.room_height, np.random.RandomState(8))
    timed = []
    real = _lib.lines_count_multi

    def timed_multi(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()          # (the ensemble's batched steps run on torch's current stream)
        real(*a, **k)
        e1.record()
        timed.append((e0, e1))
    _lib.lines_count_multi = timed_multi
    modes = {"off": None, "lines_16": lines}
    acc = {m: dict(wall=0.0, gcfm_ms=0.0, steps=0, passes=0, kernel_ms=0.0, launches=0) for m in modes}
    crossings = 0
    try:
        for p in range(args.warmup + args.passes):
            for mode, ln in modes.items():
                timed.clear()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ens = ensemble.ensemble([room] * n, args.T, seeds, max_wave=n, lines=ln)
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
                if ln is not None:
                    crossings = int(sum(r["lines"]["to_left"].sum() + r["lines"]["to_right"].sum() for r in res.values()))
    finally:
        _lib.lines_count_multi = real
    out = {"arm": "b_ensemble_512sq_x%d" % n, "members": n, "T": args.T, "grid": [probe.Ny, probe.Nx],
           "agents": int(probe.N), "reps": args.reps,
           "frame": {"ms_per_wave_frame_off": frame["off"], "ms_per_wave_frame_velocity": frame["velocity"],
                     "velocity_overhead": frame["velocity"] / frame["off"] - 1}}
    for mode, a in acc.items():
        row = {"s_per_pass": a["wall"] / a["passes"], "ms_per_wave_step": a["gcfm_ms"] / a["steps"]}
        if a["launches"]:
            row.update(count_kernel_ms_per_wave_step=a["kernel_ms"] / a["launches"], crossings_per_pass=crossings)
        out[mode] = row
    out["lines_overhead"] = out["lines_16"]["ms_per_wave_step"] / out["off"]["ms_per_wave_step"] - 1
    probe._ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5, help="timed frame launches per pass")
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
        raise SystemExit("bench_flow_stats.py measures the GPU: no CUDA device")
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
