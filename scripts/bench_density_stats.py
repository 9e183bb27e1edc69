"""Density statistics on the device: what accumulating the density frames of a run costs.

Arm (a): ensembles of 128 members of the configs[4] room (``synthetic.ensemble_room(512, 1000)``), T = 1 s, no re-solves,
  batched steps, with the statistics off, ``every=10`` and ``every=1``.  Seconds per pass (wall clock of ``run()``; the
  arms alternate after a warm-up pass of each) and the accumulate kernel's time from CUDA events around every
  ``oc_density_accum_multi`` launch: per wave-frame (one launch = the frame of every member of the wave) and per
  member-frame.
Arm (b): bench.py's one-GPU slalom room (16384 x 2048 nodes, 12 500 agents) through ``simulation.advance()``: K steps
  with the statistics off and K steps with ``every=10`` (wall clock, alternating), and the frame kernel alone (CUDA events
  around R ``oc_density_accum`` launches on the room's state after the timed steps).
Work: the node-agent pairs the kernel evaluates -- those its tile culling at r_zero keeps, counted on the host from the
positions with the kernel's own rule -- per second of kernel time, and the FP64 rate as a share of the peak
``oc_fp64_peak`` measures in the same run, counted as bench.py counts gcfm.roofline (FP64-pipe instructions per pair x
2 flops).  One JSON line per arm, with the card's name and power limit read in the same run.

    python scripts/bench_density_stats.py [--members 128] [--T 1.0] [--passes 2] [--steps 20] [--reps 5] [--arms a,b]
                                          [--out FILE]
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import math
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

# FP64-pipe instructions per evaluated pair, from the SASS of density_tile (cuobjdump -sass of oc_gcfm.o, sm_100a): the
# unrolled loop body issues 23 per pair (DADD, DMUL, DFMA of the distance and the two divisions) and ocm_exp about 47 on
# its common path (range checks, reduction, polynomial, division, scaling).  A static count, not a measured one.
FP64_INST_PER_PAIR = 70.0
DN_TX, DN_TY = 32, 8   # the kernel's tile


def kernel_pairs(X, Y, Vg_shape, x, y, sigma):
    """node-agent pairs density_tile evaluates for agents (x, y) inside: per tile, its in-grid nodes times the agents in
    its box widened by r_zero (or with a NaN coordinate), exactly the kernel's culling test"""
    Ny, Nx = Vg_shape
    two_s2 = 2 * (sigma * sigma)
    r = math.sqrt(745.2 * two_s2) * (1.0 + 1e-9) + 1e-9
    nan = np.isnan(x) | np.isnan(y)
    n_nan = int(nan.sum())
    x, y = x[~nan], y[~nan]
    order = np.argsort(x, kind="stable")
    xs, ys = x[order], y[order]
    total = 0
    jx0 = np.arange(0, Nx, DN_TX)
    jx1 = np.minimum(jx0 + DN_TX, Nx) - 1
    bx0, bx1 = X[jx0] - r, X[jx1] + r
    wx = jx1 - jx0 + 1
    for jy0 in range(0, Ny, DN_TY):
        jy1 = min(jy0 + DN_TY, Ny) - 1
        sel = (ys >= Y[jy0] - r) & (ys <= Y[jy1] + r)
        xr = xs[sel]
        cnt = np.searchsorted(xr, bx1, side="right") - np.searchsorted(xr, bx0, side="left") + n_nan
        total += int((cnt * wx).sum()) * (jy1 - jy0 + 1)
    return total


def arm_a(args, fp64_peak):
    import torch
    from optimal_crowds_b200 import _lib, ensemble, synthetic
    n = args.members
    room = synthetic.ensemble_room(512, 1000)
    seeds = list(range(n))
    modes = {"off": None, "every_10": {"every": 10}, "every_1": {"every": 1}}
    timed = []   # (wave members, start event, end event) of every batched accumulate launch
    real = _lib.density_accum_multi

    def timed_multi(ctxs, stats, states, stream=None):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()          # (the ensemble's batched steps run on torch's current stream)
        real(ctxs, stats, states, stream)
        e1.record()
        timed.append((len(ctxs), e0, e1))
    _lib.density_accum_multi = timed_multi
    acc = {m: dict(wall=0.0, kernel_ms=0.0, launches=0, member_frames=0, passes=0) for m in modes}
    last = {}
    try:
        for p in range(args.warmup + args.passes):
            for mode, ds in modes.items():
                timed.clear()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = ensemble.ensemble([room] * n, args.T, seeds, max_wave=n, density_stats=ds).run(gather=False)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                if p < args.warmup:
                    continue
                a = acc[mode]
                a["wall"] += wall
                a["passes"] += 1
                a["launches"] += len(timed)
                a["member_frames"] += sum(k for k, _, _ in timed)
                a["kernel_ms"] += sum(e0.elapsed_time(e1) for _, e0, e1 in timed)
                last[mode] = res
    finally:
        _lib.density_accum_multi = real
    # pairs of one member-frame, from the members' final positions (in T = 1 s the crowd moves about a metre)
    from optimal_crowds_b200 import simulations
    res = last["every_1"]
    with contextlib.redirect_stdout(io.StringIO()):
        probe = simulations.simulation(room, args.T, rng=np.random.RandomState(0))
    X, Y = probe._ctx.X, probe._ctx.Y
    sigma = probe.sigma_convolution
    pairs = [kernel_pairs(X, Y, (probe.Ny, probe.Nx), r["final"][r["exit_step"] < 0, 0], r["final"][r["exit_step"] < 0, 1],
                          sigma) for r in res.values()]
    pairs_per_member_frame = float(np.mean(pairs))
    out = {"arm": "a_ensemble_512sq_x%d" % n, "members": n, "T": args.T, "grid": [probe.Ny, probe.Nx],
           "agents": int(probe.N), "all_inside": all(int(r["inside"]) == r["N"] for r in res.values()),
           "frames_per_member": {m: last[m][0].get("density", {}).get("frames", 0) for m in modes}}
    for mode, a in acc.items():
        row = {"s_per_pass": a["wall"] / a["passes"]}
        if a["launches"]:
            k_s = a["kernel_ms"] * 1e-3
            row.update(ms_per_wave_frame=a["kernel_ms"] / a["launches"], ms_per_member_frame=a["kernel_ms"] / a["member_frames"],
                       kernel_s_per_pass=k_s / a["passes"], pairs_per_s=pairs_per_member_frame * a["member_frames"] / k_s,
                       fp64_tflops=pairs_per_member_frame * a["member_frames"] * FP64_INST_PER_PAIR * 2 / k_s / 1e12)
            row["fp64_frac_of_peak"] = row["fp64_tflops"] / fp64_peak
        out[mode] = row
    out["pairs_per_member_frame"] = pairs_per_member_frame
    return out


def arm_b(args, fp64_peak):
    import torch
    from optimal_crowds_b200 import _lib, simulations, synthetic
    room = synthetic.slalom_room(16384, 2048, agents=12500)
    np.random.seed(1000)
    with contextlib.redirect_stdout(io.StringIO()):
        simu = simulations.simulation(room, 2.0, density_stats={"every": 10})
        simu._solve_all()
    stats = simu._dstats
    simu.advance(3)                       # warm-up of both paths' kernels
    simu._dstats = None
    simu.advance(3)
    walls = {"off": [], "every_10": []}
    frames_on = 0
    for p in range(args.passes):
        for mode in ("off", "every_10"):
            simu._dstats = stats if mode == "every_10" else None
            f0 = stats.frames
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            done = simu.advance(args.steps)
            torch.cuda.synchronize()
            walls[mode].append((time.perf_counter() - t0) / max(done, 1))
            frames_on += stats.frames - f0
    simu._dstats = stats
    # the frame kernel alone on the current state, into scratch accumulators
    st = simu._state
    scratch = _lib.DensityStats(simu._ctx, simu._d_Vglobal, simu.sigma_convolution, 10)
    simu._ctx.density_accum(scratch, st["x"], st["y"], st["status"])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.reps):
        simu._ctx.density_accum(scratch, st["x"], st["y"], st["status"])
    e1.record()
    torch.cuda.synchronize()
    ms_frame = e0.elapsed_time(e1) / args.reps
    now, inside = simu._h_now, simu._h_status.astype(bool)
    pairs = kernel_pairs(simu._ctx.X, simu._ctx.Y, (simu.Ny, simu.Nx), now[inside, 0], now[inside, 1],
                         simu.sigma_convolution)
    step_off, step_on = float(np.median(walls["off"])), float(np.median(walls["every_10"]))
    return {"arm": "b_slalom_16384x2048", "grid": [simu.Ny, simu.Nx], "agents": int(simu.N),
            "agents_inside": int(inside.sum()), "steps_per_pass": args.steps, "passes": args.passes,
            "off": {"ms_per_step": step_off * 1e3},
            "every_10": {"ms_per_step": step_on * 1e3, "frames": frames_on,
                         "ms_per_frame_from_steps": (step_on - step_off) * 1e3 * 10},
            "frame_kernel": {"ms_per_frame": ms_frame, "reps": args.reps, "pairs_per_frame": pairs,
                             "pairs_per_s": pairs / (ms_frame * 1e-3),
                             "fp64_tflops": pairs * FP64_INST_PER_PAIR * 2 / (ms_frame * 1e-3) / 1e12,
                             "fp64_frac_of_peak": pairs * FP64_INST_PER_PAIR * 2 / (ms_frame * 1e-3) / 1e12 / fp64_peak}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--members", type=int, default=128)
    ap.add_argument("--T", type=float, default=1.0)
    ap.add_argument("--passes", type=int, default=2, help="timed passes of every mode (alternating)")
    ap.add_argument("--warmup", type=int, default=1, help="untimed passes of every mode of arm (a) first")
    ap.add_argument("--steps", type=int, default=20,
                    help="arm (b): steps per timed advance() (all passes stay inside the T = 2 s horizon)")
    ap.add_argument("--reps", type=int, default=5, help="arm (b): timed launches of the frame kernel")
    ap.add_argument("--arms", default="a,b")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    from optimal_crowds_b200 import _lib
    from scripts.bench_sweep import card
    if not torch.cuda.is_available():
        raise SystemExit("bench_density_stats.py measures the GPU: no CUDA device")
    torch.cuda.set_device(0)
    os.chdir(REPO)                 # config.json resolves as for the library's users
    info = card()
    peak_ctx = _lib.Context(10.0, 6.0, 0.05)
    fp64_peak = peak_ctx.fp64_peak()
    peak_ctx.close()
    lines = []
    for arm in args.arms.split(","):
        row = (arm_a if arm == "a" else arm_b)(args, fp64_peak)
        row.update(card=info, fp64_peak_tflops=fp64_peak, fp64_inst_per_pair=FP64_INST_PER_PAIR,
                   fp64_inst_source="static SASS count of density_tile (not measured)")
        lines.append(json.dumps(row))
        print(lines[-1], flush=True)
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
