"""Parameter-sweep ensembles on one GPU: what per-member configurations cost (``ensemble(..., configs=...)``).

Four arms, run alternately in one process after a warm-up pass of each, 128 members of the configs[4] room
(``synthetic.ensemble_room(512, 1000)``), T = 2 s, periodic re-solves (``recompute=True``):
  a  configs=None                      -- every member runs config.json
  b  128 identical ``{}`` overrides    -- the configuration path with nothing to change
  c  g swept over 128 values in [-0.05, 0]
  d  dt alternating 0.02 / 0.01        -- members re-solve at different iterations, so the re-solve batches split
One JSON line per arm: seconds per pass, HJB Gcell-updates/s over the solve calls, GCFM agent-steps/s over the rest of
the run loop, batched solve calls per pass (the solve at t = 0 included) and rooms per call, and the card's name and
power limit read in the same run.

    python scripts/bench_sweep.py [--members 128] [--T 2.0] [--passes 3] [--warmup 1] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def card():
    """name, power limit and max SM clock of cuda:0 (nvidia-smi queries only; None where unavailable)"""
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, mhz = (v.strip() for v in out.strip().splitlines()[0].split(","))
        info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(mhz)
    except Exception:
        pass
    return info


def arms(n):
    import numpy as np
    gs = np.linspace(-0.05, 0.0, n)
    return {"a_none": None,
            "b_identical": [{} for _ in range(n)],
            "c_g_sweep": [{"hjb_params": {"g": float(g)}} for g in gs],
            "d_dt_alternating": [{"dt": 0.02 if i % 2 == 0 else 0.01} for i in range(n)]}


def one_pass(room, T, n, configs):
    import torch
    from optimal_crowds_b200 import ensemble
    ens = ensemble.ensemble(room, T, list(range(n)), recompute=True, max_wave=128, configs=configs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = ens.run(gather=False)
    torch.cuda.synchronize()
    return ens.stats, res, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--members", type=int, default=128)
    ap.add_argument("--T", type=float, default=2.0)
    ap.add_argument("--passes", type=int, default=3, help="timed passes of every arm (alternating)")
    ap.add_argument("--warmup", type=int, default=1, help="untimed passes of every arm first")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    from optimal_crowds_b200 import synthetic
    if not torch.cuda.is_available():
        raise SystemExit("bench_sweep.py measures the GPU: no CUDA device")
    torch.cuda.set_device(0)
    os.chdir(REPO)                 # config.json and rooms resolve as for the library's users
    room = synthetic.ensemble_room(512, 1000)
    plan = arms(args.members)
    for _ in range(args.warmup):
        for cfgs in plan.values():
            one_pass(room, args.T, args.members, cfgs)
    keys = ("hjb_call_ms", "hjb_ms", "gcfm_ms", "build_ms", "cell_updates", "agent_steps", "hjb_calls", "hjb_call_rooms")
    acc = {name: dict({k: 0.0 for k in keys}, wall_s=[], evac=None) for name in plan}
    for _ in range(args.passes):
        for name, cfgs in plan.items():
            st, res, wall = one_pass(room, args.T, args.members, cfgs)
            a = acc[name]
            for k in keys:
                a[k] += st.get(k, 0)
            a["wall_s"].append(wall)
            a["evac"] = [res[i]["evac_time"] for i in sorted(res)[:4]]
    gpu = card()
    lines = []
    for name, a in acc.items():
        # solve calls: host clock around each batched call, which ends in a device synchronise; the GCFM run loop is the
        # rest of the time after the first solve (hjb_ms: the first solve, gcfm_ms: the run loop incl. re-solves)
        loop_ms = a["hjb_ms"] + a["gcfm_ms"] - a["hjb_call_ms"]
        lines.append({
            "arm": name, "members": args.members, "T": args.T, "passes": args.passes, "warmup": args.warmup,
            "s_per_pass": sum(a["wall_s"]) / len(a["wall_s"]), "s_per_pass_min": min(a["wall_s"]),
            "s_per_pass_max": max(a["wall_s"]),
            "hjb_gcell_updates_per_s": a["cell_updates"] / (a["hjb_call_ms"] * 1e-3) / 1e9,
            "gcfm_agent_steps_per_s": a["agent_steps"] / (loop_ms * 1e-3),
            "solve_calls_per_pass": a["hjb_calls"] / args.passes,
            "rooms_per_solve_call": a["hjb_call_rooms"] / max(a["hjb_calls"], 1),
            "first_evac_times": a["evac"], "gpu": gpu,
            "workload": "synthetic.ensemble_room(512, 1000), seeds 0..%d, recompute=True, max_wave=128" % (args.members - 1)})
    for line in lines:
        print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
