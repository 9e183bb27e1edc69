"""Ensembles over room layouts on one GPU: what mixing grid shapes in one ensemble costs and saves.

Three arms, run alternately in one process after a warm-up pass of each, T = 2 s, periodic re-solves (``recompute=True``):
  A  128 members of the configs[4] room (``synthetic.ensemble_room(512, 1000)``)           -- one shape
  B  128 members over 8 shapes in ONE ensemble: square rooms of 384, 416, 448, 480, 544, 608 nodes and two rectangular
     ones (384 x 640, 448 x 576), 16 members each, 1000 agents each                       -- one batched solve per step
  C  the members of B as 8 single-shape ensembles run one after the other                 -- what a user had to do before
One JSON line per arm: seconds per pass, HJB Gcell-updates/s over the solve calls, GCFM agent-steps/s over the rest of
the run loop, batched solve calls per pass, and the card's name and power limit read in the same run.

    python scripts/bench_shapes.py [--members 128] [--T 2.0] [--passes 2] [--warmup 1] [--arms A,B,C] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

SHAPES = [(384, 384), (416, 416), (448, 448), (480, 480), (544, 544), (608, 608), (384, 640), (448, 576)]  # (ny, nx)


def shaped_room(ny, nx, agents=1000):
    """the configs[4] room on an (ny, nx) grid: one door on the right wall, 3 cylinders, one square box of `agents` --
    20 x 20 m (2.5 ped/m^2) as in ensemble_room, or 70 % of the shorter side where the room is too small for that"""
    from optimal_crowds_b200 import synthetic
    L, H = synthetic.nodes_to_length(nx), synthetic.nodes_to_length(ny)
    room = synthetic.ensemble_room(512, agents)
    side = min(20.0, 0.7 * min(L, H))
    room.update(room_length=L, room_height=H)
    room["initial_boxes"]["box"] = [L / 2 - 1.5, H / 2, side, side, (agents + 0.5) / side ** 2, "door"]
    room["targets"]["door"] = [L, H / 2, 0.6, 2.0]
    room["cylinders"] = {"c1": [L - 2.0, H / 2 + 2.0, 0.3], "c2": [L - 2.0, H / 2 - 2.0, 0.3], "c3": [L - 3.5, H / 2, 0.3]}
    return room


def run_ensembles(groups, T):
    """run the (rooms, seeds) groups as one ensemble each, one after the other; summed stats, results, wall seconds"""
    import torch
    from optimal_crowds_b200 import ensemble
    stats, res = {}, {}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for rooms, seeds in groups:
        ens = ensemble.ensemble(rooms, T, seeds, recompute=True, max_wave=128)
        for i, r in ens.run(gather=False).items():
            res[seeds[i]] = r
        for k, v in ens.stats.items():
            stats[k] = stats.get(k, 0) + v
    torch.cuda.synchronize()
    return stats, res, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--members", type=int, default=128)
    ap.add_argument("--T", type=float, default=2.0)
    ap.add_argument("--passes", type=int, default=2, help="timed passes of every arm (alternating)")
    ap.add_argument("--warmup", type=int, default=1, help="untimed passes of every arm first")
    ap.add_argument("--arms", default="A,B,C", help="which arms to run (A alone also runs on builds without mixed shapes)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    from optimal_crowds_b200 import synthetic
    from scripts.bench_sweep import card
    if not torch.cuda.is_available():
        raise SystemExit("bench_shapes.py measures the GPU: no CUDA device")
    torch.cuda.set_device(0)
    os.chdir(REPO)                 # config.json resolves as for the library's users
    n = args.members
    seeds = list(range(n))
    mixed_rooms = [shaped_room(*SHAPES[i % len(SHAPES)]) for i in range(n)]
    plan = {
        "A_one_shape": [([synthetic.ensemble_room(512, 1000)] * n, seeds)],
        "B_8_shapes_one_ensemble": [(mixed_rooms, seeds)],
        "C_8_shapes_in_sequence": [([mixed_rooms[i] for i in seeds[s::len(SHAPES)]], seeds[s::len(SHAPES)])
                                   for s in range(len(SHAPES))],
    }
    plan = {name: g for name, g in plan.items() if name[0] in args.arms.split(",")}
    for _ in range(args.warmup):
        for groups in plan.values():
            run_ensembles(groups, args.T)
    keys = ("hjb_call_ms", "hjb_ms", "gcfm_ms", "cell_updates", "agent_steps", "hjb_calls")
    acc = {name: dict({k: 0.0 for k in keys}, wall_s=[], res=None) for name in plan}
    for _ in range(args.passes):
        for name, groups in plan.items():
            st, res, wall = run_ensembles(groups, args.T)
            a = acc[name]
            for k in keys:
                a[k] += st.get(k, 0)
            a["wall_s"].append(wall)
            a["res"] = res
    # B and C run the same members: their results must agree bit for bit
    same = None
    if "B_8_shapes_one_ensemble" in acc and "C_8_shapes_in_sequence" in acc:
        rb, rc = acc["B_8_shapes_one_ensemble"]["res"], acc["C_8_shapes_in_sequence"]["res"]
        same = sorted(rb) == sorted(rc) and all(
            rb[i]["steps"] == rc[i]["steps"] and (rb[i]["final"] == rc[i]["final"]).all() for i in rb)
    gpu = card()
    lines = []
    for name, a in acc.items():
        loop_ms = a["hjb_ms"] + a["gcfm_ms"] - a["hjb_call_ms"]
        lines.append({
            "arm": name, "members": n, "T": args.T, "passes": args.passes, "warmup": args.warmup,
            "s_per_pass": sum(a["wall_s"]) / len(a["wall_s"]), "s_per_pass_min": min(a["wall_s"]),
            "s_per_pass_max": max(a["wall_s"]),
            "hjb_gcell_updates_per_s": a["cell_updates"] / (a["hjb_call_ms"] * 1e-3) / 1e9,
            "gcfm_agent_steps_per_s": a["agent_steps"] / (loop_ms * 1e-3),
            "solve_calls_per_pass": a["hjb_calls"] / args.passes,
            "b_equals_c": same, "gpu": gpu,
            "workload": "A: synthetic.ensemble_room(512, 1000); B, C: shaped_room over %s; seeds 0..%d, recompute=True, "
                        "max_wave=128" % (SHAPES, n - 1)})
    for line in lines:
        print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
