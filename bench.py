#!/usr/bin/env python
"""bench.py -- headline benchmark of the two hot paths (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # our arm (B200, CUDA library)
    python bench.py --impl reference --steps K --warmup W    # CPU arm (C port of the reference's algorithm)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write what the timed steps computed to DIR/*.npy

Workload (config.workload): BASELINE.json configs[3], the slalom cylinder field.  The 16384 x 16384 grid with
100k agents is row-decomposed into bands of 2048 rows; one band (16384 x 2048 nodes, 12.5k agents, T = 2 s
-> nt = 100 field slices) is what one GPU holds, so the bench is WEAK scaling: N GPUs solve the
16384 x (2048 N) room and N = 8 is exactly configs[3].  A "step" is one full HJB solve
(optimals.compute_optimal_velocity: RK45 backward from T to 0 with dense output and the velocity epilogue).
metric = HJB Gcell-updates/s (cell-update = one RHS evaluation at one node; a solve does nfev*Ny*Nx).
The GCFM agent-steps/s figure is reported in the same JSON line under "gcfm".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)


class StdoutToStderr:
    """stdout must carry exactly ONE JSON line: while the benchmark runs, file descriptor 1 is pointed at stderr so
    that banners printed by libraries (e.g. NCCL's version line) cannot precede it; restored for the final print."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False

BAND_NX, BAND_NY, BAND_AGENTS, T_DEFAULT = 16384, 2048, 12500, 2.0
CPU_SAMPLE_NX, CPU_SAMPLE_NY, CPU_SAMPLE_T = 2048, 1024, 0.5   # per-thread sample of the multi-core CPU arm
CPU_BASELINE_T = 1.5                                            # single-core cpu_baseline sample (~12 s)


def ncu_traffic(fused=True):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the latest ncu --set full
    capture summarised under profiles/ (scripts/summarize_ncu.py); None if no capture is tracked."""
    tr_file = os.path.join(REPO, "profiles", "traffic.json")
    try:
        with open(tr_file) as f:
            tj = json.load(f)
        for tag in sorted(tj, reverse=True):
            for kname, v in tj[tag].items():
                if "hjb_" in kname and ("hjb_fused_kernel" in kname) == bool(fused):
                    return v, f"profiles/{tag}.md ({kname.strip()}, 16384x2048, per launch)"
    except Exception:
        pass
    return None, None


def load_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, interval_ms=200):
        self.index, self.rows, self.proc, self.interval_ms = index, [], None, int(interval_ms)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.interval_ms)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_hjb_sample(T=CPU_SAMPLE_T):
    """Bounded sample of the same workload on the host: the slalom room at 2048 x 1024 nodes, short horizon,
    solved by the C port of the reference's algorithm (oracle/oc_oracle_hjb.c)."""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import synthetic
    room = synthetic.slalom_room(CPU_SAMPLE_NX, CPU_SAMPLE_NY, agents=200)
    L, H = room["room_length"], room["room_height"]
    X, Y = np.linspace(0, L, CPU_SAMPLE_NX), np.linspace(0, H, CPU_SAMPLE_NY)
    V = co.create_potential(X, Y, [], [], list(room["cylinders"].values()), list(room["targets"].values()))
    V[V < 0] = -100; V[V > 0] = 1
    nt = round(T / 0.02)
    t0 = time.perf_counter()
    _, st, _, _ = co.hjb_solve(V, None, T, nt)
    dt = time.perf_counter() - t0
    cu = st["nfev"] * CPU_SAMPLE_NX * CPU_SAMPLE_NY
    return cu / dt / 1e9, dt, st, f"slalom room at {CPU_SAMPLE_NX}x{CPU_SAMPLE_NY} nodes, T={T} (nfev={st['nfev']}), {dt:.1f} s"


def cpu_gcfm_sample(n_agents=150, steps=2):
    """GCFM steps of the C port on the same sample room (full-grid wall argmin + O(N^2) pair loop, as the reference)."""
    from oracle import cpu_oracle as co
    from optimal_crowds_b200 import synthetic
    with open(os.path.join(REPO, "optimal_crowds_b200", "config.json")) as f:
        cfg = json.load(f)
    nx, ny = 1024, 512
    room = synthetic.slalom_room(nx, ny, agents=n_agents)
    L, H = room["room_length"], room["room_height"]
    X, Y = np.linspace(0, L, nx), np.linspace(0, H, ny)
    doors = np.array(list(room["targets"].values()))
    V = co.create_potential(X, Y, [], [], list(room["cylinders"].values()), doors)
    V[V < 0] = -100; V[V > 0] = 1
    P = co.gcfm_params(cfg, L, H, ny, nx)
    rng = np.random.RandomState(0)
    key = co.KeyData(V, rng.normal(size=(steps + 1, ny - 2, nx - 2)) * 0.1, rng.normal(size=(steps + 1, ny - 2, nx - 2)) * 0.1,
                     steps + 2, doors)
    st = dict(x=rng.uniform(2, L - 2, n_agents), y=rng.uniform(2, H - 2, n_agents), vx=rng.normal(0, .3, n_agents),
              vy=rng.normal(0, .3, n_agents), time=np.zeros(n_agents), status=np.ones(n_agents, dtype=np.uint8))
    vdes = rng.normal(1.34, 0.26, n_agents)
    t0 = time.perf_counter()
    for s in range(steps):
        co.gcfm_step(P, st, vdes, np.zeros(n_agents, dtype=np.int32), [key], X, Y, rng.permutation(n_agents),
                     rng.normal(size=(n_agents, 2)), s)
    dt = time.perf_counter() - t0
    return n_agents * steps / dt, f"{n_agents} agents x {steps} steps on a {nx}x{ny} grid, {dt:.1f} s"


def run_reference_arm(args):
    """CPU arm: the reference is single-threaded per solve (numpy ufuncs), so all host cores are used the way a
    user of the reference would use them -- one independent solve per core, aggregate throughput."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from concurrent.futures import ThreadPoolExecutor
    from oracle import cpu_oracle as co
    co.lib()
    cores = max(1, min(os.cpu_count() or 1, 64))
    vals, dts, last = [], [], None
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        with ThreadPoolExecutor(cores) as ex:  # ctypes releases the GIL inside the C solve
            outs = list(ex.map(lambda _: cpu_hjb_sample(), range(cores)))
        dt = time.perf_counter() - t0
        cu = sum(o[2]["nfev"] for o in outs) * CPU_SAMPLE_NX * CPU_SAMPLE_NY
        if it >= args.warmup:
            vals.append(cu / dt / 1e9); dts.append(dt)
        last = f"{cores} concurrent independent solves (one per core), each: " + outs[0][3]
    v = float(np.mean(vals))
    gc, gsample = cpu_gcfm_sample()
    line = {"impl": "reference", "metric": "hjb_gcell_updates_per_s", "value": v, "unit": "Gcell-updates/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(dts) * 1e3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "slalom (configs[3]) cylinder field; CPU arm runs a bounded sample", "sample": last},
            "cpu_baseline": {"value": v, "unit": "Gcell-updates/s", "cores": cores, "kind": "port", "sample": last},
            "e2e": {"value": v, "unit": "Gcell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gcfm": {"value": gc, "unit": "agent-steps/s", "sample": gsample, "cores": 1, "kind": "port"}}
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------- GPU arm
FP64_INST_PER_PAIR = 733.0    # FP64-pipe warp instructions per lane of one pair_force call, measured with ncu
                              # (profiles/r2_gcfm_pair_fp64.md: sm__inst_executed_pipe_fp64 of pair_probe_kernel / pairs)


def pin_numa(local_rank):
    """bind this process to the CPUs of the NUMA node its GPU hangs off (pinned host buffers are then allocated next to
    the GPU's PCIe root: 8 ranks uploading at once do not cross the socket interconnect)"""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read())
        if node < 0:
            return None
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, ids)
        return node
    except Exception:
        return None


def smooth_density(nx, rows, row0):
    """synthetic crowd density m >= 0 of the band starting at global row row0: smooth bumps, 0 <= m <= 1 (the live density
    of simulations.py:432-435 has the same range)"""
    x = np.arange(nx, dtype=np.float64) * 0.05
    y = (row0 + np.arange(rows, dtype=np.float64)) * 0.05
    return 0.5 * (1.0 + np.sin(2 * np.pi * x / 97.0)[None, :] * np.cos(2 * np.pi * y / 61.0)[:, None])


DUMP_FIELD_BYTES, DUMP_AGENT_BYTES = 48 << 20, 8 << 20   # --dump-outputs: at most 56 MB of float64 in all


def field_sample(opt):
    """--dump-outputs: what a caller of compute_optimal_velocity reads after the solve, vx_opt / vy_opt (nt-1, Ny-2, Nx-2),
    at the same fixed, seeded sample of nodes in every slice (the full field of the bench room is ~27 GB per component),
    and the solve's step counts"""
    import torch
    n_sl = opt.nt_opt - 1
    per = max(1, DUMP_FIELD_BYTES // (16 * max(n_sl, 1)))
    rng = np.random.RandomState(20240)
    ii = torch.from_numpy(rng.randint(0, opt.Ny - 2, per)).cuda()
    jj = torch.from_numpy(rng.randint(0, opt.Nx - 2, per)).cuda()
    vx = torch.empty((n_sl, per), dtype=torch.float64, device="cuda")
    vy = torch.empty_like(vx)
    for s in range(n_sl):   # slice s of vx_opt, as optimals.choose_optimal_velocity reads it
        if opt.d_vx is not None:
            sx, sy = opt.d_vx[s], opt.d_vy[s]
        else:
            sx, sy = opt._ctx.hjb_vels(opt.d_phi[opt.nt_opt - 1 - s], opt._prm)
        vx[s], vy[s] = sx[ii, jj], sy[ii, jj]
    st = opt.last_stats
    return {"hjb_vx_opt_sample": vx.cpu().numpy(), "hjb_vy_opt_sample": vy.cpu().numpy(),
            "hjb_nfev_accepted_rejected": np.array([st["nfev"], st["n_accepted"], st["n_rejected"]], dtype=np.float64)}


def agent_sample(simu):
    """--dump-outputs: the agents' state after simulation.advance() -- x, y, vx, vy, time, status and the step at which each
    agent left (-1: still inside) -- all agents, or a fixed, seeded sample of them if that would exceed DUMP_AGENT_BYTES"""
    idx = np.arange(simu.N)
    if simu.N * 7 * 8 > DUMP_AGENT_BYTES:
        idx = np.sort(np.random.RandomState(20241).choice(simu.N, DUMP_AGENT_BYTES // (7 * 8), replace=False))
    now = simu._h_now[idx]
    return {"gcfm_x": now[:, 0], "gcfm_y": now[:, 1], "gcfm_vx": now[:, 2], "gcfm_vy": now[:, 3],
            "gcfm_time": simu._h_timev[idx], "gcfm_status": simu._h_status[idx].astype(np.float64),
            "gcfm_exit_step": simu._exit_step[idx].astype(np.float64)}


def write_dump(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def parity_block(world, rank, note):
    """untimed multi-GPU parity, through the same code path the timed region used (peer-memory step kernel):
    (1) HJB: a reduced room (2048 x 256 N nodes, smooth random density > 0, a wall straddling every band edge) solved by
        the N ranks == the virtual-band solve of the whole grid done locally on every GPU, bit for bit (phi samples,
        step sizes, error norms); the single-GPU tests tie the virtual-band solve to the oracle;
    (2) GCFM: simulation(room, T, band=True) == simulation(room, T) on one GPU, bit for bit, incl. the exit order, on a
        room where agents leave in every band."""
    import contextlib, io
    import torch
    import torch.distributed as dist
    from optimal_crowds_b200 import _lib, dist as ocd, simulations, synthetic
    with open(os.path.join(REPO, "optimal_crowds_b200", "config.json")) as f:
        cfg = json.load(f)
    out = {}
    # ---- (1)
    Nx, rows, T = 2048, 256, 0.6
    Ny = rows * world
    L, H = (Nx - 1) * 0.05 + 0.025, (Ny - 1) * 0.05 + 0.025
    rng = np.random.RandomState(11)
    V = np.zeros((Ny, Nx)); V[0] = V[-1] = -100; V[:, 0] = V[:, -1] = -100
    for b in range(1, world):
        V[b * rows - 8: b * rows + 8, 100:1500] = -100       # walls straddling every band edge
        V[b * rows - 3: b * rows + 3, 1700:1760] = 1.0        # and a target cut by it
    V[Ny // 2 - 10: Ny // 2 + 10, -1] = 1.0; V[0, 20:40] = 1.0
    m = 0.2 + 0.8 * rng.uniform(0, 1, (Ny, Nx))
    m = 0.25 * (m + np.roll(m, 1, 0) + np.roll(m, 1, 1) + np.roll(m, -1, 0))
    nt = round(T / 0.02)
    ctx = _lib.Context(L, H, 0.05)
    own0, own1 = ocd.init_context(ctx)
    prm = _lib.hjb_params(cfg, fused=1, chunk_rows=32)
    res = ctx.hjb_solve_band(ctx.to_device(V[own0:own1]), ctx.to_device(m[own0:own1]), prm, T, nt, own=(own0, own1),
                             trace=True)
    ctx2 = _lib.Context(L, H, 0.05)
    ref = ctx2.hjb_solve_band(ctx2.to_device(V), ctx2.to_device(m), prm, T, nt, n_virtual=world, trace=True)
    ok = np.array_equal(res["trace_h"], ref["trace_h"]) and np.array_equal(res["trace_err"], ref["trace_err"])
    ok = ok and torch.equal(res["phi"][:, 1:-1], ref["phi"][:, own0:own1])
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["hjb_bitwise"] = bool(flag.item() == 1)
    out["hjb_case"] = (f"{Nx}x{Ny} nodes, T={T}, {len(res['trace_h'])} attempts, peer-memory exchange: "
                       f"{bool(getattr(ctx, 'peer_memory', False))}")
    del res, ref
    ctx.close(); ctx2.close()
    # ---- (2)
    room = synthetic.parity_room(2048, 256 * world, world)

    def run(band):
        np.random.seed(5)
        with contextlib.redirect_stdout(io.StringIO()):
            simu = simulations.simulation(room, 1.7, record=False, chunk_rows=32, band=band)
            simu._solve_all()
            for _ in range(80):
                simu.step(simu.dt)
        return simu

    a, b = run(True), run(False)
    ok_state = np.array_equal(a._h_now, b._h_now) and np.array_equal(a._h_timev, b._h_timev) and a.inside == b.inside
    ok_order = a._exit_order == b._exit_order and len(a._exit_order) > 0
    own = a._band
    exits_by_band = np.bincount(np.clip((a._h_now[a._exit_order, 1] / 0.05).astype(int) // (256), 0, world - 1),
                                minlength=world) if a._exit_order else np.zeros(world, dtype=int)
    flag = torch.tensor([1 if ok_state else 0, 1 if ok_order else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["gcfm_bitwise"] = bool(flag[0].item() == 1)
    out["gcfm_exit_order"] = bool(flag[1].item() == 1)
    out["gcfm_case"] = (f"{a.N} agents, 80 steps, {len(a._exit_order)} exits (per band: {exits_by_band.tolist()}), "
                        f"band rows {own}")
    note(f"parity: {out}")
    a._ctx.close(); b._ctx.close()
    return out


def run_slalom(args, world, rank, local_rank):
    """BASELINE configs[3] through the drop-in API: simulations.simulation(room, T) on one GPU, and
    simulations.simulation(room, T, band=True) under torchrun -- the same room row-decomposed over N GPUs."""
    import contextlib, io
    import torch
    import torch.distributed as dist
    from optimal_crowds_b200 import _lib, simulations, synthetic
    W, K = max(args.warmup, 0), args.steps
    nx, ny = args.nx, args.band_ny
    Ny = ny * world
    t_start = time.perf_counter()

    def note(msg):
        if rank == 0:
            print(f"[bench {time.perf_counter() - t_start:7.1f}s] {msg}", file=sys.stderr, flush=True)

    if world > 1 and os.environ.get("OC_BENCH_PARITY_ONLY"):  # development aid: only the untimed parity block
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ.get("OC_BENCH_WATCHDOG", "120")), exit=True)
        par = parity_block(world, rank, note)
        dist.destroy_process_group()
        return 0 if all(v for k, v in par.items() if isinstance(v, bool)) else 1
    numa = pin_numa(local_rank)
    room = synthetic.slalom_room(nx, Ny, agents=args.agents * world)
    np.random.seed(1000)   # every rank of a row-decomposed run uses the same seed (replicated, deterministic sweep)
    with contextlib.redirect_stdout(io.StringIO()):
        kw = dict(band=True) if world > 1 else {}
        if args.field != "phi":
            kw["field_storage"] = args.field
        # (record: the API default on one GPU -- the run loop then executes blocks of steps inside one library call)
        simu = simulations.simulation(room, args.T, recompute=False, record=world == 1, fused=args.fused, **kw)
    note(f"simulation built: N={simu.N} agents, grid {simu.Ny}x{simu.Nx}, keys={len(simu.targets)}, numa node {numa}")
    opt = list(simu.targets.values())[0]
    opt._prm.profile = 1
    cells = nx * Ny
    own0 = simu._band[0] if simu._band else 0
    # density input of the solve, m >= 0 and smooth: this rank's rows, as a pinned HOST array (the reference-facing
    # signature takes a numpy array) and as a device copy
    m_host = torch.from_numpy(smooth_density(nx, ny, own0)).pin_memory()
    m_dev = m_host.to("cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def solve(m):
        with contextlib.redirect_stdout(io.StringIO()):
            opt.compute_optimal_velocity(0.0, m)
        return opt.last_stats

    # ---- device-resident timing: inputs already in HBM ------------------------------------------
    for _ in range(W):
        solve(m_dev)
    barrier()
    note(f"warm-up done: {opt.last_stats}")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _lib.launch_count(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cls_ms, cls_bytes, cls_n = np.zeros(3), np.zeros(3), np.zeros(3)
    nfev_total = 0
    barrier()
    ev0.record()
    for _ in range(K):
        st = solve(m_dev)
        nfev_total += st["nfev"]
        cls_ms += st["cls_ms"]; cls_bytes += st["cls_bytes"]; cls_n += st["cls_launches"]
    ev1.record()
    barrier()
    launches = _lib.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    ms_max, step_ms_max = allmax([ev0.elapsed_time(ev1), cls_ms[0]])
    value = nfev_total * cells / (ms_max * 1e-3) / 1e9
    note(f"device-resident: {value:.2f} Gcu/s, {ms_max / K:.1f} ms/solve")
    dump = field_sample(opt) if args.dump_outputs else None   # the field of the last timed solve, before e2e overwrites it

    # ---- end to end: host m -> H2D, solve, D2H of a scalar checksum of the t = 0 field slice ----------
    def checksum():
        if opt.d_vx is not None:
            return float(opt.d_vx[0].sum().item())
        sl = opt.d_phi[opt.nt_opt - 1]
        return float((sl[1:-2] if simu._band else sl).sum().item())

    # every step gets its input from a different page-locked host buffer, uploaded inside the timed region
    m_hosts = [m_host.numpy(), torch.from_numpy(smooth_density(nx, ny, own0)[::-1].copy()).pin_memory().numpy()]
    for it in range(max(min(W, 2), 1)):  # warm-up of the whole e2e step (first use of the reduction loads its module)
        solve(m_hosts[it % 2])
        checksum()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nfev_e2e = 0
    opt._prefetched = None
    t_wall = time.perf_counter()
    e0.record()
    for it in range(K):
        if it + 1 < K and os.environ.get("OC_BENCH_PREFETCH"):
            # optional (measured slower, see DESIGN.md section 5): start the H2D of the next step's input so that it
            # overlaps this solve
            opt.prefetch_density(m_hosts[(it + 1) % 2])
        st = solve(m_hosts[it % 2])                        # uploads its input (one DMA from page-locked memory), solves
        nfev_e2e += st["nfev"]
        chk = checksum()
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    e2e_ms, = allmax([max(e0.elapsed_time(e1), wall_ms)])
    e2e_value = nfev_e2e * cells / (e2e_ms * 1e-3) / 1e9
    note(f"e2e: {e2e_value:.2f} Gcu/s")

    # ---- GCFM: agent-steps/s through simulation.step (host RNG + H2D + sweep + exit log D2H) -----------
    fp64_peak = simu._ctx.fp64_peak()
    agent_steps, dev_ms, pairs = 0, 0.0, 0
    if world == 1:
        # the body of simulation.run()'s loop (history frame + step) through the public block call it uses
        simu.advance(3)
        barrier()
        g0 = time.perf_counter()
        n0, s0 = int(simu._h_status.sum()), simu.simu_step
        done = simu.advance(args.gcfm_steps)
        ex = simu._exit_step[simu._exit_step >= s0]
        agent_steps = sum(n0 - int((ex < s0 + k).sum()) for k in range(done))
        dev_ms, pairs = simu.last_run_stats["device_ms"], simu.last_run_stats["pairs"]
        args.gcfm_steps = max(done, 1)
    else:
        for _ in range(3):
            simu.step(simu.dt)
        barrier()
        g0 = time.perf_counter()
        for _ in range(args.gcfm_steps):
            agent_steps += int(simu._h_status.sum())
            simu.step(simu.dt)
            dev_ms += simu._ctx.gcfm_last_ms()
            pairs += simu._ctx.gcfm_last_pairs()
    barrier()
    g_wall, g_dev = allmax([time.perf_counter() - g0, dev_ms * 1e-3])
    if dump is not None:
        dump.update(agent_sample(simu))
        write_dump(args.dump_outputs, dump)
        note(f"outputs written to {args.dump_outputs}: {sorted(dump)}")
    pair_tflops = pairs * FP64_INST_PER_PAIR * 2.0 / g_dev / 1e12   # FMA-equivalent flops of the FP64-pipe instructions
    gcfm = {"metric": "gcfm_agent_steps_per_s", "value": agent_steps / g_dev, "unit": "agent-steps/s",
            "e2e_value": agent_steps / g_wall, "agents": simu.N, "steps": args.gcfm_steps,
            "ms_per_step": g_dev * 1e3 / args.gcfm_steps, "pairs_per_step": pairs / args.gcfm_steps,
            "roofline": {"bound": "fp64", "unit": "TFLOP/s", "peak": fp64_peak,
                         "peak_source": "measured here (oc_fp64_peak: 8 independent DFMA chains x 16 warps/SM)",
                         "achieved": pair_tflops, "frac": pair_tflops / fp64_peak,
                         "work": f"{FP64_INST_PER_PAIR:.0f} FP64-pipe instructions per interacting pair (ncu) x pairs; the "
                                 "sweep is a dependency chain (sequential-sweep semantics), so the pipe is latency- not "
                                 "throughput-bound"},
            "note": ("value = CUDA-event time of oc_gcfm_step (H2D perm/noise + kernels + exit log); e2e_value = wall clock of "
                     "simulation.advance(steps), the block call of simulation.run(): legacy-RNG draws, staging, sweep, exit "
                     "bookkeeping, trajectory record, history frames; parity mode (sequential-sweep semantics, host RNG stream)"
                     + ("; ONE room of %d agents on %d GPUs: field samples and wall searches sharded by row band, the "
                        "sweep replicated on every rank (a room's sweep is one dependency chain)" % (simu.N, world)
                        if world > 1 else ""))}
    note(f"gcfm: {gcfm['value']:.0f} agent-steps/s device, {gcfm['e2e_value']:.0f} e2e, fp64 peak {fp64_peak:.1f} TF/s")

    parity = None
    if world > 1:
        del m_dev
        for o in simu.targets.values():
            o.d_phi = None
        torch.cuda.empty_cache()
        parity = parity_block(world, rank, note)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0 if (parity is None or all(v for k, v in parity.items() if isinstance(v, bool))) else 1
    peak, peak_src = load_peaks()
    dom = 0  # RK step kernels
    band_cells = nx * ny
    if cls_bytes[dom] == 0:  # the row-band solver reports times only: 40 B/cell/attempt + 8 B/cell/emitted phi slice
        cls_bytes[dom] = 40.0 * band_cells * ((nfev_total - 2 * K) // 6) + 8.0 * band_cells * round(args.T / 0.02) * K
    achieved = cls_bytes[dom] / (step_ms_max * 1e-3) / 1e9 if step_ms_max > 0 else 0.0
    p2p = bool(getattr(simu._ctx, "peer_memory", False))
    roof = {"bound": "hbm", "kernel": "hjb_stage_kernel<N,MODE> (RK45 stage: combination + stencil [+ y_new, error])"
            if not args.fused else "fused::hjb_fused_kernel<NE> (TMA-staged stage-fused RK45 step)", "achieved": achieved,
            "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs: 1:1 copy; a streaming kernel with this kernel's 3-read : "
            "5-write mix reaches 0.92 of it, profiles/r2_hbm_mix.md)" if peak_src == "measured" else "fallback (B200_PROFILING.md)",
            "traffic": None, "launches": int(cls_n[dom]), "avg_launch_ms": float(step_ms_max / max(cls_n[dom], 1)),
            "algorithmic_bytes_per_launch": float(cls_bytes[dom] / max(cls_n[dom], 1)),
            "share_of_step": float(step_ms_max / ms_max) if ms_max > 0 else None,
            "other_classes": {"dense_output+velocity": {"ms": float(cls_ms[1]), "launches": int(cls_n[1])},
                              "reductions": {"ms": float(cls_ms[2]), "launches": int(cls_n[2])}}}
    if world > 1:
        roof["note"] = ("the launch contains the halo exchange (NVLink peer stores) and the cross-GPU error-sum all-gather: its "
                        "duration includes waiting for the slowest rank") if p2p else \
                       "halo exchange and all-gather run as an NCCL group after the launch"
    roof["traffic"], roof["traffic_source"] = ncu_traffic(args.fused)
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        g, dt, stc, sample = cpu_hjb_sample(CPU_BASELINE_T)
        cpu = {"value": g, "unit": "Gcell-updates/s", "cores": 1, "kind": "port", "sample": sample}
        try:
            gc, gsample = cpu_gcfm_sample(n_agents=300, steps=4)
            gcfm["cpu_baseline"] = {"value": gc, "unit": "agent-steps/s", "cores": 1, "kind": "port", "sample": gsample}
        except Exception as e:  # pragma: no cover
            gcfm["cpu_baseline"] = {"error": str(e)}
    api = "simulations.simulation(room, T" + (", band=True" if world > 1 else "") + ") -> targets[key].compute_optimal_velocity(t, m)"
    line = {"metric": "hjb_gcell_updates_per_s", "value": value, "unit": "Gcell-updates/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"slalom (BASELINE configs[3]) cylinder field, {nx}x{Ny} grid "
                                   f"({nx}x{ny} band per GPU; N=8 is the 16384^2 / 100k-agent config), T={args.T} "
                                   f"(nt={round(args.T / 0.02)} slices), {args.agents * world} agents, smooth density input "
                                   "0 <= m <= 1",
                       "parallelism": "1 GPU" if world == 1 else
                       (f"one room, row bands over {world} GPUs; halo rows (6 of y_new, f_new per side) and the per-chunk error "
                        "sums are exchanged INSIDE the step launch as NVLink peer stores (CUDA IPC), NCCL only at solve start"
                        if p2p else f"one room, row bands over {world} GPUs, NCCL halo exchange + all-gather per attempt"),
                       "l2": "inputs larger than L2 (each field 268 MB > 126 MB)", "formulation":
                       "stage-wise RK45 (52 B/cell-update)" if not args.fused else
                       "stage-fused RK45 step (40 B/cell/attempt + 8 B/cell/emitted phi slice)",
                       "field_storage": opt.field_storage + " (the API default)", "api": api,
                       "nfev_per_solve": nfev_total // K},
            "e2e": {"value": e2e_value, "unit": "Gcell-updates/s", "h2d_bytes_per_step": int(m_host.numel() * 8) * world,
                    "d2h_bytes_per_step": 8 * world, "checksum": chk,
                    "api": api + " with m a pinned host numpy array (every step a different buffer, one DMA per step inside the "
                           "timed region); the result stays on the device (it is the GCFM sampler's input), the read-back is a "
                           "checksum of the t = 0 slice"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "gcfm": gcfm}
    if parity is not None:
        line["parity"] = parity
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0 if (parity is None or all(v for k, v in parity.items() if isinstance(v, bool))) else 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="slalom", choices=["slalom", "metro", "ensemble"],
                    help="slalom = BASELINE configs[3] (the headline line); metro = configs[2]; ensemble = configs[4]")
    ap.add_argument("--T", type=float, default=None)
    ap.add_argument("--band-ny", type=int, default=BAND_NY)
    ap.add_argument("--nx", type=int, default=BAND_NX)
    ap.add_argument("--agents", type=int, default=BAND_AGENTS)
    ap.add_argument("--gcfm-steps", type=int, default=50)
    ap.add_argument("--rooms", type=int, default=1024, help="ensemble: members in total (sharded over the GPUs)")
    ap.add_argument("--fused", type=int, default=int(os.environ.get("OC_FUSED", "1")),
                    help="1: stage-fused RK45 step kernel (default), 0: one kernel per RK stage")
    ap.add_argument("--field", default=os.environ.get("OC_FIELD", "phi"), choices=["phi", "velocity"],
                    help="field storage: phi samples (API default; sampler differentiates) or vx/vy slices")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed as DIR/<name>.npy (float64, <= 56 MB): a fixed, "
                         "seeded sample of vx_opt / vy_opt of the last timed HJB solve, its step counts, and the agents' "
                         "state after the timed GCFM steps (slalom workload on one GPU)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "slalom" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs supports the slalom workload of the CUDA library on one GPU")
    if args.impl == "reference":
        if args.T is None:
            args.T = T_DEFAULT
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.workload == "metro":
        from scripts import bench_workloads
        return bench_workloads.run_metro(args, world, rank, local_rank)
    if args.workload == "ensemble":
        from scripts import bench_workloads
        return bench_workloads.run_ensemble(args, world, rank, local_rank)
    if args.T is None:
        args.T = T_DEFAULT
    return run_slalom(args, world, rank, local_rank)


_EMITTED = []


def emit(text):
    """JSON lines of the workloads in scripts/bench_workloads.py: collected in the process-wide `bench` module the
    workloads import, and printed by the __main__ block once stdout has been restored"""
    _EMITTED.append(text)


if __name__ == "__main__":
    _lines = []
    _real_print = print

    def print(*a, **k):  # noqa: A001 -- JSON lines are collected and emitted after stdout is restored
        if k.get("file") is None:
            _lines.append(" ".join(str(x) for x in a))
        else:
            _real_print(*a, **k)

    with StdoutToStderr():
        _rc = main()
    # scripts/bench_workloads.py imports this file as module `bench` (here it runs as __main__): its lines are there
    _extra = list(getattr(sys.modules.get("bench"), "_EMITTED", [])) if "bench" in sys.modules else []
    for _l in _lines + _extra:
        _real_print(_l, flush=True)
    sys.exit(_rc)
