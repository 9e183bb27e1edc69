"""ctypes binding of liboc_b200.so (include/optimal_crowds.h).

The library is built in-tree by optimal_crowds_b200/build.py.  There is no CPU fallback: if the shared
object is missing, or no CUDA device is present when a compute entry point is called, this raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# OC_B200_LIB: alternative build of the same library (kernel-variant experiments, scripts/build_variants.sh)
LIB_PATH = os.environ.get("OC_B200_LIB") or os.path.join(_HERE, "liboc_b200.so")

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)
u8p = C.POINTER(C.c_uint8)


class OcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liboc_b200 error {code}: {msg}")
        self.code = code


OC_ERR_SAMPLER_RANGE = -4
OC_ERR_STEP_TOO_SMALL = -5


class HjbParams(C.Structure):
    _fields_ = [("sigma", C.c_double), ("mu", C.c_double), ("g", C.c_double), ("rtol", C.c_double),
                ("atol", C.c_double), ("lim", C.c_double), ("fused", C.c_int), ("profile", C.c_int),
                ("forced_h", dp), ("n_forced_h", C.c_int), ("chunk_rows", C.c_int)]

    def force_steps(self, h):
        """teacher-forced controller: replay the signed step sequence `h` (parity tests; see optimal_crowds.h)"""
        if h is None:
            self._keep = None
            self.forced_h, self.n_forced_h = None, 0
        else:
            self._keep = np.ascontiguousarray(h, dtype=np.float64)
            self.forced_h, self.n_forced_h = self._keep.ctypes.data_as(dp), len(self._keep)
        return self


class HjbStats(C.Structure):
    _fields_ = [("nfev", C.c_int), ("n_accepted", C.c_int), ("n_rejected", C.c_int), ("status", C.c_int),
                ("n_out", C.c_int), ("launches", C.c_int), ("h0", C.c_double), ("gpu_ms", C.c_double),
                ("cls_launches", C.c_int * 3), ("pad_", C.c_int), ("cls_ms", C.c_double * 3),
                ("cls_bytes", C.c_double * 3)]

    def asdict(self):
        d = {f: getattr(self, f) for f, _ in self._fields_ if not f.startswith(("cls_", "pad_"))}
        for f in ("cls_launches", "cls_ms", "cls_bytes"):
            d[f] = list(getattr(self, f))
        return d


class HjbRoom(C.Structure):
    _fields_ = [("sigma", C.c_double), ("mu", C.c_double), ("g", C.c_double), ("T", C.c_double), ("t_eval", dp),
                ("nt", C.c_int), ("chunk_rows", C.c_int)]


class BandCfg(C.Structure):
    _fields_ = [("n_virtual", C.c_int), ("own0", C.c_int), ("own1", C.c_int), ("phi_extra_hi", C.c_int)]


class GcfmParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in
                ("dt", "dt2", "half_noise", "relaxation", "v_max", "cutoff", "a_min", "tau_a", "b_min", "b_max",
                 "eta", "eta_walls", "cos_fov", "one_minus_cos_fov", "dx", "dy", "room_length", "room_height")] + \
               [("Ny", C.c_int), ("Nx", C.c_int), ("own0", C.c_int), ("own1", C.c_int), ("key_mod", C.c_int),
                ("key_rem", C.c_int)]


class Key(C.Structure):
    _fields_ = [("d_V", C.c_void_p), ("d_wall_tiles", C.c_void_p), ("v_min", C.c_double), ("d_vx", C.c_void_p),
                ("d_vy", C.c_void_p), ("nt_opt", C.c_int), ("n_slices", C.c_int), ("d_phi", C.c_void_p),
                ("n_phi", C.c_int), ("pad_", C.c_int), ("mu", C.c_double), ("lim", C.c_double), ("doors", dp),
                ("n_doors", C.c_int), ("phi_row0", C.c_int), ("phi_rows", C.c_int)]


_lib = None

EXPORTS = ["oc_abi_version", "oc_last_error", "oc_launch_count", "oc_ctx_create", "oc_ctx_destroy", "oc_ctx_set_int", "oc_rasterise",
           "oc_hjb_solve", "oc_hjb_rhs", "oc_hjb_vels", "oc_wall_tiles_bytes", "oc_wall_tiles", "oc_gcfm_step",
           "oc_wall_force", "oc_pair_force", "oc_density", "oc_gcfm_last_ms", "oc_dist_unique_id", "oc_dist_init",
           "oc_dist_finalize", "oc_dist_p2p_export", "oc_dist_p2p_import", "oc_dist_p2p_enabled", "oc_dist_p2p_disable", "oc_hjb_solve_band", "oc_rasterise_band", "oc_upload", "oc_hjb_solve_batch", "oc_hjb_solve_multi", "oc_hjb_solve_grids", "oc_gcfm_step_launch",
           "oc_gcfm_step_finish", "oc_gcfm_last_pairs", "oc_gcfm_last_redos", "oc_state_pack", "oc_fp64_peak", "oc_place_box", "oc_hjb_plan_chunk_rows", "oc_rng_step_draw", "oc_rng_step_draw_ckpt", "oc_gcfm_step_multi_launch", "oc_gcfm_step_multi_finish", "oc_gcfm_run"]


def load():
    """Load the shared library (raises if it has not been built -- there is no fallback path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build it with `python -m optimal_crowds_b200.build` "
                          "(the CUDA library is the only implementation; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.oc_last_error.restype = C.c_char_p
    lib.oc_launch_count.restype = C.c_longlong
    lib.oc_wall_tiles_bytes.restype = C.c_longlong
    lib.oc_gcfm_last_ms.restype = C.c_double
    lib.oc_gcfm_last_ms.argtypes = [C.c_void_p]
    lib.oc_gcfm_last_pairs.restype = C.c_longlong
    lib.oc_gcfm_last_pairs.argtypes = [C.c_void_p]
    lib.oc_gcfm_last_redos.argtypes = [C.c_void_p]
    lib.oc_state_pack.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 6
    lib.oc_fp64_peak.argtypes = [C.c_void_p, dp]
    lib.oc_hjb_plan_chunk_rows.argtypes = [C.c_void_p, C.c_int]
    vpp_ = C.POINTER(C.c_void_p)
    lib.oc_gcfm_step_multi_launch.argtypes = [C.c_int, vpp_, vpp_, ip] + [vpp_] * 9 + [ip, vpp_, ip, ip, dp, ip, ip,
                                                                                     C.c_int, C.c_void_p]
    lib.oc_gcfm_step_multi_finish.argtypes = [C.c_int, vpp_, vpp_, ip, ip]
    lib.oc_gcfm_run.argtypes = [C.c_void_p, C.POINTER(GcfmParams), C.c_int] + [C.c_void_p] * 8 + [C.c_void_p, C.c_int,
                                C.POINTER(C.c_uint32), ip, ip, dp, C.c_int, C.c_int, C.c_int, vpp_, ip, ip, ip, ip, dp,
                                C.POINTER(C.c_longlong), C.c_void_p]
    lib.oc_rng_step_draw.argtypes = [C.POINTER(C.c_uint32), ip, ip, dp, C.c_int, C.c_int, ip, dp]
    lib.oc_rng_step_draw_ckpt.argtypes = [C.POINTER(C.c_uint32), ip, ip, dp, C.c_int, C.c_int, ip, dp, C.c_int,
                                          C.POINTER(C.c_uint32), ip, ip, dp]
    lib.oc_place_box.restype = C.c_longlong
    lib.oc_place_box.argtypes = [dp, dp, C.c_int, dp, C.c_int, dp, C.c_double, C.POINTER(C.c_uint32), ip, dp, dp, C.c_int]
    lib.oc_wall_tiles_bytes.argtypes = [C.c_void_p]
    lib.oc_ctx_set_int.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    lib.oc_ctx_destroy.restype = None
    lib.oc_ctx_destroy.argtypes = [C.c_void_p]
    lib.oc_ctx_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, dp, dp,
                                  C.POINTER(C.c_void_p)]
    lib.oc_rasterise.argtypes = [C.c_void_p, dp, C.c_int, dp, C.c_int, dp, C.c_int, dp, C.c_int, C.c_int, C.c_double,
                                 C.c_double, C.c_void_p, C.c_void_p]
    lib.oc_hjb_solve.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(HjbParams), C.c_double, dp, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(HjbStats), dp, dp, C.c_int, ip,
                                 C.c_void_p]
    lib.oc_hjb_solve_band.argtypes = [C.c_void_p, C.POINTER(BandCfg), C.c_void_p, C.c_void_p, C.POINTER(HjbParams),
                                      C.c_double, dp, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(HjbStats),
                                      dp, dp, C.c_int, ip, C.c_void_p]
    lib.oc_rasterise_band.argtypes = [C.c_void_p, dp, C.c_int, dp, C.c_int, dp, C.c_int, dp, C.c_int, C.c_int,
                                      C.c_double, C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    vpp = C.POINTER(C.c_void_p)
    lib.oc_hjb_solve_batch.argtypes = [C.c_void_p, C.c_int, vpp, vpp, C.POINTER(HjbParams), C.c_double, dp, C.c_int,
                                       vpp, vpp, vpp, C.POINTER(HjbStats), C.c_void_p]
    lib.oc_hjb_solve_multi.argtypes = [C.c_void_p, C.c_int, vpp, vpp, C.POINTER(HjbRoom), C.POINTER(HjbParams), vpp, vpp,
                                       vpp, C.POINTER(HjbStats), C.c_void_p]
    lib.oc_hjb_solve_grids.argtypes = [C.c_void_p, C.c_int, vpp, vpp, vpp, C.POINTER(HjbRoom), C.POINTER(HjbParams), vpp,
                                       vpp, vpp, C.POINTER(HjbStats), C.c_void_p]
    lib.oc_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]
    lib.oc_dist_unique_id.argtypes = [C.c_void_p]
    lib.oc_dist_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.oc_dist_finalize.argtypes = [C.c_void_p]
    lib.oc_dist_p2p_export.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.oc_dist_p2p_import.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.oc_dist_p2p_enabled.argtypes = [C.c_void_p]
    lib.oc_dist_p2p_disable.argtypes = [C.c_void_p]
    lib.oc_hjb_rhs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(HjbParams), C.c_void_p,
                               C.c_void_p]
    lib.oc_hjb_vels.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(HjbParams), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.oc_wall_tiles.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, dp, C.c_void_p]
    lib.oc_gcfm_step.argtypes = [C.c_void_p, C.POINTER(GcfmParams), C.c_int] + [C.c_void_p] * 8 + \
                                [C.POINTER(Key), C.c_int, ip, dp, C.c_int, C.c_int, ip, ip, C.c_void_p]
    lib.oc_gcfm_step_launch.argtypes = [C.c_void_p, C.POINTER(GcfmParams), C.c_int] + [C.c_void_p] * 8 + \
                                       [C.POINTER(Key), C.c_int, ip, dp, C.c_int, C.c_int, C.c_void_p]
    lib.oc_gcfm_step_finish.argtypes = [C.c_void_p, ip, ip]
    lib.oc_wall_force.argtypes = [C.c_void_p, C.POINTER(GcfmParams), C.c_void_p, C.c_int] + [C.c_void_p] * 8 + \
                                 [C.c_void_p]
    lib.oc_pair_force.argtypes = [C.c_void_p, C.POINTER(GcfmParams), C.c_int] + [C.c_void_p] * 6 + [C.c_void_p]
    lib.oc_density.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                               C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = lib
    return lib


def check(rc, allow=()):
    if rc != 0 and rc not in allow:
        raise OcError(rc, load().oc_last_error().decode())
    return rc


def _hp(a):
    """host pointer of a contiguous float64 numpy array (or NULL)"""
    return None if a is None else a.ctypes.data_as(dp)


def _dev(t):
    """device pointer of a torch CUDA tensor (or NULL)"""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA tensor"
    return C.c_void_p(t.data_ptr())


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptrs(ts, B):
    """host array of B device pointers of CUDA tensors (None entries: NULL), or NULL for ts None"""
    if ts is None:
        return None
    arr = (C.c_void_p * B)()
    for q, t in enumerate(ts):
        if t is not None:
            assert t.is_cuda and t.is_contiguous()
            arr[q] = t.data_ptr()
    return arr


def _batch_results(rc, st, out_phi, out_vx, out_vy):
    check(rc, allow=(OC_ERR_STEP_TOO_SMALL,))
    return [{"stats": st[q].asdict(), "phi": out_phi[q] if out_phi is not None else None,
             "vx": out_vx[q] if out_vx is not None else None, "vy": out_vy[q] if out_vx is not None else None,
             "rc": rc if st[q].status == -1 else 0} for q in range(len(st))]


def _room_spec(rooms, B):
    """oc_hjb_room entries of dict(sigma, mu, g, T, nt[, chunk_rows]) rooms, t_eval = np.linspace(T, 0, nt) as
    optimals.py:194 builds it; returns the array and the t_eval arrays it points to (alive until the call returns)"""
    if len(rooms) != B:
        raise ValueError("one rooms entry per room expected")
    t_evals = [np.linspace(r["T"], 0, int(r["nt"])) for r in rooms]
    spec = (HjbRoom * B)()
    for q, (r, te) in enumerate(zip(rooms, t_evals)):
        spec[q] = HjbRoom(float(r["sigma"]), float(r["mu"]), float(r["g"]), float(r["T"]),
                          _hp(te) if len(te) else None, int(r["nt"]), int(r.get("chunk_rows", 0)))
    return spec, t_evals


def grid_shape(room_length, room_height, grid_step):
    """simulations.py:63-64 / optimals.py:55-56 (float floor division quirk kept)."""
    return int(room_height // grid_step + 1), int(room_length // grid_step + 1)


class Context:
    """One (GPU, grid) context; owns the library workspace."""

    def __init__(self, room_length, room_height, grid_step, device=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("optimal_crowds_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        lib = load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.Ny, self.Nx = grid_shape(room_length, room_height, grid_step)
        self.dx = self.dy = grid_step
        self.room_length, self.room_height = room_length, room_height
        self.X = np.linspace(0, room_length, self.Nx)  # simulations.py:69
        self.Y = np.linspace(0, room_height, self.Ny)  # simulations.py:70
        h = C.c_void_p()
        check(lib.oc_ctx_create(self.device, self.Ny, self.Nx, self.dx, self.dy, float(room_length),
                                float(room_height), _hp(self.X), _hp(self.Y), C.byref(h)))
        self.h = h
        self.torch_device = torch.device("cuda", self.device)
        # development aid: OC_KNOBS="gcfm_graph=0,gcfm_split=0" presets oc_ctx_set_int options of every context
        for kv in filter(None, os.environ.get("OC_KNOBS", "").split(",")):
            k, v = kv.split("=")
            self.set_int(k.strip(), int(v))

    def set_int(self, key: str, value: int):
        check(load().oc_ctx_set_int(self.h, key.encode(), int(value)))

    def close(self):
        if getattr(self, "h", None):
            load().oc_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers
    def empty(self, *shape, dtype=None):
        import torch
        return torch.empty(*shape, dtype=dtype or torch.float64, device=self.torch_device)

    def to_device(self, a, dtype=None):
        """numpy -> new device tensor (torch's copy path: DMA from page-locked memory, staged otherwise)"""
        import torch
        t = torch.from_numpy(np.ascontiguousarray(a))
        if dtype is not None:
            t = t.to(dtype)
        return t.to(self.torch_device)

    def upload(self, a, out):
        """numpy array -> existing device tensor `out` of the same dtype/size through oc_upload (one DMA from
        page-locked memory, pipelined staging otherwise).  Asynchronous on the current stream for page-locked
        sources: the next library call that synchronises (e.g. the solve) covers it."""
        a = np.ascontiguousarray(a)
        assert a.nbytes == out.numel() * out.element_size() and out.is_contiguous()
        check(load().oc_upload(self.h, a.ctypes.data_as(C.c_void_p), C.c_void_p(out.data_ptr()), a.nbytes, _stream()))
        return a  # keep alive until the stream has been synchronised

    # ---- K8
    def rasterise(self, walls, holes, cyls, targets, remap=False, wall_value=-100.0, target_value=1.0, out=None):
        w, h, c, t = (np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1, k))
                      for a, k in ((walls, 4), (holes, 4), (cyls, 3), (targets, 4)))
        V = out if out is not None else self.empty(self.Ny, self.Nx)
        check(load().oc_rasterise(self.h, _hp(w), len(w), _hp(h), len(h), _hp(c), len(c), _hp(t), len(t),
                                  int(bool(remap)), float(wall_value), float(target_value), _dev(V), _stream()))
        return V

    def rasterise_band(self, walls, holes, cyls, targets, row0, rows, remap=False, wall_value=-100.0,
                       target_value=1.0):
        """rows [row0, row0+rows) of the grid only (band-shaped result), for the row-decomposed solver"""
        w, h, c, t = (np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1, k))
                      for a, k in ((walls, 4), (holes, 4), (cyls, 3), (targets, 4)))
        V = self.empty(rows, self.Nx)
        check(load().oc_rasterise_band(self.h, _hp(w), len(w), _hp(h), len(h), _hp(c), len(c), _hp(t), len(t),
                                       int(bool(remap)), float(wall_value), float(target_value), int(row0), int(rows),
                                       _dev(V), _stream()))
        return V

    # ---- row-decomposed HJB (multi-GPU or virtual bands)
    def dist_init(self, id_bytes: bytes, rank: int, nranks: int):
        buf = C.create_string_buffer(bytes(id_bytes), 128)
        check(load().oc_dist_init(self.h, buf, int(rank), int(nranks)))
        self.rank, self.nranks = int(rank), int(nranks)

    def p2p_export(self, band_rows: int) -> bytes:
        """allocate this rank's peer-memory band arrays and return their 64-byte CUDA IPC handle"""
        buf = C.create_string_buffer(64)
        check(load().oc_dist_p2p_export(self.h, int(band_rows), buf))
        return buf.raw

    def p2p_import(self, handles):
        """map the band arrays of all ranks (handles in rank order); the row-band solve then exchanges halos and
        error sums inside the step launch over NVLink peer memory"""
        blob = b"".join(bytes(h) for h in handles)
        check(load().oc_dist_p2p_import(self.h, C.create_string_buffer(blob, len(blob)), len(handles)))

    def p2p_enabled(self) -> bool:
        return bool(load().oc_dist_p2p_enabled(self.h))

    def p2p_disable(self):
        load().oc_dist_p2p_disable(self.h)

    def hjb_solve_band(self, V, m, prm: HjbParams, T, nt, n_virtual=0, own=None, want_phi=True, want_vel=False,
                       trace=False, out_phi=None, phi_extra_hi=0):
        """V, m: full-grid tensors (virtual bands) or this rank's band (distributed, after dist_init).
        phi_extra_hi=1: phi slices hold rows+3 rows (one more halo row above the band, for the GCFM sampler)."""
        t_eval = np.linspace(T, 0, nt)
        if n_virtual and n_virtual > 1 or own is None:
            rows, prow, own0, own1 = self.Ny, self.Ny, 0, self.Ny
            vshape = (max(nt - 1, 0), self.Ny - 2, self.Nx - 2)
        else:
            own0, own1 = own
            rows = own1 - own0
            prow = rows + 2 + int(phi_extra_hi)
            vshape = (max(nt - 1, 0), rows, self.Nx - 2)
        phi = out_phi if out_phi is not None else (self.empty(nt, prow, self.Nx) if want_phi else None)
        vx = vy = None
        if want_vel:
            import torch
            vx = torch.zeros(vshape, dtype=torch.float64, device=self.torch_device)
            vy = torch.zeros(vshape, dtype=torch.float64, device=self.torch_device)
        cfg = BandCfg(int(n_virtual or 0), int(own0), int(own1), int(phi_extra_hi))
        st = HjbStats()
        cap = 1 << 16 if trace else 0
        th = np.empty(max(cap, 1)); te = np.empty(max(cap, 1))
        ntr = C.c_int()
        rc = load().oc_hjb_solve_band(self.h, C.byref(cfg), _dev(V), _dev(m), C.byref(prm), float(T), _hp(t_eval),
                                      int(nt), _dev(phi), _dev(vx), _dev(vy), C.byref(st), _hp(th) if trace else None,
                                      _hp(te) if trace else None, cap, C.byref(ntr), _stream())
        check(rc, allow=(OC_ERR_STEP_TOO_SMALL,))
        res = {"stats": st.asdict(), "phi": phi, "vx": vx, "vy": vy, "rc": rc}
        if trace:
            k = min(ntr.value, cap)
            res["trace_h"], res["trace_err"] = th[:k].copy(), te[:k].copy()
        return res

    # ---- HJB
    def hjb_solve(self, V, m, prm: HjbParams, T, nt, want_phi=False, want_vel=True, trace=False, out_vx=None,
                  out_vy=None, out_phi=None):
        t_eval = np.linspace(T, 0, nt)  # optimals.py:194
        n = self.Ny * self.Nx
        phi = out_phi if out_phi is not None else (self.empty(nt, self.Ny, self.Nx) if want_phi else None)
        vx = vy = None
        if want_vel:
            vx = out_vx if out_vx is not None else self.empty(max(nt - 1, 0), self.Ny - 2, self.Nx - 2)
            vy = out_vy if out_vy is not None else self.empty(max(nt - 1, 0), self.Ny - 2, self.Nx - 2)
        st = HjbStats()
        cap = 1 << 16 if trace else 0
        th = np.empty(max(cap, 1)); te = np.empty(max(cap, 1))
        ntr = C.c_int()
        rc = load().oc_hjb_solve(self.h, _dev(V), _dev(m), C.byref(prm), float(T), _hp(t_eval), int(nt), _dev(phi),
                                 _dev(vx), _dev(vy), C.byref(st), _hp(th) if trace else None,
                                 _hp(te) if trace else None, cap, C.byref(ntr), _stream())
        check(rc, allow=(OC_ERR_STEP_TOO_SMALL,))
        res = {"stats": st.asdict(), "phi": phi, "vx": vx, "vy": vy, "rc": rc}
        if trace:
            k = min(ntr.value, cap)
            res["trace_h"], res["trace_err"] = th[:k].copy(), te[:k].copy()
        return res

    def hjb_solve_batch(self, Vs, ms, prm: HjbParams, T, nt, out_phi=None, out_vx=None, out_vy=None, want_vel=False):
        """Independent solves of len(Vs) rooms on this context's grid, overlapped on the GPU (oc_hjb_solve_batch).
        Vs: list of (Ny,Nx) CUDA tensors; ms: None or list of tensors / None; out_*: lists of tensors or None
        (phi slices (nt,Ny,Nx) are allocated when no output is given).  Returns a list of per-room dicts."""
        B = len(Vs)
        t_eval = np.linspace(T, 0, nt)
        out_phi, out_vx, out_vy = self._batch_outputs([self] * B, [nt] * B, out_phi, out_vx, out_vy, want_vel)
        st = (HjbStats * B)()
        rc = load().oc_hjb_solve_batch(self.h, B, _ptrs(Vs, B), _ptrs(ms, B), C.byref(prm), float(T), _hp(t_eval),
                                       int(nt), _ptrs(out_phi, B), _ptrs(out_vx, B), _ptrs(out_vy, B), st, _stream())
        return _batch_results(rc, st, out_phi, out_vx, out_vy)

    def hjb_solve_multi(self, Vs, ms, rooms, prm: HjbParams, out_phi=None, out_vx=None, out_vy=None, want_vel=False):
        """hjb_solve_batch with per-room model parameters and horizons (oc_hjb_solve_multi).  rooms: one
        dict(sigma, mu, g, T, nt) per room, t_eval = np.linspace(T, 0, nt) as optimals.py:194 builds it; prm gives the
        shared rtol, atol, lim and chunk_rows (its sigma, mu and g are not used).  Outputs as hjb_solve_batch, sized by
        each room's nt."""
        B = len(Vs)
        spec, keep = _room_spec(rooms, B)
        out_phi, out_vx, out_vy = self._batch_outputs([self] * B, [int(r["nt"]) for r in rooms], out_phi, out_vx, out_vy,
                                                      want_vel)
        st = (HjbStats * B)()
        rc = load().oc_hjb_solve_multi(self.h, B, _ptrs(Vs, B), _ptrs(ms, B), spec, C.byref(prm), _ptrs(out_phi, B),
                                       _ptrs(out_vx, B), _ptrs(out_vy, B), st, _stream())
        return _batch_results(rc, st, out_phi, out_vx, out_vy)

    def hjb_solve_grids(self, grids, Vs, ms, rooms, prm: HjbParams, out_phi=None, out_vx=None, out_vy=None,
                        want_vel=False):
        """hjb_solve_multi over rooms of different grids (oc_hjb_solve_grids): room q is solved on the grid of the
        Context grids[q] (its shape and spacing); this context only lends the workspace, streams and result slots.
        rooms: dict(sigma, mu, g, T, nt) and optionally chunk_rows (0 = prm.chunk_rows, then the room's own plan).
        Outputs as hjb_solve_multi, each sized by its room's grid and nt."""
        B = len(Vs)
        if len(grids) != B:
            raise ValueError("one grid per room expected")
        spec, keep = _room_spec(rooms, B)
        out_phi, out_vx, out_vy = self._batch_outputs(grids, [int(r["nt"]) for r in rooms], out_phi, out_vx, out_vy,
                                                      want_vel)
        st = (HjbStats * B)()
        hs = (C.c_void_p * B)(*[g.h.value for g in grids])
        rc = load().oc_hjb_solve_grids(self.h, B, hs, _ptrs(Vs, B), _ptrs(ms, B), spec, C.byref(prm), _ptrs(out_phi, B),
                                       _ptrs(out_vx, B), _ptrs(out_vy, B), st, _stream())
        return _batch_results(rc, st, out_phi, out_vx, out_vy)

    @staticmethod
    def _batch_outputs(grids, nts, out_phi, out_vx, out_vy, want_vel):
        """the outputs of a batched solve: phi slices (nt,Ny,Nx) of each room's grid when no output is given"""
        if out_phi is None and not (want_vel or out_vx is not None):
            out_phi = [g.empty(nt, g.Ny, g.Nx) for g, nt in zip(grids, nts)]
        if want_vel and out_vx is None:
            out_vx = [g.empty(max(nt - 1, 0), g.Ny - 2, g.Nx - 2) for g, nt in zip(grids, nts)]
            out_vy = [g.empty(max(nt - 1, 0), g.Ny - 2, g.Nx - 2) for g, nt in zip(grids, nts)]
        return out_phi, out_vx, out_vy

    def plan_chunk_rows(self, copies=1):
        """chunk height the fused solver picks for `copies` rooms of this grid side by side (oc_hjb_plan_chunk_rows)"""
        rc = int(load().oc_hjb_plan_chunk_rows(self.h, int(copies)))
        check(min(rc, 0))
        return rc

    def hjb_rhs(self, phi, V, m, prm: HjbParams):
        out = self.empty(self.Ny, self.Nx)
        check(load().oc_hjb_rhs(self.h, _dev(phi), _dev(V), _dev(m), C.byref(prm), _dev(out), _stream()))
        return out

    def hjb_vels(self, phi, prm: HjbParams):
        vx = self.empty(self.Ny - 2, self.Nx - 2); vy = self.empty(self.Ny - 2, self.Nx - 2)
        check(load().oc_hjb_vels(self.h, _dev(phi), C.byref(prm), _dev(vx), _dev(vy), _stream()))
        return vx, vy

    # ---- GCFM
    def wall_tiles(self, V):
        import torch
        nb = load().oc_wall_tiles_bytes(self.h)
        tiles = torch.empty(nb, dtype=torch.uint8, device=self.torch_device)
        vmin = C.c_double()
        check(load().oc_wall_tiles(self.h, _dev(V), _dev(tiles), C.byref(vmin), _stream()))
        return tiles, vmin.value

    def gcfm_step(self, prm: GcfmParams, state, vdes, key_id, keys, perm, noise, simu_step):
        """state: dict of CUDA tensors x,y,vx,vy,time (float64) and status (uint8), updated in place.
        keys: list of dicts(V, tiles, v_min, vx, vy | phi, nt_opt, doors(np (n,4)))."""
        return self.gcfm_step_finish(self.gcfm_step_launch(prm, state, vdes, key_id, keys, perm, noise, simu_step))

    @staticmethod
    def make_keys(keys):
        """marshal the per-target-set descriptors (dicts, see optimals.field_key) once; returns (Key array, keep-alive)"""
        karr = (Key * len(keys))()
        keep = []
        for q, k in enumerate(keys):
            doors = np.ascontiguousarray(np.asarray(k["doors"], dtype=np.float64).reshape(-1, 4))
            keep.append(doors)
            phi = k.get("phi")
            karr[q] = Key(k["V"].data_ptr(), k["tiles"].data_ptr(), float(k["v_min"]),
                          k["vx"].data_ptr() if k.get("vx") is not None else None,
                          k["vy"].data_ptr() if k.get("vy") is not None else None, int(k["nt_opt"]),
                          int(k["vx"].shape[0]) if k.get("vx") is not None else 0,
                          phi.data_ptr() if phi is not None else None, int(phi.shape[0]) if phi is not None else 0, 0,
                          float(k.get("mu", 5.0)), float(k.get("lim", 10e-3)), _hp(doors), len(doors),
                          int(k.get("phi_row0", 0)), int(k.get("phi_rows", 0)))
        keep.append([k.get(n) for k in keys for n in ("V", "tiles", "vx", "vy", "phi")])  # tensors stay alive
        return karr, keep

    def gcfm_step_launch(self, prm: GcfmParams, state, vdes, key_id, keys, perm, noise, simu_step, stream=None):
        """enqueue one step and return at once; pass the result to gcfm_step_finish().  `keys`: list of descriptor
        dicts, or the result of make_keys() (marshalled once and reused by the run loop); `stream`: raw CUDA stream
        handle (default: torch's current stream)"""
        N = state["x"].numel()
        karr, keep = keys if isinstance(keys, tuple) else self.make_keys(keys)
        perm = np.ascontiguousarray(perm, dtype=np.int32)
        noise = np.ascontiguousarray(noise, dtype=np.float64).reshape(-1, 2)
        check(load().oc_gcfm_step_launch(self.h, C.byref(prm), N, _dev(state["x"]), _dev(state["y"]),
                                         _dev(state["vx"]), _dev(state["vy"]), _dev(state["time"]),
                                         _dev(state["status"]), _dev(vdes), _dev(key_id), karr, len(karr),
                                         perm.ctypes.data_as(ip), _hp(noise), len(noise), int(simu_step),
                                         _stream() if stream is None else C.c_void_p(stream)))
        return (N, perm, noise, karr, keep)  # keeps the host buffers alive until the step has finished

    def gcfm_step_finish(self, pending):
        N = pending[0]
        exit_log = np.empty(max(N, 1), dtype=np.int32)
        n_exit = C.c_int()
        rc = load().oc_gcfm_step_finish(self.h, exit_log.ctypes.data_as(ip), C.byref(n_exit))
        check(rc, allow=(OC_ERR_SAMPLER_RANGE,))
        return exit_log[: n_exit.value].copy(), rc

    def gcfm_run(self, prm: GcfmParams, state, vdes, key_id, keys, rng_state, n_steps, simu_step0, n_active, rows=None,
                 stream=None):
        """up to n_steps steps of the run loop in one call (oc_gcfm_run): randomness drawn in C from the legacy MT19937
        state tuple `rng_state` (np.random.get_state()), next step's draws overlapped with the GPU.  rows: optional list of
        n_steps (N,4) CUDA tensors receiving the packed state after each step.  Returns dict(steps, exits (agent ids in
        exit order), exit_step (0-based step within the call), rc, rng_state (to be set_state()d), device_ms, pairs)."""
        N = state["x"].numel()
        karr, keep = keys if isinstance(keys, tuple) else self.make_keys(keys)
        key = np.ascontiguousarray(rng_state[1], dtype=np.uint32).copy()
        pos, has, cached = C.c_int(int(rng_state[2])), C.c_int(int(rng_state[3])), C.c_double(float(rng_state[4]))
        rows_arr = None
        if rows is not None:
            rows_arr = (C.c_void_p * n_steps)()
            for q, r in enumerate(rows):
                assert r.is_cuda and r.is_contiguous() and r.numel() == 4 * N
                rows_arr[q] = r.data_ptr()
        ex_a, ex_s = np.empty(max(N, 1), dtype=np.int32), np.empty(max(N, 1), dtype=np.int32)
        n_ex, done, ms, pairs = C.c_int(), C.c_int(), C.c_double(), C.c_longlong()
        rc = load().oc_gcfm_run(self.h, C.byref(prm), N, _dev(state["x"]), _dev(state["y"]), _dev(state["vx"]),
                                _dev(state["vy"]), _dev(state["time"]), _dev(state["status"]), _dev(vdes), _dev(key_id), karr,
                                len(karr), key.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(pos), C.byref(has),
                                C.byref(cached), int(n_steps), int(simu_step0), int(n_active), rows_arr,
                                ex_a.ctypes.data_as(ip), ex_s.ctypes.data_as(ip), C.byref(n_ex), C.byref(done), C.byref(ms),
                                C.byref(pairs), _stream() if stream is None else C.c_void_p(stream))
        check(rc, allow=(OC_ERR_SAMPLER_RANGE,))
        return dict(steps=done.value, exits=ex_a[: n_ex.value].copy(), exit_step=ex_s[: n_ex.value].copy(), rc=rc,
                    rng_state=("MT19937", key, pos.value, has.value, cached.value), device_ms=ms.value, pairs=pairs.value)

    def gcfm_last_ms(self):
        return float(load().oc_gcfm_last_ms(self.h))

    def gcfm_last_pairs(self):
        """interacting pairs (ped.agents_repulsion calls of the reference) evaluated by the last step"""
        return int(load().oc_gcfm_last_pairs(self.h))

    def gcfm_last_redos(self):
        """how often the last step was redone on the exact slow path (oc_gcfm_last_redos)"""
        return int(load().oc_gcfm_last_redos(self.h))

    def state_pack(self, state, out, stream=None):
        """out (N,4) <- packed (x, y, vx, vy): one row of the device-resident trajectory record"""
        N = state["x"].numel()
        assert out.is_contiguous() and out.numel() == 4 * N
        check(load().oc_state_pack(self.h, N, _dev(state["x"]), _dev(state["y"]), _dev(state["vx"]), _dev(state["vy"]),
                                   _dev(out), _stream() if stream is None else C.c_void_p(stream)))
        return out

    def fp64_peak(self):
        """measured FP64 FMA throughput of this GPU in TFLOP/s (roofline denominator of the pair forces)"""
        v = C.c_double()
        check(load().oc_fp64_peak(self.h, C.byref(v)))
        return float(v.value)

    def wall_force(self, prm: GcfmParams, V, x, y, vx, vy, vdes):
        import torch
        N = x.numel()
        fx = self.empty(N); fy = self.empty(N)
        ind = torch.empty(N, dtype=torch.int64, device=self.torch_device)
        check(load().oc_wall_force(self.h, C.byref(prm), _dev(V), N, _dev(x), _dev(y), _dev(vx), _dev(vy), _dev(vdes),
                                   _dev(fx), _dev(fy), _dev(ind), _stream()))
        return fx, fy, ind

    def pair_force(self, prm: GcfmParams, pi, vi, vdes, pj, vj):
        N = vdes.numel()
        f = self.empty(N, 2)
        check(load().oc_pair_force(self.h, C.byref(prm), N, _dev(pi), _dev(vi), _dev(vdes), _dev(pj), _dev(vj),
                                   _dev(f), _stream()))
        return f

    def density(self, x, y, status, sigma, Vglobal, out=None):
        N = 0 if x is None else x.numel()
        d = out if out is not None else self.empty(self.Ny, self.Nx)
        Cn = float(np.sqrt(4 * np.pi ** 2 * sigma ** 2))  # simulations.py:482
        check(load().oc_density(self.h, N, _dev(x), _dev(y), _dev(status), float(sigma), Cn, _dev(Vglobal), _dev(d),
                                _stream()))
        return d


class GcfmBatch:
    """Batched GCFM steps of several simulations on one GPU (oc_gcfm_step_multi_*): marshals the members' pointers once
    and keeps their legacy MT19937 states in numpy arrays that the C side advances (ensemble.py).  ``members``: list of
    dicts with ctx (Context), prm (GcfmParams), state, vdes, key_id, keys (Context.make_keys result), rng (RandomState)."""

    def __init__(self, members, sweep_ctas=8):
        self.members = members
        self.sweep_ctas = int(sweep_ctas)
        W = len(members)
        self.mt_key = np.empty((W, 624), dtype=np.uint32)
        self.mt_pos = np.empty(W, dtype=np.int32)
        self.has_gauss = np.empty(W, dtype=np.int32)
        self.cached = np.empty(W, dtype=np.float64)
        for q, m in enumerate(members):
            st = m["rng"].get_state()
            assert st[0] == "MT19937"
            self.mt_key[q], self.mt_pos[q], self.has_gauss[q], self.cached[q] = st[1], st[2], st[3], st[4]
        self.maxN = max(m["state"]["x"].numel() for m in members)
        self.exit_log = np.empty((W, max(self.maxN, 1)), dtype=np.int32)
        self._live = None

    def _bind(self, live):
        """compact pointer arrays of the live members (rebuilt when the live set or a member's keys changed)"""
        n = len(live)
        vp = lambda: (C.c_void_p * n)()
        a = dict(ctx=vp(), prm=vp(), x=vp(), y=vp(), vx=vp(), vy=vp(), tim=vp(), status=vp(), vdes=vp(), key=vp(),
                 keys=vp(), mt=vp(), elog=vp())
        a["N"] = np.empty(n, dtype=np.int32); a["nk"] = np.empty(n, dtype=np.int32)
        for i, q in enumerate(live):
            m = self.members[q]
            st = m["state"]
            a["ctx"][i] = m["ctx"].h.value if hasattr(m["ctx"].h, "value") else m["ctx"].h
            a["prm"][i] = C.addressof(m["prm"])
            for name, t in (("x", st["x"]), ("y", st["y"]), ("vx", st["vx"]), ("vy", st["vy"]), ("tim", st["time"]),
                            ("status", st["status"]), ("vdes", m["vdes"]), ("key", m["key_id"])):
                a[name][i] = t.data_ptr()
            karr = m["keys"][0]
            a["keys"][i] = C.addressof(karr); a["nk"][i] = len(karr)
            a["N"][i] = st["x"].numel()
            a["mt"][i] = self.mt_key[q].ctypes.data
            a["elog"][i] = self.exit_log[q].ctypes.data
        a["pos"] = np.empty(n, dtype=np.int32); a["hg"] = np.empty(n, dtype=np.int32); a["cg"] = np.empty(n)
        a["n_exit"] = np.zeros(n, dtype=np.int32); a["rc"] = np.zeros(n, dtype=np.int32)
        self._live, self._a = list(live), a

    def launch(self, live, n_active, simu_step, stream=None, rebind=False):
        if rebind or self._live != list(live):
            self._bind(live)
        a, idx = self._a, np.asarray(live, dtype=np.intp)
        a["pos"][:], a["hg"][:], a["cg"][:] = self.mt_pos[idx], self.has_gauss[idx], self.cached[idx]
        na = np.ascontiguousarray(n_active, dtype=np.int32); ss = np.ascontiguousarray(simu_step, dtype=np.int32)
        I = lambda v: v.ctypes.data_as(ip)
        check(load().oc_gcfm_step_multi_launch(len(live), a["ctx"], a["prm"], I(a["N"]), a["x"], a["y"], a["vx"], a["vy"],
                                               a["tim"], a["status"], a["vdes"], a["key"], a["keys"], I(a["nk"]), a["mt"],
                                               I(a["pos"]), I(a["hg"]), _hp(a["cg"]), I(na), I(ss), self.sweep_ctas,
                                               _stream() if stream is None else C.c_void_p(stream)))
        self.mt_pos[idx], self.has_gauss[idx], self.cached[idx] = a["pos"], a["hg"], a["cg"]
        self._keep = (na, ss)

    def finish(self):
        """-> list of (exit ids in sweep order, rc) for the live members of the last launch"""
        a, n = self._a, len(self._live)
        I = lambda v: v.ctypes.data_as(ip)
        rc = load().oc_gcfm_step_multi_finish(n, a["ctx"], a["elog"], I(a["n_exit"]), I(a["rc"]))
        check(rc, allow=(OC_ERR_SAMPLER_RANGE,))
        return [(self.exit_log[q, :a["n_exit"][i]].copy() if a["n_exit"][i] else self.exit_log[q, :0], int(a["rc"][i]))
                for i, q in enumerate(self._live)]

    def write_back_rng(self):
        """hand the advanced generator states back to the members' RandomState objects"""
        for q, m in enumerate(self.members):
            m["rng"].set_state(("MT19937", self.mt_key[q].copy(), int(self.mt_pos[q]), int(self.has_gauss[q]),
                                float(self.cached[q])))


def gcfm_params(cfg: dict, room_length: float, room_height: float, Ny: int, Nx: int) -> GcfmParams:
    """Scalars evaluated with the reference's own Python expressions
    (simulations.py:81-97,303,314; pedestrians.py:74,262) so they are bit-identical."""
    p = GcfmParams()
    dt = cfg["dt"]
    p.dt, p.dt2 = dt, dt ** 2
    p.half_noise = cfg["hjb_params"]["sigma"] / 2
    p.relaxation, p.v_max, p.cutoff = cfg["relaxation"], cfg["v_max"], cfg["repulsion_cutoff"]
    p.a_min, p.tau_a, p.b_min, p.b_max = cfg["b_min"], cfg["tau_a"], cfg["b_min"], cfg["b_max"]
    p.eta, p.eta_walls = cfg["eta"], cfg["eta_walls"]
    c = float(np.cos(0.7 * np.pi))
    p.cos_fov, p.one_minus_cos_fov = c, 1 - c
    p.dx = p.dy = cfg["grid_step"]
    p.room_length, p.room_height, p.Ny, p.Nx = room_length, room_height, Ny, Nx
    p.own0 = p.own1 = 0   # single-GPU step; a row-decomposed run sets its band here
    p.key_mod = p.key_rem = 0  # all target sets local; a key-sharded run (one HJB key per GPU) sets its share here
    return p


def hjb_params(cfg: dict, fused: int = 0, profile: int = 0, chunk_rows: int = 0) -> HjbParams:
    h = cfg["hjb_params"]
    return HjbParams(h["sigma"], h["mu"], h["g"], 1e-3, 1e-6, 10e-3, int(fused), int(profile), None, 0,
                     int(chunk_rows))


def launch_count(reset=False):
    return int(load().oc_launch_count(int(bool(reset))))
