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


class DensityAcc(C.Structure):
    _fields_ = [("d_sum", C.c_void_p), ("d_max", C.c_void_p), ("d_above", C.c_void_p), ("d_Vglobal", C.c_void_p),
                ("threshold", C.c_double), ("sigma", C.c_double), ("C", C.c_double), ("every", C.c_int),
                ("pad_", C.c_int)]


class VelocityAcc(C.Structure):
    _fields_ = [("d_vx_sum", C.c_void_p), ("d_vy_sum", C.c_void_p), ("d_speed_sum", C.c_void_p)]


class LinesAcc(C.Structure):
    _fields_ = [("lines", dp), ("d_counts", C.c_void_p), ("d_px", C.c_void_p), ("d_py", C.c_void_p),
                ("d_inside", C.c_void_p), ("n_lines", C.c_int), ("capacity", C.c_int)]


class AreasAcc(C.Structure):
    _fields_ = [("verts", dp), ("d_verts", C.c_void_p), ("offsets", ip), ("d_count", C.c_void_p),
                ("d_speed_sum", C.c_void_p), ("d_vx_sum", C.c_void_p), ("d_vy_sum", C.c_void_p),
                ("d_partials", C.c_void_p), ("n_areas", C.c_int), ("capacity", C.c_int), ("partial_blocks", C.c_int),
                ("pad_", C.c_int)]


class VoronoiAcc(C.Structure):
    _fields_ = [("d_ring", C.c_void_p), ("d_tris", C.c_void_p), ("d_area_info", C.c_void_p), ("tri_offsets", ip),
                ("d_tri_offsets", C.c_void_p), ("d_bin_count", C.c_void_p), ("d_bin_start", C.c_void_p),
                ("d_slot", C.c_void_p), ("d_order", C.c_void_p), ("d_partials", C.c_void_p), ("d_rows", C.c_void_p),
                ("cutoff", C.c_double), ("edges", C.c_int), ("n_areas", C.c_int), ("bins_x", C.c_int),
                ("bins_y", C.c_int), ("bin_capacity", C.c_int), ("agent_capacity", C.c_int),
                ("partial_blocks", C.c_int), ("capacity", C.c_int)]


class VormapAcc(C.Structure):
    _fields_ = [("d_density_sum", C.c_void_p), ("d_density_max", C.c_void_p), ("d_covered", C.c_void_p),
                ("d_speed_sum", C.c_void_p), ("d_vx_sum", C.c_void_p), ("d_vy_sum", C.c_void_p),
                ("d_Vglobal", C.c_void_p), ("d_ring", C.c_void_p), ("d_bin_count", C.c_void_p),
                ("d_bin_start", C.c_void_p), ("d_slot", C.c_void_p), ("d_order", C.c_void_p), ("d_vol", C.c_void_p),
                ("cutoff", C.c_double), ("edges", C.c_int), ("every", C.c_int), ("bins_x", C.c_int),
                ("bins_y", C.c_int), ("bin_capacity", C.c_int), ("agent_capacity", C.c_int)]


class Observers(C.Structure):
    _fields_ = [("density", C.POINTER(DensityAcc)), ("velocity", C.POINTER(VelocityAcc)),
                ("lines", C.POINTER(LinesAcc)), ("areas", C.POINTER(AreasAcc)), ("voronoi", C.POINTER(VoronoiAcc))]


_lib = None

EXPORTS = ["oc_abi_version", "oc_last_error", "oc_launch_count", "oc_ctx_create", "oc_ctx_destroy", "oc_ctx_set_int", "oc_rasterise",
           "oc_hjb_solve", "oc_hjb_rhs", "oc_hjb_vels", "oc_wall_tiles_bytes", "oc_wall_tiles", "oc_gcfm_step",
           "oc_wall_force", "oc_pair_force", "oc_density", "oc_gcfm_last_ms", "oc_dist_unique_id", "oc_dist_init",
           "oc_dist_finalize", "oc_dist_p2p_export", "oc_dist_p2p_import", "oc_dist_p2p_enabled", "oc_dist_p2p_disable", "oc_hjb_solve_band", "oc_rasterise_band", "oc_upload", "oc_hjb_solve_batch", "oc_hjb_solve_multi", "oc_hjb_solve_grids", "oc_gcfm_step_launch",
           "oc_gcfm_step_finish", "oc_gcfm_last_pairs", "oc_gcfm_last_redos", "oc_state_pack", "oc_fp64_peak", "oc_place_box", "oc_hjb_plan_chunk_rows", "oc_rng_step_draw", "oc_rng_step_draw_ckpt", "oc_gcfm_step_multi_launch", "oc_gcfm_step_multi_finish", "oc_gcfm_run",
           "oc_gcfm_run_acc", "oc_density_accum", "oc_density_accum_multi", "oc_density_accum_vel",
           "oc_density_accum_vel_multi", "oc_lines_count", "oc_lines_count_multi", "oc_gcfm_run_flow",
           "oc_areas_measure", "oc_areas_measure_multi", "oc_gcfm_run_obs",
           "oc_voronoi_measure", "oc_voronoi_measure_multi", "oc_gcfm_run_observed",
           "oc_vormap_accum", "oc_vormap_accum_multi", "oc_gcfm_run_observed_maps"]


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
    lib.oc_gcfm_run_acc.argtypes = lib.oc_gcfm_run.argtypes[:-1] + [C.POINTER(DensityAcc), C.c_void_p]
    lib.oc_density_accum.argtypes = [C.c_void_p, C.POINTER(DensityAcc), C.c_int] + [C.c_void_p] * 4
    lib.oc_density_accum_multi.argtypes = [C.c_int, vpp_, vpp_, ip, vpp_, vpp_, vpp_, C.c_void_p]
    lib.oc_gcfm_run_flow.argtypes = lib.oc_gcfm_run_acc.argtypes[:-1] + [C.POINTER(VelocityAcc), C.POINTER(LinesAcc),
                                                                         C.c_void_p]
    lib.oc_density_accum_vel.argtypes = [C.c_void_p, C.POINTER(DensityAcc), C.POINTER(VelocityAcc), C.c_int] + \
                                        [C.c_void_p] * 6
    lib.oc_density_accum_vel_multi.argtypes = [C.c_int, vpp_, vpp_, vpp_, ip, vpp_, vpp_, vpp_, vpp_, vpp_, C.c_void_p]
    lib.oc_lines_count.argtypes = [C.c_void_p, C.POINTER(LinesAcc), C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    lib.oc_lines_count_multi.argtypes = [C.c_int, vpp_, vpp_, ip, vpp_, vpp_, vpp_, ip, C.c_void_p]
    lib.oc_gcfm_run_obs.argtypes = lib.oc_gcfm_run_flow.argtypes[:-1] + [C.POINTER(AreasAcc), C.c_void_p]
    lib.oc_gcfm_run_observed.argtypes = lib.oc_gcfm_run_acc.argtypes[:-2] + [C.POINTER(Observers), C.c_void_p]
    lib.oc_gcfm_run_observed_maps.argtypes = lib.oc_gcfm_run_observed.argtypes[:-1] + [C.POINTER(VormapAcc),
                                                                                     C.c_void_p]
    lib.oc_vormap_accum.argtypes = [C.c_void_p, C.POINTER(VormapAcc), C.c_int] + [C.c_void_p] * 6
    lib.oc_vormap_accum_multi.argtypes = [C.c_int, vpp_, vpp_, ip, vpp_, vpp_, vpp_, vpp_, vpp_, C.c_void_p]
    lib.oc_voronoi_measure.argtypes = [C.c_void_p, C.POINTER(VoronoiAcc), C.c_int] + [C.c_void_p] * 5 + [C.c_int,
                                                                                                       C.c_void_p]
    lib.oc_voronoi_measure_multi.argtypes = lib.oc_areas_measure_multi.argtypes
    lib.oc_areas_measure.argtypes = [C.c_void_p, C.POINTER(AreasAcc), C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p]
    lib.oc_areas_measure_multi.argtypes = [C.c_int, vpp_, vpp_, ip, vpp_, vpp_, vpp_, vpp_, vpp_, ip, C.c_void_p]
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
                 stream=None, density=None, lines=None, areas=None, voronoi=None, maps=None):
        """up to n_steps steps of the run loop in one call (oc_gcfm_run_observed): randomness drawn in C from the legacy MT19937
        state tuple `rng_state` (np.random.get_state()), next step's draws overlapped with the GPU.  rows: optional list of
        n_steps (N,4) CUDA tensors receiving the packed state after each step.  density: optional DensityStats that
        receives the frame of every due step (with its velocity maps when it has them).  lines: optional LineCounts that
        receives the crossings of every step (its capacity must cover simu_step0 + n_steps).  areas: optional AreaStats
        that receives the measurement of the state every step starts from (the same capacity rule); voronoi: optional
        VoronoiStats that receives that state's Voronoi measures (the same capacity rule); maps: optional VoronoiMaps
        that receives a frame before every due step.  Returns dict(steps,
        exits (agent ids in exit order), exit_step (0-based step within the call), rc, rng_state (to be set_state()d),
        device_ms, pairs)."""
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
        obs = Observers()
        for field, owner, attr in (("density", density, "acc"), ("velocity", density, "vel"), ("lines", lines, "acc"),
                                   ("areas", areas, "acc"), ("voronoi", voronoi, "acc")):
            acc = None if owner is None else getattr(owner, attr)
            if acc is not None:
                setattr(obs, field, C.pointer(acc))
        rc = load().oc_gcfm_run_observed_maps(self.h, C.byref(prm), N, _dev(state["x"]), _dev(state["y"]),
                                         _dev(state["vx"]), _dev(state["vy"]), _dev(state["time"]),
                                         _dev(state["status"]), _dev(vdes), _dev(key_id), karr, len(karr),
                                         key.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(pos), C.byref(has),
                                         C.byref(cached), int(n_steps), int(simu_step0), int(n_active), rows_arr,
                                         ex_a.ctypes.data_as(ip), ex_s.ctypes.data_as(ip), C.byref(n_ex), C.byref(done),
                                         C.byref(ms), C.byref(pairs), C.byref(obs),
                                         None if maps is None else C.byref(maps.acc),
                                         _stream() if stream is None else C.c_void_p(stream))
        check(rc, allow=(OC_ERR_SAMPLER_RANGE,))
        for acc in (density, maps):
            if acc is not None:
                acc.frames += acc.count(simu_step0, done.value)
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

    def density_accum(self, stats, x, y, status, stream=None, vx=None, vy=None):
        """add the density frame of the crowd (x, y, status; None for no agents) to `stats` (oc_density_accum_vel; vx, vy:
        the agents' velocities, read when `stats` has velocity maps)"""
        N = 0 if x is None else x.numel()
        check(load().oc_density_accum_vel(self.h, C.byref(stats.acc), None if stats.vel is None else C.byref(stats.vel),
                                          N, _dev(x), _dev(y), _dev(vx), _dev(vy), _dev(status),
                                          _stream() if stream is None else C.c_void_p(stream)))
        stats.frames += 1

    def lines_count(self, lines, state, step, stream=None):
        """count the crossings of the step with simu_step `step` (state: the crowd after it) in `lines` (oc_lines_count)"""
        check(load().oc_lines_count(self.h, C.byref(lines.acc), state["x"].numel(), _dev(state["x"]), _dev(state["y"]),
                                    _dev(state["status"]), int(step), _stream() if stream is None else C.c_void_p(stream)))

    def areas_measure(self, areas, state, step, stream=None):
        """measure the crowd `state` (the state the step with simu_step `step` starts from) into row `step` of `areas`
        (oc_areas_measure)"""
        N = state["x"].numel()
        P = (lambda k: None) if N == 0 else (lambda k: _dev(state[k]))
        check(load().oc_areas_measure(self.h, C.byref(areas.acc), N, P("x"), P("y"), P("vx"), P("vy"), P("status"),
                                      int(step), _stream() if stream is None else C.c_void_p(stream)))

    def voronoi_measure(self, voronoi, state, step, stream=None):
        """the Voronoi measures of the crowd `state` (the state the step with simu_step `step` starts from) into row
        `step` of `voronoi` (oc_voronoi_measure)"""
        N = state["x"].numel()
        P = (lambda k: None) if N == 0 else (lambda k: _dev(state[k]))
        check(load().oc_voronoi_measure(self.h, C.byref(voronoi.acc), N, P("x"), P("y"), P("vx"), P("vy"), P("status"),
                                        int(step), _stream() if stream is None else C.c_void_p(stream)))


    def vormap_accum(self, maps, state, stream=None):
        """add the Voronoi map frame of the crowd `state` (dict with x, y, vx, vy, status) to `maps` (oc_vormap_accum)"""
        N = state["x"].numel()
        P = (lambda k: None) if N == 0 else (lambda k: _dev(state[k]))
        check(load().oc_vormap_accum(self.h, C.byref(maps.acc), N, P("x"), P("y"), P("vx"), P("vy"), P("status"),
                                     _stream() if stream is None else C.c_void_p(stream)))
        maps.frames += 1


def vormap_accum_multi(ctxs, maps, states, stream=None):
    """one Voronoi map frame per member in six launches (oc_vormap_accum_multi): member q's crowd `states[q]` (dict with
    x, y, vx, vy, status) on the grid of ctxs[q], added to maps[q]"""
    n = len(ctxs)
    if not (len(maps) == len(states) == n and n):
        raise ValueError("one context, map accumulator and state per member expected")
    vp = lambda: (C.c_void_p * n)()
    hs, accs, xs, ys, vxs, vys, sts = vp(), vp(), vp(), vp(), vp(), vp(), vp()
    Ns = np.empty(n, dtype=np.int32)
    for q, (c, a, st) in enumerate(zip(ctxs, maps, states)):
        hs[q] = c.h.value
        accs[q] = C.addressof(a.acc)
        Ns[q] = st["x"].numel()
        if Ns[q]:
            xs[q], ys[q], sts[q] = st["x"].data_ptr(), st["y"].data_ptr(), st["status"].data_ptr()
            vxs[q], vys[q] = st["vx"].data_ptr(), st["vy"].data_ptr()
    check(load().oc_vormap_accum_multi(n, hs, accs, Ns.ctypes.data_as(ip), xs, ys, vxs, vys, sts,
                                       _stream() if stream is None else C.c_void_p(stream)))
    for a in maps:
        a.frames += 1


def density_accum_multi(ctxs, stats, states, stream=None):
    """one density frame per member in one launch per variant (oc_density_accum_vel_multi): member q's crowd `states[q]`
    (dict with x, y, status, and vx, vy when stats[q] has velocity maps) on the grid of ctxs[q], added to stats[q]"""
    n = len(ctxs)
    if not (len(stats) == len(states) == n and n):
        raise ValueError("one context, statistics and state per member expected")
    vp = lambda: (C.c_void_p * n)()
    hs, accs, vels, xs, ys, vxs, vys, sts = vp(), vp(), vp(), vp(), vp(), vp(), vp(), vp()
    Ns = np.empty(n, dtype=np.int32)
    for q, (c, s, st) in enumerate(zip(ctxs, stats, states)):
        hs[q] = c.h.value
        accs[q] = C.addressof(s.acc)
        Ns[q] = st["x"].numel()
        xs[q], ys[q], sts[q] = st["x"].data_ptr(), st["y"].data_ptr(), st["status"].data_ptr()
        if s.vel is not None:
            vels[q] = C.addressof(s.vel)
            vxs[q], vys[q] = st["vx"].data_ptr(), st["vy"].data_ptr()
    check(load().oc_density_accum_vel_multi(n, hs, accs, vels, Ns.ctypes.data_as(ip), xs, ys, vxs, vys, sts,
                                            _stream() if stream is None else C.c_void_p(stream)))
    for s in stats:
        s.frames += 1


def lines_count_multi(ctxs, lines, states, steps, stream=None):
    """the crossings of one step per member in one launch (oc_lines_count_multi): member q's crowd after its step
    `steps[q]` (`states[q]`: dict with x, y, status) counted in lines[q]"""
    n = len(ctxs)
    if not (len(lines) == len(states) == len(steps) == n and n):
        raise ValueError("one context, line counter, state and step per member expected")
    vp = lambda: (C.c_void_p * n)()
    hs, accs, xs, ys, sts = vp(), vp(), vp(), vp(), vp()
    Ns = np.empty(n, dtype=np.int32)
    ss = np.ascontiguousarray(steps, dtype=np.int32)
    for q, (c, lc, st) in enumerate(zip(ctxs, lines, states)):
        hs[q] = c.h.value
        accs[q] = C.addressof(lc.acc)
        Ns[q] = st["x"].numel()
        xs[q], ys[q], sts[q] = st["x"].data_ptr(), st["y"].data_ptr(), st["status"].data_ptr()
    check(load().oc_lines_count_multi(n, hs, accs, Ns.ctypes.data_as(ip), xs, ys, sts, ss.ctypes.data_as(ip),
                                      _stream() if stream is None else C.c_void_p(stream)))


def voronoi_measure_multi(ctxs, voronoi, states, steps, stream=None):
    """one Voronoi measurement per member in six launches (oc_voronoi_measure_multi): member q's crowd `states[q]`
    (dict with x, y, vx, vy, status) measured into row steps[q] of voronoi[q]"""
    _measure_multi(load().oc_voronoi_measure_multi, ctxs, voronoi, states, steps, stream)


def areas_measure_multi(ctxs, areas, states, steps, stream=None):
    """one measurement per member in two launches (oc_areas_measure_multi): member q's crowd `states[q]` (dict with x, y,
    vx, vy, status) measured into row steps[q] of areas[q]"""
    _measure_multi(load().oc_areas_measure_multi, ctxs, areas, states, steps, stream)


def _measure_multi(fn, ctxs, accs_, states, steps, stream):
    """marshal the members of a batched measurement (oc_areas_measure_multi, oc_voronoi_measure_multi) and call fn"""
    n = len(ctxs)
    if not (len(accs_) == len(states) == len(steps) == n and n):
        raise ValueError("one context, accumulator, state and step per member expected")
    vp = lambda: (C.c_void_p * n)()
    hs, accs, xs, ys, vxs, vys, sts = vp(), vp(), vp(), vp(), vp(), vp(), vp()
    Ns = np.empty(n, dtype=np.int32)
    ss = np.ascontiguousarray(steps, dtype=np.int32)
    for q, (c, a, st) in enumerate(zip(ctxs, accs_, states)):
        hs[q] = c.h.value
        accs[q] = C.addressof(a.acc)
        Ns[q] = st["x"].numel()
        if Ns[q]:
            xs[q], ys[q], sts[q] = st["x"].data_ptr(), st["y"].data_ptr(), st["status"].data_ptr()
            vxs[q], vys[q] = st["vx"].data_ptr(), st["vy"].data_ptr()
    check(fn(n, hs, accs, Ns.ctypes.data_as(ip), xs, ys, vxs, vys, sts, ss.ctypes.data_as(ip),
             _stream() if stream is None else C.c_void_p(stream)))


class DensityStats:
    """Device accumulators of a run's density frames (oc_density_acc): per node of the (Ny, Nx) grid the sum and the
    maximum of the frames (float64) and, with a threshold, the number of frames above it (int32); zero at creation.
    sigma: the run's sigma_convolution; Vglobal: its simulation.V on the device; every: frames are taken at the steps
    whose simu_step is a multiple of it.  velocity: also the velocity maps of the frames (oc_velocity_acc: per node the
    density-weighted sums of vx, vy and the speed, float64)."""

    def __init__(self, ctx, Vglobal, sigma, every=1, threshold=None, velocity=False):
        import torch
        shape = (ctx.Ny, ctx.Nx)
        self.sum = torch.zeros(shape, dtype=torch.float64, device=ctx.torch_device)
        self.max = torch.zeros(shape, dtype=torch.float64, device=ctx.torch_device)
        self.above = None if threshold is None else torch.zeros(shape, dtype=torch.int32, device=ctx.torch_device)
        self.vx_sum = self.vy_sum = self.speed_sum = self.vel = None
        if velocity:
            self.vx_sum, self.vy_sum, self.speed_sum = (torch.zeros(shape, dtype=torch.float64, device=ctx.torch_device)
                                                        for _ in range(3))
            self.vel = VelocityAcc(self.vx_sum.data_ptr(), self.vy_sum.data_ptr(), self.speed_sum.data_ptr())
        self.Vglobal = Vglobal
        self.every, self.threshold, self.frames = int(every), threshold, 0
        Cn = float(np.sqrt(4 * np.pi ** 2 * sigma ** 2))  # simulations.py:482, as Context.density
        self.acc = DensityAcc(self.sum.data_ptr(), self.max.data_ptr(),
                              None if self.above is None else self.above.data_ptr(), Vglobal.data_ptr(),
                              0.0 if threshold is None else float(threshold), float(sigma), Cn, self.every, 0)

    def due(self, simu_step):
        return simu_step % self.every == 0

    def count(self, simu_step0, steps):
        """frames taken by `steps` consecutive steps from simu_step0"""
        return sum(1 for k in range(simu_step0, simu_step0 + steps) if k % self.every == 0)

    def result(self):
        """dict(frames, sum, max, above (None without a threshold), mean = sum / frames (None without frames)), read back
        from the device (the caller has synchronised the streams that added frames)"""
        s = self.sum.cpu().numpy()
        r = dict(frames=self.frames, sum=s, max=self.max.cpu().numpy(),
                 above=None if self.above is None else self.above.cpu().numpy(),
                 mean=s / self.frames if self.frames else None)
        if self.vel is not None:
            # + vx_sum, vy_sum, speed_sum and the density-weighted means velocity = (vx_sum, vy_sum) / sum (Ny, Nx, 2) and
            # speed = speed_sum / sum, NaN where sum == 0
            vx, vy, sp = self.vx_sum.cpu().numpy(), self.vy_sum.cpu().numpy(), self.speed_sum.cpu().numpy()
            zero = s == 0
            with np.errstate(divide="ignore", invalid="ignore"):
                mean = lambda a: np.where(zero, np.nan, a / np.where(zero, 1.0, s))
                r.update(vx_sum=vx, vy_sum=vy, speed_sum=sp, velocity=np.stack([mean(vx), mean(vy)], axis=-1),
                         speed=mean(sp))
        return r

    @staticmethod
    def nbytes(Ny, Nx, threshold=None, velocity=False):
        """device bytes of the accumulators of an (Ny, Nx) grid"""
        return Ny * Nx * (16 + (4 if threshold is not None else 0) + (24 if velocity else 0))


class LineCounts:
    """Device accumulator of pedestrian counts through measurement lines (oc_lines_acc): per step and line the crossings
    to the left and to the right (int32 (capacity, n_lines, 2), zero at creation), and per agent the previous position
    and whether it was inside (initialised from `state`, the crowd before its first step).  names: the lines' names;
    lines: (n_lines, 4) array of (x0, y0, x1, y1) in metres; capacity: rows (steps) allocated, grown by ensure()."""

    def __init__(self, ctx, names, lines, state, capacity):
        import torch
        self.names = list(names)
        self.lines = np.ascontiguousarray(lines, dtype=np.float64).reshape(-1, 4)
        self.px, self.py = state["x"].clone(), state["y"].clone()
        self.inside = state["status"].clone()
        self.device = ctx.torch_device
        self.counts = torch.zeros((max(int(capacity), 1), len(self.lines), 2), dtype=torch.int32, device=self.device)
        self.acc = LinesAcc(self.lines.ctypes.data_as(dp), self.counts.data_ptr(), self.px.data_ptr() or None,
                            self.py.data_ptr() or None, self.inside.data_ptr() or None, len(self.lines),
                            self.counts.shape[0])

    def ensure(self, steps):
        """grow the count rows (on the host: rare) so that steps 0 .. steps-1 fit"""
        import torch
        have = self.counts.shape[0]
        if steps <= have:
            return
        torch.cuda.synchronize(self.device)   # (no update of the old rows may be in flight on any stream)
        grown = torch.zeros((max(steps, 2 * have), len(self.lines), 2), dtype=torch.int32, device=self.device)
        grown[:have] = self.counts
        torch.cuda.synchronize(self.device)
        self.counts = grown
        self.acc.d_counts, self.acc.capacity = grown.data_ptr(), grown.shape[0]

    def result(self, steps):
        """dict(names, to_left, to_right): int32 (steps, n_lines) arrays, row k = the step with simu_step k (the caller
        has synchronised the streams that counted)"""
        c = self.counts[:steps].cpu().numpy()
        return dict(names=list(self.names), to_left=np.ascontiguousarray(c[:, :, 0]),
                    to_right=np.ascontiguousarray(c[:, :, 1]))

    @staticmethod
    def nbytes(N, n_lines, capacity):
        """device bytes of the accumulator of N agents: previous positions and inside bytes, and the count rows"""
        return 17 * N + 8 * n_lines * max(int(capacity), 1)


AREA_BLOCK = 256   # agents per block of the fixed summation order (oc_areas_acc)


def polygon_area(v):
    """|shoelace area| of a polygon given as an (n, 2) array of vertices"""
    x, y = v[:, 0], v[:, 1]
    return abs(float(np.sum(x * np.roll(y, -1) - np.roll(x, -1) * y))) / 2


class AreaStats:
    """Device accumulator of measurement areas (oc_areas_acc): per step and area the pedestrians inside (int32) and the
    sums of their speeds, vx and vy (float64), rows (capacity, n_areas), grown by ensure(); the vertices on the device
    (uploaded once) and the per-block scratch of a crowd of N agents.  names: the areas' names; verts: (V, 2) array of
    all vertices in metres, area after area; offsets: (n_areas + 1) int array (simulations.areas_spec)."""

    def __init__(self, ctx, names, verts, offsets, N, capacity):
        import torch
        self.names = list(names)
        self.verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 2)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        self.device = ctx.torch_device
        na = len(self.names)
        self.d_verts = torch.from_numpy(self.verts).to(self.device)
        self.partials = torch.empty((max(-(-int(N) // AREA_BLOCK), 1), na, 4), dtype=torch.float64, device=self.device)
        self._rows(max(int(capacity), 1))
        self.acc = AreasAcc(self.verts.ctypes.data_as(dp), self.d_verts.data_ptr(), self.offsets.ctypes.data_as(ip),
                            self.count.data_ptr(), self.speed_sum.data_ptr(), self.vx_sum.data_ptr(),
                            self.vy_sum.data_ptr(), self.partials.data_ptr(), na, self.count.shape[0],
                            self.partials.shape[0], 0)

    def _rows(self, cap, old=None):
        import torch
        na = len(self.names)
        self.count = torch.zeros((cap, na), dtype=torch.int32, device=self.device)
        self.speed_sum, self.vx_sum, self.vy_sum = (torch.zeros((cap, na), dtype=torch.float64, device=self.device)
                                                    for _ in range(3))
        if old is not None:
            for new, o in zip((self.count, self.speed_sum, self.vx_sum, self.vy_sum), old):
                new[:o.shape[0]] = o

    def ensure(self, steps):
        """grow the rows (on the host: rare) so that steps 0 .. steps-1 fit"""
        import torch
        have = self.count.shape[0]
        if steps <= have:
            return
        torch.cuda.synchronize(self.device)   # (no measurement of the old rows may be in flight on any stream)
        self._rows(max(steps, 2 * have), (self.count, self.speed_sum, self.vx_sum, self.vy_sum))
        torch.cuda.synchronize(self.device)
        self.acc.d_count, self.acc.d_speed_sum = self.count.data_ptr(), self.speed_sum.data_ptr()
        self.acc.d_vx_sum, self.acc.d_vy_sum = self.vx_sum.data_ptr(), self.vy_sum.data_ptr()
        self.acc.capacity = self.count.shape[0]

    def result(self, steps):
        """dict(names, area (n_areas,) in m^2, count (steps, n_areas) int32, speed_sum, vx_sum, vy_sum (float64),
        density = count / area in ped/m^2, speed = speed_sum / count and velocity (steps, n_areas, 2) = (vx_sum, vy_sum)
        / count, NaN where count is 0); row k = the state the step with simu_step k started from (the caller has
        synchronised the streams that measured)"""
        area = np.array([polygon_area(self.verts[a:b]) for a, b in zip(self.offsets[:-1], self.offsets[1:])])
        c = self.count[:steps].cpu().numpy()
        sp, vx, vy = (t[:steps].cpu().numpy() for t in (self.speed_sum, self.vx_sum, self.vy_sum))
        zero = c == 0
        with np.errstate(divide="ignore", invalid="ignore"):
            mean = lambda a: np.where(zero, np.nan, a / np.where(zero, 1, c))
            return dict(names=list(self.names), area=area, count=c, speed_sum=sp, vx_sum=vx, vy_sum=vy,
                        density=c / area, speed=mean(sp), velocity=np.stack([mean(vx), mean(vy)], axis=-1))

    @staticmethod
    def nbytes(N, n_areas, n_verts, capacity):
        """device bytes of the accumulator of N agents: vertices, per-block scratch and the rows"""
        return 16 * n_verts + 32 * n_areas * max(-(-int(N) // AREA_BLOCK), 1) + 28 * n_areas * max(int(capacity), 1)


VORONOI_MAX_BINS = 256          # bins per axis at most (oc_voronoi_acc)
VORONOI_BIN_MARGIN = 1.0 + 1e-6  # bin side >= 2 * cutoff * margin


def voronoi_bins(length, cutoff):
    """bins along a room side of `length` metres for the Voronoi neighbour search: as many as fit with a side of at
    least 2 * cutoff * VORONOI_BIN_MARGIN, between 1 and VORONOI_MAX_BINS"""
    bound = 2.0 * cutoff * VORONOI_BIN_MARGIN
    nb = int(min(max(length // bound, 1), VORONOI_MAX_BINS))
    while nb > 1 and length / nb < bound:
        nb -= 1
    return nb


class VoronoiStats:
    """Device accumulator of the Voronoi measures of measurement areas (oc_voronoi_acc): per step and area the Voronoi
    density, speed, velocity and covered fraction (float64 rows (capacity, n_areas, 5), grown by ensure()); the cut-off
    polygon, the areas' triangles and bounding boxes on the device (uploaded once); the neighbour bins and per-block
    scratch of a crowd of N agents.  verts / offsets: the areas (simulations.areas_spec); tris: (T, 3, 2)
    counter-clockwise triangles and tri_offsets (n_areas + 1) (simulations.voronoi_triangles)."""

    def __init__(self, ctx, verts, offsets, tris, tri_offsets, cutoff, edges, N, capacity):
        import torch
        self.cutoff, self.edges = float(cutoff), int(edges)
        self.device = ctx.torch_device
        offsets = np.asarray(offsets)
        na = len(offsets) - 1
        self.n_areas = na
        k = np.arange(self.edges)
        ring = np.stack([self.cutoff * np.cos(2 * np.pi * k / self.edges),
                         self.cutoff * np.sin(2 * np.pi * k / self.edges)], axis=1)
        tris = np.asarray(tris, dtype=np.float64).reshape(-1, 3, 2)
        tri_rows = np.concatenate([tris.reshape(-1, 6), tris[:, :, 0].min(1)[:, None], tris[:, :, 0].max(1)[:, None],
                                   tris[:, :, 1].min(1)[:, None], tris[:, :, 1].max(1)[:, None]], axis=1)
        info = np.zeros((na, 5))
        for a in range(na):
            v = np.asarray(verts[offsets[a]:offsets[a + 1]], dtype=np.float64)
            info[a] = (v[:, 0].min(), v[:, 0].max(), v[:, 1].min(), v[:, 1].max(), polygon_area(v))
        self.area = info[:, 4].copy()
        self.tri_offsets = np.ascontiguousarray(tri_offsets, dtype=np.int32)
        dev = lambda a, dt=torch.float64: torch.from_numpy(np.ascontiguousarray(a)).to(self.device, dt)
        self.d_ring, self.d_tris, self.d_info = dev(ring), dev(tri_rows), dev(info)
        self.d_toff = dev(self.tri_offsets, torch.int32)
        bx, by = voronoi_bins(ctx.room_length, self.cutoff), voronoi_bins(ctx.room_height, self.cutoff)
        n = max(int(N), 1)
        self.bin_count = torch.zeros(bx * by + 1, dtype=torch.int32, device=self.device)
        self.bin_start = torch.empty(bx * by + 1, dtype=torch.int32, device=self.device)
        self.slot = torch.empty((n, 2), dtype=torch.int32, device=self.device)
        self.order = torch.empty(2 * n, dtype=torch.int32, device=self.device)
        self.partials = torch.empty((max(-(-int(N) // AREA_BLOCK), 1), na, 5), dtype=torch.float64,
                                    device=self.device)
        self.rows = torch.zeros((max(int(capacity), 1), na, 5), dtype=torch.float64, device=self.device)
        self.acc = VoronoiAcc(self.d_ring.data_ptr(), self.d_tris.data_ptr(), self.d_info.data_ptr(),
                              self.tri_offsets.ctypes.data_as(ip), self.d_toff.data_ptr(), self.bin_count.data_ptr(),
                              self.bin_start.data_ptr(), self.slot.data_ptr(), self.order.data_ptr(),
                              self.partials.data_ptr(), self.rows.data_ptr(), self.cutoff, self.edges, na, bx, by,
                              bx * by + 1, n, self.partials.shape[0], self.rows.shape[0])

    def ensure(self, steps):
        """grow the rows (on the host: rare) so that steps 0 .. steps-1 fit"""
        import torch
        have = self.rows.shape[0]
        if steps <= have:
            return
        torch.cuda.synchronize(self.device)   # (no measurement of the old rows may be in flight on any stream)
        rows = torch.zeros((max(steps, 2 * have),) + tuple(self.rows.shape[1:]), dtype=torch.float64,
                           device=self.device)
        rows[:have] = self.rows
        torch.cuda.synchronize(self.device)
        self.rows = rows
        self.acc.d_rows, self.acc.capacity = rows.data_ptr(), rows.shape[0]

    def result(self, steps):
        """dict(cutoff, edges, density, speed, covered (steps, n_areas) and velocity (steps, n_areas, 2)), float64; row k
        = the state the step with simu_step k started from (the caller has synchronised the streams that measured)"""
        r = self.rows[:steps].cpu().numpy()
        return dict(cutoff=self.cutoff, edges=self.edges, density=r[:, :, 0].copy(), speed=r[:, :, 1].copy(),
                    velocity=r[:, :, 2:4].copy(), covered=r[:, :, 4].copy())

    @staticmethod
    def nbytes(N, n_areas, n_tris, edges, bins, capacity):
        """device bytes of the accumulator of N agents: cut-off polygon, triangles, area boxes, bins, per-agent and
        per-block scratch and the rows"""
        n = max(int(N), 1)
        return (16 * edges + 80 * n_tris + 44 * n_areas + 4 + 8 * (bins + 1) + 16 * n
                + 40 * n_areas * max(-(-int(N) // AREA_BLOCK), 1) + 40 * n_areas * max(int(capacity), 1))


class VoronoiMaps:
    """Device accumulators of a run's Voronoi maps (oc_vormap_acc): per node of the (Ny, Nx) grid the sum and the maximum
    of the Voronoi density 1/|V|, the number of frames in which the node lay in a cell (int32), and the sums of the
    owner's speed, vx and vy over those frames (float64); zero at creation.  Vglobal: the run's simulation.V on the
    device; every: frames are taken at the steps whose simu_step is a multiple of it; N: the crowd size (per-agent
    scratch: bins, order, cell areas)."""

    def __init__(self, ctx, Vglobal, cutoff=1.0, edges=12, every=1, N=0):
        import torch
        self.cutoff, self.edges, self.every, self.frames = float(cutoff), int(edges), int(every), 0
        dev = ctx.torch_device
        shape = (ctx.Ny, ctx.Nx)
        self.density_sum, self.density_max, self.speed_sum, self.vx_sum, self.vy_sum = (
            torch.zeros(shape, dtype=torch.float64, device=dev) for _ in range(5))
        self.covered = torch.zeros(shape, dtype=torch.int32, device=dev)
        self.Vglobal = Vglobal
        k = np.arange(self.edges)
        ring = np.stack([self.cutoff * np.cos(2 * np.pi * k / self.edges),
                         self.cutoff * np.sin(2 * np.pi * k / self.edges)], axis=1)   # as VoronoiStats
        self.d_ring = torch.from_numpy(np.ascontiguousarray(ring)).to(dev)
        bx, by = voronoi_bins(ctx.room_length, self.cutoff), voronoi_bins(ctx.room_height, self.cutoff)
        n = max(int(N), 1)
        self.bin_count = torch.zeros(bx * by + 1, dtype=torch.int32, device=dev)
        self.bin_start = torch.empty(bx * by + 1, dtype=torch.int32, device=dev)
        self.slot = torch.empty((n, 2), dtype=torch.int32, device=dev)
        self.order = torch.empty(2 * n, dtype=torch.int32, device=dev)
        self.vol = torch.empty(n, dtype=torch.float64, device=dev)
        self.acc = VormapAcc(self.density_sum.data_ptr(), self.density_max.data_ptr(), self.covered.data_ptr(),
                             self.speed_sum.data_ptr(), self.vx_sum.data_ptr(), self.vy_sum.data_ptr(),
                             Vglobal.data_ptr(), self.d_ring.data_ptr(), self.bin_count.data_ptr(),
                             self.bin_start.data_ptr(), self.slot.data_ptr(), self.order.data_ptr(),
                             self.vol.data_ptr(), self.cutoff, self.edges, self.every, bx, by, bx * by + 1, n)

    def due(self, simu_step):
        return simu_step % self.every == 0

    def count(self, simu_step0, steps):
        """frames taken by `steps` consecutive steps from simu_step0"""
        return sum(1 for k in range(simu_step0, simu_step0 + steps) if k % self.every == 0)

    def result(self):
        """dict(cutoff, edges, frames, density_sum, density_max, covered, speed_sum, vx_sum, vy_sum and the means
        density = density_sum / frames (None without frames), speed = speed_sum / covered and velocity = (vx_sum,
        vy_sum) / covered (Ny, Nx, 2), NaN where covered == 0), read back from the device (the caller has synchronised
        the streams that added frames)"""
        ds, cov = self.density_sum.cpu().numpy(), self.covered.cpu().numpy()
        sp, vx, vy = self.speed_sum.cpu().numpy(), self.vx_sum.cpu().numpy(), self.vy_sum.cpu().numpy()
        zero = cov == 0
        with np.errstate(divide="ignore", invalid="ignore"):
            mean = lambda a: np.where(zero, np.nan, a / np.where(zero, 1, cov))
            return dict(cutoff=self.cutoff, edges=self.edges, frames=self.frames, density_sum=ds,
                        density_max=self.density_max.cpu().numpy(), covered=cov, speed_sum=sp, vx_sum=vx, vy_sum=vy,
                        density=ds / self.frames if self.frames else None, speed=mean(sp),
                        velocity=np.stack([mean(vx), mean(vy)], axis=-1))

    @staticmethod
    def nbytes(Ny, Nx, N, edges, bins):
        """device bytes of the accumulator of an (Ny, Nx) grid and N agents: 5 float64 and 1 int32 per node, the
        cut-off polygon, the bins and 24 bytes of per-agent scratch (slot, order, cell area)"""
        return 44 * Ny * Nx + 16 * edges + 8 * (bins + 1) + 24 * max(int(N), 1)


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
