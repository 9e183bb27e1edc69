"""HJB optimal-velocity field -- mirror of the reference's ``optimals.optimals`` (optimals.py:11-250) whose
solve runs on the GPU through liboc_b200.so (oc_hjb_solve).

Same constructor, methods and attributes as the reference:
``optimals(room, V, T, target)``, ``compute_optimal_velocity(t, m)``, ``choose_optimal_velocity(pos, t)``,
``draw_optimal_velocity()``, ``vx_opt, vy_opt, nt_opt, V, phi_T, lim, ...``.

Differences that do not change results:
  * the field lives on the device, by default as the value-function samples ``d_phi`` (nt, Ny, Nx) from which the
    GCFM sampler and ``vx_opt`` / ``vy_opt`` (numpy arrays materialised on first access after a solve) are derived
    with the reference's ``vels`` formula, bit-identically; ``field_storage='velocity'`` stores ``d_vx``, ``d_vy``
    (nt-1, Ny-2, Nx-2) like the reference instead;
  * ``V`` may be handed over as a numpy array (mutated in place like optimals.py:89-91) or a CUDA tensor.
"""
from __future__ import annotations

import json
import os

import numpy as np

from . import _lib


def _load_config():
    """optimals.py:36: 'optimal_crowds/config.json' relative to the CWD; falls back to the packaged copy."""
    for p in ("optimal_crowds/config.json", os.path.join(os.path.dirname(__file__), "config.json")):
        if os.path.exists(p):
            with open(p) as f:
                return json.loads(f.read())
    raise FileNotFoundError("config.json")


def _merge_config(base, overrides):
    """``base`` (a loaded config.json) with ``overrides`` applied: a new dict, ``base`` is left as it is.  Nested dicts
    (``hjb_params``) are merged key by key.  A key that ``base`` does not have raises KeyError: a misspelt parameter
    must not run the default silently."""
    merged = dict(base)
    for k, v in (overrides or {}).items():
        if k not in base:
            raise KeyError(f"unknown configuration key {k!r} (config.json has {sorted(base)})")
        if isinstance(base[k], dict):
            if not isinstance(v, dict):
                raise TypeError(f"configuration key {k!r} takes a dict of overrides")
            merged[k] = _merge_config(base[k], v)
        else:
            merged[k] = v
    return merged


def _load_room(room):
    if isinstance(room, dict):
        return room
    with open(os.path.join(os.environ.get("OC_ROOMS_DIR", "rooms"), room + ".json")) as f:  # optimals.py:41
        return json.loads(f.read())


class optimals:
    def __init__(self, room, V, T, target, _ctx=None, _config=None, field_storage="phi", fused=1, band=None, owned=True):
        """``band = (own0, own1)``: this process holds only node rows [own0, own1) of the field (one rank of a
        row-decomposed run, SURVEY.md section 8e; the context must carry a communicator, dist.init_context).
        ``owned = False``: another rank solves and holds this target set's field (key-sharded run, one HJB key per
        GPU): no field is allocated here and compute_optimal_velocity only keeps ``nt_opt`` in step."""
        var_config = _config if _config is not None else _load_config()
        var_room = _load_room(room)
        self.room_length = var_room['room_length']
        self.room_height = var_room['room_height']
        self.grid_step = var_config['grid_step']
        self.Ny, self.Nx = _lib.grid_shape(self.room_length, self.room_height, self.grid_step)  # optimals.py:55-56
        self.dx = self.dy = self.grid_step
        hp = var_config['hjb_params']
        self.sigma, self.mu, self.g = hp['sigma'], hp['mu'], hp['g']
        self.pot, self.pot_target = hp['wall_potential'], hp['target_potential']
        self.dt = var_config['dt']
        self.T = T
        self.nt_opt = round(self.T / self.dt)  # optimals.py:76
        self.target = target
        self.lim = 10e-3                       # optimals.py:95
        self._config = var_config
        self._ctx = _ctx if _ctx is not None else _lib.Context(self.room_length, self.room_height, self.grid_step)
        self._prm = _lib.hjb_params(var_config, fused=fused)
        if field_storage not in ("velocity", "phi"):
            raise ValueError("field_storage must be 'velocity' or 'phi'")
        self.band = tuple(band) if band is not None else None
        if self.band is not None and field_storage != "phi":
            raise ValueError("a row-decomposed field is stored as phi samples (field_storage='phi')")
        # 'velocity': (nt-1,Ny-2,Nx-2) x 2 slices exactly like the reference (optimals.py:80-81).
        # 'phi': the (nt,Ny,Nx) value-function samples only (half the memory, no conversion pass); the GCFM
        # sampler differentiates on the fly and vx_opt / vy_opt are produced on demand by the same kernel.
        self.field_storage = field_storage
        # potential: remap in place (optimals.py:89-91) and keep a device copy
        import torch
        if isinstance(V, np.ndarray):
            V[V < 0] = self.pot
            V[V > 0] = self.pot_target
            self.V = V
            self.d_V = self._ctx.to_device(V)
        else:
            V[V < 0] = self.pot
            V[V > 0] = self.pot_target
            self.d_V = V
            self.V = None  # materialised on demand by V_host()
        self.d_tiles, self.v_min = self._ctx.wall_tiles(self.d_V)
        n_slices = max(self.nt_opt - 1, 0)
        self._n_slices = n_slices
        self.owned = bool(owned)
        if not self.owned:
            self.d_vx = self.d_vy = self.d_phi = None
        elif field_storage == "velocity":
            self.d_vx = torch.empty((n_slices, self.Ny - 2, self.Nx - 2), dtype=torch.float64, device=self.d_V.device)
            self.d_vy = torch.empty_like(self.d_vx)
            self.d_phi = None
        else:
            self.d_vx = self.d_vy = None
            # band: owned rows + one halo row below + two above (the sampler reads owner-1 .. owner+2)
            rows = self.Ny if self.band is None else self.band[1] - self.band[0] + 3
            self.d_phi = torch.empty((n_slices + 1, rows, self.Nx), dtype=torch.float64, device=self.d_V.device)
        self._h_vx = self._h_vy = None
        self._d_m = None            # two device buffers for host densities (double-buffered uploads)
        self._d_m_flip = 0
        self._prefetched = None
        self._copy_stream = None
        self.phi_T = np.zeros((self.Ny, self.Nx), dtype=float).reshape(self.Nx * self.Ny) + 1  # optimals.py:83,93
        self.last_stats = None

    # ---- lazily materialised host views -------------------------------------------------------------
    @property
    def X_opt(self):
        return np.meshgrid(self._ctx.X, self._ctx.Y)[0]

    @property
    def Y_opt(self):
        return np.meshgrid(self._ctx.X, self._ctx.Y)[1]

    def _materialise(self):
        if self._h_vx is not None:
            return
        if self.d_vx is not None:
            self._h_vx, self._h_vy = self.d_vx.cpu().numpy(), self.d_vy.cpu().numpy()
            return
        if self.band is not None:
            raise NotImplementedError("vx_opt / vy_opt of a row-decomposed field: every rank holds only its band")
        # phi storage: vx_opt[s] = vels(sol.y[:, nt-1-s]) for s < nt-1 (optimals.py:200-204); later slices were
        # never written by the last solve (np.empty in the reference) and are left as zeros here
        vx = np.zeros((self._n_slices, self.Ny - 2, self.Nx - 2)); vy = np.zeros_like(vx)
        for s in range(min(self.nt_opt - 1, self._n_slices)):
            a, b = self._ctx.hjb_vels(self.d_phi[self.nt_opt - 1 - s], self._prm)
            vx[s], vy[s] = a.cpu().numpy(), b.cpu().numpy()
        self._h_vx, self._h_vy = vx, vy

    @property
    def vx_opt(self):
        self._materialise()
        return self._h_vx

    @property
    def vy_opt(self):
        self._materialise()
        return self._h_vy

    def field_key(self, doors):
        """descriptor of this target set for oc_gcfm_step"""
        key = dict(V=self.d_V, tiles=self.d_tiles, v_min=self.v_min, vx=self.d_vx, vy=self.d_vy, phi=self.d_phi,
                   mu=self.mu, lim=self.lim, nt_opt=self.nt_opt, doors=doors)
        if self.band is not None:
            key.update(phi_row0=self.band[0] - 1, phi_rows=self.band[1] - self.band[0] + 3)
        return key

    # ---- host density input ----------------------------------------------------------------------------
    def _band_rows_of(self, m):
        """the rows of a host density array this process needs: (Ny,Nx), flat, or already band shaped"""
        mh = np.asarray(m, dtype=np.float64)
        if self.band is not None and mh.size == (self.band[1] - self.band[0]) * self.Nx:
            return mh.reshape(-1, self.Nx)                                 # already this rank's rows
        mh = mh.reshape(self.Ny, self.Nx)
        return mh[self.band[0]:self.band[1]] if self.band is not None else mh

    def _m_buffer(self, shape, which):
        if self._d_m is None:
            self._d_m = [None, None]
        if self._d_m[which] is None or tuple(self._d_m[which].shape) != tuple(shape):
            self._d_m[which] = self._ctx.empty(*shape)
        return self._d_m[which]

    def prefetch_density(self, m):
        """Start the host -> device copy of the density a LATER ``compute_optimal_velocity(t, m)`` will be given (same
        numpy array, page-locked for a truly asynchronous copy) on a side stream, into the buffer the current solve does
        not use: the upload of the next solve's input overlaps the running solve (double-buffered input).  Optional; a
        solve whose density was not announced uploads it itself."""
        import torch
        mh = self._band_rows_of(m)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
        buf = self._m_buffer(mh.shape, self._d_m_flip ^ 1)
        with torch.cuda.stream(self._copy_stream):
            keep = self._ctx.upload(mh, buf)
            ev = torch.cuda.Event()
            ev.record()
        self._prefetched = ((mh.__array_interface__["data"][0], mh.shape), buf, ev, keep)

    def V_host(self):
        return self.V if self.V is not None else self.d_V.cpu().numpy()

    # ---- optimals.py:124-206 --------------------------------------------------------------------------
    def compute_optimal_velocity(self, t, m):
        """Solve the HJB equation backward from T to 0 and fill the first nt-1 slices of the field.

        ``m``: density as a numpy array (Ny,Nx), a CUDA tensor, or None / scalar 0 for no density."""
        import torch
        self.t = t
        self.nt_opt = round((self.T - self.t) / self.dt)  # optimals.py:140
        nt = self.nt_opt
        if nt < 1:
            # reference: np.linspace(T,0,0) -> solve_ivp raises on an empty t_eval
            raise ValueError("Values in `t_eval` are not within `t_span`.")
        if not self.owned:
            return  # the owning rank solves (and prints); only nt_opt changes here
        if m is None or (np.isscalar(m) and m == 0):
            d_m = None
        elif isinstance(m, np.ndarray):
            # host density -> device buffer; the solve below synchronises the stream, which also covers the
            # (asynchronous) copy from a page-locked source.  A row-decomposed field only needs (and only uploads) the
            # rows of its band.  An array announced with prefetch_density() is already on its way (or there).
            mh = self._band_rows_of(m)
            pf, self._prefetched = self._prefetched, None
            if pf is not None and pf[0] == (mh.__array_interface__["data"][0], mh.shape):
                torch.cuda.current_stream().wait_event(pf[2])
                d_m = pf[1]
                self._d_m_flip ^= 1
            else:
                d_m = self._m_buffer(mh.shape, self._d_m_flip)
                _keep = self._ctx.upload(mh, d_m)
        else:
            d_m = m if (self.band is not None and m.shape[0] == self.band[1] - self.band[0]) else m.reshape(self.Ny, self.Nx)
        if nt - 1 > self._n_slices:
            raise IndexError("re-solve asks for more slices than the field was allocated for")  # as numpy would
        if self.band is not None:
            own0, own1 = self.band
            if d_m is not None and d_m.shape[0] != own1 - own0:
                d_m = d_m[own0:own1].contiguous()   # a full-grid device density: this rank's rows
            res = self._ctx.hjb_solve_band(self.d_V[own0:own1], d_m, self._prm, self.T, nt, own=(own0, own1),
                                           out_phi=self.d_phi, phi_extra_hi=1)
        elif self.field_storage == "velocity":
            res = self._ctx.hjb_solve(self.d_V, d_m, self._prm, self.T, nt, want_phi=False, want_vel=nt > 1,
                                      out_vx=self.d_vx, out_vy=self.d_vy)
        else:
            res = self._ctx.hjb_solve(self.d_V, d_m, self._prm, self.T, nt, want_vel=False, out_phi=self.d_phi)
        self._h_vx = self._h_vy = None
        self.last_stats = res["stats"]
        if res["rc"] == _lib.OC_ERR_STEP_TOO_SMALL:
            # the reference ignores sol.status and then fails in its fill loop on the short sol.y (App. C #15)
            raise IndexError("RK45 stopped early (required step size is less than spacing between numbers)")
        print('Optimal trajectories have been learnt for ' + self.target)  # optimals.py:206

    # ---- optimals.py:212-250 --------------------------------------------------------------------------
    def choose_optimal_velocity(self, pos, t):
        """Host-side sampler with the reference's exact index semantics (diagonal pair, one-node shift).
        The GCFM step uses the device version of this function inside liboc_b200.so."""
        x, y = pos
        if t >= self.nt_opt - 1:
            return np.array((0., 0.), dtype=float)
        cols = self._axis_nodes(x, self.room_length, self.dx, self.Nx)
        rows = self._axis_nodes(y, self.room_height, self.dy, self.Ny)
        # numpy pairs two index lists element-wise; a scalar broadcasts against a list
        n = max(len(rows), len(cols))
        rows = rows * (n // len(rows))
        cols = cols * (n // len(cols))
        if t >= self._n_slices or t < -self._n_slices:
            raise IndexError(f"index {t} is out of bounds for axis 0 with size {self._n_slices}")
        H, W = self.Ny - 2, self.Nx - 2
        for i, j in zip(rows, cols):
            if not (-H <= i < H and -W <= j < W):
                raise IndexError(f"index ({i},{j}) is out of bounds for the field of shape ({H},{W})")
        import torch
        if self.d_vx is not None:
            sx, sy = self.d_vx[t], self.d_vy[t]
        else:
            sx, sy = self._ctx.hjb_vels(self.d_phi[self.nt_opt - 1 - t], self._prm)
        ii = torch.tensor(rows, device=sx.device); jj = torch.tensor(cols, device=sx.device)
        vals = torch.stack([sx[ii, jj], sy[ii, jj]]).cpu().numpy()
        return np.array((np.mean(vals[0]), np.mean(vals[1])), dtype=float)

    @staticmethod
    def _axis_nodes(c, extent, step, n_nodes):
        if c < extent - step:
            k = int(c // step)
            return [k, k + 1] if c > step else [k]
        return [n_nodes - 3]

    # ---- optimals.py:97-118 ---------------------------------------------------------------------------
    def draw_optimal_velocity(self):
        """Quiver plot of the field per time slice (needs matplotlib; visualisation only)."""
        import matplotlib.pyplot as plt
        X, Y = self.X_opt[1:-1, 1:-1], self.Y_opt[1:-1, 1:-1]
        for i in range(self.nt_opt - 1):
            if i < self.nt_opt - 2:
                plt.quiver(X, Y, self.vx_opt[i], self.vy_opt[i])
            else:
                plt.plot()
            plt.xlim([0, self.room_length])
            plt.ylim([0, self.room_height])
            plt.title('t = {:.2f}s'.format(i * self.dt))
            plt.show()
