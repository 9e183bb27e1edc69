/* optimal_crowds.h -- C ABI of liboc_b200.so, the B200 (sm_100a) implementation of the two
 * data-parallel hot paths of matteobutano/optimal_crowds.
 *
 * The reference is pure Python and has no FFI of its own (SURVEY.md section 8b); the boundary this
 * library replaces is the Python-internal one between simulations.py / optimals.py / pedestrians.py
 * and numpy/scipy.  Each entry point names the reference code it stands in for (file:line under
 * /root/reference, or scipy 1.18.1 for the un-vendored integrator).  The Python shim in
 * optimal_crowds_b200/{optimals,simulations,pedestrians}.py binds these with ctypes
 * (INTEGRATION.md shows the stub a maintainer of the reference would add).
 *
 * Conventions
 *   - every call returns OC_OK (0) or a negative oc_status; oc_last_error() gives the text.
 *   - one oc_ctx per (GPU, grid); a context is not thread-safe.
 *   - "d_" pointers are DEVICE pointers owned by the caller (e.g. torch tensors); all others are host.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls that return a
 *     host-visible scalar (solve statistics, exit log) synchronise that stream before returning;
 *     the others are asynchronous on it.
 *   - grid arrays are C-order (Ny,Nx) float64, y the slow axis, exactly like the reference's numpy arrays.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with OC_ERR_CUDA.
 */
#ifndef OPTIMAL_CROWDS_H
#define OPTIMAL_CROWDS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OC_ABI_VERSION 2

typedef enum {
    OC_OK = 0,
    OC_ERR_CUDA = -1,           /* CUDA runtime error (text in oc_last_error) */
    OC_ERR_ARG = -2,            /* invalid argument */
    OC_ERR_NOMEM = -3,          /* device or host allocation failed */
    OC_ERR_SAMPLER_RANGE = -4,  /* an agent position would make the reference's sampler raise IndexError
                                   (optimals.py:234-248, SURVEY App. C #7; negative indices wrap like numpy's) */
    OC_ERR_STEP_TOO_SMALL = -5, /* RK45 TOO_SMALL_STEP (scipy rk.py:133-134): solve_ivp status -1 */
    OC_ERR_NCCL = -6
} oc_status;

typedef struct oc_ctx oc_ctx;

int oc_abi_version(void);
const char *oc_last_error(void);
/* number of this library's kernels launched since the last call with reset != 0 (bench.py gpu_launches) */
long long oc_launch_count(int reset);

/* Grid context.  X (Nx) and Y (Ny) are the np.linspace node coordinates of simulations.py:69-70 /
 * optimals.py:61-62, computed by the host with numpy so they are bit-identical to the reference's. */
int oc_ctx_create(int device, int Ny, int Nx, double dx, double dy, double room_length, double room_height,
                  const double *X, const double *Y, oc_ctx **out);
void oc_ctx_destroy(oc_ctx *ctx);
/* Integer tuning options of a context.  No result depends on any of them.
 *   "gcfm_sweep_ctas"  upper bound of the GCFM sweep kernel's grid (0 = fill the GPU, the default); ensembles set it so
 *                      that the concurrent sweeps of many small crowds share the SMs
 *   "gcfm_poll_ns"     back-off between polls of a neighbour's done-flag (default 100)
 *   "gcfm_margin_mm"   displacement margin (2 x the per-axis bound) of the first attempt of a step, in mm (default 250;
 *                      a step that exceeds it is redone with 1000, then on the exact slow path)
 *   "gcfm_fov_cull"    1 (default): candidates that cannot enter the agent's field of view are not waited for
 *   "gcfm_split"       1 (default): sweep = candidate-list kernel + dependency-chain kernel; 0: one-kernel sweep
 *   "gcfm_graph"       1 (default): a step's launches are replayed as one CUDA graph
 *   "gcfm_overlap"     1 (default): wall search / sampler / noise index on side streams next to the cell list
 *   "gcfm_ws_pair"     1 (default): the wall search scans two tiles per memory round trip */
int oc_ctx_set_int(oc_ctx *ctx, const char *key, int value);

/* Host -> device copy of a caller-owned input array (e.g. the density `m` that
 * optimals.compute_optimal_velocity(t, m) receives as a numpy array, optimals.py:124) onto `stream`.
 * Page-locked `host` memory goes to the copy engine directly and must stay valid until `stream` has passed the
 * copy; pageable memory is staged by the driver and has been read completely when the call returns. */
int oc_upload(oc_ctx *ctx, const void *host, void *d_dst, long long bytes, void *stream);

/* ------------------------------------------------------------------ crowd placement (host code, no CUDA)
 * One initial box of simulation.__init__ (simulations.py:122-138): rejection-samples loc_N = int(rho*w*h) positions with
 * the reference's exact use of numpy's legacy MT19937 stream and its node-mask occupancy rule.  box = cx,cy,w,h,rho;
 * X (Nx), Y (Ny): linspace node coordinates; place_ped (Ny,Nx) float64 occupancy mask shared by all boxes, updated in
 * place; mt_key (624 words) / mt_pos: np.random.get_state()[1:3], advanced in place.  Returns the number of trials
 * (>= loc_N) or a negative oc_status. */
long long oc_place_box(const double *box, const double *X, int Nx, const double *Y, int Ny, double *place_ped, double r_in,
                       uint32_t *mt_key, int *mt_pos, double *xs, double *ys, int loc_N);

/* The random numbers of one GCFM step from numpy's legacy MT19937 stream (host code): the permutation of
 * simulations.py:271 and one normal pair per agent inside (:303).  mt_key/mt_pos/has_gauss/cached_gauss =
 * np.random.get_state()[1:5], advanced in place; perm (N ints) and noise (n_active,2) are outputs. */
int oc_rng_step_draw(uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int N, int n_active, int *perm,
                     double *noise);
/* The same, plus n_ckpt snapshots of the generator state as it is after n_active - q pairs (q = 0 .. n_ckpt-1; snapshot q:
 * ckpt_key + 624 q, ckpt_pos[q], ckpt_has[q], ckpt_cached[q]): look-ahead draws for an upper bound of agents. */
int oc_rng_step_draw_ckpt(uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int N, int n_active,
                          int *perm, double *noise, int n_ckpt, uint32_t *ckpt_key, int *ckpt_pos, int *ckpt_has,
                          double *ckpt_cached);

/* ------------------------------------------------------------------ room rasteriser (K8)
 * Replaces simulation.create_potential (simulations.py:516-576) followed by the value remap of
 * optimals.__init__ (optimals.py:89-91) when remap != 0 (V<0 -> wall_value, V>0 -> target_value).
 * Shapes are flat host arrays in JSON order: walls/holes/targets (n,4) = cx,cy,w,h; cylinders (n,3) = cx,cy,r. */
int oc_rasterise(oc_ctx *ctx, const double *walls, int n_walls, const double *holes, int n_holes,
                 const double *cyls, int n_cyls, const double *targets, int n_targets, int remap,
                 double wall_value, double target_value, double *d_V, void *stream);

/* ------------------------------------------------------------------ HJB solve (K1, K2, K3)
 * Replaces optimals.compute_optimal_velocity (optimals.py:124-206) including scipy's
 * solve_ivp(method='RK45', t_eval=...) (scipy rk.py / common.py / ivp.py, see oracle/oc_oracle_hjb.c). */
typedef struct {
    double sigma, mu, g;  /* config.json hjb_params            optimals.py:66-70 */
    double rtol, atol;    /* solve_ivp defaults 1e-3 / 1e-6    optimals.py:196 */
    double lim;           /* 10e-3                             optimals.py:95 */
    int fused;            /* 0: one kernel per RK stage; 1: stage-fused step kernel (temporal blocking) */
    int profile;          /* != 0: bracket every kernel with CUDA events and fill the per-class times below */
    /* Teacher-forced controller (parity tests): signed step h to use for attempt i < n_forced_h instead of the
     * controller's own value; accept/reject is still decided by the computed error norm.  NULL/0 = free-running.
     * (The adaptive controller operates at the explicit-stability limit and amplifies rounding-level
     * differences of the error norm ~10x per 40 attempts, so long solves are compared step-for-step.) */
    const double *forced_h;
    int n_forced_h;
    int chunk_rows;       /* fused path: rows per CTA chunk (0 = chosen per grid).  Fixing it makes the error-norm
                             summation order, and therefore every bit of the result, independent of how the grid
                             is split into row bands (bands must be multiples of it) */
} oc_hjb_params;

typedef struct {
    int nfev;        /* RHS evaluations, = 6*attempts + 2 (scipy's sol.nfev) */
    int n_accepted;  /* accepted steps */
    int n_rejected;  /* rejected step attempts */
    int status;      /* solve_ivp status: 0 finished, -1 step too small */
    int n_out;       /* t_eval samples emitted (== nt on success) */
    int launches;    /* kernels launched by this solve */
    double h0;       /* select_initial_step result */
    double gpu_ms;   /* CUDA-event time of the whole solve on `stream` */
    /* per kernel class (only when prm->profile): launches, summed CUDA-event ms, summed algorithmic bytes
     * (compulsory unique reads + writes, SURVEY.md section 8d).  class 0: RK stage kernels (K2),
     * class 1: dense output + velocity epilogue (K3), class 2: reductions / setup */
    int cls_launches[3];
    int pad_;
    double cls_ms[3];
    double cls_bytes[3];
} oc_hjb_stats;

/* d_V: remapped potential {wall_value,0,target_value}; d_m: density or NULL (== zeros).
 * t_eval: nt decreasing host values, np.linspace(T,0,nt) (optimals.py:194).
 * Outputs (each nullable): d_phi (nt,Ny,Nx): slice k = sol.y[:,k];
 *   d_vx,d_vy (nt-1,Ny-2,Nx-2): slice s = vels(sol.y[:,nt-1-s]) = the reference's vx_opt[s] (optimals.py:200-204).
 * trace_h/trace_err (nullable, capacity trace_cap): signed h and error norm of every step attempt. */
int oc_hjb_solve(oc_ctx *ctx, const double *d_V, const double *d_m, const oc_hjb_params *prm, double T,
                 const double *t_eval, int nt, double *d_phi, double *d_vx, double *d_vy, oc_hjb_stats *stats,
                 double *trace_h, double *trace_err, int trace_cap, int *trace_n, void *stream);

/* ------------------------------------------------------------------ batched HJB solves (ensembles)
 * n_rooms independent solves on the context's grid shape (BASELINE configs[4]: ensembles of rooms / seeds, one
 * batch per GPU; the reference would call optimals.compute_optimal_velocity once per room, optimals.py:124-206).
 * Every room keeps its own RK45 controller state and runs on its own CUDA stream, so the rooms' kernels overlap
 * and the host's per-attempt round trip is hidden behind the other rooms' work.  A room's result is bit-identical
 * to oc_hjb_solve of that room alone with the same prm->chunk_rows (same kernels, same reduction order).
 * d_V[b], d_m[b] (d_m or entries nullable), d_phi[b] (nt,Ny,Nx), d_vx[b], d_vy[b] (nt-1,Ny-2,Nx-2): arrays of
 * n_rooms device pointers held in HOST memory; d_phi or (d_vx and d_vy) may be NULL.  stats: n_rooms entries.
 * prm->fused, forced_h and profile are ignored (always the stage-fused kernel, free-running controller).
 * Without d_phi a step attempt may emit at most 6 t_eval samples (OC_ERR_ARG otherwise: pass d_phi for a dense t_eval).
 * Returns OC_ERR_STEP_TOO_SMALL if any room's integration stopped early (its stats.status == -1). */
/* Chunk height (prm->chunk_rows) that balances halo recomputation against wave quantisation for `copies` rooms solved
 * side by side; the default of a single solve is oc_hjb_plan_chunk_rows(ctx, 1). */
int oc_hjb_plan_chunk_rows(oc_ctx *ctx, int copies);
/* All rooms with the model parameters of prm and the one horizon (T, t_eval, nt): oc_hjb_solve_multi with n_rooms
 * identical oc_hjb_room entries. */
int oc_hjb_solve_batch(oc_ctx *ctx, int n_rooms, const double *const *d_V, const double *const *d_m,
                       const oc_hjb_params *prm, double T, const double *t_eval, int nt, double *const *d_phi,
                       double *const *d_vx, double *const *d_vy, oc_hjb_stats *stats, void *stream);

/* What one room of oc_hjb_solve_multi / oc_hjb_solve_grids does not share with the others: its model parameters (sigma,
 * mu, g of its config.json, optimals.py:66-70), its horizon and its chunking.  d_phi[b] holds rooms[b].nt slices,
 * d_vx[b] / d_vy[b] nt-1. */
typedef struct {
    double sigma, mu, g;        /* config.json hjb_params of this room */
    double T;                   /* t_span = (T, 0) */
    const double *t_eval;       /* host, nt decreasing values: np.linspace(T, 0, nt) (optimals.py:194) */
    int nt;
    int chunk_rows;             /* rows per CTA chunk of this room's fused step (>= 0): 0 = prm->chunk_rows, and when that
                                   is 0 too, the plan a stand-alone oc_hjb_solve of the room's grid makes.  The room's
                                   result is bit-identical to oc_hjb_solve with prm->chunk_rows set to the value used */
} oc_hjb_room;
/* The batched solve with per-room model parameters and horizons (ensembles whose members have their own
 * configuration).  Each room's result is bit-identical to oc_hjb_solve of that room alone with prm's sigma, mu, g
 * replaced by the room's and the room's (T, t_eval, nt).  Shared by all rooms: prm->rtol, atol, lim and, for rooms whose
 * own chunk_rows is 0, prm->chunk_rows; prm->sigma, mu and g are not read.  Step attempts of rooms with different nt still share the batched
 * launches, which are grouped by the number of samples per launch.  Without d_phi the limit of 6 t_eval samples per
 * attempt applies to every room.  OC_ERR_ARG if rooms is NULL, a room's t_eval is NULL or its nt < 1, sigma or mu is not
 * a finite positive number, or g is not finite.  A negative prm->chunk_rows means the grid's own plan, as in oc_hjb_solve.
 * Everything else as oc_hjb_solve_batch. */
int oc_hjb_solve_multi(oc_ctx *ctx, int n_rooms, const double *const *d_V, const double *const *d_m,
                       const oc_hjb_room *rooms, const oc_hjb_params *prm, double *const *d_phi, double *const *d_vx,
                       double *const *d_vy, oc_hjb_stats *stats, void *stream);
/* The batched solve over rooms of different grids (ensembles of different room layouts): room b is solved on the grid
 * of the context grids[b] -- its Ny, Nx, dx, dy -- and is bit-identical to oc_hjb_solve(grids[b], ...) with the room's
 * sigma, mu, g, horizon and chunk_rows.  d_V[b], d_m[b] and the outputs are shaped by that grid: (Ny,Nx), d_phi[b]
 * (nt,Ny,Nx), d_vx[b] / d_vy[b] (nt-1,Ny-2,Nx-2).  `ctx` owns everything the call uses (workspace, streams, events,
 * page-locked sums, final-reduction slots); the grid contexts are only read.  Step attempts of rooms of every shape share
 * the batched launches (one flattened grid of all their CTAs, up to 24 rooms per launch).  A negative chunk_rows is an
 * error here (the room's or prm's; oc_hjb_solve_multi keeps treating a negative prm->chunk_rows as 0).  oc_hjb_solve_multi is this
 * call with grids[b] = ctx.  OC_ERR_ARG, besides the cases of oc_hjb_solve_multi, if grids or an entry is NULL, a grid
 * lives on another device than ctx, a grid is too small for the stage-fused kernel (Ny <= 7 or Nx <= 9), or a
 * chunk_rows (the room's or prm's) is negative. */
int oc_hjb_solve_grids(oc_ctx *ctx, int n_rooms, oc_ctx *const *grids, const double *const *d_V,
                       const double *const *d_m, const oc_hjb_room *rooms, const oc_hjb_params *prm,
                       double *const *d_phi, double *const *d_vx, double *const *d_vy, oc_hjb_stats *stats,
                       void *stream);

/* ------------------------------------------------------------------ row-decomposed HJB solve (multi-GPU)
 * The grid of the context is split into bands of rows (SURVEY.md section 8e).  Two modes:
 *  - distributed: one process per GPU; call oc_dist_unique_id on rank 0, broadcast the 128 bytes (e.g. with
 *    torch.distributed), then oc_dist_init on every rank.  Arrays passed to oc_hjb_solve_band are BAND shaped:
 *    d_V, d_m (rows, Nx); d_phi (nt, rows+2, Nx) with one halo row on each side filled by the library;
 *    d_vx, d_vy (nt-1, rows, Nx-2), row j <-> global row own0+j (global frame rows are not written).
 *  - virtual (cfg.n_virtual > 1, no communicator needed): one process emulates n_virtual bands on one GPU with
 *    device copies as the halo exchange; arrays are FULL-grid shaped as for oc_hjb_solve.  Used by the tests to
 *    show that the decomposition does not change a bit of the result (with prm.chunk_rows fixed).
 * Only the stage-fused path exists here (prm.fused is ignored).  Bands are equal and multiples of 16 rows.  Without
 * d_phi an accepted step may emit at most 6 t_eval samples (OC_ERR_ARG otherwise). */
typedef struct {
    int n_virtual;   /* > 1: virtual bands in one process; otherwise the communicator of oc_dist_init is used */
    int own0, own1;  /* distributed mode: global rows [own0, own1) of this rank (= rank*rows .. (rank+1)*rows) */
    int phi_extra_hi; /* distributed mode: 1 = d_phi slices are (rows+3, Nx): one more halo row above the band (global
                         row own1+1), as the distributed GCFM sampler needs (oc_key.phi_row0 / phi_rows); 0 = (rows+2, Nx) */
} oc_band_cfg;
int oc_dist_unique_id(void *out128);
int oc_dist_init(oc_ctx *ctx, const void *id128, int rank, int nranks);
int oc_dist_finalize(oc_ctx *ctx);
/* NVLink peer-memory mode of the distributed row-band solve (optional; all ranks on one NVSwitch box, <= 8).
 * After oc_dist_init every rank calls oc_dist_p2p_export(ctx, rows, handle) -- it allocates the band's time-stepping
 * arrays for bands of `rows` rows in one block and returns its 64-byte CUDA IPC handle -- the ranks exchange the
 * handles (e.g. torch.distributed.all_gather_object) and call oc_dist_p2p_import(ctx, handles /(n x 64 bytes, rank
 * order)/, n).  From then on oc_hjb_solve_band does the per-attempt halo exchange and the error-norm all-gather INSIDE
 * the stage-fused step launch, as peer stores over NVLink, instead of an NCCL group after it; results are bit-identical.
 * Every rank must call oc_hjb_solve_band the same number of times. */
int oc_dist_p2p_export(oc_ctx *ctx, int band_rows, void *handle_out64);
int oc_dist_p2p_import(oc_ctx *ctx, const void *handles, int n);
int oc_dist_p2p_enabled(oc_ctx *ctx);
int oc_dist_p2p_disable(oc_ctx *ctx);   /* back to the NCCL exchange (collective decision of the caller) */
int oc_hjb_solve_band(oc_ctx *ctx, const oc_band_cfg *cfg, const double *d_V, const double *d_m,
                      const oc_hjb_params *prm, double T, const double *t_eval, int nt, double *d_phi, double *d_vx,
                      double *d_vy, oc_hjb_stats *stats, double *trace_h, double *trace_err, int trace_cap,
                      int *trace_n, void *stream);
/* Rasterise only rows [row0, row0+rows) of the context's grid into a band-shaped array (rows, Nx). */
int oc_rasterise_band(oc_ctx *ctx, const double *walls, int n_walls, const double *holes, int n_holes,
                      const double *cyls, int n_cyls, const double *targets, int n_targets, int remap,
                      double wall_value, double target_value, int row0, int rows, double *d_V, void *stream);

/* One RHS evaluation, the `hjb` closure (optimals.py:144-164). d_phi,d_out: (Ny,Nx). */
int oc_hjb_rhs(oc_ctx *ctx, const double *d_phi, const double *d_V, const double *d_m, const oc_hjb_params *prm,
               double *d_out, void *stream);
/* `vels` (optimals.py:168-186): d_phi (Ny,Nx) -> d_vx,d_vy (Ny-2,Nx-2). */
int oc_hjb_vels(oc_ctx *ctx, const double *d_phi, const oc_hjb_params *prm, double *d_vx, double *d_vy,
                void *stream);

/* ------------------------------------------------------------------ GCFM step (K4, K5, K6)
 * Replaces simulation.step (simulations.py:252-339) with ped.agents_repulsion / wall_repulsion /
 * check_status / evolve (pedestrians.py:121-136,166-191,216-334) and
 * optimals.choose_optimal_velocity (optimals.py:212-250), keeping the sequential random-order
 * in-place sweep semantics.  Scalars are computed by the host with the reference's own Python
 * expressions (dt**2, noise_intensity/2, np.cos(0.7*np.pi)). */
typedef struct {
    double dt, dt2, half_noise, relaxation, v_max, cutoff;
    double a_min, tau_a, b_min, b_max, eta, eta_walls;
    double cos_fov, one_minus_cos_fov;
    double dx, dy, room_length, room_height;
    int Ny, Nx;
    /* Distributed step (one room on several GPUs, SURVEY.md section 8e): the agents are replicated on every rank; a
     * rank evaluates the field sample and the wall force only for the agents it owns: those whose first sampled node
     * row i0 + 1 lies in [own0, own1), its band of the row-decomposed field.  i0 is the sampler's own row index after
     * numpy's wrap of a negative index (an agent at y < 0 reads the last rows, so the last band owns it), and the
     * band's phi slices hold every row the sampler then reads.  A row index out of range even after the wrap is
     * clamped into [0, Ny-1], so every agent has exactly one owner.  The per-agent terms are merged bit-exactly over the
     * communicator of oc_dist_init, and every rank then runs the identical sequential sweep (a room's sweep is one
     * dependency chain).  own0 = own1 = 0: single-GPU step, everything local. */
    int own0, own1;
    /* Target sets sharded over the ranks (BASELINE configs[2]: one HJB key per GPU; the reference builds and solves one
     * optimals object per key, simulations.py:113-121,424-425): with key_mod > 0 a rank evaluates the field sample and
     * the wall force only for agents whose key index k satisfies k % key_mod == key_rem -- the keys whose fields it
     * solved and holds -- and the terms are merged exactly like the row-band case.  key_mod = 0: all keys are local. */
    int key_mod, key_rem;
} oc_gcfm_params;

typedef struct {
    const double *d_V;            /* (Ny,Nx) remapped potential of this target set (simulation.Vs[key]) */
    const uint8_t *d_wall_tiles;  /* oc_wall_tiles() occupancy map of d_V (accelerates the exact argmin) */
    double v_min;                 /* min(V) over the grid, from oc_wall_tiles() */
    const double *d_vx, *d_vy;    /* (n_slices,Ny-2,Nx-2) optimal velocity field, or NULL when d_phi is given */
    int nt_opt;                   /* optimals.nt_opt (optimals.py:140,231) */
    int n_slices;
    /* phi storage (half the memory, no conversion pass): (n_phi,Ny,Nx) samples as written by oc_hjb_solve's
     * d_phi (slice k = sol.y[:,k]); the sampler differentiates on the fly with the same device function the
     * velocity epilogue uses: vx_opt[s] == vels(d_phi[nt_opt-1-s]) (optimals.py:200-204), mu/lim below */
    const double *d_phi;
    int n_phi;
    int pad_;
    double mu, lim;
    const double *doors;          /* host (n_doors,4): cx,cy,w,h of the box's targets (pedestrians.py:132-135) */
    int n_doors;
    /* row-band storage of d_phi (distributed runs): every slice holds node rows [phi_row0, phi_row0 + phi_rows) only,
     * as oc_hjb_solve_band writes them with phi_extra_hi = 1 (phi_row0 = own0 - 1, phi_rows = rows + 3).
     * phi_rows = 0: full-grid slices (Ny rows). */
    int phi_row0, phi_rows;
} oc_key;

/* Occupancy map used by the exact nearest-wall search (pedestrians.py:311-313): one byte per
 * OC_WALL_TILE x OC_WALL_TILE block of nodes = 1 + ring distance (in tiles, capped) to the nearest block that holds
 * a node with V < 0 (1 = the block itself holds one); the content is private to the library.
 * d_tiles: device buffer of oc_wall_tiles_bytes(ctx) bytes, caller-owned.  Synchronises `stream`. */
#define OC_WALL_TILE 16
long long oc_wall_tiles_bytes(oc_ctx *ctx);
int oc_wall_tiles(oc_ctx *ctx, const double *d_V, uint8_t *d_tiles, double *v_min, void *stream);

/* Agent state is SoA on the device: d_x,d_y,d_vx,d_vy,d_time (N doubles), d_status (N bytes, 1 inside),
 * d_vdes (N), d_key (N ints: index into keys).  perm (N) and noise (n_noise,2) are host arrays drawn by the
 * host from numpy's legacy global RNG exactly as simulations.py:271,303 would (n_noise = agents inside at
 * step start).  exit_log (host, capacity N) receives the ids of agents that left during this step, in
 * sweep order; *n_exit their count.  Returns OC_ERR_SAMPLER_RANGE (state still advanced with a zero
 * desired velocity for the offending agents) if the reference would have raised/wrapped. */
int oc_gcfm_step(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx,
                 double *d_vy, double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key,
                 const oc_key *keys, int n_keys, const int *perm, const double *noise, int n_noise,
                 int simu_step, int *exit_log, int *n_exit, void *stream);

/* The same step split in two so that the host can work (e.g. draw the next step's random numbers) while the GPU
 * runs: _launch enqueues everything on `stream` and returns without waiting (perm / noise must stay valid until
 * _finish); _finish waits for the step and returns the exit log and status exactly like oc_gcfm_step. */
int oc_gcfm_step_launch(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx,
                        double *d_vy, double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key,
                        const oc_key *keys, int n_keys, const int *perm, const double *noise, int n_noise,
                        int simu_step, void *stream);
int oc_gcfm_step_finish(oc_ctx *ctx, int *exit_log, int *n_exit);

/* The body of simulations.run()'s loop (simulations.py:427-441: history row, step; the periodic re-solve stays with the
 * caller) for up to n_steps consecutive steps in one call.  Per step the permutation and the normal pairs are drawn in C
 * from the caller's legacy MT19937 state (np.random.get_state()[1:5]: mt_key 624 words, *mt_pos, *has_gauss,
 * *cached_gauss; advanced in place exactly as the reference's draws would), with the next step's draws made while the
 * GPU runs the current one (speculation on "nobody leaves" + generator snapshots, see oc_rng.h).  n_active0: agents
 * inside at the start; d_rows (nullable): n_steps device pointers, d_rows[k] receives the packed state after step k
 * (oc_state_pack).  Stops early when nobody is inside.  exit_agent / exit_step (host, capacity N): agents in exit order
 * and the step (0-based within the call) they left in; *steps_done: steps executed; *device_ms: sum of their CUDA-event
 * times; *pairs: interacting pairs.  Returns OC_ERR_SAMPLER_RANGE like oc_gcfm_step (the offending step counts). */
int oc_gcfm_run(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx, double *d_vy,
                double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key, const oc_key *keys, int n_keys,
                uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int n_steps, int simu_step0,
                int n_active0, double *const *d_rows, int *exit_agent, int *exit_step, int *n_exits, int *steps_done,
                double *device_ms, long long *pairs, void *stream);

/* Batched step for ensembles of independent rooms (BASELINE configs[4]): ONE launch per kernel for all n members
 * (blockIdx.y = member) instead of 7 launches per member, and the members' per-step randomness drawn in C from their own
 * legacy MT19937 states (mt_key[m]: 624 words; mt_pos, has_gauss, cached_gauss: arrays of n = get_state()[2:5]; all
 * advanced in place) exactly as oc_rng_step_draw / the reference would.  Every member keeps its own context (workspace,
 * grid); all on one device.  Members may differ in grid, crowd size, target sets, field storage (velocity or phi slices)
 * and displacement margin.  Arrays are indexed by member: ctxs, prms, Ns, the SoA state pointers, keys / n_keys,
 * n_active (agents inside at step start) and simu_step.  sweep_ctas: CTAs of the sweep per member (0 = 8).  The
 * launch-wide knobs (gcfm_split, gcfm_overlap, gcfm_ws_pair) are read from ctxs[0].
 * _finish waits, returns every member's exit log (exit_log[m]: capacity Ns[m]) and status rc_out[m] (OC_OK or
 * OC_ERR_SAMPLER_RANGE as oc_gcfm_step); a member whose fast attempt was void is redone alone, after the batch, with
 * the single-step kernels on its own context's settings (margin, knobs, gcfm_sweep_ctas), as oc_gcfm_step would.
 * Results are bit-identical to stepping every member with oc_gcfm_step. */
int oc_gcfm_step_multi_launch(int n, oc_ctx *const *ctxs, const oc_gcfm_params *const *prms, const int *Ns,
                              double *const *x, double *const *y, double *const *vx, double *const *vy,
                              double *const *tim, uint8_t *const *status, const double *const *vdes,
                              const int *const *key, const oc_key *const *keys, const int *n_keys,
                              uint32_t *const *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss,
                              const int *n_active, const int *simu_step, int sweep_ctas, void *stream);
int oc_gcfm_step_multi_finish(int n, oc_ctx *const *ctxs, int *const *exit_log, int *n_exit, int *rc_out);

/* CUDA-event time (ms) of the last oc_gcfm_step on this context (H2D of perm/noise, all kernels, exit-log copy). */
double oc_gcfm_last_ms(oc_ctx *ctx);
/* Interacting pairs of the last step: calls of ped.agents_repulsion the reference would have made
 * (simulations.py:291-295) -- the work unit of the pair-force roofline (bench.py "gcfm.roofline"). */
long long oc_gcfm_last_pairs(oc_ctx *ctx);
/* How many times the last step was redone.  The fast path keeps at most 512 candidates per agent and assumes that no
 * agent moves more than 12.5 cm per axis in one step; a step that moves an agent further is restored from its snapshot
 * and redone with a 0.5 m bound, and a step that breaks that bound or the candidate limit is redone with global-memory
 * candidate lists and a search radius covering the measured displacement, until self-consistent (the reference has
 * neither limit: simulations.py:285-303). */
int oc_gcfm_last_redos(oc_ctx *ctx);
/* Packed copy of the crowd state, d_out (N,4) = x,y,vx,vy (32-byte aligned): one row of the device-resident record
 * behind ped.traj / ped.vels (pedestrians.py:106-110,189-190) and simulation.history (simulations.py:579-589). */
int oc_state_pack(oc_ctx *ctx, int N, const double *d_x, const double *d_y, const double *d_vx, const double *d_vy,
                  double *d_out, void *stream);
/* Measured FP64 FMA throughput of the context's GPU in TFLOP/s (2 flops per FMA): denominator of the GCFM
 * pair-force roofline (SURVEY.md section 8d).  Takes ~2 ms; synchronises the device. */
int oc_fp64_peak(oc_ctx *ctx, double *tflops);

/* Nearest-wall search + wall force only (pedestrians.py:282-334) for N independent probes (unit parity):
 * d_ind (nullable, N int64): the np.argmin flat index. */
int oc_wall_force(oc_ctx *ctx, const oc_gcfm_params *prm, const double *d_V, int N, const double *d_x,
                  const double *d_y, const double *d_vx, const double *d_vy, const double *d_vdes, double *d_fx,
                  double *d_fy, long long *d_ind, void *stream);
/* Pair force only (pedestrians.py:216-280) for N independent (i,j) probes (unit parity). */
int oc_pair_force(oc_ctx *ctx, const oc_gcfm_params *prm, int N, const double *d_pi, const double *d_vi,
                  const double *d_vdes, const double *d_pj, const double *d_vj, double *d_f, void *stream);

/* ------------------------------------------------------------------ Gaussian density (K7)
 * Replaces simulation.gaussian_density (simulations.py:453-487). C = sqrt(4*pi**2*sigma**2) from the host. */
int oc_density(oc_ctx *ctx, int N, const double *d_x, const double *d_y, const uint8_t *d_status, double sigma,
               double C, const double *d_Vglobal, double *d_out, void *stream);

/* Density statistics of a run (the frames simulation.write_history stores, simulations.py:579-589, accumulated on the
 * device instead of kept).  One frame d is oc_density(ctx, N, x, y, status, sigma, C, d_Vglobal) bit for bit; adding it
 * does, per node, d_sum += d, d_max = np.maximum(d_max, d) (a NaN propagates) and, when d_above is given,
 * d_above += (d > threshold).  All arrays (Ny,Nx) of the member's grid, caller-owned and initialised by the caller
 * (zeros).  `every`: oc_gcfm_run_acc adds a frame before the steps whose simu_step is a multiple of it. */
typedef struct {
    double *d_sum, *d_max;        /* float64 */
    int *d_above;                 /* int32 count of frames above threshold, or NULL */
    const double *d_Vglobal;      /* simulation.V: nodes where it is < 0 are walls (density 0) */
    double threshold;             /* finite when d_above is given */
    double sigma, C;              /* sigma_convolution and sqrt(4*pi**2*sigma**2) from the host; finite, > 0 */
    int every;                    /* >= 1 */
    int pad_;
} oc_density_acc;
/* Adds one frame of the crowd (d_x, d_y, d_status: N agents, NULL allowed when N = 0) to acc.  Asynchronous on stream.
 * OC_ERR_ARG for a NULL required pointer, every < 1, a sigma or C that is not finite and positive, or a non-finite
 * threshold with d_above. */
int oc_density_accum(oc_ctx *ctx, const oc_density_acc *acc, int N, const double *d_x, const double *d_y,
                     const uint8_t *d_status, void *stream);
/* One frame for each of n members in ONE launch: member m's crowd (Ns[m] agents at x[m], y[m], status[m]) on the grid
 * of ctxs[m] into accs[m].  Members may differ in grid shape, sigma, C, crowd size (0 included) and Vglobal; each result
 * is bit-identical to oc_density_accum of that member alone.  ctxs[0] owns the member table.  OC_ERR_ARG as
 * oc_density_accum, and for a member context on another device than ctxs[0]. */
int oc_density_accum_multi(int n, oc_ctx *const *ctxs, const oc_density_acc *const *accs, const int *Ns,
                           const double *const *x, const double *const *y, const uint8_t *const *status, void *stream);
/* oc_gcfm_run plus density statistics: before step k it adds a frame to acc when (simu_step0 + k) % acc->every == 0, on
 * `stream`, ahead of the step's randomness and sweep (nothing else changes).  acc = NULL is oc_gcfm_run. */
int oc_gcfm_run_acc(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx, double *d_vy,
                    double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key, const oc_key *keys,
                    int n_keys, uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int n_steps,
                    int simu_step0, int n_active0, double *const *d_rows, int *exit_agent, int *exit_step, int *n_exits,
                    int *steps_done, double *device_ms, long long *pairs, const oc_density_acc *acc, void *stream);

/* Velocity maps of the density frames (density_stats=dict(velocity=True)).  One frame adds, per node, over the agents of
 * the density frame (same order, culling and wall rule) with w the value the density frame adds for agent i
 * (ocm_exp(-r*r / (2*sigma*sigma)) / C): d_vx_sum += sum w*vx_i, d_vy_sum += sum w*vy_i, d_speed_sum += sum w*s_i,
 * s_i = sqrt(vx_i*vx_i + vy_i*vy_i); 0 on walls.  float64 (Ny,Nx) arrays, caller-owned and zero-initialised. */
typedef struct {
    double *d_vx_sum, *d_vy_sum, *d_speed_sum;
} oc_velocity_acc;
/* oc_density_accum plus, when vel is not NULL, the frame's velocity maps (vx, vy: the agents' velocities in the state
 * the frame describes).  The density sum is computed with the same operations in the same order, so acc receives exactly
 * what oc_density_accum adds.  OC_ERR_ARG as oc_density_accum, and for a NULL vel array or NULL d_vx / d_vy with vel. */
int oc_density_accum_vel(oc_ctx *ctx, const oc_density_acc *acc, const oc_velocity_acc *vel, int N, const double *d_x,
                         const double *d_y, const double *d_vx, const double *d_vy, const uint8_t *d_status,
                         void *stream);
/* oc_density_accum_multi with velocity maps: vels (NULL, or per member NULL / the member's maps), vx / vy (read for the
 * members with maps).  Members with and without maps run as one launch each; every result equals the member's
 * oc_density_accum_vel alone.  oc_density_accum / oc_density_accum_multi forward here with no maps. */
int oc_density_accum_vel_multi(int n, oc_ctx *const *ctxs, const oc_density_acc *const *accs,
                               const oc_velocity_acc *const *vels, const int *Ns, const double *const *x,
                               const double *const *y, const double *const *vx, const double *const *vy,
                               const uint8_t *const *status, void *stream);

/* Pedestrian counts through measurement lines.  With o(u,v,w) = (v.x-u.x)*(w.y-u.y) - (v.y-u.y)*(w.x-u.x) (FP64, no
 * contraction) and a line's endpoints a, b, an agent inside at the start of a step that moves from p (kept in d_px /
 * d_py) to q (its position after the step, the step it leaves in included) crosses the line when
 * (o(a,b,p) > 0) != (o(a,b,q) > 0) and (o(p,q,a) > 0) != (o(p,q,b) > 0): to the left when o(a,b,q) > 0, else to the
 * right.  Points on the line count as the right side; NaN positions never cross.  d_counts[(step*n_lines + l)*2 + 0] /
 * [... + 1] count the step's crossings of line l to the left / right.  d_px, d_py, d_inside (17 bytes per agent):
 * initialised by the caller with the crowd's x, y and status before its first counted step; each update compares them
 * with the current state and then overwrites them. */
typedef struct {
    const double *lines;       /* HOST: n_lines x (x0, y0, x1, y1) in metres; finite, non-zero length */
    int *d_counts;             /* int32 (capacity, n_lines, 2), caller-owned, zero-initialised */
    double *d_px, *d_py;       /* (N) previous positions */
    uint8_t *d_inside;         /* (N) inside at the start of the step */
    int n_lines;               /* 1..64 */
    int capacity;              /* steps d_counts has rows for */
} oc_lines_acc;
/* Counts the crossings of the step with simu_step `step` (the crowd's state after it, once final: after
 * oc_gcfm_step_finish).  Asynchronous on stream.  OC_ERR_ARG for a NULL required pointer, n_lines outside 1..64, a
 * non-finite or zero-length line and step outside [0, capacity). */
int oc_lines_count(oc_ctx *ctx, const oc_lines_acc *acc, int N, const double *d_x, const double *d_y,
                   const uint8_t *d_status, int step, void *stream);
/* oc_lines_count for each of n members (step steps[m]) in ONE launch; ctxs[0] owns the member table.  OC_ERR_ARG as
 * oc_lines_count, and for a member context on another device than ctxs[0]. */
int oc_lines_count_multi(int n, oc_ctx *const *ctxs, const oc_lines_acc *const *accs, const int *Ns,
                         const double *const *x, const double *const *y, const uint8_t *const *status, const int *steps,
                         void *stream);
/* oc_gcfm_run_acc plus the velocity maps of its frames (vel, needs acc) and the line counts of its steps (lines: every
 * step simu_step0 + k is counted once final; simu_step0 + n_steps must not exceed lines->capacity, checked before any
 * step).  oc_gcfm_run and oc_gcfm_run_acc forward here; this forwards to oc_gcfm_run_obs. */
int oc_gcfm_run_flow(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx, double *d_vy,
                     double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key, const oc_key *keys,
                     int n_keys, uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int n_steps,
                     int simu_step0, int n_active0, double *const *d_rows, int *exit_agent, int *exit_step, int *n_exits,
                     int *steps_done, double *device_ms, long long *pairs, const oc_density_acc *acc,
                     const oc_velocity_acc *vel, const oc_lines_acc *lines, void *stream);

/* Measurement areas: per step and polygon, the pedestrians inside and the sums of their speeds and velocities.
 * Membership (even-odd rule, FP64, no contraction, o as for the measurement lines): for every edge (a, b) of the polygon
 * (vertex k to vertex k+1, the last to the first), when (a.y <= p.y) != (b.y <= p.y), `inside` toggles if
 * (b.y > a.y) ? o(a,b,p) > 0 : o(a,b,p) < 0.  Points on an edge fall where this puts them; a NaN position is outside.
 * Only agents with status 1 count.  Row `step`, area a: d_count = agents inside, d_speed_sum = sum of
 * sqrt(vx*vx + vy*vy), d_vx_sum / d_vy_sum = sums of vx / vy.  The float sums have one order, whatever the launch:
 * agents in blocks of 256; in a block each warp of 32 sums by an xor butterfly (16, 8, 4, 2, 1; agents outside, left or
 * beyond N add +0.0), the 8 warp sums are added in warp order from 0.0, and the block sums in block order from 0.0.
 * A measurement writes its row (no accumulation), so rows need no initialisation. */
typedef struct {
    const double *verts;         /* HOST: (x, y) vertices in metres, area after area; finite */
    const double *d_verts;       /* the same vertices on the device (owned by the caller, uploaded once) */
    const int *offsets;          /* HOST: n_areas + 1; area a is vertices offsets[a] .. offsets[a+1]-1: 3..64 of them,
                                    1024 in all, non-zero area */
    int *d_count;                /* int32 (capacity, n_areas) */
    double *d_speed_sum, *d_vx_sum, *d_vy_sum;   /* float64 (capacity, n_areas) */
    double *d_partials;          /* scratch: float64 (partial_blocks, n_areas, 4), the per-block sums */
    int n_areas;                 /* 1..64 */
    int capacity;                /* rows (steps) of the arrays above */
    int partial_blocks;          /* blocks of 256 agents d_partials has room for: >= ceil(N / 256) */
    int pad_;
} oc_areas_acc;
/* Measures the crowd's state (N agents; the state a step starts from) into row `step`.  Asynchronous on stream: two
 * launches (per-block sums, then the block-order reduction).  OC_ERR_ARG for a NULL required pointer, n_areas outside
 * 1..64, an area with fewer than 3 or more than 64 vertices, more than 1024 vertices, a non-finite vertex, a zero area,
 * step outside [0, capacity) and too few partial blocks for N. */
int oc_areas_measure(oc_ctx *ctx, const oc_areas_acc *acc, int N, const double *d_x, const double *d_y,
                     const double *d_vx, const double *d_vy, const uint8_t *d_status, int step, void *stream);
/* oc_areas_measure for each of n members (row steps[m]) in two launches; ctxs[0] owns the member table.  Every row
 * equals the member's oc_areas_measure alone.  OC_ERR_ARG as oc_areas_measure, and for a member context on another
 * device than ctxs[0]. */
int oc_areas_measure_multi(int n, oc_ctx *const *ctxs, const oc_areas_acc *const *accs, const int *Ns,
                           const double *const *x, const double *const *y, const double *const *vx,
                           const double *const *vy, const uint8_t *const *status, const int *steps, void *stream);
/* Voronoi density, speed and velocity in the measurement areas (Steffen & Seyfried 2010, jpsreport's method D), per step
 * and area.  FP64 without contraction, every formula evaluated exactly as written; o(a,b,p) =
 * (b.x-a.x)*(p.y-a.y) - (b.y-a.y)*(p.x-a.x); r = cutoff, n = edges.
 *  1. Generators G: agents with status 1 and finite x and y.  Others neither own a cell nor clip one.
 *  2. Cut-off polygon: d_ring holds ox[k] = r*cos(2*pi*k/n), oy[k] = r*sin(2*pi*k/n), k = 0..n-1, computed on the host;
 *     agent i starts from P = [(x_i + ox[k], y_i + oy[k])], counter-clockwise.
 *  3. Clip(P, s), one Sutherland-Hodgman pass keeping s <= 0: for k = 0..m-1 (m vertices), a = P[k], b = P[(k+1) % m],
 *     each vertex's s evaluated once: emit a if sa <= 0; if (sa <= 0) != (sb <= 0) emit a + t*(b - a) per component with
 *     t = sa / (sa - sb).  Fewer than 3 output vertices make the polygon empty (empty stays empty).  A clip whose output
 *     would exceed 64 vertices overflows: the polygon's area is NaN.
 *  4. The cell V_i: P clipped by s = -p.x, s = p.x - L, s = -p.y, s = p.y - H (the room [0, L] x [0, H] of the
 *     context, in this order), then by every j in G, j != i, in ascending agent index, with dx = x_j - x_i,
 *     dy = y_j - y_i, dx*dx + dy*dy <= (2*r)*(2*r) and not (dx == 0 && dy == 0) (coincident agents do not clip each
 *     other): s = dx*(p.x - mx) + dy*(p.y - my), mx = 0.5*(x_i + x_j), my = 0.5*(y_i + y_j).
 *  5. |V| = 0.5 * (sum over k of x_k*y_{k+1} - x_{k+1}*y_k, in k order from 0.0); 0.0 for an empty polygon.
 *  6. Areas as triangles (d_tris, counter-clockwise, a fixed order per area; simulations.voronoi_triangles): for
 *     triangle t = (a, b, c), |V_i n t| = +0.0 when the square [x_i - r, x_i + r] x [y_i - r, y_i + r] does not meet t's
 *     bounding box (closed intervals: x_i - r <= xmax && x_i + r >= xmin, the same in y); else V_i clipped by
 *     s = -o(a,b,p), -o(b,c,p), -o(c,a,p) in that order, and its |.|.  w_ia = sum over the area's triangles in order
 *     from 0.0.  An overflowed cell gives w_ia = NaN for the areas with a triangle its square meets.
 *  7. Per-agent terms of area a, s_i = sqrt(vx*vx + vy*vy): w, w / |V_i|, w*s_i, w*vx_i, w*vy_i; +0.0 (all five) for
 *     non-generators, for cells with |V_i| <= 0 and wherever w == 0.
 *  8. The five sums per area in the measurement areas' order (blocks of 256 agents, xor butterfly per warp, warp sums in
 *     warp order from 0.0, block sums in block order from 0.0), each divided by |A| (d_area_info[a*5 + 4], the area's
 *     shoelace area): row `step`, area a of d_rows holds density = sum(w/|V|) / |A|, speed = sum(w*s) / |A|,
 *     vx = sum(w*vx) / |A|, vy = sum(w*vy) / |A|, covered = sum(w) / |A|.  A NaN means a cell touching the area
 *     overflowed (or a NaN velocity of an agent whose cell covers part of it, in speed and velocity).
 * Neighbour search: the generators are binned on a bins_x x bins_y grid over the room (bin index clamped in double, so
 * agents outside the room land in edge bins) with sides of at least 2r*(1 + 1e-6), sorted by index inside each bin,
 * and the 3x3 bins around a cell's bin are merged in ascending index.  Cells whose square meets no area's bounding box
 * are not built (their terms are +0.0 by rule 6). */
typedef struct {
    const double *d_ring;        /* (edges, 2): ox, oy of rule 2 */
    const double *d_tris;        /* (n_tris, 10): ax, ay, bx, by, cx, cy, xmin, xmax, ymin, ymax of every triangle */
    const double *d_area_info;   /* (n_areas, 5): xmin, xmax, ymin, ymax of the area's vertices, |A| (> 0) */
    const int *tri_offsets;      /* HOST: n_areas + 1; area a is triangles tri_offsets[a] .. tri_offsets[a+1]-1 (>= 1
                                    each), 992 in all */
    const int *d_tri_offsets;    /* the same offsets on the device */
    int *d_bin_count;            /* int32 (bin_capacity): zero before the first measurement, left zero by every one */
    int *d_bin_start;            /* int32 (bin_capacity) */
    int *d_slot;                 /* int32 (agent_capacity, 2): each generator's bin and place in it */
    int *d_order;                /* int32 (2 * agent_capacity): the binned generators, then the same sorted by index */
    double *d_partials;          /* scratch: float64 (partial_blocks, n_areas, 5), the per-block sums */
    double *d_rows;              /* float64 (capacity, n_areas, 5): density, speed, vx, vy, covered */
    double cutoff;               /* r: finite, in (0, 100] metres */
    int edges;                   /* n: 4..32 */
    int n_areas;                 /* 1..64 */
    int bins_x, bins_y;          /* >= 1; bins_x == 1 or L / bins_x >= 2r*(1 + 1e-6) (the same for y) */
    int bin_capacity;            /* >= bins_x * bins_y + 1 */
    int agent_capacity;          /* >= N */
    int partial_blocks;          /* >= ceil(N / 256) */
    int capacity;                /* rows (steps) of d_rows */
} oc_voronoi_acc;
/* Measures the crowd's state (N agents; the state a step starts from) into row `step` of acc->d_rows.  Asynchronous on
 * stream: six launches (bin, scan, place, sort, cells, block-order reduction).  OC_ERR_ARG for a NULL required pointer,
 * a cutoff that is not finite or outside (0, 100], edges outside 4..32, n_areas outside 1..64, bad triangle offsets
 * (an area without triangles, more than 992 in all), bins too small or too many, too small agent or partial capacities
 * for N and step outside [0, capacity). */
int oc_voronoi_measure(oc_ctx *ctx, const oc_voronoi_acc *acc, int N, const double *d_x, const double *d_y,
                       const double *d_vx, const double *d_vy, const uint8_t *d_status, int step, void *stream);
/* oc_voronoi_measure for each of n members (row steps[m]) in six launches; ctxs[0] owns the member table.  Every row
 * equals the member's oc_voronoi_measure alone.  OC_ERR_ARG as oc_voronoi_measure, for a member context on another
 * device than ctxs[0] and for two members sharing d_bin_count, d_bin_start, d_slot, d_order or d_partials. */
int oc_voronoi_measure_multi(int n, oc_ctx *const *ctxs, const oc_voronoi_acc *const *accs, const int *Ns,
                             const double *const *x, const double *const *y, const double *const *vx,
                             const double *const *vy, const uint8_t *const *status, const int *steps, void *stream);

/* Voronoi maps: per grid node, statistics of the Voronoi density 1/|V_i| and velocity of the pedestrian whose cell
 * holds the node (Steffen & Seyfried's method D as a field; jpsreport's profiles), accumulated over frames like the
 * density statistics.  FP64 without contraction, o and the symbols as for oc_voronoi_acc; r = cutoff.
 *  1. Generators, ring and the cell V_i are rules 1-5 of oc_voronoi_acc, unchanged; every generator gets its cell.
 *  2. A node is p = (X[ix], Y[iy]), the context's node coordinates the density uses.  Nodes where d_Vglobal < 0 are
 *     walls: never covered, all their terms 0.
 *  3. Owner: for each generator j, d2_j = (X-x_j)*(X-x_j) + (Y-y_j)*(Y-y_j); among those with d2_j <= r*r the one with
 *     the smallest d2_j, the lowest index on ties.  With none, p is uncovered.
 *  4. p must lie in the owner's cut-off polygon: o(a_k, a_{k+1}, p) >= 0 for every ring edge, a_k = (x_i + ox[k],
 *     y_i + oy[k]), a_n = a_0.  Otherwise p is uncovered.
 *  5. A covered node takes rho = 1/|V_i|, s_i = sqrt(vx*vx + vy*vy), vx_i and vy_i.  |V_i| <= 0 makes it uncovered;
 *     |V_i| NaN (an overflowed cell) leaves it covered with all four terms NaN.
 *  6. Per frame and node, in this order: d_density_sum += rho; d_density_max = np.maximum(d_density_max, rho) with
 *     rho = 0 when uncovered (the first NaN wins); d_covered += 1; d_speed_sum += s, d_vx_sum += vx, d_vy_sum += vy.
 *     Nothing but d_density_max changes at an uncovered node.
 * Consequences: of coincident generators the lower index owns the nodes (in the area measures both cells count); and
 * ownership is decided by distances while |V_i| is decided by the clip, which agree up to rounding on cell boundaries.
 * Cells are not clipped by internal walls, holes or cylinders.  Neighbour search as oc_voronoi_acc: the bins hold every
 * generator within r of a node in the 3x3 bins around the node's bin.  A frame is six launches: bin, scan, place,
 * sort, the cells' areas into d_vol (one thread per generator), and the nodes (tiles of 32 x 8). */
typedef struct {
    double *d_density_sum, *d_density_max;   /* float64 (Ny, Nx) of the context's grid */
    int *d_covered;                           /* int32 (Ny, Nx): frames in which the node lay in a cell */
    double *d_speed_sum, *d_vx_sum, *d_vy_sum;   /* float64 (Ny, Nx), sums over the covered frames */
    const double *d_Vglobal;     /* simulation.V: nodes where it is < 0 are walls */
    const double *d_ring;        /* (edges, 2): ox, oy of oc_voronoi_acc's rule 2 */
    int *d_bin_count;            /* int32 (bin_capacity): zero before the first frame, left zero by every one */
    int *d_bin_start;            /* int32 (bin_capacity) */
    int *d_slot;                 /* int32 (agent_capacity, 2) */
    int *d_order;                /* int32 (2 * agent_capacity) */
    double *d_vol;               /* float64 (agent_capacity): |V_i| of the frame */
    double cutoff;               /* r: finite, in (0, 100] metres */
    int edges;                   /* 4..32 */
    int every;                   /* >= 1: run loops take a frame before the steps whose simu_step is a multiple of it */
    int bins_x, bins_y;          /* as oc_voronoi_acc */
    int bin_capacity;            /* >= bins_x * bins_y + 1 */
    int agent_capacity;          /* >= N */
} oc_vormap_acc;
/* Adds one frame of the crowd (N agents; NULL arrays allowed when N = 0) to acc.  Asynchronous on stream.  The
 * accumulators are caller-owned and initialised by the caller (zeros).  OC_ERR_ARG, before any launch, for a NULL
 * required pointer, a cutoff that is not finite or outside (0, 100], edges outside 4..32, every < 1, bins too small or
 * too many and too small an agent capacity for N. */
int oc_vormap_accum(oc_ctx *ctx, const oc_vormap_acc *acc, int N, const double *d_x, const double *d_y,
                    const double *d_vx, const double *d_vy, const uint8_t *d_status, void *stream);
/* oc_vormap_accum for each of n members in six launches; ctxs[0] owns the member tables.  Members may differ in grid
 * shape, crowd size (0 included), cutoff, edges and bins; each result equals the member's oc_vormap_accum alone.
 * OC_ERR_ARG as oc_vormap_accum, for a member context on another device than ctxs[0] and for two members sharing a
 * bin, scratch or accumulator buffer. */
int oc_vormap_accum_multi(int n, oc_ctx *const *ctxs, const oc_vormap_acc *const *accs, const int *Ns,
                          const double *const *x, const double *const *y, const double *const *vx,
                          const double *const *vy, const uint8_t *const *status, void *stream);

/* The observers of a run loop, each nullable: density frames (acc) and their velocity maps (vel, needs acc), line
 * counts, measurement areas and their Voronoi measures. */
typedef struct {
    const oc_density_acc *density;
    const oc_velocity_acc *velocity;
    const oc_lines_acc *lines;
    const oc_areas_acc *areas;
    const oc_voronoi_acc *voronoi;
} oc_observers;
/* oc_gcfm_run_flow plus the measurement areas and their Voronoi measures (obs: every pointer nullable; obs itself
 * nullable): before step k, next to the density frame and ahead of the step's randomness, the state the step starts
 * from is measured into row simu_step0 + k.  simu_step0 + n_steps must not exceed the capacity of the areas' and the
 * Voronoi rows, checked before any step.  oc_gcfm_run_obs forwards here; this forwards to oc_gcfm_run_observed_maps. */
int oc_gcfm_run_observed(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx,
                         double *d_vy, double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key,
                         const oc_key *keys, int n_keys, uint32_t *mt_key, int *mt_pos, int *has_gauss,
                         double *cached_gauss, int n_steps, int simu_step0, int n_active0, double *const *d_rows,
                         int *exit_agent, int *exit_step, int *n_exits, int *steps_done, double *device_ms,
                         long long *pairs, const oc_observers *obs, void *stream);
/* The run loop's only implementation: oc_gcfm_run_observed plus Voronoi maps (maps, nullable): before the steps whose
 * simu_step is a multiple of maps->every, next to the density frame and ahead of the step's randomness, a frame of the
 * state the step starts from is added to maps.  maps is checked before any step.  oc_gcfm_run_observed forwards here. */
int oc_gcfm_run_observed_maps(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx,
                              double *d_vy, double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key,
                              const oc_key *keys, int n_keys, uint32_t *mt_key, int *mt_pos, int *has_gauss,
                              double *cached_gauss, int n_steps, int simu_step0, int n_active0, double *const *d_rows,
                              int *exit_agent, int *exit_step, int *n_exits, int *steps_done, double *device_ms,
                              long long *pairs, const oc_observers *obs, const oc_vormap_acc *maps, void *stream);
/* oc_gcfm_run_flow plus the measurement areas (areas, nullable): forwards to oc_gcfm_run_observed. */
int oc_gcfm_run_obs(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx, double *d_vy,
                    double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key, const oc_key *keys,
                    int n_keys, uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int n_steps,
                    int simu_step0, int n_active0, double *const *d_rows, int *exit_agent, int *exit_step, int *n_exits,
                    int *steps_done, double *device_ms, long long *pairs, const oc_density_acc *acc,
                    const oc_velocity_acc *vel, const oc_lines_acc *lines, const oc_areas_acc *areas, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* OPTIMAL_CROWDS_H */
