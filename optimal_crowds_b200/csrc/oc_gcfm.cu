// oc_gcfm.cu -- GCFM pedestrian update on sm_100a (K4 wall search, K5 per-agent terms, K6 sweep = candidate-list
// kernel + dependency-chain kernel; one CUDA graph per step; oc_gcfm_run: blocks of run-loop steps) and the
// Gaussian density splat (K7).  Compile with -fmad=false: every formula is evaluated with exactly the
// operations written here, in the reference's order, so results are bit-identical to the CPU restatement
// used by the tests (two-oracle protocol, SURVEY.md section 8c).
//
// Reference: simulations.py:252-339 (step), pedestrians.py:216-280 (agents_repulsion), :282-334
// (wall_repulsion), :121-136 (check_status), :166-191 (evolve), optimals.py:212-250 (sampler),
// simulations.py:453-487 (gaussian_density).
//
// Sweep semantics.  The reference visits agents one by one in a random permutation and updates them in
// place, so agent i sees the NEW state of every agent earlier in the permutation and the OLD state of the
// others (SURVEY.md section 0 #3).  The sweep kernel keeps those semantics exactly while running thousands
// of agents concurrently: warps draw tickets in permutation order; an agent only needs the new state of
// earlier agents that can be within the interaction cutoff, and spins on their per-agent "done" flags
// (release/acquire).  A warp only ever waits on lower tickets, which are held by resident warps or
// finished, so the schedule cannot deadlock.  The pair sum runs in ascending agent index like the
// reference's `for j in range(N)` loop (simulations.py:287-295).
#include <chrono>
#include <cmath>
#include <cstdint>
#include <algorithm>
#include <thread>
#include <vector>

#include "oc_common.h"
#include "oc_math.h"
#include "oc_rng.h"
#include "oc_vels.h"

namespace {

constexpr int WT = OC_WALL_TILE;
constexpr double DISP_MARGIN = 1.0;  // displacement per step (2 x per-axis bound) the FAST candidate search assumes (checked)
constexpr int SWEEP_WARPS = 4;       // warps per block in the sweep
constexpr int CAND_CAP = 512;        // fast path: candidates (agents within cutoff + margin of the old position) per agent
constexpr int CAND_CAP_MAX = 65536;  // exact slow path: candidate lists in global memory, 16-bit slot indices
constexpr int OUT_HDR = 8;           // ints in front of the exit ids in the host-visible step result
constexpr size_t SWEEP_SLOT_BYTES = 2 * sizeof(double) + 2 * sizeof(int) + 2 * sizeof(unsigned short);  // 28 B
constexpr size_t SWEEP_SMEM = (size_t)SWEEP_WARPS * CAND_CAP * SWEEP_SLOT_BYTES;  // 56 KB: 4 CTAs (16 warps) per SM
static_assert(CAND_CAP <= 65536, "slot indices are stored as 16-bit");

struct KeyDev {
    const double *V;
    const uint8_t *tiles;
    const double *vx, *vy;
    const double *phi;  // alternative field storage: phi samples, differentiated on the fly
    int nt_opt, n_slices, door_off, n_doors, n_phi;
    double off_min;  // v_min * 10e3
    double mu, lim;
    int phi_row0, phi_rows;  // node rows held by every phi slice (phi_rows = 0: the whole grid)
};

struct Ws {  // device workspace carved out of ctx->gcfm_ws
    double4 *snap4, *live4;                 // packed (x,y,vx,vy): snapshot at step start / state after the agent's turn
    double4 *cell_state;                    // snapshot of the agents in cell-list order (coalesced candidate scan)
    int2 *cell_jr;                          // (agent id, sweep rank) in cell-list order
    double *x0, *y0, *vx0, *vy0;            // snapshot at step start (SoA, used by prepare)
    double *des_x, *des_y, *wfx, *wfy;      // per-agent precomputed terms
    double *noise;                          // (N,2) device copy, consumption order
    double *doors;                          // flattened door rectangles of all keys
    int *perm, *rank, *nzidx, *flags, *exit_mark, *agent_bin, *cell_agents, *bin_start, *bin_cursor;
    uint8_t *status0;
    long long *wall_ind;  // flat index of the nearest wall node (wall_search_kernel -> agent_terms_kernel)
    // two-kernel sweep: per agent the candidate list in processing order, (agent j, position in the summation order),
    // LIST_CAP entries; (candidates, of which later in the sweep); (|v|, a_i, b_i, beta_i) of pedestrians.py:242-243,267
    int2 *lst, *lhdr;
    double4 *ell;
    // [0] done-flag generation (tag) of the attempt [1] simu_step; uploaded in front of perm / noise in one copy, so that a
    // captured graph of the step has no per-step kernel arguments
    int *hdr;
    double *time0;   // per-agent clock at step start (restored when a step is redone on the exact slow path)
    KeyDev *keys;
    // [0] ticket [1] flags: bit0 sampler range, bit1 list overflow, bit2 displacement > margin [2] interacting pairs
    // evaluated (pair_force calls) [3] largest candidate count [4..5] largest per-axis displacement (bits of a double)
    int *counters;
};

__device__ __forceinline__ int ld_acquire(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int *p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// CPython / numpy float floor division (exact floor of the real quotient; fmod is exact)
__device__ __forceinline__ double py_floordiv(double vx, double wx) {
    double mod = fmod(vx, wx);
    double div = (vx - mod) / wx;
    if (mod != 0.0) {
        if ((wx < 0) != (mod < 0)) div -= 1.0;
    }
    if (div != 0.0) {
        double fl = floor(div);
        if (div - fl > 0.5) fl += 1.0;
        return fl;
    }
    return copysign(0.0, vx / wx);
}

// optimals.py:234-248, one axis of the sampler's index rule, for the sampler and for the owner of an agent in a
// row-decomposed run alike: the (up to) two indices k0, k1 into the interior field (n - 2 nodes along the axis) with the
// top clamp, CPython's floor division and numpy's wrap of a negative index (an agent at c < 0, where k1 == k0).  The
// result can still be out of range (the reference raises IndexError): the caller checks it.
__device__ __forceinline__ void sampler_axis(double c, double extent, double step, int n, long long &k0, long long &k1) {
    if (c < extent - step) {
        k0 = (long long)py_floordiv(c, step);
        k1 = (c > step) ? k0 + 1 : k0;
    } else {
        k0 = k1 = n - 3;
    }
    if (k0 < 0) { k0 += n - 2; k1 = k0; }  // silently, no exception (App. C #7)
}

// optimals.py:212-250 -- returns 1 if the reference would raise IndexError (negative indices wrap like numpy's)
__device__ int choose_velocity(const oc_gcfm_params &p, const KeyDev &k, double x, double y, int t, double &ox,
                               double &oy) {
    ox = 0.0;
    oy = 0.0;
    if (t >= k.nt_opt - 1) return 0;
    long long j0, j1, i0, i1;
    sampler_axis(x, p.room_length, p.dx, p.Nx, j0, j1);
    sampler_axis(y, p.room_height, p.dy, p.Ny, i0, i1);
    const int W = p.Nx - 2, H = p.Ny - 2;
    if (j0 < 0 || j1 >= W || i0 < 0 || i1 >= H || t < 0) return 1;
    double ax, ay, bx, by;
    if (k.vx) {
        if (t >= k.n_slices) return 1;
        const double *sx = k.vx + (size_t)t * W * H, *sy = k.vy + (size_t)t * W * H;
        ax = sx[i0 * W + j0]; ay = sy[i0 * W + j0];
        bx = sx[i1 * W + j1]; by = sy[i1 * W + j1];
    } else {
        // vx_opt[t] = vels(sol.y[:, nt_opt-1-t]) (optimals.py:200-204), evaluated at the two sampled nodes
        const int kd = k.nt_opt - 1 - t;
        if (kd < 0 || kd >= k.n_phi) return 1;
        // slices hold the whole grid or (row-decomposed runs) node rows [phi_row0, phi_row0 + phi_rows)
        const int rows = k.phi_rows ? k.phi_rows : p.Ny, row0 = k.phi_rows ? k.phi_row0 : 0;
        if (i0 < row0 || i1 + 2 >= row0 + rows) return 1;  // not this band's agent (the caller only asks for its own)
        const double *ph = k.phi + (size_t)kd * rows * p.Nx - (long long)row0 * p.Nx;
        const double i2x = 1.0 / (2 * p.dx), i2y = 1.0 / (2 * p.dy);
        {
            const double *c = ph + (size_t)(i0 + 1) * p.Nx + (j0 + 1);
            vels_point(clamp_lim(c[0], k.lim), clamp_lim(c[-1], k.lim), clamp_lim(c[1], k.lim),
                       clamp_lim(c[-p.Nx], k.lim), clamp_lim(c[p.Nx], k.lim), k.mu, k.lim, i2x, i2y, ax, ay);
        }
        {
            const double *c = ph + (size_t)(i1 + 1) * p.Nx + (j1 + 1);
            vels_point(clamp_lim(c[0], k.lim), clamp_lim(c[-1], k.lim), clamp_lim(c[1], k.lim),
                       clamp_lim(c[-p.Nx], k.lim), clamp_lim(c[p.Nx], k.lim), k.mu, k.lim, i2x, i2y, bx, by);
        }
    }
    if (j0 == j1 && i0 == i1) {
        ox = ax;
        oy = ay;
    } else {  // two fancy-index lists pair up element-wise: (i0,j0),(i1,j1); np.mean = (a+b)/2
        ox = (ax + bx) / 2.0;
        oy = (ay + by) / 2.0;
    }
    return 0;
}

struct AgentEllipse {  // quantities of agent i that do not depend on the partner (pedestrians.py:242-243,267)
    double ni, a_i, b_i, beta_i;
};
__device__ __forceinline__ AgentEllipse ellipse_of(const oc_gcfm_params &p, double vx, double vy, double v_des) {
    AgentEllipse e;
    e.ni = ocm_norm2(vx, vy);
    e.a_i = p.a_min + p.tau_a * e.ni;
    e.b_i = p.b_max - (p.b_max - p.b_min) * ocm_npmin(e.ni / v_des, 1.0);
    e.beta_i = ocm_atan2(vy, vx);
    return e;
}

// pedestrians.py:237-280
__device__ void pair_force(const oc_gcfm_params &p, const AgentEllipse &ei, double xi, double yi, double vxi,
                           double vyi, double v_des_i, double xj, double yj, double vxj, double vyj, double &fx,
                           double &fy) {
    double nj = ocm_norm2(vxj, vyj);
    double a_j = p.a_min + p.tau_a * nj;
    double b_j = p.b_max - (p.b_max - p.b_min) * ocm_npmin(nj / v_des_i, 1.0);  // v_des of i: pedestrians.py:245
    double Rx = xj - xi, Ry = yj - yi;
    double nR = ocm_norm2(Rx, Ry);
    double ex = Rx / nR, ey = Ry / nR;
    double wx = vxj - vxi, wy = vyj - vyi;
    double d = wx * (-ex) + wy * (-ey);
    double v_rel = 0.5 * (d + fabs(d));
    double k = 0.0;
    if (ei.ni > 0) k = ocm_npmax((vxi * ex + vyi * ey) / ei.ni - p.cos_fov, 0.0) / p.one_minus_cos_fov;
    // alpha_i = atan2(Ry,Rx), alpha_j = atan2(-Ry,-Rx): one arctangent core, same bits as two calls
    double alpha_i, alpha_j;
    ocm_atan2_both(Ry, Rx, &alpha_i, &alpha_j);
    double beta_j = ocm_atan2(vyj, vxj);
    double sni, csi, snj, csj;
    ocm_sincos(alpha_i - ei.beta_i, &sni, &csi);
    ocm_sincos(alpha_j - beta_j, &snj, &csj);
    double ci = csi / ei.a_i, si = sni / ei.b_i;
    double q_i = sqrt(1.0 / (ci * ci + si * si));
    double cj = csj / a_j, sj = snj / b_j;
    double q_j = sqrt(1.0 / (cj * cj + sj * sj));
    double dist = nR - q_i - q_j;
    double rep = ocm_npmin(k * ocm_exp(-dist / (p.eta * (1.0 + v_rel))), 1.0);
    fx = -rep * Rx;
    fy = -rep * Ry;
}

// pedestrians.py:315-334 given the nearest wall node (wxp, wyp)
__device__ void wall_force_from_node(const oc_gcfm_params &p, const AgentEllipse &ei, double xi, double yi,
                                     double vxi, double vyi, double wxp, double wyp, double &fx, double &fy) {
    double Rx = wxp - xi, Ry = wyp - yi;
    double nR = ocm_norm2(Rx, Ry);
    double ex = Rx / nR, ey = Ry / nR;
    double d = vxi * ex + vyi * ey;
    double v_rel = 0.5 * (d + fabs(d));
    double alpha = ocm_atan2(Ry, Rx);
    double sn, cs;
    ocm_sincos(alpha - ei.beta_i, &sn, &cs);
    double c = cs / ei.a_i, s = sn / ei.b_i;
    double q_i = 1.0 / (c * c + s * s);  // no sqrt: pedestrians.py:328
    double dist = nR - q_i;
    double rep = ocm_npmin(ocm_exp(-dist / (p.eta_walls * (1.0 + v_rel))), 1.0);
    fx = -3.0 * rep * Rx;
    fy = -3.0 * rep * Ry;
}

// K4: exact np.argmin(sqrt((X-x)^2+(Y-y)^2) + V*10e3) (pedestrians.py:311-313), one warp per agent.
// Only nodes with V<0 can win (their offset is <= -|pot|*1e4, the host checks that this exceeds the room
// diagonal).  Returns the flat index (first index among equal keys, like np.argmin) on every lane.
//
// Search (round 2, v2).  tiles[] holds per WT x WT node tile 1 + the ring distance (in tiles) to the nearest tile with a
// wall node, so the rings below that distance are skipped.  Phase 1 scans the first ring that holds wall nodes, which
// gives an upper bound `wbest` of the minimum key.  Phase 2 then determines in ONE step the last ring K that can still
// hold a node with a key <= wbest (the rounded distance to anything outside the square of radius K exceeds it) and
// scans the tiles of rings k+1..K that (a) hold wall nodes and (b) whose nearest possible node is not farther than
// wbest -- occupancy bytes of up to 128 tiles per memory round trip, two tiles (16 independent loads per lane) per round
// trip of the node scan.  The result is the global argmin whatever superset of the necessary tiles is scanned, so the
// pruning only has to be conservative: for a node of a tile, |X[ix] - x| >= gx := max(X[ix0] - x, x - X[ix1], 0) in
// floating point as well (rounding is monotonic), hence its computed distance is >= sqrt(gx*gx + gy*gy) evaluated with
// the same operations, and its key >= that + off_min (the most negative potential x 10e3).
template <bool PAIR>
struct WallSearch {
    const double *__restrict__ X, *__restrict__ Y, *__restrict__ V;
    const uint8_t *__restrict__ tiles;
    int Ny, Nx, ntx, nty, lane;
    double x, y, off_min;
    double best, wbest;
    long long best_i;

    __device__ __forceinline__ double tile_lb(int ttx, int tty) const {
        const int ix0 = ttx * WT, ix1 = min(ix0 + WT - 1, Nx - 1), iy0 = tty * WT, iy1 = min(iy0 + WT - 1, Ny - 1);
        const double gx = fmax(fmax(X[ix0] - x, x - X[ix1]), 0.0), gy = fmax(fmax(Y[iy0] - y, y - Y[iy1]), 0.0);
        return sqrt(gx * gx + gy * gy);
    }
    // strict: a node with an equal key and a lower flat index would win the tie
    __device__ __forceinline__ bool cannot_win(double lb) const { return wbest < lb * (1.0 - 0x1p-50) + off_min; }
    __device__ __forceinline__ void load_tile(int ttx, int tty, double (&vv)[8]) const {
        static_assert(WT * WT == 8 * 32, "tile scan: 8 nodes per lane");
        // nodes c = lane, lane + 32, ...: coalesced rows of the tile, ascending flat index inside a lane
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int c = lane + 32 * q, iy = tty * WT + c / WT, ix = ttx * WT + (c % WT);
            vv[q] = (iy < Ny && ix < Nx) ? __ldg(V + (size_t)iy * Nx + ix) : 0.0;
        }
    }
    __device__ __forceinline__ void eval_tile(int ttx, int tty, const double (&vv)[8]) {
        const int ix = ttx * WT + (lane % WT);
        const double ddx = (ix < Nx) ? X[ix] - x : 0.0;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            if (vv[q] < 0) {
                const int iy = tty * WT + (lane + 32 * q) / WT;
                const double ddy = Y[iy] - y;
                const double key = sqrt(ddx * ddx + ddy * ddy) + vv[q] * 10e3;
                const long long fi = (long long)iy * Nx + ix;
                if (key < best || (key == best && fi < best_i)) { best = key; best_i = fi; }
            }
        }
    }
    __device__ __forceinline__ void refresh_wbest() {
        double wb = best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wb = fmin(wb, __shfl_xor_sync(0xffffffffu, wb, o));
        wbest = wb;
    }
    // position r on ring k (border of the (2k+1)^2 tile square around (tcx, tcy)) -> tile
    __device__ __forceinline__ static void ring_tile(int tcx, int tcy, int k, int r, int &tx, int &ty) {
        const int side = 2 * k + 1;
        if (k == 0) { tx = tcx; ty = tcy; }
        else if (r < side) { tx = tcx - k + r; ty = tcy - k; }
        else if (r < 2 * side) { tx = tcx - k + (r - side); ty = tcy + k; }
        else if (r < 2 * side + (side - 2)) { tx = tcx - k; ty = tcy - k + 1 + (r - 2 * side); }
        else { tx = tcx + k; ty = tcy - k + 1 + (r - 2 * side - (side - 2)); }
    }
    // scan the tiles of rings ka..kb that hold wall nodes and can still win
    __device__ void scan_rings(int tcx, int tcy, int ka, int kb) {
        int total = 0;
        for (int k = ka; k <= kb; k++) total += (k == 0) ? 1 : 8 * k;
        constexpr int U = 2;
        for (int base = 0; base < total; base += 32 * U) {
            int tx[U], ty[U];
            double lb[U];
            bool cand[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                int t = base + 32 * u + lane, k = ka;
                tx[u] = ty[u] = -1;
                if (t < total) {
                    while (t >= ((k == 0) ? 1 : 8 * k)) { t -= (k == 0) ? 1 : 8 * k; k++; }
                    ring_tile(tcx, tcy, k, t, tx[u], ty[u]);
                }
                cand[u] = tx[u] >= 0 && tx[u] < ntx && ty[u] >= 0 && ty[u] < nty && tiles[ty[u] * ntx + tx[u]] == 1;
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                lb[u] = 0.0;
                if (cand[u]) {
                    lb[u] = tile_lb(tx[u], ty[u]);
                    cand[u] = !cannot_win(lb[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                unsigned todo = __ballot_sync(0xffffffffu, cand[u]);
                while (todo) {
                    // up to two tiles per memory round trip; a tile that the bound found meanwhile rules out is dropped
                    int ax = -1, ay = -1, bx = -1, by = -1;
                    while (todo && (PAIR ? bx < 0 : ax < 0)) {
                        const int src = __ffs(todo) - 1;
                        todo &= todo - 1;
                        const double l = __shfl_sync(0xffffffffu, lb[u], src);
                        const int sx_ = __shfl_sync(0xffffffffu, tx[u], src), sy_ = __shfl_sync(0xffffffffu, ty[u], src);
                        if (cannot_win(l)) continue;
                        if (ax < 0) { ax = sx_; ay = sy_; } else { bx = sx_; by = sy_; }
                    }
                    if (ax < 0) break;
                    double va[8];
                    load_tile(ax, ay, va);
                    if (PAIR) {
                        double vb[8];
                        if (bx >= 0) load_tile(bx, by, vb);
                        eval_tile(ax, ay, va);
                        if (bx >= 0) eval_tile(bx, by, vb);
                    } else {
                        eval_tile(ax, ay, va);
                    }
                    refresh_wbest();
                }
            }
        }
    }
};

template <bool PAIR>
__device__ long long wall_argmin_warp(const double *__restrict__ X, const double *__restrict__ Y,
                                      const double *__restrict__ V, const uint8_t *__restrict__ tiles, int Ny,
                                      int Nx, double x, double y, double off_min) {
    WallSearch<PAIR> ws;
    ws.X = X; ws.Y = Y; ws.V = V; ws.tiles = tiles; ws.Ny = Ny; ws.Nx = Nx;
    ws.lane = threadIdx.x & 31;
    ws.ntx = (Nx + WT - 1) / WT; ws.nty = (Ny + WT - 1) / WT;
    ws.x = x; ws.y = y; ws.off_min = off_min;
    ws.best = INFINITY; ws.wbest = INFINITY; ws.best_i = (long long)Ny * Nx;
    const int ntx = ws.ntx, nty = ws.nty, lane = ws.lane;
    // tile containing the node nearest to (x,y); any centre is correct, a near one is fast
    const double sx = X[1] - X[0], sy = Y[1] - Y[0];
    int cx = (int)fmin(fmax(x / sx, 0.0), (double)(Nx - 1)), cy = (int)fmin(fmax(y / sy, 0.0), (double)(Ny - 1));
    const int tcx = cx / WT, tcy = cy / WT;
    const int kmax = max(max(tcx, ntx - 1 - tcx), max(tcy, nty - 1 - tcy));
    // tiles[t] = 1 + (ring distance, in tiles, from t to the nearest tile holding a wall node, capped at RING_CAP):
    // the rings below that distance are known to be empty and are skipped (no memory round trips for them)
    int k = max(min((int)tiles[tcy * ntx + tcx] - 1, kmax), 0);
    // (one call site of scan_rings for both phases: the scan is inlined once)
    int ka = k, kb = k;
    bool last = false;
    for (;;) {
        ws.scan_rings(tcx, tcy, ka, kb);
        if (last || kb >= kmax) break;
        if (!(ws.wbest < INFINITY)) {  // ---- phase 1: ring by ring until one holds a wall node
            ka = kb = kb + 1;
            continue;
        }
        // ---- phase 2: last ring K that can hold a node with a key <= wbest.  ring_lb(kk) = lower bound of the distance
        // to any node outside the square of radius kk (32 radii per round trip, one per lane)
        int K = kmax;
        for (int k2 = kb; k2 <= kmax; k2 += 32) {
            const int kk = k2 + lane;
            bool stop = false;
            if (kk <= kmax) {
                double lb = INFINITY;
                const int ix_lo = (tcx - kk) * WT - 1, ix_hi = (tcx + kk + 1) * WT, iy_lo = (tcy - kk) * WT - 1,
                          iy_hi = (tcy + kk + 1) * WT;
                if (ix_lo >= 0) lb = fmin(lb, x - X[ix_lo]);
                if (ix_hi < Nx) lb = fmin(lb, X[ix_hi] - x);
                if (iy_lo >= 0) lb = fmin(lb, y - Y[iy_lo]);
                if (iy_hi < Ny) lb = fmin(lb, Y[iy_hi] - y);
                stop = lb == INFINITY || ws.cannot_win(lb);
            }
            const unsigned m = __ballot_sync(0xffffffffu, stop);
            if (m) { K = k2 + __ffs(m) - 1; break; }
        }
        if (K <= kb) break;
        ka = kb + 1;
        kb = K;
        last = true;
    }
    double best = ws.best;
    long long best_i = ws.best_i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ob = __shfl_xor_sync(0xffffffffu, best, o);
        long long oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (ob < best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
    }
    return best_i;
}

// ------------------------------------------------------------------------------------------------ kernels
__global__ void tiles_kernel(const double *__restrict__ V, int Ny, int Nx, uint8_t *__restrict__ tiles,
                             double *__restrict__ vmin_out) {
    // one warp per tile
    const int ntx = (Nx + WT - 1) / WT, nty = (Ny + WT - 1) / WT;
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= ntx * nty) return;
    int ty = w / ntx, tx = w % ntx;
    int any = 0;
    double vm = INFINITY;
    for (int c = lane; c < WT * WT; c += 32) {
        int iy = ty * WT + c / WT, ix = tx * WT + (c % WT);
        if (iy < Ny && ix < Nx) {
            double v = V[(size_t)iy * Nx + ix];
            any |= (v < 0);
            vm = fmin(vm, v);
        }
    }
    any = __any_sync(0xffffffffu, any);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vm = fmin(vm, __shfl_xor_sync(0xffffffffu, vm, o));
    if (lane == 0) {
        tiles[w] = (uint8_t)any;
        vmin_out[w] = vm;
    }
}

// ring distance (Chebyshev, in tiles, capped) from every tile to the nearest occupied tile; out = 1 + distance
constexpr int RING_CAP = 64;
__global__ void tile_ring_kernel(const uint8_t *__restrict__ occ, int ntx, int nty, uint8_t *__restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntx * nty) return;
    const int ty = t / ntx, tx = t % ntx;
    int d = RING_CAP;
    for (int k = 0; k < RING_CAP && d == RING_CAP; k++) {
        bool hit = false;
        for (int q = -k; q <= k && !hit; q++) {
            const int xs = tx + q, ys = ty + q;
            if (xs >= 0 && xs < ntx) {
                if (ty - k >= 0 && occ[(ty - k) * ntx + xs]) hit = true;
                if (ty + k < nty && occ[(ty + k) * ntx + xs]) hit = true;
            }
            if (ys >= 0 && ys < nty) {
                if (tx - k >= 0 && occ[ys * ntx + tx - k]) hit = true;
                if (tx + k < ntx && occ[ys * ntx + tx + k]) hit = true;
            }
        }
        if (hit) d = k;
    }
    out[t] = (uint8_t)(1 + d);
}

// rank = inverse permutation; snapshot; bin histogram
__device__ __forceinline__ void setup_body(int N, const double *__restrict__ x, const double *__restrict__ y,
                                           const double *__restrict__ vx, const double *__restrict__ vy,
                                           const double *__restrict__ tim, const uint8_t *__restrict__ status, const Ws &w,
                                           double inv_cs, int nbx, int nby) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    w.rank[w.perm[i]] = i;
    double xi = x[i], yi = y[i];
    const double vxi = vx[i], vyi = vy[i];
    w.x0[i] = xi; w.y0[i] = yi; w.vx0[i] = vxi; w.vy0[i] = vyi;
    w.snap4[i] = make_double4(xi, yi, vxi, vyi);
    uint8_t s = status[i];
    w.status0[i] = s;
    w.time0[i] = tim[i];
    if (s && !(fabs(vxi) < 16.0 && fabs(vyi) < 16.0)) w.counters[6] = 1;  // `wild`: the sweep then culls nothing
    int bx = min(max((int)floor(xi * inv_cs), 0), nbx - 1), by = min(max((int)floor(yi * inv_cs), 0), nby - 1);
    int b = by * nbx + bx;
    w.agent_bin[i] = b;
    if (s) atomicAdd(&w.bin_start[b + 1], 1);  // histogram shifted by one: scanned in place afterwards
}

// single-block inclusive scan in place over a[0..n) (a[0] must be 0 => exclusive offsets)
__device__ __forceinline__ void scan_body(int *a, int n) {
    __shared__ int tot[1024];
    int t = threadIdx.x;
    int per = (n + 1023) / 1024;
    int lo = min(t * per, n), hi = min(lo + per, n);
    int s = 0;
    for (int i = lo; i < hi; i++) s += a[i];
    tot[t] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        int v = (t >= o) ? tot[t - o] : 0;
        __syncthreads();
        tot[t] += v;
        __syncthreads();
    }
    int run = tot[t] - s;
    for (int i = lo; i < hi; i++) { run += a[i]; a[i] = run; }
}

__device__ __forceinline__ void scatter_body(int N, const Ws &w) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N || !w.status0[i]) return;
    int b = w.agent_bin[i];
    int pos = w.bin_start[b] + atomicAdd(&w.bin_cursor[b], 1);
    w.cell_agents[pos] = i;
    w.cell_state[pos] = w.snap4[i];
    w.cell_jr[pos] = make_int2(i, w.rank[i]);
}

// undo a step that the fast path could not complete exactly (candidate-list overflow or a displacement beyond the
// search margin): the state goes back to the snapshot taken by setup_kernel, then the step is redone (slow path)
__global__ void restore_kernel(int N, Ws w, double *__restrict__ x, double *__restrict__ y, double *__restrict__ vx,
                               double *__restrict__ vy, double *__restrict__ tim, uint8_t *__restrict__ status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const double4 s = w.snap4[i];
    x[i] = s.x; y[i] = s.y; vx[i] = s.z; vy[i] = s.w;
    tim[i] = w.time0[i];
    status[i] = w.status0[i];
    if (i == 0) {  // the sampler-range flag (bit 0, set by agent_terms_kernel) survives a redo; everything else restarts
        w.counters[0] = 0;
        w.counters[1] &= 1;
        for (int q = 2; q < 8; q++) w.counters[q] = 0;
    }
}

// nzidx[agent] = number of agents active at step start that precede it in the sweep (simulations.py:303
// draws one normal pair per active agent in sweep order).  Single block.
__device__ __forceinline__ void noise_index_body(int N, const Ws &w) {
    __shared__ int tot[1024];
    int t = threadIdx.x;
    int per = (N + 1023) / 1024;
    int lo = min(t * per, N), hi = min(lo + per, N);
    int s = 0;
    for (int r = lo; r < hi; r++) s += w.status0[w.perm[r]];
    tot[t] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        int v = (t >= o) ? tot[t - o] : 0;
        __syncthreads();
        tot[t] += v;
        __syncthreads();
    }
    int run = tot[t] - s;
    for (int r = lo; r < hi; r++) {
        int a = w.perm[r];
        w.nzidx[a] = run;
        run += w.status0[a];
    }
}

// K5: per-agent terms that depend only on the agent's own old state: desired velocity (sampler) and wall force.
// Two kernels: the nearest-wall search with one WARP per agent (memory-latency bound: few registers, many resident
// warps), then sampler + wall force with one THREAD per agent (round 1 ran them on lane 0 of the search warp).
__device__ __forceinline__ bool agent_owned(const oc_gcfm_params &p, int key, double yi) {
    // key-sharded run: the rank that solved this agent's target set evaluates it
    if (p.key_mod > 0 && key % p.key_mod != p.key_rem) return false;
    if (p.own1 > p.own0) {
        // row-decomposed run: the rank whose band holds node row i0 + 1 of the sampler's (wrapped) row indices; its phi
        // slices hold node rows own0 - 1 .. own1 + 1, i.e. every row the sampler reads (i0 .. i1 + 2).  A row index the
        // sampler refuses is clamped into the grid: the sampler raises the range flag before it reads anything, so any
        // single owner will do
        long long i0, i1;
        sampler_axis(yi, p.room_height, p.dy, p.Ny, i0, i1);
        const long long orow = i0 + 1 < 0 ? 0 : (i0 + 1 > p.Ny - 1 ? p.Ny - 1 : i0 + 1);
        if (orow < p.own0 || orow >= p.own1) return false;
    }
    return true;
}
template <bool PAIR>
__device__ __forceinline__ void wall_search_body(const oc_gcfm_params &p, int N, const Ws &w,
                                                 const double *__restrict__ X, const double *__restrict__ Y,
                                                 const int *__restrict__ key_id) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= N || !w.status0[i]) return;
    const int key = key_id[i];
    const double xi = w.x0[i], yi = w.y0[i];
    if (!agent_owned(p, key, yi)) return;
    const KeyDev *k = w.keys + key;
    const long long ind = wall_argmin_warp<PAIR>(X, Y, k->V, k->tiles, p.Ny, p.Nx, xi, yi, k->off_min);
    if ((threadIdx.x & 31) == 0) w.wall_ind[i] = ind;
}
__device__ __forceinline__ void agent_terms_body(const oc_gcfm_params &p, int N, const Ws &w,
                                                 const double *__restrict__ X, const double *__restrict__ Y,
                                                 const double *__restrict__ vdes, const int *__restrict__ key_id,
                                                 int simu_step) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N || !w.status0[i]) return;
    const int key = key_id[i];
    const double xi = w.x0[i], yi = w.y0[i], vxi = w.vx0[i], vyi = w.vy0[i];
    if (!agent_owned(p, key, yi)) {  // all-zero bits for the bit-exact merge over the ranks
        w.des_x[i] = 0.0; w.des_y[i] = 0.0; w.wfx[i] = 0.0; w.wfy[i] = 0.0;
        return;
    }
    const KeyDev k = w.keys[key];
    long long ind = w.wall_ind[i];
    if (ind < 0 || ind >= (long long)p.Ny * p.Nx) ind = 0;  // no comparable key at all (NaN position): np.argmin gives 0
    double ux, uy;
    const int bad = choose_velocity(p, k, xi, yi, simu_step, ux, uy);
    if (bad) atomicOr(&w.counters[1], 1);
    w.des_x[i] = vdes[i] * ux;  // simulations.py:281
    w.des_y[i] = vdes[i] * uy;
    const AgentEllipse ei = ellipse_of(p, vxi, vyi, vdes[i]);
    double fx, fy;
    wall_force_from_node(p, ei, xi, yi, vxi, vyi, X[ind % p.Nx], Y[ind / p.Nx], fx, fy);
    w.wfx[i] = fx;
    w.wfy[i] = fy;
}

// ascending bitonic sort of a[0..n) (64-bit keys, n <= m2 = power of two, a[n..m2) is overwritten with padding) by one warp
__device__ __forceinline__ void warp_sort_u64(unsigned long long *a, int n, int lane) {
    int m2 = 1;
    while (m2 < n) m2 <<= 1;
    for (int t = n + lane; t < m2; t += 32) a[t] = ~0ull;
    __syncwarp();
    for (int k = 2; k <= m2; k <<= 1)
        for (int jj = k >> 1; jj > 0; jj >>= 1) {
            for (int t = lane; t < m2; t += 32) {
                const int u = t ^ jj;
                if (u > t) {
                    const unsigned long long x = a[t], y = a[u];
                    if ((x > y) == ((t & k) == 0)) { a[t] = y; a[u] = x; }
                }
            }
            __syncwarp();
        }
}

// Candidate search of one agent (stage A of the sweep), shared by the one-kernel sweep and the two-kernel path.
struct CandSearch {
    int span;
    double rho_s, reach2, sin_fov, cos_fov;
    bool cull_ok;
    __device__ __forceinline__ CandSearch(const oc_gcfm_params &p, const Ws &w, double margin, double inv_cs, int fov_cull) {
        const double reach = p.cutoff + margin;
        const int span = (int)ceil(reach * inv_cs);
        // No agent moves more than margin/2 per axis in one step (checked below; a violation voids the attempt), i.e. not
        // more than rho = margin/sqrt(2).  A candidate can therefore only come within the cutoff if its OLD position is
        // within cutoff + rho of i's old position ...
        const double rho_s = margin * 0.70710678118654757 * (1.0 + 1e-6) + 1e-12;
        const double reach_c = p.cutoff + rho_s + 1e-9, reach2 = reach_c * reach_c;
        // ... and can only be inside i's field of view (k > 0, pedestrians.py:259-262) if the direction to its old position
        // is within the half-angle of the field of view plus the angle asin(rho/d) that a disc of radius rho subtends.  A
        // candidate outside contributes exactly -+0.0 whatever its new state is (k = 0 and exp(.) finite), so it is neither
        // waited for nor evaluated.  Only applied when every quantity involved is tame, so that 0 * exp(.) cannot be NaN:
        // setup_kernel's `wild` flag (counters[6]: some |velocity component| >= 16 m/s or NaN) is clear, the semi-axes are
        // positive and bounded (q <= max(a, b), a <= a_min + 23 tau_a, b in [b_min, b_max] for v_des > 0) and
        // (q_i + q_j)/eta stays below the overflow threshold of exp; otherwise every candidate within reach is kept.
        const double sin_fov = sqrt(fmax(1.0 - p.cos_fov * p.cos_fov, 0.0));
        const bool cull_ok = fov_cull && w.counters[6] == 0 && p.cos_fov < 0.0 && p.cos_fov > -1.0 && p.v_max <= 16.0 &&
                             p.a_min > 0.0 && p.tau_a >= 0.0 && p.b_min > 0.0 && p.b_max >= p.b_min &&
                             2.0 * (p.a_min + 23.0 * p.tau_a) + 2.0 * p.b_max < 600.0 * p.eta;
        this->span = span; this->rho_s = rho_s; this->reach2 = reach2; this->sin_fov = sin_fov; this->cos_fov = p.cos_fov;
        this->cull_ok = cull_ok;
    }
    // fills ckk / cj / the two sort-key lists for agent i (sweep rank r); returns the number of candidates kept (<= cap;
    // on overflow the attempt is flagged void and the list truncated)
    __device__ __forceinline__ int gather(const oc_gcfm_params &p, const Ws &w, int i, int r, double xi, double yi,
                                          double vxi, double vyi, double vd, double ni, int nbx, int nby, int cap,
                                          int *ckk, int *cj, unsigned long long *sort_a, unsigned long long *sort_b) const {
        const int lane = threadIdx.x & 31;
        const unsigned lt_mask = (1u << lane) - 1;
        const bool do_cull = cull_ok && ni < 32.0 && vd > 0.0;  // (false for a NaN speed; v_des > 0 keeps b_i, b_j in [b_min, b_max])
        // ---- A. candidates.  Each of the (2 span + 1) bin rows is one contiguous range of the cell list; lanes fetch the
        // range bounds in parallel, then the concatenated ranges are scanned 32 entries at a time.
        int nc = 0;
        const int b = w.agent_bin[i];
        const int bix = b % nbx, biy = b / nbx;
        const int by0 = max(biy - span, 0), nrows = min(biy + span, nby - 1) - by0 + 1;
        int my_beg = 0, my_len = 0;
        if (lane < nrows) {
            const int by = by0 + lane;
            my_beg = w.bin_start[by * nbx + max(bix - span, 0)];
            my_len = w.bin_start[by * nbx + min(bix + span, nbx - 1) + 1] - my_beg;  // bins of one row are contiguous
        }
        int my_off = my_len;  // inclusive scan over the (few) rows
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, my_off, o);
            if (lane >= o) my_off += v;
        }
        const int total = __shfl_sync(0xffffffffu, my_off, 7);  // nrows <= 7
        my_off -= my_len;                                        // exclusive
        for (int base_t = 0; base_t < total; base_t += 32) {
            const int t = base_t + lane;
            int kk = -1;
            for (int q = 0; q < nrows; q++) {
                const int o = __shfl_sync(0xffffffffu, my_off, q), l = __shfl_sync(0xffffffffu, my_len, q),
                          bq = __shfl_sync(0xffffffffu, my_beg, q);
                if (t >= o && t < o + l) kk = bq + (t - o);
            }
            bool keep = false;
            int2 jr = make_int2(-1, 0);
            if (kk >= 0) {
                const double2 pj = *reinterpret_cast<const double2 *>(w.cell_state + kk);  // (x, y)
                const double ox = pj.x - xi, oy = pj.y - yi;
                const double d2 = ox * ox + oy * oy;
                if (d2 < reach2) {
                    bool cull = false;
                    if (do_cull) {
                        if (ni == 0.0) cull = true;  // k = 0 (pedestrians.py:259-261)
                        else {
                            const double d = sqrt(d2), sn = rho_s / d;
                            if (sn < 0.999 * sin_fov) {  // fov half-angle + asin(sn) stays below pi
                                const double cs = sqrt(1.0 - sn * sn);
                                const double cos_lim = p.cos_fov * cs - sin_fov * sn;  // cos(fov half-angle + asin(sn))
                                cull = (vxi * ox + vyi * oy) / (ni * d) < cos_lim - 1e-9;
                            }
                        }
                    }
                    if (!cull) {
                        jr = w.cell_jr[kk];
                        keep = jr.x != i;  // j != i (simulations.py:291)
                    }
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            const bool later = jr.y > r;
            if (keep) {
                const int pos = nc + __popc(m & lt_mask);
                if (pos < cap) {
                    ckk[pos] = kk;
                    cj[pos] = jr.x;
                    // processing key: later candidates first (key 0), earlier ones by ascending sweep rank
                    sort_a[pos] = ((unsigned long long)(later ? 0u : (unsigned)jr.y + 1u) << 32) | (unsigned)pos;
                    sort_b[pos] = ((unsigned long long)(unsigned)jr.x << 32) | (unsigned)pos;  // summation key: agent index
                }
            }
            nc += __popc(m);
        }
        if (nc > cap) {  // uniform across the warp
            if (lane == 0) { atomicOr(&w.counters[1], 2); atomicMax(&w.counters[3], nc); }
            // too many neighbours for the lists: this attempt is void (flag; the host redoes the step with lists sized for
            // counters[3]); the agent still advances with the first `cap` candidates so that later agents do not wait forever
            nc = cap;
        }
        return nc;
    }
};

// K6: the sweep (simulations.py:271-332).  Per agent (one warp):
//  A. gather the candidates -- agents whose OLD position is within cutoff + margin of i's old position -- from the
//     cell list into shared memory (no waiting: only the immutable snapshot is read);
//  B. two sorts, still without waiting: the PROCESSING order (candidates later in the sweep first -- they are in
//     their snapshot state -- then the earlier ones by ascending sweep rank, i.e. roughly in the order in which they
//     will publish) and the SUMMATION order (ascending agent index, `for j in range(N)`, simulations.py:287);
//  C. forces, 32 candidates at a time in processing order: an earlier candidate must have finished (acquire on its
//     done-flag, which also carries its inside/exited status), then its NEW packed state is read.  Cutoff test and
//     pair force (simulations.py:291-295) go to the candidate's slot, +0.0 if it does not interact (adding +0.0 to
//     the running sum changes no bit: the sum starts at +0.0 and can never become -0.0);
//  D. ascending-j sum, Euler step, exit test, publish.
// The sweep is a chain of dependencies (an agent needs the new state of every earlier neighbour), so what matters is
// the time from "my last dependency published" to "I publish": with this ordering it is ONE batch of pair forces plus
// the sum, instead of all remaining batches plus the sort.
__device__ __forceinline__ void
sweep_body(const oc_gcfm_params &p, int N, const Ws &w, double *__restrict__ x, double *__restrict__ y,
           double *__restrict__ vx, double *__restrict__ vy, double *__restrict__ tim,
           uint8_t *__restrict__ status, const double *__restrict__ vdes, const int *__restrict__ key_id, int tag,
           double inv_cs, int nbx, int nby, unsigned poll_ns, double margin, int cap, unsigned char *glists,
           int fov_cull) {
    extern __shared__ __align__(16) unsigned char sweep_smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // per warp: fx, fy (doubles; reused as the 64-bit sort buffers before the forces exist), ckk, cj (ints), proc, ord
    // (16-bit slot indices).  Fast path: `cap` = CAND_CAP slots in shared memory; exact slow path (glists != NULL): `cap`
    // slots per warp in global memory, sized from the candidate count the refused fast attempt measured
    unsigned char *base = glists ? glists + ((size_t)blockIdx.x * SWEEP_WARPS + wid) * cap * SWEEP_SLOT_BYTES
                                 : sweep_smem + (size_t)wid * CAND_CAP * SWEEP_SLOT_BYTES;
    double *lfx = reinterpret_cast<double *>(base), *lfy = lfx + cap;
    int *ckk = reinterpret_cast<int *>(lfy + cap), *cj = ckk + cap;
    unsigned short *proc = reinterpret_cast<unsigned short *>(cj + cap), *ord = proc + cap;
    unsigned long long *sort_a = reinterpret_cast<unsigned long long *>(lfx), *sort_b = reinterpret_cast<unsigned long long *>(lfy);
    const CandSearch cs_(p, w, margin, inv_cs, fov_cull);
    const unsigned lt_mask = (1u << lane) - 1;
    int pairs_total = 0;
    for (;;) {
        int r = 0;
        if (lane == 0) r = atomicAdd(&w.counters[0], 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r >= N) break;
        const int i = w.perm[r];
        if (!w.status0[i]) continue;  // simulations.py:277
        const double4 si = w.snap4[i];
        const double xi = si.x, yi = si.y, vxi = si.z, vyi = si.w, vd = vdes[i];
        const AgentEllipse ei = ellipse_of(p, vxi, vyi, vd);
        // ---- A. candidates
        int n_later = 0;
        const int nc = cs_.gather(p, w, i, r, xi, yi, vxi, vyi, vd, ei.ni, nbx, nby, cap, ckk, cj, sort_a, sort_b);
        __syncwarp();
        // everything the final Euler step needs that does not depend on the neighbours is fetched now, so that no global
        // load sits between "last dependency published" and "I publish"
        double nz_x = 0.0, nz_y = 0.0, wf_x = 0.0, wf_y = 0.0, de_x = 0.0, de_y = 0.0, tim_i = 0.0;
        int door_off = 0, n_doors = 0;
        if (lane == 0) {
            const int nz = w.nzidx[i];
            nz_x = w.noise[2 * nz]; nz_y = w.noise[2 * nz + 1];
            wf_x = w.wfx[i]; wf_y = w.wfy[i];
            de_x = w.des_x[i]; de_y = w.des_y[i];
            tim_i = tim[i];
            const KeyDev *kp = w.keys + key_id[i];
            door_off = kp->door_off; n_doors = kp->n_doors;
        }
        // ---- B. processing order and summation order (no waiting yet)
        if (nc > 1) {
            warp_sort_u64(sort_a, nc, lane);
            warp_sort_u64(sort_b, nc, lane);
        }
        for (int t0 = 0; t0 < nc; t0 += 32) {
            const int t = t0 + lane;
            bool is_later = false;
            if (t < nc) {
                const unsigned long long ka = sort_a[t];
                proc[t] = (unsigned short)ka;
                ord[t] = (unsigned short)sort_b[t];
                is_later = (ka >> 32) == 0;  // key 0 <=> later in the sweep: no waiting
            }
            n_later += __popc(__ballot_sync(0xffffffffu, is_later));
        }
        __syncwarp();
        // ---- C. forces in processing order
        int n_pairs = 0;
        for (int base_c = 0; base_c < nc; base_c += 32) {
            const int c = base_c + lane;
            double fx = 0.0, fy = 0.0;
            int slot = -1;
            bool hit = false;
            if (c < nc) {
                slot = proc[c];
                const int kk = ckk[slot], j = cj[slot];
                double4 sj;
                bool alive = true;
                if (c >= n_later) {  // earlier in the sweep: needs j's NEW state
                    int f;
                    while (((f = ld_acquire(&w.flags[j])) >> 1) != tag) __nanosleep(poll_ns);
                    alive = (f & 1) != 0;
                    const double2 a = __ldcg(reinterpret_cast<const double2 *>(w.live4 + j));
                    const double2 bb = __ldcg(reinterpret_cast<const double2 *>(w.live4 + j) + 1);
                    sj = make_double4(a.x, a.y, bb.x, bb.y);
                } else {  // later: still in its old state
                    sj = w.cell_state[kk];
                }
                if (alive) {
                    const double ddx = sj.x - xi, ddy = sj.y - yi;
                    if (sqrt(ddx * ddx + ddy * ddy) < p.cutoff) {  // pedestrians.py:354, simulations.py:291
                        pair_force(p, ei, xi, yi, vxi, vyi, vd, sj.x, sj.y, sj.z, sj.w, fx, fy);
                        hit = true;
                    } else { fx = 0.0; fy = 0.0; }
                }
            }
            n_pairs += __popc(__ballot_sync(0xffffffffu, hit));
            if (slot >= 0) { lfx[slot] = fx; lfy[slot] = fy; }  // the sort buffers are dead: proc/ord were extracted
        }
        __syncwarp();
        // ---- D. ascending-j sum (simulations.py:285-295).  Most slots hold +-0.0 (beyond the cutoff, or outside the field
        // of view: k = 0).  Adding a zero never changes a bit of the running sum (it starts at +0.0 and can never become
        // -0.0; x + (+-0.0) == x for every other x, NaN and inf included), so the zero terms are squeezed out in parallel
        // first and only the remaining ones -- still in ascending-j order -- go through the sequential, order-sensitive
        // additions.  proc[] is dead by now and receives the kept slots.
        int nnz = 0;
        for (int t0 = 0; t0 < nc; t0 += 32) {
            const int t = t0 + lane;
            int sl = 0;
            bool nz = false;
            if (t < nc) {
                sl = ord[t];
                nz = !(lfx[sl] == 0.0 && lfy[sl] == 0.0);   // NaN terms are kept
            }
            const unsigned mz = __ballot_sync(0xffffffffu, nz);
            if (nz) proc[nnz + __popc(mz & lt_mask)] = (unsigned short)sl;
            nnz += __popc(mz);
        }
        __syncwarp();
        double acc = 0.0;
        if (lane < 2) {  // lane 0 -> x component, lane 1 -> y component
            const double *src = lane == 0 ? lfx : lfy;
            for (int t = 0; t < nnz; t++) acc = acc + src[proc[t]];
        }
        const double rx = __shfl_sync(0xffffffffu, acc, 0), ry = __shfl_sync(0xffffffffu, acc, 1);
        if (lane == 0) {
            double cx = vxi + p.half_noise * nz_x + rx + wf_x;  // simulations.py:303
            double cy = vyi + p.half_noise * nz_y + ry + wf_y;
            double ax = (de_x - cx) / p.relaxation, ay = (de_y - cy) / p.relaxation;  // :307-308
            double nx_ = xi + cx * p.dt + 0.5 * ax * p.dt2;  // :314-315
            double ny_ = yi + cy * p.dt + 0.5 * ay * p.dt2;
            double nvx = cx + ax * p.dt, nvy = cy + ay * p.dt;  // :316-317
            double nr = sqrt(nvx * nvx + nvy * nvy);            // :321
            if (!(nr < p.v_max)) {                              // :323-326
                double sc = p.v_max / nr;
                nvx = nvx * sc;
                nvy = nvy * sc;
            }
            // the candidate search of every agent assumed that nobody moves more than margin/2 per axis in one step
            const double disp = fmax(fabs(nx_ - xi), fabs(ny_ - yi));
            if (!(disp <= margin * 0.5)) {
                atomicOr(&w.counters[1], 4);
                // (NaN displacements stay flagged with the largest margin: the host then gives up with an error)
                atomicMax(reinterpret_cast<unsigned long long *>(w.counters + 4), (unsigned long long)__double_as_longlong(disp));
            }
            pairs_total += n_pairs;  // (one atomic per warp at the end: an atomic here would sit in front of the fence below)
            bool out = false;
            for (int d = 0; d < n_doors; d++) {  // pedestrians.py:132-136
                const double *door = w.doors + 4 * (door_off + d);
                if (fabs(nx_ - door[0]) < door[2] * 0.5 && fabs(ny_ - door[1]) < door[3] * 0.5) out = true;
            }
            // publish first: the release store orders the two 16-byte stores of the new state before the flag; everything
            // that only the host / the next kernel reads is written afterwards, off the dependency chain
            w.live4[i] = make_double4(nx_, ny_, nvx, nvy);
            st_release(&w.flags[i], tag * 2 + (out ? 0 : 1));
            x[i] = nx_; y[i] = ny_; vx[i] = nvx; vy[i] = nvy;
            tim[i] = tim_i + p.dt;  // pedestrians.py:191
            if (out) {
                status[i] = 0;
                w.exit_mark[r] = i + 1;  // simulations.py:331-332, ordered by sweep position
            }
        }
        __syncwarp();
    }
    if (lane == 0 && pairs_total) atomicAdd(&w.counters[2], pairs_total);
}

// ---- two-kernel form of the sweep (the default fast path).  The candidate search, its two sorts and the agent's own
// ellipse need only the step-start snapshot, so cand_kernel does them for all agents at once -- fully parallel, next to
// the wall search on the side stream -- and leaves per agent a list in PROCESSING order of (candidate, position in the
// SUMMATION order).  chain_kernel is then the dependency chain only: wait, pair force, ordered sum, Euler step, publish.
// Its body is less than half of the one-kernel sweep's instructions (which overflowed the 32 KB instruction cache level
// behind L0: ncu `no_instruction` was a quarter of all stall cycles), and it needs neither sort buffers nor cell lists.
constexpr int LIST_CAP = CAND_CAP;
constexpr size_t CAND_SMEM = (size_t)SWEEP_WARPS * CAND_CAP * (2 * sizeof(unsigned long long) + 2 * sizeof(int) + sizeof(unsigned short));
constexpr size_t CHAIN_SMEM = (size_t)SWEEP_WARPS * CAND_CAP * (2 * sizeof(double) + sizeof(unsigned short));

__device__ __forceinline__ void cand_body(const oc_gcfm_params &p, int N, const Ws &w, const double *__restrict__ vdes,
                                          double inv_cs, int nbx, int nby, double margin, int fov_cull) {
    extern __shared__ __align__(16) unsigned char sweep_smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int i = blockIdx.x * SWEEP_WARPS + wid;
    if (i >= N || !w.status0[i]) return;
    unsigned char *base = sweep_smem + (size_t)wid * (CAND_SMEM / SWEEP_WARPS);
    unsigned long long *sort_a = reinterpret_cast<unsigned long long *>(base), *sort_b = sort_a + CAND_CAP;
    int *ckk = reinterpret_cast<int *>(sort_b + CAND_CAP), *cj = ckk + CAND_CAP;
    unsigned short *pos_of = reinterpret_cast<unsigned short *>(cj + CAND_CAP);
    const CandSearch cs_(p, w, margin, inv_cs, fov_cull);
    const int r = w.rank[i];
    const double4 si = w.snap4[i];
    const double vd = vdes[i];
    const AgentEllipse ei = ellipse_of(p, si.z, si.w, vd);
    const int nc = cs_.gather(p, w, i, r, si.x, si.y, si.z, si.w, vd, ei.ni, nbx, nby, CAND_CAP, ckk, cj, sort_a, sort_b);
    __syncwarp();
    if (nc > 1) {
        warp_sort_u64(sort_a, nc, lane);
        warp_sort_u64(sort_b, nc, lane);
    }
    for (int t = lane; t < nc; t += 32) pos_of[(unsigned short)sort_b[t]] = (unsigned short)t;  // slot -> summation position
    __syncwarp();
    int n_later = 0;
    int2 *out = w.lst + (size_t)i * LIST_CAP;
    for (int t0 = 0; t0 < nc; t0 += 32) {
        const int t = t0 + lane;
        bool is_later = false;
        if (t < nc) {
            const unsigned long long ka = sort_a[t];
            const int slot = (unsigned short)ka;
            out[t] = make_int2(cj[slot], pos_of[slot]);
            is_later = (ka >> 32) == 0;  // key 0 <=> later in the sweep: no waiting
        }
        n_later += __popc(__ballot_sync(0xffffffffu, is_later));
    }
    if (lane == 0) {
        w.lhdr[i] = make_int2(nc, n_later);
        w.ell[i] = make_double4(ei.ni, ei.a_i, ei.b_i, ei.beta_i);
    }
}

__device__ __forceinline__ void
chain_body(const oc_gcfm_params &p, int N, const Ws &w, double *__restrict__ x, double *__restrict__ y,
           double *__restrict__ vx, double *__restrict__ vy, double *__restrict__ tim, uint8_t *__restrict__ status,
           const double *__restrict__ vdes, const int *__restrict__ key_id, int tag, unsigned poll_ns, double margin) {
    extern __shared__ __align__(16) unsigned char sweep_smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned char *base = sweep_smem + (size_t)wid * (CHAIN_SMEM / SWEEP_WARPS);
    double *lfx = reinterpret_cast<double *>(base), *lfy = lfx + CAND_CAP;  // forces by summation position
    unsigned short *nzl = reinterpret_cast<unsigned short *>(lfy + CAND_CAP);  // positions of the non-zero terms
    const unsigned lt_mask = (1u << lane) - 1;
    int pairs_total = 0;
    for (;;) {
        int r = 0;
        if (lane == 0) r = atomicAdd(&w.counters[0], 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r >= N) break;
        const int i = w.perm[r];
        if (!w.status0[i]) continue;  // simulations.py:277
        const int2 hdr = w.lhdr[i];
        const int nc = hdr.x, n_later = hdr.y;
        const double4 si = w.snap4[i];
        const double xi = si.x, yi = si.y, vxi = si.z, vyi = si.w, vd = vdes[i];
        const double4 el = w.ell[i];
        AgentEllipse ei;
        ei.ni = el.x; ei.a_i = el.y; ei.b_i = el.z; ei.beta_i = el.w;
        const int2 *lst = w.lst + (size_t)i * LIST_CAP;
        // everything the final Euler step needs that does not depend on the neighbours is fetched now, so that no global
        // load sits between "last dependency published" and "I publish"
        double nz_x = 0.0, nz_y = 0.0, wf_x = 0.0, wf_y = 0.0, de_x = 0.0, de_y = 0.0, tim_i = 0.0;
        int door_off = 0, n_doors = 0;
        if (lane == 0) {
            const int nz = w.nzidx[i];
            nz_x = w.noise[2 * nz]; nz_y = w.noise[2 * nz + 1];
            wf_x = w.wfx[i]; wf_y = w.wfy[i];
            de_x = w.des_x[i]; de_y = w.des_y[i];
            tim_i = tim[i];
            const KeyDev *kp = w.keys + key_id[i];
            door_off = kp->door_off; n_doors = kp->n_doors;
        }
        // ---- forces in processing order (later candidates first: snapshot state, no waiting), stored by summation position
        int n_pairs = 0;
        for (int base_c = 0; base_c < nc; base_c += 32) {
            const int c = base_c + lane;
            double fx = 0.0, fy = 0.0;
            int pos = -1;
            bool hit = false;
            if (c < nc) {
                const int2 e = lst[c];
                const int j = e.x;
                pos = e.y;
                double4 sj;
                bool alive = true;
                if (c >= n_later) {  // earlier in the sweep: needs j's NEW state
                    int f;
                    while (((f = ld_acquire(&w.flags[j])) >> 1) != tag) __nanosleep(poll_ns);
                    alive = (f & 1) != 0;
                    const double2 a = __ldcg(reinterpret_cast<const double2 *>(w.live4 + j));
                    const double2 bb = __ldcg(reinterpret_cast<const double2 *>(w.live4 + j) + 1);
                    sj = make_double4(a.x, a.y, bb.x, bb.y);
                } else {  // later: still in its old state
                    sj = w.snap4[j];
                }
                if (alive) {
                    const double ddx = sj.x - xi, ddy = sj.y - yi;
                    if (sqrt(ddx * ddx + ddy * ddy) < p.cutoff) {  // pedestrians.py:354, simulations.py:291
                        pair_force(p, ei, xi, yi, vxi, vyi, vd, sj.x, sj.y, sj.z, sj.w, fx, fy);
                        hit = true;
                    } else { fx = 0.0; fy = 0.0; }
                }
            }
            n_pairs += __popc(__ballot_sync(0xffffffffu, hit));
            if (pos >= 0) { lfx[pos] = fx; lfy[pos] = fy; }
        }
        __syncwarp();
        // ---- ascending-j sum (simulations.py:285-295); exact zeros are squeezed out first (see the one-kernel sweep)
        int nnz = 0;
        for (int t0 = 0; t0 < nc; t0 += 32) {
            const int t = t0 + lane;
            const bool nz = t < nc && !(lfx[t] == 0.0 && lfy[t] == 0.0);  // NaN terms are kept
            const unsigned mz = __ballot_sync(0xffffffffu, nz);
            if (nz) nzl[nnz + __popc(mz & lt_mask)] = (unsigned short)t;
            nnz += __popc(mz);
        }
        __syncwarp();
        double acc = 0.0;
        if (lane < 2) {  // lane 0 -> x component, lane 1 -> y component
            const double *src = lane == 0 ? lfx : lfy;
            for (int t = 0; t < nnz; t++) acc = acc + src[nzl[t]];
        }
        const double rx = __shfl_sync(0xffffffffu, acc, 0), ry = __shfl_sync(0xffffffffu, acc, 1);
        if (lane == 0) {
            double cx = vxi + p.half_noise * nz_x + rx + wf_x;  // simulations.py:303
            double cy = vyi + p.half_noise * nz_y + ry + wf_y;
            double ax = (de_x - cx) / p.relaxation, ay = (de_y - cy) / p.relaxation;  // :307-308
            double nx_ = xi + cx * p.dt + 0.5 * ax * p.dt2;  // :314-315
            double ny_ = yi + cy * p.dt + 0.5 * ay * p.dt2;
            double nvx = cx + ax * p.dt, nvy = cy + ay * p.dt;  // :316-317
            double nr = sqrt(nvx * nvx + nvy * nvy);            // :321
            if (!(nr < p.v_max)) {                              // :323-326
                double sc = p.v_max / nr;
                nvx = nvx * sc;
                nvy = nvy * sc;
            }
            // the candidate search of every agent assumed that nobody moves more than margin/2 per axis in one step
            const double disp = fmax(fabs(nx_ - xi), fabs(ny_ - yi));
            if (!(disp <= margin * 0.5)) {
                atomicOr(&w.counters[1], 4);
                atomicMax(reinterpret_cast<unsigned long long *>(w.counters + 4), (unsigned long long)__double_as_longlong(disp));
            }
            pairs_total += n_pairs;
            bool out = false;
            for (int d = 0; d < n_doors; d++) {  // pedestrians.py:132-136
                const double *door = w.doors + 4 * (door_off + d);
                if (fabs(nx_ - door[0]) < door[2] * 0.5 && fabs(ny_ - door[1]) < door[3] * 0.5) out = true;
            }
            w.live4[i] = make_double4(nx_, ny_, nvx, nvy);
            st_release(&w.flags[i], tag * 2 + (out ? 0 : 1));
            x[i] = nx_; y[i] = ny_; vx[i] = nvx; vy[i] = nvy;
            tim[i] = tim_i + p.dt;  // pedestrians.py:191
            if (out) {
                status[i] = 0;
                w.exit_mark[r] = i + 1;  // simulations.py:331-332, ordered by sweep position
            }
        }
        __syncwarp();
    }
    if (lane == 0 && pairs_total) atomicAdd(&w.counters[2], pairs_total);
}

// ordered compaction of the exit marks (by sweep position) into host-visible memory: out[0]=count, out[1..5]=counters[1..5]
__device__ __forceinline__ void exit_compact_body(int N, const Ws &w, int *__restrict__ out) {
    __shared__ int tot[1024];
    int t = threadIdx.x;
    int per = (N + 1023) / 1024;
    int lo = min(t * per, N), hi = min(lo + per, N);
    int s = 0;
    for (int r = lo; r < hi; r++) s += (w.exit_mark[r] != 0);
    tot[t] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        int v = (t >= o) ? tot[t - o] : 0;
        __syncthreads();
        tot[t] += v;
        __syncthreads();
    }
    int run = tot[t] - s;
    for (int r = lo; r < hi; r++)
        if (w.exit_mark[r]) out[OUT_HDR + run++] = w.exit_mark[r] - 1;
    if (t == 1023) out[0] = tot[1023];
    if (t < 5) out[1 + t] = w.counters[1 + t];  // flags, pairs, largest candidate count, largest displacement (2 ints)
}

// ---- kernel entry points.  Single room: arguments by value.  Ensembles (BASELINE configs[4]): ONE launch per kernel for
// all members of a wave, blockIdx.y = member, every member described by a GcfmMember record in device memory -- the
// members' sweeps then run side by side without one stream (and one of the 32 hardware queues) per member, and a step
// of 128 members costs 8 launches instead of 128 x 7.
struct GcfmMember {
    oc_gcfm_params prm;
    Ws w;
    double *x, *y, *vx, *vy, *tim;
    uint8_t *status;
    const double *vdes, *X, *Y;
    const int *key;
    int *out;          // host-visible step result (exit log)
    int N, simu_step, tag, nbx, nby, nbins;
    double inv_cs;
    unsigned poll_ns;
    int fov_cull;
    double margin;  // displacement margin of this member's fast attempt
};

__global__ void setup_kernel(int N, const double *__restrict__ x, const double *__restrict__ y,
                             const double *__restrict__ vx, const double *__restrict__ vy,
                             const double *__restrict__ tim, const uint8_t *__restrict__ status, Ws w, double inv_cs,
                             int nbx, int nby) {
    setup_body(N, x, y, vx, vy, tim, status, w, inv_cs, nbx, nby);
}
__global__ void __launch_bounds__(1024) scan_kernel(int *a, int n) { scan_body(a, n); }
__global__ void scatter_kernel(int N, Ws w) { scatter_body(N, w); }
__global__ void __launch_bounds__(1024) noise_index_kernel(int N, Ws w) { noise_index_body(N, w); }
// PAIR: two tiles per round trip of the node scan (96 registers, 5 CTAs/SM) or one (80 registers, 6 CTAs/SM)
template <bool PAIR>
__global__ void __launch_bounds__(128, PAIR ? 5 : 6)
wall_search_kernel(oc_gcfm_params p, int N, Ws w, const double *__restrict__ X, const double *__restrict__ Y,
                   const int *__restrict__ key_id) {
    wall_search_body<PAIR>(p, N, w, X, Y, key_id);
}
__global__ void __launch_bounds__(128) agent_terms_kernel(oc_gcfm_params p, int N, Ws w, const double *__restrict__ X,
                                                          const double *__restrict__ Y, const double *__restrict__ vdes,
                                                          const int *__restrict__ key_id) {
    agent_terms_body(p, N, w, X, Y, vdes, key_id, w.hdr[1]);
}
__global__ void __launch_bounds__(SWEEP_WARPS * 32)
sweep_kernel(oc_gcfm_params p, int N, Ws w, double *__restrict__ x, double *__restrict__ y, double *__restrict__ vx,
             double *__restrict__ vy, double *__restrict__ tim, uint8_t *__restrict__ status,
             const double *__restrict__ vdes, const int *__restrict__ key_id, double inv_cs, int nbx, int nby,
             unsigned poll_ns, double margin, int cap, unsigned char *glists, int fov_cull) {
    sweep_body(p, N, w, x, y, vx, vy, tim, status, vdes, key_id, w.hdr[0], inv_cs, nbx, nby, poll_ns, margin, cap, glists,
               fov_cull);
}
__global__ void __launch_bounds__(SWEEP_WARPS * 32)
cand_kernel(oc_gcfm_params p, int N, Ws w, const double *__restrict__ vdes, double inv_cs, int nbx, int nby, double margin,
            int fov_cull) {
    cand_body(p, N, w, vdes, inv_cs, nbx, nby, margin, fov_cull);
}
__global__ void __launch_bounds__(SWEEP_WARPS * 32)
chain_kernel(oc_gcfm_params p, int N, Ws w, double *__restrict__ x, double *__restrict__ y, double *__restrict__ vx,
             double *__restrict__ vy, double *__restrict__ tim, uint8_t *__restrict__ status,
             const double *__restrict__ vdes, const int *__restrict__ key_id, unsigned poll_ns, double margin) {
    chain_body(p, N, w, x, y, vx, vy, tim, status, vdes, key_id, w.hdr[0], poll_ns, margin);
}
__global__ void __launch_bounds__(1024) exit_compact_kernel(int N, Ws w, int *__restrict__ out) {
    exit_compact_body(N, w, out);
}

// batched variants: blockIdx.y = member
__global__ void clear_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int i = t0; i <= m.nbins; i += stride) { m.w.bin_start[i] = 0; m.w.bin_cursor[i] = 0; }
    for (int i = t0; i < m.N; i += stride) m.w.exit_mark[i] = 0;
    if (t0 < 8) m.w.counters[t0] = 0;
}
__global__ void setup_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    setup_body(m.N, m.x, m.y, m.vx, m.vy, m.tim, m.status, m.w, m.inv_cs, m.nbx, m.nby);
}
__global__ void __launch_bounds__(1024) scan_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    scan_body(m.w.bin_start, m.nbins + 1);
}
__global__ void scatter_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    scatter_body(m.N, m.w);
}
__global__ void __launch_bounds__(1024) noise_index_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    noise_index_body(m.N, m.w);
}
template <bool PAIR>
__global__ void __launch_bounds__(128, PAIR ? 5 : 6) wall_search_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    wall_search_body<PAIR>(m.prm, m.N, m.w, m.X, m.Y, m.key);
}
__global__ void __launch_bounds__(128) agent_terms_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    agent_terms_body(m.prm, m.N, m.w, m.X, m.Y, m.vdes, m.key, m.simu_step);
}
__global__ void __launch_bounds__(SWEEP_WARPS * 32) sweep_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    sweep_body(m.prm, m.N, m.w, m.x, m.y, m.vx, m.vy, m.tim, m.status, m.vdes, m.key, m.tag, m.inv_cs, m.nbx, m.nby,
               m.poll_ns, m.margin, CAND_CAP, nullptr, m.fov_cull);
}
__global__ void __launch_bounds__(SWEEP_WARPS * 32) cand_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    cand_body(m.prm, m.N, m.w, m.vdes, m.inv_cs, m.nbx, m.nby, m.margin, m.fov_cull);
}
__global__ void __launch_bounds__(SWEEP_WARPS * 32) chain_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    chain_body(m.prm, m.N, m.w, m.x, m.y, m.vx, m.vy, m.tim, m.status, m.vdes, m.key, m.tag, m.poll_ns, m.margin);
}
__global__ void __launch_bounds__(1024) exit_compact_multi_kernel(const GcfmMember *__restrict__ ms) {
    const GcfmMember &m = ms[blockIdx.y];
    exit_compact_body(m.N, m.w, m.out);
}

// unit-probe kernels ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
wall_probe_kernel(oc_gcfm_params p, int N, const double *__restrict__ X, const double *__restrict__ Y,
                  const double *__restrict__ V, const uint8_t *__restrict__ tiles, double off_min,
                  const double *__restrict__ px, const double *__restrict__ py, const double *__restrict__ pvx,
                  const double *__restrict__ pvy, const double *__restrict__ vdes, double *__restrict__ fx,
                  double *__restrict__ fy, long long *__restrict__ ind_out) {
    int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= N) return;
    long long ind = wall_argmin_warp<true>(X, Y, V, tiles, p.Ny, p.Nx, px[i], py[i], off_min);
    if ((threadIdx.x & 31) == 0) {
        AgentEllipse ei = ellipse_of(p, pvx[i], pvy[i], vdes[i]);
        double ax, ay;
        wall_force_from_node(p, ei, px[i], py[i], pvx[i], pvy[i], X[ind % p.Nx], Y[ind / p.Nx], ax, ay);
        fx[i] = ax;
        fy[i] = ay;
        if (ind_out) ind_out[i] = ind;
    }
}

__global__ void pair_probe_kernel(oc_gcfm_params p, int N, const double *__restrict__ pi, const double *__restrict__ vi,
                                  const double *__restrict__ vdes, const double *__restrict__ pj,
                                  const double *__restrict__ vj, double *__restrict__ f) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= N) return;
    AgentEllipse ei = ellipse_of(p, vi[2 * q], vi[2 * q + 1], vdes[q]);
    double fx, fy;
    pair_force(p, ei, pi[2 * q], pi[2 * q + 1], vi[2 * q], vi[2 * q + 1], vdes[q], pj[2 * q], pj[2 * q + 1],
               vj[2 * q], vj[2 * q + 1], fx, fy);
    f[2 * q] = fx;
    f[2 * q + 1] = fy;
}

// K7 density (simulations.py:469-487): per node, sum over active agents in agent order.  exp underflows to
// exactly 0 beyond r_zero, so agents farther than that from the whole tile are culled without changing a bit.
constexpr int DN_TX = 32, DN_TY = 8, DN_CHUNK = 256;
__global__ void __launch_bounds__(256)
density_kernel(int N, const double *__restrict__ ax, const double *__restrict__ ay, const uint8_t *__restrict__ status,
               const double *__restrict__ X, const double *__restrict__ Y, const double *__restrict__ Vg, int Ny,
               int Nx, double two_s2, double C, double r_zero, double *__restrict__ out) {
    __shared__ double lx[DN_CHUNK], ly[DN_CHUNK];
    __shared__ int wcnt[8];
    const int ix = blockIdx.x * DN_TX + (threadIdx.x & 31), iy = blockIdx.y * DN_TY + (threadIdx.x >> 5);
    const bool in = ix < Nx && iy < Ny;
    const double x = in ? X[ix] : 0.0, y = in ? Y[iy] : 0.0;
    const int jx0 = blockIdx.x * DN_TX, jx1 = min(jx0 + DN_TX, Nx) - 1, jy0 = blockIdx.y * DN_TY,
              jy1 = min(jy0 + DN_TY, Ny) - 1;
    const double bx0 = X[jx0] - r_zero, bx1 = X[jx1] + r_zero, by0 = Y[jy0] - r_zero, by1 = Y[jy1] + r_zero;
    double d = 0.0;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int base = 0; base < N; base += DN_CHUNK) {
        int a = base + threadIdx.x;
        bool keep = false;
        double px = 0, py = 0;
        if (a < N && status[a]) {
            px = ax[a]; py = ay[a];
            keep = (px >= bx0 && px <= bx1 && py >= by0 && py <= by1) || !(px == px) || !(py == py);
        }
        unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) wcnt[wid] = __popc(m);
        __syncthreads();
        int off = 0, total = 0;
        for (int q = 0; q < 8; q++) { if (q < wid) off += wcnt[q]; total += wcnt[q]; }
        if (keep) {
            int pos = off + __popc(m & ((1u << lane) - 1));  // preserves agent order
            lx[pos] = px; ly[pos] = py;
        }
        __syncthreads();
        if (in)
            for (int q = 0; q < total; q++) {
                double cx = x - lx[q], cy = y - ly[q];
                d += ocm_exp(-(cx * cx + cy * cy) / two_s2) / C;  // :480-483
            }
        __syncthreads();
    }
    if (in) {
        size_t g = (size_t)iy * Nx + ix;
        out[g] = (Vg[g] < 0) ? 0.0 : d;  // :485
    }
}

template <class T>
T *carve(char *&p, size_t n) {
    T *r = reinterpret_cast<T *>(p);
    p += ((n * sizeof(T) + 255) / 256) * 256;
    return r;
}

}  // namespace

extern "C" long long oc_wall_tiles_bytes(oc_ctx *ctx) {
    if (!ctx) return 0;
    return (long long)((ctx->Nx + WT - 1) / WT) * ((ctx->Ny + WT - 1) / WT);
}

extern "C" int oc_wall_tiles(oc_ctx *ctx, const double *d_V, uint8_t *d_tiles, double *v_min, void *stream) {
    OC_ARG(ctx && d_V && d_tiles, "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    int nt = (int)oc_wall_tiles_bytes(ctx);
    double *d_vm = nullptr;
    OC_CUDA(cudaMalloc(&d_vm, sizeof(double) * nt + nt));
    uint8_t *d_occ = reinterpret_cast<uint8_t *>(d_vm + nt);
    const int ntx = (ctx->Nx + WT - 1) / WT, nty = (ctx->Ny + WT - 1) / WT;
    tiles_kernel<<<(nt * 32 + 127) / 128, 128, 0, st>>>(d_V, ctx->Ny, ctx->Nx, d_occ, d_vm);
    tile_ring_kernel<<<(nt + 127) / 128, 128, 0, st>>>(d_occ, ntx, nty, d_tiles);
    oc::count_launch(2);
    std::vector<double> h(nt);
    cudaError_t e = cudaMemcpyAsync(h.data(), d_vm, sizeof(double) * nt, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_vm);
    OC_CUDA(e);
    double vm = INFINITY;
    for (double v : h) vm = std::min(vm, v);
    if (v_min) *v_min = vm;
    return OC_OK;
}

static int gcfm_workspace(oc_ctx *ctx, int N, int n_keys, int n_doors, int nbins, Ws &w, int **pinned, cudaStream_t st) {
    size_t need = 0;
    auto al = [&](size_t b) { need += ((b + 255) / 256) * 256; };
    for (int q = 0; q < 10; q++) al(sizeof(double) * N);
    al(sizeof(double4) * N);
    al(sizeof(double4) * N);
    al(sizeof(double4) * N);
    al(sizeof(int2) * N);
    al(sizeof(double) * 2 * N);
    al(sizeof(double) * 4 * std::max(n_doors, 1));
    for (int q = 0; q < 7; q++) al(sizeof(int) * N);
    al(sizeof(int) * (nbins + 1));
    al(sizeof(int) * (nbins + 1));
    al(N);
    al(sizeof(KeyDev) * std::max(n_keys, 1));
    al(sizeof(int) * 8);
    al(sizeof(int) * 16);
    al(sizeof(int2) * N);
    al(sizeof(double4) * N);
    al(sizeof(int2) * (size_t)N * LIST_CAP);
    if (ctx->gcfm_ws_bytes < need) {
        if (ctx->gcfm_ws) cudaFree(ctx->gcfm_ws);
        ctx->gcfm_ws = nullptr;
        ctx->gcfm_ws_bytes = 0;
        OC_CUDA(cudaMalloc(&ctx->gcfm_ws, need));
        // done-flags start at 0; tags are never 0.  On the step's own stream: a legacy-stream cudaMemset is not ordered
        // against kernels of a non-blocking stream (ensembles step every member on its own stream)
        OC_CUDA(cudaMemsetAsync(ctx->gcfm_ws, 0, need, st));
        ctx->gcfm_ws_bytes = need;
        ctx->gcfm_keys_dev = nullptr;  // the cached key descriptors are gone
    } else if (ctx->gcfm_N != N || ctx->gcfm_nbins != nbins || ctx->gcfm_nkeys != n_keys || ctx->gcfm_ndoors != n_doors) {
        OC_CUDA(cudaMemsetAsync(ctx->gcfm_ws, 0, ctx->gcfm_ws_bytes, st));  // layout changes: done-flags must restart at 0
        ctx->gcfm_keys_dev = nullptr;
    }
    ctx->gcfm_N = N; ctx->gcfm_nbins = nbins; ctx->gcfm_nkeys = n_keys; ctx->gcfm_ndoors = n_doors;
    char *p = (char *)ctx->gcfm_ws;
    // flags first so that it keeps its place (and contents) while N is unchanged
    w.flags = carve<int>(p, N);
    w.snap4 = carve<double4>(p, N);
    w.live4 = carve<double4>(p, N);
    w.cell_state = carve<double4>(p, N);
    w.cell_jr = carve<int2>(p, N);
    w.x0 = carve<double>(p, N); w.y0 = carve<double>(p, N); w.vx0 = carve<double>(p, N); w.vy0 = carve<double>(p, N);
    w.des_x = carve<double>(p, N); w.des_y = carve<double>(p, N); w.wfx = carve<double>(p, N); w.wfy = carve<double>(p, N);
    w.time0 = carve<double>(p, N);
    w.wall_ind = carve<long long>(p, N);
    w.hdr = carve<int>(p, 16);   // hdr | perm | noise: one host-to-device copy per step (gcfm_stage mirrors the layout)
    w.perm = carve<int>(p, N);
    w.noise = carve<double>(p, 2 * (size_t)N);
    w.doors = carve<double>(p, 4 * (size_t)std::max(n_doors, 1));
    w.rank = carve<int>(p, N); w.nzidx = carve<int>(p, N);
    w.agent_bin = carve<int>(p, N); w.cell_agents = carve<int>(p, N);
    w.counters = carve<int>(p, 8);   // counters | bin_start | bin_cursor | exit_mark: one memset per attempt
    w.bin_start = carve<int>(p, nbins + 1); w.bin_cursor = carve<int>(p, nbins + 1);
    w.exit_mark = carve<int>(p, N);
    w.status0 = carve<uint8_t>(p, N);
    w.keys = carve<KeyDev>(p, std::max(n_keys, 1));
    w.lhdr = carve<int2>(p, N);
    w.ell = carve<double4>(p, N);
    w.lst = carve<int2>(p, (size_t)N * LIST_CAP);
    size_t pin = sizeof(int) * ((size_t)N + OUT_HDR + 8);
    if (ctx->gcfm_pinned_bytes < pin) {
        if (ctx->gcfm_pinned) cudaFreeHost(ctx->gcfm_pinned);
        OC_CUDA(cudaMallocHost(&ctx->gcfm_pinned, pin));
        ctx->gcfm_pinned_bytes = pin;
    }
    *pinned = (int *)ctx->gcfm_pinned;
    return OC_OK;
}

namespace {
// what oc_gcfm_step_finish needs to redo a step on the exact slow path (kept per context between _launch and _finish)
struct GcfmLaunch {
    oc_gcfm_params prm;
    int N, n_keys, n_doors, nbins_alloc;
    double *x, *y, *vx, *vy, *tim;
    uint8_t *status;
    const double *vdes;
    const int *key;
    Ws w;
    int *pinned;
    double margin;  // displacement margin of the fast attempt in flight
    int simu_step;
};

// displacement margin of the next fast attempt: the small one (oc_ctx_set_int "gcfm_margin_mm", default 0.25 m: no agent
// moves more than 12.5 cm per axis and step) unless a recent step overflowed it, then DISP_MARGIN for a while
double gcfm_fast_margin(oc_ctx *ctx) {
    if (ctx->gcfm_margin_hold > 0) { ctx->gcfm_margin_hold--; return DISP_MARGIN; }
    return std::min(DISP_MARGIN, std::max(0.02, ctx->gcfm_margin_mm * 1e-3));
}
// bin table size that fits every margin a fast or slow attempt may use (smaller margin = smaller cells = more bins)
int gcfm_max_bins(const oc_ctx *ctx, double cutoff, int *nbx_out = nullptr, int *nby_out = nullptr) {
    const double reach = cutoff + std::min(DISP_MARGIN, std::max(0.02, ctx->gcfm_margin_mm * 1e-3));
    const double inv_cs = 2.0 / reach;
    const int nbx = std::max(1, (int)std::ceil(ctx->room_length * inv_cs)),
              nby = std::max(1, (int)std::ceil(ctx->room_height * inv_cs));
    if (nbx_out) *nbx_out = nbx;
    if (nby_out) *nby_out = nby;
    return nbx * nby;
}

// side streams of a step: the per-agent terms (wall search, sampler, wall force) and the noise index only need the
// step-start snapshot and run next to the cell-list / candidate-list kernels of the main stream
int gcfm_streams(oc_ctx *ctx) {
    if (ctx->gcfm_side) return OC_OK;
    OC_CUDA(cudaStreamCreateWithFlags(&ctx->gcfm_side, cudaStreamNonBlocking));
    OC_CUDA(cudaStreamCreateWithFlags(&ctx->gcfm_side2, cudaStreamNonBlocking));
    OC_CUDA(cudaStreamCreateWithFlags(&ctx->gcfm_cap, cudaStreamNonBlocking));
    OC_CUDA(cudaEventCreateWithFlags(&ctx->gcfm_ev_fork, cudaEventDisableTiming));
    OC_CUDA(cudaEventCreateWithFlags(&ctx->gcfm_ev_join, cudaEventDisableTiming));
    OC_CUDA(cudaEventCreateWithFlags(&ctx->gcfm_ev_join2, cudaEventDisableTiming));
    return OC_OK;
}
int gcfm_fork(oc_ctx *ctx, cudaStream_t st, cudaStream_t *side, cudaStream_t *side2) {
    *side = *side2 = st;
    if (!ctx->gcfm_overlap) return OC_OK;
    int rc = gcfm_streams(ctx);
    if (rc) return rc;
    OC_CUDA(cudaEventRecord(ctx->gcfm_ev_fork, st));
    OC_CUDA(cudaStreamWaitEvent(ctx->gcfm_side, ctx->gcfm_ev_fork, 0));
    OC_CUDA(cudaStreamWaitEvent(ctx->gcfm_side2, ctx->gcfm_ev_fork, 0));
    *side = ctx->gcfm_side;
    *side2 = ctx->gcfm_side2;
    return OC_OK;
}
int gcfm_join(oc_ctx *ctx, cudaStream_t st, cudaStream_t side, cudaStream_t side2) {
    if (side == st) return OC_OK;
    OC_CUDA(cudaEventRecord(ctx->gcfm_ev_join, side));
    OC_CUDA(cudaEventRecord(ctx->gcfm_ev_join2, side2));
    OC_CUDA(cudaStreamWaitEvent(st, ctx->gcfm_ev_join, 0));
    OC_CUDA(cudaStreamWaitEvent(st, ctx->gcfm_ev_join2, 0));
    return OC_OK;
}

// per device and context, once: dynamic shared memory limits and the resident grids of the sweep kernels (kept out of
// the per-step path, and out of stream capture)
int gcfm_device_setup(oc_ctx *ctx) {
    if (ctx->gcfm_grid_chain) return OC_OK;
    int n_sm = 0, occ = 0;
    OC_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device));
    OC_CUDA(cudaFuncSetAttribute(sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SWEEP_SMEM));
    OC_CUDA(cudaFuncSetAttribute(cand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAND_SMEM));
    OC_CUDA(cudaFuncSetAttribute(chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CHAIN_SMEM));
    OC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sweep_kernel, SWEEP_WARPS * 32, SWEEP_SMEM));
    ctx->gcfm_grid_sweep = n_sm * std::max(occ, 1);
    OC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sweep_kernel, SWEEP_WARPS * 32, 0));
    ctx->gcfm_grid_sweep_slow = n_sm * std::max(occ, 1);
    OC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, chain_kernel, SWEEP_WARPS * 32, CHAIN_SMEM));
    ctx->gcfm_grid_chain = n_sm * std::max(occ, 1);
    return OC_OK;
}

int gcfm_next_tag(oc_ctx *ctx) {  // per context: the done-flags live in the context's workspace
    if (++ctx->gcfm_tag >= 0x3fffffff) ctx->gcfm_tag = 1;
    return ctx->gcfm_tag;
}

// bins + cell list (+ the candidate lists of the two-kernel sweep) of one attempt of the current step.
// margin: displacement (2 x per axis) the candidate search allows for.  first = true: the step's first attempt (the done-flag
// generation and simu_step are already in w.hdr, uploaded with perm / noise; the per-agent terms run on the side streams);
// first = false: the state is restored, a new generation is uploaded, the per-agent terms are kept.
int gcfm_sweep_attempt(oc_ctx *ctx, GcfmLaunch &L, cudaStream_t st, double margin, bool first, bool split) {
    const int N = L.N;
    Ws &w = L.w;
    const double reach = L.prm.cutoff + margin;
    const double cs = reach / 2.0, inv_cs = 1.0 / cs;  // candidate bins: cell size (cutoff + margin)/2, search +-2 cells
    const int nbx = std::max(1, (int)std::ceil(ctx->room_length * inv_cs)),
              nby = std::max(1, (int)std::ceil(ctx->room_height * inv_cs));
    const int nbins = nbx * nby;
    if (nbins > L.nbins_alloc) { oc::set_error("internal: GCFM bin table too small"); return OC_ERR_ARG; }
    const int nb = (N + 255) / 256;
    if (!first) {
        if (!ctx->gcfm_stage) {  // (a member of a batched step: its first attempt was staged by the batch)
            OC_CUDA(cudaMallocHost(&ctx->gcfm_stage, 64));
            ctx->gcfm_stage_bytes = 64;
        }
        int *hs = static_cast<int *>(ctx->gcfm_stage);  // (the previous attempt has been synchronised: the staging is free)
        hs[1] = L.simu_step;
        hs[0] = gcfm_next_tag(ctx);
        OC_CUDA(cudaMemcpyAsync(w.hdr, hs, 2 * sizeof(int), cudaMemcpyHostToDevice, st));
        restore_kernel<<<nb, 256, 0, st>>>(N, w, L.x, L.y, L.vx, L.vy, L.tim, L.status);
        oc::count_launch();
    }
    // counters | bin_start | bin_cursor | exit_mark are carved back to back (a redo resets the counters in restore_kernel)
    char *z0 = reinterpret_cast<char *>(first ? w.counters : w.bin_start);
    OC_CUDA(cudaMemsetAsync(z0, 0, reinterpret_cast<char *>(w.exit_mark + N) - z0, st));
    setup_kernel<<<nb, 256, 0, st>>>(N, L.x, L.y, L.vx, L.vy, L.tim, L.status, w, inv_cs, nbx, nby);
    cudaStream_t side = st, side2 = st;
    if (first) {  // per-agent terms of the step (not repeated by a redo: they depend on the step-start state only)
        int rc = gcfm_fork(ctx, st, &side, &side2);
        if (rc) return rc;
        if (ctx->gcfm_ws_pair) wall_search_kernel<true><<<(N * 32 + 127) / 128, 128, 0, side>>>(L.prm, N, w, ctx->d_X, ctx->d_Y, L.key);
        else wall_search_kernel<false><<<(N * 32 + 127) / 128, 128, 0, side>>>(L.prm, N, w, ctx->d_X, ctx->d_Y, L.key);
        agent_terms_kernel<<<nb * 2, 128, 0, side>>>(L.prm, N, w, ctx->d_X, ctx->d_Y, L.vdes, L.key);
        noise_index_kernel<<<1, 1024, 0, side2>>>(N, w);
        oc::count_launch(3);
    }
    scan_kernel<<<1, 1024, 0, st>>>(w.bin_start, nbins + 1);
    scatter_kernel<<<nb, 256, 0, st>>>(N, w);
    oc::count_launch(3);
    if (split) {  // two-kernel sweep: candidate lists of all agents, next to the wall search on the side stream
        cand_kernel<<<(N + SWEEP_WARPS - 1) / SWEEP_WARPS, SWEEP_WARPS * 32, CAND_SMEM, st>>>(L.prm, N, w, L.vdes, inv_cs, nbx, nby,
                                                                                             margin, ctx->gcfm_fov_cull);
        oc::count_launch();
    }
    if (first) {
        int rc = gcfm_join(ctx, st, side, side2);
        if (rc) return rc;
    }
    return OC_OK;
}
}  // namespace

extern "C" int oc_gcfm_step(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx,
                            double *d_vy, double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key,
                            const oc_key *keys, int n_keys, const int *perm, const double *noise, int n_noise,
                            int simu_step, int *exit_log, int *n_exit, void *stream) {
    int rc = oc_gcfm_step_launch(ctx, prm, N, d_x, d_y, d_vx, d_vy, d_time, d_status, d_vdes, d_key, keys, n_keys, perm,
                                 noise, n_noise, simu_step, stream);
    if (rc) return rc;
    return oc_gcfm_step_finish(ctx, exit_log, n_exit);
}

// the sweep launch of one attempt.  fast + split: the chain kernel of the two-kernel sweep (cand_kernel ran in
// gcfm_sweep_attempt); fast: one-kernel sweep with shared-memory lists of CAND_CAP slots; slow: one-kernel sweep with
// global-memory lists of `cap` slots
static int gcfm_launch_sweep(oc_ctx *ctx, GcfmLaunch &L, cudaStream_t st, double margin, int cap, bool slow, bool split) {
    const int N = L.N;
    const int want = (N + SWEEP_WARPS - 1) / SWEEP_WARPS;
    // ensembles: many small crowds sweep concurrently, each with far fewer runnable agents than the GPU has warp slots
    // (the sweep's dependency DAG is ~200 deep for 1000 agents at 2.5 ped/m^2); a capped grid lets them share the SMs.
    // Tickets are drawn in sweep order by resident warps only, so any grid size >= 1 is deadlock-free.
    auto capped = [&](int resident) {
        int g = std::max(1, std::min(resident, want));
        if (ctx->gcfm_sweep_ctas > 0) g = std::min(g, ctx->gcfm_sweep_ctas);
        return g;
    };
    if (split && !slow) {
        chain_kernel<<<capped(ctx->gcfm_grid_chain), SWEEP_WARPS * 32, CHAIN_SMEM, st>>>(
            L.prm, N, L.w, L.x, L.y, L.vx, L.vy, L.tim, L.status, L.vdes, L.key, (unsigned)ctx->gcfm_poll_ns, margin);
        exit_compact_kernel<<<1, 1024, 0, st>>>(N, L.w, L.pinned);
        oc::count_launch(2);
        OC_CUDA(cudaGetLastError());
        return OC_OK;
    }
    const double reach = L.prm.cutoff + margin, inv_cs = 2.0 / reach;
    const int nbx = std::max(1, (int)std::ceil(ctx->room_length * inv_cs)),
              nby = std::max(1, (int)std::ceil(ctx->room_height * inv_cs));
    const size_t smem = slow ? 0 : SWEEP_SMEM;
    int grid = capped(slow ? ctx->gcfm_grid_sweep_slow : ctx->gcfm_grid_sweep);
    unsigned char *glists = nullptr;
    if (slow) {
        const size_t per_warp = (size_t)cap * SWEEP_SLOT_BYTES;
        const size_t budget = (size_t)1 << 30;  // at most 1 GiB of candidate lists: fewer resident warps instead
        grid = (int)std::max<size_t>(1, std::min<size_t>(grid, budget / (per_warp * SWEEP_WARPS)));
        const size_t need = per_warp * SWEEP_WARPS * grid;
        if (ctx->gcfm_glist_bytes < need) {
            if (ctx->gcfm_glist) cudaFree(ctx->gcfm_glist);
            ctx->gcfm_glist = nullptr; ctx->gcfm_glist_bytes = 0;
            if (cudaMalloc(&ctx->gcfm_glist, need) != cudaSuccess) {
                cudaGetLastError();
                oc::set_error("cannot allocate %zu bytes of candidate lists for the exact slow path", need);
                return OC_ERR_NOMEM;
            }
            ctx->gcfm_glist_bytes = need;
        }
        glists = (unsigned char *)ctx->gcfm_glist;
    }
    sweep_kernel<<<grid, SWEEP_WARPS * 32, smem, st>>>(L.prm, N, L.w, L.x, L.y, L.vx, L.vy, L.tim, L.status, L.vdes, L.key,
                                                      inv_cs, nbx, nby, (unsigned)ctx->gcfm_poll_ns, margin, cap, glists,
                                                      ctx->gcfm_fov_cull);
    exit_compact_kernel<<<1, 1024, 0, st>>>(N, L.w, L.pinned);
    oc::count_launch(2);
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}

// everything the first (fast) attempt of a step enqueues after the key descriptors: the staged header / permutation /
// normal pairs in one copy, bins, cell list, per-agent terms, candidate lists, sweep, exit log.  Run directly, or captured
// once into a CUDA graph and replayed (the step is ~13 launches of 3-150 us: enqueueing them costs the host more than
// the small ones take to run)
static int gcfm_enqueue_first(oc_ctx *ctx, GcfmLaunch &L, cudaStream_t st, size_t stage_bytes, bool split, bool dist) {
    Ws &w = L.w;
    OC_CUDA(cudaMemcpyAsync(w.hdr, ctx->gcfm_stage, stage_bytes, cudaMemcpyHostToDevice, st));
    int rc = gcfm_sweep_attempt(ctx, L, st, L.margin, true, split);
    if (rc) return rc;
    if (dist) {
        // merge the per-agent terms over the ranks: des_x, des_y, wfx, wfy are carved back to back (padding is zero),
        // every agent was written by exactly one rank and is all-zero bits elsewhere; the sampler-range flag likewise
        const size_t words = (size_t)((w.wfy + L.N) - w.des_x);
        if ((rc = oc_dist_allreduce_max_u64(ctx, w.des_x, words, st))) return rc;
        if ((rc = oc_dist_allreduce_max_u64(ctx, w.counters, 4, st))) return rc;  // 8 ints
    }
    return gcfm_launch_sweep(ctx, L, st, L.margin, CAND_CAP, false, split);
}

extern "C" int oc_gcfm_step_launch(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y,
                                   double *d_vx, double *d_vy, double *d_time, uint8_t *d_status, const double *d_vdes,
                                   const int *d_key, const oc_key *keys, int n_keys, const int *perm,
                                   const double *noise, int n_noise, int simu_step, void *stream) {
    OC_ARG(ctx && prm && d_x && d_y && d_vx && d_vy && d_time && d_status && d_vdes && d_key && keys && perm,
           "NULL argument");
    OC_ARG(N >= 1 && n_keys >= 1 && n_noise >= 0 && n_noise <= N, "bad sizes");
    OC_ARG(prm->Ny == ctx->Ny && prm->Nx == ctx->Nx, "params grid != context grid");
    OC_ARG(!ctx->gcfm_pending, "the previous GCFM step has not been finished (oc_gcfm_step_finish)");
    OC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = gcfm_device_setup(ctx);
    if (rc) return rc;
    // the bin table is sized for the smallest cells any attempt uses (a wider margin means larger cells, i.e. fewer bins)
    const int nbins = gcfm_max_bins(ctx, prm->cutoff);
    int n_doors = 0;
    for (int k = 0; k < n_keys; k++) n_doors += keys[k].n_doors;
    if (!ctx->gcfm_last) ctx->gcfm_last = new GcfmLaunch();
    GcfmLaunch &L = *static_cast<GcfmLaunch *>(ctx->gcfm_last);
    Ws &w = L.w;
    int *pinned = nullptr;
    rc = gcfm_workspace(ctx, N, n_keys, n_doors, nbins, w, &pinned, st);
    if (rc) return rc;
    L.prm = *prm; L.N = N; L.n_keys = n_keys; L.n_doors = n_doors; L.nbins_alloc = nbins;
    L.x = d_x; L.y = d_y; L.vx = d_vx; L.vy = d_vy; L.tim = d_time; L.status = d_status; L.vdes = d_vdes; L.key = d_key;
    L.pinned = pinned;
    // target-set descriptors (KeyDev records + door rectangles): uploaded only when they changed (a re-solve changes nt_opt)
    std::vector<char> sig(sizeof(KeyDev) * n_keys + sizeof(double) * 4 * std::max(n_doors, 1), 0);
    {
        KeyDev *hk = reinterpret_cast<KeyDev *>(sig.data());
        double *hd = reinterpret_cast<double *>(sig.data() + sizeof(KeyDev) * n_keys);
        int off = 0;
        for (int k = 0; k < n_keys; k++) {
            OC_ARG(keys[k].d_V && keys[k].d_wall_tiles, "key without potential / wall tiles");
            OC_ARG(!keys[k].d_vx == !keys[k].d_vy, "d_vx and d_vy must be given together");
            hk[k] = KeyDev{keys[k].d_V, keys[k].d_wall_tiles, keys[k].d_vx, keys[k].d_vy,
                           keys[k].d_vx ? nullptr : keys[k].d_phi, keys[k].nt_opt, keys[k].d_vx ? keys[k].n_slices : 0, off,
                           keys[k].n_doors, (keys[k].d_vx || !keys[k].d_phi) ? 0 : keys[k].n_phi, keys[k].v_min * 10e3,
                           keys[k].mu, keys[k].lim, keys[k].phi_row0, keys[k].phi_rows};
            OC_ARG(keys[k].phi_rows >= 0 && (keys[k].phi_rows == 0 || !keys[k].d_vx), "row-band storage needs phi samples");
            for (int d = 0; d < 4 * keys[k].n_doors; d++) hd[4 * (size_t)off + d] = keys[k].doors[d];
            off += keys[k].n_doors;
        }
    }
    OC_CUDA(cudaEventRecord(ctx->ev0, st));
    if (ctx->gcfm_keys_sig != sig || ctx->gcfm_keys_dev != (void *)w.keys) {
        ctx->gcfm_keys_sig = sig;  // the vector stays alive: pageable source of the asynchronous copies below
        ctx->gcfm_keys_dev = (void *)w.keys;
        OC_CUDA(cudaMemcpyAsync(w.keys, ctx->gcfm_keys_sig.data(), sizeof(KeyDev) * n_keys, cudaMemcpyHostToDevice, st));
        OC_CUDA(cudaMemcpyAsync(w.doors, ctx->gcfm_keys_sig.data() + sizeof(KeyDev) * n_keys,
                                sizeof(double) * 4 * std::max(n_doors, 1), cudaMemcpyHostToDevice, st));
    }
    L.margin = gcfm_fast_margin(ctx);
    L.simu_step = simu_step;
    // staging: header, permutation, normal pairs, laid out like w.hdr .. w.noise
    const size_t off_perm = (size_t)(reinterpret_cast<char *>(w.perm) - reinterpret_cast<char *>(w.hdr)),
                 off_noise = (size_t)(reinterpret_cast<char *>(w.noise) - reinterpret_cast<char *>(w.hdr));
    const size_t stage_full = off_noise + sizeof(double) * 2 * (size_t)N;
    if (ctx->gcfm_stage_bytes < stage_full) {
        if (ctx->gcfm_stage) cudaFreeHost(ctx->gcfm_stage);
        ctx->gcfm_stage = nullptr; ctx->gcfm_stage_bytes = 0;
        OC_CUDA(cudaMallocHost(&ctx->gcfm_stage, stage_full));
        memset(ctx->gcfm_stage, 0, stage_full);
        ctx->gcfm_stage_bytes = stage_full;
    }
    {
        char *hs = static_cast<char *>(ctx->gcfm_stage);
        int *hh = reinterpret_cast<int *>(hs);
        hh[0] = gcfm_next_tag(ctx);
        hh[1] = simu_step;
        memcpy(hs + off_perm, perm, sizeof(int) * (size_t)N);
        if (n_noise) memcpy(hs + off_noise, noise, sizeof(double) * 2 * (size_t)n_noise);
    }
    const bool split = ctx->gcfm_split != 0;
    const bool dist = (prm->own1 > prm->own0 || prm->key_mod > 0) && ctx->nccl_comm && ctx->nranks > 1;
    if (ctx->gcfm_use_graph && !dist) {
        // everything a node of the captured graph depends on
        struct Key {
            oc_gcfm_params prm;
            const void *p[12];
            int N, n_keys, nbins, knobs[8];
            double margin;
            size_t stage;
        } key;
        memset(&key, 0, sizeof(key));
        key.prm = *prm;
        const void *ptrs[12] = {d_x, d_y, d_vx, d_vy, d_time, d_status, d_vdes, d_key, ctx->gcfm_ws, pinned, ctx->gcfm_stage, ctx->d_X};
        memcpy(key.p, ptrs, sizeof(ptrs));
        key.N = N; key.n_keys = n_keys; key.nbins = nbins;
        const int knobs[8] = {ctx->gcfm_split, ctx->gcfm_fov_cull, ctx->gcfm_ws_pair, ctx->gcfm_overlap, ctx->gcfm_poll_ns,
                              ctx->gcfm_sweep_ctas, n_doors, 0};
        memcpy(key.knobs, knobs, sizeof(knobs));
        key.margin = L.margin;
        key.stage = stage_full;
        std::vector<char> kb(reinterpret_cast<char *>(&key), reinterpret_cast<char *>(&key) + sizeof(key));
        if (!ctx->gcfm_graph || kb != ctx->gcfm_graph_key) {
            if (ctx->gcfm_graph) { cudaGraphExecDestroy(ctx->gcfm_graph); ctx->gcfm_graph = nullptr; }
            if ((rc = gcfm_streams(ctx))) return rc;
            const long long l0 = oc::g_launches.load();
            OC_CUDA(cudaStreamBeginCapture(ctx->gcfm_cap, cudaStreamCaptureModeRelaxed));
            rc = gcfm_enqueue_first(ctx, L, ctx->gcfm_cap, stage_full, split, false);
            cudaGraph_t g = nullptr;
            cudaError_t e = cudaStreamEndCapture(ctx->gcfm_cap, &g);
            const int per_replay = (int)(oc::g_launches.load() - l0);
            oc::g_launches.fetch_add(-per_replay);  // (captured, not launched)
            if (rc) { if (g) cudaGraphDestroy(g); return rc; }
            OC_CUDA(e);
            e = cudaGraphInstantiate(&ctx->gcfm_graph, g, 0);
            cudaGraphDestroy(g);
            OC_CUDA(e);
            ctx->gcfm_graph_key = kb;
            ctx->gcfm_graph_launches = per_replay;
        }
        OC_CUDA(cudaGraphLaunch(ctx->gcfm_graph, st));
        oc::count_launch(ctx->gcfm_graph_launches);
    } else {
        const size_t used = off_noise + sizeof(double) * 2 * (size_t)n_noise;
        if ((rc = gcfm_enqueue_first(ctx, L, st, used, split, dist))) return rc;
    }
    OC_CUDA(cudaEventRecord(ctx->ev1, st));
    ctx->gcfm_stream = st;
    ctx->gcfm_pending = true;
    return OC_OK;
}

static int gcfm_finish_member(oc_ctx *ctx, int *exit_log, int *n_exit, bool synced, bool timed) {
    OC_ARG(ctx && ctx->gcfm_pending && ctx->gcfm_last, "no GCFM step in flight");
    OC_CUDA(cudaSetDevice(ctx->device));
    ctx->gcfm_pending = false;
    cudaStream_t st = (cudaStream_t)ctx->gcfm_stream;
    GcfmLaunch &L = *static_cast<GcfmLaunch *>(ctx->gcfm_last);
    if (!synced) OC_CUDA(cudaStreamSynchronize(st));  // host-visible exit log
    const int *pinned = (const int *)ctx->gcfm_pinned;
    // Exact slow path (rare).  The fast attempt keeps at most CAND_CAP candidates per agent in shared memory and
    // searches them within cutoff + DISP_MARGIN of the agent's old position.  An attempt that met more candidates, or
    // moved an agent further than the margin covers, is void: the state is restored from the step-start snapshot and
    // the step is redone with global-memory lists sized from the measured candidate count and with a margin that
    // covers the measured displacement, until an attempt is self-consistent.  The reference has neither limit
    // (simulations.py:285-303: all pairs, repulsions add to the velocity unclipped).
    double margin = L.margin;
    int cap = CAND_CAP;
    ctx->gcfm_redos = 0;
    for (int redo = 0; (pinned[1] & 6) != 0; redo++) {
        const double room_diag = std::sqrt(ctx->room_length * ctx->room_length + ctx->room_height * ctx->room_height);
        if (redo >= 14 || margin > 4.0 * room_diag + 8.0) {
            oc::set_error("GCFM step: no self-consistent candidate search (displacement %g m, %d candidates)", margin * 0.5, cap);
            return OC_ERR_ARG;
        }
        if ((pinned[1] & 6) == 4 && margin < DISP_MARGIN && cap == CAND_CAP) {
            // only the SMALL margin of the fast path was exceeded: redo on the fast path with the full DISP_MARGIN, and
            // keep that margin for the next steps (a crowd that kicks an agent > margin/2 once tends to do it again)
            double disp;
            memcpy(&disp, pinned + 4, sizeof(double));
            if (disp == disp && disp <= 0.45 * DISP_MARGIN) {
                margin = DISP_MARGIN;
                ctx->gcfm_margin_hold = 64;
                const bool split = ctx->gcfm_split != 0;
                int rc = gcfm_sweep_attempt(ctx, L, st, margin, false, split);
                if (rc) return rc;
                if ((rc = gcfm_launch_sweep(ctx, L, st, margin, CAND_CAP, false, split))) return rc;
                if (timed) OC_CUDA(cudaEventRecord(ctx->ev1, st));
                OC_CUDA(cudaStreamSynchronize(st));
                ctx->gcfm_redos = redo + 1;
                continue;
            }
        }
        if (pinned[1] & 4) {
            double disp;
            memcpy(&disp, pinned + 4, sizeof(double));
            // NaN / inf displacement: widen geometrically up to the whole room, then give up above
            margin = (disp == disp && disp < 1e300) ? std::max(2.0 * margin, 2.2 * disp) : 4.0 * margin;
        }
        {   // lists for every candidate the void attempt counted; a wider search finds more: the loop adapts
            long long want = std::max<long long>(pinned[3], cap);
            if (pinned[1] & 4) want = std::max<long long>(want, 2 * (long long)pinned[3]);
            int c2 = CAND_CAP;
            while (c2 < want && c2 < CAND_CAP_MAX) c2 <<= 1;
            if (want > CAND_CAP_MAX) {
                oc::set_error("more than %d agents within the repulsion reach of one agent", CAND_CAP_MAX);
                return OC_ERR_ARG;
            }
            cap = c2;
        }
        int rc = gcfm_sweep_attempt(ctx, L, st, margin, false, false);
        if (rc) return rc;
        if ((rc = gcfm_launch_sweep(ctx, L, st, margin, cap, true, false))) return rc;
        if (timed) OC_CUDA(cudaEventRecord(ctx->ev1, st));
        OC_CUDA(cudaStreamSynchronize(st));
        ctx->gcfm_redos = redo + 1;
    }
    if (timed) {
        float ms = 0;
        OC_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        ctx->gcfm_last_ms = ms;
    }
    ctx->gcfm_last_pairs = pinned[2];
    int ne = pinned[0], fl = pinned[1];
    if (n_exit) *n_exit = ne;
    if (exit_log)
        for (int q = 0; q < ne; q++) exit_log[q] = pinned[OUT_HDR + q];
    if (fl & 1) {
        oc::set_error("agent position outside the sampler's index range (the reference raises IndexError here)");
        return OC_ERR_SAMPLER_RANGE;
    }
    return OC_OK;
}

extern "C" int oc_gcfm_step_finish(oc_ctx *ctx, int *exit_log, int *n_exit) {
    return gcfm_finish_member(ctx, exit_log, n_exit, false, true);
}

// ------------------------------------------------------------------------------------------------ batched step (ensembles)
// One GCFM step of n independent members (each with its own context, crowd, fields and legacy RNG stream) with ONE launch
// per kernel (blockIdx.y = member).  The host part -- per member: the step's permutation and normal pairs from the
// member's MT19937 state (oc_rng.h: numpy's legacy stream, simulations.py:271,303), the staging of both, the member
// record -- runs in C; perm / noise of all members travel in one host-to-device copy.
extern "C" int oc_gcfm_step_multi_launch(int n, oc_ctx *const *ctxs, const oc_gcfm_params *const *prms, const int *Ns,
                                         double *const *x, double *const *y, double *const *vx, double *const *vy,
                                         double *const *tim, uint8_t *const *status, const double *const *vdes,
                                         const int *const *key, const oc_key *const *keys, const int *n_keys,
                                         uint32_t *const *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss,
                                         const int *n_active, const int *simu_step, int sweep_ctas, void *stream) {
    OC_ARG(n >= 1 && ctxs && prms && Ns && x && y && vx && vy && tim && status && vdes && key && keys && n_keys && mt_key &&
           mt_pos && has_gauss && cached_gauss && n_active && simu_step, "NULL argument");
    oc_ctx *c0 = ctxs[0];
    OC_CUDA(cudaSetDevice(c0->device));
    cudaStream_t st = (cudaStream_t)stream;
    // ---- staging arena: per member perm (N ints, padded to 8 bytes) + noise (2 n_active doubles)
    // OC_DEBUG_TIMING=1: host time of the three parts of a batched launch, printed every 100 calls
    static const bool dbg_t = getenv("OC_DEBUG_TIMING") != nullptr;
    static double dbg_acc[3] = {0, 0, 0};
    static int dbg_n = 0;
    auto dbg_now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double dbg_t0 = dbg_t ? dbg_now() : 0.0;
    std::vector<size_t> off(n + 1, 0);
    int max_N = 0;
    for (int m = 0; m < n; m++) {
        OC_ARG(ctxs[m] && ctxs[m]->device == c0->device && Ns[m] >= 1 && n_active[m] >= 0 && n_active[m] <= Ns[m] &&
               prms[m]->own1 <= prms[m]->own0 && prms[m]->key_mod == 0, "bad member");
        off[m + 1] = off[m] + (((size_t)Ns[m] * sizeof(int) + 7) / 8) * 8 + (size_t)2 * n_active[m] * sizeof(double);
        max_N = std::max(max_N, Ns[m]);
    }
    // a void member attempt is redone in oc_gcfm_step_multi_finish with the single-step kernels: their shared-memory
    // limits and the member's resident grids must be set even if this context never took a single step
    for (int m = 0; m < n; m++) {
        int rc = gcfm_device_setup(ctxs[m]);
        if (rc) return rc;
    }
    const size_t arena = off[n] + 64, rec_bytes = sizeof(GcfmMember) * (size_t)n;
    if (c0->multi_bytes < arena + rec_bytes) {
        if (c0->multi_pinned) cudaFreeHost(c0->multi_pinned);
        if (c0->multi_dev) cudaFree(c0->multi_dev);
        c0->multi_pinned = c0->multi_dev = nullptr; c0->multi_bytes = 0;
        const size_t cap = (arena + rec_bytes) * 2;
        OC_CUDA(cudaMallocHost(&c0->multi_pinned, cap));
        OC_CUDA(cudaMalloc(&c0->multi_dev, cap));
        c0->multi_bytes = cap;
    }
    char *hp = (char *)c0->multi_pinned, *dp = (char *)c0->multi_dev;
    GcfmMember *recs = reinterpret_cast<GcfmMember *>(hp + ((arena + 63) / 64) * 64);
    GcfmMember *recs_dev = reinterpret_cast<GcfmMember *>(dp + ((arena + 63) / 64) * 64);
    OC_CUDA(cudaEventRecord(c0->ev0, st));
    int max_bins = 0;
    for (int m = 0; m < n; m++) {
        oc_ctx *ctx = ctxs[m];
        const oc_gcfm_params *prm = prms[m];
        const int N = Ns[m];
        OC_ARG(prm->Ny == ctx->Ny && prm->Nx == ctx->Nx, "params grid != context grid");
        const double margin = gcfm_fast_margin(ctx);
        const double reach = prm->cutoff + margin, inv_cs = 2.0 / reach;
        const int nbx = std::max(1, (int)std::ceil(ctx->room_length * inv_cs)),
                  nby = std::max(1, (int)std::ceil(ctx->room_height * inv_cs));
        const int nbins = nbx * nby, nbins_alloc = gcfm_max_bins(ctx, prm->cutoff);
        int n_doors = 0;
        for (int k = 0; k < n_keys[m]; k++) n_doors += keys[m][k].n_doors;
        if (!ctx->gcfm_last) ctx->gcfm_last = new GcfmLaunch();
        GcfmLaunch &L = *static_cast<GcfmLaunch *>(ctx->gcfm_last);
        int *pinned = nullptr;
        int rc = gcfm_workspace(ctx, N, n_keys[m], n_doors, nbins_alloc, L.w, &pinned, st);
        if (rc) return rc;
        L.prm = *prm; L.N = N; L.n_keys = n_keys[m]; L.n_doors = n_doors; L.nbins_alloc = nbins_alloc; L.margin = margin;
        L.simu_step = simu_step[m];
        L.x = x[m]; L.y = y[m]; L.vx = vx[m]; L.vy = vy[m]; L.tim = tim[m]; L.status = status[m]; L.vdes = vdes[m];
        L.key = key[m]; L.pinned = pinned;
        // target-set descriptors: uploaded only when they changed (a re-solve changes nt_opt)
        std::vector<char> sig(sizeof(KeyDev) * n_keys[m] + sizeof(double) * 4 * std::max(n_doors, 1), 0);
        KeyDev *hk = reinterpret_cast<KeyDev *>(sig.data());
        double *hd = reinterpret_cast<double *>(sig.data() + sizeof(KeyDev) * n_keys[m]);
        int doff = 0;
        for (int k = 0; k < n_keys[m]; k++) {
            const oc_key &kk = keys[m][k];
            OC_ARG(kk.d_V && kk.d_wall_tiles && (!kk.d_vx == !kk.d_vy), "bad key");
            hk[k] = KeyDev{kk.d_V, kk.d_wall_tiles, kk.d_vx, kk.d_vy, kk.d_vx ? nullptr : kk.d_phi, kk.nt_opt,
                           kk.d_vx ? kk.n_slices : 0, doff, kk.n_doors, (kk.d_vx || !kk.d_phi) ? 0 : kk.n_phi, kk.v_min * 10e3,
                           kk.mu, kk.lim, kk.phi_row0, kk.phi_rows};
            for (int d = 0; d < 4 * kk.n_doors; d++) hd[4 * (size_t)doff + d] = kk.doors[d];
            doff += kk.n_doors;
        }
        if (ctx->gcfm_keys_sig != sig || ctx->gcfm_keys_dev != (void *)L.w.keys) {
            ctx->gcfm_keys_sig = sig;   // the vector stays alive: pageable source of the asynchronous copies below
            ctx->gcfm_keys_dev = (void *)L.w.keys;
            OC_CUDA(cudaMemcpyAsync(L.w.keys, ctx->gcfm_keys_sig.data(), sizeof(KeyDev) * n_keys[m], cudaMemcpyHostToDevice, st));
            OC_CUDA(cudaMemcpyAsync(L.w.doors, ctx->gcfm_keys_sig.data() + sizeof(KeyDev) * n_keys[m],
                                    sizeof(double) * 4 * std::max(n_doors, 1), cudaMemcpyHostToDevice, st));
        }
        // (this step's randomness is drawn below, by a few host threads, straight into the staging arena)
        L.w.perm = reinterpret_cast<int *>(dp + off[m]);
        L.w.noise = reinterpret_cast<double *>(dp + off[m] + (((size_t)N * sizeof(int) + 7) / 8) * 8);
        if (++ctx->gcfm_tag >= 0x3fffffff) ctx->gcfm_tag = 1;
        GcfmMember &r = recs[m];
        r.prm = *prm; r.w = L.w; r.x = x[m]; r.y = y[m]; r.vx = vx[m]; r.vy = vy[m]; r.tim = tim[m]; r.status = status[m];
        r.vdes = vdes[m]; r.X = ctx->d_X; r.Y = ctx->d_Y; r.key = key[m]; r.out = pinned; r.N = N;
        r.simu_step = simu_step[m]; r.tag = ctx->gcfm_tag; r.nbx = nbx; r.nby = nby; r.nbins = nbins; r.inv_cs = inv_cs;
        r.poll_ns = (unsigned)ctx->gcfm_poll_ns; r.fov_cull = ctx->gcfm_fov_cull; r.margin = margin;
        max_bins = std::max(max_bins, nbins);
        ctx->gcfm_stream = st;
        ctx->gcfm_pending = true;
    }
    const double dbg_t1 = dbg_t ? dbg_now() : 0.0;
    {   // the members' streams are independent: draw them in parallel (simulations.py:271,303 per member)
        const int n_thr = std::max(1, std::min({n, 8, (int)std::thread::hardware_concurrency()}));
        auto work = [&](int t) {
            for (int m = t; m < n; m += n_thr) {
                const int N = Ns[m];
                int *perm_h = reinterpret_cast<int *>(hp + off[m]);
                double *noise_h = reinterpret_cast<double *>(hp + off[m] + (((size_t)N * sizeof(int) + 7) / 8) * 8);
                ocrng::Mt mt{mt_key[m], mt_pos[m], has_gauss[m], cached_gauss[m]};
                mt.permutation(N, perm_h);
                for (int q = 0; q < 2 * n_active[m]; q++) noise_h[q] = mt.gauss();
                mt_pos[m] = mt.pos; has_gauss[m] = mt.has_gauss; cached_gauss[m] = mt.gauss_;
            }
        };
        std::vector<std::thread> pool;
        for (int t = 1; t < n_thr; t++) pool.emplace_back(work, t);
        work(0);
        for (auto &th : pool) th.join();
    }
    const double dbg_t2 = dbg_t ? dbg_now() : 0.0;
    OC_CUDA(cudaMemcpyAsync(dp, hp, ((arena + 63) / 64) * 64 + rec_bytes, cudaMemcpyHostToDevice, st));
    OC_CUDA(cudaFuncSetAttribute(sweep_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SWEEP_SMEM));
    const int nb = (max_N + 255) / 256;
    const int ctas = std::max(1, std::min(sweep_ctas > 0 ? sweep_ctas : 8, (max_N + SWEEP_WARPS - 1) / SWEEP_WARPS));
    clear_multi_kernel<<<dim3(std::max(1, std::min(8, (std::max(max_N, max_bins) + 255) / 256)), n), 256, 0, st>>>(recs_dev);
    setup_multi_kernel<<<dim3(nb, n), 256, 0, st>>>(recs_dev);
    cudaStream_t side = st, side2 = st;
    {
        int rc = gcfm_fork(c0, st, &side, &side2);
        if (rc) return rc;
    }
    noise_index_multi_kernel<<<dim3(1, n), 1024, 0, side2>>>(recs_dev);
    if (c0->gcfm_ws_pair) wall_search_multi_kernel<true><<<dim3((max_N * 32 + 127) / 128, n), 128, 0, side>>>(recs_dev);
    else wall_search_multi_kernel<false><<<dim3((max_N * 32 + 127) / 128, n), 128, 0, side>>>(recs_dev);
    agent_terms_multi_kernel<<<dim3(nb * 2, n), 128, 0, side>>>(recs_dev);
    scan_multi_kernel<<<dim3(1, n), 1024, 0, st>>>(recs_dev);
    scatter_multi_kernel<<<dim3(nb, n), 256, 0, st>>>(recs_dev);
    const bool split = c0->gcfm_split != 0;
    if (split) {
        OC_CUDA(cudaFuncSetAttribute(cand_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAND_SMEM));
        OC_CUDA(cudaFuncSetAttribute(chain_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CHAIN_SMEM));
        cand_multi_kernel<<<dim3((max_N + SWEEP_WARPS - 1) / SWEEP_WARPS, n), SWEEP_WARPS * 32, CAND_SMEM, st>>>(recs_dev);
    }
    {
        int rc = gcfm_join(c0, st, side, side2);
        if (rc) return rc;
    }
    if (split) chain_multi_kernel<<<dim3(ctas, n), SWEEP_WARPS * 32, CHAIN_SMEM, st>>>(recs_dev);
    else sweep_multi_kernel<<<dim3(ctas, n), SWEEP_WARPS * 32, SWEEP_SMEM, st>>>(recs_dev);
    exit_compact_multi_kernel<<<dim3(1, n), 1024, 0, st>>>(recs_dev);
    oc::count_launch(split ? 10 : 9);
    OC_CUDA(cudaGetLastError());
    OC_CUDA(cudaEventRecord(c0->ev1, st));
    if (dbg_t) {
        const double t3 = dbg_now();
        dbg_acc[0] += dbg_t1 - dbg_t0; dbg_acc[1] += dbg_t2 - dbg_t1; dbg_acc[2] += t3 - dbg_t2;
        if (++dbg_n % 100 == 0) {
            fprintf(stderr, "[oc multi launch x100, %d members] member records %.2f ms, rng draws %.2f ms, enqueue %.2f ms per call\n",
                    n, dbg_acc[0] / 100, dbg_acc[1] / 100, dbg_acc[2] / 100);
            dbg_acc[0] = dbg_acc[1] = dbg_acc[2] = 0;
        }
    }
    return OC_OK;
}

extern "C" int oc_gcfm_step_multi_finish(int n, oc_ctx *const *ctxs, int *const *exit_log, int *n_exit, int *rc_out) {
    OC_ARG(n >= 1 && ctxs && exit_log && n_exit && rc_out && ctxs[0] && ctxs[0]->gcfm_pending, "no batched GCFM step in flight");
    oc_ctx *c0 = ctxs[0];
    OC_CUDA(cudaSetDevice(c0->device));
    OC_CUDA(cudaStreamSynchronize((cudaStream_t)c0->gcfm_stream));
    float ms = 0;
    OC_CUDA(cudaEventElapsedTime(&ms, c0->ev0, c0->ev1));
    int worst = OC_OK;
    for (int m = 0; m < n; m++) {
        // (a member whose fast attempt was void is redone alone on the exact slow path, like a single step)
        rc_out[m] = gcfm_finish_member(ctxs[m], exit_log[m], &n_exit[m], true, false);
        if (rc_out[m] != OC_OK && rc_out[m] != OC_ERR_SAMPLER_RANGE) worst = rc_out[m];
    }
    c0->gcfm_last_ms = ms;
    return worst;
}

// ------------------------------------------------------------------------------------------------ run loop
// Up to n_steps consecutive steps of simulations.run()'s loop body (simulations.py:427-441 minus the periodic re-solve)
// without returning to the host language between them.  Per step: the permutation and the normal pairs of the agents
// inside from the caller's legacy MT19937 state (np.random.get_state()[1:5], advanced in place; oc_rng.h), the step,
// the exit bookkeeping and -- when d_rows is given -- one row of the trajectory record (oc_state_pack into d_rows[k]).
// While the GPU runs step k this thread draws step k+1's randomness from a COPY of the generator state for the upper
// bound "nobody leaves", with snapshots of the state after n - q pairs (q < 64): when step k's exit count q is known,
// the first n - q pairs are exactly the reference's draws and the generator continues from snapshot q; otherwise the
// step is drawn afresh.  The stream of random numbers is the reference's whatever happens.
// Stops early when nobody is inside (the reference's loop condition) or on an error; *steps_done steps were executed
// (on OC_ERR_SAMPLER_RANGE including the offending one, as oc_gcfm_step).  exit_agent / exit_step (capacity N): agents in
// exit order and the index (0-based within this call) of the step they left in.  *device_ms: sum of the steps' CUDA-event
// times; *pairs: interacting pairs evaluated.
extern "C" int oc_gcfm_run(oc_ctx *ctx, const oc_gcfm_params *prm, int N, double *d_x, double *d_y, double *d_vx,
                           double *d_vy, double *d_time, uint8_t *d_status, const double *d_vdes, const int *d_key,
                           const oc_key *keys, int n_keys, uint32_t *mt_key, int *mt_pos, int *has_gauss,
                           double *cached_gauss, int n_steps, int simu_step0, int n_active0, double *const *d_rows,
                           int *exit_agent, int *exit_step, int *n_exits, int *steps_done, double *device_ms,
                           long long *pairs, void *stream) {
    OC_ARG(ctx && prm && mt_key && mt_pos && has_gauss && cached_gauss && exit_agent && exit_step && n_exits && steps_done,
           "NULL argument");
    OC_ARG(N >= 1 && n_steps >= 0 && n_active0 >= 0 && n_active0 <= N && *mt_pos >= 0 && *mt_pos <= 624, "bad sizes");
    constexpr int N_CKPT = 64;
    *n_exits = 0;
    *steps_done = 0;
    if (device_ms) *device_ms = 0.0;
    if (pairs) *pairs = 0;
    std::vector<int> perm(N), perm2(N), log_(N);
    std::vector<double> noise(2 * (size_t)N), noise2(2 * (size_t)N);
    std::vector<uint32_t> ck_key((size_t)N_CKPT * 624), key2(624);
    int ck_pos[N_CKPT], ck_has[N_CKPT];
    double ck_cached[N_CKPT];
    bool spec = false;   // perm2 / noise2 / snapshots hold a look-ahead draw for n_spec pairs
    int n_spec = 0, n_ckpt = 0;
    int n_active = n_active0;
    int rc = OC_OK;
    for (int k = 0; k < n_steps && n_active > 0; k++) {
        // ---- this step's randomness (simulations.py:271,303)
        const int q = n_spec - n_active;
        if (spec && q >= 0 && q < n_ckpt) {
            perm.swap(perm2);
            noise.swap(noise2);
            memcpy(mt_key, ck_key.data() + (size_t)624 * q, 624 * sizeof(uint32_t));
            *mt_pos = ck_pos[q]; *has_gauss = ck_has[q]; *cached_gauss = ck_cached[q];
        } else {
            ocrng::Mt mt{mt_key, *mt_pos, *has_gauss, *cached_gauss};
            mt.permutation(N, perm.data());
            mt.gauss_fill(noise.data(), 2ll * n_active);
            *mt_pos = mt.pos; *has_gauss = mt.has_gauss; *cached_gauss = mt.gauss_;
        }
        spec = false;
        rc = oc_gcfm_step_launch(ctx, prm, N, d_x, d_y, d_vx, d_vy, d_time, d_status, d_vdes, d_key, keys, n_keys, perm.data(),
                                 noise.data(), n_active, simu_step0 + k, stream);
        if (rc) return rc;
        // ---- look-ahead: the next step's draws while the GPU sweeps (not after the last step of this call)
        if (k + 1 < n_steps) {
            memcpy(key2.data(), mt_key, 624 * sizeof(uint32_t));
            ocrng::Mt mt2{key2.data(), *mt_pos, *has_gauss, *cached_gauss};
            mt2.permutation(N, perm2.data());
            n_spec = n_active;
            n_ckpt = std::min(N_CKPT, n_spec + 1);
            mt2.gauss_fill(noise2.data(), 2ll * n_spec, n_ckpt, ck_key.data(), ck_pos, ck_has, ck_cached);
            spec = true;
        }
        int ne = 0;
        rc = oc_gcfm_step_finish(ctx, log_.data(), &ne);
        if (rc != OC_OK && rc != OC_ERR_SAMPLER_RANGE) return rc;
        for (int e = 0; e < ne; e++) {
            exit_agent[*n_exits] = log_[e];
            exit_step[*n_exits] = k;
            (*n_exits)++;
        }
        n_active -= ne;
        if (device_ms) *device_ms += ctx->gcfm_last_ms;
        if (pairs) *pairs += ctx->gcfm_last_pairs;
        if (d_rows && d_rows[k]) {
            int r2 = oc_state_pack(ctx, N, d_x, d_y, d_vx, d_vy, d_rows[k], stream);
            if (r2) return r2;
        }
        (*steps_done)++;
        if (rc == OC_ERR_SAMPLER_RANGE) return rc;
    }
    return OC_OK;
}

extern "C" double oc_gcfm_last_ms(oc_ctx *ctx) { return ctx ? ctx->gcfm_last_ms : 0.0; }
extern "C" long long oc_gcfm_last_pairs(oc_ctx *ctx) { return ctx ? ctx->gcfm_last_pairs : 0; }
extern "C" int oc_gcfm_last_redos(oc_ctx *ctx) { return ctx ? ctx->gcfm_redos : 0; }
void oc_gcfm_free_launch_state(oc_ctx *ctx) {  // oc_ctx_destroy (oc_api.cu)
    if (ctx && ctx->gcfm_last) { delete static_cast<GcfmLaunch *>(ctx->gcfm_last); ctx->gcfm_last = nullptr; }
    if (ctx && ctx->gcfm_glist) { cudaFree(ctx->gcfm_glist); ctx->gcfm_glist = nullptr; ctx->gcfm_glist_bytes = 0; }
}

extern "C" int oc_wall_force(oc_ctx *ctx, const oc_gcfm_params *prm, const double *d_V, int N, const double *d_x,
                             const double *d_y, const double *d_vx, const double *d_vy, const double *d_vdes,
                             double *d_fx, double *d_fy, long long *d_ind, void *stream) {
    OC_ARG(ctx && prm && d_V && d_x && d_y && d_vx && d_vy && d_vdes && d_fx && d_fy, "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *d_tiles = nullptr;
    OC_CUDA(cudaMalloc(&d_tiles, (size_t)oc_wall_tiles_bytes(ctx)));
    double vmin = 0;
    int rc = oc_wall_tiles(ctx, d_V, d_tiles, &vmin, stream);
    if (rc == OC_OK) {
        wall_probe_kernel<<<(N * 32 + 127) / 128, 128, 0, st>>>(*prm, N, ctx->d_X, ctx->d_Y, d_V, d_tiles, vmin * 10e3,
                                                                 d_x, d_y, d_vx, d_vy, d_vdes, d_fx, d_fy, d_ind);
        oc::count_launch();
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { oc::set_error("wall_probe_kernel: %s", cudaGetErrorString(e)); rc = OC_ERR_CUDA; }
    }
    cudaFree(d_tiles);
    return rc;
}

extern "C" int oc_pair_force(oc_ctx *ctx, const oc_gcfm_params *prm, int N, const double *d_pi, const double *d_vi,
                             const double *d_vdes, const double *d_pj, const double *d_vj, double *d_f, void *stream) {
    OC_ARG(ctx && prm && d_pi && d_vi && d_vdes && d_pj && d_vj && d_f, "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    pair_probe_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*prm, N, d_pi, d_vi, d_vdes, d_pj, d_vj, d_f);
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}

extern "C" int oc_density(oc_ctx *ctx, int N, const double *d_x, const double *d_y, const uint8_t *d_status,
                          double sigma, double C, const double *d_Vglobal, double *d_out, void *stream) {
    OC_ARG(ctx && d_Vglobal && d_out && (N == 0 || (d_x && d_y && d_status)), "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    const double two_s2 = 2 * (sigma * sigma);
    // ocm_exp(x) == 0 exactly for x < -745.14: r^2/two_s2 > 745.2  =>  contribution is exactly 0.0
    const double r_zero = std::sqrt(745.2 * two_s2) * (1.0 + 1e-9) + 1e-9;
    dim3 grid((ctx->Nx + DN_TX - 1) / DN_TX, (ctx->Ny + DN_TY - 1) / DN_TY);
    density_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(N, d_x, d_y, d_status, ctx->d_X, ctx->d_Y, d_Vglobal,
                                                           ctx->Ny, ctx->Nx, two_s2, C, r_zero, d_out);
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}
