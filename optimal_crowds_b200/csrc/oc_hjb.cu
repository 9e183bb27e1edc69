// oc_hjb.cu -- HJB solve on sm_100a: RHS stencil (K1), RK45 stage kernels with the stage combination
// fused into the stencil load (K2, stage-wise formulation), dense output + velocity epilogue (K3), and the host
// drivers of the single-room and batched solves.  Both drivers (and the row-band solve, oc_hjb_dist.cu) step
// scipy's RK45 controller rk45::Controller (oc_rk45.h) and fill the fused step's per-attempt constants with
// fused::set_attempt (oc_hjb_fused.cuh).
//
// Reference: optimals.py:124-206 (compute_optimal_velocity) + scipy 1.18.1 solve_ivp/RK45
// (rk.py:14-71,85-180,538-565,715-737; common.py:63-134; ivp.py:604-621,659-728; base.py:179-210).
//
// Data layout in HBM: every field is a dense C-order (Ny,Nx) FP64 array.  Workspace = y, y_new, K[0..6],
// coef (10 arrays).  coef = (V + g*m)/(mu*sigma^2), with NaN marking wall cells (V<0 -> k = 0, optimals.py:162).
//
// Error norm: per-tile partial sums -> per-tile-row sums (fixed order) -> sequential sum over tile rows on
// the host.  The order depends only on global tile indices, so a row-band decomposition whose bands are
// multiples of TY rows reproduces the single-GPU sum bit for bit.
#include <cmath>
#include <algorithm>
#include <vector>

#include "oc_common.h"
#include "oc_hjb_fused.cuh"
#include "oc_hjb_final.h"
#include "oc_rk45.h"
#include "oc_vels.h"

namespace {

constexpr int TX = 128, TY = 16, NTHREADS = 256;  // stage tile
constexpr int SW = TX + 2;                        // smem row pitch (doubles)

// y + h * sum_j a[j]*k[j]  (rk.py:63-64: dy = np.dot(K[:s].T, a[:s]) * h ; y + dy)
struct Comb {
    const double *y;
    const double *k[6];
    double a[6];
    double h;
};

template <int N>
__device__ __forceinline__ double comb_eval(const Comb &c, size_t idx) {
    if (N == 0) return c.y[idx];
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < N; j++) acc += __ldg(c.k[j] + idx) * c.a[j];
    return c.y[idx] + acc * c.h;
}

struct ErrArgs {        // MODE 1 only
    const double *k[6];  // K[0..5] (K[6] is the kernel's own output)
    double e[7];
    double h, rtol, atol;
};

__device__ __forceinline__ double block_sum(double v, double *red) {
    // fixed-order tree: warp shuffle, then warp 0 over the 8 warp sums
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) red[w] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < NTHREADS / 32; i++) s += red[i];
    }
    return s;  // valid on thread 0
}

// MODE 0: kout = f(comb)                         (one RK stage, rk.py:62-64)
// MODE 1: ynew = comb; kout = f(ynew); partial[tile] = sum((h*K.E/scale)^2)   (rk.py:66-69,146-147)
template <int N, int MODE>
__global__ void __launch_bounds__(NTHREADS)
hjb_stage_kernel(Comb c, const double *__restrict__ coef, double *__restrict__ kout, double *__restrict__ ynew,
                 ErrArgs ea, double *__restrict__ partial, int Ny, int Nx, double diff_over_dxdy) {
    __shared__ double tile[(TY + 2) * SW];
    __shared__ double red[NTHREADS / 32];
    const int tx0 = blockIdx.x * TX, ty0 = blockIdx.y * TY;
    for (int idx = threadIdx.x; idx < (TY + 2) * SW; idx += NTHREADS) {
        int ly = idx / SW, lx = idx - ly * SW;
        int gy = ty0 + ly - 1, gx = tx0 + lx - 1;
        // mirror ghosts (optimals.py:149-152): row -1 := row 1, row Ny := row Ny-2; same for columns
        if (gy < 0) gy = 1;
        if (gy == Ny) gy = Ny - 2;
        if (gx < 0) gx = 1;
        if (gx == Nx) gx = Nx - 2;
        double v = 0.0;
        if (gy < Ny && gx < Nx) v = comb_eval<N>(c, (size_t)gy * Nx + gx);
        tile[idx] = v;
    }
    __syncthreads();
    double acc = 0.0;
    const int lx = threadIdx.x & (TX - 1);
    const int gx = tx0 + lx;
#pragma unroll 2
    for (int ly = threadIdx.x / TX; ly < TY; ly += NTHREADS / TX) {
        int gy = ty0 + ly;
        if (gy >= Ny || gx >= Nx) continue;
        size_t g = (size_t)gy * Nx + gx;
        const double *t = tile + (ly + 1) * SW + (lx + 1);
        double C = t[0];
        // optimals.py:154-160 (same summation order: up + down + left + right - 4C)
        double lap = t[-SW] + t[SW] + t[-1] + t[1] - 4.0 * C;
        double cf = coef[g];
        double r = diff_over_dxdy * lap - cf * C;
        if (cf != cf) r = 0.0;  // wall: optimals.py:162
        kout[g] = r;
        if (MODE == 1) {
            ynew[g] = C;
            double e = r * ea.e[6];
#pragma unroll
            for (int j = 5; j >= 0; j--)
                if (j != 1) e += __ldg(ea.k[j] + g) * ea.e[j];
            double sc = ea.atol + fmax(fabs(c.y[g]), fabs(C)) * ea.rtol;
            double q = (e * ea.h) / sc;
            acc += q * q;
        }
    }
    if (MODE == 1) {
        double s = block_sum(acc, red);
        if (threadIdx.x == 0) partial[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = s;
    }
}

// sum of the tile partials of one tile row, in fixed order -> rowsum[tile_row]
__global__ void __launch_bounds__(NTHREADS) rowgroup_sum_kernel(const double *__restrict__ partial, int nbx,
                                                                double *__restrict__ rowsum) {
    __shared__ double red[NTHREADS / 32];
    double v = 0.0;
    for (int i = threadIdx.x; i < nbx; i += NTHREADS) v += partial[(size_t)blockIdx.x * nbx + i];
    double s = block_sum(v, red);
    if (threadIdx.x == 0) rowsum[blockIdx.x] = s;
}

// select_initial_step norms (common.py:109-127): mode 0: (y/sc)^2 and (f/sc)^2 ; mode 1: ((f1-f0)/sc)^2
__global__ void __launch_bounds__(NTHREADS)
init_norm_kernel(const double *__restrict__ y, const double *__restrict__ f0, const double *__restrict__ f1,
                 double rtol, double atol, int Ny, int Nx, double *__restrict__ partial, int mode) {
    __shared__ double red[NTHREADS / 32];
    const int tx0 = blockIdx.x * TX, ty0 = blockIdx.y * TY;
    const int gx = tx0 + (threadIdx.x & (TX - 1));
    double a0 = 0.0, a1 = 0.0;
    for (int ly = threadIdx.x / TX; ly < TY; ly += NTHREADS / TX) {
        int gy = ty0 + ly;
        if (gy >= Ny || gx >= Nx) continue;
        size_t g = (size_t)gy * Nx + gx;
        double sc = atol + fabs(y[g]) * rtol;
        if (mode == 0) {
            double q0 = y[g] / sc, q1 = f0[g] / sc;
            a0 += q0 * q0;
            a1 += q1 * q1;
        } else {
            double q = (f1[g] - f0[g]) / sc;
            a0 += q * q;
        }
    }
    size_t nb = (size_t)gridDim.x * gridDim.y, b = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
    double s0 = block_sum(a0, red);
    if (threadIdx.x == 0) partial[b] = s0;
    __syncthreads();
    if (mode == 0) {
        double s1 = block_sum(a1, red);
        if (threadIdx.x == 0) partial[nb + b] = s1;
    }
}

// coef = (V<0) ? NaN : (V + g*m)/(mu*sigma^2); y = 1 (optimals.py:83)
__global__ void prep_kernel(const double *__restrict__ V, const double *__restrict__ m, double g, double inv_den,
                            size_t n, double *__restrict__ coef, double *__restrict__ y) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double v = V[i];
    double mm = m ? m[i] : 0.0;
    coef[i] = (v < 0) ? __longlong_as_double(0x7ff8000000000000LL) : (v + g * mm) * inv_den;
    if (y) y[i] = 1.0;
}

// ---------------------------------------------------------------------------------------------------
// K3: dense output (rk.py:178-180,723-737) + vels (optimals.py:168-186), up to DMAX t_eval points per launch.
constexpr int DTX = 64, DTY = 8, DSW = DTX + 2, DMAX = 6;
constexpr int DCELLS = (DTY + 2) * DSW;                      // 660
constexpr int DPER = (DCELLS + NTHREADS - 1) / NTHREADS;     // 3

struct DenseArgs {
    const double *yold;
    const double *k[7];
    double P[7][4];
    double h;  // t - t_old (RkDenseOutput.h)
    int n_emit;
    double x[DMAX];       // (t_eval - t_old)/h
    double *phi[DMAX];    // (Ny,Nx) slice or NULL
    double *vx[DMAX];     // (Ny-2,Nx-2) slice or NULL
    double *vy[DMAX];
    double mu, lim, inv_two_dx, inv_two_dy;
};

__global__ void __launch_bounds__(NTHREADS) hjb_dense_kernel(DenseArgs a, int Ny, int Nx) {
    __shared__ double tile[DCELLS];
    const int tx0 = blockIdx.x * DTX, ty0 = blockIdx.y * DTY;
    double q[DPER][4], y0[DPER];
#pragma unroll
    for (int s = 0; s < DPER; s++) {
        int idx = threadIdx.x + s * NTHREADS;
        q[s][0] = q[s][1] = q[s][2] = q[s][3] = 0.0;
        y0[s] = 0.0;
        if (idx < DCELLS) {
            int ly = idx / DSW, lx = idx - ly * DSW;
            int gy = ty0 + ly - 1, gx = tx0 + lx - 1;
            if (gy >= 0 && gy < Ny && gx >= 0 && gx < Nx) {
                size_t g = (size_t)gy * Nx + gx;
                y0[s] = a.yold[g];
#pragma unroll
                for (int j = 0; j < 7; j++) {
                    if (j == 1) continue;  // P[1,:] == 0
                    double kj = __ldg(a.k[j] + g);
#pragma unroll
                    for (int p = 0; p < 4; p++) q[s][p] += kj * a.P[j][p];
                }
            }
        }
    }
    for (int e = 0; e < a.n_emit; e++) {
        double x = a.x[e];
        double p1 = x, p2 = p1 * x, p3 = p2 * x, p4 = p3 * x;  // np.cumprod
        __syncthreads();
#pragma unroll
        for (int s = 0; s < DPER; s++) {
            int idx = threadIdx.x + s * NTHREADS;
            if (idx < DCELLS) {
                double d = q[s][0] * p1 + q[s][1] * p2 + q[s][2] * p3 + q[s][3] * p4;
                double ph = a.h * d + y0[s];
                int ly = idx / DSW, lx = idx - ly * DSW;
                int gy = ty0 + ly - 1, gx = tx0 + lx - 1;
                if (a.phi[e] && ly >= 1 && ly <= DTY && lx >= 1 && lx <= DTX && gy < Ny && gx < Nx)
                    a.phi[e][(size_t)gy * Nx + gx] = ph;
                tile[idx] = clamp_lim(ph, a.lim);
            }
        }
        __syncthreads();
        if (a.vx[e]) {
#pragma unroll
            for (int r = 0; r < (DTX * DTY) / NTHREADS; r++) {
                int cell = threadIdx.x + r * NTHREADS;
                int ly = cell / DTX, lx = cell - ly * DTX;
                int gy = ty0 + ly, gx = tx0 + lx;
                if (gy >= 1 && gy < Ny - 1 && gx >= 1 && gx < Nx - 1) {
                    const double *t = tile + (ly + 1) * DSW + (lx + 1);
                    double ox, oy;
                    vels_point(t[0], t[-1], t[1], t[-DSW], t[DSW], a.mu, a.lim, a.inv_two_dx, a.inv_two_dy, ox, oy);
                    size_t o = (size_t)(gy - 1) * (Nx - 2) + (gx - 1);
                    a.vx[e][o] = ox;
                    a.vy[e][o] = oy;
                }
            }
        }
    }
}

// standalone vels (optimals.py:168-186) for unit parity
__global__ void __launch_bounds__(NTHREADS)
vels_kernel(const double *__restrict__ phi, int Ny, int Nx, double mu, double lim, double inv_two_dx,
            double inv_two_dy, double *__restrict__ vx, double *__restrict__ vy) {
    int gx = blockIdx.x * 64 + (threadIdx.x & 63) + 1, gy = blockIdx.y * 4 + (threadIdx.x >> 6) + 1;
    if (gy >= Ny - 1 || gx >= Nx - 1) return;
    size_t g = (size_t)gy * Nx + gx;
    double ox, oy;
    vels_point(clamp_lim(phi[g], lim), clamp_lim(phi[g - 1], lim), clamp_lim(phi[g + 1], lim),
               clamp_lim(phi[g - Nx], lim), clamp_lim(phi[g + Nx], lim), mu, lim, inv_two_dx, inv_two_dy, ox, oy);
    size_t o = (size_t)(gy - 1) * (Nx - 2) + (gx - 1);
    vx[o] = ox;
    vy[o] = oy;
}

// ---------------------------------------------------------------------------------------------------
struct Solver {
    oc_ctx *ctx;
    cudaStream_t st;
    int Ny, Nx, nbx, nby;
    size_t n;
    double *y, *ynew, *K[7], *coef;
    double *partial, *rowsum_d, *rowsum_h;
    double diff_over_dxdy;
    int launches = 0;
    bool profile = false;
    struct Rec { int cls; double bytes; cudaEvent_t a, b; };
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> pool;
    size_t pool_used = 0;
    cudaEvent_t get_event() {
        if (pool_used == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
        return pool[pool_used++];
    }
    void begin(int cls, double bytes) {
        if (!profile) return;
        Rec r{cls, bytes, get_event(), get_event()};
        cudaEventRecord(r.a, st);
        recs.push_back(r);
    }
    void end() {
        if (!profile) return;
        cudaEventRecord(recs.back().b, st);
    }
    void collect(oc_hjb_stats *out) {
        for (auto &r : recs) {
            float ms = 0;
            cudaEventElapsedTime(&ms, r.a, r.b);
            out->cls_launches[r.cls]++;
            out->cls_ms[r.cls] += ms;
            out->cls_bytes[r.cls] += r.bytes;
        }
        for (auto e : pool) cudaEventDestroy(e);
        pool.clear(); recs.clear();
    }

    template <int N, int MODE>
    void launch_stage(const Comb &c, double *kout, double *yn, const ErrArgs &ea) {
        dim3 grid(nbx, nby);
        // algorithmic words per cell: y + N k's + coef in, k out (+ y_new out, K[0..5] re-used for the error)
        begin(0, 8.0 * (double)n * (MODE == 1 ? 9 : N + 3));
        hjb_stage_kernel<N, MODE><<<grid, NTHREADS, 0, st>>>(c, coef, kout, yn, ea, partial, Ny, Nx, diff_over_dxdy);
        end();
        launches++;
    }
    void stage(int N, const Comb &c, double *kout) {
        ErrArgs ea{};
        switch (N) {
            case 0: launch_stage<0, 0>(c, kout, nullptr, ea); break;
            case 1: launch_stage<1, 0>(c, kout, nullptr, ea); break;
            case 2: launch_stage<2, 0>(c, kout, nullptr, ea); break;
            case 3: launch_stage<3, 0>(c, kout, nullptr, ea); break;
            case 4: launch_stage<4, 0>(c, kout, nullptr, ea); break;
            case 5: launch_stage<5, 0>(c, kout, nullptr, ea); break;
        }
    }
    // ---- stage-fused step (oc_hjb_fused.cuh)
    int fused_rc = 0, fused_gx = 0, fused_gy = 0;
    void fused_plan(int n_sm, int forced_rc = 0) {
        fused_gx = (Nx + fused::VX - 1) / fused::VX;
        fused_rc = forced_rc > 0 ? forced_rc : fused::plan_chunk_rows(Nx, Ny, n_sm, 1, 0);
        fused_gy = (Ny + fused_rc - 1) / fused_rc;
    }
    fused::MapCache maps;  // TMA descriptors of this solve's arrays
    int launch_fused(int ne, fused::Args &a) {
        fused::set_tensor_maps(a, Ny, &maps);
        dim3 grid(fused_gx, fused_gy);
        begin(0, 8.0 * (double)n * (5 + ne));  // y, f, coef in; y_new, f_new, NE phi slices out
        OC_CUDA(fused::launch<false>(ne, a, grid, st));
        end();
        launches++;
        return OC_OK;
    }
    // sum over tile rows of per-tile partials located at partial+off; host-visible after sync
    int reduce_to_host(size_t off, double *out, int gx = -1, int gy = -1) {
        if (gx < 0) { gx = nbx; gy = nby; }
        begin(2, 8.0 * ((double)gx * gy + gy));
        rowgroup_sum_kernel<<<gy, NTHREADS, 0, st>>>(partial + off, gx, rowsum_d);
        end();
        launches++;
        OC_CUDA(cudaMemcpyAsync(rowsum_h, rowsum_d, sizeof(double) * gy, cudaMemcpyDeviceToHost, st));
        OC_CUDA(cudaStreamSynchronize(st));
        double s = 0.0;
        for (int i = 0; i < gy; i++) s += rowsum_h[i];  // fixed global order
        *out = s;
        return OC_OK;
    }
};

int ensure_ws(oc_ctx *ctx, size_t n, int nbx, int nby) {
    int rc = oc_ensure_buffer(ctx->hjb_ws, ctx->hjb_ws_bytes, 10 * n * sizeof(double), false, "HJB workspace");
    if (rc) return rc;
    // large enough for the stage tiles and for any fused-step plan (>= 32-row chunks, 240-column tiles)
    size_t np = (size_t)2 * nbx * nby + nby + 64;
    {
        size_t fgx = (size_t)(nbx * TX + fused::VX - 1) / fused::VX + 1, fgy = (size_t)(nby * TY + 15) / 16 + 1;
        np = std::max(np, 2 * fgx * fgy + fgy + 64);
    }
    if ((rc = oc_ensure_buffer(ctx->hjb_partial, ctx->hjb_partial_bytes, np * sizeof(double), false, "HJB partial sums")))
        return rc;
    size_t hp = (size_t)std::max(nby, (nby * TY + 15) / 16 + 1) + 16;
    return oc_ensure_buffer(ctx->h_pinned, ctx->h_pinned_bytes, hp * sizeof(double), true, "pinned host scratch");
}

int ensure_final_reduce(oc_ctx *ctx, int slots) { return ocfinal::ensure(ctx, slots); }
void final_reduce_args(oc_ctx *ctx, int slot, fused::Args &fa) { ocfinal::set_args(ctx, slot, ++ctx->fr_seq, fa); }
inline bool final_ready(oc_ctx *ctx, int slot, unsigned long long seq, double *out) { return ocfinal::ready(ctx, slot, seq, out); }
int wait_final(oc_ctx *ctx, int slot, unsigned long long seq, cudaStream_t st, double *out) {
    return ocfinal::wait(ctx, slot, seq, st, out);
}

}  // namespace

extern "C" int oc_hjb_rhs(oc_ctx *ctx, const double *d_phi, const double *d_V, const double *d_m,
                          const oc_hjb_params *prm, double *d_out, void *stream) {
    OC_ARG(ctx && d_phi && d_V && prm && d_out, "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    Solver s{};
    s.ctx = ctx; s.st = (cudaStream_t)stream; s.Ny = ctx->Ny; s.Nx = ctx->Nx;
    s.n = (size_t)s.Ny * s.Nx;
    s.nbx = (s.Nx + TX - 1) / TX; s.nby = (s.Ny + TY - 1) / TY;
    int rc = ensure_ws(ctx, s.n, s.nbx, s.nby);
    if (rc) return rc;
    s.coef = ctx->hjb_ws;
    s.partial = ctx->hjb_partial;
    double s2 = prm->sigma * prm->sigma;
    s.diff_over_dxdy = (-0.5 * s2) / (ctx->dx * ctx->dy);
    prep_kernel<<<(unsigned)((s.n + 255) / 256), 256, 0, s.st>>>(d_V, d_m, prm->g, 1.0 / (prm->mu * s2), s.n, s.coef, nullptr);
    Comb c{};
    c.y = d_phi;
    s.stage(0, c, d_out);
    oc::count_launch(2);
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}

// rows per CTA chunk the stage-fused kernel would choose for `copies` independent solves of this context's grid running
// side by side (ensembles).  A caller that wants member results independent of the batch size fixes prm->chunk_rows
// to this value for the stand-alone solve too (the chunking defines the order of the error-norm sum).
extern "C" int oc_hjb_plan_chunk_rows(oc_ctx *ctx, int copies) {
    if (!ctx || copies < 1) return OC_ERR_ARG;
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device);
    return fused::plan_chunk_rows(ctx->Nx, ctx->Ny, n_sm, copies, 0);
}

extern "C" int oc_hjb_vels(oc_ctx *ctx, const double *d_phi, const oc_hjb_params *prm, double *d_vx, double *d_vy,
                           void *stream) {
    OC_ARG(ctx && d_phi && prm && d_vx && d_vy, "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    dim3 grid((ctx->Nx - 2 + 63) / 64, (ctx->Ny - 2 + 3) / 4);
    vels_kernel<<<grid, NTHREADS, 0, (cudaStream_t)stream>>>(d_phi, ctx->Ny, ctx->Nx, prm->mu, prm->lim,
                                                             1.0 / (2 * ctx->dx), 1.0 / (2 * ctx->dy), d_vx, d_vy);
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}

extern "C" int oc_hjb_solve(oc_ctx *ctx, const double *d_V, const double *d_m, const oc_hjb_params *prm, double T,
                            const double *t_eval, int nt, double *d_phi, double *d_vx, double *d_vy,
                            oc_hjb_stats *stats, double *trace_h, double *trace_err, int trace_cap, int *trace_n,
                            void *stream) {
    OC_ARG(ctx && d_V && prm && stats, "NULL argument");
    OC_ARG(nt >= 1 && t_eval, "t_eval required");
    OC_CUDA(cudaSetDevice(ctx->device));
    Solver s{};
    s.ctx = ctx; s.st = (cudaStream_t)stream; s.Ny = ctx->Ny; s.Nx = ctx->Nx;
    const size_t n = s.n = (size_t)s.Ny * s.Nx;
    s.nbx = (s.Nx + TX - 1) / TX; s.nby = (s.Ny + TY - 1) / TY;
    int rc = ensure_ws(ctx, n, s.nbx, s.nby);
    if (rc) return rc;
    double *ws = ctx->hjb_ws;
    s.coef = ws; s.y = ws + n; s.ynew = ws + 2 * n;
    for (int j = 0; j < 7; j++) s.K[j] = ws + (3 + j) * n;
    s.partial = ctx->hjb_partial;
    s.rowsum_d = ctx->hjb_partial + (size_t)2 * s.nbx * s.nby;
    s.rowsum_h = ctx->h_pinned;
    const double s2 = prm->sigma * prm->sigma;
    s.diff_over_dxdy = (-0.5 * s2) / (ctx->dx * ctx->dy);
    const double rtol = prm->rtol, atol = prm->atol;
    const double sqrt_n = std::sqrt((double)n);
    memset(stats, 0, sizeof(*stats));
    s.profile = prm->profile != 0;
    OC_CUDA(cudaEventRecord(ctx->ev0, s.st));

    prep_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s.st>>>(d_V, d_m, prm->g, 1.0 / (prm->mu * s2), n, s.coef, s.y);
    s.launches++;
    rk45::Controller ctl(T, t_eval, nt);
    // rk.py:94: f = fun(t0, y0)
    {
        Comb c{};
        c.y = s.y;
        s.stage(0, c, s.K[0]);
        stats->nfev++;
    }
    // common.py:109-134 select_initial_step
    if (ctl.needs_initial_step()) {
        dim3 grid(s.nbx, s.nby);
        init_norm_kernel<<<grid, NTHREADS, 0, s.st>>>(s.y, s.K[0], nullptr, rtol, atol, s.Ny, s.Nx, s.partial, 0);
        s.launches++;
        double s0, s1, sq2;
        if ((rc = s.reduce_to_host(0, &s0))) return rc;
        if ((rc = s.reduce_to_host((size_t)s.nbx * s.nby, &s1))) return rc;
        const double d1 = std::sqrt(s1) / sqrt_n;
        const double h0 = ctl.initial_h0(std::sqrt(s0) / sqrt_n, d1);
        Comb c{};
        c.y = s.y; c.k[0] = s.K[0]; c.a[0] = 1.0; c.h = h0 * ctl.direction;  // y1 = y0 + h0*direction*f0
        s.stage(1, c, s.K[1]);
        stats->nfev++;
        init_norm_kernel<<<grid, NTHREADS, 0, s.st>>>(s.y, s.K[0], s.K[1], rtol, atol, s.Ny, s.Nx, s.partial, 1);
        s.launches++;
        if ((rc = s.reduce_to_host(0, &sq2))) return rc;
        ctl.set_initial_step(h0, d1, std::sqrt(sq2) / sqrt_n / h0);
    }
    stats->h0 = ctl.h_abs;

    // stage-fused path (prm->fused): needs room for NE_MAX phi slices when only velocities are requested
    // the fused kernel mirrors up to 6 rows / 8 columns across the boundary: tiny grids take the stage-wise path
    bool use_fused = prm->fused != 0 && s.Ny > fused::HY + 1 && s.Nx > fused::HX + 1, fused_attempt = false;
    double *phi_scratch = nullptr;
    if (use_fused) {
        int n_sm = 148;
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device);
        s.fused_plan(n_sm, prm->chunk_rows);
        size_t np_need = (size_t)2 * s.fused_gx * s.fused_gy + s.fused_gy;
        if (ctx->hjb_partial_bytes < np_need * sizeof(double) || ctx->h_pinned_bytes < ((size_t)s.fused_gy + 16) * sizeof(double)) {
            oc::set_error("internal: fused partial buffers too small");
            return OC_ERR_ARG;
        }
        if (!d_phi && d_vx && d_vy) {
            size_t need = (size_t)fused::NE_MAX * n * sizeof(double);
            if ((rc = oc_ensure_buffer(ctx->hjb_scratch, ctx->hjb_scratch_bytes, need, false, "phi scratch"))) return rc;
            phi_scratch = ctx->hjb_scratch;
        }
    }
    const size_t n_int = (size_t)(s.Ny - 2) * (s.Nx - 2);
    const bool final_in_kernel = use_fused && s.fused_gy <= fused::MAX_FINAL_ROWS;
    if (final_in_kernel && (rc = ensure_final_reduce(ctx, 1))) return rc;
    const bool want_out = d_phi || (d_vx && d_vy);

    while (ctl.begin_step()) {
        bool accepted = false;
        while (!accepted && ctl.propose(prm->forced_h, prm->n_forced_h)) {  // forced_h: teacher-forced (tests)
            const double h = ctl.h;
            // more than NE_MAX samples: with a phi output the step is launched again for the remaining samples (as the
            // batched and row-band solves do, so their results stay bit-identical); the NE_MAX scratch slices of a
            // velocity-only solve cannot hold them, that attempt takes the stage-wise path
            fused_attempt = use_fused && (!want_out || d_phi || ctl.n_emit() <= fused::NE_MAX);
            double se;
            if (fused_attempt) {
                // one launch per NE_MAX samples: 6 RHS evaluations, y_new, f_new, error partial sums and the
                // (speculative) dense output samples; a rejected attempt's samples are overwritten by the step that
                // finally covers them.  A repeated launch recomputes identical y_new / f_new / error sums.
                fused::Args fa{};
                fa.y = s.y; fa.k1 = s.K[0]; fa.coef = s.coef; fa.ynew = s.ynew; fa.k7 = s.K[6]; fa.partial = s.partial;
                fa.A = s.diff_over_dxdy; fa.rtol = rtol; fa.atol = atol;
                fa.Ny = s.Ny; fa.Nx = s.Nx; fa.RC = s.fused_rc;
                fa.row_base = 0; fa.own0 = 0; fa.own1 = s.Ny; fa.phi_row_base = 0;
                const int n_emit = want_out ? ctl.n_emit() : 0;
                int e0 = 0;
                do {
                    const int ne = std::min(n_emit - e0, fused::NE_MAX);
                    fused::set_attempt(fa, ctl, e0, ne, d_phi, phi_scratch, n);
                    // every launch finishes its own reduction (one ticket round, one sequence number); the same stream
                    // orders them, the host waits for the last one's
                    if (final_in_kernel) final_reduce_args(ctx, 0, fa);
                    if ((rc = s.launch_fused(ne, fa))) return rc;
                    e0 += ne;
                } while (e0 < n_emit);
                stats->nfev += 6;
                if (final_in_kernel) {
                    if ((rc = wait_final(ctx, 0, fa.seq, s.st, &se))) return rc;
                } else if ((rc = s.reduce_to_host(0, &se, s.fused_gx, s.fused_gy))) return rc;
            } else {
            // rk_step (rk.py:61-69): K[0] = f already in place
            for (int sgi = 1; sgi < 6; sgi++) {
                Comb c{};
                c.y = s.y; c.h = h;
                for (int j = 0; j < sgi; j++) { c.k[j] = s.K[j]; c.a[j] = rk45::A[sgi][j]; }
                s.stage(sgi, c, s.K[sgi]);
            }
            {
                // y_new = y + h*dot(K[:-1].T,B) with B[1]=0 dropped; K[6] = f(y_new); error partials
                Comb c{};
                c.y = s.y; c.h = h;
                int m = 0;
                for (int j = 0; j < 6; j++)
                    if (j != 1) { c.k[m] = s.K[j]; c.a[m] = rk45::B[j]; m++; }
                ErrArgs ea{};
                for (int j = 0; j < 6; j++) ea.k[j] = s.K[j];
                for (int j = 0; j < 7; j++) ea.e[j] = rk45::E[j];
                ea.h = h; ea.rtol = rtol; ea.atol = atol;
                s.launch_stage<5, 1>(c, s.K[6], s.ynew, ea);
            }
            stats->nfev += 6;
            if ((rc = s.reduce_to_host(0, &se))) return rc;
            }
            const double error_norm = std::sqrt(se) / sqrt_n;  // rk.py:147, common.py:63-65
            const int ntr = ctl.attempts();
            if (trace_h && ntr < trace_cap) { trace_h[ntr] = h; trace_err[ntr] = error_norm; }
            accepted = ctl.judge(error_norm);
        }
        if (!accepted) break;  // step too small

        if (fused_attempt) {
            // samples were written by the step kernel; only the gradient-to-velocity conversion is left
            for (int e = 0; e < ctl.n_emit(); e++) {
                const int kd = ctl.sample_column(e);
                if (d_vx && d_vy && kd >= 1) {
                    const double *ph = fused::sample_slice(ctl, e, d_phi, phi_scratch, n);
                    const int sl = nt - 1 - kd;
                    dim3 grid((s.Nx - 2 + 63) / 64, (s.Ny - 2 + 3) / 4);
                    s.begin(1, 8.0 * (double)n * 3);
                    vels_kernel<<<grid, NTHREADS, 0, s.st>>>(ph, s.Ny, s.Nx, prm->mu, prm->lim, 1.0 / (2 * ctx->dx), 1.0 / (2 * ctx->dy),
                                                             d_vx + (size_t)sl * n_int, d_vy + (size_t)sl * n_int);
                    s.end();
                    s.launches++;
                }
            }
        } else {
            int e = 0;
            while (e < ctl.n_emit()) {
                DenseArgs a{};
                a.yold = s.y;
                for (int j = 0; j < 7; j++) { a.k[j] = s.K[j]; for (int p = 0; p < 4; p++) a.P[j][p] = rk45::P[j][p]; }
                a.h = ctl.h; a.mu = prm->mu; a.lim = prm->lim; a.inv_two_dx = 1.0 / (2 * ctx->dx); a.inv_two_dy = 1.0 / (2 * ctx->dy);
                int m = 0;
                bool any = false;
                for (; m < DMAX && e < ctl.n_emit(); e++) {
                    int kd = ctl.sample_column(e);  // column of sol.y
                    a.x[m] = ctl.sample_x(e);
                    a.phi[m] = d_phi ? d_phi + (size_t)kd * n : nullptr;
                    int sl = nt - 1 - kd;  // vx_opt slice (optimals.py:200-204); column 0 (phi_T) has none
                    bool has_v = d_vx && d_vy && kd >= 1;
                    a.vx[m] = has_v ? d_vx + (size_t)sl * n_int : nullptr;
                    a.vy[m] = has_v ? d_vy + (size_t)sl * n_int : nullptr;
                    if (a.phi[m] || a.vx[m]) { any = true; m++; }
                }
                a.n_emit = m;
                if (any) {
                    dim3 grid((s.Nx + DTX - 1) / DTX, (s.Ny + DTY - 1) / DTY);
                    double words = 7.0;  // y_old + K[0], K[2..6]
                    for (int q = 0; q < m; q++) words += (a.phi[q] ? 1.0 : 0.0) + (a.vx[q] ? 2.0 : 0.0);
                    s.begin(1, 8.0 * (double)n * words);
                    hjb_dense_kernel<<<grid, NTHREADS, 0, s.st>>>(a, s.Ny, s.Nx);
                    s.end();
                    s.launches++;
                }
            }
        }
        // accept (rk.py:167-174): y <- y_new, f <- f_new (FSAL: pointer swaps)
        ctl.accept();
        std::swap(s.y, s.ynew);
        std::swap(s.K[0], s.K[6]);
    }
    OC_CUDA(cudaEventRecord(ctx->ev1, s.st));
    OC_CUDA(cudaStreamSynchronize(s.st));
    OC_CUDA(cudaGetLastError());
    float ms = 0;
    OC_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    stats->gpu_ms = ms;
    s.collect(stats);
    ctl.report(stats);
    stats->launches = s.launches;
    oc::count_launch(s.launches);
    if (trace_n) *trace_n = ctl.attempts();
    if (ctl.status == -1) {
        oc::set_error("RK45: required step size is less than spacing between numbers (t=%g)", ctl.t);
        return OC_ERR_STEP_TOO_SMALL;
    }
    return OC_OK;
}

// ---------------------------------------------------------------------------------------------------
// Batched solve for ensembles of independent rooms (BASELINE configs[4], SURVEY 8e).
// Every room keeps its own RK45 controller (t, h, accept/reject, t_eval cursor: the reference integrates each
// room separately, optimals.py:193-196) and its own CUDA stream; a room's step attempt is one launch of the
// stage-fused kernel per 6 samples followed by the fixed-order reduction, exactly the launches oc_hjb_solve issues, so
// every room's result is bit-identical to solving it alone (with the same chunk_rows).  The host serves the rooms
// round-robin: while it reads room b's error norm and enqueues b's next attempt, the other rooms' kernels keep
// the GPU busy -- small grids (512^2: ~10 us of device work per attempt) are launch-latency bound one at a time.
// oc_hjb_solve_grids is the one implementation: every room brings its own grid (shape and spacing: every size, tile
// grid, workspace offset and norm below is the room's), its own sigma, mu, g (prep_kernel's coefficients, the diffusion
// constant of the step kernel, vels_kernel's mu -- all kernel arguments already) and its own horizon (its controller);
// oc_hjb_solve_multi gives every room the context's grid, oc_hjb_solve_batch also the same parameters.
namespace {

struct BatchRoom {
    Solver s;
    enum Phase { START, INIT0, INIT1, STEP, DONE } phase = START;
    const double *V = nullptr, *m = nullptr;
    double *phi = nullptr, *scratch = nullptr, *vx = nullptr, *vy = nullptr;  // scratch: NE_MAX slices, without phi
    double *rs_d = nullptr, *rs_h = nullptr;  // row-group sums (device / pinned host), 3 regions of `rs_stride`
    int rs_stride = 0;
    size_t n_int = 0;                    // interior cells: one vx / vy slice
    double sqrt_n = 0, dx = 0, dy = 0;   // the room's grid
    bool final_in_kernel = false;        // its fused step finishes the error sum in the launch (fused_gy small enough)
    cudaEvent_t ev = nullptr;
    unsigned long long wait_seq = 0;     // sequence number of the step attempt in flight (in-kernel final reduction)
    rk45::Controller ctl;                // the room's horizon: T, t_eval, nt
    double g = 0, inv_mu_s2 = 0, mu = 0; // prep_kernel's coefficients, vels_kernel's mu (s.diff_over_dxdy: its sigma)
    double h0 = 0, d1 = 0;               // select_initial_step between its two norm reductions
    double step_sum = 0.0;               // error sum delivered by the last CTA of the attempt
    fused::Args fa{};                    // the attempt waiting in a bucket for its batched launch
    oc_hjb_stats st{};
};

}  // namespace

extern "C" int oc_hjb_solve_batch(oc_ctx *ctx, int n_rooms, const double *const *d_V, const double *const *d_m,
                                  const oc_hjb_params *prm, double T, const double *t_eval, int nt,
                                  double *const *d_phi, double *const *d_vx, double *const *d_vy,
                                  oc_hjb_stats *stats, void *stream) {
    OC_ARG(prm && n_rooms >= 1, "NULL argument");
    std::vector<oc_hjb_room> same(n_rooms, oc_hjb_room{prm->sigma, prm->mu, prm->g, T, t_eval, nt, 0});
    return oc_hjb_solve_multi(ctx, n_rooms, d_V, d_m, same.data(), prm, d_phi, d_vx, d_vy, stats, stream);
}

extern "C" int oc_hjb_solve_multi(oc_ctx *ctx, int n_rooms, const double *const *d_V, const double *const *d_m,
                                  const oc_hjb_room *spec, const oc_hjb_params *prm, double *const *d_phi,
                                  double *const *d_vx, double *const *d_vy, oc_hjb_stats *stats, void *stream) {
    OC_ARG(ctx && prm && n_rooms >= 1, "NULL argument");
    std::vector<oc_ctx *> grids(n_rooms, ctx);
    oc_hjb_params p = *prm;
    if (p.chunk_rows < 0) p.chunk_rows = 0;  // as oc_hjb_solve: a negative chunk_rows means the grid's own plan
    return oc_hjb_solve_grids(ctx, n_rooms, grids.data(), d_V, d_m, spec, &p, d_phi, d_vx, d_vy, stats, stream);
}

extern "C" int oc_hjb_solve_grids(oc_ctx *ctx, int n_rooms, oc_ctx *const *grids, const double *const *d_V,
                                  const double *const *d_m, const oc_hjb_room *spec, const oc_hjb_params *prm,
                                  double *const *d_phi, double *const *d_vx, double *const *d_vy, oc_hjb_stats *stats,
                                  void *stream) {
    OC_ARG(ctx && d_V && prm && stats && n_rooms >= 1, "NULL argument");
    OC_ARG(grids, "grids (one context per room) required");
    OC_ARG(spec, "rooms (per-room parameters and horizons) required");
    OC_ARG(prm->chunk_rows >= 0, "chunk_rows must not be negative");
    for (int b = 0; b < n_rooms; b++) {
        const oc_hjb_room &p = spec[b];
        OC_ARG(p.nt >= 1 && p.t_eval, "t_eval required");
        OC_ARG(std::isfinite(p.sigma) && p.sigma > 0, "sigma must be a finite positive number");
        OC_ARG(std::isfinite(p.mu) && p.mu > 0, "mu must be a finite positive number");
        OC_ARG(std::isfinite(p.g), "g must be finite");
        OC_ARG(p.chunk_rows >= 0, "a room's chunk_rows must not be negative");
        OC_ARG(grids[b], "NULL grid");
        OC_ARG(grids[b]->device == ctx->device, "a room's grid lives on another device than ctx");
        OC_ARG(grids[b]->Ny > fused::HY + 1 && grids[b]->Nx > fused::HX + 1, "grid too small for the stage-fused kernel");
    }
    OC_ARG(d_phi || (d_vx && d_vy), "an output (d_phi or d_vx,d_vy) is required");
    OC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t main_st = (cudaStream_t)stream;
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device);
    // per room: coef, y, y_new, f, f_new (+ NE_MAX phi slices when only velocities are kept) ; partial sums ; row sums
    const bool need_scratch = !d_phi;
    const bool want_v = d_vx && d_vy;
    std::vector<BatchRoom> rooms(n_rooms);
    std::vector<size_t> ws_off(n_rooms + 1, 0);
    std::vector<size_t> pin_off(n_rooms + 1, 0), np_room(n_rooms);
    bool any_final = false;
    for (int b = 0; b < n_rooms; b++) {
        const oc_ctx *gr = grids[b];
        BatchRoom &r = rooms[b];
        Solver &s = r.s;
        // the expressions of oc_hjb_solve, with the room's grid
        s.Ny = gr->Ny; s.Nx = gr->Nx;
        s.n = (size_t)s.Ny * s.Nx;
        r.n_int = (size_t)(s.Ny - 2) * (s.Nx - 2);
        s.nbx = (s.Nx + TX - 1) / TX; s.nby = (s.Ny + TY - 1) / TY;
        const int rc_rows = spec[b].chunk_rows > 0 ? spec[b].chunk_rows : prm->chunk_rows;
        s.fused_plan(n_sm, rc_rows);
        r.dx = gr->dx; r.dy = gr->dy;
        r.sqrt_n = std::sqrt((double)s.n);
        r.final_in_kernel = s.fused_gy <= fused::MAX_FINAL_ROWS;
        any_final = any_final || r.final_in_kernel;
        // (even numbers of doubles: every room's arrays stay 16-byte aligned for the TMA descriptors)
        const size_t np = np_room[b] = ((std::max((size_t)2 * s.nbx * s.nby, (size_t)s.fused_gx * s.fused_gy) + 8) + 1) & ~(size_t)1;
        r.rs_stride = ((std::max(s.nby, s.fused_gy) + 8) + 1) & ~1;
        const size_t per_room = (5 + (need_scratch ? fused::NE_MAX : 0)) * s.n + np + 3 * (size_t)r.rs_stride;
        ws_off[b + 1] = ws_off[b] + ((per_room + 1) & ~(size_t)1);
        pin_off[b + 1] = pin_off[b] + 3 * (size_t)r.rs_stride;
    }
    int rc = oc_ensure_buffer(ctx->batch_ws, ctx->batch_ws_bytes, ws_off[n_rooms] * sizeof(double), false,
                              "batched HJB workspace");
    if (rc) return rc;
    if ((rc = oc_ensure_buffer(ctx->batch_pinned, ctx->batch_pinned_bytes, pin_off[n_rooms] * sizeof(double), true,
                               "batched HJB host sums")))
        return rc;
    constexpr int MAX_STREAMS = 32;
    const int n_streams = std::min(n_rooms, MAX_STREAMS);
    while ((int)ctx->batch_streams.size() < n_streams) {
        cudaStream_t s;
        OC_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        ctx->batch_streams.push_back(s);
    }
    while ((int)ctx->batch_events.size() < n_rooms + 1) {
        cudaEvent_t e;
        OC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->batch_events.push_back(e);
    }
    // inputs produced on the caller's stream are visible to the room streams
    OC_CUDA(cudaEventRecord(ctx->ev0, main_st));
    cudaEvent_t ev_in = ctx->batch_events[n_rooms];
    OC_CUDA(cudaEventRecord(ev_in, main_st));
    for (int q = 0; q < n_streams; q++) OC_CUDA(cudaStreamWaitEvent(ctx->batch_streams[q], ev_in, 0));

    const double rtol = prm->rtol, atol = prm->atol;
    if (any_final && (rc = ensure_final_reduce(ctx, n_rooms))) return rc;
    for (int b = 0; b < n_rooms; b++) {
        BatchRoom &r = rooms[b];
        OC_ARG(d_V[b] && (!d_phi || d_phi[b]) && (!want_v || (d_vx[b] && d_vy[b])), "NULL room pointer");
        double *ws = ctx->batch_ws + ws_off[b];
        Solver &s = r.s;
        const size_t n = s.n;
        s.ctx = ctx; s.st = ctx->batch_streams[b % n_streams];
        s.coef = ws; s.y = ws + n; s.ynew = ws + 2 * n; s.K[0] = ws + 3 * n; s.K[6] = ws + 4 * n;
        s.K[1] = s.K[6];  // f(y0 + h0 f0) of select_initial_step lives in the (still unused) f_new array
        s.partial = ws + (5 + (need_scratch ? fused::NE_MAX : 0)) * n;
        r.rs_d = s.partial + np_room[b];
        r.rs_h = ctx->batch_pinned + pin_off[b];
        const double s2 = spec[b].sigma * spec[b].sigma;   // the expressions of oc_hjb_solve, with the room's values
        s.diff_over_dxdy = (-0.5 * s2) / (r.dx * r.dy);
        r.g = spec[b].g; r.inv_mu_s2 = 1.0 / (spec[b].mu * s2); r.mu = spec[b].mu;
        r.V = d_V[b]; r.m = d_m ? d_m[b] : nullptr;
        r.phi = d_phi ? d_phi[b] : nullptr;
        r.scratch = need_scratch ? ws + 5 * n : nullptr;
        r.vx = want_v ? d_vx[b] : nullptr; r.vy = want_v ? d_vy[b] : nullptr;
        r.ev = ctx->batch_events[b];
        r.ctl = rk45::Controller(spec[b].T, spec[b].t_eval, spec[b].nt);
    }
    // room-local helpers ------------------------------------------------------------------------------
    auto reduce_async = [&](BatchRoom &r, size_t off, int gx, int gy, int slot) {
        rowgroup_sum_kernel<<<gy, NTHREADS, 0, r.s.st>>>(r.s.partial + off, gx, r.rs_d + (size_t)slot * r.rs_stride);
        r.s.launches++;
        cudaMemcpyAsync(r.rs_h + (size_t)slot * r.rs_stride, r.rs_d + (size_t)slot * r.rs_stride, sizeof(double) * gy,
                        cudaMemcpyDeviceToHost, r.s.st);
    };
    auto host_sum = [&](BatchRoom &r, int gy, int slot) {
        double s = 0.0;
        const double *p = r.rs_h + (size_t)slot * r.rs_stride;
        for (int i = 0; i < gy; i++) s += p[i];  // fixed global order
        return s;
    };
    // Batched launches: the step attempts that become ready during one polling sweep are grouped by their number of
    // dense-output samples NE and their staging variant (TMA for even Nx, LDGSTS otherwise) and launched together, up to
    // fused::BATCH_MAX rooms of any grid shapes per launch (a flattened grid of all their CTAs; fewer when the launch's
    // CTA-to-room table cannot describe them, see fused::set_batch_table), instead of one launch per
    // room: 512^2 rooms need ~10 us of device work per attempt, less than a launch round trip.  Only with phi output
    // (velocity-only storage converts scratch slices on the room's own stream) and for rooms with the in-kernel final
    // reduction; a room's arithmetic is unchanged (same kernel body, same chunking, same reduction order).
    const bool batched = d_phi != nullptr && !getenv("OC_BATCH_PER_ROOM");
    std::vector<BatchRoom *> buckets[fused::NE_MAX + 1][2];
    std::vector<fused::BatchArgs> host_ba(1);
    int bucket_launches = 0;
    auto flush = [&]() -> int {
        for (int ne = 0; ne <= fused::NE_MAX; ne++) {
            for (int bulk = 0; bulk < 2; bulk++) {
                auto &bk = buckets[ne][bulk];
                for (size_t off = 0; off < bk.size();) {
                    int nb = (int)std::min<size_t>(fused::BATCH_MAX, bk.size() - off);
                    int ngx[fused::BATCH_MAX], ngy[fused::BATCH_MAX];
                    for (int q = 0; q < nb; q++) { ngx[q] = bk[off + q]->s.fused_gx; ngy[q] = bk[off + q]->s.fused_gy; }
                    int ctas;
                    while ((ctas = fused::set_batch_table(host_ba[0], nb, ngx, ngy)) == 0) nb--;
                    for (int q = 0; q < nb; q++) host_ba[0].a[q] = bk[off + q]->fa;
                    cudaStream_t st = ctx->batch_streams[(bucket_launches++) % n_streams];
                    OC_CUDA(fused::launch_batch(ne, bulk != 0, host_ba[0], ctas, st));
                    rooms[0].s.launches++;
                    off += nb;
                }
                bk.clear();
            }
        }
        return OC_OK;
    };
    // enqueue one step attempt of room r (fused kernel + reduction); the room is DONE when its step became too small
    auto attempt = [&](BatchRoom &r) -> int {
        rk45::Controller &c = r.ctl;
        if (!c.propose()) { r.phase = BatchRoom::DONE; return OC_OK; }
        fused::Args fa{};
        Solver &s = r.s;
        fa.y = s.y; fa.k1 = s.K[0]; fa.coef = s.coef; fa.ynew = s.ynew; fa.k7 = s.K[6]; fa.partial = s.partial;
        fa.A = s.diff_over_dxdy; fa.rtol = rtol; fa.atol = atol;
        fa.Ny = s.Ny; fa.Nx = s.Nx; fa.RC = s.fused_rc;
        fa.row_base = 0; fa.own0 = 0; fa.own1 = s.Ny; fa.phi_row_base = 0;
        // the samples this attempt emits if accepted, NE_MAX per launch; with more than NE_MAX samples inside one
        // step (only when h >> dt) the step is simply launched again for the remaining samples: the re-launch
        // recomputes identical y_new / f_new / error sums
        if (!d_phi && c.n_emit() > fused::NE_MAX) {
            oc::set_error("batched solve without a phi output supports at most %d samples per step", fused::NE_MAX);
            return OC_ERR_ARG;
        }
        // an attempt waits in a bucket only when ALL its samples fit one launch.  The launches of a longer attempt
        // share the room's ticket counter and result slot, so they must not overlap: they go out in order on the
        // room's own stream (the sequence OC_BATCH_PER_ROOM gives every attempt).
        const bool to_bucket = batched && r.final_in_kernel && c.n_emit() <= fused::NE_MAX;
        int e0 = 0;
        do {
            const int ne = std::min(c.n_emit() - e0, fused::NE_MAX);
            // without a phi output the samples go to the room's scratch slices (velocities are derived on accept)
            fused::set_attempt(fa, c, e0, ne, r.phi, r.scratch, s.n);
            if (r.final_in_kernel) { final_reduce_args(ctx, (int)(&r - rooms.data()), fa); r.wait_seq = fa.seq; }
            if (to_bucket) {
                fused::set_tensor_maps(fa, s.Ny, &s.maps);
                r.fa = fa;
                buckets[ne][fused::bulk_ok(fa) ? 1 : 0].push_back(&r);
                break;
            }
            int rc = s.launch_fused(ne, fa);
            if (rc) return rc;
            e0 += ne;
        } while (e0 < c.n_emit());
        r.st.nfev += 6;
        if (!r.final_in_kernel) {
            reduce_async(r, 0, s.fused_gx, s.fused_gy, 0);
            cudaEventRecord(r.ev, s.st);
        }
        r.phase = BatchRoom::STEP;
        return OC_OK;
    };
    auto start_step = [&](BatchRoom &r) -> int {  // base.py:179-210 step(): one call of _step_impl
        if (!r.ctl.begin_step()) { r.phase = BatchRoom::DONE; return OC_OK; }
        return attempt(r);
    };
    auto advance = [&](BatchRoom &r) -> int {
        Solver &s = r.s;
        const size_t n = s.n;
        const int Ny = s.Ny, Nx = s.Nx, nbx = s.nbx, nby = s.nby;
        switch (r.phase) {
        case BatchRoom::START: {
            prep_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s.st>>>(r.V, r.m, r.g, r.inv_mu_s2, n, s.coef, s.y);
            s.launches++;
            Comb c{};
            c.y = s.y;
            s.stage(0, c, s.K[0]);  // rk.py:94
            r.st.nfev++;
            if (!r.ctl.needs_initial_step()) { r.st.h0 = 0.0; return start_step(r); }
            init_norm_kernel<<<dim3(nbx, nby), NTHREADS, 0, s.st>>>(s.y, s.K[0], nullptr, rtol, atol, Ny, Nx, s.partial, 0);
            s.launches++;
            reduce_async(r, 0, nbx, nby, 0);
            reduce_async(r, (size_t)nbx * nby, nbx, nby, 1);
            cudaEventRecord(r.ev, s.st);
            r.phase = BatchRoom::INIT0;
            return OC_OK;
        }
        case BatchRoom::INIT0: {  // common.py:109-127
            r.d1 = std::sqrt(host_sum(r, nby, 1)) / r.sqrt_n;
            r.h0 = r.ctl.initial_h0(std::sqrt(host_sum(r, nby, 0)) / r.sqrt_n, r.d1);
            Comb c{};
            c.y = s.y; c.k[0] = s.K[0]; c.a[0] = 1.0; c.h = r.h0 * r.ctl.direction;
            s.stage(1, c, s.K[1]);
            r.st.nfev++;
            init_norm_kernel<<<dim3(nbx, nby), NTHREADS, 0, s.st>>>(s.y, s.K[0], s.K[1], rtol, atol, Ny, Nx, s.partial, 1);
            s.launches++;
            reduce_async(r, 0, nbx, nby, 2);
            cudaEventRecord(r.ev, s.st);
            r.phase = BatchRoom::INIT1;
            return OC_OK;
        }
        case BatchRoom::INIT1: {  // common.py:127-134
            r.ctl.set_initial_step(r.h0, r.d1, std::sqrt(host_sum(r, nby, 2)) / r.sqrt_n / r.h0);
            r.st.h0 = r.ctl.h_abs;
            return start_step(r);
        }
        case BatchRoom::STEP: {  // rk.py:146-165
            const double error_norm = std::sqrt(r.final_in_kernel ? r.step_sum : host_sum(r, s.fused_gy, 0)) / r.sqrt_n;
            rk45::Controller &c = r.ctl;
            if (!c.judge(error_norm)) return attempt(r);
            for (int e = 0; e < c.n_emit(); e++) {
                const int kd = c.sample_column(e);
                if (want_v && kd >= 1) {  // slice s = vels(sol.y[:, nt-1-s]) (optimals.py:200-204)
                    const double *ph = fused::sample_slice(c, e, r.phi, r.scratch, n);
                    const int sl = c.nt - 1 - kd;
                    dim3 grid((Nx - 2 + 63) / 64, (Ny - 2 + 3) / 4);
                    vels_kernel<<<grid, NTHREADS, 0, s.st>>>(ph, Ny, Nx, r.mu, prm->lim, 1.0 / (2 * r.dx), 1.0 / (2 * r.dy),
                                                             r.vx + (size_t)sl * r.n_int, r.vy + (size_t)sl * r.n_int);
                    s.launches++;
                }
            }
            c.accept();
            std::swap(s.y, s.ynew);
            std::swap(s.K[0], s.K[6]);
            return start_step(r);
        }
        default: return OC_OK;
        }
    };
    int live = n_rooms;
    for (int b = 0; b < n_rooms && !rc; b++) {
        rc = advance(rooms[b]);
        if (rooms[b].phase == BatchRoom::DONE) live--;
    }
    if (!rc) rc = flush();
    unsigned long long idle = 0;
    while (live > 0 && !rc) {
        bool progressed = false;
        for (int b = 0; b < n_rooms && !rc; b++) {
            BatchRoom &r = rooms[b];
            if (r.phase == BatchRoom::DONE) continue;
            if (r.final_in_kernel && r.phase == BatchRoom::STEP) {
                // the attempt's last CTA publishes the error sum in mapped host memory: no event, no copy
                if (!final_ready(ctx, b, r.wait_seq, &r.step_sum)) continue;
            } else {
                cudaError_t e = cudaEventQuery(r.ev);
                if (e == cudaErrorNotReady) continue;
                OC_CUDA(e);
            }
            progressed = true;
            rc = advance(r);
            if (r.phase == BatchRoom::DONE) live--;
        }
        if (!rc) rc = flush();  // one batched launch per NE class for everything that became ready in this sweep
        if (progressed) { idle = 0; continue; }
        if ((++idle & 0x3ffff) == 0) {  // nothing became ready for a long time: make sure no launch has failed
            bool all_idle = true;
            for (int q = 0; q < n_streams && !rc; q++) {
                cudaError_t e = cudaStreamQuery(ctx->batch_streams[q]);
                if (e == cudaErrorNotReady) all_idle = false;
                else if (e != cudaSuccess) {
                    oc::set_error("batched HJB solve: %s", cudaGetErrorString(e));
                    cudaGetLastError();
                    rc = OC_ERR_CUDA;
                }
            }
            // every stream has drained, so every launched attempt has published its error sum (ocfinal::wait): a room
            // still waiting after one more look never gets one -- an error instead of a host that spins for ever
            for (int b = 0; b < n_rooms && !rc && all_idle; b++) {
                BatchRoom &r = rooms[b];
                if (r.final_in_kernel && r.phase == BatchRoom::STEP && !final_ready(ctx, b, r.wait_seq, &r.step_sum)) {
                    oc::set_error("batched HJB solve: room %d: fused RK45 step did not deliver its error sum", b);
                    rc = OC_ERR_CUDA;
                }
            }
        }
    }
    // the caller's stream continues after every room stream
    for (int q = 0; q < n_streams; q++) {
        cudaEventRecord(ctx->batch_events[q], ctx->batch_streams[q]);
        cudaStreamWaitEvent(main_st, ctx->batch_events[q], 0);
    }
    OC_CUDA(cudaEventRecord(ctx->ev1, main_st));
    OC_CUDA(cudaStreamSynchronize(main_st));
    OC_CUDA(cudaGetLastError());
    if (rc) return rc;
    float ms = 0;
    OC_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    int bad = -1, total_launches = 0;
    for (int b = 0; b < n_rooms; b++) {
        BatchRoom &r = rooms[b];
        r.ctl.report(&r.st);
        r.st.launches = r.s.launches; r.st.gpu_ms = ms;
        total_launches += r.s.launches;
        stats[b] = r.st;
        if (r.ctl.status == -1 && bad < 0) bad = b;
    }
    oc::count_launch(total_launches);
    if (bad >= 0) {
        oc::set_error("RK45: required step size is less than spacing between numbers (room %d, t=%g)", bad, rooms[bad].ctl.t);
        return OC_ERR_STEP_TOO_SMALL;
    }
    return OC_OK;
}
