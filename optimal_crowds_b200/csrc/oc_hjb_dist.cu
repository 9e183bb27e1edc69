// oc_hjb_dist.cu -- row-decomposed HJB solve (SURVEY.md section 8e): the grid is split into bands of rows,
// one band per GPU (one process per GPU, NCCL over NVLink) or, for tests on one GPU, several "virtual" bands in
// one process.  Every band runs the stage-fused RK45 step kernel (oc_hjb_fused.cuh) on its rows.  After each
// attempt ONE ncclGroup carries (a) the all-gather of the per-chunk error partial sums, which every rank adds
// in global chunk order, so each rank takes the same accept/reject decision and -- with prm.chunk_rows fixed --
// the result is bit-identical to the undecomposed solve, and (b) speculatively, the 6 boundary rows of y_new and
// f_new for the neighbouring bands (if the attempt is rejected they are never used), so that an accepted step
// needs no further communication before the next attempt can be launched.
//
// Exchange traffic per accepted step and neighbour: 2 arrays x 6 rows x Nx x 8 B (1.5 MB at Nx = 16384) plus
// one row per emitted phi slice when velocities are requested; all messages of a step go out in ONE
// ncclGroup on the compute stream.  The scalar reduction is one ncclAllGather of (chunks per band) doubles.
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "oc_common.h"
#include "oc_hjb_fused.cuh"
#include "oc_hjb_final.h"
#include "oc_rk45.h"
#include "oc_vels.h"

namespace {

// ---- minimal NCCL binding, resolved at run time from the libnccl torch has already loaded ---------------
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { ncclFloat64 = 8, ncclUint64 = 5, ncclMax = 2 };
struct Nccl {
    void *h = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Send)(const void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load() {
        if (h) return true;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (!h) return false;
#define SYM(f) *(void **)(&f) = dlsym(h, "nccl" #f); if (!f) return false;
        SYM(GetUniqueId) SYM(CommInitRank) SYM(CommDestroy) SYM(GroupStart) SYM(GroupEnd) SYM(Send) SYM(Recv)
        SYM(AllGather) SYM(AllReduce) SYM(GetErrorString)
#undef SYM
        return true;
    }
} g_nccl;

#define OC_NCCL(expr)                                                                                   \
    do {                                                                                                \
        int _r = (expr);                                                                                \
        if (_r != 0) {                                                                                  \
            oc::set_error("%s failed: %s", #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "?"); \
            return OC_ERR_NCCL;                                                                         \
        }                                                                                               \
    } while (0)

constexpr int HB = fused::HY;  // halo rows exchanged per side
constexpr int NT = 256;
constexpr int TXS = 128, TYS = 16;  // tiles of the (rarely used) single-stage kernels, same as oc_hjb.cu

__device__ __forceinline__ int mirror_idx(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * (n - 1) - i : i); }

struct BandView {
    int Ny, Nx;          // global grid
    int row_base;        // global row of storage row 0
    int own0, own1;      // rows owned
};

// coef = (V<0) ? NaN : (V + g*m)/(mu sigma^2) on the owned rows; y = 1 on every storage row (phi_T, optimals.py:83)
__global__ void prep_band_kernel(const double *__restrict__ V, const double *__restrict__ m, int io_row0, double g,
                                 double inv_den, BandView b, int rows_store, double *__restrict__ coef,
                                 double *__restrict__ y) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t n = (size_t)rows_store * b.Nx;
    if (i >= n) return;
    int lr = (int)(i / b.Nx), c = (int)(i - (size_t)lr * b.Nx);
    int row = b.row_base + lr;
    y[i] = 1.0;
    if (row >= b.own0 && row < b.own1) {
        size_t s = (size_t)(row - io_row0) * b.Nx + c;
        double v = V[s], mm = m ? m[s] : 0.0;
        coef[i] = (v < 0) ? __longlong_as_double(0x7ff8000000000000LL) : (v + g * mm) * inv_den;
    }
}

__device__ __forceinline__ double block_sum(double v, double *red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < NT / 32; i++) s += red[i];
    return s;
}

// out = f(y + c*f0) on owned rows (c = 0, f0 = NULL: f(y)).  optimals.py:144-164.  Used for the two RHS evaluations of
// the start-up (rk.py:94, common.py:126); tile partial sums in the same 128x16 layout as the single-GPU solver:
// mode 0: (y/sc)^2 -> partial[0..), (out/sc)^2 -> partial[nb..)   (d0, d1 with out = f0)
// mode 1: ((out - f0)/sc)^2 -> partial[0..)                        (d2 with out = f1)
__global__ void __launch_bounds__(NT)
rhs_band_kernel(const double *__restrict__ y, const double *__restrict__ f0, double c, const double *__restrict__ coef,
                double *__restrict__ out, BandView b, double A, double rtol, double atol, double *__restrict__ partial,
                int mode) {
    __shared__ double red[NT / 32];
    const int gx = blockIdx.x * TXS + (threadIdx.x & (TXS - 1));
    double a0 = 0.0, a1 = 0.0;
    for (int ly = threadIdx.x / TXS; ly < TYS; ly += NT / TXS) {
        const int row = b.own0 + blockIdx.y * TYS + ly;
        if (row >= b.own1 || gx >= b.Nx) continue;
        auto at = [&](int r, int cidx) {
            size_t s = (size_t)(mirror_idx(r, b.Ny) - b.row_base) * b.Nx + mirror_idx(cidx, b.Nx);
            return f0 ? fma(c, f0[s], y[s]) : y[s];
        };
        const size_t s = (size_t)(row - b.row_base) * b.Nx + gx;
        const double C = at(row, gx);
        const double lap = at(row - 1, gx) + at(row + 1, gx) + at(row, gx - 1) + at(row, gx + 1) - 4.0 * C;
        const double cf = coef[s];
        double r = A * lap - cf * C;
        if (cf != cf) r = 0.0;
        out[s] = r;
        const double sc = atol + fabs(y[s]) * rtol;
        if (mode == 0) {
            double q0 = y[s] / sc, q1 = r / sc;
            a0 += q0 * q0;
            a1 += q1 * q1;
        } else {
            double q = (r - f0[s]) / sc;
            a0 += q * q;
        }
    }
    const size_t nb = (size_t)gridDim.x * gridDim.y, bi = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
    double s0 = block_sum(a0, red);
    if (threadIdx.x == 0) partial[bi] = s0;
    __syncthreads();
    if (mode == 0) {
        double s1 = block_sum(a1, red);
        if (threadIdx.x == 0) partial[nb + bi] = s1;
    }
}

__global__ void __launch_bounds__(NT) rowsum_band_kernel(const double *__restrict__ partial, int nbx,
                                                         double *__restrict__ rowsum) {
    __shared__ double red[NT / 32];
    double v = 0.0;
    for (int i = threadIdx.x; i < nbx; i += NT) v += partial[(size_t)blockIdx.x * nbx + i];
    double s = block_sum(v, red);
    if (threadIdx.x == 0) rowsum[blockIdx.x] = s;
}

// phi slice (first row = global row phi_row_base) -> vx, vy rows (first row = global row v_row_base), interior only
__global__ void __launch_bounds__(NT)
vels_band_kernel(const double *__restrict__ phi, int phi_row_base, BandView b, double mu, double lim, double i2x,
                 double i2y, double *__restrict__ vx, double *__restrict__ vy, int v_row_base) {
    const int gx = blockIdx.x * 64 + (threadIdx.x & 63) + 1;
    const int row = b.own0 + blockIdx.y * 4 + (threadIdx.x >> 6);
    if (row >= b.own1 || row < 1 || row >= b.Ny - 1 || gx >= b.Nx - 1) return;
    const double *p = phi + (size_t)(row - phi_row_base) * b.Nx + gx;
    double ox, oy;
    vels_point(clamp_lim(p[0], lim), clamp_lim(p[-1], lim), clamp_lim(p[1], lim), clamp_lim(p[-b.Nx], lim),
               clamp_lim(p[b.Nx], lim), mu, lim, i2x, i2y, ox, oy);
    const size_t o = (size_t)(row - v_row_base) * (b.Nx - 2) + (gx - 1);
    vx[o] = ox;
    vy[o] = oy;
}

struct Band {
    BandView v;
    int rows_store;
    double *coef, *y, *ynew, *f, *fnew;  // storage (rows_store x Nx)
    double *partial;                     // per-band tile/chunk partial sums
    int gy_fused, gy_tiles;
    const double *V, *m;                 // inputs; element (row, col) at [(row - io_row0)*Nx + col]
    int io_row0;
    int phi_row_base, v_row_base;
    size_t phi_slice, v_slice;           // elements per output slice
    double *scratch;                     // NE_MAX phi slices when only velocities are requested
};

}  // namespace

extern "C" int oc_dist_unique_id(void *out128) {
    OC_ARG(out128, "NULL id");
    if (!g_nccl.load()) { oc::set_error("cannot load libnccl.so.2 (import torch first, or set LD_LIBRARY_PATH)"); return OC_ERR_NCCL; }
    ncclUniqueId id;
    OC_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(out128, &id, sizeof(id));
    return OC_OK;
}

extern "C" int oc_dist_init(oc_ctx *ctx, const void *id128, int rank, int nranks) {
    OC_ARG(ctx && id128 && nranks >= 1 && rank >= 0 && rank < nranks, "bad arguments");
    if (!g_nccl.load()) { oc::set_error("cannot load libnccl.so.2"); return OC_ERR_NCCL; }
    OC_CUDA(cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ncclComm_t comm = nullptr;
    OC_NCCL(g_nccl.CommInitRank(&comm, nranks, id, rank));
    ctx->nccl_comm = comm;
    ctx->rank = rank;
    ctx->nranks = nranks;
    return OC_OK;
}

// In-place element-wise maximum of `count` 64-bit words over all ranks.  The distributed GCFM step merges per-agent
// terms that exactly one rank computed (the others hold all-zero bits), so the maximum of the bit patterns is a
// bit-exact merge -- unlike a floating-point sum, which would turn -0.0 into +0.0.
int oc_dist_allreduce_max_u64(oc_ctx *ctx, void *d_buf, size_t count, cudaStream_t st) {
    if (!ctx->nccl_comm || ctx->nranks <= 1) return OC_OK;
    OC_NCCL(g_nccl.AllReduce(d_buf, d_buf, count, ncclUint64, ncclMax, (ncclComm_t)ctx->nccl_comm, st));
    return OC_OK;
}

// ---- NVLink peer-memory mode --------------------------------------------------------------------------------
// One cudaMalloc block per rank holds the four time-stepping arrays of its band (y, y_new, f, f_new: rows_store x Nx
// each) and the inboxes of the cross-GPU error-sum exchange.  The block is exported through CUDA IPC; every rank maps
// the blocks of all ranks (same layout everywhere, so a peer address is peer_base + local offset).
// Deferred halo exchange of the emitted phi samples (distributed GCFM sampler: every slice carries one row of the band
// above and 1 + xhi rows of the band below).  The rows are gathered from all nt slices into four contiguous buffers,
// exchanged with ONE NCCL group per solve, and scattered back -- instead of one small NCCL group per accepted step,
// which put ~50 us of launch latency on the critical path of every step.
// pack = 1: staging <- slice rows ; pack = 0: slice rows <- staging.  rows [r0, r0 + nr) of every slice.
__global__ void phi_halo_rows_kernel(double *__restrict__ phi, size_t slice, int nt, int Nx, int r0, int nr,
                                     double *__restrict__ staging, int pack) {
    const size_t per = (size_t)nr * Nx, total = per * nt;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t k = i / per, o = i - k * per;
        double *p = phi + k * slice + (size_t)r0 * Nx + o;
        if (pack) staging[i] = *p;
        else *p = staging[i];
    }
}

static size_t p2p_inbox_doubles() { return (size_t)2 * fused::P2P_MAX_RANKS * fused::P2P_INBOX_STRIDE; }

extern "C" int oc_dist_p2p_export(oc_ctx *ctx, int band_rows, void *handle_out64) {
    OC_ARG(ctx && handle_out64 && band_rows > 0, "bad arguments");
    OC_ARG(ctx->nranks >= 1 && ctx->nranks <= fused::P2P_MAX_RANKS, "peer-memory mode supports up to 8 ranks");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    OC_CUDA(cudaSetDevice(ctx->device));
    const size_t n_store = (size_t)(band_rows + 2 * HB) * ctx->Nx;
    const size_t bytes = (4 * n_store + p2p_inbox_doubles()) * sizeof(double);
    if (ctx->p2p_buf) { cudaFree(ctx->p2p_buf); ctx->p2p_buf = nullptr; }
    ctx->p2p_on = false;
    if (cudaMalloc(&ctx->p2p_buf, bytes) != cudaSuccess) {
        cudaGetLastError();
        oc::set_error("cannot allocate %zu bytes for the peer-memory band arrays", bytes);
        return OC_ERR_NOMEM;
    }
    OC_CUDA(cudaMemset(ctx->p2p_buf, 0, bytes));
    OC_CUDA(cudaDeviceSynchronize());
    ctx->p2p_bytes = bytes;
    ctx->p2p_n_store = n_store;
    cudaIpcMemHandle_t h;
    OC_CUDA(cudaIpcGetMemHandle(&h, ctx->p2p_buf));
    memcpy(handle_out64, &h, sizeof(h));
    return OC_OK;
}

extern "C" int oc_dist_p2p_import(oc_ctx *ctx, const void *handles, int n) {
    OC_ARG(ctx && handles && ctx->p2p_buf && n == ctx->nranks, "export first; one handle per rank expected");
    OC_CUDA(cudaSetDevice(ctx->device));
    for (int q = 0; q < n; q++) {
        if (q == ctx->rank) { ctx->p2p_peer[q] = ctx->p2p_buf; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles + (size_t)q * sizeof(h), sizeof(h));
        void *p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            oc::set_error("cudaIpcOpenMemHandle(rank %d) failed: %s", q, cudaGetErrorString(e));
            return OC_ERR_CUDA;
        }
        ctx->p2p_peer[q] = p;
    }
    ctx->p2p_on = true;
    ctx->p2p_seq = 0;
    return OC_OK;
}

extern "C" int oc_dist_p2p_enabled(oc_ctx *ctx) { return ctx && ctx->p2p_on ? 1 : 0; }
extern "C" int oc_dist_p2p_disable(oc_ctx *ctx) {
    if (ctx) ctx->p2p_on = false;  // back to the NCCL exchange (the mapped blocks are released by oc_dist_finalize)
    return OC_OK;
}

extern "C" int oc_dist_finalize(oc_ctx *ctx) {
    if (ctx && ctx->p2p_buf) {
        cudaSetDevice(ctx->device);
        for (int q = 0; q < ctx->nranks && q < 8; q++)
            if (q != ctx->rank && ctx->p2p_peer[q]) cudaIpcCloseMemHandle(ctx->p2p_peer[q]);
        cudaFree(ctx->p2p_buf);
        ctx->p2p_buf = nullptr;
        ctx->p2p_on = false;
    }
    if (ctx && ctx->nccl_comm) {
        g_nccl.CommDestroy((ncclComm_t)ctx->nccl_comm);
        ctx->nccl_comm = nullptr;
    }
    return OC_OK;
}

extern "C" int oc_hjb_solve_band(oc_ctx *ctx, const oc_band_cfg *cfg, const double *d_V, const double *d_m,
                                 const oc_hjb_params *prm, double T, const double *t_eval, int nt, double *d_phi,
                                 double *d_vx, double *d_vy, oc_hjb_stats *stats, double *trace_h, double *trace_err,
                                 int trace_cap, int *trace_n, void *stream) {
    OC_ARG(ctx && cfg && d_V && prm && stats && t_eval && nt >= 1, "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int Ny = ctx->Ny, Nx = ctx->Nx;
    const bool dist = ctx->nccl_comm != nullptr && cfg->n_virtual <= 1;
    const int nranks = dist ? ctx->nranks : 1, rank = dist ? ctx->rank : 0;
    ncclComm_t comm = (ncclComm_t)ctx->nccl_comm;
    const int nb_local = dist ? 1 : std::max(1, cfg->n_virtual);
    const int nbands = dist ? nranks : nb_local;
    OC_ARG(Ny > 2 * HB + 2 && Nx > 2 * fused::HX + 2, "grid too small for the fused step");
    // band layout: equal heights, multiples of 16 rows (tile rows) and of the chunk size
    int band_rows;
    if (dist) {
        band_rows = cfg->own1 - cfg->own0;
        OC_ARG(band_rows > 0 && cfg->own0 == rank * band_rows && band_rows * nranks == Ny, "bands must tile the grid equally");
    } else {
        OC_ARG(Ny % nbands == 0, "n_virtual must divide Ny");
        band_rows = Ny / nbands;
    }
    OC_ARG(nbands == 1 || (band_rows % TYS == 0 && band_rows >= 2 * HB), "band height must be a multiple of 16 and >= 12");
    const int gx_f = (Nx + fused::VX - 1) / fused::VX, gx_t = (Nx + TXS - 1) / TXS;
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device);
    int rc_rows = prm->chunk_rows;
    if (rc_rows <= 0) rc_rows = fused::plan_chunk_rows(Nx, band_rows, n_sm, dist ? 1 : nb_local, nbands > 1);
    OC_ARG(nbands == 1 || band_rows % rc_rows == 0, "band height must be a multiple of chunk_rows");
    const int gy_f = (band_rows + rc_rows - 1) / rc_rows, gy_t = (band_rows + TYS - 1) / TYS;
    const int rows_store = band_rows + 2 * HB;
    const size_t n_store = (size_t)rows_store * Nx, n_glob = (size_t)Ny * Nx;
    int rc0 = 0;
    const bool want_v = d_vx && d_vy, want_out = d_phi || want_v;
    // phi slices of a distributed band hold one halo row below and 1 + phi_extra_hi rows above the owned rows (the
    // GCFM sampler of an agent owned by this band reads up to two rows past it, oc_gcfm.cu)
    const int xhi = dist ? cfg->phi_extra_hi : 0;
    OC_ARG(xhi == 0 || xhi == 1, "phi_extra_hi must be 0 or 1");
    // phi samples with GCFM halo rows and no velocity conversion: their halo rows are exchanged once, after the solve
    const bool defer_phi_halo = dist && xhi && d_phi && !want_v && !getenv("OC_PHI_HALO_PER_STEP");

    // peer-memory mode: the band arrays live in the IPC-exported block, halos and error sums travel inside the step launch
    const bool use_p2p = dist && nranks > 1 && ctx->p2p_on && ctx->p2p_n_store == n_store && gy_f <= fused::P2P_INBOX_STRIDE - 2 &&
                         gy_f <= fused::MAX_FINAL_ROWS && !prm->forced_h;
    if (use_p2p && (rc0 = ocfinal::ensure(ctx, 1))) return rc0;
    // ---- workspace: per local band 5 arrays + partials (+ phi scratch)
    // (every piece is an even number of doubles: the band arrays stay 16-byte aligned for the TMA descriptors)
    const size_t n_partial = (((size_t)2 * gx_t * gy_t + (size_t)gx_f * gy_f + 64) + 1) & ~(size_t)1;
    const size_t per_band = 5 * n_store + n_partial + ((want_v && !d_phi) ? (size_t)fused::NE_MAX * (band_rows + 2) * Nx : 0);
    const int seg = (std::max(gy_f, gy_t) + 1) & ~1;  // row sums per band
    const size_t need = (per_band * nb_local + (size_t)2 * seg * nbands + 64) * sizeof(double);
    if ((rc0 = oc_ensure_buffer(ctx->dist_ws, ctx->dist_ws_bytes, need, false, "banded HJB workspace"))) return rc0;
    const size_t pin_need = ((size_t)seg * nbands + 16) * sizeof(double);
    if ((rc0 = oc_ensure_buffer(ctx->h_pinned, ctx->h_pinned_bytes, pin_need, true, "pinned host scratch"))) return rc0;
    double *wsp = (double *)ctx->dist_ws;
    double *rowsum_loc = wsp; wsp += (size_t)seg * nbands;   // this process's band sums (virtual: all bands)
    double *rowsum_all = wsp; wsp += (size_t)seg * nbands;   // gathered over all ranks
    double *rowsum_h = ctx->h_pinned;
    std::vector<Band> bands(nb_local);
    for (int q = 0; q < nb_local; q++) {
        Band &b = bands[q];
        const int bi = dist ? rank : q;
        b.v = BandView{Ny, Nx, bi * band_rows - HB, bi * band_rows, (bi + 1) * band_rows};
        b.rows_store = rows_store;
        b.coef = wsp; b.y = wsp + n_store; b.ynew = wsp + 2 * n_store; b.f = wsp + 3 * n_store; b.fnew = wsp + 4 * n_store;
        wsp += 5 * n_store;
        if (use_p2p) {
            double *pb = (double *)ctx->p2p_buf;
            b.y = pb; b.ynew = pb + n_store; b.f = pb + 2 * n_store; b.fnew = pb + 3 * n_store;
        }
        b.partial = wsp; wsp += n_partial;
        b.gy_fused = gy_f; b.gy_tiles = gy_t;
        b.V = d_V; b.m = d_m;
        b.io_row0 = dist ? b.v.own0 : 0;
        if (dist) {
            b.phi_row_base = b.v.own0 - 1; b.phi_slice = (size_t)(band_rows + 2 + xhi) * Nx;
            b.v_row_base = b.v.own0; b.v_slice = (size_t)band_rows * (Nx - 2);
        } else {
            b.phi_row_base = 0; b.phi_slice = n_glob;
            b.v_row_base = 1; b.v_slice = (size_t)(Ny - 2) * (Nx - 2);
        }
        b.scratch = nullptr;
        if (want_v && !d_phi) { b.scratch = wsp; wsp += (size_t)fused::NE_MAX * (band_rows + 2) * Nx; }
    }

    memset(stats, 0, sizeof(*stats));
    int launches = 0;
    const double s2 = prm->sigma * prm->sigma;
    const double A = (-0.5 * s2) / (ctx->dx * ctx->dy);
    const double rtol = prm->rtol, atol = prm->atol, sqrt_n = std::sqrt((double)n_glob);
    OC_CUDA(cudaEventRecord(ctx->ev0, st));

    // ---- halo exchange of `rows` boundary rows of one array per band (arr(b) selects the array)
    bool in_group = false;  // the caller has already opened an ncclGroup
    auto exchange = [&](std::initializer_list<double *Band::*> arrays, int phi_ne, double *const *phi_ptrs) -> int {
        // phi_ptrs: per local band, phi_ne slice pointers (only in dist mode, 1 halo row each side)
        if (nbands == 1) return OC_OK;
        if (!dist) {
            for (int q = 0; q + 1 < nb_local; q++) {
                Band &u = bands[q], &d = bands[q + 1];  // u above (smaller rows), d below
                for (auto arr : arrays) {
                    // d's top halo <- u's last HB owned rows ; u's bottom halo <- d's first HB owned rows
                    OC_CUDA(cudaMemcpyAsync(d.*arr, u.*arr + (size_t)band_rows * Nx, sizeof(double) * HB * Nx,
                                            cudaMemcpyDeviceToDevice, st));
                    OC_CUDA(cudaMemcpyAsync(u.*arr + (size_t)(HB + band_rows) * Nx, d.*arr + (size_t)HB * Nx,
                                            sizeof(double) * HB * Nx, cudaMemcpyDeviceToDevice, st));
                }
            }
            return OC_OK;
        }
        Band &b = bands[0];
        if (!in_group) OC_NCCL(g_nccl.GroupStart());
        for (auto arr : arrays) {
            double *p = b.*arr;
            if (rank > 0) {
                OC_NCCL(g_nccl.Send(p + (size_t)HB * Nx, (size_t)HB * Nx, ncclFloat64, rank - 1, comm, st));
                OC_NCCL(g_nccl.Recv(p, (size_t)HB * Nx, ncclFloat64, rank - 1, comm, st));
            }
            if (rank + 1 < nranks) {
                OC_NCCL(g_nccl.Send(p + (size_t)band_rows * Nx, (size_t)HB * Nx, ncclFloat64, rank + 1, comm, st));
                OC_NCCL(g_nccl.Recv(p + (size_t)(HB + band_rows) * Nx, (size_t)HB * Nx, ncclFloat64, rank + 1, comm, st));
            }
        }
        for (int e = 0; e < phi_ne; e++) {  // slice storage: row 0 = own0-1 (halo), rows 1..band_rows owned, last = halo
            double *p = phi_ptrs[e];
            if (rank > 0) {  // my first 1 + xhi owned rows are the upper neighbour's high halo
                OC_NCCL(g_nccl.Send(p + (size_t)1 * Nx, (size_t)(1 + xhi) * Nx, ncclFloat64, rank - 1, comm, st));
                OC_NCCL(g_nccl.Recv(p, Nx, ncclFloat64, rank - 1, comm, st));
            }
            if (rank + 1 < nranks) {
                OC_NCCL(g_nccl.Send(p + (size_t)band_rows * Nx, Nx, ncclFloat64, rank + 1, comm, st));
                OC_NCCL(g_nccl.Recv(p + (size_t)(band_rows + 1) * Nx, (size_t)(1 + xhi) * Nx, ncclFloat64, rank + 1, comm, st));
            }
        }
        if (!in_group) OC_NCCL(g_nccl.GroupEnd());
        return OC_OK;
    };

    // ---- sum of per-band partial sums (layout gx x gy per band at partial+off) in global order, on every rank
    // with_halo: also ship the boundary rows of y_new / f_new in the SAME ncclGroup (one launch latency per
    // attempt).  The exchange is speculative: if the attempt is rejected the received rows are simply never used.
    auto reduce = [&](size_t off, int gx, int gy, double *out, bool with_halo = false) -> int {
        for (int q = 0; q < nb_local; q++) {
            rowsum_band_kernel<<<gy, NT, 0, st>>>(bands[q].partial + off, gx, rowsum_loc + (size_t)q * gy);
            launches++;
        }
        const double *src = rowsum_loc;
        if (dist && nranks > 1) {
            OC_NCCL(g_nccl.GroupStart());
            OC_NCCL(g_nccl.AllGather(rowsum_loc, rowsum_all, gy, ncclFloat64, comm, st));
            if (with_halo) {
                in_group = true;
                int erc = exchange({&Band::ynew, &Band::fnew}, 0, nullptr);
                in_group = false;
                if (erc) return erc;
            }
            OC_NCCL(g_nccl.GroupEnd());
            src = rowsum_all;
        } else if (with_halo) {
            int erc = exchange({&Band::ynew, &Band::fnew}, 0, nullptr);
            if (erc) return erc;
        }
        OC_CUDA(cudaMemcpyAsync(rowsum_h, src, sizeof(double) * gy * nbands, cudaMemcpyDeviceToHost, st));
        OC_CUDA(cudaStreamSynchronize(st));
        double s = 0.0;
        for (int i = 0; i < gy * nbands; i++) s += rowsum_h[i];  // global chunk order
        *out = s;
        return OC_OK;
    };

    int rc;
    for (Band &b : bands) {
        prep_band_kernel<<<(unsigned)((n_store + 255) / 256), 256, 0, st>>>(b.V, b.m, b.io_row0, prm->g, 1.0 / (prm->mu * s2),
                                                                             b.v, rows_store, b.coef, b.y);
        launches++;
    }
    if ((rc = exchange({&Band::coef}, 0, nullptr))) return rc;

    rk45::Controller ctl(T, t_eval, nt);
    dim3 grid_t(gx_t, gy_t);
    const size_t nb_t = (size_t)gx_t * gy_t;
    // rk.py:94 f0 = fun(t0, y0) and the d0, d1 norms of select_initial_step (common.py:109-118)
    for (Band &b : bands) {
        rhs_band_kernel<<<grid_t, NT, 0, st>>>(b.y, nullptr, 0.0, b.coef, b.f, b.v, A, rtol, atol, b.partial, 0);
        launches++;
    }
    stats->nfev++;
    if ((rc = exchange({&Band::f}, 0, nullptr))) return rc;
    if (ctl.needs_initial_step()) {
        double s0, s1, sq2;
        if ((rc = reduce(0, gx_t, gy_t, &s0))) return rc;
        if ((rc = reduce(nb_t, gx_t, gy_t, &s1))) return rc;
        const double d1 = std::sqrt(s1) / sqrt_n;
        const double h0 = ctl.initial_h0(std::sqrt(s0) / sqrt_n, d1);
        for (Band &b : bands) {  // f1 = fun(t0 + h0*dir, y0 + h0*dir*f0) into ynew (scratch)
            rhs_band_kernel<<<grid_t, NT, 0, st>>>(b.y, b.f, h0 * ctl.direction, b.coef, b.ynew, b.v, A, rtol, atol,
                                                  b.partial, 1);
            launches++;
        }
        stats->nfev++;
        if ((rc = reduce(0, gx_t, gy_t, &sq2))) return rc;
        ctl.set_initial_step(h0, d1, std::sqrt(sq2) / sqrt_n / h0);
    }
    stats->h0 = ctl.h_abs;

    fused::MapCache maps;  // TMA descriptors of the band arrays
    auto launch_fused = [&](int ne, fused::Args &fa, dim3 grid) -> int {
        fused::set_tensor_maps(fa, rows_store, &maps);
        OC_CUDA(use_p2p ? fused::launch<true>(ne, fa, grid, st) : fused::launch<false>(ne, fa, grid, st));
        launches++;
        return OC_OK;
    };
    // peer addresses: same layout in every rank's block
    auto peer_of = [&](int q, const double *mine) -> double * {
        return (double *)ctx->p2p_peer[q] + (mine - (const double *)ctx->p2p_buf);
    };

    unsigned long long p2p_wait_seq = 0;
    cudaEvent_t pe0 = nullptr, pe1 = nullptr;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof;  // one pair per attempt, read after the final synchronisation
    double step_ms = 0.0;
    int step_launches = 0;

    while (ctl.begin_step()) {
        bool accepted = false;
        while (!accepted && ctl.propose(prm->forced_h, prm->n_forced_h)) {
            const int n_emit = want_out ? ctl.n_emit() : 0;
            // samples beyond NE_MAX per launch: repeat the (identical) step for the next batch
            int done = 0;
            do {
                const int ne = std::min(n_emit - done, (int)fused::NE_MAX);
                for (int q = 0; q < nb_local; q++) {
                    Band &b = bands[q];
                    fused::Args fa{};
                    fa.y = b.y; fa.k1 = b.f; fa.coef = b.coef; fa.ynew = b.ynew; fa.k7 = b.fnew;
                    fa.partial = b.partial + 2 * nb_t;
                    fa.A = A; fa.rtol = rtol; fa.atol = atol;
                    fa.Ny = Ny; fa.Nx = Nx; fa.RC = rc_rows;
                    fa.row_base = b.v.row_base; fa.own0 = b.v.own0; fa.own1 = b.v.own1; fa.phi_row_base = b.phi_row_base;
                    fused::set_attempt(fa, ctl, done, ne, d_phi, b.scratch, b.phi_slice);
                    if (use_p2p) {
                        // sequence numbers of this mode carry bit 62, so a value left in the result slot by a
                        // single-GPU solve on the same context (its own counter) can never look like an answer
                        ocfinal::set_args(ctx, 0, (1ull << 62) | ++ctx->p2p_seq, fa);
                        p2p_wait_seq = fa.seq;
                        fa.nranks = nranks; fa.my_rank = rank;
                        for (int r2 = 0; r2 < nranks; r2++)
                            fa.peer_inbox[r2] = (double *)ctx->p2p_peer[r2] + 4 * n_store;
                        if (rank > 0) {
                            fa.peer_ynew[0] = peer_of(rank - 1, b.ynew); fa.peer_k7[0] = peer_of(rank - 1, b.fnew);
                            fa.peer_row_base[0] = b.v.row_base - band_rows;
                        }
                        if (rank + 1 < nranks) {
                            fa.peer_ynew[1] = peer_of(rank + 1, b.ynew); fa.peer_k7[1] = peer_of(rank + 1, b.fnew);
                            fa.peer_row_base[1] = b.v.row_base + band_rows;
                        }
                    }
                    if (prm->profile && q == 0 && done == 0) {
                        cudaEventCreate(&pe0); cudaEventCreate(&pe1);
                        prof.emplace_back(pe0, pe1);
                        cudaEventRecord(pe0, st);
                    }
                    if ((rc = launch_fused(ne, fa, dim3(gx_f, gy_f)))) return rc;
                    if (prm->profile && q == nb_local - 1 && done == 0) {
                        cudaEventRecord(pe1, st);
                    }
                }
                done += ne;
            } while (done < n_emit && !(want_v && !d_phi));  // scratch holds one batch only (see below)
            stats->nfev += 6;
            double se;
            if (use_p2p) {
                // halos and the gathered error sums arrived inside the launch; the last CTA hands over the total
                if ((rc = ocfinal::wait(ctx, 0, p2p_wait_seq, st, &se))) return rc;
            } else if ((rc = reduce(2 * nb_t, gx_f, gy_f, &se, true))) return rc;
            if (prm->profile) step_launches += nb_local;
            const double error_norm = std::sqrt(se) / sqrt_n;
            const int ntr = ctl.attempts();
            if (trace_h && ntr < trace_cap) { trace_h[ntr] = ctl.h; trace_err[ntr] = error_norm; }
            accepted = ctl.judge(error_norm);
        }
        if (!accepted) break;  // step too small
        // ---- accepted: velocities of the emitted samples, halo exchange of the new state
        const int n_emit = ctl.n_emit();
        if (want_v && !d_phi && n_emit > fused::NE_MAX) {
            oc::set_error("banded solve: more than %d samples in one step need d_phi storage", fused::NE_MAX);
            return OC_ERR_ARG;
        }
        std::vector<double *> phis;
        if (want_v)
            for (int e = 0; e < n_emit; e++) {
                if (ctl.sample_column(e) < 1) continue;
                for (Band &b : bands) phis.push_back(fused::sample_slice(ctl, e, d_phi, b.scratch, b.phi_slice));
            }
        for (Band &b : bands) { std::swap(b.y, b.ynew); std::swap(b.f, b.fnew); }  // FSAL (rk.py:167-174)
        // the halo rows of the new y, f travelled with the error sums; only the halo rows of the emitted phi slices are
        // left: needed by the velocity conversion below and, with phi_extra_hi, by the distributed GCFM sampler
        if (dist && want_v && !phis.empty() && (rc = exchange({}, (int)phis.size(), phis.data()))) return rc;
        if (dist && !want_v && xhi && d_phi && !defer_phi_halo) {
            std::vector<double *> hp;
            for (int e = 0; e < n_emit; e++) hp.push_back(fused::sample_slice(ctl, e, d_phi, nullptr, bands[0].phi_slice));
            if (!hp.empty() && (rc = exchange({}, (int)hp.size(), hp.data()))) return rc;
        }
        if (want_v) {
            size_t pi = 0;
            for (int e = 0; e < n_emit; e++) {
                const int kd = ctl.sample_column(e);
                if (kd < 1) continue;
                const int sl = nt - 1 - kd;
                for (Band &b : bands) {
                    dim3 grid((Nx - 2 + 63) / 64, (band_rows + 3) / 4);
                    vels_band_kernel<<<grid, NT, 0, st>>>(phis[pi++], b.phi_row_base, b.v, prm->mu, prm->lim,
                                                          1.0 / (2 * ctx->dx), 1.0 / (2 * ctx->dy),
                                                          d_vx + (size_t)sl * b.v_slice, d_vy + (size_t)sl * b.v_slice,
                                                          b.v_row_base);
                    launches++;
                }
            }
        }
        ctl.accept();
    }
    if (defer_phi_halo && ctl.status == 0 && nranks > 1) {
        // all nt samples are final now: one packed exchange of their halo rows (see phi_halo_rows_kernel)
        Band &b = bands[0];
        const int up = 1 + xhi;                       // rows I send up / receive from below
        const size_t n_up = (size_t)nt * up * Nx, n_dn = (size_t)nt * Nx;
        const size_t need = 2 * (n_up + n_dn) * sizeof(double);
        if ((rc = oc_ensure_buffer(ctx->dist_halo, ctx->dist_halo_bytes, need, false, "phi halo exchange staging")))
            return rc;
        double *s_up = (double *)ctx->dist_halo, *s_dn = s_up + n_up, *r_up = s_dn + n_dn, *r_dn = r_up + n_dn;
        const int blocks = 592;
        if (rank > 0) phi_halo_rows_kernel<<<blocks, 256, 0, st>>>(d_phi, b.phi_slice, nt, Nx, 1, up, s_up, 1);
        if (rank + 1 < nranks) phi_halo_rows_kernel<<<blocks, 256, 0, st>>>(d_phi, b.phi_slice, nt, Nx, band_rows, 1, s_dn, 1);
        OC_NCCL(g_nccl.GroupStart());
        if (rank > 0) {
            OC_NCCL(g_nccl.Send(s_up, n_up, ncclFloat64, rank - 1, comm, st));
            OC_NCCL(g_nccl.Recv(r_up, n_dn, ncclFloat64, rank - 1, comm, st));
        }
        if (rank + 1 < nranks) {
            OC_NCCL(g_nccl.Send(s_dn, n_dn, ncclFloat64, rank + 1, comm, st));
            OC_NCCL(g_nccl.Recv(r_dn, n_up, ncclFloat64, rank + 1, comm, st));
        }
        OC_NCCL(g_nccl.GroupEnd());
        if (rank > 0) phi_halo_rows_kernel<<<blocks, 256, 0, st>>>(d_phi, b.phi_slice, nt, Nx, 0, 1, r_up, 0);
        if (rank + 1 < nranks) phi_halo_rows_kernel<<<blocks, 256, 0, st>>>(d_phi, b.phi_slice, nt, Nx, band_rows + 1, up, r_dn, 0);
        launches += (rank > 0 ? 2 : 0) + (rank + 1 < nranks ? 2 : 0);
    }
    OC_CUDA(cudaEventRecord(ctx->ev1, st));
    OC_CUDA(cudaStreamSynchronize(st));
    OC_CUDA(cudaGetLastError());
    float ms = 0;
    OC_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    for (auto &pr : prof) {
        float pms = 0;
        if (cudaEventElapsedTime(&pms, pr.first, pr.second) == cudaSuccess) step_ms += pms;
        cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
    }
    cudaGetLastError();
    stats->gpu_ms = ms;
    ctl.report(stats);
    stats->launches = launches;
    stats->cls_launches[0] = step_launches;
    stats->cls_ms[0] = step_ms;
    stats->cls_bytes[0] = 0;  // filled by the caller from nfev (40 B/cell/attempt + 8 B/cell/sample)
    oc::count_launch(launches);
    if (trace_n) *trace_n = ctl.attempts();
    if (ctl.status == -1) {
        oc::set_error("RK45: required step size is less than spacing between numbers (t=%g)", ctl.t);
        return OC_ERR_STEP_TOO_SMALL;
    }
    return OC_OK;
}
