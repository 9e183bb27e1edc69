// oc_api.cu -- context management, error text, rasteriser (K8) and density (K7) of liboc_b200.so.
#include <algorithm>
#include <cmath>
#include <mutex>

#include "oc_common.h"
#include "oc_math.h"
#include "oc_rng.h"

namespace oc {
static thread_local char g_err[1024] = "";
std::atomic<long long> g_launches{0};
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace oc

extern "C" int oc_abi_version(void) { return OC_ABI_VERSION; }
extern "C" const char *oc_last_error(void) { return oc::g_err; }
extern "C" long long oc_launch_count(int reset) {
    return reset ? oc::g_launches.exchange(0) : oc::g_launches.load();
}

extern "C" int oc_ctx_create(int device, int Ny, int Nx, double dx, double dy, double room_length,
                             double room_height, const double *X, const double *Y, oc_ctx **out) {
    OC_ARG(out != nullptr, "out is NULL");
    OC_ARG(Ny >= 3 && Nx >= 3, "grid must be at least 3x3");
    OC_ARG(X != nullptr && Y != nullptr, "X/Y linspace arrays required");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        oc::set_error("no CUDA device available (%s); liboc_b200 has no CPU fallback",
                      e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return OC_ERR_CUDA;
    }
    OC_ARG(device >= 0 && device < ndev, "device index out of range");
    OC_CUDA(cudaSetDevice(device));
    oc_ctx *c = new oc_ctx();
    c->device = device;
    c->Ny = Ny;
    c->Nx = Nx;
    c->dx = dx;
    c->dy = dy;
    c->room_length = room_length;
    c->room_height = room_height;
    c->X.assign(X, X + Nx);
    c->Y.assign(Y, Y + Ny);
    OC_CUDA(cudaMalloc(&c->d_X, sizeof(double) * Nx));
    OC_CUDA(cudaMalloc(&c->d_Y, sizeof(double) * Ny));
    OC_CUDA(cudaMemcpy(c->d_X, X, sizeof(double) * Nx, cudaMemcpyHostToDevice));
    OC_CUDA(cudaMemcpy(c->d_Y, Y, sizeof(double) * Ny, cudaMemcpyHostToDevice));
    OC_CUDA(cudaEventCreate(&c->ev0));
    OC_CUDA(cudaEventCreate(&c->ev1));
    *out = c;
    return OC_OK;
}

extern "C" int oc_ctx_set_int(oc_ctx *ctx, const char *key, int value) {
    OC_ARG(ctx && key, "NULL argument");
    if (!strcmp(key, "gcfm_sweep_ctas")) {
        OC_ARG(value >= 0, "gcfm_sweep_ctas must be >= 0");
        ctx->gcfm_sweep_ctas = value;
        return OC_OK;
    }
    if (!strcmp(key, "gcfm_poll_ns")) {
        OC_ARG(value >= 0 && value <= 1000000, "gcfm_poll_ns out of range");
        ctx->gcfm_poll_ns = value;
        return OC_OK;
    }
    if (!strcmp(key, "gcfm_margin_mm")) {
        OC_ARG(value >= 20 && value <= 1000, "gcfm_margin_mm out of range (20..1000)");
        ctx->gcfm_margin_mm = value;
        ctx->gcfm_margin_hold = 0;
        return OC_OK;
    }
    if (!strcmp(key, "gcfm_fov_cull")) {
        ctx->gcfm_fov_cull = value != 0;
        return OC_OK;
    }
    if (!strcmp(key, "gcfm_ws_pair")) {
        ctx->gcfm_ws_pair = value != 0;
        return OC_OK;
    }
    if (!strcmp(key, "gcfm_split")) {
        ctx->gcfm_split = value != 0;
        return OC_OK;
    }
    if (!strcmp(key, "gcfm_graph")) {
        ctx->gcfm_use_graph = value != 0;
        return OC_OK;
    }
    if (!strcmp(key, "gcfm_overlap")) {
        ctx->gcfm_overlap = value != 0;
        return OC_OK;
    }
    oc::set_error("unknown option '%s'", key);
    return OC_ERR_ARG;
}

extern "C" void oc_ctx_destroy(oc_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaFree(c->d_X);
    cudaFree(c->d_Y);
    cudaFree(c->hjb_ws);
    cudaFree(c->hjb_partial);
    cudaFree(c->hjb_scratch);
    cudaFree(c->dist_ws);
    cudaFree(c->dist_halo);
    oc_dist_finalize(c);
    cudaFree(c->gcfm_ws);
    oc_gcfm_free_launch_state(c);
    if (c->multi_pinned) cudaFreeHost(c->multi_pinned);
    cudaFree(c->multi_dev);
    if (c->dens_ev) cudaEventSynchronize(c->dens_ev);
    if (c->dens_pinned) cudaFreeHost(c->dens_pinned);
    cudaFree(c->dens_dev);
    if (c->dens_ev) cudaEventDestroy(c->dens_ev);
    if (c->lines_ev) cudaEventSynchronize(c->lines_ev);
    if (c->lines_pinned) cudaFreeHost(c->lines_pinned);
    cudaFree(c->lines_dev);
    if (c->lines_ev) cudaEventDestroy(c->lines_ev);
    if (c->areas_ev) cudaEventSynchronize(c->areas_ev);
    if (c->areas_pinned) cudaFreeHost(c->areas_pinned);
    cudaFree(c->areas_dev);
    if (c->areas_ev) cudaEventDestroy(c->areas_ev);
    if (c->vor_ev) cudaEventSynchronize(c->vor_ev);
    if (c->vor_pinned) cudaFreeHost(c->vor_pinned);
    cudaFree(c->vor_dev);
    if (c->vor_ev) cudaEventDestroy(c->vor_ev);
    if (c->vmap_ev) cudaEventSynchronize(c->vmap_ev);
    if (c->vmap_pinned) cudaFreeHost(c->vmap_pinned);
    cudaFree(c->vmap_dev);
    if (c->vmap_ev) cudaEventDestroy(c->vmap_ev);
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    if (c->gcfm_pinned) cudaFreeHost(c->gcfm_pinned);
    cudaFree(c->fr_ticket);
    if (c->fr_result) cudaFreeHost(c->fr_result);
    cudaFree(c->batch_ws);
    if (c->batch_pinned) cudaFreeHost(c->batch_pinned);
    for (auto s : c->batch_streams) cudaStreamDestroy(s);
    for (auto e : c->batch_events) cudaEventDestroy(e);
    if (c->gcfm_graph) cudaGraphExecDestroy(c->gcfm_graph);
    if (c->gcfm_side) cudaStreamDestroy(c->gcfm_side);
    if (c->gcfm_side2) cudaStreamDestroy(c->gcfm_side2);
    if (c->gcfm_cap) cudaStreamDestroy(c->gcfm_cap);
    if (c->gcfm_ev_fork) cudaEventDestroy(c->gcfm_ev_fork);
    if (c->gcfm_ev_join) cudaEventDestroy(c->gcfm_ev_join);
    if (c->gcfm_ev_join2) cudaEventDestroy(c->gcfm_ev_join2);
    if (c->gcfm_stage) cudaFreeHost(c->gcfm_stage);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    delete c;
}

// ------------------------------------------------------------------------------------------------
// Host -> device transfer of an input array (the density `m` of optimals.compute_optimal_velocity arrives as a
// numpy array, optimals.py:124) into a caller-owned device buffer on `stream`.  Page-locked sources go to the copy
// engine directly (measured 51.7 GB/s on the B200 box); pageable ones are staged by the driver (25.9 GB/s measured,
// faster than a hand-rolled double-buffered memcpy pipeline on one host thread, 18 GB/s) and have been read
// completely when the call returns.
extern "C" int oc_upload(oc_ctx *ctx, const void *host, void *d_dst, long long bytes, void *stream) {
    OC_ARG(ctx && (bytes == 0 || (host && d_dst)) && bytes >= 0, "NULL argument");
    if (bytes == 0) return OC_OK;
    OC_CUDA(cudaSetDevice(ctx->device));
    // OC_UPLOAD_CHUNK_MB > 0: the copy is issued in pieces, so that launches of a solve running on another stream can
    // slip in between them instead of queueing behind one 268 MB transfer (prefetch of the next solve's density)
    static const long long chunk = [] {
        const char *e = getenv("OC_UPLOAD_CHUNK_MB");
        return e ? (long long)atoll(e) << 20 : 0ll;
    }();
    if (chunk <= 0 || bytes <= chunk) {
        OC_CUDA(cudaMemcpyAsync(d_dst, host, (size_t)bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
        return OC_OK;
    }
    for (long long off = 0; off < bytes; off += chunk)
        OC_CUDA(cudaMemcpyAsync((char *)d_dst + off, (const char *)host + off, (size_t)std::min(chunk, bytes - off),
                                cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return OC_OK;
}

// ------------------------------------------------------------------------------------------------
// Crowd placement of one initial box (simulations.py:122-138) on the host, in C: the reference's rejection sampling with
// its exact consumption of numpy's legacy MT19937 stream -- two uniform(lo, hi, 1) draws per trial, x first (:130-131) --
// and its occupancy test on the node mask (:132,135), restricted to the window of nodes that can lie within r_in of
// the trial.  The generator state (624 key words + position) is passed in and out, so that the Python host continues
// with np.random exactly where the reference would be.  ~50 ns per trial instead of ~8 us in numpy: 100k agents are
// placed in milliseconds (SURVEY.md section 8 f2).  No CUDA involved.
extern "C" long long oc_place_box(const double *box, const double *X, int Nx, const double *Y, int Ny, double *place_ped,
                                  double r_in, uint32_t *mt_key, int *mt_pos, double *xs, double *ys, int loc_N) {
    if (!box || !X || !Y || !place_ped || !mt_key || !mt_pos || (loc_N > 0 && (!xs || !ys)) || Nx < 2 || Ny < 2 ||
        *mt_pos < 0 || *mt_pos > 624) {
        oc::set_error("bad argument: oc_place_box");
        return OC_ERR_ARG;
    }
    ocrng::Mt mt{mt_key, *mt_pos, 0, 0.0};
    const double lox = box[0] - box[2] / 2, hix = box[0] + box[2] / 2, loy = box[1] - box[3] / 2, hiy = box[1] + box[3] / 2;
    const double sx = hix - lox, sy = hiy - loy;  // legacy uniform: low + (high - low) * next_double
    const double stepx = X[1] - X[0], stepy = Y[1] - Y[0];
    long long trials = 0;
    int placed = 0;
    while (placed < loc_N) {
        trials++;
        const double x = lox + sx * mt.next_double();
        const double y = loy + sy * mt.next_double();
        const int j0 = std::max((int)std::floor((x - r_in) / stepx) - 2, 0), j1 = std::min((int)std::ceil((x + r_in) / stepx) + 3, Nx);
        const int i0 = std::max((int)std::floor((y - r_in) / stepy) - 2, 0), i1 = std::min((int)std::ceil((y + r_in) / stepy) + 3, Ny);
        bool taken = false;
        for (int i = i0; i < i1 && !taken; i++) {
            const double dy = Y[i] - y, dy2 = dy * dy;
            for (int j = j0; j < j1; j++) {
                const double dx = X[j] - x;
                if (std::sqrt(dx * dx + dy2) < r_in && place_ped[(size_t)i * Nx + j] == 1.0) { taken = true; break; }
            }
        }
        if (taken) continue;                                                  // simulations.py:132
        for (int i = i0; i < i1; i++) {
            const double dy = Y[i] - y, dy2 = dy * dy;
            for (int j = j0; j < j1; j++) {
                const double dx = X[j] - x;
                if (std::sqrt(dx * dx + dy2) < r_in) place_ped[(size_t)i * Nx + j] = 1.0;   // :135
            }
        }
        xs[placed] = x; ys[placed] = y;
        placed++;
    }
    *mt_pos = mt.pos;
    return trials;
}

// The randomness of one GCFM step, drawn from a legacy MT19937 state exactly as the reference does (simulations.py:271:
// np.random.choice(np.arange(N), N, replace=False); :303: one np.random.normal(size=2) per agent inside, in sweep order).
// State = np.random.get_state()[1:5], advanced in place.  perm: N ints; noise: (n_active, 2) doubles.
extern "C" int oc_rng_step_draw(uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int N, int n_active,
                                int *perm, double *noise) {
    return oc_rng_step_draw_ckpt(mt_key, mt_pos, has_gauss, cached_gauss, N, n_active, perm, noise, 0, nullptr, nullptr,
                                 nullptr, nullptr);
}

// The same draw with snapshots of the generator state as it is after n_active - q pairs, q = 0 .. n_ckpt-1: a caller that
// draws a step's randomness ahead of time for an UPPER BOUND of agents (nobody leaves) can later continue the stream
// exactly where the reference would be once the true count (n_active - q) is known (look-ahead RNG of the run loop).
extern "C" int oc_rng_step_draw_ckpt(uint32_t *mt_key, int *mt_pos, int *has_gauss, double *cached_gauss, int N,
                                     int n_active, int *perm, double *noise, int n_ckpt, uint32_t *ckpt_key,
                                     int *ckpt_pos, int *ckpt_has, double *ckpt_cached) {
    OC_ARG(mt_key && mt_pos && has_gauss && cached_gauss && perm && (n_active == 0 || noise) && N >= 0 && n_active >= 0 &&
           *mt_pos >= 0 && *mt_pos <= 624 && n_ckpt >= 0 && (n_ckpt == 0 || (ckpt_key && ckpt_pos && ckpt_has && ckpt_cached)),
           "oc_rng_step_draw");
    ocrng::Mt mt{mt_key, *mt_pos, *has_gauss, *cached_gauss};
    mt.permutation(N, perm);
    mt.gauss_fill(noise, 2ll * n_active, n_ckpt, ckpt_key, ckpt_pos, ckpt_has, ckpt_cached);
    *mt_pos = mt.pos; *has_gauss = mt.has_gauss; *cached_gauss = mt.gauss_;
    return OC_OK;
}

// ------------------------------------------------------------------------------------------------
// FP64 pipe peak of this GPU, measured: the roofline denominator of the GCFM pair forces (SURVEY.md section 8d asks
// for a measured FP64 FMA peak; MEASURED_PEAKS.json only carries HBM and bf16 tensor figures).  8 independent DFMA
// chains per thread, 16 warps per SM, ~10^9 FMAs: B200 sustains ~1.84 warp-DFMA per clock and SM (34 TFLOP/s).
namespace {
__global__ void __launch_bounds__(512) fp64_peak_kernel(double *out, int iters, double a, double b) {
    double v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = threadIdx.x * 1e-9 + i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 16; u++)
#pragma unroll
            for (int i = 0; i < 8; i++) v[i] = fma(v[i], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s += v[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
}  // namespace

extern "C" int oc_fp64_peak(oc_ctx *ctx, double *tflops) {
    OC_ARG(ctx && tflops, "NULL argument");
    OC_CUDA(cudaSetDevice(ctx->device));
    int n_sm = 0;
    OC_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device));
    double *d = nullptr;
    OC_CUDA(cudaMalloc(&d, sizeof(double) * 512 * n_sm));
    const int iters = 4000;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        OC_CUDA(cudaEventRecord(ctx->ev0, 0));
        fp64_peak_kernel<<<n_sm, 512>>>(d, iters, 0.999, 1e-3);
        OC_CUDA(cudaEventRecord(ctx->ev1, 0));
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { cudaFree(d); OC_CUDA(e); }
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaFree(d);
    oc::count_launch(4);
    *tflops = 2.0 * (double)iters * 16 * 8 * 512 * n_sm / (best * 1e-3) / 1e12;
    return OC_OK;
}

// ------------------------------------------------------------------------------------------------
// Packed copy of the crowd state: out[i] = (x, y, vx, vy) of agent i, one row of the device-resident trajectory
// record (ped.traj / ped.vels, pedestrians.py:189-190; history frames, simulations.py:579-589).
namespace {
__global__ void state_pack_kernel(int N, const double *__restrict__ x, const double *__restrict__ y,
                                  const double *__restrict__ vx, const double *__restrict__ vy, double4 *__restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = make_double4(x[i], y[i], vx[i], vy[i]);
}
}  // namespace

extern "C" int oc_state_pack(oc_ctx *ctx, int N, const double *d_x, const double *d_y, const double *d_vx,
                             const double *d_vy, double *d_out, void *stream) {
    OC_ARG(ctx && N >= 0 && (N == 0 || (d_x && d_y && d_vx && d_vy && d_out)), "NULL argument");
    OC_ARG(((uintptr_t)d_out % 32) == 0, "d_out must be 32-byte aligned");
    if (N == 0) return OC_OK;
    OC_CUDA(cudaSetDevice(ctx->device));
    state_pack_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(N, d_x, d_y, d_vx, d_vy,
                                                                         reinterpret_cast<double4 *>(d_out));
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}

// ------------------------------------------------------------------------------------------------
// K8 rasteriser: one thread per node, shapes staged in shared memory in chunks.
// simulations.py:536-576: walls add -1 (:538-547), holes set 0 (:549-555), cylinders add -1 (:557-563),
// frame = -1 (:565-568), targets = 1 (:570-574); strict '<' on the linspace coordinates.
// optimals.py:89-91 remap: V<0 -> pot, V>0 -> pot_target.
namespace {
constexpr int RAST_CHUNK = 256;

struct RastArgs {
    const double *walls, *holes, *cyls, *targets;  // device copies
    int n_walls, n_holes, n_cyls, n_targets;
    int remap;
    double wall_value, target_value;
};

// Stage into shared memory the shapes of one chunk whose bounding box touches the block's node rectangle
// (conservative, non-strict test; the per-node test below is the reference's strict one).  Order inside a
// class does not matter: walls/cylinders add -1 (exact integer sums), holes/targets assign a constant.
template <int W>
__device__ __forceinline__ int stage_shapes(const double *__restrict__ src, int base, int n_total, double x0,
                                            double x1, double y0, double y1, double *sh, int *cnt) {
    if (threadIdx.x == 0) *cnt = 0;
    __syncthreads();
    int k = base + threadIdx.x;
    if (k < n_total) {
        const double *s = src + (size_t)k * W;
        double hx = (W == 4) ? s[2] / 2 : s[2], hy = (W == 4) ? s[3] / 2 : s[2];
        if (s[0] - hx <= x1 && s[0] + hx >= x0 && s[1] - hy <= y1 && s[1] + hy >= y0) {
            int pos = atomicAdd(cnt, 1);
            for (int q = 0; q < W; q++) sh[pos * W + q] = s[q];
        }
    }
    __syncthreads();
    return *cnt;
}

// rows [row0, row0+rows) of the (Ny,Nx) grid are written to V (rows, Nx)
__global__ void __launch_bounds__(256) rasterise_kernel(const double *__restrict__ X, const double *__restrict__ Y,
                                                        int Ny, int Nx, RastArgs a, int row0, int rows,
                                                        double *__restrict__ V) {
    __shared__ double sh[RAST_CHUNK * 4];
    __shared__ int cnt;
    const int j = blockIdx.x * 32 + (threadIdx.x & 31);
    const int il = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int i = row0 + il;
    const bool in = (il < rows && i < Ny && j < Nx);
    const double x = in ? X[j] : 0.0, y = in ? Y[i] : 0.0;
    const double bx0 = X[blockIdx.x * 32], bx1 = X[min(blockIdx.x * 32 + 31, Nx - 1)];
    const double by0 = Y[min(row0 + blockIdx.y * 8, Ny - 1)], by1 = Y[min(row0 + blockIdx.y * 8 + 7, Ny - 1)];
    double v = 0.0;
    for (int base = 0; base < a.n_walls; base += RAST_CHUNK) {  // simulations.py:538-547
        int n = stage_shapes<4>(a.walls, base, a.n_walls, bx0, bx1, by0, by1, sh, &cnt);
        for (int k = 0; k < n; k++)
            if (fabs(x - sh[4 * k]) < sh[4 * k + 2] / 2 && fabs(y - sh[4 * k + 1]) < sh[4 * k + 3] / 2) v += -1.0;
        __syncthreads();
    }
    for (int base = 0; base < a.n_holes; base += RAST_CHUNK) {  // :549-555
        int n = stage_shapes<4>(a.holes, base, a.n_holes, bx0, bx1, by0, by1, sh, &cnt);
        for (int k = 0; k < n; k++)
            if (fabs(x - sh[4 * k]) < sh[4 * k + 2] / 2 && fabs(y - sh[4 * k + 1]) < sh[4 * k + 3] / 2) v = 0.0;
        __syncthreads();
    }
    for (int base = 0; base < a.n_cyls; base += RAST_CHUNK) {  // :557-563
        int n = stage_shapes<3>(a.cyls, base, a.n_cyls, bx0, bx1, by0, by1, sh, &cnt);
        for (int k = 0; k < n; k++) {
            double ddx = x - sh[3 * k], ddy = y - sh[3 * k + 1];
            if (sqrt(ddx * ddx + ddy * ddy) < sh[3 * k + 2]) v += -1.0;
        }
        __syncthreads();
    }
    if (in && (j == 0 || j == Nx - 1 || i == 0 || i == Ny - 1)) v = -1.0;  // :565-568
    for (int base = 0; base < a.n_targets; base += RAST_CHUNK) {  // :570-574
        int n = stage_shapes<4>(a.targets, base, a.n_targets, bx0, bx1, by0, by1, sh, &cnt);
        for (int k = 0; k < n; k++)
            if (fabs(x - sh[4 * k]) < sh[4 * k + 2] / 2 && fabs(y - sh[4 * k + 1]) < sh[4 * k + 3] / 2) v = 1.0;
        __syncthreads();
    }
    if (!in) return;
    if (a.remap) {  // optimals.py:89-91
        if (v < 0) v = a.wall_value;
        else if (v > 0) v = a.target_value;
    }
    V[(size_t)il * Nx + j] = v;
}
}  // namespace

extern "C" int oc_rasterise(oc_ctx *ctx, const double *walls, int n_walls, const double *holes, int n_holes,
                            const double *cyls, int n_cyls, const double *targets, int n_targets, int remap,
                            double wall_value, double target_value, double *d_V, void *stream) {
    OC_ARG(ctx, "ctx NULL");
    return oc_rasterise_band(ctx, walls, n_walls, holes, n_holes, cyls, n_cyls, targets, n_targets, remap, wall_value,
                             target_value, 0, ctx->Ny, d_V, stream);
}

extern "C" int oc_rasterise_band(oc_ctx *ctx, const double *walls, int n_walls, const double *holes, int n_holes,
                                 const double *cyls, int n_cyls, const double *targets, int n_targets, int remap,
                                 double wall_value, double target_value, int row0, int rows, double *d_V,
                                 void *stream) {
    OC_ARG(ctx && d_V, "ctx/d_V NULL");
    OC_ARG(row0 >= 0 && rows >= 1 && row0 + rows <= ctx->Ny, "row range outside the grid");
    cudaStream_t st = (cudaStream_t)stream;
    OC_CUDA(cudaSetDevice(ctx->device));
    size_t nd = (size_t)4 * n_walls + 4 * n_holes + 3 * n_cyls + 4 * n_targets;
    double *d_sh = nullptr;
    std::vector<double> h(nd ? nd : 1);
    size_t o = 0;
    RastArgs a{};
    if (nd) OC_CUDA(cudaMalloc(&d_sh, nd * sizeof(double)));
    auto put = [&](const double *src, int n, int w, const double *&dst) {
        dst = d_sh + o;
        if (n) memcpy(h.data() + o, src, sizeof(double) * n * w);
        o += (size_t)n * w;
    };
    put(walls, n_walls, 4, a.walls);
    put(holes, n_holes, 4, a.holes);
    put(cyls, n_cyls, 3, a.cyls);
    put(targets, n_targets, 4, a.targets);
    a.n_walls = n_walls; a.n_holes = n_holes; a.n_cyls = n_cyls; a.n_targets = n_targets;
    a.remap = remap; a.wall_value = wall_value; a.target_value = target_value;
    if (nd) OC_CUDA(cudaMemcpyAsync(d_sh, h.data(), nd * sizeof(double), cudaMemcpyHostToDevice, st));
    dim3 grid((ctx->Nx + 31) / 32, (rows + 7) / 8);
    rasterise_kernel<<<grid, 256, 0, st>>>(ctx->d_X, ctx->d_Y, ctx->Ny, ctx->Nx, a, row0, rows, d_V);
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    OC_CUDA(cudaStreamSynchronize(st));  // h / d_sh lifetimes
    if (d_sh) cudaFree(d_sh);
    return OC_OK;
}
