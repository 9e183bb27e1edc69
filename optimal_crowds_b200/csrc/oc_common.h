// oc_common.h -- shared host-side plumbing of liboc_b200.so (context, error text, launch counter).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../include/optimal_crowds.h"

struct oc_ctx {
    int device;
    int Ny, Nx;
    double dx, dy, room_length, room_height;
    double *d_X = nullptr, *d_Y = nullptr;  // linspace node coordinates (device copies)
    std::vector<double> X, Y;               // host copies
    // HJB workspace (lazily allocated, reused across solves)
    double *hjb_ws = nullptr;
    size_t hjb_ws_bytes = 0;
    double *hjb_scratch = nullptr;  // phi slices of the fused step when only velocities are stored
    size_t hjb_scratch_bytes = 0;
    double *hjb_partial = nullptr;  // per-tile error partial sums
    size_t hjb_partial_bytes = 0;
    double *h_pinned = nullptr;  // pinned host scratch (row-group sums, flags)
    size_t h_pinned_bytes = 0;
    // GCFM workspace
    void *gcfm_ws = nullptr;
    size_t gcfm_ws_bytes = 0;
    int gcfm_N = -1, gcfm_nbins = -1, gcfm_nkeys = -1, gcfm_ndoors = -1;  // layout the workspace was carved for
    void *gcfm_pinned = nullptr;
    size_t gcfm_pinned_bytes = 0;
    // row-band (multi-GPU) solver
    void *nccl_comm = nullptr;
    int rank = 0, nranks = 1;
    void *dist_ws = nullptr;
    size_t dist_ws_bytes = 0;
    void *dist_halo = nullptr;      // staging of the deferred phi halo exchange (oc_hjb_dist.cu)
    size_t dist_halo_bytes = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    double gcfm_last_ms = 0.0;
    void *gcfm_stream = nullptr;
    bool gcfm_pending = false;
    void *gcfm_last = nullptr;        // launch state of the step in flight (oc_gcfm.cu: GcfmLaunch), for the slow-path redo
    void *gcfm_glist = nullptr;       // global-memory candidate lists of the exact slow path
    size_t gcfm_glist_bytes = 0;
    int gcfm_tag = 0;                 // generation of the sweep's done-flags (they live in this context's workspace)
    int gcfm_redos = 0;               // slow-path redos of the last step
    long long gcfm_last_pairs = 0;    // interacting pairs evaluated by the last step
    std::vector<char> gcfm_keys_sig;  // batched step: the target-set descriptors last uploaded (KeyDev records + doors)
    void *gcfm_keys_dev = nullptr;    //   and where they were uploaded to
    void *multi_pinned = nullptr, *multi_dev = nullptr;  // batched step: staging arena (perm, noise, member records)
    size_t multi_bytes = 0;
    int gcfm_poll_ns = 100;    // oc_ctx_set_int("gcfm_poll_ns"): back-off between polls of a neighbour's done-flag
    int gcfm_sweep_ctas = 0;  // oc_ctx_set_int("gcfm_sweep_ctas"): cap of the sweep grid (0 = fill the GPU)
    int gcfm_margin_mm = 250;  // oc_ctx_set_int("gcfm_margin_mm"): displacement margin (2 x per-axis bound) of the fast attempt
    int gcfm_margin_hold = 0;  // steps left on the full margin after a step that exceeded the small one
    int gcfm_fov_cull = 1;     // oc_ctx_set_int("gcfm_fov_cull"): drop candidates that cannot enter the field of view
    int gcfm_overlap = 1;      // oc_ctx_set_int("gcfm_overlap"): wall search / sampler on a side stream next to the cell list
    int gcfm_ws_pair = 1;      // oc_ctx_set_int("gcfm_ws_pair"): wall search scans two tiles per memory round trip
    int gcfm_split = 1;        // oc_ctx_set_int("gcfm_split"): two-kernel sweep (candidate lists, then the dependency chain)
    int gcfm_use_graph = 1;    // oc_ctx_set_int("gcfm_graph"): replay the step's launches as one CUDA graph
    cudaStream_t gcfm_side = nullptr, gcfm_side2 = nullptr, gcfm_cap = nullptr;  // side streams of a step, capture stream
    cudaEvent_t gcfm_ev_fork = nullptr, gcfm_ev_join = nullptr, gcfm_ev_join2 = nullptr;
    void *gcfm_stage = nullptr;       // pinned staging of one step's header (tag, simu_step), permutation and normal pairs
    size_t gcfm_stage_bytes = 0;
    cudaGraphExec_t gcfm_graph = nullptr;  // the captured fast attempt of a step ...
    std::vector<char> gcfm_graph_key;      // ... and everything its nodes depend on (pointers, sizes, margin, options)
    int gcfm_graph_launches = 0;           // kernels per replay (launch counter)
    int gcfm_grid_chain = 0, gcfm_grid_sweep = 0, gcfm_grid_sweep_slow = 0;  // resident grids of the sweep kernels on this device
    // in-kernel final reduction of the fused step (oc_hjb_fused.cuh): ticket counters on the device, results in
    // mapped page-locked host memory (slot b: value at [2b], sequence number at [2b+1])
    unsigned *fr_ticket = nullptr;
    double *fr_result = nullptr;
    int fr_slots = 0;
    unsigned long long fr_seq = 0;
    // row-band solve over NVLink peer memory (oc_dist_p2p_*): y, y_new, f, f_new of this rank's band + the inboxes live
    // in ONE cudaMalloc block that the other ranks map through CUDA IPC
    void *p2p_buf = nullptr;
    size_t p2p_bytes = 0, p2p_n_store = 0;
    void *p2p_peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool p2p_on = false;
    unsigned long long p2p_seq = 0;
    // batched (ensemble) HJB solve: per-room workspace, streams and events
    double *batch_ws = nullptr;
    size_t batch_ws_bytes = 0;
    double *batch_pinned = nullptr;
    size_t batch_pinned_bytes = 0;
    std::vector<cudaStream_t> batch_streams;
    std::vector<cudaEvent_t> batch_events;
};

int oc_dist_allreduce_max_u64(oc_ctx *ctx, void *d_buf, size_t count, cudaStream_t st);  // oc_hjb_dist.cu
void oc_gcfm_free_launch_state(oc_ctx *ctx);                                               // oc_gcfm.cu

namespace oc {
void set_error(const char *fmt, ...);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }
}  // namespace oc

#define OC_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            oc::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return OC_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

// Grows a reusable device buffer (or, with `pinned`, page-locked host buffer) to at least `need` bytes.  The old
// buffer is released and forgotten before the new allocation, so after a failed one no freed buffer stays on record.
template <typename T>
inline int oc_ensure_buffer(T *&buf, size_t &bytes, size_t need, bool pinned, const char *what) {
    if (bytes >= need) return OC_OK;
    if (pinned) cudaFreeHost(buf);
    else cudaFree(buf);
    buf = nullptr;
    bytes = 0;
    void *p = nullptr;
    if ((pinned ? cudaMallocHost(&p, need) : cudaMalloc(&p, need)) != cudaSuccess) {
        cudaGetLastError();
        oc::set_error("cannot allocate %zu bytes of %s", need, what);
        return OC_ERR_NOMEM;
    }
    buf = (T *)p;
    bytes = need;
    return OC_OK;
}

#define OC_ARG(cond, msg)                  \
    do {                                   \
        if (!(cond)) {                     \
            oc::set_error("bad argument: %s", msg); \
            return OC_ERR_ARG;             \
        }                                  \
    } while (0)
