// oc_voronoi.cu -- Voronoi density, speed and velocity in the measurement areas (oc_voronoi_acc in
// include/optimal_crowds.h states the rule; tests/voronoi_oracle.py restates it in numpy).  Compile with -fmad=false:
// every formula is evaluated with exactly the operations written here.
//
// One measurement is six launches on the caller's stream:
//   vor_bin      one thread per agent: a generator's bin (index clamped in double) and its place in the bin (atomicAdd,
//                so the order inside a bin is not yet fixed);
//   vor_scan     one block per crowd: bin starts by an exclusive scan; the counts are zeroed for the next measurement;
//   vor_place    one thread per agent: the generators' indices into their bins' slices;
//   vor_sort     one warp per bin: the slice sorted by agent index (rank sort), so that the cell kernel can merge the 3x3
//                bins around an agent in ascending index without a candidate list;
//   vor_cells    one thread per agent in blocks of VO_BLOCK = 256 (part of the summation order, not a tuning parameter):
//                the cell in per-thread local memory (three 64-vertex buffers: the cell, and the two a clip alternates
//                between), its area, its clip by every triangle whose bounding box the cut-off square meets, the five
//                terms per area summed by warp butterflies and warp order into per-block partials;
//   vor_reduce   one block per crowd: the block sums in block order, divided by |A|, written to the step's row.
// The triangles (up to 992, 80 bytes each with their bounding boxes) do not fit in static shared memory; they are read
// from global memory through the read-only cache.  Every thread of a warp reads the same triangle at the same time, so
// a load is one broadcast from L1.  The _multi kernels run a whole ensemble wave: a block finds its member by binary
// search in a member table in device memory, as areas_measure_multi_kernel does.
//
// A frame of the Voronoi maps (oc_vormap_acc) is six launches too: the bin, scan, place and sort kernels above on the
// maps' own scratch, then
//   vor_volume   one thread per agent: |V_i| of every generator into the maps' per-agent buffer (the cell built by
//                cell(), the one copy of rules 2-4 that vor_cells also uses);
//   vormap_node  one thread per node in tiles of 32 x 8, as density_tile: the owner among the generators of the 3x3 bins
//                around the node's bin, the cut-off test and the accumulation.
#include <cmath>
#include <cstdint>
#include <climits>

#include "oc_common.h"

namespace {

constexpr int VO_BLOCK = 256, VO_WARPS = VO_BLOCK / 32, VO_MAX_AREAS = 64, VO_MAX_TRIS = 992, VO_CAP = 64;
constexpr int VO_MAX_BINS_AXIS = 256;          // bins per axis at most (a bin side grows past 2r when the room is long)
constexpr double VO_BIN_MARGIN = 1.0 + 1e-6;   // bin side >= 2r * margin: rounding in x / side cannot skip a bin
constexpr int VO_SORT_WARPS = 8;               // bins per block of vor_sort

struct VorMember {
    const double *x, *y, *vx, *vy;
    const uint8_t *status;
    const double *ring, *tris, *info;
    const int *toff;
    int *count, *start, *slot, *order;
    double *partials, *row;
    double *vol;                // per-agent cell areas of the maps (oc_vormap_acc), NULL for the areas' measures
    double r, L, H, sx, sy;     // cut-off, room, bin sides
    int N, edges, na, bx, by;
    int blk0, bin0, pad_;       // first agent block and first sort block of the member in a batched launch
};

__device__ __forceinline__ bool generator(const VorMember &m, int i) {
    return m.status[i] == 1 && isfinite(m.x[i]) && isfinite(m.y[i]);
}
__device__ __forceinline__ int bin_axis(double v, double side, int nb) {
    return (int)fmin(fmax(floor(v / side), 0.0), (double)(nb - 1));
}

// one Sutherland-Hodgman pass keeping s <= 0; returns the vertex count (0: empty), or -1 when the output would exceed
// VO_CAP vertices
template <class S>
__device__ __forceinline__ int vclip(const double2 *in, int n, double2 *out, S s) {
    if (n < 3) return n < 0 ? n : 0;
    int m = 0;
    const double2 p0 = in[0];
    const double s0 = s(p0);
    double2 a = p0;
    double sa = s0;
    for (int k = 0; k < n; k++) {
        const bool last = k + 1 == n;
        const double2 b = last ? p0 : in[k + 1];
        const double sb = last ? s0 : s(b);
        if (sa <= 0) {
            if (m == VO_CAP) return -1;
            out[m++] = a;
        }
        if ((sa <= 0) != (sb <= 0)) {
            if (m == VO_CAP) return -1;
            const double t = sa / (sa - sb);
            out[m++] = make_double2(a.x + t * (b.x - a.x), a.y + t * (b.y - a.y));
        }
        a = b;
        sa = sb;
    }
    return m < 3 ? 0 : m;
}
__device__ __forceinline__ double shoelace(const double2 *p, int n) {
    double s = 0.0;
    for (int k = 0; k < n; k++) {
        const double2 a = p[k], b = p[k + 1 == n ? 0 : k + 1];
        s += a.x * b.y - b.x * a.y;
    }
    return 0.5 * s;
}
__device__ __forceinline__ double warp_butterfly(double v) {
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// ---------------------------------------------------------------------------------------------------- neighbour bins
__device__ __forceinline__ void bin_agent(const VorMember &m, int i) {
    if (i >= m.N) return;
    int b = -1, s = 0;
    if (generator(m, i)) {
        b = bin_axis(m.y[i], m.sy, m.by) * m.bx + bin_axis(m.x[i], m.sx, m.bx);
        s = atomicAdd(m.count + b, 1);
    }
    m.slot[2 * i] = b;
    m.slot[2 * i + 1] = s;
}
// exclusive scan of the bx*by counts into start[0 .. bx*by] (one block of 1024 threads), counts zeroed
__device__ __forceinline__ void scan_bins(const VorMember &m) {
    __shared__ int wsum[32];
    __shared__ int carry;
    const int nb = m.bx * m.by, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nb; base += 1024) {
        const int t = base + threadIdx.x;
        const int c = t < nb ? m.count[t] : 0;
        int v = c;
        for (int off = 1; off < 32; off <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, v, off);
            if (lane >= off) v += u;
        }
        if (lane == 31) wsum[wid] = v;
        __syncthreads();
        if (wid == 0) {
            int w = wsum[lane];
            for (int off = 1; off < 32; off <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, w, off);
                if (lane >= off) w += u;
            }
            wsum[lane] = w;
        }
        __syncthreads();
        const int incl = v + (wid ? wsum[wid - 1] : 0) + carry;
        if (t < nb) {
            m.start[t] = incl - c;
            m.count[t] = 0;
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) m.start[nb] = carry;
}
__device__ __forceinline__ void place_agent(const VorMember &m, int i) {
    if (i >= m.N) return;
    const int b = m.slot[2 * i];
    if (b >= 0) m.order[m.start[b] + m.slot[2 * i + 1]] = i;
}
// warp `w` of the sort blocks: bin b's slice of order (unsorted) into order + N (sorted), by rank
__device__ __forceinline__ void sort_bin(const VorMember &m, int b) {
    if (b >= m.bx * m.by) return;
    const int lane = threadIdx.x & 31, s0 = m.start[b], n = m.start[b + 1] - s0;
    const int *in = m.order + s0;
    int *out = m.order + m.N + s0;
    for (int e = lane; e < n; e += 32) {
        const int v = in[e];
        int rank = 0;
        for (int f = 0; f < n; f++) rank += in[f] < v;
        out[rank] = v;
    }
}

// ---------------------------------------------------------------------------------------------------- cells
// The cell V_i of generator i at (x, y), rules 2-4 of oc_voronoi_acc: the cut-off polygon, clipped by the room, then by
// the generators of the 3x3 bins around i's bin merged in ascending index.  cur and tmp point at the thread's two VO_CAP
// buffers; on return cur holds the cell and tmp is free.  Returns its vertex count: 0 empty, -1 overflowed.
__device__ __forceinline__ int cell(const VorMember &m, int i, double x, double y, double2 *&cur, double2 *&tmp) {
    const double r = m.r;
    double2 *A = cur, *B = tmp;
    for (int k = 0; k < m.edges; k++) A[k] = make_double2(x + __ldg(m.ring + 2 * k), y + __ldg(m.ring + 2 * k + 1));
    const double L = m.L, H = m.H;
    int n = vclip(A, m.edges, B, [](double2 p) { return -p.x; });
    n = vclip(B, n, A, [L](double2 p) { return p.x - L; });
    n = vclip(A, n, B, [](double2 p) { return -p.y; });
    n = vclip(B, n, A, [H](double2 p) { return p.y - H; });
    // the 3x3 bins around i's bin, merged in ascending agent index
    const int cx = bin_axis(x, m.sx, m.bx), cy = bin_axis(y, m.sy, m.by);
    const int *sorted = m.order + m.N;
    int ptr[9], end[9], head[9], nq = 0;
    for (int yy = max(cy - 1, 0); yy <= min(cy + 1, m.by - 1); yy++)
        for (int xx = max(cx - 1, 0); xx <= min(cx + 1, m.bx - 1); xx++) {
            const int b = yy * m.bx + xx;
            ptr[nq] = m.start[b];
            end[nq] = m.start[b + 1];
            head[nq] = ptr[nq] < end[nq] ? sorted[ptr[nq]] : INT_MAX;
            nq++;
        }
    const double d2 = (2.0 * r) * (2.0 * r);
    while (n > 0) {
        int q = 0;
        for (int k = 1; k < nq; k++)
            if (head[k] < head[q]) q = k;
        const int j = head[q];
        if (j == INT_MAX) break;
        ptr[q]++;
        head[q] = ptr[q] < end[q] ? sorted[ptr[q]] : INT_MAX;
        if (j == i) continue;
        const double xj = m.x[j], yj = m.y[j];
        const double dx = xj - x, dy = yj - y;
        if (!(dx * dx + dy * dy <= d2) || (dx == 0 && dy == 0)) continue;
        const double mx = 0.5 * (x + xj), my = 0.5 * (y + yj);
        n = vclip(cur, n, tmp, [dx, dy, mx, my](double2 p) { return dx * (p.x - mx) + dy * (p.y - my); });
        double2 *t = cur; cur = tmp; tmp = t;
    }
    return n;
}

// The five terms of agent i for every area, summed over block `blk` into partials (blk, na, 5).
__device__ __forceinline__ void cells_block(const VorMember &m, int blk) {
    __shared__ double W[VO_WARPS][VO_MAX_AREAS][5];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int i = blk * VO_BLOCK + threadIdx.x;
    const double r = m.r;
    double2 A[VO_CAP], B[VO_CAP], C[VO_CAP];
    double2 *cur = A, *tmp = B;
    int n = 0;                    // cell vertices: 0 empty, -1 overflowed
    double x = 0.0, y = 0.0, u = 0.0, v = 0.0, sp = 0.0, vol = 0.0;
    bool live = false;            // a generator whose square meets some area's bounding box
    if (i < m.N && generator(m, i)) {
        x = m.x[i]; y = m.y[i];
        const double xl = x - r, xh = x + r, yl = y - r, yh = y + r;
        for (int a = 0; a < m.na && !live; a++) {
            const double *bb = m.info + 5 * a;
            live = xl <= __ldg(bb + 1) && xh >= __ldg(bb) && yl <= __ldg(bb + 3) && yh >= __ldg(bb + 2);
        }
    }
    if (live) {
        u = m.vx[i]; v = m.vy[i];
        sp = sqrt(u * u + v * v);
        n = cell(m, i, x, y, cur, tmp);
        vol = n < 0 ? NAN : shoelace(cur, n);
        live = n < 0 || vol > 0;
    }
    for (int a = 0; a < m.na; a++) {
        double w = 0.0;
        if (live) {
            const double *bb = m.info + 5 * a;
            const double xl = x - r, xh = x + r, yl = y - r, yh = y + r;
            if (xl <= __ldg(bb + 1) && xh >= __ldg(bb) && yl <= __ldg(bb + 3) && yh >= __ldg(bb + 2)) {
                for (int t = __ldg(m.toff + a), t1 = __ldg(m.toff + a + 1); t < t1; t++) {
                    const double *T = m.tris + 10 * t;
                    if (!(xl <= __ldg(T + 7) && xh >= __ldg(T + 6) && yl <= __ldg(T + 9) && yh >= __ldg(T + 8))) continue;
                    if (n < 0) {
                        w = NAN;
                        break;
                    }
                    const double ax = __ldg(T), ay = __ldg(T + 1), bx = __ldg(T + 2), by = __ldg(T + 3);
                    const double qx = __ldg(T + 4), qy = __ldg(T + 5);
                    int k = vclip(cur, n, tmp, [=](double2 p) { return -((bx - ax) * (p.y - ay) - (by - ay) * (p.x - ax)); });
                    k = vclip(tmp, k, C, [=](double2 p) { return -((qx - bx) * (p.y - by) - (qy - by) * (p.x - bx)); });
                    k = vclip(C, k, tmp, [=](double2 p) { return -((ax - qx) * (p.y - qy) - (ay - qy) * (p.x - qx)); });
                    w += k < 0 ? NAN : shoelace(tmp, k);
                }
            }
        }
        const bool any = !(w == 0.0);
        double t5[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
        if (any) {
            t5[0] = w / vol; t5[1] = w * sp; t5[2] = w * u; t5[3] = w * v; t5[4] = w;
        }
        if (__ballot_sync(0xffffffffu, any)) {   // (warp-uniform: a warp of +0.0 terms sums to +0.0)
            for (int q = 0; q < 5; q++) t5[q] = warp_butterfly(t5[q]);
        }
        if (lane == 0)
            for (int q = 0; q < 5; q++) W[wid][a][q] = t5[q];
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 5 * m.na; t += VO_BLOCK) {
        const int a = t / 5, q = t % 5;
        double s = 0.0;
        for (int k = 0; k < VO_WARPS; k++) s += W[k][a][q];
        m.partials[((size_t)blk * m.na + a) * 5 + q] = s;
    }
}
// the row of a crowd of N agents from its block sums
__device__ __forceinline__ void reduce_rows(const VorMember &m) {
    const int nb = (m.N + VO_BLOCK - 1) / VO_BLOCK;
    for (int t = threadIdx.x; t < 5 * m.na; t += blockDim.x) {
        const int a = t / 5, q = t % 5;
        double s = 0.0;
        for (int b = 0; b < nb; b++) s += m.partials[((size_t)b * m.na + a) * 5 + q];
        m.row[t] = s / m.info[5 * a + 4];
    }
}

// ---------------------------------------------------------------------------------------------------- maps
// Voronoi maps (oc_vormap_acc): |V_i| of every agent into m.vol (0.0 for non-generators, NaN for overflowed cells), then
// per node the owner among the generators of the 3x3 bins around the node's bin and the accumulation of rules 3-6.
constexpr int VM_TX = 32, VM_TY = 8;   // nodes per tile of the node kernel: a warp is 32 nodes of one row

__device__ __forceinline__ void volume_agent(const VorMember &m, int i) {
    if (i >= m.N) return;
    double vol = 0.0;
    if (generator(m, i)) {
        double2 A[VO_CAP], B[VO_CAP];
        double2 *cur = A, *tmp = B;
        const int n = cell(m, i, m.x[i], m.y[i], cur, tmp);
        vol = n < 0 ? NAN : shoelace(cur, n);
    }
    m.vol[i] = vol;
}

struct VorMapMember {
    const double *x, *y, *vx, *vy, *vol, *ring, *X, *Y, *Vg;
    const int *start, *order;
    double *dsum, *dmax, *ssum, *vxsum, *vysum;
    int *cov;
    double r, sx, sy;
    int N, edges, bx, by, Ny, Nx, ntx, tile0;
};

// tile (tx, ty) of VM_TX x VM_TY nodes.  The warp's 32 nodes lie in one row and mostly in one bin, so the candidates'
// loads are broadcasts; no staging in shared memory.
__device__ __forceinline__ void vormap_tile(const VorMapMember &m, int tx, int ty) {
    __shared__ double2 ring[32];
    for (int k = threadIdx.x; k < m.edges; k += blockDim.x) ring[k] = make_double2(m.ring[2 * k], m.ring[2 * k + 1]);
    __syncthreads();
    const int ix = tx * VM_TX + (threadIdx.x & 31), iy = ty * VM_TY + (threadIdx.x >> 5);
    if (ix >= m.Nx || iy >= m.Ny) return;
    const size_t g = (size_t)iy * m.Nx + ix;
    int owner = -1;
    if (!(m.Vg[g] < 0) && m.N > 0) {
        // rule 3: the nearest generator within r, the lowest index on ties
        const double X = m.X[ix], Y = m.Y[iy], rr = m.r * m.r;
        const int cx = bin_axis(X, m.sx, m.bx), cy = bin_axis(Y, m.sy, m.by);
        const int *sorted = m.order + m.N;
        double best = 0.0;
        for (int yy = max(cy - 1, 0); yy <= min(cy + 1, m.by - 1); yy++)
            for (int xx = max(cx - 1, 0); xx <= min(cx + 1, m.bx - 1); xx++) {
                const int b = yy * m.bx + xx;
                for (int e = m.start[b], e1 = m.start[b + 1]; e < e1; e++) {
                    const int j = sorted[e];
                    const double dx = X - m.x[j], dy = Y - m.y[j];
                    const double d2 = dx * dx + dy * dy;
                    if (d2 <= rr && (owner < 0 || d2 < best || (d2 == best && j < owner))) {
                        best = d2;
                        owner = j;
                    }
                }
            }
        // rule 4: inside the owner's cut-off polygon
        if (owner >= 0) {
            const double xi = m.x[owner], yi = m.y[owner];
            for (int k = 0; k < m.edges; k++) {
                const double2 a = ring[k], b = ring[k + 1 == m.edges ? 0 : k + 1];
                const double ax = xi + a.x, ay = yi + a.y, bx = xi + b.x, by = yi + b.y;
                if (!((bx - ax) * (Y - ay) - (by - ay) * (X - ax) >= 0)) {
                    owner = -1;
                    break;
                }
            }
        }
    }
    // rules 5 and 6 (each term is added as soon as it is known: fewer values live across the division and the square
    // root, whose slow paths are calls)
    const double vol = owner >= 0 ? m.vol[owner] : 0.0;
    const bool nan = vol != vol;
    if (!nan && !(vol > 0)) {                   // uncovered: d_density_max = np.maximum(d_density_max, 0.0)
        if (0.0 > m.dmax[g]) m.dmax[g] = 0.0;   // (it changes only where it is below 0)
        return;
    }
    const double rho = nan ? NAN : 1.0 / vol;
    m.dsum[g] = m.dsum[g] + rho;
    const double mx = m.dmax[g];
    m.dmax[g] = (mx != mx) ? mx : ((rho != rho || rho > mx) ? rho : mx);   // np.maximum(mx, rho): the first NaN wins
    m.cov[g] += 1;
    const double u = nan ? NAN : m.vx[owner], v = nan ? NAN : m.vy[owner];
    m.vxsum[g] = m.vxsum[g] + u;
    m.vysum[g] = m.vysum[g] + v;
    const double s = nan ? NAN : sqrt(u * u + v * v);
    m.ssum[g] = m.ssum[g] + s;
}

__global__ void __launch_bounds__(VO_BLOCK) vor_volume_kernel(VorMember m) { volume_agent(m, blockIdx.x * VO_BLOCK + threadIdx.x); }
__global__ void __launch_bounds__(VM_TX * VM_TY) vormap_node_kernel(VorMapMember m) {
    vormap_tile(m, blockIdx.x, blockIdx.y);
}

__global__ void __launch_bounds__(VO_BLOCK) vor_bin_kernel(VorMember m) { bin_agent(m, blockIdx.x * VO_BLOCK + threadIdx.x); }
__global__ void __launch_bounds__(1024) vor_scan_kernel(VorMember m) { scan_bins(m); }
__global__ void __launch_bounds__(VO_BLOCK) vor_place_kernel(VorMember m) { place_agent(m, blockIdx.x * VO_BLOCK + threadIdx.x); }
__global__ void __launch_bounds__(VO_SORT_WARPS * 32) vor_sort_kernel(VorMember m) {
    sort_bin(m, blockIdx.x * VO_SORT_WARPS + (threadIdx.x >> 5));
}
__global__ void __launch_bounds__(VO_BLOCK) vor_cells_kernel(VorMember m) { cells_block(m, blockIdx.x); }
__global__ void __launch_bounds__(256) vor_reduce_kernel(VorMember m) { reduce_rows(m); }

// batched: the member owning block b of a launch whose members start at blocks first(m) (non-decreasing)
template <bool BINS>
__device__ __forceinline__ int member_of(const VorMember *__restrict__ ms, int n, int b) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((BINS ? ms[mid].bin0 : ms[mid].blk0) <= b) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}
__global__ void __launch_bounds__(VO_BLOCK) vor_bin_multi_kernel(const VorMember *__restrict__ ms, int n) {
    const VorMember &m = ms[member_of<false>(ms, n, blockIdx.x)];
    bin_agent(m, (blockIdx.x - m.blk0) * VO_BLOCK + threadIdx.x);
}
__global__ void __launch_bounds__(1024) vor_scan_multi_kernel(const VorMember *__restrict__ ms) { scan_bins(ms[blockIdx.x]); }
__global__ void __launch_bounds__(VO_BLOCK) vor_place_multi_kernel(const VorMember *__restrict__ ms, int n) {
    const VorMember &m = ms[member_of<false>(ms, n, blockIdx.x)];
    place_agent(m, (blockIdx.x - m.blk0) * VO_BLOCK + threadIdx.x);
}
__global__ void __launch_bounds__(VO_SORT_WARPS * 32) vor_sort_multi_kernel(const VorMember *__restrict__ ms, int n) {
    const VorMember &m = ms[member_of<true>(ms, n, blockIdx.x)];
    sort_bin(m, (blockIdx.x - m.bin0) * VO_SORT_WARPS + (threadIdx.x >> 5));
}
__global__ void __launch_bounds__(VO_BLOCK) vor_cells_multi_kernel(const VorMember *__restrict__ ms, int n) {
    const VorMember &m = ms[member_of<false>(ms, n, blockIdx.x)];
    cells_block(m, blockIdx.x - m.blk0);
}
__global__ void __launch_bounds__(256) vor_reduce_multi_kernel(const VorMember *__restrict__ ms) { reduce_rows(ms[blockIdx.x]); }

__global__ void __launch_bounds__(VO_BLOCK) vor_volume_multi_kernel(const VorMember *__restrict__ ms, int n) {
    const VorMember &m = ms[member_of<false>(ms, n, blockIdx.x)];
    volume_agent(m, (blockIdx.x - m.blk0) * VO_BLOCK + threadIdx.x);
}
__global__ void __launch_bounds__(VM_TX * VM_TY) vormap_node_multi_kernel(const VorMapMember *__restrict__ ms, int n) {
    const int b = blockIdx.x;
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (ms[mid].tile0 <= b) lo = mid;
        else hi = mid - 1;
    }
    const VorMapMember &m = ms[lo];
    const int t = b - m.tile0;
    vormap_tile(m, t % m.ntx, t / m.ntx);
}

int args_check(const oc_ctx *ctx, const oc_voronoi_acc *a, int N, bool ptrs, int step) {
    if (int rc = oc_voronoi_check(ctx, a, N)) return rc;
    OC_ARG(N == 0 || ptrs, "NULL argument");
    OC_ARG(step >= 0 && step < a->capacity, "Voronoi measures: step beyond the row capacity");
    return OC_OK;
}

VorMember member(const oc_ctx *ctx, const oc_voronoi_acc *a, int N, const double *x, const double *y, const double *vx,
                 const double *vy, const uint8_t *status, int step) {
    VorMember m{};
    m.x = x; m.y = y; m.vx = vx; m.vy = vy; m.status = status;
    m.ring = a->d_ring; m.tris = a->d_tris; m.info = a->d_area_info; m.toff = a->d_tri_offsets;
    m.count = a->d_bin_count; m.start = a->d_bin_start; m.slot = a->d_slot; m.order = a->d_order;
    m.partials = a->d_partials;
    m.row = a->d_rows + (size_t)step * a->n_areas * 5;
    m.r = a->cutoff; m.L = ctx->room_length; m.H = ctx->room_height;
    m.sx = ctx->room_length / a->bins_x; m.sy = ctx->room_height / a->bins_y;
    m.N = N; m.edges = a->edges; m.na = a->n_areas; m.bx = a->bins_x; m.by = a->bins_y;
    return m;
}

VorMember map_member(const oc_ctx *ctx, const oc_vormap_acc *a, int N, const double *x, const double *y,
                     const double *vx, const double *vy, const uint8_t *status) {
    VorMember m{};
    m.x = x; m.y = y; m.vx = vx; m.vy = vy; m.status = status;
    m.ring = a->d_ring;
    m.count = a->d_bin_count; m.start = a->d_bin_start; m.slot = a->d_slot; m.order = a->d_order;
    m.vol = a->d_vol;
    m.r = a->cutoff; m.L = ctx->room_length; m.H = ctx->room_height;
    m.sx = ctx->room_length / a->bins_x; m.sy = ctx->room_height / a->bins_y;
    m.N = N; m.edges = a->edges; m.bx = a->bins_x; m.by = a->bins_y;
    return m;
}
VorMapMember node_member(const oc_ctx *ctx, const oc_vormap_acc *a, const VorMember &c) {
    return VorMapMember{c.x, c.y, c.vx, c.vy, a->d_vol, a->d_ring, ctx->d_X, ctx->d_Y, a->d_Vglobal, a->d_bin_start,
                        a->d_order, a->d_density_sum, a->d_density_max, a->d_speed_sum, a->d_vx_sum, a->d_vy_sum,
                        a->d_covered, c.r, c.sx, c.sy, c.N, c.edges, c.bx, c.by, ctx->Ny, ctx->Nx,
                        (ctx->Nx + VM_TX - 1) / VM_TX, 0};
}

bool bins_cover(double len, int nb, double r) { return nb == 1 || len / nb >= 2.0 * r * VO_BIN_MARGIN; }

}  // namespace

int oc_voronoi_check(const oc_ctx *ctx, const oc_voronoi_acc *a, int N) {
    OC_ARG(ctx && a && a->d_ring && a->d_tris && a->d_area_info && a->tri_offsets && a->d_tri_offsets &&
           a->d_bin_count && a->d_bin_start && a->d_slot && a->d_order && a->d_partials && a->d_rows, "NULL argument");
    OC_ARG(std::isfinite(a->cutoff) && a->cutoff > 0 && a->cutoff <= 100, "Voronoi measures: cutoff must be in (0, 100]");
    OC_ARG(a->edges >= 4 && a->edges <= 32, "Voronoi measures: edges must be in 4..32");
    OC_ARG(a->n_areas >= 1 && a->n_areas <= VO_MAX_AREAS, "Voronoi measures: n_areas must be in 1..64");
    OC_ARG(a->tri_offsets[0] == 0, "Voronoi measures: triangle offsets must start at 0");
    for (int k = 0; k < a->n_areas; k++)
        OC_ARG(a->tri_offsets[k + 1] > a->tri_offsets[k] && a->tri_offsets[k + 1] <= VO_MAX_TRIS,
               "Voronoi measures: every area needs triangles, 992 in all at most");
    OC_ARG(a->bins_x >= 1 && a->bins_y >= 1 && a->bins_x <= VO_MAX_BINS_AXIS && a->bins_y <= VO_MAX_BINS_AXIS &&
           a->bin_capacity >= a->bins_x * a->bins_y + 1, "Voronoi measures: bad bin grid");
    OC_ARG(bins_cover(ctx->room_length, a->bins_x, a->cutoff) && bins_cover(ctx->room_height, a->bins_y, a->cutoff),
           "Voronoi measures: bins narrower than twice the cutoff");
    OC_ARG(N >= 0 && N <= a->agent_capacity, "Voronoi measures: too small an agent capacity for N");
    OC_ARG((N + VO_BLOCK - 1) / VO_BLOCK <= a->partial_blocks, "Voronoi measures: too few partial blocks for N");
    OC_ARG(a->capacity >= 0, "Voronoi measures: negative capacity");
    return OC_OK;
}

int oc_voronoi_enqueue(oc_ctx *ctx, const oc_voronoi_acc *a, int N, const double *d_x, const double *d_y,
                       const double *d_vx, const double *d_vy, const uint8_t *d_status, int step, cudaStream_t st) {
    OC_CUDA(cudaSetDevice(ctx->device));
    const VorMember m = member(ctx, a, N, d_x, d_y, d_vx, d_vy, d_status, step);
    const int nb = (N + VO_BLOCK - 1) / VO_BLOCK;
    if (nb) {
        vor_bin_kernel<<<nb, VO_BLOCK, 0, st>>>(m);
        vor_scan_kernel<<<1, 1024, 0, st>>>(m);
        vor_place_kernel<<<nb, VO_BLOCK, 0, st>>>(m);
        vor_sort_kernel<<<(m.bx * m.by + VO_SORT_WARPS - 1) / VO_SORT_WARPS, VO_SORT_WARPS * 32, 0, st>>>(m);
        vor_cells_kernel<<<nb, VO_BLOCK, 0, st>>>(m);
        oc::count_launch(5);
    }
    vor_reduce_kernel<<<1, 256, 0, st>>>(m);
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}

extern "C" int oc_voronoi_measure(oc_ctx *ctx, const oc_voronoi_acc *acc, int N, const double *d_x, const double *d_y,
                                  const double *d_vx, const double *d_vy, const uint8_t *d_status, int step,
                                  void *stream) {
    if (int rc = args_check(ctx, acc, N, d_x && d_y && d_vx && d_vy && d_status, step)) return rc;
    return oc_voronoi_enqueue(ctx, acc, N, d_x, d_y, d_vx, d_vy, d_status, step, (cudaStream_t)stream);
}

extern "C" int oc_voronoi_measure_multi(int n, oc_ctx *const *ctxs, const oc_voronoi_acc *const *accs, const int *Ns,
                                        const double *const *x, const double *const *y, const double *const *vx,
                                        const double *const *vy, const uint8_t *const *status, const int *steps,
                                        void *stream) {
    OC_ARG(n >= 1 && ctxs && accs && Ns && x && y && vx && vy && status && steps && ctxs[0], "NULL argument");
    oc_ctx *c0 = ctxs[0];
    for (int q = 0; q < n; q++) {
        OC_ARG(ctxs[q], "NULL argument");
        OC_ARG(ctxs[q]->device == c0->device, "Voronoi measures: member context on another device");
        if (int rc = args_check(ctxs[q], accs[q], Ns[q], x[q] && y[q] && vx[q] && vy[q] && status[q], steps[q]))
            return rc;
        // the members' launches run concurrently: no two may share bins or scratch
        for (int p = 0; p < q; p++)
            OC_ARG(accs[p]->d_bin_count != accs[q]->d_bin_count && accs[p]->d_bin_start != accs[q]->d_bin_start &&
                   accs[p]->d_slot != accs[q]->d_slot && accs[p]->d_order != accs[q]->d_order &&
                   accs[p]->d_partials != accs[q]->d_partials, "Voronoi measures: members share bins or scratch");
    }
    OC_CUDA(cudaSetDevice(c0->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = sizeof(VorMember) * (size_t)n;
    // the table (staging and device copy) is reused once the previous call's kernels have read it, whatever its stream
    if (!c0->vor_ev) OC_CUDA(cudaEventCreateWithFlags(&c0->vor_ev, cudaEventDisableTiming));
    OC_CUDA(cudaEventSynchronize(c0->vor_ev));
    if (int rc = oc_ensure_buffer(c0->vor_pinned, c0->vor_pinned_bytes, bytes, true, "Voronoi member table")) return rc;
    if (int rc = oc_ensure_buffer(c0->vor_dev, c0->vor_dev_bytes, bytes, false, "Voronoi member table")) return rc;
    VorMember *recs = static_cast<VorMember *>(c0->vor_pinned);
    long long blocks = 0, sort_blocks = 0;
    for (int q = 0; q < n; q++) {
        recs[q] = member(ctxs[q], accs[q], Ns[q], x[q], y[q], vx[q], vy[q], status[q], steps[q]);
        recs[q].blk0 = (int)blocks;
        recs[q].bin0 = (int)sort_blocks;
        blocks += (Ns[q] + VO_BLOCK - 1) / VO_BLOCK;
        if (Ns[q]) sort_blocks += (recs[q].bx * recs[q].by + VO_SORT_WARPS - 1) / VO_SORT_WARPS;
        OC_ARG(blocks < 0x7fffffff && sort_blocks < 0x7fffffff, "Voronoi measures: too many agents for one launch");
    }
    OC_CUDA(cudaMemcpyAsync(c0->vor_dev, recs, bytes, cudaMemcpyHostToDevice, st));
    const VorMember *dev = static_cast<const VorMember *>(c0->vor_dev);
    if (blocks) {
        vor_bin_multi_kernel<<<(unsigned)blocks, VO_BLOCK, 0, st>>>(dev, n);
        vor_scan_multi_kernel<<<n, 1024, 0, st>>>(dev);
        vor_place_multi_kernel<<<(unsigned)blocks, VO_BLOCK, 0, st>>>(dev, n);
        vor_sort_multi_kernel<<<(unsigned)sort_blocks, VO_SORT_WARPS * 32, 0, st>>>(dev, n);
        vor_cells_multi_kernel<<<(unsigned)blocks, VO_BLOCK, 0, st>>>(dev, n);
        oc::count_launch(5);
    }
    vor_reduce_multi_kernel<<<n, 256, 0, st>>>(dev);
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    OC_CUDA(cudaEventRecord(c0->vor_ev, st));
    return OC_OK;
}

// ------------------------------------------------------------------------------------------------ Voronoi maps
int oc_vormap_check(const oc_ctx *ctx, const oc_vormap_acc *a, int N) {
    OC_ARG(ctx && a && a->d_density_sum && a->d_density_max && a->d_covered && a->d_speed_sum && a->d_vx_sum &&
           a->d_vy_sum && a->d_Vglobal && a->d_ring && a->d_bin_count && a->d_bin_start && a->d_slot && a->d_order &&
           a->d_vol, "NULL argument");
    OC_ARG(std::isfinite(a->cutoff) && a->cutoff > 0 && a->cutoff <= 100, "Voronoi maps: cutoff must be in (0, 100]");
    OC_ARG(a->edges >= 4 && a->edges <= 32, "Voronoi maps: edges must be in 4..32");
    OC_ARG(a->every >= 1, "Voronoi maps: every must be >= 1");
    OC_ARG(a->bins_x >= 1 && a->bins_y >= 1 && a->bins_x <= VO_MAX_BINS_AXIS && a->bins_y <= VO_MAX_BINS_AXIS &&
           a->bin_capacity >= a->bins_x * a->bins_y + 1, "Voronoi maps: bad bin grid");
    OC_ARG(bins_cover(ctx->room_length, a->bins_x, a->cutoff) && bins_cover(ctx->room_height, a->bins_y, a->cutoff),
           "Voronoi maps: bins narrower than twice the cutoff");
    OC_ARG(N >= 0 && N <= a->agent_capacity, "Voronoi maps: too small an agent capacity for N");
    return OC_OK;
}

int oc_vormap_enqueue(oc_ctx *ctx, const oc_vormap_acc *a, int N, const double *d_x, const double *d_y,
                      const double *d_vx, const double *d_vy, const uint8_t *d_status, cudaStream_t st) {
    OC_CUDA(cudaSetDevice(ctx->device));
    const VorMember m = map_member(ctx, a, N, d_x, d_y, d_vx, d_vy, d_status);
    const int nb = (N + VO_BLOCK - 1) / VO_BLOCK;
    if (nb) {
        vor_bin_kernel<<<nb, VO_BLOCK, 0, st>>>(m);
        vor_scan_kernel<<<1, 1024, 0, st>>>(m);
        vor_place_kernel<<<nb, VO_BLOCK, 0, st>>>(m);
        vor_sort_kernel<<<(m.bx * m.by + VO_SORT_WARPS - 1) / VO_SORT_WARPS, VO_SORT_WARPS * 32, 0, st>>>(m);
        vor_volume_kernel<<<nb, VO_BLOCK, 0, st>>>(m);
        oc::count_launch(5);
    }
    const dim3 grid((ctx->Nx + VM_TX - 1) / VM_TX, (ctx->Ny + VM_TY - 1) / VM_TY);
    vormap_node_kernel<<<grid, VM_TX * VM_TY, 0, st>>>(node_member(ctx, a, m));
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    return OC_OK;
}

extern "C" int oc_vormap_accum(oc_ctx *ctx, const oc_vormap_acc *acc, int N, const double *d_x, const double *d_y,
                               const double *d_vx, const double *d_vy, const uint8_t *d_status, void *stream) {
    if (int rc = oc_vormap_check(ctx, acc, N)) return rc;
    OC_ARG(N == 0 || (d_x && d_y && d_vx && d_vy && d_status), "NULL argument");
    return oc_vormap_enqueue(ctx, acc, N, d_x, d_y, d_vx, d_vy, d_status, (cudaStream_t)stream);
}

// One frame per member: the five per-agent launches over the members' agent blocks (the VorMember table) and one node
// launch over their tiles (the VorMapMember table after it).  Members may differ in grid shape, crowd size, cutoff,
// edges and bins.
extern "C" int oc_vormap_accum_multi(int n, oc_ctx *const *ctxs, const oc_vormap_acc *const *accs, const int *Ns,
                                     const double *const *x, const double *const *y, const double *const *vx,
                                     const double *const *vy, const uint8_t *const *status, void *stream) {
    OC_ARG(n >= 1 && ctxs && accs && Ns && x && y && vx && vy && status && ctxs[0], "NULL argument");
    oc_ctx *c0 = ctxs[0];
    for (int q = 0; q < n; q++) {
        OC_ARG(ctxs[q] && accs[q], "NULL argument");
        OC_ARG(ctxs[q]->device == c0->device, "Voronoi maps: member context on another device");
        if (int rc = oc_vormap_check(ctxs[q], accs[q], Ns[q])) return rc;
        OC_ARG(Ns[q] == 0 || (x[q] && y[q] && vx[q] && vy[q] && status[q]), "NULL argument");
        // the members run concurrently: no two may share bins, scratch or accumulators
        const oc_vormap_acc *b = accs[q];
        for (int p = 0; p < q; p++) {
            const oc_vormap_acc *a = accs[p];
            OC_ARG(a->d_bin_count != b->d_bin_count && a->d_bin_start != b->d_bin_start && a->d_slot != b->d_slot &&
                   a->d_order != b->d_order && a->d_vol != b->d_vol && a->d_density_sum != b->d_density_sum &&
                   a->d_density_max != b->d_density_max && a->d_covered != b->d_covered &&
                   a->d_speed_sum != b->d_speed_sum && a->d_vx_sum != b->d_vx_sum && a->d_vy_sum != b->d_vy_sum,
                   "Voronoi maps: members share bins, scratch or accumulators");
        }
    }
    OC_CUDA(cudaSetDevice(c0->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = (sizeof(VorMember) + sizeof(VorMapMember)) * (size_t)n;
    // the tables (staging and device copy) are reused once the previous call's kernels have read them
    if (!c0->vmap_ev) OC_CUDA(cudaEventCreateWithFlags(&c0->vmap_ev, cudaEventDisableTiming));
    OC_CUDA(cudaEventSynchronize(c0->vmap_ev));
    if (int rc = oc_ensure_buffer(c0->vmap_pinned, c0->vmap_pinned_bytes, bytes, true, "Voronoi map member table"))
        return rc;
    if (int rc = oc_ensure_buffer(c0->vmap_dev, c0->vmap_dev_bytes, bytes, false, "Voronoi map member table"))
        return rc;
    VorMember *recs = static_cast<VorMember *>(c0->vmap_pinned);
    VorMapMember *nodes = reinterpret_cast<VorMapMember *>(recs + n);
    long long blocks = 0, sort_blocks = 0, tiles = 0;
    for (int q = 0; q < n; q++) {
        recs[q] = map_member(ctxs[q], accs[q], Ns[q], x[q], y[q], vx[q], vy[q], status[q]);
        recs[q].blk0 = (int)blocks;
        recs[q].bin0 = (int)sort_blocks;
        blocks += (Ns[q] + VO_BLOCK - 1) / VO_BLOCK;
        if (Ns[q]) sort_blocks += (recs[q].bx * recs[q].by + VO_SORT_WARPS - 1) / VO_SORT_WARPS;
        nodes[q] = node_member(ctxs[q], accs[q], recs[q]);
        nodes[q].tile0 = (int)tiles;
        tiles += (long long)nodes[q].ntx * ((ctxs[q]->Ny + VM_TY - 1) / VM_TY);
        OC_ARG(blocks < 0x7fffffff && sort_blocks < 0x7fffffff && tiles < 0x7fffffff,
               "Voronoi maps: too many agents or nodes for one launch");
    }
    OC_CUDA(cudaMemcpyAsync(c0->vmap_dev, recs, bytes, cudaMemcpyHostToDevice, st));
    const VorMember *dev = static_cast<const VorMember *>(c0->vmap_dev);
    const VorMapMember *dnodes = reinterpret_cast<const VorMapMember *>(dev + n);
    if (blocks) {
        vor_bin_multi_kernel<<<(unsigned)blocks, VO_BLOCK, 0, st>>>(dev, n);
        vor_scan_multi_kernel<<<n, 1024, 0, st>>>(dev);
        vor_place_multi_kernel<<<(unsigned)blocks, VO_BLOCK, 0, st>>>(dev, n);
        vor_sort_multi_kernel<<<(unsigned)sort_blocks, VO_SORT_WARPS * 32, 0, st>>>(dev, n);
        vor_volume_multi_kernel<<<(unsigned)blocks, VO_BLOCK, 0, st>>>(dev, n);
        oc::count_launch(5);
    }
    vormap_node_multi_kernel<<<(unsigned)tiles, VM_TX * VM_TY, 0, st>>>(dnodes, n);
    oc::count_launch();
    OC_CUDA(cudaGetLastError());
    OC_CUDA(cudaEventRecord(c0->vmap_ev, st));
    return OC_OK;
}
