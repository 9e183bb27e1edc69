// oc_hjb_fused.cuh -- stage-fused RK45 step kernel (temporal blocking across the 6 new RHS evaluations).
//
// One launch performs a whole Dormand-Prince step attempt (scipy rk.py:14-71 rk_step + :146-147 error
// estimate) and the dense-output samples phi(t_e) of the t_eval points that fall inside the step
// (rk.py:178-180,723-737), reading y, f = K[0] and coef once and writing y_new, f_new = K[6] and the
// phi slices once: 40 B/cell/attempt + 8 B/cell/emitted slice instead of the 312 B/cell/attempt of the
// stage-wise formulation (SURVEY.md section 8d (iii)).
//
// Scheme ("2.5-D" streaming): a CTA owns BX = 128 consecutive columns and marches down a chunk of rows.
// Thread t owns ONE column; all RK state of that column lives in its registers as short row windows.
// At iteration r the CTA receives row r (stage 1 input), and stage s = 2..7 evaluates the stencil on row
// r-(s-1), i.e. every stage lags one row behind the previous one, so the 3-row stencil windows of all
// six stage inputs are register-resident.  Only the left/right neighbours cross threads: the stage
// input rows are published once per row to a double-buffered shared-memory line, two stages per 16-byte
// element (3 STS.128 + 6 LDS.128 per thread and row; one __syncthreads per row).
// Rows of y, f, coef are staged ahead of use in shared memory by the TMA unit: tiles of GR = 6 rows x 128 columns,
// one `cp.async.bulk.tensor.2d` per field and row group, issued by one elected thread while the previous group is
// being consumed (double buffered, completion tracked by one mbarrier per buffer; SASS: UTMALDG + SYNCS).  Columns
// outside the grid are zero-filled by the TMA unit and never read: the mirror ghost columns are read from the
// mirrored position inside the staged row.  Row groups that reach across the top or bottom edge of the grid (mirror
// ghost rows: a different, descending source row each) are staged row by row with 1-D bulk copies (UBLKCP) on the
// same mbarrier.  Grids with an odd number of columns (rows not 16-byte aligned) take the per-thread `cp.async`
// (LDGSTS) variant of the same kernel (template parameter BULK = false).
// Six stencil applications consume HALO = 6 columns per side (8 allocated for 64-byte aligned rows) and
// 6 rows above/below the chunk, which are recomputed redundantly.
//
// Arithmetic: FP64, FMA contraction allowed.  The stage combination is evaluated as
// y + (h a_s1) k_1 + (h a_s2) k_2 + ... with premultiplied coefficients, and the RHS (optimals.py:154-162)
// as  A_w * (N + S + W + E) + d_w * C  with A_w = A, d_w = -(4 A + coef) in the room and A_w = d_w = 0 in
// walls; both differ from the reference's evaluation order by rounding only (parity bar 1e-10, observed
// ~1e-13).
#pragma once
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstddef>
#include <cstdint>

#include "oc_rk45.h"

namespace fused {

#ifndef OC_BX
#define OC_BX 128
#endif
#ifndef OC_PF
#define OC_PF 6
#endif
#ifndef OC_PD
#define OC_PD (OC_PF - 1)
#endif
constexpr int BX = OC_BX;           // threads per CTA = columns per tile incl. halo
constexpr int HX = 8;               // halo columns per side (6 needed)
constexpr int VX = BX - 2 * HX;     // valid output columns per tile (112)
constexpr int HY = 6;               // halo rows per side
constexpr int PF = OC_PF;           // LDGSTS variant: staging ring depth (rows): rows r .. r+PD
constexpr int PD = OC_PD;           // LDGSTS variant: prefetch distance (rows in flight)
constexpr int GR = 6;               // TMA variant: rows per staged tile (row group)
constexpr int NG = 2;               // TMA variant: tile buffers (one in use, one in flight)
constexpr int UNROLL = 12;          // rows per unrolled loop body (multiple of PF, of NG*GR and of 2)
static_assert(UNROLL % PF == 0 && UNROLL % 2 == 0 && PD < PF && UNROLL == NG * GR && PF == GR, "ring / unroll geometry");
#ifndef OC_CTAS
#define OC_CTAS 2
#endif
#ifndef OC_VREGCONST
#define OC_VREGCONST 3
#endif
// 2 CTAs (8 warps) per SM with ~216 registers/thread beat 3 CTAs at 164: the row body is one long straight-line block
// and the extra registers buy instruction-level parallelism across the six stage chains (profiles/r1_fused_v4.md)
constexpr int CTAS_PER_SM = OC_CTAS;
constexpr int NE_MAX = 6;           // dense-output samples per launch

// rows per CTA chunk: balance the tail of the last wave (slots = SMs x resident CTAs) against the 2*HY halo rows
// each chunk recomputes.  `rows` = rows of the band, `copies` = bands launched back to back on this GPU.
inline int plan_chunk_rows(int Nx, int rows, int n_sm, int copies, int must_divide) {
    static const int cand[] = {16, 32, 48, 64, 96, 128, 160, 192, 224, 256, 320, 384, 448, 512, 640, 768, 1024, 2048};
    constexpr int UNROLL = 12;  // rows per unrolled loop body of the kernel (see below)
    const long long slots = (long long)n_sm * CTAS_PER_SM;
    const int gx = (Nx + VX - 1) / VX;
    double best = 1e300;
    int rc = 16;
    for (int c : cand) {
        if (must_divide && rows % c) continue;
        const int cc = c < rows ? c : rows;
        const long long blocks = (long long)gx * ((rows + cc - 1) / cc) * copies;
        // a CTA walks its chunk + 2 HY halo rows in whole unrolled bodies of UNROLL rows
        const int walked = (cc + 2 * HY + UNROLL - 1) / UNROLL * UNROLL;
        const double cost = (double)((blocks + slots - 1) / slots) * walked;
        if (cost < best) { best = cost; rc = cc; }
    }
    return rc;
}

constexpr int P2P_MAX_RANKS = 8;    // one NVSwitch box
constexpr int P2P_INBOX_STRIDE = 64; // doubles per (parity, rank) inbox slot: <= 62 chunk-row sums + the sequence number

struct alignas(64) Args {
    // TMA descriptors of y, k1, coef as 2-D (storage rows, Nx) FP64 tensors with a (GR, BX) box; valid when tma != 0
    CUtensorMap tm_y, tm_k1, tm_coef;
    int tma;
    const double *y, *k1, *coef;
    double *ynew, *k7, *partial;
    double *phi[NE_MAX];
    double ha21;
    double ha3[2], ha4[3], ha5[4], ha6[5];
    double hb[6];            // h*B (B[1] = 0 unused)
    double he[7];            // h*E (E[1] = 0 unused)
    double w[NE_MAX][7];     // h * sum_q P[j][q] x_e^(q+1)
    double A;                // -0.5 sigma^2 / (dx dy)
    double rtol, atol;
    int Ny, Nx, RC;          // global grid, RC = rows per chunk
    // row band (multi-GPU / virtual ranks): rows [own0, own1) are computed; y, k1, coef, ynew, k7 point to storage
    // whose first row is global row `row_base` (halo rows from the neighbouring bands included); phi slices
    // start at global row `phi_row_base`.  Single GPU: row_base = phi_row_base = 0, own = [0, Ny).
    int row_base, own0, own1, phi_row_base;
    // Final reduction inside the launch (single-GPU and batched solves): the CTA that finishes last adds the per-CTA
    // partial sums in the library's fixed order (per chunk row: 256 strided accumulators, shuffle tree, 8 warp sums left
    // to right; then the chunk rows top to bottom -- exactly rowgroup_sum_kernel + the host loop) and publishes the
    // scalar in page-locked host memory, where the host polls for it: no reduction launch, no copy, no stream
    // synchronisation per step attempt.  ticket == NULL: partial sums only (row-band solver: NCCL all-gather).
    unsigned *ticket;
    double *result;                 // mapped host memory: result[0] = sum
    unsigned long long *result_seq; // mapped host memory: set to `seq` after result[0] is visible
    unsigned long long seq;
    // Row-band solve over NVLink peer memory (template parameter P2P; oc_hjb_dist.cu): the halo exchange and the
    // error-norm all-gather are part of this launch.  (a) A CTA whose chunk touches a band edge copies the rows of
    // y_new / f_new lying within HY rows of that edge straight into the neighbouring GPU's halo rows when its row loop ends.  (b) The last
    // CTA writes this band's chunk-row sums into the inbox of every rank (peer stores, then a system fence, then the
    // sequence number), waits for the inboxes of all ranks, adds the sums in global chunk order and hands the total to
    // the host.  A rank that has seen every rank's sequence number also knows that every rank's kernel -- and with it
    // every halo store aimed at this rank -- has completed.
    double *peer_ynew[2], *peer_k7[2];  // [0]: rank-1 (rows above), [1]: rank+1; NULL at the ends of the grid
    int peer_row_base[2];               // global row of storage row 0 of the neighbour's arrays
    int nranks, my_rank;
    double *peer_inbox[P2P_MAX_RANKS];  // inbox of rank q as seen from this GPU; [my_rank] is the local one
};
constexpr int MAX_FINAL_ROWS = 2 * 6 * (BX + 2) - 8;  // chunk-row sums are staged in the (then idle) exchange buffer

// Where sample e of the controller's current attempt goes: column kd of `phi` (slices of `slice` elements), or, when
// only velocities are stored (phi == NULL), scratch slot e % NE_MAX.
inline double *sample_slice(const rk45::Controller &c, int e, double *phi, double *scratch, size_t slice) {
    return phi ? phi + (size_t)c.sample_column(e) * slice : scratch + (size_t)(e % NE_MAX) * slice;
}
// The per-attempt constants of one launch for the controller's current attempt: the tableau times h, and for samples
// [e0, e0 + ne) the dense-output weights (RkDenseOutput, rk.py:723-737) and destination slices.  The caller sets the
// arrays, geometry, tickets and peer pointers.
inline void set_attempt(Args &a, const rk45::Controller &c, int e0, int ne, double *phi, double *scratch, size_t slice) {
    const double h = c.h;
    a.ha21 = h * rk45::A[1][0];
    for (int j = 0; j < 2; j++) a.ha3[j] = h * rk45::A[2][j];
    for (int j = 0; j < 3; j++) a.ha4[j] = h * rk45::A[3][j];
    for (int j = 0; j < 4; j++) a.ha5[j] = h * rk45::A[4][j];
    for (int j = 0; j < 5; j++) a.ha6[j] = h * rk45::A[5][j];
    for (int j = 0; j < 6; j++) a.hb[j] = h * rk45::B[j];
    for (int j = 0; j < 7; j++) a.he[j] = h * rk45::E[j];
    for (int i = 0; i < ne; i++) {
        const double x = c.sample_x(e0 + i);
        const double pw[4] = {x, x * x, x * x * x, x * x * x * x};
        for (int j = 0; j < 7; j++) {
            double acc = 0.0;
            for (int q = 0; q < 4; q++) acc += rk45::P[j][q] * pw[q];
            a.w[i][j] = h * acc;
        }
        a.phi[i] = sample_slice(c, e0 + i, phi, scratch, slice);
    }
}

// ---- per-thread cp.async (LDGSTS) staging: the BULK = false variant
// predicated forms: the unrolled row body has no divergent region (a branch around the loads / stores makes ptxas save
// and restore the uniform registers that hold the RK coefficients on both sides of it)
__device__ __forceinline__ void cp_async8_if(void *smem, const void *gmem, bool ok) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %2, 0; @p cp.async.ca.shared.global [%0], [%1], 8; }"
                 ::"r"(s), "l"(gmem), "r"((int)ok) : "memory");
}
__device__ __forceinline__ void st_if(double *p, double v, bool ok) {
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %2, 0; @p st.global.f64 [%0], %1; }" ::"l"(p), "d"(v), "r"((int)ok) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- bulk-async (TMA) staging: the BULK = true variant
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
// one row segment global -> shared; completion (bytes) is signalled on `bar`.  16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void *smem, const void *gmem, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem), "r"(bytes),
                   "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
// one (GR x BX) tile global -> shared through a tensor map; out-of-range elements are zero-filled
__device__ __forceinline__ void tma_g2s_2d(unsigned smem, const CUtensorMap *map, int cx, int cy, unsigned bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem), "l"(reinterpret_cast<uint64_t>(map)), "r"(cx), "r"(cy), "r"(bar) : "memory");
}
// true on exactly one lane of a converged warp (uniform predicate: the region it guards is issued once per warp)
__device__ __forceinline__ bool elect_one() {
    unsigned pred;
    asm volatile("{ .reg .pred p; elect.sync _|p, 0xffffffff; selp.u32 %0, 1, 0, p; }" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_expect_tx_u32(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s_u32(unsigned smem, const void *gmem, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem), "l"(gmem), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "OC_WAITU_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra OC_DONEU_%=;\n"
        "bra OC_WAITU_%=;\n"
        "OC_DONEU_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "OC_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra OC_DONE_%=;\n"
        "bra OC_WAIT_%=;\n"
        "OC_DONE_%=:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}

// optimals.py:154-162.  Mirror ghosts (:149-152) need no special case here: rows/columns outside the grid
// are LOADED from their mirror image (row -j -> row j, row Ny-1+j -> Ny-1-j), the stencil commutes with
// that reflection, so every stage input is automatically even about the boundary and the value the
// reference reads from its ghost cell (ghost(-1) = value(1)) is exactly what sits in the halo.
// The newest row `dn` of the stage input is produced in the same iteration, so the evaluation is split
// into a part that does not depend on it (`pre`) and one FMA that does: the serial chain through the six
// stages of one row iteration is 2 FMAs per stage, with no select on it (walls: A_w = d_w = 0).
__device__ __forceinline__ double rhs_pre(double up, double lf, double rt, double C, double Aw, double dw) {
    return fma(Aw, (up + lf) + rt, dw * C);
}
__device__ __forceinline__ double rhs_fin(double pre, double dn, double Aw) { return fma(Aw, dn, pre); }

// 1/x for finite x > 0 (the error scale is >= atol): hardware seed + two Newton steps (~1e-16), no slow path
__device__ __forceinline__ double rcp_pos(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    return r;
}

struct __align__(128) Smem {
    double pf[NG][3][GR][BX];  // staged rows of y, k1, coef: NG tiles (TMA) / one ring of PF = GR row slots (LDGSTS)
    double2 ex[2][3][BX + 2];  // published stage-input rows, double buffered: (u2,u3), (u4,u5), (u6,y_new)
    double cst[(1 + NE_MAX) * 6];  // h*E and the dense-output weights (made opaque to the compiler, see below)
    double red[BX / 32];
    unsigned long long full[NG];   // one mbarrier per tile buffer (TMA)
    unsigned tile[4];              // bx, by, ngx, ngy of the batched kernel (hjb_fused_body<..., STASH = true>)
};
static_assert(sizeof(double2) * 2 * 3 * (BX + 2) >= sizeof(double) * MAX_FINAL_ROWS, "final reduction staging");

__device__ __forceinline__ int mirror(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * (n - 1) - i : i); }

// (bx, by): this CTA's tile column and chunk row; (ngx, ngy): the tile grid of its room.  STASH: keep the four in shared
// memory across the row loop (the batched kernel derives them from its launch table: they cannot be re-read from special
// registers as blockIdx / gridDim can, and the row loop needs every register)
template <int NE, bool P2P, bool BULK, bool STASH = false>
__device__ __forceinline__ void hjb_fused_body(const Args &a, unsigned bx, unsigned by, unsigned ngx, unsigned ngy) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
    const int tid = threadIdx.x;
    const int x0 = bx * VX - HX;                            // global column of tile position 0
    const int gx = x0 + tid;
    const int c0 = max(x0, 0), c1 = min(x0 + BX, a.Nx);             // columns of the grid this tile covers
    const int gxm = min(max(mirror(gx, a.Nx), c0), c1 - 1);         // column this thread's state comes from
    const int lt = BULK ? gxm - x0 : tid;                           // its position in the staged row
    const int y0 = a.own0 + by * a.RC;
    const int y1 = min(y0 + a.RC, a.own1);
    const bool col_out = tid >= HX && tid < BX - HX && gx < a.Nx;  // columns this thread stores
    const int phi_shift = (a.row_base - a.phi_row_base) * a.Nx;    // phi slices may start at another global row

    for (int i = tid; i < 2 * 3 * (BX + 2); i += BX) (&sm.ex[0][0][0])[i] = make_double2(0.0, 0.0);
    if (tid < 6) {
        const int j = tid == 0 ? 0 : tid + 1;  // stages 1,3,4,5,6,7 (B[1] = E[1] = P[1] = 0)
        sm.cst[tid] = a.he[j];
#pragma unroll
        for (int ee = 0; ee < NE; ee++) sm.cst[6 * (ee + 1) + tid] = a.w[ee][j];
    }
    if (STASH && tid == 0) { sm.tile[0] = bx; sm.tile[1] = by; sm.tile[2] = ngx; sm.tile[3] = ngy; }
    if (BULK && tid == 0) {
#pragma unroll
        for (int s = 0; s < NG; s++) mbar_init(&sm.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // shared-memory window addresses, computed once (opaque: ptxas would otherwise re-derive them from SR_CgaCtaId at every use)
    unsigned sm_pf = (unsigned)__cvta_generic_to_shared(&sm.pf[0][0][0][0]);
    unsigned sm_full = (unsigned)__cvta_generic_to_shared(&sm.full[0]);
    asm volatile("" : "+r"(sm_pf), "+r"(sm_full));

    // windows, indexed by lag (row r - lag)
    // all windows are registers.  Shared memory is the bottleneck resource of this kernel (every LDS.64 of a
    // warp costs 2 cycles of the SM's 128 B/cycle), so each loaded value is read from the ring exactly once.
    double yw[7], k1w[7], Aw[7], dw[7], k2w[5], k3w[7], k4w[7], k5w[7], k6w[7];
    double u2[3], u3[4], u4[5], u5[6], u6[7], un[8];
#pragma unroll
    for (int i = 0; i < 7; i++) { yw[i] = 0; k1w[i] = 0; Aw[i] = 0; dw[i] = 0; k3w[i] = 0; k4w[i] = 0; k5w[i] = 0; k6w[i] = 0; }
#pragma unroll
    for (int i = 0; i < 5; i++) k2w[i] = 0;
    u2[0] = u2[1] = u2[2] = 0; u3[1] = u3[2] = u3[3] = 0; u4[2] = u4[3] = u4[4] = 0;
    u5[3] = u5[4] = u5[5] = 0; u6[4] = u6[5] = u6[6] = 0; un[5] = un[6] = un[7] = 0;

    const int r_begin = y0 - HY, r_end = y1 + HY;  // rows loaded: [r_begin, r_end)
    const unsigned row_bytes = (unsigned)(c1 - c0) * 8u;
    // ring slot of row `row` = (row - r_begin) mod PF, tracked incrementally (PF is not a power of two)
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp-uniform
    constexpr unsigned TILE_BYTES = 3u * GR * BX * 8u, FIELD_BYTES = GR * BX * 8u, ROW_BYTES = BX * 8u;
    // TMA variant: stage the row group that starts at row `ga` into tile buffer `slot` (one elected thread)
    auto issue_group = [&](int ga, int slot) {
        if (warp == 0 && ga < r_end && elect_one()) {
            const unsigned bar = sm_full + 8u * slot, dst = sm_pf + TILE_BYTES * slot;
            if (ga >= 0 && ga + GR <= a.Ny) {
                mbar_expect_tx_u32(bar, TILE_BYTES);
                tma_g2s_2d(dst, &a.tm_y, x0, ga - a.row_base, bar);
                tma_g2s_2d(dst + FIELD_BYTES, &a.tm_k1, x0, ga - a.row_base, bar);
                tma_g2s_2d(dst + 2u * FIELD_BYTES, &a.tm_coef, x0, ga - a.row_base, bar);
            } else {  // the group reaches across the top / bottom edge of the grid: mirror ghost rows, one source row each
                mbar_expect_tx_u32(bar, 3u * GR * row_bytes);
#pragma unroll 1
                for (int j = 0; j < GR; j++) {
                    const int rm = min(max(mirror(ga + j, a.Ny), 0), a.Ny - 1);
                    const int g = (rm - a.row_base) * a.Nx + c0;  // element offsets fit 32 bits (one field < 2^31 elements)
                    const unsigned d = dst + ROW_BYTES * j + 8u * (c0 - x0);
                    bulk_g2s_u32(d, a.y + g, row_bytes, bar);
                    bulk_g2s_u32(d + FIELD_BYTES, a.k1 + g, row_bytes, bar);
                    bulk_g2s_u32(d + 2u * FIELD_BYTES, a.coef + g, row_bytes, bar);
                }
            }
        }
    };
    // LDGSTS variant: ring slot of row `row` = (row - r_begin) mod PF
    auto issue = [&](int row, int slot) {
        const int rm = min(max(mirror(row, a.Ny), 0), a.Ny - 1);
        const int g = (rm - a.row_base) * a.Nx + gxm;
        const bool ok = row < r_end;
        cp_async8_if(&sm.pf[0][0][slot][tid], a.y + g, ok);
        cp_async8_if(&sm.pf[0][1][slot][tid], a.k1 + g, ok);
        cp_async8_if(&sm.pf[0][2][slot][tid], a.coef + g, ok);
        cp_async_commit();  // one group per iteration, possibly empty
    };

    if (BULK) issue_group(r_begin, 0);
    else {
#pragma unroll 1
        for (int q = 0; q < PD; q++) issue(r_begin + q, q);
    }

    // The ~47 FP64 constants of the body do not fit the uniform register file (ptxas then spills uniform registers
    // through MOV.SPILL / R2UR.FILL every row).  With 2 CTAs/SM there are spare vector registers: the dense-output
    // weights of the first OC_VREGCONST samples (and h*E) are pinned there by making them opaque to the compiler
    // (read back from shared memory: a value ptxas could re-derive from the constant bank would not stay in a register).
    constexpr int NV = NE < OC_VREGCONST ? NE : OC_VREGCONST;
    double wv[NV > 0 ? NV : 1][6], hev[6];
#pragma unroll
    for (int ee = 0; ee < NV; ee++)
#pragma unroll
        for (int j = 0; j < 6; j++) wv[ee][j] = sm.cst[6 * (ee + 1) + j];
#pragma unroll
    for (int j = 0; j < 6; j++) hev[j] = a.he[j == 0 ? 0 : j + 1];
    const double dwall = -4.0 * a.A;  // d_w = -(4A + coef)

    double acc = 0.0;
    unsigned ph_base = 0;  // mbarrier phase of the tile buffers during this unrolled body
    // The row loop is unrolled by (a multiple of) the ring depth: inside the unrolled body the ring slot of every row,
    // the exchange buffer and the register holding each window entry are compile-time constants -- no address
    // arithmetic and no register moves for the shifting windows.
#pragma unroll 1
    for (int rb = r_begin; rb < r_end; rb += UNROLL) {
#pragma unroll
      for (int uu = 0; uu < UNROLL; uu++) {
        const int r = rb + uu;
        // rows past r_end are harmless (no loads are issued, every store is guarded): no early exit, so the
        // unrolled body is one straight-line block and the window shifts below are pure register renaming
        const int s0 = uu % PF;      // ring slot of row r: (r - r_begin) mod PF
        const int buf = uu & 1;
        const int gi = uu / GR, gj = uu % GR;  // TMA variant: tile buffer and row inside the tile
        if (BULK) {
            if (gj == 0) {
                // the other buffer was released by the barrier that ended the previous group: refill it, then make sure
                // this group's tile (in flight since the previous group started) has landed
                issue_group(r + GR, gi ^ 1);
                if (r < r_end) mbar_wait_u32(sm_full + 8u * gi, ph_base);
            }
        } else {
            issue(r + PD, (s0 + PD) % PF);
            cp_async_wait<PD>();
        }
        const double *ring = BULK ? &sm.pf[gi][0][gj][lt] : &sm.pf[0][0][s0][lt];
        yw[0] = ring[0];
        k1w[0] = ring[GR * BX];
        {
            const double cf = ring[2 * GR * BX];
            const bool wall = cf != cf;             // wall marker written by prep_kernel (optimals.py:162)
            Aw[0] = wall ? 0.0 : a.A;
            dw[0] = wall ? 0.0 : dwall - cf;
        }
        const double2 *exp_ = &sm.ex[buf ^ 1][0][tid];  // previous iteration's rows: [p*(BX+2)] left, [+2] right
        double2 *exc = &sm.ex[buf][0][tid + 1];
#ifdef OC_ABL_NOEX  // ablation (wrong results): no neighbour exchange
        const double2 l23 = make_double2(u2[1], u3[2]), r23 = l23, l45 = make_double2(u4[3], u5[4]), r45 = l45,
                      l6n = make_double2(u6[5], un[6]), r6n = l6n;
#else
        const double2 l23 = exp_[0], r23 = exp_[2];
        const double2 l45 = exp_[BX + 2], r45 = exp_[BX + 2 + 2];
        const double2 l6n = exp_[2 * (BX + 2)], r6n = exp_[2 * (BX + 2) + 2];
#endif
        // parts of the six stencils that do not depend on this iteration's new rows
        const double p2 = rhs_pre(u2[2], l23.x, r23.x, u2[1], Aw[1], dw[1]);
        const double p3 = rhs_pre(u3[3], l23.y, r23.y, u3[2], Aw[2], dw[2]);
        const double p4 = rhs_pre(u4[4], l45.x, r45.x, u4[3], Aw[3], dw[3]);
        const double p5 = rhs_pre(u5[5], l45.y, r45.y, u5[4], Aw[4], dw[4]);
        const double p6 = rhs_pre(u6[6], l6n.x, r6n.x, u6[5], Aw[5], dw[5]);
        const double p7 = rhs_pre(un[7], l6n.y, r6n.y, un[6], Aw[6], dw[6]);
        // stage-input partial sums that do not depend on this iteration's new k's (rk.py:63-64, premultiplied by h)
        const double q3 = fma(a.ha3[0], k1w[1], yw[1]);
        const double q4 = fma(a.ha4[1], k2w[2], fma(a.ha4[0], k1w[2], yw[2]));
        const double q5 = fma(a.ha5[2], k3w[3], fma(a.ha5[1], k2w[3], fma(a.ha5[0], k1w[3], yw[3])));
        const double q6 = fma(a.ha6[3], k4w[4], fma(a.ha6[2], k3w[4], fma(a.ha6[1], k2w[4], fma(a.ha6[0], k1w[4], yw[4]))));
        const double qn = fma(a.hb[4], k5w[5], fma(a.hb[3], k4w[5], fma(a.hb[2], k3w[5], fma(a.hb[0], k1w[5], yw[5]))));
        // ---- the serial chain of this row iteration
        u2[0] = fma(a.ha21, k1w[0], yw[0]);            // stage 2 input on row r
#ifdef OC_CHAIN1
        // one FMA per stage on the chain: k_s = (A_w h a) k_{s-1} + (A_w q + p); the stage input itself is off the chain
        k2w[1] = rhs_fin(p2, u2[0], Aw[1]);            // k2 on row r-1
        k3w[2] = fma(Aw[2] * a.ha3[1], k2w[1], fma(Aw[2], q3, p3));
        k4w[3] = fma(Aw[3] * a.ha4[2], k3w[2], fma(Aw[3], q4, p4));
        k5w[4] = fma(Aw[4] * a.ha5[3], k4w[3], fma(Aw[4], q5, p5));
        k6w[5] = fma(Aw[5] * a.ha6[4], k5w[4], fma(Aw[5], q6, p6));
        u3[1] = fma(a.ha3[1], k2w[1], q3);
        u4[2] = fma(a.ha4[2], k3w[2], q4);
        u5[3] = fma(a.ha5[3], k4w[3], q5);
        u6[4] = fma(a.ha6[4], k5w[4], q6);
        un[5] = fma(a.hb[5], k6w[5], qn);              // y_new on row r-5 (rk.py:66; B[1] = 0)
        const double k7 = fma(Aw[6] * a.hb[5], k6w[5], fma(Aw[6], qn, p7));  // k7 = f(y_new) on row r-6
#else
        k2w[1] = rhs_fin(p2, u2[0], Aw[1]);            // k2 on row r-1
        u3[1] = fma(a.ha3[1], k2w[1], q3);
        k3w[2] = rhs_fin(p3, u3[1], Aw[2]);            // k3 on row r-2
        u4[2] = fma(a.ha4[2], k3w[2], q4);
        k4w[3] = rhs_fin(p4, u4[2], Aw[3]);            // k4 on row r-3
        u5[3] = fma(a.ha5[3], k4w[3], q5);
        k5w[4] = rhs_fin(p5, u5[3], Aw[4]);            // k5 on row r-4
        u6[4] = fma(a.ha6[4], k5w[4], q6);
        k6w[5] = rhs_fin(p6, u6[4], Aw[5]);            // k6 on row r-5
        un[5] = fma(a.hb[5], k6w[5], qn);              // y_new on row r-5 (rk.py:66; B[1] = 0)
        const double k7 = rhs_fin(p7, un[5], Aw[6]);   // k7 = f(y_new) on row r-6
#endif
#ifndef OC_ABL_NOEX
        exc[0] = make_double2(u2[0], u3[1]);
        exc[BX + 2] = make_double2(u4[2], u5[3]);
        exc[2 * (BX + 2)] = make_double2(u6[4], un[5]);
#endif
        // ---- outputs on row r-6.  The arithmetic is unconditional (halo threads compute values nobody reads) and only
        // the stores and the error accumulation are predicated: no divergent region inside the unrolled body
        {
            const int row = r - 6;
#ifdef OC_ABL_NOSTORE  // ablation (wrong results): nothing is stored
            const bool ok = col_out && row >= y0 && row < y1 && a.Nx < 0;
#else
            const bool ok = col_out && row >= y0 && row < y1;
#endif
            const int g = (row - a.row_base) * a.Nx + gx;
            // rk.py:106,146-147: err = h * K.E ; scale = atol + max(|y|,|y_new|) * rtol
            double e = fma(hev[5], k7, fma(hev[4], k6w[6], fma(hev[3], k5w[6], fma(hev[2], k4w[6], fma(hev[1], k3w[6], hev[0] * k1w[6])))));
            double sc = fma(fmax(fabs(yw[6]), fabs(un[6])), a.rtol, a.atol);
            double qq = e * rcp_pos(sc);
            acc = ok ? fma(qq, qq, acc) : acc;
            st_if(a.ynew + g, un[6], ok);
            st_if(a.k7 + g, k7, ok);
#pragma unroll
            for (int ee = 0; ee < NE; ee++) {
                // rk.py:723-737: y_old + h * Q.p with Q = K^T P, regrouped per stage
                double ph;
#ifdef OC_ABL_NOPHI  // ablation (wrong results): no dense-output arithmetic
                if (true) ph = k7; else
#endif
                if (ee < NV)
                    ph = fma(wv[ee][5], k7, fma(wv[ee][4], k6w[6], fma(wv[ee][3], k5w[6], fma(wv[ee][2], k4w[6],
                             fma(wv[ee][1], k3w[6], fma(wv[ee][0], k1w[6], yw[6]))))));
                else
                    ph = fma(a.w[ee][6], k7, fma(a.w[ee][5], k6w[6], fma(a.w[ee][4], k5w[6],
                             fma(a.w[ee][3], k4w[6], fma(a.w[ee][2], k3w[6], fma(a.w[ee][0], k1w[6], yw[6]))))));
                st_if(a.phi[ee] + (g + phi_shift), ph, ok);
            }
        }
#ifndef OC_ABL_NOSYNC
        __syncthreads();
#endif
        // ---- shift windows by one row (pure renaming inside the unrolled body)
#pragma unroll
        for (int l = 6; l > 0; l--) { yw[l] = yw[l - 1]; k1w[l] = k1w[l - 1]; Aw[l] = Aw[l - 1]; dw[l] = dw[l - 1]; }
        k2w[4] = k2w[3]; k2w[3] = k2w[2]; k2w[2] = k2w[1];
        k3w[6] = k3w[5]; k3w[5] = k3w[4]; k3w[4] = k3w[3]; k3w[3] = k3w[2];
        k4w[6] = k4w[5]; k4w[5] = k4w[4]; k4w[4] = k4w[3];
        k5w[6] = k5w[5]; k5w[5] = k5w[4];
        k6w[6] = k6w[5];
        u2[2] = u2[1]; u2[1] = u2[0];
        u3[3] = u3[2]; u3[2] = u3[1];
        u4[4] = u4[3]; u4[3] = u4[2];
        u5[5] = u5[4]; u5[4] = u5[3];
        u6[6] = u6[5]; u6[5] = u6[4];
        un[7] = un[6]; un[6] = un[5];
      }
      ph_base ^= 1u;  // every tile buffer is used once per unrolled body
    }
    if (!BULK) cp_async_wait<0>();
    if (P2P && col_out) {
        // Halo exchange over NVLink: the rows of y_new / f_new within HY of a band edge are copied into the neighbouring
        // GPU's halo rows with peer stores.  Done here, after the row loop, by the thread that wrote them (it re-reads its
        // own stores, L2 hits), so that the hot loop of the row-band variant is the single-GPU loop.  Speculative like
        // the step itself: the rows of a rejected attempt are never read.
        if (y0 == a.own0 && a.peer_ynew[0] != nullptr)
            for (int row = a.own0; row < min(a.own0 + HY, y1); row++) {
                const int g = (row - a.row_base) * a.Nx + gx, gp = (row - a.peer_row_base[0]) * a.Nx + gx;
                a.peer_ynew[0][gp] = a.ynew[g];
                a.peer_k7[0][gp] = a.k7[g];
            }
        if (y1 == a.own1 && a.peer_ynew[1] != nullptr)
            for (int row = max(a.own1 - HY, y0); row < a.own1; row++) {
                const int g = (row - a.row_base) * a.Nx + gx, gp = (row - a.peer_row_base[1]) * a.Nx + gx;
                a.peer_ynew[1][gp] = a.ynew[g];
                a.peer_k7[1][gp] = a.k7[g];
            }
    }
    if (STASH) { bx = sm.tile[0]; by = sm.tile[1]; ngx = sm.tile[2]; ngy = sm.tile[3]; }
    // fixed-order CTA reduction of the error partial sum
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((tid & 31) == 0) sm.red[tid >> 5] = acc;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < BX / 32; i++) s += sm.red[i];
        a.partial[(size_t)by * ngx + bx] = s;
    }
    if (a.ticket == nullptr) return;
    // ---- last CTA: fixed-order final reduction (see Args)
    __shared__ int is_last;
    if (tid == 0) {
        if (P2P) __threadfence_system();  // this CTA's peer stores are ordered before its ticket
        else __threadfence();
        const unsigned t = atomicAdd(a.ticket, 1u);
        is_last = (t == ngx * ngy - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    double *rows = reinterpret_cast<double *>(&sm.ex[0][0][0]);
    const int ntx = ngx, gy = ngy, lane = tid & 31;
    for (int row = tid >> 5; row < gy; row += BX / 32) {
        // the 8 warps of rowgroup_sum_kernel's 256 threads, emulated by this warp: all loads first (independent, in
        // flight together), then the 8 shuffle trees, then the left-to-right sum of the 8 warp totals
        double v[8];
#pragma unroll
        for (int vw = 0; vw < 8; vw++) {
            v[vw] = 0.0;
            for (int i = vw * 32 + lane; i < ntx; i += 256) v[vw] += __ldcg(a.partial + (size_t)row * ntx + i);
        }
        double srow = 0.0;
#pragma unroll
        for (int vw = 0; vw < 8; vw++) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[vw] += __shfl_down_sync(0xffffffffu, v[vw], o);
            srow += v[vw];  // meaningful on lane 0
        }
        if (lane == 0) rows[row] = srow;
    }
    __syncthreads();
    if (P2P) {
        // all-gather of the chunk-row sums through the ranks' inboxes (double buffered by the parity of seq)
        const int par = (int)(a.seq & 1ull);
        if (tid < a.nranks) {
            double *dst = a.peer_inbox[tid] + (size_t)(par * P2P_MAX_RANKS + a.my_rank) * P2P_INBOX_STRIDE;
            for (int r = 0; r < gy; r++) *reinterpret_cast<volatile double *>(dst + r) = rows[r];
            __threadfence_system();
            *reinterpret_cast<volatile unsigned long long *>(dst + P2P_INBOX_STRIDE - 1) = a.seq;
            const volatile unsigned long long *flag = reinterpret_cast<const volatile unsigned long long *>(
                a.peer_inbox[a.my_rank] + (size_t)(par * P2P_MAX_RANKS + tid) * P2P_INBOX_STRIDE + P2P_INBOX_STRIDE - 1);
            // bounded wait (>= 8 s): a rank that died must not leave the others spinning in a kernel for ever
            long long it = 0;
            while (*flag != a.seq) {
                if (++it > 40000000ll) { is_last = 2; break; }
                __nanosleep(200);
            }
            __threadfence_system();
        }
        __syncthreads();
        if (tid == 0 && is_last == 2) {  // peer time-out: tell the host (sequence number with the top bit set)
            *a.ticket = 0u;
            *reinterpret_cast<volatile unsigned long long *>(a.result_seq) = a.seq | (1ull << 63);
        } else if (tid == 0) {
            double tot = 0.0;
            for (int q = 0; q < a.nranks; q++) {  // global chunk order: ranks top to bottom, chunk rows top to bottom
                const volatile double *src = a.peer_inbox[a.my_rank] + (size_t)(par * P2P_MAX_RANKS + q) * P2P_INBOX_STRIDE;
                for (int r = 0; r < gy; r++) tot += src[r];
            }
            *a.ticket = 0u;
            *reinterpret_cast<volatile double *>(a.result) = tot;
            __threadfence_system();
            *reinterpret_cast<volatile unsigned long long *>(a.result_seq) = a.seq;
        }
        return;
    }
    if (tid == 0) {
        double tot = 0.0;
        for (int r = 0; r < gy; r++) tot += rows[r];
        *a.ticket = 0u;
        *reinterpret_cast<volatile double *>(a.result) = tot;
        __threadfence_system();
        *reinterpret_cast<volatile unsigned long long *>(a.result_seq) = a.seq;
    }
}

template <int NE, bool P2P = false, bool BULK = true>
__global__ void __launch_bounds__(BX, CTAS_PER_SM) hjb_fused_kernel(const __grid_constant__ Args a) {
    hjb_fused_body<NE, P2P, BULK>(a, blockIdx.x, blockIdx.y, gridDim.x, gridDim.y);
}

// Ensembles (BASELINE configs[4]): the same step for up to BATCH_MAX independent rooms in ONE launch.  The rooms may
// differ in grid shape: the launch is a flattened 1-D grid holding exactly the sum of the rooms' tile grids, room q owning
// CTAs [first[q], first[q + 1]) in its own row-major (chunk row, tile column) order -- the chunking and CTA order of its
// stand-alone launch.  Every room brings its own Args (its own grid, step size, dense-output weights, arrays, ticket and
// result slot: the rooms' RK45 controllers are independent), all in kernel-parameter space, so the per-room constants are
// still uniform-register operands.  Rooms are grouped by their number of dense-output samples NE and by the staging
// variant (BULK needs an even Nx; see bulk_ok).
// A CTA finds its room with ONE load from a CTA-to-room table indexed by blockIdx.x >> shift: ptxas repeats that load
// where the row loop needs the room's Args instead of keeping the room index in a register (a scan of the prefix sums
// cannot be repeated that way, and the index then spilled inside the row loop).  The table has one entry per 2^shift
// CTAs, so every room's first CTA must be a multiple of 2^shift (set_batch_table).
constexpr int BATCH_MAX = 24;
constexpr int BATCH_PARAM_BYTES = 32704;  // the 32764-byte kernel-parameter limit, rounded down to Args' 64-byte alignment
constexpr int BATCH_TABLE = BATCH_PARAM_BYTES - BATCH_MAX * (int)sizeof(Args) - (3 * BATCH_MAX + 1) * (int)sizeof(int);
struct BatchArgs {
    Args a[BATCH_MAX];
    int first[BATCH_MAX];       // first CTA of room q (prefix sum); INT_MAX past the last room of the launch
    int ngx[BATCH_MAX], ngy[BATCH_MAX];  // tile grid of room q: tile columns, chunk rows
    int shift;
    unsigned char room_of[BATCH_TABLE];  // room of CTAs [c << shift, (c + 1) << shift)
};
static_assert(BATCH_TABLE >= 1024 && sizeof(BatchArgs) <= 32764, "kernel parameter space");
template <int NE, bool BULK>
__global__ void __launch_bounds__(BX, CTAS_PER_SM) hjb_fused_batch_kernel(const __grid_constant__ BatchArgs ba) {
    const int cta = blockIdx.x;
    const int q = ba.room_of[cta >> ba.shift];
    const int local = cta - ba.first[q], ngx = ba.ngx[q];
    hjb_fused_body<NE, false, BULK, true>(ba.a[q], local % ngx, local / ngx, ngx, ba.ngy[q]);
}

// Launch of one step attempt.  BULK staging needs 16-byte aligned rows: an even number of columns and 16-byte aligned
// field pointers (phi slices are only stored to, with 8-byte stores).
inline bool bulk_ok(const Args &a) {
#ifdef OC_NO_BULK
    return false;
#else
    return a.tma != 0 && (a.Nx % 2 == 0) && (((uintptr_t)a.y | (uintptr_t)a.k1 | (uintptr_t)a.coef) % 16 == 0);
#endif
}

// Host side of the TMA staging: descriptor of one field stored as (rows, Nx) FP64 with a (GR, BX) box.  The encoder is
// a driver entry point (no link-time dependency on libcuda).  Returns false when the field cannot be described
// (odd Nx: row pitch not a multiple of 16 bytes) -- the solver then launches the LDGSTS variant.
inline bool make_tensor_map(CUtensorMap *tm, const double *base, int rows, int Nx) {
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static encode_fn encode = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            encode = reinterpret_cast<encode_fn>(fn);
        else
            cudaGetLastError();
    }
    if (!encode || Nx % 2 != 0 || ((uintptr_t)base % 16) != 0) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)Nx, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)Nx * sizeof(double)};
    const cuuint32_t box[2] = {(cuuint32_t)BX, (cuuint32_t)GR};
    const cuuint32_t estr[2] = {1, 1};
    return encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// descriptors of the three fields an attempt reads (storage of `rows` rows each); sets a.tma.  A solve alternates between
// a handful of arrays (y / y_new, f / f_new, coef): the encoded descriptors are kept in a small per-solve cache.
struct MapCache {
    static constexpr int CAP = 8;
    const double *base[CAP];
    int rows[CAP], n = 0;
    CUtensorMap tm[CAP];
    bool get(const double *b, int r, int Nx, CUtensorMap *out) {
        for (int i = 0; i < n; i++)
            if (base[i] == b && rows[i] == r) { *out = tm[i]; return true; }
        CUtensorMap t;
        if (!make_tensor_map(&t, b, r, Nx)) return false;
        if (n < CAP) { base[n] = b; rows[n] = r; tm[n] = t; n++; }
        *out = t;
        return true;
    }
};
inline void set_tensor_maps(Args &a, int rows, MapCache *cache = nullptr) {
    MapCache local;
    MapCache &c = cache ? *cache : local;
    a.tma = c.get(a.y, rows, a.Nx, &a.tm_y) && c.get(a.k1, rows, a.Nx, &a.tm_k1) && c.get(a.coef, rows, a.Nx, &a.tm_coef);
}
template <int NE, bool P2P, bool BULK>
inline cudaError_t launch_one(const Args &a, dim3 grid, cudaStream_t st) {
    if (sizeof(Smem) > 48 * 1024) {  // per device, cheap: set on every launch (only deep rings need it)
        cudaError_t e = cudaFuncSetAttribute(hjb_fused_kernel<NE, P2P, BULK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)sizeof(Smem));
        if (e != cudaSuccess) return e;
    }
    hjb_fused_kernel<NE, P2P, BULK><<<grid, BX, sizeof(Smem), st>>>(a);
    return cudaSuccess;
}
template <bool P2P>
inline cudaError_t launch(int ne, const Args &a, dim3 grid, cudaStream_t st) {
    const bool bulk = bulk_ok(a);
#define OC_FUSED_CASE(NE) \
    case NE: return bulk ? launch_one<NE, P2P, true>(a, grid, st) : launch_one<NE, P2P, false>(a, grid, st);
    switch (ne) {
        OC_FUSED_CASE(0) OC_FUSED_CASE(1) OC_FUSED_CASE(2) OC_FUSED_CASE(3) OC_FUSED_CASE(4) OC_FUSED_CASE(5)
        default: return bulk ? launch_one<6, P2P, true>(a, grid, st) : launch_one<6, P2P, false>(a, grid, st);
    }
#undef OC_FUSED_CASE
}

// one launch for `nb` rooms (all with `ne` samples), all TMA-capable (bulk) or none; ba.first / ngx / ngy set by
// set_batch_table
template <int NE, bool BULK>
inline cudaError_t launch_batch_one(const BatchArgs &ba, int ctas, cudaStream_t st) {
    if (sizeof(Smem) > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(hjb_fused_batch_kernel<NE, BULK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)sizeof(Smem));
        if (e != cudaSuccess) return e;
    }
    hjb_fused_batch_kernel<NE, BULK><<<ctas, BX, sizeof(Smem), st>>>(ba);
    return cudaSuccess;
}
// the launch table of rooms [0, nb) with tile grids (ngx[q], ngy[q]); returns the number of CTAs of the launch, or 0 when
// the CTA-to-room table cannot describe these rooms (more than BATCH_TABLE entries at the coarsest shift their first CTAs
// allow): the caller then launches fewer rooms.  One room always fits.
inline int set_batch_table(BatchArgs &ba, int nb, const int *ngx, const int *ngy) {
    int ctas = 0, align = 30;  // align: the largest shift every room's first CTA is a multiple of
    for (int q = 0; q < BATCH_MAX; q++) {
        ba.first[q] = q < nb ? ctas : INT_MAX;
        ba.ngx[q] = q < nb ? ngx[q] : 1;
        ba.ngy[q] = q < nb ? ngy[q] : 1;
        if (q > 0 && q < nb) align = std::min(align, __builtin_ctz((unsigned)ctas));
        if (q < nb) ctas += ngx[q] * ngy[q];
    }
    int shift = 0;
    while (((ctas - 1) >> shift) + 1 > BATCH_TABLE) shift++;
    if (shift > align) return 0;
    ba.shift = shift;
    for (int q = 0; q < nb; q++)
        for (int c = ba.first[q] >> shift; c <= (ba.first[q] + ngx[q] * ngy[q] - 1) >> shift; c++) ba.room_of[c] = (unsigned char)q;
    return ctas;
}
inline cudaError_t launch_batch(int ne, bool bulk, const BatchArgs &ba, int ctas, cudaStream_t st) {
#define OC_FUSED_CASE(NE) \
    case NE: return bulk ? launch_batch_one<NE, true>(ba, ctas, st) : launch_batch_one<NE, false>(ba, ctas, st);
    switch (ne) {
        OC_FUSED_CASE(0) OC_FUSED_CASE(1) OC_FUSED_CASE(2) OC_FUSED_CASE(3) OC_FUSED_CASE(4) OC_FUSED_CASE(5)
        default: return bulk ? launch_batch_one<6, true>(ba, ctas, st) : launch_batch_one<6, false>(ba, ctas, st);
    }
#undef OC_FUSED_CASE
}

}  // namespace fused
