// splash_upslope.cuh -- upslope contributing area (SURVEY 8f-2, second slice): depression filling and Quinn et al.
// (1991) multiple-flow-direction accumulation on the DEM.  The definition (and what is assumed about topmodel's
// sinkfill / topidx, PARITY UNPINNED) is in include/splash_cuda.h above splash_upslope_area_run.
//
// Every per-row metric (dx, dy, the diagonal, the cell area, the contour lengths and the fill steps eps) is computed
// once on the host and read from `rows`, so the kernels only add, subtract, multiply, divide and compare operands
// that a numpy restatement can reproduce bit for bit (-fmad=false).
#pragma once

#include <cooperative_groups.h>

namespace upslope {

namespace cg = cooperative_groups;

// per-row metrics, [n_rows * UR_N] row-major
enum { UR_DX = 0, UR_DY, UR_DD, UR_AREA, UR_LC, UR_LD, UR_EX, UR_EY, UR_ED, UR_N };

// neighbours in D8 code order: E, SE, S, SW, W, NW, N, NE (north row first, so S is row + 1)
__device__ __forceinline__ int d8_dr(int k) { return (k >= 1 && k <= 3) ? 1 : ((k >= 5 && k <= 7) ? -1 : 0); }
__device__ __forceinline__ int d8_dc(int k) { return (k == 0 || k == 1 || k == 7) ? 1 : ((k >= 3 && k <= 5) ? -1 : 0); }
// column of `rows` that holds the distance of direction k (E, W: dx; S, N: dy; diagonals: dd)
__device__ __forceinline__ int d8_dist(int k) { return (k & 1) ? UR_DD : ((k & 2) ? UR_DY : UR_DX); }

// ---- fill: the least W >= Z with W = Z on boundary cells and W(c) >= W(n) + eps(c->n) for some neighbour n -------
// Jacobi sweeps from above (W = +inf on non-boundary cells at the start) over 32 x 32 shared-memory tiles with a
// one-cell halo.  Inside a tile the update W(c) = max(Z(c), min_n W(n) + eps(c->n)) is iterated, with the halo held
// at the sweep's input, until the tile is stable or for at most the tile's perimeter; the sweep writes the other
// buffer of a ping-pong pair.  Every update lowers W and stays above the fixpoint, which is unique (eps > 0), so the
// result does not depend on the tiling or the iteration count; the sweep count does not depend on scheduling either
// (each in-tile iteration is a synchronous Jacobi step).
constexpr int kFT = 32;             // tile edge (cells)
constexpr int kFRows = 8;           // threadIdx.y extent; a thread owns kFT / kFRows cells of its column
constexpr int kFCells = kFT / kFRows;
constexpr int kFH = kFT + 2;        // tile + halo
constexpr int kFIter = 4 * kFT;     // in-tile iteration bound: the tile's perimeter

struct FillParams {
    const double* z;
    const double* rows;
    int n_rows, n_cols;
};

__device__ __forceinline__ bool is_boundary(const double* z, int nr, int nc, int r, int c) {
    if (r == 0 || c == 0 || r == nr - 1 || c == nc - 1) return true;
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if (isnan(z[(int64_t)(r + d8_dr(k)) * nc + c + d8_dc(k)])) return true;
    return false;
}

// W = Z on boundary cells, +inf on the other valid cells, NaN where Z is NA.  *err = 1 when an elevation is +-inf
// (rejected: the fill and the weights need finite values); *n_valid counts the valid cells.
__global__ void __launch_bounds__(256) k_fill_init(FillParams p, double* w, int* err, int* n_valid) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = false;
    if (i < (int64_t)p.n_rows * p.n_cols) {
        const int r = (int)(i / p.n_cols), c = (int)(i - (int64_t)r * p.n_cols);
        const double z = p.z[i];
        valid = !isnan(z);
        if (isinf(z)) *err = 1;
        w[i] = !valid ? z : (is_boundary(p.z, p.n_rows, p.n_cols, r, c) ? z : (double)INFINITY);
    }
    const int nv = __syncthreads_count(valid);
    if (threadIdx.x == 0 && nv) atomicAdd(n_valid, nv);
}

// One global sweep: reads w_in, writes w_out; flags[sweep] = 1 when a cell changed.  A sweep whose predecessor
// changed nothing returns at once (the batch the host launched between two reads of the flags went past the
// fixpoint).
__global__ void __launch_bounds__(kFT * kFRows) k_fill_sweep(FillParams p, const double* __restrict__ w_in,
                                                              double* __restrict__ w_out, int* flags, int sweep) {
    if (__ldcg(flags + sweep - 1) == 0) return;
    __shared__ double sz[kFH][kFH];
    __shared__ double sw[kFH][kFH];
    const int nr = p.n_rows, nc = p.n_cols;
    const int r0 = (int)blockIdx.y * kFT - 1, c0 = (int)blockIdx.x * kFT - 1;
    const int tid = threadIdx.y * kFT + threadIdx.x;
    for (int h = tid; h < kFH * kFH; h += kFT * kFRows) {
        const int hr = h / kFH, hc = h - hr * kFH, r = r0 + hr, c = c0 + hc;
        const bool in = r >= 0 && r < nr && c >= 0 && c < nc;
        const int64_t g = (int64_t)r * nc + c;
        sz[hr][hc] = in ? p.z[g] : (double)NAN;
        sw[hr][hc] = in ? w_in[g] : (double)NAN;
    }
    __syncthreads();
    const int hc = 1 + threadIdx.x, c = c0 + hc;
    bool upd[kFCells];
    double eps[kFCells][3];
#pragma unroll
    for (int j = 0; j < kFCells; ++j) {
        const int hr = 1 + threadIdx.y + j * kFRows, r = r0 + hr;
        upd[j] = false;
        if (r < nr && c < nc && !isnan(sz[hr][hc]) && r > 0 && c > 0 && r < nr - 1 && c < nc - 1) {
            bool b = false;
#pragma unroll
            for (int k = 0; k < 8; ++k) b |= isnan(sz[hr + d8_dr(k)][hc + d8_dc(k)]);
            upd[j] = !b;
        }
        if (upd[j]) {
            eps[j][0] = p.rows[(int64_t)r * UR_N + UR_EX];
            eps[j][1] = p.rows[(int64_t)r * UR_N + UR_EY];
            eps[j][2] = p.rows[(int64_t)r * UR_N + UR_ED];
        }
    }
    bool changed = false;
    for (int it = 0; it < kFIter; ++it) {
        double nv[kFCells];
        bool any = false;
#pragma unroll
        for (int j = 0; j < kFCells; ++j) {
            const int hr = 1 + threadIdx.y + j * kFRows;
            nv[j] = sw[hr][hc];
            if (!upd[j]) continue;
            double m = (double)INFINITY;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const double e = (k & 1) ? eps[j][2] : ((k & 2) ? eps[j][1] : eps[j][0]);
                const double v = sw[hr + d8_dr(k)][hc + d8_dc(k)] + e;
                if (v < m) m = v;
            }
            const double zc = sz[hr][hc];
            const double w = (m > zc) ? m : zc;
            any |= (w != nv[j]);
            nv[j] = w;
        }
        __syncthreads();  // every read of this iteration is done
#pragma unroll
        for (int j = 0; j < kFCells; ++j) sw[1 + threadIdx.y + j * kFRows][hc] = nv[j];
        changed |= any;
        if (!__syncthreads_or(any)) break;
    }
#pragma unroll
    for (int j = 0; j < kFCells; ++j) {
        const int hr = 1 + threadIdx.y + j * kFRows, r = r0 + hr;
        if (r < nr && c < nc) w_out[(int64_t)r * nc + c] = sw[hr][hc];
    }
    if (__syncthreads_or(changed) && tid == 0) flags[sweep] = 1;
}

// ---- accumulation (Quinn et al. 1991 MFD on the filled surface) ----------------------------------------------------
// A cell's donors are its valid neighbours with a strictly higher W; it passes dx*dy plus what it received to its
// strictly lower valid neighbours n, each the share w / S with w = ((W(c) - W(n)) / dist) * L and S the sum of its w
// in D8 order.  Kahn's algorithm, level-synchronous: a frontier cell pulls area(u) * (w_uc / S_u) from its donors in
// D8 order (they are final: every donor left the frontier in an earlier round), so the bits do not depend on the
// schedule; then it decrements its receivers' donor counts, and the thread that takes a count to 0 appends that
// receiver to the next frontier.  The atomics only schedule.
constexpr int kAccThreads = 256;
constexpr int kSoloEnter = kAccThreads;      // frontier this small: one CTA goes on alone with __syncthreads
constexpr int kSoloLeave = 4 * kAccThreads;  // ... until the frontier grows past this: the next launch takes the grid

// control words of the accumulation (device int array)
enum { AC_CNT = 0 /* 3 frontier counters */, AC_CUR = 3, AC_ROUNDS, AC_DONE, AC_NVALID, AC_ERR, AC_BADZ, AC_N };

struct AccumParams {
    const double* w;     // filled surface (NaN = NA)
    const double* rows;
    double* s;           // weight sum of each cell (prep writes it)
    double* area;
    int* ndon;           // donors not yet final
    int* front[2];       // frontiers (ping-pong; each valid cell enters exactly one)
    int* ctl;
    int n_rows, n_cols;
};

// S, the donor count and the first frontier (cells without donors); area = NaN where W is NA.
__global__ void __launch_bounds__(256) k_flow_prep(AccumParams p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.n_rows * p.n_cols) return;
    const int r = (int)(i / p.n_cols), c = (int)(i - (int64_t)r * p.n_cols);
    const double w0 = p.w[i];
    if (isnan(w0)) {
        p.area[i] = w0;
        return;
    }
    const double* rw = p.rows + (int64_t)r * UR_N;
    double s = 0.0;
    int nd = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int rr = r + d8_dr(k), cc = c + d8_dc(k);
        if (rr < 0 || rr >= p.n_rows || cc < 0 || cc >= p.n_cols) continue;
        const double wn = p.w[(int64_t)rr * p.n_cols + cc];
        if (wn < w0)
            s = s + ((w0 - wn) / rw[d8_dist(k)]) * rw[(k & 1) ? UR_LD : UR_LC];
        else if (wn > w0)
            ++nd;
    }
    p.s[i] = s;
    p.ndon[i] = nd;
    if (nd == 0) p.front[0][atomicAdd(p.ctl + AC_CNT, 1)] = (int)i;
}

__device__ __forceinline__ void accum_cell(const AccumParams& p, int i, int* fout, int* cnt_next) {
    const int r = i / p.n_cols, c = i - r * p.n_cols;
    const double w0 = p.w[i];
    double a = p.rows[(int64_t)r * UR_N + UR_AREA];
#pragma unroll
    for (int k = 0; k < 8; ++k) {  // pull from the donors
        const int rr = r + d8_dr(k), cc = c + d8_dc(k);
        if (rr < 0 || rr >= p.n_rows || cc < 0 || cc >= p.n_cols) continue;
        const int n = rr * p.n_cols + cc;
        const double wn = p.w[n];
        if (wn > w0) {  // the donor's weight towards c, with the donor's row metrics (direction k + 4: same kind)
            const double* rn = p.rows + (int64_t)rr * UR_N;
            const double wt = ((wn - w0) / rn[d8_dist(k)]) * rn[(k & 1) ? UR_LD : UR_LC];
            a = a + __ldcg(p.area + n) * (wt / p.s[n]);
        }
    }
    __stcg(p.area + i, a);
#pragma unroll
    for (int k = 0; k < 8; ++k) {  // release the receivers
        const int rr = r + d8_dr(k), cc = c + d8_dc(k);
        if (rr < 0 || rr >= p.n_rows || cc < 0 || cc >= p.n_cols) continue;
        const int n = rr * p.n_cols + cc;
        if (p.w[n] < w0 && atomicSub(p.ndon + n, 1) == 1) fout[atomicAdd(cnt_next, 1)] = n;
    }
}

// Cooperative launch sized with the occupancy API.  Rounds over the whole grid with grid.sync(); once the frontier
// fits one CTA, block 0 goes on alone with __syncthreads() (long rivers give thousands of rounds of a few cells) and
// hands back to the next launch if the frontier grows past kSoloLeave.  The round, the frontier parity and the
// counters live in ctl, so a launch resumes where the last one stopped.  Every loop ends on an empty frontier, on
// the round bound (n_valid: a longer chain would need a cycle) or on a solo hand-back.
__global__ void __launch_bounds__(kAccThreads) k_accum(AccumParams p) {
    cg::grid_group g = cg::this_grid();
    int* ctl = p.ctl;
    const bool lead = blockIdx.x == 0 && threadIdx.x == 0;
    int cur = __ldcg(ctl + AC_CUR), rounds = __ldcg(ctl + AC_ROUNDS);
    const int n_valid = __ldcg(ctl + AC_NVALID);
    bool solo = false;
    while (true) {
        const int n = __ldcg(ctl + AC_CNT + cur % 3);
        if (n == 0) {
            if (lead) ctl[AC_DONE] = 1;
            break;
        }
        if (rounds >= n_valid) {
            if (lead) ctl[AC_ERR] = 1;
            break;
        }
        if (!solo && n <= kSoloEnter) {
            g.sync();  // every CTA has read n before block 0 moves the counters on
            if (blockIdx.x != 0) return;
            solo = true;
        } else if (solo && n > kSoloLeave) {
            break;
        }
        const int stride = solo ? (int)blockDim.x : (int)(gridDim.x * blockDim.x);
        const int first = solo ? (int)threadIdx.x : (int)(blockIdx.x * blockDim.x + threadIdx.x);
        const int* fin = (cur & 1) ? p.front[1] : p.front[0];
        int* fout = (cur & 1) ? p.front[0] : p.front[1];
        for (int j = first; j < n; j += stride) accum_cell(p, __ldcg(fin + j), fout, ctl + AC_CNT + (cur + 1) % 3);
        if (lead) ctl[AC_CNT + (cur + 2) % 3] = 0;  // read in the previous round, appended to in the next
        if (solo)
            __syncthreads();
        else
            g.sync();
        ++cur;
        ++rounds;
    }
    if (lead) {
        ctl[AC_CUR] = cur;
        ctl[AC_ROUNDS] = rounds;
    }
}

}  // namespace upslope
