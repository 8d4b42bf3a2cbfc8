// splash_upslope.cuh -- upslope contributing area (SURVEY 8f-2): depression filling, then either Quinn et al. (1991)
// multiple-flow-direction accumulation (second slice) or Tarboton (1997) D-infinity accumulation with flat resolution
// (third slice).  The definitions (and what is assumed about topmodel's sinkfill / topidx and TauDEM's PitRemove /
// DinfFlowDir / AreaDinf, PARITY UNPINNED) are in include/splash_cuda.h above splash_upslope_area_run and
// splash_upslope_dinf_run.
//
// Every per-row metric (dx, dy, the diagonal, the cell area, the contour lengths, the fill steps eps and the facet
// angles) is computed once on the host and read from `rows`, so the kernels only add, subtract, multiply, divide and
// compare operands that a numpy restatement can reproduce bit for bit (-fmad=false); the one exception is the D8
// angle inside a D-infinity facet, atan(s2 / s1).
#pragma once

#include <cooperative_groups.h>

namespace upslope {

namespace cg = cooperative_groups;

// per-row metrics, [n_rows * UR_N] row-major
// UR_TX = atan2(dy, dx), UR_TY = atan2(dx, dy): the angle of a D-infinity facet whose cardinal step is E-W / N-S
enum { UR_DX = 0, UR_DY, UR_DD, UR_AREA, UR_LC, UR_LD, UR_EX, UR_EY, UR_ED, UR_TX, UR_TY, UR_N };

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
// (each in-tile iteration is a synchronous Jacobi step).  With eps = 0 (D-infinity: PitRemove fills to flat) the
// equation has other solutions too (a closed flat floor is one), but every iterate from above stays above the minimax
// spill elevation, which is itself a solution, and takes its values from the finite set of Z; the descent therefore
// stops, and only at that greatest solution, whatever the tiling.
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

struct MfdRule : AccumParams {
    __device__ __forceinline__ void visit(int i, int* fout, int* cnt_next) const { accum_cell(*this, i, fout, cnt_next); }
};

// Level-synchronous frontier rounds; Rule::visit(i, fout, cnt_next) does one frontier cell's work and appends the
// cells it completes to fout.  Instantiated for the MFD and D-infinity accumulations and for the breadth-first
// distances over flats.  Cooperative launch sized with the occupancy API.  Rounds over the whole grid with
// grid.sync(); once the frontier fits one CTA, block 0 goes on alone with __syncthreads() (long rivers give thousands
// of rounds of a few cells) and hands back to the next launch if the frontier grows past kSoloLeave.  The round, the
// frontier parity and the counters live in ctl, so a launch resumes where the last one stopped.  Every loop ends on
// an empty frontier, on the round bound (n_valid: a longer chain would need a cycle) or on a solo hand-back.
template <class Rule>
__device__ __forceinline__ void frontier_rounds(const Rule& p) {
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
        for (int j = first; j < n; j += stride) p.visit(__ldcg(fin + j), fout, ctl + AC_CNT + (cur + 1) % 3);
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

template <class Rule>
__global__ void __launch_bounds__(kAccThreads) k_accum(Rule p) {
    frontier_rounds(p);
}

// ---- D-infinity (Tarboton 1997) on the surface filled with eps = 0, flats resolved as Garbrecht and Martz (1997) in
// the formulation of Barnes, Lehman and Mulla (2014) ------------------------------------------------------------------
// Flat: a valid non-boundary cell without a strictly lower neighbour.  Outlet: a non-flat (or boundary) neighbour of a
// flat cell at the same W.  The flats get two breadth-first distances, towards lower (from the outlets: their flat
// neighbours are 1) and away from higher (flat cells next to higher ground are 1), both as frontier rounds of
// k_accum; labels (the least cell index of each 8-connected flat) give the per-flat maximum H of the away distance,
// and M = 2 * towards + (H - away) is the surface a flat cell's direction is taken on (outlets M = 0).
enum { FL_FLAT = 1, FL_HIGH = 2 };  // cell class bits; FL_HIGH: a flat cell with a strictly higher neighbour
// receiver codes, one byte per cell: cardinal receiver (D8 code in bits 0-2, present: bit 3), diagonal (bits 4-6, 7)
enum { REC_C = 0x08, REC_D = 0x80 };

constexpr double kHalfPi = 1.5707963267948966;  // pi / 2 rounded to double
constexpr double kTwoPi = 4.0 * kHalfPi;

struct FlatParams {
    const double* w;     // filled surface (NaN = NA)
    unsigned char* cls;
    int* tow;            // towards-lower distance (-1: unset); k_flat_mask turns it into M
    int* away;           // away-from-higher distance (-1: unset)
    int* hmax;           // per-flat maximum of away, at the flat's label
    int n_rows, n_cols;
};

// classes; label = own index on flat cells, -1 elsewhere; distances unset; hmax 0
__global__ void __launch_bounds__(256) k_flat_mark(FlatParams p, int* label) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.n_rows * p.n_cols) return;
    const int r = (int)(i / p.n_cols), c = (int)(i - (int64_t)r * p.n_cols);
    const double w0 = p.w[i];
    unsigned char k = 0;
    if (!isnan(w0) && !is_boundary(p.w, p.n_rows, p.n_cols, r, c)) {
        bool lower = false, higher = false;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const double wn = p.w[(int64_t)(r + d8_dr(j)) * p.n_cols + c + d8_dc(j)];
            lower |= wn < w0;
            higher |= wn > w0;
        }
        if (!lower) k = FL_FLAT | (higher ? FL_HIGH : 0);
    }
    p.cls[i] = k;
    label[i] = (k & FL_FLAT) ? (int)i : -1;
    p.tow[i] = -1;
    p.away[i] = -1;
    p.hmax[i] = 0;
}

// One Jacobi sweep of the flat labels: the least label among the cell and its flat neighbours, and the label of the
// cell its label names (pointer jumping: that cell is in the same flat).  Labels only fall and stay cell indices of
// the same flat, so the sweeps end with every flat at its least index.  flags as k_fill_sweep.
__global__ void __launch_bounds__(256) k_flat_label(FlatParams p, const int* __restrict__ lin, int* __restrict__ lout,
                                                    int* flags, int sweep) {
    if (__ldcg(flags + sweep - 1) == 0) return;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool changed = false;
    if (i < (int64_t)p.n_rows * p.n_cols) {
        int l = lin[i];
        if (l >= 0) {  // a flat cell: not on the edge, every neighbour exists
            const int r = (int)(i / p.n_cols), c = (int)(i - (int64_t)r * p.n_cols);
            int m = lin[l];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int64_t n = (int64_t)(r + d8_dr(k)) * p.n_cols + c + d8_dc(k);
                if (p.cls[n] & FL_FLAT) m = min(m, lin[n]);
            }
            changed = m < l;
            l = min(l, m);
        }
        lout[i] = l;
    }
    if (__syncthreads_or(changed) && threadIdx.x == 0) flags[sweep] = 1;
}

// First frontier of a breadth-first distance: flat cells next to an outlet (towards) or to higher ground (away) get 1.
template <bool kAway>
__global__ void __launch_bounds__(256) k_flat_seed(FlatParams p, int* front0, int* ctl) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.n_rows * p.n_cols) return;
    const unsigned char k = p.cls[i];
    if (!(k & FL_FLAT)) return;
    bool seed = (k & FL_HIGH) != 0;
    if (!kAway) {
        const int r = (int)(i / p.n_cols), c = (int)(i - (int64_t)r * p.n_cols);
        const double w0 = p.w[i];
        seed = false;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int64_t n = (int64_t)(r + d8_dr(j)) * p.n_cols + c + d8_dc(j);
            seed |= !(p.cls[n] & FL_FLAT) && p.w[n] == w0;
        }
    }
    if (seed) {
        (kAway ? p.away : p.tow)[i] = 1;
        front0[atomicAdd(ctl + AC_CNT, 1)] = (int)i;
    }
}

// A frontier cell at distance d gives d + 1 to its flat neighbours that have none (the CAS only decides who appends
// a cell; every claimant of a round writes the same distance).
struct FlatBfs {
    const unsigned char* cls;
    int* dist;
    int* front[2];
    int* ctl;
    int n_rows, n_cols;
    __device__ __forceinline__ void visit(int i, int* fout, int* cnt_next) const {
        const int r = i / n_cols, c = i - r * n_cols;
        const int d = __ldcg(dist + i) + 1;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int n = (r + d8_dr(k)) * n_cols + c + d8_dc(k);
            if ((cls[n] & FL_FLAT) && atomicCAS(dist + n, -1, d) == -1) fout[atomicAdd(cnt_next, 1)] = n;
        }
    }
};

__global__ void __launch_bounds__(256) k_flat_height(FlatParams p, const int* label) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.n_rows * p.n_cols || !(p.cls[i] & FL_FLAT)) return;
    const int a = p.away[i];
    if (a > 0) atomicMax(p.hmax + label[i], a);
}

// M = 2 * towards + (H - away) on flat cells (away and H are 0 on a flat without higher ground), 0 elsewhere; in place
// of the towards distance.
__global__ void __launch_bounds__(256) k_flat_mask(FlatParams p, const int* label) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.n_rows * p.n_cols) return;
    if (!(p.cls[i] & FL_FLAT)) {
        p.tow[i] = 0;
        return;
    }
    const int a = p.away[i];
    p.tow[i] = 2 * p.tow[i] + p.hmax[label[i]] - (a > 0 ? a : 0);
}

// facet f (Tarboton's order): cardinal neighbour e1, diagonal neighbour e2, angle ac * pi/2 + af * r
__device__ __forceinline__ int facet_e1(int f) { return (8 - 2 * ((f + 1) >> 1)) & 7; }
__device__ __forceinline__ int facet_e2(int f) { return 7 - 2 * (f >> 1); }
__device__ __forceinline__ double facet_angle(int f, double r) {
    const double b = (double)((f + 1) >> 1) * kHalfPi;
    const double a = (f & 1) ? b - r : b + r;
    return a >= kTwoPi ? a - kTwoPi : a;  // facet 8 at r = 0: east
}

struct DinfParams {
    const double* w;
    const double* rows;
    const unsigned char* cls;
    const int* mask;     // M (0 off the flats)
    unsigned char* rec;  // receiver codes
    double* pd;          // proportion of the diagonal receiver (1 - pd: the cardinal one)
    double* angle;       // optional (NULL): radians counter-clockwise from east, NaN without a direction
    int n_rows, n_cols;
};

// The D-infinity facet rule on W (on M, for a flat cell, over the facets whose neighbours are at its W); the
// clipping cases are decided by comparisons only, and only the angle inside the chosen facet goes through atan.
__global__ void __launch_bounds__(256) k_dinf_dir(DinfParams p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.n_rows * p.n_cols) return;
    const int r = (int)(i / p.n_cols), c = (int)(i - (int64_t)r * p.n_cols);
    const double w0 = p.w[i];
    unsigned char code = 0;
    double pd = 0.0, ang = (double)NAN;
    if (!isnan(w0) && !is_boundary(p.w, p.n_rows, p.n_cols, r, c)) {
        const double* rw = p.rows + (int64_t)r * UR_N;
        const double dx = rw[UR_DX], dy = rw[UR_DY], dd = rw[UR_DD];
        const bool flat = (p.cls[i] & FL_FLAT) != 0;
        const double e0 = flat ? (double)p.mask[i] : w0;
        double best = 0.0, bs1 = 0.0, bs2 = 0.0;
        int bf = -1, bk = 0;
#pragma unroll
        for (int f = 0; f < 8; ++f) {
            const int k1 = facet_e1(f), k2 = facet_e2(f);
            const int64_t n1 = (int64_t)(r + d8_dr(k1)) * p.n_cols + c + d8_dc(k1);
            const int64_t n2 = (int64_t)(r + d8_dr(k2)) * p.n_cols + c + d8_dc(k2);
            double e1 = p.w[n1], e2 = p.w[n2];
            if (flat) {
                if (e1 != w0 || e2 != w0) continue;
                e1 = (double)p.mask[n1];
                e2 = (double)p.mask[n2];
            }
            const bool ew = (k1 & 2) == 0;  // cardinal step E or W
            const double d1 = ew ? dx : dy, d2 = ew ? dy : dx;
            const double s1 = (e0 - e1) / d1, s2 = (e1 - e2) / d2;
            double s;
            int kind;  // 0: clipped to the cardinal, 1: clipped to the diagonal, 2: inside the facet
            if (s2 > 0.0 && s1 > 0.0 && s2 * d1 < s1 * d2) {
                kind = 2;
                s = sqrt(s1 * s1 + s2 * s2);
            } else if (s2 > 0.0) {
                kind = 1;
                s = (e0 - e2) / dd;
            } else {
                kind = 0;
                s = s1;
            }
            if (s > best) {
                best = s;
                bf = f;
                bk = kind;
                bs1 = s1;
                bs2 = s2;
            }
        }
        if (bf >= 0) {
            const int k1 = facet_e1(bf), k2 = facet_e2(bf);
            const double th = ((k1 & 2) == 0) ? rw[UR_TX] : rw[UR_TY];
            double rr;
            if (bk == 0) {
                code = REC_C | k1;
                rr = 0.0;
            } else if (bk == 1) {
                code = REC_D | (k2 << 4);
                pd = 1.0;
                rr = th;
            } else {
                code = REC_C | k1 | REC_D | (k2 << 4);
                rr = atan(bs2 / bs1);
                pd = fmin(rr / th, 1.0);  // the device atan may land a few ulp past theta_f: no negative share
            }
            ang = facet_angle(bf, rr);
        } else if (flat) {  // steepest descent in M over the neighbours at W (Barnes: one is lower)
            double g = 0.0;
            int bk8 = -1;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int64_t n = (int64_t)(r + d8_dr(k)) * p.n_cols + c + d8_dc(k);
                if (p.w[n] != w0) continue;
                const double v = (e0 - (double)p.mask[n]) / rw[d8_dist(k)];
                if (v > g) {
                    g = v;
                    bk8 = k;
                }
            }
            if (bk8 >= 0) {
                // the first facet with that receiver, clipped to it
                const int f = bk8 == 0 ? 0 : 7 - bk8;
                if (bk8 & 1) {
                    code = REC_D | (bk8 << 4);
                    pd = 1.0;
                    ang = facet_angle(f, ((facet_e1(f) & 2) == 0) ? rw[UR_TX] : rw[UR_TY]);
                } else {
                    code = REC_C | bk8;
                    ang = facet_angle(f, 0.0);
                }
            }
        }
    }
    p.rec[i] = code;
    p.pd[i] = pd;
    if (p.angle) p.angle[i] = ang;
}

// Accumulation on the receivers: area(c) = dx*dy + sum over donors u in D8 order of area(u) * p(u -> c).
struct DinfRule {
    const unsigned char* rec;
    const double* pd;
    const double* rows;
    double* area;
    int* ndon;
    int* front[2];
    int* ctl;
    int n_rows, n_cols;
    // whether the neighbour in direction k is a receiver of u
    __device__ __forceinline__ bool gives(int u, int k) const {
        const unsigned char q = rec[u];
        return (k & 1) ? ((q & REC_D) && ((q >> 4) & 7) == k) : ((q & REC_C) && (q & 7) == k);
    }
    __device__ __forceinline__ void visit(int i, int* fout, int* cnt_next) const {
        const int r = i / n_cols, c = i - r * n_cols;
        double a = rows[(int64_t)r * UR_N + UR_AREA];
#pragma unroll
        for (int k = 0; k < 8; ++k) {  // pull from the donors
            const int rr = r + d8_dr(k), cc = c + d8_dc(k);
            if (rr < 0 || rr >= n_rows || cc < 0 || cc >= n_cols) continue;
            const int n = rr * n_cols + cc;
            const int back = (k + 4) & 7;
            if (gives(n, back)) a = a + __ldcg(area + n) * ((back & 1) ? pd[n] : 1.0 - pd[n]);
        }
        __stcg(area + i, a);
        const unsigned char q = rec[i];  // release the receivers (they exist: a receiver is a valid neighbour)
        if (q & REC_C) {
            const int k = q & 7, n = (r + d8_dr(k)) * n_cols + c + d8_dc(k);
            if (atomicSub(ndon + n, 1) == 1) fout[atomicAdd(cnt_next, 1)] = n;
        }
        if (q & REC_D) {
            const int k = (q >> 4) & 7, n = (r + d8_dr(k)) * n_cols + c + d8_dc(k);
            if (atomicSub(ndon + n, 1) == 1) fout[atomicAdd(cnt_next, 1)] = n;
        }
    }
};

// At the default bound ptxas keeps this instantiation to 32 registers and spills; one CTA per SM is the floor the
// cooperative launch needs anyway (the occupancy API sizes the grid).
template <>
__global__ void __launch_bounds__(kAccThreads, 1) k_accum<DinfRule>(DinfRule p) {
    frontier_rounds(p);
}

// donor counts and the first frontier (cells without donors); area = NaN where W is NA.
__global__ void __launch_bounds__(256) k_dinf_prep(DinfRule p, const double* w) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.n_rows * p.n_cols) return;
    if (isnan(w[i])) {
        p.area[i] = w[i];
        return;
    }
    const int r = (int)(i / p.n_cols), c = (int)(i - (int64_t)r * p.n_cols);
    int nd = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int rr = r + d8_dr(k), cc = c + d8_dc(k);
        if (rr < 0 || rr >= p.n_rows || cc < 0 || cc >= p.n_cols) continue;
        nd += p.gives(rr * p.n_cols + cc, (k + 4) & 7);
    }
    p.ndon[i] = nd;
    if (nd == 0) p.front[0][atomicAdd(p.ctl + AC_CNT, 1)] = (int)i;
}

}  // namespace upslope
