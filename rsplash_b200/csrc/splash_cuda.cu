// splash_cuda.cu -- libsplash_cuda: kernels and the C-ABI host library (see include/splash_cuda.h).
//
// Kernels (sm_100a, FP64 CUDA cores; no tensor cores -- the path is not a contraction):
//   k_cell_setup      one-shot per cell: pedotransfer soil properties, soil_info, every per-cell
//                     invariant of the day step (splash_model.cuh: cell_setup)
//   k_snow_threshold  per cell: Tt = max(tc[p_snow >= 0.5]) over the whole series
//                     (R/splash.point.R:120-122), a column reduction over the tc matrix
//   k_spin_first      per cell: the aridity year + pass 0 of the second spin_up (730 uniform days)
//   k_spin_check/rest one lock-step year pass of the cells that still spin: the check day (which is
//                     also day 1 of the next pass) with compaction, then days 2..365 of the survivors;
//                     the list sizes stay on the device, the host never waits for them
//   k_run_bulk        the run_all day loop of every cell whose spin-up is finished: 768 threads per SM, state in
//                     registers, the state half's constants in shared memory and the forcing half's read from
//                     the constant matrix (HybridCC), optionally in regime-sorted order (k_regime_*), next day's
//                     forcing staged by cp.async, outputs written with streaming stores (daily) or reduced per
//                     month in registers (monthly)
//   k_run_list        per-thread state machine (rest of the spin-up, then the day loop) for the few cells
//                     that outlive the lock-step passes; lanes fetch cells from a device-side queue
//   k_pool_*          move those stragglers (constants, state, forcing columns) into a context-wide
//                     pool so that their tile's buffers can be reused while they finish; k_pool_table computes the
//                     forcing half of their cyclic spin-up year once, k_pool_spin iterates the state half in stages,
//                     the last of which runs the branch-light day step (splash_model.cuh: day_state_fast)
//
// Host side: a context owns streams and grow-only device buffers.  A call splits the block into
// cell tiles and enqueues, per tile, a fixed kernel sequence on one of several compute streams
//   H2D(tile t+1)  ||  kernels(tiles t, t-1, ..)  ||  straggler pool  ||  D2H(tile t-1)
// without any host round trip.  With SPLASH_MEM_DEVICE the kernels read and write the caller's
// device arrays in place (no copies).  There is no host implementation of the model in this library.
#include "../../include/splash_cuda.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <map>
#include <mutex>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "splash_model.cuh"
#include "splash_host_tables.h"
#include "splash_upslope.cuh"

using namespace splash;

namespace {

constexpr int kThreads = 128;  // threads per CTA of the list-mode (non-uniform) day-loop kernels
#ifndef SPLASH_MIN_BLOCKS
#define SPLASH_MIN_BLOCKS 4
#endif
constexpr int kMinBlocks = SPLASH_MIN_BLOCKS;  // resident CTAs per SM the register allocation aims for
// Uniform kernels (every thread of the CTA runs the same days): one large CTA per SM whose warps are
// kept together by a CTA barrier per day (SPLASH_SYNC=1; 0 = none), so that they walk through the ~60 KB
// loop body together and share instruction-cache lines instead of each streaming the body from L2 on
// its own (the body is larger than the 32 KB L1.5 instruction cache; profiles/README.md).
#ifndef SPLASH_SYNC
#define SPLASH_SYNC 1
#endif
#ifndef SPLASH_UTHREADS
#define SPLASH_UTHREADS 512
#endif
#ifndef SPLASH_UBLOCKS
#define SPLASH_UBLOCKS 1
#endif
constexpr int kListThreads = 32;  // list mode: one warp per CTA, so that the few long-running warps spread over all SMs
#ifndef SPLASH_SYNC_EVERY
#define SPLASH_SYNC_EVERY 1  // barrier every n-th day (power of two)
#endif
constexpr int kSyncMask = SPLASH_SYNC_EVERY - 1;
constexpr int kSync = SPLASH_SYNC;
constexpr int kUThreads = SPLASH_UTHREADS;
constexpr int kUBlocks = SPLASH_UBLOCKS;
// Register budget of the uniform kernels: they are compiled for a CTA `kURegSlack` threads larger than
// the one launched, so that a full CTA leaves room on its SM for one-warp CTAs of the straggler pool
// (list mode, 128 registers/thread).  Without the slack a 512-thread CTA owns the whole register file
// and the long-running pool warps and the uniform kernels would exclude each other from an SM.
#ifndef SPLASH_UREG_SLACK
#define SPLASH_UREG_SLACK 64
#endif
constexpr int kUBound = kUThreads + SPLASH_UREG_SLACK;
// SPLASH_UREGS: the register cap of the uniform kernels.  A full 512-thread CTA at 104 registers leaves 12 288 registers
// of its SM free: three one-warp CTAs of the straggler pool (128 registers per thread).  Measured on the resident
// benchmark (profiles/README.md): 96 registers (what a launch bound of 576 threads gives) 3.09 s per pass, 104: 2.92 s,
// 112 / 120 / 128: faster bulk kernel alone (up to +15 %) but 3.1 - 3.9 s per pass, because pool warps and such CTAs then
// exclude each other from an SM and the straggler chain ends after the bulk launches.  SPLASH_UREGS=0: launch bound.
#ifndef SPLASH_UREGS
#define SPLASH_UREGS (SPLASH_UTHREADS > 512 ? 80 : 104)
#endif
// the bulk launch (k_run_bulk) has its own shape, see kBThreads below (the literal-order day step, SPLASH_LEVEL=0, reads
// five more constants per cell: its 39 hot ones do not fit 768 threads, so it keeps the shape of the other kernels)
#ifndef SPLASH_BULK_THREADS
#define SPLASH_BULK_THREADS (SPLASH_L1_RECIP ? 768 : SPLASH_UTHREADS)
#endif
#ifndef SPLASH_BULK_REGS
#define SPLASH_BULK_REGS (SPLASH_BULK_THREADS > 512 ? 80 : 104)
#endif
#ifndef SPLASH_BULK_RELOAD
#define SPLASH_BULK_RELOAD 1
#endif
#define SPLASH_BULK_BOUNDS __maxnreg__(SPLASH_BULK_REGS)
#if SPLASH_UREGS > 0
#define SPLASH_UNIFORM_BOUNDS __maxnreg__(SPLASH_UREGS)
#else
#define SPLASH_UNIFORM_BOUNDS __launch_bounds__(kUBound, kUBlocks)
#endif
constexpr int kSpinYear = 365; // R/splash.point.R:141-152: the spin-up year is always 365 days

__constant__ MonthTab c_month_tab;

// -DSPLASH_BOUNDS_CHECK: every index that comes out of a device-side list, queue or pool range is checked before it
// is used; the first violation is recorded (site id) and fails the call.  compute-sanitizer is not available on the
// pool's boxes, this build stands in for it in one GPU test (tests/test_cluster_gpu.py).
#ifdef SPLASH_BOUNDS_CHECK
__device__ unsigned long long g_bounds_err = 0;
#define SPLASH_CHECK(cond, site)                                          \
    do {                                                                  \
        if (!(cond)) {                                                    \
            atomicCAS(&g_bounds_err, 0ULL, (unsigned long long)(site));   \
            return;                                                       \
        }                                                                 \
    } while (0)
#else
#define SPLASH_CHECK(cond, site) \
    do {                         \
    } while (0)
#endif

// ---------------------------------------------------------------------------------------------
// accessors for the per-cell constant matrix
// ---------------------------------------------------------------------------------------------
struct StridedCC {  // column of a [NCC][stride] matrix (shared or global memory)
    double* base;
    int64_t stride;
    __device__ __forceinline__ double& operator()(int k) const { return base[(int64_t)k * stride]; }
};

// Shapes of the uniform kernels.  The day step keeps 52 constants per cell; as private shared-memory columns they cap a
// CTA at 512 cells (213 KB), i.e. four warps per scheduler -- too few to hide the FP64 dependency latency (ncu r02:
// 3.6 cycles of fixed-latency wait per issued instruction).  A kernel compiled for more than 512 threads keeps only the
// constants of the state half (the dependent chain) in shared memory and reads the 18 that the forcing half and the
// output stage use -- state-independent, so their loads are issued at the top of the day and are not waited for until
// the forcing half needs them -- from the constant matrix in global memory (L2 hits: 15 MB for the whole device).
// The bulk launch runs 768 threads x 80 registers = six warps per scheduler (+8 % on the kernel alone, measured; the
// spin-up kernels keep 512 threads: their late rounds are short lists, where larger CTAs were measured slower).
constexpr int kBThreads = SPLASH_BULK_THREADS;
template <int NT> __host__ __device__ constexpr bool hybrid_cc() { return NT > 512; }

// constants that only day_forcing (and the output stage) read
__host__ __device__ constexpr bool cc_cold(int k) {
    return k == C_ELEV_K || k == C_LAT_K || k == C_TT || k == C_COS_LAT || k == C_SIN_LAT || k == C_SIN_S || k == C_COS_S ||
           k == C_COS_A || k == C_SIN_A || k == C_TAU_O || k == C_TAU_A || k == C_PATM || k == C_PBAR || k == C_PBARF ||
           k == C_VISC0 || k == C_INTPERM || k == C_INV_TAU_B || k == C_WRR;
}
__host__ __device__ constexpr int cc_hot_slot(int k) {  // rank of constant k among the hot ones
    int n = 0;
    for (int j = 0; j < k; ++j) n += cc_cold(j) ? 0 : 1;
    return n;
}
constexpr int kHotCC = cc_hot_slot(NCC_DAY);
static_assert(kHotCC + 18 == NCC_DAY && cc_hot_slot(0) == 0 && !cc_cold(C_RES) && cc_cold(C_WRR) && cc_cold(C_TT),
              "hot / cold split of the day step's constants");

template <int NT>
struct HybridCC {  // read-only: hot constants from the thread's shared-memory column, cold ones from the global matrix
    const double* hot;
    const double* cold;  // p.cc + c
    int64_t gstride;
    __device__ __forceinline__ double operator()(int k) const {
        return cc_cold(k) ? __ldg(cold + (int64_t)k * gstride) : hot[cc_hot_slot(k) * NT];
    }
};

template <typename T>
__device__ __forceinline__ double ld_stream(const T* p) {
    return (double)__ldcs(p);
}

// ---------------------------------------------------------------------------------------------
// K1: per-cell setup
// ---------------------------------------------------------------------------------------------
struct SetupParams {
    const double *lat, *elev, *slop, *asp, *resolution;
    const double* soil;  // [6][soil_pitch]
    int64_t soil_pitch;
    const double* au;    // [au_layers][au_pitch]
    int64_t au_pitch;
    int au_layers;
    int n_cells;
    double* cc;          // [NCC][cpitch]
    int64_t cpitch;
    double* diag;        // [SPLASH_NDIAG][dpitch] or null
    int64_t dpitch;
};

__global__ void __launch_bounds__(128) k_cell_setup(SetupParams p) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cells) return;
    CellInputs in;
    in.lat = p.lat[c];
    in.elev = p.elev[c];
    in.slop = p.slop[c];
    in.asp = p.asp[c];
    in.resolution = p.resolution[c];
    in.sand = p.soil[0 * p.soil_pitch + c];
    in.clay = p.soil[1 * p.soil_pitch + c];
    in.om = p.soil[2 * p.soil_pitch + c];
    in.gravel = p.soil[3 * p.soil_pitch + c];
    in.bd = p.soil[4 * p.soil_pitch + c];
    in.depth = p.soil[5 * p.soil_pitch + c];
    in.au = p.au[c];
    if (p.au_layers == 1) {  // R/splash.point.R:106-110
        in.cellin = 3;
        in.cellout = 3;
    } else {                 // :111-115
        in.cellin = p.au[1 * p.au_pitch + c];
        in.cellout = p.au[2 * p.au_pitch + c];
    }
    StridedCC cc{p.cc + c, p.cpitch};
    CellDiag dg;
    cell_setup(cc, in, dg);
    if (p.diag) {
        double* d = p.diag + c;
        d[SPLASH_DIAG_SAT * p.dpitch] = dg.sat;
        d[SPLASH_DIAG_WP * p.dpitch] = dg.wp;
        d[SPLASH_DIAG_FC * p.dpitch] = dg.fc;
        d[SPLASH_DIAG_KSAT * p.dpitch] = dg.ksat;
        d[SPLASH_DIAG_LAMBDA * p.dpitch] = dg.lambda;
        d[SPLASH_DIAG_DEPTH * p.dpitch] = dg.depth;
        d[SPLASH_DIAG_BUB * p.dpitch] = dg.bub;
        d[SPLASH_DIAG_RES * p.dpitch] = dg.res;
        d[SPLASH_DIAG_WMAX_R * p.dpitch] = dg.wmax_r;
    }
}

// ---------------------------------------------------------------------------------------------
// K0: snowfall threshold temperature
// ---------------------------------------------------------------------------------------------
template <typename FT>
__global__ void __launch_bounds__(256) k_snow_threshold(const FT* __restrict__ tc, int64_t fpitch, int n_days,
                                                        int n_cells, double* cc, int64_t cpitch, double* diag,
                                                        int64_t dpitch, int* frost) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells) return;
    StridedCC ccg{cc + c, cpitch};
    // Tt <- max(tc[p_snow >= 0.5]); an NA probability makes the result NA, an empty set gives -Inf
    double Tt = -INFINITY;
    bool any_na = false;
    int n_snow = 0, n_frost = 0;
    const FT* col = tc + c;
#pragma unroll 4
    for (int d = 0; d < n_days; ++d) {
        const double t = ld_stream(col + (int64_t)d * fpitch);
        n_frost += (t < 0.0) ? 1 : 0;
        const int snowy = snow_class(ccg, t);
        if (snowy < 0) {
            any_na = true;
        } else if (snowy) {
            ++n_snow;
            if (t > Tt) Tt = t;
        }
    }
    if (any_na) Tt = nan("");
    ccg(C_TT) = Tt;
    if (frost) frost[c] = n_frost;
    if (diag) {
        diag[SPLASH_DIAG_TT * dpitch + c] = Tt;
        diag[SPLASH_DIAG_SNOW_DAYS * dpitch + c] = (double)n_snow;
    }
}

// ---------------------------------------------------------------------------------------------
// Spin-up and daily integration
//
// Per-cell work state kept in global memory between launches (pitch = tile pitch):
//   st[5]      wn, snow, qin, td, nd at the end of the last completed year pass (E_k)
//   w1         wn after day 1 of that pass (wn_vec[0], SPLASH.cpp:1672,1727)
//   snap[5]    snapshot of an earlier E_j for exact cycle detection
//   passes     completed year passes k of the second spin_up call (spin_count, SPLASH.cpp:1696)
//   snap_pass  j
//   status     ST_ACTIVE (still spinning) / ST_READY_BULK / ST_READY_LATE (spin-up finished)
// ---------------------------------------------------------------------------------------------
enum : int { ST_ACTIVE = 0, ST_READY_BULK = 1, ST_EXPORTED = 3 };
constexpr int kMaxRounds = 32;  // upper bound of lock-step year passes per tile
constexpr int kRegimeKeys = 128; // buckets of the regime sort (k_regime_*)

// Device-resident control block of one tile.  Everything the kernels of a tile need to know about
// the sizes of its lists lives here, so the host enqueues the whole tile without waiting.
struct TileCtl {
    unsigned long long cnt[kMaxRounds + 2];  // cnt[r]: cells in spin list r (cnt[0] = cells of the tile)
    unsigned long long spin_days;            // spin-up cell-days executed (incl. check days)
    unsigned long long unconverged;          // cells that hit the pass limit
    unsigned long long cycles;               // cells cut short by exact cycle detection
    unsigned long long pool_base, pool_end;  // this tile's range of the straggler pool
    unsigned long long pool_head;            // work-fetch cursor of the pool's daily-integration launch
    unsigned long long spin_head;            // work-fetch cursor of the pool's first spin-up stage
    unsigned long long hard_n[4], hard_head[4];  // hard_n[s]: cells that exceeded stage s's pass budget; cursor of the stage that reads them
    unsigned long long decl_n, decl_head;    // cells of the last stage that keep declining the branch-light day step (guarded route)
    unsigned long long tail_head, tail_end;  // leftovers that did not fit the pool: finished in the tile
    unsigned long long max_chain;            // most year passes executed by one thread of a list-mode launch
    unsigned long long n_ready;              // cells in the regime-sorted order of the bulk launch
    unsigned long long regime[kRegimeKeys];  // regime sort: bucket counts, then bucket cursors
};

struct Work {
    double* st;
    double* w1;
    double* snap;
    int* passes;
    int* snap_pass;
    int* status;
    int* frost;          // days with tc < 0 (k_snow_threshold): a key of the regime sort (null in the pool's view)
    unsigned char* key;  // regime-sort bucket of the cell
    int64_t pitch;
};

struct RunParams {
    const void *sw, *pn;       // [n_days][fpitch]
    int64_t fpitch;
    const void* tc;            // [n_days][tpitch]
    int64_t tpitch;
    const void *sw1, *pn1;     // the first min(n_days, 365) rows of sw / pn, [..][f1pitch]: all the spin-up reads of them
    int64_t f1pitch;           // (host-fed calls upload them ahead of the full series; otherwise sw1 == sw, pn1 == pn)
    double* cc;                // [NCC][cpitch]
    int64_t cpitch;
    const DayTab* dtab;        // [n_days]
    const DayTab* dtab_spin;   // [365], year = year[0], n = 1..365
    int n_days;
    int n_cells;               // cells of the tile
    Work w;
    int* lists[2];             // ping-pong spin lists of the tile: list r lives in lists[r & 1] (list 0 = identity)
    const int* order;          // k_run_bulk: regime-sorted cell order (ctl->n_ready entries); null = identity
    int* order_w;              // ... as written by k_regime_scatter
    int round;                 // k_spin_check / k_spin_rest: lock-step round r
    TileCtl* ctl;              // the tile's control block
    // k_run_list: lanes fetch i from *q_head while i < *q_end; cell = q_list ? q_list[i] : i
    unsigned long long* q_head;
    const unsigned long long* q_end;
    const int* q_list;
    double* out[9];            // [n_out][opitch]; null = skip
    int64_t opitch;
    double* diag;              // [SPLASH_NDIAG][dpitch] or null
    int64_t dpitch;
    int max_spin;
    double spin_tol;
};

// Neumaier-compensated sum: R's sum() accumulates in 80-bit long double (summary.c), the device
// has no such type; the compensation keeps the aridity index within an ulp of that result.
struct CompSum {
    double s = 0.0, c = 0.0;
    __device__ __forceinline__ void add(double x) {
        const double t = s + x;
        c += (fabs(s) >= fabs(x)) ? ((s - t) + x) : ((x - t) + s);
        s = t;
    }
    __device__ __forceinline__ double value() const { return s + c; }
};

__device__ __forceinline__ void load_cc(const RunParams& p, int c, const StridedCC& cc) {
#pragma unroll 4
    for (int k = 0; k < NCC_DAY; ++k) cc(k) = p.cc[(int64_t)k * p.cpitch + c];
}

__device__ __forceinline__ CellState load_state(const Work& w, int c) {
    CellState s;
    s.wn = w.st[0 * w.pitch + c];
    s.snow = w.st[1 * w.pitch + c];
    s.qin = w.st[2 * w.pitch + c];
    s.td = w.st[3 * w.pitch + c];
    s.nd = w.st[4 * w.pitch + c];
    return s;
}

__device__ __forceinline__ void store_state(const Work& w, int c, const CellState& s) {
    w.st[0 * w.pitch + c] = s.wn;
    w.st[1 * w.pitch + c] = s.snow;
    w.st[2 * w.pitch + c] = s.qin;
    w.st[3 * w.pitch + c] = s.td;
    w.st[4 * w.pitch + c] = s.nd;
}

__device__ __forceinline__ bool same_bits(double a, double b) {
    return __double_as_longlong(a) == __double_as_longlong(b);
}

// forcing of spin-up day d (0..364): x[1:365] pads short series with NA, R/splash.point.R:141-144
template <typename FT>
__device__ __forceinline__ void spin_forcing(const RunParams& p, int c, int d, double& f_sw, double& f_tc, double& f_pn) {
    if (d < p.n_days) {
        const int64_t off = (int64_t)d * p.f1pitch + c;
        f_sw = ld_stream((const FT*)p.sw1 + off);
        f_tc = ld_stream((const FT*)p.tc + (int64_t)d * p.tpitch + c);
        f_pn = ld_stream((const FT*)p.pn1 + off);
    } else {
        f_sw = f_tc = f_pn = nan("");
    }
}

// Next-day forcing in flight: the uniform kernels load day d+1's three values RAW (still float / double as stored) before
// they compute day d and convert them at the top of the next iteration, so that the HBM latency of the load hides behind
// a whole day step (in capture r02 the first use of the freshly loaded forcing -- its float-to-double conversion right
// after the day barrier -- held 12.7 % of all stall samples).  `spin`: rows of the spin-up year (sw1 / tc / pn1, NA-padded).
template <typename FT>
struct RawForcing {
    FT sw, tc, pn;
};

template <typename FT>
__device__ __forceinline__ RawForcing<FT> ld_raw_main(const RunParams& p, int c, int d) {
    RawForcing<FT> r;
    const int64_t off = (int64_t)d * p.fpitch + c;
    r.sw = __ldcs((const FT*)p.sw + off);
    r.tc = __ldcs((const FT*)p.tc + (int64_t)d * p.tpitch + c);
    r.pn = __ldcs((const FT*)p.pn + off);
    return r;
}

template <typename FT>
__device__ __forceinline__ RawForcing<FT> ld_raw_spin(const RunParams& p, int c, int d) {
    RawForcing<FT> r;
    if (d < p.n_days) {
        const int64_t off = (int64_t)d * p.f1pitch + c;
        r.sw = __ldcs((const FT*)p.sw1 + off);
        r.tc = __ldcs((const FT*)p.tc + (int64_t)d * p.tpitch + c);
        r.pn = __ldcs((const FT*)p.pn1 + off);
    } else {  // x[1:365] pads short series with NA, R/splash.point.R:141-144
        r.sw = r.tc = r.pn = (FT)nan("");
    }
    return r;
}

// f32 forcing of the bulk kernel: the same one-day-ahead pipeline through shared memory with cp.async (LDGSTS): every thread
// copies its own three values of day d+1 into a two-slot ring behind the cell constants (2 x 3 x 512 x 4 B = 12 KB, which
// fits beside the 208 KB of constants; the f64 ring would not) while day d computes, and waits for its own copy group at the
// top of the next day -- no registers held across the day step, no barrier (a thread reads only what it copied itself).
__device__ __forceinline__ void cp_async_f32(float* smem_dst, const float* gmem_src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <typename FT>
struct BulkForcing {  // generic: raw values in registers (f64 forcing)
    RawForcing<FT> nxt{};
    __device__ __forceinline__ void start(const RunParams& p, int c, bool live, void*) {
        if (live && p.n_days > 0) nxt = ld_raw_main<FT>(p, c, 0);
    }
    __device__ __forceinline__ void next(const RunParams& p, int c, int d, bool live, double& f_sw, double& f_tc, double& f_pn) {
        const RawForcing<FT> cur = nxt;
        if (live && d + 1 < p.n_days) nxt = ld_raw_main<FT>(p, c, d + 1);
        f_sw = (double)cur.sw;
        f_tc = (double)cur.tc;
        f_pn = (double)cur.pn;
    }
};

template <>
struct BulkForcing<float> {  // f32: cp.async ring in shared memory
    float* ring = nullptr;   // [2][3][kBThreads], this thread's column
    __device__ __forceinline__ void issue(const RunParams& p, int c, int d) {
        float* slot = ring + (d & 1) * 3 * kBThreads;
        const int64_t off = (int64_t)d * p.fpitch + c;
        cp_async_f32(slot, (const float*)p.sw + off);
        cp_async_f32(slot + kBThreads, (const float*)p.tc + (int64_t)d * p.tpitch + c);
        cp_async_f32(slot + 2 * kBThreads, (const float*)p.pn + off);
        cp_async_commit();
    }
    __device__ __forceinline__ void start(const RunParams& p, int c, bool live, void* smem_after_cc) {
        ring = (float*)smem_after_cc + threadIdx.x;
        if (live && p.n_days > 0) issue(p, c, 0);
    }
    __device__ __forceinline__ void next(const RunParams& p, int c, int d, bool live, double& f_sw, double& f_tc, double& f_pn) {
        f_sw = f_tc = f_pn = 0.0;
        if (!live) return;
        cp_async_wait_all();
        const float* slot = ring + (d & 1) * 3 * kBThreads;
        f_sw = (double)slot[0];
        f_tc = (double)slot[kBThreads];
        f_pn = (double)slot[2 * kBThreads];
        if (d + 1 < p.n_days) issue(p, c, d + 1);
    }
};

// The loop condition of SPLASH::spin_up (SPLASH.cpp:1697) evaluated after the check day, plus exact
// cycle detection.  `Ek` is the end-of-pass state the check day started from, `chk_wn` the check
// day's soil moisture.  Returns true when another year pass has to run.
//
// Cycle detection: the year map E_{k+1} = F(E_k) is deterministic, so if E_k equals an earlier E_j
// bit for bit the sequence is periodic with p = k - j, and so is every later check (the check after
// pass q only depends on E_{q-1} and E_q).  All checks of one full period [j+1, k] have then been
// seen to fail, hence the reference would run to its pass limit; whole periods are skipped and the
// remainder simulated, which lands on exactly the state the reference reaches (Brent's scheme:
// the snapshot is refreshed at powers of two, and every 64 passes so that a cycle entered late is
// still found within 64 + period passes).
__device__ __forceinline__ bool spin_decide(const CellState& Ek, double chk_wn, double w1, int& passes, int& snap_pass,
                                            const StridedCC& snap, double tol, int max_spin, bool& hit_limit,
                                            bool& cycle_found) {
    double diff = chk_wn - w1;
    if (diff < 0) diff = w1 - chk_wn;
    bool cont = (diff > tol) && (passes < max_spin);
    cycle_found = false;
    if (cont) {
        if (snap_pass > 0 && passes > snap_pass && same_bits(Ek.wn, snap(0)) && same_bits(Ek.snow, snap(1)) &&
            same_bits(Ek.qin, snap(2)) && same_bits(Ek.td, snap(3)) && same_bits(Ek.nd, snap(4))) {
            const int period = passes - snap_pass;
            passes += ((max_spin - passes) / period) * period;
            cycle_found = true;
            if (passes >= max_spin) cont = false;
        } else if ((passes & (passes - 1)) == 0 || (passes & 63) == 0) {
            snap(0) = Ek.wn;
            snap(1) = Ek.snow;
            snap(2) = Ek.qin;
            snap(3) = Ek.td;
            snap(4) = Ek.nd;
            snap_pass = passes;
        }
    }
    hit_limit = (!cont) && (diff > tol);
    return cont;
}

// a uniform kernel's constants: all of them (StridedCC) or the hot ones (HybridCC) into the thread's shared-memory column
template <int NT>
__device__ __forceinline__ void stage_cc(const RunParams& p, int c, bool live, double* s_cc, StridedCC& cc) {
    cc = StridedCC{s_cc + threadIdx.x, NT};
    if (live) load_cc(p, c, cc);
}
template <int NT>
__device__ __forceinline__ void stage_cc(const RunParams& p, int c, bool live, double* s_cc, HybridCC<NT>& cc) {
    cc = HybridCC<NT>{s_cc + threadIdx.x, p.cc + c, p.cpitch};
    if (live) {
#pragma unroll
        for (int k = 0; k < NCC_DAY; ++k)
            if (!cc_cold(k)) s_cc[cc_hot_slot(k) * NT + threadIdx.x] = p.cc[(int64_t)k * p.cpitch + c];
    }
}
template <int NT> using ShapeCC = std::conditional_t<hybrid_cc<NT>(), HybridCC<NT>, StridedCC>;
template <int NT> __host__ __device__ constexpr int staged_cc() { return hybrid_cc<NT>() ? kHotCC : (int)NCC_DAY; }  // constants per cell in shared memory

// lateral_consts on a uniform kernel's constants: the four results go to the thread's shared-memory column and to the
// constant matrix (HybridCC is read-only, so the arithmetic runs on a scratch copy of the three inputs)
struct ScratchCC {
    double v[NCC];
    __device__ __forceinline__ double& operator()(int k) { return v[k]; }
};
template <int NT>
__device__ __forceinline__ void apply_lateral(const RunParams& p, int c, double* s_cc, const ShapeCC<NT>& cc, double AI) {
    ScratchCC t;
    t(C_SIDOCT) = cc(C_SIDOCT);
    t(C_DEPTH) = cc(C_DEPTH);
    t(C_AI) = cc(C_AI);
    lateral_consts(t, AI);
    constexpr int out[4] = {C_CELLOUT, C_CQ0, C_ACSQS, C_CT};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int k = out[j];
        s_cc[(hybrid_cc<NT>() ? cc_hot_slot(k) : k) * NT + threadIdx.x] = t(k);
        p.cc[(int64_t)k * p.cpitch + c] = t(k);
    }
}

// ---- K2a: aridity pass + pass 0 of the second spin_up, all cells, 730 uniform days ---------------
template <typename FT>
__global__ void SPLASH_UNIFORM_BOUNDS k_spin_first(RunParams p) {
    extern __shared__ double s_cc[];
    const int c = blockIdx.x * kUThreads + threadIdx.x;
    const bool live = c < p.n_cells;  // threads past the tile's end idle through the loop: every thread reaches every barrier
    ShapeCC<kUThreads> cc;
    stage_cc<kUThreads>(p, live ? c : 0, live, s_cc, cc);
    const double RES = live ? cc(C_RES) : 0.0;
    CellState st;
    st.wn = RES;  // cold start of SPLASH::spin_up, SPLASH.cpp:1633-1639
    st.snow = st.qin = st.td = st.nd = 0.0;
    CompSum sum_pet, sum_p;  // aridity index, R/splash.point.R:147-150
    double AI = nan("");
    double w1 = 0.0;
    RawForcing<FT> nxt{};
    if (live) nxt = ld_raw_spin<FT>(p, c, 0);
    for (int it = 0; it < 2 * kSpinYear; ++it) {
        const int d = (it < kSpinYear) ? it : it - kSpinYear;
        const RawForcing<FT> cur = nxt;
        if (live && it + 1 < 2 * kSpinYear) nxt = ld_raw_spin<FT>(p, c, (d + 1 == kSpinYear) ? 0 : d + 1);
        const double f_sw = (double)cur.sw, f_tc = (double)cur.tc, f_pn = (double)cur.pn;
        const DayTab dt = p.dtab_spin[d];
        DayOut o;
        double rain, snowfall;
        if (kSync >= 1 && (it & kSyncMask) == 0) __syncthreads();
        if (!live) continue;
        splash_day(cc, dt, c_month_tab, f_sw, f_tc, f_pn, st, o, rain, snowfall);
        if (it < kSpinYear) {
            // first spin_up call: only its pass-0 pet is consumed (R/splash.point.R:148-150)
            if (!isnan(o.pet)) sum_pet.add(o.pet);
            const double P = rain + snowfall;
            if (!isnan(P)) sum_p.add(P);
            if (it == kSpinYear - 1) {
                AI = sum_pet.value() / sum_p.value();
                apply_lateral<kUThreads>(p, c, s_cc, cc, AI);  // soil_info[12] <- AI lands in the `cellout` slot (SURVEY B-3)
                st.wn = RES;
                st.snow = st.qin = st.td = st.nd = 0.0;
            }
        } else if (it == kSpinYear) {
            w1 = st.wn;
        }
    }
    if (!live) return;
    store_state(p.w, c, st);
    p.w.w1[c] = w1;
    p.w.passes[c] = 1;
    p.w.snap_pass[c] = 0;
    p.w.status[c] = ST_ACTIVE;
    if (p.diag) p.diag[SPLASH_DIAG_AI * p.dpitch + c] = AI;
    atomicAdd(&p.ctl->spin_days, (unsigned long long)(2 * kSpinYear));
}

// ---- K2b: round r, the check day of every cell of spin list r, then compaction into list r+1 ---------
template <typename FT>
__global__ void __launch_bounds__(kThreads, kMinBlocks) k_spin_check(RunParams p) {
    extern __shared__ double s_cc[];
    const int r = p.round;
    const unsigned long long i = (unsigned long long)blockIdx.x * kThreads + threadIdx.x;
    if (i >= p.ctl->cnt[r]) return;
    const int c = (r == 0) ? (int)i : p.lists[r & 1][i];
    SPLASH_CHECK(c >= 0 && c < p.n_cells, 101);
    StridedCC cc{s_cc + threadIdx.x, kThreads};
    load_cc(p, c, cc);
    const CellState Ek = load_state(p.w, c);
    CellState st = Ek;
    double f_sw, f_tc, f_pn;
    spin_forcing<FT>(p, c, 0, f_sw, f_tc, f_pn);
    const DayTab dt = p.dtab_spin[0];
    DayOut o;
    double rain, snowfall;
    // quick_run(1, ...) from the day-365 state, SPLASH.cpp:1674,1729; it is also day 1 of the next pass
    splash_day(cc, dt, c_month_tab, f_sw, f_tc, f_pn, st, o, rain, snowfall);
    int passes = p.w.passes[c], snap_pass = p.w.snap_pass[c];
    StridedCC snap{p.w.snap + c, p.w.pitch};
    bool hit_limit, cycle_found;
    const bool cont = spin_decide(Ek, st.wn, p.w.w1[c], passes, snap_pass, snap, p.spin_tol, p.max_spin, hit_limit, cycle_found);
    p.w.passes[c] = passes;
    p.w.snap_pass[c] = snap_pass;
    if (cycle_found) atomicAdd(&p.ctl->cycles, 1ULL);
    if (cont) {
        store_state(p.w, c, st);  // state after day 1 of pass k+1: k_spin_rest of this round continues from it
        p.w.w1[c] = st.wn;
        const unsigned long long k = atomicAdd(&p.ctl->cnt[r + 1], 1ULL);
        SPLASH_CHECK(k < (unsigned long long)p.w.pitch, 102);
        p.lists[(r + 1) & 1][k] = c;
    } else {
        // the day-365 state is handed over, not the check day's (R/splash.point.R:164-172): st stays
        p.w.status[c] = ST_READY_BULK;
        if (hit_limit) atomicAdd(&p.ctl->unconverged, 1ULL);
    }
    atomicAdd(&p.ctl->spin_days, 1ULL);
}

// ---- K2c: days 2..365 of a year pass for the (compacted) cells that continue ----------------------
template <typename FT>
__global__ void SPLASH_UNIFORM_BOUNDS k_spin_rest(RunParams p) {
    extern __shared__ double s_cc[];
    const int r = p.round;
    const unsigned long long i = (unsigned long long)blockIdx.x * kUThreads + threadIdx.x;
    const unsigned long long n_list = p.ctl->cnt[r + 1];
    if ((unsigned long long)blockIdx.x * kUThreads >= n_list) return;  // surplus CTA: all of its threads leave together
    const bool live = i < n_list;  // the list's last CTA: idle threads still reach every barrier
    const int c = live ? p.lists[(r + 1) & 1][i] : 0;
    SPLASH_CHECK(c >= 0 && c < p.n_cells && n_list <= (unsigned long long)p.n_cells, 103);
    ShapeCC<kUThreads> cc;
    stage_cc<kUThreads>(p, c, live, s_cc, cc);
    CellState st{};
    if (live) st = load_state(p.w, c);
    RawForcing<FT> nxt{};
    if (live) nxt = ld_raw_spin<FT>(p, c, 1);
    for (int d = 1; d < kSpinYear; ++d) {
        const RawForcing<FT> cur = nxt;
        if (live && d + 1 < kSpinYear) nxt = ld_raw_spin<FT>(p, c, d + 1);
        const double f_sw = (double)cur.sw, f_tc = (double)cur.tc, f_pn = (double)cur.pn;
        const DayTab dt = p.dtab_spin[d];
        DayOut o;
        double rain, snowfall;
        if (kSync >= 1 && (d & kSyncMask) == 0) __syncthreads();
        if (!live) continue;
        splash_day(cc, dt, c_month_tab, f_sw, f_tc, f_pn, st, o, rain, snowfall);
    }
    if (!live) return;
    store_state(p.w, c, st);  // E_{k+1}: end of the pass
    p.w.passes[c] += 1;
    atomicAdd(&p.ctl->spin_days, (unsigned long long)(kSpinYear - 1));
}

// ---- K2d: daily integration (run_all) ---------------------------------------------------------------
// Output stage shared by the two day-loop kernels: sm_lim (R/splash.point.R:197-200), then either the daily
// layers or the monthly reduction in registers (mean(wn, snow, sm_lim) / sum(rest), na.rm = TRUE, :210-211).
struct MonthAcc {
    double acc[9];
    int cnt[3];
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int k = 0; k < 9; ++k) acc[k] = 0.0;
        cnt[0] = cnt[1] = cnt[2] = 0;
    }
};

template <bool kMonthly>
__device__ __forceinline__ void emit_day(const RunParams& p, int c, int d, const DayTab& dt, double wrr, double RES,
                                         const CellState& st, const DayOut& o, MonthAcc& m) {
    double sm_lim = (st.wn - RES) / wrr;  // R/splash.point.R:197-200
    if (sm_lim < 0) sm_lim = 0.0;
    if (sm_lim > 1) sm_lim = 1.0;
    const double v[9] = {st.wn, o.ro, o.pet, o.aet, st.snow, o.cond, o.bflow, o.netr, sm_lim};
    if (kMonthly) {
#ifdef SPLASH_MACC_LOCAL  // experiment: a rolled loop keeps the nine sums in local memory instead of 18 registers
#pragma unroll 1
#else
#pragma unroll
#endif
        for (int k = 0; k < 9; ++k)
            if (!isnan(v[k])) m.acc[k] += v[k];
        if (!isnan(v[0])) ++m.cnt[0];
        if (!isnan(v[4])) ++m.cnt[1];
        if (!isnan(v[8])) ++m.cnt[2];
        const bool last = (d + 1 == p.n_days) || (p.dtab[d + 1].group != dt.group);
        if (last) {
            const int64_t off = (int64_t)dt.group * p.opitch + c;
            const double m0 = m.cnt[0] ? m.acc[0] / m.cnt[0] : nan("");
            const double m4 = m.cnt[1] ? m.acc[4] / m.cnt[1] : nan("");
            const double m8 = m.cnt[2] ? m.acc[8] / m.cnt[2] : nan("");
            const double w[9] = {m0, m.acc[1], m.acc[2], m.acc[3], m4, m.acc[5], m.acc[6], m.acc[7], m8};
#pragma unroll
            for (int k = 0; k < 9; ++k)
                if (p.out[k]) __stcs(p.out[k] + off, w[k]);
            m.clear();
        }
    } else {
        const int64_t off = (int64_t)d * p.opitch + c;
#pragma unroll
        for (int k = 0; k < 9; ++k)
            if (p.out[k]) __stcs(p.out[k] + off, v[k]);
    }
}

// Bulk launch: the run_all day loop of every cell of the tile whose spin-up is finished, one thread per cell,
// uniform day loop (every live thread of the CTA runs days 0..n_days-1; the CTA meets at a barrier per day).
// Thread i integrates cell p.order[i] (i < ctl->n_ready): the tile's cells regime-sorted by k_regime_*, so that
// the cells of a warp take the same branches of the day step more often (flat / sloped, deep / shallow soil,
// frost and snow frequency, aridity); without an order (the default: the sort was measured slower on the synthetic grid,
// whose divergence is day-to-day weather, not regime), cell i.
template <typename FT, bool kMonthly>
__global__ void SPLASH_BULK_BOUNDS k_run_bulk(RunParams p) {
    extern __shared__ double s_cc[];
    const long long i0 = (long long)blockIdx.x * kBThreads;
    const long long n_run = p.order ? (long long)p.ctl->n_ready : (long long)p.n_cells;
    if (i0 >= n_run) return;  // surplus CTA: all of its threads leave together
    const long long i = i0 + threadIdx.x;
    int c = 0;
    bool live = i < n_run;
    if (live) {
        c = p.order ? p.order[i] : (int)i;
        SPLASH_CHECK(c >= 0 && c < p.n_cells && n_run <= (long long)p.n_cells, 104);
        live = p.w.status[c] == ST_READY_BULK;
    }
    ShapeCC<kBThreads> cc;
    stage_cc<kBThreads>(p, c, live, s_cc, cc);
    CellState st{};
    double RES = 0.0, wrr = 1.0;
    if (live) {
        RES = cc(C_RES);
        wrr = cc(C_WRR);
        st = load_state(p.w, c);
    }
    int n_snowfall = 0;
    MonthAcc macc;
    macc.clear();
    BulkForcing<FT> pipe;
    pipe.start(p, c, live, s_cc + (size_t)staged_cc<kBThreads>() * kBThreads);
    for (int d = 0; d < p.n_days; ++d) {
        double f_sw, f_tc, f_pn;
        pipe.next(p, c, d, live, f_sw, f_tc, f_pn);
        const DayTab dt = p.dtab[d];
        if (kSync >= 1 && (d & kSyncMask) == 0) __syncthreads();
        if (!live) continue;
        DayOut o;
        double rain, snowfall;
        splash_day(cc, dt, c_month_tab, f_sw, f_tc, f_pn, st, o, rain, snowfall);
        if (snowfall > 0.0) ++n_snowfall;
#if SPLASH_BULK_RELOAD  // RES and Wmax_R - RES re-read per day: four registers less across the day step (+1.5 %, measured)
        emit_day<kMonthly>(p, c, d, dt, cc(C_WRR), cc(C_RES), st, o, macc);
#else
        emit_day<kMonthly>(p, c, d, dt, wrr, RES, st, o, macc);
#endif
    }
    if (!live) return;
    store_state(p.w, c, st);
    if (p.diag) p.diag[SPLASH_DIAG_SNOWFALL_DAYS * p.dpitch + c] = (double)n_snowfall;
}

// List mode: a per-thread state machine for the few cells that outlive the lock-step rounds (the straggler pool,
// and leftovers that did not fit into it).  Each lane fetches a cell from the device-side queue
// (q_head/q_end/q_list), finishes its spin-up if it is still ST_ACTIVE (per-thread loop with the reference's
// convergence test and exact cycle detection), integrates its days, and fetches the next one.
enum Phase : int { PH_DONE = -1, PH_SPIN = 1, PH_MAIN = 2 };

template <typename FT, bool kMonthly>
__global__ void __launch_bounds__(kListThreads, 16) k_run_list(RunParams p) {
    constexpr int NT = kListThreads;
    extern __shared__ double s_cc[];
    StridedCC cc{s_cc + threadIdx.x, NT};
    StridedCC snap{s_cc + (int64_t)NCC_DAY * NT + threadIdx.x, NT};  // 5 private slots after the constants
    unsigned long long spin_days = 0;
    int max_chain = 0;

    for (;;) {
        const unsigned long long i = atomicAdd(p.q_head, 1ULL);
        if (i >= *p.q_end) break;
        const int c = p.q_list ? p.q_list[i] : (int)i;
        SPLASH_CHECK(c >= 0 && c < p.n_cells, 105);
        const int status = p.w.status[c];
        load_cc(p, c, cc);

        const FT* sw_col = (const FT*)p.sw + c;
        const FT* tc_col = (const FT*)p.tc + c;
        const FT* pn_col = (const FT*)p.pn + c;

        const double RES = cc(C_RES), wrr = cc(C_WRR);
        CellState st = load_state(p.w, c);
        CellState saved = st;
        int phase = (status == ST_ACTIVE) ? PH_SPIN : PH_MAIN;
        int passes = 0, snap_pass = 0, chain = 0;
        double w1 = 0.0;
        if (phase == PH_SPIN) {
            passes = p.w.passes[c];
            snap_pass = p.w.snap_pass[c];
            w1 = p.w.w1[c];
#pragma unroll
            for (int k = 0; k < 5; ++k) snap(k) = p.w.snap[(int64_t)k * p.w.pitch + c];
        }
        int d = 0;
        int n_snowfall = 0;
        MonthAcc macc;
        macc.clear();
        if (phase == PH_MAIN && p.n_days == 0) phase = PH_DONE;

        while (phase != PH_DONE) {
            // ---- forcing and day table of (phase, d) ---------------------------------------------------
            DayTab dt;
            double f_sw, f_tc, f_pn;
            if (phase == PH_MAIN) {
                dt = p.dtab[d];
                const int64_t off = (int64_t)d * p.fpitch;
                f_sw = ld_stream(sw_col + off);
                f_tc = ld_stream(tc_col + (int64_t)d * p.tpitch);
                f_pn = ld_stream(pn_col + off);
            } else {
                dt = p.dtab_spin[d];
                spin_forcing<FT>(p, c, d, f_sw, f_tc, f_pn);
                if (d == 0) saved = st;  // E_k: state of day 365 before the check day
            }
            DayOut o;
            double rain, snowfall;
            splash_day(cc, dt, c_month_tab, f_sw, f_tc, f_pn, st, o, rain, snowfall);

            if (phase == PH_MAIN) {
                if (snowfall > 0.0) ++n_snowfall;
                emit_day<kMonthly>(p, c, d, dt, wrr, RES, st, o, macc);
                if (++d == p.n_days) phase = PH_DONE;
            } else {  // PH_SPIN: the rest of the second spin_up call, SPLASH.cpp:1697-1743
                ++spin_days;
                bool cont = true;
                if (d == 0) {
                    bool hit_limit, cycle_found;
                    cont = spin_decide(saved, st.wn, w1, passes, snap_pass, snap, p.spin_tol, p.max_spin, hit_limit, cycle_found);
                    if (hit_limit) atomicAdd(&p.ctl->unconverged, 1ULL);
                    if (cycle_found) atomicAdd(&p.ctl->cycles, 1ULL);
                    w1 = st.wn;
                }
                if (!cont) {
                    st = saved;  // hand over the day-365 state, not the check day's
                    d = 0;
                    phase = (p.n_days > 0) ? PH_MAIN : PH_DONE;
                } else if (++d == kSpinYear) {
                    d = 0;
                    ++passes;
                    ++chain;
                }
            }
        }

        store_state(p.w, c, st);
        if (p.diag) p.diag[SPLASH_DIAG_SNOWFALL_DAYS * p.dpitch + c] = (double)n_snowfall;
        if (status == ST_ACTIVE) {
            p.w.passes[c] = passes;
            if (p.diag) p.diag[SPLASH_DIAG_SPIN_PASSES * p.dpitch + c] = (double)passes;
        }
        if (chain > max_chain) max_chain = chain;
    }
    if (spin_days) atomicAdd(&p.ctl->spin_days, spin_days);
    if (max_chain) atomicMax(&p.ctl->max_chain, (unsigned long long)max_chain);
}

// ---- regime sort: a counting sort of the tile's finished cells by a key that predicts which branches of the
//      day step a cell takes (k_run_bulk runs the cells in this order; results do not depend on it) -------------
__device__ __forceinline__ int regime_key(const RunParams& p, int c) {
    const double tan_s = p.cc[(int64_t)C_TAN_S * p.cpitch + c];
    const double depth = p.cc[(int64_t)C_DEPTH * p.cpitch + c];
    const double ai = p.cc[(int64_t)C_CELLOUT * p.cpitch + c];  // the aridity index sits in the cellout slot (SURVEY B-3)
    const double sat = p.cc[(int64_t)C_SAT * p.cpitch + c];
    if (isnan(sat) || isnan(ai) || isnan(tan_s)) return kRegimeKeys - 1;  // NA cells together
    const int flat = (tan_s == 0.0) ? 1 : 0;
    const int deep = (depth >= 2.0) ? 1 : 0;
    const int nd = p.n_days > 0 ? p.n_days : 1;
    const int frost = p.w.frost[c];  // days with tc < 0 (viscosity is a cell constant there), k_snow_threshold
    const int fq = (frost == 0) ? 0 : ((8 * (long long)frost) / nd >= 7 ? 3 : ((2 * (long long)frost >= nd) ? 2 : 1));
    const int wq = (ai < 0.6) ? 0 : (ai < 1.2) ? 1 : (ai < 2.5) ? 2 : 3;  // humid ... arid
    return ((flat * 2 + deep) * 4 + fq) * 4 + wq;  // 0..63
}

__global__ void __launch_bounds__(256) k_regime_count(RunParams p) {
    __shared__ unsigned int h[kRegimeKeys];
    for (int k = threadIdx.x; k < kRegimeKeys; k += blockDim.x) h[k] = 0;
    __syncthreads();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < p.n_cells && p.w.status[c] == ST_READY_BULK) {
        const int key = regime_key(p, c);
        p.w.key[c] = (unsigned char)key;
        atomicAdd(&h[key], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < kRegimeKeys; k += blockDim.x)
        if (h[k]) atomicAdd(&p.ctl->regime[k], (unsigned long long)h[k]);
}

__global__ void k_regime_scan(TileCtl* ctl) {  // one thread: bucket counts -> bucket cursors
    unsigned long long run = 0;
    for (int k = 0; k < kRegimeKeys; ++k) {
        const unsigned long long n = ctl->regime[k];
        ctl->regime[k] = run;
        run += n;
    }
    ctl->n_ready = run;
}

__global__ void __launch_bounds__(256) k_regime_scatter(RunParams p) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < p.n_cells && p.w.status[c] == ST_READY_BULK) {
        const unsigned long long k = atomicAdd(&p.ctl->regime[p.w.key[c]], 1ULL);
        SPLASH_CHECK(p.w.key[c] < kRegimeKeys && k < (unsigned long long)p.n_cells, 106);
        p.order_w[k] = c;
    }
}

// ---------------------------------------------------------------------------------------------
// Straggler pool.  The cells still spinning after a tile's lock-step rounds (a fraction of a
// percent, but each may need up to 1000 year passes) are copied out of the tile -- constants, work
// state and their forcing columns -- so that the tile's buffers can be reused while list-mode
// launches finish them on their own streams.  Results are scattered to the caller's arrays at the
// end of the call.
// ---------------------------------------------------------------------------------------------
constexpr int kDayPrePad = (kDayPreDoubles + 1) / 2 * 2;  // DayPre padded to whole 16-byte words

struct Pool {
    void* f[3];          // [n_days][cap] forcing columns (same element type as the call's forcing)
    double* cc;          // [NCC][cap]
    Work w;              // pitch = cap
    double* out[9];      // [n_out][cap]; null = layer not requested
    double* diag;        // [SPLASH_NDIAG][cap] (only the rows written by list mode are used)
    long long* cell;     // [cap] index of the cell in the caller's arrays
    double* table;       // [cap][365][kDayPrePad] forcing half of the cyclic spin-up year (k_pool_table): one
                         // contiguous 176-byte record per (cell, day), read by its lane with eleven 16-byte loads
    int* hard[2];        // [cap] each, per tile range, ping-pong: pool cells handed from one spin-up stage to the next
    unsigned long long* count;  // entries handed out so far
    long long cap;
};

// one thread: reserve this tile's range of the pool for the leftovers of its last spin list
__global__ void k_pool_reserve(TileCtl* ctl, int last_list, unsigned long long* pool_count, long long cap) {
    const unsigned long long n = ctl->cnt[last_list];
    const unsigned long long base = atomicAdd(pool_count, n);
    unsigned long long fit = 0;
    if (base < (unsigned long long)cap) fit = ((unsigned long long)cap - base < n) ? (unsigned long long)cap - base : n;
    ctl->pool_base = base;
    ctl->pool_end = base + fit;
    ctl->pool_head = base;
    ctl->spin_head = base;
    ctl->tail_head = fit;  // entries [fit, n) of the last list stay in the tile
    ctl->tail_end = n;
}

// part 1: per-entry records and the spin-up year's forcing rows (from sw1 / tc / pn1); part 2: the forcing rows
// of the whole series (from sw / tc / pn).  Host-fed calls run part 1 as soon as a tile has spun up and part 2
// once the tile's full series has arrived; otherwise both run together (part 3).
template <typename FT>
__global__ void __launch_bounds__(256) k_pool_export(RunParams p, Pool pool, int last_list, long long cell0, int part) {
    const TileCtl* ctl = p.ctl;
    const unsigned long long base = ctl->pool_base;
    const long long n = (long long)(ctl->pool_end - base);
    if (n <= 0) return;
    const int* list = (last_list == 0) ? nullptr : p.lists[last_list & 1];
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // per-entry records
    for (long long e = tid; (part & 1) && e < n; e += nthreads) {
        const int c = list ? list[e] : (int)e;
        const long long j = (long long)base + e;
        SPLASH_CHECK(c >= 0 && c < p.n_cells && j >= 0 && j < pool.cap, 107);
        for (int k = 0; k < NCC; ++k) pool.cc[(long long)k * pool.cap + j] = p.cc[(int64_t)k * p.cpitch + c];
        for (int k = 0; k < 5; ++k) {
            pool.w.st[(long long)k * pool.cap + j] = p.w.st[(int64_t)k * p.w.pitch + c];
            pool.w.snap[(long long)k * pool.cap + j] = p.w.snap[(int64_t)k * p.w.pitch + c];
        }
        pool.w.w1[j] = p.w.w1[c];
        pool.w.passes[j] = p.w.passes[c];
        pool.w.snap_pass[j] = p.w.snap_pass[c];
        pool.w.status[j] = ST_ACTIVE;
        pool.cell[j] = cell0 + c;
        p.w.status[c] = ST_EXPORTED;
    }
    // forcing columns: consecutive threads write consecutive pool entries of one day
    const bool whole = (part & 2) != 0;
    const long long rows = whole ? (long long)p.n_days : (long long)(p.n_days < kSpinYear ? p.n_days : kSpinYear);
    const void* src_sw = whole ? p.sw : p.sw1;
    const void* src_pn = whole ? p.pn : p.pn1;
    const long long spitch = whole ? p.fpitch : p.f1pitch;
    for (long long q = tid; q < n * rows; q += nthreads) {
        const long long d = q / n, e = q - d * n;
        const int c = list ? list[e] : (int)e;
        const long long dst = d * pool.cap + (long long)base + e;
        SPLASH_CHECK(c >= 0 && c < p.n_cells && (long long)base + e < pool.cap, 108);
        ((FT*)pool.f[0])[dst] = ((const FT*)src_sw)[d * spitch + c];
        ((FT*)pool.f[1])[dst] = ((const FT*)p.tc)[d * p.tpitch + c];
        ((FT*)pool.f[2])[dst] = ((const FT*)src_pn)[d * spitch + c];
    }
}

// The spin-up year is cyclic: the forcing half of each of its 365 days (day_forcing) is the same in
// every pass, and a straggler runs up to 1000 of them.  One thread per (pool cell, day) computes it
// once; k_pool_spin then only iterates the state half.  `p` is the pool's view (arrays of pitch cap).
template <typename FT>
__global__ void __launch_bounds__(128) k_pool_table(RunParams p, Pool pool) {
    const TileCtl* ctl = p.ctl;
    const long long base = (long long)ctl->pool_base;
    const long long n = (long long)ctl->pool_end - base;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n * kSpinYear; q += nthreads) {
        const int d = (int)(q / n);
        const int j = (int)(base + (q - (long long)d * n));
        SPLASH_CHECK(j >= 0 && j < pool.cap, 109);
        StridedCC cc{p.cc + j, p.cpitch};
        double f_sw, f_tc, f_pn;
        spin_forcing<FT>(p, j, d, f_sw, f_tc, f_pn);
        DayPre pre;
        day_forcing(cc, p.dtab_spin[d], c_month_tab, f_sw, f_tc, f_pn, pre);
        day_forcing_recession(cc, pre);
        const double* v = reinterpret_cast<const double*>(&pre);
        double* dst = pool.table + ((long long)j * kSpinYear + d) * kDayPrePad;
#pragma unroll
        for (int k = 0; k < kDayPreDoubles; ++k) dst[k] = v[k];
    }
}

constexpr int kFastDeclineLimit = 36;  // days of the probe pass (10 %) the branch-light route may decline before the cell goes to the guarded list
// SPLASH_CHAIN_FAST: the chain's state half through the branch-light route (day_state_fast, splash_model.cuh)
#ifndef SPLASH_CHAIN_FAST
#define SPLASH_CHAIN_FAST 1
#endif
#ifdef SPLASH_CHAIN_SHARED_MATH
using ChainMath = MathShared;
#else
using ChainMath = MathInline;
#endif

// The rest of the second spin_up call (SPLASH.cpp:1697-1743) for the pool's cells: a per-thread loop over
// year passes with the reference's convergence test and exact cycle detection, the forcing half of every
// day read from the table.  This is the longest sequential chain of the whole job (up to 1000 x 365 day
// steps for a cell that never converges), so the loop body is kept to the state half only.
//
// Stages keep the lanes busy: most pool cells converge within a few dozen more passes, a few percent
// run for hundreds.  Stage s gives every cell it receives `budget` passes; the cells that exceed it
// are appended to the tile's next `hard` list and stage s+1 runs only those, so that the warps which
// live for seconds are few and full instead of many and nearly empty (they hold SM resources all the
// while).  The last stage is launched with enough shared memory per CTA that no 512-thread CTA of the
// uniform kernels fits beside it: its warps (at most four per SM) own their SM and run the chain at
// its uncontended latency, roughly half the time per day step of a warp squeezed in beside 16 others.
//
// kBoth (the last stage when SPLASH_CHAIN_FAST): the state half through day_state_fast (splash_model.cuh), which
// shortens a lone warp's dependent chain by ~1.7x -- for the cells whose days stay inside its fast ranges.  A cell
// that keeps declining it (a column at its residual moisture, a zero air-entry pressure ...) would pay for both
// routes every day, and so would its warp.  So the last stage is two launches: a PROBE (stage 3) runs one year pass
// of every cell on the fast route and sorts the cells into two lists by the number of days declined; the FINAL
// launch (stage 4) gives its first `ctas_a` CTAs the fast route on the first list and the others the guarded route
// on the second, fewer cells per warp.  (The interleaved chains want registers: 255 per thread, no spills; the
// warps of these stages own their SM anyway.)
constexpr int kStageProbe = 3, kStageFinal = 4;
// kBoth: the next day's table record travels into a two-slot shared-memory ring (cp.async, 16-byte chunks, one column per
// lane) while the current day computes: the record's L2 latency was the loop's one long-scoreboard stall
constexpr int kTabChunks = kDayPrePad / 2;
constexpr size_t kSmemChainRing = (size_t)2 * kTabChunks * kListThreads * 16;
constexpr int kPoolDeclinerLanes = 2;  // cells per warp on the guarded route of the final launch (divergence is what it pays for)
template <bool kBoth>
__global__ void __launch_bounds__(kListThreads, kBoth ? 8 : 16) k_pool_spin(RunParams p, Pool pool, int stage, int budget, int lanes,
                                                                            int ctas_a, int lanes_b) {
    extern __shared__ double s_cc[];
    const bool role_b = kBoth && stage == kStageFinal && (int)blockIdx.x >= ctas_a;  // guarded route on the decliners
    const bool fast = kBoth && !role_b;
    if ((int)threadIdx.x >= (role_b ? lanes_b : lanes)) return;  // last stage: fewer cells per warp = fewer divergent paths per day step
    StridedCC cc{s_cc + threadIdx.x, kListThreads};
    StridedCC snap{s_cc + (int64_t)NCC_DAY * kListThreads + threadIdx.x, kListThreads};
    unsigned long long spin_days = 0;
    int max_chain = 0;
    for (;;) {
        int c;
        if (stage == 1) {
            const unsigned long long i = atomicAdd(&p.ctl->spin_head, 1ULL);
            if (i >= p.ctl->pool_end) break;
            c = (int)i;
        } else if (role_b) {  // the decliners' list grows down from the end of the tile's range
            const unsigned long long i = atomicAdd(&p.ctl->decl_head, 1ULL);
            if (i >= p.ctl->decl_n) break;
            c = pool.hard[(stage - 1) & 1][p.ctl->pool_end - 1 - i];
        } else {
            const unsigned long long i = atomicAdd(&p.ctl->hard_head[stage - 1], 1ULL);
            if (i >= p.ctl->hard_n[stage - 1]) break;
            c = pool.hard[(stage - 1) & 1][p.ctl->pool_base + i];
        }
        SPLASH_CHECK(c >= 0 && c < pool.cap && (unsigned long long)c >= p.ctl->pool_base && (unsigned long long)c < p.ctl->pool_end, 110);
        load_cc(p, c, cc);
        CellState st = load_state(p.w, c);
        CellState saved = st;
        int passes = p.w.passes[c], snap_pass = p.w.snap_pass[c], chain = 0;
        double w1 = p.w.w1[c];
#pragma unroll
        for (int k = 0; k < 5; ++k) snap(k) = p.w.snap[(int64_t)k * p.w.pitch + c];
        const double2* tab = reinterpret_cast<const double2*>(pool.table + (long long)c * kSpinYear * kDayPrePad);
        bool cont = true;
        int d = 0;
        int declined = 0;  // days of this stage that day_state_fast handed to the guarded route
        double2* const ring = reinterpret_cast<double2*>(s_cc + (size_t)(NCC_DAY + 5) * kListThreads) + threadIdx.x;  // [2][kTabChunks][lanes]
        int slot = 0;
        auto fetch = [&](int day, int into) {
#pragma unroll
            for (int k = 0; k < kTabChunks; ++k) cp_async_16(ring + (into * kTabChunks + k) * kListThreads, tab + day * kTabChunks + k);
            cp_async_commit();
        };
        if constexpr (kBoth) fetch(0, 0);
        while (cont) {
            DayPre pre;
            if constexpr (kBoth) {
                cp_async_wait_all();
                double* v = reinterpret_cast<double*>(&pre);
#pragma unroll
                for (int k = 0; k < kTabChunks; ++k) {
                    const double2 w = ring[(slot * kTabChunks + k) * kListThreads];
                    v[2 * k] = w.x;
                    if (2 * k + 1 < kDayPreDoubles) v[2 * k + 1] = w.y;
                }
                fetch((d + 1 == kSpinYear) ? 0 : d + 1, slot ^ 1);
                slot ^= 1;
            } else {
                double* v = reinterpret_cast<double*>(&pre);
                const double2* src = tab + d * (kDayPrePad / 2);
#pragma unroll
                for (int k = 0; k < kDayPrePad / 2; ++k) {
                    const double2 w = __ldg(src + k);
                    v[2 * k] = w.x;
                    if (2 * k + 1 < kDayPreDoubles) v[2 * k + 1] = w.y;
                }
                // next day's record on its way while this day computes
                const double2* nxt = tab + ((d + 1 == kSpinYear) ? 0 : d + 1) * (kDayPrePad / 2);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(nxt));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(nxt + kDayPrePad / 2 - 1));
            }
            if (d == 0) saved = st;  // E_k: state of day 365 before the check day
            DayOut o;
            if constexpr (kBoth) {
                declined += day_state_auto<ChainMath>(cc, pre, st, o, fast) ? 0 : 1;
            } else {
                day_state<ChainMath>(cc, pre, st, o);
            }
            ++spin_days;
            if (d == 0) {
                bool hit_limit, cycle_found;
                cont = spin_decide(saved, st.wn, w1, passes, snap_pass, snap, p.spin_tol, p.max_spin, hit_limit, cycle_found);
                if (hit_limit) atomicAdd(&p.ctl->unconverged, 1ULL);
                if (cycle_found) atomicAdd(&p.ctl->cycles, 1ULL);
                w1 = st.wn;
            }
            if (cont && ++d == kSpinYear) {
                d = 0;
                ++passes;
                ++chain;
                if (chain >= budget) break;  // st == E_k, the end of a pass: the next stage resumes from it
            }
        }
        if constexpr (kBoth) cp_async_wait_all();  // the record fetched ahead: its slot is free for the next cell
        if (cont) {  // budget exhausted: park the cell for the next stage
            store_state(p.w, c, st);
            p.w.w1[c] = w1;
            p.w.passes[c] = passes;
            p.w.snap_pass[c] = snap_pass;
#pragma unroll
            for (int k = 0; k < 5; ++k) p.w.snap[(int64_t)k * p.w.pitch + c] = snap(k);
            if (kBoth && stage == kStageProbe && declined > kFastDeclineLimit) {
                const unsigned long long k2 = atomicAdd(&p.ctl->decl_n, 1ULL);
                pool.hard[stage & 1][p.ctl->pool_end - 1 - k2] = c;
            } else {
                const unsigned long long k2 = atomicAdd(&p.ctl->hard_n[stage], 1ULL);
                SPLASH_CHECK(p.ctl->pool_base + k2 < p.ctl->pool_end, 111);
                pool.hard[stage & 1][p.ctl->pool_base + k2] = c;
            }
            continue;
        }
        store_state(p.w, c, saved);  // the day-365 state is handed over, not the check day's
        p.w.passes[c] = passes;
        p.w.status[c] = ST_READY_BULK;
        if (p.diag) p.diag[SPLASH_DIAG_SPIN_PASSES * p.dpitch + c] = (double)passes;
        if (chain > max_chain) max_chain = chain;
    }
    if (spin_days) atomicAdd(&p.ctl->spin_days, spin_days);
    if (max_chain) atomicMax(&p.ctl->max_chain, (unsigned long long)max_chain);
}

// device-resident outputs: write the pool's results into the caller's arrays
struct Out9 {
    double* p[9];
};

__global__ void k_pool_scatter(Pool pool, long long n, long long n_out, Out9 o9, long long ostride,
                               double* state_final, double* cell_diag, long long nc) {
    double* const* out9 = o9.p;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (int k = 0; k < 9; ++k) {
        if (!pool.out[k] || !out9[k]) continue;
        for (long long q = tid; q < n * n_out; q += nthreads) {
            const long long r = q / n, j = q - r * n;
            out9[k][r * ostride + pool.cell[j]] = pool.out[k][r * pool.cap + j];
        }
    }
    for (long long j = tid; j < n; j += nthreads) {
        const long long c = pool.cell[j];
        if (state_final) {
            for (int k = 0; k < 5; ++k) state_final[(long long)k * nc + c] = pool.w.st[(long long)k * pool.cap + j];
            state_final[5LL * nc + c] = pool.cc[(long long)C_CELLOUT * pool.cap + j];
            state_final[6LL * nc + c] = pool.cc[(long long)C_TT * pool.cap + j];
        }
        if (cell_diag) {
            cell_diag[(long long)SPLASH_DIAG_SPIN_PASSES * nc + c] = pool.diag[(long long)SPLASH_DIAG_SPIN_PASSES * pool.cap + j];
            cell_diag[(long long)SPLASH_DIAG_SNOWFALL_DAYS * nc + c] = pool.diag[(long long)SPLASH_DIAG_SNOWFALL_DAYS * pool.cap + j];
        }
    }
}

__global__ void k_finish_diag(const int* passes, double* diag, int64_t dpitch, int n) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n) diag[SPLASH_DIAG_SPIN_PASSES * dpitch + c] = (double)passes[c];
}

// ---------------------------------------------------------------------------------------------
// unSWC.grid (R/unsSWC.grid.R:14-141): unsaturated-zone diagnostics of the simulated soil water.
// A per-cell-layer map: one thread per cell keeps the cell's Brooks-Corey parameters in registers
// and walks the layers (day-major wn: each load / store is a coalesced row segment per warp).
// R's ifelse() semantics are kept: a condition on an NA operand yields NA.
// ---------------------------------------------------------------------------------------------
struct UnswcParams {
    const double* soil;  // [6][soil_pitch]
    int64_t soil_pitch;
    const double* wn;    // [n_layers][wpitch]
    int64_t wpitch;
    double *theta_i, *wtd, *w_z, *se;  // [n_layers][opitch] each; null = not wanted
    int64_t opitch;
    int64_t n_cells, n_layers;
    double uns_depth;
};

__device__ __forceinline__ double unswc_wtd(double psi_m, double totdepth, double bub) {  // :49-50, :113-115
    const double wtdini = (bub - psi_m) / 1000;
    if (isnan(wtdini) || isnan(totdepth)) return nan("");
    if (wtdini > totdepth) return totdepth;
    return (wtdini < 0) ? 0.0 : wtdini;
}

__global__ void __launch_bounds__(256) k_unswc(UnswcParams p) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cells) return;
    // soil_hydro(sand, clay, OM, fgravel = soil_data[[4]] * 0, bd), :78
    const SoilHydro sh = soil_hydro(p.soil[0 * p.soil_pitch + c], p.soil[1 * p.soil_pitch + c], p.soil[2 * p.soil_pitch + c],
                                    p.soil[3 * p.soil_pitch + c] * 0, p.soil[4 * p.soil_pitch + c]);
    const double theta_s = sh.sat, theta_r = sh.res_frac, lambda = 1 / sh.coef_B, bub = sh.bubbling_p;
    const double depth = p.soil[5 * p.soil_pitch + c];
    const double ilam = (1 / lambda);
    const double ud = p.uns_depth;
    for (int64_t l = 0; l < p.n_layers; ++l) {
        const double w = __ldcs(p.wn + l * p.wpitch + c);
        // calc_thetai, :96-103
        const double theta_o = (w / (depth * 1000));
        double theta_i;
        if (isnan(theta_o) || isnan(theta_s)) {
            theta_i = nan("");
        } else if (theta_o >= theta_s) {
            theta_i = theta_s - 0.0001;
        } else if (isnan(theta_r)) {
            theta_i = nan("");
        } else {
            theta_i = (theta_o <= theta_r) ? theta_r + 0.0001 : theta_o;
        }
#if SPLASH_LEVEL >= 1 && !defined(SPLASH_LIBDEVICE_MATH)
        // x^y as exp(y*log(x)) with the library's own exp/log (level-1 arithmetic, DESIGN.md)
        const double x = ((theta_i - theta_r) / (theta_s - theta_r));
        const double psi_m = bub / fm::pow_core(x, ilam);  // :109
#else
        const double psi_m = bub / pow((((theta_i - theta_r) / (theta_s - theta_r))), ilam);  // :109
#endif
        const double wtd = unswc_wtd(psi_m, depth, bub);                                        // :121
        // UnsWater(psi_m, z_uns, theta_r, theta_s, bub_press, lambda, depth = uns_depth), :47-70 as called at :129
        const double wtd2 = unswc_wtd(psi_m, ud, bub);
        const bool na2 = isnan(wtd2) || isnan(ud);
        const bool shallow = !na2 && (wtd2 <= ud);
        const double z_uns = na2 ? nan("") : (shallow ? wtd2 * 1000 : ud * 1000);
#if SPLASH_LEVEL >= 1 && !defined(SPLASH_LIBDEVICE_MATH)
        // both powers through the same function: at z_uns == 0 the two terms must cancel exactly, as in R
        const double pz = fm::pow_core(bub / (psi_m + z_uns), lambda);
        const double p0 = fm::pow_core(bub / (psi_m + 0), lambda);
#else
        const double pz = pow((bub / (psi_m + z_uns)), lambda);
        const double p0 = pow((bub / (psi_m + 0)), lambda);
#endif
        const double w_uns_z = theta_r * z_uns + (((psi_m + z_uns) * (theta_r - theta_s) * pz) / (lambda - 1));
        const double w_uns_0 = theta_r * 0 + (((psi_m + 0) * (theta_r - theta_s) * p0) / (lambda - 1));
        const double w_uns = w_uns_z - w_uns_0;
        const double sat_swc = na2 ? nan("") : (shallow ? theta_s * (ud - wtd2) * 1000 : 0.0);
        const double w_z = w_uns + sat_swc;
        // calc_Se, :133-138
        const double theta_top = w_z / (ud * 1000);
        double Se = theta_top / theta_s;
        if (!isnan(Se)) Se = (Se > 1) ? 1.0 : ((Se < 0) ? 0.0 : Se);
        const int64_t o = l * p.opitch + c;
        if (p.theta_i) __stcs(p.theta_i + o, theta_i);
        if (p.wtd) __stcs(p.wtd + o, wtd);
        if (p.w_z) __stcs(p.w_z + o, w_z);
        if (p.se) __stcs(p.se + o, Se);
    }
}

// ---------------------------------------------------------------------------------------------
// Terrain preprocessing, first slice (SURVEY 8f-2; see include/splash_cuda.h: PARITY UNPINNED, raster::terrain /
// raster::area are not in the reference tree).  One thread per cell, a 3x3 stencil over the DEM: an HBM-bound map
// (8 B read + <= 40 B written per cell; the eight neighbour reads hit L1/L2).
// ---------------------------------------------------------------------------------------------
struct TerrainParams {
    const double* elev;
    double *slope, *aspect, *lat, *resolution, *flowdir, *ncellin, *ncellout;
    int64_t n_rows, n_cols;
    double ymax, xres, yres;
    int lonlat;
};

constexpr double kEarthR = 6378137.0;  // raster's default sphere for lon/lat distances

__device__ __forceinline__ void terrain_cell_size(const TerrainParams& p, int64_t r, double& dx, double& dy, double& lat_c) {
    lat_c = p.ymax - ((double)r + 0.5) * p.yres;
    if (p.lonlat) {
        dy = kEarthR * (p.yres * kpir);
        dx = kEarthR * cos(lat_c * kpir) * (p.xres * kpir);
    } else {
        dy = p.yres;
        dx = p.xres;
    }
}

__global__ void __launch_bounds__(256) k_terrain(TerrainParams p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_rows * p.n_cols) return;
    const int64_t r = i / p.n_cols, c = i - r * p.n_cols;
    const double z0 = p.elev[i];
    double dx, dy, lat_c;
    terrain_cell_size(p, r, dx, dy, lat_c);
    const bool valid = !isnan(z0);
    if (p.lat) p.lat[i] = valid ? lat_c : nan("");                       // lat <- elev * 0; lat[!is.na(lat)] <- y
    if (p.resolution) p.resolution[i] = sqrt(dx * dy);                   // sqrt(area km2) * 1000
    double slope = nan(""), aspect = nan(""), fd = nan("");
    if (r > 0 && r + 1 < p.n_rows && c > 0 && c + 1 < p.n_cols) {
        const double* e = p.elev + i;
        const int64_t nc = p.n_cols;
        const double z1 = e[-nc - 1], z2 = e[-nc], z3 = e[-nc + 1], z4 = e[-1], z6 = e[1], z7 = e[nc - 1], z8 = e[nc], z9 = e[nc + 1];
        const bool all_ok = valid && !(isnan(z1) || isnan(z2) || isnan(z3) || isnan(z4) || isnan(z6) || isnan(z7) || isnan(z8) || isnan(z9));
        if (all_ok) {
            // Horn (1981), 8 neighbours: east-minus-west and north-minus-south gradients
            const double zx = ((z3 + 2.0 * z6 + z9) - (z1 + 2.0 * z4 + z7)) / (8.0 * dx);
            const double zy = ((z1 + 2.0 * z2 + z3) - (z7 + 2.0 * z8 + z9)) / (8.0 * dy);
            slope = atan(sqrt(zx * zx + zy * zy)) / kpir;
            // downslope direction clockwise from north; flat cells: 90 degrees (the model multiplies it by sin(slope) = 0)
            double a = (kPI / 2.0 - atan2(-zy, -zx)) / kpir;
            if (a < 0.0) a += 360.0;
            if (a >= 360.0) a -= 360.0;
            if (zx == 0.0 && zy == 0.0) a = 90.0;
            aspect = a;
            // D8: steepest drop over distance; codes 1 E, 2 SE, 4 S, 8 SW, 16 W, 32 NW, 64 N, 128 NE; ties: lowest code
            const double dd = sqrt(dx * dx + dy * dy);
            const double drop[8] = {(z0 - z6) / dx, (z0 - z9) / dd, (z0 - z8) / dy, (z0 - z7) / dd,
                                    (z0 - z4) / dx, (z0 - z1) / dd, (z0 - z2) / dy, (z0 - z3) / dd};
            int best = 0;
#pragma unroll
            for (int k = 1; k < 8; ++k)
                if (drop[k] > drop[best]) best = k;
            fd = (double)(1 << best);
        }
    }
    if (valid && isnan(slope)) slope = 0.0;    // terraines[is.na(terraines) & !is.na(elev)] <- 0, R/splash.grid.R:107
    if (valid && isnan(aspect)) aspect = 0.0;
    if (p.slope) p.slope[i] = slope;
    if (p.aspect) p.aspect[i] = aspect;
    if (p.flowdir) p.flowdir[i] = fd;
}

// ncellflow(flowdir, inout, met = 'top'), R/upslope_area.R:140-165: focal 3x3 count of the neighbours whose direction
// equals the template (column-major fill of matrix(c(2,1,128,4,0,64,8,16,32), nrow = 3): NW 2, W 1, SW 128, N 4, S 64,
// NE 8, E 16, SE 32 -- each neighbour pointing at the centre; 'out' uses the reversed vector), zero matches -> 1, and NA
// where all nine values are NA.  Cells outside the grid count as NA (raster::focal pads with NA).
__global__ void __launch_bounds__(256) k_ncellflow(TerrainParams p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_rows * p.n_cols) return;
    const int64_t r = i / p.n_cols, c = i - r * p.n_cols;
    // window in raster::focal's order read column by column to match the column-major template
    const int dr[9] = {-1, 0, 1, -1, 0, 1, -1, 0, 1};
    const int dc[9] = {-1, -1, -1, 0, 0, 0, 1, 1, 1};
    const double t_in[9] = {2, 1, 128, 4, 0, 64, 8, 16, 32};
    int n_na = 0, m_in = 0, m_out = 0;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int64_t rr = r + dr[k], cc2 = c + dc[k];
        double v = nan("");
        if (rr >= 0 && rr < p.n_rows && cc2 >= 0 && cc2 < p.n_cols) v = p.flowdir[rr * p.n_cols + cc2];
        if (isnan(v)) {
            ++n_na;
        } else {
            m_in += (v == t_in[k]) ? 1 : 0;
            m_out += (v == t_in[8 - k]) ? 1 : 0;
        }
    }
    const double vin = (n_na == 9) ? nan("") : (double)(m_in == 0 ? 1 : m_in);
    const double vout = (n_na == 9) ? nan("") : (double)(m_out == 0 ? 1 : m_out);
    if (p.ncellin) p.ncellin[i] = vin;
    if (p.ncellout) p.ncellout[i] = vout;
}

// diagnostic: the day step's transcendental functions applied to an array (splash_debug_math)
__global__ void k_debug_math(int op, int64_t n, const double* x, double* y) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    const double w = x[(i * 7919 + 13) % n];  // second operand of the division checks
    switch (op) {
        case 0: y[i] = f_exp(v); break;
        case 1: y[i] = f_log(v); break;
        case 2: y[i] = f_acos(v); break;
        case 3: y[i] = f_sin(v); break;
        // the branch-light bodies against what they stand for (bit for bit inside their guards, NaN outside)
        case 4: y[i] = fm::acos_ok(v) ? fm::acos_body(v) : nan(""); break;
        case 5: y[i] = fm::sqrt_ok(v) ? fm::sqrt_body(v) : nan(""); break;
        case 6: y[i] = fm::sqrt_ok(v) ? sqrt(v) : nan(""); break;
        case 7: y[i] = fm::div_ok(v, w) ? fm::div_body(v, w) : nan(""); break;
        case 8: y[i] = fm::div_ok(v, w) ? v / w : nan(""); break;
        case 9: y[i] = fm::exp_ok(v) ? fm::exp_body(v) : nan(""); break;
        default: y[i] = fm::log_ok(v) ? fm::log_body(v) : nan(""); break;
    }
}

__global__ void k_init_tables() {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kSnowAgeTab) g_snow_age_tab[i] = snow_age_factor_formula((double)i);
}

__global__ void k_tile_begin(TileCtl* ctl, int n_cells) {  // (the control blocks are zeroed once per call)
    ctl->cnt[0] = (unsigned long long)n_cells;
}

// resume: the carried aridity index (row 5 of state_init, parked in w.w1) goes where the interrupted run
// had it, soil_info[12] == `cellout` (R/splash.point.R:150, SURVEY B-3)
// ... and the carried snowfall threshold (row 6, parked in w.snap) replaces the one k_snow_threshold took from this
// segment of the series alone: Tt is a reduction over the WHOLE series (R/splash.point.R:120-122)
__global__ void k_init_resume(Work w, double* cc, int64_t cpitch, double* diag, int64_t dpitch, int n) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    w.status[c] = ST_READY_BULK;
    w.passes[c] = 0;
    StridedCC ccg{cc + c, cpitch};
    const double AI = w.w1[c];
    lateral_consts(ccg, AI);
    const double Tt = w.snap[c];
    ccg(C_TT) = Tt;
    if (diag) {
        diag[SPLASH_DIAG_AI * dpitch + c] = AI;
        diag[SPLASH_DIAG_TT * dpitch + c] = Tt;
    }
}

// ---------------------------------------------------------------------------------------------
// Monthly -> daily forcing: stats::approx(time_index_month, x, time_index, method = "linear", rule = 2)$y as
// splash.point applies it to monthly tc and sw_in (R/splash.point.R:74-84).  The knots are the non-NA months
// (approx drops NA pairs), the interpolant is R's y[i] + (y[j] - y[i]) * ((v - x[i]) / (x[j] - x[i])), a day
// that falls on a knot takes the knot's value, and days outside the knots hold the end values (rule = 2).  Fewer
// than two non-NA months: the series is NA (:75-76).
//   k_m2d_knots   per cell: first and last non-NA month (or -1 when fewer than two)
//   k_month2day   one thread per cell and chunk of days; CTAs of one chunk are launched next to each other, so
//                 the rows being written at any moment are few (the day-major layout puts consecutive days of a
//                 cell n_cells elements apart)
// HBM-bound: 8 (or 4) bytes written per cell-day, ~8 bytes read per cell-month.  The quotient is an integer
// ratio a/b with 0 < a < b: for b <= 40000 the correctly rounded value is q0 + fma(-b, q0, a) * rb with
// rb = 1/b rounded once per knot interval and q0 = a * rb (checked exhaustively, tools/m2d_divcheck.c), which
// keeps the FP64 pipe below the store stream; longer gaps take the IEEE division.
// ---------------------------------------------------------------------------------------------
struct M2dParams {
    const double* monthly;  // [n_months][ipitch]
    int64_t ipitch;
    void* out;              // [day - out_day0][opitch], double or float
    int64_t opitch;
    const int32_t* xs;      // [n_months] day index of each month's first day
    int2* knots;            // [n_cells] first / last non-NA month
    int64_t n_cells;
    int n_months;
    int64_t day0, day1;     // days this launch covers
    int64_t out_day0;       // day held by row 0 of `out`
    int64_t chunk;          // days per blockIdx.y
};

__global__ void __launch_bounds__(256) k_m2d_knots(M2dParams p) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cells) return;
    const double* y = p.monthly + c;
    int n_ok = 0, first = -1, last = -1;
    for (int m = 0; m < p.n_months; ++m) {
        if (!isnan(__ldcs(y + (int64_t)m * p.ipitch))) {
            ++n_ok;
            if (first < 0) first = m;
            last = m;
        }
    }
    p.knots[c] = (n_ok < 2) ? make_int2(-1, -1) : make_int2(first, last);
}

template <typename OT, int V>
struct M2dVec;
template <> struct M2dVec<double, 1> { using T = double; };
template <> struct M2dVec<double, 2> { using T = double2; };
template <> struct M2dVec<float, 1> { using T = float; };
template <> struct M2dVec<float, 2> { using T = float2; };
template <> struct M2dVec<float, 4> { using T = float4; };

// V adjacent cells per thread (one 8/16-byte store per day); kSync > 0 keeps the warps of a CTA within kSync
// days of each other, so that a CTA writes whole 256*V-cell row segments close in time.
template <typename OT, int V, int kSync>
__global__ void __launch_bounds__(256) k_month2day(M2dParams p) {
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * V;
    const bool active = c < p.n_cells;  // the host picks V so that n_cells % V == 0
    if (kSync == 0 && !active) return;
    const int64_t d0 = p.day0 + (int64_t)blockIdx.y * p.chunk;
    const int64_t d1 = (d0 + p.chunk < p.day1) ? d0 + p.chunk : p.day1;
    if (d0 >= d1) return;
    struct Knot {
        int j, last;
        double x_lo, x_hi, y_lo, y_hi, xi, yi, xj, yj, b, rb, dy;
    } k[V];
    const double* y = p.monthly + c;
    if (active) {
#pragma unroll
        for (int u = 0; u < V; ++u) {
            const int2 kn = p.knots[c + u];
            const int first = kn.x, last = kn.y;
            k[u].last = last;
            if (first < 0) continue;
            const double* yu = y + u;
            k[u].x_lo = p.xs[first];
            k[u].x_hi = p.xs[last];
            k[u].y_lo = yu[(int64_t)first * p.ipitch];
            k[u].y_hi = yu[(int64_t)last * p.ipitch];
            // left knot of the chunk's first day: the last non-NA month that starts on or before d0
            int i = first;
            if ((double)d0 > k[u].x_lo) {
                int lo = first, hi = last;
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (p.xs[mid] <= d0) lo = mid; else hi = mid - 1;
                }
                i = lo;
                while (isnan(yu[(int64_t)i * p.ipitch])) --i;  // stops at `first` at the latest
            }
            int j = i;
            if (i < last) do ++j; while (isnan(yu[(int64_t)j * p.ipitch]));
            k[u].j = j;
            k[u].xi = p.xs[i];
            k[u].yi = yu[(int64_t)i * p.ipitch];
            k[u].xj = p.xs[j];
            k[u].yj = yu[(int64_t)j * p.ipitch];
            k[u].b = k[u].xj - k[u].xi;
            k[u].rb = 1.0 / k[u].b;
            k[u].dy = k[u].yj - k[u].yi;
        }
    }
    OT* o = (OT*)p.out + c + (d0 - p.out_day0) * p.opitch;
    for (int64_t d = d0; d < d1; ++d, o += p.opitch) {
        if (active) {
            const double v = (double)d;
            OT r[V];
#pragma unroll
            for (int u = 0; u < V; ++u) {
                Knot& q = k[u];
                double w;
                if (q.last < 0) {
                    w = nan("");
                } else if (v < q.x_lo) {
                    w = q.y_lo;
                } else if (v >= q.x_hi) {
                    w = q.y_hi;
                } else {
                    while (v >= q.xj) {  // x[i] <= v < x[j], neighbouring knots (j <= last because v < x_hi)
                        q.xi = q.xj;
                        q.yi = q.yj;
                        int j = q.j;
                        do ++j; while (isnan(y[u + (int64_t)j * p.ipitch]));
                        q.j = j;
                        q.xj = p.xs[j];
                        q.yj = y[u + (int64_t)j * p.ipitch];
                        q.b = q.xj - q.xi;
                        q.rb = 1.0 / q.b;
                        q.dy = q.yj - q.yi;
                    }
                    const double a = v - q.xi;
                    double t;
                    if (q.b <= 40000.0) {
                        const double t0 = a * q.rb;
                        t = fma(fma(-q.b, t0, a), q.rb, t0);  // == a / b (see above)
                    } else {
                        t = a / q.b;
                    }
                    w = (v == q.xi) ? q.yi : q.yi + q.dy * t;
                }
                r[u] = (OT)w;
            }
            typename M2dVec<OT, V>::T pack;
            memcpy(&pack, r, sizeof(pack));
            __stcs((typename M2dVec<OT, V>::T*)o, pack);
        }
        if (kSync > 0 && ((d - d0) % kSync) == kSync - 1) __syncthreads();
    }
}

// Row-band form of the same interpolation.  The month that holds a day, and the quotient (v - x_i)/(x_j - x_i)
// when both of its neighbouring months are present, depend on the day only: the host tabulates them (IEEE
// division, as R does it).  A CTA then sweeps a band of D day-rows over K*256 adjacent cells, row by row: a
// cell-day is two cached monthly values, one multiply-add pair and one store, and a warp's consecutive stores
// stay inside one row.  Cells with NA months next to the day take the general search below (knots from
// k_m2d_knots), which follows approx1() as the walk kernel does.
struct M2dBand {
    const double* monthly;
    int64_t ipitch;
    void* out;
    int64_t opitch;
    const int32_t* xs;
    const int2* knots;
    const int32_t* day_m;  // [n_days] month that holds the day (largest m with xs[m] <= d), -1 before the first month
    const double* day_q;   // [n_days] (d - xs[m]) / (xs[m+1] - xs[m]); 0 on a month's first day and in the last month
    int64_t n_cells;
    int n_months;
    int64_t day0, day1, out_day0;
    int D;
};

__device__ __noinline__ double m2d_general(const double* y, int64_t ipitch, const int32_t* xs, int2 kn, int m, int64_t d) {
    if (kn.x < 0) return nan("");  // fewer than two non-NA months, R/splash.point.R:75-76
    const double v = (double)d;
    const double x_lo = xs[kn.x], x_hi = xs[kn.y];
    if (v < x_lo) return y[(int64_t)kn.x * ipitch];   // rule = 2
    if (v >= x_hi) return y[(int64_t)kn.y * ipitch];
    int i = m, j = m + 1;                              // kn.x <= m < kn.y here
    while (isnan(y[(int64_t)i * ipitch])) --i;         // stops at kn.x at the latest
    while (isnan(y[(int64_t)j * ipitch])) ++j;         // stops at kn.y at the latest
    const double xi = xs[i], xj = xs[j], yi = y[(int64_t)i * ipitch], yj = y[(int64_t)j * ipitch];
    if (v == xi) return yi;
    return yi + (yj - yi) * ((v - xi) / (xj - xi));
}

template <typename OT, int K>
__global__ void __launch_bounds__(256) k_month2day_band(M2dBand p) {
    const int64_t cbase = (int64_t)blockIdx.x * (256 * K) + threadIdx.x;
    const int64_t d0 = p.day0 + (int64_t)blockIdx.y * p.D;
    const int64_t d1 = (d0 + p.D < p.day1) ? d0 + p.D : p.day1;
    int cur_m = INT_MIN;
    double yi[K], yj[K];
    OT* o = (OT*)p.out + (d0 - p.out_day0) * p.opitch + cbase;
    for (int64_t d = d0; d < d1; ++d, o += p.opitch) {
        const int m = __ldg(p.day_m + d);
        const double q = __ldg(p.day_q + d);
        if (m != cur_m) {
            cur_m = m;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int64_t c = cbase + k * 256;
                yi[k] = yj[k] = nan("");
                if (c < p.n_cells && m >= 0) {
                    yi[k] = p.monthly[(int64_t)m * p.ipitch + c];
                    yj[k] = (m + 1 < p.n_months) ? p.monthly[(int64_t)(m + 1) * p.ipitch + c] : yi[k];
                }
            }
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int64_t c = cbase + k * 256;
            if (c >= p.n_cells) continue;
            double r;
            if (!isnan(yi[k]) && !isnan(yj[k]))
                r = (q == 0.0) ? yi[k] : yi[k] + (yj[k] - yi[k]) * q;
            else
                r = m2d_general(p.monthly + c, p.ipitch, p.xs, p.knots[c], m, d);
            __stcs(o + k * 256, (OT)r);
        }
    }
}


// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

constexpr int kSlots = 3;         // forcing / output buffer sets in flight when they stream from / to the host
constexpr int kRunStreams = 8;    // compute streams the tiles are dealt to
constexpr int kPoolStreams = 16;  // streams of the straggler-pool launches: a tile's pool work must not queue behind
                                  // another tile's seconds-long chain, so calls are cut into at most 16 tiles when possible
#ifndef SPLASH_ROUNDS
#define SPLASH_ROUNDS 20
#endif
constexpr int kRounds = SPLASH_ROUNDS;  // lock-step year passes per tile before the leftovers go to the pool
// Pass budgets of the pool's first two spin-up stages and the shape of the third, which runs to the reference's pass
// limit on SMs of its own.  Two presets, chosen per call by its size (profiles/README.md R2.2):
//   large calls (the straggler chain hides behind seconds of bulk work): 8 / 128 passes, 16 cells per last-stage warp on 48
//     CTAs -- few SMs taken away from the uniform kernels (resident benchmark: 2.83 s per pass against 2.97 s);
//   small calls (chain-bound: row blocks of host-fed runs, shards of a strong-scaling run): 4 / 32 passes, 8 cells per
//     warp on 96 CTAs -- the long runners reach their uncontended SMs sooner and share their warp, hence every divergent
//     branch of the day step, with fewer cells (583 200 cells x 2 years: 1.59 s against 1.83 s).
constexpr int kPoolStage1Passes = 8, kPoolStage2Passes = 128, kPoolLastLanes = 16, kPoolLastCtas = 48;
constexpr int kPoolStage1Small = 2, kPoolStage2Small = 8, kPoolLastLanesSmall = 8, kPoolLastCtasSmall = 96;
constexpr double kPoolSmallCallCellDays = 5e9;  // n_cells * n_days below which a call counts as chain-bound
static_assert(kRounds <= kMaxRounds, "kRounds");
// cells per tile aimed for: two full waves of the 512-thread uniform kernels (the bulk launches of several tiles run side
// by side on their streams, so a 768-thread bulk CTA shape needs no whole number of waves per tile)
#ifndef SPLASH_TILE_TARGET
#define SPLASH_TILE_TARGET (148LL * 512 * 2)
#endif
constexpr int64_t kTileTarget = SPLASH_TILE_TARGET;

constexpr int kWorkInts = 8;  // int arrays of a work set: passes, snap_pass, status, 2 spin lists, frost days, bulk order, sort keys
struct WorkSet {  // per-tile work arrays (per slot when the inputs stream from the host)
    DevBuf cc, work_d, work_i, diag;
};

}  // namespace

struct splash_cluster;

struct splash_ctx {
    int device = 0;
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaStream_t s_run[kRunStreams] = {};
    cudaStream_t s_pool[kPoolStreams] = {};
    std::string err;
    splash_stats stats{};
    int sm_count = 0;
    bool month_tab_set = false;
    // grow-only device buffers
    DevBuf forcing[kSlots][3], cellin[kSlots], outs[kSlots];
    std::vector<WorkSet> work;
    DevBuf dtab, dtab_spin, ctl, pool_mem, ahead_mem;
    // tuning knobs (environment overrides for experiments, read once at creation)
    int n_run_streams = kRunStreams;      // SPLASH_RUN_STREAMS
    int pool_stage1 = kPoolStage1Passes;  // SPLASH_POOL_STAGE1 (0 = single stage)
    int pool_stage2 = kPoolStage2Passes;  // SPLASH_POOL_STAGE2
    int pool_excl_smem = 0;               // dynamic shared memory of a last-stage CTA (SPLASH_POOL_EXCL=0: no exclusivity)
    int pool_last_lanes = kPoolLastLanes, pool_last_ctas = kPoolLastCtas;  // SPLASH_POOL_LANES, SPLASH_POOL_CTAS
    int chain_fast = SPLASH_CHAIN_FAST;  // SPLASH_CHAIN_FAST=0/1: the pool's last stage on the branch-light day step (k_pool_spin)
    bool pool_auto = true;                // none of the four was set in the environment: preset by call size
    int two_pass = 1;                     // SPLASH_TWO_PASS
    int n_rounds = kRounds;               // SPLASH_ROUNDS_RT (<= kRounds)
    int64_t pool_cap = 0;                 // SPLASH_POOL_CAP: force the pool capacity (tests of the overflow path)
    int spin_ahead = 1;                   // SPLASH_SPIN_AHEAD=0: host-fed calls upload tile by tile (no spin-up data first)
    int regime_sort = 0;                  // SPLASH_REGIME_SORT=1: the bulk launch takes the cells in regime-sorted order (measured
                                          // slower on the synthetic grid, whose divergence is day-to-day weather: profiles/README.md)
    double mem_share = 1.0;               // share of the device's memory this context may plan with (lanes of a cluster)
    // a context over several GPUs (splash_ctx_create_multi): the work goes to the cluster's lanes
    splash_cluster* multi = nullptr;
};

namespace {

std::string g_create_err = "";

int fail(splash_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx)
        ctx->err = buf;
    else
        g_create_err = buf;
    return code;
}

#define CU(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess)                                                                        \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? SPLASH_ERR_NOMEM : SPLASH_ERR_CUDA,     \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);  \
    } while (0)

int ensure(splash_ctx* ctx, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap) return SPLASH_OK;
    if (b.p) {
        CU(cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    CU(cudaMalloc(&b.p, bytes));
    b.cap = bytes;
    return SPLASH_OK;
}

struct TmpDev {  // a temporary device buffer that is released on every return path
    void* p = nullptr;
    ~TmpDev() {
        if (p) cudaFree(p);
    }
};

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
inline unsigned grid_for(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }
inline unsigned ugrid_for(int64_t n) { return (unsigned)((n + kUThreads - 1) / kUThreads); }

constexpr size_t kSmemSpin = sizeof(double) * NCC_DAY * kThreads;             // k_spin_check
constexpr size_t kSmemUniform = sizeof(double) * staged_cc<kUThreads>() * kUThreads;  // k_spin_first, k_spin_rest
constexpr size_t kSmemBulkCC = sizeof(double) * staged_cc<kBThreads>() * kBThreads;   // bulk launch: staged constants
inline unsigned bgrid_for(int64_t n) { return (unsigned)((n + kBThreads - 1) / kBThreads); }
constexpr size_t kSmemBulkF32 = kSmemBulkCC + sizeof(float) * 2 * 3 * kBThreads;  // f32 forcing: + the cp.async ring
template <typename FT> constexpr size_t bulk_smem() { return sizeof(FT) == 4 ? kSmemBulkF32 : kSmemBulkCC; }
static_assert(kSmemBulkF32 <= 227 * 1024, "bulk launch: shared memory per CTA");
constexpr size_t kSmemList = sizeof(double) * (NCC_DAY + 5) * kListThreads;  // list mode: + cycle snapshot

template <typename FT>
cudaError_t prepare_kernels() {
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_spin_first<FT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemUniform))) return e;
    if ((e = cudaFuncSetAttribute(k_spin_check<FT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemSpin))) return e;
    if ((e = cudaFuncSetAttribute(k_spin_rest<FT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemUniform))) return e;
    if ((e = cudaFuncSetAttribute(k_run_bulk<FT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bulk_smem<FT>()))) return e;
    if ((e = cudaFuncSetAttribute(k_run_bulk<FT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bulk_smem<FT>()))) return e;
    if ((e = cudaFuncSetAttribute(k_run_list<FT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemList))) return e;
    if ((e = cudaFuncSetAttribute(k_run_list<FT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemList))) return e;
    if ((e = cudaFuncSetAttribute(k_pool_spin<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024))) return e;
    if ((e = cudaFuncSetAttribute(k_pool_spin<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024))) return e;
    return cudaSuccess;
}

// bulk launch: every ST_READY_BULK cell of the tile, uniform day loop
template <typename FT>
void launch_bulk(const RunParams& rp, bool monthly, cudaStream_t s) {
    if (rp.n_cells <= 0) return;
    if (monthly)
        k_run_bulk<FT, true><<<bgrid_for(rp.n_cells), kBThreads, bulk_smem<FT>(), s>>>(rp);
    else
        k_run_bulk<FT, false><<<bgrid_for(rp.n_cells), kBThreads, bulk_smem<FT>(), s>>>(rp);
}

// list-mode launch: `warps` one-warp CTAs whose lanes fetch cells from the queue in rp
template <typename FT>
void launch_list(const RunParams& rp, bool monthly, int warps, cudaStream_t s) {
    if (monthly)
        k_run_list<FT, true><<<(unsigned)warps, kListThreads, kSmemList, s>>>(rp);
    else
        k_run_list<FT, false><<<(unsigned)warps, kListThreads, kSmemList, s>>>(rp);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int splash_abi_version(void) { return SPLASH_ABI_VERSION; }

static splash_ctx* first_lane(splash_ctx* ctx);

static int ctx_create_impl(int device, splash_ctx* ctx, const cudaDeviceProp& prop);

int splash_ctx_create(int device, splash_ctx** out_ctx) {
    splash_ctx* ctx = nullptr;
    if (!out_ctx) return fail(nullptr, SPLASH_ERR_BAD_ARG, "splash_ctx_create: out_ctx is NULL");
    *out_ctx = nullptr;
    // The call keeps ~25 streams busy (tiles, straggler pool, copies).  With the default of 8 hardware
    // work queues several streams share one, and a tile's next kernel then waits behind another
    // stream's seconds-long pool kernel (measured: tiles 4..7 started 2.6 s late).  The host process
    // exports CUDA_DEVICE_MAX_CONNECTIONS=32 before it initialises CUDA (include/splash_cuda.h,
    // INTEGRATION.md); the library does not touch the environment.
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(nullptr, SPLASH_ERR_NO_DEVICE,
                    "no CUDA device available (%s); libsplash_cuda has no CPU implementation",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= n) return fail(nullptr, SPLASH_ERR_BAD_ARG, "device %d out of range [0,%d)", device, n);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, SPLASH_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10 || prop.minor != 0)  // the library embeds sm_100a SASS only (no PTX to JIT for other parts)
        return fail(nullptr, SPLASH_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    ctx = new splash_ctx();
    const int rc = ctx_create_impl(device, ctx, prop);
    if (rc != SPLASH_OK) {  // the message must outlive the context
        g_create_err = ctx->err;
        splash_ctx_destroy(ctx);
        return rc;
    }
    *out_ctx = ctx;
    return SPLASH_OK;
}

static int ctx_create_impl(int device, splash_ctx* ctx, const cudaDeviceProp& prop) {
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (const char* v = getenv("SPLASH_RUN_STREAMS")) ctx->n_run_streams = std::max(1, std::min(kRunStreams, atoi(v)));
    ctx->pool_auto = !getenv("SPLASH_POOL_STAGE1") && !getenv("SPLASH_POOL_STAGE2") && !getenv("SPLASH_POOL_LANES") && !getenv("SPLASH_POOL_CTAS");
    if (const char* v = getenv("SPLASH_POOL_STAGE1")) ctx->pool_stage1 = std::max(0, atoi(v));
    if (const char* v = getenv("SPLASH_TWO_PASS")) ctx->two_pass = atoi(v) != 0;
    if (const char* v = getenv("SPLASH_POOL_STAGE2")) ctx->pool_stage2 = std::max(1, atoi(v));
    if (const char* v = getenv("SPLASH_POOL_LANES")) ctx->pool_last_lanes = std::max(1, std::min(32, atoi(v)));
    if (const char* v = getenv("SPLASH_CHAIN_FAST")) ctx->chain_fast = atoi(v) != 0;
    if (const char* v = getenv("SPLASH_POOL_CTAS")) ctx->pool_last_ctas = std::max(1, atoi(v));
    {
        // a quarter of the SM's shared memory per last-stage CTA: four of them fill an SM, and none fits
        // beside a uniform CTA (kSmemUniform)
        const char* v = getenv("SPLASH_POOL_EXCL");
        const bool excl = !v || atoi(v) != 0;
        const int quarter = ((int)prop.sharedMemPerMultiprocessor - 4 * 1024) / 4 / 1024 * 1024;
        ctx->pool_excl_smem = excl ? std::max<int>((int)kSmemList, std::min<int>(quarter, (int)prop.sharedMemPerBlockOptin)) : (int)kSmemList;
    }
    if (const char* v = getenv("SPLASH_ROUNDS_RT")) ctx->n_rounds = std::max(0, std::min(kRounds, atoi(v)));
    if (const char* v = getenv("SPLASH_POOL_CAP")) ctx->pool_cap = std::max<int64_t>(32, atoll(v));
    if (const char* v = getenv("SPLASH_SPIN_AHEAD")) ctx->spin_ahead = atoi(v) != 0;
    if (const char* v = getenv("SPLASH_REGIME_SORT")) ctx->regime_sort = atoi(v) != 0;
    CU(cudaSetDevice(device));
    int prio_lo = 0, prio_hi = 0;
    CU(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    CU(cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking));
    // Stragglers first (the chain of the slowest cell is the critical path of a call); the tiles abreast.
    // SPLASH_TILE_PRIO=1 ranks tile t's stream above tile t+1's (earlier chain starts for the first tiles): measured
    // WORSE on the resident benchmark (4.0 - 4.5 s per pass against 2.9 s: the later tiles' spin-ups starve and their
    // chains end after everything else), kept as a knob only.
    const bool tile_prio = getenv("SPLASH_TILE_PRIO") && atoi(getenv("SPLASH_TILE_PRIO")) != 0;
    for (int i = 0; i < kRunStreams; ++i)
        CU(cudaStreamCreateWithPriority(&ctx->s_run[i], cudaStreamNonBlocking, tile_prio ? std::min(prio_lo, prio_hi + 1 + i) : prio_lo));
    for (auto& s : ctx->s_pool) CU(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, prio_hi));
    k_init_tables<<<(kSnowAgeTab + 255) / 256, 256>>>();
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    CU(prepare_kernels<double>());
    CU(prepare_kernels<float>());
    return SPLASH_OK;
}

void splash_ctx_destroy(splash_ctx* ctx) {
    if (!ctx) return;
    if (ctx->multi) {
        splash_cluster_destroy(ctx->multi);
        delete ctx;
        return;
    }
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    auto fr = [](DevBuf& b) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    };
    for (int i = 0; i < kSlots; ++i) {
        for (int k = 0; k < 3; ++k) fr(ctx->forcing[i][k]);
        fr(ctx->cellin[i]);
        fr(ctx->outs[i]);
    }
    for (auto& w : ctx->work) {
        fr(w.cc);
        fr(w.work_d);
        fr(w.work_i);
        fr(w.diag);
    }
    fr(ctx->dtab);
    fr(ctx->dtab_spin);
    fr(ctx->ctl);
    fr(ctx->pool_mem);
    fr(ctx->ahead_mem);
    if (ctx->s_h2d) cudaStreamDestroy(ctx->s_h2d);
    if (ctx->s_d2h) cudaStreamDestroy(ctx->s_d2h);
    for (auto s : ctx->s_run)
        if (s) cudaStreamDestroy(s);
    for (auto s : ctx->s_pool)
        if (s) cudaStreamDestroy(s);
    delete ctx;
}

const char* splash_last_error(const splash_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int64_t splash_count_months(const int32_t* year, const int32_t* month, int64_t n_days) {
    if (!year || !month || n_days <= 0) return 0;
    int64_t n = 1;
    for (int64_t d = 1; d < n_days; ++d)
        if (year[d] != year[d - 1] || month[d] != month[d - 1]) ++n;
    return n;
}

int splash_last_stats(const splash_ctx* ctx, splash_stats* out) {
    if (!ctx || !out) return SPLASH_ERR_BAD_ARG;
    *out = ctx->stats;
    return SPLASH_OK;
}

int splash_debug_math(splash_ctx* ctx, int op, int64_t n, const double* x, double* y) {
    if (ctx && ctx->multi) {  // single-GPU work: the context's first lane does it
        splash_ctx* lane = first_lane(ctx);
        const int rc = splash_debug_math(lane, op, n, x, y);
        ctx->err = lane->err;
        return rc;
    }
    if (!ctx || !x || !y || n < 0 || op < 0 || op > 10) return SPLASH_ERR_BAD_ARG;
    if (n == 0) return SPLASH_OK;
    CU(cudaSetDevice(ctx->device));
    TmpDev dx, dy;  // freed on every return path
    CU(cudaMalloc(&dx.p, (size_t)n * 8));
    CU(cudaMalloc(&dy.p, (size_t)n * 8));
    CU(cudaMemcpy(dx.p, x, (size_t)n * 8, cudaMemcpyHostToDevice));
    k_debug_math<<<(unsigned)((n + 255) / 256), 256>>>(op, n, (const double*)dx.p, (double*)dy.p);
    CU(cudaGetLastError());
    CU(cudaMemcpy(y, dy.p, (size_t)n * 8, cudaMemcpyDeviceToHost));
    return SPLASH_OK;
}

int splash_unswc_grid_run(splash_ctx* ctx, const splash_unswc_in* in, splash_unswc_out* out) {
    if (ctx && ctx->multi) {  // single-GPU work: the context's first lane does it
        splash_ctx* lane = first_lane(ctx);
        const int rc = splash_unswc_grid_run(lane, in, out);
        ctx->err = lane->err;
        return rc;
    }
    if (!ctx) return SPLASH_ERR_BAD_ARG;
    ctx->err.clear();
    if (!in || !out) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_unswc_grid_run: NULL in/out");
    const int64_t nc = in->n_cells, nl = in->n_layers;
    if (nc < 0 || nl < 0) return fail(ctx, SPLASH_ERR_BAD_ARG, "negative n_cells/n_layers");
    const int64_t istride = in->cell_stride ? in->cell_stride : nc, ostride = out->cell_stride ? out->cell_stride : nc;
    if (istride < nc || ostride < nc) return fail(ctx, SPLASH_ERR_BAD_ARG, "cell_stride smaller than n_cells");
    if ((in->mem_kind != SPLASH_MEM_HOST && in->mem_kind != SPLASH_MEM_DEVICE) || out->mem_kind != in->mem_kind)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "mem_kind must be SPLASH_MEM_HOST or SPLASH_MEM_DEVICE, the same for in and out");
    if (nc == 0 || nl == 0) return SPLASH_OK;
    if (!in->soil || !in->wn) return fail(ctx, SPLASH_ERR_BAD_ARG, "NULL soil/wn");
    CU(cudaSetDevice(ctx->device));
    double* const optr[4] = {out->theta_i, out->wtd, out->w_z, out->se};
    UnswcParams p{};
    p.n_cells = nc;
    p.uns_depth = in->uns_depth;
    cudaStream_t S = ctx->s_run[0];
    if (in->mem_kind == SPLASH_MEM_DEVICE) {
        p.soil = in->soil;
        p.soil_pitch = nc;
        p.wn = in->wn;
        p.wpitch = istride;
        p.theta_i = optr[0];
        p.wtd = optr[1];
        p.w_z = optr[2];
        p.se = optr[3];
        p.opitch = ostride;
        p.n_layers = nl;
        k_unswc<<<(unsigned)((nc + 255) / 256), 256, 0, S>>>(p);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(S));
        return SPLASH_OK;
    }
    // host arrays: chunks of layers through a device staging area (H2D, kernel, D2H per chunk)
    int n_o = 0;
    for (auto q : optr) n_o += q ? 1 : 0;
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(nl, ((int64_t)1 << 30) / std::max<int64_t>(1, nc * 8 * (1 + n_o))));
    TmpDev t_soil, t_wn, t_out;  // freed on every return path
    CU(cudaMalloc(&t_soil.p, (size_t)6 * nc * 8));
    CU(cudaMalloc(&t_wn.p, (size_t)chunk * nc * 8));
    if (n_o) CU(cudaMalloc(&t_out.p, (size_t)n_o * chunk * nc * 8));
    double *d_soil = (double*)t_soil.p, *d_wn = (double*)t_wn.p, *d_out = (double*)t_out.p;
    CU(cudaMemcpyAsync(d_soil, in->soil, (size_t)6 * nc * 8, cudaMemcpyHostToDevice, S));
    p.soil = d_soil;
    p.soil_pitch = nc;
    p.wn = d_wn;
    p.wpitch = nc;
    p.opitch = nc;
    double** pp[4] = {&p.theta_i, &p.wtd, &p.w_z, &p.se};
    int rc = SPLASH_OK;
    for (int64_t l0 = 0; l0 < nl && rc == SPLASH_OK; l0 += chunk) {
        const int64_t n = std::min<int64_t>(chunk, nl - l0);
        int k = 0;
        for (int i = 0; i < 4; ++i) *pp[i] = optr[i] ? d_out + (size_t)(k++) * chunk * nc : nullptr;
        p.n_layers = n;
        if (cudaMemcpy2DAsync(d_wn, (size_t)nc * 8, in->wn + l0 * istride, (size_t)istride * 8, (size_t)nc * 8, (size_t)n,
                              cudaMemcpyHostToDevice, S) != cudaSuccess) rc = SPLASH_ERR_CUDA;
        k_unswc<<<(unsigned)((nc + 255) / 256), 256, 0, S>>>(p);
        for (int i = 0; i < 4 && rc == SPLASH_OK; ++i)
            if (optr[i] && cudaMemcpy2DAsync(optr[i] + l0 * ostride, (size_t)ostride * 8, *pp[i], (size_t)nc * 8, (size_t)nc * 8, (size_t)n,
                                             cudaMemcpyDeviceToHost, S) != cudaSuccess) rc = SPLASH_ERR_CUDA;
        if (cudaStreamSynchronize(S) != cudaSuccess) rc = SPLASH_ERR_CUDA;
    }
    if (rc != SPLASH_OK) return fail(ctx, rc, "splash_unswc_grid_run: %s", cudaGetErrorString(cudaGetLastError()));
    return SPLASH_OK;
}

int splash_terrain_run(splash_ctx* ctx, const splash_terrain_in* in, splash_terrain_out* out) {
    if (ctx && ctx->multi) {  // single-GPU work: the context's first lane does it
        splash_ctx* lane = first_lane(ctx);
        const int rc = splash_terrain_run(lane, in, out);
        ctx->err = lane->err;
        return rc;
    }
    if (!ctx) return SPLASH_ERR_BAD_ARG;
    ctx->err.clear();
    if (!in || !out) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_terrain_run: NULL in/out");
    const int64_t nr = in->n_rows, ncol = in->n_cols;
    if (nr < 0 || ncol < 0 || nr > (int64_t)1 << 31 || ncol > (int64_t)1 << 31) return fail(ctx, SPLASH_ERR_BAD_ARG, "bad n_rows/n_cols");
    if (in->mem_kind != SPLASH_MEM_HOST && in->mem_kind != SPLASH_MEM_DEVICE)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "mem_kind must be SPLASH_MEM_HOST or SPLASH_MEM_DEVICE");
    if (!(in->xres > 0) || !(in->yres > 0)) return fail(ctx, SPLASH_ERR_BAD_ARG, "xres and yres must be positive");
    const int64_t n = nr * ncol;
    if (n == 0) return SPLASH_OK;
    if (!in->elev) return fail(ctx, SPLASH_ERR_BAD_ARG, "NULL elev");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t S = ctx->s_run[0];
    double* const optr[7] = {out->slope, out->aspect, out->lat, out->resolution, out->flowdir, out->ncellin, out->ncellout};
    TerrainParams p{};
    p.n_rows = nr;
    p.n_cols = ncol;
    p.ymax = in->ymax;
    p.xres = in->xres;
    p.yres = in->yres;
    p.lonlat = in->lonlat;
    const bool need_fd = out->flowdir || out->ncellin || out->ncellout;
    const unsigned grid = (unsigned)((n + 255) / 256);
    TmpDev t_elev, t_out, t_fd;  // freed on every return path
    double** slot[7] = {&p.slope, &p.aspect, &p.lat, &p.resolution, &p.flowdir, &p.ncellin, &p.ncellout};
    if (in->mem_kind == SPLASH_MEM_DEVICE) {
        p.elev = in->elev;
        for (int k = 0; k < 7; ++k) *slot[k] = optr[k];
        if (need_fd && !p.flowdir) {
            CU(cudaMalloc(&t_fd.p, (size_t)n * 8));
            p.flowdir = (double*)t_fd.p;
        }
    } else {
        CU(cudaMalloc(&t_elev.p, (size_t)n * 8));
        CU(cudaMalloc(&t_out.p, (size_t)n * 8 * 7));
        CU(cudaMemcpyAsync(t_elev.p, in->elev, (size_t)n * 8, cudaMemcpyHostToDevice, S));
        p.elev = (const double*)t_elev.p;
        for (int k = 0; k < 7; ++k) *slot[k] = (optr[k] || (k == 4 && need_fd)) ? (double*)t_out.p + (size_t)k * n : nullptr;
    }
    k_terrain<<<grid, 256, 0, S>>>(p);
    if (out->ncellin || out->ncellout) k_ncellflow<<<grid, 256, 0, S>>>(p);
    CU(cudaGetLastError());
    if (in->mem_kind == SPLASH_MEM_HOST)
        for (int k = 0; k < 7; ++k)
            if (optr[k]) CU(cudaMemcpyAsync(optr[k], *slot[k], (size_t)n * 8, cudaMemcpyDeviceToHost, S));
    CU(cudaStreamSynchronize(S));
    return SPLASH_OK;
}

// Per-row metrics of the upslope area (splash_upslope.cuh: UR_*), on the host with libm so that the kernels and a
// numpy restatement (Python's math module is the same libm) share every operand.  No contraction into FMA.
__attribute__((optimize("fp-contract=off"))) static void upslope_rows(int64_t n_rows, double ymax, double xres, double yres,
                                                                      int lonlat, double min_slope_deg, std::vector<double>& rows) {
    using namespace upslope;
    const double t = tan(min_slope_deg * kpir);
    rows.resize((size_t)n_rows * UR_N);
    for (int64_t r = 0; r < n_rows; ++r) {
        double* m = rows.data() + r * UR_N;
        const double lat_c = ymax - ((double)r + 0.5) * yres;
        const double dy = lonlat ? kEarthR * (yres * kpir) : yres;
        const double dx = lonlat ? kEarthR * cos(lat_c * kpir) * (xres * kpir) : xres;
        const double dd = sqrt(dx * dx + dy * dy);
        const double rl = sqrt(dx * dy);
        m[UR_DX] = dx;
        m[UR_DY] = dy;
        m[UR_DD] = dd;
        m[UR_AREA] = dx * dy;
        m[UR_LC] = 0.5 * rl;
        m[UR_LD] = 0.354 * rl;
        m[UR_EX] = dx * t;
        m[UR_EY] = dy * t;
        m[UR_ED] = dd * t;
        m[UR_TX] = atan2(dy, dx);
        m[UR_TY] = atan2(dx, dy);
    }
}

// The DEM geometry both upslope entry points take (splash_upslope_in / splash_dinf_in).
struct UpslopeGeom {
    int64_t n_rows, n_cols;
    const double* elev;
    double ymax, xres, yres;
    int32_t lonlat, mem_kind;
};

static int upslope_check(splash_ctx* ctx, const UpslopeGeom& g) {
    if (g.n_rows < 0 || g.n_cols < 0 || g.n_rows > (int64_t)upslope::kFT * 65535 || (g.n_cols > 0 && g.n_rows > INT32_MAX / g.n_cols))
        return fail(ctx, SPLASH_ERR_BAD_ARG, "bad n_rows/n_cols (n_rows*n_cols must fit in int32, n_rows <= %d)", upslope::kFT * 65535);
    if (g.mem_kind != SPLASH_MEM_HOST && g.mem_kind != SPLASH_MEM_DEVICE)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "mem_kind must be SPLASH_MEM_HOST or SPLASH_MEM_DEVICE");
    if (!(g.xres > 0) || !(g.yres > 0) || !std::isfinite(g.xres) || !std::isfinite(g.yres))
        return fail(ctx, SPLASH_ERR_BAD_ARG, "xres and yres must be positive and finite");
    if (g.lonlat && !(g.ymax <= 90.0 && g.ymax - (double)g.n_rows * g.yres >= -90.0))
        return fail(ctx, SPLASH_ERR_BAD_ARG, "lonlat: the rows must lie between -90 and 90 degrees");
    return SPLASH_OK;
}

constexpr int kUpslopeBatch = 64;  // sweeps launched between two reads of their flags

// The temporaries of one upslope call (freed on every return path) and the device views of its DEM and area.
struct UpslopeRun {
    const char* fn;
    cudaStream_t S;
    int64_t n;
    bool host;
    std::vector<double> rows;
    TmpDev t_z, t_w0, t_w1, t_area, t_rows, t_ctl;
    const double* z = nullptr;
    const double* d_rows = nullptr;
    double* area = nullptr;
    double* w[2] = {nullptr, nullptr};
    int* ctl = nullptr;    // upslope::AC_* control words
    int* flags = nullptr;  // flags[0]: "the sweep before this batch changed something"; flags[1..batch]: the batch
    int hctl[upslope::AC_N + 1 + kUpslopeBatch];
};

// Device buffers, per-row metrics, W's initial state; +-inf elevations are rejected here.
static int upslope_begin(splash_ctx* ctx, UpslopeRun& u, const UpslopeGeom& g, double min_slope_deg, double* out_area) {
    using namespace upslope;
    CU(cudaSetDevice(ctx->device));
    u.S = ctx->s_run[0];
    u.n = g.n_rows * g.n_cols;
    u.host = g.mem_kind == SPLASH_MEM_HOST;
    upslope_rows(g.n_rows, g.ymax, g.xres, g.yres, g.lonlat, min_slope_deg, u.rows);
    const size_t nb = (size_t)u.n * 8;
    if (u.host) {
        CU(cudaMalloc(&u.t_z.p, nb));
        CU(cudaMalloc(&u.t_area.p, nb));
        CU(cudaMemcpyAsync(u.t_z.p, g.elev, nb, cudaMemcpyHostToDevice, u.S));
    }
    CU(cudaMalloc(&u.t_w0.p, nb));
    CU(cudaMalloc(&u.t_w1.p, nb));
    CU(cudaMalloc(&u.t_rows.p, u.rows.size() * 8));
    CU(cudaMalloc(&u.t_ctl.p, (AC_N + 1 + kUpslopeBatch) * sizeof(int)));
    CU(cudaMemcpyAsync(u.t_rows.p, u.rows.data(), u.rows.size() * 8, cudaMemcpyHostToDevice, u.S));
    u.ctl = (int*)u.t_ctl.p;
    u.flags = u.ctl + AC_N;
    CU(cudaMemsetAsync(u.ctl, 0, AC_N * sizeof(int), u.S));
    u.z = u.host ? (const double*)u.t_z.p : g.elev;
    u.d_rows = (const double*)u.t_rows.p;
    u.area = u.host ? (double*)u.t_area.p : out_area;
    u.w[0] = (double*)u.t_w0.p;
    u.w[1] = (double*)u.t_w1.p;
    FillParams fp{u.z, u.d_rows, (int)g.n_rows, (int)g.n_cols};
    k_fill_init<<<(unsigned)((u.n + 255) / 256), 256, 0, u.S>>>(fp, u.w[0], u.ctl + AC_BADZ, u.ctl + AC_NVALID);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(u.hctl, u.ctl, AC_N * sizeof(int), cudaMemcpyDeviceToHost, u.S));
    CU(cudaStreamSynchronize(u.S));
    if (u.hctl[AC_BADZ]) return fail(ctx, SPLASH_ERR_BAD_ARG, "%s: elev has +-inf values (NaN is NA)", u.fn);
    return SPLASH_OK;
}

extern "C++" {  // templates inside the file's extern "C" block
// Jacobi sweeps launched in batches between reads of their changed flags (no host round trip per sweep), until a
// sweep changes nothing; at most n sweeps.  launch(j, s) enqueues global sweep s as sweep j of the batch.
template <class Launch>
static int run_sweeps(splash_ctx* ctx, UpslopeRun& u, const char* what, Launch launch, int64_t* sweeps_out) {
    int64_t sweeps = 0;
    bool converged = false;
    for (int batch = 4; !converged;) {
        const int one = 1;
        CU(cudaMemcpyAsync(u.flags, &one, sizeof(int), cudaMemcpyHostToDevice, u.S));
        CU(cudaMemsetAsync(u.flags + 1, 0, batch * sizeof(int), u.S));
        for (int j = 1; j <= batch; ++j) launch(j, sweeps + j - 1);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(u.hctl, u.flags + 1, batch * sizeof(int), cudaMemcpyDeviceToHost, u.S));
        CU(cudaStreamSynchronize(u.S));
        for (int j = 0; j < batch && !converged; ++j) {
            ++sweeps;
            converged = u.hctl[j] == 0;
        }
        if (!converged && sweeps >= u.n)
            return fail(ctx, SPLASH_ERR_CUDA, "%s: %s did not converge in %lld sweeps", u.fn, what, (long long)u.n);
        batch = std::min(2 * batch, kUpslopeBatch);
    }
    *sweeps_out = sweeps;
    return SPLASH_OK;
}

// The fill; *wf: the filled surface (written by the last sweep, equal to its input: nothing changed).
static int upslope_fill(splash_ctx* ctx, UpslopeRun& u, int n_rows, int n_cols, int64_t* sweeps, const double** wf) {
    using namespace upslope;
    FillParams fp{u.z, u.d_rows, n_rows, n_cols};
    const dim3 fgrid((unsigned)((n_cols + kFT - 1) / kFT), (unsigned)((n_rows + kFT - 1) / kFT)), fblock(kFT, kFRows);
    const int rc = run_sweeps(ctx, u, "the fill", [&](int j, int64_t s) {
        k_fill_sweep<<<fgrid, fblock, 0, u.S>>>(fp, u.w[s & 1], u.w[(s + 1) & 1], u.flags, j);
    }, sweeps);
    if (rc) return rc;
    *wf = u.w[*sweeps & 1];
    return SPLASH_OK;
}

// Clear the frontier words of ctl before a seed kernel fills the first frontier (n_valid stays).
static int rounds_reset(splash_ctx* ctx, UpslopeRun& u) {
    CU(cudaMemsetAsync(u.ctl, 0, upslope::AC_NVALID * sizeof(int), u.S));
    return SPLASH_OK;
}

// The frontier rounds of k_accum<Rule> in cooperative launches until the frontier is empty; a launch that does not
// finish runs at least one round, and there are at most n rounds.
template <class Rule>
static int run_rounds(splash_ctx* ctx, UpslopeRun& u, Rule p, const char* what, int64_t* rounds) {
    using namespace upslope;
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_accum<Rule>, kAccThreads, 0));
    if (per_sm < 1) return fail(ctx, SPLASH_ERR_CUDA, "%s: k_accum does not fit an SM", u.fn);
    const unsigned agrid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((int64_t)per_sm * ctx->sm_count, (u.n + kAccThreads - 1) / kAccThreads));
    void* args[] = {&p};
    int64_t launches = 0;
    for (int batch = 2;; batch = std::min(2 * batch, 16)) {
        if (launches > u.n + 1) return fail(ctx, SPLASH_ERR_CUDA, "%s: the %s did not finish", u.fn, what);
        for (int j = 0; j < batch; ++j) CU(cudaLaunchCooperativeKernel((const void*)k_accum<Rule>, agrid, kAccThreads, args, 0, u.S));
        launches += batch;
        CU(cudaMemcpyAsync(u.hctl, u.ctl, AC_N * sizeof(int), cudaMemcpyDeviceToHost, u.S));
        CU(cudaStreamSynchronize(u.S));
        if (u.hctl[AC_ERR]) return fail(ctx, SPLASH_ERR_CUDA, "%s: more %s rounds than valid cells", u.fn, what);
        if (u.hctl[AC_DONE]) break;
    }
    *rounds = u.hctl[AC_ROUNDS];
    return SPLASH_OK;
}

}  // extern "C++"

// area (and the optional filled surface) to the caller's arrays, then wait for the stream.
static int upslope_finish(splash_ctx* ctx, UpslopeRun& u, double* area, double* filled, const double* wf) {
    const size_t nb = (size_t)u.n * 8;
    if (u.host) {
        CU(cudaMemcpyAsync(area, u.area, nb, cudaMemcpyDeviceToHost, u.S));
        if (filled) CU(cudaMemcpyAsync(filled, wf, nb, cudaMemcpyDeviceToHost, u.S));
    } else if (filled) {
        CU(cudaMemcpyAsync(filled, wf, nb, cudaMemcpyDeviceToDevice, u.S));
    }
    CU(cudaStreamSynchronize(u.S));
    return SPLASH_OK;
}

int splash_upslope_area_run(splash_ctx* ctx, const splash_upslope_in* in, splash_upslope_out* out) {
    using namespace upslope;
    if (ctx && ctx->multi) {  // single-GPU work: the context's first lane does it
        splash_ctx* lane = first_lane(ctx);
        const int rc = splash_upslope_area_run(lane, in, out);
        ctx->err = lane->err;
        return rc;
    }
    if (!ctx) return SPLASH_ERR_BAD_ARG;
    ctx->err.clear();
    if (!in || !out) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_upslope_area_run: NULL in/out");
    out->fill_sweeps = 0;
    out->accum_rounds = 0;
    UpslopeRun u;
    u.fn = "splash_upslope_area_run";
    const UpslopeGeom g{in->n_rows, in->n_cols, in->elev, in->ymax, in->xres, in->yres, in->lonlat, in->mem_kind};
    if (int rc = upslope_check(ctx, g)) return rc;
    if (!std::isfinite(in->min_slope_deg) || !(in->min_slope_deg > 0.0) || !(in->min_slope_deg < 90.0))
        return fail(ctx, SPLASH_ERR_BAD_ARG, "min_slope_deg must be in (0, 90)");
    const int nr = (int)in->n_rows, ncol = (int)in->n_cols;
    if ((int64_t)nr * ncol == 0) return SPLASH_OK;
    if (!in->elev || !out->area) return fail(ctx, SPLASH_ERR_BAD_ARG, "NULL elev/area");
    if (int rc = upslope_begin(ctx, u, g, in->min_slope_deg, out->area)) return rc;
    const double* wf = nullptr;
    if (int rc = upslope_fill(ctx, u, nr, ncol, &out->fill_sweeps, &wf)) return rc;

    // accumulation
    TmpDev t_s, t_ndon, t_f0, t_f1;
    CU(cudaMalloc(&t_s.p, (size_t)u.n * 8));
    CU(cudaMalloc(&t_ndon.p, (size_t)u.n * 4));
    CU(cudaMalloc(&t_f0.p, (size_t)u.n * 4));
    CU(cudaMalloc(&t_f1.p, (size_t)u.n * 4));
    MfdRule ap{};
    ap.w = wf;
    ap.rows = u.d_rows;
    ap.s = (double*)t_s.p;
    ap.area = u.area;
    ap.ndon = (int*)t_ndon.p;
    ap.front[0] = (int*)t_f0.p;
    ap.front[1] = (int*)t_f1.p;
    ap.ctl = u.ctl;
    ap.n_rows = nr;
    ap.n_cols = ncol;
    if (int rc = rounds_reset(ctx, u)) return rc;
    k_flow_prep<<<(unsigned)((u.n + 255) / 256), 256, 0, u.S>>>(ap);
    CU(cudaGetLastError());
    if (int rc = run_rounds(ctx, u, ap, "accumulation", &out->accum_rounds)) return rc;
    return upslope_finish(ctx, u, out->area, out->filled, wf);
}

int splash_upslope_dinf_run(splash_ctx* ctx, const splash_dinf_in* in, splash_dinf_out* out) {
    using namespace upslope;
    if (ctx && ctx->multi) {  // single-GPU work: the context's first lane does it
        splash_ctx* lane = first_lane(ctx);
        const int rc = splash_upslope_dinf_run(lane, in, out);
        ctx->err = lane->err;
        return rc;
    }
    if (!ctx) return SPLASH_ERR_BAD_ARG;
    ctx->err.clear();
    if (!in || !out) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_upslope_dinf_run: NULL in/out");
    out->fill_sweeps = 0;
    out->flat_rounds = 0;
    out->accum_rounds = 0;
    UpslopeRun u;
    u.fn = "splash_upslope_dinf_run";
    const UpslopeGeom g{in->n_rows, in->n_cols, in->elev, in->ymax, in->xres, in->yres, in->lonlat, in->mem_kind};
    if (int rc = upslope_check(ctx, g)) return rc;
    const int nr = (int)in->n_rows, ncol = (int)in->n_cols;
    if ((int64_t)nr * ncol == 0) return SPLASH_OK;
    if (!in->elev || !out->area) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_upslope_dinf_run: NULL elev/area");
    if (int rc = upslope_begin(ctx, u, g, 0.0, out->area)) return rc;  // eps = 0: PitRemove fills to flat
    const double* wf = nullptr;
    if (int rc = upslope_fill(ctx, u, nr, ncol, &out->fill_sweeps, &wf)) return rc;
    const int64_t n = u.n;
    const unsigned grid = (unsigned)((n + 255) / 256);

    // flats: classes, labels, the two distances, the per-flat maximum, the mask M (in place of the towards distance)
    TmpDev t_cls, t_lab0, t_lab1, t_tow, t_away, t_hmax, t_ndon, t_f0, t_f1, t_rec, t_pd, t_angle;
    CU(cudaMalloc(&t_cls.p, (size_t)n));
    for (TmpDev* t : {&t_lab0, &t_lab1, &t_tow, &t_away, &t_hmax, &t_ndon, &t_f0, &t_f1}) CU(cudaMalloc(&t->p, (size_t)n * 4));
    CU(cudaMalloc(&t_rec.p, (size_t)n));
    CU(cudaMalloc(&t_pd.p, (size_t)n * 8));
    unsigned char* cls = (unsigned char*)t_cls.p;
    int* lab[2] = {(int*)t_lab0.p, (int*)t_lab1.p};
    int* front[2] = {(int*)t_f0.p, (int*)t_f1.p};
    FlatParams fp{wf, cls, (int*)t_tow.p, (int*)t_away.p, (int*)t_hmax.p, nr, ncol};
    k_flat_mark<<<grid, 256, 0, u.S>>>(fp, lab[0]);
    CU(cudaGetLastError());
    int64_t label_sweeps = 0, tow_rounds = 0, away_rounds = 0;
    if (int rc = run_sweeps(ctx, u, "the flat labelling", [&](int j, int64_t s) {
            k_flat_label<<<grid, 256, 0, u.S>>>(fp, lab[s & 1], lab[(s + 1) & 1], u.flags, j);
        }, &label_sweeps))
        return rc;
    const int* label = lab[label_sweeps & 1];
    if (int rc = rounds_reset(ctx, u)) return rc;
    k_flat_seed<false><<<grid, 256, 0, u.S>>>(fp, front[0], u.ctl);
    CU(cudaGetLastError());
    if (int rc = run_rounds(ctx, u, FlatBfs{cls, fp.tow, {front[0], front[1]}, u.ctl, nr, ncol}, "flat distance", &tow_rounds)) return rc;
    if (int rc = rounds_reset(ctx, u)) return rc;
    k_flat_seed<true><<<grid, 256, 0, u.S>>>(fp, front[0], u.ctl);
    CU(cudaGetLastError());
    if (int rc = run_rounds(ctx, u, FlatBfs{cls, fp.away, {front[0], front[1]}, u.ctl, nr, ncol}, "flat distance", &away_rounds)) return rc;
    k_flat_height<<<grid, 256, 0, u.S>>>(fp, label);
    k_flat_mask<<<grid, 256, 0, u.S>>>(fp, label);
    CU(cudaGetLastError());
    out->flat_rounds = label_sweeps + tow_rounds + away_rounds;

    // directions
    double* angle = out->angle;
    if (angle && u.host) {
        CU(cudaMalloc(&t_angle.p, (size_t)n * 8));
        angle = (double*)t_angle.p;
    }
    DinfParams dp{wf, u.d_rows, cls, fp.tow, (unsigned char*)t_rec.p, (double*)t_pd.p, angle, nr, ncol};
    k_dinf_dir<<<grid, 256, 0, u.S>>>(dp);
    CU(cudaGetLastError());

    // accumulation
    DinfRule ar{dp.rec, dp.pd, u.d_rows, u.area, (int*)t_ndon.p, {front[0], front[1]}, u.ctl, nr, ncol};
    if (int rc = rounds_reset(ctx, u)) return rc;
    k_dinf_prep<<<grid, 256, 0, u.S>>>(ar, wf);
    CU(cudaGetLastError());
    if (int rc = run_rounds(ctx, u, ar, "accumulation", &out->accum_rounds)) return rc;
    if (out->angle && u.host) CU(cudaMemcpyAsync(out->angle, angle, (size_t)n * 8, cudaMemcpyDeviceToHost, u.S));
    return upslope_finish(ctx, u, out->area, out->filled, wf);
}

int splash_month2day_linear(splash_ctx* ctx, const splash_m2d_in* in, void* daily_out) {
    if (ctx && ctx->multi) {  // single-GPU work: the context's first lane does it
        splash_ctx* lane = first_lane(ctx);
        const int rc = splash_month2day_linear(lane, in, daily_out);
        ctx->err = lane->err;
        return rc;
    }
    if (!ctx) return SPLASH_ERR_BAD_ARG;
    ctx->err.clear();
    if (!in) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_month2day_linear: NULL in");
    const int64_t nc = in->n_cells, nm = in->n_months, nd = in->n_days;
    if (nc < 0 || nm < 0 || nd < 0 || nm > INT32_MAX) return fail(ctx, SPLASH_ERR_BAD_ARG, "negative or oversized n_cells/n_months/n_days");
    const int64_t istride = in->in_stride ? in->in_stride : nc, ostride = in->out_stride ? in->out_stride : nc;
    if (istride < nc || ostride < nc) return fail(ctx, SPLASH_ERR_BAD_ARG, "stride smaller than n_cells");
    if (in->mem_kind != SPLASH_MEM_HOST && in->mem_kind != SPLASH_MEM_DEVICE)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "mem_kind must be SPLASH_MEM_HOST or SPLASH_MEM_DEVICE");
    if (nc == 0 || nd == 0) return SPLASH_OK;
    if (!daily_out || (nm > 0 && (!in->monthly || !in->month_start))) return fail(ctx, SPLASH_ERR_BAD_ARG, "NULL monthly/month_start/daily_out");
    for (int64_t m = 1; m < nm; ++m)
        if (in->month_start[m] <= in->month_start[m - 1]) return fail(ctx, SPLASH_ERR_BAD_ARG, "month_start must be strictly increasing");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t S = ctx->s_run[0];
    const size_t osz = in->out_f32 ? 4 : 8;
    int32_t* d_xs = nullptr;
    int2* d_knots = nullptr;
    double* d_monthly = nullptr;
    void* d_out = nullptr;
    int32_t* d_day_m = nullptr;
    double* d_day_q = nullptr;
    int rc = SPLASH_OK;
    auto cu = [&](cudaError_t e) {
        if (e != cudaSuccess && rc == SPLASH_OK) {
            rc = (e == cudaErrorMemoryAllocation) ? SPLASH_ERR_NOMEM : SPLASH_ERR_CUDA;
            fail(ctx, rc, "splash_month2day_linear: %s", cudaGetErrorString(e));
        }
        return e == cudaSuccess;
    };
    M2dParams p{};
    p.ipitch = istride;
    p.n_cells = nc;
    p.n_months = (int)nm;
    const int64_t day_chunk = getenv("SPLASH_M2D_CHUNK") ? std::max(1, atoi(getenv("SPLASH_M2D_CHUNK"))) : 512;
    // launch shape (measured in profiles/README.md: one cell per thread, 512-day chunks, no lock-step is the most
    // repeatable; the other shapes stay selectable for the round-2 study of the row-strided store stream)
    const int want_v = getenv("SPLASH_M2D_VEC") ? atoi(getenv("SPLASH_M2D_VEC")) : 1;
    const int sync_days = getenv("SPLASH_M2D_SYNC") ? atoi(getenv("SPLASH_M2D_SYNC")) : 0;
    if (cu(cudaMalloc(&d_xs, (size_t)std::max<int64_t>(nm, 1) * 4)) && cu(cudaMalloc(&d_knots, (size_t)nc * sizeof(int2))) &&
        (nm == 0 || cu(cudaMemcpyAsync(d_xs, in->month_start, (size_t)nm * 4, cudaMemcpyHostToDevice, S)))) {
        p.xs = d_xs;
        p.knots = d_knots;
        bool have_knots = false;
        const char* kern = getenv("SPLASH_M2D_KERNEL");
        const bool band = kern && !strcmp(kern, "band");
        const int band_d = getenv("SPLASH_M2D_BAND_D") ? std::max(1, atoi(getenv("SPLASH_M2D_BAND_D"))) : 16;
        const int band_k = getenv("SPLASH_M2D_BAND_K") ? atoi(getenv("SPLASH_M2D_BAND_K")) : 4;
        auto launch_band = [&](int64_t day0, int64_t day1) {
            if (!d_day_m) {  // per-day table: month index and quotient, host arithmetic (IEEE division like R)
                std::vector<int32_t> dm((size_t)nd);
                std::vector<double> dq((size_t)nd);
                int64_t m = -1;
                for (int64_t d = 0; d < nd; ++d) {
                    while (m + 1 < nm && in->month_start[m + 1] <= d) ++m;
                    dm[(size_t)d] = (int32_t)m;
                    dq[(size_t)d] = (m >= 0 && m + 1 < nm)
                                        ? (double)(d - in->month_start[m]) / (double)(in->month_start[m + 1] - in->month_start[m]) : 0.0;
                }
                if (!cu(cudaMalloc(&d_day_m, (size_t)nd * 4)) || !cu(cudaMalloc(&d_day_q, (size_t)nd * 8)) ||
                    !cu(cudaMemcpy(d_day_m, dm.data(), (size_t)nd * 4, cudaMemcpyHostToDevice)) ||
                    !cu(cudaMemcpy(d_day_q, dq.data(), (size_t)nd * 8, cudaMemcpyHostToDevice)))
                    return false;
            }
            M2dBand b{};
            b.monthly = p.monthly; b.ipitch = p.ipitch; b.out = p.out; b.opitch = p.opitch; b.xs = p.xs; b.knots = p.knots;
            b.day_m = d_day_m; b.day_q = d_day_q; b.n_cells = nc; b.n_months = (int)nm; b.out_day0 = p.out_day0; b.D = band_d;
            const int K = (band_k >= 4) ? 4 : (band_k >= 2 ? 2 : 1);
            const int64_t cta_x = (nc + 256 * K - 1) / (256 * K);
            for (int64_t a = day0; a < day1 && rc == SPLASH_OK; a += (int64_t)band_d * 65535) {
                b.day0 = a;
                b.day1 = std::min(day1, a + (int64_t)band_d * 65535);
                dim3 grid((unsigned)cta_x, (unsigned)((b.day1 - b.day0 + band_d - 1) / band_d));
#define M2D_BAND(OT) \
    do { \
        if (K == 4) k_month2day_band<OT, 4><<<grid, 256, 0, S>>>(b); \
        else if (K == 2) k_month2day_band<OT, 2><<<grid, 256, 0, S>>>(b); \
        else k_month2day_band<OT, 1><<<grid, 256, 0, S>>>(b); \
    } while (0)
                if (in->out_f32) M2D_BAND(float);
                else M2D_BAND(double);
#undef M2D_BAND
            }
            return cu(cudaGetLastError());
        };
        auto launch = [&](int64_t day0, int64_t day1) {
            if (!have_knots) {
                k_m2d_knots<<<(unsigned)((nc + 255) / 256), 256, 0, S>>>(p);
                have_knots = true;
            }
            if (band) return launch_band(day0, day1);
            // cells per thread: as many as one aligned 16-byte store holds, when the rows allow it
            int V = 1;
            for (int v = (int)(16 / osz); v > 1; v >>= 1)
                if (v <= want_v && nc % v == 0 && (p.opitch * osz) % (v * osz) == 0 && ((uintptr_t)p.out % (v * osz)) == 0) {
                    V = v;
                    break;
                }
            const int64_t cta_x = (nc / V + 255) / 256;
            p.chunk = day_chunk;
            for (int64_t a = day0; a < day1 && rc == SPLASH_OK; a += p.chunk * 65535) {  // grid.y limit
                p.day0 = a;
                p.day1 = std::min(day1, a + p.chunk * 65535);
                dim3 grid((unsigned)cta_x, (unsigned)((p.day1 - p.day0 + p.chunk - 1) / p.chunk));
#define M2D_LAUNCH(OT, VV) \
    do { \
        if (sync_days > 0) k_month2day<OT, VV, 8><<<grid, 256, 0, S>>>(p); \
        else k_month2day<OT, VV, 0><<<grid, 256, 0, S>>>(p); \
    } while (0)
                if (in->out_f32) {
                    if (V == 4) M2D_LAUNCH(float, 4);
                    else if (V == 2) M2D_LAUNCH(float, 2);
                    else M2D_LAUNCH(float, 1);
                } else {
                    if (V == 2) M2D_LAUNCH(double, 2);
                    else M2D_LAUNCH(double, 1);
                }
#undef M2D_LAUNCH
            }
            return cu(cudaGetLastError());
        };
        if (in->mem_kind == SPLASH_MEM_DEVICE) {
            p.monthly = in->monthly;
            p.out = daily_out;
            p.opitch = ostride;
            p.out_day0 = 0;
            launch(0, nd);
        } else {
            // host arrays: the monthly block goes up once, the daily series come back in chunks of days
            const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(nd, ((int64_t)1 << 30) / std::max<int64_t>(1, nc * (int64_t)osz)));
            if (cu(cudaMalloc(&d_monthly, (size_t)std::max<int64_t>(nm, 1) * nc * 8)) && cu(cudaMalloc(&d_out, (size_t)chunk * nc * osz)) &&
                (nm == 0 || cu(cudaMemcpy2DAsync(d_monthly, (size_t)nc * 8, in->monthly, (size_t)istride * 8, (size_t)nc * 8, (size_t)nm,
                                                 cudaMemcpyHostToDevice, S)))) {
                p.monthly = d_monthly;
                p.ipitch = nc;
                p.out = d_out;
                p.opitch = nc;
                for (int64_t a = 0; a < nd && rc == SPLASH_OK; a += chunk) {
                    const int64_t b = std::min(nd, a + chunk);
                    p.out_day0 = a;
                    if (!launch(a, b)) break;
                    cu(cudaMemcpy2DAsync((char*)daily_out + (size_t)a * ostride * osz, (size_t)ostride * osz, d_out, (size_t)nc * osz,
                                         (size_t)nc * osz, (size_t)(b - a), cudaMemcpyDeviceToHost, S));
                    cu(cudaStreamSynchronize(S));
                }
            }
        }
    }
    cu(cudaStreamSynchronize(S));
    cudaFree(d_xs);
    cudaFree(d_knots);
    cudaFree(d_monthly);
    cudaFree(d_out);
    cudaFree(d_day_m);
    cudaFree(d_day_q);
    return rc;
}


}  // extern "C"

namespace {

// Everything one call needs; run() enqueues the whole job and waits once at the end.
template <typename FT>
struct GridJob {
    splash_ctx* ctx;
    const splash_grid_in* in;
    splash_grid_out* out;
    splash_opts opts;
    int64_t nc, nd, n_out, istride, ostride;
    int64_t apitch, xpitch, spitch;  // layer pitches of soil/au, of state_final/cell_diag, of state_init
    bool in_dev, out_dev, monthly;
    int max_spin;
    double spin_tol;
    double* out_ptr[9];
    int n_out_layers = 0;
    int64_t tile = 0, n_tiles = 0, pitch = 0;
    int n_work = 0;
    // host-fed calls: the data every tile's spin-up needs (the whole tc series for the snow threshold, the
    // first year of sw and pn, the per-cell inputs) is uploaded for ALL tiles before the bulk of the forcing,
    // so that every tile's stragglers start their chain early instead of when their tile's turn comes
    bool ahead = false;
    int64_t ncp = 0, nd1 = 0;        // pitch of the call-wide buffers, rows of the first-year copies
    void *a_tc = nullptr, *a_sw1 = nullptr, *a_pn1 = nullptr;
    double* a_cellin = nullptr;
    Pool pool{};
    int64_t launches = 0;

    struct TileEv {
        cudaEvent_t h2d0, h2d1, h2da, h2db;       // h2d stream: the tile's uploads (`ahead` mode: h2d0..h2da spin-up data, h2db..h2d1 the rest)
        cudaEvent_t k0, kf0, kf1, kr1, kb0, kb1;  // run stream: begin, k_spin_first begin/end, rounds end, bulk begin/end
        cudaEvent_t exported, exported_b, run, d2h0, d2h1;  // stragglers exported (state / whole forcing); kernels done; downloads
        cudaEvent_t ps1, ps2, pm;                 // pool stream: spin stage 1 done, stage 2 done, daily integration done
    };
    std::vector<TileEv> ev;
    std::vector<RunParams> rps, pps;  // per tile: the tile's view, the pool's view
    std::vector<SetupParams> sps;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;

    TileCtl* ctl(int64_t t) const { return (TileCtl*)ctx->ctl.p + t; }
    cudaStream_t run_stream(int64_t t) const { return ctx->s_run[t % ctx->n_run_streams]; }
    int work_of(int64_t t) const { return (in_dev || ahead) ? (int)t : (int)(t % kSlots); }
    int64_t cells_of(int64_t t) const { return std::min<int64_t>(tile, nc - t * tile); }

    int plan() {
        const size_t fsz = sizeof(FT);
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        size_t held = ctx->pool_mem.cap + ctx->ctl.cap + ctx->ahead_mem.cap;
        for (int i = 0; i < kSlots; ++i) {
            for (int k = 0; k < 3; ++k) held += ctx->forcing[i][k].cap;
            held += ctx->cellin[i].cap + ctx->outs[i].cap;
        }
        for (auto& w : ctx->work) held += w.cc.cap + w.work_d.cap + w.work_i.cap + w.diag.cap;
        // (a lane of a cluster shares its device with the other lanes)
        double budget = 0.80 * (double)(free_b + held) * ctx->mem_share;

        // ---- straggler pool: a slice of the budget, ~4 % of the cells -----------------------------------
        const double per_entry = 3.0 * (double)std::max<int64_t>(nd, 1) * fsz + (double)(NCC + 11 + SPLASH_NDIAG + 1) * 8.0 + 12.0 +
                                 (double)n_out_layers * (double)std::max<int64_t>(n_out, 1) * 8.0 +
                                 (double)kSpinYear * kDayPrePad * 8.0;
        int64_t cap = std::min<int64_t>(std::max<int64_t>(nc / 24, 2048), 131072);
        cap = std::min<int64_t>(cap, (int64_t)(0.10 * budget / per_entry));
        cap = std::min<int64_t>(std::max<int64_t>(cap, 32), round_up(nc, 32));
        if (ctx->pool_cap > 0) cap = ctx->pool_cap;
        cap = round_up(cap, 32);
        if (opts.skip_spinup) cap = 32;  // nothing spins
        {
            size_t off = 0;
            auto carve = [&](size_t bytes) {
                const size_t o = off;
                off += (bytes + 255) / 256 * 256;
                return o;
            };
            const size_t o_f = carve(3 * (size_t)std::max<int64_t>(nd, 1) * cap * fsz);
            const size_t o_cc = carve((size_t)NCC * cap * 8);
            const size_t o_wd = carve((size_t)11 * cap * 8);
            const size_t o_wi = carve((size_t)3 * cap * 4);
            const size_t o_out = carve((size_t)n_out_layers * std::max<int64_t>(n_out, 1) * cap * 8);
            const size_t o_dg = carve((size_t)SPLASH_NDIAG * cap * 8);
            const size_t o_cell = carve((size_t)cap * 8);
            const size_t o_tab = carve((size_t)kSpinYear * kDayPrePad * cap * 8);
            const size_t o_hard = carve((size_t)cap * 4 * 2);
            const size_t o_cnt = carve(256);
            if (int rc = ensure(ctx, ctx->pool_mem, off)) return rc;
            char* b = (char*)ctx->pool_mem.p;
            for (int k = 0; k < 3; ++k) pool.f[k] = b + o_f + (size_t)k * std::max<int64_t>(nd, 1) * cap * fsz;
            pool.cc = (double*)(b + o_cc);
            double* wd = (double*)(b + o_wd);
            int* wi = (int*)(b + o_wi);
            pool.w.st = wd;
            pool.w.w1 = wd + 5 * cap;
            pool.w.snap = wd + 6 * cap;
            pool.w.passes = wi;
            pool.w.snap_pass = wi + cap;
            pool.w.status = wi + 2 * cap;
            pool.w.frost = nullptr;
            pool.w.key = nullptr;
            pool.w.pitch = cap;
            int li = 0;
            for (int k = 0; k < 9; ++k)
                pool.out[k] = out_ptr[k] ? (double*)(b + o_out) + (size_t)(li++) * std::max<int64_t>(n_out, 1) * cap : nullptr;
            pool.diag = (double*)(b + o_dg);
            pool.cell = (long long*)(b + o_cell);
            pool.table = (double*)(b + o_tab);
            pool.hard[0] = (int*)(b + o_hard);
            pool.hard[1] = pool.hard[0] + cap;
            pool.count = (unsigned long long*)(b + o_cnt);
            pool.cap = cap;
            budget -= (double)off;
        }

        // ---- host-fed calls: spin-up data of all tiles ahead of the bulk of the forcing, if it fits --------
        const double work_cell = (double)(NCC + 11 + SPLASH_NDIAG) * 8.0 + kWorkInts * 4.0;
        nd1 = std::min<int64_t>(nd, kSpinYear);
        ncp = round_up(nc, 32);
        const double ahead_bytes = (double)ncp * ((double)(nd + 2 * nd1) * fsz + 14 * 8.0);
        {
            // worth it only if what is left still gives decent tiles (three slots of sw + pn [+ outputs])
            const double left = budget - ahead_bytes - work_cell * (double)nc;
            const double slot1 = 2.0 * (double)nd * (double)fsz + (out_dev ? 0.0 : (double)n_out_layers * (double)n_out * 8.0);
            const double tile_left = left / ((double)kSlots * std::max(slot1, 1.0));
            ahead = !in_dev && !opts.skip_spinup && ctx->spin_ahead && nd > 0 && left > 0 &&
                    tile_left >= (double)std::min<int64_t>(nc, std::max<int64_t>(32768, nc / 16));
        }
        if (ahead) budget -= ahead_bytes;
        // ---- tile size ------------------------------------------------------------------------------------
        double slot_cell = 0.0;  // bytes per cell held once per slot
        if (!in_dev) slot_cell += (ahead ? 2.0 * (double)nd * (double)fsz : 3.0 * (double)nd * (double)fsz + 14 * 8.0);
        if (!out_dev) slot_cell += (double)n_out_layers * (double)n_out * 8.0;
        if (in_dev || ahead) budget -= work_cell * (double)nc;  // one work set per tile
        else slot_cell += work_cell;                            // one work set per slot
        if (budget <= 0) return fail(ctx, SPLASH_ERR_NOMEM, "not enough device memory for the per-cell work arrays");
        int64_t t_auto = std::min<int64_t>(kTileTarget, std::max<int64_t>(16384, round_up((nc + 3) / 4, 1024)));
        t_auto = std::max<int64_t>(t_auto, round_up((nc + kPoolStreams - 1) / kPoolStreams, 1024));  // <= 16 tiles: one pool stream each
        if (slot_cell > 0) t_auto = std::min<int64_t>(t_auto, (int64_t)(budget / ((double)kSlots * slot_cell)));
        tile = opts.tile_cells > 0 ? opts.tile_cells : t_auto;
        tile = std::min<int64_t>(tile, nc);
        if (tile < nc) {
            int64_t t2 = tile / 1024 * 1024;
            if (t2 == 0) t2 = tile / 128 * 128;
            tile = std::max<int64_t>(128, t2);
        }
        if (tile <= 0) return fail(ctx, SPLASH_ERR_NOMEM, "not enough device memory for one tile");
        if (tile > (int64_t)INT32_MAX / 2) tile = (int64_t)INT32_MAX / 2 / 1024 * 1024;
        n_tiles = (nc + tile - 1) / tile;
        pitch = round_up(tile, 32);
        n_work = (in_dev || ahead) ? (int)n_tiles : (int)std::min<int64_t>(kSlots, n_tiles);
        return SPLASH_OK;
    }

    int allocate() {
        const size_t fsz = sizeof(FT);
        if ((int)ctx->work.size() < n_work) ctx->work.resize((size_t)n_work);
        for (int w = 0; w < n_work; ++w) {
            WorkSet& ws = ctx->work[(size_t)w];
            if (int rc = ensure(ctx, ws.cc, (size_t)NCC * pitch * 8)) return rc;
            if (int rc = ensure(ctx, ws.work_d, (size_t)11 * pitch * 8)) return rc;
            if (int rc = ensure(ctx, ws.work_i, (size_t)kWorkInts * pitch * 4)) return rc;
            if (int rc = ensure(ctx, ws.diag, (size_t)SPLASH_NDIAG * pitch * 8)) return rc;
        }
        const int n_slots = (int)std::min<int64_t>(kSlots, n_tiles);
        for (int s = 0; s < n_slots; ++s) {
            if (!in_dev) {
                for (int k = 0; k < 3; ++k)
                    if (!(ahead && k == 1))  // (the tc series lives in the call-wide buffer)
                        if (int rc = ensure(ctx, ctx->forcing[s][k], (size_t)std::max<int64_t>(nd, 1) * pitch * fsz)) return rc;
                if (!ahead)
                    if (int rc = ensure(ctx, ctx->cellin[s], (size_t)14 * pitch * 8)) return rc;
            }
            if (!out_dev && n_out_layers)
                if (int rc = ensure(ctx, ctx->outs[s], (size_t)n_out_layers * std::max<int64_t>(n_out, 1) * pitch * 8)) return rc;
        }
        if (ahead) {
            const size_t b_tc = (size_t)nd * ncp * fsz, b_1 = (size_t)nd1 * ncp * fsz;
            if (int rc = ensure(ctx, ctx->ahead_mem, b_tc + 2 * b_1 + (size_t)14 * ncp * 8 + 1024)) return rc;
            char* b = (char*)ctx->ahead_mem.p;
            a_tc = b;
            a_sw1 = b + b_tc;
            a_pn1 = b + b_tc + b_1;
            a_cellin = (double*)(b + (b_tc + 2 * b_1 + 255) / 256 * 256);
        }
        if (int rc = ensure(ctx, ctx->ctl, sizeof(TileCtl) * (size_t)n_tiles)) return rc;
        CU(cudaMemsetAsync(ctx->ctl.p, 0, sizeof(TileCtl) * (size_t)n_tiles, ctx->s_h2d));
        CU(cudaMemsetAsync(pool.count, 0, 256, ctx->s_h2d));
        CU(cudaStreamSynchronize(ctx->s_h2d));
        ev.resize((size_t)n_tiles);
        for (auto& t : ev) {
            cudaEvent_t* timed[13] = {&t.h2d0, &t.h2d1, &t.k0, &t.kf0, &t.kf1, &t.kr1, &t.kb0, &t.kb1, &t.d2h0, &t.d2h1, &t.ps1, &t.ps2, &t.pm};
            for (auto* e : timed) CU(cudaEventCreate(e));
            CU(cudaEventCreate(&t.h2da));
            CU(cudaEventCreate(&t.h2db));
            CU(cudaEventCreateWithFlags(&t.exported_b, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&t.exported, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&t.run, cudaEventDisableTiming));
        }
        CU(cudaEventCreate(&ev_begin));
        CU(cudaEventCreate(&ev_end));
        rps.resize((size_t)n_tiles);
        pps.resize((size_t)n_tiles);
        sps.resize((size_t)n_tiles);
        return SPLASH_OK;
    }

    void release() {
        for (auto& t : ev) {
            cudaEvent_t all[18] = {t.h2d0, t.h2d1, t.k0, t.kf0, t.kf1, t.kr1, t.kb0, t.kb1, t.d2h0, t.d2h1, t.exported, t.run, t.ps1, t.ps2, t.pm, t.h2da, t.exported_b, t.h2db};
            for (auto e : all)
                if (e) cudaEventDestroy(e);
        }
        ev.clear();
        if (ev_begin) cudaEventDestroy(ev_begin);
        if (ev_end) cudaEventDestroy(ev_end);
        ev_begin = ev_end = nullptr;
    }

    // `ahead` mode, phase A: what the tile's spin-up needs, into the call-wide buffers
    int enqueue_h2d_ahead(int64_t t) {
        const size_t fsz = sizeof(FT);
        const int64_t c0 = t * tile, nct = cells_of(t);
        cudaStream_t H = ctx->s_h2d;
        CU(cudaEventRecord(ev[(size_t)t].h2d0, H));
        CU(cudaMemcpy2DAsync((char*)a_tc + (size_t)c0 * fsz, (size_t)ncp * fsz, (const char*)in->tc + (size_t)c0 * fsz, (size_t)istride * fsz,
                             (size_t)nct * fsz, (size_t)nd, cudaMemcpyHostToDevice, H));
        CU(cudaMemcpy2DAsync((char*)a_sw1 + (size_t)c0 * fsz, (size_t)ncp * fsz, (const char*)in->sw_in + (size_t)c0 * fsz,
                             (size_t)istride * fsz, (size_t)nct * fsz, (size_t)nd1, cudaMemcpyHostToDevice, H));
        CU(cudaMemcpy2DAsync((char*)a_pn1 + (size_t)c0 * fsz, (size_t)ncp * fsz, (const char*)in->pn + (size_t)c0 * fsz, (size_t)istride * fsz,
                             (size_t)nct * fsz, (size_t)nd1, cudaMemcpyHostToDevice, H));
        ctx->stats.h2d_bytes += (int64_t)nct * (nd + 2 * nd1) * (int64_t)fsz;
        double* ci = a_cellin + c0;
        const double* vec[5] = {in->lat, in->elev, in->slop, in->asp, in->resolution};
        for (int k = 0; k < 5; ++k)
            CU(cudaMemcpyAsync(ci + (size_t)k * ncp, vec[k] + c0, (size_t)nct * 8, cudaMemcpyHostToDevice, H));
        CU(cudaMemcpy2DAsync(ci + (size_t)5 * ncp, (size_t)ncp * 8, in->soil + c0, (size_t)apitch * 8, (size_t)nct * 8, 6, cudaMemcpyHostToDevice, H));
        CU(cudaMemcpy2DAsync(ci + (size_t)11 * ncp, (size_t)ncp * 8, in->au + c0, (size_t)apitch * 8, (size_t)nct * 8, (size_t)in->au_layers,
                             cudaMemcpyHostToDevice, H));
        ctx->stats.h2d_bytes += (int64_t)nct * 8 * (5 + 6 + in->au_layers);
        CU(cudaEventRecord(ev[(size_t)t].h2da, H));
        return SPLASH_OK;
    }

    // uploads of tile t into its slot (in `ahead` mode: the whole sw and pn series; tc is already there)
    int enqueue_h2d(int64_t t) {
        const size_t fsz = sizeof(FT);
        const int s = (int)(t % kSlots);
        const int64_t c0 = t * tile, nct = cells_of(t);
        cudaStream_t H = ctx->s_h2d;
        if (in_dev) {
            CU(cudaEventRecord(ev[(size_t)t].h2d0, H));
        } else {
            if (t >= kSlots) CU(cudaStreamWaitEvent(H, ev[(size_t)(t - kSlots)].run, 0));  // the slot's previous kernels are done
            CU(cudaEventRecord(ahead ? ev[(size_t)t].h2db : ev[(size_t)t].h2d0, H));
            const char* src[3] = {(const char*)in->sw_in, (const char*)in->tc, (const char*)in->pn};
            for (int k = 0; k < 3; ++k) {
                if (ahead && k == 1) continue;
                if (nd > 0)
                    CU(cudaMemcpy2DAsync(ctx->forcing[s][k].p, (size_t)pitch * fsz, src[k] + (size_t)c0 * fsz, (size_t)istride * fsz,
                                         (size_t)nct * fsz, (size_t)nd, cudaMemcpyHostToDevice, H));
                ctx->stats.h2d_bytes += (int64_t)nct * nd * (int64_t)fsz;
            }
            if (!ahead) {
                double* ci = (double*)ctx->cellin[s].p;
                const double* vec[5] = {in->lat, in->elev, in->slop, in->asp, in->resolution};
                for (int k = 0; k < 5; ++k)
                    CU(cudaMemcpyAsync(ci + (size_t)k * pitch, vec[k] + c0, (size_t)nct * 8, cudaMemcpyHostToDevice, H));
                CU(cudaMemcpy2DAsync(ci + (size_t)5 * pitch, (size_t)pitch * 8, in->soil + c0, (size_t)apitch * 8, (size_t)nct * 8, 6,
                                     cudaMemcpyHostToDevice, H));
                CU(cudaMemcpy2DAsync(ci + (size_t)11 * pitch, (size_t)pitch * 8, in->au + c0, (size_t)apitch * 8, (size_t)nct * 8,
                                     (size_t)in->au_layers, cudaMemcpyHostToDevice, H));
                ctx->stats.h2d_bytes += (int64_t)nct * 8 * (5 + 6 + in->au_layers);
            }
        }
        CU(cudaEventRecord(ev[(size_t)t].h2d1, H));
        return SPLASH_OK;
    }

    // kernel parameters of tile t (no CUDA calls)
    void setup_params(int64_t t) {
        const size_t fsz = sizeof(FT);
        const int s = (int)(t % kSlots);
        const int64_t c0 = t * tile, nct = cells_of(t);
        SetupParams& sp = sps[(size_t)t];
        RunParams& rp = rps[(size_t)t];
        sp = SetupParams{};
        rp = RunParams{};
        if (in_dev) {
            rp.sw = (const char*)in->sw_in + (size_t)c0 * fsz;
            rp.tc = (const char*)in->tc + (size_t)c0 * fsz;
            rp.pn = (const char*)in->pn + (size_t)c0 * fsz;
            rp.fpitch = rp.tpitch = rp.f1pitch = istride;
            rp.sw1 = rp.sw;
            rp.pn1 = rp.pn;
            sp.lat = in->lat + c0;
            sp.elev = in->elev + c0;
            sp.slop = in->slop + c0;
            sp.asp = in->asp + c0;
            sp.resolution = in->resolution + c0;
            sp.soil = in->soil + c0;
            sp.soil_pitch = apitch;
            sp.au = in->au + c0;
            sp.au_pitch = apitch;
        } else {
            rp.sw = ctx->forcing[s][0].p;
            rp.pn = ctx->forcing[s][2].p;
            rp.fpitch = pitch;
            const double* ci;
            int64_t cp;
            if (ahead) {
                rp.tc = (const char*)a_tc + (size_t)c0 * fsz;
                rp.sw1 = (const char*)a_sw1 + (size_t)c0 * fsz;
                rp.pn1 = (const char*)a_pn1 + (size_t)c0 * fsz;
                rp.tpitch = rp.f1pitch = ncp;
                ci = a_cellin + c0;
                cp = ncp;
            } else {
                rp.tc = ctx->forcing[s][1].p;
                rp.sw1 = rp.sw;
                rp.pn1 = rp.pn;
                rp.tpitch = rp.f1pitch = pitch;
                ci = (const double*)ctx->cellin[s].p;
                cp = pitch;
            }
            sp.lat = ci;
            sp.elev = ci + cp;
            sp.slop = ci + 2 * cp;
            sp.asp = ci + 3 * cp;
            sp.resolution = ci + 4 * cp;
            sp.soil = ci + 5 * cp;
            sp.soil_pitch = cp;
            sp.au = ci + 11 * cp;
            sp.au_pitch = cp;
        }

        // ---- kernel parameters of the tile ----------------------------------------------------------------
        WorkSet& ws = ctx->work[(size_t)work_of(t)];
        sp.au_layers = in->au_layers;
        sp.n_cells = (int)nct;
        sp.cc = (double*)ws.cc.p;
        sp.cpitch = pitch;
        sp.diag = (double*)ws.diag.p;
        sp.dpitch = pitch;
        rp.cc = sp.cc;
        rp.cpitch = pitch;
        rp.dtab = (const DayTab*)ctx->dtab.p;
        rp.dtab_spin = (const DayTab*)ctx->dtab_spin.p;
        rp.n_days = (int)nd;
        rp.n_cells = (int)nct;
        double* wd = (double*)ws.work_d.p;
        int* wi = (int*)ws.work_i.p;
        rp.w.st = wd;
        rp.w.w1 = wd + 5 * pitch;
        rp.w.snap = wd + 6 * pitch;
        rp.w.passes = wi;
        rp.w.snap_pass = wi + pitch;
        rp.w.status = wi + 2 * pitch;
        rp.w.frost = wi + 5 * pitch;
        rp.w.key = (unsigned char*)(wi + 7 * pitch);
        rp.w.pitch = pitch;
        rp.lists[0] = wi + 3 * pitch;
        rp.lists[1] = wi + 4 * pitch;
        rp.order = nullptr;
        rp.order_w = wi + 6 * pitch;
        rp.ctl = ctl(t);
        int li = 0;
        for (int k = 0; k < 9; ++k) {
            if (!out_ptr[k])
                rp.out[k] = nullptr;
            else if (out_dev)
                rp.out[k] = out_ptr[k] + c0;
            else
                rp.out[k] = (double*)ctx->outs[s].p + (size_t)(li++) * std::max<int64_t>(n_out, 1) * pitch;
        }
        rp.opitch = out_dev ? ostride : pitch;
        rp.diag = sp.diag;
        rp.dpitch = pitch;
        rp.max_spin = max_spin;
        rp.spin_tol = spin_tol;
    }

    // setup, spin-up (first year pair, lock-step rounds), hand-over of the leftovers to the pool
    int enqueue_spin(int64_t t) {
        const int64_t c0 = t * tile, nct = cells_of(t);
        TileEv& e = ev[(size_t)t];
        RunParams& rp = rps[(size_t)t];
        cudaStream_t R = run_stream(t);
        CU(cudaStreamWaitEvent(R, ahead ? e.h2da : e.h2d1, 0));
        if (t >= kSlots && !(in_dev && out_dev) && !ahead) {
            // slot t % kSlots (forcing, work set, output staging) was last used by tile t - kSlots
            CU(cudaStreamWaitEvent(R, ev[(size_t)(t - kSlots)].run, 0));
            if (!out_dev) CU(cudaStreamWaitEvent(R, ev[(size_t)(t - kSlots)].d2h1, 0));
        }
        CU(cudaEventRecord(e.k0, R));
        k_tile_begin<<<1, 1, 0, R>>>(rp.ctl, (int)nct);
        k_cell_setup<<<(unsigned)((nct + 127) / 128), 128, 0, R>>>(sps[(size_t)t]);
        CU(cudaGetLastError());
        k_snow_threshold<FT><<<(unsigned)((nct + 255) / 256), 256, 0, R>>>((const FT*)rp.tc, rp.tpitch, rp.n_days, (int)nct, rp.cc,
                                                                            rp.cpitch, rp.diag, rp.dpitch, rp.w.frost);
        CU(cudaGetLastError());
        launches += 3;
        CU(cudaEventRecord(e.kf0, R));
        if (opts.skip_spinup) {
            // resume: run_all starts from the caller's state (SPLASH.cpp:1833-1835 wn_last ... nds_last)
            CU(cudaMemcpy2DAsync(rp.w.st, (size_t)pitch * 8, opts.state_init + c0, (size_t)spitch * 8, (size_t)nct * 8, 5,
                                 cudaMemcpyHostToDevice, R));
            CU(cudaMemcpyAsync(rp.w.w1, opts.state_init + 5 * spitch + c0, (size_t)nct * 8, cudaMemcpyHostToDevice, R));
            CU(cudaMemcpyAsync(rp.w.snap, opts.state_init + 6 * spitch + c0, (size_t)nct * 8, cudaMemcpyHostToDevice, R));
            k_init_resume<<<(unsigned)((nct + 255) / 256), 256, 0, R>>>(rp.w, rp.cc, rp.cpitch, rp.diag, rp.dpitch, (int)nct);
            CU(cudaGetLastError());
            ++launches;
            CU(cudaEventRecord(e.kf1, R));
            CU(cudaEventRecord(e.kr1, R));
            CU(cudaEventRecord(e.exported, R));
            return SPLASH_OK;
        }
        // ---- aridity year + pass 0 for every cell ---------------------------------------------------------
        k_spin_first<FT><<<ugrid_for(nct), kUThreads, kSmemUniform, R>>>(rp);
        CU(cudaGetLastError());
        ++launches;
        CU(cudaEventRecord(e.kf1, R));
        // ---- lock-step year passes; the list sizes stay on the device (grids are sized for the worst case,
        //      surplus CTAs exit at once) --------------------------------------------------------------------
        // a round can keep at most the cells of the previous one: after a few rounds a fraction of the grid suffices
        const int n_rounds = ctx->n_rounds;
        for (int r = 0; r < n_rounds; ++r) {
            RunParams q = rp;
            q.round = r;
            k_spin_check<FT><<<grid_for(nct), kThreads, kSmemSpin, R>>>(q);
            k_spin_rest<FT><<<ugrid_for(nct), kUThreads, kSmemUniform, R>>>(q);
            CU(cudaGetLastError());
            launches += 2;
        }
        CU(cudaEventRecord(e.kr1, R));
        // ---- leftovers: into the pool (their own streams), or finished here if the pool is full -----------
        k_pool_reserve<<<1, 1, 0, R>>>(rp.ctl, n_rounds, pool.count, pool.cap);
        k_pool_export<FT><<<(unsigned)(ctx->sm_count * 4), 256, 0, R>>>(rp, pool, n_rounds, (long long)c0, ahead ? 1 : 3);
        CU(cudaGetLastError());
        launches += 2;
        CU(cudaEventRecord(e.exported, R));
        {
            cudaStream_t Q = ctx->s_pool[t % kPoolStreams];
            CU(cudaStreamWaitEvent(Q, e.exported, 0));
            RunParams& pp = pps[(size_t)t];
            pp = rp;
            pp.sw = pp.sw1 = pool.f[0];
            pp.tc = pool.f[1];
            pp.pn = pp.pn1 = pool.f[2];
            pp.fpitch = pp.tpitch = pp.f1pitch = pool.cap;
            pp.cc = pool.cc;
            pp.cpitch = pool.cap;
            pp.w = pool.w;
            for (int k = 0; k < 9; ++k) pp.out[k] = pool.out[k];
            pp.opitch = pool.cap;
            pp.diag = pool.diag;
            pp.dpitch = pool.cap;
            pp.n_cells = (int)pool.cap;
            pp.q_head = &rp.ctl->pool_head;
            pp.q_end = &rp.ctl->pool_end;
            pp.q_list = nullptr;
            // forcing half of the cyclic year once, the spin-up chain on the state half, then the daily integration
            k_pool_table<FT><<<(unsigned)(ctx->sm_count * 2), 128, 0, Q>>>(pp, pool);
            // stage budgets: a short first look, a long second one, then the cells that may run to the pass limit
            const bool small_call = ctx->pool_auto && (double)nc * (double)nd < kPoolSmallCallCellDays;
            const int s1 = small_call ? kPoolStage1Small : ctx->pool_stage1, s2 = small_call ? kPoolStage2Small : ctx->pool_stage2;
            const int lanes3 = small_call ? kPoolLastLanesSmall : ctx->pool_last_lanes, ctas3 = small_call ? kPoolLastCtasSmall : ctx->pool_last_ctas;
            const int b1 = s1 > 0 ? s1 : (1 << 30);
            k_pool_spin<false><<<(unsigned)(ctx->sm_count * 2), kListThreads, kSmemList, Q>>>(pp, pool, 1, b1, 32, 0, 0);
            CU(cudaEventRecord(e.ps1, Q));
            k_pool_spin<false><<<(unsigned)(ctx->sm_count * 2), kListThreads, kSmemList, Q>>>(pp, pool, 2, s2, 32, 0, 0);
            if (ctx->chain_fast) {  // probe pass, then the fast route and the guarded route side by side (see k_pool_spin)
                const int ctas_b = std::max(8, ctas3 / 4);
                const size_t smem3 = std::max<size_t>((size_t)ctx->pool_excl_smem, kSmemList + kSmemChainRing);
                k_pool_spin<true><<<(unsigned)ctas3, kListThreads, smem3, Q>>>(pp, pool, kStageProbe, 1, lanes3, 0, 0);
                k_pool_spin<true><<<(unsigned)(ctas3 + ctas_b), kListThreads, smem3, Q>>>(pp, pool, kStageFinal, 1 << 30, lanes3, ctas3, kPoolDeclinerLanes);
                ++launches;
            } else {
                k_pool_spin<false><<<(unsigned)ctas3, kListThreads, ctx->pool_excl_smem, Q>>>(pp, pool, 3, 1 << 30, lanes3, 0, 0);
            }
            CU(cudaEventRecord(e.ps2, Q));
            CU(cudaGetLastError());
            launches += 4;
        }
        return SPLASH_OK;
    }

    // daily integration of every cell of the tile that finished its spin-up, then the tile's downloads
    int enqueue_main(int64_t t) {
        const int64_t c0 = t * tile, nct = cells_of(t);
        TileEv& e = ev[(size_t)t];
        RunParams& rp = rps[(size_t)t];
        cudaStream_t R = run_stream(t), D = ctx->s_d2h;
        if (ahead) {
            // the tile's whole sw / pn series has to be in its slot, and the slot's previous outputs downloaded
            CU(cudaStreamWaitEvent(R, e.h2d1, 0));
            if (t >= kSlots && !out_dev) CU(cudaStreamWaitEvent(R, ev[(size_t)(t - kSlots)].d2h1, 0));
        }
        if (!opts.skip_spinup) {
            const int n_rounds = ctx->n_rounds;
            // ---- the stragglers' day loop needs their whole forcing columns in the pool -----------------------
            if (ahead) {
                k_pool_export<FT><<<(unsigned)(ctx->sm_count * 4), 256, 0, R>>>(rp, pool, n_rounds, (long long)c0, 2);
                CU(cudaGetLastError());
                ++launches;
            }
            CU(cudaEventRecord(e.exported_b, R));
            cudaStream_t Q = ctx->s_pool[t % kPoolStreams];
            CU(cudaStreamWaitEvent(Q, e.exported_b, 0));
            launch_list<FT>(pps[(size_t)t], monthly, ctx->sm_count * 2, Q);
            CU(cudaEventRecord(e.pm, Q));
            CU(cudaGetLastError());
            ++launches;
            // ---- leftovers that did not fit the pool: rest of their spin-up and their day loop, in the tile ---
            RunParams tp = rp;
            tp.q_head = &rp.ctl->tail_head;
            tp.q_end = &rp.ctl->tail_end;
            tp.q_list = n_rounds ? rp.lists[n_rounds & 1] : nullptr;
            launch_list<FT>(tp, monthly, ctx->sm_count * 2, R);
            CU(cudaGetLastError());
            ++launches;
        }
        if (ctx->regime_sort && nd > 0) {
            // the finished cells in regime order (exported stragglers and, after a resume, nothing are left out)
            CU(cudaMemsetAsync(&rp.ctl->n_ready, 0, sizeof(unsigned long long) * (1 + kRegimeKeys), R));
            k_regime_count<<<(unsigned)((nct + 255) / 256), 256, 0, R>>>(rp);
            k_regime_scan<<<1, 1, 0, R>>>(rp.ctl);
            k_regime_scatter<<<(unsigned)((nct + 255) / 256), 256, 0, R>>>(rp);
            CU(cudaGetLastError());
            launches += 3;
            rp.order = rp.order_w;
        }
        CU(cudaEventRecord(e.kb0, R));
        launch_bulk<FT>(rp, monthly, R);
        CU(cudaGetLastError());
        CU(cudaEventRecord(e.kb1, R));
        k_finish_diag<<<(unsigned)((nct + 255) / 256), 256, 0, R>>>(rp.w.passes, rp.diag, rp.dpitch, (int)nct);
        CU(cudaGetLastError());
        launches += 2;
        CU(cudaEventRecord(e.run, R));

        CU(cudaStreamWaitEvent(D, e.run, 0));
        CU(cudaEventRecord(e.d2h0, D));
        const cudaMemcpyKind okind = out_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
        if (!out_dev) {
            for (int k = 0; k < 9; ++k) {
                if (!out_ptr[k] || n_out == 0) continue;
                CU(cudaMemcpy2DAsync(out_ptr[k] + c0, (size_t)ostride * 8, rp.out[k], (size_t)pitch * 8, (size_t)nct * 8, (size_t)n_out,
                                     cudaMemcpyDeviceToHost, D));
                ctx->stats.d2h_bytes += (int64_t)nct * n_out * 8;
            }
        }
        if (out->state_final) {
            CU(cudaMemcpy2DAsync(out->state_final + c0, (size_t)xpitch * 8, rp.w.st, (size_t)pitch * 8, (size_t)nct * 8, 5, okind, D));
            CU(cudaMemcpyAsync(out->state_final + 5 * xpitch + c0, rp.cc + (size_t)C_CELLOUT * pitch, (size_t)nct * 8, okind, D));
            CU(cudaMemcpyAsync(out->state_final + 6 * xpitch + c0, rp.cc + (size_t)C_TT * pitch, (size_t)nct * 8, okind, D));
            if (!out_dev) ctx->stats.d2h_bytes += (int64_t)nct * SPLASH_NSTATE * 8;
        }
        if (out->cell_diag) {
            CU(cudaMemcpy2DAsync(out->cell_diag + c0, (size_t)xpitch * 8, rp.diag, (size_t)pitch * 8, (size_t)nct * 8, SPLASH_NDIAG, okind, D));
            if (!out_dev) ctx->stats.d2h_bytes += (int64_t)nct * SPLASH_NDIAG * 8;
        }
        CU(cudaEventRecord(e.d2h1, D));
        return SPLASH_OK;
    }

    // results of the pool's cells into the caller's arrays (after everything else has drained)
    int scatter_pool(int64_t n_pool) {
        if (n_pool <= 0) return SPLASH_OK;
        if (out_dev) {
            Out9 o9;
            for (int k = 0; k < 9; ++k) o9.p[k] = out_ptr[k];
            k_pool_scatter<<<(unsigned)(ctx->sm_count * 2), 256, 0, ctx->s_d2h>>>(pool, (long long)n_pool, (long long)n_out, o9,
                                                                                 (long long)ostride, out->state_final, out->cell_diag,
                                                                                 (long long)xpitch);
            CU(cudaGetLastError());
            ++launches;
            CU(cudaStreamSynchronize(ctx->s_d2h));
            return SPLASH_OK;
        }
        std::vector<long long> cell((size_t)n_pool);
        CU(cudaMemcpy(cell.data(), pool.cell, (size_t)n_pool * 8, cudaMemcpyDeviceToHost));
        std::vector<double> buf((size_t)std::max<int64_t>(n_out, SPLASH_NDIAG) * (size_t)n_pool);
        for (int k = 0; k < 9; ++k) {
            if (!out_ptr[k] || n_out == 0) continue;
            CU(cudaMemcpy2D(buf.data(), (size_t)n_pool * 8, pool.out[k], (size_t)pool.cap * 8, (size_t)n_pool * 8, (size_t)n_out,
                            cudaMemcpyDeviceToHost));
            ctx->stats.d2h_bytes += n_pool * n_out * 8;
            // rows are independent: a few host threads hide the cache misses of the scattered stores
            const int n_thr = (int)std::max<int64_t>(1, std::min<int64_t>({8, (int64_t)std::thread::hardware_concurrency(), n_out}));
            auto rows = [&](int64_t r0, int64_t r1) {
                for (int64_t r = r0; r < r1; ++r) {
                    double* dst = out_ptr[k] + r * ostride;
                    const double* src = buf.data() + r * n_pool;
                    for (int64_t j = 0; j < n_pool; ++j) dst[cell[(size_t)j]] = src[j];
                }
            };
            if (n_thr == 1 || n_pool * n_out < (1 << 16)) {
                rows(0, n_out);
            } else {
                std::vector<std::thread> th;
                for (int i = 0; i < n_thr; ++i) th.emplace_back(rows, n_out * i / n_thr, n_out * (i + 1) / n_thr);
                for (auto& t : th) t.join();
            }
        }
        if (out->state_final) {
            CU(cudaMemcpy2D(buf.data(), (size_t)n_pool * 8, pool.w.st, (size_t)pool.cap * 8, (size_t)n_pool * 8, 5, cudaMemcpyDeviceToHost));
            for (int k = 0; k < 5; ++k)
                for (int64_t j = 0; j < n_pool; ++j) out->state_final[(int64_t)k * xpitch + cell[(size_t)j]] = buf[(size_t)(k * n_pool + j)];
            CU(cudaMemcpy(buf.data(), pool.cc + (size_t)C_CELLOUT * pool.cap, (size_t)n_pool * 8, cudaMemcpyDeviceToHost));
            for (int64_t j = 0; j < n_pool; ++j) out->state_final[5 * xpitch + cell[(size_t)j]] = buf[(size_t)j];
            CU(cudaMemcpy(buf.data(), pool.cc + (size_t)C_TT * pool.cap, (size_t)n_pool * 8, cudaMemcpyDeviceToHost));
            for (int64_t j = 0; j < n_pool; ++j) out->state_final[6 * xpitch + cell[(size_t)j]] = buf[(size_t)j];
        }
        if (out->cell_diag) {
            CU(cudaMemcpy2D(buf.data(), (size_t)n_pool * 8, pool.diag, (size_t)pool.cap * 8, (size_t)n_pool * 8, SPLASH_NDIAG,
                            cudaMemcpyDeviceToHost));
            const int rows[2] = {SPLASH_DIAG_SPIN_PASSES, SPLASH_DIAG_SNOWFALL_DAYS};
            for (int r : rows)
                for (int64_t j = 0; j < n_pool; ++j) out->cell_diag[(int64_t)r * xpitch + cell[(size_t)j]] = buf[(size_t)(r * n_pool + j)];
        }
        return SPLASH_OK;
    }

    int run() {
        if (int rc = plan()) return rc;
        if (int rc = allocate()) return rc;
        CU(cudaEventRecord(ev_begin, ctx->s_h2d));
        for (auto s : ctx->s_run) CU(cudaStreamWaitEvent(s, ev_begin, 0));  // (idle streams included: harmless)
        for (int64_t t = 0; t < n_tiles; ++t) setup_params(t);
        if (in_dev && out_dev && ctx->two_pass) {
            // resident data: every tile's spin-up first, so that the stragglers (up to 1000 sequential year
            // passes) start as early as possible and run beside the daily integration of all tiles
            for (int64_t t = 0; t < n_tiles; ++t) {
                if (int rc = enqueue_h2d(t)) return rc;
                if (int rc = enqueue_spin(t)) return rc;
            }
            for (int64_t t = 0; t < n_tiles; ++t)
                if (int rc = enqueue_main(t)) return rc;
        } else if (ahead) {
            // host-fed: the spin-up data of every tile goes up first (40 % of the bytes of a 10-year call), all
            // tiles spin up while the rest of the forcing follows tile by tile through the slots
            for (int64_t t = 0; t < n_tiles; ++t)
                if (int rc = enqueue_h2d_ahead(t)) return rc;
            for (int64_t t = 0; t < n_tiles; ++t)
                if (int rc = enqueue_spin(t)) return rc;
            for (int64_t t = 0; t < n_tiles; ++t) {
                if (int rc = enqueue_h2d(t)) return rc;   // waits for the slot (tile t - kSlots enqueued below)
                if (int rc = enqueue_main(t)) return rc;
            }
        } else {
            for (int64_t t = 0; t < n_tiles; ++t) {
                if (int rc = enqueue_h2d(t)) return rc;
                if (int rc = enqueue_spin(t)) return rc;
                if (int rc = enqueue_main(t)) return rc;
            }
        }
        // ---- drain -------------------------------------------------------------------------------------------
        CU(cudaStreamSynchronize(ctx->s_h2d));
        for (auto s : ctx->s_run) CU(cudaStreamSynchronize(s));
        const auto t_pool0 = std::chrono::steady_clock::now();
        for (auto s : ctx->s_pool) CU(cudaStreamSynchronize(s));
        const double pool_wait_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_pool0).count();
        CU(cudaStreamSynchronize(ctx->s_d2h));
        unsigned long long pool_count = 0;
        CU(cudaMemcpy(&pool_count, pool.count, 8, cudaMemcpyDeviceToHost));
        const int64_t n_pool = (int64_t)std::min<unsigned long long>(pool_count, (unsigned long long)pool.cap);
        const auto t_sc0 = std::chrono::steady_clock::now();
        if (int rc = scatter_pool(n_pool)) return rc;
        ctx->stats.scatter_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_sc0).count();
        CU(cudaEventRecord(ev_end, ctx->s_d2h));
        CU(cudaEventSynchronize(ev_end));

#ifdef SPLASH_BOUNDS_CHECK
        {
            unsigned long long site = 0;
            CU(cudaMemcpyFromSymbol(&site, g_bounds_err, sizeof(site)));
            if (site) return fail(ctx, SPLASH_ERR_CUDA, "bounds check failed in a kernel (site %llu)", site);
        }
#endif
        // ---- accounting --------------------------------------------------------------------------------------
        std::vector<TileCtl> h_ctl((size_t)n_tiles);
        CU(cudaMemcpy(h_ctl.data(), ctx->ctl.p, sizeof(TileCtl) * (size_t)n_tiles, cudaMemcpyDeviceToHost));
        splash_stats& st = ctx->stats;
        for (int64_t t = 0; t < n_tiles; ++t) {
            const TileCtl& c = h_ctl[(size_t)t];
            st.spin_cell_days += (int64_t)c.spin_days;
            st.unconverged_cells += (int64_t)c.unconverged;
            st.cycle_cells += (int64_t)c.cycles;
            st.pool_cells += (int64_t)(c.pool_end - c.pool_base);
            st.pool_overflow_cells += (int64_t)c.tail_end - (int64_t)(c.pool_end - c.pool_base);
            st.pool_max_passes = std::max<int64_t>(st.pool_max_passes, (int64_t)c.max_chain);
            const TileEv& e = ev[(size_t)t];
            float ms = 0;
            if (ahead) {
                if (cudaEventElapsedTime(&ms, e.h2d0, e.h2da) == cudaSuccess) st.h2d_ms += ms;
                if (cudaEventElapsedTime(&ms, e.h2db, e.h2d1) == cudaSuccess) st.h2d_ms += ms;
            } else if (cudaEventElapsedTime(&ms, e.h2d0, e.h2d1) == cudaSuccess) {
                st.h2d_ms += ms;
            }
            if (cudaEventElapsedTime(&ms, e.k0, e.kf0) == cudaSuccess) st.setup_ms += ms;
            if (cudaEventElapsedTime(&ms, e.kf0, e.kf1) == cudaSuccess) st.first_ms += ms;
            if (cudaEventElapsedTime(&ms, e.kf1, e.kr1) == cudaSuccess) st.rounds_ms += ms;
            if (cudaEventElapsedTime(&ms, e.kb0, e.kb1) == cudaSuccess) st.bulk_ms += ms;
            if (cudaEventElapsedTime(&ms, e.d2h0, e.d2h1) == cudaSuccess) st.d2h_ms += ms;
        }
        if (getenv("SPLASH_TRACE")) {  // per-tile timeline, ms since the first enqueue
            for (int64_t t = 0; t < n_tiles; ++t) {
                const TileEv& e = ev[(size_t)t];
                const TileCtl& c = h_ctl[(size_t)t];
                auto at = [&](cudaEvent_t x) {
                    float m = -1;
                    return cudaEventElapsedTime(&m, ev_begin, x) == cudaSuccess ? (double)m : -1.0;
                };
                fprintf(stderr,
                        "[splash trace] tile %2lld: start %7.1f first %7.1f..%7.1f rounds_end %7.1f bulk %7.1f..%7.1f | pool n=%llu last_stage=%llu declining=%llu "
                        "stage1_end %7.1f stage2_end %7.1f main_end %7.1f max_chain %llu\n",
                        (long long)t, at(e.k0), at(e.kf0), at(e.kf1), at(e.kr1), at(e.kb0), at(e.kb1), c.pool_end - c.pool_base, c.hard_n[2], c.decl_n,
                        opts.skip_spinup ? -1.0 : at(e.ps1), opts.skip_spinup ? -1.0 : at(e.ps2), opts.skip_spinup ? -1.0 : at(e.pm), c.max_chain);
                // the cells (indices in the caller's arrays) that declined the branch-light day step: tools/decliners.py looks at them
                for (unsigned long long k = 0; pool.cap > 0 && k < c.decl_n && k < 16; ++k) {
                    int pc = -1;
                    long long cell = -1;
                    int passes = -1;
                    if (cudaMemcpy(&pc, pool.hard[kStageProbe & 1] + (c.pool_end - 1 - k), sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess && pc >= 0 &&
                        pc < pool.cap && cudaMemcpy(&cell, pool.cell + pc, sizeof(long long), cudaMemcpyDeviceToHost) == cudaSuccess &&
                        cudaMemcpy(&passes, pool.w.passes + pc, sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess)
                        fprintf(stderr, "[splash trace]   declining cell %lld (tile %lld) passes %d\n", cell, (long long)t, passes);
                }
            }
        }
        float ms = 0;
        for (int64_t t0 = 0; t0 < std::min<int64_t>(kRunStreams, n_tiles); ++t0)
            for (int64_t t = 0; t < n_tiles; ++t)
                if (cudaEventElapsedTime(&ms, ev[(size_t)t0].kb0, ev[(size_t)t].kb1) == cudaSuccess)
                    st.bulk_span_ms = std::max(st.bulk_span_ms, (double)ms);
        if (cudaEventElapsedTime(&ms, ev_begin, ev_end) == cudaSuccess) st.gpu_ms = ms;
        st.pool_wait_ms = pool_wait_ms;
        st.main_cell_days = nc * nd;
        st.kernel_launches = launches;
        st.n_tiles = n_tiles;
        st.tile_cells = tile;
        return SPLASH_OK;
    }
};

}  // namespace

extern "C" {

static int multi_grid_run(splash_ctx* ctx, const splash_grid_in* in, const splash_opts* opts_in, splash_grid_out* out);

int splash_grid_run(splash_ctx* ctx, const splash_grid_in* in, const splash_opts* opts_in, splash_grid_out* out) {
    if (!ctx) return SPLASH_ERR_BAD_ARG;
    if (ctx->multi) return multi_grid_run(ctx, in, opts_in, out);
    const auto t_begin = std::chrono::steady_clock::now();
    ctx->err.clear();
    ctx->stats = splash_stats{};
    if (!in || !out) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_grid_run: NULL in/out");
    splash_opts opts{};
    if (opts_in) opts = *opts_in;
    const int64_t nc = in->n_cells, nd = in->n_days;
    if (nc < 0 || nd < 0) return fail(ctx, SPLASH_ERR_BAD_ARG, "negative n_cells/n_days");
    if (nd > (1 << 30) || nc > (int64_t)1 << 40) return fail(ctx, SPLASH_ERR_BAD_ARG, "n_days/n_cells too large");
    if (in->au_layers != 1 && in->au_layers != 3) return fail(ctx, SPLASH_ERR_BAD_ARG, "au_layers must be 1 or 3");
    if (in->forcing_dtype != SPLASH_F64 && in->forcing_dtype != SPLASH_F32)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "forcing_dtype must be SPLASH_F64 or SPLASH_F32");
    if ((in->mem_kind != SPLASH_MEM_HOST && in->mem_kind != SPLASH_MEM_DEVICE) ||
        (out->mem_kind != SPLASH_MEM_HOST && out->mem_kind != SPLASH_MEM_DEVICE))
        return fail(ctx, SPLASH_ERR_BAD_ARG, "mem_kind must be SPLASH_MEM_HOST or SPLASH_MEM_DEVICE");
    const int64_t istride = in->cell_stride ? in->cell_stride : nc;
    const int64_t ostride = out->cell_stride ? out->cell_stride : nc;
    if (istride < nc || ostride < nc) return fail(ctx, SPLASH_ERR_BAD_ARG, "cell_stride smaller than n_cells");
    const int64_t apitch = in->attr_stride ? in->attr_stride : nc;
    const int64_t xpitch = out->aux_stride ? out->aux_stride : nc;
    const int64_t spitch = opts.state_stride ? opts.state_stride : nc;
    if (apitch < nc || xpitch < nc || spitch < nc) return fail(ctx, SPLASH_ERR_BAD_ARG, "attr_stride/aux_stride/state_stride smaller than n_cells");
    if (nc > 0 && (!in->lat || !in->elev || !in->slop || !in->asp || !in->resolution || !in->soil || !in->au))
        return fail(ctx, SPLASH_ERR_BAD_ARG, "NULL per-cell input array");
    if (nd > 0 && (!in->year || !in->doy || !in->month)) return fail(ctx, SPLASH_ERR_BAD_ARG, "NULL time array (year/doy/month)");
    if (nc > 0 && nd > 0 && (!in->sw_in || !in->tc || !in->pn)) return fail(ctx, SPLASH_ERR_BAD_ARG, "NULL forcing array");
    for (int64_t d = 0; d < nd; ++d)
        if (in->month[d] < 1 || in->month[d] > 12 || in->doy[d] < 1 || in->doy[d] > 366)
            return fail(ctx, SPLASH_ERR_BAD_ARG, "month/doy out of range at day %lld", (long long)d);
    const int64_t n_months = splash_count_months(in->year, in->month, nd);
    const int64_t n_out = opts.monthly_out ? n_months : nd;
    if (out->n_out != n_out)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "out->n_out is %lld, expected %lld", (long long)out->n_out, (long long)n_out);
    if (opts.skip_spinup && !opts.state_init) return fail(ctx, SPLASH_ERR_BAD_ARG, "skip_spinup needs state_init");
    if (nc == 0) return SPLASH_OK;

    CU(cudaSetDevice(ctx->device));

    // ---- day tables ---------------------------------------------------------------------------------
    std::vector<DayTab> h_tab, h_spin;
    build_day_tables(in->year, in->doy, in->month, nd, kSpinYear, h_tab, h_spin);
    if (!ctx->month_tab_set) {
        const MonthTab mt = build_month_table();
        CU(cudaMemcpyToSymbol(c_month_tab, &mt, sizeof(mt)));
        ctx->month_tab_set = true;
    }
    if (int rc = ensure(ctx, ctx->dtab, sizeof(DayTab) * h_tab.size())) return rc;
    if (int rc = ensure(ctx, ctx->dtab_spin, sizeof(DayTab) * kSpinYear)) return rc;
    CU(cudaMemcpyAsync(ctx->dtab.p, h_tab.data(), sizeof(DayTab) * h_tab.size(), cudaMemcpyHostToDevice, ctx->s_h2d));
    CU(cudaMemcpyAsync(ctx->dtab_spin.p, h_spin.data(), sizeof(DayTab) * kSpinYear, cudaMemcpyHostToDevice, ctx->s_h2d));
    CU(cudaStreamSynchronize(ctx->s_h2d));

    auto fill = [&](auto& job) {
        job.ctx = ctx;
        job.in = in;
        job.out = out;
        job.opts = opts;
        job.nc = nc;
        job.nd = nd;
        job.n_out = n_out;
        job.istride = istride;
        job.ostride = ostride;
        job.apitch = apitch;
        job.xpitch = xpitch;
        job.spitch = spitch;
        job.in_dev = (in->mem_kind == SPLASH_MEM_DEVICE);
        job.out_dev = (out->mem_kind == SPLASH_MEM_DEVICE);
        job.monthly = opts.monthly_out != 0;
        job.max_spin = opts.max_spin > 0 ? opts.max_spin : 1000;
        job.spin_tol = opts.spin_tol_mm > 0 ? opts.spin_tol_mm : 1.0;
        double* const op[9] = {out->wn, out->ro, out->pet, out->aet, out->snow, out->cond, out->bflow, out->netr, out->sm_lim};
        for (int k = 0; k < 9; ++k) {
            job.out_ptr[k] = op[k];
            job.n_out_layers += op[k] ? 1 : 0;
        }
    };
    int rc;
    if (in->forcing_dtype == SPLASH_F32) {
        GridJob<float> job{};
        fill(job);
        rc = job.run();
        if (rc != SPLASH_OK) cudaDeviceSynchronize();
        job.release();
    } else {
        GridJob<double> job{};
        fill(job);
        rc = job.run();
        if (rc != SPLASH_OK) cudaDeviceSynchronize();
        job.release();
    }
    if (rc != SPLASH_OK) return rc;
    ctx->stats.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    return SPLASH_OK;
}

int splash_point_run(splash_ctx* ctx, int64_t n_days, const int32_t* year, const int32_t* doy, const int32_t* month,
                     const double* sw_in, const double* tc, const double* pn, double lat, double elev, double slop,
                     double asp, const double* soil_data, const double* au, int32_t au_len, double resolution,
                     const splash_opts* opts, splash_grid_out* out) {
    if (!ctx) return SPLASH_ERR_BAD_ARG;
    if (!soil_data || !au || !out) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_point_run: NULL soil_data/au/out");
    splash_grid_in in{};
    in.n_cells = 1;
    in.n_days = n_days;
    in.cell_stride = 1;
    in.year = year;
    in.doy = doy;
    in.month = month;
    in.sw_in = sw_in;
    in.tc = tc;
    in.pn = pn;
    in.lat = &lat;
    in.elev = &elev;
    in.slop = &slop;
    in.asp = &asp;
    in.resolution = &resolution;
    in.soil = soil_data;  // 6 layers of one cell: layer-major with n_cells == 1 is the plain vector
    in.au = au;
    in.au_layers = au_len;
    in.mem_kind = SPLASH_MEM_HOST;
    in.forcing_dtype = SPLASH_F64;
    splash_grid_out o = *out;
    o.cell_stride = 1;
    o.mem_kind = SPLASH_MEM_HOST;
    return splash_grid_run(ctx, &in, opts, &o);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Block scheduler (splash_cluster_*): the reference's sendCall / recvOneData loop over its workers
// (R/splash.grid.R:312-314, 359-400).  Lanes are single-GPU contexts with a worker thread each; blocks
// wait in one FIFO and go to whichever lane is free next, as the reference's blocks go to whichever
// worker has returned.  Cells are independent: lanes share nothing but the caller's (disjoint) arrays.
// ---------------------------------------------------------------------------------------------
namespace {

struct ClusterJob {
    int64_t ticket = 0;
    splash_grid_in in{};
    splash_opts opts{};
    splash_grid_out out{};
    int rc = SPLASH_OK;
    splash_stats stats{};
    std::string err;
    bool done = false;
};

}  // namespace

struct splash_cluster {
    std::vector<splash_ctx*> lanes;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::deque<ClusterJob*> fifo;
    std::map<int64_t, ClusterJob*> jobs;  // submitted and not yet waited for
    int64_t next_ticket = 1;
    bool stop = false;
    std::string err;
    int n_devices = 0;
};

namespace {

void cluster_worker(splash_cluster* cl, int lane) {
    splash_ctx* ctx = cl->lanes[(size_t)lane];
    for (;;) {
        ClusterJob* job = nullptr;
        {
            std::unique_lock<std::mutex> lk(cl->mu);
            cl->cv_work.wait(lk, [&] { return cl->stop || !cl->fifo.empty(); });
            if (cl->fifo.empty()) return;  // stop requested and nothing left to run
            job = cl->fifo.front();
            cl->fifo.pop_front();
        }
        const int rc = splash_grid_run(ctx, &job->in, &job->opts, &job->out);
        {
            std::lock_guard<std::mutex> lk(cl->mu);
            job->rc = rc;
            job->stats = ctx->stats;
            if (rc != SPLASH_OK) job->err = ctx->err;
            job->done = true;
        }
        cl->cv_done.notify_all();
    }
}

void add_stats(splash_stats& a, const splash_stats& b) {
    a.h2d_ms = std::max(a.h2d_ms, b.h2d_ms);
    a.setup_ms = std::max(a.setup_ms, b.setup_ms);
    a.first_ms = std::max(a.first_ms, b.first_ms);
    a.rounds_ms = std::max(a.rounds_ms, b.rounds_ms);
    a.bulk_ms = std::max(a.bulk_ms, b.bulk_ms);
    a.bulk_span_ms = std::max(a.bulk_span_ms, b.bulk_span_ms);
    a.d2h_ms = std::max(a.d2h_ms, b.d2h_ms);
    a.pool_wait_ms = std::max(a.pool_wait_ms, b.pool_wait_ms);
    a.scatter_ms = std::max(a.scatter_ms, b.scatter_ms);
    a.gpu_ms = std::max(a.gpu_ms, b.gpu_ms);
    a.h2d_bytes += b.h2d_bytes;
    a.d2h_bytes += b.d2h_bytes;
    a.spin_cell_days += b.spin_cell_days;
    a.main_cell_days += b.main_cell_days;
    a.kernel_launches += b.kernel_launches;
    a.unconverged_cells += b.unconverged_cells;
    a.cycle_cells += b.cycle_cells;
    a.n_tiles += b.n_tiles;
    a.tile_cells = std::max(a.tile_cells, b.tile_cells);
    a.pool_cells += b.pool_cells;
    a.pool_overflow_cells += b.pool_overflow_cells;
    a.pool_max_passes = std::max(a.pool_max_passes, b.pool_max_passes);
}

}  // namespace

extern "C" {

int splash_cluster_create(const int* devices, int n_devices, int lanes_per_device, splash_cluster** out) {
    if (!out) return fail(nullptr, SPLASH_ERR_BAD_ARG, "splash_cluster_create: out is NULL");
    *out = nullptr;
    if (!devices || n_devices <= 0 || n_devices > 64 || lanes_per_device <= 0 || lanes_per_device > 4)
        return fail(nullptr, SPLASH_ERR_BAD_ARG, "splash_cluster_create: need 1..64 devices and 1..4 lanes per device");
    for (int i = 0; i < n_devices; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return fail(nullptr, SPLASH_ERR_BAD_ARG, "splash_cluster_create: device %d listed twice", devices[i]);
    splash_cluster* cl = new splash_cluster();
    cl->n_devices = n_devices;
    // lanes of one device are interleaved with the other devices' (lane l -> device l % n): the first blocks of a
    // call spread over all GPUs
    for (int l = 0; l < n_devices * lanes_per_device; ++l) {
        splash_ctx* ctx = nullptr;
        const int rc = splash_ctx_create(devices[l % n_devices], &ctx);
        if (rc != SPLASH_OK) {
            for (auto* c : cl->lanes) splash_ctx_destroy(c);
            delete cl;
            return rc;  // (the message is splash_last_error(NULL))
        }
        ctx->mem_share = 1.0 / lanes_per_device;
        cl->lanes.push_back(ctx);
    }
    for (int l = 0; l < (int)cl->lanes.size(); ++l) cl->workers.emplace_back(cluster_worker, cl, l);
    *out = cl;
    return SPLASH_OK;
}

void splash_cluster_destroy(splash_cluster* cl) {
    if (!cl) return;
    {
        std::lock_guard<std::mutex> lk(cl->mu);
        cl->stop = true;
    }
    cl->cv_work.notify_all();
    for (auto& t : cl->workers) t.join();  // outstanding blocks are run to completion first
    for (auto& kv : cl->jobs) delete kv.second;
    for (auto* c : cl->lanes) splash_ctx_destroy(c);
    delete cl;
}

int splash_cluster_lanes(const splash_cluster* cl) { return cl ? (int)cl->lanes.size() : 0; }

const char* splash_cluster_last_error(const splash_cluster* cl) { return cl ? cl->err.c_str() : g_create_err.c_str(); }

int splash_cluster_submit(splash_cluster* cl, const splash_grid_in* in, const splash_opts* opts, const splash_grid_out* out,
                          int64_t* ticket) {
    if (!cl) return SPLASH_ERR_BAD_ARG;
    if (!in || !out || !ticket) {
        cl->err = "splash_cluster_submit: NULL in/out/ticket";
        return SPLASH_ERR_BAD_ARG;
    }
    if (in->mem_kind != SPLASH_MEM_HOST || out->mem_kind != SPLASH_MEM_HOST) {
        cl->err = "splash_cluster_submit: blocks of a cluster take HOST arrays (device arrays belong to one GPU: use splash_grid_run on that GPU's context)";
        return SPLASH_ERR_BAD_ARG;
    }
    ClusterJob* job = new ClusterJob();
    job->in = *in;
    if (opts) job->opts = *opts;
    job->out = *out;
    {
        std::lock_guard<std::mutex> lk(cl->mu);
        job->ticket = cl->next_ticket++;
        cl->jobs[job->ticket] = job;
        cl->fifo.push_back(job);
        *ticket = job->ticket;
    }
    cl->cv_work.notify_one();
    return SPLASH_OK;
}

int splash_cluster_wait(splash_cluster* cl, int64_t ticket, int64_t* done_ticket, splash_stats* stats) {
    if (!cl) return SPLASH_ERR_BAD_ARG;
    std::unique_lock<std::mutex> lk(cl->mu);
    ClusterJob* job = nullptr;
    if (ticket >= 0) {
        auto it = cl->jobs.find(ticket);
        if (it == cl->jobs.end()) {
            cl->err = "splash_cluster_wait: unknown ticket";
            return SPLASH_ERR_BAD_ARG;
        }
        job = it->second;
        cl->cv_done.wait(lk, [&] { return job->done; });
    } else {
        if (cl->jobs.empty()) {
            cl->err = "splash_cluster_wait: nothing outstanding";
            return SPLASH_ERR_BAD_ARG;
        }
        cl->cv_done.wait(lk, [&] {
            for (auto& kv : cl->jobs)
                if (kv.second->done) {
                    job = kv.second;
                    return true;
                }
            return false;
        });
    }
    cl->jobs.erase(job->ticket);
    if (done_ticket) *done_ticket = job->ticket;
    if (stats) *stats = job->stats;
    const int rc = job->rc;
    if (rc != SPLASH_OK) cl->err = job->err;
    delete job;
    return rc;
}

int splash_ctx_create_multi(const int* devices, int n_devices, splash_ctx** out_ctx) {
    if (!out_ctx) return fail(nullptr, SPLASH_ERR_BAD_ARG, "splash_ctx_create_multi: out_ctx is NULL");
    *out_ctx = nullptr;
    splash_cluster* cl = nullptr;
    // two lanes per GPU: the upload of a block overlaps the tail (straggler chain) of the previous one
    const int rc = splash_cluster_create(devices, n_devices, 2, &cl);
    if (rc != SPLASH_OK) return rc;
    splash_ctx* ctx = new splash_ctx();
    ctx->device = devices[0];
    ctx->multi = cl;
    *out_ctx = ctx;
    return SPLASH_OK;
}

int splash_ctx_device_count(const splash_ctx* ctx) { return !ctx ? 0 : (ctx->multi ? ctx->multi->n_devices : 1); }

// splash_grid_run on a multi-GPU context: the block is cut into row blocks (two per lane, like
// blockSize(minblocks = nodes * 2), R/splash.grid.R:264-268), which are scheduled over the lanes; every block
// reads and writes its own cell range of the caller's arrays through the strides of the structs.
static int multi_grid_run(splash_ctx* ctx, const splash_grid_in* in, const splash_opts* opts_in, splash_grid_out* out) {
    const auto t_begin = std::chrono::steady_clock::now();
    ctx->err.clear();
    ctx->stats = splash_stats{};
    if (!in || !out) return fail(ctx, SPLASH_ERR_BAD_ARG, "splash_grid_run: NULL in/out");
    if (in->mem_kind != SPLASH_MEM_HOST || out->mem_kind != SPLASH_MEM_HOST)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "a multi-GPU context takes HOST arrays (device arrays belong to one GPU)");
    splash_opts opts{};
    if (opts_in) opts = *opts_in;
    const int64_t nc = in->n_cells;
    if (nc < 0 || in->n_days < 0) return fail(ctx, SPLASH_ERR_BAD_ARG, "negative n_cells/n_days");
    if (in->forcing_dtype != SPLASH_F64 && in->forcing_dtype != SPLASH_F32)
        return fail(ctx, SPLASH_ERR_BAD_ARG, "forcing_dtype must be SPLASH_F64 or SPLASH_F32");
    splash_cluster* cl = ctx->multi;
    const int64_t fsz = in->forcing_dtype == SPLASH_F32 ? 4 : 8;
    const int64_t istride = in->cell_stride ? in->cell_stride : nc, ostride = out->cell_stride ? out->cell_stride : nc;
    const int64_t apitch = in->attr_stride ? in->attr_stride : nc, xpitch = out->aux_stride ? out->aux_stride : nc;
    const int64_t spitch = opts.state_stride ? opts.state_stride : nc;
    const int64_t lanes = (int64_t)cl->lanes.size();
    int64_t n_blocks = std::max<int64_t>(1, std::min<int64_t>(2 * lanes, (nc + 4095) / 4096));
    const int64_t bsz = std::max<int64_t>(1, round_up((nc + n_blocks - 1) / n_blocks, 1024));
    n_blocks = nc > 0 ? (nc + bsz - 1) / bsz : 1;
    int first_rc = SPLASH_OK;
    std::vector<int64_t> tickets;
    for (int64_t b = 0; b < n_blocks; ++b) {
        const int64_t b0 = b * bsz, n = std::max<int64_t>(0, std::min<int64_t>(bsz, nc - b0));
        splash_grid_in bi = *in;
        bi.n_cells = n;
        bi.cell_stride = istride;
        bi.attr_stride = apitch;
        auto adv = [&](const void* p, int64_t bytes) { return p ? (const void*)((const char*)p + bytes) : nullptr; };
        bi.sw_in = adv(in->sw_in, b0 * fsz);
        bi.tc = adv(in->tc, b0 * fsz);
        bi.pn = adv(in->pn, b0 * fsz);
        bi.lat = (const double*)adv(in->lat, b0 * 8);
        bi.elev = (const double*)adv(in->elev, b0 * 8);
        bi.slop = (const double*)adv(in->slop, b0 * 8);
        bi.asp = (const double*)adv(in->asp, b0 * 8);
        bi.resolution = (const double*)adv(in->resolution, b0 * 8);
        bi.soil = (const double*)adv(in->soil, b0 * 8);
        bi.au = (const double*)adv(in->au, b0 * 8);
        splash_grid_out bo = *out;
        bo.cell_stride = ostride;
        bo.aux_stride = xpitch;
        double** layers[11] = {&bo.wn, &bo.ro, &bo.pet, &bo.aet, &bo.snow, &bo.cond, &bo.bflow, &bo.netr, &bo.sm_lim, &bo.state_final, &bo.cell_diag};
        for (auto** q : layers)
            if (*q) *q += b0;
        splash_opts bopt = opts;
        bopt.state_stride = spitch;
        if (bopt.state_init) bopt.state_init += b0;
        int64_t tk = 0;
        const int rc = splash_cluster_submit(cl, &bi, &bopt, &bo, &tk);
        if (rc != SPLASH_OK) {
            first_rc = rc;
            ctx->err = cl->err;
            break;
        }
        tickets.push_back(tk);
    }
    for (int64_t tk : tickets) {
        splash_stats st{};
        const int rc = splash_cluster_wait(cl, tk, nullptr, &st);
        if (rc != SPLASH_OK && first_rc == SPLASH_OK) {
            first_rc = rc;
            ctx->err = cl->err;
        }
        if (rc == SPLASH_OK) add_stats(ctx->stats, st);
    }
    ctx->stats.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    return first_rc;
}

}  // extern "C"

static splash_ctx* first_lane(splash_ctx* ctx) { return ctx->multi->lanes[0]; }
