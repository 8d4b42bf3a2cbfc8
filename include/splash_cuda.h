/*
 * splash_cuda.h -- C ABI of libsplash_cuda, the B200 drop-in for the splash.grid()/splash.point()
 * hot path of dsval/rsplash (SPLASH v2.0).
 *
 * What each entry point replaces in the reference (paths relative to /root/reference):
 *
 *   splash_grid_run   <- the per-block worker body `clFun`: mapply(splash.point, sw_in=, tc=, pn=,
 *                        lat=, elev=, slop=, asp=, soil_data=, Au=, resolution=, MoreArgs=...)
 *                        R/splash.grid.R:277-308, and for every cell the three Rcpp-module calls it
 *                        makes, R/splash.point.R:92 (new(SPLASH,lat,elev)), :148/:152
 *                        ($spin_up, src/SPLASH.cpp:1594-1749) and :158-172 ($run_all,
 *                        src/SPLASH.cpp:1833-1916), plus the per-cell R arithmetic around them
 *                        (R/splash.point.R:96-131 soil_hydro / snow partition, :147-150 aridity
 *                        quirk, :182-214 sm_lim and monthly aggregation).
 *   splash_point_run  <- splash.point() itself, R/splash.point.R:29-225 (one cell).
 *   splash_ctx_create / _destroy <- raster::beginCluster / endCluster, R/splash.grid.R:32-39
 *                        (the PSOCK worker pool is what the GPU context stands in for).
 *   splash_last_error <- the only error path of the reference scheduler,
 *                        `stop('cluster error:')`, R/splash.grid.R:363-365.
 *
 * Layout contract: forcing matrices are DAY-MAJOR with cells contiguous, element (day d, cell c) at
 * [d * cell_stride + c].  This is exactly what raster::getValues(brick, row, nrows) hands to R
 * (column-major [cells x layers], R/splash.grid.R:278-280), so the R glue passes REAL() pointers
 * through unchanged.  Outputs use the same layout with n_out layers (= n_days, or the number of
 * calendar months when monthly_out is set), matching do.call(rbind, value[k,]) at
 * R/splash.grid.R:370-378.
 *
 * Ownership: the caller owns every buffer it passes in (inputs and outputs); the library keeps no
 * pointer after a call returns.  Device buffers, pinned staging memory and streams live in the
 * context.  A context is bound to one CUDA device and is not re-entrant: one call at a time.
 * There is no CPU fallback: without a usable CUDA device splash_ctx_create fails.
 *
 *   splash_cluster_*  <- the block scheduler of splash.grid over its N workers: sendCall(cl[[i]], clFun, i)
 *                        for the first `nodes` blocks, then recvOneData() / sendCall() of the next block until
 *                        all blocks are in (R/splash.grid.R:264-268, 312-314, 359-400).  A cluster is a set of
 *                        lanes (GPUs x calls in flight per GPU); submit == sendCall, wait == recvOneData.
 *   splash_ctx_create_multi <- the same scheduler driven by the library itself: splash_grid_run on such a
 *                        context cuts the call into row blocks (two per lane, like blockSize(minblocks =
 *                        nodes * 2), :264-268), runs them over all its GPUs and writes disjoint ranges of the
 *                        caller's arrays.  Cells are independent: there is no data-path collective and no NCCL.
 *
 * Process environment: a call keeps ~26 CUDA streams busy; with CUDA's default of 8 hardware work queues
 * streams share queues and kernels of one stream wait behind seconds-long kernels of another.  Export
 * CUDA_DEVICE_MAX_CONNECTIONS=32 before the process initialises CUDA (the library does not touch the
 * environment; rsplash_b200/__init__.py and the R shim in INTEGRATION.md do it for their processes).
 *
 * NaN inputs are data, not errors: they propagate exactly as in the reference (per-layer NA masks).
 */
#ifndef SPLASH_CUDA_H
#define SPLASH_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPLASH_ABI_VERSION 7
#define SPLASH_NSTATE 7

/* status codes */
enum {
    SPLASH_OK = 0,
    SPLASH_ERR_BAD_ARG = 1,  /* NULL/negative/inconsistent argument */
    SPLASH_ERR_CUDA = 2,     /* a CUDA runtime call failed (see splash_last_error) */
    SPLASH_ERR_NOMEM = 3,    /* device or pinned-host allocation failed */
    SPLASH_ERR_NO_DEVICE = 4 /* no usable sm_100 device: there is no CPU fallback */
};

/* where the caller's pointers live */
enum { SPLASH_MEM_HOST = 0, SPLASH_MEM_DEVICE = 1 };
/* element type of the three forcing matrices (everything else is always f64) */
enum { SPLASH_F64 = 0, SPLASH_F32 = 1 };

/* layers of splash_grid_out.cell_diag, [SPLASH_NDIAG * n_cells], layer-major */
enum {
    SPLASH_DIAG_SAT = 0,   /* soil_info[0]  saturation, mm            R/splash.point.R:98  */
    SPLASH_DIAG_WP = 1,    /* soil_info[1]  wilting point, mm         :99  */
    SPLASH_DIAG_FC = 2,    /* soil_info[2]  field capacity, mm        :100 */
    SPLASH_DIAG_KSAT = 3,  /* soil_info[3]  mm/h                      :355-363 */
    SPLASH_DIAG_LAMBDA = 4,/* soil_info[4]  1/B                       :104 */
    SPLASH_DIAG_DEPTH = 5, /* soil_info[5]  m                         :97  */
    SPLASH_DIAG_BUB = 6,   /* soil_info[6]  air-entry pressure, mm    :369-380 */
    SPLASH_DIAG_RES = 7,   /* soil_info[7]  residual, mm              :101 */
    SPLASH_DIAG_WMAX_R = 8,/* theta_c*depth*1000 used by sm_lim       :102,197 */
    SPLASH_DIAG_TT = 9,    /* snowfall threshold temperature Tt       :122 */
    SPLASH_DIAG_AI = 10,   /* sum(pet)/sum(P) of the first spin-up    :150 */
    SPLASH_DIAG_SPIN_PASSES = 11, /* year passes executed by the 2nd spin_up (1..1000) */
    SPLASH_DIAG_SNOW_DAYS = 12,   /* number of days with p_snow >= 0.5 (occurrence flags) */
    SPLASH_DIAG_SNOWFALL_DAYS = 13, /* number of days with snowfall > 0 */
    SPLASH_NDIAG = 14
};

typedef struct splash_ctx splash_ctx;

/* Inputs of one block of cells == the mapply() argument set of R/splash.grid.R:291-304. */
typedef struct splash_grid_in {
    int64_t n_cells;        /* cells in this block */
    int64_t n_days;         /* length of the daily series */
    int64_t cell_stride;    /* elements between consecutive days in sw_in/tc/pn; 0 means n_cells */
    const int32_t* year;    /* [n_days] calendar year of each day   (format(time_index,'%Y'), splash.point.R:59) */
    const int32_t* doy;     /* [n_days] day of year 1..366          (format(time_index,'%j'), :57) */
    const int32_t* month;   /* [n_days] month 1..12                 (format(time_index,'%m'), :547) */
    const void* sw_in;      /* [n_days*cell_stride] shortwave radiation, W m-2 */
    const void* tc;         /* [n_days*cell_stride] air temperature, deg C */
    const void* pn;         /* [n_days*cell_stride] precipitation, mm day-1 */
    const double* lat;      /* [n_cells] latitude, deg */
    const double* elev;     /* [n_cells] elevation, m */
    const double* slop;     /* [n_cells] slope, deg */
    const double* asp;      /* [n_cells] aspect, deg clockwise from north (library applies asp-180, splash.point.R:131) */
    const double* resolution; /* [n_cells] cell size, m */
    const double* soil;     /* [6*n_cells] layer-major: sand %, clay %, OM %, gravel %, bulk density g cm-3 (NaN = derive), depth m */
    const double* au;       /* [au_layers*n_cells] layer-major: upslope area m2 [, n cells draining in, n cells draining out] */
    int32_t au_layers;      /* 1 (length(Au)==1 branch, splash.point.R:106-110) or 3 (:111-115) */
    int32_t mem_kind;       /* SPLASH_MEM_HOST or SPLASH_MEM_DEVICE: applies to every pointer above except year/doy/month (always host) */
    int32_t forcing_dtype;  /* SPLASH_F64 (what R passes) or SPLASH_F32 (rasters are FLT4S on disk) */
    int32_t reserved;
    int64_t attr_stride;    /* elements between consecutive layers of soil and au; 0 means n_cells (a block that is a
                             * column range of a larger matrix passes the matrix's cell count) */
} splash_grid_in;

/* Outputs: the nine layers of R/splash.grid.R:449 (any pointer may be NULL = not wanted). */
typedef struct splash_grid_out {
    int64_t n_out;          /* layers the caller allocated: n_days, or splash_count_months() when monthly_out */
    int64_t cell_stride;    /* elements between consecutive layers; 0 means n_cells */
    double* wn;             /* soil water content, mm */
    double* ro;             /* runoff, mm */
    double* pet;            /* potential evapotranspiration, mm */
    double* aet;            /* actual evapotranspiration, mm */
    double* snow;           /* snow water equivalent, mm */
    double* cond;           /* condensation, mm */
    double* bflow;          /* lateral drainage, mm */
    double* netr;           /* daytime net radiation, MJ m-2 */
    double* sm_lim;         /* relative soil moisture limitation 0..1 */
    double* state_final;    /* optional [SPLASH_NSTATE*aux_stride] layer-major: wn, snow, qin, td, nd after the last day (the carried
                             * arguments of run_all, SPLASH.cpp:1833-1835), the value of soil_info[12] (the aridity index
                             * R/splash.point.R:150 writes there) and the snowfall threshold temperature Tt the series was
                             * partitioned with (a reduction over the WHOLE tc series, R/splash.point.R:120-122, which a
                             * later segment cannot recompute): everything a later call needs to continue the series */
    double* cell_diag;      /* optional [SPLASH_NDIAG*aux_stride] layer-major */
    int32_t mem_kind;       /* SPLASH_MEM_HOST or SPLASH_MEM_DEVICE for every pointer above */
    int32_t reserved;
    int64_t aux_stride;     /* elements between consecutive layers of state_final and cell_diag; 0 means n_cells */
} splash_grid_out;

typedef struct splash_opts {
    int32_t monthly_out;    /* sim.control$monthly_out, R/splash.grid.R:28,173-181: 1 = monthly mean(wn,snow,sm_lim)/sum(rest) */
    int32_t max_spin;       /* spin-up pass limit; 0 means the reference's 1000 (SPLASH.cpp:1697) */
    double spin_tol_mm;     /* spin-up tolerance on |delta wn(day 1)|; 0 means the reference's 1.0 mm */
    int64_t tile_cells;     /* cells per device tile; 0 = choose from free device memory */
    int32_t skip_spinup;    /* 1 = start run_all from state_init instead of spinning up (resume) */
    int32_t reserved;
    const double* state_init; /* [SPLASH_NSTATE*state_stride] layer-major, a previous call's state_final (host); used when
                               * skip_spinup.  The resumed segment is partitioned into rain and snow with the carried Tt
                               * (row 6), so that a series run in pieces equals the series run at once */
    int64_t state_stride;   /* elements between consecutive layers of state_init; 0 means n_cells */
} splash_opts;

/* Timing / accounting of the last call, filled by splash_last_stats (all times in milliseconds).
 * Tiles overlap on several streams, so the per-kernel-class times are sums of per-tile stream intervals
 * (they may add up to more than gpu_ms). */
typedef struct splash_stats {
    double h2d_ms;          /* host->device copies (sum over tiles, stream time) */
    double setup_ms;        /* cell-setup + snow-threshold kernels */
    double first_ms;        /* k_spin_first: aridity year + pass 0, 730 uniform days for every cell */
    double rounds_ms;       /* lock-step spin-up rounds (check + rest kernels) */
    double bulk_ms;         /* the bulk daily-integration kernels (CUDA events on their streams), summed over tiles */
    double bulk_span_ms;    /* first bulk kernel start to last bulk kernel end (== their run time when nothing else runs, e.g. a resume call) */
    double d2h_ms;          /* device->host copies */
    double pool_wait_ms;    /* host wait for the straggler pool after every tile stream had drained */
    double scatter_ms;      /* host time to move the pool's results into the caller's arrays */
    double gpu_ms;          /* first enqueue to last completion, CUDA events */
    double total_ms;        /* wall clock of the call */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    int64_t spin_cell_days; /* cell-days executed in spin-up (incl. check days) */
    int64_t main_cell_days; /* n_cells * n_days */
    int64_t kernel_launches;/* kernels of this library launched by the call */
    int64_t unconverged_cells; /* cells that hit the pass limit */
    int64_t cycle_cells;    /* cells whose spin-up was cut short by exact cycle detection */
    int64_t n_tiles;
    int64_t tile_cells;
    int64_t pool_cells;     /* cells that outlived the lock-step rounds and finished in the straggler pool */
    int64_t pool_overflow_cells; /* ... that did not fit the pool and finished inside their tile */
    int64_t pool_max_passes;/* longest chain of year passes one thread executed after the rounds */
} splash_stats;

int splash_abi_version(void);

/* Create a context on CUDA device `device` (ordinal).  Fails with SPLASH_ERR_NO_DEVICE when there
 * is no CUDA device: the library has no host implementation of the model. */
int splash_ctx_create(int device, splash_ctx** out_ctx);
/* A context over several GPUs of one host (SURVEY 8b).  splash_grid_run / splash_point_run on it accept HOST
 * arrays only; the call is cut into row blocks that are scheduled over the devices (see splash_cluster_*),
 * every block writes its own cell range of the caller's arrays.  n_devices == 1 is allowed. */
int splash_ctx_create_multi(const int* devices, int n_devices, splash_ctx** out_ctx);
void splash_ctx_destroy(splash_ctx* ctx);
/* Number of GPUs behind a context (1 for splash_ctx_create). */
int splash_ctx_device_count(const splash_ctx* ctx);

/* Message of the last failure on this context (or of the last failed splash_ctx_create when ctx is
 * NULL).  Never NULL; valid until the next call on the same context. */
const char* splash_last_error(const splash_ctx* ctx);

/* Number of calendar-month groups in the day axis = length(ztime.months); what n_out must be for
 * monthly_out (run-length of (year, month), like fastmatch::ctapply over format(time,'%Y-%m'),
 * R/splash.point.R:208-211).  Pure host arithmetic. */
int64_t splash_count_months(const int32_t* year, const int32_t* month, int64_t n_days);

/* Run a block of cells.  Returns SPLASH_OK or an error code; on error outputs are unspecified. */
int splash_grid_run(splash_ctx* ctx, const splash_grid_in* in, const splash_opts* opts, splash_grid_out* out);

/* Run one cell: splash.point(sw_in, tc, pn, lat, elev, slop, asp, soil_data, Au, resolution, ...).
 * soil_data[6] as in splash_grid_in.soil; au has au_len (1 or 3) elements.  out is a splash_grid_out
 * with n_cells = 1 semantics (host pointers). */
int splash_point_run(splash_ctx* ctx, int64_t n_days, const int32_t* year, const int32_t* doy,
                     const int32_t* month, const double* sw_in, const double* tc, const double* pn,
                     double lat, double elev, double slop, double asp, const double* soil_data,
                     const double* au, int32_t au_len, double resolution, const splash_opts* opts,
                     splash_grid_out* out);

/* Accounting of the last splash_grid_run / splash_point_run on this context (multi-GPU contexts: byte, cell-day
 * and launch counts summed over the blocks, times are the maximum over the lanes). */
int splash_last_stats(const splash_ctx* ctx, splash_stats* out);

/* ---- block scheduler: the reference's sendCall / recvOneData loop (R/splash.grid.R:312-314, 359-400) ----
 * A cluster owns `lanes_per_device` single-GPU contexts on each listed device, each with a worker thread.
 * submit() hands a block (HOST arrays, which must stay valid and untouched until the block has been waited
 * for) to the least-loaded lane and returns at once with a ticket; wait() blocks until the given ticket (or,
 * with ticket < 0, any outstanding one) has finished and returns its status, ticket and accounting.  With two
 * lanes per device the upload of block k+1 overlaps the tail of block k (its last stragglers' spin-up chain),
 * which a sequence of synchronous splash_grid_run calls leaves exposed. */
typedef struct splash_cluster splash_cluster;
int splash_cluster_create(const int* devices, int n_devices, int lanes_per_device, splash_cluster** out);
void splash_cluster_destroy(splash_cluster* cl);
int splash_cluster_lanes(const splash_cluster* cl);
int splash_cluster_submit(splash_cluster* cl, const splash_grid_in* in, const splash_opts* opts, const splash_grid_out* out,
                          int64_t* ticket);
/* Returns the block's status code (SPLASH_OK, ...) or SPLASH_ERR_BAD_ARG when nothing is outstanding.
 * done_ticket / stats may be NULL. */
int splash_cluster_wait(splash_cluster* cl, int64_t ticket, int64_t* done_ticket, splash_stats* stats);
const char* splash_cluster_last_error(const splash_cluster* cl);

/* ---- unSWC.grid: unsaturated-zone diagnostics of the simulated soil water (R/unsSWC.grid.R:14-141) ----
 * Replaces the four raster::overlay() passes of unSWC.grid (calc_thetai :96-103, calcwtd :112-121, UnsWater
 * :47-70 as called at :129, calc_Se :133-139) and its soil_hydro() call (:78); the netCDF writing stays in R.
 * All arrays layer-major with cells contiguous (raster::getValues layout); any output pointer may be NULL. */
typedef struct splash_unswc_in {
    int64_t n_cells;
    int64_t n_layers;       /* time steps (daily or monthly) of wn */
    int64_t cell_stride;    /* elements between consecutive layers of wn; 0 means n_cells */
    const double* soil;     /* [6*n_cells] layer-major as in splash_grid_in.soil (gravel is ignored: fgravel*0, :78) */
    const double* wn;       /* [n_layers*cell_stride] soil water content of the whole profile, mm */
    double uns_depth;       /* depth to integrate the water content to, m */
    int32_t mem_kind;       /* SPLASH_MEM_HOST or SPLASH_MEM_DEVICE (inputs and outputs alike) */
    int32_t reserved;
} splash_unswc_in;

typedef struct splash_unswc_out {
    int64_t cell_stride;    /* elements between consecutive layers of the outputs; 0 means n_cells */
    double* theta_i;        /* mean volumetric moisture of the profile, m3/m3 (theta_mean file, :103) */
    double* wtd;            /* water table depth, m (:121) */
    double* w_z;            /* water content from the surface to uns_depth, mm (:129) */
    double* se;             /* effective saturation of that layer, 0..1 (:139) */
    int32_t mem_kind;
    int32_t reserved;
} splash_unswc_out;

int splash_unswc_grid_run(splash_ctx* ctx, const splash_unswc_in* in, splash_unswc_out* out);

/* ---- monthly -> daily forcing: the deterministic half of splash.point's step 01 (R/splash.point.R:66-86) ----
 * When the forcing is monthly, splash.point interpolates air temperature and shortwave radiation onto the daily
 * axis with stats::approx(time_index_month, x, time_index, method = "linear", rule = 2)$y (:77, :83): knots at the
 * first day of each month, NA months dropped, the end values held outside the knots, and an all-NA series when
 * fewer than two months are present (:75-76, :81-82).  This entry does that for a block of cells on the device,
 * so that monthly grids (the CRU example of the package) cross the PCIe bus as monthly data and the daily series
 * exist only in HBM, in the layout splash_grid_in takes (pass the result as device forcing).  Precipitation goes
 * through month2day_rain (:460-516), which draws from rgamma and stays with the caller. */
typedef struct splash_m2d_in {
    int64_t n_cells;
    int64_t n_months;
    int64_t n_days;
    int64_t in_stride;          /* elements between consecutive months of `monthly`; 0 means n_cells */
    int64_t out_stride;         /* elements between consecutive days of the output; 0 means n_cells */
    const int32_t* month_start; /* [n_months] HOST: 0-based index on the daily axis of each month's first day
                                 * (time_index_month - time_index[1]); strictly increasing */
    const double* monthly;      /* [n_months*in_stride] month-major, cells contiguous */
    int32_t mem_kind;           /* SPLASH_MEM_HOST or SPLASH_MEM_DEVICE, for `monthly` and the output alike */
    int32_t out_f32;            /* 0: the output is double[]; 1: float[] (the f32 forcing layout of splash_grid_in) */
} splash_m2d_in;

/* daily_out: [n_days*out_stride] double or float according to in->out_f32. */
int splash_month2day_linear(splash_ctx* ctx, const splash_m2d_in* in, void* daily_out);

/* ---- terrain preprocessing, first slice (SURVEY 8f-2): what splash.grid derives from the DEM before the hot path ----
 * Small-grid branch of splash.grid (R/splash.grid.R:95-110): resolution <- sqrt(area(elev)) * 1000, lat from the cell
 * centres, terrain(elev, opt = c('slope', 'aspect'), unit = 'degrees') with NA slopes of valid cells set to 0 (:107), and
 * of upslope_area() (R/upslope_area.R:12-58) the flow direction terrain(elev, opt = 'flowdir') and the in-tree focal
 * counts ncellflow(flowdir, 'in' | 'out', met = 'top') (:140-165).  The contributing area itself (topmodel::sinkfill /
 * topidx) is splash_upslope_area_run below.
 * PARITY UNPINNED: raster::terrain and raster::area are third-party code that is not in /root/reference; the kernels
 * follow their published formulas (Horn 1981 slope/aspect on 8 neighbours with metric cell sizes from the latitude,
 * D8 flow direction with codes 1 = E, 2 = SE, 4 = S, ... 128 = NE, drop over distance), and where raster is random (ties
 * of the steepest drop) the lowest code wins. */
typedef struct splash_terrain_in {
    int64_t n_rows, n_cols;
    const double* elev;     /* [n_rows*n_cols] row-major, north row first (raster order); NaN = NA */
    double ymax;            /* northern edge of the grid (degrees, or metres when lonlat == 0) */
    double xres, yres;      /* cell size (degrees, or metres when lonlat == 0) */
    int32_t lonlat;         /* 1: geographic coordinates (cell sizes in metres follow from the latitude) */
    int32_t mem_kind;       /* SPLASH_MEM_HOST or SPLASH_MEM_DEVICE, inputs and outputs alike */
} splash_terrain_in;

typedef struct splash_terrain_out {  /* every layer [n_rows*n_cols] row-major; any pointer may be NULL */
    double* slope;          /* degrees; NA (border / NA neighbour) of a valid cell -> 0, R/splash.grid.R:107 */
    double* aspect;         /* degrees clockwise from north; same NA rule */
    double* lat;            /* latitude of the cell centre where elev is valid, else NA (:101-104) */
    double* resolution;     /* sqrt(cell area) in m (:98) */
    double* flowdir;        /* D8 code, NA on the border and where a neighbour is NA */
    double* ncellin;        /* cells draining in, at least 1 (ncellflow's nmatch[nmatch==0] <- 1); NA where all nine flowdir are NA */
    double* ncellout;       /* ncellflow(flowdir, 'out', 'top') */
} splash_terrain_out;

int splash_terrain_run(splash_ctx* ctx, const splash_terrain_in* in, splash_terrain_out* out);

/* ---- upslope contributing area (SURVEY 8f-2, second slice): the Au layer of splash_grid_in ----
 * What upslope_area() gets from topmodel::sinkfill(dem, res, degree) and topidx(filled, res)$area
 * (R/upslope_area.R:12-58): depression filling, then multiple-flow-direction accumulation.  Au[1] of the reference;
 * Au[2], Au[3] are splash_terrain_run's ncellin / ncellout.
 *
 * PARITY UNPINNED: topmodel is CRAN code that is not in the reference tree, so this is a precise published definition:
 *   Cells.  Per-row metric sizes dx, dy as splash_terrain_run (lonlat: a sphere of 6 378 137 m at the row's centre
 *     latitude), diagonal distance dd = sqrt(dx^2 + dy^2), cell area dx*dy.  Flow runs between valid cells only, over
 *     8 neighbours; distances and contour lengths of a step are those of the row the step starts in.
 *   Boundary.  A valid cell is a boundary cell if it is on the grid edge or has an NA neighbour.
 *   Fill.  The filled surface W is the least surface with W >= Z, W = Z on boundary cells, and for every other valid
 *     cell a valid neighbour n with W(c) >= W(n) + eps(c->n), eps = dist(c->n) * tan(min_slope_deg) (Planchon and
 *     Darboux 2001): the fixpoint of W(c) = max(Z(c), min_n W(n) + eps(c->n)), unique because eps > 0 (and for
 *     floating point as long as W + eps > W, i.e. eps above half an ulp of the elevations).
 *   Accumulation.  Quinn et al. (1991), as topidx: every valid neighbour n with W(n) < W(c) receives the share
 *     w / S of c's area, w = tan(beta) * L, tan(beta) = (W(c) - W(n)) / dist, L = 0.5 r (cardinal) or 0.354 r
 *     (diagonal), r = sqrt(dx*dy), S the sum of c's w.  area(c) = dx*dy + sum over donors u of area(u) * (w_uc / S_u).
 *     The area of a cell without a lower valid neighbour leaves the grid there.
 *   Evaluation order.  Neighbours in D8 code order (E, SE, S, SW, W, NW, N, NE) for both sums, each a left-to-right
 *     sum starting from 0 (S) or dx*dy (area); w = ((W(c) - W(n)) / dist) * L.  tan(), cos() and every per-row value
 *     are computed once on the host; the kernels use no FMA and IEEE division, so the result is reproducible bit
 *     for bit and does not depend on the schedule.
 * To be checked against a real R run of upslope_area(): the 0.354 literal for the diagonal contour length; per-row
 * metric cell sizes (topmodel takes one square `res`); the edge and NA treatment (R/upslope_area.R sets NA to -9999
 * before the call); and the `degree` R passes to sinkfill (0.1 is assumed, also the Python default).
 *
 * Elevations must be finite or NaN (+-inf is SPLASH_ERR_BAD_ARG); n_rows * n_cols must fit in int32 and n_rows in
 * 2 097 120.  The fill runs at most n_rows * n_cols sweeps and the accumulation at most one round per valid cell;
 * reaching either bound is SPLASH_ERR_CUDA, not a loop.  Multi-GPU contexts run it on their first GPU. */
typedef struct splash_upslope_in {
    int64_t n_rows, n_cols;
    const double* elev;     /* [n_rows*n_cols] row-major, north row first; NaN = NA (as splash_terrain_in) */
    double ymax, xres, yres;/* as splash_terrain_in */
    int32_t lonlat;
    int32_t mem_kind;       /* SPLASH_MEM_HOST or SPLASH_MEM_DEVICE, inputs and outputs alike */
    double min_slope_deg;   /* minimum drop the fill enforces, degrees, in (0, 90) (topmodel::sinkfill's `degree`) */
} splash_upslope_in;

typedef struct splash_upslope_out {
    double* area;           /* [n_rows*n_cols] contributing area m2 (own cell included); NA where elev is NA */
    double* filled;         /* optional [n_rows*n_cols]: the filled DEM W (NULL = not wanted) */
    int64_t fill_sweeps;    /* written by the call: global fill sweeps run, the last of which changed no cell */
    int64_t accum_rounds;   /* written by the call: accumulation rounds (= cells on the longest flow path) */
} splash_upslope_out;

int splash_upslope_area_run(splash_ctx* ctx, const splash_upslope_in* in, splash_upslope_out* out);

/* ---- D-infinity contributing area (SURVEY 8f-2, third slice): Au for coarse or large grids ----
 * What upslope_areav2() (R/upslope_area.R:59-137) gets from TauDEM through mpiexec (:76-81): PitRemove, DinfFlowDir
 * (which resolves flats) and AreaDinf.  Same cells, boundary and output as splash_upslope_area_run; the Python
 * api.upslope_areav2 adds splash_terrain_run's ncellin / ncellout as Au[2], Au[3].
 *
 * PARITY UNPINNED: TauDEM and the lines of R/upslope_area.R that call it are not in this tree, so this is a precise
 * published definition:
 *   Cells, distances, boundary.  As splash_upslope_area_run: per-row dx, dy, dd = sqrt(dx^2 + dy^2), area dx*dy, the
 *     metrics of a step taken from the row it starts in; a boundary cell is a valid cell on the grid edge or next to
 *     an NA cell.
 *   Fill.  W(c) = the least, over 8-connected paths of valid cells from c to a boundary cell, of the highest Z on the
 *     path (the minimax spill elevation; W = Z on boundary cells).  It is the greatest solution of
 *     W(c) = max(Z(c), min_n W(n)), the Planchon-Darboux fixpoint with eps = 0, which the sweeps reach from above.
 *   Directions.  Boundary cells have none: their area leaves the grid (as TauDEM leaves edge cells without one).  Every
 *     other valid cell with a strictly lower neighbour takes the D-infinity facet rule on W (Tarboton 1997).  Facets in
 *     Tarboton's order, (cardinal e1, diagonal e2, ac, af): 1 (E, NE, 0, 1), 2 (N, NE, 1, -1), 3 (N, NW, 1, 1),
 *     4 (W, NW, 2, -1), 5 (W, SW, 2, 1), 6 (S, SW, 3, -1), 7 (S, SE, 3, 1), 8 (E, SE, 4, -1).  d1, d2 = dx, dy when
 *     e1 is E or W, dy, dx when it is N or S; theta_f = atan2(d2, d1), per row on the host.
 *     s1 = (e0 - e1) / d1, s2 = (e1 - e2) / d2, then, by comparisons only:
 *       s2 > 0, s1 > 0 and s2 * d1 < s1 * d2:  inside the facet, s = sqrt(s1*s1 + s2*s2), r = atan(s2 / s1);
 *       otherwise s2 > 0:                       clipped to the diagonal, s = (e0 - e2) / dd, r = theta_f;
 *       otherwise:                              clipped to the cardinal, s = s1, r = 0.
 *     The facet of largest s > 0 wins, ties to the lowest facet.  Angle = ac * (pi/2) + af * r (2 pi is reported as
 *     0).  atan(s2 / s1) is the only transcendental the device evaluates.
 *   Proportions.  Inside a facet the cardinal receiver gets 1 - p and the diagonal one p = min(r / theta_f, 1)
 *     (TauDEM's angle split for square cells, its natural generalisation for others; the min keeps a share from going
 *     negative when atan rounds r a few ulp past theta_f); a clipped cell has one receiver, with 1.
 *   Flats.  A flat cell is a valid non-boundary cell without a strictly lower neighbour.  Each 8-connected set of flat
 *     cells is level and has an outlet: a non-flat or boundary neighbour at the same W.  Flats are resolved as
 *     Garbrecht and Martz (1997) in the formulation of Barnes, Lehman and Mulla (2014): breadth-first distances
 *     towards lower (1 next to an outlet) and away from higher (1 on flat cells next to higher ground), H = the
 *     largest away distance of the flat (0, with away = 0, on a flat without higher ground), and the mask
 *     M = 2 * towards + (H - away); outlets count as M = 0.  A flat cell takes the facet rule on M instead of W, over
 *     the facets whose two neighbours are at its W.  If no facet gives s > 0, everything goes to the neighbour at its W
 *     of steepest descent (M(c) - M(n)) / dist, ties to the lowest D8 code, with the angle of the first facet that has
 *     that neighbour, clipped to it (Barnes: such a neighbour exists).
 *   Accumulation.  area(c) = dx*dy + sum over donors u in D8 code order of area(u) * p(u->c), a left-to-right sum,
 *     no FMA, IEEE division.  Every receiver is strictly lower in W or, on a flat, in M, so the graph is acyclic and
 *     the result does not depend on the schedule.
 * To be checked against a real R + TauDEM run of upslope_areav2(), in this order:
 *   1. which TauDEM tool's grid becomes Au[1] (AreaDinf's is assumed, not AreaD8's);
 *   2. the conversion of TauDEM's specific catchment area (per unit contour width) to m2 (here: the area itself);
 *   3. edge contamination: assumed off, i.e. the area is reported everywhere, as TauDEM's -nc;
 *   4. that edge cells have no direction;
 *   5. the proportion rule on non-square cells;
 *   6. the weighting of the two gradients of Garbrecht and Martz: TauDEM's own flat code may weight them otherwise;
 *   7. that Au[2..3] are still ncellflow's counts.
 *
 * Arguments, limits and multi-GPU contexts as splash_upslope_area_run.  The fill and the flat labelling run at most
 * n_rows * n_cols sweeps each, the distances and the accumulation at most one round per valid cell; reaching a bound
 * is SPLASH_ERR_CUDA, not a loop. */
typedef struct splash_dinf_in {
    int64_t n_rows, n_cols;
    const double* elev;     /* as splash_upslope_in */
    double ymax, xres, yres;
    int32_t lonlat;
    int32_t mem_kind;       /* SPLASH_MEM_HOST or SPLASH_MEM_DEVICE, inputs and outputs alike */
} splash_dinf_in;

typedef struct splash_dinf_out {
    double* area;           /* [n_rows*n_cols] contributing area m2 (own cell included); NA where elev is NA */
    double* filled;         /* optional [n_rows*n_cols]: the filled DEM W (NULL = not wanted) */
    double* angle;          /* optional [n_rows*n_cols]: flow angle, radians counter-clockwise from east in [0, 2 pi);
                               NaN where a cell has no direction */
    int64_t fill_sweeps;    /* written by the call: global fill sweeps run, the last of which changed no cell */
    int64_t flat_rounds;    /* written by the call: flat labelling sweeps + rounds of the two distances */
    int64_t accum_rounds;   /* written by the call: accumulation rounds (= cells on the longest flow path) */
} splash_dinf_out;

int splash_upslope_dinf_run(splash_ctx* ctx, const splash_dinf_in* in, splash_dinf_out* out);

/* Diagnostic (used by tests/test_math_gpu.py, not by the R glue): apply one of the day step's
 * transcendental functions to a host array on the device.  op: 0 exp, 1 log, 2 acos, 3 sin (hour
 * angles, [0, pi]).  These are the library's own implementations (csrc/splash_math.cuh), which stand
 * in for the libm calls of src/SPLASH.cpp, src/EVAP.cpp and src/SOLAR.cpp.  op 4..10: the guard-free
 * bodies of the branch-light day step and what they must equal bit for bit -- 4 acos body, 5 sqrt
 * body, 6 sqrt, 7 division body, 8 division (second operand x[(7919 i + 13) mod n]), 9 exp body,
 * 10 log body; NaN where an argument is outside the body's guard. */
int splash_debug_math(splash_ctx* ctx, int op, int64_t n, const double* x, double* y);

#ifdef __cplusplus
}
#endif
#endif /* SPLASH_CUDA_H */
