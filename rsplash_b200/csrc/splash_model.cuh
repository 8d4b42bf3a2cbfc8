// splash_model.cuh -- device-side SPLASH v2.0 cell model for sm_100a (FP64 CUDA cores).
//
// One thread owns one cell.  Per-cell constants live in shared memory as private columns
// (cc[k * blockDim.x + threadIdx.x]: conflict-free, no synchronisation), the five state scalars
// (wn, snow, qin, td, nd) stay in registers across the day loop.
//
// What is restated here (reference paths relative to /root/reference, see also SURVEY.md App. A):
//   cell_setup()      R/splash.point.R:96-115 (soil_info) + soil_hydro :232-416, the per-cell
//                     invariants of SPLASH::run_one_day (src/SPLASH.cpp:946-1029, 1291-1356),
//                     EVAP::elv2pres (src/EVAP.cpp:319-336), SOLAR tau_o (src/SOLAR.cpp:170)
//   lateral_consts()  the terms of run_one_day that depend on `cellout`, which R overwrites with
//                     the aridity index between the two spin-ups (R/splash.point.R:150)
//   snow_class()      snowfall_prob, R/splash.point.R:560-578 (NA / p_snow >= 0.5 / not)
//   splash_day()      one day: snow partition (R/splash.point.R:120-128,547-555), then
//                     SOLAR::calculate_daily_fluxes (src/SOLAR.cpp:129-255),
//                     EVAP::calculate_daily_fluxes (src/EVAP.cpp:100-263),
//                     SPLASH::run_one_day (src/SPLASH.cpp:984-1583) incl. moist_surf (:1921-1961)
//                     and inf_GA (:1963-2023)
//
// Numerics: the formulas and their order follow the reference; the file is compiled with -fmad=false
// (the reference build has no FMA contraction, SURVEY B-9).  With -DSPLASH_LEVEL=0 every operation is the
// reference's and hoisting is limited to sub-expressions that are bit-identical when computed once; the
// differences against the CPU reference are then libdevice vs glibc transcendentals (<= 2 ulp each).
// The DEFAULT, level 1, additionally evaluates x^y as exp(y log x) with shared logarithms, divides by
// guarded reciprocal multiplication, uses the library's own exp/log/acos (<= 1.5 ulp) and reproduces five
// floating-point accidents of the reference explicitly (DESIGN.md section 5): a few tens of ulp per
// operation, which only ill-conditioned cells turn into more than the gates
// (profiles/r02_level_table.json: 91 cells of 12 000 against 22 at level 0 and 102 for the reference's own
// -mfma build).
#pragma once

// SPLASH_LEVEL selects how literally the day step follows the reference's floating-point recipe:
//   0  every operation in the reference's order, libdevice pow() where the reference calls pow()
//   1  (default) same formulas, but x^y is evaluated as exp(y*log(x)) with the logarithm shared
//      between powers of the same base, divisions by per-cell constants become multiplications
//      by reciprocals computed once, and the Kunsat power is skipped where the reference never
//      uses it.  Each rewrite perturbs a result by a few ulp (1e-16 relative), three orders of
//      magnitude inside the parity budget; tests/test_parity_gpu.py runs the gates on both.
#ifndef SPLASH_LEVEL
#define SPLASH_LEVEL 1
#endif
// the two halves of level 1
#define SPLASH_L1_POW (SPLASH_LEVEL >= 1)    // x^y as exp(y*log(x)) with shared logarithms
#define SPLASH_L1_RECIP (SPLASH_LEVEL >= 1)  // reciprocals of per-cell constants, consistent theta scaling
// SPLASH_FAST_STATE: the uniform kernels' state half through day_state_fast (branch-light, same bits) with day_state as
// the fallback; the straggler chain has its own switch (SPLASH_CHAIN_FAST, splash_cuda.cu)
#ifndef SPLASH_FAST_STATE
#define SPLASH_FAST_STATE 0
#endif

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <type_traits>

#include "splash_math.cuh"
#include "splash_consts.cuh"

namespace splash {

// ------------------------------------------------------------------------------------------------
// Global constants, reference src/global.cpp:51-82
// ------------------------------------------------------------------------------------------------
constexpr double kA = 91.86328;
constexpr double kalb_sw = 0.30;
constexpr double kb = 0.2012435;
constexpr double kc = 0.25;
constexpr double kd = 0.50;
constexpr double kkfus = 334000;
constexpr double kG = 9.80665;
constexpr double kGsc = 1360.8;
constexpr double kL = 0.0065;
constexpr double kMa = 0.028963;
constexpr double kMv = 0.01802;
constexpr double kPo = 101325;
constexpr double kR = 8.31447;
constexpr double kTo = 288.15;
constexpr double kPI = 3.141592653589793;
constexpr double kpir = (kPI / 180.0);
constexpr double kfluidity = 35187037;

// ------------------------------------------------------------------------------------------------
// Per-cell constant slots (rows of the [NCC][pitch] constant matrix)
// ------------------------------------------------------------------------------------------------
enum CellConst : int {
    // snow partition
    C_ELEV_K = 0,  // elev * 0.0004596581
    C_LAT_K,       // |lat| * 0.0110592101
    C_TT,          // threshold temperature Tt (written by the snow-threshold kernel)
    // geometry
    C_COS_LAT, C_SIN_LAT, C_SIN_S, C_COS_S, C_COS_A, C_SIN_A, C_TAN_S, C_COS2_S,
    // atmosphere
    C_TAU_O, C_TAU_A, C_PATM, C_PBAR, C_PBARF, C_VISC0,
    // soil column
    C_SAT, C_RES, C_DEPTH, C_THS, C_THR, C_DTH, C_ILAM, C_NLAM, C_E3, C_BUB,
    C_WMAX, C_THWMAX, C_INTPERM, C_HF, C_KUEXP,
    // lateral flow
    C_BRQ0, C_BRW, C_ACSW, C_CW, C_SIDOCT, C_AI, C_AU,
    C_CELLOUT, C_CQ0, C_ACSQS, C_CT,  // depend on cellout (recomputed after the aridity pass)
    // output stage
    C_WRR,         // Wmax_R - RES, denominator of sm_lim (R/splash.point.R:197)
    // level-1 reciprocals and cached powers
    C_INV_D1000, C_INV_DTH, C_INV_WMR, C_INV_TAU_B, C_INV_AI, C_INV_DENKB, C_TEN_BP, C_KU_WMAX,
    // only read by the level-0 day step (and by cell_setup)
    C_D1000, C_WMR, C_TAU_B, C_DENKB, C_BP10,
    NCC,
#if SPLASH_L1_RECIP
    NCC_DAY = C_D1000  // constants the day step reads: what the kernels stage in shared memory
#else
    NCC_DAY = NCC
#endif
};

// Sections of day_forcing that read constants an accessor may keep outside its directly addressable storage: the bulk
// launch holds them in tensor memory and moves each group into registers at the top of its section (splash_cuda.cu,
// TmemCC).  day_forcing calls cc_fetch where every lane of a warp reaches it; accessors without such storage ignore it.
enum CCGroup : int { CCG_SNOW, CCG_GEOMETRY, CCG_PRESSURE, CCG_OUTPUT };
template <class CC>
__device__ __forceinline__ void cc_fetch(const CC&, CCGroup) {}

struct DayTab {      // per-day values that do not depend on the cell (host-built, SOLAR.cpp:98-124)
    double dr;       // distance factor
    double sd;       // sin(delta*pir)
    double cd;       // cos(delta*pir)
    int32_t month;   // 0..11
    int32_t group;   // month-group id of the day (monthly output)
};

struct MonthTab {    // frain_func's month factors (R/splash.point.R:549-550), host-built
    double s1[12];   // dsin((m+2)/1.91)
    double trm14[12];// 1.4 * (13.3*(0.55+dsin(m+4))*0.6)
};

struct CellState {
    double wn, snow, qin, td, nd;
};

struct DayOut {
    double ro, pet, aet, cond, bflow, netr;
};

#if SPLASH_L1_RECIP
#define SPLASH_FDIV(a, b) fm::fdiv((a), (b))       // a/b to ~1.5 ulp, IEEE behaviour for 0/inf/NaN denominators
#define SPLASH_DIVC_1000(a) ((a) * kD.k_1em3)     // divisions by compile-time constants: a * (1.0 / c), the reciprocal
#define SPLASH_DIVC_6(a) ((a) * kD.k_sixth)        // folded at compile time (and kept in constant memory)
#define SPLASH_DIVC_1E6(a) ((a) * kD.k_1em6)
#define SPLASH_TO_DEG(x) ((x) * kD.to_deg)
#define SPLASH_DIV_D1000(x) ((x) * cc(C_INV_D1000))
#define SPLASH_DIV_DTH(x) ((x) * cc(C_INV_DTH))
#define SPLASH_DIV_TAU_B(x) ((x) * cc(C_INV_TAU_B))
#define SPLASH_DIV_1000(x) ((x) * kD.k_1em3)
#else
#define SPLASH_FDIV(a, b) ((a) / (b))
#define SPLASH_DIVC_1000(a) ((a) / (1000.0))
#define SPLASH_DIVC_6(a) ((a) / (6.0))
#define SPLASH_DIVC_1E6(a) ((a) / (1e6))
#define SPLASH_TO_DEG(x) ((x) / kpir)
#define SPLASH_DIV_D1000(x) ((x) / cc(C_D1000))
#define SPLASH_DIV_DTH(x) ((x) / cc(C_DTH))
#define SPLASH_DIV_TAU_B(x) ((x) / cc(C_TAU_B))
#define SPLASH_DIV_1000(x) ((x) / 1000.0)
#endif

// One shared copy of each transcendental instead of ~25 inlined expansions: the day step is a
// single long loop body and its code size, not its arithmetic, was the first bottleneck (ncu:
// 48 % of warp-stall samples were `no_instruction` with a 91 KB kernel, profiles/README.md).
#if SPLASH_LEVEL >= 1
using fm::f_acos;  // splash_math.cuh: coefficients in __constant__ memory instead of 64-bit immediates
using fm::f_exp;
using fm::f_log;
using fm::f_sin;
#else
__device__ __noinline__ double f_exp(double x) { return exp(x); }
__device__ __noinline__ double f_log(double x) { return log(x); }
__device__ __noinline__ double f_acos(double x) { return acos(x); }
__device__ __noinline__ double f_sin(double x) { return sin(x); }
#endif

// Snow-age factor of the albedo, SOLAR.cpp:208: exp(-0.895189 * nd).  nd counts the days since the last snowfall
// (0, 1, 2, ...), so the factor only takes the values of a table, which k_init_tables fills with the very
// function the day step would call (bit-identical); beyond the table the factor has underflowed to exactly 0.
constexpr int kSnowAgeTab = 1024;
__device__ double g_snow_age_tab[kSnowAgeTab];

__device__ __forceinline__ double snow_age_factor_formula(double nd) { return f_exp(-0.895189 * nd); }

__device__ __forceinline__ double snow_age_factor(double nd) {
#if SPLASH_LEVEL >= 1
    if (nd >= 0.0 && nd < (double)kSnowAgeTab) {
        const int i = (int)nd;
        if ((double)i == nd) return g_snow_age_tab[i];
    }
#endif
    return snow_age_factor_formula(nd);
}

// Hour angle h = acos(x) (degrees) together with sin(h): the reference evaluates sin(h * pir) after
// h = acos(x) / pir; level 1 takes sin(acos(x)) = sqrt((1 - x)(1 + x)) instead (accurate to ~1.5 ulp for
// every |x| < 1, no cancellation), and the reference's own values at the clamps: sin(0) = 0 and
// sin(180 * pir) = sin(fl(pi)) = 1.2246467991473532e-16.
#define SPLASH_SIN_180 kD.sin_180

// How the day step reaches its transcendentals.  MathShared: calls of the shared out-of-line copies.
// MathInline: the same algorithms expanded in place -- no call, no argument shuffling -- what the day-loop
// kernels use.  Both evaluate identical operation sequences: results are bit-equal.
struct MathShared {
    static __device__ __forceinline__ double exp(double x) { return f_exp(x); }
    static __device__ __forceinline__ double log(double x) { return f_log(x); }
    static __device__ __forceinline__ double acos(double x) { return f_acos(x); }
    static __device__ __forceinline__ double sin(double x) { return f_sin(x); }
};
#if SPLASH_LEVEL >= 1
struct MathInline {
    static __device__ __forceinline__ double exp(double x) { return fm::exp_core(x); }
    static __device__ __forceinline__ double log(double x) { return fm::log_core(x); }
    static __device__ __forceinline__ double acos(double x) { return fm::acos_core(x); }
    static __device__ __forceinline__ double sin(double x) { return fm::sin_core(x); }
};
#else
using MathInline = MathShared;
#endif

// std::max / std::min semantics of the reference (NaN in the first argument wins, SURVEY B-1)
__device__ __forceinline__ double cxx_max(double a, double b) { return (a < b) ? b : a; }
__device__ __forceinline__ double cxx_min(double a, double b) { return (b < a) ? b : a; }

// ------------------------------------------------------------------------------------------------
// glibc expf, bit-exact.  EVAP::calc_viscosity_h2o ends in std::f_exp(float) (src/EVAP.cpp:451),
// i.e. glibc's expf, whose result differs from the correctly rounded one in a fraction of a
// percent of arguments; viscosity scales every conductivity, so a 1-ulp float error (6e-8) would
// dominate the error budget (SURVEY B-4).  This follows the published algorithm of glibc 2.28+
// (sysdeps/ieee754/flt-32/e_expf.c, N = 32 table, degree-3 polynomial in double) with the FMA
// contraction pattern of the x86-64 `-mfma` build that the ifunc selects on the CPUs used here.
// ------------------------------------------------------------------------------------------------
__device__ __constant__ double kExp2Tab[32] = {
    0x1.0000000000000p+0, 0x1.059b0d3158574p+0, 0x1.0b5586cf9890fp+0, 0x1.11301d0125b51p+0,
    0x1.172b83c7d517bp+0, 0x1.1d4873168b9aap+0, 0x1.2387a6e756238p+0, 0x1.29e9df51fdee1p+0,
    0x1.306fe0a31b715p+0, 0x1.371a7373aa9cbp+0, 0x1.3dea64c123422p+0, 0x1.44e086061892dp+0,
    0x1.4bfdad5362a27p+0, 0x1.5342b569d4f82p+0, 0x1.5ab07dd485429p+0, 0x1.6247eb03a5585p+0,
    0x1.6a09e667f3bcdp+0, 0x1.71f75e8ec5f74p+0, 0x1.7a11473eb0187p+0, 0x1.82589994cce13p+0,
    0x1.8ace5422aa0dbp+0, 0x1.93737b0cdc5e5p+0, 0x1.9c49182a3f090p+0, 0x1.a5503b23e255dp+0,
    0x1.ae89f995ad3adp+0, 0x1.b7f76f2fb5e47p+0, 0x1.c199bdd85529cp+0, 0x1.cb720dcef9069p+0,
    0x1.d5818dcfba487p+0, 0x1.dfc97337b9b5fp+0, 0x1.ea4afa2a490dap+0, 0x1.f50765b6e4540p+0};

__device__ __forceinline__ float glibc_expf(float x) {
    const double xd = (double)x;
    if (!(fabsf(x) < 88.0f)) return (float)f_exp(xd);  // overflow/underflow/NaN tails: not reached by viscosity
    const double InvLn2N = kD.ef_inv, Shift = 0x1.8p+52;
    const double C0 = kD.ef_c0, C1 = kD.ef_c1, C2 = kD.ef_c2;
    double kd = fma(InvLn2N, xd, Shift);
    const uint64_t ki = (uint64_t)__double_as_longlong(kd);
    kd = kd - Shift;
    const double r = fma(InvLn2N, xd, -kd);
    const double z = fma(r, C0, C1);
    const double r2 = r * r;
    double y = fma(r, C2, 1.0);
    y = fma(z, r2, y);
    const uint64_t i = ki & 31u;
    const uint64_t t = (uint64_t)__double_as_longlong(kExp2Tab[i]) - (i << 47) + (ki << 47);
    y = y * __longlong_as_double((long long)t);
    return (float)y;
}

// ------------------------------------------------------------------------------------------------
// EVAP helpers
// ------------------------------------------------------------------------------------------------
struct DensityPoly {
    double po, ko, ca, cb;
};

// temperature polynomials of EVAP::density_h2o, src/EVAP.cpp:349-378 (power sums as written)
__device__ __forceinline__ DensityPoly density_poly(double tc) {
    DensityPoly q;
    // (the literals live in constant memory, splash_consts.cuh: same values, same operations)
    double po = kD.po0;
    po += kD.po1 * tc;
    po += kD.po2 * tc * tc;
    po += kD.po3 * tc * tc * tc;
    po += kD.po4 * tc * tc * tc * tc;
    po += kD.po5 * tc * tc * tc * tc * tc;
    po += kD.po6 * tc * tc * tc * tc * tc * tc;
    po += kD.po7 * tc * tc * tc * tc * tc * tc * tc;
    po += kD.po8 * tc * tc * tc * tc * tc * tc * tc * tc;
    double ko = kD.ko0;
    ko += kD.ko1 * tc;
    ko += kD.ko2 * tc * tc;
    ko += kD.ko3 * tc * tc * tc;
    ko += kD.ko4 * tc * tc * tc * tc;
    ko += kD.ko5 * tc * tc * tc * tc * tc;
    double ca = kD.ca0;
    ca += kD.ca1 * tc;
    ca += kD.ca2 * tc * tc;
    ca += kD.ca3 * tc * tc * tc;
    ca += kD.ca4 * tc * tc * tc * tc;
    double cb = kD.cb0;
    cb += kD.cb1 * tc;
    cb += kD.cb2 * tc * tc;
    cb += kD.cb3 * tc * tc * tc;
    cb += kD.cb4 * tc * tc * tc * tc;
    q.po = po;
    q.ko = ko;
    q.ca = ca;
    q.cb = cb;
    return q;
}

// pressure part of EVAP::density_h2o, src/EVAP.cpp:381-388 (pbar = 1e-5 * p)
// kExact: the IEEE division, for the value that is narrowed to float in the viscosity routine.
template <bool kExact = false>
__device__ __forceinline__ double density_at(const DensityPoly& q, double pbar) {
    const double num = (q.ko + q.ca * pbar + q.cb * (pbar * pbar));
    double pw = num;
    pw = kExact ? pw / (num - pbar) : SPLASH_FDIV(pw, num - pbar);
    pw *= (1.0e3) * q.po;
    return pw;
}

// EVAP::calc_viscosity_h2o, src/EVAP.cpp:405-462, with its FP32 roundings.  `tcf` is the float
// the reference narrows tw to, `rho_d` = density_h2o((double)tcf, (double)pf) in double.
__device__ __forceinline__ double viscosity_h2o(float tcf, double rho_d) {
    const float rho = (float)rho_d;
    const float tbar = (float)(((double)tcf + kD.lv_a) / kD.vs_tk);
    const float tbarx = (float)sqrt((double)tbar);  // pow(tbar, 0.5) in double, narrowed
    const float tbar2 = tbar * tbar;
    const float tbar3 = tbar * tbar * tbar;
    const float rbar = rho / 322.0f;
    float mu0 = (float)(kD.vs_m0 + kD.vs_m1 / (double)tbar + kD.vs_m2 / (double)tbar2 - kD.vs_m3 / (double)tbar3);
    mu0 = (float)(1e2 * (double)tbarx / (double)mu0);
    const float ctbar = (float)((1.0 / (double)tbar) - 1.0);
    // integer powers of (rbar - 1.0) in double, j = 0..6
    const double rb = (double)rbar - 1.0;
    const double rb2 = rb * rb, rb3 = rb2 * rb, rb4 = rb3 * rb, rb5 = rb4 * rb, rb6 = rb5 * rb;
    // integer powers of ctbar in double narrowed to float, i = 0..5
    const double ct = (double)ctbar;
    const double ct2 = ct * ct, ct3 = ct2 * ct, ct4 = ct3 * ct, ct5 = ct4 * ct;
    // coef2_i = sum_j h[j][i] * (rbar-1)^j, accumulated in the reference's order with a float
    // round after every add; the table's zero entries add an exact 0 and are skipped.
    // (h: the float table entry widened to double, (double)0.520094f etc.; constant memory holds those doubles)
#define SPLASH_H(acc, h, p) acc = (float)((double)(acc) + (h) * (p))
    float c2_0 = 0.0f, c2_1 = 0.0f, c2_2 = 0.0f, c2_3 = 0.0f, c2_4 = 0.0f, c2_5 = 0.0f;
    SPLASH_H(c2_0, kD.h00, 1.0); SPLASH_H(c2_0, kD.h10, rb); SPLASH_H(c2_0, kD.h20, rb2);
    SPLASH_H(c2_0, kD.h30, rb3); SPLASH_H(c2_0, kD.h40, rb4);
    SPLASH_H(c2_1, kD.h01, 1.0); SPLASH_H(c2_1, (double)0.999115f, rb); SPLASH_H(c2_1, kD.h21, rb2);
    SPLASH_H(c2_1, kD.h31, rb3);
    SPLASH_H(c2_2, kD.h02, 1.0); SPLASH_H(c2_2, (double)1.88797f, rb); SPLASH_H(c2_2, kD.h22, rb2);
    SPLASH_H(c2_3, kD.h03, 1.0); SPLASH_H(c2_3, kD.h13, rb); SPLASH_H(c2_3, kD.h23, rb2);
    SPLASH_H(c2_3, (double)0.0698452f, rb4); SPLASH_H(c2_3, kD.h63, rb6);
    SPLASH_H(c2_4, kD.h24, rb2); SPLASH_H(c2_4, kD.h54, rb5);
    SPLASH_H(c2_5, kD.h15, rb); SPLASH_H(c2_5, kD.h65, rb6);
#undef SPLASH_H
    float mu1 = 0.0f;
    mu1 = __fadd_rn(mu1, __fmul_rn(1.0f, c2_0));         // pow(ctbar, 0) == 1
    mu1 = __fadd_rn(mu1, __fmul_rn((float)ct, c2_1));
    mu1 = __fadd_rn(mu1, __fmul_rn((float)ct2, c2_2));
    mu1 = __fadd_rn(mu1, __fmul_rn((float)ct3, c2_3));
    mu1 = __fadd_rn(mu1, __fmul_rn((float)ct4, c2_4));
    mu1 = __fadd_rn(mu1, __fmul_rn((float)ct5, c2_5));
    mu1 = glibc_expf(__fmul_rn(rbar, mu1));
    const float mu_bar = __fmul_rn(mu0, mu1);
    const float mu = __fmul_rn(mu_bar, 1e-6f);
    return (double)mu;
}

// EVAP::specific_heat, src/EVAP.cpp:491-515
__device__ __forceinline__ double specific_heat(double tc) {
    double cp;
    if (tc < 0) {
        cp = kD.cp_lo;
    } else if (tc > 100) {
        cp = kD.cp_hi;
    } else {
        cp = kD.cp0;
        cp += kD.cp1 * tc;
        cp += kD.cp2 * tc * tc;
        cp += kD.cp3 * tc * tc * tc;
        cp += kD.cp4 * tc * tc * tc * tc;
        cp += kD.cp5 * tc * tc * tc * tc * tc;
        cp *= (1.0e3);
    }
    return cp;
}

// ------------------------------------------------------------------------------------------------
// Brooks-Corey column transmittance: the block repeated at src/SPLASH.cpp:1406-1426 and
// :1511-1531.  Returns T_uns (after the flux-density scaling and the <0/NaN failsafe) and Acs_out.
// ------------------------------------------------------------------------------------------------
struct Transm {
    double t_uns, acs_out;
};

template <class M, class CC>
__device__ __forceinline__ Transm column_transmittance_core(const CC& cc, double sm, double ksat_visc) {
    const double bub = cc(C_BUB);
    const double e3 = cc(C_E3);
    const double depth = cc(C_DEPTH);
    Transm r;
#if SPLASH_L1_POW
    const double theta_i = SPLASH_DIV_D1000(sm);
    const double x = SPLASH_DIV_DTH(theta_i - cc(C_THR));
    const double a = cc(C_ILAM) * M::log(x);  // log shared by x^(1/lambda) and (x^(1/lambda))^(3 lambda + 1)
    const double psi_m = SPLASH_FDIV(bub, M::exp(a));
    double wtd = SPLASH_DIV_1000(bub - psi_m);
    bool clamped = false;
    if (wtd < 0.0 || isnan(wtd)) {
        wtd = kD.k_01b;
        clamped = true;
    } else if (wtd > depth) {
        wtd = depth;
        clamped = true;
    }
    r.acs_out = (depth - wtd) * cc(C_SIDOCT) * cc(C_CELLOUT);
    const double r1 = M::exp(e3 * a);  // (bub/psi_m)^e3 with bub/psi_m == x^(1/lambda)
    const double den = psi_m + (wtd * 1000.0);
    double dr;  // (bub/psi_m)^e3 - (bub/den)^e3
    if (!clamped) {
        // the second base is 1 up to rounding noise (den == bub): first-order expansion
        const double q = SPLASH_FDIV(bub, den);
        const double qm1 = q - 1.0;
        const double r2 = (fabs(qm1) < kD.k_1em7) ? (1.0 + e3 * qm1) : M::exp(e3 * M::log(q));
        dr = r1 - r2;
    } else {
        // wtd was clamped: on dry soil both bases are x^(1/lambda)-small and differ by depth/psi_m ~ 1e-15 relative.
        // Two separately composed powers (|e3 ln b| ulp each) lose that difference -- and whether the drainage Q
        // below is tiny or exactly 0 decides between a finite and an infinite t_drain (:1470).  The ratio form
        // r1 * ((den_ratio)^e3 - 1) keeps it, as the reference's two pow() of nearly equal bases do.
        const double t = e3 * M::log(SPLASH_FDIV(psi_m, den));
        const double em1 = (fabs(t) < kD.k_1em5) ? t * (1.0 + 0.5 * t) : M::exp(t) - 1.0;
        dr = -(r1 * em1);
    }
    double t_uns = (ksat_visc * bub / e3) * dr;
#else
    const double theta_i = (sm) / cc(C_D1000);
    const double psi_m = bub / pow((((theta_i - cc(C_THR)) / cc(C_DTH))), cc(C_ILAM));
    double wtd = ((bub - psi_m) / 1000.0);
    if (wtd < 0.0 || isnan(wtd)) {
        wtd = 0.01;
    } else if (wtd > depth) {
        wtd = depth;
    }
    r.acs_out = (depth - wtd) * cc(C_SIDOCT) * cc(C_CELLOUT);
    double t_uns = (ksat_visc * bub / e3) * (pow((bub / psi_m), e3) - pow((bub / (psi_m + (wtd * 1000.0))), e3));
#endif
    t_uns *= cc(C_CT);
    if (t_uns < 0.0 || isnan(t_uns)) {
        t_uns = 0.0;
    }
    r.t_uns = t_uns;
    return r;
}

template <class CC>
__device__ __noinline__ Transm column_transmittance_shared(const CC& cc, double sm, double ksat_visc) {
    return column_transmittance_core<MathShared>(cc, sm, ksat_visc);
}
template <class M, class CC>
__device__ __forceinline__ Transm column_transmittance(const CC& cc, double sm, double ksat_visc) {
    if constexpr (std::is_same<M, MathShared>::value)
        return column_transmittance_shared(cc, sm, ksat_visc);
    else
        return column_transmittance_core<M>(cc, sm, ksat_visc);
}

// snowfall_prob, R/splash.point.R:576: p_snow = 1 / (1 + exp(z)).  The path only ever asks whether p_snow is NA
// and whether p_snow >= 0.5 (:122,124).  p_snow >= 0.5 <=> exp(z) <= 1 <=> z <= 0, so away from z == 0 the sign of
// the exponent decides and no exp / division is needed; within 1e-9 of zero the expression is evaluated as
// written.  Returns -1 (NA), 1 (snow-probable day) or 0.
template <class CC>
__device__ __forceinline__ int snow_class(const CC& cc, double tc) {
    const double z = kD.snow_a + kD.snow_b * tc - cc(C_ELEV_K) - cc(C_LAT_K);
    if (isnan(z)) return -1;
    if (z < kD.snow_lo) return 1;
    if (z > kD.snow_hi) return 0;
    return (1 / (1 + exp(z)) >= 0.5) ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
// One day of one cell, in two halves.
//
//   day_forcing   everything that depends on the day's forcing and the cell's constants only: snow
//                 partition, solar geometry up to the net longwave flux, the thermodynamic
//                 coefficients and the water viscosity.  It is the same in every spin-up pass over
//                 the cyclic first year, which the straggler pool exploits (k_pool_table).
//   day_state     the part that carries the state: albedo, net radiation, evapotranspiration,
//                 snowmelt, infiltration, runoff, lateral flow, soil-water update.
//
// splash_day = day_forcing + day_state is what every other kernel inlines; splitting it moves no
// floating-point operation, so both routes give bit-identical results.
//   cc     accessor for the cell's constants
//   dt     day table entry (dr, sin/cos of declination, month)
//   mt     month table of frain_func
//   sw_in, tc, pn   raw forcing of the day (pn = total precipitation before the snow partition)
// ------------------------------------------------------------------------------------------------
struct DayPre {
    double snowfall, rain;            // R/splash.point.R:127-128
    double ru, rv, ruv, hs, sin_hs;   // SOLAR.cpp:129-159 (hs in degrees)
    double tau, dr;                   // transmittivity, distance factor
    double r_in, rw_den;              // 86400*sw_in;  (86400/pi)*(ru*pir*hs + rv*sin(hs)), SOLAR.cpp:223
    double rw_dark;                   // != 0 when sw_in == 0 or hs == 0 (first branch of SOLAR.cpp:220)
    double rnl;                       // net longwave, SOLAR.cpp:203
    double tc;
    double s, g, econ, pw, eet_k, rx; // EVAP.cpp:110-145
    double ksat_visc;                 // SPLASH.cpp:1260
#if SPLASH_L1_RECIP
    // level 1: reciprocals of forcing-only denominators of the state half (computed once per day here; for a
    // straggler once per spin-up year, in the pool's table)
    double inv_rw_den, inv_rx, inv_econ, inv_pwk, inv_k24;
    // the recession / drainage terms of run_one_day that depend on Ksat_visc and the cell only (SPLASH.cpp:1303-1360):
    // read by day_state_fast (the straggler chain takes them from its table once per spin-up year; in the fused
    // kernels they are dead values unless that route is compiled in)
    double kbe3, kb, lkb, qo_sum;
#endif
};
constexpr int kDayPreDoubles = sizeof(DayPre) / sizeof(double);

template <class M = MathShared, class CC>
__device__ __forceinline__ void day_forcing(const CC& cc, const DayTab& dt, const MonthTab& mt, double sw_in, double tc,
                                            double pn, DayPre& q) {
    // ---- snow partition, R/splash.point.R:120-128 with frain_func :547-555 ------------------------
    cc_fetch(cc, CCG_SNOW);  // C_ELEV_K, C_LAT_K, C_TT
    const int snowy = snow_class(cc, tc);
    double f_rain;
    if (snowy < 0) {
        f_rain = nan("");  // ifelse(NA, ., .) is NA
    } else if (snowy) {
        const double Tt = cc(C_TT);
        const double Ttm = Tt + (Tt * mt.s1[dt.month]);
        const double x = SPLASH_FDIV(tc - Ttm, mt.trm14[dt.month]);
        double frain;
        if (tc <= Ttm) {
            frain = 5 * (x * x * x) + kD.fr_a * (x * x) + kD.fr_b * x + 0.5;
        } else {
            frain = 5 * (x * x * x) - kD.fr_a * (x * x) + kD.fr_b * x + 0.5;
        }
        if (frain < 0) frain = 0;
        if (frain > 1) frain = 1;
        f_rain = frain;
    } else {
        f_rain = 1;
    }
    q.snowfall = pn * (1 - f_rain);
    q.rain = pn * f_rain;
    q.tc = tc;

    // ---- SOLAR::calculate_daily_fluxes, SOLAR.cpp:129-203 ------------------------------------------
    cc_fetch(cc, CCG_GEOMETRY);  // the six trig constants, C_TAU_O, C_TAU_A, C_INV_TAU_B
    const double a = dt.sd * cc(C_COS_LAT) * cc(C_SIN_S) * cc(C_COS_A) - dt.sd * cc(C_SIN_LAT) * cc(C_COS_S);
    const double b = dt.cd * cc(C_COS_LAT) * cc(C_COS_S) + dt.cd * cc(C_SIN_LAT) * cc(C_SIN_S) * cc(C_COS_A);
    const double c = dt.cd * cc(C_SIN_S) * cc(C_SIN_A);
    const double d = b * b + c * c - a * a;
    double sinfirst;
    if (d < 0) {
        sinfirst = SPLASH_FDIV(a * c, b * b + c * c);
    } else {
        sinfirst = SPLASH_FDIV(a * c + b * sqrt(d), b * b + c * c);
    }
    const double ru = -1 * a + c * sinfirst;
    const double rv = b;
    double hs;
    const double ruv = SPLASH_FDIV(ru, rv);
#if SPLASH_L1_POW
    double sin_hs;
    if (ruv >= 1.0) {
        hs = 180.0;
        sin_hs = SPLASH_SIN_180;
    } else if (ruv <= -1.0) {
        hs = 0.0;
        sin_hs = 0.0;
    } else {
        const double x = -1.0 * ruv;
        hs = SPLASH_TO_DEG(M::acos(x));
        sin_hs = sqrt((1.0 - x) * (1.0 + x));
    }
#else
    if (ruv >= 1.0) {
        hs = 180.0;
    } else if (ruv <= -1.0) {
        hs = 0.0;
    } else {
        hs = -1.0 * ruv;
        hs = f_acos(hs);
        hs = SPLASH_TO_DEG(hs);
    }
    const double sin_hs = f_sin(hs * kpir);
#endif
    double ra_d = kD.k_ra * dt.dr * kD.gsc;
    ra_d *= (ru * hs * kD.pir + rv * sin_hs);
    const double tau_o = cc(C_TAU_O);
    const double r_in = 86400 * sw_in;
    double tau;
    if (isnan(ra_d) || r_in == 0 || ra_d < r_in) {
        tau = tau_o;
    } else {
        tau = SPLASH_FDIV(r_in, ra_d);
    }
#if SPLASH_L1_POW
    double sf = M::exp(kD.sf_exp * M::log(SPLASH_DIV_TAU_B(tau - cc(C_TAU_A))));
#else
    double sf = pow(((tau - cc(C_TAU_A)) / cc(C_TAU_B)), (1 / 0.7410));
#endif
    if (isnan(sf)) {
        sf = 0.0;
    } else if (sf > 1.0) {
        sf = 1.0;
    }
    q.rnl = (kD.rnl_a + kD.rnl_b * sf) * (kD.rnl_A + kD.rnl_c * tc);
    q.ru = ru;
    q.rv = rv;
    q.ruv = ruv;
    q.hs = hs;
    q.sin_hs = sin_hs;
    q.tau = tau;
    q.dr = dt.dr;
    q.r_in = r_in;
    q.rw_den = (kD.k_ra * (ru * kD.pir * hs + rv * sin_hs));
    q.rw_dark = ((sw_in == 0.0) || (hs == 0.0)) ? 1.0 : 0.0;

    // ---- EVAP::calculate_daily_fluxes, EVAP.cpp:100-145 --------------------------------------------
    cc_fetch(cc, CCG_PRESSURE);  // C_PATM, C_PBAR, C_PBARF, C_VISC0, C_INTPERM
    const double patm = cc(C_PATM);
    double s = M::exp(SPLASH_FDIV(tc * kD.ss_a, tc + kD.ss_b));  // sat_slope, :299-301
    s = SPLASH_FDIV(s, (tc + kD.ss_b) * (tc + kD.ss_b));
    s *= kD.ss_k;
    double lv = SPLASH_FDIV(tc + kD.lv_a, tc + kD.lv_a - kD.lv_b);  // enthalpy_vap, :313-315
    lv = lv * lv;
    lv *= 1.91846e6;
    const DensityPoly qd = density_poly(tc);
    const double pw = density_at(qd, cc(C_PBAR));
    const double cp = specific_heat(tc);
    const double g = SPLASH_FDIV(kD.ma * cp * patm, kD.mv * lv);  // psychro, :486
    const double econ = SPLASH_FDIV(s, lv * pw * (s + g));
    // viscosity at tw = max(tc, 0) narrowed to float, :100-105,120,413
    double visc;
    if (tc < 0.0) {
        visc = cc(C_VISC0);  // tw == 0: a function of the cell's pressure only
    } else {
        const float tcf = (float)tc;
        double rho_d;
        if ((double)tcf == tc) {
            rho_d = density_at<true>(qd, cc(C_PBARF));  // same temperature polynomials, float-rounded pressure
        } else {
            rho_d = density_at<true>(density_poly((double)tcf), cc(C_PBARF));
        }
        visc = viscosity_h2o(tcf, rho_d);
    }
    q.s = s;
    q.g = g;
    q.econ = econ;
    q.pw = pw;
    q.eet_k = (1.0e3) * SPLASH_FDIV(s, lv * pw * (s + kD.eet_c * g));  // EVAP.cpp:129-131: eet_d = eet_k * rn_d
    q.rx = (3.6e6) * econ;
    q.ksat_visc = cc(C_INTPERM) * SPLASH_FDIV(pw * kD.grav, visc) * kD.k36;  // SPLASH.cpp:1260
#if SPLASH_L1_RECIP
    q.inv_rw_den = SPLASH_FDIV(1.0, q.rw_den);
    q.inv_rx = SPLASH_FDIV(1.0, q.rx);
    q.inv_econ = SPLASH_FDIV(1.0, econ);
    q.inv_pwk = SPLASH_FDIV(1.0, pw * kkfus);
    q.inv_k24 = SPLASH_FDIV(1.0, q.ksat_visc * 24);
#endif
}

#if SPLASH_L1_RECIP
// The recession / drainage terms of the state half that depend on the day's viscosity and the cell only (DayPre::kbe3,
// kb, lkb, qo_sum), for day_state_fast: computed once per spin-up year by the straggler pool's table kernel.  Kept out of
// day_forcing so that the fused kernels, which never read them, compile exactly as they did without them.
template <class M = MathShared, class CC>
__device__ __forceinline__ void day_forcing_recession(const CC& cc, DayPre& q) {
    {   // the same operations, in the same order, as day_state's sections 5.2.1 / 5.2.2
        const double Ksat_visc = q.ksat_visc, hyd_grad_in = cc(C_TAN_S);
        const double kbe3 = (Ksat_visc * cc(C_BUB) / cc(C_E3));
        const double T_q0 = kbe3 * cc(C_BRQ0);
        const double Q_q0 = T_q0 * hyd_grad_in * cc(C_CQ0);
        const double Q_qs = SPLASH_DIVC_1000(hyd_grad_in * Ksat_visc * 24.0 * cc(C_ACSQS));
        const double z_kb = (Q_q0 - Q_qs) * cc(C_INV_DENKB);
        const double Kb = (fabs(z_kb) < 0x1p-20) ? 1.0 + fma(0.5 * z_kb, z_kb, z_kb) : M::exp(z_kb);
        const double To_uns = kbe3 * cc(C_BRW);
        const double Qo_uns = To_uns * cc(C_CW);
        const double Qo_sat = SPLASH_DIVC_1000(Ksat_visc * 24.0 * cc(C_ACSW));
        q.kbe3 = kbe3;
        q.kb = Kb;
        q.lkb = M::log(Kb);
        q.qo_sum = Qo_sat + Qo_uns;
    }
}
#endif

template <class M = MathShared, class CC>
__device__ __forceinline__ void day_state(const CC& cc, const DayPre& q, CellState& st, DayOut& o) {
    const double wn = st.wn;
    const double tc = q.tc;
    // ---- 00/03. theta_i clamp and supply rate, SPLASH.cpp:984-990, 1042-1048 ----------------------
    const double theta_s = cc(C_THS);
    const double theta_mean = SPLASH_DIV_D1000(wn);
    double theta_i = theta_mean;
    if (theta_i >= theta_s) {
        theta_i = theta_s - kD.k_001;
    } else if (theta_i <= cc(C_THR)) {
        theta_i = cc(C_THR) + kD.k_001;
    }
#if SPLASH_L1_RECIP
    double sw = ((wn - cc(C_RES)) * cc(C_INV_WMR));
#else
    double sw = ((wn - cc(C_RES)) / cc(C_WMR));
#endif
    if (sw < 0.0 || isnan(sw)) {
        sw = 0.0;
    } else if (sw > 1.0) {
        sw = 1.0;
    }
    // ---- 04. snowpack, :1225-1231 ---------------------------------------------------------------
    double nd = st.nd;
    if (q.snowfall > 0.0) {
        nd = 0.0;
    } else {
        nd += 1.0;
    }
    double snow = st.snow + q.snowfall;

    // ---- SOLAR::calculate_daily_fluxes, SOLAR.cpp:208-255 ------------------------------------------
    const double ru = q.ru, rv = q.rv, hs = q.hs, sin_hs = q.sin_hs, rnl = q.rnl;
    const double max_alb_snw = kD.alb_a + (kD.alb_b * snow_age_factor(nd));
    const double sfc = SPLASH_FDIV(snow, 140.0 + snow);
    const double alb_v = kD.alb_sw - kD.alb_c * sw;
    const double alb = alb_v * (1.0 - sfc) + sfc * max_alb_snw;
    double rw;
    if (q.rw_dark != 0.0) {
        rw = (1.0 - alb) * q.tau * q.dr * kD.gsc;
    } else {
#if SPLASH_L1_RECIP
        rw = (1.0 - alb) * (q.r_in) * q.inv_rw_den;
#else
        rw = SPLASH_FDIV((1.0 - alb) * (q.r_in), q.rw_den);
#endif
    }
    double hn;
#if SPLASH_L1_RECIP
    const double inv_rwrv = SPLASH_FDIV(1.0, rw * rv);  // shared by qn and cos_hi
    const double qn = (rnl - rw * ru) * inv_rwrv;
#else
    const double qn = SPLASH_FDIV(rnl - rw * ru, rw * rv);
#endif
#if SPLASH_L1_POW
    double sin_hn;
    if (qn >= 1.0) {
        hn = 0;
        sin_hn = 0.0;
    } else if (qn <= -1.0) {
        hn = 180.0;
        sin_hn = SPLASH_SIN_180;
    } else {
        hn = SPLASH_TO_DEG(M::acos(qn));
        sin_hn = sqrt((1.0 - qn) * (1.0 + qn));
    }
#else
    if (qn >= 1.0) {
        hn = 0;
    } else if (qn <= -1.0) {
        hn = 180.0;
    } else {
        hn = M::acos(qn);
        hn = SPLASH_TO_DEG(hn);
    }
    const double sin_hn = M::sin(hn * kpir);
#endif
    double rn_d = kD.pir * hn * (rw * ru - rnl) + rw * rv * sin_hn;
    rn_d *= kD.k_ra;
    double rnn_d = rw * rv * (sin_hs - sin_hn);
    rnn_d += rw * ru * (hs - hn) * kD.pir;
    rnn_d -= rnl * (kD.k_pi - hn * kD.pir);
    rnn_d *= kD.k_ra;

    // ---- EVAP::calculate_daily_fluxes, EVAP.cpp:124-263 --------------------------------------------
    const double s = q.s, g = q.g, econ = q.econ, pw = q.pw, rx = q.rx;
    const double cn = (1.0e3) * econ * fabs(rnn_d) * kD.k_01;
    const double eet_d = q.eet_k * rn_d;
    const double pet_max = rx * ((rw * (ru + rv)) - rnl);
#if SPLASH_L1_RECIP
    // EF = 1 / (g / (sw s) + 1) = sw s / (g + sw s): one division; sw == 0 gives 0 either way
    const double EF = SPLASH_FDIV(sw * s, g + sw * s);
#else
    const double B_r = SPLASH_FDIV(g, sw * s);
    const double EF = SPLASH_FDIV(1.0, B_r + 1.0);
#endif
    double swp = pet_max * EF;
    if (swp < 0.0 || isnan(swp)) {
        swp = 0.0;
    }
#if SPLASH_L1_RECIP
    const double cos_hi = swp * inv_rwrv * q.inv_rx + rnl * inv_rwrv - q.ruv;
#else
    const double cos_hi = SPLASH_FDIV(swp, rw * rv * rx) + SPLASH_FDIV(rnl, rw * rv) - q.ruv;  // ru/rv: same operands as in day_forcing
#endif
    double hi;
#if SPLASH_L1_POW
    double sin_hi;
    if (cos_hi >= 1.0) {
        hi = 0.0;
        sin_hi = 0.0;
    } else if (cos_hi <= -1.0) {
        hi = 180.0;
        sin_hi = SPLASH_SIN_180;
    } else {
        hi = SPLASH_TO_DEG(M::acos(cos_hi));
        sin_hi = sqrt((1.0 - cos_hi) * (1.0 + cos_hi));
    }
#else
    if (cos_hi >= 1.0) {
        hi = 0.0;
    } else if (cos_hi <= -1.0) {
        hi = 180.0;
    } else {
        hi = M::acos(cos_hi);
        hi = SPLASH_TO_DEG(hi);
    }
    const double sin_hi = M::sin(hi * kpir);
#endif
    double snowmelt_tot;
    if (tc >= 3.0) {
#if SPLASH_L1_RECIP
        snowmelt_tot = cxx_min(snow, (rn_d * q.inv_pwk) * 1000.0);
#else
        snowmelt_tot = cxx_min(snow, SPLASH_FDIV(rn_d, pw * kkfus) * 1000.0);
#endif
    } else {
        snowmelt_tot = 0.0;
    }
    double melt_enrg = SPLASH_DIVC_1000(snowmelt_tot) * pw * kkfus;
    const double AE = rn_d - melt_enrg;
    const double sublimation = cxx_min(snowmelt_tot, (AE * econ) * 1000.0);
#if SPLASH_L1_RECIP
    melt_enrg += SPLASH_DIVC_1000(sublimation) * q.inv_econ;
#else
    melt_enrg += SPLASH_FDIV(SPLASH_DIVC_1000(sublimation), econ);
#endif
    double aet_d = swp * hi * kD.pir;
    aet_d += rx * rw * rv * (sin_hn - sin_hi);
    aet_d += (rx * rw * ru - rx * rnl) * (hn - hi) * kD.pir;
    aet_d *= kD.k_24pi;
#if SPLASH_L1_RECIP
    // Days without melt and without an evaporation integral (polar night): sublimation = (AE*econ)*1000 is negative
    // (deposition) and aet becomes ((sublimation/1000)/econ * econ) * 1000 -- the same operations run backwards and
    // forwards again, which return sublimation exactly for 99.8 % of the values, so that aet == inflow and
    // R = infi - aet (SPLASH.cpp:1283) is exactly 0.  `R > 0` would switch the same-day upslope input on (:1468,
    // a jump of Qt/Ai ~ 1e-3 mm); with reciprocal multiplications the round trip is off by an ulp on 22 % of the
    // days.  Take the round trip's fixed point.
    if (aet_d == 0.0 && snowmelt_tot == 0.0)
        aet_d = 0.0 - sublimation;
    else
#endif
    aet_d -= (melt_enrg * econ * 1000.0);
    if (aet_d < 0.0) {
        aet_d = 0.0;
    }

    // ---- back in SPLASH::run_one_day, SPLASH.cpp:1236-1284 -----------------------------------------
    snow -= snowmelt_tot;
    const double snowmelt = snowmelt_tot - sublimation;
    const double Ksat_visc = q.ksat_visc;
    const double inflow = q.rain + cn + snowmelt;
    // moist_surf(depth, 10, bub, wn, SAT, RES, lambda), :1935-1957
    double surf_moist;
    {
        const double theta_r = cc(C_THR);
#if SPLASH_L1_POW
        // head/bp = (bp/u + 10)/bp = 1/u + 10/bp with u = x^(1/lambda); 1/u = M::exp(-M::log(x)/lambda)
        const double lx = M::log(SPLASH_DIV_DTH(theta_mean - theta_r));
        const double inv_u = M::exp(-(cc(C_ILAM) * lx));
        double head = inv_u + cc(C_TEN_BP);
        // the reference forms bp/u first (:1945), which overflows to -inf once |bp|/u > DBL_MAX (dry soil with a
        // tiny lambda: u = x^(1/lambda) ~ 1e-306); head/bp is then +inf and theta_BC collapses onto theta_r
        if (inv_u > fabs(cc(C_TEN_BP)) * kD.k_ovf) head = INFINITY;
        double hp = M::exp(cc(C_NLAM) * M::log(head));
        // an air-entry pressure of exactly 0 (pedotransfer result of some sandy, gravelly soils) makes the base -inf:
        // pow(-inf, y) is +0 for y < 0, +inf for y > 0 and 1 for y == 0 (C11 F.10.4.4), not NaN
        if (head == -INFINITY) hp = (cc(C_NLAM) < 0.0) ? 0.0 : ((cc(C_NLAM) > 0.0) ? INFINITY : ((cc(C_NLAM) == 0.0) ? 1.0 : hp));
        double theta_BC = cc(C_DTH) * hp + theta_r;
#else
        const double bp = cc(C_BP10);
        const double water_pot_BC = bp / pow((((theta_mean - theta_r) / cc(C_DTH))), cc(C_ILAM));
        const double total_head_BC = water_pot_BC + 10.0;
        double theta_BC = cc(C_DTH) * pow((total_head_BC / bp), cc(C_NLAM)) + theta_r;
#endif
        if (theta_mean < theta_r) {
            theta_BC = theta_r;
        } else if (isnan(theta_BC)) {
            theta_BC = theta_s;
        }
        surf_moist = theta_BC;
    }
    const double theta_m = cxx_max(cc(C_THWMAX), theta_i);
    // inf_GA(bub, surf_moist, Ksat_visc, theta_s, lambda, inflow, 6.0, slop), :1984-2022
    double infi;
    {
        const double P = inflow;
        const double r = SPLASH_DIVC_6(P);
        const double h_f = cc(C_HF);
        const double delta_theta = (theta_s - surf_moist);
        double I = 0.0;
        if (r <= Ksat_visc) {
            I = P;
        } else {
            if (delta_theta <= 0.0) {
                I = Ksat_visc * 6.0;
            } else {
                double tp = SPLASH_FDIV(Ksat_visc * delta_theta * -1.0 * h_f, r * (r - Ksat_visc));
                if (tp <= 0.0 || isnan(tp)) {
                    tp = kD.k_01b;
                }
                const double tp_s = tp / cc(C_COS2_S);
                I = r * tp_s + (Ksat_visc * (6.0 - tp_s) - (h_f * delta_theta * M::log(1 - SPLASH_FDIV(r * tp_s, h_f * delta_theta))));
            }
        }
        if (I > P) {
            I = P;
        }
        infi = I;
    }
    const double ro_h = cxx_max(inflow - infi, 0.0);
    double R = infi - aet_d;
    const bool deep = (cc(C_DEPTH) >= 2.0);
#if SPLASH_L1_POW
    // Kunsat only enters T_uns when depth >= 2 (:1433-1435); below field capacity its power is a cell constant
    double Kunsat = 0.0;
    if (deep) {
        const double kp = (theta_i <= cc(C_THWMAX) || isnan(theta_i)) ? cc(C_KU_WMAX) : M::exp(cc(C_KUEXP) * M::log(theta_m / theta_s));
        Kunsat = Ksat_visc * kp;
    }
#else
    const double Kunsat = Ksat_visc * pow((theta_m / theta_s), cc(C_KUEXP));
#endif
    const double hyd_grad_in = cc(C_TAN_S);
#if SPLASH_L1_RECIP
    const double hyd_grad_z = infi * q.inv_k24 - 1.0;
#else
    const double hyd_grad_z = SPLASH_FDIV(infi, Ksat_visc * 24) - 1.0;
#endif
    const double hyd_grad_out = sqrt((hyd_grad_z * hyd_grad_z) + (hyd_grad_in * hyd_grad_in));

    // ---- 5.2.1 recession constant, :1303-1326 ------------------------------------------------------
    const double kbe3 = (Ksat_visc * cc(C_BUB) / cc(C_E3));
    const double T_q0 = kbe3 * cc(C_BRQ0);
    const double Q_q0 = T_q0 * hyd_grad_in * cc(C_CQ0);
    const double Q_qs = SPLASH_DIVC_1000(hyd_grad_in * Ksat_visc * 24.0 * cc(C_ACSQS));
#if SPLASH_L1_RECIP
    // 5.7 takes log(Kb) back (:1470): on gentle slopes the exponent is ~1e-8 and every bit of Kb counts.  There
    // 1 + z + z^2/2 rounds to the correctly rounded exp(z) (as glibc's exp does) with probability 1 - |z|.
    const double z_kb = (Q_q0 - Q_qs) * cc(C_INV_DENKB);
    const double Kb = (fabs(z_kb) < 0x1p-20) ? 1.0 + fma(0.5 * z_kb, z_kb, z_kb) : M::exp(z_kb);
#else
    const double Kb = M::exp((Q_q0 - Q_qs) / cc(C_DENKB));
#endif
    // ---- 5.2.2 drainage at Wmax, :1346-1360 --------------------------------------------------------
    const double To_uns = kbe3 * cc(C_BRW);
    const double Qo_uns = To_uns * cc(C_CW);
    const double Qo_sat = SPLASH_DIVC_1000(Ksat_visc * 24.0 * cc(C_ACSW));
    const double Qt = (Qo_sat + Qo_uns) * hyd_grad_out;
    // ---- 5.2.3 upslope input of the previous day, :1365-1372 ---------------------------------------
    double q_in_o = 0.0;
    if ((st.td <= 0.0) || (st.qin <= 0.0)) {
        q_in_o = 0.0;
    } else {
        q_in_o = st.qin * Kb;
    }
    // ---- 5.3/5.4 soil moisture and Dunne runoff, :1377-1397 ----------------------------------------
    const double SAT = cc(C_SAT), RES = cc(C_RES);
    double sm = wn + q_in_o + R;
    double ro_d = 0.0;
    if (sm > SAT) {
        ro_d = (sm - SAT);
        sm = SAT;
        if (R > 0) {
            R -= ro_d;
        }
    } else if (sm < RES) {
        sm = RES;
        ro_d = 0.0;
    }
#if SPLASH_L1_RECIP
#define SPLASH_DIV_AI(x) ((x) * cc(C_INV_AI))
#else
#define SPLASH_DIV_AI(x) ((x) / Ai)
#endif
    // ---- 5.6 transmittance after recharge, :1406-1457 ----------------------------------------------
    const double Ai = cc(C_AI);
    Transm tr = column_transmittance<M>(cc, sm, Ksat_visc);
    double T;
    {
        double T_uns = tr.t_uns;
        double T_sat;
        if (deep) {
            T_uns += Kunsat * 24.0;
            T_sat = Ksat_visc * 24.0 * SPLASH_DIV_AI(tr.acs_out + Ai);
        } else {
            T_sat = Ksat_visc * 24.0 * SPLASH_DIV_AI(tr.acs_out);
        }
        T = (T_sat + T_uns) * hyd_grad_out;
    }
    const double Q = SPLASH_DIVC_1000(T * Ai);
    // ---- 5.7 same-day upslope input, :1465-1483 ----------------------------------------------------
    double t_drain = 0.0;
    double q_in_f = 0.0;
    const double td = st.td - 1.0;
    if ((R > 0.0) && (sm > cc(C_WMAX))) {
        const double lkb = M::log(Kb);
        const double Au = cc(C_AU);
        t_drain = SPLASH_FDIV(-1.0 * M::log(1.0 - (lkb * SPLASH_FDIV(Au * R, Q))), lkb);
        q_in_f = SPLASH_DIV_AI(Qt - Au * R * lkb);
    }
    if (q_in_f < 0.0 || isnan(q_in_f)) {
        q_in_f = 0.0;
    }
    const double tdrain_out = cxx_max((td + t_drain) / 2, 0.0);
    // ---- 5.8 update soil moisture, :1488-1506 ------------------------------------------------------
    const double sm_before = sm;
    sm += (q_in_f);
    if (sm > SAT) {
        ro_d += (sm - SAT);
        sm = SAT;
    } else if (sm < RES) {
        sm = RES;
    }
    const double ro = ro_d + ro_h;
    // ---- 5.6' transmittance after upslope input, :1511-1547.  When sm did not move the block
    //      recomputes exactly the values of 5.6, so they are reused (bit-identical). -----------------
    if (!(sm == sm_before)) {
        tr = column_transmittance<M>(cc, sm, Ksat_visc);
    }
    {
        const double T_sat = Ksat_visc * 24.0 * SPLASH_DIV_AI(tr.acs_out);
        T = (T_sat + tr.t_uns) * hyd_grad_out;
    }
    // ---- 5.8' drain, :1552-1567 --------------------------------------------------------------------
    sm -= (T);
    if (sm > SAT) {
        sm = SAT;
    } else if (sm < RES) {
        sm = RES;
    }
    // ---- 5.9 next-day input and outputs, :1573-1583, 1898-1908 -------------------------------------
    st.wn = sm;
    st.snow = snow;
    st.qin = cxx_max(cxx_max(q_in_o, q_in_f), 0.0);
    st.td = tdrain_out;
    st.nd = nd;
    o.ro = ro;
    o.pet = eet_d;
    o.aet = aet_d;
    o.cond = cn;
    o.bflow = T;
    o.netr = SPLASH_DIVC_1E6(rn_d);
#undef SPLASH_DIV_AI
}

// ------------------------------------------------------------------------------------------------
// The branch-light state half (level 1 only).
//
// day_state above is ~100 basic blocks: every transcendental and every guarded division carries its own range check
// and fallback branch, and every `if` of the reference is a branch.  A scheduler's warps then each run ONE dependent
// FP64 chain (ncu r02: 3.6 cycles of fixed-latency wait per issued instruction at four warps per scheduler; for the
// straggler chain, one warp per scheduler, every cycle of it is exposed).  day_state_fast computes the same values with
// the same operations, organised so that independent chains share a basic block and overlap:
//   * the fast-range bodies of exp/log/acos/fdiv (splash_math.cuh) without their guards; every guard is and-ed into
//     one flag `ok`, gated by the condition under which the guarded value is actually used;
//   * the reference's two-way and three-way `if`s as selects over both results;
//   * the blocks that are rare and long stay branches and keep the guarded primitives: infiltration excess (inf_GA),
//     the clamped-water-table tail of the transmittance, the second transmittance when the upslope input moved sm.
// When `ok` comes out false (a NaN, a zero denominator, an argument outside a fast range: the reference's failsafe
// territory) nothing has been written and the caller runs day_state on the same inputs.  Selected paths perform
// day_state's operations in day_state's order, so both routes give the same bits (tools/emul_snapshot.py, the host
// build with -DSPLASH_FAST_STATE=0/1; tests/test_level1_host_cpu.py).
// ------------------------------------------------------------------------------------------------
#if SPLASH_L1_POW && SPLASH_L1_RECIP
#ifdef SPLASH_HOST_EMUL
// host build only: how often each guard sends a day to the guarded path (tools/fast_state_stats.py)
extern "C" long long g_fast_guard_trips[32];
extern "C" long long g_fast_days;
#define SPLASH_GUARD(k, cond)                                  \
    do {                                                       \
        if (!(cond)) {                                         \
            ok = false;                                        \
            __atomic_fetch_add(&g_fast_guard_trips[k], 1LL, __ATOMIC_RELAXED); \
        }                                                      \
    } while (0)
#else
#define SPLASH_GUARD(k, cond) ok = ok & (cond)  // (conditions are written with | and &: no short-circuit branches)
#endif

template <class M, class CC>
__device__ __forceinline__ Transm column_transmittance_fast(const CC& cc, double sm, double kbe3, bool& ok_io) {
    bool ok = ok_io;
    const double bub = cc(C_BUB);
    const double e3 = cc(C_E3);
    const double depth = cc(C_DEPTH);
    Transm r;
    const double theta_i = SPLASH_DIV_D1000(sm);
    const double x = SPLASH_DIV_DTH(theta_i - cc(C_THR));
    const double a = cc(C_ILAM) * fm::log_body(x);
    const double e3a = e3 * a;
    // Two regimes of a column at (or a rounding error below) its residual moisture are closed forms of the guarded
    // route, which reaches them through its IEEE fallbacks every day the soil stays that dry:
    //   negx  x < 0: log x, psi_m, wtd, both powers and dr are NaN -> wtd takes the `wtd < 0 || isnan` clamp (0.01)
    //         and T_uns the `< 0 || isnan` failsafe (0)
    //   dry   x == 0, or x^(1/lambda) underflows to 0 (a <= -746): psi_m = bub / 0 = -inf, wtd = +inf clamps to the
    //         depth, the first power is exp(e3 a) = 0 and the second is built on (-inf) / (-inf) = NaN, so dr is
    //         NaN and T_uns again the failsafe's 0.  Needs bub < 0, e3 > 0 and 1/lambda > 0, which holds for every
    //         soil the pedotransfer functions return but is checked (a zero air-entry pressure goes the guarded way).
    const bool negx = (x < 0.0);
    //   dry   also with x^(1/lambda) = exp(a) below 2^-930 but not 0 (a <= -645): psi_m = bub / exp(a) is finite but so
    //         large that psi_m + 1000 wtd == psi_m, the ratio of the two bases is exactly 1, dr = -(r1 * 0) = -0 and
    //         T_uns = kbe3 * (-0) * CT = +0 for kbe3 < 0 < CT -- the failsafe's value again (and -inf / -inf = NaN if
    //         psi_m overflows: same result), wtd the depth as before
    const bool regular = (bub < -1e-100) & (e3 > 0.0) & (cc(C_ILAM) > 0.0) & (cc(C_ILAM) < INFINITY) & (depth < INFINITY) &
                         (kbe3 < 0.0) & (kbe3 > -INFINITY) & (cc(C_CT) > 0.0) & (cc(C_CT) < INFINITY);
    const bool dry = regular & ((x == 0.0) | (fm::log_ok(x) & (a <= -645.0)));
    const bool closed = negx | dry;
    SPLASH_GUARD(16, closed | fm::log_ok(x));
    SPLASH_GUARD(17, closed | fm::exp_ok(a));
    const double ea = fm::exp_body(a);
    SPLASH_GUARD(18, closed | fm::fdiv_ok(ea));
    const double psi_m = bub * fm::rcp(ea);
    const double wtd0 = SPLASH_DIV_1000(bub - psi_m);
    const bool below = (wtd0 < 0.0) | isnan(wtd0);
    const bool above = !below & (wtd0 > depth);
    const bool clamped = below | above;
    const double wtd = negx ? kD.k_01b : (dry ? depth : (below ? kD.k_01b : (above ? depth : wtd0)));
    r.acs_out = (depth - wtd) * cc(C_SIDOCT) * cc(C_CELLOUT);
    SPLASH_GUARD(19, closed | fm::exp_ok(e3a));
    const double r1 = fm::exp_body(e3a);
    const double den = psi_m + (wtd * 1000.0);
    // water table inside the column: the second base is 1 up to rounding noise, first-order expansion
    const double qq = bub * fm::rcp(den);
    const double qm1 = qq - 1.0;
    double dr = r1 - (1.0 + e3 * qm1);
    const bool expansion = fm::fdiv_ok(den) & (fabs(qm1) < kD.k_1em7);
    if ((clamped | !expansion) & !closed) {  // the rare, long cases as in column_transmittance_core
        if (clamped) {
            const double t = e3 * M::log(SPLASH_FDIV(psi_m, den));
            const double em1 = (fabs(t) < kD.k_1em5) ? t * (1.0 + 0.5 * t) : M::exp(t) - 1.0;
            dr = -(r1 * em1);
        } else {
            const double q = SPLASH_FDIV(bub, den);
            const double q1 = q - 1.0;
            const double r2 = (fabs(q1) < kD.k_1em7) ? (1.0 + e3 * q1) : M::exp(e3 * M::log(q));
            dr = r1 - r2;
        }
    }
    double t_uns = kbe3 * dr;
    t_uns *= cc(C_CT);
    r.t_uns = (closed | (t_uns < 0.0) | isnan(t_uns)) ? 0.0 : t_uns;
    ok_io = ok;
    return r;
}

// returns false (st, o untouched) when the day needs the guarded path
template <class M, class CC>
__device__ __forceinline__ bool day_state_fast(const CC& cc, const DayPre& q, CellState& st, DayOut& o) {
    bool ok = true;
    const double wn = st.wn;
    const double tc = q.tc;
    const double Ksat_visc = q.ksat_visc;
    const double theta_s = cc(C_THS), theta_r = cc(C_THR);
    const double theta_mean = SPLASH_DIV_D1000(wn);
    const double theta_i =
        (theta_mean >= theta_s) ? theta_s - kD.k_001 : ((theta_mean <= theta_r) ? theta_r + kD.k_001 : theta_mean);
    // the IEEE division of the day (fm::div_body: the compiler's own sequence without its fix-up branch)
    const double theta_m = cxx_max(cc(C_THWMAX), theta_i);
    const double ku_ratio = fm::div_body(theta_m, theta_s);
    const double kbe3 = q.kbe3;
    double sw = ((wn - cc(C_RES)) * cc(C_INV_WMR));
    sw = ((sw < 0.0) | isnan(sw)) ? 0.0 : ((sw > 1.0) ? 1.0 : sw);
    const double nd = (q.snowfall > 0.0) ? 0.0 : st.nd + 1.0;
    double snow = st.snow + q.snowfall;

    // ---- chain A: albedo -> shortwave -> net radiation cross-over hour angle ---------------------------------
    const double ru = q.ru, rv = q.rv, hs = q.hs, sin_hs = q.sin_hs, rnl = q.rnl;
    const int ndi = (int)nd;
    SPLASH_GUARD(0, (nd >= 0.0) & ((double)ndi == nd));  // else: snow_age_factor's formula path
    const double saf = (ndi < kSnowAgeTab) ? g_snow_age_tab[ndi & (kSnowAgeTab - 1)] : 0.0;  // exp(-0.895 nd) == 0 beyond
    const double max_alb_snw = kD.alb_a + (kD.alb_b * saf);
    const double d_sfc = 140.0 + snow;
    SPLASH_GUARD(1, fm::fdiv_ok(d_sfc));
    const double sfc = snow * fm::rcp(d_sfc);
    const double alb_v = kD.alb_sw - kD.alb_c * sw;
    const double alb = alb_v * (1.0 - sfc) + sfc * max_alb_snw;
    const double rw = (q.rw_dark != 0.0) ? (1.0 - alb) * q.tau * q.dr * kD.gsc : (1.0 - alb) * (q.r_in) * q.inv_rw_den;
    const double rwrv = rw * rv;
    SPLASH_GUARD(2, fm::fdiv_ok(rwrv));
    const double inv_rwrv = 1.0 * fm::rcp(rwrv);
    const double qn = (rnl - rw * ru) * inv_rwrv;
    const bool qn_hi = (qn >= 1.0), qn_lo = (qn <= -1.0);
    SPLASH_GUARD(3, qn_hi | qn_lo | fm::acos_ok(qn));
    // (every arm of a select is a value computed beforehand: `c ? a : f(x)` would be a branch around f)
    const double hn_mid = SPLASH_TO_DEG(fm::acos_body(qn));
    const double sq_hn = (1.0 - qn) * (1.0 + qn);
    const double sin_hn_mid = fm::sqrt_body(sq_hn);
    SPLASH_GUARD(15, qn_hi | qn_lo | fm::sqrt_ok(sq_hn));
    const double hn = qn_hi ? 0.0 : (qn_lo ? 180.0 : hn_mid);
    const double sin_hn = qn_hi ? 0.0 : (qn_lo ? SPLASH_SIN_180 : sin_hn_mid);
    double rn_d = kD.pir * hn * (rw * ru - rnl) + rw * rv * sin_hn;
    rn_d *= kD.k_ra;
    double rnn_d = rw * rv * (sin_hs - sin_hn);
    rnn_d += rw * ru * (hs - hn) * kD.pir;
    rnn_d -= rnl * (kD.k_pi - hn * kD.pir);
    rnn_d *= kD.k_ra;
    const double s = q.s, g = q.g, econ = q.econ, pw = q.pw, rx = q.rx;
    const double cn = (1.0e3) * econ * fabs(rnn_d) * kD.k_01;
    const double eet_d = q.eet_k * rn_d;
    const double pet_max = rx * ((rw * (ru + rv)) - rnl);
    const double ef_den = g + sw * s;
    SPLASH_GUARD(4, fm::fdiv_ok(ef_den));
    const double EF = (sw * s) * fm::rcp(ef_den);
    double swp = pet_max * EF;
    swp = ((swp < 0.0) | isnan(swp)) ? 0.0 : swp;
    const double cos_hi = swp * inv_rwrv * q.inv_rx + rnl * inv_rwrv - q.ruv;
    const bool ch_hi = (cos_hi >= 1.0), ch_lo = (cos_hi <= -1.0);
    SPLASH_GUARD(5, ch_hi | ch_lo | fm::acos_ok(cos_hi));
    const double hi_mid = SPLASH_TO_DEG(fm::acos_body(cos_hi));
    const double sq_hi = (1.0 - cos_hi) * (1.0 + cos_hi);
    const double sin_hi_mid = fm::sqrt_body(sq_hi);
    SPLASH_GUARD(21, ch_hi | ch_lo | fm::sqrt_ok(sq_hi));
    const double hi = ch_hi ? 0.0 : (ch_lo ? 180.0 : hi_mid);
    const double sin_hi = ch_hi ? 0.0 : (ch_lo ? SPLASH_SIN_180 : sin_hi_mid);
    const double melt_cap = cxx_min(snow, (rn_d * q.inv_pwk) * 1000.0);
    const double snowmelt_tot = (tc >= 3.0) ? melt_cap : 0.0;
    double melt_enrg = SPLASH_DIVC_1000(snowmelt_tot) * pw * kkfus;
    const double AE = rn_d - melt_enrg;
    const double sublimation = cxx_min(snowmelt_tot, (AE * econ) * 1000.0);
    melt_enrg += SPLASH_DIVC_1000(sublimation) * q.inv_econ;
    double aet_d = swp * hi * kD.pir;
    aet_d += rx * rw * rv * (sin_hn - sin_hi);
    aet_d += (rx * rw * ru - rx * rnl) * (hn - hi) * kD.pir;
    aet_d *= kD.k_24pi;
    const double aet_fix = 0.0 - sublimation, aet_gen = aet_d - (melt_enrg * econ * 1000.0);
    aet_d = ((aet_d == 0.0) & (snowmelt_tot == 0.0)) ? aet_fix : aet_gen;
    aet_d = (aet_d < 0.0) ? 0.0 : aet_d;
    snow -= snowmelt_tot;
    const double snowmelt = snowmelt_tot - sublimation;
    const double inflow = q.rain + cn + snowmelt;

    // ---- chain B: moist_surf (two logs, two exps of the relative saturation) ---------------------------------
    double surf_moist;
    {
        const double xms = SPLASH_DIV_DTH(theta_mean - theta_r);
        const bool below = (theta_mean < theta_r);  // the result is theta_r whatever the powers give
        const double lx = fm::log_body(xms);
        const double a1 = -(cc(C_ILAM) * lx);
        const double inv_u = fm::exp_body(a1);
        double head = inv_u + cc(C_TEN_BP);
        head = (inv_u > fabs(cc(C_TEN_BP)) * kD.k_ovf) ? INFINITY : head;
        const double a2 = cc(C_NLAM) * fm::log_body(head);
        const double hp = fm::exp_body(a2);
        // a negative head (|10 / bp| > 1/u: a coarse soil near saturation) makes log, the power and theta_BC NaN, which the
        // reference's failsafe turns into theta_s
        const bool neg_head = (head < 0.0) & (head > -INFINITY);
        // at the residual moisture (x == 0) or with 1/u = exp(a1) overflowing (a1 >= 710) the head is +inf and
        // (head/bp)^(-lambda) = exp(-lambda * inf) = 0: theta_BC = DTH * 0 + theta_r (for lambda > 0, 1/lambda > 0)
        const bool inf_head = ((xms == 0.0) | (fm::log_ok(xms) & (a1 >= 710.0))) & (cc(C_ILAM) > 0.0) & (cc(C_NLAM) < 0.0) &
                              (cc(C_NLAM) > -INFINITY) & (fabs(cc(C_DTH)) < INFINITY);
        SPLASH_GUARD(6, below | inf_head | (fm::log_ok(xms) & fm::exp_ok(a1)));
        SPLASH_GUARD(7, below | inf_head | neg_head | fm::log_ok(head));  // (head == 0, +-inf: guarded path)
        SPLASH_GUARD(12, below | inf_head | !fm::log_ok(head) | fm::exp_ok(a2));
        const double theta_BC = cc(C_DTH) * (inf_head ? 0.0 : hp) + theta_r;
        surf_moist = below ? theta_r : ((!inf_head & (neg_head | isnan(theta_BC))) ? theta_s : theta_BC);
    }

    // ---- chain C: Kunsat above field capacity (deep columns) -------------------------------------------------
    const bool deep = (cc(C_DEPTH) >= 2.0);
    const bool ku_const = (theta_i <= cc(C_THWMAX)) | isnan(theta_i);
    const double ku_l = cc(C_KUEXP) * fm::log_body(ku_ratio);
    SPLASH_GUARD(8, !deep | ku_const | (fm::div_ok(theta_m, theta_s) & fm::log_ok(ku_ratio) & fm::exp_ok(ku_l)));
    const double kp_pow = fm::exp_body(ku_l);
    const double kp = ku_const ? cc(C_KU_WMAX) : kp_pow;
    const double Kunsat = deep ? Ksat_visc * kp : 0.0;

    // ---- recession constant and drainage at Wmax: forcing and constants only, computed by day_forcing --------------
    const double hyd_grad_in = cc(C_TAN_S);
    const double Kb = q.kb, lkb = q.lkb;
    // flat cells: Kb == 1, log Kb == 0; soils with a vanishing air-entry pressure: Kb == 0 or +inf, log Kb == -+inf
    const bool kb_sat = (Kb == 0.0) | (Kb == INFINITY);

    // ---- inf_GA, SPLASH.cpp:1984-2022: the infiltration-excess case stays a branch ---------------------------
    double infi;
    {
        const double P = inflow;
        const double r = SPLASH_DIVC_6(P);
        const double h_f = cc(C_HF);
        const double delta_theta = (theta_s - surf_moist);
        double I = (r <= Ksat_visc) ? P : Ksat_visc * 6.0;
        if (!(r <= Ksat_visc) && !(delta_theta <= 0.0)) {
            double tp = SPLASH_FDIV(Ksat_visc * delta_theta * -1.0 * h_f, r * (r - Ksat_visc));
            if (tp <= 0.0 || isnan(tp)) {
                tp = kD.k_01b;
            }
            const double tp_s = tp / cc(C_COS2_S);
            I = r * tp_s + (Ksat_visc * (6.0 - tp_s) - (h_f * delta_theta * M::log(1 - SPLASH_FDIV(r * tp_s, h_f * delta_theta))));
        }
        infi = (I > P) ? P : I;
    }
    const double ro_h = cxx_max(inflow - infi, 0.0);
    double R = infi - aet_d;
    const double hyd_grad_z = infi * q.inv_k24 - 1.0;
    const double hg2 = (hyd_grad_z * hyd_grad_z) + (hyd_grad_in * hyd_grad_in);
    SPLASH_GUARD(22, fm::sqrt_ok(hg2));
    const double hyd_grad_out = fm::sqrt_body(hg2);
    const double Qt = q.qo_sum * hyd_grad_out;
    const double qin_kb = st.qin * Kb;
    const double q_in_o = ((st.td <= 0.0) | (st.qin <= 0.0)) ? 0.0 : qin_kb;
    const double SAT = cc(C_SAT), RES = cc(C_RES);
    double sm = wn + q_in_o + R;
    const bool over = (sm > SAT);
    const double excess = sm - SAT;
    double ro_d = over ? excess : 0.0;
    const double R_less = R - ro_d;
    R = (over & (R > 0)) ? R_less : R;
    sm = over ? SAT : ((sm < RES) ? RES : sm);
    const double Ai = cc(C_AI);
    Transm tr = column_transmittance_fast<M>(cc, sm, kbe3, ok);
    double T;
    {
        const double T_uns = deep ? tr.t_uns + Kunsat * 24.0 : tr.t_uns;
        const double T_sat = Ksat_visc * 24.0 * ((deep ? tr.acs_out + Ai : tr.acs_out) * cc(C_INV_AI));
        T = (T_sat + T_uns) * hyd_grad_out;
    }
    const double Q = SPLASH_DIVC_1000(T * Ai);
    // ---- 5.7 same-day upslope input, :1465-1483 --------------------------------------------------------------
    const double td = st.td - 1.0;
    const bool drain = (R > 0.0) & (sm > cc(C_WMAX));
    const double AuR = cc(C_AU) * R;
    const double arg = 1.0 - (lkb * (AuR * fm::rcp(Q)));
    // flat cells: Kb == 1, log Kb == 0 and t_drain = -log(1 - 0 * x) / 0 is NaN whatever x is (0/0, or NaN/0); with
    // log Kb == +-inf the logarithm's argument is +-inf or NaN and t_drain = (+-inf or NaN) / +-inf is NaN as well
    const bool lkb_zero = (lkb == 0.0) | kb_sat;
    // no outflow at all (Q == +0: a column whose transmittance is the failsafe's 0): Au R / 0 = +inf; for lkb < 0 the
    // argument of the logarithm is 1 - lkb * inf = +inf and t_drain = (-inf) / lkb = +inf, for lkb > 0 it is -inf and
    // the logarithm, hence t_drain, NaN
    const bool q_zero = (__double_as_longlong(Q) == 0LL) & (AuR > 0.0) & (AuR < INFINITY) & fm::fdiv_ok(lkb);
    // a negative argument gives log = NaN and t_drain = NaN (lkb finite)
    const bool arg_neg = (arg < 0.0) & fm::fdiv_ok(Q) & fm::fdiv_ok(lkb);
    SPLASH_GUARD(10, !drain | ((fm::log_ok(Kb) | kb_sat) & (lkb_zero | q_zero | fm::fdiv_ok(Q))));  // (Kb NaN: guarded route)
    SPLASH_GUARD(11, !drain | lkb_zero | q_zero | arg_neg | (fm::log_ok(arg) & fm::fdiv_ok(lkb)));
    const double t_drain_v = (-1.0 * fm::log_body(arg)) * fm::rcp(lkb);
    const double t_drain = drain ? ((lkb_zero | arg_neg | (q_zero & (lkb > 0.0))) ? nan("") : (q_zero ? INFINITY : t_drain_v)) : 0.0;
    const double q_in_f_v = (Qt - AuR * lkb) * cc(C_INV_AI);
    double q_in_f = drain ? q_in_f_v : 0.0;
    q_in_f = ((q_in_f < 0.0) | isnan(q_in_f)) ? 0.0 : q_in_f;
    const double tdrain_out = cxx_max((td + t_drain) / 2, 0.0);
    // ---- 5.8 update soil moisture, :1488-1506 ----------------------------------------------------------------
    const double sm_before = sm;
    sm += (q_in_f);
    const bool over2 = (sm > SAT);
    const double ro_d2 = ro_d + (sm - SAT);
    ro_d = over2 ? ro_d2 : ro_d;
    sm = over2 ? SAT : ((sm < RES) ? RES : sm);
    const double ro = ro_d + ro_h;
    if (!(sm == sm_before)) {
        tr = column_transmittance_fast<M>(cc, sm, kbe3, ok);
    }
    {
        const double T_sat = Ksat_visc * 24.0 * (tr.acs_out * cc(C_INV_AI));
        T = (T_sat + tr.t_uns) * hyd_grad_out;
    }
    sm -= (T);
    sm = (sm > SAT) ? SAT : ((sm < RES) ? RES : sm);
#ifdef SPLASH_HOST_EMUL
    __atomic_fetch_add(&g_fast_days, 1LL, __ATOMIC_RELAXED);
#endif
    if (!ok) return false;
    st.wn = sm;
    st.snow = snow;
    st.qin = cxx_max(cxx_max(q_in_o, q_in_f), 0.0);
    st.td = tdrain_out;
    st.nd = nd;
    o.ro = ro;
    o.pet = eet_d;
    o.aet = aet_d;
    o.cond = cn;
    o.bflow = T;
    o.netr = SPLASH_DIVC_1E6(rn_d);
    return true;
}
#undef SPLASH_GUARD

// the state half as the kernels call it: the branch-light route when `try_fast`, and the guarded route (one inline
// copy behind it: no call, the day's inputs stay in their registers) for the days it declines.  Returns whether the
// branch-light route took the day.
template <class M, class CC>
__device__ __forceinline__ bool day_state_auto(const CC& cc, const DayPre& q, CellState& st, DayOut& o, bool try_fast = true) {
    bool done = false;
    if (try_fast) done = day_state_fast<M>(cc, q, st, o);
    if (!done) day_state<M>(cc, q, st, o);
    return done;
}
#else
template <class M, class CC>
__device__ __forceinline__ bool day_state_auto(const CC& cc, const DayPre& q, CellState& st, DayOut& o, bool try_fast = true) {
    day_state<M>(cc, q, st, o);
    return false;
}
#endif

//   st     state in/out;  o  fluxes of the day;  rain_out / snowfall_out  the partitioned precipitation
//   (for the aridity index and the occurrence flags)
// The uniform kernels expand the transcendentals in place, as the chain kernel does (measured +6 % over the shared
// out-of-line copies once the literals moved to constant memory: no argument shuffling, no call / return).

template <class CC>
__device__ __forceinline__ void splash_day(const CC& cc, const DayTab& dt, const MonthTab& mt, double sw_in, double tc,
                                           double pn, CellState& st, DayOut& o, double& rain_out,
                                           double& snowfall_out) {
    DayPre q;
    day_forcing<MathInline>(cc, dt, mt, sw_in, tc, pn, q);
    rain_out = q.rain;
    snowfall_out = q.snowfall;
#if SPLASH_FAST_STATE
    day_forcing_recession<MathInline>(cc, q);
    day_state_auto<MathInline>(cc, q, st, o);
#else
    day_state<MathInline>(cc, q, st, o);
#endif
}

// ------------------------------------------------------------------------------------------------
// Terms of run_one_day that depend on `cellout` (SPLASH.cpp:1305, 1319, 1420, 1426).
// ------------------------------------------------------------------------------------------------
template <class CC>
__device__ __forceinline__ void lateral_consts(CC& cc, double cellout) {
    const double sid_oct = cc(C_SIDOCT);
    cc(C_CELLOUT) = cellout;
    cc(C_CQ0) = ((24.0 * sid_oct * cellout) / (1.0e6));
    cc(C_ACSQS) = (cc(C_DEPTH)) * sid_oct * cellout;
    cc(C_CT) = ((24.0 * cellout * sid_oct) / (1000.0 * cc(C_AI)));
}

// ------------------------------------------------------------------------------------------------
// One-shot per-cell setup: pedotransfer functions, soil_info, and every per-cell invariant of the
// day step.  Inputs as in splash_grid_in (raw user values).
// ------------------------------------------------------------------------------------------------
struct CellInputs {
    double lat, elev, slop, asp, resolution;
    double sand, clay, om, gravel, bd, depth;
    double au, cellin, cellout;
};

struct CellDiag {
    double sat, wp, fc, ksat, lambda, depth, bub, res, wmax_r;
};

// soil_hydro(sand, clay, OM, fgravel, bd), R/splash.point.R:232-416: the pedotransfer functions.  Shared by
// the per-cell setup of the hot path and by the unSWC diagnostics (which call it with fgravel = 0).
struct SoilHydro {
    double sat, fc, wp, res_frac, ksat, coef_A, coef_B, theta_c, bubbling_p;
};

__device__ __forceinline__ SoilHydro soil_hydro(double sand, double clay, double om, double gravel, double bd_in) {
    // ---- R/splash.point.R:261-380, 410 -------------------------------------------------------------
    const double fsand = sand / 100;
    const double fclay = clay / 100;
    const double fOM = om / 100;
    const double fgravel = gravel / 100;
    const double dp = 1 / ((fOM / 1.3) + ((1 - fOM) / 2.65));
    double bd = bd_in;
    if (isnan(bd)) {
        bd = (1.5 + (dp - 1.5 - 1.10 * (1 - fclay)) * (1 - exp(-0.022 * 30.0))) / (1 + 6.27 * fOM);
    }
    if (bd < 0.81) bd = 0.81;
    double sat = 1 - (bd / dp);
    const double sq_clay = sqrt(fclay);  // fclay^0.5
    double fc = (sat / bd) * (0.4760944 + (0.9402962 - 0.4760944) * sq_clay) *
                exp(-1 * (0.05472678 * fsand - 0.01 * fOM) / (sat / bd));
    const double wp_Ball = fc * (0.2018522 + (0.7809203 - 0.2018522) * sq_clay);
    double wp = -2.464e-05 * sand + 3.650e-03 * clay + 8.680e-03 * om + 9.393e-03 * bd;
    if (!isnan(wp) && wp >= fc) wp = wp_Ball;
    const double coef_B = (log(1500.0) - log(33.0)) / (log(fc) - log(wp));
    const double coef_A = exp(log(33.0) + coef_B * log(fc));
    const double coef_lambda = 1 / coef_B;
    const double coeff_c = 1000.0 / (997 * 9.80665);
    const double theta_c = pow((coeff_c * coef_A / 2.0), (1 / (1 + coef_B)));
    double theta_r0 = (0.0285 + 0.00336 * (clay)) * bd;
    if (!isnan(theta_r0) && theta_r0 > wp) theta_r0 = wp;
    sat = sat * (1 - fgravel);
    fc = fc * (1 - fgravel);
    wp = wp * (1 - fgravel);
    const double ksat = 857.48454 / (1 + exp(-2.70927 * fsand + 3.62264 * bd + 7.33398 * fclay + -8.11795 * (sat - fc) +
                                            18.75552 * fOM + 1.03319 * coef_lambda));
    const double m33i = 0.278 * fsand + 0.034 * fclay + 0.022 * fOM - 0.018 * (fsand * fOM) - 0.027 * (fclay * fOM) -
                        0.584 * (fsand * fclay) + 0.078;
    const double m33 = m33i + (0.636 * m33i - 0.107);
    const double bub_init = -21.6 * fsand - 27.93 * fclay - 81.97 * m33 + 71.12 * (fsand * m33) + 8.29 * (fclay * m33) +
                            14.05 * (fsand * fclay) + 27.16;
    double bubbling_p = bub_init + (0.02 * (bub_init * bub_init) - 0.113 * bub_init - 0.7);
    bubbling_p = bubbling_p * -101.97162129779;
    if (!isnan(bubbling_p) && bubbling_p > 0) bubbling_p = coef_A * -101.97162129779;
    const double res_frac = theta_r0 * (1 - fgravel);

    SoilHydro h;
    h.sat = sat;
    h.fc = fc;
    h.wp = wp;
    h.res_frac = res_frac;
    h.ksat = ksat;
    h.coef_A = coef_A;
    h.coef_B = coef_B;
    h.theta_c = theta_c;
    h.bubbling_p = bubbling_p;
    return h;
}

template <class CC>
__device__ __forceinline__ void cell_setup(CC& cc, const CellInputs& in, CellDiag& dg) {
    const SoilHydro sh = soil_hydro(in.sand, in.clay, in.om, in.gravel, in.bd);
    const double sat = sh.sat, fc = sh.fc, wp = sh.wp, res_frac = sh.res_frac, ksat = sh.ksat, coef_B = sh.coef_B,
                 theta_c = sh.theta_c, bubbling_p = sh.bubbling_p;

    // ---- soil_info, R/splash.point.R:97-115 --------------------------------------------------------
    const double depth = in.depth;
    const double SAT = sat * depth * 1000;
    const double WP = wp * depth * 1000;
    const double FC = fc * depth * 1000;
    const double RES = res_frac * depth * 1000;
    const double Wmax_R = theta_c * depth * 1000;
    const double lambda = 1 / coef_B;
    const double bub = bubbling_p;
    const double Ai = in.resolution * in.resolution;
    dg.sat = SAT;
    dg.wp = WP;
    dg.fc = FC;
    dg.ksat = ksat;
    dg.lambda = lambda;
    dg.depth = depth;
    dg.bub = bub;
    dg.res = RES;
    dg.wmax_r = Wmax_R;

    // ---- snow partition and geometry ---------------------------------------------------------------
    cc(C_ELEV_K) = in.elev * 0.0004596581;
    cc(C_LAT_K) = fabs(in.lat) * 0.0110592101;
    const double asp = in.asp - 180;  // R/splash.point.R:131
    cc(C_COS_LAT) = cos(in.lat * kpir);
    cc(C_SIN_LAT) = sin(in.lat * kpir);
    cc(C_SIN_S) = sin(in.slop * kpir);
    const double cos_s = cos(in.slop * kpir);
    cc(C_COS_S) = cos_s;
    cc(C_COS_A) = cos(asp * kpir);
    cc(C_SIN_A) = sin(asp * kpir);
    cc(C_TAN_S) = tan(in.slop * kpir);
    cc(C_COS2_S) = cos_s * cos_s;
    // ---- atmosphere: SOLAR.cpp:170,197; EVAP.cpp:331-334 -------------------------------------------
    const double tau_o = (kc + kd) * (1.0 + (2.67e-5) * in.elev);
    cc(C_TAU_O) = tau_o;
    cc(C_TAU_A) = tau_o * 0.1898;
    cc(C_TAU_B) = (tau_o * (1 - 0.1898));
    const double ep = (kG * kMa) / (kR * kL);
    double patm = (1.0 - in.elev * kL / kTo);
    patm = pow(patm, ep);
    patm *= kPo;
    cc(C_PATM) = patm;
    cc(C_PBAR) = (1.0e-5) * patm;
    const double pbarf = (1.0e-5) * (double)(float)patm;
    cc(C_PBARF) = pbarf;
    cc(C_VISC0) = viscosity_h2o(0.0f, density_at<true>(density_poly(0.0), pbarf));
    // ---- soil column: SPLASH.cpp:971-1029 ----------------------------------------------------------
    const double d1000 = depth * 1000.0;
    const double theta_s = SAT / d1000;
    const double theta_r = RES / d1000;
    const double theta_fc = FC / d1000;
    const double theta_wp = WP / d1000;
    const double dth = (theta_s - theta_r);
    const double ilam = (1 / lambda);
    const double e3 = (3.0 * lambda + 1.0);
    cc(C_SAT) = SAT;
    cc(C_RES) = RES;
    cc(C_DEPTH) = depth;
    cc(C_D1000) = d1000;
#if SPLASH_L1_RECIP
    // The day step forms theta = w * (1/d1000).  theta_s and theta_r are scaled by the same multiply so
    // that a bucket sitting exactly at SAT (or RES) -- the clamps make that a common state -- still gives
    // (theta_i - theta_r)/(theta_s - theta_r) == 1 (or 0) and never a ratio one ulp above 1, which
    // would trip the reference's discontinuous failsafe `wtd < 0 -> 0.01` (SPLASH.cpp:1412-1413).
    const double inv_d1000 = 1.0 / d1000;
    const double theta_s1 = SAT * inv_d1000, theta_r1 = RES * inv_d1000;
    cc(C_INV_D1000) = inv_d1000;
    cc(C_THS) = theta_s1;
    cc(C_THR) = theta_r1;
    cc(C_DTH) = (theta_s1 - theta_r1);
    cc(C_INV_DTH) = 1.0 / (theta_s1 - theta_r1);
#else
    cc(C_THS) = theta_s;
    cc(C_THR) = theta_r;
    cc(C_DTH) = dth;
    cc(C_INV_D1000) = 1.0 / d1000;
    cc(C_INV_DTH) = 1.0 / dth;
#endif
    cc(C_ILAM) = ilam;
    cc(C_NLAM) = (-1 * lambda);
    cc(C_E3) = e3;
    cc(C_BUB) = bub;
    cc(C_BP10) = bub / 10;
    const double KG_o = 1000.0 / (997 * kG);
    const double coeff_A = exp(log(33.0) + (1.0 / lambda) * log(theta_fc));
    const double Wmax = pow((coeff_A * KG_o / (depth)), (1.0 / ((1 / lambda) + 1.0))) * (depth * 1000.0);
    cc(C_WMAX) = Wmax;
    cc(C_WMR) = (Wmax - RES);
#if SPLASH_L1_RECIP
    cc(C_THWMAX) = Wmax * inv_d1000;
#else
    cc(C_THWMAX) = Wmax / (depth * 1000.0);
#endif
    cc(C_INTPERM) = ksat / kfluidity;
    cc(C_HF) = ((2 + 3 * lambda) / (1 + 3 * lambda)) * (bub / 2);
    cc(C_KUEXP) = (3.0 + (2.0 / lambda));
    // ---- lateral flow invariants: SPLASH.cpp:993, 1291-1303, 1326, 1334-1356 -----------------------
    const double sid_oct = sqrt(Ai / (2.0 * (1 + sqrt(2.0))));
    cc(C_SIDOCT) = sid_oct;
    cc(C_AI) = Ai;
    cc(C_AU) = in.au;
    {
        const double theta_q0 = theta_wp + 0.001;
        const double psi_q0 = bub / pow((((theta_q0 - theta_r) / dth)), ilam);
        double wtd_q0 = ((bub - psi_q0) / 1000.0);
        if (wtd_q0 < 0.0 || isnan(wtd_q0)) {
            wtd_q0 = 0.0;
        } else if (wtd_q0 > depth) {
            wtd_q0 = depth;
        }
        cc(C_BRQ0) = (pow((bub / psi_q0), e3) - pow((bub / (psi_q0 + (wtd_q0 * 1000.0))), e3));
        cc(C_DENKB) = ((SAT - WP) * (Ai / 1000.0));
    }
    {
        const double theta_w = (Wmax) / (depth * 1000.0);
        const double psi_m = bub / pow((((theta_w - theta_r) / dth)), ilam);
        double wtd = ((bub - psi_m) / 1000.0);
        if (wtd < 0.0 || isnan(wtd)) {
            wtd = 0.01;
        } else if (wtd > depth) {
            wtd = depth;
        }
        cc(C_ACSW) = (depth - wtd) * in.cellin * sid_oct;
        cc(C_BRW) = (pow((bub / psi_m), e3) - pow((bub / (psi_m + (wtd * 1000.0))), e3));
        cc(C_CW) = ((24.0 * in.cellin * sid_oct) / (1.0e6));
    }
    lateral_consts(cc, in.cellout);
    cc(C_WRR) = (Wmax_R - RES);
    cc(C_INV_WMR) = 1.0 / (Wmax - RES);
    cc(C_INV_TAU_B) = 1.0 / (tau_o * (1 - 0.1898));
    cc(C_INV_AI) = 1.0 / Ai;
    cc(C_INV_DENKB) = 1.0 / ((SAT - WP) * (Ai / 1000.0));
    cc(C_TEN_BP) = 10.0 / (bub / 10);
    cc(C_KU_WMAX) = pow((cc(C_THWMAX) / cc(C_THS)), (3.0 + (2.0 / lambda)));
    cc(C_TT) = nan("");
}

}  // namespace splash
