// tg_device.cuh -- device-side building blocks: vehicle model, analytic/FD linearisation,
// reference windows, Philox4x32-10 sensor noise.  sm_100a, fp64.
//
// Reference (paths relative to the reference root):
//   tire_forces / f_cont        MPC/mpc_6stati.py:25-71, generation_type1.py:38-68, generation_type2.py:52-86
//   numerical_jacobian          MPC/mpc_6stati.py:73-97
//   linearize_discretize        MPC/mpc_6stati.py:99-109
//   vref profiles / ref window  MPC/main.py:28-47, 51-68 ; MPC/README.md:68-76
//   plant clipping              generation_type1.py:81-82, generation_type2.py:186-187
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/trajgen.h"

#define TG_LIN 20  // compact per-stage linearisation record (see tg_lin_expand); g is kept separately (6 per stage)
#define TG_TAB_NI 64   // the tyre-curve table has TG_TAB_NI + 1 intervals, centred on alpha_i = -maxAlpha + i * 2 maxAlpha / TG_TAB_NI
#define TG_TAB_NC 10   // coefficients per interval (degree 9 in the local variable s in [-1, 1])
#define TG_ATAN_NI 128 // likewise the atan table on [-TG_ATAN_T0, TG_ATAN_T0]: TG_ATAN_NI + 1 intervals
#define TG_ATAN_T0 4.0
#define TG_TAB_ROWS (TG_TAB_NI + 1)
#define TG_ATAN_ROWS (TG_ATAN_NI + 1)

// controller settings: tg_ctrl_spec with R and Rd replaced by their symmetric parts.  The handle's own are DevCfg::ctl; the
// ctrl instances of tw_solver.cuh read a problem's own record of the same type
struct TwCtrl { double q_c, q_phi, q_vx, Rs[4], Rds[4], u_lo[2], u_hi[2], du_lo[2], du_hi[2], x_lo[6], x_hi[6]; };
static_assert(sizeof(TwCtrl) == sizeof(tg_ctrl_spec), "TwCtrl mirrors tg_ctrl_spec field by field");

struct DevCfg {
    int N, n;         // horizon, 2N
    int model, plant, jacobian;
    int ns;           // number of state components with a finite bound
    int sidx[6];      // their indices
    int ms, m;        // ns*N state rows, 4N + ms rows in total
    int max_iter, check_every, adaptive_rho, adaptive_rho_min_iter, warm_start, vref_advance;
    int free_mode;    // start solves that have no active row with rho = 1e-6, alpha = 1 (tw_solver.cuh)
    double Ts;
    double p[TG_NPARAMS];
    double inv_m, inv_Iz;   // 1.0/m, 1.0/Iz (the MPC variant multiplies by them, MPC/mpc_6stati.py:67-69)
    const double *tyre_tab; // [2][TG_TAB_NI][TG_TAB_NC] piecewise polynomials of sin(C atan(B alpha)) on [-maxAlpha, maxAlpha], or null
    double tab_scale;       // TG_TAB_NI / (2 maxAlpha)
    const double *atan_tab; // [TG_ATAN_NI][TG_TAB_NC] piecewise polynomials of atan on [-TG_ATAN_T0, TG_ATAN_T0], or null
    TwCtrl ctl;             // weights and bounds
    double rho, sigma, alpha, alpha_warm, eps_abs, eps_rel, eps_pinf, adapt_tol;
    double noise_std[6];
    unsigned long long seed_base;
};

enum { P_Cm1 = 0, P_Cm2, P_Cr0, P_Cr2, P_Br, P_Cr, P_Dr, P_Bf, P_Cf, P_Df, P_m, P_Iz, P_lf, P_lr, P_g, P_maxAlpha, P_vx_zero };

__device__ __forceinline__ double tg_clamp(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// The fp64 transcendentals are inlined at every call.  One out-of-line copy of each per kernel shrinks the step from 11.1 k to
// 9.3 k SASS instructions but measured 2.3 % slower (DESIGN.md section 8): with the problems of a CTA walking the code
// together, instruction fetch no longer limits the step.
__device__ __forceinline__ double2 tg_sincos2(double x) { double s_, c_; sincos(x, &s_, &c_); return make_double2(s_, c_); }
__device__ __forceinline__ double tg_atan2(double y, double x) { return atan2(y, x); }
__device__ __forceinline__ double tg_atan(double x) { return atan(x); }
__device__ __forceinline__ double tg_sin(double x) { return sin(x); }
__device__ __forceinline__ void TG_SINCOS(double x_, double &s_, double &c_) { const double2 r_ = tg_sincos2(x_); s_ = r_.x; c_ = r_.y; }

// ------------------------------------------------------------------------------------------------
// f_cont: continuous-time dynamics, all three variants.  sd/cd = sin/cos(delta) are passed in because
// the controller evaluates the whole horizon at the same delta (ubar_k = u_prev, mpc_6stati.py:170).
__device__ __noinline__ void tg_f_cont(const double *__restrict__ p, int variant, const double x[6], double d,
                                          double delta, double sd, double cd, double f[6])
{
    const double phi = x[2], vx = x[3], vy = x[4], om = x[5];
    const double vmag = fmax(fabs(vx), p[P_vx_zero]);
    double vx_eff;
    if (variant == TG_MODEL_MPC) {
        const double sgn = (double)((vx > 0.0) - (vx < 0.0));  // np.sign: sign(0) = 0  (:33)
        vx_eff = sgn * vmag;
    } else {
        vx_eff = vmag;  // generation_type1.py:41
    }
    double af = -tg_atan2(om * p[P_lf] + vy, vx_eff) + delta;
    double ar = tg_atan2(om * p[P_lr] - vy, vx_eff);
    af = tg_clamp(af, -p[P_maxAlpha], p[P_maxAlpha]);
    if (variant != TG_MODEL_GEN1) ar = tg_clamp(ar, -p[P_maxAlpha], p[P_maxAlpha]);  // gen1 leaves alpha_r free (:46)
    const double Fyf = p[P_Df] * tg_sin(p[P_Cf] * tg_atan(p[P_Bf] * af));
    const double Fyr = p[P_Dr] * tg_sin(p[P_Cr] * tg_atan(p[P_Br] * ar));
    const double vl = (variant == TG_MODEL_MPC) ? vx : vx_eff;  // :51 vs generation_type1.py:53
    const double Frx = (p[P_Cm1] - p[P_Cm2] * vl) * d - p[P_Cr0] - p[P_Cr2] * (vl * vl);
    double sp, cp;
    TG_SINCOS(phi, sp, cp);
    const double m = p[P_m], Iz = p[P_Iz];
    f[0] = vx * cp - vy * sp;
    f[1] = vx * sp + vy * cp;
    f[2] = om;
    if (variant == TG_MODEL_MPC) {
        f[3] = (1.0 / m) * (Frx - Fyf * sd + m * vy * om);
        f[4] = (1.0 / m) * (Fyr + Fyf * cd - m * vx * om);
        f[5] = (1.0 / Iz) * (Fyf * p[P_lf] * cd - Fyr * p[P_lr]);
    } else {
        f[3] = (Frx - Fyf * sd + m * vy * om) / m;
        f[4] = (Fyr + Fyf * cd - m * vx * om) / m;
        f[5] = (Fyf * p[P_lf] * cd - Fyr * p[P_lr]) / Iz;
    }
}

// plant step: x <- x + Ts f(x,u) (+ clipping for the generator plants) for the vehicle p (the handle's c.p or a row of a
// per-trajectory plant table); c supplies Ts and the plant variant
__device__ __forceinline__ void tg_plant_step(const DevCfg &c, const double *p, double x[6], double d, double delta)
{
    double sd, cd, f[6];
    TG_SINCOS(delta, sd, cd);
    tg_f_cont(p, c.plant, x, d, delta, sd, cd, f);
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = x[i] + c.Ts * f[i];
    if (c.plant != TG_PLANT_MPC) {
        x[3] = fmax(x[3], 0.0);
        x[5] = tg_clamp(x[5], -6.0, 6.0);
    }
}

// f_cont evaluated by the 4 lanes of a quad in SIMD: lane role 0 = front tyre chain (atan2 -> atan -> sin),
// role 1 = rear tyre chain, roles 2/3 = tg_sin(phi) / tg_sin(phi + pi/2) = cos(phi) sharing the final sin with the
// tyre lanes; three transcendental latencies instead of eight on the sequential rollout / plant path.  Must be
// called by all 32 lanes of a warp; every lane returns the full f.
__device__ __forceinline__ void tg_f_cont_lanes(const double *__restrict__ p, double inv_m, double inv_Iz, int variant,
                                                const double x[6], double d, double delta, double sd, double cd, int lane,
                                                double f[6], double *aux = nullptr)
{
    const int role = lane & 3, base = lane & ~3;
    const double phi = x[2], vx = x[3], vy = x[4], om = x[5];
    const double vmag = fmax(fabs(vx), p[P_vx_zero]);
    const double vx_eff = (variant == TG_MODEL_MPC) ? (double)((vx > 0.0) - (vx < 0.0)) * vmag : vmag;
    const bool front = (role == 0);
    const double Lt = front ? p[P_lf] : p[P_lr];
    const double nl = front ? (om * Lt + vy) : (om * Lt - vy);
    const double at = tg_atan2(nl, vx_eff);
    double alpha = front ? (-at + delta) : at;
    const double alpha_raw = alpha;
    if (front || variant != TG_MODEL_GEN1) alpha = tg_clamp(alpha, -p[P_maxAlpha], p[P_maxAlpha]);
    const double th = (front ? p[P_Cf] : p[P_Cr]) * tg_atan((front ? p[P_Bf] : p[P_Br]) * alpha);
    const double arg = (role < 2) ? th : ((role == 2) ? phi : phi + 1.5707963267948966);
    const double sv = tg_sin(arg);
    if (aux && lane < 4) {   // hand the transcendental intermediates of this stage to the linearisation (one predicate,
        // no divergence): tyre lanes store (slip angle before the clamp, C atan(B alpha)), lanes 2/3 sin(phi) / cos(phi)
        const bool tyre = role < 2;
        aux[tyre ? 2 * role : 2 + role] = tyre ? alpha_raw : sv;
        aux[tyre ? 2 * role + 1 : 2 + role] = tyre ? th : sv;
    }
    const double F = (front ? p[P_Df] : p[P_Dr]) * sv;
    const double Fyf = __shfl_sync(0xffffffffu, F, base), Fyr = __shfl_sync(0xffffffffu, F, base + 1);
    const double sp = __shfl_sync(0xffffffffu, sv, base + 2), cp = __shfl_sync(0xffffffffu, sv, base + 3);
    const double vl = (variant == TG_MODEL_MPC) ? vx : vx_eff;
    const double Frx = (p[P_Cm1] - p[P_Cm2] * vl) * d - p[P_Cr0] - p[P_Cr2] * (vl * vl);
    const double m = p[P_m], Iz = p[P_Iz];
    f[0] = vx * cp - vy * sp;
    f[1] = vx * sp + vy * cp;
    f[2] = om;
    if (variant == TG_MODEL_MPC) {
        f[3] = inv_m * (Frx - Fyf * sd + m * vy * om);       // (1.0/m) * (...), MPC/mpc_6stati.py:67
        f[4] = inv_m * (Fyr + Fyf * cd - m * vx * om);
        f[5] = inv_Iz * (Fyf * p[P_lf] * cd - Fyr * p[P_lr]);
    } else {
        f[3] = (Frx - Fyf * sd + m * vy * om) / m;
        f[4] = (Fyr + Fyf * cd - m * vx * om) / m;
        f[5] = (Fyf * p[P_lf] * cd - Fyr * p[P_lr]) / Iz;
    }
}

// ------------------------------------------------------------------------------------------------
// Tyre curve from a table.  The Pacejka term g(alpha) = sin(C atan(B alpha)) is only ever evaluated on the clamped
// slip angle |alpha| <= maxAlpha (MPC/mpc_6stati.py:42-47), a compact interval on which g is analytic (nearest
// singularity at alpha = +-i/B), so a piecewise degree-9 polynomial on 64 intervals reproduces it to ~1e-16
// (built in long double at tg_create, verified there against libm; the handle falls back to atan/sin if the fit is
// not at rounding level for the caller's B, C).  It replaces two of the three dependent fp64 transcendentals of
// every stage of the sequential nominal rollout -- the longest dependent chain of an MPC step -- by an index
// computation and nine FMAs, and gives the linearisation dg/dalpha for free.
// Row and local variable of a table look-up.  Interval i is CENTRED on the grid point u = i (u = (x - lo) * scale, i = 0 .. NI),
// so the index is round-to-nearest of u: adding 1.5 * 2^52 leaves it in the low mantissa word (no F2I / I2F on the chain)
// and subtracting it again gives the rounded value; s = 2 (u - i) lies in [-1, 1].  0 <= u <= NI is the caller's duty.
__device__ __forceinline__ const double *tg_tab_row(const double *__restrict__ tab, double u, double &s_)
{
    const double MAGIC = 6755399441055744.0;   // 1.5 * 2^52
    const double m = u + MAGIC;
    const int i = __double2loint(m);
    s_ = 2.0 * (u - (m - MAGIC));
    return tab + i * TG_TAB_NC;
}
// value of a table row at s: two interleaved Horner chains in s^2 (even / odd coefficients), half the dependent depth
__device__ __forceinline__ double tg_tab_val(const double *__restrict__ row, double s_)
{
    const double2 *c2 = reinterpret_cast<const double2 *>(row);
    const double2 c01 = __ldg(c2), c23 = __ldg(c2 + 1), c45 = __ldg(c2 + 2), c67 = __ldg(c2 + 3), c89 = __ldg(c2 + 4);
    const double s2 = s_ * s_;
    double ev = fma(c89.x, s2, c67.x), od = fma(c89.y, s2, c67.y);
    ev = fma(ev, s2, c45.x); od = fma(od, s2, c45.y);
    ev = fma(ev, s2, c23.x); od = fma(od, s2, c23.y);
    ev = fma(ev, s2, c01.x); od = fma(od, s2, c01.y);
    return fma(od, s_, ev);
}

__device__ __forceinline__ void tg_tyre_tab(const double *__restrict__ tab, double alpha, double ma, double scale,
                                            double &g, double &dg)
{
    double s_;
    const double2 *c2 = reinterpret_cast<const double2 *>(tg_tab_row(tab, (alpha + ma) * scale, s_));
    const double2 c01 = __ldg(c2), c23 = __ldg(c2 + 1), c45 = __ldg(c2 + 2), c67 = __ldg(c2 + 3), c89 = __ldg(c2 + 4);
    double v = c89.y, d_ = 0.0;   // Horner for the value and its derivative together
    d_ = fma(d_, s_, v); v = fma(v, s_, c89.x);
    d_ = fma(d_, s_, v); v = fma(v, s_, c67.y);
    d_ = fma(d_, s_, v); v = fma(v, s_, c67.x);
    d_ = fma(d_, s_, v); v = fma(v, s_, c45.y);
    d_ = fma(d_, s_, v); v = fma(v, s_, c45.x);
    d_ = fma(d_, s_, v); v = fma(v, s_, c23.y);
    d_ = fma(d_, s_, v); v = fma(v, s_, c23.x);
    d_ = fma(d_, s_, v); v = fma(v, s_, c01.y);
    d_ = fma(d_, s_, v); v = fma(v, s_, c01.x);
    g = v;
    dg = d_ * (2.0 * scale);
}
// the value alone (nominal rollout, plant): short dependent chain
__device__ __forceinline__ double tg_tyre_val(const double *__restrict__ tab, double alpha, double ma, double scale)
{
    double s_;
    const double *row = tg_tab_row(tab, fma(alpha, scale, ma * scale), s_);
    return tg_tab_val(row, s_);
}

// 1 / x for x > 0 to ~1 ulp without the IEEE division sequence: hardware seed + two Newton steps
__device__ __forceinline__ double tg_rcp_pos(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;
}

// atan(t) for |t| <= TG_ATAN_T0 from the table (1e-16; nearest singularities of atan are at +-i, far from every interval)
__device__ __forceinline__ double tg_atan_tab(const double *__restrict__ tab, double t)
{
    double s_;
    const double *row = tg_tab_row(tab, fma(t, TG_ATAN_NI / (2.0 * TG_ATAN_T0), TG_ATAN_NI / 2.0), s_);
    return tg_tab_val(row, s_);
}

// atan2(y, x) for the slip angles: x = vx_eff.  With x > 0 (always for the generator variants, and for the MPC variant
// while the vehicle moves forward) atan2(y, x) = atan(y / x); the table covers |y / x| <= 4, anything else takes libdevice.
__device__ __forceinline__ double tg_slip_atan(const double *__restrict__ atan_tab, double y, double x)
{
    if (atan_tab && x > 0.0) {
        const double t = y * tg_rcp_pos(x);
        if (fabs(t) <= TG_ATAN_T0) return tg_atan_tab(atan_tab, t);
    }
    return tg_atan2(y, x);
}

// sin / cos of phi + dphi from sin / cos of phi, |dphi| <= 0.25 (Taylor to x^13 / x^12: < 3e-18)
__device__ __forceinline__ void tg_rotate_small(double &sp, double &cp, double dphi)
{
    const double x2 = dphi * dphi;
    double ps = -1.0 / 6227020800.0;
    ps = fma(ps, x2, 1.0 / 39916800.0); ps = fma(ps, x2, -1.0 / 362880.0); ps = fma(ps, x2, 1.0 / 5040.0);
    ps = fma(ps, x2, -1.0 / 120.0); ps = fma(ps, x2, 1.0 / 6.0);
    const double sn = fma(-dphi * x2, ps, dphi);                        // dphi - dphi^3 (1/6 - ...)
    double pc = 1.0 / 479001600.0;
    pc = fma(pc, x2, -1.0 / 3628800.0); pc = fma(pc, x2, 1.0 / 40320.0); pc = fma(pc, x2, -1.0 / 720.0);
    pc = fma(pc, x2, 1.0 / 24.0); pc = fma(pc, x2, -0.5);
    const double cm1 = pc * x2;                                          // cos(dphi) - 1
    const double ns = fma(sp, cm1, fma(cp, sn, sp));
    const double nc = fma(cp, cm1, fma(-sp, sn, cp));
    sp = ns; cp = nc;
}

// f_cont by a lane pair (lane & 1: 0 = front tyre, 1 = rear tyre) with the tyre table and sin/cos(phi) supplied by
// the caller.  GEN1 leaves the rear slip angle unclamped (generation_type1.py:46): inside the clamp interval the table still
// applies, outside it that lane evaluates atan / sin.
// aux (optional, shared memory) receives {alpha_f raw, alpha_r raw, sin phi, cos phi} for the linearisation.
// p, inv_m = 1/m, inv_Iz = 1/Iz: the vehicle; tyre_tab / atan_tab: the handle's tables (c.tab_scale is their scale), which
// only serve a vehicle whose B, C and maxAlpha are the handle's (tg_plant_row_tables).  atan_tab may be null.
__device__ __forceinline__ void tg_f_cont_tab(const DevCfg &c, const double *__restrict__ p, double inv_m, double inv_Iz,
                                              const double *__restrict__ tyre_tab, const double *__restrict__ atan_tab, int variant,
                                              const double x[6], double d, double delta, double sd, double cd, double sp, double cp,
                                              int lane, double f[6], double *aux = nullptr)
{
    const int rear = lane & 1, base = lane & ~1;
    const double vx = x[3], vy = x[4], om = x[5];
    const double vmag = fmax(fabs(vx), p[P_vx_zero]);
    const double vx_eff = (variant == TG_MODEL_MPC) ? (double)((vx > 0.0) - (vx < 0.0)) * vmag : vmag;
    const double nl = rear ? (om * p[P_lr] - vy) : (om * p[P_lf] + vy);
    const double at = tg_slip_atan(atan_tab, nl, vx_eff);
    const double alpha_raw = rear ? at : (-at + delta);
    const bool free_rear = rear && variant == TG_MODEL_GEN1;
    const double alpha = free_rear ? alpha_raw : tg_clamp(alpha_raw, -p[P_maxAlpha], p[P_maxAlpha]);
    double g, dg;
    if (free_rear && fabs(alpha) > p[P_maxAlpha]) g = tg_sin(p[P_Cr] * tg_atan(p[P_Br] * alpha));
    else tg_tyre_tab(tyre_tab + rear * (TG_TAB_ROWS * TG_TAB_NC), alpha, p[P_maxAlpha], c.tab_scale, g, dg);
    const double F = (rear ? p[P_Dr] : p[P_Df]) * g;
    if (aux && lane < 2) { aux[rear] = alpha_raw; aux[2 + rear] = rear ? cp : sp; }
    const double Fyf = __shfl_sync(0xffffffffu, F, base), Fyr = __shfl_sync(0xffffffffu, F, base + 1);
    const double vl = (variant == TG_MODEL_MPC) ? vx : vx_eff;
    const double Frx = (p[P_Cm1] - p[P_Cm2] * vl) * d - p[P_Cr0] - p[P_Cr2] * (vl * vl);
    const double m = p[P_m];
    f[0] = vx * cp - vy * sp;
    f[1] = vx * sp + vy * cp;
    f[2] = om;
    if (variant == TG_MODEL_MPC) {
        f[3] = inv_m * (Frx - Fyf * sd + m * vy * om);       // (1.0/m) * (...), MPC/mpc_6stati.py:67
        f[4] = inv_m * (Fyr + Fyf * cd - m * vx * om);
        f[5] = inv_Iz * (Fyf * p[P_lf] * cd - Fyr * p[P_lr]);
    } else {
        f[3] = (Frx - Fyf * sd + m * vy * om) / m;
        f[4] = (Fyr + Fyf * cd - m * vx * om) / m;
        f[5] = (Fyf * p[P_lf] * cd - Fyr * p[P_lr]) / p[P_Iz];
    }
}

// One Euler stage of the velocity recurrence (vx, vy, omega) <- (vx, vy, omega) + Ts f_{3..5} by a lane pair (lane & 1:
// 0 = front tyre, 1 = rear tyre), written for the SHORTEST dependent chain: this recurrence is the longest sequential chain
// of an MPC step (N stages, nothing else of the step can start before it ends).  Per-step constants are hoisted into
// TgRoll; the tables are indexed without F2I / I2F; clamps are compare-selects; the force exchange is one xor-shuffle; the
// sums are re-associated so that two FMAs follow the tyre force (results differ from tg_f_cont_tab's in the last bit only).
// Variants MPC / GEN2 (both slip angles clamped).  aux (optional, shared memory) receives the slip angle before the clamp.
struct TgRoll {
    double L, svy, sa, da, D, ma, tscale, toff, Ts_im, Ts_iI5f, Ts_iI5r, cdm, d, sd;
    const double *tyre;
    int rear;
};
__device__ __forceinline__ TgRoll tg_roll_setup(const DevCfg &c, double d, double delta, double sd, double cd, int lane)
{
    const double *__restrict__ p = c.p;
    TgRoll k;
    k.rear = lane & 1;
    k.L = k.rear ? p[P_lr] : p[P_lf];
    k.svy = k.rear ? -1.0 : 1.0;                       // n = omega L + svy vy
    k.sa = k.rear ? 1.0 : -1.0; k.da = k.rear ? 0.0 : delta;   // alpha = sa atan(n / vx_eff) + da
    k.D = k.rear ? p[P_Dr] : p[P_Df];
    k.ma = p[P_maxAlpha]; k.tscale = c.tab_scale; k.toff = p[P_maxAlpha] * c.tab_scale;
    k.tyre = c.tyre_tab + k.rear * (TG_TAB_ROWS * TG_TAB_NC);
    k.Ts_im = c.Ts * c.inv_m;
    k.Ts_iI5f = c.Ts * c.inv_Iz * p[P_lf] * cd; k.Ts_iI5r = c.Ts * c.inv_Iz * p[P_lr];
    k.cdm = cd; k.d = d; k.sd = sd;
    return k;
}
__device__ __forceinline__ void tg_roll_stage(const DevCfg &c, const TgRoll &k, int variant, double &vx, double &vy, double &om,
                                              int lane, double *aux)
{
    const double *__restrict__ p = c.p;
    const double vz = p[P_vx_zero];
    double veff = vx;                                    // sign(vx) max(|vx|, vx_zero) = vx while vx >= vx_zero
    if (!(vx >= vz)) {
        const double vmag = fmax(fabs(vx), vz);
        veff = (variant == TG_MODEL_MPC) ? (double)((vx > 0.0) - (vx < 0.0)) * vmag : vmag;
    }
    const double n = fma(om, k.L, k.svy * vy);
    double at;
    {
        const double t = n * tg_rcp_pos(veff);
        if (c.atan_tab && veff > 0.0 && fabs(t) <= TG_ATAN_T0) at = tg_atan_tab(c.atan_tab, t);
        else at = tg_atan2(n, veff);
    }
    const double araw = fma(k.sa, at, k.da);
    double al = araw > k.ma ? k.ma : araw;
    al = al < -k.ma ? -k.ma : al;
    double s_;
    const double *row = tg_tab_row(k.tyre, fma(al, k.tscale, k.toff), s_);
    const double F = k.D * tg_tab_val(row, s_);
    if (aux && lane < 2) aux[k.rear] = araw;
    // everything that does not wait for the tyre force
    const double vl = (variant == TG_MODEL_MPC) ? vx : veff;
    const double Frx = (p[P_Cm1] - p[P_Cm2] * vl) * k.d - p[P_Cr0] - p[P_Cr2] * (vl * vl);
    const double m = p[P_m];
    const double b3 = fma(m * vy, om, Frx), b4 = -m * vx * om;
    const double vx0 = fma(k.Ts_im, b3, vx), vy0 = fma(k.Ts_im, b4, vy);
    const double Fo = __shfl_xor_sync(0xffffffffu, F, 1);
    const double Fyf = k.rear ? Fo : F, Fyr = k.rear ? F : Fo;
    // vx' = vx + Ts/m (Frx - Fyf sin(delta) + m vy om);  vy' = vy + Ts/m (Fyr + Fyf cos(delta) - m vx om);
    // om' = om + Ts/Iz (Fyf lf cos(delta) - Fyr lr)
    vx = fma(-k.Ts_im * k.sd, Fyf, vx0);
    vy = fma(k.Ts_im, fma(Fyf, k.cdm, Fyr), vy0);
    om = fma(k.Ts_iI5f, Fyf, fma(-k.Ts_iI5r, Fyr, om));
}

// Which tables a row of a per-trajectory plant table (p = the row) may use: the handle's, when the row's tyre constants Bf, Cf,
// Br, Cr and maxAlpha equal the handle's bit for bit (the tables are fitted and verified for those constants only); none
// otherwise, and none when the handle has none -- the row's plant then evaluates atan2 / atan / sin with libdevice, as a handle
// without tables does.  Either way row b computes what a handle created with params = row b computes.
__device__ __forceinline__ bool tg_plant_row_tables(const DevCfg &c, const double *__restrict__ p)
{
    if (!c.tyre_tab) return false;
    auto same = [&](int i) { return __double_as_longlong(p[i]) == __double_as_longlong(c.p[i]); };
    return same(P_Bf) && same(P_Cf) && same(P_Br) && same(P_Cr) && same(P_maxAlpha);
}

// plant step by a whole warp (see tg_f_cont_lanes) for the vehicle p with 1/m, 1/Iz and the tables tyre_tab / atan_tab
// (null: libdevice)
__device__ __forceinline__ void tg_plant_step_lanes(const DevCfg &c, const double *__restrict__ p, double inv_m, double inv_Iz,
                                                    const double *tyre_tab, const double *atan_tab, double x[6], double d,
                                                    double delta, int lane)
{
    double sd, cd, f[6];
    TG_SINCOS(delta, sd, cd);
    if (tyre_tab) {
        double sp, cp;
        TG_SINCOS(x[2], sp, cp);
        tg_f_cont_tab(c, p, inv_m, inv_Iz, tyre_tab, atan_tab, c.plant, x, d, delta, sd, cd, sp, cp, lane, f);
    } else {
        tg_f_cont_lanes(p, inv_m, inv_Iz, c.plant, x, d, delta, sd, cd, lane, f);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = x[i] + c.Ts * f[i];
    if (c.plant != TG_PLANT_MPC) {
        x[3] = fmax(x[3], 0.0);
        x[5] = tg_clamp(x[5], -6.0, 6.0);
    }
}

// Plant step of the generator plants (TG_PLANT_GEN1 / GEN2) by ONE thread, for the open-loop kernels where a thread owns
// a trajectory.  vx_eff = max(|vx|, vx_zero) > 0 there (generation_type1.py:41), so atan2(y, vx_eff) = atan(y / vx_eff),
// and the tyre curve comes from the table (tyre_tab: the handle's, or null for libdevice; pv: the vehicle) wherever the slip
// angle lies inside the clamp interval (always for the front tyre and for GEN2's rear tyre; GEN1 leaves the rear angle free,
// :46, and falls back to atan / sin outside).
__device__ __forceinline__ void tg_plant_step_gen(const DevCfg &c, const double *pv, const double *tyre_tab,
                                                  const double *atan_tab, double x[6], double d, double delta)
{
    const double *__restrict__ p = pv;
    const double vx = x[3], vy = x[4], om = x[5];
    const double ma = p[P_maxAlpha];
    const double vmag = fmax(fabs(vx), p[P_vx_zero]);
    const double af = tg_clamp(delta - tg_slip_atan(atan_tab, om * p[P_lf] + vy, vmag), -ma, ma);
    double ar = tg_slip_atan(atan_tab, om * p[P_lr] - vy, vmag);
    if (c.plant != TG_PLANT_GEN1) ar = tg_clamp(ar, -ma, ma);
    double gf, gr, dg;
    if (tyre_tab) {
        tg_tyre_tab(tyre_tab, af, ma, c.tab_scale, gf, dg);
        if (fabs(ar) <= ma) tg_tyre_tab(tyre_tab + TG_TAB_ROWS * TG_TAB_NC, ar, ma, c.tab_scale, gr, dg);
        else gr = tg_sin(p[P_Cr] * tg_atan(p[P_Br] * ar));
    } else {
        gf = tg_sin(p[P_Cf] * tg_atan(p[P_Bf] * af));
        gr = tg_sin(p[P_Cr] * tg_atan(p[P_Br] * ar));
    }
    const double Fyf = p[P_Df] * gf, Fyr = p[P_Dr] * gr;
    const double Frx = (p[P_Cm1] - p[P_Cm2] * vmag) * d - p[P_Cr0] - p[P_Cr2] * (vmag * vmag);
    double sd, cd, sp, cp;
    TG_SINCOS(delta, sd, cd);
    TG_SINCOS(x[2], sp, cp);
    const double m = p[P_m], Ts = c.Ts;
    const double f0 = vx * cp - vy * sp, f1 = vx * sp + vy * cp;
    const double f3 = (Frx - Fyf * sd + m * vy * om) / m;
    const double f4 = (Fyr + Fyf * cd - m * vx * om) / m;
    const double f5 = (Fyf * p[P_lf] * cd - Fyr * p[P_lr]) / p[P_Iz];
    x[0] = x[0] + Ts * f0;
    x[1] = x[1] + Ts * f1;
    x[2] = x[2] + Ts * om;
    x[3] = fmax(x[3] + Ts * f3, 0.0);                 // generation_type1.py:81-82
    x[4] = x[4] + Ts * f4;
    x[5] = tg_clamp(x[5] + Ts * f5, -6.0, 6.0);
}

// ------------------------------------------------------------------------------------------------
// Compact linearisation record of one stage.  For every variant and both Jacobian modes the full
// 6x6 / 6x2 matrices have this sparsity exactly (f does not depend on X,Y; phi enters rows 0,1 only;
// rows 0-2 do not depend on u; rows 4,5 do not depend on d), so nothing is lost:
//   [0..2]  A[0][2],A[0][3],A[0][4]   [3..5] A[1][2],A[1][3],A[1][4]   [6] A[2][5]
//   [7..15] A[3..5][3..5] row-major   [16] B[3][0]  [17] B[3][1]  [18] B[4][1]  [19] B[5][1]
//   A[i][i] = 1 for i<3, everything else 0.   g[0..5] goes to a separate array (only the taps / X_opt need it:
//   the nominal rollout IS the affine recursion, x_k = xbar_k + sum_j G_kj dU_j).
__device__ __forceinline__ void tg_lin_expand(const double *__restrict__ r, const double *__restrict__ gv, double *A, double *Bm, double *g)
{
    if (A) {
        for (int i = 0; i < 36; ++i) A[i] = 0.0;
        A[0] = 1.0; A[7] = 1.0; A[14] = 1.0;
        A[2] = r[0]; A[3] = r[1]; A[4] = r[2];
        A[8] = r[3]; A[9] = r[4]; A[10] = r[5];
        A[17] = r[6];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) A[(3 + i) * 6 + 3 + j] = r[7 + 3 * i + j];
    }
    if (Bm) {
        for (int i = 0; i < 12; ++i) Bm[i] = 0.0;
        Bm[6] = r[16]; Bm[7] = r[17]; Bm[9] = r[18]; Bm[11] = r[19];
    }
    if (g && gv)
        for (int i = 0; i < 6; ++i) g[i] = gv[i];
}

// Analytic linearisation at (x, u): Ad = I + Ts df/dx, Bd = Ts df/du, g = Ts (f - Jx x - Ju u).
// `aux` (optional) = {alpha_f before the clamp, Cf atan(Bf alpha_f), alpha_r before the clamp, Cr atan(Br alpha_r),
// sin(phi), cos(phi)} as the nominal rollout left them for this stage: the rollout has just evaluated f at exactly
// this point, so the two atan2, two atan and one sincos of the linearisation are not recomputed.
// With `tab_aux` = {alpha_f, alpha_r before the clamp, sin(phi), cos(phi)} (table path) the tyre force and its slope
// come from the table and no transcendental is evaluated at all.
// Returns true when the reference's central-difference stencil (MPC/mpc_6stati.py:73-97, eps = 1e-5 on every state and
// input) straddles a CONTINUOUS kink of f -- |vx| = vx_zero or a slip-angle clamp -- where the reference's Jacobian is a
// blend of the two one-sided slopes.  The caller re-evaluates such a stage with tg_linearize_fd: parity is with what the
// reference computes.  NOT covered, on purpose: stencils that straddle a JUMP of f (the atan2 branch cut behind
// vx_eff < 0, the sign flip at vx = 0; a nominal rollout that brakes through standstill ends up there with n ~ 0).  The
// reference then returns jump / (2 eps) -- entries of ~2e5 in Ad, cond(H) 1e13..1e15 after condensing -- which no
// condensed solver can carry in fp64; the closed form keeps the one-sided derivative there (DESIGN.md section 5).
__device__ bool tg_linearize_analytic(const DevCfg &c, const double x[6], double d, double delta, double sd,
                                      double cd, double *__restrict__ rec, double *__restrict__ gout,
                                      const double *__restrict__ aux = nullptr, const double *__restrict__ tab_aux = nullptr)
{
    const double *p = c.p;
    const int variant = c.model;
    const double phi = x[2], vx = x[3], vy = x[4], om = x[5];
    const double lf = p[P_lf], lr = p[P_lr], m = p[P_m], ma = p[P_maxAlpha];
    const double im = c.inv_m, iI = c.inv_Iz;
    const double avx = fabs(vx);
    const double vmag = fmax(avx, p[P_vx_zero]);
    const double sgn = (double)((vx > 0.0) - (vx < 0.0));
    const bool free_v = avx > p[P_vx_zero];
    double vx_eff, dveff;  // d vx_eff / d vx
    if (variant == TG_MODEL_MPC) { vx_eff = sgn * vmag; dveff = free_v ? 1.0 : 0.0; }
    else                         { vx_eff = vmag;       dveff = free_v ? sgn : 0.0; }
    const double nf = om * lf + vy, nr = om * lr - vy;
    const double denf = nf * nf + vx_eff * vx_eff, denr = nr * nr + vx_eff * vx_eff;
    double af = tab_aux ? tab_aux[0] : (aux ? aux[0] : -tg_atan2(nf, vx_eff) + delta);
    double ar = tab_aux ? tab_aux[1] : (aux ? aux[2] : tg_atan2(nr, vx_eff));
    // partials of the slip angles (zero where the clamp is active)
    double af_vx = (nf / denf) * dveff, af_vy = -vx_eff / denf, af_om = -lf * vx_eff / denf, af_de = 1.0;
    double ar_vx = -(nr / denr) * dveff, ar_vy = -vx_eff / denr, ar_om = lr * vx_eff / denr;
    bool near_kink;
    {
        const double eps = 1e-5;                                   // the reference's eps_x = eps_u
        const double da = 1.0001 * eps * fmax(1.0, 1.0 / vmag);    // first-order reach of a slip angle over the stencil
        near_kink = fabs(avx - p[P_vx_zero]) <= eps || fabs(fabs(af) - ma) <= da ||
                    (variant != TG_MODEL_GEN1 && fabs(fabs(ar) - ma) <= da);
    }
    if (af > ma || af < -ma) { af = tg_clamp(af, -ma, ma); af_vx = af_vy = af_om = af_de = 0.0; }
    if (variant != TG_MODEL_GEN1 && (ar > ma || ar < -ma)) { ar = tg_clamp(ar, -ma, ma); ar_vx = ar_vy = ar_om = 0.0; }
    double Fyf, Fyr, dFf, dFr;   // forces and dF / d alpha
    if (tab_aux) {
        double g, dg;
        tg_tyre_tab(c.tyre_tab, af, ma, c.tab_scale, g, dg);
        Fyf = p[P_Df] * g; dFf = p[P_Df] * dg;
        tg_tyre_tab(c.tyre_tab + TG_TAB_ROWS * TG_TAB_NC, ar, ma, c.tab_scale, g, dg);
        Fyr = p[P_Dr] * g; dFr = p[P_Dr] * dg;
    } else {
        double s1, c1, s2, c2;
        const double Bf = p[P_Bf], Br = p[P_Br];
        TG_SINCOS(aux ? aux[1] : p[P_Cf] * tg_atan(Bf * af), s1, c1);
        TG_SINCOS(aux ? aux[3] : p[P_Cr] * tg_atan(Br * ar), s2, c2);
        Fyf = p[P_Df] * s1; Fyr = p[P_Dr] * s2;
        dFf = p[P_Df] * c1 * p[P_Cf] * Bf / (1.0 + (Bf * af) * (Bf * af));
        dFr = p[P_Dr] * c2 * p[P_Cr] * Br / (1.0 + (Br * ar) * (Br * ar));
    }
    const double Ff_vx = dFf * af_vx, Ff_vy = dFf * af_vy, Ff_om = dFf * af_om, Ff_de = dFf * af_de;
    const double Fr_vx = dFr * ar_vx, Fr_vy = dFr * ar_vy, Fr_om = dFr * ar_om;
    double vl, dvl;
    if (variant == TG_MODEL_MPC) { vl = vx; dvl = 1.0; } else { vl = vx_eff; dvl = dveff; }
    const double Frx = (p[P_Cm1] - p[P_Cm2] * vl) * d - p[P_Cr0] - p[P_Cr2] * (vl * vl);
    const double Frx_vx = (-p[P_Cm2] * d - 2.0 * p[P_Cr2] * vl) * dvl;
    const double Frx_d = p[P_Cm1] - p[P_Cm2] * vl;
    double sp, cp;
    if (tab_aux) { sp = tab_aux[2]; cp = tab_aux[3]; } else if (aux) { sp = aux[4]; cp = aux[5]; } else TG_SINCOS(phi, sp, cp);
    double f[6];
    f[0] = vx * cp - vy * sp;
    f[1] = vx * sp + vy * cp;
    f[2] = om;
    f[3] = (Frx - Fyf * sd + m * vy * om) * im;
    f[4] = (Fyr + Fyf * cd - m * vx * om) * im;
    f[5] = (Fyf * lf * cd - Fyr * lr) * iI;
    // continuous Jacobian entries (rows 3..5)
    const double j33 = (Frx_vx - Ff_vx * sd) * im, j34 = (-Ff_vy * sd + m * om) * im, j35 = (-Ff_om * sd + m * vy) * im;
    const double j43 = (Fr_vx + Ff_vx * cd - m * om) * im, j44 = (Fr_vy + Ff_vy * cd) * im, j45 = (Fr_om + Ff_om * cd - m * vx) * im;
    const double j53 = (Ff_vx * lf * cd - Fr_vx * lr) * iI, j54 = (Ff_vy * lf * cd - Fr_vy * lr) * iI,
                 j55 = (Ff_om * lf * cd - Fr_om * lr) * iI;
    const double b30 = Frx_d * im, b31 = (-Ff_de * sd - Fyf * cd) * im;
    const double b41 = (Ff_de * cd - Fyf * sd) * im;
    const double b51 = (Ff_de * lf * cd - Fyf * lf * sd) * iI;
    const double Ts = c.Ts;
    rec[0] = -Ts * f[1]; rec[1] = Ts * cp; rec[2] = -Ts * sp;
    rec[3] = Ts * f[0];  rec[4] = Ts * sp; rec[5] = Ts * cp;
    rec[6] = Ts;
    rec[7] = 1.0 + Ts * j33; rec[8] = Ts * j34;        rec[9] = Ts * j35;
    rec[10] = Ts * j43;      rec[11] = 1.0 + Ts * j44; rec[12] = Ts * j45;
    rec[13] = Ts * j53;      rec[14] = Ts * j54;       rec[15] = 1.0 + Ts * j55;
    const double B30 = Ts * b30, B31 = Ts * b31, B41 = Ts * b41, B51 = Ts * b51;
    rec[16] = B30; rec[17] = B31; rec[18] = B41; rec[19] = B51;
    if (gout) {   // g = x + Ts f - Ad x - Bd u = Ts f - (Ad - I) x - Bd u
        gout[0] = Ts * f[0] - (rec[0] * phi + rec[1] * vx + rec[2] * vy);
        gout[1] = Ts * f[1] - (rec[3] * phi + rec[4] * vx + rec[5] * vy);
        gout[2] = Ts * f[2] - rec[6] * om;
        gout[3] = Ts * f[3] - (Ts * j33 * vx + Ts * j34 * vy + Ts * j35 * om) - (B30 * d + B31 * delta);
        gout[4] = Ts * f[4] - (Ts * j43 * vx + Ts * j44 * vy + Ts * j45 * om) - (B41 * delta);
        gout[5] = Ts * f[5] - (Ts * j53 * vx + Ts * j54 * vy + Ts * j55 * om) - (B51 * delta);
    }
    return near_kink;
}

// Central-difference linearisation, the reference's arithmetic verbatim (mpc_6stati.py:73-109):
// 12 + 4 + 1 evaluations of f_cont, eps = 1e-5, g = xbar + Ts f - Ad xbar - Bd ubar.
__device__ __noinline__ void tg_linearize_fd(const DevCfg &c, const double x[6], double d, double delta, double *__restrict__ rec, double *__restrict__ gout)
{
    const double eps = 1e-5;
    double Jx[6][6], Ju[6][2], f0[6], fp[6], fm[6], xx[6];
    double sd, cd;
    TG_SINCOS(delta, sd, cd);
    for (int i = 0; i < 6; ++i) {
        for (int j = 0; j < 6; ++j) xx[j] = x[j];
        xx[i] = x[i] + eps;
        tg_f_cont(c.p, c.model, xx, d, delta, sd, cd, fp);
        xx[i] = x[i] - eps;
        tg_f_cont(c.p, c.model, xx, d, delta, sd, cd, fm);
        for (int r = 0; r < 6; ++r) Jx[r][i] = (fp[r] - fm[r]) / (2.0 * eps);
    }
    tg_f_cont(c.p, c.model, x, d + eps, delta, sd, cd, fp);
    tg_f_cont(c.p, c.model, x, d - eps, delta, sd, cd, fm);
    for (int r = 0; r < 6; ++r) Ju[r][0] = (fp[r] - fm[r]) / (2.0 * eps);
    {
        double s2, c2;
        TG_SINCOS(delta + eps, s2, c2);
        tg_f_cont(c.p, c.model, x, d, delta + eps, s2, c2, fp);
        TG_SINCOS(delta - eps, s2, c2);
        tg_f_cont(c.p, c.model, x, d, delta - eps, s2, c2, fm);
        for (int r = 0; r < 6; ++r) Ju[r][1] = (fp[r] - fm[r]) / (2.0 * eps);
    }
    tg_f_cont(c.p, c.model, x, d, delta, sd, cd, f0);
    const double Ts = c.Ts;
    double Ad[6][6], Bd[6][2], g[6];
    for (int r = 0; r < 6; ++r) {
        for (int j = 0; j < 6; ++j) Ad[r][j] = ((r == j) ? 1.0 : 0.0) + Ts * Jx[r][j];
        Bd[r][0] = Ts * Ju[r][0];
        Bd[r][1] = Ts * Ju[r][1];
    }
    for (int r = 0; r < 6; ++r) {
        double ax = 0.0;
        for (int j = 0; j < 6; ++j) ax += Ad[r][j] * x[j];
        g[r] = x[r] + Ts * f0[r] - ax - (Bd[r][0] * d + Bd[r][1] * delta);
    }
    rec[0] = Ad[0][2]; rec[1] = Ad[0][3]; rec[2] = Ad[0][4];
    rec[3] = Ad[1][2]; rec[4] = Ad[1][3]; rec[5] = Ad[1][4];
    rec[6] = Ad[2][5];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) rec[7 + 3 * i + j] = Ad[3 + i][3 + j];
    rec[16] = Bd[3][0]; rec[17] = Bd[3][1]; rec[18] = Bd[4][1]; rec[19] = Bd[5][1];   // Bd[4][0] = Bd[5][0] = 0 exactly (f4, f5 do not see d)
    if (gout)
        for (int i = 0; i < 6; ++i) gout[i] = g[i];
}

// ------------------------------------------------------------------------------------------------
// Reference generators (MPC/main.py:28-47, 51-68)
__device__ __forceinline__ double tg_vref_at(int kind, const double *__restrict__ v, double t, double vx0)
{
    switch (kind) {
        case TG_VREF_HOLD: return vx0;
        case TG_VREF_CONST: return v[0];
        case TG_VREF_RAMP: return v[0] + (v[1] - v[0]) * tg_clamp(t / v[2], 0.0, 1.0);
        case TG_VREF_TRAPEZOID: {
            const double v0 = v[0], vmax = v[1], t_acc = v[2], t_flat = v[3], t_dec = v[4];
            double r = (t <= t_acc) ? v0 + (vmax - v0) * (t / t_acc) : vmax;
            if (t > t_acc + t_flat) r = vmax - (vmax - v0) * ((t - (t_acc + t_flat)) / t_dec);
            return tg_clamp(r, v0, vmax);
        }
        default: return v[0] + v[1] * tg_sin(2.0 * 3.141592653589793 * t / v[2]);
    }
}

__device__ __forceinline__ void tg_path_at(const tg_ref_spec &s, const double *__restrict__ brk,
                                           const double *__restrict__ coef, double xs, double &y, double &dy)
{
    if (s.path_kind == TG_PATH_PARABOLA) {
        y = s.path[0] * (xs * xs) + s.path[1] * xs + s.path[2];
        dy = 2.0 * s.path[0] * xs + s.path[1];
    } else if (s.path_kind == TG_PATH_SINE) {
        double sn, cs;
        TG_SINCOS(s.path[1] * xs + s.path[2], sn, cs);
        y = s.path[0] * sn + s.path[3];
        dy = s.path[0] * s.path[1] * cs;
    } else {
        int lo = 0;
        const int K = s.spline_count;
        const double *b = brk + s.spline_first;
        while (lo + 1 < K && xs >= b[lo + 1]) ++lo;
        const double *cc = coef + 4 * (size_t)(s.spline_first + lo);
        const double dx = xs - b[lo];
        y = ((cc[0] * dx + cc[1]) * dx + cc[2]) * dx + cc[3];
        dy = (3.0 * cc[0] * dx + 2.0 * cc[1]) * dx + cc[2];
    }
}

// Parametric path (TG_PATH_ARC): x(s) in pieces [first, first + K), y(s) in pieces [first + K, first + 2K) of the coefficient
// table, one set of breaks (the first K entries).  `lo` is the caller's running piece index (s mostly advances).
__device__ __forceinline__ void tg_arc_eval(const tg_ref_spec &s, const double *__restrict__ brk, const double *__restrict__ coef,
                                            double sv, int &lo, double &x, double &y, double &dx, double &dy)
{
    const int K = s.spline_count;
    const double *b = brk + s.spline_first;
    if (sv < b[lo]) lo = 0;
    while (lo + 1 < K && sv >= b[lo + 1]) ++lo;
    const double *cx = coef + 4 * (size_t)(s.spline_first + lo), *cy = cx + 4 * (size_t)K;
    const double d = sv - b[lo];
    x = ((cx[0] * d + cx[1]) * d + cx[2]) * d + cx[3];
    y = ((cy[0] * d + cy[1]) * d + cy[2]) * d + cy[3];
    dx = (3.0 * cx[0] * d + 2.0 * cx[1]) * d + cx[2];
    dy = (3.0 * cy[0] * d + 2.0 * cy[1]) * d + cy[2];
}
#define TG_ARC_PROJECT_ITERS 4
// parameter of the path point closest to (X, Y): a fixed number of Gauss-Newton steps from s_guess (oracle/refgen.py arc_project)
__device__ __forceinline__ double tg_arc_project(const tg_ref_spec &s, const double *__restrict__ brk, const double *__restrict__ coef,
                                                 double s_guess, double X, double Y, int &lo)
{
    double sv = s_guess;
    for (int it = 0; it < TG_ARC_PROJECT_ITERS; ++it) {
        double x, y, dx, dy;
        tg_arc_eval(s, brk, coef, sv, lo, x, y, dx, dy);
        sv = sv + ((X - x) * dx + (Y - y) * dy) / (dx * dx + dy * dy);
    }
    return sv;
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller with fixed polynomial kernels: bit-identical to oracle/philox_ref.c
// (same operations in the same order; __d*_rn / __fma_rn keep nvcc from contracting differently).
__device__ __forceinline__ void tg_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1, uint32_t out[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ double tg_log_u(uint32_t r)
{
    const unsigned long long mm = 2ull * r + 1ull;
    int e = 63 - __clzll((long long)mm);
    double f = __dmul_rn((double)mm, __longlong_as_double((long long)(1023 - e) << 52));  // exact scaling by 2^-e
    if (f > 1.4142135623730951) { f = __dmul_rn(f, 0.5); e += 1; }
    const double s = __ddiv_rn(__dadd_rn(f, -1.0), __dadd_rn(f, 1.0));
    const double s2 = __dmul_rn(s, s);
    double pl = 1.0 / 27.0;
    pl = __fma_rn(pl, s2, 1.0 / 25.0);
    pl = __fma_rn(pl, s2, 1.0 / 23.0);
    pl = __fma_rn(pl, s2, 1.0 / 21.0);
    pl = __fma_rn(pl, s2, 1.0 / 19.0);
    pl = __fma_rn(pl, s2, 1.0 / 17.0);
    pl = __fma_rn(pl, s2, 1.0 / 15.0);
    pl = __fma_rn(pl, s2, 1.0 / 13.0);
    pl = __fma_rn(pl, s2, 1.0 / 11.0);
    pl = __fma_rn(pl, s2, 1.0 / 9.0);
    pl = __fma_rn(pl, s2, 1.0 / 7.0);
    pl = __fma_rn(pl, s2, 1.0 / 5.0);
    pl = __fma_rn(pl, s2, 1.0 / 3.0);
    pl = __fma_rn(pl, s2, 1.0);
    const double lf = __dmul_rn(__dmul_rn(2.0, s), pl);
    return __fma_rn((double)(e - 33), 0.6931471805599453, lf);
}

__device__ __forceinline__ void tg_sincos_2pi_u(uint32_t r, double &sn, double &cs)
{
    const unsigned long long mm = 2ull * r + 1ull;
    const uint32_t oct = (uint32_t)(mm >> 30);
    const unsigned long long frac = mm & ((1ull << 30) - 1);
    double t = __dmul_rn((double)frac, 9.313225746154785e-10);  // 2^-30
    if (oct & 1u) t = __dadd_rn(1.0, -t);
    const double a = __dmul_rn(t, 0.7853981633974483);
    const double a2 = __dmul_rn(a, a);
    double ps = -1.0 / 1307674368000.0;
    ps = __fma_rn(ps, a2, 1.0 / 6227020800.0);
    ps = __fma_rn(ps, a2, -1.0 / 39916800.0);
    ps = __fma_rn(ps, a2, 1.0 / 362880.0);
    ps = __fma_rn(ps, a2, -1.0 / 5040.0);
    ps = __fma_rn(ps, a2, 1.0 / 120.0);
    ps = __fma_rn(ps, a2, -1.0 / 6.0);
    ps = __fma_rn(ps, a2, 1.0);
    const double sk = __dmul_rn(a, ps);
    double pc = 1.0 / 20922789888000.0;
    pc = __fma_rn(pc, a2, -1.0 / 87178291200.0);
    pc = __fma_rn(pc, a2, 1.0 / 479001600.0);
    pc = __fma_rn(pc, a2, -1.0 / 3628800.0);
    pc = __fma_rn(pc, a2, 1.0 / 40320.0);
    pc = __fma_rn(pc, a2, -1.0 / 720.0);
    pc = __fma_rn(pc, a2, 1.0 / 24.0);
    pc = __fma_rn(pc, a2, -0.5);
    const double ck = __fma_rn(pc, a2, 1.0);
    // octant symmetries without a branch (lanes of a warp hold different octants): sin takes the cosine kernel in
    // octants 1,2,5,6; sin < 0 in octants 4-7; cos < 0 in octants 2-5.  Same values as an 8-way switch.
    const bool swap = ((oct + 1u) & 2u) != 0u;
    const double s0 = swap ? ck : sk, c0 = swap ? sk : ck;
    sn = (oct & 4u) ? -s0 : s0;
    cs = ((oct + 2u) & 4u) ? -c0 : c0;
}

__device__ __forceinline__ void tg_box_muller(uint32_t r0, uint32_t r1, double &n0, double &n1)
{
    const double rad = __dsqrt_rn(__dmul_rn(-2.0, tg_log_u(r0)));
    double sn, cs;
    tg_sincos_2pi_u(r1, sn, cs);
    n0 = __dmul_rn(rad, cs);
    n1 = __dmul_rn(rad, sn);
}

// six standard normals of (seed,row): X, Y, phi, vx, vy, omega
__device__ __forceinline__ void tg_noise_row(unsigned long long seed, uint32_t row, double out[6])
{
    uint32_t a[4], b[4];
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    tg_philox4x32_10(row, 0u, 0u, 0u, k0, k1, a);
    tg_philox4x32_10(row, 1u, 0u, 0u, k0, k1, b);
    tg_box_muller(a[0], a[1], out[0], out[1]);
    tg_box_muller(a[2], a[3], out[2], out[3]);
    tg_box_muller(b[0], b[1], out[4], out[5]);
}
