/* trajgen.h -- C ABI of libtrajgen.so: batched closed-loop MPC trajectory generation on B200 (sm_100a).
 *
 * Drop-in boundary for ONE hot path of DorianaG01/trajectory_generation (paths below are relative to
 * the reference root).  The reference has no FFI of its own: the path is plain Python,
 *   MPC/mpc_6stati.py:120-275  mpc_step(x0, u_prev, path_ref, Ts, N, params, q_c, q_phi, q_vx, R, Rd,
 *                                       vref, u_bounds, du_bounds, x_lo, x_hi, solver, verbose)
 *                               -> (u_cmd[2], status:str, info:dict)
 *   MPC/main.py:85-101          the closed loop that calls it and integrates the plant
 *   generation_traj/generation_type{1,2}.py  the dataset shell (x0, clipping, noise, CSV rows)
 * so the entry points here are what a ctypes binding of that path needs (INTEGRATION.md shows the stub).
 *
 * Conventions: plain pointers and sizes, no framework types.  Functions without a suffix take DEVICE
 * pointers and enqueue on the handle's stream (asynchronous); *_host functions take HOST pointers and
 * return after the results are in the caller's buffers.  All arrays are C-contiguous fp64 unless noted,
 * one contiguous block per problem ("[B][6]" = B rows of 6).  Return value: 0 = ok, <0 = error
 * (tg_last_error() gives the message).  A handle is bound to one device and one stream and is not
 * thread-safe; use one handle per thread/stream.
 *
 * Environment variables read by the library (development / measurement knobs; none is needed in production and none changes
 * results beyond rounding -- the GPU tests pin that for TRAJGEN_PPC).  tg_create reads them: a handle keeps what they were
 * when it was created.
 *   TRAJGEN_PPC=<p>            problems per CTA of the fused kernels (default: chosen per launch, 1-4)
 *   TRAJGEN_DYNAMIC_N=1        use the run-time-horizon kernel where a compile-time-horizon instance (N = 10, 20, 40, 50) exists
 *   TRAJGEN_NO_TYRE_TABLE=1    evaluate the tyre curve / slip-angle atan with libdevice instead of the handle's tables
 *   TRAJGEN_LIB=<path>         (Python layer only) load this shared library instead of the in-tree libtrajgen.so
 */
#ifndef TRAJGEN_H
#define TRAJGEN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TG_VERSION 100

/* error codes */
#define TG_OK 0
#define TG_ERR_INVALID (-1)      /* bad argument / config */
#define TG_ERR_UNSUPPORTED (-2)  /* horizon / state-bound rows do not fit the kernel's shared memory */
#define TG_ERR_CUDA (-3)         /* CUDA runtime error */
#define TG_ERR_NOMEM (-4)

/* per-problem solver status (mpc_step's status strings, MPC/mpc_6stati.py:257-262) */
#define TG_STATUS_OPTIMAL 0            /* "optimal" */
#define TG_STATUS_OPTIMAL_INACCURATE 1 /* "optimal_inaccurate" (accepted, :261) */
#define TG_STATUS_INFEASIBLE 2         /* "infeasible"  -> u_cmd = u_prev */
#define TG_STATUS_UNBOUNDED 3          /* "unbounded"   (cannot occur: R > 0; kept for the mapping) */
#define TG_STATUS_USER_LIMIT 4         /* "user_limit"  (max_iter reached) -> u_cmd = u_prev */
#define TG_STATUS_NAN 5                /* "Solver Error: ..." (non-finite data or diverged iteration) -> u_cmd = u_prev */
#define TG_NUM_STATUS 6

/* dynamics variants (SURVEY.md section 2.1) */
#define TG_MODEL_MPC 0   /* MPC/mpc_6stati.py:25-71 */
#define TG_MODEL_GEN1 1  /* generation_traj/generation_type1.py:38-68 */
#define TG_MODEL_GEN2 2  /* generation_traj/generation_type2.py:52-86 */
/* plant post-step clipping: MPC/main.py:97 has none; generation_type1.py:81-82 / type2:186-187 clip */
#define TG_PLANT_MPC 0   /* MPC model, no clipping */
#define TG_PLANT_GEN1 1  /* gen1 model + vx>=0, |omega|<=6 */
#define TG_PLANT_GEN2 2  /* gen2 model + vx>=0, |omega|<=6 */

#define TG_JAC_ANALYTIC 0 /* closed-form Jacobians of f_cont */
#define TG_JAC_FD 1       /* central differences eps=1e-5, MPC/mpc_6stati.py:73-97 verbatim */

/* reference path kinds (MPC/main.py:64-66, MPC/README.md:68-76) */
#define TG_PATH_PARABOLA 0 /* y = p0 x^2 + p1 x + p2 */
#define TG_PATH_SINE 1     /* y = p0 sin(p1 x + p2) + p3 */
#define TG_PATH_SPLINE 2   /* piecewise cubic y(x): breaks/coef table, scipy PPoly layout */
#define TG_PATH_ARC 3      /* arclength-parameterised path (x(s), y(s)): two cubic-spline tables over s, see tg_ref_spec */
/* velocity-reference kinds (MPC/mpc_6stati.py:158-163, MPC/main.py:28-47) */
#define TG_VREF_HOLD 0      /* vref=None -> x0[3] */
#define TG_VREF_CONST 1     /* v[0] */
#define TG_VREF_RAMP 2      /* v0=v[0], v_cruise=v[1], tramp=v[2] */
#define TG_VREF_TRAPEZOID 3 /* v0, vmax, t_acc, t_flat, t_dec */
#define TG_VREF_SINE 4      /* v_mean, v_amp, period_s */

#define TG_INF 1e20

/* Order of params[]: Cm1 Cm2 Cr0 Cr2 Br Cr Dr Bf Cf Df m Iz lf lr g maxAlpha vx_zero (MPC/mpc_6stati.py:9-19) */
#define TG_NPARAMS 17

typedef struct tg_config {
    int32_t N;               /* horizon (mpc_step N=20; MPC/main.py uses 40) */
    int32_t model;           /* TG_MODEL_* used by the controller's linearisation */
    int32_t plant;           /* TG_PLANT_* used by tg_closed_loop */
    int32_t jacobian;        /* TG_JAC_* */
    double Ts;
    double params[TG_NPARAMS];
    double q_c, q_phi, q_vx; /* MPC/mpc_6stati.py:128-130 */
    double R[4], Rd[4];      /* row-major 2x2, :131-132 (symmetric part is used, like cp.quad_form) */
    double u_lo[2], u_hi[2];   /* :135-136 */
    double du_lo[2], du_hi[2]; /* :137-138 */
    double x_lo[6], x_hi[6];   /* :139-140; <= -TG_INF / >= TG_INF = absent */
    /* ADMM (OSQP-style) settings */
    double rho, sigma, alpha, eps_abs, eps_rel, eps_prim_inf, adaptive_rho_tol;
    double alpha_warm;       /* relaxation of the first 4 check intervals of a WARM-started solve (then alpha); <= 0 = alpha */
    int32_t max_iter, check_every, adaptive_rho, adaptive_rho_min_iter;
    int32_t warm_start;      /* closed loop: shift-warm-start across steps; step API: keep per-problem state */
    int32_t vref_advance;    /* 0 = the reference's behaviour (window never advances, MPC/main.py:87) */
    /* sensor noise (generation_type1.py:25-32,255) */
    double noise_std[6];
    uint64_t noise_seed_base;
    int32_t threads_per_problem; /* reserved, must be 0: the launch geometry follows from N (tg_info reports it) */
    int32_t solver_flags;        /* bit 0: do NOT start solves that have no active row in "free" mode (rho 1e-6, alpha 1; DESIGN.md 2) */
} tg_config;

/* one reference scenario per trajectory (closed loop) */
typedef struct tg_ref_spec {
    int32_t path_kind;
    int32_t vref_kind;
    int32_t spline_first;  /* first piece of this trajectory in the spline tables */
    int32_t spline_count;  /* number of pieces K: spl_breaks[first+i] = start of piece i, spl_coef[first+i][4] =
                              (c0,c1,c2,c3) of y = ((c0 dx + c1) dx + c2) dx + c3, dx = x - start; either end extrapolates
                              its end piece (scipy PPoly behaviour).
                              TG_PATH_ARC: the path is (x(s), y(s)); x(s) = pieces [first, first + K), y(s) = pieces
                              [first + K, first + 2K) of spl_coef over the breaks spl_breaks[first .. first + K); path[0] = the
                              parameter s from which the point closest to the vehicle is searched on the first step (the
                              closed loop tracks it afterwards).  The window of MPC/main.py:51-68 then advances along the
                              path by the arclength vref Ts, and phi* = atan2(y', x') is unwrapped along the window, starting
                              within pi of the vehicle's heading (csrc/tw_solver.cuh tw_ref_window_warp; oracle/refgen.py) */
    double path[4];
    double vref[6];
} tg_ref_spec;

/* per-problem (step API) / per-trajectory (closed loop) controller settings for the *_ctrl entry points.  The fields mean
 * what the same fields of tg_config mean, and the symmetric parts of R and Rd are used.  +-TG_INF = absent.  Everything else
 * stays per handle: N, Ts, model, plant, Jacobian mode, vehicle parameters, noise, the solver settings, and WHICH state
 * components carry bounds (tg_config's x_lo / x_hi fix that set, and with it the shared-memory layout).  A row may give any
 * finite or infinite bound on a component the handle bounds.  Rules (checked by tg_check_ctrl and by the *_host entry points,
 * which return TG_ERR_INVALID naming the first bad row and field before anything is launched; preconditions of the
 * device-pointer ones): weights finite and >= 0; R, Rd finite, the symmetric part of R positive definite, that of Rd positive
 * semidefinite; lo <= hi for every bound; no finite x_lo / x_hi on a state component the handle does not bound.
 * (The vehicle that the closed loop integrates -- its plant -- can be set per trajectory as well: see tg_closed_loop_params.) */
typedef struct tg_ctrl_spec {
    double q_c, q_phi, q_vx;
    double R[4], Rd[4];        /* row-major 2x2 */
    double u_lo[2], u_hi[2];
    double du_lo[2], du_hi[2];
    double x_lo[6], x_hi[6];
} tg_ctrl_spec;

/* the rules of tg_ctrl_spec for the host table ctrl[B], for a handle that bounds state component i when bit i of
 * bounded_states is set.  TG_OK, or TG_ERR_INVALID with tg_last_error() = "ctrl row b: <field> <why>" for the first bad row.
 * Needs no handle and no GPU. */
int tg_check_ctrl(int B, const tg_ctrl_spec *ctrl, uint32_t bounded_states);

/* ---- per-trajectory plant parameters (the *_params entry points).  plant[B][TG_NPARAMS] (fp64, the order of params[]): row b
 * is the vehicle that trajectory b's ground truth integrates for all of its steps -- the closed-loop plant step (MPC/main.py:97,
 * with the clipping of generation_type1.py:81-82 / generation_type2.py:186-187 for the generator plants), tg_plant_rollout's
 * integration and the open-loop generators' (generation_type1.py:70-84, generation_type2.py:180-187).  NULL = the handle's
 * params for every trajectory.  The table changes nothing else: the controller's rollout, linearisation and QP keep the
 * handle's params (a plant that differs from the controller's model), and so do the reference windows, the sensor noise,
 * tg_make_scenarios' u0 and the plant variant.  g is unused, as everywhere.
 * Tyre curve: a row whose Bf, Cf, Br, Cr and maxAlpha equal the handle's bit for bit, on a handle whose tables are in use
 * (tg_tyre_table_info), evaluates the handle's tyre-curve and slip-angle tables; any other row evaluates atan2 / atan / sin with
 * libdevice (the tables are fitted and verified for the handle's constants only).  So row b gives the bits that a handle created
 * with params = row b gives -- with TRAJGEN_NO_TYRE_TABLE=1 when its tyre constants differ from the handle's.  Varying masses,
 * inertias, motor / drag constants or tyre peaks (D) keeps the tables; varying B, C or maxAlpha costs libdevice in the plant.
 * Rules: every entry finite; m, Iz, vx_zero and maxAlpha > 0.  tg_check_plant_params checks them (no handle, no GPU needed):
 * TG_OK, or TG_ERR_INVALID with tg_last_error() = "plant row b: <name> <why>" for the first bad row.  The *_host entry points
 * check them before anything is launched; for the device-pointer ones they are a precondition. */
int tg_check_plant_params(int B, const double *plant);

typedef struct tg_handle tg_handle;

const char *tg_last_error(void);
int tg_version(void);
void tg_default_config(tg_config *cfg); /* mpc_step's defaults (N=20, Ts=0.02, weights, bounds) + OSQP-like solver settings */

int tg_create(const tg_config *cfg, int device, tg_handle **out);
int tg_destroy(tg_handle *h);
int tg_set_stream(tg_handle *h, void *cuda_stream);
int tg_synchronize(tg_handle *h);
int tg_kernel_launches(tg_handle *h, int64_t *count); /* kernels launched through this handle so far */
/* launch geometry of one problem: resident problems per SM, threads per problem, dynamic shared memory per problem, SM count
 * (the 64-thread kernels place up to 8 problems side by side in one CTA; DESIGN.md section 3) */
/* the tyre-curve table of this handle (DESIGN.md section 3): whether the kernels use it (in_use bit 0; bit 1 = the
 * slip-angle atan table is in use as well), and its largest deviation
 * from libm (value of sin(C atan(B alpha)), slope) on the check grid of tg_create */
int tg_tyre_table_info(tg_handle *h, int32_t *in_use, double *max_value_err, double *max_slope_err);
int tg_info(tg_handle *h, int32_t *ctas_per_sm, int32_t *threads_per_cta, int32_t *smem_bytes, int32_t *num_sms);

/* K1 tap -- replaces MPC/mpc_6stati.py:165-178 (rollout + N x linearize_discretize).
 * x0[B][6], u_prev[B][2] -> A[B][N][6][6], Bm[B][N][6][2], g[B][N][6], xbar[B][N+1][6] (any output may be NULL) */
int tg_linearize(tg_handle *h, int B, const double *x0, const double *u_prev,
                 double *A, double *Bm, double *g, double *xbar);

/* K2 tap -- condensed form of the QP of MPC/mpc_6stati.py:180-252 in dU = U - u_prev:
 * min 1/2 dU'H dU + q'dU + c0,  l <= [I; D; Gs] dU <= u.   H[B][n][n], q[B][n], c0[B], l/u[B][m], Gs[B][ms][n]
 * with n = 2N, m = 4N + ms, ms = (#bounded states) * N.  Outputs may be NULL. */
int tg_assemble(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref,
                const double *vref, double *H, double *q, double *c0, double *l, double *u, double *Gs);

/* K1+K2+K3 -- replaces mpc_step (MPC/mpc_6stati.py:120-275), batched.
 * x0[B][6], u_prev[B][2], path_ref[B][N+1][3], vref[B][N+1] (NULL = hold x0[3], :158-159)
 * -> u_cmd[B][2], status[B], iters[B], objective[B], U_opt[B][N][2], X_opt[B][N+1][6], y_opt[B][m] (optional outputs may be NULL) */
int tg_mpc_step(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref,
                const double *vref, double *u_cmd, int32_t *status, int32_t *iters, double *objective,
                double *U_opt, double *X_opt, double *y_opt);
int tg_mpc_step_host(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref,
                     const double *vref, double *u_cmd, int32_t *status, int32_t *iters, double *objective,
                     double *U_opt, double *X_opt, double *y_opt);
/* the same with problem b solved under its own settings ctrl[b] (tg_ctrl_spec); ctrl == NULL is tg_mpc_step[_host] */
int tg_mpc_step_ctrl(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref,
                     const double *vref, const tg_ctrl_spec *ctrl, double *u_cmd, int32_t *status, int32_t *iters,
                     double *objective, double *U_opt, double *X_opt, double *y_opt);
int tg_mpc_step_ctrl_host(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref,
                          const double *vref, const tg_ctrl_spec *ctrl, double *u_cmd, int32_t *status, int32_t *iters,
                          double *objective, double *U_opt, double *X_opt, double *y_opt);

/* a10 tap -- MPC/main.py:28-47,51-68: reference window for the current state.
 * x0[B][6], spec[B], step index t -> path_ref[B][N+1][3], vref[B][N+1] */
int tg_ref_window(tg_handle *h, int B, const double *x0, const tg_ref_spec *spec, const double *spl_breaks,
                  const double *spl_coef, int t_index, double *path_ref, double *vref);

/* fused K1..K4 -- replaces the loop MPC/main.py:85-101 plus the dataset shell
 * (generation_type2.py:180-200): T closed-loop steps for B trajectories.
 * x0[B][6], u0[B][2], spec[B], spline tables (may be NULL), traj_id0 = global id of trajectory 0 of this batch
 * -> clean[B][T+1][6] (row 0 = x0), noisy[B][T+1][6], U[B][T][2], status_counts[B][TG_NUM_STATUS], iters_total[B] */
int tg_closed_loop(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                   const double *spl_breaks, const double *spl_coef, int64_t traj_id0, double *clean,
                   double *noisy, double *U, int32_t *status_counts, int64_t *iters_total);
int tg_closed_loop_host(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                        const double *spl_breaks, int64_t n_breaks, const double *spl_coef, int64_t n_coef,
                        int64_t traj_id0, double *clean, double *noisy, double *U, int32_t *status_counts,
                        int64_t *iters_total);
/* the same with trajectory b controlled under its own settings ctrl[b] (tg_ctrl_spec) for all its T steps;
 * ctrl == NULL is tg_closed_loop[_host] */
int tg_closed_loop_ctrl(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                        const tg_ctrl_spec *ctrl, const double *spl_breaks, const double *spl_coef, int64_t traj_id0,
                        double *clean, double *noisy, double *U, int32_t *status_counts, int64_t *iters_total);
int tg_closed_loop_ctrl_host(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                             const tg_ctrl_spec *ctrl, const double *spl_breaks, int64_t n_breaks, const double *spl_coef,
                             int64_t n_coef, int64_t traj_id0, double *clean, double *noisy, double *U,
                             int32_t *status_counts, int64_t *iters_total);
/* the same with trajectory b's plant integrated with the vehicle plant[b] (see tg_check_plant_params) while its controller keeps
 * the handle's model.  ctrl and plant may each be NULL; (NULL, NULL) is tg_closed_loop[_host].  ctrl == NULL runs the handle's
 * own kernel instances (the compile-time horizons included), ctrl != NULL the ctrl instances. */
int tg_closed_loop_params(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                          const tg_ctrl_spec *ctrl, const double *plant, const double *spl_breaks, const double *spl_coef,
                          int64_t traj_id0, double *clean, double *noisy, double *U, int32_t *status_counts,
                          int64_t *iters_total);
int tg_closed_loop_params_host(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                               const tg_ctrl_spec *ctrl, const double *plant, const double *spl_breaks, int64_t n_breaks,
                               const double *spl_coef, int64_t n_coef, int64_t traj_id0, double *clean, double *noisy,
                               double *U, int32_t *status_counts, int64_t *iters_total);

/* ---- scenario + initial-state generation on the device (SURVEY.md 8(d) configs 2, 3, 5): x0 from the ranges of
 * generation_type1.py:260-265 / generation_type2.py:171-174 (Y and phi relative to the reference path), one reference path
 * per trajectory (natural cubic spline through random knots / sinusoid / parabola, by id mod n_cycle), ramp-cruise speed
 * profile.  Every number is a function of seed_base + global trajectory id (Philox4x32-10; layout in csrc/tg_scenarios.cuh,
 * restated by oracle/scenarios.py).  spline tables: spl_knots - 1 pieces per trajectory, trajectory b at [b * (spl_knots - 1)]. */
typedef struct tg_scenario_rules {
    double x0_lo[6], x0_hi[6];   /* X, -, -, vx, vy, omega ranges (entries 1, 2 unused: Y, phi follow the path) */
    double lat_off[2], head_off[2]; /* lateral / heading offset from the path at X */
    double vref0, vcruise[2], t_ramp; /* vref ramps from vref0 to U(vcruise) over t_ramp seconds (MPC/main.py:28-32) */
    double sine_A[2], sine_k[2], sine_psi[2]; /* y = A sin(k x + psi), MPC/README.md:75 has A = k = 0.5 */
    double parab_c[2];           /* y = c x^2, MPC/main.py:64 has c = 0.1 */
    double spl_x0, spl_dx[2], spl_sigma; /* knots from x = spl_x0 every U(spl_dx) m, ordinates N(0, spl_sigma^2) */
    int32_t spl_knots;           /* 3 .. 32 */
    int32_t n_cycle, cycle[4];   /* path kind of trajectory id i = cycle[i mod n_cycle] (TG_PATH_PARABOLA / SINE / SPLINE) */
    int32_t reserved;
    uint64_t seed_base;
} tg_scenario_rules;
void tg_default_scenario_rules(tg_scenario_rules *r); /* BASELINE config 2: spline / sinusoid by id parity, generation_type1's x0 ranges */
/* DEVICE pointers: x0[B][6], u0[B][2] (steady-state duty cycle at vx, 0), spec[B], spl_breaks[B][spl_knots-1], spl_coef[B][spl_knots-1][4] */
int tg_make_scenarios(tg_handle *h, int B, int64_t traj_id0, const tg_scenario_rules *rules, double *x0, double *u0,
                      tg_ref_spec *spec, double *spl_breaks, double *spl_coef);
int tg_make_scenarios_host(tg_handle *h, int B, int64_t traj_id0, const tg_scenario_rules *rules, double *x0, double *u0,
                           tg_ref_spec *spec, double *spl_breaks, double *spl_coef);

/* K4 taps -- plant + noise.  tg_plant_rollout: open-loop Euler integration with the configured plant
 * (generation_type1.py:70-84): x0[B][6], U[B][T][2] -> X[B][T+1][6].
 * tg_sensor_noise: standard normals [n_traj][n_rows][6] for seeds seed_base + traj_id0 + i (Philox4x32-10).
 * tg_philox_u32: raw stream, out[n][4] = philox(ctr=(first+i, block, 0, 0), key=seed). */
int tg_plant_rollout(tg_handle *h, int B, int T, const double *x0, const double *U, double *X);
/* the same with trajectory b integrated with the vehicle plant[b][TG_NPARAMS] (NULL = tg_plant_rollout; see tg_check_plant_params) */
int tg_plant_rollout_params(tg_handle *h, int B, int T, const double *x0, const double *U, const double *plant, double *X);
int tg_sensor_noise(tg_handle *h, int64_t traj_id0, int n_traj, int n_rows, double *out);
int tg_philox_u32(tg_handle *h, uint64_t seed, uint32_t first, uint32_t block, int n, uint32_t *out);

/* ---- open-loop generators (SURVEY.md section 8(f) rank 2): the control synthesis of the two generator scripts, fused
 * with the plant integration and the sensor noise.  The handle supplies Ts, the plant (TG_PLANT_GEN1 / TG_PLANT_GEN2),
 * params, noise_std and noise_seed_base; N and the MPC settings are ignored.  Random numbers: Philox4x32-10 keyed by
 * ctrl_seed_base + traj_id0 + i (controls) and noise_seed_base + traj_id0 + i (sensor noise) -- the reference's
 * distributions and seeding contract with a counter-based stream (layout: oracle/openloop.py). */
typedef struct tg_type1_rules {          /* generation_type1.py */
    double d_mean, d_std, delta_mean, delta_std; /* mpc_stats :250 */
    double du_lo[2], du_hi[2];           /* slew per step (d, delta) :251 */
    double u_lo[2], u_hi[2];             /* final clip :288-289 */
    double transient_s[2];               /* duration of the spline transient, uniform :110 */
    double checkpoint_s[2];              /* knot spacing of the transient spline, uniform :90 */
    double period_s[2], amp_frac[2];     /* steering sinusoid: period, amplitude / delta_std :122 */
    double p_straight;                   /* P(mode = straight) :108 */
    double tr_d_frac, tr_delta_frac;     /* knot sigma / (d_std, delta_std) :115 */
    double st_d_frac;                    /* steady d sigma / d_std :118 */
    double sin_noise_frac, straight_frac;/* steady delta sigma / delta_std, sinusoid :124 and straight :128 */
    double ctrl_noise_frac;              /* high-frequency control noise sigma / std :283-284 */
    int32_t mode;                        /* -1 = 'random', 0 = 'straight', 1 = 'sinusoid' (:105) */
    int32_t reserved;
} tg_type1_rules;

typedef struct tg_type2_rules {          /* generation_type2.py: ControlRules :21-30 + the literals of :97-149 */
    double v_turn_max, v_high;
    double d_range[2], delta_turn_range[2];
    double delta_straight_noise;
    double delta_rate_max;               /* rad/s :97 */
    double v_floor, d_boost_min;         /* :100 */
    double seg_s[2];                     /* segment duration, uniform :114 */
    double p_modes[4];                   /* accelerate, cruise, turn_left, turn_right :111-112 */
    double p_after_turn[2];              /* accelerate, cruise :109 */
    double acc_d_lo;                     /* accelerate: d ~ U(acc_d_lo, d_range[1]) :120 */
    double cruise_d[2];                  /* :122 */
    double turn_d_fast[2], turn_d_slow[2]; /* v > v_turn_max / otherwise :124 */
    double stall_v, stall_d[2], stall_min_s; /* :131-133 */
    double delta_clip;                   /* :141 */
} tg_type2_rules;

void tg_default_type1_rules(tg_type1_rules *r);
void tg_default_type2_rules(tg_type2_rules *r);

/* generation_type1.py:279-306 for B trajectories: x0[B][6] -> clean[B][T+1][6] (row 0 = x0), noisy[B][T+1][6],
 * U[B][T][2], modes[B] (0 straight / 1 sinusoid).  Outputs may be NULL; non-NULL clean/noisy/U must be 16-byte aligned. */
int tg_openloop_type1(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules, uint64_t ctrl_seed_base,
                      int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes);
/* generation_type2.py:95-157,176-200 for B trajectories; modes[B][T]: 0 accelerate, 1 cruise, 2 turn_left, 3 turn_right. */
int tg_openloop_type2(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules, uint64_t ctrl_seed_base,
                      int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes);
int tg_openloop_type1_host(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules, uint64_t ctrl_seed_base,
                           int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes);
int tg_openloop_type2_host(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules, uint64_t ctrl_seed_base,
                           int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes);
/* the same with trajectory b's ground truth integrated with the vehicle plant[b][TG_NPARAMS] (generation_type1.py:70-84,
 * generation_type2.py:180-187; NULL = the functions above; see tg_check_plant_params).  The control synthesis is unchanged;
 * type 2's shadow simulation reads the plant's state, so its controls follow the row's vehicle. */
int tg_openloop_type1_params(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules, uint64_t ctrl_seed_base,
                             int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes);
int tg_openloop_type2_params(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules, uint64_t ctrl_seed_base,
                             int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes);
int tg_openloop_type1_params_host(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules,
                                  uint64_t ctrl_seed_base, int64_t traj_id0, const double *plant, double *clean, double *noisy,
                                  double *U, int8_t *modes);
int tg_openloop_type2_params_host(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules,
                                  uint64_t ctrl_seed_base, int64_t traj_id0, const double *plant, double *clean, double *noisy,
                                  double *U, int8_t *modes);

/* ---- estimator-side physics (SURVEY.md section 8(f) rank 4): KalmanNet's prior step, fused.  DEVICE pointers (e.g. the
 * data_ptr() of torch CUDA tensors), dtype 0 = fp64, 1 = fp32 (torch's default, what the reference runs in); Ts and the
 * vehicle parameters come from the handle, the data-set limits (Params["x_min"] ... ["omega_max"],
 * KalmanNet/training.py:60-90) from `lim`. */
typedef struct tg_state_limits { double lo[6], hi[6]; } tg_state_limits;
/* VehicleModel.f, KalmanNet/vehicle_model.py:109-134 (with pt_f_cont :43-79): x[B][6], u[B][2] -> x_next[B][6] */
int tg_estimator_step(tg_handle *h, int B, int dtype, const void *x, const void *u, const tg_state_limits *lim, void *x_next);
/* its vector-Jacobian product as torch.autograd computes it: grad_x[B][6] = (d x_next / d x)^T grad_next, grad_u[B][2]
 * likewise (either may be NULL) -- lets the fused step sit inside KalmanNet's back-propagation through time */
int tg_estimator_step_vjp(tg_handle *h, int B, int dtype, const void *x, const void *u, const tg_state_limits *lim,
                          const void *grad_next, void *grad_x, void *grad_u);
/* rollout_open_loop, KalmanNet/test_prediction.py:68-87: x0[B][6], U[B][2][T_u] -> preds[B][6][Hn] with
 * Hn = min(H, T_u - t_start) (returned in *H_out; the caller sizes preds for H) */
int tg_estimator_rollout(tg_handle *h, int B, int dtype, int T_u, int t_start, int H, const void *x0, const void *U,
                         const tg_state_limits *lim, void *preds, int32_t *H_out);

/* host-side dataset writer -- replaces the DataFrame concat + to_csv of generation_type1.py:315-339 /
 * generation_type2.py:202-218,309-322.  HOST pointers clean[B][T+1][6], noisy[B][T+1][6], U[B][T][2]; writes the
 * clean file (with phi) and the noisy file (without), byte-identical to pandas' output for the same numbers
 * (shortest-repr floats, empty d/delta on each trajectory's last row, ids traj_id0 + i).  append != 0 continues an
 * existing file without a header (sharded / chunked generation).  Either path may be NULL.  n_threads <= 0 = all cores. */
int tg_write_csv(const char *clean_path, const char *noisy_path, int B, int T, double Ts, int64_t traj_id0,
                 const double *clean, const double *noisy, const double *U, int append, int n_threads);

/* host-side merge -- replaces generation_traj/merge_datasets.py:33-52 for one pair of files: out = rows of `first`
 * verbatim + rows of `second` with trajectory_id += offset, offset = id_offset if >= 0 else max(trajectory_id of first) + 1
 * (:42-45; the reference re-uses the clean files' offset for the noisy pair, :62-63).  Both files must have the same
 * header.  Text is copied, not re-parsed, so every number keeps its digits.  Outputs may be NULL. */
int tg_merge_csv(const char *first_path, const char *second_path, const char *out_path, int64_t id_offset,
                 int64_t *id_offset_used, int64_t *rows_written);

/* measured FMA peak of this GPU (roofline denominator): TFLOP/s for dtype 0 = fp64, 1 = fp32 */
int tg_fma_peak(tg_handle *h, int dtype, double *tflops);

/* host<->device helpers so a ctypes caller needs no other CUDA binding */
int tg_device_count(int *n);
int tg_malloc(void **dptr, int64_t bytes);                  /* on the calling thread's current device */
int tg_malloc_on(tg_handle *h, void **dptr, int64_t bytes); /* on the handle's device (use this one when several GPUs are in play) */
int tg_free(void *dptr);
int tg_memcpy_h2d(tg_handle *h, void *dst, const void *src, int64_t bytes);
int tg_memcpy_d2h(tg_handle *h, void *dst, const void *src, int64_t bytes);
int tg_malloc_host(void **hptr, int64_t bytes); /* pinned */
int tg_free_host(void *hptr);

#ifdef __cplusplus
}
#endif
#endif /* TRAJGEN_H */
