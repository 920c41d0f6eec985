// trajgen.cu -- kernels + C ABI (include/trajgen.h) of libtrajgen.so.  sm_100a only.
//
// Kernels (one CTA per problem / trajectory, persistent grid-stride over the batch):
//   tg_mpc_step_kernel     K1+K2+K3: replaces mpc_step, MPC/mpc_6stati.py:120-275
//   tg_closed_loop_kernel  fused K1..K4: replaces the loop MPC/main.py:85-101 + the dataset shell
//                          generation_type2.py:180-200 (plant clipping, sensor noise)
//   tg_ref_window_kernel   MPC/main.py:28-47,51-68
//   tg_plant_kernel        generation_type1.py:70-84 (open-loop integration with clipping; per-trajectory plant parameters)
//   tg_noise_kernel / tg_philox_kernel   Philox4x32-10 sensor-noise stream
//   tg_fma_peak_kernel     FMA micro-benchmark (roofline denominator)
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <initializer_list>
#include <new>
#include <string>
#include <vector>

#include "tw_solver.cuh"
#include "tg_openloop.cuh"
#include "tg_scenarios.cuh"
#include "tg_estimator.cuh"

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
void tg_internal_set_error(const char *msg) { g_err = msg; }   // for tg_csv.cpp
#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail(TG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

struct StepArgs {
    int B;
    const double *x0, *u_prev, *path_ref, *vref;
    double *u_cmd; int *status; int *iters; double *objective; double *U_opt, *X_opt, *y_opt;
    // taps
    double *A, *Bm, *g, *xbar, *H, *q, *c0, *l, *u, *Gs;
    int stop;
    double *ws_x, *ws_y; int *ws_valid;   // per-problem warm-start state (step API), may be null
    int ppc;                              // problems per CTA
    const tg_ctrl_spec *ctrl;             // [B] per-problem settings: read by the ctrl instances only (appended last, so that the
                                          // parameter offsets of every other instance stay as they were)
};

struct LoopArgs {
    int B, T;
    const double *x0, *u0;
    const tg_ref_spec *spec;
    const double *brk, *coef;
    long long traj_id0;
    double *clean, *noisy, *U;
    int *status_counts;
    long long *iters_total;
    int ppc;   // problems per CTA
    const tg_ctrl_spec *ctrl;   // [B] per-trajectory settings: read by the ctrl instances only (appended last, like StepArgs::ctrl)
    const double *plant;        // [B][TG_NPARAMS] per-trajectory plant parameters or null (appended last for the same reason)
};

// ------------------------------------------------------------------------------------------------ warp-per-problem kernels
// tw_solver.cuh: W warps per problem (W = 1 for N <= 14), P problems per CTA side by side, each with its own shared-memory
// block (and, for W > 1, its own named barrier TW_BAR_PROB + p).  Problems of a CTA are re-aligned at every step boundary
// (TW_BAR_STEP) so that they fetch the same instruction lines at the same time (the step body is ~100 KB of straight code).
#define TW_CTA_THREADS 512
enum { TW_BAR_PROB = 1, TW_BAR_STEP = 15 };
// register budget: 128 per thread on every shape (the tile takes 32 of them with S = 1, 64 with S = 2).  The kernels state it
// next to __launch_bounds__, so that ptxas gets both .maxntid and .maxnreg (without .maxntid the single-problem instances
// compile to different code, without .maxnreg all of them do); nvcc accepts the two qualifiers together only with a value
// that depends on a template parameter, hence the function template.
template <int S> constexpr int tw_regs() { return 128; }

// P1 = true: the single-problem-per-CTA instance.  Its only barrier id is the constant 1, so the kernel is built with 2
// hardware barriers instead of 16 (a barrier id held in a register makes ptxas reserve all 16, and an SM has 64: four
// resident CTAs at most, whatever the registers and the shared memory would allow).
// CT = true: the ctrl instance.  Each problem stages its own tg_ctrl_spec (a.ctrl[b]) behind its shared-memory block
// (tw_stage_ctrl, stride tw_stride(L) + TW_CTRL_DBL) and the solver takes its weights and bounds from there.
template <int W, int S, int NC, bool P1 = false, bool HS = (NC == 0), bool CT = false>
__global__ void __launch_bounds__(TW_CTA_THREADS) __maxnreg__(tw_regs<S>())
tw_mpc_step_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ WLayout L, const __grid_constant__ StepArgs a)
{
    extern __shared__ __align__(16) double sm_all[];
    constexpr int NT = 32 * W;
    const int P = P1 ? 1 : a.ppc;
    int prob = P1 ? 0 : threadIdx.x / NT, tid = P1 ? threadIdx.x : threadIdx.x % NT;
    unsigned sm_off = (unsigned)prob * (unsigned)(tw_stride(L) + (CT ? TW_CTRL_DBL : 0)) * 8u;
    if constexpr (!P1) asm volatile("" : "+r"(tid), "+r"(prob), "+r"(sm_off));   // kept in registers instead of being re-derived at every use
    const int bar = P1 ? TW_BAR_PROB : TW_BAR_PROB + prob;
    double *sm = reinterpret_cast<double *>(reinterpret_cast<char *>(sm_all) + sm_off);
    const int N = NC > 0 ? NC : c.N, n = 2 * N, ms = HS ? c.ms : 0;
    if (prob >= P) return;
    const TwMap<S> mp = tw_make_map<W, S>(LF(nb), tid);
    for (int b0 = blockIdx.x * P; b0 < a.B; b0 += gridDim.x * P) {
        const int b = b0 + prob;
        if (b >= a.B) break;
        tw_sync<W>(bar);
        if (tid < 6) sm[LF(x0) + tid] = a.x0[6 * (size_t)b + tid];
        if (tid < 2) sm[LF(uprev) + tid] = a.u_prev[2 * (size_t)b + tid];
        if constexpr (CT) tw_stage_ctrl(sm + tw_stride(L), a.ctrl + b, tid);
        const double vx0 = a.x0[6 * (size_t)b + 3];
        for (int k = tid; k <= N; k += NT) {
            if (a.path_ref) {
                const double *pr = a.path_ref + 3 * ((size_t)b * (N + 1) + k);
                sm[LF(Xr) + k] = pr[0]; sm[LF(Yr) + k] = pr[1]; sm[LF(Pr) + k] = pr[2];
            } else { sm[LF(Xr) + k] = 0.0; sm[LF(Yr) + k] = 0.0; sm[LF(Pr) + k] = 0.0; }
            sm[LF(vref) + k] = a.vref ? a.vref[(size_t)b * (N + 1) + k] : vx0;
        }
        bool warm = false, warm_free = false;
        if (a.ws_valid && c.warm_start && a.ws_valid[b]) {
            warm = true; warm_free = a.ws_valid[b] == 2;
            const size_t m = 2 * (size_t)n + ms;
            for (int i = tid; i < n; i += NT) sm[LF(x) + i] = a.ws_x[(size_t)b * n + i];
            for (int i = tid; i < 2 * n; i += NT) sm[LF(y) + i] = a.ws_y[b * m + i];
            for (int i = tid; i < ms; i += NT) sm[L.ys + i] = a.ws_y[b * m + 2 * n + i];
        }
        tw_sync<W>(bar);
        StepTaps tap;
        tap.A = a.A ? a.A + (size_t)b * N * 36 : nullptr;
        tap.Bm = a.Bm ? a.Bm + (size_t)b * N * 12 : nullptr;
        tap.g = a.g ? a.g + (size_t)b * N * 6 : nullptr;
        tap.xbar = a.xbar ? a.xbar + (size_t)b * (N + 1) * 6 : nullptr;
        tap.H = a.H ? a.H + (size_t)b * n * n : nullptr;
        tap.q = a.q ? a.q + (size_t)b * n : nullptr;
        tap.c0 = a.c0 ? a.c0 + b : nullptr;
        tap.l = a.l ? a.l + (size_t)b * (2 * n + ms) : nullptr;
        tap.u = a.u ? a.u + (size_t)b * (2 * n + ms) : nullptr;
        tap.Gs = a.Gs ? a.Gs + (size_t)b * c.ms * n : nullptr;
        tap.stop = a.stop;
        const StepResult r = tw_step_body<W, S, NC, HS, CT>(c, L, sm, mp, warm, warm_free, tap, nullptr, tid, bar,
                                                             CT ? reinterpret_cast<const TwCtrl *>(sm + tw_stride(L)) : nullptr);
        if (a.stop) continue;
        const bool ok = (r.status == TG_STATUS_OPTIMAL || r.status == TG_STATUS_OPTIMAL_INACCURATE);  // :261
        const double ud = sm[LF(uprev)], udel = sm[LF(uprev) + 1];
        if (tid == 0) {
            a.u_cmd[2 * (size_t)b] = ok ? ud + sm[LF(xt)] : ud;          // :265 / fallback :262
            a.u_cmd[2 * (size_t)b + 1] = ok ? udel + sm[LF(xt) + 1] : udel;
            if (a.status) a.status[b] = r.status;
            if (a.iters) a.iters[b] = r.iters;
            if (a.objective) a.objective[b] = ok ? r.objective : nan("");
        }
        if (a.U_opt)
            for (int i = tid; i < n; i += NT) a.U_opt[(size_t)b * n + i] = ok ? ((i & 1) ? udel : ud) + sm[LF(xt) + i] : nan("");
        if (a.y_opt) {
            const size_t m = 2 * (size_t)n + ms;
            for (int i = tid; i < 2 * n; i += NT) a.y_opt[b * m + i] = ok ? sm[LF(y) + i] : nan("");
            for (int i = tid; i < ms; i += NT) a.y_opt[b * m + 2 * n + i] = ok ? sm[L.ys + i] : nan("");
        }
        if (a.X_opt && tid == 0) {
            // X_k of the QP (x_{k+1} = A_k x_k + B_k u_k + g_k, :189-192).  The nominal rollout satisfies the same recursion
            // with u = u_prev, so X_k = xbar_k + dx_k with dx_{k+1} = A_k dx_k + B_k dU_k, dx_0 = 0.
            double *X = a.X_opt + (size_t)b * (N + 1) * 6;
            double dx[6] = {0, 0, 0, 0, 0, 0};
            for (int i = 0; i < 6; ++i) X[i] = ok ? sm[LF(xbar) + i] : nan("");
            for (int k = 0; k < N; ++k) {
                const double *r_ = sm + LF(lin) + TG_LIN * k;
                const double d0 = sm[LF(xt) + 2 * k], d1 = sm[LF(xt) + 2 * k + 1];
                double nx[6];
                nx[0] = dx[0] + r_[0] * dx[2] + r_[1] * dx[3] + r_[2] * dx[4];
                nx[1] = dx[1] + r_[3] * dx[2] + r_[4] * dx[3] + r_[5] * dx[4];
                nx[2] = dx[2] + r_[6] * dx[5];
                nx[3] = r_[7] * dx[3] + r_[8] * dx[4] + r_[9] * dx[5] + r_[16] * d0 + r_[17] * d1;
                nx[4] = r_[10] * dx[3] + r_[11] * dx[4] + r_[12] * dx[5] + r_[18] * d1;
                nx[5] = r_[13] * dx[3] + r_[14] * dx[4] + r_[15] * dx[5] + r_[19] * d1;
                for (int i = 0; i < 6; ++i) { dx[i] = nx[i]; X[6 * (k + 1) + i] = ok ? sm[LF(xbar) + 6 * (k + 1) + i] + dx[i] : nan(""); }
            }
        }
        if (a.ws_valid && c.warm_start) {
            const size_t m = 2 * (size_t)n + ms;
            for (int i = tid; i < n; i += NT) a.ws_x[(size_t)b * n + i] = sm[LF(xt) + i];
            for (int i = tid; i < 2 * n; i += NT) a.ws_y[b * m + i] = sm[LF(y) + i];
            for (int i = tid; i < ms; i += NT) a.ws_y[b * m + 2 * n + i] = sm[L.ys + i];
            if (tid == 0) a.ws_valid[b] = ok ? (r.free_end ? 2 : 1) : 0;
        }
    }
}

// PT = true: the plant instance.  Trajectory b's plant integrates the row a.plant[b] (tg_closed_loop_params); the controller
// keeps c.p.  A template flag rather than a run-time branch: the second inlined plant step made the compile-time instances
// spill more (N = 20: 60 / 84 B of spill stores / loads instead of 48 / 60 B), so the instances a launch without a plant table
// runs stay as they were.
template <int W, int S, int NC, bool P1 = false, bool HS = (NC == 0), bool CT = false, bool PT = false>
__global__ void __launch_bounds__(TW_CTA_THREADS) __maxnreg__(tw_regs<S>())
tw_closed_loop_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ WLayout L, const __grid_constant__ LoopArgs a)
{
    extern __shared__ __align__(16) double sm_all[];
    constexpr int NT = 32 * W;
    const int P = P1 ? 1 : a.ppc;
    int prob = P1 ? 0 : threadIdx.x / NT, tid = P1 ? threadIdx.x : threadIdx.x % NT;
    unsigned sm_off = (unsigned)prob * (unsigned)(tw_stride(L) + (CT ? TW_CTRL_DBL : 0)) * 8u;
    if constexpr (!P1) asm volatile("" : "+r"(tid), "+r"(prob), "+r"(sm_off));
    const int bar = P1 ? TW_BAR_PROB : TW_BAR_PROB + prob;
    double *sm = reinterpret_cast<double *>(reinterpret_cast<char *>(sm_all) + sm_off);
    const int N = NC > 0 ? NC : c.N, n = 2 * N, ms = HS ? c.ms : 0, ns = HS ? c.ns : 0, T = a.T;
    if (prob >= P) return;
    const TwMap<S> mp = tw_make_map<W, S>(LF(nb), tid);
    const StepTaps tap = {};
    int *cnt = reinterpret_cast<int *>(sm + LF(misc) + M_CNT);                 // 6 status counters
    long long *itsum = reinterpret_cast<long long *>(sm + LF(misc) + M_CNT + 3);
    const bool my = tid < N;
    const int j0 = 2 * tid;
    // Trajectories are dealt round-robin over the CTAs: slot `prob` of CTA c takes b = c + G (round P + prob), G = gridDim.x;
    // `active` (the busy slots of this CTA in this round) is what the step barrier counts.
    const int G = gridDim.x;
    for (int round = 0; blockIdx.x + (long long)G * round * P < a.B; ++round) {
        const long long bfirst = blockIdx.x + (long long)G * round * P;
        const long long left = (a.B - 1 - bfirst) / G + 1;                   // slots with a trajectory, >= 1
        const int active = left < P ? (int)left : P;
        const bool lockstep = !P1 && active > 1;
        if (prob >= active) break;                                           // later rounds have no work for this slot either
        const int b = (int)(bfirst + (long long)G * prob);
        tw_sync<W>(bar);
        if (tid < 12) sm[LF(spec) + tid] = reinterpret_cast<const double *>(a.spec + b)[tid];   // scenario -> shared memory
        if (tid < 6) { const double v_ = a.x0[6 * (size_t)b + tid]; sm[LF(x0) + tid] = v_; a.clean[(size_t)b * (T + 1) * 6 + tid] = v_; }
        if (tid < 2) sm[LF(uprev) + tid] = a.u0[2 * (size_t)b + tid];
        if constexpr (CT) tw_stage_ctrl(sm + tw_stride(L), a.ctrl + b, tid);   // the trajectory's settings, once
        if (tid < TG_NUM_STATUS) cnt[tid] = 0;
        if (tid == 0) *itsum = 0;
        bool warm = false, warm_free = false;
        tw_sync<W>(bar);
#pragma unroll 1
        for (int t = 0; t <= T; ++t) {
            FusedCtx fx;
            fx.brk = a.brk; fx.coef = a.coef;
            fx.noisy_row = a.noisy + ((size_t)b * (T + 1) + t) * 6;
            fx.seed = c.seed_base + (unsigned long long)(a.traj_id0 + b);
            fx.t_index = t;
            if (t == T) {   // last row: only its noisy copy remains to be written
                if (tid < 3) {
                    uint32_t r4[4];
                    tg_philox4x32_10((uint32_t)t, (uint32_t)(tid >> 1), 0u, 0u, (uint32_t)fx.seed, (uint32_t)(fx.seed >> 32), r4);
                    double n0, n1;
                    tg_box_muller(r4[(tid & 1) * 2], r4[(tid & 1) * 2 + 1], n0, n1);
                    fx.noisy_row[2 * tid] = sm[LF(x0) + 2 * tid] + c.noise_std[2 * tid] * n0;
                    fx.noisy_row[2 * tid + 1] = sm[LF(x0) + 2 * tid + 1] + c.noise_std[2 * tid + 1] * n1;
                }
                break;
            }
            const StepResult r = tw_step_body<W, S, NC, HS, CT>(c, L, sm, mp, warm, warm_free, tap, &fx, tid, bar,
                                                                 CT ? reinterpret_cast<const TwCtrl *>(sm + tw_stride(L)) : nullptr);
            const bool ok = (r.status == TG_STATUS_OPTIMAL || r.status == TG_STATUS_OPTIMAL_INACCURATE);
            if (tid == 0) { cnt[r.status] += 1; *itsum += r.iters; }
            // shifted warm start for the next step, in the next step's dU coordinates
            double2 nx = make_double2(0.0, 0.0), nyb = nx, nyr = nx;
            if (my) {
                const double2 d0 = tw_ld2(sm + LF(xt));
                const double2 xs_ = tw_ld2(sm + LF(xt) + ((tid + 1 < N) ? j0 + 2 : j0));
                nx = make_double2(xs_.x - d0.x, xs_.y - d0.y);
                if (tid + 1 < N) { nyb = tw_ld2(sm + LF(y) + j0 + 2); nyr = tw_ld2(sm + LF(y) + n + j0 + 2); }
            }
            if (tid < 32) {   // plant (MPC/main.py:97) + outputs, warp 0 (lane-parallel f_cont)
                const double ud = sm[LF(uprev)], udel = sm[LF(uprev) + 1];
                const double u0 = ok ? ud + sm[LF(xt)] : ud, u1 = ok ? udel + sm[LF(xt) + 1] : udel;
                double xs[6];
#pragma unroll
                for (int i = 0; i < 6; ++i) xs[i] = sm[LF(x0) + i];
                if constexpr (PT) {   // the trajectory's own plant: row b (global memory, stays in L1 / L2); the controller keeps c.p
                    const double *__restrict__ pr = a.plant + (size_t)b * TG_NPARAMS;
                    const bool tab = tg_plant_row_tables(c, pr);
                    // 1.0 / m is IEEE-rounded in fp64 on the device: the inv_m / inv_Iz tg_create stores for the same m, Iz
                    tg_plant_step_lanes(c, pr, 1.0 / pr[P_m], 1.0 / pr[P_Iz], tab ? c.tyre_tab : nullptr, tab ? c.atan_tab : nullptr,
                                        xs, u0, u1, tid);
                } else {
                    tg_plant_step_lanes(c, c.p, c.inv_m, c.inv_Iz, c.tyre_tab, c.atan_tab, xs, u0, u1, tid);
                }
                if (tid == 0) {
                    double *clean = a.clean + ((size_t)b * (T + 1) + t + 1) * 6;
#pragma unroll
                    for (int i = 0; i < 6; ++i) { sm[LF(misc) + M_XNEXT + i] = xs[i]; clean[i] = xs[i]; }
                    a.U[((size_t)b * T + t) * 2] = u0; a.U[((size_t)b * T + t) * 2 + 1] = u1;
                    sm[LF(misc) + M_UCMD] = u0; sm[LF(misc) + M_UCMD + 1] = u1;
                }
            }
            tw_sync<W>(bar);
            // commit the new state / warm start
            if (tid < 6) sm[LF(x0) + tid] = sm[LF(misc) + M_XNEXT + tid];
            if (tid < 2) sm[LF(uprev) + tid] = sm[LF(misc) + M_UCMD + tid];
            if (my) { tw_st2(sm + LF(x) + j0, nx.x, nx.y); tw_st2(sm + LF(y) + j0, nyb.x, nyb.y); tw_st2(sm + LF(y) + n + j0, nyr.x, nyr.y); }
            if (ms > 0) {   // shift the state-row duals by one stage (ns rows), in place: ascending order, one thread
                if (tid == 0) {
                    for (int i = 0; i + ns < ms; ++i) sm[L.ys + i] = sm[L.ys + i + ns];
                    for (int i = (ms > ns ? ms - ns : 0); i < ms; ++i) sm[L.ys + i] = 0.0;
                }
            }
            warm = ok && c.warm_start;
            warm_free = warm && r.free_end;
            if constexpr (P1) tw_sync<W>(bar);
            else if (lockstep) tg_sync(TW_BAR_STEP, NT * active); else tw_sync<W>(bar);
        }
        tw_sync<W>(bar);
        if (tid < TG_NUM_STATUS && a.status_counts) a.status_counts[(size_t)b * TG_NUM_STATUS + tid] = cnt[tid];
        if (tid == 0 && a.iters_total) a.iters_total[b] = *itsum;
    }
}

// a10 tap: the reference window of tw_ref_window_warp for B states, one warp per problem
__global__ void tg_ref_window_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ WLayout L, int B,
                                     const double *x0, const tg_ref_spec *spec, const double *brk, const double *coef,
                                     int t_index, double *path_ref, double *vref)
{
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x, N = c.N;
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        __syncwarp();
        if (lane < 6) sm[L.x0 + lane] = x0[6 * (size_t)b + lane];
        __syncwarp();
        const tg_ref_spec sp = spec[b];
        tw_ref_window_warp<0, 1>(c, L, sm, sp, brk, coef, t_index, lane);
        __syncwarp();
        for (int k = lane; k <= N; k += 32) {
            double *pr = path_ref + 3 * ((size_t)b * (N + 1) + k);
            pr[0] = sm[L.Xr + k]; pr[1] = sm[L.Yr + k]; pr[2] = sm[L.Pr + k];
            vref[(size_t)b * (N + 1) + k] = sm[L.vref + k];
        }
    }
}

// plant: [B][TG_NPARAMS] per-trajectory parameters or null (every trajectory integrates the handle's c.p)
__global__ void tg_plant_kernel(const __grid_constant__ DevCfg c, int B, int T, const double *x0, const double *U,
                                const double *plant, double *X)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double *__restrict__ pv = plant ? plant + (size_t)b * TG_NPARAMS : c.p;
    const bool tab = plant ? tg_plant_row_tables(c, pv) : true;
    const double *tyre_tab = tab ? c.tyre_tab : nullptr, *atan_tab = tab ? c.atan_tab : nullptr;
    double xs[6];
    double *Xo = X + (size_t)b * (T + 1) * 6;
    for (int i = 0; i < 6; ++i) { xs[i] = x0[6 * (size_t)b + i]; Xo[i] = xs[i]; }
    for (int t = 0; t < T; ++t) {
        if (c.plant == TG_PLANT_MPC) tg_plant_step(c, pv, xs, U[((size_t)b * T + t) * 2], U[((size_t)b * T + t) * 2 + 1]);
        else tg_plant_step_gen(c, pv, tyre_tab, atan_tab, xs, U[((size_t)b * T + t) * 2], U[((size_t)b * T + t) * 2 + 1]);
        for (int i = 0; i < 6; ++i) Xo[6 * (size_t)(t + 1) + i] = xs[i];
    }
}

__global__ void tg_noise_kernel(unsigned long long seed0, int n_traj, int n_rows, double *out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n_traj * n_rows) return;
    const int tr = (int)(i / n_rows), row = (int)(i % n_rows);
    double nz[6];
    tg_noise_row(seed0 + (unsigned long long)tr, (uint32_t)row, nz);
    for (int k = 0; k < 6; ++k) out[6 * i + k] = nz[k];
}

__global__ void tg_philox_kernel(unsigned long long seed, uint32_t first, uint32_t block, int n, uint32_t *out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t r[4];
    tg_philox4x32_10(first + (uint32_t)i, block, 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    for (int k = 0; k < 4; ++k) out[4 * (size_t)i + k] = r[k];
}

template <typename T>
__global__ void tg_fma_peak_kernel(T *out, int iters)
{
    T a0 = (T)threadIdx.x * (T)1e-3, a1 = a0 + (T)1, a2 = a0 + (T)2, a3 = a0 + (T)3, a4 = a0 + (T)4, a5 = a0 + (T)5,
      a6 = a0 + (T)6, a7 = a0 + (T)7;
    const T b = (T)0.999, cc = (T)1e-4;
    for (int i = 0; i < iters; ++i) {
        a0 = a0 * b + cc; a1 = a1 * b + cc; a2 = a2 * b + cc; a3 = a3 * b + cc;
        a4 = a4 * b + cc; a5 = a5 * b + cc; a6 = a6 * b + cc; a7 = a7 * b + cc;
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------------------------------------ host side
// Tyre-curve table (tg_device.cuh: tg_tyre_tab): per interval the degree-(NC-1) Chebyshev interpolant of
// g(alpha) = sin(C atan(B alpha)) in long double, converted to monomials of s in [-1, 1].  Returns the largest
// deviation from libm on a dense check grid (value and slope) so the caller can refuse a table that is not at
// rounding level for unusual B, C.
static double build_cheb_table(const std::function<long double(long double)> &fun, const std::function<long double(long double)> &dfun,
                               long double lo, long double hi, int NI, double *tab /*[NI + 1][NC]*/, double *slope_err)
{
    // NI + 1 intervals of width h = (hi - lo) / NI, interval i centred on lo + i h (tg_tab_row): the end intervals reach half
    // an interval beyond [lo, hi], where fun is still analytic
    const int NC = TG_TAB_NC;
    const long double PI = 3.141592653589793238462643383279502884L;
    long double T[TG_TAB_NC][TG_TAB_NC] = {};   // T[k][i] = coefficient of s^i in T_k(s)
    T[0][0] = 1.0L;
    if (NC > 1) T[1][1] = 1.0L;
    for (int k = 2; k < NC; ++k)
        for (int i = 0; i < NC; ++i) T[k][i] = (i > 0 ? 2.0L * T[k - 1][i - 1] : 0.0L) - T[k - 2][i];
    const long double hw = (hi - lo) / (2 * NI);
    double worst = 0.0, worst_d = 0.0;
    for (int it = 0; it <= NI; ++it) {
        const long double ctr = lo + 2 * it * hw;
        long double fv[TG_TAB_NC], a[TG_TAB_NC];
        for (int j = 0; j < NC; ++j) {
            const long double sj = cosl(PI * (j + 0.5L) / NC);
            fv[j] = fun(ctr + hw * sj);
        }
        for (int k = 0; k < NC; ++k) {
            long double acc = 0.0L;
            for (int j = 0; j < NC; ++j) acc += fv[j] * cosl(PI * k * (j + 0.5L) / NC);
            a[k] = acc * (k == 0 ? 1.0L : 2.0L) / NC;
        }
        for (int i = 0; i < NC; ++i) {
            long double m = 0.0L;
            for (int k = 0; k < NC; ++k) m += a[k] * T[k][i];
            tab[it * NC + i] = (double)m;
        }
        for (int q = 0; q <= 16; ++q) {   // check grid incl. the interval ends
            const double sq = -1.0 + q / 8.0;
            double v = tab[it * NC + NC - 1], dv = 0.0;
            for (int i = NC - 2; i >= 0; --i) { dv = dv * sq + v; v = v * sq + tab[it * NC + i]; }
            const long double al = ctr + hw * sq;
            worst = fmax(worst, fabs((double)(v - fun(al))));
            worst_d = fmax(worst_d, fabs((double)(dv / (double)hw - dfun(al))));
        }
    }
    if (slope_err) *slope_err = worst_d;
    return worst;
}

static double build_tyre_table(double B, double C, double ma, double *tab /*[TG_TAB_ROWS][NC]*/, double *slope_err)
{
    auto f = [=](long double al) { return sinl((long double)C * atanl((long double)B * al)); };
    auto df = [=](long double al) { const long double ba = (long double)B * al; return cosl((long double)C * atanl(ba)) * C * B / (1.0L + ba * ba); };
    return build_cheb_table(f, df, -(long double)ma, (long double)ma, TG_TAB_NI, tab, slope_err);
}

// atan on [-TG_ATAN_T0, TG_ATAN_T0] (the slip-angle argument n / vx_eff of the sequential nominal rollout): same form
static double build_atan_table(double *tab /*[TG_ATAN_ROWS][NC]*/)
{
    auto f = [](long double t) { return atanl(t); };
    auto df = [](long double t) { return 1.0L / (1.0L + t * t); };
    return build_cheb_table(f, df, -(long double)TG_ATAN_T0, (long double)TG_ATAN_T0, TG_ATAN_NI, tab, nullptr);
}

// the warp-per-problem kernel instances of a handle: several problems per CTA, and P1 (one problem per CTA); null where the
// instance is not compiled
typedef void (*TwStepKernel)(DevCfg, WLayout, StepArgs);
typedef void (*TwLoopKernel)(DevCfg, WLayout, LoopArgs);
struct TwKernels {
    TwStepKernel step, step_p1;
    TwLoopKernel loop, loop_p1;
    TwLoopKernel loop_pt, loop_pt_p1;   // the same loop kernels with per-trajectory plant parameters (PT)
};
// what a launch of one set of instances needs: the kernels, the shared memory per problem, and the most problems per CTA
// (0: one problem does not fit)
struct TwLaunch {
    TwKernels k;
    size_t smem;
    int ppc_max;
};

struct tg_handle {
    tg_config cfg;
    DevCfg dc;
    int device, num_sms, grid_cap;
    int ppc_env;              // TRAJGEN_PPC override of the problems per CTA (0 = automatic)
    // warp-per-problem kernels (tw_solver.cuh): W warps per problem, S tile blocks per thread
    int W, S;
    TwLaunch tw;              // the instances of the handle's own settings
    TwLaunch tw_ctrl;         // the ctrl instances of the shape (per-problem settings, tg_mpc_step_ctrl / tg_closed_loop_ctrl)
    WLayout WL;
    WLayout Lref;             // layout of the reference-window tap kernel (no state rows, one warp)
    size_t smem_optin;
    cudaStream_t stream;
    long long launches;
    double *tyre_tab;   // device copy of the tyre-curve table, or null (fit not at rounding level -> atan/sin path)
    double tab_err[2];  // max |table - libm| of value and slope on the check grid
    // warm-start state for the step API
    double *ws_x, *ws_y; int *ws_valid; int ws_B;
    // staging for *_host entry points
    void *dstage; size_t dstage_bytes;
    void *hstage; size_t hstage_bytes;
};

// kernel instances: (W, S) for a run-time horizon, plus the horizons of the reference / the BASELINE configurations compiled in
// (NC = N: shared-memory offsets become immediates, horizon loops get constant trip counts: 25-50 % faster).  The compile-time
// instances serve the standard controller only -- MPC tyre model from the tables, analytic Jacobians (tw_standard_controller) --
// and come without (HS = false) or with (HS = true) the code of the state-bound rows.
static bool tw_standard_controller(const DevCfg &d)
{
    return d.model == TG_MODEL_MPC && d.jacobian == TG_JAC_ANALYTIC && d.tyre_tab && d.atan_tab;
}
// the kernels of one (W, S, NC, HS, CT).  Single-problem-per-CTA instances exist for the one- and two-warp shapes, where four
// CTAs per SM would leave most of the register file and shared memory unused, except for a compile-time horizon without
// state-bound rows.  A compile-time horizon with state-bound rows on those shapes has only that instance (problems with
// state-bound rows always run one per CTA, choose_tw_ppc).  The ctrl instances (CT, per-problem settings staged in shared
// memory) exist for the run-time horizon with the code of the state-bound rows only.
template <int W, int S, int NC, bool HS, bool CT = false>
static TwKernels tw_instance()
{
    static_assert(NC == 0 || (tw_shape(NC).W == W && tw_shape(NC).S == S), "a compile-time horizon runs on its tw_shape");
    static_assert(!CT || (NC == 0 && HS), "ctrl instances: run-time horizon with state-bound rows only");
    TwKernels k = {};
    if constexpr (!(HS && NC > 0 && W <= 2)) {
        k.step = tw_mpc_step_kernel<W, S, NC, false, HS, CT>;
        k.loop = tw_closed_loop_kernel<W, S, NC, false, HS, CT>;
        k.loop_pt = tw_closed_loop_kernel<W, S, NC, false, HS, CT, true>;
    }
    if constexpr (W <= 2 && (NC == 0 || HS)) {
        k.step_p1 = tw_mpc_step_kernel<W, S, NC, true, HS, CT>;
        k.loop_p1 = tw_closed_loop_kernel<W, S, NC, true, HS, CT>;
        k.loop_pt_p1 = tw_closed_loop_kernel<W, S, NC, true, HS, CT, true>;
    }
    return k;
}
// the run-time-horizon instances of the five shapes
template <bool CT>
static TwKernels tw_runtime(int W, int S)
{
    if (W == 1 && S == 1) return tw_instance<1, 1, 0, true, CT>();
    if (W == 2 && S == 1) return tw_instance<2, 1, 0, true, CT>();
    if (W == 4 && S == 1) return tw_instance<4, 1, 0, true, CT>();
    if (W == 8 && S == 1) return tw_instance<8, 1, 0, true, CT>();
    if (W == 8 && S == 2) return tw_instance<8, 2, 0, true, CT>();
    return TwKernels{};
}
// every compiled instance.  ct selects the ctrl instances.  Otherwise fixed_n selects the compile-time-horizon instances where
// one exists: mpc_step's default horizon (20), MPC/main.py's (40), BASELINE config 4's (10, 50).  No instance: every pointer
// null.
static TwKernels tw_kernels(int W, int S, int N, int ms, bool fixed_n, bool ct)
{
    if (fixed_n && !ct && ms == 0) {
        if (W == 2 && S == 1 && N == 20) return tw_instance<2, 1, 20, false>();
        if (W == 1 && S == 1 && N == 10) return tw_instance<1, 1, 10, false>();
        if (W == 8 && S == 1 && N == 40) return tw_instance<8, 1, 40, false>();
        if (W == 8 && S == 2 && N == 50) return tw_instance<8, 2, 50, false>();
    }
    if (fixed_n && !ct && ms > 0) {
        if (W == 2 && S == 1 && N == 20) return tw_instance<2, 1, 20, true>();
        if (W == 1 && S == 1 && N == 10) return tw_instance<1, 1, 10, true>();
        if (W == 8 && S == 2 && N == 50) return tw_instance<8, 2, 50, true>();
    }
    if (!ct) return tw_runtime<false>(W, S);
    return tw_runtime<true>(W, S);
}
// a TwLaunch of the instances k with `smem` bytes per problem.  Problems per CTA: within the CTA's threads, a barrier id per
// problem for W > 1, and the opt-in shared memory.  The shared-memory attributes are per kernel function and process-wide:
// always raise them to the device limit so that handles with different layouts can be used side by side.
static int make_tw_launch(const tg_handle *h, const TwKernels &k, size_t smem, TwLaunch &out)
{
    out.k = k; out.smem = smem; out.ppc_max = 0;
    if (smem > h->smem_optin) return TG_OK;
    int p = TW_CTA_THREADS / (32 * h->W);
    if (h->W > 1) p = std::min(p, TW_BAR_STEP - TW_BAR_PROB);
    while (p > 1 && (size_t)p * smem > h->smem_optin) p -= 1;
    out.ppc_max = p;
    for (const void *f : {(const void *)k.step, (const void *)k.step_p1, (const void *)k.loop, (const void *)k.loop_p1,
                          (const void *)k.loop_pt, (const void *)k.loop_pt_p1}) {
        if (!f) continue;
        CK(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_optin));
        CK(cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    return TG_OK;
}

// warp-per-problem kernels: problems per CTA.  Resident problems per SM are bounded by registers (512 threads x 128) and
// shared memory either way; larger CTAs share more instruction fetches, smaller ones spread a small batch over more SMs.
static int choose_tw_ppc(const tg_handle *h, int B, int ppc_max)
{
    if (h->ppc_env) return h->ppc_env < ppc_max ? h->ppc_env : ppc_max;
    // problems with state-bound rows have long, unequal solves (tens to hundreds of ADMM iterations): free-running
    // single-problem CTAs beat problems that wait for one another at every step boundary
    if (h->dc.ms > 0) return 1;
    // measured at N = 20 (two warps per problem): 4 problems per CTA 2.65e7 steps/s (B = 2368), 8 per CTA 2.37e7 (B = 4736),
    // 2 per CTA 2.24e7 and 1 per CTA 1.43e7 (B = 1024): sharing instruction fetches matters, waiting for 7 neighbours costs more
    int p = ppc_max < 4 ? ppc_max : 4;
    while (p > 1 && (B + p - 1) / p < h->num_sms) p >>= 1;   // every SM gets a CTA before CTAs get wider
    return p < 1 ? 1 : p;
}

// the single-problem instance where there is no other or where one problem per CTA is chosen, else `multi` with
// choose_tw_ppc problems per CTA; `multi` and `p1` are kernels of `t`
template <typename Args>
static int launch_tw(tg_handle *h, const TwLaunch &t, void (*multi)(DevCfg, WLayout, Args), void (*p1)(DevCfg, WLayout, Args),
                     Args &a)
{
    // tg_create refuses a handle whose own problems do not fit, so only the ctrl instances can get here without a fit
    if (t.ppc_max < 1) return fail(TG_ERR_UNSUPPORTED, "per-problem settings: the record does not fit beside the problem's shared memory");
    int ppc = choose_tw_ppc(h, a.B, t.ppc_max);
    void (*kern)(DevCfg, WLayout, Args) = multi;
    if (p1 && (!multi || ppc == 1)) { kern = p1; ppc = 1; }
    a.ppc = ppc;
    const int threads = 32 * h->W * ppc;
    const size_t smem = (size_t)ppc * t.smem;
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1) return fail(TG_ERR_UNSUPPORTED, "kernel does not fit on an SM with this configuration");
    const int cap = per_sm * h->num_sms, ctas = (a.B + ppc - 1) / ppc;
    kern<<<ctas < cap ? ctas : cap, threads, smem, h->stream>>>(h->dc, h->WL, a);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

extern "C" {

const char *tg_last_error(void) { return g_err.c_str(); }
int tg_version(void) { return TG_VERSION; }

void tg_default_config(tg_config *c)
{
    memset(c, 0, sizeof(*c));
    c->N = 20; c->model = TG_MODEL_MPC; c->plant = TG_PLANT_MPC; c->jacobian = TG_JAC_ANALYTIC;
    c->Ts = 0.02;
    const double p[TG_NPARAMS] = {0.287, 0.0545, 0.0518, 0.00035, 3.3852, 1.2691, 0.1737, 2.579, 1.2, 0.192,
                                  0.041, 27.8e-6, 0.029, 0.033, 9.81, 0.6, 0.3};
    memcpy(c->params, p, sizeof(p));
    c->q_c = 6.0; c->q_phi = 0.5; c->q_vx = 0.5;
    c->R[0] = 0.02; c->R[3] = 2.0; c->Rd[0] = 0.01; c->Rd[3] = 5.0;
    c->u_lo[0] = -1.0; c->u_hi[0] = 1.0; c->u_lo[1] = -0.6; c->u_hi[1] = 0.6;
    c->du_lo[0] = -0.5; c->du_hi[0] = 0.5; c->du_lo[1] = -0.3; c->du_hi[1] = 0.3;
    for (int i = 0; i < 6; ++i) { c->x_lo[i] = -TG_INF; c->x_hi[i] = TG_INF; }
    c->rho = 0.1; c->sigma = 1e-6; c->alpha = 1.6; c->eps_abs = 1e-6; c->eps_rel = 1e-6; c->eps_prim_inf = 1e-4;   // eps: one decade tighter than CVXPY's OSQP setting (1e-5), DESIGN.md 2
    c->adaptive_rho_tol = 5.0; c->alpha_warm = 1.2; c->max_iter = 10000; c->check_every = 5; c->adaptive_rho = 1; c->adaptive_rho_min_iter = 20;
    c->warm_start = 0; c->vref_advance = 0;
    const double sd[6] = {0.05, 0.05, 0.003, 0.010, 0.003, 0.030};
    memcpy(c->noise_std, sd, sizeof(sd));
    c->noise_seed_base = 12345ull;
}

int tg_device_count(int *n) { CK(cudaGetDeviceCount(n)); return TG_OK; }

int tg_create(const tg_config *cfg, int device, tg_handle **out)
{
    if (!cfg || !out) return fail(TG_ERR_INVALID, "null argument");
    if (cfg->N < 1) return fail(TG_ERR_INVALID, "N must be >= 1");
    if (!(cfg->Ts > 0)) return fail(TG_ERR_INVALID, "Ts must be > 0");
    if (cfg->max_iter < 1 || cfg->check_every < 1) return fail(TG_ERR_INVALID, "max_iter and check_every must be >= 1");
    if (!(cfg->rho > 0) || !(cfg->sigma > 0) || !(cfg->alpha > 0 && cfg->alpha < 2)) return fail(TG_ERR_INVALID, "rho, sigma > 0 and 0 < alpha < 2 required");
    const TwShape shape = tw_shape(cfg->N);
    if (shape.W == 0) return fail(TG_ERR_UNSUPPORTED, "horizon N > 56 is not supported");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (ndev == 0) return fail(TG_ERR_CUDA, "no CUDA device: libtrajgen has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(TG_ERR_INVALID, "bad device index");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(TG_ERR_UNSUPPORTED, "libtrajgen is built for sm_100a (B200) only");

    tg_handle *h = new (std::nothrow) tg_handle();
    if (!h) return fail(TG_ERR_NOMEM, "out of host memory");
    memset(h, 0, sizeof(*h));
    struct Guard { tg_handle *p; ~Guard() { if (p) { cudaFree(p->tyre_tab); delete p; } } } guard{h};   // released on success
    h->cfg = *cfg; h->W = shape.W; h->S = shape.S; h->device = device; h->num_sms = prop.multiProcessorCount;
    DevCfg &d = h->dc;
    d.N = cfg->N; d.n = 2 * cfg->N; d.model = cfg->model; d.plant = cfg->plant; d.jacobian = cfg->jacobian;
    d.ns = 0;
    for (int i = 0; i < 6; ++i)
        if (cfg->x_lo[i] > -TG_INF || cfg->x_hi[i] < TG_INF) d.sidx[d.ns++] = i;
    d.ms = d.ns * d.N; d.m = 4 * d.N + d.ms;
    d.max_iter = cfg->max_iter; d.check_every = cfg->check_every; d.adaptive_rho = cfg->adaptive_rho;
    d.adaptive_rho_min_iter = cfg->adaptive_rho_min_iter; d.warm_start = cfg->warm_start; d.vref_advance = cfg->vref_advance;
    d.Ts = cfg->Ts;
    memcpy(d.p, cfg->params, sizeof(d.p));
    d.inv_m = 1.0 / d.p[P_m]; d.inv_Iz = 1.0 / d.p[P_Iz];
    d.tyre_tab = nullptr; d.tab_scale = 0.0;
    if (d.p[P_maxAlpha] > 0.0 && !getenv("TRAJGEN_NO_TYRE_TABLE")) {
        std::vector<double> tab(2 * TG_TAB_ROWS * TG_TAB_NC + TG_ATAN_ROWS * TG_TAB_NC);
        double se_f = 0.0, se_r = 0.0;
        const double e_f = build_tyre_table(d.p[P_Bf], d.p[P_Cf], d.p[P_maxAlpha], tab.data(), &se_f);
        const double e_r = build_tyre_table(d.p[P_Br], d.p[P_Cr], d.p[P_maxAlpha], tab.data() + TG_TAB_ROWS * TG_TAB_NC, &se_r);
        const double e_at = build_atan_table(tab.data() + 2 * TG_TAB_ROWS * TG_TAB_NC);
        h->tab_err[0] = fmax(e_f, e_r); h->tab_err[1] = fmax(se_f, se_r);
        if (h->tab_err[0] <= 4e-16 && h->tab_err[1] <= 1e-12) {
            CK(cudaMalloc(&h->tyre_tab, tab.size() * sizeof(double)));
            CK(cudaMemcpy(h->tyre_tab, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
            d.tyre_tab = h->tyre_tab;
            d.tab_scale = TG_TAB_NI / (2.0 * d.p[P_maxAlpha]);
            if (e_at <= 4e-16) d.atan_tab = h->tyre_tab + 2 * TG_TAB_ROWS * TG_TAB_NC;
        }
    }
    d.ctl.q_c = cfg->q_c; d.ctl.q_phi = cfg->q_phi; d.ctl.q_vx = cfg->q_vx;
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j) {
            d.ctl.Rs[i * 2 + j] = 0.5 * (cfg->R[i * 2 + j] + cfg->R[j * 2 + i]);
            d.ctl.Rds[i * 2 + j] = 0.5 * (cfg->Rd[i * 2 + j] + cfg->Rd[j * 2 + i]);
        }
    memcpy(d.ctl.u_lo, cfg->u_lo, 16); memcpy(d.ctl.u_hi, cfg->u_hi, 16); memcpy(d.ctl.du_lo, cfg->du_lo, 16); memcpy(d.ctl.du_hi, cfg->du_hi, 16);
    memcpy(d.ctl.x_lo, cfg->x_lo, 48); memcpy(d.ctl.x_hi, cfg->x_hi, 48);
    d.rho = cfg->rho; d.sigma = cfg->sigma; d.alpha = cfg->alpha;
    d.alpha_warm = (cfg->alpha_warm > 0.0 && cfg->alpha_warm < 2.0) ? cfg->alpha_warm : cfg->alpha; d.eps_abs = cfg->eps_abs; d.eps_rel = cfg->eps_rel;
    d.eps_pinf = cfg->eps_prim_inf; d.adapt_tol = cfg->adaptive_rho_tol > 1.0 ? cfg->adaptive_rho_tol : 5.0;
    memcpy(d.noise_std, cfg->noise_std, 48);
    d.seed_base = cfg->noise_seed_base;

    d.free_mode = (cfg->solver_flags & 1) ? 0 : 1;
    h->smem_optin = (size_t)prop.sharedMemPerBlockOptin;
    h->Lref = tw_make_layout(d.N, 0, TwShape{1, 1});
    CK(cudaFuncSetAttribute(tg_ref_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_optin));
    h->ppc_env = 0;   // TRAJGEN_PPC pins the number of problems per CTA (measurement knob)
    {
        h->WL = tw_make_layout(d.N, d.ms, shape);
        const size_t stride = (size_t)tw_stride(h->WL) * sizeof(double);
        const TwKernels k = tw_kernels(h->W, h->S, d.N, d.ms, tw_standard_controller(d) && !getenv("TRAJGEN_DYNAMIC_N"), false);
        int rc = make_tw_launch(h, k, stride, h->tw);
        if (rc != TG_OK) return rc;
        if (h->tw.ppc_max < 1) return fail(TG_ERR_UNSUPPORTED, "state-bound rows x horizon exceed the 227 KB shared memory of one CTA");
        if (const char *e = getenv("TRAJGEN_PPC")) { const int v = atoi(e); if (v >= 1 && v <= h->tw.ppc_max) h->ppc_env = v; }
        if (!k.loop && !k.loop_p1) return fail(TG_ERR_UNSUPPORTED, "no kernel shape for this horizon");
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k.loop_p1 ? k.loop_p1 : k.loop, 32 * h->W, stride));
        if (occ < 1) return fail(TG_ERR_UNSUPPORTED, "kernel does not fit on an SM with this configuration");
        h->grid_cap = occ * h->num_sms;     // resident problems with one problem per CTA
        // the ctrl instances: the block plus the staged record (launch_tw takes the occupancy per launch)
        rc = make_tw_launch(h, tw_kernels(h->W, h->S, d.N, d.ms, false, true), stride + TW_CTRL_DBL * sizeof(double), h->tw_ctrl);
        if (rc != TG_OK) return rc;
    }
    h->stream = 0;
    guard.p = nullptr;
    *out = h;
    return TG_OK;
}

int tg_destroy(tg_handle *h)
{
    if (!h) return TG_OK;
    cudaSetDevice(h->device);
    cudaFree(h->tyre_tab); cudaFree(h->ws_x); cudaFree(h->ws_y); cudaFree(h->ws_valid); cudaFree(h->dstage);
    if (h->hstage) cudaFreeHost(h->hstage);
    delete h;
    return TG_OK;
}

int tg_set_stream(tg_handle *h, void *s) { if (!h) return fail(TG_ERR_INVALID, "null handle"); h->stream = (cudaStream_t)s; return TG_OK; }
int tg_synchronize(tg_handle *h) { if (!h) return fail(TG_ERR_INVALID, "null handle"); CK(cudaStreamSynchronize(h->stream)); return TG_OK; }
int tg_info(tg_handle *h, int32_t *ctas_per_sm, int32_t *threads_per_cta, int32_t *smem_bytes, int32_t *num_sms)
{
    if (!h) return fail(TG_ERR_INVALID, "null handle");
    if (ctas_per_sm) *ctas_per_sm = h->grid_cap / h->num_sms;
    if (threads_per_cta) *threads_per_cta = 32 * h->W;
    if (smem_bytes) *smem_bytes = (int32_t)h->tw.smem;
    if (num_sms) *num_sms = h->num_sms;
    return TG_OK;
}
#ifdef TG_PHASE_TIMING
int tg_debug_phases(long long *out16, int reset)
{
    if (out16) CK(cudaMemcpyFromSymbol(out16, g_tg_phase, sizeof(long long) * 16));
    if (reset) { long long z[16] = {0}; CK(cudaMemcpyToSymbol(g_tg_phase, z, sizeof(z))); }
    return TG_OK;
}
#endif
int tg_tyre_table_info(tg_handle *h, int32_t *in_use, double *max_value_err, double *max_slope_err)
{
    if (!h) return fail(TG_ERR_INVALID, "null handle");
    if (in_use) *in_use = (h->dc.tyre_tab ? 1 : 0) | (h->dc.atan_tab ? 2 : 0);   // bit 0: tyre curve, bit 1: slip-angle atan
    if (max_value_err) *max_value_err = h->tab_err[0];
    if (max_slope_err) *max_slope_err = h->tab_err[1];
    return TG_OK;
}
int tg_kernel_launches(tg_handle *h, int64_t *count) { if (!h || !count) return fail(TG_ERR_INVALID, "null argument"); *count = h->launches; return TG_OK; }

static int launch_step(tg_handle *h, StepArgs &a)
{
    if (a.B <= 0) return TG_OK;   // empty batch: nothing to do
    CK(cudaSetDevice(h->device));
    const TwLaunch &t = a.ctrl ? h->tw_ctrl : h->tw;
    return launch_tw(h, t, t.k.step, t.k.step_p1, a);
}

// the rules of tg_ctrl_spec (include/trajgen.h), row by row: TG_ERR_INVALID naming the first bad row and field
int tg_check_ctrl(int B, const tg_ctrl_spec *ctrl, uint32_t bounded_states)
{
    if (B > 0 && !ctrl) return fail(TG_ERR_INVALID, "bad argument: ctrl is null");
    for (int b = 0; b < B; ++b) {
        const tg_ctrl_spec &r = ctrl[b];
        auto bad = [&](const std::string &field, const char *why) { return fail(TG_ERR_INVALID, "ctrl row " + std::to_string(b) + ": " + field + " " + why); };
        const double *q[3] = {&r.q_c, &r.q_phi, &r.q_vx};
        const char *qn[3] = {"q_c", "q_phi", "q_vx"};
        for (int i = 0; i < 3; ++i)
            if (!(std::isfinite(*q[i]) && *q[i] >= 0.0)) return bad(qn[i], "must be finite and >= 0");
        for (int i = 0; i < 4; ++i) {
            if (!std::isfinite(r.R[i])) return bad("R[" + std::to_string(i) + "]", "must be finite");
            if (!std::isfinite(r.Rd[i])) return bad("Rd[" + std::to_string(i) + "]", "must be finite");
        }
        {   // symmetric parts, as the kernels use them
            const double a = r.R[0], c = 0.5 * (r.R[1] + r.R[2]), d = r.R[3];
            if (!(a > 0.0 && a * d - c * c > 0.0)) return bad("R", "symmetric part is not positive definite");
            const double ad = r.Rd[0], cd = 0.5 * (r.Rd[1] + r.Rd[2]), dd = r.Rd[3];
            if (!(ad >= 0.0 && dd >= 0.0 && ad * dd - cd * cd >= 0.0)) return bad("Rd", "symmetric part is not positive semidefinite");
        }
        for (int i = 0; i < 2; ++i) {
            if (!(r.u_lo[i] <= r.u_hi[i])) return bad("u_lo[" + std::to_string(i) + "] / u_hi[" + std::to_string(i) + "]", "lo > hi");
            if (!(r.du_lo[i] <= r.du_hi[i])) return bad("du_lo[" + std::to_string(i) + "] / du_hi[" + std::to_string(i) + "]", "lo > hi");
        }
        for (int i = 0; i < 6; ++i) {
            const std::string f = "x_lo[" + std::to_string(i) + "] / x_hi[" + std::to_string(i) + "]";
            if (!(r.x_lo[i] <= r.x_hi[i])) return bad(f, "lo > hi");
            if (!(bounded_states >> i & 1u) && (r.x_lo[i] > -TG_INF || r.x_hi[i] < TG_INF)) return bad(f, "finite bound on a state component the handle does not bound");
        }
    }
    return TG_OK;
}
// tg_check_ctrl's bounded_states of a handle: bit i set when it bounds state component i
static uint32_t bounded_states(const tg_handle *h)
{
    uint32_t m = 0;
    for (int si = 0; si < h->dc.ns; ++si) m |= 1u << h->dc.sidx[si];
    return m;
}

int tg_linearize(tg_handle *h, int B, const double *x0, const double *u_prev, double *A, double *Bm, double *g, double *xbar)
{
    if (!h || B < 0 || (B > 0 && (!x0 || !u_prev))) return fail(TG_ERR_INVALID, "bad argument");
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.x0 = x0; a.u_prev = u_prev; a.path_ref = nullptr; a.vref = nullptr;
    a.A = A; a.Bm = Bm; a.g = g; a.xbar = xbar; a.stop = 1;
    return launch_step(h, a);
}

int tg_assemble(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref, const double *vref,
                double *H, double *q, double *c0, double *l, double *u, double *Gs)
{
    if (!h || B < 0 || (B > 0 && (!x0 || !u_prev || !path_ref))) return fail(TG_ERR_INVALID, "bad argument");
    if ((l == nullptr) != (u == nullptr)) return fail(TG_ERR_INVALID, "l and u must be given together");
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.x0 = x0; a.u_prev = u_prev; a.path_ref = path_ref; a.vref = vref;
    a.H = H; a.q = q; a.c0 = c0; a.l = l; a.u = u; a.Gs = Gs; a.stop = 2;
    return launch_step(h, a);
}

static int ensure_ws(tg_handle *h, int B)
{
    if (!h->cfg.warm_start || B <= h->ws_B) return TG_OK;
    cudaFree(h->ws_x); cudaFree(h->ws_y); cudaFree(h->ws_valid);
    h->ws_x = h->ws_y = nullptr; h->ws_valid = nullptr; h->ws_B = 0;
    CK(cudaMalloc(&h->ws_x, (size_t)B * h->dc.n * sizeof(double)));
    CK(cudaMalloc(&h->ws_y, (size_t)B * h->dc.m * sizeof(double)));
    CK(cudaMalloc(&h->ws_valid, (size_t)B * sizeof(int)));
    CK(cudaMemsetAsync(h->ws_valid, 0, (size_t)B * sizeof(int), h->stream));
    h->ws_B = B;
    return TG_OK;
}

int tg_mpc_step(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref, const double *vref,
                double *u_cmd, int32_t *status, int32_t *iters, double *objective, double *U_opt, double *X_opt, double *y_opt)
{
    return tg_mpc_step_ctrl(h, B, x0, u_prev, path_ref, vref, nullptr, u_cmd, status, iters, objective, U_opt, X_opt, y_opt);
}

int tg_mpc_step_ctrl(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref, const double *vref,
                     const tg_ctrl_spec *ctrl, double *u_cmd, int32_t *status, int32_t *iters, double *objective, double *U_opt,
                     double *X_opt, double *y_opt)
{
    if (!h || B < 0 || (B > 0 && (!x0 || !u_prev || !path_ref || !u_cmd))) return fail(TG_ERR_INVALID, "bad argument");
    CK(cudaSetDevice(h->device));
    int rc = ensure_ws(h, B);
    if (rc != TG_OK) return rc;
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.x0 = x0; a.u_prev = u_prev; a.path_ref = path_ref; a.vref = vref;
    a.u_cmd = u_cmd; a.status = status; a.iters = iters; a.objective = objective; a.U_opt = U_opt; a.X_opt = X_opt; a.y_opt = y_opt;
    a.ws_x = h->ws_x; a.ws_y = h->ws_y; a.ws_valid = h->ws_valid;
    a.ctrl = ctrl;
    return launch_step(h, a);
}

int tg_ref_window(tg_handle *h, int B, const double *x0, const tg_ref_spec *spec, const double *brk, const double *coef,
                  int t_index, double *path_ref, double *vref)
{
    if (!h || B < 0 || (B > 0 && (!x0 || !spec || !path_ref || !vref))) return fail(TG_ERR_INVALID, "bad argument");
    if (B == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    const int grid = B < 8 * h->num_sms ? B : 8 * h->num_sms;
    tg_ref_window_kernel<<<grid, 32, (size_t)h->Lref.total * sizeof(double), h->stream>>>(h->dc, h->Lref, B, x0, spec, brk, coef, t_index, path_ref, vref);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

int tg_closed_loop(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                   const double *brk, const double *coef, int64_t traj_id0, double *clean, double *noisy, double *U,
                   int32_t *status_counts, int64_t *iters_total)
{
    return tg_closed_loop_ctrl(h, B, T, x0, u0, spec, nullptr, brk, coef, traj_id0, clean, noisy, U, status_counts, iters_total);
}

int tg_closed_loop_ctrl(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                        const tg_ctrl_spec *ctrl, const double *brk, const double *coef, int64_t traj_id0, double *clean,
                        double *noisy, double *U, int32_t *status_counts, int64_t *iters_total)
{
    return tg_closed_loop_params(h, B, T, x0, u0, spec, ctrl, nullptr, brk, coef, traj_id0, clean, noisy, U, status_counts, iters_total);
}

int tg_closed_loop_params(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                          const tg_ctrl_spec *ctrl, const double *plant, const double *brk, const double *coef, int64_t traj_id0,
                          double *clean, double *noisy, double *U, int32_t *status_counts, int64_t *iters_total)
{
    if (!h || B < 0 || T < 0 || (B > 0 && (!x0 || !u0 || !spec || !clean || !noisy || (T > 0 && !U)))) return fail(TG_ERR_INVALID, "bad argument");
    if (B == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    LoopArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.T = T; a.x0 = x0; a.u0 = u0; a.spec = spec; a.brk = brk; a.coef = coef; a.traj_id0 = traj_id0;
    a.clean = clean; a.noisy = noisy; a.U = U; a.status_counts = status_counts; a.iters_total = (long long *)iters_total;
    a.ctrl = ctrl;
    a.plant = plant;
    const TwLaunch &t = ctrl ? h->tw_ctrl : h->tw;   // a plant table alone keeps the handle's own (compile-time-horizon) instances
    return plant ? launch_tw(h, t, t.k.loop_pt, t.k.loop_pt_p1, a) : launch_tw(h, t, t.k.loop, t.k.loop_p1, a);
}

// the rules of a plant table (include/trajgen.h): TG_ERR_INVALID naming the first bad row and field
int tg_check_plant_params(int B, const double *plant)
{
    static const char *const names[TG_NPARAMS] = {"Cm1", "Cm2", "Cr0", "Cr2", "Br", "Cr", "Dr", "Bf", "Cf", "Df", "m", "Iz", "lf",
                                                  "lr", "g", "maxAlpha", "vx_zero"};
    if (B < 0) return fail(TG_ERR_INVALID, "bad argument: B < 0");
    if (B > 0 && !plant) return fail(TG_ERR_INVALID, "bad argument: plant is null");
    for (int b = 0; b < B; ++b) {
        const double *r = plant + (size_t)b * TG_NPARAMS;
        auto bad = [&](int i, const char *why) { return fail(TG_ERR_INVALID, "plant row " + std::to_string(b) + ": " + names[i] + " " + why); };
        for (int i = 0; i < TG_NPARAMS; ++i)
            if (!std::isfinite(r[i])) return bad(i, "must be finite");
        for (int i : {P_m, P_Iz, P_vx_zero, P_maxAlpha})
            if (!(r[i] > 0.0)) return bad(i, "must be > 0");
    }
    return TG_OK;
}

int tg_plant_rollout(tg_handle *h, int B, int T, const double *x0, const double *U, double *X)
{
    return tg_plant_rollout_params(h, B, T, x0, U, nullptr, X);
}

int tg_plant_rollout_params(tg_handle *h, int B, int T, const double *x0, const double *U, const double *plant, double *X)
{
    if (!h || B < 0 || T < 0 || (B > 0 && (!x0 || !X || (T > 0 && !U)))) return fail(TG_ERR_INVALID, "bad argument");
    if (B == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    tg_plant_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(h->dc, B, T, x0, U, plant, X);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

int tg_sensor_noise(tg_handle *h, int64_t traj_id0, int n_traj, int n_rows, double *out)
{
    if (!h || n_traj < 0 || n_rows < 0 || ((long long)n_traj * n_rows > 0 && !out)) return fail(TG_ERR_INVALID, "bad argument");
    const long long tot = (long long)n_traj * n_rows;
    if (tot == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    tg_noise_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(h->dc.seed_base + (unsigned long long)traj_id0, n_traj, n_rows, out);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

// ---- scenario generation (tg_scenarios.cuh)
void tg_default_scenario_rules(tg_scenario_rules *r)
{
    memset(r, 0, sizeof(*r));
    const double lo[6] = {-2.0, 0.0, 0.0, 0.4, -0.05, -1.0}, hi[6] = {2.0, 0.0, 0.0, 1.5, 0.05, 1.0};   // generation_type1.py:260-265
    memcpy(r->x0_lo, lo, sizeof(lo)); memcpy(r->x0_hi, hi, sizeof(hi));
    r->lat_off[0] = -0.2; r->lat_off[1] = 0.2; r->head_off[0] = -0.2; r->head_off[1] = 0.2;
    r->vref0 = 0.8; r->vcruise[0] = 0.8; r->vcruise[1] = 2.0; r->t_ramp = 2.0;                          // MPC/main.py:87
    r->sine_A[0] = 0.2; r->sine_A[1] = 1.0; r->sine_k[0] = 0.3; r->sine_k[1] = 1.0; r->sine_psi[0] = 0.0; r->sine_psi[1] = 6.283185307179586;
    r->parab_c[0] = -0.2; r->parab_c[1] = 0.2;
    r->spl_x0 = -6.0; r->spl_dx[0] = 1.0; r->spl_dx[1] = 3.0; r->spl_sigma = 0.3; r->spl_knots = 27;
    r->n_cycle = 2; r->cycle[0] = TG_PATH_SPLINE; r->cycle[1] = TG_PATH_SINE;
    r->seed_base = 2025ull;
}

static int scenario_check(tg_handle *h, int B, const tg_scenario_rules *r)
{
    if (!h || !r || B < 0) return fail(TG_ERR_INVALID, "bad argument");
    if (r->spl_knots < 3 || r->spl_knots > TG_SCN_MAX_KNOTS) return fail(TG_ERR_INVALID, "scenario rules: 3 <= spl_knots <= 32");
    if (r->n_cycle < 1 || r->n_cycle > 4) return fail(TG_ERR_INVALID, "scenario rules: 1 <= n_cycle <= 4");
    for (int i = 0; i < r->n_cycle; ++i)
        if (r->cycle[i] < TG_PATH_PARABOLA || r->cycle[i] > TG_PATH_SPLINE) return fail(TG_ERR_INVALID, "scenario rules: cycle entries must be parabola / sine / spline");
    if (!(r->spl_dx[0] > 0) || r->spl_dx[1] < r->spl_dx[0]) return fail(TG_ERR_INVALID, "scenario rules: knot spacing must be positive");
    if ((long long)B * (r->spl_knots - 1) > 2147483647LL) return fail(TG_ERR_INVALID, "scenario rules: spline table index overflow");
    return TG_OK;
}

int tg_make_scenarios(tg_handle *h, int B, int64_t traj_id0, const tg_scenario_rules *rules, double *x0, double *u0,
                      tg_ref_spec *spec, double *spl_breaks, double *spl_coef)
{
    int rc = scenario_check(h, B, rules);
    if (rc != TG_OK) return rc;
    if (B == 0) return TG_OK;
    if (!x0 || !u0 || !spec || !spl_breaks || !spl_coef) return fail(TG_ERR_INVALID, "null output");
    CK(cudaSetDevice(h->device));
    tg_scenario_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(h->dc, *rules, B, (long long)traj_id0, x0, u0, spec, spl_breaks, spl_coef);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

// ---- open-loop generators (tg_openloop.cuh)
void tg_default_type1_rules(tg_type1_rules *r)
{
    memset(r, 0, sizeof(*r));
    r->d_mean = 0.2161; r->d_std = 0.1314; r->delta_mean = 0.0035; r->delta_std = 0.0338;    // generation_type1.py:250
    r->du_lo[0] = -0.1; r->du_hi[0] = 0.1; r->du_lo[1] = -0.04; r->du_hi[1] = 0.04;           // :251
    r->u_lo[0] = -1.0; r->u_hi[0] = 1.0; r->u_lo[1] = -0.6; r->u_hi[1] = 0.6;                 // :288-289
    r->transient_s[0] = 1.5; r->transient_s[1] = 3.0; r->checkpoint_s[0] = 3.0; r->checkpoint_s[1] = 5.0;
    r->period_s[0] = 4.0; r->period_s[1] = 8.0; r->amp_frac[0] = 0.5; r->amp_frac[1] = 1.5;
    r->p_straight = 0.5; r->tr_d_frac = 0.2; r->tr_delta_frac = 0.3; r->st_d_frac = 0.05;
    r->sin_noise_frac = 0.1; r->straight_frac = 0.01; r->ctrl_noise_frac = 0.1; r->mode = -1;
}

void tg_default_type2_rules(tg_type2_rules *r)
{
    memset(r, 0, sizeof(*r));
    r->v_turn_max = 1.2; r->v_high = 4.0; r->d_range[0] = 0.0; r->d_range[1] = 0.33;          // generation_type2.py:24-27
    r->delta_turn_range[0] = 0.015; r->delta_turn_range[1] = 0.04; r->delta_straight_noise = 0.004;
    r->delta_rate_max = 0.30; r->v_floor = 0.35; r->d_boost_min = 0.15;                         // :97,:100
    r->seg_s[0] = 0.4; r->seg_s[1] = 1.5;                                                       // :114
    r->p_modes[0] = 0.35; r->p_modes[1] = 0.35; r->p_modes[2] = 0.15; r->p_modes[3] = 0.15;     // :112
    r->p_after_turn[0] = 0.5; r->p_after_turn[1] = 0.5;                                         // :109
    r->acc_d_lo = 0.3; r->cruise_d[0] = -0.05; r->cruise_d[1] = 0.2;                            // :120,:122
    r->turn_d_fast[0] = 0.0; r->turn_d_fast[1] = 0.15; r->turn_d_slow[0] = 0.05; r->turn_d_slow[1] = 0.25;   // :124
    r->stall_v = 0.5; r->stall_d[0] = 0.5; r->stall_d[1] = 1.0; r->stall_min_s = 0.3;           // :131-133
    r->delta_clip = 0.6;                                                                        // :141
}

static int openloop_check(tg_handle *h, int B, int T, const double *x0, const void *rules, const double *clean,
                          const double *noisy, const double *U)
{
    if (!h || B < 0 || T < 1 || !rules || (B > 0 && !x0)) return fail(TG_ERR_INVALID, "bad argument (T >= 1 required)");
    if (((uintptr_t)clean | (uintptr_t)noisy | (uintptr_t)U) & 15) return fail(TG_ERR_INVALID, "clean / noisy / U must be 16-byte aligned");
    return TG_OK;
}

extern "C++" {
template <int KIND, typename Rules>
static int openloop_launch(tg_handle *h, int B, int T, const double *x0, const Rules &rules, uint64_t ctrl_seed_base,
                           int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes)
{
    if (B == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    OpenLoopArgs a;
    a.B = B; a.T = T; a.x0 = x0; a.traj_id0 = traj_id0; a.ctrl_seed_base = ctrl_seed_base;
    a.clean = clean; a.noisy = noisy; a.U = U; a.modes = (signed char *)modes; a.plant = plant;
    const int per_cta = 32 * TG_OL_WARPS;
    const size_t smem = TG_OL_WARPS * TG_OL_TILE * sizeof(double);
    if (plant) tg_openloop_kernel<KIND, Rules, true><<<(B + per_cta - 1) / per_cta, per_cta, smem, h->stream>>>(h->dc, rules, a);
    else tg_openloop_kernel<KIND, Rules, false><<<(B + per_cta - 1) / per_cta, per_cta, smem, h->stream>>>(h->dc, rules, a);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}
}  // extern "C++"

int tg_openloop_type1(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules, uint64_t ctrl_seed_base,
                      int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes)
{
    return tg_openloop_type1_params(h, B, T, x0, rules, ctrl_seed_base, traj_id0, nullptr, clean, noisy, U, modes);
}

int tg_openloop_type1_params(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules, uint64_t ctrl_seed_base,
                             int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes)
{
    int rc = openloop_check(h, B, T, x0, rules, clean, noisy, U);
    if (rc != TG_OK) return rc;
    const tg_type1_rules &r = *rules;
    const double Ts = h->dc.Ts;
    if (!(r.transient_s[0] > 0) || r.transient_s[1] < r.transient_s[0] || !(r.checkpoint_s[0] > 0) || r.checkpoint_s[1] < r.checkpoint_s[0] ||
        !(r.period_s[0] > 0) || r.period_s[1] < r.period_s[0] || r.mode < -1 || r.mode > 1)
        return fail(TG_ERR_INVALID, "type-1 rules: bad range");
    if ((int)(r.transient_s[0] / Ts) < 1) return fail(TG_ERR_INVALID, "type-1 rules: the transient must last at least one step");
    {   // knots of the transient spline in the worst case (longest transient, densest checkpoints)
        const double n_tr = std::min((double)T, std::floor(r.transient_s[1] / Ts));
        const double every = std::max(1.0, std::nearbyint(r.checkpoint_s[0] / Ts));
        if (std::ceil(n_tr / every) + 1 > TG_OL_MAX_KNOTS) return fail(TG_ERR_UNSUPPORTED, "type-1 rules: more than 16 spline knots in the transient");
    }
    return openloop_launch<1>(h, B, T, x0, r, ctrl_seed_base, traj_id0, plant, clean, noisy, U, modes);
}

int tg_openloop_type2(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules, uint64_t ctrl_seed_base,
                      int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes)
{
    return tg_openloop_type2_params(h, B, T, x0, rules, ctrl_seed_base, traj_id0, nullptr, clean, noisy, U, modes);
}

int tg_openloop_type2_params(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules, uint64_t ctrl_seed_base,
                             int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes)
{
    int rc = openloop_check(h, B, T, x0, rules, clean, noisy, U);
    if (rc != TG_OK) return rc;
    const tg_type2_rules &r = *rules;
    double tot4 = 0, tot2 = 0;
    for (int i = 0; i < 4; ++i) { if (!(r.p_modes[i] >= 0)) return fail(TG_ERR_INVALID, "type-2 rules: negative probability"); tot4 += r.p_modes[i]; }
    for (int i = 0; i < 2; ++i) { if (!(r.p_after_turn[i] >= 0)) return fail(TG_ERR_INVALID, "type-2 rules: negative probability"); tot2 += r.p_after_turn[i]; }
    if (!(tot4 > 0) || !(tot2 > 0) || !(r.seg_s[0] > 0) || r.seg_s[1] < r.seg_s[0]) return fail(TG_ERR_INVALID, "type-2 rules: bad range");
    return openloop_launch<2>(h, B, T, x0, r, ctrl_seed_base, traj_id0, plant, clean, noisy, U, modes);
}

// ---- estimator physics (tg_estimator.cuh)
extern "C++" {
template <typename T>
static EstCfg<T> make_est_cfg(const tg_handle *h, const tg_state_limits *lim)
{
    EstCfg<T> e;
    const double *p = h->cfg.params;
    e.Ts = (T)h->cfg.Ts;
    for (int i = 0; i < 6; ++i) { e.lo[i] = (T)lim->lo[i]; e.hi[i] = (T)lim->hi[i]; }
    e.Cm1 = (T)p[P_Cm1]; e.Cm2 = (T)p[P_Cm2]; e.Cr0 = (T)p[P_Cr0]; e.Cr2 = (T)p[P_Cr2];
    e.Br = (T)p[P_Br]; e.Cr = (T)p[P_Cr]; e.Dr = (T)p[P_Dr]; e.Bf = (T)p[P_Bf]; e.Cf = (T)p[P_Cf]; e.Df = (T)p[P_Df];
    e.m = (T)p[P_m]; e.Iz = (T)p[P_Iz]; e.lf = (T)p[P_lf]; e.lr = (T)p[P_lr]; e.maxAlpha = (T)p[P_maxAlpha];
    // KalmanNet/vehicle_model.py:26 builds the threshold as a float32 tensor whatever the state dtype
    e.vx_zero = (T)(float)p[P_vx_zero];
    return e;
}
}  // extern "C++"

static bool est_aligned(int dtype, std::initializer_list<const void *> ptrs)
{
    const uintptr_t mask = dtype == 0 ? 15 : 7;      // the kernels move pairs of values
    for (const void *p : ptrs)
        if ((uintptr_t)p & mask) return false;
    return true;
}

static int est_check(tg_handle *h, int B, int dtype, const tg_state_limits *lim)
{
    if (!h || B < 0 || !lim || (dtype != 0 && dtype != 1)) return fail(TG_ERR_INVALID, "bad argument (dtype: 0 = fp64, 1 = fp32)");
    for (int i = 0; i < 6; ++i)
        if (!(lim->lo[i] <= lim->hi[i])) return fail(TG_ERR_INVALID, "state limits: lo > hi");
    return TG_OK;
}

int tg_estimator_step(tg_handle *h, int B, int dtype, const void *x, const void *u, const tg_state_limits *lim, void *x_next)
{
    int rc = est_check(h, B, dtype, lim);
    if (rc != TG_OK) return rc;
    if (B == 0) return TG_OK;
    if (!x || !u || !x_next) return fail(TG_ERR_INVALID, "null argument");
    if (!est_aligned(dtype, {x, u, x_next})) return fail(TG_ERR_INVALID, "buffers must be aligned to two elements (8 B fp32 / 16 B fp64)");
    CK(cudaSetDevice(h->device));
    const int blocks = (B + 127) / 128;
    if (dtype == 0) tg_estimator_step_kernel<double><<<blocks, 128, 0, h->stream>>>(make_est_cfg<double>(h, lim), B, (const double *)x, (const double *)u, (double *)x_next);
    else tg_estimator_step_kernel<float><<<blocks, 128, 0, h->stream>>>(make_est_cfg<float>(h, lim), B, (const float *)x, (const float *)u, (float *)x_next);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

int tg_estimator_step_vjp(tg_handle *h, int B, int dtype, const void *x, const void *u, const tg_state_limits *lim,
                          const void *grad_next, void *grad_x, void *grad_u)
{
    int rc = est_check(h, B, dtype, lim);
    if (rc != TG_OK) return rc;
    if (B == 0) return TG_OK;
    if (!x || !u || !grad_next) return fail(TG_ERR_INVALID, "null argument");
    if (!est_aligned(dtype, {x, u, grad_next, grad_x, grad_u})) return fail(TG_ERR_INVALID, "buffers must be aligned to two elements (8 B fp32 / 16 B fp64)");
    CK(cudaSetDevice(h->device));
    const int blocks = (B + 127) / 128;
    if (dtype == 0) tg_estimator_vjp_kernel<double><<<blocks, 128, 0, h->stream>>>(make_est_cfg<double>(h, lim), B, (const double *)x, (const double *)u, (const double *)grad_next, (double *)grad_x, (double *)grad_u);
    else tg_estimator_vjp_kernel<float><<<blocks, 128, 0, h->stream>>>(make_est_cfg<float>(h, lim), B, (const float *)x, (const float *)u, (const float *)grad_next, (float *)grad_x, (float *)grad_u);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

int tg_estimator_rollout(tg_handle *h, int B, int dtype, int T_u, int t_start, int H, const void *x0, const void *U,
                         const tg_state_limits *lim, void *preds, int32_t *H_out)
{
    int rc = est_check(h, B, dtype, lim);
    if (rc != TG_OK) return rc;
    if (T_u < 0 || t_start < 0 || H < 0) return fail(TG_ERR_INVALID, "bad argument");
    const int Hn = std::max(0, std::min(H, T_u - t_start));       // test_prediction.py:79: stop at the end of u
    if (H_out) *H_out = Hn;
    if (B == 0 || Hn == 0) return TG_OK;
    if (!x0 || !U || !preds) return fail(TG_ERR_INVALID, "null argument");
    CK(cudaSetDevice(h->device));
    const int blocks = (B + 63) / 64;
    if (dtype == 0) tg_estimator_rollout_kernel<double><<<blocks, 64, 0, h->stream>>>(make_est_cfg<double>(h, lim), B, T_u, t_start, Hn, (const double *)x0, (const double *)U, (double *)preds);
    else tg_estimator_rollout_kernel<float><<<blocks, 64, 0, h->stream>>>(make_est_cfg<float>(h, lim), B, T_u, t_start, Hn, (const float *)x0, (const float *)U, (float *)preds);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

int tg_philox_u32(tg_handle *h, uint64_t seed, uint32_t first, uint32_t block, int n, uint32_t *out)
{
    if (!h || n < 0 || (n > 0 && !out)) return fail(TG_ERR_INVALID, "bad argument");
    if (n == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    tg_philox_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(seed, first, block, n, out);
    h->launches += 1;
    CK(cudaGetLastError());
    return TG_OK;
}

int tg_fma_peak(tg_handle *h, int dtype, double *tflops)
{
    if (!h || !tflops) return fail(TG_ERR_INVALID, "null argument");
    CK(cudaSetDevice(h->device));
    const int blocks = h->num_sms * 8, threads = 256, iters = 1 << 15;
    void *buf = nullptr;
    CK(cudaMalloc(&buf, (size_t)blocks * threads * 8));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(e0, h->stream));
        if (dtype == 0) tg_fma_peak_kernel<double><<<blocks, threads, 0, h->stream>>>((double *)buf, iters);
        else tg_fma_peak_kernel<float><<<blocks, threads, 0, h->stream>>>((float *)buf, iters);
        CK(cudaEventRecord(e1, h->stream));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
        h->launches += 1;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf);
    *tflops = 2.0 * 8.0 * (double)iters * blocks * threads / (best * 1e-3) / 1e12;
    return TG_OK;
}

int tg_malloc(void **p, int64_t bytes) { if (!p || bytes < 0) return fail(TG_ERR_INVALID, "bad argument"); *p = nullptr; if (bytes == 0) return TG_OK; CK(cudaMalloc(p, (size_t)bytes)); return TG_OK; }
int tg_malloc_on(tg_handle *h, void **p, int64_t bytes)
{
    if (!h) return fail(TG_ERR_INVALID, "null handle");
    CK(cudaSetDevice(h->device));
    return tg_malloc(p, bytes);
}
int tg_free(void *p) { if (p) CK(cudaFree(p)); return TG_OK; }
int tg_malloc_host(void **p, int64_t bytes) { if (!p || bytes < 0) return fail(TG_ERR_INVALID, "bad argument"); *p = nullptr; if (bytes == 0) return TG_OK; CK(cudaMallocHost(p, (size_t)bytes)); return TG_OK; }
int tg_free_host(void *p) { if (p) CK(cudaFreeHost(p)); return TG_OK; }
int tg_memcpy_h2d(tg_handle *h, void *dst, const void *src, int64_t bytes)
{
    if (!h || bytes < 0) return fail(TG_ERR_INVALID, "bad argument");
    if (bytes == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return TG_OK;
}
int tg_memcpy_d2h(tg_handle *h, void *dst, const void *src, int64_t bytes)
{
    if (!h || bytes < 0) return fail(TG_ERR_INVALID, "bad argument");
    if (bytes == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return TG_OK;
}

// ---- host-buffer entry points: stage through one device arena, copies on the handle's stream
static int ensure_dstage(tg_handle *h, size_t bytes)
{
    if (bytes <= h->dstage_bytes) return TG_OK;
    if (h->dstage) { CK(cudaStreamSynchronize(h->stream)); CK(cudaFree(h->dstage)); h->dstage = nullptr; h->dstage_bytes = 0; }
    CK(cudaMalloc(&h->dstage, bytes));
    h->dstage_bytes = bytes;
    return TG_OK;
}

// The buffers of one *_host call, each listed once: in() before the launch, out() after it.  stage() sizes the arena from
// the list, points each device pointer at its slot and enqueues the host-to-device copies; finish() enqueues the
// device-to-host copies and synchronises.  A null host pointer or zero bytes gives a null device pointer and no copy, so an
// optional output the caller leaves out is one the kernel does not store.  Slots start on 256-byte boundaries (the open-loop
// kernels store double2).
extern "C++" {
class HostStage {
public:
    explicit HostStage(tg_handle *h) : h_(h) {}
    template <typename T> void in(T *&dev, const T *host, size_t bytes) { add(dev, const_cast<T *>(host), bytes, true); }
    // alias: where the kernel stores straight into the caller's (pinned) buffer; nothing is staged or copied then
    template <typename T> void out(T *&dev, T *host, size_t bytes, T *alias = nullptr)
    {
        if (alias) dev = alias;
        else add(dev, host, bytes, false);
    }
    int stage()
    {
        const int rc = ensure_dstage(h_, end_);
        if (rc != TG_OK) return rc;
        for (const Buf &b : bufs_) {
            char *p = (char *)h_->dstage + b.off;
            b.set(b.dev, p);
            if (b.in) CK(cudaMemcpyAsync(p, b.host, b.bytes, cudaMemcpyHostToDevice, h_->stream));
        }
        return TG_OK;
    }
    int finish()
    {
        for (const Buf &b : bufs_)
            if (!b.in) CK(cudaMemcpyAsync(b.host, (char *)h_->dstage + b.off, b.bytes, cudaMemcpyDeviceToHost, h_->stream));
        CK(cudaStreamSynchronize(h_->stream));
        return TG_OK;
    }

private:
    struct Buf { void *dev; void (*set)(void *, char *); void *host; size_t bytes, off; bool in; };
    template <typename T> static void set_ptr(void *dev, char *p) { *static_cast<T **>(dev) = reinterpret_cast<T *>(p); }
    template <typename T> void add(T *&dev, T *host, size_t bytes, bool in)
    {
        dev = nullptr;
        if (!host || !bytes) return;
        bufs_.push_back({&dev, &set_ptr<T>, host, bytes, end_, in});
        end_ = (end_ + bytes + 255) & ~(size_t)255;
    }
    tg_handle *h_;
    std::vector<Buf> bufs_;
    size_t end_ = 0;
};
}  // extern "C++"

int tg_mpc_step_host(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref, const double *vref,
                     double *u_cmd, int32_t *status, int32_t *iters, double *objective, double *U_opt, double *X_opt, double *y_opt)
{
    return tg_mpc_step_ctrl_host(h, B, x0, u_prev, path_ref, vref, nullptr, u_cmd, status, iters, objective, U_opt, X_opt, y_opt);
}

int tg_mpc_step_ctrl_host(tg_handle *h, int B, const double *x0, const double *u_prev, const double *path_ref, const double *vref,
                          const tg_ctrl_spec *ctrl, double *u_cmd, int32_t *status, int32_t *iters, double *objective,
                          double *U_opt, double *X_opt, double *y_opt)
{
    if (!h || B < 0 || (B > 0 && (!x0 || !u_prev || !path_ref || !u_cmd))) return fail(TG_ERR_INVALID, "bad argument");
    if (ctrl) { const int rc = tg_check_ctrl(B, ctrl, bounded_states(h)); if (rc != TG_OK) return rc; }
    if (B == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    const int N = h->dc.N, n = h->dc.n, m = h->dc.m;
    const size_t b8 = sizeof(double);
    double *d_x0, *d_up, *d_pr, *d_vr, *d_uc, *d_ob, *d_U, *d_X, *d_y;
    int32_t *d_st, *d_it;
    tg_ctrl_spec *d_ct;
    HostStage s(h);
    s.in(d_x0, x0, (size_t)B * 6 * b8);
    s.in(d_up, u_prev, (size_t)B * 2 * b8);
    s.in(d_pr, path_ref, (size_t)B * (N + 1) * 3 * b8);
    s.in(d_vr, vref, (size_t)B * (N + 1) * b8);
    s.in(d_ct, ctrl, (size_t)B * sizeof(tg_ctrl_spec));
    s.out(d_uc, u_cmd, (size_t)B * 2 * b8);
    s.out(d_st, status, (size_t)B * 4);
    s.out(d_it, iters, (size_t)B * 4);
    s.out(d_ob, objective, (size_t)B * b8);
    s.out(d_U, U_opt, (size_t)B * n * b8);
    s.out(d_X, X_opt, (size_t)B * (N + 1) * 6 * b8);
    s.out(d_y, y_opt, (size_t)B * m * b8);
    int rc = s.stage();
    if (rc != TG_OK) return rc;
    rc = tg_mpc_step_ctrl(h, B, d_x0, d_up, d_pr, d_vr, d_ct, d_uc, d_st, d_it, d_ob, d_U, d_X, d_y);
    if (rc != TG_OK) return rc;
    return s.finish();
}

// device alias of a pinned (cudaHostAlloc'ed / registered) host buffer, or null for pageable memory
static void *pinned_device_alias(const void *p)
{
    cudaPointerAttributes at;
    if (!p || cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

int tg_closed_loop_host(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                        const double *brk, int64_t n_breaks, const double *coef, int64_t n_coef, int64_t traj_id0,
                        double *clean, double *noisy, double *U, int32_t *status_counts, int64_t *iters_total)
{
    return tg_closed_loop_ctrl_host(h, B, T, x0, u0, spec, nullptr, brk, n_breaks, coef, n_coef, traj_id0, clean, noisy, U,
                                    status_counts, iters_total);
}

int tg_closed_loop_ctrl_host(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                             const tg_ctrl_spec *ctrl, const double *brk, int64_t n_breaks, const double *coef, int64_t n_coef,
                             int64_t traj_id0, double *clean, double *noisy, double *U, int32_t *status_counts,
                             int64_t *iters_total)
{
    return tg_closed_loop_params_host(h, B, T, x0, u0, spec, ctrl, nullptr, brk, n_breaks, coef, n_coef, traj_id0, clean, noisy, U,
                                      status_counts, iters_total);
}

int tg_closed_loop_params_host(tg_handle *h, int B, int T, const double *x0, const double *u0, const tg_ref_spec *spec,
                               const tg_ctrl_spec *ctrl, const double *plant, const double *brk, int64_t n_breaks,
                               const double *coef, int64_t n_coef, int64_t traj_id0, double *clean, double *noisy, double *U,
                               int32_t *status_counts, int64_t *iters_total)
{
    if (!h || B < 0 || T < 0 || (B > 0 && (!x0 || !u0 || !spec || !clean || !noisy || (T > 0 && !U)))) return fail(TG_ERR_INVALID, "bad argument");
    if (ctrl) { const int rc = tg_check_ctrl(B, ctrl, bounded_states(h)); if (rc != TG_OK) return rc; }
    if (plant) { const int rc = tg_check_plant_params(B, plant); if (rc != TG_OK) return rc; }
    if (B == 0) return TG_OK;
    {   // the scenario table is host memory here: reject what would send the device out of bounds
        const int64_t n_tab = (brk && coef) ? (n_breaks < n_coef ? n_breaks : n_coef) : 0;
        for (int b = 0; b < B; ++b) {
            const tg_ref_spec &sp = spec[b];
            if (sp.path_kind < TG_PATH_PARABOLA || sp.path_kind > TG_PATH_ARC || sp.vref_kind < TG_VREF_HOLD || sp.vref_kind > TG_VREF_SINE)
                return fail(TG_ERR_INVALID, "scenario " + std::to_string(b) + ": unknown path_kind / vref_kind");
            if (sp.path_kind == TG_PATH_SPLINE || sp.path_kind == TG_PATH_ARC) {
                const int64_t need_c = (int64_t)sp.spline_first + (sp.path_kind == TG_PATH_ARC ? 2 : 1) * (int64_t)sp.spline_count;
                if (sp.spline_count < 1 || sp.spline_first < 0 || (int64_t)sp.spline_first + sp.spline_count > n_tab || need_c > n_coef || !coef)
                    return fail(TG_ERR_INVALID, "scenario " + std::to_string(b) + ": spline pieces outside the break / coefficient tables");
            }
        }
    }
    CK(cudaSetDevice(h->device));
    const size_t b8 = sizeof(double);
    const size_t s_cl = (size_t)B * (T + 1) * 6 * b8;
    // Rows leave the SM at ~1 GB/s (112 B per MPC step), far below what PCIe carries, so when the caller's result buffers
    // are pinned the kernel stores straight into them (posted writes overlap the computation) and the device-to-host copy
    // of the rows after the kernel disappears.  Pageable buffers are staged through the device arena.
    double *a_cl = (double *)pinned_device_alias(clean), *a_no = (double *)pinned_device_alias(noisy), *a_U = (double *)pinned_device_alias(U);
    const bool direct = a_cl && a_no && (a_U || T == 0);
    double *d_x0, *d_u0, *d_bk, *d_cf, *d_cl, *d_no, *d_U, *d_pl;
    tg_ref_spec *d_sp;
    int32_t *d_sc;
    int64_t *d_it;
    tg_ctrl_spec *d_ct;
    HostStage s(h);
    s.in(d_x0, x0, (size_t)B * 6 * b8);
    s.in(d_u0, u0, (size_t)B * 2 * b8);
    s.in(d_sp, spec, (size_t)B * sizeof(tg_ref_spec));
    s.in(d_bk, brk, (size_t)(n_breaks > 0 ? n_breaks : 0) * b8);
    s.in(d_cf, coef, (size_t)(n_coef > 0 ? n_coef : 0) * 4 * b8);
    s.in(d_ct, ctrl, (size_t)B * sizeof(tg_ctrl_spec));
    s.in(d_pl, plant, (size_t)B * TG_NPARAMS * b8);
    s.out(d_cl, clean, s_cl, direct ? a_cl : nullptr);
    s.out(d_no, noisy, s_cl, direct ? a_no : nullptr);
    s.out(d_U, U, (size_t)B * T * 2 * b8, direct ? a_U : nullptr);
    s.out(d_sc, status_counts, (size_t)B * TG_NUM_STATUS * 4);
    s.out(d_it, iters_total, (size_t)B * 8);
    int rc = s.stage();
    if (rc != TG_OK) return rc;
    rc = tg_closed_loop_params(h, B, T, d_x0, d_u0, d_sp, d_ct, d_pl, d_bk, d_cf, traj_id0, d_cl, d_no, d_U, d_sc, d_it);
    if (rc != TG_OK) return rc;
    return s.finish();
}

int tg_make_scenarios_host(tg_handle *h, int B, int64_t traj_id0, const tg_scenario_rules *rules, double *x0, double *u0,
                           tg_ref_spec *spec, double *spl_breaks, double *spl_coef)
{
    int rc = scenario_check(h, B, rules);
    if (rc != TG_OK) return rc;
    if (B == 0) return TG_OK;
    if (!x0 || !u0 || !spec || !spl_breaks || !spl_coef) return fail(TG_ERR_INVALID, "null output");
    CK(cudaSetDevice(h->device));
    const size_t P = (size_t)rules->spl_knots - 1;
    double *d_x0, *d_u0, *d_bk, *d_cf;
    tg_ref_spec *d_sp;
    HostStage s(h);
    s.out(d_x0, x0, (size_t)B * 48);
    s.out(d_u0, u0, (size_t)B * 16);
    s.out(d_sp, spec, (size_t)B * sizeof(tg_ref_spec));
    s.out(d_bk, spl_breaks, (size_t)B * P * 8);
    s.out(d_cf, spl_coef, (size_t)B * P * 32);
    rc = s.stage();
    if (rc != TG_OK) return rc;
    rc = tg_make_scenarios(h, B, traj_id0, rules, d_x0, d_u0, d_sp, d_bk, d_cf);
    if (rc != TG_OK) return rc;
    return s.finish();
}

extern "C++" {
template <typename Rules>
static int openloop_host(int (*launch)(tg_handle *, int, int, const double *, const Rules *, uint64_t, int64_t, const double *,
                                       double *, double *, double *, int8_t *),
                         tg_handle *h, int B, int T, const double *x0, const Rules *rules, uint64_t ctrl_seed_base,
                         int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes,
                         size_t n_modes)
{
    if (!h || B < 0 || T < 1 || !rules || (B > 0 && !x0)) return fail(TG_ERR_INVALID, "bad argument (T >= 1 required)");
    if (plant) { const int rc = tg_check_plant_params(B, plant); if (rc != TG_OK) return rc; }
    if (B == 0) return TG_OK;
    CK(cudaSetDevice(h->device));
    const size_t b8 = sizeof(double), s_cl = (size_t)B * (T + 1) * 6 * b8;
    double *d_x0, *d_pl, *d_cl, *d_no, *d_U;
    int8_t *d_m;
    HostStage s(h);
    s.in(d_x0, x0, (size_t)B * 6 * b8);
    s.out(d_cl, clean, s_cl);
    s.out(d_no, noisy, s_cl);
    s.out(d_U, U, (size_t)B * T * 2 * b8);
    s.out(d_m, modes, n_modes);
    s.in(d_pl, plant, (size_t)B * TG_NPARAMS * b8);
    int rc = s.stage();
    if (rc != TG_OK) return rc;
    rc = launch(h, B, T, d_x0, rules, ctrl_seed_base, traj_id0, d_pl, d_cl, d_no, d_U, d_m);
    if (rc != TG_OK) return rc;
    return s.finish();
}
}  // extern "C++"

int tg_openloop_type1_host(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules, uint64_t ctrl_seed_base,
                           int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes)
{
    return tg_openloop_type1_params_host(h, B, T, x0, rules, ctrl_seed_base, traj_id0, nullptr, clean, noisy, U, modes);
}

int tg_openloop_type1_params_host(tg_handle *h, int B, int T, const double *x0, const tg_type1_rules *rules, uint64_t ctrl_seed_base,
                                  int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes)
{
    return openloop_host(tg_openloop_type1_params, h, B, T, x0, rules, ctrl_seed_base, traj_id0, plant, clean, noisy, U, modes,
                         (size_t)(B > 0 ? B : 0));
}

int tg_openloop_type2_host(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules, uint64_t ctrl_seed_base,
                           int64_t traj_id0, double *clean, double *noisy, double *U, int8_t *modes)
{
    return tg_openloop_type2_params_host(h, B, T, x0, rules, ctrl_seed_base, traj_id0, nullptr, clean, noisy, U, modes);
}

int tg_openloop_type2_params_host(tg_handle *h, int B, int T, const double *x0, const tg_type2_rules *rules, uint64_t ctrl_seed_base,
                                  int64_t traj_id0, const double *plant, double *clean, double *noisy, double *U, int8_t *modes)
{
    return openloop_host(tg_openloop_type2_params, h, B, T, x0, rules, ctrl_seed_base, traj_id0, plant, clean, noisy, U, modes,
                         (size_t)(B > 0 ? B : 0) * (size_t)(T > 0 ? T : 0));
}

}  // extern "C"
