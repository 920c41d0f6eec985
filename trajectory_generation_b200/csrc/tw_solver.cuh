// tw_solver.cuh -- one MPC step for one problem by W warps; W = 1 (horizons N <= 14) is a warp per problem with no CTA
// barrier anywhere on the path (sm_100a, fp64).
//
// Replaces MPC/mpc_6stati.py:165-275 (nominal rollout, N x linearize_discretize, CVXPY problem construction, OSQP solve,
// receding-horizon output) with
//   K1  nominal rollout (one lane pair: front / rear tyre chain, tables), reference window and sensor noise of the row,
//       per-stage linearisation (one lane per stage, compact 20-word records in shared memory)
//   K2  condensing in dU = U - u_prev.  Lane j owns column j of G_k (6 registers) and walks the horizon; per stage it emits
//       three scaled rows W (lateral error, heading, speed); H = sum_k W_k' W_k + band terms accumulates in the tile
//   K3  ADMM (the OSQP iteration) on K = H + sigma I + A' diag(rho) A.
// The n x n symmetric matrix (n = 2N) lives in registers as its LOWER TRIANGLE only: 4 x 4 blocks (I, J), J <= I, dealt
// row-major over the 32 W threads, S blocks ("slots") per thread (tw_shape) -- n = 40 is 55 blocks on the 64 threads of two
// warps, 16 doubles per thread.  K^-1 comes from n symmetric sweep steps on that tile (one shared-memory round trip per pivot, the
// pivot-row index inside a block is a compile-time constant); x~ = K^-1 rhs is 2 x 16 FMAs per off-diagonal block, with
// the block partials exchanged through shared memory.  The ADMM vectors live in shared memory, lane t owns stage t (the
// entries 2t, 2t+1 of dU and its two box and two rate rows).
#pragma once
#include <type_traits>
#include "tg_device.cuh"

// optional phase timing (development): -DTG_PHASE_TIMING accumulates clock64 deltas of CTA 0 / thread 0 per phase
#ifdef TG_PHASE_TIMING
__device__ long long g_tg_phase[16];
#define TG_TICK(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) { const long long t__ = clock64(); g_tg_phase[i] += t__ - tg_last_tick; tg_last_tick = t__; } } while (0)
#define TG_TICK_DECL long long tg_last_tick = clock64()
#else
#define TG_TICK(i) do { } while (0)
#define TG_TICK_DECL do { } while (0)
#endif

// misc slots (doubles): 0 c0, 2 rho scale, 8..13 next state, 14..15 applied input, 16..19 counters (as 32/64-bit ints)
enum { M_C0 = 0, M_RHOSCALE = 2, M_XNEXT = 8, M_UCMD = 14, M_CNT = 16 };

struct StepTaps {   // optional debug/parity outputs of this problem (global memory, may be null)
    double *A, *Bm, *g, *xbar;          // tg_linearize
    double *H, *q, *c0, *l, *u, *Gs;    // tg_assemble
    int stop;                           // 0 = full step, 1 = stop after linearisation, 2 = stop after assembly
};

struct FusedCtx {   // closed-loop extras handled inside the step body
    const double *brk, *coef;   // spline tables (global)
    double *noisy_row;          // where the noisy copy of the CURRENT state goes (global), or null
    unsigned long long seed;
    int t_index;
};

struct StepResult {
    int status, iters;
    double objective;
    bool free_end;              // the solve ended with every dual at zero (no active row)
};

// barrier of a thread group of the CTA
__device__ __forceinline__ void tg_sync(int bar, int nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(nthreads) : "memory");
}

#define TW_WARM_RESTART_ITER 300
#define TW_FREE_RHO 1e-6         // rho scale of a solve that starts with no active row (see tw_step_body)
#define TW_POLISH_MARGIN 1e-3    // a converged standard solve is polished if every row is this far inside its bounds

// shared-memory layout of one problem (offsets in doubles) on a shape, identical on host and device.  Everything that does not
// depend on the number of state-bound rows ms comes first, so that for a compile-time horizon (template parameter NC of the
// kernels) every offset of the fixed part is an immediate in the load / store instructions; the state-row arrays form the tail.
struct WLayout {
    int x0, uprev, misc, spec, xbar, lin, rr, sn, cs, q, x, xt, v, z, y, rho, rinv, dyr, piv, wb, red;
    int aux, Xr, Yr, Pr, vref, P;   // inside the wb region (dead before / after K2)
    int dH, dsc;                    // dH aliases v, dsc aliases xt
    int NV, nb, nbuf;
    int zs, ys, rhos, rinvs, ls, us, zts, dys, tv, gt, Gs;   // tail: state rows (ms each; tv ms; gt 3 NV; Gs packed, tw_gs_*)
    int total;
};

__host__ __device__ constexpr int tw_even(int v) { return (v + 1) & ~1; }   // keep 16-byte alignment

// State-bound rows (mpc_6stati.py:216-221).  Row i = k ns + si is row sidx[si] of G_{k+1} (k = 0 .. N-1); it vanishes in the
// columns >= 2 (k + 1) (inputs that come later), so the rows are stored PACKED: the ns rows of stage k have length
// len_k = 4 ceil((k + 1) / 2) (zero-padded to whole 4-blocks of the tile) and start at ns off_k, off_k = sum_{k' < k} len_k'.
// Half the dense ms x NV block: N = 50 with two bounded states is 41 KB instead of 80 KB.
__host__ __device__ constexpr int tw_gs_len(int k) { return 4 * ((k >> 1) + 1); }
__host__ __device__ constexpr int tw_gs_off(int k) { return 4 * (k >> 1) * ((k >> 1) + 1) + ((k & 1) ? 4 * ((k >> 1) + 1) : 0); }

// shape of the solver for horizon N: W warps per problem, S tile blocks per thread (28, 55, 120 and 253 blocks on 32 W
// threads, 406 on 512 slots); W = 0: N is not supported
struct TwShape { int W, S; };
__host__ __device__ constexpr TwShape tw_shape(int N)
{ return N <= 14 ? TwShape{1, 1} : N <= 20 ? TwShape{2, 1} : N <= 30 ? TwShape{4, 1} : N <= 44 ? TwShape{8, 1} : N <= 56 ? TwShape{8, 2} : TwShape{0, 0}; }

// Block vectors that every thread reads at its block row AND its block column (the pivot rows of the sweep, the staging rows of
// the condensing) are stored PADDED: the four entries of block I at 6 I .. 6 I + 3.  The 16-byte pieces that the lanes of a warp
// read then fall into distinct banks (stride 48 bytes: 8 block rows cover the 32 banks once) instead of colliding pairwise
// (stride 32 bytes: block rows I and I + 4 share their banks): one wavefront per 128-bit load instead of two.
// (Not on the two-tiles-per-thread shape, N > 44, whose constrained problems need the shared memory for their second resident
// CTA, and not on the one-warp shape, N <= 14, where it gains nothing and costs the sixteenth resident CTA.)
__host__ __device__ constexpr int tw_ps(int W, int S) { return (S >= 2 || W == 1) ? 4 : 6; }   // doubles per block in a padded vector
#define TW_PAD(i, PS_) ((PS_) * ((i) >> 2) + ((i) & 3))
// horizon stages condensed per synchronisation in K2: twice as many on the eight-warp, one-tile shape, N = 31 .. 44, whose
// synchronisations are the costliest (config 1 53.4 -> 51.8 us per step)
__host__ __device__ constexpr int tw_kb(int W, int S) { return (W >= 8 && S == 1) ? 8 : 4; }

__host__ __device__ constexpr WLayout tw_make_layout(int N, int ms, TwShape sh)
{
    WLayout L = {};
    int o = 0;
    const int n = 2 * N, W = sh.W, ps = tw_ps(sh.W, sh.S);
    const int nb = (n + 3) / 4, NV = 4 * nb;
    L.nb = nb; L.NV = NV; L.nbuf = (W == 1) ? 1 : 2;
    L.x0 = o; o += 6; L.uprev = o; o += 2; L.misc = o; o += 24; L.spec = o; o += 12;
    L.xbar = o; o += tw_even(6 * (N + 1)); L.lin = o; o += tw_even(TG_LIN * N);
    L.rr = o; o += tw_even(3 * (N + 1)); L.sn = o; o += tw_even(N + 1); L.cs = o; o += tw_even(N + 1);
    L.q = o; o += NV; L.x = o; o += NV; L.xt = o; o += NV; L.v = o; o += NV;
    L.z = o; o += 2 * NV; L.y = o; o += 2 * NV; L.rho = o; o += 2 * NV + 2; L.rinv = o; o += 2 * NV + 2;   // box rows, then rate rows at + n
    L.dyr = o; o += NV + 2;
    L.piv = o; o += 2 * (4 * ps * nb + 16);   // two panel buffers of the sweep (up to 4 padded columns + the 4 x 4 inverse)
    int wbn = L.nbuf * tw_kb(sh.W, sh.S) * 3 * ps * nb;   // padded staging rows (TW_PAD)
    if (wbn < nb * nb * 4) wbn = nb * nb * 4;
    const int k1n = tw_even(6 * N) + 4 * tw_even(N + 2);
    if (wbn < k1n) wbn = k1n;
    L.wb = o; o += wbn;
    L.aux = L.wb; L.Xr = L.wb + tw_even(6 * N); L.Yr = L.Xr + tw_even(N + 2); L.Pr = L.Yr + tw_even(N + 2); L.vref = L.Pr + tw_even(N + 2);
    L.P = L.wb;
    L.dH = L.v; L.dsc = L.xt;
    L.red = o; o += (W > 1 ? 32 * W : 0);
    const int mse = tw_even(ms);
    L.zs = o; o += mse; L.ys = o; o += mse; L.rhos = o; o += mse; L.rinvs = o; o += mse;
    L.ls = o; o += mse; L.us = o; o += mse; L.zts = o; o += mse; L.dys = o; o += mse;
    L.tv = o; o += mse; L.gt = o; o += (ms > 0 ? 3 * NV : 0);
    L.Gs = o; o += (ms > 0 ? (ms / N) * tw_gs_off(N) : 0);
    L.total = o;
    return L;
}

// compile-time geometry of horizon NC on its shape (NC = 0: run-time horizon, everything comes from the WLayout kernel argument)
template <int NC, int W>
struct TwFix { static_assert(NC == 0 || tw_shape(NC).W == W, "a compile-time horizon runs on its tw_shape");
               static constexpr WLayout L = tw_make_layout(NC, 0, tw_shape(NC)); };
// doubles of shared memory per problem: the problems of a CTA lie side by side, each block 16-byte aligned
__host__ __device__ constexpr int tw_stride(const WLayout &L) { return tw_even(L.total); }
// offset of a FIXED-part array / a geometry constant
#define LF(f) (NC > 0 ? TwFix<NC, W>::L.f : L.f)

// Per-problem controller settings (TwCtrl, tg_device.cuh).  The ctrl instances (template flag CT) stage a problem's record in
// shared memory right after its block, at sm + tw_stride(L), so that their stride is tw_stride(L) + TW_CTRL_DBL; every other
// instance reads the handle's settings, DevCfg::ctl.  TWC(f) is the field f of whichever applies.  It names c.ctl.f directly:
// a reference to c.ctl would take the address of the __grid_constant__ parameter and can turn its loads into generic ones.
constexpr int TW_CTRL_DBL = tw_even((int)(sizeof(TwCtrl) / sizeof(double)));
#define TWC(f) (CT ? cr->f : c.ctl.f)
// thread i < 31 stages field i of the record; the caller synchronises before the record is read
__device__ __forceinline__ void tw_stage_ctrl(double *rec, const tg_ctrl_spec *src, int tid)
{
    const double *s = reinterpret_cast<const double *>(src);
    if (tid < 31) {
        double v = s[tid];
        if (tid >= 3 && tid < 11) {   // R, Rd: 0.5 (M_ij + M_ji)
            const int k = (tid - 3) & 3;
            v = 0.5 * (v + s[tid - k + (((k & 1) << 1) | (k >> 1))]);
        }
        rec[tid] = v;
    }
}

// synchronise the threads of ONE problem: a warp for W = 1, a named barrier otherwise
template <int W>
__device__ __forceinline__ void tw_sync(int bar)
{
    if constexpr (W == 1) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(bar), "n"(32 * W) : "memory");
}

__device__ __forceinline__ void tw_ld4(const double *p, double (&o)[4])
{
    const double2 *p2 = reinterpret_cast<const double2 *>(p);
    const double2 a = p2[0], b = p2[1];
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
}
__device__ __forceinline__ void tw_st4(double *p, double a, double b, double c, double d)
{
    double2 *p2 = reinterpret_cast<double2 *>(p);
    p2[0] = make_double2(a, b); p2[1] = make_double2(c, d);
}
__device__ __forceinline__ double2 tw_ld2(const double *p) { return *reinterpret_cast<const double2 *>(p); }
// Explicit shared-space accesses for the innermost loops.  The compiler re-derives the CTA's shared-memory window base
// (S2R SR_CgaCtaId + LEA, tens of cycles) next to ordinary shared accesses inside loops instead of keeping it in a register,
// which put it on the dependent chain of every sweep pivot; a 32-bit shared address computed once avoids that.
__device__ __forceinline__ unsigned tw_saddr(const double *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tw_lds4(unsigned a, double (&o)[4])
{
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%4];\n\tld.shared.v2.f64 {%2, %3}, [%4+16];" : "=d"(o[0]), "=d"(o[1]), "=d"(o[2]), "=d"(o[3]) : "r"(a));
}
__device__ __forceinline__ double tw_lds1(unsigned a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v; }
__device__ __forceinline__ void tw_sts4(unsigned a, double x0, double x1, double x2, double x3)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};\n\tst.shared.v2.f64 [%0+16], {%3, %4};" ::"r"(a), "d"(x0), "d"(x1), "d"(x2), "d"(x3) : "memory");
}
__device__ __forceinline__ void tw_sts1(unsigned a, double x0) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(x0) : "memory"); }
// 1 / x for x > 0: hardware seed (~2^-22) + one cubic step, e = 1 - x r, r <- r (1 + e + e^2): ~2^-66, three dependent FMAs
__device__ __forceinline__ double tw_rcp3(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);
    return fma(r, fma(e, e, e), r);
}
__device__ __forceinline__ void tw_st2(double *p, double a, double b) { *reinterpret_cast<double2 *>(p) = make_double2(a, b); }

// max of NRED non-negative values over the threads of a problem.  The norms only feed the termination / rho tests, so they
// are reduced in fp32 (rounded up): non-negative floats order like their bit patterns -> one REDUX per value.
template <int W, int NRED>
__device__ __forceinline__ void tw_reduce_max(double (&vals)[NRED], double *red, int tid, int bar)
{
    unsigned int u[NRED];
#pragma unroll
    for (int i = 0; i < NRED; ++i) u[i] = __reduce_max_sync(0xffffffffu, __float_as_uint(__double2float_ru(fabs(vals[i]))));
    if constexpr (W > 1) {
        unsigned int *ured = reinterpret_cast<unsigned int *>(red);
        const int lane = tid & 31, wid = tid >> 5;
        if (lane == 0)
#pragma unroll
            for (int i = 0; i < NRED; ++i) ured[wid * 16 + i] = u[i];
        tw_sync<W>(bar);
#pragma unroll
        for (int i = 0; i < NRED; ++i) {
            unsigned int v = ured[i];
#pragma unroll
            for (int w = 1; w < W; ++w) v = max(v, ured[w * 16 + i]);
            u[i] = v;
        }
        tw_sync<W>(bar);
    }
#pragma unroll
    for (int i = 0; i < NRED; ++i) vals[i] = (double)__uint_as_float(u[i]);
}

// true if `pred` holds for any thread of the problem
template <int W>
__device__ __forceinline__ bool tw_any(bool pred, double *red, int tid, int bar)
{
    bool r = __any_sync(0xffffffffu, pred);
    if constexpr (W > 1) {
        int *ired = reinterpret_cast<int *>(red);
        if ((tid & 31) == 0) ired[(tid >> 5) * 32] = r ? 1 : 0;
        tw_sync<W>(bar);
        int v = 0;
#pragma unroll
        for (int w = 0; w < W; ++w) v |= ired[w * 32];
        tw_sync<W>(bar);
        r = v != 0;
    }
    return r;
}

template <int W>
__device__ __forceinline__ double tw_reduce_sum(double v, double *red, int tid, int bar)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if constexpr (W > 1) {
        const int lane = tid & 31, wid = tid >> 5;
        if (lane == 0) red[wid * 8] = v;
        tw_sync<W>(bar);
        v = red[0];
#pragma unroll
        for (int w = 1; w < W; ++w) v += red[w * 8];
        tw_sync<W>(bar);
    }
    return v;
}

// block coordinates of a thread's S slots: slot s holds block e = s * NT + tid of the row-major lower triangle
template <int S>
struct TwMap {
    int ro[S], co[S];   // first row / column of the block (multiples of 4)
    int act[S];         // e < number of blocks (an inactive slot shadows block (0, 0) and never publishes anything)
};

template <int W, int S>
__device__ __forceinline__ TwMap<S> tw_make_map(int nb, int tid)
{
    TwMap<S> mp;
    const int nblk = nb * (nb + 1) / 2;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const int e = s * 32 * W + tid;
        int I = (int)((sqrtf(8.0f * (float)e + 1.0f) - 1.0f) * 0.5f);
        while ((I + 1) * (I + 2) / 2 <= e) ++I;
        while (I * (I + 1) / 2 > e) --I;
        const int J = e - I * (I + 1) / 2;
        int act = e < nblk ? 1 : 0, ro = act ? 4 * I : 0, co = act ? 4 * J : 0;
        asm volatile("" : "+r"(act), "+r"(ro), "+r"(co));   // kept in registers instead of being re-derived from e at every use
        mp.act[s] = act; mp.ro[s] = ro; mp.co[s] = co;
    }
    return mp;
}

// reference window by ONE warp (MPC/main.py:87-90): vref over the horizon, xs by sequential accumulation (the reference's own
// summation order), y = path(xs), phi* = atan(path'(xs)), and sin / cos(phi*).
// TG_PATH_ARC (a path that is not a graph over X, SURVEY.md 8(f) rank 3): the anchor is the path parameter s0 of the point
// closest to the vehicle, found from the guess in sp.path[0] and written back to *s_anchor (when given) so that the closed
// loop tracks it from step to step; the window advances by the arclength vref Ts (ds = vref Ts / |p'(s)|) and
// phi* = atan2(y', x') is unwrapped along the window, starting within pi of the vehicle's heading (oracle/refgen.py
// ref_window_arc states the same arithmetic).
template <int NC, int W>
__device__ __forceinline__ void tw_ref_window_warp(const DevCfg &c, const WLayout &L, double *sm, const tg_ref_spec &sp,
                                                   const double *brk, const double *coef, int t_index, int lane,
                                                   double *s_anchor = nullptr)
{
    const int N = NC > 0 ? NC : c.N;
    const double t0 = c.vref_advance ? (double)t_index * c.Ts : 0.0;
    const double vx0 = sm[LF(x0) + 3];
    for (int k = lane; k <= N; k += 32) sm[LF(vref) + k] = tg_vref_at(sp.vref_kind, sp.vref, t0 + (double)k * c.Ts, vx0);
    __syncwarp();
    if (sp.path_kind == TG_PATH_ARC) {
        if (lane == 0) {
            int lo = 0;
            double sv = tg_arc_project(sp, brk, coef, sp.path[0], sm[LF(x0)], sm[LF(x0) + 1], lo);
            double prev = sm[LF(x0) + 2];
            const double two_pi = 6.283185307179586;
            for (int k = 0; k <= N; ++k) {
                double x, y, dx, dy;
                tg_arc_eval(sp, brk, coef, sv, lo, x, y, dx, dy);
                const double raw = atan2(dy, dx);
                const double ph = raw + two_pi * rint((prev - raw) / two_pi);
                sm[LF(Xr) + k] = x; sm[LF(Yr) + k] = y; sm[LF(Pr) + k] = ph;
                prev = ph;
                if (k == 0 && s_anchor) *s_anchor = sv;
                if (k < N) sv = sv + sm[LF(vref) + k] * c.Ts / sqrt(dx * dx + dy * dy);
            }
        }
        __syncwarp();
        for (int k = lane; k <= N; k += 32) {
            double s_, c_;
            TG_SINCOS(sm[LF(Pr) + k], s_, c_);
            sm[LF(sn) + k] = s_; sm[LF(cs) + k] = c_;
        }
        return;
    }
    if (lane == 0) {
        double xs = sm[LF(x0)];
        sm[LF(Xr)] = xs;
        for (int k = 0; k < N; ++k) { xs = xs + sm[LF(vref) + k] * c.Ts; sm[LF(Xr) + k + 1] = xs; }   // :59-61
    }
    __syncwarp();
    for (int k = lane; k <= N; k += 32) {
        double y, dy, s_, c_;
        tg_path_at(sp, brk, coef, sm[LF(Xr) + k], y, dy);
        const double ph = tg_atan(dy);   // :66
        TG_SINCOS(ph, s_, c_);
        sm[LF(Yr) + k] = y; sm[LF(Pr) + k] = ph; sm[LF(sn) + k] = s_; sm[LF(cs) + k] = c_;
    }
}

// ---------------------------------------------------------------------------------------------------------------- K2
// H = sum_k W_k' W_k on the tile (W rows carry sqrt(2 q)); optionally q and the state-bound rows.  Thread j owns column j of G
// (n <= 32 W on every shape).
template <int W, int S, int NC, bool HS, bool CT = false>
__device__ __forceinline__ void tw_condense(const DevCfg &c, const WLayout &L, double *sm, const TwMap<S> &mp, double (&a)[S][4][4],
                                            bool first, int tid, int bar, const TwCtrl *cr = nullptr)
{
    constexpr int KB = tw_kb(W, S);   // stages per synchronisation (the layout reserves the staging rows: tw_make_layout)
    constexpr int PS = tw_ps(W, S);
    const int NVP = PS * LF(nb);                                  // padded length of a staging row
    constexpr int NT = 32 * W;
    const int N = NC > 0 ? NC : c.N, n = 2 * N, NV = LF(NV), ns = HS ? c.ns : 0, ms_ = HS ? c.ms : 0;   // HS: the instance carries the code of the state-bound rows
    const double *lin = sm + LF(lin), *sn = sm + LF(sn), *cs = sm + LF(cs), *rr = sm + LF(rr);
    double *wbuf = sm + LF(wb), *Gs = sm + L.Gs;
    const double sqp = sqrt(2.0 * TWC(q_phi)), sqv = sqrt(2.0 * TWC(q_vx));
    double G[6], qacc = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) G[i] = 0.0;
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) a[s][r][cc] = 0.0;
    if (NV > n) {   // pad columns of the staging rows (and of the state rows) must read as zero
        const int np = (NV - n) > 0 ? NV - n : 1;
        for (int i = tid; i < LF(nbuf) * KB * 3 * np; i += NT) wbuf[(i / np) * NVP + TW_PAD(n + i % np, PS)] = 0.0;
        tw_sync<W>(bar);
    }
    if (first)   // zero pads of the packed state rows (len_k - 2 (k + 1) = 0 or 2 entries per row)
        for (int i = tid; i < ms_; i += NT) {
            const int k = i / (ns > 0 ? ns : 1), si = i - k * ns;
            double *row = Gs + ns * tw_gs_off(k) + si * tw_gs_len(k);
            for (int j = 2 * (k + 1); j < tw_gs_len(k); ++j) row[j] = 0.0;
        }
    // compile-time horizon that is a multiple of KB: the stage loops below have a constant trip count and are unrolled, so that
    // the loads of a stage are issued under the arithmetic of the previous one
    constexpr bool FULLKB = NC > 0 && NC % KB == 0;
    constexpr int UNR = FULLKB ? KB : 1;
    // unrolling the rounds as well measured 1 % slower (more code, no extra overlap)
#pragma unroll 1
    for (int k0 = 0; k0 < N; k0 += KB) {
        const int kb = FULLKB ? KB : ((N - k0 < KB) ? N - k0 : KB);
        double *wblk = wbuf + ((LF(nbuf) == 2) ? ((k0 / KB) & 1) * KB * 3 * NVP : 0);
        const int j = tid;
        if (j < n && k0 + kb > (tid & ~31) / 2) {   // nothing to do before the first column of this warp is born
            const int c1 = j & 1, jb = j >> 1, pj = TW_PAD(j, PS);
#pragma unroll UNR
            for (int s_i = 0; s_i < kb; ++s_i) {
                const int k = k0 + s_i;
                const double *r = lin + TG_LIN * k;
                double A_[16];
#pragma unroll
                for (int i = 0; i < 8; ++i) { const double2 t = tw_ld2(r + 2 * i); A_[2 * i] = t.x; A_[2 * i + 1] = t.y; }
                // G_{k+1} = A_k G_k; the column is born at stage jb as a column of B_k (it holds zeros before, A 0 = 0)
                const double bm = (jb == k) ? 1.0 : 0.0;
                const double b3 = r[16 + c1], b4 = c1 ? r[18] : 0.0, b5 = c1 ? r[19] : 0.0;
                const double n0 = G[0] + A_[0] * G[2] + A_[1] * G[3] + A_[2] * G[4];
                const double n1 = G[1] + A_[3] * G[2] + A_[4] * G[3] + A_[5] * G[4];
                const double n2 = G[2] + A_[6] * G[5];
                const double n3 = fma(bm, b3, A_[7] * G[3] + A_[8] * G[4] + A_[9] * G[5]);
                const double n4 = fma(bm, b4, A_[10] * G[3] + A_[11] * G[4] + A_[12] * G[5]);
                const double n5 = fma(bm, b5, A_[13] * G[3] + A_[14] * G[4] + A_[15] * G[5]);
                G[0] = n0; G[1] = n1; G[2] = n2; G[3] = n3; G[4] = n4; G[5] = n5;
                const int kk = k + 1;
                const double wc = sn[kk] * n0 - cs[kk] * n1, wp = sqp * n2, wv = sqv * n3;   // sn, cs carry sqrt(2 q_c)
                double *wrow = wblk + s_i * 3 * NVP;
                wrow[pj] = wc; wrow[NVP + pj] = wp; wrow[2 * NVP + pj] = wv;
                if (first) {
                    qacc = fma(rr[3 * kk], wc, fma(rr[3 * kk + 1], wp, fma(rr[3 * kk + 2], wv, qacc)));
                    if (jb <= k)
                        for (int si = 0; si < ns; ++si) {
                            const int sx = c.sidx[si];
                            const double gv = (sx == 0) ? n0 : (sx == 1) ? n1 : (sx == 2) ? n2 : (sx == 3) ? n3 : (sx == 4) ? n4 : n5;
                            Gs[ns * tw_gs_off(k) + si * tw_gs_len(k) + j] = gv;
                        }
                }
            }
        } else if (j < n) {   // not born in this block of stages: its W entries are zero
            for (int s_i = 0; s_i < kb; ++s_i) {
                double *wrow = wblk + s_i * 3 * NVP;
                wrow[TW_PAD(j, PS)] = 0.0; wrow[NVP + TW_PAD(j, PS)] = 0.0; wrow[2 * NVP + TW_PAD(j, PS)] = 0.0;
            }
        }
        tw_sync<W>(bar);
#pragma unroll UNR
        for (int s_i = 0; s_i < kb; ++s_i) {
            const int lim = 2 * (k0 + s_i) + 2;   // columns born so far
            const double *wrow = wblk + s_i * 3 * NVP;
#pragma unroll
            for (int s = 0; s < S; ++s) {
                if (mp.act[s] && mp.ro[s] < lim) {   // rank-3 update of the block: 3 x (4 + 4) operands, 48 FMAs (co <= ro)
#pragma unroll
                    for (int rI = 0; rI < 3; ++rI) {
                        double rw[4], cw[4];
                        tw_ld4(wrow + rI * NVP + (mp.ro[s] >> 2) * PS, rw);   // TW_PAD of a multiple of 4
                        tw_ld4(wrow + rI * NVP + (mp.co[s] >> 2) * PS, cw);
#pragma unroll
                        for (int r = 0; r < 4; ++r)
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc) a[s][r][cc] = fma(rw[r], cw[cc], a[s][r][cc]);
                    }
                }
            }
        }
        if (LF(nbuf) == 1) tw_sync<W>(bar);   // single staging buffer: the next block of stages overwrites it
    }
    if (first) {
#pragma unroll
        for (int p = 0; p < 1; ++p) {   // a one-trip loop only because it keeps the generated code unchanged
            const int j = tid;
            if (j < n) {
                const int cc = j & 1;
                sm[LF(q) + j] = qacc + 2.0 * (TWC(Rs[cc * 2]) * sm[LF(uprev)] + TWC(Rs[cc * 2 + 1]) * sm[LF(uprev) + 1]);
            }
        }
    }
    // input and input-rate penalties (mpc_6stati.py:238-245) in dU: 2 Rs + (4 | 2) Rds on a stage's own 2x2 block, -2 Rds
    // between neighbouring stages.  A 4x4 tile block holds two stages, so the touched entries are static.
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const int st0 = mp.ro[s] >> 1;   // first stage of the block's rows
        if (mp.ro[s] == mp.co[s]) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const int sr = r >> 1, sc = cc >> 1, ar = r & 1, ac = cc & 1;
                    const int str = st0 + sr, stc = st0 + sc;
                    if (str < N && stc < N) {
                        double add;
                        if (sr == sc) add = 2.0 * TWC(Rs[ar * 2 + ac]) + ((str < N - 1) ? 4.0 : 2.0) * TWC(Rds[ar * 2 + ac]);
                        else add = -2.0 * TWC(Rds[ar * 2 + ac]);
                        a[s][r][cc] += add;
                    }
                }
        } else if (mp.ro[s] == mp.co[s] + 4) {   // rows: stages st0, st0 + 1; columns: stages st0 - 2, st0 - 1
            if (st0 < N) {
#pragma unroll
                for (int r = 0; r < 2; ++r)
#pragma unroll
                    for (int cc = 2; cc < 4; ++cc) a[s][r][cc] += -2.0 * TWC(Rds[(r & 1) * 2 + (cc & 1)]);
            }
        }
    }
}

// K = H + sigma I + A' diag(rho) A on the tile (rho vectors in shared memory)
template <int W, int S, int NC, bool HS>
__device__ __forceinline__ void tw_build_K(const DevCfg &c, const WLayout &L, const double *sm, const TwMap<S> &mp, double (&a)[S][4][4])
{
    const int n = NC > 0 ? 2 * NC : c.n, NV = LF(NV);
    const double *rho_b = sm + LF(rho), *rho_r = sm + LF(rho) + n, *rho_s = sm + L.rhos;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const int R0 = mp.ro[s];
        if (R0 == mp.co[s]) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = R0 + r;
                if (i < n) a[s][r][r] += c.sigma + rho_b[i] + rho_r[i] + ((i + 2 < n) ? rho_r[i + 2] : 0.0);
            }
            if (R0 + 2 < n) { const double t = rho_r[R0 + 2]; a[s][2][0] -= t; a[s][0][2] -= t; }
            if (R0 + 3 < n) { const double t = rho_r[R0 + 3]; a[s][3][1] -= t; a[s][1][3] -= t; }
        } else if (R0 == mp.co[s] + 4) {   // (row R0 + r, column R0 - 2 + r), r = 0, 1
            if (R0 < n) a[s][0][2] -= rho_r[R0];
            if (R0 + 1 < n) a[s][1][3] -= rho_r[R0 + 1];
        }
    }
    const double *Gs = sm + L.Gs;
    const int ns = HS ? c.ns : 0, N = NC > 0 ? NC : c.N;
    if (ns > 0)
        for (int k = 0; k < N; ++k) {
            const int len = tw_gs_len(k);
            for (int si = 0; si < ns; ++si) {
                const double rs = rho_s[k * ns + si];
                const double *row = Gs + ns * tw_gs_off(k) + si * len;
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    if (mp.ro[s] < len) {   // the row vanishes beyond column 2 (k + 1) <= len (co <= ro)
                        double gr[4], gc[4];
                        tw_ld4(row + mp.ro[s], gr);
                        tw_ld4(row + mp.co[s], gc);
#pragma unroll
                        for (int r = 0; r < 4; ++r) {
                            const double t = gr[r] * rs;
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc) a[s][r][cc] = fma(t, gc[cc], a[s][r][cc]);
                        }
                    }
                }
            }
        }
}

// ------------------------------------------------------------------------------------------- state-row products (ms > 0)
// Thread geometry of the two products with the packed state rows, chosen once per step: NG threads (a power of two, lanes of
// one warp) share a column pair in G_s' v, TPR threads share a row in G_s x.
struct TwGsGeo { int ng, lg_ng, tpr, lg_tpr; };
template <int W>
__device__ __forceinline__ TwGsGeo tw_gs_geo(int N, int ms)
{
    constexpr int NT = 32 * W;
    TwGsGeo g; g.ng = 1; g.lg_ng = 0; g.tpr = 1; g.lg_tpr = 0;
    while (g.ng * 2 * N <= NT && g.ng < 8) { g.ng *= 2; g.lg_ng += 1; }
    while (g.tpr * 2 * ms <= NT && g.tpr < 4) { g.tpr *= 2; g.lg_tpr += 1; }
    return g;
}
// gt[v NV + j] = sum_i Gs[i][j] vec_v[i] for v < NVEC and every column j < n, by all threads of the problem: thread (jp, g)
// sums the stages k = jp + g, jp + g + NG, ... (rows of earlier stages vanish in column pair jp), then the NG partials are
// folded with shuffles.  The caller synchronises before reading gt.  (32-bit shared addresses and explicit ld.shared: with
// generic pointers every access of these loops carried 64-bit address arithmetic, ~30 instructions per row.)
__device__ __forceinline__ double2 tw_lds2(unsigned a) { double2 v; asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a)); return v; }
template <int W, int NVEC>
__device__ __forceinline__ void tw_gs_tmul(const WLayout &L, double *sm, const TwGsGeo &geo, int N, int ns, int NV,
                                           const double *const (&vec)[NVEC], int tid)
{
    const unsigned gs_a = tw_saddr(sm + L.Gs);
    unsigned vec_a[NVEC];
#pragma unroll
    for (int v = 0; v < NVEC; ++v) vec_a[v] = tw_saddr(vec[v]);
    double *gt = sm + L.gt;
    const int jp = tid >> geo.lg_ng, g = tid & (geo.ng - 1);
    double a0[NVEC], a1[NVEC];
#pragma unroll
    for (int v = 0; v < NVEC; ++v) { a0[v] = 0.0; a1[v] = 0.0; }
    if (jp < N) {
        for (int k = jp + g; k < N; k += geo.ng) {
            const unsigned len8 = 8u * (unsigned)tw_gs_len(k);
            unsigned ra = gs_a + 8u * (unsigned)(ns * tw_gs_off(k) + 2 * jp), va = 8u * (unsigned)(k * ns);
            for (int si = 0; si < ns; ++si, ra += len8, va += 8u) {
                const double2 g2 = tw_lds2(ra);
#pragma unroll
                for (int v = 0; v < NVEC; ++v) {
                    const double t = tw_lds1(vec_a[v] + va);
                    a0[v] = fma(g2.x, t, a0[v]); a1[v] = fma(g2.y, t, a1[v]);
                }
            }
        }
    }
    for (int o = geo.ng >> 1; o > 0; o >>= 1)
#pragma unroll
        for (int v = 0; v < NVEC; ++v) { a0[v] += __shfl_xor_sync(0xffffffffu, a0[v], o); a1[v] += __shfl_xor_sync(0xffffffffu, a1[v], o); }
    if (jp < N && g == 0)
#pragma unroll
        for (int v = 0; v < NVEC; ++v) tw_st2(gt + v * NV + 2 * jp, a0[v], a1[v]);
}
// (G_s x)_r for the row r = r0 + (tid >> lg_tpr) (0 if r >= ms), summed over the TPR threads of the row; every thread of the
// problem must call it (shuffles)
template <int W>
__device__ __forceinline__ double tw_gs_row_dot(const WLayout &L, const double *sm, const TwGsGeo &geo, int ns, int ms, const double *x,
                                                int r, int tid)
{
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (r < ms) {
        const int k = r / ns, si = r - k * ns, h = tid & (geo.tpr - 1);
        const unsigned st = 16u * (unsigned)geo.tpr;                 // bytes between the column pairs of one thread
        unsigned ga = tw_saddr(sm + L.Gs) + 8u * (unsigned)(ns * tw_gs_off(k) + si * tw_gs_len(k)) + 16u * (unsigned)h;
        unsigned xa = tw_saddr(x) + 16u * (unsigned)h;
        int d = h;
        for (; d + geo.tpr <= k; d += 2 * geo.tpr, ga += 2u * st, xa += 2u * st) {   // column pairs d and d + TPR (both <= k)
            const double2 g_a = tw_lds2(ga), x_a = tw_lds2(xa), g_b = tw_lds2(ga + st), x_b = tw_lds2(xa + st);
            s0 = fma(g_a.x, x_a.x, s0); s1 = fma(g_a.y, x_a.y, s1); s2 = fma(g_b.x, x_b.x, s2); s3 = fma(g_b.y, x_b.y, s3);
        }
        if (d <= k) { const double2 g_a = tw_lds2(ga), x_a = tw_lds2(xa); s0 = fma(g_a.x, x_a.x, s0); s1 = fma(g_a.y, x_a.y, s1); }
    }
    double acc = (s0 + s1) + (s2 + s3);
    for (int o = geo.tpr >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return acc;
}

// a <- D a D with the diagonal D in dsc: the Jacobi scaling of the tile before the sweeps and the un-scaling after them
template <int S>
__device__ __forceinline__ void tw_scale_tile(const double *dsc, const TwMap<S> &mp, double (&a)[S][4][4])
{
#pragma unroll
    for (int s = 0; s < S; ++s) {
        double dr[4], dc[4];
        tw_ld4(dsc + mp.ro[s], dr);
        tw_ld4(dsc + mp.co[s], dc);
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) a[s][r][cc] *= dr[r] * dc[cc];
    }
}
// K^ = D K D with D = diag(K)^-1/2 (zero in the pad rows), published in dsc for the un-scaling K^-1 = D K^^-1 D: the unpivoted
// sweep is only as accurate as cond(K), and K inherits the variable scaling of H
template <int W, int S>
__device__ __forceinline__ void tw_jacobi_scale(double *dsc, const TwMap<S> &mp, double (&a)[S][4][4], int n, int bar)
{
#pragma unroll
    for (int s = 0; s < S; ++s)
        if (mp.act[s] && mp.ro[s] == mp.co[s])
            tw_st4(dsc + mp.ro[s], (mp.ro[s] + 0 < n) ? rsqrt(a[s][0][0]) : 0.0, (mp.ro[s] + 1 < n) ? rsqrt(a[s][1][1]) : 0.0,
                   (mp.ro[s] + 2 < n) ? rsqrt(a[s][2][2]) : 0.0, (mp.ro[s] + 3 < n) ? rsqrt(a[s][3][3]) : 0.0);
    tw_sync<W>(bar);
    tw_scale_tile<S>(dsc, mp, a);
}

// In-register inversion of the SPD tile by n symmetric sweeps (SWP_k: a_kk <- -1/a_kk, a_ik <- a_ik/a_kk,
// a_ij <- a_ij - a_ik a_kj / a_kk); on return a = -K^-1 (lower-triangle blocks).
// Step k = 4 K + kr: the threads holding block row K (their row kr) and block column K (their column kr) publish row k of
// the matrix (= column k by symmetry) with v[k] = a_kk - 1, the reciprocal pivot beside it; everybody then does one rank-1
// update of each slot with w_i = v_i / a_kk (w = 1 - 1/a_kk on the pivot row) and the pivot is repaired in place.
// K is Jacobi-scaled first and un-scaled afterwards.
template <int W, int S, int NC>
__device__ __forceinline__ void tw_sweep_invert_scalar(const DevCfg &c, const WLayout &L, double *sm, const TwMap<S> &mp,
                                                       double (&a)[S][4][4], int bar)
{
    const int n = NC > 0 ? 2 * NC : c.n, NV = LF(NV), nb = LF(nb);
    double *vb = sm + LF(piv), *dsc = sm + LF(dsc);
    tw_jacobi_scale<W, S>(dsc, mp, a, n, bar);
    // the reciprocal of pivot k+1 is started as soon as that entry has been updated in step k, so that its latency overlaps
    // the rest of the rank-1 update
    double rp_next = 0.0;
#pragma unroll
    for (int s = 0; s < S; ++s)
        if (mp.act[s] && mp.ro[s] == 0 && mp.co[s] == 0) rp_next = tw_rcp3(a[s][0][0]);
    // shared-space addresses of this thread's operands in the two pivot-row buffers (buffer = pivot parity)
    constexpr unsigned PS = tw_ps(W, S);
    const unsigned NVP = PS * (unsigned)nb;   // padded pivot rows (TW_PAD)
    const unsigned vb_a = tw_saddr(vb), stride_a = (NVP + 2u) * 8u;
    unsigned ro_a[S], co_a[S];
#pragma unroll
    for (int s = 0; s < S; ++s) { ro_a[s] = vb_a + 2u * PS * (unsigned)mp.ro[s]; co_a[s] = vb_a + 2u * PS * (unsigned)mp.co[s]; }
#pragma unroll 1
    for (int K = 0; K < nb; ++K) {
        const int K4 = 4 * K;
#pragma unroll
        for (int kr = 0; kr < 4; ++kr) {
            const int k = K4 + kr;
            if (k < n) {   // uniform
                const unsigned boff = (kr & 1) ? stride_a : 0u;   // k & 1 == kr & 1 (K4 is even)
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    if (mp.act[s]) {
                        if (mp.ro[s] == K4) {          // block row K: row kr of the block is a_{k, co..co+3}
                            tw_sts4(co_a[s] + boff, a[s][kr][0], a[s][kr][1], a[s][kr][2], a[s][kr][3]);
                            if (mp.co[s] == K4) { tw_sts1(vb_a + boff + 8u * PS * (unsigned)K + 8u * (unsigned)kr, a[s][kr][kr] - 1.0); tw_sts1(vb_a + boff + 8u * NVP, rp_next); }
                        } else if (mp.co[s] == K4) {   // block column K below the diagonal: column kr is a_{ro..ro+3, k}
                            tw_sts4(ro_a[s] + boff, a[s][0][kr], a[s][1][kr], a[s][2][kr], a[s][3][kr]);
                        }
                    }
                }
                tw_sync<W>(bar);
                const double p = tw_lds1(vb_a + boff + 8u * NVP);
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    double vr[4], vc[4];
                    tw_lds4(ro_a[s] + boff, vr);
                    tw_lds4(co_a[s] + boff, vc);
#pragma unroll
                    for (int r = 0; r < 4; ++r) vr[r] *= p;
                    if (mp.ro[s] == K4) vr[kr] = 1.0 - p;
                    {   // next pivot first
                        const int nx = (kr + 1) & 3;                   // static after unrolling
                        const int nK4 = (kr == 3) ? K4 + 4 : K4;
                        if (mp.act[s] && mp.ro[s] == nK4 && mp.co[s] == nK4) rp_next = tw_rcp3(fma(-vr[nx], vc[nx], a[s][nx][nx]));   // K is SPD: pivots > 0
                    }
#pragma unroll
                    for (int r = 0; r < 4; ++r)
#pragma unroll
                        for (int cc = 0; cc < 4; ++cc) a[s][r][cc] = fma(-vr[r], vc[cc], a[s][r][cc]);
                    if (mp.ro[s] == K4 && mp.co[s] == K4) a[s][kr][kr] = -p;
                }
            }
        }
    }
    tw_scale_tile<S>(dsc, mp, a);   // K^-1 = D K^^-1 D
    tw_sync<W>(bar);
}

// BLOCKED sweep: the pivots of a 4 x 4 diagonal block in two groups of two (two synchronisations per block instead of four).
// Sweeping the index set P of a group:
//     A_PP <- -D^-1 (D = A_PP),   A_iP <- A_iP D^-1,   A_ij <- A_ij - A_iP D^-1 A_Pj.
// The panel V = A_.P (n x 2) is published column-wise (VT[m][i] = A_{i, P_m}; block column K below the diagonal, block row K
// left of it by symmetry), with D - I in the rows of P itself, and the owner of the diagonal block publishes D^-1 (inverted in
// its registers).  With that patch every block (I, J) -- panel blocks included -- does the same update
//     A_IJ <- A_IJ - (V_I D^-1) V_J',
// and only the diagonal block is repaired afterwards (<- -D^-1).  The panel and the inverse of the next group are published
// right after a thread's update of the current one, into the other buffer.
// inverse of the 2 x 2 SPD block a[o .. o+1][o .. o+1] (closed form)
__device__ __forceinline__ void tw_inv_spd(const double (&a)[4][4], int o, double (&di)[2][2])
{
    const double a00 = o ? a[2][2] : a[0][0], a01 = o ? a[3][2] : a[1][0], a11 = o ? a[3][3] : a[1][1];
    const double r = tw_rcp3(fma(a00, a11, -a01 * a01));   // SPD: det > 0
    di[0][0] = a11 * r; di[1][1] = a00 * r; di[0][1] = -a01 * r; di[1][0] = di[0][1];
}

template <int W, int S, int NC>
__device__ __forceinline__ void tw_sweep_invert(const DevCfg &c, const WLayout &L, double *sm, const TwMap<S> &mp,
                                                double (&a)[S][4][4], int bar)
{
    // measured (DESIGN.md section 8, profiles/r02_sweep_variants.txt): with one or two warps per problem the scalar sweep is fastest
    // (the blocked forms add fp64 work that the 7-8 problems of an SM have to share the fp64 pipe for); with four or eight warps
    // per problem the synchronisation is costlier and the 2-pivot form wins (config 1: 52.0 -> 49.6 us per step; N = 30: +2 %);
    // the 4-pivot form loses everywhere.  Two tiles per thread (N > 44) keep the scalar form.
    if constexpr (!(W >= 4 && S == 1)) {
        tw_sweep_invert_scalar<W, S, NC>(c, L, sm, mp, a, bar);
        return;
    } else {
    constexpr int PB = 2;   // pivots per group
    const int n = NC > 0 ? 2 * NC : c.n, NV = LF(NV), nb = LF(nb);
    double *vb = sm + LF(piv), *dsc = sm + LF(dsc);
    tw_jacobi_scale<W, S>(dsc, mp, a, n, bar);
#pragma unroll
    for (int s = 0; s < S; ++s)
        if (mp.ro[s] == mp.co[s])   // pad rows (odd horizons) become identity rows: they pass through the block inverse unchanged
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (mp.ro[s] + r >= n) a[s][r][r] = 1.0;
    // panel buffer of one pivot group: PB columns of NV (VT[m][i] = A_{i, P_m}) + the PB x PB inverse; two buffers, alternating
    constexpr unsigned PS = tw_ps(W, S);
    const unsigned NVP = PS * (unsigned)nb;   // padded panel columns (TW_PAD)
    const unsigned vb_a = tw_saddr(vb), stride_a = ((unsigned)PB * NVP + (unsigned)(PB * PB)) * 8u, nv8 = NVP * 8u, dinv_o = (unsigned)PB * nv8;
    unsigned ro_a[S], co_a[S];
#pragma unroll
    for (int s = 0; s < S; ++s) { ro_a[s] = vb_a + 2u * PS * (unsigned)mp.ro[s]; co_a[s] = vb_a + 2u * PS * (unsigned)mp.co[s]; }
    // publish the panel of pivot group h (compile-time) of block K4 into the buffer at boff
    auto publish = [&](int K4, auto h_, unsigned boff) {
        constexpr int h = decltype(h_)::value, o = h * PB;
#pragma unroll
        for (int s = 0; s < S; ++s) {
            if (mp.act[s]) {
                if (mp.ro[s] == K4) {
                    if (mp.co[s] == K4) {   // diagonal block: D - I in the pivot rows, D^-1 beside the panel
                        double di[PB][PB];
                        tw_inv_spd(a[s], o, di);
#pragma unroll
                        for (int m = 0; m < PB; ++m) {
                            tw_sts4(ro_a[s] + boff + (unsigned)m * nv8, a[s][0][o + m] - (o + m == 0 ? 1.0 : 0.0), a[s][1][o + m] - (o + m == 1 ? 1.0 : 0.0),
                                    a[s][2][o + m] - (o + m == 2 ? 1.0 : 0.0), a[s][3][o + m] - (o + m == 3 ? 1.0 : 0.0));
#pragma unroll
                            for (int q = 0; q < PB; ++q) tw_sts1(vb_a + boff + dinv_o + 8u * (unsigned)(m * PB + q), di[m][q]);
                        }
                    } else {                // block row K left of the diagonal: V_{j, m} = a[o + m][j]
#pragma unroll
                        for (int m = 0; m < PB; ++m) tw_sts4(co_a[s] + boff + (unsigned)m * nv8, a[s][o + m][0], a[s][o + m][1], a[s][o + m][2], a[s][o + m][3]);
                    }
                } else if (mp.co[s] == K4) {   // block column K below the diagonal: V_{i, m} = a[i][o + m]
#pragma unroll
                    for (int m = 0; m < PB; ++m) tw_sts4(ro_a[s] + boff + (unsigned)m * nv8, a[s][0][o + m], a[s][1][o + m], a[s][2][o + m], a[s][3][o + m]);
                }
            }
        }
    };
    // one pivot group: A_IJ <- A_IJ - (V_I D^-1) V_J' for every block, then the pivot sub-block of the diagonal block <- -D^-1
    auto update = [&](int K4, auto h_, unsigned boff) {
        constexpr int h = decltype(h_)::value, o = h * PB;
        double di[PB][PB];
#pragma unroll
        for (int m = 0; m < PB; ++m)
#pragma unroll
            for (int q = 0; q < PB; ++q) di[m][q] = tw_lds1(vb_a + boff + dinv_o + 8u * (unsigned)(m * PB + q));
#pragma unroll
        for (int s = 0; s < S; ++s) {
            double vi[PB][4];
#pragma unroll
            for (int m = 0; m < PB; ++m) tw_lds4(ro_a[s] + boff + (unsigned)m * nv8, vi[m]);
#pragma unroll
            for (int q = 0; q < PB; ++q) {
                double vj[4], w[4];
                tw_lds4(co_a[s] + boff + (unsigned)q * nv8, vj);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    double t = vi[0][r] * di[0][q];
#pragma unroll
                    for (int m = 1; m < PB; ++m) t = fma(vi[m][r], di[m][q], t);
                    w[r] = t;
                }
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int cc = 0; cc < 4; ++cc) a[s][r][cc] = fma(-w[r], vj[cc], a[s][r][cc]);
            }
            if (mp.ro[s] == K4 && mp.co[s] == K4) {
#pragma unroll
                for (int m = 0; m < PB; ++m)
#pragma unroll
                    for (int q = 0; q < PB; ++q) a[s][o + m][o + q] = -di[m][q];
            }
        }
    };
    using std::integral_constant;
    publish(0, integral_constant<int, 0>(), 0u);
#pragma unroll 1
    for (int K = 0; K < nb; ++K) {
        const int K4 = 4 * K;
        // the buffer alternates with every group: group h of a block uses buffer h
        tw_sync<W>(bar);
        update(K4, integral_constant<int, 0>(), 0u);
        publish(K4, integral_constant<int, 1>(), stride_a);
        tw_sync<W>(bar);
        update(K4, integral_constant<int, 1>(), stride_a);
        if (K + 1 < nb) publish(K4 + 4, integral_constant<int, 0>(), 0u);
    }
    tw_scale_tile<S>(dsc, mp, a);   // K^-1 = D K^^-1 D
    tw_sync<W>(bar);
    }
}

// block partials of x~ = K^-1 v (a = -K^-1): P[(seg * nb + other) * 4 + r]; summed per entry by tw_matvec_sum
template <int W, int S, int NC>
__device__ __forceinline__ void tw_matvec_partials(const WLayout &L, double *sm, const TwMap<S> &mp, const double (&a)[S][4][4])
{
    const int nb = LF(nb);
    const double *v = sm + LF(v);
    double *P = sm + LF(P);
#pragma unroll
    for (int s = 0; s < S; ++s) {
        double vi[4], vj[4], pi_[4], pj[4];
        tw_ld4(v + mp.ro[s], vi);
        tw_ld4(v + mp.co[s], vj);
#pragma unroll
        for (int r = 0; r < 4; ++r) pi_[r] = a[s][r][0] * vj[0] + a[s][r][1] * vj[1] + a[s][r][2] * vj[2] + a[s][r][3] * vj[3];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) pj[cc] = a[s][0][cc] * vi[0] + a[s][1][cc] * vi[1] + a[s][2][cc] * vi[2] + a[s][3][cc] * vi[3];
        if (mp.act[s]) {
            const int I = mp.ro[s] >> 2, J = mp.co[s] >> 2;
            tw_st4(P + (I * nb + J) * 4, pi_[0], pi_[1], pi_[2], pi_[3]);
            if (I != J) tw_st4(P + (J * nb + I) * 4, pj[0], pj[1], pj[2], pj[3]);
        }
    }
}
// entries 2t, 2t+1 of x~ (t = stage)
template <int W, int NC>
__device__ __forceinline__ double2 tw_matvec_sum(const WLayout &L, const double *sm, int t)
{
    const int nb = LF(nb);
    const double *P = sm + LF(P) + ((t >> 1) * nb) * 4 + 2 * (t & 1);
    double s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int o = 0; o < nb; ++o) { const double2 p = tw_ld2(P + 4 * o); s0 += p.x; s1 += p.y; }
    return make_double2(-s0, -s1);
}

// ------------------------------------------------------------------------------------------------------------ the step
// On entry shared memory holds x0, uprev and -- unless `fx` is given, in which case the body builds it from the scenario in
// sm[LF(spec)] -- the reference window (Xr, Yr, Pr, vref); if `warm`, the warm-start dU in sm[LF(x)] and duals in sm[LF(y)].
// On exit sm[LF(xt)] holds dU*, sm[LF(y)] the duals, and the result is returned to every thread.  CT: the weights and bounds
// come from the problem's record `cr` (TwCtrl, in shared memory) instead of DevCfg; nothing else changes.
//
// Solver: the OSQP iteration on the condensed problem with per-row rho_i = rho / max_j(a_ij^2 / H_jj).  A solve that starts
// with every dual at zero (cold start, or a warm start from a solution with no active row: 99.9 % of the steps of the
// dataset workloads) first runs in "free" mode: rho = TW_FREE_RHO, alpha = 1.  With no row active the iteration map is then
// x <- x - K^-1 (H x + q) with K = H + O(1e-6), so two iterations land on the unconstrained optimum to ~1e-12 -- the EXACT
// optimum of the QP whenever it satisfies every row, which the standard residual test then certifies (r_prim = 0).  As soon
// as a row clamps, the solve falls back to the standard settings (rho, alpha) and refactors.
template <int W, int S, int NC, bool HS, bool CT = false>
__device__ StepResult tw_step_body(const DevCfg &c, const WLayout &L, double *sm, const TwMap<S> &mp, bool warm, bool warm_free,
                                   const StepTaps &tap, const FusedCtx *fx, int tid, int bar, const TwCtrl *cr = nullptr)
{
    constexpr int NT = 32 * W;
    const int N = NC > 0 ? NC : c.N, n = 2 * N, NV = LF(NV), ms = HS ? c.ms : 0, ns = HS ? c.ns : 0;   // HS: the instance carries the code of the state-bound rows
    StepResult res;
    res.status = TG_STATUS_NAN; res.iters = 0; res.objective = 0.0; res.free_end = false;

    double *misc = sm + LF(misc), *xbar = sm + LF(xbar), *lin = sm + LF(lin);
    double *sn = sm + LF(sn), *cs = sm + LF(cs), *rr = sm + LF(rr);
    double *q = sm + LF(q), *x = sm + LF(x), *xt = sm + LF(xt), *v = sm + LF(v);
    double *z = sm + LF(z), *y = sm + LF(y), *rho = sm + LF(rho), *rinv = sm + LF(rinv), *dyr = sm + LF(dyr);
    double *zs = sm + L.zs, *ys = sm + L.ys, *rhos = sm + L.rhos, *rinvs = sm + L.rinvs;     // state rows (tail of the layout)
    double *ls = sm + L.ls, *us = sm + L.us, *zts = sm + L.zts, *dys = sm + L.dys, *Gs = sm + L.Gs, *red = sm + LF(red);
    double *tv = sm + L.tv, *gt = sm + L.gt;
    const TwGsGeo geo = tw_gs_geo<W>(N, ms);
    TG_TICK_DECL;

    // ---------------- K1a: reference window + sensor noise of the row (closed loop), nominal rollout (mpc_6stati.py:167-172)
    const int roll_warp = 0, ref_warp = (W > 1) ? 1 : 0, noise_warp = (W > 2) ? 2 : ref_warp;
    const int wid = tid >> 5, lane = tid & 31;
    if (wid == ref_warp) {
        if (fx) {
            const tg_ref_spec &sp = *reinterpret_cast<const tg_ref_spec *>(sm + LF(spec));
            tw_ref_window_warp<NC, W>(c, L, sm, sp, fx->brk, fx->coef, fx->t_index, lane, sm + LF(spec) + 2);   // + 2: sp.path[0]
        } else {
            for (int i = lane; i <= N; i += 32) { double s_, c_; TG_SINCOS(sm[LF(Pr) + i], s_, c_); sn[i] = s_; cs[i] = c_; }
        }
    }
    if (wid == noise_warp && fx && fx->noisy_row && lane < 3) {   // never fed back
        uint32_t r4[4];
        tg_philox4x32_10((uint32_t)fx->t_index, (uint32_t)(lane >> 1), 0u, 0u, (uint32_t)fx->seed, (uint32_t)(fx->seed >> 32), r4);
        double n0, n1;
        tg_box_muller(r4[(lane & 1) * 2], r4[(lane & 1) * 2 + 1], n0, n1);
        fx->noisy_row[2 * lane] = sm[LF(x0) + 2 * lane] + c.noise_std[2 * lane] * n0;
        fx->noisy_row[2 * lane + 1] = sm[LF(x0) + 2 * lane + 1] + c.noise_std[2 * lane + 1] * n1;
    }
    if (wid == roll_warp) {
        const double ud = sm[LF(uprev)], udel = sm[LF(uprev) + 1];
        double sd, cd, xs[6], f[6];
        TG_SINCOS(udel, sd, cd);
#pragma unroll
        for (int i = 0; i < 6; ++i) xs[i] = sm[LF(x0) + i];
        if (lane < 6) xbar[lane] = sm[LF(x0) + lane];
        // kernels with a compile-time horizon serve the standard controller only (MPC tyre model from the tables, analytic
        // Jacobians: checked by the dispatcher), so the other variants' code is not even compiled into them
        const bool use_tab = (NC > 0) ? true : (c.tyre_tab && c.model != TG_MODEL_GEN1);
        const int model = (NC > 0) ? TG_MODEL_MPC : c.model;
        if (use_tab) {
            // (vx, vy, omega) do not depend on the pose, so only they ride the sequential chain (slip angle -> tyre force ->
            // Euler update, from tables); heading and position are recovered afterwards in the reference's summation order.
            double vx = xs[3], vy = xs[4], om = xs[5];
            const TgRoll rk = tg_roll_setup(c, ud, udel, sd, cd, lane);
#pragma unroll 1
            for (int k = 0; k < N; ++k) {
                tg_roll_stage(c, rk, model, vx, vy, om, lane, sm + LF(aux) + 6 * k);
                if (lane == 0) { xbar[6 * (k + 1) + 3] = vx; xbar[6 * (k + 1) + 4] = vy; xbar[6 * (k + 1) + 5] = om; }
            }
            __syncwarp();
            if (lane == 0) {
                double phi = xs[2];
                for (int k = 0; k < N; ++k) { phi = phi + c.Ts * xbar[6 * k + 5]; xbar[6 * (k + 1) + 2] = phi; }
            }
            __syncwarp();
            for (int k = lane; k < N; k += 32) {
                double s_, c_;
                TG_SINCOS(xbar[6 * k + 2], s_, c_);
                const double vxk = xbar[6 * k + 3], vyk = xbar[6 * k + 4];
                double *ax = sm + LF(aux) + 6 * k;
                ax[2] = s_; ax[3] = c_;
                ax[4] = vxk * c_ - vyk * s_;          // Xdot, Ydot of the stage
                ax[5] = vxk * s_ + vyk * c_;
            }
            __syncwarp();
            if (lane < 2) {
                double pos = xs[lane];
                for (int k = 0; k < N; ++k) { pos = pos + c.Ts * sm[LF(aux) + 6 * k + 4 + lane]; xbar[6 * (k + 1) + lane] = pos; }
            }
        } else {
#pragma unroll 1
            for (int k = 0; k < N; ++k) {
                tg_f_cont_lanes(c.p, c.inv_m, c.inv_Iz, model, xs, ud, udel, sd, cd, lane, f, sm + LF(aux) + 6 * k);
#pragma unroll
                for (int i = 0; i < 6; ++i) xs[i] = xs[i] + c.Ts * f[i];
                if (lane == 0) {
#pragma unroll
                    for (int i = 0; i < 6; ++i) xbar[6 * (k + 1) + i] = xs[i];
                }
            }
        }
    }
    tw_sync<W>(bar);
    TG_TICK(0);

    // ---------------- K1b: linearise every stage (mpc_6stati.py:175-178) + tracking residuals at xbar (rows carry sqrt(2 q))
    const double sqc = sqrt(2.0 * TWC(q_c)), sqp = sqrt(2.0 * TWC(q_phi)), sqv = sqrt(2.0 * TWC(q_vx));
    {
        const double ud = sm[LF(uprev)], udel = sm[LF(uprev) + 1];
        for (int k = tid; k < N; k += NT) {
            double xs[6];
#pragma unroll
            for (int i = 0; i < 6; ++i) xs[i] = xbar[6 * k + i];
            double *gout = tap.g ? tap.g + 6 * k : nullptr;
            if (NC == 0 && c.jacobian == TG_JAC_FD) {
                tg_linearize_fd(c, xs, ud, udel, lin + TG_LIN * k, gout);
            } else {
                double sd, cd;
                TG_SINCOS(udel, sd, cd);
                bool kink;
                if (NC > 0 || (c.tyre_tab && c.model != TG_MODEL_GEN1)) kink = tg_linearize_analytic(c, xs, ud, udel, sd, cd, lin + TG_LIN * k, gout, nullptr, sm + LF(aux) + 6 * k);
                else kink = tg_linearize_analytic(c, xs, ud, udel, sd, cd, lin + TG_LIN * k, gout, sm + LF(aux) + 6 * k);
                if (kink) tg_linearize_fd(c, xs, ud, udel, lin + TG_LIN * k, gout);   // rare: the reference's own arithmetic at a kink
            }
        }
        double c0_part = 0.0;
        for (int k = NT - 1 - tid; k <= N; k += NT) {   // from the last thread down: overlaps the linearisation when W > 1
            const double *xk = xbar + 6 * k;
            const double s_ = sn[k], c_ = cs[k];
            const double rc = sqc * (s_ * (xk[0] - sm[LF(Xr) + k]) - c_ * (xk[1] - sm[LF(Yr) + k]));  // lateral_error :111-117
            const double rp = sqp * (xk[2] - sm[LF(Pr) + k]), rv = sqv * (xk[3] - sm[LF(vref) + k]);
            c0_part += 0.5 * (rc * rc + rp * rp + rv * rv);
            rr[3 * k] = rc; rr[3 * k + 1] = rp; rr[3 * k + 2] = rv;
        }
        tw_sync<W>(bar);   // everybody is done with the unscaled sn / cs and the window
        for (int k = NT - 1 - tid; k <= N; k += NT) { sn[k] *= sqc; cs[k] *= sqc; }
        if (!fx) {   // constant term: stage costs at xbar + N u_prev' R u_prev (only the step API reports the objective)
            double c0 = tw_reduce_sum<W>(c0_part, red, tid, bar);
            c0 += (double)N * (ud * (TWC(Rs[0]) * ud + TWC(Rs[1]) * udel) + udel * (TWC(Rs[2]) * ud + TWC(Rs[3]) * udel));
            if (tid == 0) misc[M_C0] = c0;
        }
    }
    if (tap.A || tap.Bm) {
        for (int k = tid; k < N; k += NT)
            tg_lin_expand(lin + TG_LIN * k, nullptr, tap.A ? tap.A + 36 * k : nullptr, tap.Bm ? tap.Bm + 12 * k : nullptr, nullptr);
    }
    if (tap.xbar)
        for (int i = tid; i < 6 * (N + 1); i += NT) tap.xbar[i] = xbar[i];
    tw_sync<W>(bar);
    if (tap.stop == 1) return res;
    TG_TICK(1);

    // ---------------- K2 + bounds + rho, K3: factor; ADMM.  The factor pass is re-entered when rho changes.
    double a[S][4][4];
    const double lb0 = TWC(u_lo[0]) - sm[LF(uprev)], ub0 = TWC(u_hi[0]) - sm[LF(uprev)];
    const double lb1 = TWC(u_lo[1]) - sm[LF(uprev) + 1], ub1 = TWC(u_hi[1]) - sm[LF(uprev) + 1];
    const double sigma = c.sigma;
    bool x0_infeasible = false;
    for (int si = 0; si < ns; ++si) {
        const int sx = c.sidx[si];
        const double xv = sm[LF(x0) + sx];
        // k = 0 rows (:217,:220): x0 itself outside its box.  The reference hands these rows to OSQP, which accepts a violation
        // below its primal tolerance (CVXPY's settings: eps_abs = eps_rel = 1e-5) as "optimal" -- e.g. the plant landing 1e-6
        // outside a bound that the previous step's plan touched -- so the same tolerance applies here, whatever tighter
        // tolerance this library's own iteration runs at.
        const double ea = fmax(c.eps_abs, 1e-5), er = fmax(c.eps_rel, 1e-5);
        if (xv < TWC(x_lo[sx]) - (ea + er * fmax(fabs(xv), fabs(TWC(x_lo[sx])))) || xv > TWC(x_hi[sx]) + (ea + er * fmax(fabs(xv), fabs(TWC(x_hi[sx])))))
            x0_infeasible = true;
    }
    bool free_mode = (!warm || warm_free) && c.free_mode;
    double rho_scale = free_mode ? TW_FREE_RHO : c.rho;
    double alpha = free_mode ? 1.0 : (warm ? c.alpha_warm : c.alpha);
    const int alpha_switch = 4 * c.check_every;
    int status = TG_STATUS_USER_LIMIT, it = 0;
    int until_check = free_mode ? 2 : c.check_every;
    double obj = 0.0, nq = 0.0;
    bool first = true, done = false, all_free = false, polished = false;
    const bool my = tid < N;              // this thread owns a stage
    const int j0 = 2 * tid;               // its first entry

#pragma unroll 1
    while (!done) {
        tw_condense<W, S, NC, HS, CT>(c, L, sm, mp, a, first, tid, bar, cr);
        if (first) {
#pragma unroll
            for (int s = 0; s < S; ++s)
                if (mp.act[s] && mp.ro[s] == mp.co[s]) tw_st4(sm + LF(dH) + mp.ro[s], a[s][0][0], a[s][1][1], a[s][2][2], a[s][3][3]);
            tw_sync<W>(bar);
            // bounds (mpc_6stati.py:198-221) and per-row rho = rho0 / max_j(a_ij^2 / H_jj)
            const double *dH = sm + LF(dH);
            if (my) {
                const double h0 = dH[j0], h1 = dH[j0 + 1];
                const double g0 = (tid > 0) ? fmin(h0, dH[j0 - 2]) : h0, g1 = (tid > 0) ? fmin(h1, dH[j0 - 1]) : h1;
                tw_st2(rho + j0, rho_scale * h0, rho_scale * h1);
                tw_st2(rho + n + j0, rho_scale * g0, rho_scale * g1);
                tw_st2(rinv + j0, 1.0 / (rho_scale * h0), 1.0 / (rho_scale * h1));
                tw_st2(rinv + n + j0, 1.0 / (rho_scale * g0), 1.0 / (rho_scale * g1));
            }
            for (int i = tid; i < ms; i += NT) {
                const int nsd = ns > 0 ? ns : 1, kk = i / nsd + 1, sx = c.sidx[i % nsd];
                const double xb = xbar[6 * kk + sx];
                ls[i] = (TWC(x_lo[sx]) <= -TG_INF) ? -TG_INF : TWC(x_lo[sx]) - xb;
                us[i] = (TWC(x_hi[sx]) >= TG_INF) ? TG_INF : TWC(x_hi[sx]) - xb;
                double mx = 0.0;
                const double *grow = Gs + ns * tw_gs_off(kk - 1) + (i % nsd) * tw_gs_len(kk - 1);
                for (int j = 0; j < 2 * kk; ++j) { const double gij = grow[j]; mx = fmax(mx, gij * gij / dH[j]); }
                const double rs = rho_scale * ((mx > 1e-30) ? 1.0 / mx : 1.0);
                rhos[i] = rs; rinvs[i] = 1.0 / rs;
            }
            if (tap.H) {
#pragma unroll
                for (int s = 0; s < S; ++s)
                    if (mp.act[s])
#pragma unroll
                        for (int r = 0; r < 4; ++r)
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc) {
                                const int i = mp.ro[s] + r, j = mp.co[s] + cc;
                                if (i < n && j < n) { tap.H[i * n + j] = a[s][r][cc]; tap.H[j * n + i] = a[s][r][cc]; }
                            }
            }
            double nqp = 0.0;
            if (my) nqp = fmax(fabs(q[j0]), fabs(q[j0 + 1]));
            {
                double vals[1] = {nqp};
                tw_reduce_max<W, 1>(vals, red, tid, bar);
                nq = vals[0];
            }
            tw_sync<W>(bar);   // rho visible to every thread; dH (aliases v) no longer needed
            if (tap.q) for (int i = tid; i < n; i += NT) tap.q[i] = q[i];
            if (tap.c0 && tid == 0) tap.c0[0] = misc[M_C0];
            if (tap.l) {
                for (int i = tid; i < n; i += NT) {
                    tap.l[i] = (i & 1) ? lb1 : lb0; tap.u[i] = (i & 1) ? ub1 : ub0;
                    tap.l[n + i] = TWC(du_lo[i & 1]); tap.u[n + i] = TWC(du_hi[i & 1]);
                }
                for (int i = tid; i < ms; i += NT) { tap.l[2 * n + i] = ls[i]; tap.u[2 * n + i] = us[i]; }
            }
            if (tap.Gs)
                for (int i = tid; i < ms * n; i += NT) {
                    const int nsd = ns > 0 ? ns : 1, r_ = i / n, j = i % n, k = r_ / nsd;
                    tap.Gs[i] = (j < 2 * (k + 1)) ? Gs[ns * tw_gs_off(k) + (r_ % nsd) * tw_gs_len(k) + j] : 0.0;
                }
            if (tap.stop == 2) return res;
            TG_TICK(3);
        }
        tw_build_K<W, S, NC, HS>(c, L, sm, mp, a);
        tw_sweep_invert<W, S, NC>(c, L, sm, mp, a, bar);
        TG_TICK(4);

        if (x0_infeasible) { status = TG_STATUS_INFEASIBLE; break; }
        if (first) {
            if (!warm) {
                if (my) { tw_st2(x + j0, 0.0, 0.0); tw_st2(z + j0, 0.0, 0.0); tw_st2(z + n + j0, 0.0, 0.0); tw_st2(y + j0, 0.0, 0.0); tw_st2(y + n + j0, 0.0, 0.0); }
                for (int i = tid; i < ms; i += NT) { zs[i] = 0.0; ys[i] = 0.0; }
            } else {
                if (my) {
                    const double2 xj = tw_ld2(x + j0);
                    const double2 xp = (tid > 0) ? tw_ld2(x + j0 - 2) : make_double2(0.0, 0.0);
                    tw_st2(z + j0, tg_clamp(xj.x, lb0, ub0), tg_clamp(xj.y, lb1, ub1));
                    tw_st2(z + n + j0, tg_clamp(xj.x - xp.x, TWC(du_lo[0]), TWC(du_hi[0])), tg_clamp(xj.y - xp.y, TWC(du_lo[1]), TWC(du_hi[1])));
                }
                for (int r0 = 0; r0 < ms; r0 += NT >> geo.lg_tpr) {
                    const int r_ = r0 + (tid >> geo.lg_tpr);
                    const double acc = tw_gs_row_dot<W>(L, sm, geo, ns, ms, x, r_, tid);
                    if (r_ < ms && (tid & (geo.tpr - 1)) == 0) zs[r_] = tg_clamp(acc, ls[r_], us[r_]);
                }
            }
            tw_sync<W>(bar);
        }
        if (ms > 0) {   // t = rho_s z_s - y_s for the first right-hand side of this factorisation
            for (int i = tid; i < ms; i += NT) tv[i] = rhos[i] * zs[i] - ys[i];
            tw_sync<W>(bar);
        }
        first = false;
        TG_TICK(7);

        bool refactor = false;
#pragma unroll 1
        while (!refactor) {
            ++it;
            const bool check = (--until_check == 0) || (it == c.max_iter);
            if (check) until_check = free_mode ? 1 : c.check_every;
            if (!free_mode && it == alpha_switch + 1) alpha = c.alpha;
            if (warm && !free_mode && it == TW_WARM_RESTART_ITER) {
                // a warm start that has not converged by now is a bad start (the active set changed): restart from zero
                if (my) { tw_st2(x + j0, 0.0, 0.0); tw_st2(z + j0, 0.0, 0.0); tw_st2(z + n + j0, 0.0, 0.0); tw_st2(y + j0, 0.0, 0.0); tw_st2(y + n + j0, 0.0, 0.0); }
                for (int i = tid; i < ms; i += NT) { zs[i] = 0.0; ys[i] = 0.0; tv[i] = 0.0; }
                tw_sync<W>(bar);
            }
            // (a) rhs = sigma x - q + A'(rho z - y)
            if (ms > 0) {   // state rows: G_s' (rho_s z_s - y_s) by all threads
                const double *const vec1[1] = {tv};
                tw_gs_tmul<W, 1>(L, sm, geo, N, ns, NV, vec1, tid);
                tw_sync<W>(bar);
            }
            double2 rhs2 = make_double2(0.0, 0.0);
            if (my) {
                const double2 x2 = tw_ld2(x + j0), q2 = tw_ld2(q + j0);
                const double2 zb = tw_ld2(z + j0), yb = tw_ld2(y + j0), rb = tw_ld2(rho + j0);
                const double2 zr = tw_ld2(z + n + j0), yr = tw_ld2(y + n + j0), rr2 = tw_ld2(rho + n + j0);
                double r0 = sigma * x2.x - q2.x + (rb.x * zb.x - yb.x) + (rr2.x * zr.x - yr.x);
                double r1 = sigma * x2.y - q2.y + (rb.y * zb.y - yb.y) + (rr2.y * zr.y - yr.y);
                if (tid + 1 < N) {
                    const double2 zn_ = tw_ld2(z + n + j0 + 2), yn_ = tw_ld2(y + n + j0 + 2), rn_ = tw_ld2(rho + n + j0 + 2);
                    r0 -= rn_.x * zn_.x - yn_.x; r1 -= rn_.y * zn_.y - yn_.y;
                }
                if (ms > 0) { const double2 g2 = tw_ld2(gt + j0); r0 += g2.x; r1 += g2.y; }
                rhs2 = make_double2(r0, r1);
                tw_st2(v + j0, r0, r1);
            }
            tw_sync<W>(bar);
            // (b) x~ = K^-1 rhs
            tw_matvec_partials<W, S, NC>(L, sm, mp, a);
            tw_sync<W>(bar);
            double2 xt2 = make_double2(0.0, 0.0);
            if (my) { xt2 = tw_matvec_sum<W, NC>(L, sm, tid); tw_st2(xt + j0, xt2.x, xt2.y); }
            tw_sync<W>(bar);
            // (c) relaxation, projection, dual update; lane t: box rows 2t, 2t+1 and rate rows 2t, 2t+1
            double rp = 0.0, nzt = 0.0, nz = 0.0, ndy = 0.0, cert = 0.0;
            double2 dyb = make_double2(0.0, 0.0), dyr2 = make_double2(0.0, 0.0);
            bool clamped = false, near = false;
            if (my) {
                const double2 x2 = tw_ld2(x + j0);
                tw_st2(x + j0, alpha * xt2.x + (1.0 - alpha) * x2.x, alpha * xt2.y + (1.0 - alpha) * x2.y);
                {   // box rows
                    const double2 zo = tw_ld2(z + j0), yo = tw_ld2(y + j0), ri = tw_ld2(rinv + j0), r_ = tw_ld2(rho + j0);
                    const double zr0 = alpha * xt2.x + (1.0 - alpha) * zo.x, zr1 = alpha * xt2.y + (1.0 - alpha) * zo.y;
                    const double t0 = zr0 + yo.x * ri.x, t1 = zr1 + yo.y * ri.y;
                    const double zn0 = tg_clamp(t0, lb0, ub0), zn1 = tg_clamp(t1, lb1, ub1);
                    const double yn0 = yo.x + r_.x * (zr0 - zn0), yn1 = yo.y + r_.y * (zr1 - zn1);
                    clamped = clamped || zn0 != t0 || zn1 != t1;
                    dyb = make_double2(yn0 - yo.x, yn1 - yo.y);
                    rp = fmax(fabs(xt2.x - zn0), fabs(xt2.y - zn1));
                    nzt = fmax(fabs(xt2.x), fabs(xt2.y)); nz = fmax(fabs(zn0), fabs(zn1));
                    tw_st2(z + j0, zn0, zn1); tw_st2(y + j0, yn0, yn1);
                    if (check) {
                        ndy = fmax(fabs(dyb.x), fabs(dyb.y));
                        cert += (dyb.x > 0.0 ? ub0 : lb0) * dyb.x + (dyb.y > 0.0 ? ub1 : lb1) * dyb.y;
                        near = fmin(fmin(xt2.x - lb0, ub0 - xt2.x), fmin(xt2.y - lb1, ub1 - xt2.y)) < TW_POLISH_MARGIN;
                    }
                }
                {   // rate rows
                    const double2 xp = (tid > 0) ? tw_ld2(xt + j0 - 2) : make_double2(0.0, 0.0);
                    const double zt0 = xt2.x - xp.x, zt1 = xt2.y - xp.y;
                    const double2 zo = tw_ld2(z + n + j0), yo = tw_ld2(y + n + j0), ri = tw_ld2(rinv + n + j0), r_ = tw_ld2(rho + n + j0);
                    const double zr0 = alpha * zt0 + (1.0 - alpha) * zo.x, zr1 = alpha * zt1 + (1.0 - alpha) * zo.y;
                    const double t0 = zr0 + yo.x * ri.x, t1 = zr1 + yo.y * ri.y;
                    const double zn0 = tg_clamp(t0, TWC(du_lo[0]), TWC(du_hi[0])), zn1 = tg_clamp(t1, TWC(du_lo[1]), TWC(du_hi[1]));
                    const double yn0 = yo.x + r_.x * (zr0 - zn0), yn1 = yo.y + r_.y * (zr1 - zn1);
                    clamped = clamped || zn0 != t0 || zn1 != t1;
                    dyr2 = make_double2(yn0 - yo.x, yn1 - yo.y);
                    rp = fmax(rp, fmax(fabs(zt0 - zn0), fabs(zt1 - zn1)));
                    nzt = fmax(nzt, fmax(fabs(zt0), fabs(zt1))); nz = fmax(nz, fmax(fabs(zn0), fabs(zn1)));
                    tw_st2(z + n + j0, zn0, zn1); tw_st2(y + n + j0, yn0, yn1);
                    if (check) {
                        tw_st2(dyr + j0, dyr2.x, dyr2.y);
                        ndy = fmax(ndy, fmax(fabs(dyr2.x), fabs(dyr2.y)));
                        cert += (dyr2.x > 0.0 ? TWC(du_hi[0]) : TWC(du_lo[0])) * dyr2.x + (dyr2.y > 0.0 ? TWC(du_hi[1]) : TWC(du_lo[1])) * dyr2.y;
                        near = near || fmin(fmin(zt0 - TWC(du_lo[0]), TWC(du_hi[0]) - zt0), fmin(zt1 - TWC(du_lo[1]), TWC(du_hi[1]) - zt1)) < TW_POLISH_MARGIN;
                    }
                }
            }
            for (int r0 = 0; r0 < ms; r0 += NT >> geo.lg_tpr) {
                const int r_ = r0 + (tid >> geo.lg_tpr);
                const double ztl = tw_gs_row_dot<W>(L, sm, geo, ns, ms, xt, r_, tid);
                if (r_ >= ms || (tid & (geo.tpr - 1)) != 0) continue;
                const double zr = alpha * ztl + (1.0 - alpha) * zs[r_];
                const double t_ = zr + ys[r_] * rinvs[r_];
                const double zn = tg_clamp(t_, ls[r_], us[r_]);
                const double yn = ys[r_] + rhos[r_] * (zr - zn);
                clamped = clamped || zn != t_;
                const double d_ = yn - ys[r_];
                ys[r_] = yn; zs[r_] = zn; tv[r_] = rhos[r_] * zn - yn;
                rp = fmax(rp, fabs(ztl - zn)); nzt = fmax(nzt, fabs(ztl)); nz = fmax(nz, fabs(zn));
                if (check) {
                    zts[r_] = ztl; dys[r_] = d_;
                    ndy = fmax(ndy, fabs(d_));
                    if (d_ > 0.0) cert += (us[r_] >= TG_INF) ? 1e300 : us[r_] * d_;
                    else if (d_ < 0.0) cert += (ls[r_] <= -TG_INF) ? 1e300 : ls[r_] * d_;
                    near = near || fmin(ztl - ls[r_], us[r_] - ztl) < TW_POLISH_MARGIN;
                }
            }
            tw_sync<W>(bar);
            TG_TICK(8);
            if (free_mode && tw_any<W>(clamped, red, tid, bar)) {
                // a row is active after all: standard settings from here on
                free_mode = false; polished = true;
                rho_scale = c.rho;
                alpha = warm ? c.alpha_warm : c.alpha;
                until_check = c.check_every;
                const double f_ = c.rho / TW_FREE_RHO;
                for (int i = tid; i < 2 * n; i += NT) { rho[i] *= f_; rinv[i] = 1.0 / rho[i]; }
                for (int i = tid; i < ms; i += NT) { rhos[i] *= f_; rinvs[i] = 1.0 / rhos[i]; ys[i] = 0.0; }
                if (my) { tw_st2(y + j0, 0.0, 0.0); tw_st2(y + n + j0, 0.0, 0.0); }
                tw_sync<W>(bar);
                refactor = true;
                continue;
            }
            if (!check) continue;

            // (d) residuals at (x~, z, y):  H x~ = rhs - sigma x~ - A'(rho .* z~)
            double rd = 0.0, nh = 0.0, na = 0.0, natdy = 0.0;
            bool bad = false;
            if (ms > 0) {   // G_s' y_s, G_s' (rho_s z~_s), G_s' dy_s by all threads (zts is scaled in place: it is rewritten at the next check)
                for (int i = tid; i < ms; i += NT) zts[i] *= rhos[i];
                tw_sync<W>(bar);
                const double *const vec3[3] = {ys, zts, dys};
                tw_gs_tmul<W, 3>(L, sm, geo, N, ns, NV, vec3, tid);
                tw_sync<W>(bar);
            }
            if (my) {
                const double2 yb = tw_ld2(y + j0), yr = tw_ld2(y + n + j0), rb = tw_ld2(rho + j0), rr2 = tw_ld2(rho + n + j0);
                const double2 xp = (tid > 0) ? tw_ld2(xt + j0 - 2) : make_double2(0.0, 0.0);
                double aty0 = yb.x + yr.x, aty1 = yb.y + yr.y;
                double atr0 = rb.x * xt2.x + rr2.x * (xt2.x - xp.x), atr1 = rb.y * xt2.y + rr2.y * (xt2.y - xp.y);
                double atd0 = dyb.x + dyr2.x, atd1 = dyb.y + dyr2.y;
                if (tid + 1 < N) {
                    const double2 yn_ = tw_ld2(y + n + j0 + 2), rn_ = tw_ld2(rho + n + j0 + 2), xn_ = tw_ld2(xt + j0 + 2), dn_ = tw_ld2(dyr + j0 + 2);
                    aty0 -= yn_.x; aty1 -= yn_.y;
                    atr0 -= rn_.x * (xn_.x - xt2.x); atr1 -= rn_.y * (xn_.y - xt2.y);
                    atd0 -= dn_.x; atd1 -= dn_.y;
                }
                if (ms > 0) {
                    const double2 gy = tw_ld2(gt + j0), gr_ = tw_ld2(gt + NV + j0), gd = tw_ld2(gt + 2 * NV + j0);
                    aty0 += gy.x; aty1 += gy.y; atr0 += gr_.x; atr1 += gr_.y; atd0 += gd.x; atd1 += gd.y;
                }
                const double2 q2 = tw_ld2(q + j0);
                const double hx0 = rhs2.x - sigma * xt2.x - atr0, hx1 = rhs2.y - sigma * xt2.y - atr1;
                rd = fmax(fabs(hx0 + q2.x + aty0), fabs(hx1 + q2.y + aty1));
                nh = fmax(fabs(hx0), fabs(hx1)); na = fmax(fabs(aty0), fabs(aty1));
                natdy = fabs(atd0) * fmax(fabs(lb0), fabs(ub0)) + fabs(atd1) * fmax(fabs(lb1), fabs(ub1));
                bad = !(isfinite(hx0) && isfinite(hx1) && isfinite(aty0) && isfinite(aty1));
                if (!fx) obj = xt2.x * (0.5 * hx0 + q2.x) + xt2.y * (0.5 * hx1 + q2.y);
            }
            double vals[7] = {rp, nzt, nz, rd, nh, na, ndy};
            tw_reduce_max<W, 7>(vals, red, tid, bar);
            const bool any_bad = tw_any<W>(bad, red, tid, bar);
            const double eps_p = c.eps_abs + c.eps_rel * fmax(vals[1], vals[2]);
            const double eps_d = c.eps_abs + c.eps_rel * fmax(fmax(vals[4], vals[5]), nq);
            if (any_bad || !(vals[0] == vals[0]) || !(vals[3] == vals[3])) { status = TG_STATUS_NAN; done = true; break; }
            TG_TICK(9);
            if (vals[0] <= eps_p && vals[3] <= eps_d) {
                if (!free_mode && c.free_mode && !polished) {
                    // Polish.  A standard solve stops within eps of the optimum (a warm-started one that has just lost its last
                    // active row, e.g. the duty cycle leaving its bound, ended 4e-4 away with duals of ~1e-6 still decaying).  If
                    // every row of the final iterate is clearly inside its bounds (margin TW_POLISH_MARGIN), no row is active and
                    // the optimum is the unconstrained one: drop the duals and finish in free mode, which lands on it to
                    // rounding.  (Once per step: if the free iterate clamps after all, the solve returns to the standard
                    // settings and ends there.)
                    if (!tw_any<W>(near, red, tid, bar)) {
                        polished = true; free_mode = true; alpha = 1.0; until_check = 2;
                        const double f_ = TW_FREE_RHO / rho_scale;
                        rho_scale = TW_FREE_RHO;
                        for (int i = tid; i < 2 * n; i += NT) { rho[i] *= f_; rinv[i] = 1.0 / rho[i]; y[i] = 0.0; }
                        for (int i = tid; i < ms; i += NT) { rhos[i] *= f_; rinvs[i] = 1.0 / rhos[i]; ys[i] = 0.0; }
                        tw_sync<W>(bar);
                        refactor = true;
                        continue;
                    }
                }
                status = TG_STATUS_OPTIMAL; all_free = free_mode; done = true; break;
            }
            if (it >= c.max_iter) {
                if (vals[0] <= 10.0 * eps_p && vals[3] <= 10.0 * eps_d) status = TG_STATUS_OPTIMAL_INACCURATE;
                done = true;
                break;
            }
            // numerical failure guard: a convergent iteration stays near the input box; with relative tolerances a
            // diverging one would otherwise "converge" (eps_rel * 1e58 > any residual)
            if (vals[1] > 1e8) { status = TG_STATUS_NAN; done = true; break; }
            // primal infeasibility certificate.  OSQP (section 3.4) asks ||A'dy|| <= eps ||dy|| and u'(dy)+ + l'(dy)- < 0;
            // on this problem family ||A'dy|| / ||dy|| plateaus near 5e-3 for thousands of iterations.  Every dU_j is
            // boxed by its input row (|dU_j| <= r_j = max(|l_j|, |u_j|)), which gives a RIGOROUS, scale-free test:
            // for any feasible dU, -sum_j |A'dy|_j r_j <= dy'A dU <= u'(dy)+ + l'(dy)-, so
            //      u'(dy)+ + l'(dy)- + sum_j |(A'dy)_j| r_j < 0   proves infeasibility.
            {
                const double cert_sum = tw_reduce_sum<W>(cert + natdy, red, tid, bar);
                if (vals[6] > 1e-30 && cert_sum < -1e-9 * vals[6]) { status = TG_STATUS_INFEASIBLE; done = true; break; }
            }
            if (free_mode) continue;
            if (c.adaptive_rho && it >= c.adaptive_rho_min_iter) {
                const double sp = fmax(vals[1], vals[2]), sd = fmax(fmax(vals[4], vals[5]), nq);
                const double ratio = sqrt((vals[0] / (sp + 1e-10)) / (vals[3] / (sd + 1e-10) + 1e-10));
                const double ns_ = fmin(fmax(rho_scale * ratio, 1e-6), 1e6);
                if (ns_ > rho_scale * c.adapt_tol || ns_ * c.adapt_tol < rho_scale) {
                    const double f_ = ns_ / rho_scale;
                    rho_scale = ns_;
                    for (int i = tid; i < 2 * n; i += NT) { rho[i] *= f_; rinv[i] = 1.0 / rho[i]; }
                    for (int i = tid; i < ms; i += NT) { rhos[i] *= f_; rinvs[i] = 1.0 / rhos[i]; }
                    tw_sync<W>(bar);
                    refactor = true;   // H is rebuilt from the stage records (no copy of it is kept), then K, then K^-1
                }
            }
        }
    }
    if (!fx && (status == TG_STATUS_OPTIMAL || status == TG_STATUS_OPTIMAL_INACCURATE)) obj = tw_reduce_sum<W>(obj, red, tid, bar);
    if (!all_free && status == TG_STATUS_OPTIMAL) {   // a standard solve that ended with no active row: the next one may start free
        bool nzy = false;
        if (my) { const double2 yb = tw_ld2(y + j0), yr = tw_ld2(y + n + j0); nzy = yb.x != 0.0 || yb.y != 0.0 || yr.x != 0.0 || yr.y != 0.0; }
        for (int i = tid; i < ms; i += NT) nzy = nzy || ys[i] != 0.0;
        all_free = !tw_any<W>(nzy, red, tid, bar);
    }
    TG_TICK(5);
    if (it > c.max_iter) it = c.max_iter;
    res.status = status;
    res.iters = it;
    res.objective = obj + misc[M_C0];
    res.free_end = all_free;
    if (tid == 0) misc[M_RHOSCALE] = rho_scale;
    tw_sync<W>(bar);
    TG_TICK(6);
    return res;
}
