// tg_openloop.cuh -- the generators' open-loop control synthesis fused with the plant and the sensor noise
// (SURVEY.md section 8(f), rank 2).  sm_100a, fp64.
//
// Reference (paths relative to the reference root):
//   generation_type1.py:86-137   create_spline_signal / generate_smooth_profiles / apply_du_bounds
//   generation_type1.py:279-306  per-trajectory body of the main loop (control noise, slew, clip, simulate, sensor noise)
//   generation_type2.py:95-157   sample_controls_piecewise (accelerate / cruise / turn state machine on a shadow simulation)
//   generation_type2.py:176-200  ground-truth integration + sensor noise
//
// One thread owns one trajectory for the sequential part (control recursion + Euler plant); the 32 trajectories of
// a warp stage TG_OL_CHUNK rows in a shared-memory tile, and the warp then writes the tile out cooperatively, so
// that global stores are 16-byte, contiguous within each trajectory's run of rows, and the sensor noise (one
// Philox block + one Box-Muller per column pair) is computed by all lanes in parallel instead of serially per row.
// The random streams are Philox4x32-10 keyed by trajectory id (layout: oracle/openloop.py, which is also the CPU
// statement of what this file must produce).
#pragma once
#include "tg_device.cuh"

#define TG_OL_CHUNK 4          // rows staged per warp between cooperative write-outs
#define TG_OL_WARPS 2          // warps per CTA
#define TG_OL_STRIDE 33        // tile row stride in doubles (32 trajectories + 1: conflict-free column access)
#define TG_OL_MAX_KNOTS 16     // knots of the transient spline (the reference's ranges give 2)
#define TG_OL_TILE (TG_OL_CHUNK * 8 * TG_OL_STRIDE)

__device__ __forceinline__ double tg_u01(uint32_t r) { return ((double)r + 0.5) * 2.3283064365386963e-10; }   // (r + 0.5) 2^-32
__device__ __forceinline__ double tg_uniform(uint32_t r, double lo, double hi) { return lo + (hi - lo) * tg_u01(r); }

__device__ __forceinline__ void tg_ctrl_philox(unsigned long long key, uint32_t index, uint32_t block, uint32_t out[4])
{
    tg_philox4x32_10(index, block, 0u, 0u, (uint32_t)key, (uint32_t)(key >> 32), out);
}

// ------------------------------------------------------------------------------------------------ type 1
struct Type1Thread {
    int n_tr, K, piece, sinusoid;
    int kx[TG_OL_MAX_KNOTS];
    double y[2][TG_OL_MAX_KNOTS], m2[2][TG_OL_MAX_KNOTS];   // knot values and second derivatives (d, delta)
    double cf[2][4];                                         // coefficients of the current piece
    double w, amp, phase;
    double out[2];                                           // slew-limiter state (before the final clip)
};

__device__ __forceinline__ void tg_t1_load_piece(Type1Thread &s, int i)
{
    s.piece = i;
    const double h = (double)(s.kx[i + 1] - s.kx[i]);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const double dl = (s.y[c][i + 1] - s.y[c][i]) / h;
        s.cf[c][0] = (s.m2[c][i + 1] - s.m2[c][i]) / (6.0 * h);
        s.cf[c][1] = 0.5 * s.m2[c][i];
        s.cf[c][2] = dl - h * (2.0 * s.m2[c][i] + s.m2[c][i + 1]) / 6.0;
        s.cf[c][3] = s.y[c][i];
    }
}

// generate_smooth_profiles' draws + create_spline_signal (generation_type1.py:86-102, 104-113)
__device__ void tg_t1_setup(Type1Thread &s, const tg_type1_rules &r, unsigned long long key, int T, double Ts)
{
    uint32_t a[4], b4[4];
    tg_ctrl_philox(key, 0u, 0x10u, a);      // mode, transient, checkpoint, period
    tg_ctrl_philox(key, 1u, 0x10u, b4);     // amplitude, phase
    s.sinusoid = (r.mode >= 0) ? r.mode : (tg_u01(a[0]) < r.p_straight ? 0 : 1);               // :108
    int n_tr = (int)(tg_uniform(a[1], r.transient_s[0], r.transient_s[1]) / Ts);               // :110-111
    s.n_tr = n_tr < T ? n_tr : T;
    s.w = 6.283185307179586 / tg_uniform(a[3], r.period_s[0], r.period_s[1]);                  // :122-123
    s.amp = tg_uniform(b4[0], r.delta_std * r.amp_frac[0], r.delta_std * r.amp_frac[1]);
    s.phase = tg_uniform(b4[1], 0.0, 6.283185307179586);
    s.out[0] = s.out[1] = 0.0;
    s.K = 1; s.piece = -1;
    if (s.n_tr <= 1) return;                                                                    // :88
    const double every_d = rint(tg_uniform(a[2], r.checkpoint_s[0], r.checkpoint_s[1]) / Ts);  // :90-91
    const int every = every_d < 1.0 ? 1 : (int)every_d;
    int K = 0;
    for (int p = 0; p < s.n_tr && K < TG_OL_MAX_KNOTS; p += every) s.kx[K++] = p;             // :93
    if (s.kx[K - 1] != s.n_tr - 1 && K < TG_OL_MAX_KNOTS) s.kx[K++] = s.n_tr - 1;             // :94
    s.K = K;
    const double sd[2] = {r.d_std * r.tr_d_frac, r.delta_std * r.tr_delta_frac};
    const double mu[2] = {r.d_mean, r.delta_mean};
    for (int k = 0; k < K; ++k) {                                                              // :96
        uint32_t w4[4];
        double z0, z1;
        tg_ctrl_philox(key, (uint32_t)k, 0x11u, w4);
        tg_box_muller(w4[0], w4[1], z0, z1);
        s.y[0][k] = mu[0] + sd[0] * z0;
        s.y[1][k] = mu[1] + sd[1] * z1;
    }
    // natural cubic spline (:97): second derivatives by the Thomas algorithm, m_0 = m_{K-1} = 0
    for (int c = 0; c < 2; ++c) { s.m2[c][0] = 0.0; s.m2[c][K - 1] = 0.0; }
    if (K > 2) {
        double bb[TG_OL_MAX_KNOTS], rr[2][TG_OL_MAX_KNOTS];
        for (int i = 1; i < K - 1; ++i) {
            const double h0 = (double)(s.kx[i] - s.kx[i - 1]), h1 = (double)(s.kx[i + 1] - s.kx[i]);
            bb[i] = 2.0 * (h0 + h1);
            for (int c = 0; c < 2; ++c)
                rr[c][i] = 6.0 * ((s.y[c][i + 1] - s.y[c][i]) / h1 - (s.y[c][i] - s.y[c][i - 1]) / h0);
            if (i > 1) {
                const double wgt = h0 / bb[i - 1];            // sub-diagonal a_i = h_{i-1}; super-diagonal of row i-1 = h_{i-1}
                bb[i] -= wgt * h0;
                for (int c = 0; c < 2; ++c) rr[c][i] -= wgt * rr[c][i - 1];
            }
        }
        for (int c = 0; c < 2; ++c) {
            s.m2[c][K - 2] = rr[c][K - 2] / bb[K - 2];
            for (int i = K - 3; i >= 1; --i) {
                const double h1 = (double)(s.kx[i + 1] - s.kx[i]);
                s.m2[c][i] = (rr[c][i] - h1 * s.m2[c][i + 1]) / bb[i];
            }
        }
    }
    tg_t1_load_piece(s, 0);
}

// control of step t (generation_type1.py:113-129, 283-289): profile + control noise -> slew limiter -> clip
__device__ __forceinline__ void tg_t1_control(Type1Thread &s, const tg_type1_rules &r, unsigned long long key, int t, double Ts,
                                              double &d_cmd, double &delta_cmd)
{
    uint32_t w4[4];
    tg_ctrl_philox(key, (uint32_t)t, 0x12u, w4);
    double zn0, zn1;
    tg_box_muller(w4[2], w4[3], zn0, zn1);
    double pc[2];
    if (t < s.n_tr) {
        if (s.n_tr <= 1) { pc[0] = r.d_mean; pc[1] = r.delta_mean; }
        else {
            while (s.piece + 2 < s.K && t >= s.kx[s.piece + 1]) tg_t1_load_piece(s, s.piece + 1);
            const double dx = (double)(t - s.kx[s.piece]);
#pragma unroll
            for (int c = 0; c < 2; ++c) pc[c] = ((s.cf[c][0] * dx + s.cf[c][1]) * dx + s.cf[c][2]) * dx + s.cf[c][3];
        }
    } else {
        double z0, z1;
        tg_box_muller(w4[0], w4[1], z0, z1);
        pc[0] = r.d_mean + (r.d_std * r.st_d_frac) * z0;                                       // :118
        if (s.sinusoid) {
            const double ts = (double)(t - s.n_tr) * Ts;
            pc[1] = (r.delta_mean + s.amp * sin(s.w * ts + s.phase)) + (r.delta_std * r.sin_noise_frac) * z1;   // :124-125
        } else {
            pc[1] = r.delta_mean + (r.delta_std * r.straight_frac) * z1;                        // :128
        }
    }
    const double raw[2] = {pc[0] + (r.d_std * r.ctrl_noise_frac) * zn0, pc[1] + (r.delta_std * r.ctrl_noise_frac) * zn1};
#pragma unroll
    for (int c = 0; c < 2; ++c)
        s.out[c] = (t == 0) ? raw[c] : s.out[c] + tg_clamp(raw[c] - s.out[c], r.du_lo[c], r.du_hi[c]);   // :131-137
    d_cmd = tg_clamp(s.out[0], r.u_lo[0], r.u_hi[0]);                                          // :288-289
    delta_cmd = tg_clamp(s.out[1], r.u_lo[1], r.u_hi[1]);
}

// ------------------------------------------------------------------------------------------------ type 2
struct Type2Thread {
    int seg, left, mode, prev_mode;
    double d, delta, prev_delta;
};

__device__ __forceinline__ int tg_choice(double u, const double *p, int n)
{
    double tot = 0.0;
    for (int i = 0; i < n; ++i) tot += p[i];
    double acc = 0.0;
    int idx = 0;
    for (int i = 0; i < n; ++i) {       // cdf = cumsum(p) / cdf[-1]; searchsorted(u, side='right')
        acc += p[i];
        if (acc / tot <= u) idx = i + 1;
    }
    return idx < n ? idx : n - 1;
}

// segment header of sample_controls_piecewise (generation_type2.py:105-131)
__device__ void tg_t2_new_segment(Type2Thread &s, const tg_type2_rules &r, unsigned long long key, double v, double Ts)
{
    uint32_t a[4], b4[4];
    tg_ctrl_philox(key, (uint32_t)s.seg, 0x20u, a);
    tg_ctrl_philox(key, (uint32_t)s.seg, 0x21u, b4);
    s.seg += 1;
    double z0, z1;
    tg_box_muller(b4[0], b4[1], z0, z1);
    int mode;
    if (s.prev_mode == 2 || s.prev_mode == 3) mode = tg_choice(tg_u01(a[0]), r.p_after_turn, 2);   // :107-109
    else mode = tg_choice(tg_u01(a[0]), r.p_modes, 4);                                             // :111-112
    int len = (int)rint(tg_uniform(a[1], r.seg_s[0], r.seg_s[1]) / Ts);                            // :114
    if (len < 1) len = 1;
    double d, delta;
    if (mode == 0) {                                                                                // :118-120
        if (v >= r.v_high) mode = 1;
        d = tg_uniform(a[2], r.acc_d_lo, r.d_range[1]);
        delta = 0.0 + r.delta_straight_noise * z0;
    } else if (mode == 1) {                                                                         // :121-122
        d = tg_uniform(a[2], r.cruise_d[0], r.cruise_d[1]);
        delta = 0.0 + r.delta_straight_noise * z0;
    } else {                                                                                        // :123-128
        d = (v > r.v_turn_max) ? tg_uniform(a[2], r.turn_d_fast[0], r.turn_d_fast[1])
                               : tg_uniform(a[2], r.turn_d_slow[0], r.turn_d_slow[1]);
        const double mag = tg_uniform(a[3], r.delta_turn_range[0], r.delta_turn_range[1]);
        const double scale = fmin(1.0, r.v_turn_max / fmax(v, 1e-3));
        delta = (mode == 2 ? mag : -mag) * scale;
    }
    if (v < r.stall_v) {                                                                            // :131-133
        mode = 0;
        d = tg_uniform(b4[2], r.stall_d[0], r.stall_d[1]);
        delta = 0.0 + r.delta_straight_noise * z1;
        const int mn = (int)rint(r.stall_min_s / Ts);
        if (len < mn) len = mn;
    }
    s.mode = mode; s.left = len; s.d = d; s.delta = delta;
}

// one step of the fill loop (generation_type2.py:136-149)
__device__ __forceinline__ void tg_t2_control(Type2Thread &s, const tg_type2_rules &r, unsigned long long key, const double x[6],
                                              double Ts, double &d_cmd, double &delta_cmd)
{
    const double v = hypot(x[3], x[4]);
    if (s.left == 0) {
        s.prev_mode = s.mode;
        tg_t2_new_segment(s, r, key, v, Ts);
    }
    if (v < r.v_floor) s.d = fmax(s.d, r.d_boost_min);
    d_cmd = tg_clamp(s.d, r.d_range[0], r.d_range[1]);
    double dk = tg_clamp(s.delta, -r.delta_clip, r.delta_clip);
    const double step = r.delta_rate_max * Ts;
    dk = tg_clamp(dk, s.prev_delta - step, s.prev_delta + step);
    s.prev_delta = dk;
    delta_cmd = dk;
    s.left -= 1;
}

// ------------------------------------------------------------------------------------------------ fused kernel
struct OpenLoopArgs {
    int B, T;
    const double *x0;
    long long traj_id0;
    unsigned long long ctrl_seed_base;
    double *clean, *noisy, *U;
    signed char *modes;      // type 1: [B]; type 2: [B][T]; may be null
    const double *plant;     // [B][TG_NPARAMS] per-trajectory plant parameters, read by the PT instances only; null = c.p
};

// cooperative write-out of rows [r0, r0 + TG_OL_CHUNK) of the warp's 32 trajectories (b0 = first trajectory)
__device__ __forceinline__ void tg_ol_flush(const DevCfg &c, const OpenLoopArgs &a, const double *tile, int b0, int r0, int lane)
{
    const int T = a.T;
    constexpr int PAIRS = TG_OL_CHUNK * 3;
    for (int f = lane; f < 32 * PAIRS; f += 32) {
        const int j = f / PAIRS, q = f - j * PAIRS, r = q / 3, cp = q - 3 * r;
        const int b = b0 + j, row = r0 + r;
        if (b >= a.B || row > T) continue;
        const double v0 = tile[(r * 8 + 2 * cp) * TG_OL_STRIDE + j], v1 = tile[(r * 8 + 2 * cp + 1) * TG_OL_STRIDE + j];
        const size_t o = ((size_t)b * (T + 1) + row) * 6 + 2 * cp;
        if (a.clean) *reinterpret_cast<double2 *>(a.clean + o) = make_double2(v0, v1);
        if (a.noisy) {
            const unsigned long long seed = c.seed_base + (unsigned long long)(a.traj_id0 + b);
            uint32_t r4[4];
            tg_philox4x32_10((uint32_t)row, (uint32_t)(cp >> 1), 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r4);
            double n0, n1;
            tg_box_muller(r4[(cp & 1) * 2], r4[(cp & 1) * 2 + 1], n0, n1);
            *reinterpret_cast<double2 *>(a.noisy + o) = make_double2(v0 + c.noise_std[2 * cp] * n0, v1 + c.noise_std[2 * cp + 1] * n1);
        }
    }
    if (a.U) {
        for (int f = lane; f < 32 * TG_OL_CHUNK; f += 32) {
            const int j = f / TG_OL_CHUNK, r = f - j * TG_OL_CHUNK;
            const int b = b0 + j, row = r0 + r;
            if (b >= a.B || row >= T) continue;
            *reinterpret_cast<double2 *>(a.U + ((size_t)b * T + row) * 2) =
                make_double2(tile[(r * 8 + 6) * TG_OL_STRIDE + j], tile[(r * 8 + 7) * TG_OL_STRIDE + j]);
        }
    }
}

// KIND 1 = generation_type1, 2 = generation_type2.  PT = true: trajectory b integrates its plant with the row a.plant[b]
// (read from global memory at every step; L1 keeps it) and the tables tg_plant_row_tables gives it.  PT = false reads the
// handle's parameters from the constant bank, as the kernel did before plant tables existed (DESIGN.md section 3).
template <int KIND, typename Rules, bool PT = false>
__global__ void __launch_bounds__(32 * TG_OL_WARPS) tg_openloop_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ Rules rules,
                                                                     const OpenLoopArgs a)
{
    extern __shared__ double ol_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *tile = ol_smem + warp * TG_OL_TILE;
    const int T = a.T;
    const int b0 = (blockIdx.x * TG_OL_WARPS + warp) * 32;
    if (b0 >= a.B) return;
    const int b = b0 + lane;
    const bool live = b < a.B;
    const unsigned long long key = a.ctrl_seed_base + (unsigned long long)(a.traj_id0 + (live ? b : b0));
    double x[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = a.x0[6 * (size_t)(live ? b : b0) + i];
    const double *__restrict__ pv = PT ? a.plant + (size_t)(live ? b : b0) * TG_NPARAMS : nullptr;
    const bool row_tab = PT && tg_plant_row_tables(c, pv);
    Type1Thread s1;
    Type2Thread s2;
    if constexpr (KIND == 1) {
        tg_t1_setup(s1, rules, key, T, c.Ts);
        if (live && a.modes) a.modes[b] = (signed char)s1.sinusoid;
    } else {
        s2.seg = 0; s2.left = 0; s2.mode = -1; s2.prev_mode = -1; s2.d = 0.0; s2.delta = 0.0; s2.prev_delta = 0.0;
    }
#pragma unroll 1
    for (int r0 = 0; r0 <= T; r0 += TG_OL_CHUNK) {
#pragma unroll 1
        for (int r = 0; r < TG_OL_CHUNK; ++r) {
            const int t = r0 + r;
            if (t > T) break;
            double *col = tile + (r * 8) * TG_OL_STRIDE + lane;
#pragma unroll
            for (int i = 0; i < 6; ++i) col[i * TG_OL_STRIDE] = x[i];
            if (t < T) {
                double d_cmd, delta_cmd;
                if constexpr (KIND == 1) tg_t1_control(s1, rules, key, t, c.Ts, d_cmd, delta_cmd);
                else {
                    tg_t2_control(s2, rules, key, x, c.Ts, d_cmd, delta_cmd);
                    if (live && a.modes) a.modes[(size_t)b * T + t] = (signed char)s2.mode;
                }
                col[6 * TG_OL_STRIDE] = d_cmd;
                col[7 * TG_OL_STRIDE] = delta_cmd;
                if constexpr (PT) {
                    if (c.plant == TG_PLANT_MPC) tg_plant_step(c, pv, x, d_cmd, delta_cmd);
                    else tg_plant_step_gen(c, pv, row_tab ? c.tyre_tab : nullptr, row_tab ? c.atan_tab : nullptr, x, d_cmd, delta_cmd);
                } else {
                    if (c.plant == TG_PLANT_MPC) tg_plant_step(c, c.p, x, d_cmd, delta_cmd);
                    else tg_plant_step_gen(c, c.p, c.tyre_tab, c.atan_tab, x, d_cmd, delta_cmd);
                }
            }
        }
        __syncwarp();
        tg_ol_flush(c, a, tile, b0, r0, lane);
        __syncwarp();
    }
}
