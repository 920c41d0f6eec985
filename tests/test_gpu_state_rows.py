"""GPU (-m gpu): the state-bound rows (x_lo / x_hi) on every solver shape against the condensed reference (oracle/condensed.py).

The solver has five shapes (tw_shape: W warps, S tiles): W1 S1 for N <= 14, W2 S1 for 15-20, W4 S1 for 21-30, W8 S1 for 31-44
and W8 S2 for 45-56, each with its own condensing batch (tw_kb) and its own state-row products.  The horizons below are the
edges of every shape, plus 10, 20, 40 and 50, which run the run-time instances through jacobian=JAC_FD (the compile-time
instances serve the analytic Jacobian only).  JAC_FD linearises as the oracle does (to ~1e-9), so the QP data can be compared
exactly.  Checked here:

  a. the assembled QP (tg_assemble) equals the condensed reference row by row;
  b. every answer of tg_mpc_step is what its status claims: an optimal one passes the KKT certificate of the reference's QP
     within the bounds of the kernel's stopping rule and has the interior-point objective; an infeasible one is infeasible by
     the LP margin s*; no verdict contradicts s*;
  c. the same with a table of per-problem settings (ctrl instances) on all five shapes;
  d. TRAJGEN_PPC (problems per CTA) does not change the bits of closed loops with state rows;
  e. one closed loop per shape follows the oracle's closed loop.

An answer is never compared with the reference's active set or its U* unless the solve is certified: near-degenerate
problems have several active sets within the tolerance, and verdicts near s* = 0 are not decisive."""
import multiprocessing as mp
import os

import numpy as np
import pytest

import trajectory_generation_b200 as tg
from trajectory_generation_b200 import _lib
from oracle import condensed as oc, mpc as ompc, refgen as R
from conftest import HARD

pytestmark = pytest.mark.gpu

TS = 0.02
INF = _lib.TG_INF
TIGHT = {"eps_abs": 1e-6, "eps_rel": 1e-6}
TOL_LIN = 1e-6        # the analytic linearisation's tolerance against the oracle (test_gpu_parity.py)
TOL_QP = 1e-9         # JAC_FD: the assembled QP against the reference, relative to the largest entry of each array
# the dual of a row strictly inside its bounds is zero up to the rounding of the projection, y (1 - rho / rho) + rho ulp(z):
# at most ~1e-12, times a distance of a few units to the bound
COMP_ROUND = 1e-10
SMEM_OPTIN = 227 * 1024   # B200: opt-in shared memory of one CTA
BLAS_THREADS = ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS")
SIX_LO = [-20.0, -5.0, -1.5, 0.2, -0.15, -2.0]    # all six states bounded; only vy / omega are near their bounds
SIX_HI = [20.0, 5.0, 1.5, 3.0, 0.15, 2.0]
DU_TIGHT = ((-0.1, -0.04), (0.1, 0.04))           # conftest.HARD's rate limits as (lo, hi)
DU_LOOSE = ((-0.5, -0.3), (0.5, 0.3))             # mpc_step's default

HORIZONS = [7, 13, 16, 19, 21, 30, 31, 44, 45, 56, 10, 20, 40, 50]
CASES = [(N, "vy_omega") for N in HORIZONS] + [(44, "six"), (56, "six")]
IDS = [f"N{N}-{k}" for N, k in CASES]
B_SOLVE, B_TAP, N_OUTSIDE = 64, 16, 8


def _box(kind):
    return (HARD["x_lo"], HARD["x_hi"]) if kind == "vy_omega" else (SIX_LO, SIX_HI)


def _handle_kw(kind, tight, **kw):
    lo, hi = _box(kind)
    du = DU_TIGHT if tight else DU_LOOSE
    return dict(Ts=TS, jacobian=tg.JAC_FD, x_lo=lo, x_hi=hi, du_bounds=tuple(zip(*du)), **kw)


def _settings(kind, tight):
    lo, hi = _box(kind)
    du = DU_TIGHT if tight else DU_LOOSE
    return dict(x_lo=lo, x_hi=hi, du_lo=du[0], du_hi=du[1])


@pytest.fixture(scope="module")
def pool():
    # one BLAS thread per worker: the reference's matrices are small, and a worker per core with a BLAS thread pool each would
    # oversubscribe the CPUs many times over (the spawned workers read these variables when they start)
    saved = {k: os.environ.get(k) for k in BLAS_THREADS}
    os.environ.update({k: "1" for k in BLAS_THREADS})
    try:
        p = mp.get_context("spawn").Pool(min(16, os.cpu_count() or 1))
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    with p:
        yield p


# ------------------------------------------------------------------------------------------------ reference jobs (pool)
def _reference_job(x0, u0, pr, vr, N, settings, bounded):
    """the condensed QP of one problem (the parts the checks read), its feasibility margin s*, and the interior-point optimum
    where s* = 0"""
    c = oc.condense(x0, u0, pr, vr, TS, N, bounded=bounded, **settings)
    r = dict(H=c.H, q=c.q, c0=c.c0, l=c.l, u=c.u, Gs=c.Gs, s=oc.feasibility_margin(*c.with_k0_rows()))
    if r["s"] == 0.0:
        o = oc.exact_optimum(c)
        r.update(ipm_status=o["status"], ipm_obj=o["objective"], ipm_dU=o["dU"], ipm_y=o["y"])
    return r


def _constraint_matrix(ref):
    """A = [I; D; Gs] of a reference (condense's row order)"""
    n = ref["H"].shape[0]
    return np.vstack([np.eye(n), np.eye(n) - np.eye(n, k=-2), ref["Gs"]])


def _loop_job(x0, u0, T, N):
    X, U, st, _ = ompc.closed_loop(x0, u0, T, TS, N, path_kind=R.PATH_SINE, path_prm=(0.5, 0.5, 0.0, 0.0), **HARD)
    return X, U, st


# ------------------------------------------------------------------------------------------------ problems
def _problems(N, B, seed, vy_box=0.15, om_box=2.0):
    """lateral offsets up to 1.5 m, vy and omega started near their bounds (at least 1e-3 inside, the kernel decides the
    k = 0 rows by itself), steering that pushes vy further; the last N_OUTSIDE problems start with vy outside its box"""
    rng = np.random.default_rng(seed)
    x0 = np.zeros((B, 6))
    x0[:, 1] = rng.uniform(-1.5, 1.5, B)
    x0[:, 2] = rng.uniform(-0.1, 0.1, B)
    x0[:, 3] = rng.uniform(0.8, 1.2, B)
    sv, so = rng.choice([-1.0, 1.0], B), rng.choice([-1.0, 1.0], B)
    x0[:, 4] = sv * rng.uniform(0.667, 0.99, B) * vy_box
    x0[:, 5] = so * rng.uniform(0.6, 0.999, B) * om_box
    out = np.arange(B) >= B - N_OUTSIDE
    x0[out, 4] = sv[out] * (vy_box + rng.uniform(2e-3, 2e-2, out.sum()))
    u0 = np.stack([tg.d_steady_state(x0[:, 3]), sv * rng.uniform(0.05, 0.2, B)], 1)
    sc = tg.Scenarios(B)
    sc.set_sine(slice(0, B), rng.uniform(0.3, 0.7, B), 0.5, 0.0, 0.0)
    return x0, u0, sc


_REF = {}


def _reference(N, kind, pool):
    """the problems of (N, kind) and their condensed references (one per problem, kept for the module)"""
    if (N, kind) not in _REF:
        x0, u0, sc = _problems(N, B_SOLVE, seed=1000 + N + (7 if kind == "six" else 0))
        tight = np.arange(B_SOLVE) % 2 == 0
        gen = tg.ClosedLoopGenerator(N=N, Ts=TS, jacobian=tg.JAC_FD, x_lo=_box(kind)[0], x_hi=_box(kind)[1])
        pr, vr = gen.ref_window(x0, sc)
        bounded = gen.bounded_states
        jobs = [(x0[i], u0[i], pr[i], vr[i], N, _settings(kind, tight[i]), bounded) for i in range(B_SOLVE)]
        _REF[(N, kind)] = dict(x0=x0, u0=u0, pr=pr, vr=vr, tight=tight, refs=pool.starmap(_reference_job, jobs))
    return _REF[(N, kind)]


def _create_or_refuse(N, kind, **kw):
    """the handle, or None where six bounded states at N = 56 exceed the shared memory of a CTA: tg_create must then refuse
    it, naming the shared memory"""
    try:
        return tg.BatchedMPC(N=N, **kw)
    except tg.TrajgenError as e:
        assert kind == "six" and N == 56 and "shared memory" in str(e), (N, kind, str(e))
        print(f"N={N} {kind}: tg_create refuses the handle: {e}")
        return None


# ------------------------------------------------------------------------------------------------ a. taps
def _compare_qp(asm, i, ref, tol):
    """worst error of the assembled QP of problem i against its reference, in units of the tolerance: H relative to max|H|,
    q and Gs relative to 1 + their largest entry (the finite differences of the linearisation round relative to the
    magnitude of f, and the condensed rows multiply the stages together), l and u absolute, c0 through the objective at
    random points"""
    n = ref["H"].shape[0]
    e = {"H": np.abs(asm["H"][i] - ref["H"]).max() / np.abs(ref["H"]).max(),
         "q": np.abs(asm["q"][i] - ref["q"]).max() / (1.0 + np.abs(ref["q"]).max())}
    for f in ("l", "u"):
        got, want = asm[f][i], ref[f]
        absent = np.abs(want) >= INF
        assert np.array_equal(np.abs(got) >= INF, absent) and np.array_equal(got[absent], want[absent]), f
        e[f] = np.abs(got[~absent] - want[~absent]).max()
    e["Gs"] = np.abs(asm["Gs"][i] - ref["Gs"]).max() / (1.0 + np.abs(ref["Gs"]).max()) if ref["Gs"].size else 0.0
    rng = np.random.default_rng(i)
    for _ in range(2):
        dU = rng.normal(0, 0.1, n)
        obj = 0.5 * dU @ ref["H"] @ dU + ref["q"] @ dU + ref["c0"]
        got = 0.5 * dU @ asm["H"][i] @ dU + asm["q"][i] @ dU + asm["c0"][i]
        e["c0"] = max(e.get("c0", 0.0), abs(got - obj) / (1.0 + abs(obj)))
    return {k: v / tol for k, v in e.items()}


@pytest.mark.parametrize("N,kind", CASES, ids=IDS)
def test_assembled_qp_equals_the_condensed_reference(N, kind, pool):
    m = {t: _create_or_refuse(N, kind, **_handle_kw(kind, t)) for t in (True, False)}
    if m[True] is None:
        return
    ref = _reference(N, kind, pool)
    assert m[True].ms == ref["refs"][0]["Gs"].shape[0]
    idx = np.arange(B_TAP)
    worst = {}
    for t, h in m.items():
        rows = idx[ref["tight"][idx] == t]
        asm = h.assemble(ref["x0"][rows], ref["u0"][rows], ref["pr"][rows], ref["vr"][rows])
        for j, i in enumerate(rows):
            for k, v in _compare_qp(asm, j, ref["refs"][i], TOL_QP).items():
                worst[k] = max(worst.get(k, 0.0), v)
    print(f"N={N} {kind}: worst tap error / tolerance 1e-9: " + " ".join(f"{k} {v:.3f}" for k, v in worst.items()))
    assert max(worst.values()) <= 1.0, worst
    if kind == "vy_omega" and N in (10, 20, 50):
        # the compile-time instance with state rows (analytic Jacobian from the tyre / atan tables): linearisation error
        # TOL_LIN per stage, accumulated over the N stages that a condensed row multiplies together
        h = tg.BatchedMPC(N=N, Ts=TS, x_lo=HARD["x_lo"], x_hi=HARD["x_hi"], du_bounds=HARD["du_bounds"])
        rows = idx[ref["tight"][idx]]
        asm = h.assemble(ref["x0"][rows], ref["u0"][rows], ref["pr"][rows], ref["vr"][rows])
        wa = {}
        for j, i in enumerate(rows):
            r = ref["refs"][i]
            scale = {"H": 1.0, "q": 1.0, "l": 1 + np.abs(r["l"][np.abs(r["l"]) < INF]).max(),
                     "u": 1 + np.abs(r["u"][np.abs(r["u"]) < INF]).max(), "Gs": 1.0, "c0": 1.0}
            for k, v in _compare_qp(asm, j, r, TOL_LIN * N).items():
                wa[k] = max(wa.get(k, 0.0), v / scale[k])
        print(f"N={N} analytic compile-time instance: worst error / (N TOL_LIN scale): " + " ".join(f"{k} {v:.3f}" for k, v in wa.items()))
        assert max(wa.values()) <= 1.0, wa


# ------------------------------------------------------------------------------------------------ b. solves
def _judge(label, refs, out):
    """the checks of every answer in ``out`` (BatchedMPC.step, plus u0) against its reference (see the module docstring);
    returns the summary counts"""
    cnt = dict(optimal=0, inaccurate=0, active=0, infeasible=0, user_limit=0, other=0)
    worst, worst_obj, beyond = 0.0, 0.0, 0
    for i, r in enumerate(refs):
        st, s = int(out["status"][i]), r["s"]
        y = out["y_opt"][i]
        # no verdict contradicts the feasibility margin
        assert not (s > 1e-4 and st in (0, 1)), (label, i, st, s)
        assert not (s == 0.0 and st == 2), (label, i, st, s)
        if st not in (0, 1):   # rows that are not accepted carry NaN
            assert np.isnan(out["U_opt"][i]).all() and np.isnan(y).all(), (label, i)
        if st in (0, 1):
            dU = (out["U_opt"][i] - out["u0"][i][None, :]).reshape(-1)
            n = len(dU)
            c = oc.kkt_certificate(r["H"], r["q"], _constraint_matrix(r), r["l"], r["u"], dU, y, TIGHT["eps_abs"], TIGHT["eps_rel"])
            f = 1.0 if st == 0 else 10.0
            # the tolerance of the QP data (TOL_QP, test a) carried through the residuals
            n1, gmax = np.abs(dU).sum(), 1.0 + (np.abs(r["Gs"]).max() if r["Gs"].size else 0.0)
            dp = TOL_QP * gmax * n1
            dd = TOL_QP * (np.abs(r["H"]).max() * n1 + 1.0 + np.abs(r["q"]).max() + gmax * np.abs(y).sum())
            ratios = (c["primal"] / (f * c["eps_p"] + dp), c["stationarity"] / (f * c["eps_d"] + dd),
                      c["complementarity"] / (f * c["comp_bound"] + dp * np.abs(y).max() + COMP_ROUND))
            worst = max(worst, *ratios)
            assert max(ratios) <= 1.0, (label, i, st, c)
            assert s <= f * c["eps_p"] + dp, (label, i, s, c["eps_p"])
            # the reported objective is the reference objective at the returned point.  The kernel forms H x from its
            # factorisation (rhs - sigma x - A'(rho A x)), which differs from H x by the solve's residual; both its own and the
            # reference's stationarity residuals are within the bound, so that difference is at most 2 eps_d + dd per entry
            f_ref = 0.5 * dU @ r["H"] @ dU + r["q"] @ dU + r["c0"]
            obj = out["objective"][i]
            assert abs(obj - f_ref) <= 1e-9 * (1 + abs(f_ref)) + 0.5 * n1 * (2 * f * c["eps_d"] + dd), (label, i, obj, f_ref)
            if "ipm_status" in r:
                assert r["ipm_status"] == "optimal", (label, i, r["ipm_status"])
                # an eps-KKT point is eps-optimal: with r = H x + q + A'y and the stopping rule's bounds,
                #   f(x) - f* <= ||r|| ||x - x*||_1 + ||y||_1 eps_p   and   f* - f(x) <= ||y*||_1 eps_p,
                # which many active state rows with duals of order one make larger than 1e-5 (1 + |f*|)
                gap = f * (c["eps_d"] + dd) * np.abs(dU - r["ipm_dU"]).sum() \
                    + max(np.abs(y).sum(), np.abs(r["ipm_y"]).sum()) * (f * c["eps_p"] + dp)
                tol_obj = 1e-5 * (1 + abs(r["ipm_obj"]))
                err = abs(obj - r["ipm_obj"])
                assert err <= tol_obj + gap, (label, i, obj, r["ipm_obj"], gap)
                worst_obj = max(worst_obj, err / (tol_obj + gap))
                beyond += int(err > tol_obj)
            cnt["optimal" if st == 0 else "inaccurate"] += 1
            cnt["active"] += int(st == 0 and (np.abs(y[2 * n:]) > 1e-6).any())
        elif st == 2:
            assert s > 1e-7, (label, i, s)
            cnt["infeasible"] += 1
        elif st == 4:
            cnt["user_limit"] += 1
        else:
            cnt["other"] += 1
    print(f"{label}: worst certificate residual / bound {worst:.3g}; worst objective error / bound {worst_obj:.3g} "
          f"({beyond} beyond 1e-5 (1 + |f*|)); " + ", ".join(f"{k} {v}" for k, v in cnt.items()))
    return cnt


@pytest.mark.parametrize("N,kind", CASES, ids=IDS)
def test_every_answer_is_what_its_status_claims(N, kind, pool):
    m = {t: _create_or_refuse(N, kind, solver_opts=TIGHT, **_handle_kw(kind, t)) for t in (True, False)}
    if m[True] is None:
        return
    ref = _reference(N, kind, pool)
    out = {}
    for t, h in m.items():
        o = h.step(ref["x0"], ref["u0"], ref["pr"], ref["vr"])
        for k, v in o.items():
            out.setdefault(k, v.copy())[ref["tight"] == t] = v[ref["tight"] == t]
    out["u0"] = ref["u0"]
    cnt = _judge(f"N={N} {kind}", ref["refs"], out)
    # coverage: the inputs must keep the state rows active and reach the infeasible verdict
    assert cnt["active"] >= 8 and cnt["infeasible"] >= 1, cnt


# ------------------------------------------------------------------------------------------------ c. per-problem settings
CTRL_SETTINGS = [   # (q_c, q_phi, q_vx, R, Rd, vy box, omega box); the last drops the box
    (6.0, 0.5, 0.5, [0.02, 0.0, 0.0, 2.0], [0.01, 0.0, 0.0, 5.0], 0.15, 2.0),
    (2.0, 1.5, 0.2, [0.05, 0.01, 0.01, 1.0], [0.02, 0.0, 0.0, 2.0], 0.10, 1.0),
    (12.0, 0.3, 1.0, [0.01, 0.0, 0.0, 4.0], [0.005, 0.001, 0.001, 8.0], 0.20, 1.5),
    (4.0, 0.8, 0.5, [0.03, -0.02, 0.0, 0.5], [0.0, 0.0, 0.0, 1.0], None, None),
]


@pytest.mark.parametrize("N", [13, 16, 30, 44, 56])
def test_per_problem_settings_on_every_shape(N, pool):
    B = B_SOLVE
    which = np.arange(B) % 4
    vyb = np.array([CTRL_SETTINGS[k][5] or 0.15 for k in which])
    omb = np.array([CTRL_SETTINGS[k][6] or 2.0 for k in which])
    x0, u0, sc = _problems(N, B, seed=2000 + N)
    # near (or, for the last rows, outside) each row's own box
    x0[:, 4] = x0[:, 4] / 0.15 * vyb
    x0[:, 4] = np.where(np.arange(B) >= B - N_OUTSIDE, np.sign(x0[:, 4]) * (vyb + 5e-3), x0[:, 4])
    x0[:, 5] = x0[:, 5] / 2.0 * omb
    m = tg.BatchedMPC(N=N, solver_opts=TIGHT, **_handle_kw("vy_omega", True))
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS, jacobian=tg.JAC_FD)
    pr, vr = gen.ref_window(x0, sc)
    f = {k: np.array([CTRL_SETTINGS[w][j] for w in which], float) for j, k in enumerate(("q_c", "q_phi", "q_vx"))}
    f["R"] = np.array([CTRL_SETTINGS[w][3] for w in which]); f["Rd"] = np.array([CTRL_SETTINGS[w][4] for w in which])
    xl, xh = np.full((B, 6), -INF), np.full((B, 6), INF)
    boxed = which != 3
    xl[boxed, 4], xh[boxed, 4], xl[boxed, 5], xh[boxed, 5] = -vyb[boxed], vyb[boxed], -omb[boxed], omb[boxed]
    du = np.where((np.arange(B) // 4 % 2 == 0)[:, None, None], np.array(DU_TIGHT), np.array(DU_LOOSE))   # [B, lo/hi, 2]
    tab = m.ctrl_table(B, x_lo=xl, x_hi=xh, du_lo=du[:, 0], du_hi=du[:, 1], **f)
    out = m.step(x0, u0, pr, vr, ctrl=tab)
    out["u0"] = u0
    jobs = [(x0[i], u0[i], pr[i], vr[i], N,
             dict(q_c=f["q_c"][i], q_phi=f["q_phi"][i], q_vx=f["q_vx"][i], R=f["R"][i], Rd=f["Rd"][i], x_lo=xl[i], x_hi=xh[i],
                  du_lo=du[i, 0], du_hi=du[i, 1]), m.bounded_states) for i in range(B)]
    cnt = _judge(f"N={N} ctrl table", pool.starmap(_reference_job, jobs), out)
    assert cnt["active"] >= 8 and cnt["infeasible"] >= 1, cnt
    # the rows without a box: x0 outside the other rows' boxes is no reason to refuse them, and their state duals stay zero
    free = np.nonzero(which == 3)[0]
    assert np.isin(out["status"][free], (0, 1)).all(), out["status"][free]
    assert (out["y_opt"][free][:, 4 * N:] == 0.0).all()


# ------------------------------------------------------------------------------------------------ d. problems per CTA
def _ppc_max(h):
    """tg_create's limit on problems per CTA (make_tw_launch): threads of the CTA, barrier ids, shared memory"""
    W = h.info()["threads_per_cta"] // 32
    p = 512 // (32 * W)
    if W > 1:
        p = min(p, 14)
    while p > 1 and p * h.info()["smem_bytes"] > SMEM_OPTIN:
        p -= 1
    return p


@pytest.mark.parametrize("N", [7, 16, 30, 31, 44, 45, 56])
def test_problems_per_cta_keep_the_bits(N, monkeypatch):
    """TRAJGEN_PPC is read in tg_create; 2 and 4 problems per CTA where the shared memory allows them (a larger value is
    ignored and the problems run one per CTA)"""
    B, T = 40, 15
    x0, u0, sc = _problems(N, B, seed=3000 + N)
    kw = _handle_kw("vy_omega", True)
    monkeypatch.delenv("TRAJGEN_PPC", raising=False)
    g1 = tg.ClosedLoopGenerator(N=N, **kw)
    ref = g1.generate(x0, u0, sc, T)
    pmax = _ppc_max(g1)
    assert ref["status_counts"][:, 0].sum() > 0 and ref["status_counts"][:, 2].sum() > 0
    ran = []
    for ppc in (2, 4):
        monkeypatch.setenv("TRAJGEN_PPC", str(ppc))
        alt = tg.ClosedLoopGenerator(N=N, **kw).generate(x0, u0, sc, T)
        monkeypatch.delenv("TRAJGEN_PPC")
        for k in ("clean", "U", "status_counts", "iters_total"):
            np.testing.assert_array_equal(ref[k], alt[k], err_msg=f"N={N} ppc={ppc} {k}")
        ran.append(ppc if ppc <= pmax else None)
    print(f"N={N}: ppc_max {pmax}, problems per CTA compared with 1: {[p for p in ran if p]}")
    if N not in (44, 56):
        assert ran[0] == 2, pmax          # at least two problems per CTA were really exercised


# ------------------------------------------------------------------------------------------------ e. closed loop
@pytest.mark.parametrize("N", [13, 19, 21, 44, 56])
def test_closed_loop_follows_the_oracle(N, pool):
    """one closed loop per shape with the vy / omega box: candidates whose oracle loop is optimal at every step must match it
    to 1e-3, and at least one of them has the box active"""
    K, T = 8, 8
    rng = np.random.default_rng(4000 + N)
    x0 = np.zeros((K, 6))
    s = np.where(np.arange(K) % 2 == 0, 1.0, -1.0)
    x0[:, 1] = -s * rng.uniform(0.5, 1.5, K)
    x0[:, 3] = rng.uniform(0.9, 1.1, K)
    x0[:, 4] = s * rng.uniform(0.08, 0.14, K)
    x0[:, 5] = s * rng.uniform(0.5, 1.8, K)
    u0 = np.stack([tg.d_steady_state(x0[:, 3]), s * rng.uniform(0.0, 0.08, K)], 1)
    sc = tg.Scenarios(K)
    sc.set_sine(slice(0, K), 0.5, 0.5, 0.0, 0.0)
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS, jacobian=tg.JAC_FD, **HARD)
    res = gen.generate(x0, u0, sc, T)
    loops = pool.starmap(_loop_job, [(x0[i], u0[i], T, N) for i in range(K)])
    # the box's activity along each GPU loop: the step API at the visited states
    m = tg.BatchedMPC(N=N, Ts=TS, jacobian=tg.JAC_FD, **HARD)
    xs = res["clean"][:, :T].reshape(-1, 6)
    us = np.concatenate([u0[:, None, :], res["U"][:, :T - 1]], 1).reshape(-1, 2)
    pr, vr = gen.ref_window(xs, tg.Scenarios.from_arrays(np.repeat(sc.spec["path_kind"], T), np.repeat(sc.spec["path"], T, 0),
                                                         np.repeat(sc.spec["vref"], T, 0)))
    st = m.step(xs, us, pr, vr)
    active = (np.abs(np.nan_to_num(st["y_opt"][:, 4 * N:])) > 1e-6).any(1).reshape(K, T).any(1)
    compared, with_box = 0, 0
    for i, (Xo, Uo, sto) in enumerate(loops):
        if not all(v == "optimal" for v in sto):
            continue
        assert res["status_counts"][i, :2].sum() == T, (i, res["status_counts"][i])
        assert np.abs(res["clean"][i] - Xo).max() < 1e-3 and np.abs(res["U"][i] - Uo).max() < 1e-3, i
        compared += 1
        with_box += int(active[i])
    print(f"N={N}: {compared} of {K} closed loops compared with the oracle, {with_box} of them with the box active")
    assert with_box >= 1, (compared, active)
