"""Oracle: the condensed QP of one MPC step in dU = U - u_prev, and certificates for a claimed solution of it (fp64).

Test infrastructure -- see ``oracle/__init__.py``.  The kernels never form the sparse problem of MPC/mpc_6stati.py:180-250:
they condense it (tw_solver.cuh, K2) into

    min 1/2 dU'H dU + q'dU + c0   s.t.   l <= A dU <= u,   A = [I ; D ; Gs]

with the rows in the kernel's order: the 2N input boxes (stage-major, two per stage), the 2N rate rows, then ns rows per
stage for the states x_1 .. x_N (ns = the bounded state components, in index order).  The k = 0 state rows do not depend on
dU; the kernel decides them before its iteration (x0 outside its box means "infeasible"), so they are kept apart here.

``condense`` derives all of it from the sparse statement (``oracle.qp.build_sparse_qp`` on
``oracle.dynamics.linearize_horizon``) by eliminating the states through the equality rows -- generic linear algebra that
shares no code or ordering rule with the kernels.  ``kkt_certificate`` measures how far a claimed (dU, y) is from a KKT point
and states the bounds the kernel's stopping rule promises; ``feasibility_margin`` decides feasibility by a linear program
(HiGHS); ``exact_optimum`` is the interior-point optimum of the sparse problem, with its duals in the condensed row order.
"""
import numpy as np
from scipy.optimize import linprog

from . import dynamics as dyn
from . import qp as oqp

INF = oqp.INF   # TG_INF: a bound at or beyond it is absent


class CondensedQP:
    """H[n,n], q[n], c0, A[m,n] = [I; D; Gs], l[m], u[m], Gs[ms,n]; k0_l / k0_u[ns]: the k = 0 state rows as bounds on 0
    (x_lo - x0, x_hi - x0); sidx: the bounded state components; sparse: the SparseQP it was condensed from; M, z0: the sparse
    variables z = M dU + z0 that satisfy the equality rows; u_prev; ysel: sparse inequality row of each condensed row (-1:
    not present in the sparse problem, i.e. a state row whose two bounds are absent)."""

    def objective(self, dU):
        dU = np.asarray(dU, float).reshape(-1)
        return 0.5 * dU @ self.H @ dU + self.q @ dU + self.c0

    def sparse_point(self, dU):
        return self.M @ np.asarray(dU, float).reshape(-1) + self.z0

    def with_k0_rows(self):
        """(A, l, u) with the k = 0 state rows appended as zero rows: what ``feasibility_margin`` needs"""
        ns = len(self.sidx)
        return (np.vstack([self.A, np.zeros((ns, self.A.shape[1]))]), np.concatenate([self.l, self.k0_l]),
                np.concatenate([self.u, self.k0_u]))


def _pair(v, default):
    return np.asarray(default if v is None else v, float).reshape(2)


def condense(x0, u_prev, path_ref, vref, Ts, N, q_c=6.0, q_phi=0.5, q_vx=0.5, R=None, Rd=None, u_lo=None, u_hi=None,
             du_lo=None, du_hi=None, x_lo=None, x_hi=None, bounded=None, params=None, variant=dyn.VARIANT_MPC):
    """The condensed QP of mpc_step's problem at (x0, u_prev, path_ref[N+1,3], vref[N+1]) with the settings of one
    tg_ctrl_spec row (same field names; R, Rd as 2x2 or 4 row-major entries; None = mpc_step's default).  ``bounded[6]``:
    the state components that carry rows (a handle's bounded_states); default: those with a finite bound.  A component
    that carries rows but whose two bounds are absent gives rows with l = -INF, u = INF, as a ctrl row that drops its box."""
    p = dict(dyn.PARAMS)
    if params is not None:
        p.update(params)
    x0 = np.asarray(x0, float).reshape(6)
    up = np.asarray(u_prev, float).reshape(2)
    R = None if R is None else np.asarray(R, float).reshape(2, 2)
    Rd = None if Rd is None else np.asarray(Rd, float).reshape(2, 2)
    ulo, uhi = _pair(u_lo, (-1.0, -0.6)), _pair(u_hi, (1.0, 0.6))
    dlo, dhi = _pair(du_lo, (-0.5, -0.3)), _pair(du_hi, (0.5, 0.3))
    xl = np.full(6, -INF) if x_lo is None else np.maximum(np.asarray(x_lo, float).reshape(6), -INF)
    xh = np.full(6, INF) if x_hi is None else np.minimum(np.asarray(x_hi, float).reshape(6), INF)
    has = (xl > -INF) | (xh < INF)
    bounded = has if bounded is None else np.asarray(bounded, bool).reshape(6)
    if np.any(has & ~bounded):
        raise ValueError("a finite state bound on a component without rows")
    sidx = np.nonzero(bounded)[0]
    ns, n = len(sidx), 2 * N

    A_, B_, g_, _ = dyn.linearize_horizon(x0, up, Ts, N, p, variant)
    sparse = oqp.build_sparse_qp(x0, up, A_, B_, g_, np.asarray(path_ref, float), np.asarray(vref, float), q_c, q_phi, q_vx,
                                 R, Rd, tuple(zip(ulo, uhi)), tuple(zip(dlo, dhi)),
                                 xl if has.any() else None, xh if has.any() else None)
    # eliminate the states: E z = b with z = [X; U], U = u_prev + dU  ->  X = Ex^-1 (b - Eu U)
    nx = 6 * (N + 1)
    E, b = sparse.A[:sparse.n_eq], sparse.l[:sparse.n_eq]
    Ex, Eu = E[:, :nx], E[:, nx:]
    U0 = np.tile(up, N)
    M = np.vstack([-np.linalg.solve(Ex, Eu), np.eye(n)])
    z0 = np.concatenate([np.linalg.solve(Ex, b - Eu @ U0), U0])

    P, qs = sparse.P, sparse.q
    out = CondensedQP()
    out.H = M.T @ P @ M
    out.H = 0.5 * (out.H + out.H.T)
    out.q = M.T @ (P @ z0 + qs)
    out.c0 = 0.5 * z0 @ P @ z0 + qs @ z0 + sparse.const

    # input boxes and rates: the sparse rows come stage by stage (box j = 0, 1, rate j = 0, 1)
    Ain, lin, uin = sparse.A[sparse.n_eq:], sparse.l[sparse.n_eq:], sparse.u[sparse.n_eq:]
    box = np.array([4 * k + j for k in range(N) for j in range(2)])
    rate = box + 2
    rows = [Ain[box] @ M, Ain[rate] @ M]
    shift = lambda v, r: np.where(v <= -INF, -INF, np.where(v >= INF, INF, v - (Ain[r] @ z0)))
    lo, hi = [shift(lin[box], box), shift(lin[rate], rate)], [shift(uin[box], box), shift(uin[rate], rate)]
    # state rows k = 1 .. N: the rows of M that give x_k[i], bounds shifted by the free response z0
    st = np.array([6 * k + i for k in range(1, N + 1) for i in sidx], int).reshape(-1)
    Gs = M[st] if ns else np.zeros((0, n))
    xl_r, xh_r = np.tile(xl[sidx], N), np.tile(xh[sidx], N)
    rows.append(Gs)
    lo.append(np.where(xl_r <= -INF, -INF, xl_r - z0[st] if ns else xl_r))
    hi.append(np.where(xh_r >= INF, INF, xh_r - z0[st] if ns else xh_r))
    out.A = np.vstack(rows)
    out.l, out.u = np.concatenate(lo), np.concatenate(hi)
    out.Gs = Gs
    out.k0_l = np.where(xl[sidx] <= -INF, -INF, xl[sidx] - x0[sidx])
    out.k0_u = np.where(xh[sidx] >= INF, INF, xh[sidx] - x0[sidx])
    out.sidx, out.sparse, out.M, out.z0, out.u_prev, out.N = sidx, sparse, M, z0, up, N
    # which sparse inequality row each condensed row is (build_sparse_qp lists the state rows k = 0 .. N of the components
    # with a bound, in index order)
    comp = np.nonzero(has)[0]
    pos = {int(i): j for j, i in enumerate(comp)}
    srow = [4 * N + k * len(comp) + pos[int(i)] if int(i) in pos else -1 for k in range(1, N + 1) for i in sidx]
    out.ysel = np.concatenate([box, rate, np.array(srow, int)]).astype(int)
    return out


def kkt_certificate(H, q, A, l, u, dU, y, eps_abs, eps_rel):
    """How far (dU, y) is from a KKT point of  min 1/2 dU'H dU + q'dU  s.t.  l <= A dU <= u  (y > 0 pushes against the
    upper bound, y < 0 against the lower one, OSQP's convention), and what the kernel's stopping rule guarantees.

    The kernel (tw_solver.cuh, step (d)) stops when, at its returned point x~ = dU and dual y,
        ||A x~ - z||  <= eps_p = eps_abs + eps_rel max(||A x~||, ||z||)                     (z: A x~ projected on [l, u])
        ||H x~ + q + A'y|| <= eps_d = eps_abs + eps_rel max(||H x~||, ||A'y||, ||q||)
    (infinity norms), and its projection leaves y > 0 only on rows with z at u and y < 0 only on rows with z at l.  So the
    primal violation is at most eps_p, the stationarity residual at most eps_d, and the complementarity |y_i| times the
    distance from A_i x~ to the bound y_i points at at most ||y|| eps_p.  Returns dict(primal, stationarity,
    complementarity, eps_p, eps_d, comp_bound)."""
    dU, y = np.asarray(dU, float).reshape(-1), np.asarray(y, float).reshape(-1)
    Ax = A @ dU
    lo_ok, hi_ok = l > -INF, u < INF
    viol = np.maximum(np.where(lo_ok, l - Ax, 0.0), np.where(hi_ok, Ax - u, 0.0))
    primal = float(max(viol.max(initial=0.0), 0.0))
    Hx, Aty = H @ dU, A.T @ y
    stat = float(np.abs(Hx + q + Aty).max())
    # complementarity: a dual that points at an absent bound is infinitely wrong
    d_up = np.where(hi_ok, np.abs(u - Ax), np.inf)
    d_lo = np.where(lo_ok, np.abs(Ax - l), np.inf)
    comp_i = np.zeros_like(y)
    comp_i[y > 0] = y[y > 0] * d_up[y > 0]
    comp_i[y < 0] = -y[y < 0] * d_lo[y < 0]
    z = np.clip(Ax, np.where(lo_ok, l, -np.inf), np.where(hi_ok, u, np.inf))
    eps_p = eps_abs + eps_rel * max(np.abs(Ax).max(initial=0.0), np.abs(z).max(initial=0.0))
    eps_d = eps_abs + eps_rel * max(np.abs(Hx).max(), np.abs(Aty).max(initial=0.0), np.abs(q).max())
    return {"primal": primal, "stationarity": stat, "complementarity": float(comp_i.max(initial=0.0)),
            "eps_p": eps_p, "eps_d": eps_d, "comp_bound": eps_p * float(np.abs(y).max(initial=0.0))}


def feasibility_margin(A, l, u):
    """s* = min s >= 0 s.t. l - s <= A dU <= u + s (absent bounds dropped), by HiGHS at tight tolerances.  s* > 0: no dU
    satisfies every row; s* is by how much the least violated choice still misses.  Zero rows stand for rows that do not
    depend on dU (the k = 0 state rows)."""
    A = np.asarray(A, float)
    n = A.shape[1]
    fu, fl = u < INF, l > -INF
    A_ub = np.vstack([np.hstack([A[fu], -np.ones((fu.sum(), 1))]), np.hstack([-A[fl], -np.ones((fl.sum(), 1))])])
    b_ub = np.concatenate([u[fu], -l[fl]])
    c = np.zeros(n + 1); c[-1] = 1.0
    res = linprog(c, A_ub=A_ub, b_ub=b_ub, bounds=[(None, None)] * n + [(0.0, None)], method="highs",
                  options={"primal_feasibility_tolerance": 1e-10, "dual_feasibility_tolerance": 1e-10, "presolve": False})
    if res.status != 0:
        raise RuntimeError(f"feasibility LP: {res.message}")
    return max(float(res.x[-1]), 0.0)


def exact_optimum(cqp, tol=1e-10):
    """``oracle.qp.solve_ipm`` on the sparse problem cqp was condensed from -> dict(status, objective, U[N,2], dU[2N],
    y[m] in the condensed row order (0 on rows the sparse problem does not have)).  The long horizons are ill-conditioned
    (cond(H) ~ 1e11 at N = 50, Ts = 0.02), where the interior-point stopping test at 1e-10 can stall short of it; the
    solve is then repeated at ten times the tolerance, which still fixes the objective to ~1e-9.  An infeasible problem can
    make the method's linear systems singular: that is reported as status "error" (mpc_step's "Solver Error")."""
    try:
        z, y_s, status = oqp.solve_ipm(cqp.sparse, tol=tol)
        if status != "optimal":
            z, y_s, status = oqp.solve_ipm(cqp.sparse, tol=10.0 * tol)
    except (RuntimeError, np.linalg.LinAlgError):
        return {"status": "error", "objective": np.nan, "U": None, "dU": None, "y": None}
    X, U = cqp.sparse.split(z)
    y = np.where(cqp.ysel >= 0, y_s[np.maximum(cqp.ysel, 0)], 0.0)
    return {"status": status, "objective": float(cqp.sparse.objective(z)), "U": U.T.copy(),
            "dU": (U.T - cqp.u_prev[None, :]).reshape(-1), "y": y}
