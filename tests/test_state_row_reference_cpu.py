"""CPU: the condensed reference of the state-bound rows (oracle/condensed.py) can tell a right answer from a wrong one.

It must restate the sparse problem of MPC/mpc_6stati.py:180-250 exactly, accept the exact optimum of a problem whose vy /
omega box is active, reject that optimum after each of three small corruptions (the point moved, one state-row dual with its
sign flipped, the state rows of one stage taken from the next stage), and decide feasibility with a margin.  The horizons are
the edges of the solver's shapes (tw_shape: N <= 14, 20, 30, 44, 56)."""
import numpy as np
import pytest

from oracle import condensed as oc, dynamics as dyn, refgen as R

INF = oc.INF
TS = 0.02
EPS = 1e-6          # the kernels' default eps_abs = eps_rel
# conftest.HARD as tg_ctrl_spec fields: tight rate limits and a box on vy / omega
HARD = dict(du_lo=(-0.1, -0.04), du_hi=(0.1, 0.04), x_lo=[-INF] * 4 + [-0.15, -2.0], x_hi=[INF] * 4 + [0.15, 2.0])
HORIZONS = [7, 16, 30, 44, 56]


def _condensed(N, x, up, **kw):
    v = R.vref_profile(R.VREF_RAMP, (0.8, 2.0, 2.0), N, TS)
    pr = R.ref_window(x[0], N, TS, v, R.PATH_SINE, (0.5, 0.5, 0.0, 0.0))
    return oc.condense(x, up, pr, v, TS, N, **{**HARD, **kw}), pr, v


def _active_problem(N):
    """1.5 m right of the path, vy and omega near their bounds, steering that pushes vy up: the box is active"""
    x = np.array([0.0, -1.5, 0.05, 1.0, 0.135, 1.9])
    up = np.array([R.d_steady_state(1.0), 0.1])
    return _condensed(N, x, up)


def _passes(c, A, dU, y):
    r = oc.kkt_certificate(c.H, c.q, A, c.l, c.u, dU, y, EPS, EPS)
    return r["primal"] <= r["eps_p"] and r["stationarity"] <= r["eps_d"] and r["complementarity"] <= r["comp_bound"]


@pytest.mark.parametrize("N", HORIZONS)
def test_condensed_qp_restates_the_sparse_problem(N):
    """objective at random U to 1e-10 relative; every row, in the kernel's order, equals its sparse row at the point the
    dynamics give (states simulated forward from x0, not taken from the elimination)"""
    rng = np.random.default_rng(N)
    x = np.array([0.2, 0.8, -0.1, 1.1, 0.05, -0.7])
    up = np.array([R.d_steady_state(1.1), -0.05])
    c, pr, v = _condensed(N, x, up, x_lo=[-3.0, -3.0, -1.0, 0.2, -0.15, -2.0], x_hi=[3.0, 3.0, 1.0, 3.0, 0.15, 2.0])
    assert list(c.sidx) == [0, 1, 2, 3, 4, 5] and c.A.shape == (4 * N + 6 * N, 2 * N)
    assert np.abs(c.H - c.H.T).max() == 0.0 and np.linalg.eigvalsh(c.H).min() > 0
    A_, B_, g_, _ = dyn.linearize_horizon(x, up, TS, N)
    n = 2 * N
    D = np.eye(n) - np.eye(n, k=-2)
    np.testing.assert_array_equal(c.A[:n], np.eye(n))
    np.testing.assert_allclose(c.A[n:2 * n], D, atol=1e-15)
    for _ in range(3):
        U = up[None, :] + rng.normal(0, 0.1, (N, 2))
        dU = (U - up[None, :]).reshape(-1)
        X = np.zeros((N + 1, 6)); X[0] = x
        for k in range(N):
            X[k + 1] = A_[k] @ X[k] + B_[k] @ U[k] + g_[k]
        z = np.concatenate([X.reshape(-1), U.reshape(-1)])
        obj = c.sparse.objective(z)
        assert abs(c.objective(dU) - obj) <= 1e-10 * abs(obj)
        np.testing.assert_allclose(c.sparse_point(dU), z, atol=1e-12)
        Ac = c.A @ dU
        # box rows: U_k = u_prev + dU_k; rate rows: U_k - U_{k-1} (U_{-1} = u_prev); state rows: X_k[i], k = 1 .. N
        np.testing.assert_allclose(Ac[:n] + np.tile(up, N), U.reshape(-1), atol=1e-14)
        np.testing.assert_allclose(Ac[n:2 * n], np.diff(np.vstack([up, U]), axis=0).reshape(-1), atol=1e-14)
        np.testing.assert_allclose(Ac[2 * n:] + c.z0[6:6 * (N + 1)], X[1:].reshape(-1), atol=1e-12)
        # the bounds are the sparse ones, shifted by the same free response: row slack is preserved row by row
        sp_rows = (c.sparse.A @ z)[c.sparse.n_eq:][c.ysel]
        np.testing.assert_allclose(Ac - c.l, sp_rows - c.sparse.l[c.sparse.n_eq:][c.ysel], atol=1e-11)
        np.testing.assert_allclose(c.u - Ac, c.sparse.u[c.sparse.n_eq:][c.ysel] - sp_rows, atol=1e-11)
    np.testing.assert_allclose(c.k0_l, np.array([-3.0, -3.0, -1.0, 0.2, -0.15, -2.0]) - x, atol=0)


def test_a_dropped_box_keeps_its_rows_unbounded():
    """a ctrl row that drops its box (+-TG_INF) on a component the handle bounds: the rows stay, with absent bounds, and the
    sparse problem has no such rows (their duals map to 0)"""
    x = np.array([0.0, 0.5, 0.0, 1.0, 0.0, 0.3]); up = np.array([R.d_steady_state(1.0), 0.0])
    c, _, _ = _condensed(12, x, up, x_lo=[-INF] * 6, x_hi=[INF] * 6, bounded=[False] * 4 + [True, True])
    assert c.Gs.shape == (24, 24) and (c.l[48:] == -INF).all() and (c.u[48:] == INF).all() and (c.ysel[48:] == -1).all()
    assert c.sparse.A.shape[0] == c.sparse.n_eq + 48
    o = oc.exact_optimum(c)
    assert o["status"] == "optimal" and (o["y"][48:] == 0).all()
    assert _passes(c, c.A, o["dU"], o["y"])


@pytest.mark.parametrize("N", HORIZONS)
def test_certificate_accepts_the_optimum_and_rejects_corruptions(N):
    c, _, _ = _active_problem(N)
    o = oc.exact_optimum(c)
    assert o["status"] == "optimal"
    n = 2 * N
    ys = o["y"][2 * n:]
    act = np.nonzero(np.abs(ys) > 1e-6)[0]
    assert len(act) > 0, "the vy / omega box must be active"
    assert abs(c.objective(o["dU"]) - o["objective"]) <= 1e-10 * (1 + abs(o["objective"]))
    assert _passes(c, c.A, o["dU"], o["y"])
    # (1) the optimum moved by 1e-4 along a random direction
    d = np.random.default_rng(N).normal(size=n)
    assert not _passes(c, c.A, o["dU"] + 1e-4 * d / np.abs(d).max(), o["y"])
    # (2) the largest active state-row dual with its sign flipped
    i = act[np.argmax(np.abs(ys[act]))]
    y_bad = o["y"].copy(); y_bad[2 * n + i] = -y_bad[2 * n + i]
    assert not _passes(c, c.A, o["dU"], y_bad)
    # (3) the state rows of that dual's stage taken from the next stage (the previous one at the end of the horizon)
    ns = len(c.sidx)
    k = i // ns
    k2 = k + 1 if k + 1 < N else k - 1
    A_bad = c.A.copy()
    A_bad[2 * n + k * ns:2 * n + (k + 1) * ns] = c.Gs[k2 * ns:(k2 + 1) * ns]
    assert not _passes(c, A_bad, o["dU"], o["y"])


@pytest.mark.parametrize("N", HORIZONS)
def test_feasibility_margin(N):
    # x0 1e-3 outside the vy box, omega and the steering driving vy further out, the tight rate limit: more than 1e-3 short
    x = np.array([0.0, 0.0, 0.05, 1.0, 0.151, -1.9]); up = np.array([R.d_steady_state(1.0), -0.3])
    c, _, _ = _condensed(N, x, up)
    s = oc.feasibility_margin(*c.with_k0_rows())
    assert s > 1e-3 + 1e-6, s
    # the same x0 1e-3 inside the box and loose rate limits: an interior point exists
    x[4], x[5] = 0.149, 0.3
    c, _, _ = _condensed(N, x, np.array([R.d_steady_state(1.0), 0.0]), du_lo=(-0.5, -0.3), du_hi=(0.5, 0.3))
    assert oc.feasibility_margin(*c.with_k0_rows()) == 0.0
    # only the k = 0 rows violated (vy 1e-3 outside, nothing driving it out): exactly that violation
    x = np.array([0.0, 0.0, 0.0, 1.0, 0.151, 0.0])
    c, _, _ = _condensed(N, x, np.array([R.d_steady_state(1.0), 0.0]), du_lo=(-0.5, -0.3), du_hi=(0.5, 0.3))
    assert abs(oc.feasibility_margin(*c.with_k0_rows()) - 1e-3) < 1e-9
