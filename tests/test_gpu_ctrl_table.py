"""GPU: per-problem / per-trajectory controller settings (tg_ctrl_spec tables, tg_mpc_step_ctrl, tg_closed_loop_ctrl).

A table that repeats the handle's settings gives the bits of the run-time-horizon instance without a table; a mixed batch
gives, trajectory by trajectory, the bits of a handle created with each row's settings; non-default rows track the oracle's
exact optimum; streamed generation slices the table with the scenarios; invalid rows are refused before any launch."""
import numpy as np
import pytest

import trajectory_generation_b200 as tg
from trajectory_generation_b200 import _lib
from oracle import mpc as ompc, refgen as R

pytestmark = pytest.mark.gpu

TS = 0.02
INF = _lib.TG_INF
# config-4 style: tight rate limits (generation_type1.py:251) and a box on vy / omega
BOX = dict(du_bounds=((-0.1, 0.1), (-0.04, 0.04)), x_lo=[-INF] * 4 + [-0.15, -2.0], x_hi=[INF] * 4 + [0.15, 2.0])
LOOP_FIELDS = ("clean", "noisy", "U", "status_counts", "iters_total")
STEP_FIELDS = ("u_cmd", "status", "iters", "objective", "U_opt", "X_opt", "y_opt")


def _loop_inputs(B, seed, lat=1.0):
    rng = np.random.default_rng(seed)
    x0 = np.zeros((B, 6))
    x0[:, 1] = rng.uniform(-lat, lat, B)
    x0[:, 2] = rng.uniform(-0.1, 0.1, B)
    x0[:, 3] = rng.uniform(0.8, 1.2, B)
    u0 = np.stack([tg.d_steady_state(x0[:, 3]), np.zeros(B)], 1)
    sc = tg.Scenarios(B)
    sc.set_sine(slice(0, B), rng.uniform(0.3, 0.7, B), 0.5, 0.0, 0.0)
    return x0, u0, sc


def _same(a, b, fields):
    for f in fields:
        np.testing.assert_array_equal(a[f], b[f], err_msg=f)


@pytest.fixture
def dynamic_n(monkeypatch):
    """handles created inside the test use the run-time-horizon instance even where a compile-time one exists"""
    monkeypatch.setenv("TRAJGEN_DYNAMIC_N", "1")


# ------------------------------------------------------------------------------------------------ 1. uniform table
@pytest.mark.parametrize("box", [False, True], ids=["nobox", "box"])
@pytest.mark.parametrize("N", [8, 16, 26, 36, 52, 20])
def test_uniform_table_gives_the_bits_of_no_table(N, box, monkeypatch):
    if N == 20:
        monkeypatch.setenv("TRAJGEN_DYNAMIC_N", "1")
    kw = dict(BOX) if box else {}
    B, T = 40, 50
    x0, u0, sc = _loop_inputs(B, seed=N)
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS, **kw)
    r0 = gen.generate(x0, u0, sc, T)
    r1 = gen.generate(x0, u0, sc, T, ctrl=gen.ctrl_table(B))
    _same(r0, r1, LOOP_FIELDS)
    assert r0["status_counts"][:, :2].sum() > 0
    # the step API on the reference windows of the first closed-loop states
    m = tg.BatchedMPC(N=N, Ts=TS, **kw)
    pr, vr = gen.ref_window(x0, sc)
    s0 = m.step(x0, u0, pr, vr)
    s1 = m.step(x0, u0, pr, vr, ctrl=m.ctrl_table(B))
    _same(s0, s1, STEP_FIELDS)


# ------------------------------------------------------------------------------------------------ 2. mixed batch
def _settings(box):
    """four controller settings; with ``box`` each carries its own (finite) vy / omega box and tight rate limits"""
    s = [dict(q_c=6.0, q_phi=0.5, q_vx=0.5, R=[[0.02, 0.0], [0.0, 2.0]], Rd=[[0.01, 0.0], [0.0, 5.0]]),
         dict(q_c=2.0, q_phi=1.5, q_vx=0.2, R=[[0.05, 0.01], [0.01, 1.0]], Rd=[[0.02, 0.0], [0.0, 2.0]]),
         dict(q_c=12.0, q_phi=0.3, q_vx=1.0, R=[[0.01, 0.0], [0.0, 4.0]], Rd=[[0.005, 0.001], [0.001, 8.0]]),
         dict(q_c=4.0, q_phi=0.8, q_vx=0.5, R=[[0.03, -0.02], [0.0, 0.5]], Rd=[[0.0, 0.0], [0.0, 1.0]])]
    if box:
        boxes = [(0.15, 2.0, 0.1, 0.04), (0.10, 1.0, 0.08, 0.03), (0.20, 0.6, 0.12, 0.05), (0.08, 1.5, 0.05, 0.02)]
        for st, (vy, om, dd, ddl) in zip(s, boxes):
            st.update(du_bounds=((-dd, dd), (-ddl, ddl)), x_lo=[-INF] * 4 + [-vy, -om], x_hi=[INF] * 4 + [vy, om])
    else:
        dus = [((-0.5, 0.5), (-0.3, 0.3)), ((-0.2, 0.3), (-0.1, 0.1)), ((-0.05, 0.05), (-0.02, 0.02)), ((-0.4, 0.1), (-0.2, 0.3))]
        us = [((-1.0, 1.0), (-0.6, 0.6)), ((-0.5, 0.8), (-0.4, 0.4)), ((-1.0, 1.0), (-0.3, 0.3)), ((0.0, 0.6), (-0.6, 0.6))]
        for st, du, u in zip(s, dus, us):
            st.update(du_bounds=du, u_bounds=u)
    return s


def _table_from_settings(gen, settings, which):
    """ctrl table whose row b holds settings[which[b]]"""
    B = len(which)
    rows = [gen.ctrl_table(1, **_ctrl_fields(st))[0] for st in settings]
    return gen.ctrl_table(B, **{f: np.stack([rows[k][f] for k in which]) for f in _lib.CTRL_SPEC_DTYPE.names})


def _ctrl_fields(st):
    f = {k: st[k] for k in ("q_c", "q_phi", "q_vx", "R", "Rd") if k in st}
    if "du_bounds" in st:
        du = np.asarray(st["du_bounds"], float)
        f.update(du_lo=du[:, 0], du_hi=du[:, 1])
    if "u_bounds" in st:
        u = np.asarray(st["u_bounds"], float)
        f.update(u_lo=u[:, 0], u_hi=u[:, 1])
    if "x_lo" in st:
        f.update(x_lo=st["x_lo"], x_hi=st["x_hi"])
    return f


def _mixed_batch_check(N, box, B, T, solver_opts):
    base = dict(BOX) if box else {}
    settings = _settings(box)
    which = np.random.default_rng(7 * N + B).permutation(np.arange(B) % 4)
    x0, u0, sc = _loop_inputs(B, seed=N + 100, lat=1.5 if box else 1.0)
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS, solver_opts=solver_opts, **base)
    tab = _table_from_settings(gen, settings, which)
    mixed = gen.generate(x0, u0, sc, T, ctrl=tab)
    m = tg.BatchedMPC(N=N, Ts=TS, solver_opts=solver_opts, **base)
    pr, vr = gen.ref_window(x0, sc)
    smix = m.step(x0, u0, pr, vr, ctrl=tab)
    for k, st in enumerate(settings):
        rows = np.nonzero(which == k)[0]
        ref = tg.ClosedLoopGenerator(N=N, Ts=TS, solver_opts=solver_opts, **{**base, **st}).generate(x0, u0, sc, T)
        for f in LOOP_FIELDS:
            np.testing.assert_array_equal(mixed[f][rows], ref[f][rows], err_msg=f"setting {k}: {f}")
        sref = tg.BatchedMPC(N=N, Ts=TS, solver_opts=solver_opts, **{**base, **st}).step(x0, u0, pr, vr)
        for f in STEP_FIELDS:
            np.testing.assert_array_equal(smix[f][rows], sref[f][rows], err_msg=f"setting {k}: step {f}")
    return mixed


@pytest.mark.parametrize("N", [10, 20])
def test_mixed_batch_with_state_box_equals_one_handle_per_setting(N, dynamic_n):
    mixed = _mixed_batch_check(N, True, B=48, T=40, solver_opts={"max_iter": 150})
    tot = mixed["status_counts"].sum(0)
    assert tot[2] > 0 and tot[4] > 0, tot      # steps that end infeasible and at the iteration limit are covered
    assert tot[5] == 0


@pytest.mark.parametrize("ppc", [None, 1, 2, 4])
@pytest.mark.parametrize("N", [10, 20])
def test_mixed_batch_without_state_box_equals_one_handle_per_setting(N, ppc, dynamic_n, monkeypatch):
    if ppc is not None:
        monkeypatch.setenv("TRAJGEN_PPC", str(ppc))
    mixed = _mixed_batch_check(N, False, B=48 if ppc is None else 47, T=40, solver_opts=None)
    assert mixed["status_counts"][:, :2].sum() > 0


# ------------------------------------------------------------------------------------------------ 3. oracle
def test_closed_loop_rows_track_the_oracle():
    N, T = 20, 200
    x0 = np.array([[0.0, 0.4, 0.05, 1.0, 0.0, 0.0]])
    u0 = np.array([[tg.d_steady_state(1.0), 0.0]])
    sc = tg.Scenarios(1)
    sc.set_sine(0, 0.5, 0.5, 0.0, 0.0)
    w_a = dict(q_c=3.0, q_phi=1.0, q_vx=0.8, R=np.array([[0.05, 0.01], [0.01, 1.0]]), Rd=np.diag([0.02, 3.0]),
               du_bounds=((-0.2, 0.2), (-0.1, 0.1)))
    w_b = dict(q_c=10.0, q_phi=0.3, q_vx=0.4, R=np.diag([0.01, 3.0]), Rd=np.diag([0.02, 6.0]),
               du_bounds=((-0.3, 0.3), (-0.05, 0.05)))
    # (a) a handle without a state box
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS)
    ra = gen.generate(x0, u0, sc, T, ctrl=gen.ctrl_table(1, **_ctrl_fields(w_a)))
    # (b) a box-carrying handle whose row drops the box (+-TG_INF): the oracle runs without state bounds
    genb = tg.ClosedLoopGenerator(N=N, Ts=TS, **BOX)
    rb = genb.generate(x0, u0, sc, T, ctrl=genb.ctrl_table(1, **_ctrl_fields(w_b), x_lo=[-INF] * 6, x_hi=[INF] * 6))
    for r, w in ((ra, w_a), (rb, w_b)):
        Xo, Uo, st, _ = ompc.closed_loop(x0[0], u0[0], T, TS, N, path_kind=R.PATH_SINE, path_prm=(0.5, 0.5, 0.0, 0.0), **w)
        assert all(s == "optimal" for s in st)
        assert r["status_counts"][0, :2].sum() == T
        assert np.abs(r["clean"][0] - Xo).max() < 1e-3 and np.abs(r["U"][0] - Uo).max() < 1e-3


def test_step_batch_with_a_setting_per_problem_matches_oracle():
    N, B = 20, 12
    rng = np.random.default_rng(3)
    x0, u0, sc = _loop_inputs(B, seed=5, lat=0.8)
    x0[:, 4] = rng.uniform(-0.02, 0.02, B); x0[:, 5] = rng.uniform(-0.3, 0.3, B)
    m = tg.BatchedMPC(N=N, Ts=TS, **BOX)
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS)
    pr, vr = gen.ref_window(x0, sc)
    q = np.exp(rng.uniform(np.log(0.5), np.log(2.0), (B, 3))) * (6.0, 0.5, 0.5)
    Rm = np.exp(rng.uniform(np.log(0.5), np.log(2.0), (B, 1))) * np.array([0.02, 0.005, 0.005, 2.0])
    Rdm = np.exp(rng.uniform(np.log(0.5), np.log(2.0), (B, 1))) * np.array([0.01, 0.0, 0.0, 5.0])
    du = rng.uniform(0.5, 1.0, (B, 2)) * (0.1, 0.04)
    vy, om = rng.uniform(0.08, 0.2, B), rng.uniform(0.8, 2.0, B)
    xl = np.tile([-INF] * 6, (B, 1)); xh = -xl
    xl[:, 4], xh[:, 4], xl[:, 5], xh[:, 5] = -vy, vy, -om, om
    xl[::4, 4:] = -INF; xh[::4, 4:] = INF                    # every fourth row without the box
    tab = m.ctrl_table(B, q_c=q[:, 0], q_phi=q[:, 1], q_vx=q[:, 2], R=Rm, Rd=Rdm, du_lo=-du, du_hi=du, x_lo=xl, x_hi=xh)
    out = m.step(x0, u0, pr, vr, ctrl=tab)
    for b in range(B):
        bounded = xl[b, 4] > -INF
        u_o, st_o, _ = ompc.mpc_step(x0[b], u0[b], pr[b], Ts=TS, N=N, vref=vr[b], q_c=q[b, 0], q_phi=q[b, 1], q_vx=q[b, 2],
                                     R=Rm[b].reshape(2, 2), Rd=Rdm[b].reshape(2, 2), du_bounds=((-du[b, 0], du[b, 0]), (-du[b, 1], du[b, 1])),
                                     x_lo=xl[b] if bounded else None, x_hi=xh[b] if bounded else None, solver="ipm")
        assert _lib.STATUS_STRINGS[out["status"][b]] == st_o, b
        assert np.abs(out["u_cmd"][b] - u_o).max() < 1e-3, b


# ------------------------------------------------------------------------------------------------ 4. streaming
def test_streamed_generation_slices_the_table(tmp_path):
    N, B, T = 20, 40, 30
    x0, u0, sc = _loop_inputs(B, seed=11)
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS)
    which = np.arange(B) % 4
    tab = _table_from_settings(gen, _settings(False), which)
    one = gen.generate(x0, u0, sc, T, ctrl=tab)
    chunked = gen.generate(x0, u0, sc, T, ctrl=tab, chunk=16)
    _same(one, chunked, LOOP_FIELDS)
    tg.write_csv(one, TS, tmp_path / "c1.csv", tmp_path / "n1.csv")
    kept = gen.generate_to_csv(x0, u0, sc, T, tmp_path / "c2.csv", tmp_path / "n2.csv", chunk=16, keep=True, ctrl=tab)
    _same(one, kept, LOOP_FIELDS)
    assert (tmp_path / "c1.csv").read_bytes() == (tmp_path / "c2.csv").read_bytes()
    assert (tmp_path / "n1.csv").read_bytes() == (tmp_path / "n2.csv").read_bytes()
    # the table really is per trajectory: the settings change the rows
    plain = gen.generate(x0, u0, sc, T)
    for k in (1, 2, 3):
        assert not np.array_equal(plain["U"][which == k], one["U"][which == k])


# ------------------------------------------------------------------------------------------------ 5. rejection
BAD_ROWS = [
    ("q_c", np.nan, "q_c"), ("q_phi", -1.0, "q_phi"), ("q_vx", np.inf, "q_vx"),
    ("R", [1.0, 0.0, 0.0, -1.0], "R "), ("R", [1.0, 2.0, 0.0, 1.0], "R "), ("R", [np.nan, 0.0, 0.0, 1.0], "R[0]"),
    ("Rd", [-0.1, 0.0, 0.0, 1.0], "Rd "), ("Rd", [1.0, 3.0, 3.0, 1.0], "Rd "),
    ("u_lo", [2.0, -0.6], "u_lo[0]"), ("du_hi", [0.5, -0.4], "du_lo[1]"), ("x_lo", [-INF] * 4 + [0.5, -2.0], "x_lo[4]"),
    ("x_lo", [-5.0] + [-INF] * 3 + [-0.15, -2.0], "x_lo[0]"),
]


@pytest.mark.parametrize("field,value,name", BAD_ROWS, ids=[f"{f}-{i}" for i, (f, _, _) in enumerate(BAD_ROWS)])
def test_invalid_rows_are_refused_before_any_launch(field, value, name):
    N, B, T, bad = 10, 6, 5, 3
    x0, u0, sc = _loop_inputs(B, seed=1)
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS, **BOX)
    pr, vr = gen.ref_window(x0, sc)
    tab = gen.ctrl_table(B)
    tab[field][bad] = value
    L = _lib.load()
    n0 = gen.kernel_launches()
    out = {f: np.zeros(s) for f, s in (("u_cmd", (B, 2)), ("objective", B))}
    st, it = np.zeros(B, np.int32), np.zeros(B, np.int32)
    rc = L.tg_mpc_step_ctrl_host(gen.handle, B, _lib.ptr(x0), _lib.ptr(u0), _lib.ptr(np.ascontiguousarray(pr)), _lib.ptr(vr),
                                 tab.ctypes.data, _lib.ptr(out["u_cmd"]), _lib.ptr(st), _lib.ptr(it), _lib.ptr(out["objective"]),
                                 None, None, None)
    msg = L.tg_last_error().decode()
    assert rc == -1 and f"ctrl row {bad}" in msg and name in msg, (rc, msg)
    res = gen.alloc_result(B, T, pinned=False)
    brk, coef = sc.tables()
    rc = L.tg_closed_loop_ctrl_host(gen.handle, B, T, _lib.ptr(x0), _lib.ptr(u0), sc.spec.ctypes.data, tab.ctypes.data,
                                    None, 0, None, 0, 0, _lib.ptr(res["clean"]), _lib.ptr(res["noisy"]), _lib.ptr(res["U"]),
                                    _lib.ptr(res["status_counts"]), _lib.ptr(res["iters_total"]))
    msg = L.tg_last_error().decode()
    assert rc == -1 and f"ctrl row {bad}" in msg and name in msg, (rc, msg)
    with pytest.raises(ValueError, match=f"ctrl row {bad}"):
        gen.generate(x0, u0, sc, T, ctrl=tab)
    with pytest.raises(ValueError, match=f"ctrl row {bad}"):
        gen.generate(x0, u0, sc, T, ctrl=tab, chunk=2)
    with pytest.raises(ValueError, match=f"ctrl row {bad}"):
        gen.step(x0, u0, pr, vr, ctrl=tab)
    with pytest.raises(ValueError, match=f"ctrl row {bad}"):
        gen.ctrl_table(B, **{field: np.stack([gen.ctrl_table(1)[field][0]] * bad + [np.asarray(value, float)] * (B - bad))})
    assert gen.kernel_launches() == n0
