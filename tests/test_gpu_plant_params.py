"""GPU: per-trajectory plant parameters (tg_closed_loop_params, tg_plant_rollout_params, tg_openloop_type{1,2}_params).

A table whose rows repeat the handle's params gives the bits of the launch without a table on every kernel instance; row b
gives the bits of a handle created with params = row b (without tyre tables when the row changes B / C); the open-loop
generators agree with tg_plant_rollout and with the oracle; closed-loop rows with a plant that differs from the controller's
model track the oracle's loop (restated with a vehicle of its own for the plant: tests/plant_mismatch_loop.py); trajectories
are independent of their neighbours and of how a batch is cut; invalid tables are refused before any launch."""
import numpy as np
import pytest

import trajectory_generation_b200 as tg
from trajectory_generation_b200 import _lib
from oracle import dynamics as dyn, mpc as ompc, openloop as ool, refgen as R
import plant_mismatch_loop as pml

pytestmark = pytest.mark.gpu

TS = 0.02
INF = _lib.TG_INF
ORDER = _lib.PARAM_ORDER
BOX = dict(du_bounds=((-0.1, 0.1), (-0.04, 0.04)), x_lo=[-INF] * 4 + [-0.15, -2.0], x_hi=[INF] * 4 + [0.15, 2.0])
LOOP_FIELDS = ("clean", "noisy", "U", "status_counts", "iters_total")
PLANTS = (tg.PLANT_MPC, tg.PLANT_GEN1, tg.PLANT_GEN2)


def _loop_inputs(B, seed):
    rng = np.random.default_rng(seed)
    x0 = np.zeros((B, 6))
    x0[:, 1] = rng.uniform(-1.0, 1.0, B)
    x0[:, 2] = rng.uniform(-0.1, 0.1, B)
    x0[:, 3] = rng.uniform(0.8, 1.2, B)
    u0 = np.stack([tg.d_steady_state(x0[:, 3]), np.zeros(B)], 1)
    sc = tg.Scenarios(B)
    sc.set_sine(slice(0, B), rng.uniform(0.3, 0.7, B), 0.5, 0.0, 0.0)
    return x0, u0, sc


def _same(a, b, fields=LOOP_FIELDS):
    for f in fields:
        np.testing.assert_array_equal(a[f], b[f], err_msg=f)


def _vehicles():
    """four vehicles: two that keep the tyre constants (B, C, maxAlpha) and two that change B / C"""
    return [dict(m=0.041 * 1.15, Iz=27.8e-6 * 0.85, Cm1=0.287 * 1.1, Df=0.192 * 0.9, Dr=0.1737 * 1.12),
            dict(m=0.041 * 0.85, Iz=27.8e-6 * 1.2, Cm2=0.0545 * 1.1, Cr0=0.0518 * 0.9, Df=0.192 * 1.15, Dr=0.1737 * 0.88,
                 lf=0.031, lr=0.031),
            dict(m=0.041 * 1.05, Bf=2.579 * 1.08, Cf=1.2 * 0.95),
            dict(Iz=27.8e-6 * 0.9, Br=3.3852 * 0.93, Cr=1.2691 * 1.06, Dr=0.1737 * 1.05)]


def _row(v):
    p = dict(tg.Params)
    p.update(v)
    return [p[k] for k in ORDER]


def _mixed_table(B):
    vs = _vehicles()
    return np.array([_row(vs[b % 4]) for b in range(B)]), [b % 4 for b in range(B)]


@pytest.fixture
def no_tyre_table(monkeypatch):
    def make(fn):
        monkeypatch.setenv("TRAJGEN_NO_TYRE_TABLE", "1")
        try:
            return fn()
        finally:
            monkeypatch.delenv("TRAJGEN_NO_TYRE_TABLE")
    return make


# ------------------------------------------------------------------------------------------------ 1. uniform table
@pytest.mark.parametrize("case", ["n20", "n26", "box", "ctrl"])
def test_closed_loop_uniform_table_gives_the_bits_of_no_table(case):
    N = 26 if case == "n26" else 20
    kw = dict(BOX) if case == "box" else {}
    B, T = 40, 60
    x0, u0, sc = _loop_inputs(B, seed=N + len(case))
    gen = tg.ClosedLoopGenerator(N=N, Ts=TS, plant=tg.PLANT_GEN2, **kw)
    ctrl = gen.ctrl_table(B) if case == "ctrl" else None
    r0 = gen.generate(x0, u0, sc, T, ctrl=ctrl)
    r1 = gen.generate(x0, u0, sc, T, ctrl=ctrl, plant_params=gen.plant_table(B))
    _same(r0, r1)
    accepted = r0["status_counts"][:, :2].sum()
    assert accepted == B * T if case != "box" else accepted > B * T // 2   # the box makes some steps infeasible by construction


@pytest.mark.parametrize("plant", PLANTS)
def test_plant_rollout_and_openloop_uniform_table_give_the_bits_of_no_table(plant):
    B, T = 70, 300
    rng = np.random.default_rng(plant)
    gen = tg.ClosedLoopGenerator(N=5, Ts=0.01, plant=plant)
    x0 = np.zeros((B, 6)); x0[:, 3] = rng.uniform(0.3, 1.5, B); x0[:, 5] = rng.uniform(-1, 1, B)
    U = np.stack([rng.uniform(-0.2, 0.6, (B, T)), rng.uniform(-0.5, 0.5, (B, T))], -1)
    np.testing.assert_array_equal(gen.plant_rollout(x0, U, plant_params=gen.plant_table(B)), gen.plant_rollout(x0, U))
    for kind in ("type1", "type2"):
        og = tg.OpenLoopGenerator(kind, Ts=0.01, plant=plant)
        xo = og.sample_x0(B, seed=4)
        a, b = og.generate(xo, T), og.generate(xo, T, plant_params=og.plant_table(B))
        _same(a, b, ("clean", "noisy", "U", "modes"))


# ------------------------------------------------------------------------------------------------ 2. row b = a handle with row b
def _handle_for(v, make_plain, no_tyre_table):
    keeps = not any(k in v for k in ("Bf", "Cf", "Br", "Cr", "maxAlpha"))
    return make_plain() if keeps else no_tyre_table(make_plain)


@pytest.mark.parametrize("plant", PLANTS)
def test_plant_rollout_row_gives_the_bits_of_a_handle_with_its_params(plant, no_tyre_table):
    B, T = 48, 250
    rng = np.random.default_rng(10 + plant)
    x0 = np.zeros((B, 6)); x0[:, 3] = rng.uniform(0.3, 1.5, B); x0[:, 4] = rng.uniform(-0.05, 0.05, B)
    x0[:, 5] = rng.uniform(-1, 1, B)
    x0[::3, 3] = 0.3; x0[::3, 4] = rng.uniform(-0.5, 0.5, x0[::3].shape[0])   # slow and sliding: GEN1's unclamped rear slip
    U = np.stack([rng.uniform(-0.2, 0.6, (B, T)), rng.uniform(-0.6, 0.6, (B, T))], -1)   # angle leaves the clamp interval
    gen = tg.ClosedLoopGenerator(N=5, Ts=0.01, plant=plant)
    table, which = _mixed_table(B)
    X = gen.plant_rollout(x0, U, plant_params=table)
    for k, v in enumerate(_vehicles()):
        idx = [b for b in range(B) if which[b] == k]
        h = _handle_for(v, lambda: tg.ClosedLoopGenerator(N=5, Ts=0.01, plant=plant, params=v), no_tyre_table)
        np.testing.assert_array_equal(X[idx], h.plant_rollout(x0[idx], U[idx]), err_msg=str(v))
        assert np.abs(X[idx] - gen.plant_rollout(x0[idx], U[idx])).max() > 0
    if plant == tg.PLANT_GEN1:   # the unclamped rear slip angle has left [-maxAlpha, maxAlpha] (libdevice path of the table rows)
        p = tg.Params
        alpha_r = np.arctan2(X[..., 5] * p["lr"] - X[..., 4], np.maximum(np.abs(X[..., 3]), p["vx_zero"]))
        assert np.abs(alpha_r).max() > p["maxAlpha"]


@pytest.mark.parametrize("kind", ["type1", "type2"])
@pytest.mark.parametrize("plant", PLANTS)
def test_openloop_row_gives_the_bits_of_a_handle_with_its_params(kind, plant, no_tyre_table):
    B, T = 40, 400
    og = tg.OpenLoopGenerator(kind, Ts=0.01, plant=plant)
    x0 = og.sample_x0(B, seed=7)
    table, which = _mixed_table(B)
    res = og.generate(x0, T, plant_params=table)
    for k, v in enumerate(_vehicles()):
        idx = np.array([b for b in range(B) if which[b] == k])
        h = _handle_for(v, lambda: tg.OpenLoopGenerator(kind, Ts=0.01, plant=plant, params=v), no_tyre_table)
        for b in idx:   # one trajectory per launch: its ids (control and noise streams) are kept through traj_id0
            r = h.generate(x0[b:b + 1], T, traj_id0=int(b))
            for f in ("clean", "noisy", "U", "modes"):
                np.testing.assert_array_equal(res[f][b:b + 1], r[f], err_msg=f"{f} {b} {v}")


# ------------------------------------------------------------------------------------------------ 3. open-loop consistency
def _rules_from_struct(cls, struct):
    import ctypes
    kw = {}
    for name, _ in struct._fields_:
        if name != "reserved":
            v = getattr(struct, name)
            kw[name] = tuple(v) if isinstance(v, ctypes.Array) else v
    return cls(**kw)


@pytest.mark.parametrize("kind", ["type1", "type2"])
def test_openloop_with_table_matches_plant_rollout_and_oracle(kind):
    B, T, Ts = 24, 1200, 0.01
    og = tg.OpenLoopGenerator(kind, Ts=Ts)
    x0 = og.sample_x0(B, seed=11)
    table, which = _mixed_table(B)
    res = og.generate(x0, T, plant_params=table)
    pl = tg.ClosedLoopGenerator(N=5, Ts=Ts, plant=og.cfg.plant)
    np.testing.assert_array_equal(pl.plant_rollout(x0, res["U"], plant_params=table), res["clean"])
    rules = _rules_from_struct(ool.Type1Rules if kind == "type1" else ool.Type2Rules, og.rules)
    exact = 0
    for b in range(B):
        p = dict(zip(ORDER, table[b]))
        if kind == "type1":
            U, X, mode = ool.type1_trajectory(ool.PhiloxType1Source(tg.CTRL_SEED_BASE + b), x0[b], T, Ts, rules, p=p)
            np.testing.assert_allclose(res["U"][b], U, rtol=0, atol=1e-12)
            assert res["modes"][b] == mode
            np.testing.assert_allclose(res["clean"][b], X, rtol=1e-8, atol=1e-8)
            exact += 1
        else:
            U, X, modes = ool.type2_trajectory(ool.PhiloxType2Source(tg.CTRL_SEED_BASE + b), x0[b], T, Ts, rules, p=p)
            if not np.array_equal(res["modes"][b], modes):   # a threshold decision on the last bits of the state (libdevice vs
                continue                                      # libm) may flip on a libdevice row
            exact += 1
            np.testing.assert_allclose(res["U"][b], U, rtol=0, atol=1e-9)
            np.testing.assert_allclose(res["clean"][b], X, rtol=1e-7, atol=1e-7)
    assert exact >= B - 2


# ------------------------------------------------------------------------------------------------ 4. closed loop with mismatch
def _oracle_spline(sc, i):
    f, K = sc.spec["spline_first"][i], sc.spec["spline_count"][i]
    brk, coef = sc.tables()
    return np.append(brk[f:f + K], np.inf), coef[f:f + K]


def _oracle_check(gen, x0, u0, sc, res, b, T, plant_row, **mpc_kwargs):
    kind = int(sc.spec["path_kind"][b])
    Xo, Uo, st, _ = pml.closed_loop(x0[b], u0[b], T, gen.cfg.Ts, gen.N, path_kind=kind, path_prm=tuple(sc.spec["path"][b]),
                                     spline=_oracle_spline(sc, b) if kind == R.PATH_SPLINE else None, vref_kind=R.VREF_RAMP,
                                     vref_prm=tuple(sc.spec["vref"][b][:3]), vref_advance=True, plant=dyn.PLANT_GEN2,
                                     solver="ipm", plant_params=plant_row, **mpc_kwargs)
    assert all(s in ompc.ACCEPTED for s in st)
    assert res["status_counts"][b, :2].sum() == T
    assert np.abs(res["clean"][b, :T + 1] - Xo).max() < 1e-3 and np.abs(res["U"][b, :T] - Uo).max() < 1e-3


def test_closed_loop_with_plant_mismatch_tracks_the_oracle():
    T = 200
    gen = tg.ClosedLoopGenerator(N=20, Ts=0.01, plant=tg.PLANT_GEN2, vref_advance=True)
    x0, u0, sc = gen.make_scenarios(8)
    vs = _vehicles()
    table = gen.plant_table(8)
    for b, k in ((0, 0), (1, 1), (2, 2)):     # a spline, a sine (rows keep the tyre constants) and a spline with other B / C
        table[b] = _row(vs[k])
    res = gen.generate(x0, u0, sc, T, plant_params=table)
    assert {int(sc.spec["path_kind"][b]) for b in range(3)} == {R.PATH_SPLINE, R.PATH_SINE}
    for b in range(3):
        _oracle_check(gen, x0, u0, sc, res, b, T, table[b])


# ------------------------------------------------------------------------------------------------ 5. batch independence
def test_rows_of_the_handles_params_keep_their_bits_and_permutation_permutes():
    B, T = 64, 120
    gen = tg.ClosedLoopGenerator(N=20, Ts=0.01, plant=tg.PLANT_GEN2, vref_advance=True)
    x0, u0, sc = gen.make_scenarios(B)
    base = gen.generate(x0, u0, sc, T)
    table = gen.plant_table(B)
    changed = np.arange(B) % 3 == 1
    mixed, _ = _mixed_table(B)
    table[changed] = mixed[changed]
    r = gen.generate(x0, u0, sc, T, plant_params=table)
    for f in LOOP_FIELDS:
        np.testing.assert_array_equal(r[f][~changed], base[f][~changed], err_msg=f)
    assert all(np.abs(r["clean"][b] - base["clean"][b]).max() > 0 for b in np.flatnonzero(changed))
    perm = np.random.default_rng(5).permutation(B)
    spec = sc.spec[perm].copy()
    sp = tg.Scenarios(0); sp.spec = spec; sp._breaks, sp._coef = sc._breaks, sc._coef
    rp = gen.generate(x0[perm], u0[perm], sp, T, plant_params=table[perm])
    # the noise stream is keyed by the position in the batch: compare everything but the noisy rows
    for f in ("clean", "U", "status_counts", "iters_total"):
        np.testing.assert_array_equal(rp[f], r[f][perm], err_msg=f)


def test_chunked_streamed_and_csv_generation_equal_one_launch(tmp_path):
    B, T = 50, 80
    gen = tg.ClosedLoopGenerator(N=20, Ts=0.01, plant=tg.PLANT_GEN2, vref_advance=True)
    x0, u0, sc = gen.make_scenarios(B)
    table, _ = _mixed_table(B)
    one = gen.generate(x0, u0, sc, T, plant_params=table)
    _same(gen.generate(x0, u0, sc, T, chunk=16, plant_params=table), one)
    for lo, hi, res in gen.generate_chunks(x0, u0, sc, T, chunk=21, plant_params=table):
        for f in LOOP_FIELDS:
            np.testing.assert_array_equal(res[f], one[f][lo:hi], err_msg=f)
    out = gen.generate_to_csv(x0, u0, sc, T, tmp_path / "c.csv", tmp_path / "n.csv", chunk=13, keep=True, plant_params=table)
    _same(out, one)
    tg.write_csv(one, 0.01, tmp_path / "c1.csv", tmp_path / "n1.csv")
    assert (tmp_path / "c.csv").read_bytes() == (tmp_path / "c1.csv").read_bytes()
    assert (tmp_path / "n.csv").read_bytes() == (tmp_path / "n1.csv").read_bytes()


# ------------------------------------------------------------------------------------------------ 6. ctrl and plant together
def test_ctrl_table_with_uniform_plant_table_equals_ctrl_table_alone():
    B, T = 40, 60
    x0, u0, sc = _loop_inputs(B, seed=3)
    gen = tg.ClosedLoopGenerator(N=20, Ts=TS, plant=tg.PLANT_GEN2, **BOX)
    ctrl = gen.ctrl_table(B, q_c=np.linspace(2.0, 10.0, B))
    _same(gen.generate(x0, u0, sc, T, ctrl=ctrl), gen.generate(x0, u0, sc, T, ctrl=ctrl, plant_params=gen.plant_table(B)))


def test_ctrl_row_and_plant_row_together_track_the_oracle():
    T = 200
    gen = tg.ClosedLoopGenerator(N=20, Ts=0.01, plant=tg.PLANT_GEN2, vref_advance=True)
    x0, u0, sc = gen.make_scenarios(2)
    w = dict(q_c=3.0, q_phi=1.0, q_vx=0.8, R=np.array([[0.05, 0.01], [0.01, 1.0]]), Rd=np.diag([0.02, 3.0]))
    ctrl = gen.ctrl_table(2, q_c=w["q_c"], q_phi=w["q_phi"], q_vx=w["q_vx"], R=w["R"], Rd=w["Rd"])
    table = gen.plant_table(2)
    table[1] = _row(_vehicles()[0])
    res = gen.generate(x0, u0, sc, T, ctrl=ctrl, plant_params=table)
    _oracle_check(gen, x0, u0, sc, res, 1, T, table[1], **w)


# ------------------------------------------------------------------------------------------------ 7. refused input
@pytest.mark.parametrize("name,value,why", [("m", 0.0, "must be > 0"), ("Iz", -1.0, "must be > 0"), ("Df", np.nan, "must be finite"),
                                            ("maxAlpha", 0.0, "must be > 0"), ("vx_zero", np.inf, "must be finite")])
def test_invalid_table_is_refused_before_any_launch(name, value, why):
    B, T = 6, 10
    x0, u0, sc = _loop_inputs(B, seed=1)
    gen = tg.ClosedLoopGenerator(N=20, Ts=TS)
    og = tg.OpenLoopGenerator("type2", Ts=0.01)
    bad = gen.plant_table(B)
    bad[4, ORDER.index(name)] = value
    msg = rf"plant row 4: {name} {why}"
    n0, m0 = gen.kernel_launches(), og.kernel_launches()
    with pytest.raises(ValueError, match=msg):
        gen.generate(x0, u0, sc, T, plant_params=bad)
    with pytest.raises(ValueError, match=msg):
        gen.plant_rollout(x0, np.zeros((B, T, 2)), plant_params=bad)
    with pytest.raises(ValueError, match=msg):
        og.generate(og.sample_x0(B), T, plant_params=bad)
    # the C entry points refuse it on their own, before anything is launched
    L = _lib.load()
    spec = np.ascontiguousarray(sc.spec)
    out = gen.alloc_result(B, T, pinned=False)
    rc = L.tg_closed_loop_params_host(gen.handle, B, T, _lib.ptr(x0), _lib.ptr(np.ascontiguousarray(u0)), spec.ctypes.data, None,
                                      _lib.ptr(bad), None, 0, None, 0, 0, _lib.ptr(out["clean"]), _lib.ptr(out["noisy"]),
                                      _lib.ptr(out["U"]), None, None)
    assert rc == -1 and L.tg_last_error().decode() == msg
    xo = np.ascontiguousarray(og.sample_x0(B))
    cl = np.empty((B, T + 1, 6))
    rc = L.tg_openloop_type2_params_host(og._h, B, T, _lib.ptr(xo), __import__("ctypes").byref(og.rules), 1, 0, _lib.ptr(bad),
                                         _lib.ptr(cl), None, None, None)
    assert rc == -1 and L.tg_last_error().decode() == msg
    assert gen.kernel_launches() == n0 and og.kernel_launches() == m0
