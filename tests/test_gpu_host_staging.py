"""GPU: the host-array entry points (tg_*_host) give the bits of the device-pointer entry points on the same inputs.

The host forms copy the caller's arrays through one device arena per handle.  Each case here runs both forms and compares
every output byte: with optional outputs present and left out (NULL), with and without vref, ctrl and plant tables, spline
tables, T = 0 and B = 0 closed loops, pageable and pinned result buffers, open-loop calls that ask for U only, and batches
that grow and shrink the arena of one handle."""
import ctypes

import numpy as np
import pytest

import trajectory_generation_b200 as tg
from trajectory_generation_b200 import _lib

pytestmark = pytest.mark.gpu

TS = 0.02
INF = _lib.TG_INF
BOX = dict(du_bounds=((-0.1, 0.1), (-0.04, 0.04)), x_lo=[-INF] * 4 + [-0.15, -2.0], x_hi=[INF] * 4 + [0.15, 2.0])


class _Dev:
    """device copies of host arrays on one handle, kept alive as long as this object; None stays None (NULL)"""

    def __init__(self, h):
        self.h, self.bufs = h, []

    def put(self, a):
        if a is None:
            return None
        a = np.ascontiguousarray(a)
        b = _lib.DeviceBuffer(max(a.nbytes, 8), self.h)
        _lib.check(_lib.load().tg_memcpy_h2d(self.h, b.ptr, _lib.ptr(a), a.nbytes))
        self.bufs.append(b)
        return b.ptr

    def get(self, p, like):
        out = np.empty_like(like)
        _lib.check(_lib.load().tg_memcpy_d2h(self.h, _lib.ptr(out), p, out.nbytes))   # synchronises the handle's stream
        return out


def _sentinel(shape, dtype=np.float64, pinned=False):
    a = _lib.pinned_empty(shape, dtype) if pinned and int(np.prod(shape)) else np.empty(shape, dtype)
    a[...] = -7
    return a


def _bits(a):
    return np.ascontiguousarray(a).reshape(-1).view(np.uint8)


def _same(host, dev, names):
    for k in names:
        if host[k] is not None:
            np.testing.assert_array_equal(_bits(host[k]), _bits(dev[k]), err_msg=k)


def _inputs(B, seed, spline):
    rng = np.random.default_rng(seed)
    x0 = np.zeros((B, 6))
    x0[:, 0] = rng.uniform(-1.0, 1.0, B)
    x0[:, 1] = rng.uniform(-0.5, 0.5, B)
    x0[:, 2] = rng.uniform(-0.1, 0.1, B)
    x0[:, 3] = rng.uniform(0.8, 1.2, B)
    u0 = np.stack([tg.d_steady_state(x0[:, 3]), np.zeros(B)], 1)
    sc = tg.Scenarios(B)
    sc.set_sine(slice(0, B), rng.uniform(0.3, 0.7, B), 0.5, 0.0, 0.0)
    if spline and B:
        idx = np.arange(0, B, 2)
        kx = np.tile(np.arange(-6.0, 30.0, 2.0), (len(idx), 1))
        sc.set_splines(idx, kx, rng.normal(0.0, 0.3, kx.shape))
    return x0, u0, sc


# ------------------------------------------------------------------------------------------------ step
STEP_OUT = ("u_cmd", "status", "iters", "objective", "U_opt", "X_opt", "y_opt")
STEP_OPTIONAL = {"all": STEP_OUT, "none": ("u_cmd",), "some": ("u_cmd", "status", "objective", "X_opt")}


@pytest.mark.parametrize("ctrl", [False, True], ids=["noctrl", "ctrl"])
@pytest.mark.parametrize("vref", [False, True], ids=["novref", "vref"])
@pytest.mark.parametrize("outputs", list(STEP_OPTIONAL))
def test_step_host_equals_device(outputs, vref, ctrl):
    """two handles run the same sequence of steps (the warm start carries over), one through the host form"""
    L = _lib.load()
    gh, gd = tg.ClosedLoopGenerator(N=20, Ts=TS, **BOX), tg.ClosedLoopGenerator(N=20, Ts=TS, **BOX)
    N, m = gh.N, gh.m
    dev = _Dev(gd.handle)
    for B, seed in ((16, 1), (16, 2), (40, 3)):
        x0, u0, sc = _inputs(B, seed, spline=False)
        pr, vr = gh.ref_window(x0, sc)
        pr = np.ascontiguousarray(pr)
        vr = np.ascontiguousarray(vr) if vref else None
        tab = gh.ctrl_table(B, q_c=np.linspace(4.0, 8.0, B)) if ctrl else None
        shapes = {"u_cmd": ((B, 2), np.float64), "status": (B, np.int32), "iters": (B, np.int32), "objective": (B, np.float64),
                  "U_opt": ((B, N, 2), np.float64), "X_opt": ((B, N + 1, 6), np.float64), "y_opt": ((B, m), np.float64)}
        host = {k: _sentinel(*shapes[k]) if k in STEP_OPTIONAL[outputs] else None for k in STEP_OUT}
        dptr = {k: dev.put(_sentinel(*shapes[k])) if host[k] is not None else None for k in STEP_OUT}
        _lib.check(L.tg_mpc_step_ctrl_host(gh.handle, B, _lib.ptr(x0), _lib.ptr(u0), _lib.ptr(pr), _lib.ptr(vr), _lib.ptr(tab),
                                           *[_lib.ptr(host[k]) for k in STEP_OUT]))
        _lib.check(L.tg_mpc_step_ctrl(gd.handle, B, dev.put(x0), dev.put(u0), dev.put(pr), dev.put(vr), dev.put(tab),
                                      *[dptr[k] for k in STEP_OUT]))
        _same(host, {k: dev.get(dptr[k], host[k]) if host[k] is not None else None for k in STEP_OUT}, STEP_OUT)
        assert (host["u_cmd"] != -7).all()


# ------------------------------------------------------------------------------------------------ closed loop
LOOP_OUT = ("clean", "noisy", "U", "status_counts", "iters_total")


def _loop_both(gen, dev, B, T, seed, spline, ctrl, plant, optional, pinned):
    """one tg_closed_loop_params_host call and one tg_closed_loop_params call on the same inputs; returns both results"""
    L = _lib.load()
    x0, u0, sc = _inputs(B, seed, spline)
    spec = np.ascontiguousarray(sc.spec)
    brk, coef = sc.tables() if spline else (None, None)
    tab = gen.ctrl_table(B, q_c=np.linspace(4.0, 8.0, B)) if ctrl and B else None
    pl = gen.plant_table(B, m=0.041 * np.linspace(0.9, 1.1, B)) if plant and B else None
    shapes = {"clean": ((B, T + 1, 6), np.float64), "noisy": ((B, T + 1, 6), np.float64), "U": ((B, T, 2), np.float64),
              "status_counts": ((B, _lib.TG_NUM_STATUS), np.int32), "iters_total": (B, np.int64)}
    present = LOOP_OUT if optional else ("clean", "noisy", "U")
    host = {k: _sentinel(*shapes[k], pinned=pinned and k in ("clean", "noisy", "U")) if k in present else None for k in LOOP_OUT}
    dptr = {k: dev.put(_sentinel(*shapes[k])) if host[k] is not None else None for k in LOOP_OUT}
    # without spline tables the counts still say 7 and 3: a missing table has no pieces
    n_brk, n_coef = (len(brk), len(coef)) if spline else (7, 3)
    _lib.check(L.tg_closed_loop_params_host(gen.handle, B, T, _lib.ptr(x0), _lib.ptr(u0), spec.ctypes.data, _lib.ptr(tab), _lib.ptr(pl),
                                            _lib.ptr(brk), n_brk, _lib.ptr(coef), n_coef, 11, *[_lib.ptr(host[k]) for k in LOOP_OUT]))
    _lib.check(L.tg_closed_loop_params(gen.handle, B, T, dev.put(x0), dev.put(u0), dev.put(spec), dev.put(tab), dev.put(pl),
                                       dev.put(brk), dev.put(coef), 11, *[dptr[k] for k in LOOP_OUT]))
    if B == 0:
        return host, host
    return host, {k: dev.get(dptr[k], host[k]) if host[k] is not None else None for k in LOOP_OUT}


@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("tables", ["none", "ctrl", "plant", "ctrl+plant"])
def test_closed_loop_host_equals_device(tables, pinned):
    gen = tg.ClosedLoopGenerator(N=20, Ts=TS)
    dev = _Dev(gen.handle)
    for T in (30, 0):
        for spline in (True, False):
            for optional in (True, False):
                host, ref = _loop_both(gen, dev, 24, T, 5, spline, "ctrl" in tables, "plant" in tables, optional, pinned)
                _same(host, ref, LOOP_OUT)
                assert (host["clean"] != -7).all()
                if optional:
                    assert host["status_counts"].sum() == 24 * T
    _loop_both(gen, dev, 0, 30, 5, False, "ctrl" in tables, "plant" in tables, True, pinned)   # B = 0: nothing to do, both succeed


def test_host_arena_grows_and_is_reused():
    """a larger batch after a smaller one grows the handle's arena; a smaller one after it reuses it"""
    gen = tg.ClosedLoopGenerator(N=20, Ts=TS)
    og = tg.OpenLoopGenerator("type2", Ts=0.01)
    dev, odev = _Dev(gen.handle), _Dev(og._h)
    for B in (8, 300, 8, 64):
        host, ref = _loop_both(gen, dev, B, 25, B, True, False, False, True, False)
        _same(host, ref, LOOP_OUT)
        host, ref = _openloop_both(og, odev, B, 40, ("clean", "noisy", "U", "modes"), False)
        _same(host, ref, OL_OUT)


# ------------------------------------------------------------------------------------------------ scenarios
@pytest.mark.parametrize("B", [0, 5, 130])
def test_make_scenarios_host_equals_device(B):
    L = _lib.load()
    gen = tg.ClosedLoopGenerator(N=20, Ts=TS)
    dev = _Dev(gen.handle)
    rules = tg.scenario_rules()
    P = rules.spl_knots - 1
    names = ("x0", "u0", "spec", "brk", "coef")
    host = {"x0": _sentinel((B, 6)), "u0": _sentinel((B, 2)), "spec": np.zeros(B, _lib.REF_SPEC_DTYPE),
            "brk": _sentinel(B * P), "coef": _sentinel((B * P, 4))}
    _bits(host["spec"])[:] = 0xA5
    dptr = {k: dev.put(host[k]) for k in names}
    _lib.check(L.tg_make_scenarios_host(gen.handle, B, 3, ctypes.byref(rules), *[_lib.ptr(host[k]) for k in names]))
    _lib.check(L.tg_make_scenarios(gen.handle, B, 3, ctypes.byref(rules), *[dptr[k] for k in names]))
    if B:
        _same(host, {k: dev.get(dptr[k], host[k]) for k in names}, names)
        assert (host["x0"] != -7).all()


# ------------------------------------------------------------------------------------------------ open loop
OL_OUT = ("clean", "noisy", "U", "modes")


def _openloop_both(og, dev, B, T, want, plant):
    L = _lib.load()
    x0 = np.ascontiguousarray(og.sample_x0(B, seed=B + T))
    pl = og.plant_table(B, m=0.041 * np.linspace(0.9, 1.1, B)) if plant else None
    shapes = {"clean": ((B, T + 1, 6), np.float64), "noisy": ((B, T + 1, 6), np.float64), "U": ((B, T, 2), np.float64),
              "modes": ((B,) if og.kind == "type1" else (B, T), np.int8)}
    host = {k: _sentinel(*shapes[k]) if k in want else None for k in OL_OUT}
    dptr = {k: dev.put(_sentinel(*shapes[k])) if host[k] is not None else None for k in OL_OUT}
    fn = f"tg_openloop_{og.kind}_params"
    _lib.check(getattr(L, fn + "_host")(og._h, B, T, _lib.ptr(x0), ctypes.byref(og.rules), og.ctrl_seed_base, 2, _lib.ptr(pl),
                                        *[_lib.ptr(host[k]) for k in OL_OUT]))
    _lib.check(getattr(L, fn)(og._h, B, T, dev.put(x0), ctypes.byref(og.rules), og.ctrl_seed_base, 2, dev.put(pl),
                              *[dptr[k] for k in OL_OUT]))
    return host, {k: dev.get(dptr[k], host[k]) if host[k] is not None else None for k in OL_OUT}


@pytest.mark.parametrize("plant", [False, True], ids=["noplant", "plant"])
@pytest.mark.parametrize("kind", ["type1", "type2"])
def test_openloop_host_equals_device(kind, plant):
    og = tg.OpenLoopGenerator(kind, Ts=0.01)
    dev = _Dev(og._h)
    for want in (OL_OUT, ("U",), ("clean", "modes"), ("noisy",), ()):
        host, ref = _openloop_both(og, dev, 50, 60, want, plant)
        _same(host, ref, OL_OUT)
        for k in want:
            assert (host[k] != -7).any(), k
