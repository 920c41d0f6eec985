"""Host-side mirror of the reference's controller interface (MPC/mpc_6stati.py) over libtrajgen.so.

``mpc_step`` keeps the reference's signature, argument meaning, return tuple and failure behaviour
(MPC/mpc_6stati.py:120-143, 255-275): it never raises on a solver failure, it returns
``(u_prev, status_string, {})``.  ``BatchedMPC`` is the same controller for B problems at once.
All arithmetic happens in the CUDA kernels; this module only marshals arrays.
"""
import ctypes

import numpy as np

from . import _lib

# MPC/mpc_6stati.py:9-19
Params = {
    "Cm1": 0.287, "Cm2": 0.0545, "Cr0": 0.0518, "Cr2": 0.00035,
    "Br": 3.3852, "Cr": 1.2691, "Dr": 0.1737, "Bf": 2.579, "Cf": 1.2, "Df": 0.192,
    "m": 0.041, "Iz": 27.8e-6, "lf": 0.029, "lr": 0.033, "g": 9.81, "maxAlpha": 0.6, "vx_zero": 0.3,
}

MODEL_MPC, MODEL_GEN1, MODEL_GEN2 = 0, 1, 2
PLANT_MPC, PLANT_GEN1, PLANT_GEN2 = 0, 1, 2
JAC_ANALYTIC, JAC_FD = 0, 1


def make_config(Ts=0.02, N=20, params=None, q_c=6.0, q_phi=0.5, q_vx=0.5, R=None, Rd=None,
                u_bounds=((-1.0, 1.0), (-0.6, 0.6)), du_bounds=((-0.5, 0.5), (-0.3, 0.3)), x_lo=None, x_hi=None,
                model=MODEL_MPC, plant=PLANT_MPC, jacobian=JAC_ANALYTIC, solver_opts=None, warm_start=False,
                vref_advance=False, noise_std=None, noise_seed_base=None):
    """tg_config from mpc_step-style keyword arguments (same names and defaults, :124-140)."""
    cfg = _lib.default_config()
    cfg.N, cfg.Ts = int(N), float(Ts)
    p = dict(Params)
    if params is not None:
        p.update(params)                                   # :144-146
    for i, k in enumerate(_lib.PARAM_ORDER):
        cfg.params[i] = float(p[k])
    cfg.q_c, cfg.q_phi, cfg.q_vx = float(q_c), float(q_phi), float(q_vx)
    R = np.diag([0.02, 2.0]) if R is None else np.asarray(R, float).reshape(2, 2)
    Rd = np.diag([0.01, 5.0]) if Rd is None else np.asarray(Rd, float).reshape(2, 2)
    for i in range(4):
        cfg.R[i], cfg.Rd[i] = float(R.flat[i]), float(Rd.flat[i])
    for j in range(2):
        cfg.u_lo[j], cfg.u_hi[j] = float(u_bounds[j][0]), float(u_bounds[j][1])
        cfg.du_lo[j], cfg.du_hi[j] = float(du_bounds[j][0]), float(du_bounds[j][1])
    xl = np.full(6, -_lib.TG_INF) if x_lo is None else np.maximum(np.asarray(x_lo, float).reshape(6), -_lib.TG_INF)
    xh = np.full(6, _lib.TG_INF) if x_hi is None else np.minimum(np.asarray(x_hi, float).reshape(6), _lib.TG_INF)
    for i in range(6):
        cfg.x_lo[i], cfg.x_hi[i] = float(xl[i]), float(xh[i])
    cfg.model, cfg.plant, cfg.jacobian = int(model), int(plant), int(jacobian)
    cfg.warm_start, cfg.vref_advance = int(bool(warm_start)), int(bool(vref_advance))
    if noise_std is not None:
        for i in range(6):
            cfg.noise_std[i] = float(noise_std[i])
    if noise_seed_base is not None:
        cfg.noise_seed_base = int(noise_seed_base)
    for k, v in (solver_opts or {}).items():
        if not hasattr(cfg, k):
            raise ValueError(f"unknown solver option {k!r}")
        setattr(cfg, k, type(getattr(cfg, k))(v))
    return cfg




def check_plant_table(table):
    """The rules of a per-trajectory plant table (include/trajgen.h, tg_check_plant_params) for a C-contiguous [B, 17] fp64 array
    whose columns follow PARAM_ORDER: every entry finite, m, Iz, vx_zero and maxAlpha > 0.  Raises ValueError naming the first
    bad row and column, as the C entry points do.  Returns the table."""
    t = np.asarray(table)
    if t.dtype != np.float64 or t.ndim != 2 or t.shape[1] != _lib.TG_NPARAMS or not t.flags["C_CONTIGUOUS"]:
        raise ValueError(f"plant table: expected a C-contiguous [B, {_lib.TG_NPARAMS}] float64 array (columns in PARAM_ORDER), "
                         f"got {t.dtype} {t.shape}")
    L = _lib.load()
    if L.tg_check_plant_params(t.shape[0], _lib.ptr(t)) != 0:
        raise ValueError(L.tg_last_error().decode())
    return table


def _plant_table(params, B, columns):
    """[B, 17] plant table whose rows start as ``params`` (17 values in PARAM_ORDER); columns by name take a scalar or a [B] array"""
    B = int(B)
    t = np.empty((B, _lib.TG_NPARAMS))
    t[:] = np.asarray(params[:], float)
    for k, v in columns.items():
        if k not in _lib.PARAM_ORDER:
            raise TypeError(f"unknown plant parameter {k!r} (names: {', '.join(_lib.PARAM_ORDER)})")
        v = np.asarray(v, float)
        if v.ndim > 1 or (v.ndim == 1 and v.shape[0] != B):
            raise ValueError(f"plant parameter {k}: expected a scalar or {B} values, got shape {v.shape}")
        t[:, _lib.PARAM_ORDER.index(k)] = v
    return check_plant_table(t)


def _plant_arg(table, B):
    """a caller's plant table, checked (None stays None)"""
    if table is None:
        return None
    t = np.asarray(table)
    if t.ndim != 2 or t.shape[0] != B:
        raise ValueError(f"plant_params: expected {B} rows, got shape {t.shape}")
    return check_plant_table(np.ascontiguousarray(t) if t.dtype == np.float64 else t)


def check_ctrl_table(table, bounded):
    """The rules of include/trajgen.h::tg_ctrl_spec for every row of ``table`` (CTRL_SPEC_DTYPE), checked by the library's
    tg_check_ctrl; ``bounded[6]`` says which state components the handle bounds.  Raises ValueError naming the first bad row
    and field, as the C entry points do."""
    t = np.ascontiguousarray(table)
    if t.dtype != _lib.CTRL_SPEC_DTYPE or t.ndim != 1:
        raise ValueError("ctrl must be a table of CTRL_SPEC_DTYPE (see ctrl_table)")
    L = _lib.load()
    if L.tg_check_ctrl(len(t), _lib.ptr(t), sum(1 << i for i in range(6) if bounded[i])) != 0:
        raise ValueError(L.tg_last_error().decode())
    return table


class BatchedMPC:
    """B independent MPC problems per call on one B200.  Construction takes mpc_step's keyword
    arguments; ``step`` takes the per-problem arrays."""

    def __init__(self, device=0, **kwargs):
        self.cfg = make_config(**kwargs)
        self.N = self.cfg.N
        self._h = ctypes.c_void_p()
        _lib.check(_lib.load().tg_create(ctypes.byref(self.cfg), int(device), ctypes.byref(self._h)))
        self.n = 2 * self.N
        self.ns = sum(self.bounded_states)
        self.ms = self.ns * self.N
        self.m = 4 * self.N + self.ms

    # -- lifetime
    def close(self):
        if self._h:
            _lib.load().tg_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def set_stream(self, cuda_stream):
        _lib.check(_lib.load().tg_set_stream(self._h, ctypes.c_void_p(int(cuda_stream))))

    def synchronize(self):
        _lib.check(_lib.load().tg_synchronize(self._h))

    def kernel_launches(self):
        c = ctypes.c_int64()
        _lib.check(_lib.load().tg_kernel_launches(self._h, ctypes.byref(c)))
        return c.value

    def info(self):
        """launch geometry: dict(ctas_per_sm, threads_per_cta, smem_bytes, num_sms)."""
        v = [ctypes.c_int32() for _ in range(4)]
        _lib.check(_lib.load().tg_info(self._h, *[ctypes.byref(x) for x in v]))
        return dict(zip(("ctas_per_sm", "threads_per_cta", "smem_bytes", "num_sms"), [x.value for x in v]))

    def tyre_table_info(self):
        """dict(in_use, max_value_err, max_slope_err) of the tyre-curve table built for this handle's B, C, maxAlpha."""
        u, a, b = ctypes.c_int32(), ctypes.c_double(), ctypes.c_double()
        _lib.check(_lib.load().tg_tyre_table_info(self._h, ctypes.byref(u), ctypes.byref(a), ctypes.byref(b)))
        return {"in_use": bool(u.value & 1), "atan_in_use": bool(u.value & 2), "max_value_err": a.value, "max_slope_err": b.value}

    # -- per-problem settings
    @property
    def bounded_states(self):
        """which of the six state components this handle bounds (tg_config's finite x_lo / x_hi): the components on which a
        ctrl table may set bounds"""
        return tuple(self.cfg.x_lo[i] > -_lib.TG_INF or self.cfg.x_hi[i] < _lib.TG_INF for i in range(6))

    def ctrl_table(self, B, **fields):
        """A [B] table of per-problem controller settings (CTRL_SPEC_DTYPE, include/trajgen.h::tg_ctrl_spec) for ``step`` and
        ``ClosedLoopGenerator.generate``.  Every row starts as this handle's own settings; a keyword overrides a field with an
        array that broadcasts to [B] (q_c, q_phi, q_vx) or [B, k] (R and Rd: k = 4 row-major, or [..., 2, 2]; u_lo, u_hi,
        du_lo, du_hi: 2; x_lo, x_hi: 6).  A bound of +-TG_INF (or +-inf) is absent.  Raises ValueError naming the first row
        that breaks a rule of tg_ctrl_spec."""
        B = int(B)
        t = np.zeros(B, _lib.CTRL_SPEC_DTYPE)
        cfg = self.cfg
        for f in _lib.CTRL_SPEC_DTYPE.names:
            v = getattr(cfg, f)
            t[f] = v if isinstance(v, float) else np.asarray(v[:], float)
        for f, v in fields.items():
            if f not in _lib.CTRL_SPEC_DTYPE.names:
                raise TypeError(f"unknown ctrl field {f!r}")
            v = np.asarray(v, float)
            shape = _lib.CTRL_SPEC_DTYPE[f].shape
            if f in ("R", "Rd") and v.shape[-2:] == (2, 2):
                v = v.reshape(v.shape[:-2] + (4,))
            if f in ("x_lo", "x_hi"):
                v = np.clip(v, -_lib.TG_INF, _lib.TG_INF)
            try:
                t[f] = np.broadcast_to(v, (B,) + shape)
            except ValueError:
                raise ValueError(f"ctrl field {f}: shape {v.shape} does not broadcast to {(B,) + shape}") from None
        return check_ctrl_table(t, self.bounded_states)

    def _ctrl_arg(self, ctrl, B):
        """a caller's ctrl table, checked: a C-contiguous [B] array of CTRL_SPEC_DTYPE that satisfies tg_ctrl_spec's rules"""
        t = np.ascontiguousarray(ctrl)
        if t.shape != (B,):
            raise ValueError(f"ctrl: expected {B} rows, got shape {t.shape}")
        return check_ctrl_table(t, self.bounded_states)

    # -- host-array API
    @staticmethod
    def _arr(a, shape):
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
        if a.shape != shape:
            raise ValueError(f"expected shape {shape}, got {a.shape}")
        return a

    def _on_device(self, arrays):
        """copy host arrays into fresh device buffers; returns (buffers, pointers)."""
        L = _lib.load()
        bufs = []
        for a in arrays:
            if a is None:
                bufs.append(None)
                continue
            b = _lib.DeviceBuffer(max(a.nbytes, 8), self._h)
            _lib.check(L.tg_memcpy_h2d(self._h, b.ptr, _lib.ptr(a), a.nbytes))
            bufs.append(b)
        return bufs

    def _from_device(self, buf, shape, dtype=np.float64):
        out = np.empty(shape, dtype=dtype)
        _lib.check(_lib.load().tg_memcpy_d2h(self._h, _lib.ptr(out), buf.ptr, out.nbytes))
        return out

    def linearize(self, x0, u_prev):
        """K1 tap: -> A[B,N,6,6], Bm[B,N,6,2], g[B,N,6], xbar[B,N+1,6]  (MPC/mpc_6stati.py:165-178)."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B, N = x0.shape[0], self.N
        u_prev = self._arr(np.asarray(u_prev, float).reshape(-1, 2), (B, 2))
        if B == 0:
            return np.zeros((0, N, 6, 6)), np.zeros((0, N, 6, 2)), np.zeros((0, N, 6)), np.zeros((0, N + 1, 6))
        bx, bu = self._on_device([x0, u_prev])
        oA, oB, og, ox = (_lib.DeviceBuffer(B * N * 36 * 8, self._h), _lib.DeviceBuffer(B * N * 12 * 8, self._h),
                          _lib.DeviceBuffer(B * N * 6 * 8, self._h), _lib.DeviceBuffer(B * (N + 1) * 6 * 8, self._h))
        _lib.check(_lib.load().tg_linearize(self._h, B, bx.ptr, bu.ptr, oA.ptr, oB.ptr, og.ptr, ox.ptr))
        return (self._from_device(oA, (B, N, 6, 6)), self._from_device(oB, (B, N, 6, 2)),
                self._from_device(og, (B, N, 6)), self._from_device(ox, (B, N + 1, 6)))

    def assemble(self, x0, u_prev, path_ref, vref=None):
        """K2 tap: condensed QP in dU = U - u_prev -> dict(H, q, c0, l, u, Gs)."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B, N, n, m, ms = x0.shape[0], self.N, self.n, self.m, self.ms
        u_prev = self._arr(np.asarray(u_prev, float).reshape(-1, 2), (B, 2))
        path_ref = self._arr(path_ref, (B, N + 1, 3))
        vref = None if vref is None else self._arr(vref, (B, N + 1))
        bx, bu, bp, bv = self._on_device([x0, u_prev, path_ref, vref])
        oH, oq, oc, ol, ou = (_lib.DeviceBuffer(B * n * n * 8, self._h), _lib.DeviceBuffer(B * n * 8, self._h), _lib.DeviceBuffer(B * 8, self._h),
                              _lib.DeviceBuffer(B * m * 8, self._h), _lib.DeviceBuffer(B * m * 8, self._h))
        oG = _lib.DeviceBuffer(max(B * ms * n * 8, 8), self._h)
        _lib.check(_lib.load().tg_assemble(self._h, B, bx.ptr, bu.ptr, bp.ptr, bv.ptr if bv else None,
                                           oH.ptr, oq.ptr, oc.ptr, ol.ptr, ou.ptr, oG.ptr if ms else None))
        return {"H": self._from_device(oH, (B, n, n)), "q": self._from_device(oq, (B, n)),
                "c0": self._from_device(oc, (B,)), "l": self._from_device(ol, (B, m)), "u": self._from_device(ou, (B, m)),
                "Gs": self._from_device(oG, (B, ms, n)) if ms else np.zeros((B, 0, n))}

    def step(self, x0, u_prev, path_ref, vref=None, want_trajectory=True, ctrl=None):
        """Batched mpc_step.  x0[B,6], u_prev[B,2], path_ref[B,N+1,3], vref[B,N+1] | None
        -> dict(u_cmd[B,2], status[B] int32, iters[B], objective[B], U_opt[B,N,2], X_opt[B,N+1,6], y_opt[B,m]).
        Rows whose status is not accepted carry u_cmd = u_prev and NaN in the optional outputs.  ``ctrl``: a [B] table of
        per-problem weights and bounds (``ctrl_table``); None = the handle's settings for every problem."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B, N = x0.shape[0], self.N
        u_prev = self._arr(np.asarray(u_prev, float).reshape(-1, 2), (B, 2))
        path_ref = self._arr(path_ref, (B, N + 1, 3))                 # :151
        vref = None if vref is None else self._arr(vref, (B, N + 1))
        ctrl = None if ctrl is None else self._ctrl_arg(ctrl, B)
        out = {"u_cmd": np.empty((B, 2)), "status": np.empty(B, np.int32), "iters": np.empty(B, np.int32),
               "objective": np.empty(B)}
        if want_trajectory:
            out.update(U_opt=np.empty((B, N, 2)), X_opt=np.empty((B, N + 1, 6)), y_opt=np.empty((B, self.m)))
        _lib.check(_lib.load().tg_mpc_step_ctrl_host(
            self._h, B, _lib.ptr(x0), _lib.ptr(u_prev), _lib.ptr(path_ref), _lib.ptr(vref), _lib.ptr(ctrl),
            _lib.ptr(out["u_cmd"]), _lib.ptr(out["status"]), _lib.ptr(out["iters"]), _lib.ptr(out["objective"]),
            _lib.ptr(out.get("U_opt")), _lib.ptr(out.get("X_opt")), _lib.ptr(out.get("y_opt"))))
        return out


_SHIM_CACHE = {}


def _freeze(v):
    if v is None:
        return None
    if isinstance(v, dict):
        return tuple(sorted((k, _freeze(x)) for k, x in v.items()))
    return tuple(np.asarray(v, float).ravel().tolist())


def mpc_step(x0, u_prev, path_ref, Ts=0.02, N=20, params=None, q_c=6.0, q_phi=0.5, q_vx=0.5,
             R=np.diag([0.02, 2.0]), Rd=np.diag([0.01, 5.0]), vref=None,
             u_bounds=((-1.0, 1.0), (-0.6, 0.6)), du_bounds=((-0.5, 0.5), (-0.3, 0.3)),
             x_lo=None, x_hi=None, solver=None, verbose=False, solver_opts=None, device=0):
    """Drop-in for MPC/mpc_6stati.py:mpc_step (B = 1).  ``solver`` is accepted and ignored (the
    reference's only choice is cp.OSQP; here the CUDA ADMM always runs); ``solver_opts`` exposes
    the ADMM settings of tg_config.  Returns (u_cmd[2], status:str, info:dict) -- info has the
    reference's keys (:267-274) and is {} when the status is not accepted (:258-262)."""
    x0 = np.asarray(x0, float).reshape(6)                   # :148-151
    u_pr = np.asarray(u_prev, float).reshape(2)
    path_ref = np.asarray(path_ref, float)
    assert path_ref.shape[0] == N + 1 and path_ref.shape[1] == 3
    if vref is None:                                        # :158-163
        vref_a = np.full(N + 1, x0[3])
    elif np.isscalar(vref):
        vref_a = np.full(N + 1, float(vref))
    else:
        vref_a = np.asarray(vref, float).reshape(N + 1)
    key = (float(Ts), int(N), _freeze(params), q_c, q_phi, q_vx, _freeze(R), _freeze(Rd), _freeze(u_bounds),
           _freeze(du_bounds), _freeze(x_lo), _freeze(x_hi), _freeze(solver_opts), device)
    ctl = _SHIM_CACHE.get(key)
    if ctl is None:
        if len(_SHIM_CACHE) >= 16:                          # a caller that varies the settings every call must not leak handles
            _SHIM_CACHE.pop(next(iter(_SHIM_CACHE))).close()
        ctl = BatchedMPC(device=device, Ts=Ts, N=N, params=params, q_c=q_c, q_phi=q_phi, q_vx=q_vx, R=R, Rd=Rd,
                         u_bounds=u_bounds, du_bounds=du_bounds, x_lo=x_lo, x_hi=x_hi, solver_opts=solver_opts)
        _SHIM_CACHE[key] = ctl
    out = ctl.step(x0[None], u_pr[None], path_ref[None], vref_a[None])
    code = int(out["status"][0])
    status = _lib.STATUS_STRINGS[code]
    if code not in _lib.ACCEPTED:                           # :261-262
        return u_pr, status, {}
    u_cmd = out["u_cmd"][0].copy()
    info = {"status": status, "objective": float(out["objective"][0]), "X_opt": out["X_opt"][0].T.copy(),
            "U_opt": out["U_opt"][0].T.copy(), "path_ref": path_ref, "vref": vref_a,
            "iters": int(out["iters"][0]), "y_opt": out["y_opt"][0].copy()}
    return u_cmd, status, info
