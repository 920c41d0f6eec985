"""Closed-loop MPC dataset generation on B200: the drop-in for the generators' hot path.

Mirrors the shell of generation_traj/generation_type2.py:162-220 (x0 sampling, per-trajectory seeds,
plant clipping, Gaussian sensor noise, clean/noisy rows) and the closed loop of MPC/main.py:85-101,
with the control sequence produced by the MPC instead of the open-loop synthesis.  All T steps of all
B trajectories run inside ONE kernel launch (tg_closed_loop); this module builds the per-trajectory
scenario table, calls the C ABI and lays the results out in the reference's dataset schema.
"""
import ctypes

import numpy as np

from . import _lib
from .mpc import BatchedMPC, Params, _plant_table, _plant_arg  # noqa: F401

PATH_PARABOLA, PATH_SINE, PATH_SPLINE, PATH_ARC = 0, 1, 2, 3
VREF_HOLD, VREF_CONST, VREF_RAMP, VREF_TRAPEZOID, VREF_SINE = 0, 1, 2, 3, 4

CLEAN_COLS = ["t", "X", "Y", "phi", "vx", "vy", "omega", "d", "delta", "trajectory_id"]   # generation_type1.py:327
NOISY_COLS = ["t", "X", "Y", "vx", "vy", "omega", "d", "delta", "trajectory_id"]
# generation_type1.py:260-265 / generation_type2.py:171-174
X0_RANGES_TYPE1 = ((-2.0, 2.0), (-2.0, 2.0), (-np.pi, np.pi), (0.4, 1.5), (-0.05, 0.05), (-1.0, 1.0))
X0_RANGES_TYPE2 = ((-2.0, 2.0), (-2.0, 2.0), (-np.pi, np.pi), (0.2, 0.6), (-0.05, 0.05), (-1.0, 1.0))


def d_steady_state(v, p=Params):
    """MPC/main.py:9-18."""
    return (p["Cr0"] + p["Cr2"] * v ** 2) / (p["Cm1"] - p["Cm2"] * v)


class Scenarios:
    """Per-trajectory reference scenarios (tg_ref_spec table + shared spline tables)."""

    def __init__(self, n):
        self.spec = np.zeros(n, dtype=_lib.REF_SPEC_DTYPE)
        self.spec["path_kind"] = PATH_PARABOLA
        self.spec["path"][:, 0] = 0.1                      # MPC/main.py:64
        self.spec["vref_kind"] = VREF_RAMP
        self.spec["vref"][:, :3] = (0.8, 2.0, 2.0)         # MPC/main.py:87
        self._breaks, self._coef = [], []

    def __len__(self):
        return len(self.spec)

    @classmethod
    def from_arrays(cls, path_kind, path, vref, breaks=None, coef=None, vref_kind=None):
        """Scenario table from plain arrays: path_kind[B], path[B,4], vref[B,6] (+ vref_kind[B], default ramp); spline tables
        breaks[B,P], coef[B,P,4] with trajectory b's pieces at row b (the layout tg_make_scenarios and oracle/scenarios.py use)."""
        B = len(path_kind)
        sc = cls(B)
        sc.spec["path_kind"] = np.asarray(path_kind, np.int32)
        sc.spec["path"] = np.asarray(path, float).reshape(B, 4)
        sc.spec["vref"] = np.asarray(vref, float).reshape(B, 6)
        sc.spec["vref_kind"] = VREF_RAMP if vref_kind is None else np.asarray(vref_kind, np.int32)
        if breaks is not None:
            breaks = np.ascontiguousarray(breaks, float); coef = np.ascontiguousarray(coef, float)
            P = breaks.shape[1]
            sc._breaks, sc._coef = [breaks.reshape(-1)], [coef.reshape(-1, 4)]
            sc.spec["spline_first"] = np.arange(B) * P
            sc.spec["spline_count"] = P
        return sc

    def set_parabola(self, i, c2=0.1, c1=0.0, c0=0.0):
        self.spec["path_kind"][i] = PATH_PARABOLA
        self.spec["path"][i] = np.stack(np.broadcast_arrays(c2, c1, c0, 0.0), -1)

    def set_sine(self, i, A=0.5, k=0.5, psi=0.0, c0=0.0):
        self.spec["path_kind"][i] = PATH_SINE
        self.spec["path"][i] = np.stack(np.broadcast_arrays(A, k, psi, c0), -1)

    def set_spline(self, i, knots_x, knots_y):
        """natural cubic spline y(x) through the knots (scipy CubicSpline, as generation_type1.py:97 uses)."""
        from scipy.interpolate import CubicSpline
        cs = CubicSpline(np.asarray(knots_x, float), np.asarray(knots_y, float), bc_type="natural")
        first = sum(len(b) for b in self._breaks)
        K = cs.c.shape[1]
        self._breaks.append(np.asarray(cs.x[:K], float))
        self._coef.append(np.ascontiguousarray(cs.c.T, dtype=float))
        self.spec["path_kind"][i] = PATH_SPLINE
        self.spec["spline_first"][i] = first
        self.spec["spline_count"][i] = K

    def set_splines(self, idx, knots_x, knots_y):
        """natural cubic splines for many trajectories at once: idx[M] trajectory indices, knots_x[M,K] (increasing along
        axis 1), knots_y[M,K].  Same result as M calls of set_spline (scipy's CubicSpline(bc_type='natural') coefficients to
        rounding), but the tridiagonal systems are solved for the whole batch with array operations."""
        idx = np.asarray(idx)
        X = np.asarray(knots_x, float); Y = np.asarray(knots_y, float)
        M, K = X.shape
        h = np.diff(X, axis=1)                                  # [M, K-1]
        d = np.diff(Y, axis=1) / h
        # second derivatives m_0 = m_{K-1} = 0;  h_{i-1} m_{i-1} + 2 (h_{i-1} + h_i) m_i + h_i m_{i+1} = 6 (d_i - d_{i-1})
        n = K - 2
        m = np.zeros((M, K))
        if n > 0:
            a = h[:, :-1].copy(); b = 2.0 * (h[:, :-1] + h[:, 1:]); c = h[:, 1:].copy(); r = 6.0 * (d[:, 1:] - d[:, :-1])
            for i in range(1, n):                               # Thomas algorithm, vectorised over the batch
                w = a[:, i] / b[:, i - 1]
                b[:, i] -= w * c[:, i - 1]
                r[:, i] -= w * r[:, i - 1]
            sol = np.zeros((M, n))
            sol[:, -1] = r[:, -1] / b[:, -1]
            for i in range(n - 2, -1, -1):
                sol[:, i] = (r[:, i] - c[:, i] * sol[:, i + 1]) / b[:, i]
            m[:, 1:-1] = sol
        # piece i on [x_i, x_{i+1}]: y = c0 dx^3 + c1 dx^2 + c2 dx + c3 (scipy PPoly order)
        c0 = (m[:, 1:] - m[:, :-1]) / (6.0 * h)
        c1 = m[:, :-1] / 2.0
        c2 = d - h * (2.0 * m[:, :-1] + m[:, 1:]) / 6.0
        c3 = Y[:, :-1]
        coef = np.stack([c0, c1, c2, c3], axis=-1)              # [M, K-1, 4]
        first = sum(len(b_) for b_ in self._breaks)
        self._breaks.append(X[:, :-1].reshape(-1))
        self._coef.append(coef.reshape(-1, 4))
        self.spec["path_kind"][idx] = PATH_SPLINE
        self.spec["spline_first"][idx] = first + np.arange(M) * (K - 1)
        self.spec["spline_count"][idx] = K - 1
        return coef

    def set_arc(self, i, px, py, s_start=0.0):
        """Arclength-parameterised reference path through the way-points (px, py) -- a path that need not be a graph over X
        (U-turns, loops; SURVEY.md 8(f) rank 3): natural cubic splines x(s), y(s), s = cumulative chord length.  The window is
        anchored at the path point closest to the vehicle, searched from ``s_start`` on the first step and tracked afterwards.
        Table layout: K pieces of x(s) followed by K pieces of y(s) (the breaks are stored twice so that one index serves both
        tables)."""
        from scipy.interpolate import CubicSpline
        px = np.asarray(px, float); py = np.asarray(py, float)
        sk = np.concatenate([[0.0], np.cumsum(np.hypot(np.diff(px), np.diff(py)))])
        cx, cy = CubicSpline(sk, px, bc_type="natural"), CubicSpline(sk, py, bc_type="natural")
        first = sum(len(b) for b in self._breaks)
        K = cx.c.shape[1]
        self._breaks.append(np.concatenate([sk[:K], sk[:K]]))
        self._coef.append(np.ascontiguousarray(np.concatenate([cx.c.T, cy.c.T], axis=0), dtype=float))
        self.spec["path_kind"][i] = PATH_ARC
        self.spec["spline_first"][i] = first
        self.spec["spline_count"][i] = K
        self.spec["path"][i] = (float(s_start), 0.0, 0.0, 0.0)
        return sk

    def set_vref(self, i, kind, *prm):
        self.spec["vref_kind"][i] = kind
        cols = list(prm) + [0.0] * (6 - len(prm))
        self.spec["vref"][i] = np.stack(np.broadcast_arrays(*cols), -1)

    def tables(self):
        if not self._breaks:
            return np.zeros(0), np.zeros((0, 4))
        return np.ascontiguousarray(np.concatenate(self._breaks)), np.ascontiguousarray(np.concatenate(self._coef, axis=0))

    def slice(self, lo, hi):
        s = Scenarios(0)
        s.spec = self.spec[lo:hi].copy()
        s._breaks, s._coef = self._breaks, self._coef      # spline_first indexes the shared tables
        return s


def scenario_rules(**overrides):
    """tg_scenario_rules with the library defaults (BASELINE config 2: spline / sinusoid references by id parity, x0 from
    generation_type1.py:260-265's ranges); keyword overrides by field name, e.g. cycle=(PATH_PARABOLA, PATH_SINE, PATH_SPLINE),
    x0_lo=..., seed_base=...."""
    r = _lib.TgScenarioRules()
    _lib.load().tg_default_scenario_rules(ctypes.byref(r))
    for k, v in overrides.items():
        if k == "cycle":
            v = list(v)
            r.n_cycle = len(v)
            for i, kind in enumerate(v):
                r.cycle[i] = int(kind)
            continue
        if not hasattr(r, k):
            raise TypeError(f"unknown scenario rule {k!r}")
        cur = getattr(r, k)
        if isinstance(cur, ctypes.Array):
            v = list(np.asarray(v, float).ravel())
            if len(v) != len(cur):
                raise ValueError(f"{k}: expected {len(cur)} values")
            for i, x in enumerate(v):
                cur[i] = x
        else:
            setattr(r, k, type(cur)(v))
    return r


class ClosedLoopGenerator(BatchedMPC):
    """MPC-in-the-loop trajectory generator.  Keyword arguments are mpc_step's plus ``plant``
    (PLANT_MPC = MPC/main.py:97; PLANT_GEN1/2 = the generators' clipped plants), ``warm_start``,
    ``noise_std`` and ``noise_seed_base`` (generation_type2.py:31-43,191)."""

    def __init__(self, device=0, warm_start=True, **kwargs):
        super().__init__(device=device, warm_start=warm_start, **kwargs)

    def plant_table(self, B, **columns):
        """A [B, 17] table of per-trajectory plant parameters for ``generate`` / ``plant_rollout`` (C-contiguous fp64, columns in
        PARAM_ORDER).  Every row starts as this handle's ``params``; a keyword named as in PARAM_ORDER sets a column to a scalar or
        a [B] array, e.g. ``plant_table(B, m=0.041 * rng.uniform(0.8, 1.2, B))``.  Only the plant (the ground truth) integrates
        the table; the controller keeps the handle's model.  Rows that keep Bf, Cf, Br, Cr and maxAlpha keep the handle's tyre
        tables; rows that change them evaluate the tyre curve with libdevice (include/trajgen.h).  Checked: raises ValueError
        naming the first bad row and column."""
        return _plant_table(self.cfg.params, B, columns)

    @staticmethod
    def alloc_result(B, T, pinned=True):
        """result buffers of one generate() call: dict(clean[B,T+1,6], noisy[B,T+1,6], U[B,T,2], status_counts[B,6],
        iters_total[B]).  pinned=True: page-locked memory, into which the kernel stores its rows directly."""
        mk = _lib.pinned_empty if pinned else np.empty
        return {"clean": mk((B, T + 1, 6)), "noisy": mk((B, T + 1, 6)), "U": mk((B, T, 2)),
                "status_counts": np.zeros((B, _lib.TG_NUM_STATUS), np.int32), "iters_total": np.zeros(B, np.int64)}

    #: generate() streams batches whose result rows exceed this many bytes through two page-locked chunk buffers
    STREAM_BYTES = 1 << 30

    def generate(self, x0, u0, scenarios, T, traj_id0=0, out=None, pinned=True, chunk=None, ctrl=None, plant_params=None):
        """x0[B,6], u0[B,2], scenarios (len B), T steps -> dict(clean[B,T+1,6], noisy[B,T+1,6], U[B,T,2],
        status_counts[B,6], iters_total[B]).  Row 0 of clean is x0; noise seed = base + traj_id0 + i.
        The result arrays are page-locked by default (``pinned``), so the kernel writes its rows straight into them
        while it runs (112 B per MPC step: far below what PCIe carries) and nothing is copied afterwards; ``out`` re-uses
        the buffers of an earlier call (see ``alloc_result``).  Page-locking gigabytes takes longer than generating them, so
        a batch whose rows exceed STREAM_BYTES (or any batch when ``chunk`` is given) is generated in chunks through two
        cached page-locked chunk buffers (generate_chunks) and gathered into ordinary arrays by host threads while the next
        chunk computes.  ``ctrl``: a [B] table of per-trajectory weights and bounds (``ctrl_table``), held for all T steps;
        None = the handle's settings for every trajectory.  ``plant_params``: a [B, 17] table of per-trajectory plant
        parameters (``plant_table``): trajectory b's ground truth integrates row b while its controller keeps the handle's model;
        None = the handle's params for every plant."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B, T = x0.shape[0], int(T)
        u0 = self._arr(np.asarray(u0, float).reshape(-1, 2), (B, 2))
        if len(scenarios) != B:
            raise ValueError("one scenario per trajectory required")
        ctrl = None if ctrl is None else self._ctrl_arg(ctrl, B)
        plant_params = _plant_arg(plant_params, B)
        row_bytes = (2 * (T + 1) * 6 + T * 2) * 8
        if out is None and (chunk is not None or (pinned and B * row_bytes > self.STREAM_BYTES)):
            return self._generate_streamed(x0, u0, scenarios, T, traj_id0, chunk, ctrl=ctrl, plant_params=plant_params)
        spec = np.ascontiguousarray(scenarios.spec)
        brk, coef = scenarios.tables()
        if out is None:
            out = self.alloc_result(B, T, pinned)
        elif out["clean"].shape != (B, T + 1, 6) or out["U"].shape != (B, T, 2):
            raise ValueError("`out` was allocated for another batch size / horizon")
        _lib.check(_lib.load().tg_closed_loop_params_host(
            self._h, B, T, _lib.ptr(x0), _lib.ptr(u0), spec.ctypes.data, _lib.ptr(ctrl), _lib.ptr(plant_params),
            _lib.ptr(brk) if len(brk) else None,
            len(brk), _lib.ptr(coef) if len(coef) else None, len(coef), int(traj_id0),
            _lib.ptr(out["clean"]), _lib.ptr(out["noisy"]), _lib.ptr(out["U"]), _lib.ptr(out["status_counts"]),
            _lib.ptr(out["iters_total"])))
        return out

    def close(self):
        """destroys the handle and releases the cached page-locked chunk buffers"""
        self._chunk_bufs = None
        self._chunk_key = None
        super().close()

    def _chunk_buffers(self, nb, T):
        """two page-locked result sets for chunks of nb trajectories x T steps, cached on the generator"""
        key = (int(nb), int(T))
        if getattr(self, "_chunk_key", None) != key:
            self._chunk_bufs = None                      # release the previous pair first
            self._chunk_bufs = [self.alloc_result(nb, T), self.alloc_result(nb, T)]
            self._chunk_key = key
        return self._chunk_bufs

    def generate_chunks(self, x0, u0, scenarios, T, traj_id0=0, chunk=None, ctrl=None, plant_params=None):
        """Iterator over a large batch: yields (lo, hi, res) with res = the result dict of trajectories lo .. hi - 1 as views of
        one of two page-locked chunk buffers.  The GPU computes chunk k + 1 (a host thread sits in tg_closed_loop_host, which
        releases the GIL) while the caller consumes chunk k; a yielded view stays valid until the caller asks for the
        next-but-one chunk.  ``chunk`` defaults to 8192 trajectories (1.1 GB of rows at T = 1200).  ``ctrl`` and
        ``plant_params`` ([B] tables, see ``generate``) are sliced with the scenarios."""
        from concurrent.futures import ThreadPoolExecutor
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        u0 = np.ascontiguousarray(np.asarray(u0, float).reshape(-1, 2))
        B, T = x0.shape[0], int(T)
        ctrl = None if ctrl is None else self._ctrl_arg(ctrl, B)   # checked before the first chunk is launched
        plant_params = _plant_arg(plant_params, B)
        chunk = int(chunk) if chunk else 8192
        nb = min(chunk, B)
        bufs = self._chunk_buffers(nb, T)
        los = list(range(0, B, chunk))

        def run(k):
            lo = los[k]; hi = min(lo + chunk, B)
            res = {k_: v[:hi - lo] for k_, v in bufs[k % 2].items()}
            ClosedLoopGenerator.generate(self, x0[lo:hi], u0[lo:hi], scenarios.slice(lo, hi), T, traj_id0 + lo, out=res,
                                         ctrl=None if ctrl is None else ctrl[lo:hi],
                                         plant_params=None if plant_params is None else plant_params[lo:hi])
            return lo, hi, res

        with ThreadPoolExecutor(1) as ex:
            fut = ex.submit(run, 0)
            for k in range(len(los)):
                item = fut.result()
                if k + 1 < len(los):
                    fut = ex.submit(run, k + 1)          # into the buffer the caller released when it asked for this chunk
                yield item

    def _generate_streamed(self, x0, u0, scenarios, T, traj_id0, chunk, n_copy_threads=4, ctrl=None, plant_params=None):
        from concurrent.futures import ThreadPoolExecutor
        B = x0.shape[0]
        out = self.alloc_result(B, T, pinned=False)
        with ThreadPoolExecutor(n_copy_threads) as pool:
            for lo, hi, res in self.generate_chunks(x0, u0, scenarios, T, traj_id0, chunk, ctrl=ctrl, plant_params=plant_params):
                jobs = []
                step = max(1, (hi - lo + n_copy_threads - 1) // n_copy_threads)
                for a in range(0, hi - lo, step):        # ndarray copies release the GIL: first touch + copy on several cores
                    b = min(a + step, hi - lo)
                    for k_ in ("clean", "noisy", "U"):
                        jobs.append(pool.submit(np.copyto, out[k_][lo + a:lo + b], res[k_][a:b]))
                out["status_counts"][lo:hi] = res["status_counts"]; out["iters_total"][lo:hi] = res["iters_total"]
                for j in jobs:
                    j.result()
        return out

    def generate_to_csv(self, x0, u0, scenarios, T, clean_path, noisy_path, traj_id0=0, chunk=8192, keep=False, n_threads=0,
                        csv_ids=None, ctrl=None, plant_params=None):
        """generate() in chunks of ``chunk`` trajectories with the dataset files written as it goes (the reference holds
        every DataFrame in RAM and writes once at the end, generation_type2.py:166,216-218,319-322): while the GPU computes
        chunk k + 1 into one set of pinned buffers, the host formats chunk k from the other (tg_write_csv, all cores,
        appending).  ``csv_ids``: write only the first csv_ids trajectories to the files (BASELINE config 5: CSV for the
        first 5 000 ids, the rest stays binary).  ``ctrl``, ``plant_params``: per-trajectory tables as in ``generate`` (the
        files do not record the plant table: the caller keeps it).  Returns
        dict(status_counts[B,6], iters_total[B]) (+ the rows if ``keep``)."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B, T = x0.shape[0], int(T)
        n_csv = B if csv_ids is None else min(int(csv_ids), B)
        out = {"status_counts": np.zeros((B, _lib.TG_NUM_STATUS), np.int32), "iters_total": np.zeros(B, np.int64)}
        if keep:
            out.update({k_: v for k_, v in self.alloc_result(B, T, pinned=False).items() if k_ in ("clean", "noisy", "U")})
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(1) as writer:                # one writer: chunks are appended in order
            pending = []
            for lo, hi, res in self.generate_chunks(x0, u0, scenarios, T, traj_id0, chunk, ctrl=ctrl, plant_params=plant_params):
                out["status_counts"][lo:hi] = res["status_counts"]; out["iters_total"][lo:hi] = res["iters_total"]
                if keep:
                    for k_ in ("clean", "noisy", "U"):
                        np.copyto(out[k_][lo:hi], res[k_])
                if lo < n_csv:
                    # the rows leave the page-locked chunk buffer before they are formatted, so that the GPU gets the buffer back
                    # at once and the text is produced beside the following chunks
                    m = min(hi, n_csv) - lo
                    rows = {k_: (out[k_][lo:lo + m] if keep else res[k_][:m].copy()) for k_ in ("clean", "noisy", "U")}
                    pending.append(writer.submit(write_csv, rows, self.cfg.Ts, clean_path, noisy_path, traj_id0=traj_id0 + lo,
                                                 append=lo > 0, n_threads=n_threads))
            for f in pending:
                f.result()
        return out

    def make_scenarios(self, B, rules=None, traj_id0=0):
        """Initial states, steady-state inputs and reference scenarios for trajectory ids traj_id0 .. traj_id0 + B - 1, generated
        on the device (tg_make_scenarios: Philox draws keyed by the global id, natural-spline fits per trajectory) and returned
        as host arrays: (x0[B,6], u0[B,2], Scenarios)."""
        rules = rules if rules is not None else scenario_rules()
        P = rules.spl_knots - 1
        x0, u0 = np.empty((B, 6)), np.empty((B, 2))
        sc = Scenarios(B)
        brk, coef = np.empty(B * P), np.empty((B * P, 4))
        _lib.check(_lib.load().tg_make_scenarios_host(self._h, int(B), int(traj_id0), ctypes.byref(rules), _lib.ptr(x0), _lib.ptr(u0),
                                                      sc.spec.ctypes.data, _lib.ptr(brk), _lib.ptr(coef)))
        sc._breaks, sc._coef = [brk], [coef]
        return x0, u0, sc

    def ref_window(self, x0, scenarios, t_index=0):
        """a10 tap: -> path_ref[B,N+1,3], vref[B,N+1] (MPC/main.py:87-90)."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B, N = x0.shape[0], self.N
        spec = np.ascontiguousarray(scenarios.spec)
        brk, coef = scenarios.tables()
        bufs = self._on_device([x0, spec.view(np.uint8), brk if len(brk) else None, coef if len(coef) else None])
        op, ov = _lib.DeviceBuffer(B * (N + 1) * 3 * 8, self._h), _lib.DeviceBuffer(B * (N + 1) * 8, self._h)
        _lib.check(_lib.load().tg_ref_window(self._h, B, bufs[0].ptr, bufs[1].ptr, bufs[2].ptr if bufs[2] else None,
                                             bufs[3].ptr if bufs[3] else None, int(t_index), op.ptr, ov.ptr))
        return self._from_device(op, (B, N + 1, 3)), self._from_device(ov, (B, N + 1))

    def plant_rollout(self, x0, U, plant_params=None):
        """K4 tap: open-loop Euler integration with the configured plant (generation_type1.py:70-84); ``plant_params``: a
        [B, 17] table (``plant_table``) of per-trajectory vehicles, None = the handle's params."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B = x0.shape[0]
        U = np.ascontiguousarray(np.asarray(U, float))
        T = U.shape[1]
        plant_params = _plant_arg(plant_params, B)
        bx, bu, bp = self._on_device([x0, U, plant_params])
        oX = _lib.DeviceBuffer(B * (T + 1) * 6 * 8, self._h)
        _lib.check(_lib.load().tg_plant_rollout_params(self._h, B, T, bx.ptr, bu.ptr, bp.ptr if bp else None, oX.ptr))
        return self._from_device(oX, (B, T + 1, 6))

    def sensor_noise_normals(self, traj_id0, n_traj, n_rows):
        """K4 tap: standard normals [n_traj, n_rows, 6] of seeds noise_seed_base + traj_id0 + i."""
        o = _lib.DeviceBuffer(max(n_traj * n_rows * 6 * 8, 8), self._h)
        _lib.check(_lib.load().tg_sensor_noise(self._h, int(traj_id0), int(n_traj), int(n_rows), o.ptr))
        return self._from_device(o, (n_traj, n_rows, 6))

    def philox_u32(self, seed, first, block, n):
        o = _lib.DeviceBuffer(max(n * 16, 16), self._h)
        _lib.check(_lib.load().tg_philox_u32(self._h, int(seed), int(first), int(block), int(n), o.ptr))
        return self._from_device(o, (n, 4), np.uint32)

    def fma_peak_tflops(self, dtype="f64"):
        v = ctypes.c_double()
        _lib.check(_lib.load().tg_fma_peak(self._h, 0 if dtype == "f64" else 1, ctypes.byref(v)))
        return v.value


# ----------------------------------------------------------------------------------- dataset schema
def sample_x0(num_traj, seed=42, ranges=X0_RANGES_TYPE2):
    """generation_type2.py:164,171-174: six successive rng.uniform draws per trajectory from default_rng(seed)."""
    rng = np.random.default_rng(seed)
    out = np.zeros((num_traj, 6))
    for i in range(num_traj):
        for j, (lo, hi) in enumerate(ranges):
            out[i, j] = rng.uniform(lo, hi)
    return out


def to_frames(result, Ts, traj_id0=0):
    """-> (clean DataFrame, noisy DataFrame) in the reference schema (generation_type2.py:202-216,309-317):
    T+1 rows per trajectory, t = k Ts, last row's d, delta = NaN, noisy has no phi."""
    import pandas as pd
    clean, noisy, U = result["clean"], result["noisy"], result["U"]
    B, T1, _ = clean.shape
    t = np.tile(np.arange(T1) * Ts, B)
    tid = np.repeat(np.arange(traj_id0, traj_id0 + B), T1)
    Upad = np.concatenate([U, np.full((B, 1, 2), np.nan)], axis=1).reshape(B * T1, 2)
    frames = []
    for S in (clean, noisy):
        S2 = S.reshape(B * T1, 6)
        frames.append(pd.DataFrame({"t": t, "X": S2[:, 0], "Y": S2[:, 1], "phi": S2[:, 2], "vx": S2[:, 3],
                                    "vy": S2[:, 4], "omega": S2[:, 5], "d": Upad[:, 0], "delta": Upad[:, 1],
                                    "trajectory_id": tid}))
    return frames[0][CLEAN_COLS], frames[1][NOISY_COLS]


def write_csv(result, Ts, clean_path, noisy_path, traj_id0=0, append=False, engine="native", n_threads=0):
    """clean/noisy CSV files exactly as generation_type2.py:319-322 writes them.  engine="native": the library's
    multi-threaded writer (tg_write_csv, byte-identical to pandas for the same numbers); engine="pandas":
    DataFrame.to_csv(index=False) as the reference does."""
    if engine == "pandas":
        c, n = to_frames(result, Ts, traj_id0)
        c.to_csv(clean_path, index=False, mode="a" if append else "w", header=not append)
        n.to_csv(noisy_path, index=False, mode="a" if append else "w", header=not append)
        return
    clean = np.ascontiguousarray(result["clean"], dtype=np.float64)
    noisy = np.ascontiguousarray(result["noisy"], dtype=np.float64)
    U = np.ascontiguousarray(result["U"], dtype=np.float64)
    B, T1, _ = clean.shape
    _lib.check(_lib.load().tg_write_csv(str(clean_path).encode(), str(noisy_path).encode(), B, T1 - 1, float(Ts), int(traj_id0),
                                        _lib.ptr(clean), _lib.ptr(noisy), _lib.ptr(U) if U.size else None, int(bool(append)),
                                        int(n_threads)))


def merge_datasets(first_clean, second_clean, out_clean, first_noisy=None, second_noisy=None, out_noisy=None):
    """generation_traj/merge_datasets.py:33-70: concatenate two generation runs, re-indexing the second run's
    trajectory ids by max(id of the first clean file) + 1; the noisy pair re-uses the clean pair's offset (:62-63).
    Native streaming merge (tg_merge_csv): rows are copied as text, so no number is re-rounded.  Raises
    TrajgenError("File not found: ...") like the script's check (:23-27).  -> dict(id_offset, rows_clean, rows_noisy)."""
    L = _lib.load()
    off, rows_c, rows_n = _lib.i64(), _lib.i64(), _lib.i64()
    _lib.check(L.tg_merge_csv(str(first_clean).encode(), str(second_clean).encode(), str(out_clean).encode(), -1,
                              ctypes.byref(off), ctypes.byref(rows_c)))
    if first_noisy is not None:
        _lib.check(L.tg_merge_csv(str(first_noisy).encode(), str(second_noisy).encode(), str(out_noisy).encode(), off.value,
                                  None, ctypes.byref(rows_n)))
    return {"id_offset": off.value, "rows_clean": rows_c.value, "rows_noisy": rows_n.value}


def to_loader_tensors(result, T_steps):
    """The arrays KalmanNet/data_loader.py:33-53 would build from the CSVs, without the CSV round trip:
    y[B,5,T] noisy (X,Y,vx,vy,omega), u[B,2,T], x[B,6,T] clean; float32.  Like the loader (:51-53) it takes the first
    T_steps rows of each trajectory's T+1 rows; the controls of the last row are NaN in the files, so asking for all
    T+1 rows gives a NaN last column in u, exactly as the loader does."""
    clean, noisy, U = result["clean"], result["noisy"], result["U"]
    T1 = clean.shape[1]
    if T_steps > T1:
        raise ValueError(f"T_steps = {T_steps} exceeds the {T1} rows per trajectory")
    Upad = np.concatenate([U, np.full((U.shape[0], 1, 2), np.nan)], axis=1)
    y = noisy[:, :T_steps][:, :, [0, 1, 3, 4, 5]].transpose(0, 2, 1).astype(np.float32)
    u = Upad[:, :T_steps].transpose(0, 2, 1).astype(np.float32)
    x = clean[:, :T_steps].transpose(0, 2, 1).astype(np.float32)
    return y, u, x
