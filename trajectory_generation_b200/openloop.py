"""The generators' own open-loop modes on B200 (SURVEY.md section 8(f), rank 2).

``generation_type1.py`` (spline transient + straight / sinusoidal steady steering, slew-limited) and
``generation_type2.py`` (accelerate / cruise / turn state machine on a shadow simulation) synthesise their control
sequences without the MPC.  ``OpenLoopGenerator`` runs either synthesis, the plant integration and the sensor noise
for all trajectories in ONE kernel launch (tg_openloop_type1 / tg_openloop_type2) and returns the same result dict as
``ClosedLoopGenerator.generate`` -- so ``write_csv`` / ``to_loader_tensors`` / ``merge_datasets`` apply unchanged.
Random numbers follow the reference's distributions and seeding contract (seed = base + trajectory id) on a
counter-based Philox4x32-10 stream; ``oracle/openloop.py`` states the stream layout.
"""
import ctypes

import numpy as np

from . import _lib
from .mpc import PLANT_GEN1, PLANT_GEN2, make_config, _plant_table, _plant_arg
from .generation import X0_RANGES_TYPE1, X0_RANGES_TYPE2, sample_x0

TYPE1_MODES = ("straight", "sinusoid")                                # generation_type1.py:108
TYPE2_MODES = ("accelerate", "cruise", "turn_left", "turn_right")     # generation_type2.py:108-112
CTRL_SEED_BASE = 42                                                   # generation_type1.py:17, generation_type2.py:292


def _fill(struct, overrides):
    names = {f[0] for f in struct._fields_}
    for k, v in overrides.items():
        if k not in names:
            raise TypeError(f"unknown rule {k!r}")
        cur = getattr(struct, k)
        if isinstance(cur, ctypes.Array):
            v = list(np.asarray(v, float).reshape(-1))
            if len(v) != len(cur):
                raise ValueError(f"rule {k!r} takes {len(cur)} values")
            for i, x in enumerate(v):
                cur[i] = x
        else:
            setattr(struct, k, v)
    return struct


def type1_rules(**overrides):
    """tg_type1_rules with generation_type1.py's constants (mpc_stats :250, du_bounds :251, ...); du_bounds / u_bounds may be
    given in the reference's ((d_lo, d_hi), (delta_lo, delta_hi)) form."""
    r = _lib.TgType1Rules()
    _lib.load().tg_default_type1_rules(ctypes.byref(r))
    for key, lo, hi in (("du_bounds", "du_lo", "du_hi"), ("u_bounds", "u_lo", "u_hi")):
        if key in overrides:
            b = np.asarray(overrides.pop(key), float).reshape(2, 2)
            overrides[lo], overrides[hi] = b[:, 0], b[:, 1]
    if isinstance(overrides.get("mode"), str):
        overrides["mode"] = -1 if overrides["mode"] == "random" else TYPE1_MODES.index(overrides["mode"])
    return _fill(r, overrides)


def type2_rules(**overrides):
    """tg_type2_rules with generation_type2.py's ControlRules (:21-30) and the literals of sample_controls_piecewise."""
    r = _lib.TgType2Rules()
    _lib.load().tg_default_type2_rules(ctypes.byref(r))
    return _fill(r, overrides)


class OpenLoopGenerator:
    """kind = "type1" | "type2".  ``generate(x0, T)`` replaces the per-trajectory loop of generation_type1.py:267-312 /
    generation_type2.py:169-216 (control synthesis, ground-truth integration, sensor noise)."""

    def __init__(self, kind="type2", Ts=0.01, device=0, plant=None, params=None, noise_std=None, noise_seed_base=None,
                 ctrl_seed_base=CTRL_SEED_BASE, **rules):
        if kind not in ("type1", "type2"):
            raise ValueError("kind must be 'type1' or 'type2'")
        self.kind, self.Ts, self.ctrl_seed_base = kind, float(Ts), int(ctrl_seed_base)
        if plant is None:
            plant = PLANT_GEN1 if kind == "type1" else PLANT_GEN2
        kw = dict(N=1, Ts=Ts, plant=plant, model=plant, params=params)
        if noise_std is not None:
            kw["noise_std"] = noise_std
        if noise_seed_base is not None:
            kw["noise_seed_base"] = noise_seed_base
        self.cfg = make_config(**kw)
        self.rules = type1_rules(**rules) if kind == "type1" else type2_rules(**rules)
        self._h = _lib.vp()
        _lib.check(_lib.load().tg_create(ctypes.byref(self.cfg), int(device), ctypes.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().tg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sample_x0(self, num_traj, seed=42):
        """the generator's own initial-state ranges (generation_type1.py:260-265 / generation_type2.py:171-174)."""
        return sample_x0(num_traj, seed, X0_RANGES_TYPE1 if self.kind == "type1" else X0_RANGES_TYPE2)

    def plant_table(self, B, **columns):
        """A [B, 17] table of per-trajectory plant parameters for ``generate`` (see ClosedLoopGenerator.plant_table): rows start as
        this handle's params, keywords named as in PARAM_ORDER set a column to a scalar or a [B] array.  Checked."""
        return _plant_table(self.cfg.params, B, columns)

    def generate(self, x0, T, traj_id0=0, want=("clean", "noisy", "U", "modes"), plant_params=None):
        """x0[B,6], T steps -> dict(clean[B,T+1,6], noisy[B,T+1,6], U[B,T,2], modes): modes[B] (type 1: 0 straight,
        1 sinusoid) or modes[B,T] (type 2: index into TYPE2_MODES).  ``plant_params``: a [B, 17] table (``plant_table``) with
        which trajectory b's ground truth is integrated; None = the handle's params."""
        x0 = np.ascontiguousarray(np.asarray(x0, float).reshape(-1, 6))
        B, T = x0.shape[0], int(T)
        plant_params = _plant_arg(plant_params, B)
        out = {}
        if "clean" in want:
            out["clean"] = np.empty((B, T + 1, 6))
        if "noisy" in want:
            out["noisy"] = np.empty((B, T + 1, 6))
        if "U" in want:
            out["U"] = np.empty((B, T, 2))
        if "modes" in want:
            out["modes"] = np.zeros(B if self.kind == "type1" else (B, T), dtype=np.int8)
        fn = getattr(_lib.load(), f"tg_openloop_{self.kind}_params_host")
        _lib.check(fn(self._h, B, T, _lib.ptr(x0), ctypes.byref(self.rules), self.ctrl_seed_base, int(traj_id0),
                      _lib.ptr(plant_params), _lib.ptr(out.get("clean")), _lib.ptr(out.get("noisy")), _lib.ptr(out.get("U")), _lib.ptr(out.get("modes"))))
        return out

    def generate_device(self, x0_dev, B, T, clean_dev=None, noisy_dev=None, U_dev=None, modes_dev=None, traj_id0=0,
                        plant_dev=None):
        """device-pointer form (asynchronous on the handle's stream): tg_openloop_type{1,2}_params.  ``plant_dev``: device
        pointer of a [B, 17] plant table or None; its rules (check_plant_table) are the caller's to keep."""
        fn = getattr(_lib.load(), f"tg_openloop_{self.kind}_params")
        _lib.check(fn(self._h, int(B), int(T), x0_dev, ctypes.byref(self.rules), self.ctrl_seed_base, int(traj_id0),
                      plant_dev, clean_dev, noisy_dev, U_dev, modes_dev))

    def synchronize(self):
        _lib.check(_lib.load().tg_synchronize(self._h))

    def set_stream(self, cuda_stream):
        _lib.check(_lib.load().tg_set_stream(self._h, cuda_stream))

    def kernel_launches(self):
        n = _lib.i64()
        _lib.check(_lib.load().tg_kernel_launches(self._h, ctypes.byref(n)))
        return n.value
