"""ctypes binding of libtrajgen.so (include/trajgen.h).  No CPU fallback: if the library is missing
or no B200 is visible, the first use raises."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TRAJGEN_LIB", os.path.join(_HERE, "libtrajgen.so"))
CSRC = os.path.join(_HERE, "csrc")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "--shared", "-Xcompiler", "-fPIC"]

TG_INF = 1e20
TG_NPARAMS = 17
TG_NUM_STATUS = 6
PARAM_ORDER = ("Cm1", "Cm2", "Cr0", "Cr2", "Br", "Cr", "Dr", "Bf", "Cf", "Df", "m", "Iz", "lf", "lr", "g",
               "maxAlpha", "vx_zero")
# mpc_step's status strings (MPC/mpc_6stati.py:257-262)
STATUS_STRINGS = ("optimal", "optimal_inaccurate", "infeasible", "unbounded", "user_limit", "Solver Error: NumericalFailure")
ACCEPTED = (0, 1)

d, i32, i64, u64, vp = ctypes.c_double, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.c_void_p


class TgConfig(ctypes.Structure):
    _fields_ = [
        ("N", i32), ("model", i32), ("plant", i32), ("jacobian", i32),
        ("Ts", d), ("params", d * TG_NPARAMS),
        ("q_c", d), ("q_phi", d), ("q_vx", d), ("R", d * 4), ("Rd", d * 4),
        ("u_lo", d * 2), ("u_hi", d * 2), ("du_lo", d * 2), ("du_hi", d * 2),
        ("x_lo", d * 6), ("x_hi", d * 6),
        ("rho", d), ("sigma", d), ("alpha", d), ("eps_abs", d), ("eps_rel", d), ("eps_prim_inf", d),
        ("adaptive_rho_tol", d), ("alpha_warm", d),
        ("max_iter", i32), ("check_every", i32), ("adaptive_rho", i32), ("adaptive_rho_min_iter", i32),
        ("warm_start", i32), ("vref_advance", i32),
        ("noise_std", d * 6), ("noise_seed_base", u64),
        ("threads_per_problem", i32), ("solver_flags", i32),
    ]


class TgType1Rules(ctypes.Structure):
    """include/trajgen.h::tg_type1_rules (generation_type1.py's constants)."""
    _fields_ = [
        ("d_mean", d), ("d_std", d), ("delta_mean", d), ("delta_std", d),
        ("du_lo", d * 2), ("du_hi", d * 2), ("u_lo", d * 2), ("u_hi", d * 2),
        ("transient_s", d * 2), ("checkpoint_s", d * 2), ("period_s", d * 2), ("amp_frac", d * 2),
        ("p_straight", d), ("tr_d_frac", d), ("tr_delta_frac", d), ("st_d_frac", d),
        ("sin_noise_frac", d), ("straight_frac", d), ("ctrl_noise_frac", d),
        ("mode", i32), ("reserved", i32),
    ]


class TgType2Rules(ctypes.Structure):
    """include/trajgen.h::tg_type2_rules (generation_type2.py's ControlRules + literals)."""
    _fields_ = [
        ("v_turn_max", d), ("v_high", d), ("d_range", d * 2), ("delta_turn_range", d * 2),
        ("delta_straight_noise", d), ("delta_rate_max", d), ("v_floor", d), ("d_boost_min", d),
        ("seg_s", d * 2), ("p_modes", d * 4), ("p_after_turn", d * 2), ("acc_d_lo", d), ("cruise_d", d * 2),
        ("turn_d_fast", d * 2), ("turn_d_slow", d * 2), ("stall_v", d), ("stall_d", d * 2), ("stall_min_s", d),
        ("delta_clip", d),
    ]


class TgScenarioRules(ctypes.Structure):
    """include/trajgen.h::tg_scenario_rules."""
    _fields_ = [
        ("x0_lo", d * 6), ("x0_hi", d * 6), ("lat_off", d * 2), ("head_off", d * 2),
        ("vref0", d), ("vcruise", d * 2), ("t_ramp", d),
        ("sine_A", d * 2), ("sine_k", d * 2), ("sine_psi", d * 2), ("parab_c", d * 2),
        ("spl_x0", d), ("spl_dx", d * 2), ("spl_sigma", d),
        ("spl_knots", i32), ("n_cycle", i32), ("cycle", i32 * 4), ("reserved", i32), ("seed_base", u64),
    ]


class TgStateLimits(ctypes.Structure):
    _fields_ = [("lo", d * 6), ("hi", d * 6)]


REF_SPEC_DTYPE = np.dtype([("path_kind", np.int32), ("vref_kind", np.int32), ("spline_first", np.int32),
                           ("spline_count", np.int32), ("path", np.float64, 4), ("vref", np.float64, 6)], align=True)
assert REF_SPEC_DTYPE.itemsize == 96

# include/trajgen.h::tg_ctrl_spec: one row of per-problem / per-trajectory controller settings
CTRL_SPEC_DTYPE = np.dtype([("q_c", np.float64), ("q_phi", np.float64), ("q_vx", np.float64), ("R", np.float64, 4),
                            ("Rd", np.float64, 4), ("u_lo", np.float64, 2), ("u_hi", np.float64, 2), ("du_lo", np.float64, 2),
                            ("du_hi", np.float64, 2), ("x_lo", np.float64, 6), ("x_hi", np.float64, 6)], align=True)
assert CTRL_SPEC_DTYPE.itemsize == 248

# every symbol include/trajgen.h declares
EXPORTS = (
    "tg_last_error", "tg_version", "tg_default_config", "tg_create", "tg_destroy", "tg_set_stream", "tg_synchronize",
    "tg_kernel_launches", "tg_info", "tg_tyre_table_info", "tg_linearize", "tg_assemble", "tg_mpc_step", "tg_mpc_step_host",
    "tg_mpc_step_ctrl", "tg_mpc_step_ctrl_host", "tg_check_ctrl", "tg_ref_window",
    "tg_closed_loop", "tg_closed_loop_host", "tg_closed_loop_ctrl", "tg_closed_loop_ctrl_host", "tg_check_plant_params",
    "tg_closed_loop_params", "tg_closed_loop_params_host", "tg_plant_rollout_params", "tg_openloop_type1_params",
    "tg_openloop_type2_params", "tg_openloop_type1_params_host", "tg_openloop_type2_params_host", "tg_default_scenario_rules", "tg_make_scenarios", "tg_make_scenarios_host", "tg_default_type1_rules", "tg_default_type2_rules", "tg_openloop_type1",
    "tg_openloop_type2", "tg_openloop_type1_host", "tg_openloop_type2_host", "tg_write_csv", "tg_merge_csv", "tg_estimator_step", "tg_estimator_step_vjp",
    "tg_estimator_rollout", "tg_plant_rollout", "tg_sensor_noise", "tg_philox_u32", "tg_fma_peak",
    "tg_device_count", "tg_malloc", "tg_malloc_on", "tg_free", "tg_memcpy_h2d", "tg_memcpy_d2h", "tg_malloc_host", "tg_free_host",
)

_lib = None


class TrajgenError(RuntimeError):
    pass


def build(verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> libtrajgen.so (in-tree)."""
    src = os.path.join(CSRC, "trajgen.cu")
    src_csv = os.path.join(CSRC, "tg_csv.cpp")
    deps = [src, src_csv] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    deps.append(os.path.join(_HERE, "..", "include", "trajgen.h"))
    if os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(p) for p in deps):
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + ["-o", LIB_PATH, src, src_csv]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB_PATH


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TrajgenError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH)
    L.tg_last_error.restype = ctypes.c_char_p
    L.tg_default_config.argtypes = [ctypes.POINTER(TgConfig)]
    L.tg_default_config.restype = None
    L.tg_create.argtypes = [ctypes.POINTER(TgConfig), ctypes.c_int, ctypes.POINTER(vp)]
    L.tg_destroy.argtypes = [vp]
    L.tg_set_stream.argtypes = [vp, vp]
    L.tg_synchronize.argtypes = [vp]
    L.tg_kernel_launches.argtypes = [vp, ctypes.POINTER(i64)]
    L.tg_info.argtypes = [vp] + [ctypes.POINTER(i32)] * 4
    L.tg_tyre_table_info.argtypes = [vp, ctypes.POINTER(i32), ctypes.POINTER(d), ctypes.POINTER(d)]
    L.tg_linearize.argtypes = [vp, ctypes.c_int] + [vp] * 6
    L.tg_assemble.argtypes = [vp, ctypes.c_int] + [vp] * 10
    L.tg_mpc_step.argtypes = [vp, ctypes.c_int] + [vp] * 11
    L.tg_mpc_step_host.argtypes = [vp, ctypes.c_int] + [vp] * 11
    L.tg_mpc_step_ctrl.argtypes = [vp, ctypes.c_int] + [vp] * 12
    L.tg_mpc_step_ctrl_host.argtypes = [vp, ctypes.c_int] + [vp] * 12
    L.tg_check_ctrl.argtypes = [ctypes.c_int, vp, ctypes.c_uint32]
    L.tg_ref_window.argtypes = [vp, ctypes.c_int, vp, vp, vp, vp, ctypes.c_int, vp, vp]
    L.tg_closed_loop.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp]
    L.tg_closed_loop_host.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, i64, vp, i64, i64, vp, vp, vp, vp, vp]
    L.tg_closed_loop_ctrl.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp]
    L.tg_closed_loop_ctrl_host.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, i64, vp, i64, i64, vp, vp, vp, vp, vp]
    L.tg_check_plant_params.argtypes = [ctypes.c_int, vp]
    L.tg_closed_loop_params.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp]
    L.tg_closed_loop_params_host.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, i64, vp, i64, i64, vp, vp, vp,
                                             vp, vp]
    L.tg_default_scenario_rules.argtypes = [ctypes.POINTER(TgScenarioRules)]
    L.tg_default_scenario_rules.restype = None
    L.tg_make_scenarios.argtypes = [vp, ctypes.c_int, i64, ctypes.POINTER(TgScenarioRules), vp, vp, vp, vp, vp]
    L.tg_make_scenarios_host.argtypes = [vp, ctypes.c_int, i64, ctypes.POINTER(TgScenarioRules), vp, vp, vp, vp, vp]
    L.tg_default_type1_rules.argtypes = [ctypes.POINTER(TgType1Rules)]
    L.tg_default_type1_rules.restype = None
    L.tg_default_type2_rules.argtypes = [ctypes.POINTER(TgType2Rules)]
    L.tg_default_type2_rules.restype = None
    for name, rules in (("tg_openloop_type1", TgType1Rules), ("tg_openloop_type2", TgType2Rules)):
        for suffix in ("", "_host"):
            getattr(L, name + suffix).argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.POINTER(rules), u64, i64, vp, vp, vp, vp]
            getattr(L, name + "_params" + suffix).argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.POINTER(rules), u64, i64, vp,
                                                             vp, vp, vp, vp]
    L.tg_write_csv.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, d, i64, vp, vp, vp, ctypes.c_int, ctypes.c_int]
    L.tg_merge_csv.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, i64, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    L.tg_estimator_step.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, ctypes.POINTER(TgStateLimits), vp]
    L.tg_estimator_step_vjp.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, ctypes.POINTER(TgStateLimits), vp, vp, vp]
    L.tg_estimator_rollout.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp,
                                       ctypes.POINTER(TgStateLimits), vp, ctypes.POINTER(i32)]
    L.tg_plant_rollout.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp]
    L.tg_plant_rollout_params.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
    L.tg_sensor_noise.argtypes = [vp, i64, ctypes.c_int, ctypes.c_int, vp]
    L.tg_philox_u32.argtypes = [vp, u64, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, vp]
    L.tg_fma_peak.argtypes = [vp, ctypes.c_int, ctypes.POINTER(d)]
    L.tg_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
    L.tg_malloc.argtypes = [ctypes.POINTER(vp), i64]
    L.tg_malloc_on.argtypes = [vp, ctypes.POINTER(vp), i64]
    L.tg_free.argtypes = [vp]
    L.tg_memcpy_h2d.argtypes = [vp, vp, vp, i64]
    L.tg_memcpy_d2h.argtypes = [vp, vp, vp, i64]
    L.tg_malloc_host.argtypes = [ctypes.POINTER(vp), i64]
    L.tg_free_host.argtypes = [vp]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise TrajgenError(f"libtrajgen error {rc}: {load().tg_last_error().decode()}")


def default_config():
    cfg = TgConfig()
    load().tg_default_config(ctypes.byref(cfg))
    return cfg


def ptr(a):
    """host pointer of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data


def pinned_empty(shape, dtype=np.float64):
    """A page-locked (cudaMallocHost) NumPy array, freed when the array (and every view of it) is garbage-collected.
    The closed-loop kernel stores its rows straight into such buffers (no device-to-host copy after the kernel)."""
    import weakref
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
    if nbytes == 0:
        return np.empty(shape, dtype)
    p = vp()
    check(load().tg_malloc_host(ctypes.byref(p), nbytes))
    buf = (ctypes.c_char * nbytes).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    weakref.finalize(buf, load().tg_free_host, p.value)     # arr.base keeps buf alive
    return arr


class DeviceBuffer:
    """A cudaMalloc'ed block owned by Python (used by tests / bench to keep data resident in HBM)."""

    def __init__(self, nbytes, handle=None):
        self.nbytes = int(nbytes)
        p = vp()
        if handle is not None:                       # on the owning handle's device, whatever the thread's current device is
            check(load().tg_malloc_on(handle, ctypes.byref(p), self.nbytes))
        else:
            check(load().tg_malloc(ctypes.byref(p), self.nbytes))
        self.ptr = p.value

    def free(self):
        if self.ptr:
            load().tg_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
