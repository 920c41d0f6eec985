"""trajectory_generation_b200 -- B200-native (sm_100a) batched closed-loop MPC trajectory generation.

Drop-in for ONE hot path of DorianaG01/trajectory_generation: ``mpc_step`` (MPC/mpc_6stati.py), the
closed loop around it (MPC/main.py) and the clean/noisy dataset shell of the generators.  Python
marshals arrays; the arithmetic runs in hand-written CUDA kernels behind the C ABI of
``libtrajgen.so`` (include/trajgen.h).  There is no CPU fallback.
"""
from . import _lib
from ._lib import TrajgenError, build, CTRL_SPEC_DTYPE
from .mpc import (BatchedMPC, Params, mpc_step, make_config, check_ctrl_table, check_plant_table, MODEL_MPC, MODEL_GEN1, MODEL_GEN2, PLANT_MPC,
                  PLANT_GEN1, PLANT_GEN2, JAC_ANALYTIC, JAC_FD)
from .generation import (ClosedLoopGenerator, Scenarios, scenario_rules, PATH_ARC, d_steady_state, sample_x0, to_frames, write_csv, merge_datasets,
                         to_loader_tensors, PATH_PARABOLA, PATH_SINE, PATH_SPLINE, VREF_HOLD, VREF_CONST, VREF_RAMP,
                         VREF_TRAPEZOID, VREF_SINE, X0_RANGES_TYPE1, X0_RANGES_TYPE2, CLEAN_COLS, NOISY_COLS)
from .openloop import OpenLoopGenerator, type1_rules, type2_rules, TYPE1_MODES, TYPE2_MODES, CTRL_SEED_BASE


def __getattr__(name):          # torch is imported only when the estimator mirror is asked for
    if name in ("VehicleModel", "rollout_open_loop", "estimator"):
        import importlib
        mod = importlib.import_module(".estimator", __name__)
        return mod if name == "estimator" else getattr(mod, name)
    raise AttributeError(name)


STATUS_STRINGS = _lib.STATUS_STRINGS
__all__ = [n for n in dir() if not n.startswith("_")]
