"""Reference for the tests of per-trajectory plant parameters: the closed loop of MPC/main.py:85-101 as oracle/mpc.py's
``closed_loop`` states it, with the plant step (:97) integrating a vehicle of its own while the controller keeps
``mpc_kwargs["params"]``.  tests/test_plant_params_cpu.py pins it to ``oracle.mpc.closed_loop`` where the two vehicles agree."""
import numpy as np

from oracle import dynamics as dyn, mpc as ompc, refgen


def plant_vehicle(plant_params):
    """dyn.PARAMS updated by ``plant_params``: a dict of overrides, or 17 values in the order Cm1 Cm2 Cr0 Cr2 Br Cr Dr Bf Cf Df
    m Iz lf lr g maxAlpha vx_zero (tg_config.params); None = dyn.PARAMS"""
    p = dict(dyn.PARAMS)
    if isinstance(plant_params, dict):
        p.update(plant_params)
    elif plant_params is not None:
        p.update(zip(dyn.PARAMS.keys(), np.asarray(plant_params, float).reshape(17).tolist()))
    return p


def closed_loop(x0, u_prev, T, Ts, N, path_kind=refgen.PATH_PARABOLA, path_prm=(0.1, 0.0, 0.0, 0.0), spline=None,
                vref_kind=refgen.VREF_RAMP, vref_prm=(0.8, 2.0, 2.0), vref_advance=False, plant=dyn.PLANT_MPC, solver="ipm",
                solver_opts=None, plant_params=None, **mpc_kwargs):
    """oracle.mpc.closed_loop (graph paths) with the plant step integrating plant_vehicle(plant_params).
    Returns X[T+1,6] (row 0 = x0), U[T,2], statuses[T], iters[T]."""
    pp = plant_vehicle(plant_params)
    x = np.asarray(x0, float).copy()
    u_prev = np.asarray(u_prev, float).copy()
    Xh = np.zeros((T + 1, 6)); Uh = np.zeros((T, 2)); st = []; its = np.zeros(T, int)
    Xh[0] = x
    for t in range(T):
        t0 = t * Ts if vref_advance else 0.0
        vref_seq = refgen.vref_profile(vref_kind, vref_prm, N, Ts, t0, x[3])
        path_ref = refgen.ref_window(x[0], N, Ts, vref_seq, path_kind, path_prm, spline)
        u_cmd, status, info = ompc.mpc_step(x, u_prev, path_ref, Ts=Ts, N=N, vref=vref_seq, solver=solver,
                                            solver_opts=solver_opts, **mpc_kwargs)
        x = dyn.plant_step(x, u_cmd, Ts, p=pp, plant=plant)
        Xh[t + 1] = x; Uh[t] = u_cmd; st.append(status); its[t] = info.get("iters", 0) if info else 0
        u_prev = u_cmd
    return Xh, Uh, st, its
