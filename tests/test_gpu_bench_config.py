"""GPU (-m gpu): parity of EXACTLY what bench.py times -- BASELINE config 2 through bench.make_workload
(generation_type1's clipped plant, spline / sinusoid references, time-advancing ramp vref, N = 20, Ts = 0.01,
library-default solver settings: eps 1e-5, shifted warm start, check_every 5) over the full T = 1200 -- against the
oracle closed loop of MPC/main.py:85-101 (tests/golden/oracle_bench_config.npz, made by tests/golden/make_bench_golden.py:
32 trajectory ids, every step solved (a) to the exact optimum by the oracle's interior-point method and (b) by the
oracle's restated OSQP at CVXPY's settings, eps 1e-5, cold start)."""
import os

import numpy as np
import pytest

import bench
import trajectory_generation_b200 as tg
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

# Stated tolerance.  The closed loop is a feedback system: a per-step solver error is fed back through the plant, amplified by
# the stiff yaw dynamics for a step or two (x40 was observed where the duty cycle leaves its bound) and then rejected.  The
# oracle's own two solvers differ by |dX| 3.8e-3 / |dU| 8.0e-3 over these runs (OSQP at CVXPY's eps = 1e-5 stops up to ~1e-2
# from the optimum on single steps, SURVEY.md 7.3).  The CUDA path is held to 1e-4 of the EXACT-optimum loop over all 1200
# steps; measured 7e-7 (X) / 2e-6 (U) with the library defaults (eps 1e-6; unconstrained steps are solved to rounding).
TOL_X_VS_EXACT = 1e-4
TOL_U_VS_EXACT = 1e-4


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN, "oracle_bench_config.npz"))


def test_benchmarked_configuration_matches_oracle_closed_loop(golden):
    par = bench.parity_vs_golden(golden)
    print(par)
    assert par["n_traj"] >= 32 and par["T"] == 1200
    assert par["all_steps_accepted"] and par["workload_matches_oracle_generator"]
    # 2 of the 32 trajectories brake through standstill in the nominal rollout of one early step, where the reference's central
    # differences straddle a jump of f (fd_jump); they are compared up to that step and must have re-converged by the end
    assert len(par["fd_jump_trajectories"]) <= 5 and par["compared_steps"] >= 32400
    assert par["max_abs_err_X_last_100_steps"] <= TOL_X_VS_EXACT, par
    assert par["max_abs_err_X"] <= TOL_X_VS_EXACT, par
    assert par["max_abs_err_U"] <= TOL_U_VS_EXACT, par
    # distance to the restated OSQP at matched eps: not larger than the oracle's own IPM-vs-OSQP distance
    assert par["max_abs_err_X_vs_osqp"] <= par["oracle_ipm_vs_osqp_X"] + TOL_X_VS_EXACT
    assert par["max_abs_err_U_vs_osqp"] <= par["oracle_ipm_vs_osqp_U"] + TOL_U_VS_EXACT


def test_benchmarked_configuration_with_reference_jacobians_matches_every_step(golden):
    """Same runs with the reference's own central-difference Jacobians (TG_JAC_FD = numerical_jacobian verbatim,
    MPC/mpc_6stati.py:73-97): the kernel then reproduces the finite-difference artefact steps as well, so ALL 32 x 1200 steps
    are compared with the oracle loop, nothing excluded."""
    kw = dict(bench.GEN_KW, jacobian=tg.JAC_FD)
    par = bench.parity_vs_golden(golden, gen_kw=kw, exclude_fd_jumps=False)
    print(par)
    assert par["compared_steps"] == 32 * 1200 and par["all_steps_accepted"]
    assert par["max_abs_err_X"] <= TOL_X_VS_EXACT, par
    assert par["max_abs_err_U"] <= TOL_U_VS_EXACT, par


def test_benchmarked_configuration_is_batch_and_shard_invariant(golden):
    """the 32 golden ids inside the full B = 1024 bench batch give the same rows as the 32-trajectory run (bit-exact)."""
    n = int(golden["n_traj"])
    gen = tg.ClosedLoopGenerator(**bench.GEN_KW)
    x0, u0, sc = bench.make_workload(gen, 1024)
    big = gen.generate(x0, u0, sc, 300)
    small = gen.generate(x0[:n], u0[:n], sc.slice(0, n), 300)
    assert np.array_equal(big["clean"][:n], small["clean"]) and np.array_equal(big["U"][:n], small["U"])
    assert np.array_equal(big["noisy"][:n], small["noisy"])


def test_dump_outputs_are_the_timed_launch_results(tmp_path):
    """bench.py --dump-outputs at the benchmarked size: --steps sets the number of launches the library counts in the timed
    window, and the dump is a seeded sample of the B = 1024 trajectories (all of them would exceed 64 MB) in float64,
    bit-identical to the rows the public API returns for the same workload."""
    import json
    import subprocess
    import sys
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(bench.ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu", "--no-extra",
                        "--no-parity", "--dump-outputs", str(out)], capture_output=True, text=True, check=True)
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["timed_launches"] == 2 and line["warmup"] == 3
    d = {f.stem: np.load(f) for f in out.glob("*.npy")}
    assert set(d) == {"traj_ids", "clean", "noisy", "U", "status_counts", "iters_total"}
    assert all(a.dtype == np.float64 for a in d.values())
    assert sum(f.stat().st_size for f in out.glob("*.npy")) <= bench.DUMP_BYTES
    ids = d["traj_ids"].astype(np.int64)
    assert 32 <= len(ids) < 1024 and (np.diff(ids) > 0).all() and ids[-1] < 1024
    gen = tg.ClosedLoopGenerator(**bench.GEN_KW)
    x0, u0, sc = bench.make_workload(gen, 1024)
    ref = gen.generate(x0, u0, sc, 1200)
    for k in ("clean", "noisy", "U", "status_counts", "iters_total"):
        assert np.array_equal(d[k], ref[k][ids].astype(np.float64)), k
