"""CPU oracle for the closed-loop MPC hot path of DorianaG01/trajectory_generation.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product: only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it, and only as the checker (or as the timed CPU
baseline), never as the thing shipped.  The product path is
``trajectory_generation_b200`` -> ``libtrajgen.so`` (CUDA, sm_100a) and fails loudly
when that library is missing.

Parity status ("pinned" means checked against genuine reference outputs):

* physics / linearisation / plant / noise-shell / CSV rows  -- PINNED.  The reference's
  own NumPy code (``MPC/mpc_6stati.py``, ``generation_traj/generation_type{1,2}.py``) is
  importable in the build container with stub ``cvxpy`` / ``matplotlib`` modules
  (``oracle/refload.py``); ``tests/golden/make_golden.py`` ran it and committed the
  outputs under ``tests/golden/``; ``tests/test_oracle_vs_golden.py`` checks every
  restated function against them.
* the consumer's loader (``KalmanNet/data_loader.py``, restated in ``oracle/dataset.py``)  --
  restated from the cited lines; ``tests/golden/make_golden.py`` checks the restatement
  against the reference's own loader whenever it regenerates the fixtures.
* the QP (``MPC/mpc_6stati.py:180-262``: CVXPY problem -> OSQP)  -- PARITY UNPINNED.
  ``cvxpy`` and ``osqp`` are un-pinned third-party dependencies
  (``README.md:70``, ``MPC/README.md:84``: "pip install cvxpy osqp", no version) that are
  not installed here and cannot be installed offline, and the reference ships no test,
  fixture or stored solver output.  ``oracle/qp.py`` restates the *problem* exactly as
  the reference states it (sparse form, same rows, same cost) and solves it two ways
  (a primal-dual interior-point method to ~1e-10 = "the exact optimum", and a
  restatement of the published OSQP algorithm at CVXPY's settings); the two must agree,
  which pins the restatement to the mathematics but not to a binary of OSQP.

Every function cites the reference ``file:line`` it follows (paths relative to the
reference root).
"""
