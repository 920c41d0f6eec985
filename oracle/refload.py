"""Oracle helper: import the reference's own importable Python (build container only).

Test infrastructure -- see ``oracle/__init__.py``.  The reference tree (``REFERENCE_ROOT``)
is not part of this repository, so no test, ``smoke()`` or ``bench.py`` calls this; only
``tests/golden/make_golden.py`` does, to produce the committed fixtures and to check the
oracle's loader restatement against the reference's own loader.

``MPC/mpc_6stati.py:6`` does ``import cvxpy as cp`` and uses ``cp.OSQP`` as a default
argument (``:141``); neither cvxpy nor osqp is installed or installable offline, so a
two-attribute stub module lets the NumPy half (``tire_forces``, ``f_cont``,
``numerical_jacobian``, ``linearize_discretize``, ``lateral_error``) import.  ``mpc_step``
itself then fails at ``cp.Variable`` -- the QP half is what ``oracle/qp.py`` restates.
The generators import ``matplotlib`` (absent); stubs with the two imported names suffice.
"""
import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("TRAJGEN_REFERENCE_ROOT", "/root/reference")


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "MPC", "mpc_6stati.py"))


def _stub(name, **attrs):
    if name in sys.modules:
        return
    try:
        importlib.import_module(name)
        return
    except Exception:
        pass
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    sys.modules[name] = mod


def _import_from(subdir, modname):
    path = os.path.join(REFERENCE_ROOT, subdir)
    if path not in sys.path:
        sys.path.insert(0, path)
    return importlib.import_module(modname)


def real_cvxpy_available():
    try:
        import cvxpy  # noqa: F401
        import osqp  # noqa: F401
        return hasattr(sys.modules["cvxpy"], "Variable")
    except Exception:
        return False


def load_mpc():
    """-> the reference module MPC/mpc_6stati.py (cvxpy stubbed when absent)."""
    _stub("cvxpy", OSQP="OSQP")
    return _import_from("MPC", "mpc_6stati")


def _stub_matplotlib():
    _stub("matplotlib")
    _stub("matplotlib.pyplot")
    _stub("matplotlib.animation", FuncAnimation=object, PillowWriter=object)
    try:
        import tqdm  # noqa: F401
    except Exception:
        _stub("tqdm", tqdm=lambda it, **kw: it)


def load_gen1():
    """-> generation_traj/generation_type1.py (executes np.random.seed(42) at import, :17)."""
    _stub_matplotlib()
    return _import_from("generation_traj", "generation_type1")


def load_gen2():
    _stub_matplotlib()
    return _import_from("generation_traj", "generation_type2")


def load_data_loader():
    """-> KalmanNet/data_loader.py (imports as-is: pandas + torch are installed)."""
    return _import_from("KalmanNet", "data_loader")
