"""CPU: per-trajectory plant parameters -- the rules of a plant table (tg_check_plant_params / check_plant_table), the
column overrides of plant_table, and the reference loop with a plant that differs from the controller's model
(tests/plant_mismatch_loop.py) against the oracle's closed loop."""
import types

import numpy as np
import pytest

import trajectory_generation_b200 as tg
from trajectory_generation_b200 import _lib
from oracle import dynamics as dyn, mpc as ompc, refgen as R
import plant_mismatch_loop as pml

ORDER = _lib.PARAM_ORDER


def _default_rows(B):
    return np.tile(np.array([tg.Params[k] for k in ORDER]), (B, 1))


def _stub(**params):
    """a stand-in for a generator: plant_table reads nothing but cfg.params"""
    return types.SimpleNamespace(cfg=tg.make_config(params=params or None))


def test_default_rows_are_accepted():
    t = _default_rows(3)
    assert tg.check_plant_table(t) is t
    assert _lib.load().tg_check_plant_params(0, None) == 0


@pytest.mark.parametrize("name,value,why", [
    ("Cm1", np.nan, "must be finite"), ("Df", np.inf, "must be finite"), ("g", -np.inf, "must be finite"),
    ("m", 0.0, "must be > 0"), ("m", -0.041, "must be > 0"), ("Iz", 0.0, "must be > 0"), ("Iz", -1e-6, "must be > 0"),
    ("vx_zero", 0.0, "must be > 0"), ("vx_zero", -0.3, "must be > 0"), ("maxAlpha", 0.0, "must be > 0"),
    ("maxAlpha", -0.6, "must be > 0"), ("m", np.nan, "must be finite")])
def test_bad_entry_names_row_and_field(name, value, why):
    t = _default_rows(5)
    t[3, ORDER.index(name)] = value
    with pytest.raises(ValueError, match=rf"^plant row 3: {name} {why}$"):
        tg.check_plant_table(t)
    t[1, ORDER.index(name)] = value          # the first bad row is named
    with pytest.raises(ValueError, match=rf"^plant row 1: {name} "):
        tg.check_plant_table(t)


def test_negative_values_elsewhere_are_not_refused():
    """only m, Iz, vx_zero and maxAlpha carry a sign rule: a negative drag or tyre constant is finite, so it passes"""
    t = _default_rows(2)
    t[0, ORDER.index("Cr0")] = -0.01
    t[1, ORDER.index("Bf")] = -2.0
    tg.check_plant_table(t)


@pytest.mark.parametrize("bad", [
    np.zeros((4, 16)), np.zeros(17), np.zeros((2, 17), np.float32), np.zeros((2, 17), np.int64),
    np.asfortranarray(_default_rows(3)), np.zeros((2, 3, 17))])
def test_wrong_shape_or_dtype_is_refused(bad):
    with pytest.raises(ValueError, match="plant table"):
        tg.check_plant_table(bad)


def test_plant_table_overrides_columns():
    stub = _stub(m=0.05)
    B = 4
    base = np.array(stub.cfg.params[:])
    t = tg.ClosedLoopGenerator.plant_table(stub, B)
    assert t.shape == (B, 17) and t.dtype == np.float64 and t.flags["C_CONTIGUOUS"]
    np.testing.assert_array_equal(t, np.tile(base, (B, 1)))
    assert t[0, ORDER.index("m")] == 0.05                      # starts from the handle's params, not the reference defaults
    m = np.array([0.03, 0.04, 0.05, 0.06])
    t = tg.OpenLoopGenerator.plant_table(stub, B, m=m, Df=0.2, Iz=np.full(B, 3e-5))
    np.testing.assert_array_equal(t[:, ORDER.index("m")], m)
    assert (t[:, ORDER.index("Df")] == 0.2).all() and (t[:, ORDER.index("Iz")] == 3e-5).all()
    keep = [i for i, k in enumerate(ORDER) if k not in ("m", "Df", "Iz")]
    np.testing.assert_array_equal(t[:, keep], np.tile(base[keep], (B, 1)))


def test_plant_table_refuses_unknown_names_bad_lengths_and_bad_values():
    stub = _stub()
    with pytest.raises(TypeError, match="mass"):
        tg.ClosedLoopGenerator.plant_table(stub, 3, mass=0.05)
    with pytest.raises(ValueError, match="expected a scalar or 3 values"):
        tg.ClosedLoopGenerator.plant_table(stub, 3, m=[0.04, 0.05])
    with pytest.raises(ValueError, match="^plant row 2: Iz must be > 0$"):
        tg.ClosedLoopGenerator.plant_table(stub, 3, Iz=[1e-5, 2e-5, 0.0])


# ------------------------------------------------------------------------------------------------ reference loop
LOOP = dict(T=12, Ts=0.02, N=10, path_kind=R.PATH_SINE, path_prm=(0.5, 0.5, 0.0, 0.0))
X0 = np.array([0.0, 0.3, 0.05, 1.0, 0.0, 0.0])
U0 = np.array([0.1, 0.0])


@pytest.mark.parametrize("plant", [dyn.PLANT_MPC, dyn.PLANT_GEN2])
def test_reference_loop_with_the_models_vehicle_is_the_oracle_loop(plant):
    X0_, U0_, st0, _ = ompc.closed_loop(X0, U0, plant=plant, **LOOP)
    for pp in (None, dict(dyn.PARAMS), [dyn.PARAMS[k] for k in ORDER]):
        X1, U1, st1, _ = pml.closed_loop(X0, U0, plant=plant, plant_params=pp, **LOOP)
        np.testing.assert_array_equal(X1, X0_)
        np.testing.assert_array_equal(U1, U0_)
        assert st1 == st0


def test_reference_loop_with_another_vehicle_changes_only_the_plant():
    X0_, U0_, _, _ = ompc.closed_loop(X0, U0, **LOOP)
    row = [dyn.PARAMS[k] for k in ORDER]
    row[ORDER.index("m")] *= 1.15
    row[ORDER.index("Df")] *= 0.9
    X1, U1, st1, _ = pml.closed_loop(X0, U0, plant_params=row, **LOOP)
    np.testing.assert_array_equal(U1[0], U0_[0])          # the first decision sees x0 only: the controller's model is unchanged
    assert np.abs(X1[1] - X0_[1]).max() > 0               # the plant integrates another vehicle
    np.testing.assert_array_equal(X1[1], dyn.plant_step(X0, U0_[0], LOOP["Ts"], p=dict(zip(ORDER, row))))
    assert all(s in ompc.ACCEPTED for s in st1)
