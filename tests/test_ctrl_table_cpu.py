"""CPU: the NumPy mirror of tg_ctrl_spec has the header's layout, and the library's checks of a ctrl table (tg_check_ctrl,
which check_ctrl_table and the *_host entry points call; it needs no GPU) follow the rules the header states
(tests/test_gpu_ctrl_table.py checks the entry points on the GPU)."""
import os
import re

import numpy as np
import pytest

import trajectory_generation_b200 as tg
from trajectory_generation_b200 import _lib
from conftest import ROOT

INF = _lib.TG_INF


def _header_struct(name):
    """(field, count) of a struct of doubles in include/trajgen.h, in declaration order"""
    src = open(os.path.join(ROOT, "include", "trajgen.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, flags=re.S).group(1)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        assert decl.startswith("double "), decl
        for item in decl[len("double "):].split(","):
            m = re.fullmatch(r"\s*(\w+)\s*(?:\[(\d+)\])?\s*", item)
            fields.append((m.group(1), int(m.group(2) or 1)))
    return fields


def test_ctrl_spec_dtype_has_the_header_layout():
    fields = _header_struct("tg_ctrl_spec")
    dt = _lib.CTRL_SPEC_DTYPE
    assert [f for f, _ in fields] == list(dt.names)
    off = 0
    for f, k in fields:
        sub, o = dt.fields[f][:2]
        assert o == off, f
        assert sub.base == np.float64 and int(np.prod(sub.shape)) == k, f
        off += 8 * k
    assert dt.itemsize == off == 248


def _table(B):
    """B rows of mpc_step's defaults (include/trajgen.h: tg_default_config)"""
    t = np.zeros(B, _lib.CTRL_SPEC_DTYPE)
    t["q_c"], t["q_phi"], t["q_vx"] = 6.0, 0.5, 0.5
    t["R"] = (0.02, 0.0, 0.0, 2.0); t["Rd"] = (0.01, 0.0, 0.0, 5.0)
    t["u_lo"] = (-1.0, -0.6); t["u_hi"] = (1.0, 0.6); t["du_lo"] = (-0.5, -0.3); t["du_hi"] = (0.5, 0.3)
    t["x_lo"] = -INF; t["x_hi"] = INF
    return t


BOUNDED = (False, False, False, False, True, True)   # a handle with a vy / omega box


def test_valid_tables_pass():
    t = _table(5)
    t["x_lo"][:, 4:] = (-0.15, -2.0); t["x_hi"][:, 4:] = (0.15, 2.0)
    t["x_lo"][1, 4:] = -INF; t["x_hi"][1, 4:] = INF             # a row may drop the box of a bounded component
    t["Rd"][2] = 0.0                                            # Rd only needs to be semidefinite
    t["q_c"][3] = 0.0
    t["R"][4] = (0.05, 0.04, -0.02, 1.0)                         # only the symmetric part has to be definite
    t["u_lo"][0] = t["u_hi"][0]                                  # lo == hi is allowed
    assert tg.check_ctrl_table(t, BOUNDED) is t


@pytest.mark.parametrize("field,value,message", [
    ("q_c", np.nan, "q_c must be finite"), ("q_phi", -0.1, "q_phi must be finite and >= 0"), ("q_vx", np.inf, "q_vx"),
    ("R", (np.inf, 0, 0, 1), "R[0] must be finite"), ("Rd", (1, np.nan, 0, 1), "Rd[1] must be finite"),
    ("R", (1.0, 0.0, 0.0, 0.0), "R symmetric part is not positive definite"),
    ("R", (1.0, 3.0, -1.0, 1.0), "R symmetric part is not positive definite"),
    ("Rd", (0.0, 0.0, 0.0, -1.0), "Rd symmetric part is not positive semidefinite"),
    ("Rd", (1.0, 2.0, 2.0, 1.0), "Rd symmetric part is not positive semidefinite"),
    ("u_hi", (-2.0, 0.6), "u_lo[0] / u_hi[0] lo > hi"), ("du_lo", (-0.5, 0.4), "du_lo[1] / du_hi[1] lo > hi"),
    ("x_hi", (INF,) * 5 + (-np.inf,), "x_lo[5] / x_hi[5] lo > hi"),
    ("x_lo", (-INF,) * 3 + (0.0, -INF, -INF), "x_lo[3] / x_hi[3] finite bound on a state component the handle does not bound"),
])
def test_each_rule_names_the_first_bad_row_and_field(field, value, message):
    t = _table(6)
    t[field][4] = value
    t["q_c"][5] = -1.0                                          # a later bad row is not the one reported
    with pytest.raises(ValueError, match=re.escape(f"ctrl row 4: {message}")):
        tg.check_ctrl_table(t, BOUNDED)
