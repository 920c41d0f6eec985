"""CPU: host-side logic of the package -- scenario tables, dataset schema / CSV text, loader hand-off,
sharding.  No compute calls."""
import os

import numpy as np
import pandas as pd
import pytest

import trajectory_generation_b200 as tg
from trajectory_generation_b200 import distributed as tgd
from conftest import GOLDEN


def _reference_rows():
    c = pd.read_csv(os.path.join(GOLDEN, "reference_gen2_clean.csv"), float_precision="round_trip")
    n = pd.read_csv(os.path.join(GOLDEN, "reference_gen2_noisy.csv"), float_precision="round_trip")
    B = c["trajectory_id"].nunique()
    T1 = len(c) // B
    clean = c[["X", "Y", "phi", "vx", "vy", "omega"]].values.reshape(B, T1, 6)
    noisy = np.zeros_like(clean)
    noisy[:, :, [0, 1, 3, 4, 5]] = n[["X", "Y", "vx", "vy", "omega"]].values.reshape(B, T1, 5)
    U = c[["d", "delta"]].values.reshape(B, T1, 2)[:, :-1]
    return {"clean": clean, "noisy": noisy, "U": U}


def test_csv_writer_is_byte_identical_to_the_reference(tmp_path):
    """feeding the reference's own rows through the package's writer reproduces the reference's files."""
    res = _reference_rows()
    for engine in ("native", "pandas"):
        tg.write_csv(res, 0.01, tmp_path / "c.csv", tmp_path / "n.csv", engine=engine)
        assert open(tmp_path / "c.csv").read() == open(os.path.join(GOLDEN, "reference_gen2_clean.csv")).read()
        assert open(tmp_path / "n.csv").read() == open(os.path.join(GOLDEN, "reference_gen2_noisy.csv")).read()
    # appending shard by shard gives the same bytes as one call
    first = {k: v[:2] for k, v in res.items()}
    rest = {k: v[2:] for k, v in res.items()}
    tg.write_csv(first, 0.01, tmp_path / "c2.csv", tmp_path / "n2.csv")
    tg.write_csv(rest, 0.01, tmp_path / "c2.csv", tmp_path / "n2.csv", traj_id0=2, append=True)
    assert open(tmp_path / "c2.csv").read() == open(os.path.join(GOLDEN, "reference_gen2_clean.csv")).read()


def test_native_float_formatting_equals_python_repr(tmp_path):
    """the native writer's float text is Python's repr for awkward values (exponent thresholds, subnormals, -0.0)."""
    vals = np.array([0.0, -0.0, 1.0, -1.5, 0.1, 1e-4, 1e-5, 1.5e-7, 123456789.125, 1e15, 1e16, 1.2345678901234567e17, 5e-324,
                     1.7976931348623157e308, 0.30000000000000004, 2.0 ** -20, 1 / 3, 12345678901234567.0, np.inf, -np.inf])
    rng = np.random.default_rng(0)
    vals = np.concatenate([vals, rng.normal(size=200) * 10.0 ** rng.integers(-12, 12, 200)])
    B = len(vals)
    clean = np.zeros((B, 1, 6)); clean[:, 0, 0] = vals
    res = {"clean": clean, "noisy": clean.copy(), "U": np.zeros((B, 0, 2))}
    tg.write_csv(res, 0.5, tmp_path / "c.csv", tmp_path / "n.csv")
    lines = open(tmp_path / "c.csv").read().splitlines()[1:]
    for v, ln in zip(vals, lines):
        assert ln.split(",")[1] == repr(float(v)), (v, ln)
    c, n = tg.to_frames(res, 0.01)
    assert list(c.columns) == tg.CLEAN_COLS and list(n.columns) == tg.NOISY_COLS
    last = c[c["trajectory_id"] == 2].iloc[-1]
    assert np.isnan(last["d"]) and np.isnan(last["delta"])          # generation_type2.py:211-212


def test_loader_tensors_match_reference_loader(tmp_path):
    """the reference's rows written by the package's writer, read back by the loader (oracle/dataset.py's restatement of
    KalmanNet/data_loader.py), give the tensors to_loader_tensors hands over without the CSV round trip."""
    from oracle import dataset as odata
    res = _reference_rows()
    tg.write_csv(res, 0.01, tmp_path / "c.csv", tmp_path / "n.csv")
    y, u, x = tg.to_loader_tensors(res, 50)
    assert y.shape == (3, 5, 50) and u.shape == (3, 2, 50) and x.shape == (3, 6, 50) and y.dtype == np.float32
    ally, allu, allx, n_train = odata.load_vehicle_dataset(str(tmp_path / "n.csv"), str(tmp_path / "c.csv"), T_steps=50)
    perm = np.arange(3); np.random.default_rng(42).shuffle(perm)      # KalmanNet/data_loader.py:60-62
    np.testing.assert_array_equal(allx, x[perm])
    np.testing.assert_array_equal(ally, y[perm])
    np.testing.assert_array_equal(allu, u[perm])
    assert n_train == 2 and not np.isnan(allx).any()


@pytest.mark.parametrize("args", [["--impl", "reference"], ["--steps", "0"]])
def test_bench_refuses_dump_outputs_without_a_timed_gpu_step(tmp_path, args):
    """--dump-outputs writes the timed GPU launch's results: with the CPU arm or no timed step there is nothing to write."""
    import subprocess
    import sys
    from conftest import ROOT
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "d")] + args,
                       capture_output=True, text=True)
    assert p.returncode == 2 and "--dump-outputs needs" in p.stderr and not (tmp_path / "d").exists()


def test_sample_x0_is_the_reference_draw():
    x0 = tg.sample_x0(3, 42)
    np.testing.assert_allclose(x0[0], [1.0958241942238534, -0.24448624099179073, 2.2531371815723604,
                                       0.47894721162374554, -0.04058226521123505, 0.9512447032735118], rtol=0, atol=0)


def test_scenarios_table():
    sc = tg.Scenarios(5)
    assert (sc.spec["path_kind"] == tg.PATH_PARABOLA).all() and sc.spec["path"][0, 0] == 0.1
    sc.set_sine(slice(1, 3), A=np.array([0.3, 0.4]), k=0.5, psi=0.1)
    sc.set_spline(3, [0, 1, 2, 3], [0, 0.5, -0.2, 0.1])
    sc.set_spline(4, [0, 2, 4], [0, 1.0, 0.0])
    sc.set_vref(slice(0, 5), tg.VREF_CONST, 1.2)
    brk, coef = sc.tables()
    assert list(sc.spec["path"][2]) == [0.4, 0.5, 0.1, 0.0]
    assert len(brk) == 5 and coef.shape == (5, 4) and sc.spec["spline_first"][4] == 3 and sc.spec["spline_count"][4] == 2
    sub = sc.slice(3, 5)
    assert len(sub) == 2 and sub.spec["spline_first"][1] == 3 and np.array_equal(sub.tables()[0], brk)
    assert tg.d_steady_state(1.0) == pytest.approx(0.2243010752688172)


def test_shard_ranges_partition_the_ids():
    for B, W in ((10, 1), (10, 3), (1048576, 8), (5, 8), (0, 2)):
        r = [tgd.shard_range(B, k, W) for k in range(W)]
        assert r[0][0] == 0 and r[-1][1] == B
        assert all(r[k][1] == r[k + 1][0] for k in range(W - 1))
        assert max(h - l for l, h in r) - min(h - l for l, h in r) <= 1


def test_batched_natural_splines_equal_scipy():
    from scipy.interpolate import CubicSpline
    rng = np.random.default_rng(5)
    M, K = 7, 12
    X = np.cumsum(rng.uniform(1.0, 3.0, (M, K)), axis=1) - 6.0
    Y = rng.normal(0, 0.3, (M, K))
    sc = tg.Scenarios(10)
    sc.set_spline(0, X[0], Y[0])                        # a single one first: the batch appends after it
    coef = sc.set_splines(np.arange(2, 2 + M), X, Y)
    brk, cf = sc.tables()
    for i in range(M):
        cs = CubicSpline(X[i], Y[i], bc_type="natural")
        np.testing.assert_allclose(coef[i], cs.c.T, rtol=1e-10, atol=1e-12)
        f, n_ = sc.spec["spline_first"][2 + i], sc.spec["spline_count"][2 + i]
        assert n_ == K - 1 and np.array_equal(brk[f:f + n_], X[i, :-1]) and np.array_equal(cf[f:f + n_], coef[i])
    assert sc.spec["spline_first"][0] == 0 and sc.spec["spline_first"][2] == K - 1


def test_merge_datasets_matches_the_reference_script(tmp_path):
    """tg_merge_csv (host-only entry point) vs generation_traj/merge_datasets.py:33-70 restated with pandas.  With a
    correctly rounded parser (float_precision='round_trip') pandas' re-serialisation is the identity on the numbers,
    so the merged files must agree byte for byte; with pandas' default fast parser the reference's merge perturbs last
    digits, which the verbatim merge never does."""
    import pandas as pd
    rng = np.random.default_rng(0)

    def run(B, T):
        return {"clean": rng.normal(size=(B, T + 1, 6)), "noisy": rng.normal(size=(B, T + 1, 6)), "U": rng.normal(size=(B, T, 2))}
    p = lambda n: str(tmp_path / n)          # noqa: E731
    tg.write_csv(run(3, 5), 0.01, p("pc.csv"), p("pn.csv"))
    tg.write_csv(run(4, 7), 0.01, p("mc.csv"), p("mn.csv"))
    info = tg.merge_datasets(p("pc.csv"), p("mc.csv"), p("oc.csv"), p("pn.csv"), p("mn.csv"), p("on.csv"))
    assert info == {"id_offset": 3, "rows_clean": 3 * 6 + 4 * 8, "rows_noisy": 3 * 6 + 4 * 8}
    off = None
    for a, b, o in (("pc.csv", "mc.csv", "rc.csv"), ("pn.csv", "mn.csv", "rn.csv")):
        d1 = pd.read_csv(p(a), float_precision="round_trip")
        d2 = pd.read_csv(p(b), float_precision="round_trip")
        if off is None:
            off = d1["trajectory_id"].max() + 1                       # merge_datasets.py:42-45, re-used for the noisy pair
        d2["trajectory_id"] = d2["trajectory_id"] + off
        pd.concat([d1, d2], ignore_index=True, sort=False).to_csv(p(o), index=False)
    assert open(p("oc.csv"), "rb").read() == open(p("rc.csv"), "rb").read()
    assert open(p("on.csv"), "rb").read() == open(p("rn.csv"), "rb").read()
    merged = pd.read_csv(p("oc.csv"))
    assert sorted(merged["trajectory_id"].unique()) == list(range(7))
    with pytest.raises(tg.TrajgenError, match="File not found"):
        tg.merge_datasets(p("missing.csv"), p("mc.csv"), p("x.csv"))
    with pytest.raises(tg.TrajgenError, match="different columns"):
        tg.merge_datasets(p("pc.csv"), p("mn.csv"), p("x.csv"))
    # a second file without a trailing newline and with CRLF line ends
    open(p("crlf.csv"), "wb").write(b"t,X,trajectory_id\r\n0.0,1.5,0\r\n0.01,2.5,1")
    open(p("lf.csv"), "wb").write(b"t,X,trajectory_id\n0.0,9.5,4\n")
    tg.merge_datasets(p("lf.csv"), p("crlf.csv"), p("m.csv"))
    assert open(p("m.csv")).read() == "t,X,trajectory_id\n0.0,9.5,4\n0.0,1.5,5\n0.01,2.5,6\n"


def test_scenario_oracle_spline_is_scipys_natural_spline_and_ranges_hold():
    """oracle/scenarios.py (what tg_make_scenarios must reproduce): the Thomas-algorithm spline equals scipy's
    CubicSpline(bc_type="natural") -- the routine generation_type1.py:97 calls --, every draw lies in its range, and a
    trajectory does not depend on the batch it is generated in (ids are the only key)."""
    from scipy.interpolate import CubicSpline
    from oracle import scenarios as oscn, refgen as R
    o = oscn.make_scenarios(12)
    ru = oscn.DEFAULT_RULES
    for b in range(12):
        x0 = o["x0"][b]
        assert ru["x0_lo"][0] <= x0[0] <= ru["x0_hi"][0] and ru["x0_lo"][3] <= x0[3] <= ru["x0_hi"][3]
        assert ru["x0_lo"][4] <= x0[4] <= ru["x0_hi"][4] and ru["x0_lo"][5] <= x0[5] <= ru["x0_hi"][5]
        assert ru["vcruise"][0] <= o["vref"][b, 1] <= ru["vcruise"][1] and o["path_kind"][b] == ru["cycle"][b % 2]
        if o["path_kind"][b] == R.PATH_SPLINE:
            kx = o["breaks"][b]; ky = o["coef"][b, :, 3]
            assert (np.diff(kx) >= 1.0).all() and (np.diff(kx) <= 3.0).all() and kx[0] == -6.0
            # rebuild the last knot from the last piece, then compare with scipy on the interior pieces
            h = kx[-1] - kx[-2]
            cs = CubicSpline(kx, ky, bc_type="natural")          # natural spline through the first K-1 knots differs from
            assert cs.c.shape[1] == len(kx) - 1                  # ours only through the (dropped) last knot: compare the fit
            full = oscn.natural_spline(np.append(kx, kx[-1] + h), np.append(ky, ky[-1]))
            ref = CubicSpline(np.append(kx, kx[-1] + h), np.append(ky, ky[-1]), bc_type="natural")
            np.testing.assert_allclose(full, ref.c.T, atol=1e-12)
            # the lateral / heading offsets are applied at X
            piece = int(np.clip((kx <= x0[0]).sum() - 1, 0, len(kx) - 1)); dx = x0[0] - kx[piece]
            c0, c1, c2, c3 = o["coef"][b, piece]
            assert abs(x0[1] - (((c0 * dx + c1) * dx + c2) * dx + c3)) <= 0.2 + 1e-12
    shifted = oscn.make_scenarios(4, traj_id0=5)
    for k in ("x0", "u0", "path", "vref", "breaks", "coef"):
        assert np.array_equal(shifted[k], o[k][5:9]), k
