"""Generates the committed fixtures under tests/golden/ (run in the BUILD container only: it imports
the reference from /root/reference through oracle/refload.py, which the GPU box does not have).

  python tests/golden/make_golden.py            # reference-pinned fixtures + oracle-made QP fixtures

reference_*.npz / reference_*.csv  = outputs of the reference's OWN code (pinned parity):
    f_cont (three variants), linearize_discretize, vref profiles + reference window, gen1/gen2 plant
    integration with clipping, gen2 dataset rows and CSV text, PCG64 noise facts.
oracle_*.npz = outputs of oracle/ (the QP cannot be run through CVXPY/OSQP here -> PARITY UNPINNED):
    per-step QP optima (interior point, 1e-10) and closed-loop trajectories.
"""
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

from oracle import dynamics as dyn, mpc as ompc, refgen as R, refload  # noqa: E402


def reference_fixtures():
    m = refload.load_mpc()
    g1 = refload.load_gen1()
    g2 = refload.load_gen2()
    rng = np.random.default_rng(20251018)
    n = 64
    X = np.stack([rng.uniform(-2, 2, n), rng.uniform(-2, 2, n), rng.uniform(-np.pi, np.pi, n), rng.uniform(-0.5, 2.5, n),
                  rng.uniform(-0.5, 0.5, n), rng.uniform(-6, 6, n)], axis=1)
    U = np.stack([rng.uniform(-1, 1, n), rng.uniform(-0.6, 0.6, n)], axis=1)
    # SURVEY appendix A points first
    X[0] = [0.3, -0.2, 0.4, 1.2, 0.08, -0.7]; U[0] = [0.35, -0.12]
    X[1] = [0.0, 0.0, -1.0, 0.2, 0.25, 3.0]; U[1] = [0.8, 0.5]
    X[2] = [0.0, 0.5, 0.0, 1.0, 0.0, 0.0]; U[2] = [(0.0518 + 0.00035) / (0.287 - 0.0545), 0.0]
    X[3] = [0.0, 0.0, 0.0, 0.0, 0.1, 0.5]; U[3] = [0.5, 0.1]     # vx = 0: sign(0) = 0 branch
    F = np.zeros((3, n, 6))
    for i in range(n):
        F[0, i] = m.f_cont(X[i], U[i], m.Params)
        F[1, i] = g1.f_cont(X[i], U[i], g1.Params)
        F[2, i] = g2.f_cont(X[i], U[i], g2.Params)
    # linearisation away from the kinks (|vx| = 0.3, |alpha| = 0.6) so analytic and FD Jacobians agree
    nl = 48
    XL = np.stack([rng.uniform(-2, 2, nl), rng.uniform(-2, 2, nl), rng.uniform(-np.pi, np.pi, nl), rng.uniform(0.4, 2.5, nl),
                   rng.uniform(-0.08, 0.08, nl), rng.uniform(-1.5, 1.5, nl)], axis=1)
    UL = np.stack([rng.uniform(-1, 1, nl), rng.uniform(-0.25, 0.25, nl)], axis=1)
    XL[0], UL[0] = X[0], U[0]
    XL[1], UL[1] = X[2], U[2]
    TsL = np.where(np.arange(nl) % 2 == 0, 0.02, 0.01)
    AL = np.zeros((nl, 6, 6)); BL = np.zeros((nl, 6, 2)); GL = np.zeros((nl, 6))
    for i in range(nl):
        AL[i], BL[i], GL[i] = m.linearize_discretize(XL[i], UL[i], float(TsL[i]), m.Params)
    # horizon linearisation exactly as mpc_step does it (:165-178) for 4 start states
    N = 20
    AH = np.zeros((4, N, 6, 6)); BH = np.zeros((4, N, 6, 2)); GH = np.zeros((4, N, 6)); XB = np.zeros((4, N + 1, 6))
    for i in range(4):
        xbar = np.zeros((6, N + 1)); xbar[:, 0] = XL[i]
        for k in range(N):
            xbar[:, k + 1] = xbar[:, k] + 0.02 * m.f_cont(xbar[:, k], UL[i], m.Params)
            AH[i, k], BH[i, k], GH[i, k] = m.linearize_discretize(xbar[:, k], UL[i], 0.02, m.Params)
        XB[i] = xbar.T
    # MPC/main.py function definitions (the module body runs the CVXPY loop, so only the head is executed)
    src = open(os.path.join(refload.REFERENCE_ROOT, "MPC", "main.py")).read().split("# --- MPC SIMULATION SETUP ---")[0]
    refload._stub_matplotlib()
    ns = {}
    old = sys.stdout; sys.stdout = io.StringIO()
    try:
        exec(compile(src, "main_head", "exec"), ns)
    finally:
        sys.stdout = old
    vr40 = ns["vref_profile_ramp_cruise"](40, 0.02, v0=0.8, v_cruise=2.0, tramp=2.0)
    vtr = ns["vref_profile_trapezoid"](40, 0.1, v0=0.8, vmax=2.0, t_acc=1.0, t_flat=1.5, t_dec=1.0)
    vsn = ns["vref_profile_sine"](40, 0.1)
    win = ns["ref_window_from_x_with_vref"](0.37, 40, 0.02, vr40)
    dss = np.array([ns["d_steady_state"](v) for v in (0.5, 1.0, 2.0)])
    # generator plants (clipping) on aggressive controls so that the clips engage
    T = 300
    Usim = np.stack([np.clip(0.3 + 0.7 * np.sin(np.arange(T) * 0.05), -1, 1), 0.5 * np.sin(np.arange(T) * 0.11)], axis=1)
    x0p = np.array([0.0, 0.0, 0.3, 0.45, 0.0, 0.2])
    Xg1 = g1.simulate_trajectory(x0p, Usim, 0.01, g1.Params)
    Xg2 = np.empty((T + 1, 6)); Xg2[0] = x0p
    for k in range(T):     # generation_type2.py:180-187
        Xg2[k + 1] = Xg2[k] + 0.01 * g2.f_cont(Xg2[k], Usim[k], g2.Params)
        Xg2[k + 1, 3] = max(Xg2[k + 1, 3], 0.0)
        Xg2[k + 1, 5] = float(np.clip(Xg2[k + 1, 5], -6, 6))
    Xm = np.empty((T + 1, 6)); Xm[0] = x0p
    for k in range(T):     # MPC/main.py:97
        Xm[k + 1] = Xm[k] + 0.01 * m.f_cont(Xm[k], Usim[k], m.Params)
    np.savez_compressed(os.path.join(HERE, "reference_physics.npz"), X=X, U=U, F=F, XL=XL, UL=UL, TsL=TsL, AL=AL, BL=BL,
                        GL=GL, AH=AH, BH=BH, GH=GH, XB=XB, vr40=vr40, vtr=vtr, vsn=vsn, win=win, dss=dss,
                        Usim=Usim, x0p=x0p, Xg1=Xg1, Xg2=Xg2, Xm=Xm)
    # gen2 dataset: 3 trajectories x 0.5 s, the reference's own DataFrame -> CSV text
    old = sys.stdout; sys.stdout = io.StringIO()
    try:
        df = g2.generate_dataset(num_traj=3, T=0.5, Ts=0.01, seed=42)
    finally:
        sys.stdout = old
    clean = df[df["noise_type"] == "clean"].drop(columns=["noise_type", "mode"])       # generation_type2.py:309-317
    noisy = df[df["noise_type"] == "noisy"].drop(columns=["noise_type", "mode", "phi"])
    clean.to_csv(os.path.join(HERE, "reference_gen2_clean.csv"), index=False)
    noisy.to_csv(os.path.join(HERE, "reference_gen2_noisy.csv"), index=False)
    print("reference fixtures written")


def reference_openloop_fixtures():
    """Outputs of the reference's own open-loop generators (SURVEY.md section 8(f) rank 2) -> reference_openloop.npz.
    type 2: generate_dataset (generation_type2.py:162-220) as is; type 1: the per-trajectory body of its __main__
    loop (generation_type1.py:267-292; the loop is not in a function, so its statements are replayed here on the
    module's own functions and constants, with the legacy global RNG seeded like :17)."""
    g1 = refload.load_gen1()
    g2 = refload.load_gen2()
    out = {}
    # ---- type 2
    cases2 = ((3, 12.0, 0.01, 42), (3, 6.0, 0.02, 7))
    for c, (n, dur, Ts, seed) in enumerate(cases2):
        old = sys.stdout; sys.stdout = io.StringIO()
        try:
            df = g2.generate_dataset(num_traj=n, T=dur, Ts=Ts, seed=seed)
        finally:
            sys.stdout = old
        cl = df[df["noise_type"] == "clean"]
        T1 = len(cl) // n
        names = {"accelerate": 0, "cruise": 1, "turn_left": 2, "turn_right": 3, "": -1}
        out[f"t2_{c}_meta"] = np.array([n, T1 - 1, Ts, seed])
        out[f"t2_{c}_X"] = cl[["X", "Y", "phi", "vx", "vy", "omega"]].to_numpy().reshape(n, T1, 6)
        out[f"t2_{c}_U"] = cl[["d", "delta"]].to_numpy().reshape(n, T1, 2)[:, :-1]
        out[f"t2_{c}_modes"] = np.array([names[m] for m in cl["mode"]], dtype=np.int8).reshape(n, T1)[:, :-1]
    # ---- type 1
    stats = {'d_mean': 0.2161, 'd_std': 0.1314, 'delta_mean': 0.0035, 'delta_std': 0.0338}     # :250
    du_bounds = ((-0.1, 0.1), (-0.04, 0.04))                                                    # :251
    ranges = ((-2.0, 2.0), (-2.0, 2.0), (-np.pi, np.pi), (0.4, 1.5), (-0.05, 0.05), (-1.0, 1.0))  # :260-265
    cases1 = ((6, 1200, 0.01, 42), (4, 400, 0.02, 11))
    for c, (n, T, Ts, seed) in enumerate(cases1):
        np.random.seed(seed)
        X0 = np.zeros((n, 6)); U = np.zeros((n, T, 2)); X = np.zeros((n, T + 1, 6)); modes = np.zeros(n, dtype=np.int8)
        DC = np.zeros((n, T, 2))
        for i in range(n):
            x0 = np.array([np.random.uniform(*r) for r in ranges])
            d_clean, delta_clean, mode = g1.generate_smooth_profiles(T, Ts, stats)
            noise_d = np.random.normal(0, stats['d_std'] * 0.1, T)
            noise_delta = np.random.normal(0, stats['delta_std'] * 0.1, T)
            d_true = np.clip(g1.apply_du_bounds(d_clean + noise_d, *du_bounds[0]), -1.0, 1.0)
            delta_true = np.clip(g1.apply_du_bounds(delta_clean + noise_delta, *du_bounds[1]), -0.6, 0.6)
            Ui = np.stack([d_true, delta_true], axis=1)
            X0[i], U[i], X[i] = x0, Ui, g1.simulate_trajectory(x0, Ui, Ts, g1.Params)
            DC[i] = np.stack([d_clean, delta_clean], axis=1)
            modes[i] = {"straight": 0, "sinusoid": 1}[mode]
        out[f"t1_{c}_meta"] = np.array([n, T, Ts, seed])
        out[f"t1_{c}_x0"], out[f"t1_{c}_U"], out[f"t1_{c}_X"], out[f"t1_{c}_modes"], out[f"t1_{c}_clean_profiles"] = X0, U, X, modes, DC
    out["n_t1"], out["n_t2"] = len(cases1), len(cases2)
    np.savez_compressed(os.path.join(HERE, "reference_openloop.npz"), **out)
    print("reference open-loop fixtures written")


def reference_estimator_fixtures():
    """Outputs + autograd gradients of the reference's own KalmanNet/vehicle_model.py (VehicleModel.f) and of
    rollout_open_loop (KalmanNet/test_prediction.py:68-87, whose module body runs an evaluation, so the function's
    source is compiled on its own) -> reference_estimator.npz, in fp32 and fp64."""
    import inspect, re, torch
    vm = refload._import_from("KalmanNet", "vehicle_model")
    src = open(os.path.join(refload.REFERENCE_ROOT, "KalmanNet", "test_prediction.py")).read()
    m = re.search(r"@torch.no_grad\(\)\ndef rollout_open_loop.*?\n(?=def )", src, flags=re.S)
    ns = {"torch": torch}
    exec(compile(m.group(0), "rollout_open_loop", "exec"), ns)
    rng = np.random.default_rng(5)
    B = 96
    lo = np.array([-3.0, -3.0, -3.2, 0.05, -0.4, -5.0]); hi = np.array([3.0, 3.0, 3.2, 2.2, 0.4, 5.0])
    X = np.stack([rng.uniform(-3.5, 3.5, B), rng.uniform(-3.5, 3.5, B), rng.uniform(-3.5, 3.5, B), rng.uniform(-0.2, 2.6, B),
                  rng.uniform(-0.5, 0.5, B), rng.uniform(-6, 6, B)], axis=1)
    U = np.stack([rng.uniform(-1, 1, B), rng.uniform(-0.6, 0.6, B)], axis=1)
    G = rng.normal(size=(B, 6))
    out = {"lo": lo, "hi": hi, "X": X, "U": U, "G": G, "Ts": np.array(0.01)}
    T, H, t0 = 40, 25, 20
    Useq = np.stack([np.clip(0.25 + 0.1 * rng.normal(size=(8, T)), -1, 1), 0.05 * rng.normal(size=(8, T))], axis=1)   # [8,2,T]
    out["Useq"], out["roll_meta"] = Useq, np.array([T, H, t0])
    for name, dt in (("f32", torch.float32), ("f64", torch.float64)):
        prm = dict(vm.Params)
        for i, k in enumerate(("x", "y", "phi", "vx", "vy", "omega")):
            prm[k + "_min"], prm[k + "_max"] = float(lo[i]), float(hi[i])
        model = vm.VehicleModel(0.01, 10, 10, None, None, None, None)
        model.Params = prm
        x = torch.tensor(X, dtype=dt, requires_grad=True); u = torch.tensor(U, dtype=dt, requires_grad=True)
        y = model.f(x.unsqueeze(2), u.unsqueeze(2)).squeeze(2)
        y.backward(torch.tensor(G, dtype=dt))
        out[f"next_{name}"], out[f"gx_{name}"], out[f"gu_{name}"] = y.detach().numpy(), x.grad.numpy(), u.grad.numpy()
        out[f"h_{name}"] = model.h(x.detach().unsqueeze(2)).squeeze(2).numpy()
        x0 = torch.tensor(X[:8], dtype=dt).unsqueeze(2)
        out[f"roll_{name}"] = ns["rollout_open_loop"](model, x0, torch.tensor(Useq, dtype=dt), t0, H).numpy()     # stops at T
    np.savez_compressed(os.path.join(HERE, "reference_estimator.npz"), **out)
    print("reference estimator fixtures written")


def reference_loader_check():
    """oracle/dataset.py's load_vehicle_dataset (which the tests read the package's CSVs with) against the reference's own
    KalmanNet/data_loader.py on the committed gen2 CSVs: the same tensors in the same order, the same training split."""
    dl = refload.load_data_loader()
    from oracle import dataset as odata
    c, n = os.path.join(HERE, "reference_gen2_clean.csv"), os.path.join(HERE, "reference_gen2_noisy.csv")
    splits = dl.load_vehicle_dataset(n, c, T_steps=50)
    mine = odata.load_vehicle_dataset(n, c, T_steps=50)
    for k in range(3):                                                  # y, u, x
        ref = np.concatenate([s[k].numpy() for s in splits])
        assert ref.dtype == mine[k].dtype and np.array_equal(ref, mine[k], equal_nan=True), k
    assert len(splits[0][0]) == mine[3]
    print("loader restatement agrees with the reference loader")


def oracle_qp_fixtures():
    rng = np.random.default_rng(7)
    cases = []
    hard = dict(du_bounds=((-0.1, 0.1), (-0.04, 0.04)), x_lo=[-1e20] * 4 + [-0.15, -2.0], x_hi=[1e20] * 4 + [0.15, 2.0])
    for N, Ts, is_hard, cnt in ((20, 0.02, False, 6), (20, 0.02, True, 6), (10, 0.02, True, 3), (40, 0.02, False, 2),
                                (50, 0.02, True, 2), (20, 0.01, False, 3)):
        for _ in range(cnt):
            vx = rng.uniform(0.5, 1.5)
            x = np.array([rng.uniform(-1, 1), 0.0, rng.uniform(-0.3, 0.3), vx, rng.uniform(-0.05, 0.05), rng.uniform(-1, 1)])
            prm = (rng.uniform(0.2, 1.0), rng.uniform(0.3, 1.0), rng.uniform(0, 2 * np.pi), 0.0)
            y0, _ = R.path_eval(R.PATH_SINE, prm, x[0:1])
            x[1] = y0[0] + (rng.uniform(-1.5, 1.5) if is_hard else rng.uniform(-0.2, 0.2))
            up = np.array([R.d_steady_state(vx), rng.uniform(-0.1, 0.1)])
            v = R.vref_profile(R.VREF_RAMP, (0.8, rng.uniform(0.8, 2.0), 2.0), N, Ts)
            pr = R.ref_window(x[0], N, Ts, v, R.PATH_SINE, prm)
            kw = hard if is_hard else {}
            u_cmd, status, info = ompc.mpc_step(x, up, pr, Ts=Ts, N=N, vref=v, solver="ipm", **kw)
            if status != "optimal":
                continue
            cases.append(dict(N=N, Ts=Ts, hard=is_hard, x0=x, u_prev=up, path_ref=pr, vref=v, u_cmd=u_cmd,
                              U_opt=info["U_opt"], X_opt=info["X_opt"], objective=info["objective"], y=info["y_ineq"]))
    out = {"n": len(cases)}
    for i, c in enumerate(cases):
        for k, v in c.items():
            out[f"{k}_{i}"] = np.asarray(v)
    np.savez_compressed(os.path.join(HERE, "oracle_qp.npz"), **out)
    print("oracle QP fixtures:", len(cases))


def oracle_closed_loop_fixtures():
    # BASELINE config 1: MPC/main.py verbatim (N=40, Ts=0.02, x0=[0,.5,0,1,0,0], parabola, ramp vref), 600 steps
    x0 = np.array([0.0, 0.5, 0.0, 1.0, 0.0, 0.0]); u0 = np.array([R.d_steady_state(1.0), 0.0])
    X40, U40, st40, _ = ompc.closed_loop(x0, u0, 600, 0.02, 40)
    assert all(s == "optimal" for s in st40)
    X20, U20, st20, _ = ompc.closed_loop(x0, u0, 300, 0.02, 20, path_kind=R.PATH_SINE, path_prm=(0.5, 0.5, 0.0, 0.0))
    assert all(s == "optimal" for s in st20)
    # generator-style: Ts=0.01, gen2 plant with clipping, hard rate bounds
    x1 = np.array([0.0, 0.8, 0.1, 0.6, 0.0, 0.0]); u1 = np.array([R.d_steady_state(0.6), 0.0])
    Xg, Ug, stg, _ = ompc.closed_loop(x1, u1, 200, 0.01, 20, plant=dyn.PLANT_GEN2,
                                      du_bounds=((-0.1, 0.1), (-0.04, 0.04)))
    np.savez_compressed(os.path.join(HERE, "oracle_closed_loop.npz"), x0=x0, u0=u0, X40=X40, U40=U40, X20=X20, U20=U20,
                        x1=x1, u1=u1, Xg=Xg, Ug=Ug, stg=np.array([s == "optimal" for s in stg]))
    d, de = U40[:, 0], U40[:, 1]
    print("config-1 control statistics (cf. generation_type1.py:250: d 0.2161/0.1314, delta 0.0035/0.0338):",
          d.mean(), d.std(), de.mean(), de.std())


if __name__ == "__main__":
    if not refload.available():
        raise SystemExit("the reference tree is not mounted; fixtures can only be regenerated in the build container")
    reference_fixtures()
    reference_openloop_fixtures()
    reference_estimator_fixtures()
    reference_loader_check()
    oracle_qp_fixtures()
    oracle_closed_loop_fixtures()
