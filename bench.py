#!/usr/bin/env python
"""bench.py -- closed-loop MPC steps/s on B200 (BASELINE.json metric), roofline and CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--horizon-steps T] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: BASELINE config 2 -- B = 1024 trajectories per GPU,
spline / sinusoidal references, N = 20, Ts = 0.01, T = 1200 closed-loop MPC steps each (1.23 M MPC steps),
run by ONE launch of the fused closed-loop kernel.  `value` is timed with CUDA events on the kernel's
stream with inputs resident in HBM; `e2e` goes through the public Python API with host arrays
(ClosedLoopGenerator.generate: inputs copied host -> device inside the call, result rows stored into page-locked
host arrays while the kernel runs).  For N > 1 the driver launches this file under torchrun: each rank
owns its own block of trajectory ids (weak scaling, no collective on the solve path), time = max over
ranks.  `--impl reference` times the reference's algorithm on the host cores (oracle/ port of
MPC/main.py's loop with the restated OSQP; cvxpy/osqp are not installable offline).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_HORIZON, TS = 20, 0.01
METRIC = "closed-loop MPC steps/sec (batched QP solves/sec)"
DUMP_BYTES = 64 * 10 ** 6       # --dump-outputs writes at most this much in all


def make_workload(gen, B, traj_id0=0):
    """BASELINE config 2 (SURVEY.md section 8(d)) for trajectory ids traj_id0 .. traj_id0 + B - 1, generated ON THE DEVICE
    (tg_make_scenarios; oracle/scenarios.py restates it): even ids a natural cubic spline y(x) through 27 knots every
    U(1,3) m from x = -6 m with N(0, 0.3^2) m ordinates, odd ids y = A sin(kx + psi) with A~U(0.2,1), k~U(0.3,1),
    psi~U(0,2pi); vref ramp-cruise 0.8 -> U(0.8,2.0) m/s over 2 s, advancing in time; x0 from generation_type1.py:260-265's
    ranges with heading / lateral offset (+-0.2) relative to the path; u0 = steady-state duty cycle.  Every number is a
    function of 2025 + trajectory id.  -> (x0[B,6], u0[B,2], Scenarios)"""
    return gen.make_scenarios(B, traj_id0=traj_id0)


def workload_from_golden(golden):
    """the first n_traj ids of the same workload as the oracle generated them (stored with the golden closed loops)"""
    import trajectory_generation_b200 as tg
    sc = tg.Scenarios.from_arrays(golden["path_kind"], golden["path"], golden["vref"], golden["breaks"], golden["coef"])
    return np.ascontiguousarray(golden["x0"]), np.ascontiguousarray(golden["u0"]), sc


GEN_KW = dict(N=N_HORIZON, Ts=TS, plant=1, vref_advance=True)   # plant 1 = generation_type1's clipped plant


def parity_vs_golden(golden=None, gen_kw=None, device=0, exclude_fd_jumps=True):
    """Parity of the benchmarked configuration, measured OUTSIDE the timed region: the first n_traj ids of make_workload
    run through the public generator API for the golden file's full T and compared with the oracle closed loops stored
    in tests/golden/oracle_bench_config.npz (exact per-step optimum, and the restated OSQP at eps 1e-5)."""
    import trajectory_generation_b200 as tg
    if golden is None:
        golden = np.load(os.path.join(ROOT, "tests", "golden", "oracle_bench_config.npz"))
    n, T = int(golden["n_traj"]), int(golden["T"])
    x0, u0, sc = workload_from_golden(golden)
    gen = tg.ClosedLoopGenerator(device=device, **(gen_kw or GEN_KW))
    xg, ug, scg = make_workload(gen, n)                      # the device-made workload is the oracle-made one
    same = (np.abs(xg - x0).max() <= 1e-13 and np.array_equal(ug, u0) and np.array_equal(scg.spec["path_kind"], sc.spec["path_kind"])
            and np.abs(scg.tables()[1] - sc.tables()[1]).max() == 0.0)
    res = gen.generate(x0, u0, sc, T)
    gen.close()
    # Steps at which the reference's central differences straddle a JUMP of f_cont (golden["fd_jump"], DESIGN.md section 5)
    # are not comparable: there the reference's Jacobian is the jump divided by 2 eps.  A trajectory is compared up to its
    # first such step; what follows it is reported separately (the loops re-converge within a few steps).
    jump = golden["fd_jump"] if exclude_fd_jumps else np.zeros_like(golden["fd_jump"])
    first = np.where(jump.any(1), jump.argmax(1), T)                      # first artefact step per trajectory, T = none
    mU = np.arange(T)[None, :] < first[:, None]                             # U[t] comparable
    mX = np.arange(T + 1)[None, :] <= first[:, None]                        # X[t] comparable (X[first] is still pre-artefact)
    dX, dU = np.abs(res["clean"] - golden["X_ipm"]), np.abs(res["U"] - golden["U_ipm"])
    eX, eU = dX[mX], dU[mU]
    oX, oU = np.abs(res["clean"] - golden["X_osqp"])[mX], np.abs(res["U"] - golden["U_osqp"])[mU]
    return {"reference": "oracle closed loop (MPC/main.py:85-101 restated), exact optimum per step", "n_traj": n, "T": T,
            "max_abs_err_X": float(eX.max()), "max_abs_err_U": float(eU.max()),
            "rms_err_X": float(np.sqrt((eX ** 2).mean())), "rms_err_U": float(np.sqrt((eU ** 2).mean())),
            "max_abs_err_X_vs_osqp": float(oX.max()), "max_abs_err_U_vs_osqp": float(oU.max()),
            "oracle_ipm_vs_osqp_X": float(np.abs(golden["X_ipm"] - golden["X_osqp"])[mX].max()),
            "oracle_ipm_vs_osqp_U": float(np.abs(golden["U_ipm"] - golden["U_osqp"])[mU].max()),
            "compared_steps": int(mU.sum()), "fd_jump_trajectories": np.nonzero(jump.any(1))[0].tolist(),
            "max_abs_err_X_after_fd_jump": float(dX[~mX].max()) if (~mX).any() else 0.0,
            "max_abs_err_X_last_100_steps": float(dX[:, -100:].max()),
            "workload_matches_oracle_generator": bool(same),
            "all_steps_accepted": bool(res["status_counts"][:, :2].sum() == n * T),
            "mean_admm_iters": float(res["iters_total"].sum() / (n * T))}


def algorithmic_flops_per_step(N, iters, check_every):
    """SURVEY.md section 8(d) convention (add/mul = 1, FMA = 2, transcendental/div/sqrt = 1), analytic Jacobians."""
    F_lin = 420 * N
    F_cond = 72 * N * (N - 1) + 78 * N
    F_hess = 2 * N * (N + 1) * (2 * N + 1) + 9 * N * (N + 1)
    F_fact = (2 * N) ** 3 / 3 + (2 * N) ** 2
    F_iter = 2 * (2 * N) ** 2 + 64 * N
    F_check = 2 * (2 * N) ** 2 + 30 * N
    return F_lin + F_cond + F_hess + F_fact + iters * F_iter + (iters / check_every) * F_check + 150


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arm
CPU_CHUNK_STEPS = 40                    # closed-loop steps per chunk
CPU_CHUNK_STARTS = (0, 300, 600, 900)   # chunks start at these steps of a trajectory: transient, mid-run and late cruise
# (16 cores x 4 chunks x 40 steps = 2560 MPC steps, about 25 core-seconds)


def _cpu_chunk(args):
    """MPC/main.py:85-101 for CPU_CHUNK_STEPS steps of one trajectory of the workload, started from the oracle's own state at
    step t0 (tests/golden/oracle_bench_config.npz): oracle port, cold-started restated OSQP each step (the reference builds a
    fresh cp.Problem per call, so its warm_start=True never takes effect)."""
    b, t0, n_steps, x, u_prev, spec, brk, coef = args
    from oracle import dynamics as dyn, mpc as ompc, refgen as R
    kind = int(spec["path_kind"])
    spline = None
    if kind == R.PATH_SPLINE:
        f, K = int(spec["spline_first"]), int(spec["spline_count"])
        spline = (np.append(brk[f:f + K], np.inf), coef[f:f + K])
    tt = time.perf_counter()
    its, nopt = 0, 0
    x = np.array(x, float); u_prev = np.array(u_prev, float)
    for t in range(t0, t0 + n_steps):
        vref_seq = R.vref_profile(int(spec["vref_kind"]), tuple(spec["vref"]), N_HORIZON, TS, t * TS, x[3])
        path_ref = R.ref_window(x[0], N_HORIZON, TS, vref_seq, kind, tuple(spec["path"]), spline)
        u_cmd, status, info = ompc.mpc_step(x, u_prev, path_ref, Ts=TS, N=N_HORIZON, vref=vref_seq, solver="osqp")
        x = dyn.plant_step(x, u_cmd, TS, plant=dyn.PLANT_GEN1)
        u_prev = u_cmd
        its += info.get("iters", 0) if info else 0
        nopt += status == "optimal"
    return time.perf_counter() - tt, its, nopt


def cpu_baseline(cores, chunks_per_core=len(CPU_CHUNK_STARTS)):
    """-> (MPC steps/s over all cores, description).  The sample: `cores` trajectories of the bench workload x the chunk
    starts above x CPU_CHUNK_STEPS steps, each chunk started from the oracle's state at that step."""
    import multiprocessing as mp
    golden = np.load(os.path.join(ROOT, "tests", "golden", "oracle_bench_config.npz"))
    n_g = int(golden["n_traj"])
    x0, u0, sc = workload_from_golden(golden)
    brk, coef = sc.tables()
    X, U = golden["X_ipm"], golden["U_ipm"]
    jobs = []
    for c in range(cores):
        b = c % n_g
        for t0 in CPU_CHUNK_STARTS[:chunks_per_core]:
            up = u0[b] if t0 == 0 else U[b, t0 - 1]
            jobs.append((b, t0, CPU_CHUNK_STEPS, X[b, t0], up, sc.spec[b], brk, coef))
    if cores > 1:
        with mp.get_context("spawn").Pool(cores) as pool:     # spawn: the parent may hold a CUDA context
            pool.map(_cpu_chunk, [(j[0], j[1], 1) + j[3:] for j in jobs[:cores]])   # start-up + imports are not the workload
            t0 = time.perf_counter()
            res = pool.map(_cpu_chunk, jobs, chunksize=1)
    else:
        t0 = time.perf_counter()
        res = [_cpu_chunk(j) for j in jobs]
    wall = time.perf_counter() - t0
    steps = len(jobs) * CPU_CHUNK_STEPS
    sample = (f"{len(jobs)} chunks of {CPU_CHUNK_STEPS} closed-loop steps ({cores} trajectories of the config-2 workload, chunks "
              f"starting at steps {list(CPU_CHUNK_STARTS[:chunks_per_core])} from the oracle's state), one process per core")
    return steps / wall, {"wall_s": wall, "mean_osqp_iters": sum(r[1] for r in res) / steps,
                          "optimal_frac": sum(r[2] for r in res) / steps, "sample": sample, "mpc_steps_in_sample": steps}


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    vals, info = [], {}
    for it in range(args.warmup + args.steps):
        v, info = cpu_baseline(cores)
        if it >= args.warmup:
            vals.append(v)
    value = float(np.mean(vals))
    sample = info.pop("sample")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "MPC steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * info["mpc_steps_in_sample"] / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "BASELINE config 2: generation_type1-style spline/sinusoidal references, closed loop",
                       "horizon_N": N_HORIZON, "Ts": TS, "plant": "generation_type1 (clipped)", "sample": sample,
                       "note": "CPU port of MPC/main.py's loop under oracle/ (the oracle's restatement of the reference's "
                               "finite-difference linearisation in plain math.* calls -- faster than the reference's own NumPy "
                               "code --, the restated CVXPY problem and the restated OSQP algorithm, cold start per step); "
                               "cvxpy / osqp are not installed and cannot be installed offline, so this stands in for the "
                               "reference's CVXPY -> OSQP call and is optimistic for it"},
            "cpu_baseline": {"value": value, "unit": "MPC steps/s", "cores": cores, "kind": "port", "sample": sample, **info},
            "e2e": {"value": value, "unit": "MPC steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
def measure_widened_rows(stream, hbm_peak):
    """SURVEY.md 8(f) rows measured beside the headline (never part of `value`): the open-loop generator kernels
    (rank 2; 65536 trajectories x 1200 steps, device-resident, CUDA events, L2 flushed) against the HBM roofline on their
    algorithmic output bytes (112 B per trajectory-step)."""
    import torch
    import trajectory_generation_b200 as tg
    out, launches = {}, 0
    B, T = 65536, 1200
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for kind in ("type1", "type2"):
        g = tg.OpenLoopGenerator(kind, Ts=TS)
        g.set_stream(stream.cuda_stream)
        x0 = torch.from_numpy(np.ascontiguousarray(np.tile(g.sample_x0(1024), (B // 1024, 1)))).cuda()
        clean = torch.empty((B, T + 1, 6), dtype=torch.float64, device="cuda")
        noisy, U = torch.empty_like(clean), torch.empty((B, T, 2), dtype=torch.float64, device="cuda")
        ms = []
        with torch.cuda.stream(stream):
            for rep in range(5):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                g.generate_device(x0.data_ptr(), B, T, clean.data_ptr(), noisy.data_ptr(), U.data_ptr(), None)
                e1.record(stream)
                e1.synchronize()
                launches += 1
                if rep >= 2:
                    ms.append(e0.elapsed_time(e1))
        t = float(np.mean(ms)) * 1e-3
        nbytes = B * (T + 1) * 96 + B * T * 16 + B * 48
        out[f"openloop_{kind}"] = {"kernel": f"tg_openloop_kernel<{kind}>", "trajectory_steps_per_s": B * T / t, "kernel_ms": t * 1e3,
                                  "batch": B, "T": T, "roofline": {"bound": "hbm", "achieved": nbytes / t / 1e9, "peak": hbm_peak,
                                                                   "unit": "GB/s", "frac": nbytes / t / 1e9 / hbm_peak}}
        g.close()
        del clean, noisy, U
    return out, launches


def dump_outputs(out_dir, outputs, traj_id0):
    """--dump-outputs: the device arrays one tg_closed_loop launch returned (dict name -> tensor [B, ...]) as <name>.npy in
    float64, for a fixed, seeded sample of the B trajectories (all of them when they fit in DUMP_BYTES), plus their global ids
    as traj_ids.npy.  The workload is a function of the trajectory ids alone, so two builds run with the same arguments can be
    compared output for output."""
    import torch
    B = outputs["clean"].shape[0]
    per_traj = 8 * (1 + sum(a[0].numel() for a in outputs.values()))
    n = min(B, max(1, (DUMP_BYTES - 4096) // per_traj))            # 4096: room for the .npy headers
    rows = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    idx = torch.from_numpy(rows).to(outputs["clean"].device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "traj_ids.npy"), (traj_id0 + rows).astype(np.float64))
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.index_select(0, idx).to(torch.float64).cpu().numpy())


def run_gpu(args, rank, world, local_rank):
    import torch
    import trajectory_generation_b200 as tg
    from trajectory_generation_b200 import _lib

    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B, T, N = args.batch, args.horizon_steps, N_HORIZON
    traj_id0 = rank * B
    kw = dict(GEN_KW)
    so = {}
    if args.check_every:
        so["check_every"] = args.check_every
    for kv in args.solver_opt:
        k, v = kv.split("=")
        so[k] = float(v)
    if so:
        kw["solver_opts"] = so
    gen = tg.ClosedLoopGenerator(device=local_rank, **kw)
    x0, u0, sc = make_workload(gen, B, traj_id0)
    brk, coef = sc.tables()
    stream = torch.cuda.Stream(device=dev)
    gen.set_stream(stream.cuda_stream)
    L = _lib.load()

    # ---- resident inputs / outputs (torch = device memory plumbing)
    def dev_t(a, dtype=torch.float64):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev) if a.size else torch.zeros(1, dtype=dtype, device=dev)
    d_x0, d_u0 = dev_t(x0), dev_t(u0)
    d_spec = torch.from_numpy(np.ascontiguousarray(sc.spec).view(np.uint8)).to(dev)
    d_brk, d_coef = dev_t(brk), dev_t(coef)
    d_clean = torch.empty((B, T + 1, 6), dtype=torch.float64, device=dev)
    d_noisy = torch.empty_like(d_clean)
    d_U = torch.empty((B, T, 2), dtype=torch.float64, device=dev)
    d_sc = torch.zeros((B, 6), dtype=torch.int32, device=dev)
    d_it = torch.zeros(B, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def launch():
        _lib.check(L.tg_closed_loop(gen.handle, B, T, d_x0.data_ptr(), d_u0.data_ptr(), d_spec.data_ptr(), d_brk.data_ptr(),
                                    d_coef.data_ptr(), traj_id0, d_clean.data_ptr(), d_noisy.data_ptr(), d_U.data_ptr(),
                                    d_sc.data_ptr(), d_it.data_ptr()))

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            launch()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = gen.kernel_launches()
    evs = []
    with torch.cuda.stream(stream):
        for _ in range(args.steps):
            flush.zero_()                                            # L2 flush between timed iterations
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); launch(); e1.record(stream)
            evs.append((e0, e1))
    barrier()
    kern_ms = [a.elapsed_time(b) for a, b in evs]
    gpu_launches = gen.kernel_launches() - launches0
    timed_launches = gpu_launches                                    # counted by the library: one per timed step
    total_ms = float(np.sum(kern_ms))
    tm = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    total_ms_max = float(tm.item())
    iters_total = int(d_it.sum().item())
    status = d_sc.sum(0).cpu().numpy()
    if dist is not None:
        agg = torch.tensor([iters_total] + status.tolist(), dtype=torch.int64, device=dev)
        dist.all_reduce(agg)
        iters_total, status = int(agg[0].item()), agg[1:].cpu().numpy()
    steps_per_launch = B * T
    value = world * steps_per_launch * args.steps / (total_ms_max * 1e-3)
    mean_iters = iters_total / (world * steps_per_launch)

    # ---- e2e: the public Python API (ClosedLoopGenerator.generate -> tg_closed_loop_host) with HOST buffers: inputs are
    # copied host -> device inside the call, the result rows land in page-locked host arrays while the kernel runs
    out = gen.alloc_result(B, T, pinned=True)
    gen.generate(x0, u0, sc, T, traj_id0, out=out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        gen.generate(x0, u0, sc, T, traj_id0, out=out)
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * steps_per_launch * args.steps / float(te.item())
    h2d = x0.nbytes + u0.nbytes + sc.spec.nbytes + brk.nbytes + coef.nbytes
    d2h = 2 * B * (T + 1) * 6 * 8 + B * T * 2 * 8 + B * 6 * 4 + B * 8
    e2e_ok = bool(np.array_equal(out["clean"], d_clean.cpu().numpy()))
    gpu_launches += args.steps + 1
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:          # the e2e calls above use their own buffers: d_* still hold the last timed step
        dump_outputs(args.dump_outputs, {"clean": d_clean, "noisy": d_noisy, "U": d_U, "status_counts": d_sc, "iters_total": d_it},
                     traj_id0)

    # ---- p50 latency of one batched mpc_step call (device-resident, B problems, cold start): on the initial states of the
    # workload (large offsets: most problems have active rows) and on its states at mid-run (t = T/2: the typical case)
    lat, lat_mid = None, None
    if rank == 0:
        ctl = tg.BatchedMPC(device=local_rank, N=N, Ts=TS)
        ctl.set_stream(stream.cuda_stream)

        def p50(x_np, up_np, t_index):
            nonlocal gpu_launches
            pr, vr = gen.ref_window(x_np, sc, t_index=t_index)
            d_x, d_up, d_pr, d_vr = dev_t(x_np), dev_t(up_np), dev_t(pr), dev_t(vr)
            d_uc = torch.empty((B, 2), dtype=torch.float64, device=dev)
            d_st, d_its = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
            ev = []
            with torch.cuda.stream(stream):
                for i in range(110):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(stream)
                    _lib.check(L.tg_mpc_step(ctl.handle, B, d_x.data_ptr(), d_up.data_ptr(), d_pr.data_ptr(), d_vr.data_ptr(), d_uc.data_ptr(),
                                             d_st.data_ptr(), d_its.data_ptr(), None, None, None, None))
                    b.record(stream)
                    ev.append((a, b))
            torch.cuda.synchronize(dev)
            gpu_launches += 111
            return float(np.median([a.elapsed_time(b) for a, b in ev[10:]])), float(d_its.double().mean().item())
        lat = p50(x0, u0, 0)
        tm_ = T // 2
        if tm_ >= 1:
            lat_mid = p50(out["clean"][:, tm_].copy(), out["U"][:, tm_ - 1].copy(), tm_)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        fp64_peak = gen.fma_peak_tflops("f64")
        kms = float(np.mean(kern_ms))
        alg_bytes = steps_per_launch * 14 * 8 + B * (6 + 2) * 8 + B * 14 * 8      # 14 fp64 words out per MPC step + x0/u0 in + row 0
        flops = steps_per_launch * algorithmic_flops_per_step(N, mean_iters, gen.cfg.check_every)
        parity = None
        if not args.no_parity:
            try:
                parity = parity_vs_golden(device=local_rank)      # outside the timed region
                # the same runs with the reference's own central-difference Jacobians: every step comparable, none excluded
                pfd = parity_vs_golden(device=local_rank, gen_kw=dict(GEN_KW, jacobian=tg.JAC_FD), exclude_fd_jumps=False)
                parity["with_reference_fd_jacobians"] = {k: pfd[k] for k in ("max_abs_err_X", "max_abs_err_U", "compared_steps",
                                                                               "all_steps_accepted", "mean_admm_iters")}
                gpu_launches += 2
            except Exception as e:
                parity = {"error": repr(e)}
        widened = None
        if not args.no_extra:
            try:
                widened, n_l = measure_widened_rows(stream, hbm_peak)
                gpu_launches += n_l
            except Exception as e:          # never let a side measurement take the headline line down
                widened = {"error": repr(e)}
        cores = os.cpu_count() or 1
        cb_val, cb_info = (0.0, {"skipped": True, "sample": "skipped"}) if args.no_cpu else cpu_baseline(cores)
        cb_sample = cb_info.pop("sample")
        line = {
            "metric": METRIC, "value": value, "unit": "MPC steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "BASELINE config 2: generation_type1-style spline/sinusoidal references, fused closed loop",
                       "batch_per_gpu": B, "global_batch": world * B, "horizon_N": N, "Ts": TS, "closed_loop_steps_T": T,
                       "mpc_steps_per_bench_step": world * steps_per_launch, "plant": "generation_type1 (clipped)", "jacobian": "analytic",
                       "solver": {"eps_abs": gen.cfg.eps_abs, "eps_rel": gen.cfg.eps_rel, "rho": gen.cfg.rho, "alpha": gen.cfg.alpha,
                                  "check_every": gen.cfg.check_every, "warm_start": bool(gen.cfg.warm_start),
                                  "free_mode": not (gen.cfg.solver_flags & 1)},
                       "parallelism": f"trajectory-parallel x{world}, no collective on the solve path",
                       "l2": "256 MB buffer zeroed before every timed launch; outputs (138 MB) exceed the 126 MB L2"},
            "mean_admm_iters_per_step": mean_iters, "status_counts": {k: int(v) for k, v in zip(tg.STATUS_STRINGS, status)},
            "p50_step_latency_ms": lat[0] if lat else None,
            "p50_step_latency_note": f"one tg_mpc_step call over {B} problems, cold start, device-resident, CUDA events; the workload's initial "
                                     f"states (mean {lat[1] if lat else 0:.1f} ADMM iterations: most have active rows)",
            "p50_step_latency_ms_midrun": lat_mid[0] if lat_mid else None,
            "p50_step_latency_midrun_note": f"same call on the closed loop's states at step {T // 2} (mean {lat_mid[1] if lat_mid else 0:.1f} iterations)",
            "e2e": {"value": e2e_value, "unit": "MPC steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": "ClosedLoopGenerator.generate (host arrays in, page-locked result arrays out; tg_closed_loop_host)",
                    "matches_resident_run": e2e_ok},
            "gpu_launches": int(gpu_launches), "timed_launches": int(timed_launches),
            "parity": parity,
            # the binding roofline of this path is the fp64 CUDA-core FMA rate (SURVEY.md 8(d): neither HBM nor tensor cores;
            # the only dense contraction is a 40 x 40 SPD inversion per problem); algorithmic flops per MPC step by the
            # SURVEY's convention at the measured mean iteration count.  HBM is reported beside it.
            "roofline": {"bound": "fp64 CUDA-core FMA (tensor cores are not applicable: fp64, 40x40 per problem)",
                         "achieved": flops / (kms * 1e-3) / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": flops / (kms * 1e-3) / 1e12 / fp64_peak,
                         "peak_source": "tg_fma_peak micro-benchmark in this run (MEASURED_PEAKS.json has no fp64 entry; nominal 37)",
                         "traffic": None, "traffic_note": "DRAM bytes are an ncu metric: profiles/r02_closed_loop_ncu.txt",
                         "kernel": "tw_closed_loop_kernel<2,1,20>", "kernel_ms": kms,
                         "algorithmic_flops_per_mpc_step": flops / steps_per_launch},
            "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / (kms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes / (kms * 1e-3) / 1e9 / hbm_peak, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes,
                             "note": "112 B leave the SM per MPC step: not the bound"},
            "cpu_baseline": {"value": cb_val, "unit": "MPC steps/s", "cores": cores, "kind": "port", "sample": cb_sample, **cb_info},
            "clocks": clocks,
            "widened_rows": widened,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="trajectories per GPU")
    ap.add_argument("--horizon-steps", type=int, default=1200, help="closed-loop steps T per trajectory")
    ap.add_argument("--check-every", type=int, default=0, help="override the ADMM termination-check interval (0 = library default)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (development runs)")
    ap.add_argument("--no-extra", action="store_true", help="skip the side measurements of the widened rows (open-loop generators)")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity sample against the golden oracle loops (development runs)")
    ap.add_argument("--solver-opt", action="append", default=[], help="development: key=value override of a tg_config solver field")
    ap.add_argument("--dump-outputs", metavar="DIR", help="GPU path only: write the last timed step's outputs (clean, noisy, U, "
                    "status_counts, iters_total of rank 0's trajectories; a fixed sample of them beyond 64 MB) as DIR/<name>.npy "
                    "in float64")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs the GPU path (--impl b200) and at least one timed step (--steps >= 1)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        args.warmup = max(args.warmup, 3) if args.warmup else 0
        run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
