#!/usr/bin/env python
"""Cost of per-trajectory controller settings (tg_closed_loop_ctrl) on the bench workload.

  python tools/ctrl_table_bench.py [--batches 1024 4736] [--horizon-steps 1200] [--rounds 2] [--reps 3] [--out FILE]

bench.py's workload (BASELINE config 2, N = 20, Ts = 0.01, generation_type1's clipped plant, advancing vref) with inputs resident
in HBM, four arms timed with CUDA events around single launches (L2 flushed before each), alternated round by round:
  a  no table, compile-time-horizon instance (what bench.py times)
  b  no table, run-time-horizon instance (TRAJGEN_DYNAMIC_N=1 at handle creation)
  c  a table that repeats the handle's settings for every trajectory (the ctrl instance)
  d  a randomised table: q_c, q_phi, q_vx, R, Rd scaled log-uniformly in [0.5, 2], the du limits scaled by U(0.5, 1)
Prints one JSON object: GPU name and power limit, and per batch and arm the steps/s of every round and ADMM iterations per step.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import GEN_KW, make_workload  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": "unknown", "error": str(e)}


def random_table(gen, B, seed):
    rng = np.random.default_rng(seed)
    t = gen.ctrl_table(B)
    for f in ("q_c", "q_phi", "q_vx"):
        t[f] *= np.exp(rng.uniform(np.log(0.5), np.log(2.0), B))
    for f in ("R", "Rd"):
        t[f] *= np.exp(rng.uniform(np.log(0.5), np.log(2.0), B))[:, None]     # one factor per matrix keeps it definite
    s = rng.uniform(0.5, 1.0, (B, 2))
    t["du_lo"] *= s
    t["du_hi"] *= s
    return gen.ctrl_table(B, **{f: t[f] for f in t.dtype.names})                # through the checks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[1024, 4736])
    ap.add_argument("--horizon-steps", type=int, default=1200)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3, help="timed launches per arm and round")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import trajectory_generation_b200 as tg
    from trajectory_generation_b200 import _lib
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L = _lib.load()
    T = args.horizon_steps
    os.environ.pop("TRAJGEN_DYNAMIC_N", None)
    gen_a = tg.ClosedLoopGenerator(**GEN_KW)
    os.environ["TRAJGEN_DYNAMIC_N"] = "1"
    gen_b = tg.ClosedLoopGenerator(**GEN_KW)
    del os.environ["TRAJGEN_DYNAMIC_N"]
    stream = torch.cuda.Stream(device=dev)
    for g in (gen_a, gen_b):
        g.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"workload": f"bench.make_workload, N = {GEN_KW['N']}, Ts = {GEN_KW['Ts']}, T = {T}", **gpu_info(), "batches": {}}

    def dev_t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev) if a.size else torch.zeros(1, dtype=torch.float64, device=dev)

    for B in args.batches:
        x0, u0, sc = make_workload(gen_a, B)
        brk, coef = sc.tables()
        d_x0, d_u0, d_brk, d_coef = dev_t(x0), dev_t(u0), dev_t(brk), dev_t(coef)
        d_spec = torch.from_numpy(np.ascontiguousarray(sc.spec).view(np.uint8)).to(dev)
        d_clean = torch.empty((B, T + 1, 6), dtype=torch.float64, device=dev)
        d_noisy = torch.empty_like(d_clean)
        d_U = torch.empty((B, T, 2), dtype=torch.float64, device=dev)
        d_sc = torch.zeros((B, 6), dtype=torch.int32, device=dev)
        d_it = torch.zeros(B, dtype=torch.int64, device=dev)
        tables = {"c": gen_a.ctrl_table(B), "d": random_table(gen_a, B, seed=B)}
        d_tab = {k: torch.from_numpy(v.view(np.uint8)).to(dev) for k, v in tables.items()}

        def launch(arm):
            g = gen_b if arm == "b" else gen_a
            if arm in ("a", "b"):
                rc = L.tg_closed_loop(g.handle, B, T, d_x0.data_ptr(), d_u0.data_ptr(), d_spec.data_ptr(), d_brk.data_ptr(),
                                      d_coef.data_ptr(), 0, d_clean.data_ptr(), d_noisy.data_ptr(), d_U.data_ptr(),
                                      d_sc.data_ptr(), d_it.data_ptr())
            else:
                rc = L.tg_closed_loop_ctrl(g.handle, B, T, d_x0.data_ptr(), d_u0.data_ptr(), d_spec.data_ptr(),
                                           d_tab[arm].data_ptr(), d_brk.data_ptr(), d_coef.data_ptr(), 0, d_clean.data_ptr(),
                                           d_noisy.data_ptr(), d_U.data_ptr(), d_sc.data_ptr(), d_it.data_ptr())
            _lib.check(rc)

        arms = ("a", "b", "c", "d")
        rec = {a: {"steps_per_s": [], "iters_per_step": None} for a in arms}
        outs = {}
        with torch.cuda.stream(stream):
            for a in arms:                                   # warm-up: module load, first-touch of the outputs
                launch(a)
        torch.cuda.synchronize()
        for _ in range(args.rounds):
            for a in arms:
                evs = []
                with torch.cuda.stream(stream):
                    for _ in range(args.reps):
                        flush.zero_()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(stream); launch(a); e1.record(stream)
                        evs.append((e0, e1))
                torch.cuda.synchronize()
                ms = sum(e0.elapsed_time(e1) for e0, e1 in evs)
                rec[a]["steps_per_s"].append(B * T * args.reps / (ms * 1e-3))
                rec[a]["iters_per_step"] = int(d_it.sum().item()) / (B * T)
                outs[a] = (d_clean.cpu().numpy(), d_U.cpu().numpy())
        for a in arms:
            rec[a]["mean_steps_per_s"] = float(np.mean(rec[a]["steps_per_s"]))
        ref = rec["b"]["mean_steps_per_s"]
        rec["c_over_b"] = rec["c"]["mean_steps_per_s"] / ref
        rec["c_over_a"] = rec["c"]["mean_steps_per_s"] / rec["a"]["mean_steps_per_s"]
        rec["b_c_outputs_identical"] = bool(all(np.array_equal(x, y) for x, y in zip(outs["b"], outs["c"])))
        result["batches"][str(B)] = rec
    txt = json.dumps(result, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
