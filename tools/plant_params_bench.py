#!/usr/bin/env python
"""Cost of per-trajectory plant parameters (tg_closed_loop_params, tg_openloop_type{1,2}_params).

  python tools/plant_params_bench.py [--batches 1024 4736] [--horizon-steps 1200] [--openloop-batch 65536] [--rounds 2]
                                     [--reps 3] [--out FILE]

Closed loop: bench.py's workload (BASELINE config 2, N = 20, Ts = 0.01, generation_type1's clipped plant, advancing vref) with
inputs resident in HBM, four arms timed with CUDA events around single launches (L2 flushed before each), alternated round by
round:
  none     no table (the compile-time-horizon instance bench.py times)
  uniform  a table whose every row is the handle's params (the plant instance; rows bit-identical to `none`)
  rand     m, Iz, Cm1, Df, Dr scaled by U(0.8, 1.2) per trajectory: the tyre constants are kept, so are the tyre tables
  randbc   as rand, and Bf, Cf, Br, Cr scaled by U(0.9, 1.1): those plants evaluate the tyre curve with libdevice
Open loop: type 1 and type 2 at --openloop-batch x T with no table, rand and randbc.
Prints one JSON object: GPU name and power limit, steps/s of every round, ADMM iterations per step and status counts.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import GEN_KW, make_workload  # noqa: E402
from ctrl_table_bench import gpu_info  # noqa: E402


def random_table(gen, B, seed, bc):
    rng = np.random.default_rng(seed)
    p = dict(zip(_order(), gen.cfg.params[:]))
    cols = {k: p[k] * rng.uniform(0.8, 1.2, B) for k in ("m", "Iz", "Cm1", "Df", "Dr")}
    if bc:
        cols.update({k: p[k] * rng.uniform(0.9, 1.1, B) for k in ("Bf", "Cf", "Br", "Cr")})
    return gen.plant_table(B, **cols)


def _order():
    from trajectory_generation_b200 import _lib
    return _lib.PARAM_ORDER


def timed(launch, arms, rounds, reps, stream, flush, work):
    import torch
    rec = {a: {"steps_per_s": []} for a in arms}
    with torch.cuda.stream(stream):
        for a in arms:                                   # warm-up: module load, first-touch of the outputs
            launch(a)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for a in arms:
            evs = []
            with torch.cuda.stream(stream):
                for _ in range(reps):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream); launch(a); e1.record(stream)
                    evs.append((e0, e1))
            torch.cuda.synchronize()
            ms = sum(e0.elapsed_time(e1) for e0, e1 in evs)
            rec[a]["steps_per_s"].append(work * reps / (ms * 1e-3))
    for a in arms:
        rec[a]["mean_steps_per_s"] = float(np.mean(rec[a]["steps_per_s"]))
        rec[a]["over_none"] = rec[a]["mean_steps_per_s"] / rec[arms[0]]["mean_steps_per_s"] if a != arms[0] else 1.0
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[1024, 4736])
    ap.add_argument("--horizon-steps", type=int, default=1200)
    ap.add_argument("--openloop-batch", type=int, default=65536)
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
    gen = tg.ClosedLoopGenerator(**GEN_KW)
    stream = torch.cuda.Stream(device=dev)
    gen.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"workload": f"bench.make_workload, N = {GEN_KW['N']}, Ts = {GEN_KW['Ts']}, T = {T}", **gpu_info(),
              "closed_loop": {}, "openloop": {}}

    def dev_t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev) if a.size else torch.zeros(1, dtype=torch.float64, device=dev)

    arms = ("none", "uniform", "rand", "randbc")
    for B in args.batches:
        x0, u0, sc = make_workload(gen, B)
        brk, coef = sc.tables()
        d_x0, d_u0, d_brk, d_coef = dev_t(x0), dev_t(u0), dev_t(brk), dev_t(coef)
        d_spec = torch.from_numpy(np.ascontiguousarray(sc.spec).view(np.uint8)).to(dev)
        d_clean = torch.empty((B, T + 1, 6), dtype=torch.float64, device=dev)
        d_noisy = torch.empty_like(d_clean)
        d_U = torch.empty((B, T, 2), dtype=torch.float64, device=dev)
        d_sc = {a: torch.zeros((B, 6), dtype=torch.int32, device=dev) for a in arms}
        d_it = {a: torch.zeros(B, dtype=torch.int64, device=dev) for a in arms}
        d_tab = {"uniform": dev_t(gen.plant_table(B)), "rand": dev_t(random_table(gen, B, B, False)),
                 "randbc": dev_t(random_table(gen, B, B, True))}

        def launch(arm):
            _lib.check(L.tg_closed_loop_params(gen.handle, B, T, d_x0.data_ptr(), d_u0.data_ptr(), d_spec.data_ptr(), None,
                                               d_tab[arm].data_ptr() if arm in d_tab else None, d_brk.data_ptr(),
                                               d_coef.data_ptr(), 0, d_clean.data_ptr(), d_noisy.data_ptr(), d_U.data_ptr(),
                                               d_sc[arm].data_ptr(), d_it[arm].data_ptr()))
        rec = timed(launch, arms, args.rounds, args.reps, stream, flush, B * T)
        for a in arms:
            rec[a]["iters_per_step"] = int(d_it[a].sum().item()) / (B * T)
            rec[a]["status_counts"] = d_sc[a].sum(0).cpu().tolist()
        # the rows of the last launches of `none` and `uniform` are equal bit for bit
        with torch.cuda.stream(stream):
            launch("none")
        torch.cuda.synchronize()
        c_none = d_clean.cpu().numpy()
        with torch.cuda.stream(stream):
            launch("uniform")
        torch.cuda.synchronize()
        rec["none_uniform_rows_identical"] = bool(np.array_equal(c_none, d_clean.cpu().numpy()))
        result["closed_loop"][str(B)] = rec
        del d_clean, d_noisy, d_U
    B = args.openloop_batch
    for kind in ("type1", "type2"):
        og = tg.OpenLoopGenerator(kind, Ts=0.01)
        og.set_stream(stream.cuda_stream)
        x0 = dev_t(og.sample_x0(B, seed=1))
        d_clean = torch.empty((B, T + 1, 6), dtype=torch.float64, device=dev)
        d_noisy = torch.empty_like(d_clean)
        d_U = torch.empty((B, T, 2), dtype=torch.float64, device=dev)
        d_tab = {"rand": dev_t(random_table(og, B, 7, False)), "randbc": dev_t(random_table(og, B, 7, True))}

        def launch_ol(arm):
            og.generate_device(x0.data_ptr(), B, T, d_clean.data_ptr(), d_noisy.data_ptr(), d_U.data_ptr(), None,
                               plant_dev=d_tab[arm].data_ptr() if arm in d_tab else None)
        result["openloop"][kind] = timed(launch_ol, ("none", "rand", "randbc"), args.rounds, args.reps, stream, flush, B * T)
        result["openloop"][kind]["batch"] = B
        del d_clean, d_noisy, d_U
        og.close()
    txt = json.dumps(result, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
