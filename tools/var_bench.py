"""Development: time bench.py for library variants (tools/_var/*.so via TRAJGEN_LIB) and problems per CTA (TRAJGEN_PPC).
usage: python tools/var_bench.py lib:ppc:batch[:extra-env=val] ..."""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for spec in sys.argv[1:]:
    f = spec.split(":")
    lib, ppc, batch = f[0], f[1], f[2]
    env = dict(os.environ)
    if lib: env["TRAJGEN_LIB"] = os.path.join(ROOT, "tools", "_var", lib)
    if ppc: env["TRAJGEN_PPC"] = ppc
    for kv in f[3:]:
        k, v = kv.split("="); env[k] = v
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu", "--no-extra", "--batch", batch, "--steps", "3"],
                       env=env, capture_output=True, text=True)
    try:
        d = json.loads(p.stdout.strip().splitlines()[-1])
        print(f"{spec}: {d['value']:.3e} steps/s  {d['ms_per_step']:.1f} ms  iters {d['mean_admm_iters_per_step']:.2f}  e2e {d['e2e']['value']:.3e}  p50 step {d['p50_step_latency_ms']:.3f} ms  status {d['status_counts']}", flush=True)
    except Exception as e:
        print(f"{spec}: FAILED {e!r}\n{p.stdout[-500:]}\n{p.stderr[-1500:]}", flush=True)
