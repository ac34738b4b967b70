"""Cost of nonnegative ALS (hals_als_half_step_nonnegative) against the Cholesky routes, on bench.py's synthetic c2
(MovieLens-20M shape, rank 64) and c3 (Netflix-prize shape, rank 128) workloads.

Three routes, each from the same inputs and initial factors:
  (a) tc     the default Cholesky route (tensor-core kernels, split-form factors)
  (b) simt   the CUDA-core Cholesky route (HALS_FORCE_SIMT=1, read once per process: a child process with a timeout;
             the engine uses the fp32 stateless entry point, which that variable routes to the CUDA-core kernels)
  (c) nnls   nonnegative=True (CUDA-core kernels, block-principal-pivoting NNLS)
(c) against (b) is what the NNLS solve costs over the Cholesky solve with everything else equal.

Every route runs with CUDA graphs (as bench.py), W warm-up sweeps, then S sweeps with CUDA events around the item and
the user half-step.  Prints one JSON line per workload and route: median item / user / sweep ms, train RMSE after the
W + S sweeps, fraction of exactly-zero entries in X and Y (rows with ratings), rows that reached the NNLS iteration
cap, the ALS kernels one sweep launched, and the GPU name and power limit.
Usage: python scripts/bench_als_nonneg.py [--workloads c2 c3] [--sweeps 5] [--warmup 2] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hybrid_als_twotower_recommender_b200  # noqa: E402,F401
from bench import WORKLOADS, synth_coo  # noqa: E402
from hybrid_als_twotower_recommender_b200.als_engine import AlsEngine  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": line}


def als_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name.split("(")[0].replace("void ", "") for e in prof.events() if "als_" in e.name}
    return sorted(names)


def run_route(name, route, sweeps, warmup):
    w = WORKLOADS[name]
    dev = torch.device("cuda")
    u, i, r = synth_coo(w, dev)
    eng = AlsEngine(u, i, r, w["users"], w["items"], w["rank"], w["reg"], device=dev, nonnegative=(route == "nnls"))
    if route == "simt":
        eng.split = None          # the stateless fp32 half-step: HALS_FORCE_SIMT=1 sends it to the CUDA-core kernels
    eng.init_user_factors(1)
    kernels = als_kernels(eng.sweep)   # one eager sweep, before the graphs
    eng.enable_graphs()
    for _ in range(warmup):
        eng.sweep()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(sweeps)]
    torch.cuda.synchronize()
    for e in ev:
        e[0].record()
        eng.item_half_step()
        e[1].record()
        eng.user_half_step()
        e[2].record()
    torch.cuda.synchronize()
    item = [e[0].elapsed_time(e[1]) for e in ev]
    user = [e[1].elapsed_time(e[2]) for e in ev]
    eng.sync_factors()
    rmse = eng.rmse(u, i, r)
    X, Y = eng.X[eng.user_present], eng.Y[eng.item_present]
    out = {"workload": name, "route": route, "rank": w["rank"], "sweeps": sweeps, "warmup": warmup,
           "item_ms": statistics.median(item), "user_ms": statistics.median(user),
           "sweep_ms": statistics.median([a + b for a, b in zip(item, user)]), "train_rmse": rmse,
           "zero_frac_X": float((X == 0).float().mean()), "zero_frac_Y": float((Y == 0).float().mean()),
           "min_X": float(X.min()), "min_Y": float(Y.min()), "nnls_capped_rows": eng.nonneg_capped_rows(),
           "als_kernels": kernels}
    del eng, u, i, r
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c2", "c3"])
    ap.add_argument("--sweeps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--route", choices=["all", "tc", "simt", "nnls"], default="all")
    ap.add_argument("--timeout", type=float, default=900.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = gpu_info()
    lines = []
    for name in args.workloads:
        routes = ["tc", "simt", "nnls"] if args.route == "all" else [args.route]
        for route in routes:
            if route == "simt" and os.environ.get("HALS_FORCE_SIMT") != "1":
                cmd = [sys.executable, os.path.abspath(__file__), "--workloads", name, "--route", "simt",
                       "--sweeps", str(args.sweeps), "--warmup", str(args.warmup)]
                p = subprocess.run(cmd, env=dict(os.environ, HALS_FORCE_SIMT="1"), capture_output=True, text=True,
                                   timeout=args.timeout)
                if p.returncode != 0:
                    raise RuntimeError(f"simt child failed:\n{p.stdout}\n{p.stderr}")
                res = json.loads(p.stdout.strip().splitlines()[-1])
            else:
                res = run_route(name, route, args.sweeps, args.warmup)
                res.update(info)
            print(json.dumps(res), flush=True)
            lines.append(res)
    if args.out:
        with open(args.out, "w") as f:
            for res in lines:
                f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
