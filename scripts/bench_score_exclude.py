"""Cost of per-user exclusion lists in the hybrid top-k pass (hals_score_blend_topk_excluding) at the per-GPU
config-5 shape of scripts/bench_score.py: ka = 128, kt = 50, 1.25 M items, k = 100.

Pass 2 only (the extrema pass does not change), over slabs of 65536 users like bench.py, timed with CUDA events.
Four variants alternate within every repetition:
  plain      hals_score_blend_topk
  empty      the excluding entry point with all-empty lists
  zipf150    150 items per user (about the MovieLens-20M mean) drawn from a Zipf(1) popularity over the items
  own_top156 each user's own top-156 (from a k = 156 call): removes exactly the strongest survivors, the adversarial
             case for the candidate streams and the verification margin
Prints one JSON line per user count: median pass-2 ms, pairs/s, flagged (exactly re-run) users per variant, and the
GPU name and power limit.  Usage: python scripts/bench_score_exclude.py [--users 65536 1000000] [--reps 5]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hybrid_als_twotower_recommender_b200  # noqa: E402,F401
from hybrid_als_twotower_recommender_b200 import scoring  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": line}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, nargs="+", default=[65536])
    ap.add_argument("--items", type=int, default=1_250_000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--slab", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    I, k, ka, kt = args.items, args.k, 128, 50
    info = gpu_info()
    for U in args.users:
        g = torch.Generator(device="cuda").manual_seed(1)
        Ua = torch.randn(U, ka, device="cuda", generator=g) * ka ** -0.5
        Ia = torch.randn(I, ka, device="cuda", generator=g)
        Ut = torch.nn.functional.layer_norm(torch.randn(U, kt, device="cuda", generator=g), (kt,))
        It = torch.nn.functional.layer_norm(torch.randn(I, kt, device="cuda", generator=g), (kt,))
        sc = scoring.HybridScorer(Ua, Ia, Ut, It)
        slabs = [(u0, min(U, u0 + args.slab)) for u0 in range(0, U, args.slab)]
        ex = [sc.extrema(u0, u1) for u0, u1 in slabs]

        # exclusion lists over all U users (rowptr sliced per slab by the scorer)
        empty = (torch.zeros(U + 1, dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda"))
        per = 150
        cdf = torch.cumsum(1.0 / torch.arange(1, I + 1, device="cuda", dtype=torch.float64), 0)   # Zipf(1) by rank
        rank_item = torch.randperm(I, device="cuda", generator=g)                                  # rank -> item
        draws = torch.searchsorted(cdf, torch.rand(U * per, device="cuda", generator=g, dtype=torch.float64) * cdf[-1])
        draws.clamp_(max=I - 1)
        zipf = scoring.exclusion_lists(torch.arange(U, device="cuda").repeat_interleave(per), rank_item[draws], U)
        del draws
        top = torch.cat([sc.topk_local(e, 156, 0.8, 0.2, u0, u1)[0] for e, (u0, u1) in zip(ex, slabs)])
        own = scoring.exclusion_lists(torch.arange(U, device="cuda").repeat_interleave(156), top.reshape(-1).long(), U)
        del top
        variants = {"plain": None, "empty": empty, "zipf150": zipf, "own_top156": own}

        def run(excl):
            out = []
            for e, (u0, u1) in zip(ex, slabs):
                out.append(sc.topk_local(e, k, 0.8, 0.2, u0, u1, exclude=excl))
            return out

        # untimed: flagged users per variant (the counter is per call: read after each slab) and the empty-list check
        flagged, first = {}, {}
        for name, excl in variants.items():
            f = 0
            for e, (u0, u1) in zip(ex, slabs):
                r = sc.topk_local(e, k, 0.8, 0.2, u0, u1, exclude=excl)
                f += max(sc.flagged_users(u1 - u0, k), 0)
                if u0 == 0:
                    first[name] = r
            flagged[name] = f
        (pi, ps), (ei, es) = first["plain"], first["empty"]
        assert torch.equal(pi, ei) and torch.equal(ps.view(torch.int32), es.view(torch.int32)), "empty lists changed the result"
        times = {n: [] for n in variants}
        for rep in range(args.warmup + args.reps):
            for name, excl in variants.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(excl)
                e1.record()
                torch.cuda.synchronize()
                if rep >= args.warmup:
                    times[name].append(e0.elapsed_time(e1))
        res = {"U": U, "I": I, "k": k, "ka": ka, "kt": kt, "slab": args.slab, "reps": args.reps, **info,
               "excluded_per_user": {"zipf150": int(zipf[1].numel()) / U, "own_top156": 156}}
        base = sorted(times["plain"])[len(times["plain"]) // 2]
        for name in variants:
            t = sorted(times[name])
            med = t[len(t) // 2]
            res[name] = {"ms_pass2_median": med, "ms_min": t[0], "ms_max": t[-1], "pairs_per_s": U * I / (med * 1e-3),
                         "vs_plain": med / base, "flagged_users": flagged[name]}
        print(json.dumps(res), flush=True)
        del sc, Ua, Ia, Ut, It, zipf, own, empty, variants
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
