"""ALS top-k by raw dot product (ALSModel.recommend_for_*): one pass (hals_score_topk) against the two-pass hybrid call
it replaces for ALS-only scoring (hals_score_extrema + hals_score_blend_topk with weights (1, 0)).

Variants, alternated within every repetition, over slabs of 65536 query rows (as ALSModel.recommend_for_* runs them):
  one_pass  HybridScorer(Q, C, None, None).topk_dot(k)
  two_pass  HybridScorer(Q, C, None, None).recommend(k, 1.0, 0.0): extrema + blend.  (s - min) / (max - min) is a
            monotone map of the raw score, so the ranking is the same up to fp32 rounding of near-ties.
Shapes: MovieLens-20M (138,493 users x 26,744 items, rank 64, k = 10 and 100, both directions) and the per-GPU
config-5 shape (65,536 and 1,000,000 users x 1,250,000 items, rank 128, k = 100, users -> items).  Factors are seeded
N(0, 1/rank) for the queries and N(0, 1) for the candidates.
Timed with CUDA events: 1 warm-up, median of --reps (>= 5) repetitions.  Flagged rows (re-run exactly on the CUDA-core
kernel) are counted in an untimed pass, as is the agreement of the two variants' index lists: a row may differ only
where the raw scores of the items involved lie within `tie_tol` * |q| * max|c| of each other.
Prints one JSON line per (shape, direction, k) and the GPU name and power limit; --out also writes them as a JSON list.
Usage: python scripts/bench_als_recommend.py [--reps 5] [--out FILE] [--only ml20m|c5]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hybrid_als_twotower_recommender_b200  # noqa: E402,F401
from hybrid_als_twotower_recommender_b200 import scoring  # noqa: E402

TIE_TOL = 1e-5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": line}


def agreement(Q, C, a_idx, b_idx, detail_rows=2000):
    """Rows whose two index lists differ, and whether every difference is a near-tie of raw scores."""
    diff = torch.nonzero((a_idx != b_idx).any(1)).flatten()
    cmax = float(torch.linalg.vector_norm(C.double(), dim=1).max())
    worst, bad = 0.0, 0
    for r in diff[:detail_rows].tolist():
        a, b = a_idx[r], b_idx[r]
        items = torch.unique(torch.cat([a, b]))
        items = items[items >= 0].long()
        s = C[items].double() @ Q[r].double()
        scale = float(torch.linalg.vector_norm(Q[r].double())) * cmax
        score = dict(zip(items.tolist(), s.tolist()))
        # position by position the two lists must hold items of (nearly) the same raw score
        for x, y in zip(a.tolist(), b.tolist()):
            if x != y:
                gap = abs(score.get(x, float("inf")) - score.get(y, float("-inf"))) / scale
                worst = max(worst, gap)
                bad += gap > TIE_TOL
    return {"rows": int(a_idx.shape[0]), "rows_differing": int(diff.numel()),
            "rows_checked": int(min(diff.numel(), detail_rows)), "positions_beyond_tie_tol": int(bad),
            "max_gap_rel_to_q_norm_x_max_c_norm": worst, "tie_tol": TIE_TOL}


def measure(name, direction, Q, C, k, slab, reps, warmup, info):
    n_q, n_c, rank = Q.shape[0], C.shape[0], Q.shape[1]
    sc = scoring.HybridScorer(Q, C, None, None)
    slabs = [(u0, min(n_q, u0 + slab)) for u0 in range(0, n_q, slab)]
    variants = {"one_pass": lambda u0, u1: sc.topk_dot(k, u0, u1),
                "two_pass": lambda u0, u1: sc.recommend(k, 1.0, 0.0, u0, u1)}
    # untimed: flagged rows (the counter is per call) and the full index lists for the agreement check
    flagged, lists = {}, {}
    for v, fn in variants.items():
        f, out = 0, []
        for u0, u1 in slabs:
            out.append(fn(u0, u1)[0])
            f += max(sc.flagged_users(u1 - u0, k, dot=(v == "one_pass")), 0)
        flagged[v], lists[v] = f, torch.cat(out)
    agree = agreement(Q, C, lists["one_pass"], lists["two_pass"])
    del lists
    times = {v: [] for v in variants}
    for rep in range(warmup + reps):
        for v, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for u0, u1 in slabs:
                fn(u0, u1)
            e1.record()
            torch.cuda.synchronize()
            if rep >= warmup:
                times[v].append(e0.elapsed_time(e1))
    res = {"shape": name, "direction": direction, "n_q": n_q, "n_c": n_c, "rank": rank, "k": k, "slab": slab,
           "reps": reps, "warmup": warmup, **info}
    for v in variants:
        t = sorted(times[v])
        med = t[len(t) // 2]
        res[v] = {"ms_median": med, "ms_min": t[0], "ms_max": t[-1], "pairs_per_s": n_q * n_c / (med * 1e-3),
                  "flagged_rows": flagged[v]}
    res["one_pass_over_two_pass"] = res["one_pass"]["ms_median"] / res["two_pass"]["ms_median"]
    res["agreement"] = agree
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--slab", type=int, default=65536)
    ap.add_argument("--only", choices=["ml20m", "c5"], default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be >= 5 (the median of at least five repetitions)")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 kernels")
    info = gpu_info()
    results = []

    def emit(r):
        print(json.dumps(r), flush=True)
        results.append(r)

    g = torch.Generator(device="cuda").manual_seed(1)
    if args.only in (None, "ml20m"):
        U, I, rank = 138_493, 26_744, 64
        Uf = torch.randn(U, rank, device="cuda", generator=g) * rank ** -0.5
        If = torch.randn(I, rank, device="cuda", generator=g)
        for k in (10, 100):
            emit(measure("movielens20m", "users->items", Uf, If, k, args.slab, args.reps, args.warmup, info))
            emit(measure("movielens20m", "items->users", If, Uf, k, args.slab, args.reps, args.warmup, info))
        del Uf, If
    if args.only in (None, "c5"):
        I, rank, k = 1_250_000, 128, 100
        If = torch.randn(I, rank, device="cuda", generator=g)
        for U in (65_536, 1_000_000):
            Uf = torch.randn(U, rank, device="cuda", generator=g) * rank ** -0.5
            emit(measure("config5_per_gpu", "users->items", Uf, If, k, args.slab, args.reps, args.warmup, info))
            del Uf
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
