"""Hybrid top-k over per-user candidate lists (hals_score_blend_topk_lists, get_hybrid_recommendations_batch).

Workloads:
  rerank     1,000,000 users x 256 candidates each, drawn Zipf-popular (p ~ 1 / rank^0.9) from 1,250,000 items (ids
             shuffled, so popular rows are scattered), ka = 128, kt = 50, top_k = 100.  Timed: the blend call with
             per-user weights and with one scalar pair, and the F1 stage of a call with ratings (the two raw top-10
             calls, ALS operands alone and tower operands alone, plus hals_f1_at_k).
  reference  10,000 users x the full 9,964-item list, ka = 10, kt = 50, top_k = 5: the list call against
             HybridScorer.recommend (what recommend_batch runs) on the same operands.
  loop       get_hybrid_recommendations in a Python loop over a 200-user SAMPLE of the reference shape (synthetic
             models), against get_hybrid_recommendations_batch on the same 200 users and on all 10,000.
Kernel-level times: CUDA events, one warm-up call per shape, median of --reps.  The re-rank item operands (0.9 GB)
exceed the 126 MB L2, but the Zipf draw keeps the popular rows resident, so the gather is served partly from L2:
gathered bytes / time is reported against the 7.7 TB/s HBM data-sheet figure.
Prints one JSON line per measurement and the GPU name and power limit; --out also writes them as a JSON list.
Usage: python scripts/bench_hybrid_lists.py [--reps 5] [--out FILE] [--only rerank|reference|loop]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hybrid_als_twotower_recommender_b200 as pkg  # noqa: E402
from hybrid_als_twotower_recommender_b200 import _native as nat, scoring  # noqa: E402

HBM_TBS = 7.7


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": line}


def timed(fn, reps):
    fn()                                             # warm-up of this shape
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def rates(ms, pairs, ka, kt):
    gathered = pairs * (ka + kt) * 4
    return {"ms": round(ms, 3), "pairs_per_s": pairs / (ms * 1e-3), "gathered_bytes": gathered,
            "gathered_TB_per_s": gathered / (ms * 1e-3) / 1e12,
            "share_of_hbm_7.7TBs": gathered / (ms * 1e-3) / 1e12 / HBM_TBS}


def rerank(reps):
    U, I, L, ka, kt, k = 1_000_000, 1_250_000, 256, 128, 50, 100
    g = torch.Generator(device="cuda").manual_seed(0)
    Ua = torch.randn(U, ka, device="cuda", generator=g) * ka ** -0.5
    Ia = torch.randn(I, ka, device="cuda", generator=g)
    Ut = torch.randn(U, kt, device="cuda", generator=g)
    It = torch.randn(I, kt, device="cuda", generator=g)
    p = 1.0 / torch.arange(1, I + 1, device="cuda", dtype=torch.float64) ** 0.9
    cdf = torch.cumsum(p / p.sum(), 0)
    rank = torch.searchsorted(cdf, torch.rand(U * L, device="cuda", generator=g, dtype=torch.float64)).clamp(max=I - 1)
    cand = torch.randperm(I, device="cuda", generator=g)[rank].to(torch.int32)
    rowptr = torch.arange(U + 1, device="cuda", dtype=torch.int64) * L
    w = torch.where(torch.rand(U, 1, device="cuda", generator=g) < 0.5, 0.8, 0.2)
    w = torch.cat([w, 1 - w], 1).float().contiguous()
    pairs = U * L
    distinct = int(torch.unique(cand).numel())
    out = []
    ms = timed(lambda: scoring.blend_topk_lists(Ua, Ia, Ut, It, rowptr, cand, k, row_weights=w), reps)
    out.append({"workload": "rerank", "variant": "per_user_weights", **rates(ms, pairs, ka, kt)})
    ms_s = timed(lambda: scoring.blend_topk_lists(Ua, Ia, Ut, It, rowptr, cand, k, w_als=0.8, w_tt=0.2), reps)
    out.append({"workload": "rerank", "variant": "scalar_weights", **rates(ms_s, pairs, ka, kt)})
    a_ptr = torch.arange(U + 1, device="cuda", dtype=torch.int64) * 8        # 8 rated positions per user
    a_items = torch.sort(torch.randint(0, I, (U, 8), device="cuda", generator=g, dtype=torch.int32), 1).values.reshape(-1)
    f1 = torch.empty(U, device="cuda")
    tp = torch.empty(U, device="cuda", dtype=torch.int32)

    def f1_stage():
        for ops in ((Ua, Ia, None, None), (None, None, Ut, It)):
            pos, _ = scoring.blend_topk_lists(*ops, rowptr, cand, 10, w_als=1.0, w_tt=1.0, raw=True)
            pred = torch.where(pos >= 0, cand[pos.clamp(min=0).long()], -1).to(torch.int32)
            nat.check(nat.lib().hals_f1_at_k(nat.ptr(pred), 10, 10, nat.ptr(a_ptr), nat.ptr(a_items), U, nat.ptr(f1),
                                             nat.ptr(tp), nat.current_stream()))
    ms_f1 = timed(f1_stage, reps)
    out.append({"workload": "rerank", "variant": "f1_stage", "ms": round(ms_f1, 3),
                "f1_share_of_call_with_ratings": ms_f1 / (ms_f1 + ms),
                "gathered_TB_per_s": pairs * (ka + kt) * 4 / (ms_f1 * 1e-3) / 1e12})
    for o in out:
        o.update({"users": U, "items": I, "list_len": L, "distinct_items_drawn": distinct, "ka": ka, "kt": kt, "top_k": k})
    return out


def reference_models(U, I, ka, kt, seed=0):
    """A HybridRecommendationSystem over synthetic factors (no training): ALS rank ka, tower width kt."""
    import pandas as pd
    from hybrid_als_twotower_recommender_b200.als_model import ALSFactors
    rng = np.random.default_rng(seed)
    als = pkg.ALSModel(rank=ka)
    als.model = ALSFactors(ka, np.arange(U), np.arange(I), torch.randn(U, ka, device="cuda") * ka ** -0.5,
                           torch.randn(I, ka, device="cuda"), torch.ones(U, dtype=torch.bool, device="cuda"),
                           torch.ones(I, dtype=torch.bool, device="cuda"))
    tt = pkg.TwoTowerModel(U, I, 20, 10, embedding_size=kt)
    tt.build_model(seed=seed)
    items = pd.DataFrame({"itemId": np.arange(I), "manufacturer_id": rng.integers(0, 20, I),
                          "category_id": rng.integers(0, 10, I), "price": rng.uniform(2, 200, I),
                          "average_review_rating": rng.uniform(1, 5, I)})
    tt.scaler.fit(items[["price", "average_review_rating"]])
    hrs = pkg.HybridRecommendationSystem()
    hrs.als_model, hrs.twotower_model, hrs.models_loaded = als, tt, True
    return hrs, items


def reference(reps):
    U, I, ka, kt, k = 10_000, 9_964, 10, 50, 5
    hrs, items = reference_models(U, I, ka, kt)
    m = hrs.als_model.model
    Ua, Ia = m.user_factors, m.item_factors
    Ut, It = hrs.twotower_model.user_vectors(np.arange(U)), hrs.twotower_model.item_vectors(items)
    rowptr, cand = scoring.candidate_lists(None, np.arange(I), U, "cuda")
    ms_l = timed(lambda: scoring.blend_topk_lists(Ua, Ia, Ut, It, rowptr, cand, k, w_als=0.2, w_tt=0.8), reps)
    sc = scoring.HybridScorer(Ua, Ia, Ut, It)
    ms_s = timed(lambda: sc.recommend(k, 0.2, 0.8), reps)
    pairs = U * I
    return [{"workload": "reference", "variant": "lists", **rates(ms_l, pairs, ka, kt)},
            {"workload": "reference", "variant": "shared_candidates_recommend", **rates(ms_s, pairs, ka, kt)},
            {"workload": "reference", "variant": "ratio_lists_over_shared", "ratio": ms_l / ms_s,
             "users": U, "items": I, "ka": ka, "kt": kt, "top_k": k}]


def loop(reps):
    import contextlib
    import io
    U, I, ka, kt, k, S = 10_000, 9_964, 10, 50, 5, 200
    hrs, items = reference_models(U, I, ka, kt)
    rng = np.random.default_rng(1)
    sample = [int(x) for x in rng.choice(U, S, replace=False)]
    actual = [{int(x): 5.0 for x in rng.choice(I, 10, replace=False)} if j % 4 == 0 else None for j in range(S)]

    def run_loop():
        with contextlib.redirect_stdout(io.StringIO()):
            for u, a in zip(sample, actual):
                hrs.get_hybrid_recommendations(u, items, a, k)
        torch.cuda.synchronize()

    def wall(fn):
        fn()
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(ts))
    ms_loop = wall(run_loop)
    ms_b200 = wall(lambda: hrs.get_hybrid_recommendations_batch(sample, items, None, actual, k, as_arrays=True))
    users = list(range(U))
    act_all = [{int(x): 5.0 for x in rng.choice(I, 10, replace=False)} if j % 4 == 0 else None for j in range(U)]
    ms_all = wall(lambda: hrs.get_hybrid_recommendations_batch(users, items, None, act_all, k, as_arrays=True))
    return [{"workload": "loop", "variant": "per_user_loop_SAMPLE", "users": S, "ms": round(ms_loop, 1),
             "ms_per_user": ms_loop / S},
            {"workload": "loop", "variant": "batch_api_same_sample", "users": S, "ms": round(ms_b200, 1),
             "ms_per_user": ms_b200 / S},
            {"workload": "loop", "variant": "batch_api_all_users", "users": U, "ms": round(ms_all, 1),
             "ms_per_user": ms_all / U, "note": "end to end, host joins and copies included; 1 in 4 users rated"}]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    ap.add_argument("--only", choices=["rerank", "reference", "loop"])
    a = ap.parse_args()
    nat.require_cuda()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    res = [info]
    for name, fn in (("rerank", rerank), ("reference", reference), ("loop", loop)):
        if a.only and a.only != name:
            continue
        for r in fn(a.reps):
            print(json.dumps(r), flush=True)
            res.append(r)
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
