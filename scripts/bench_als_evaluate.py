"""Ranking evaluation of an ALS model on the device (ALSModel.evaluate_ranking) against the top-k pass it is built on
(ALSModel.recommend_for_all_users(k, exclude=..., as_arrays=True)), on the same inputs.

Every user has held-out items (the labels) and training pairs (the exclusions), so both calls rank the same users with
the same exclusions; evaluate_ranking adds the label CSR build (scoring.label_lists_by_id), one hals_ranking_metrics
launch per slab and one reduction, and brings back five numbers instead of the lists.  Also timed on their own: the
label CSR build (device work and the host syncs its sizes need) and the hals_ranking_metrics kernel over all users'
lists (already on the device), as a CUDA graph of KERNEL_LAUNCHES raw launches so that the host cost of issuing each
call does not count.
Agreement: per-row device metrics against the numpy restatement of Spark's RankingMetrics (tests/ranking_oracle.py) on
the GPU's own lists, for a sample of 10,000 users.
Shapes: MovieLens-20M (138,493 users x 26,744 items, rank 64, k = 10 and 100, ~20 M training pairs excluded, ~10
held-out items per user) and the per-GPU config-5 shape (1,000,000 users x 1,250,000 items, rank 128, k = 100, 10
training pairs excluded and 10 held-out items per user).  Factors are seeded N(0, 1/rank) for the users and N(0, 1) for
the items; id pairs are drawn from a seeded generator.
Timed with CUDA events: 1 warm-up, median of --reps (>= 5) repetitions, the two calls alternating within a repetition.
Prints one JSON line per (shape, k) and the GPU name and power limit, read in the same run; --out also writes them.
Usage: python scripts/bench_als_evaluate.py [--reps 5] [--out FILE] [--only ml20m|c5]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pandas as pd
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hybrid_als_twotower_recommender_b200 as pkg  # noqa: E402
from hybrid_als_twotower_recommender_b200 import _native as nat  # noqa: E402
from hybrid_als_twotower_recommender_b200.als_model import ALSFactors  # noqa: E402
from hybrid_als_twotower_recommender_b200.evaluation import ranking_metrics_batch  # noqa: E402
from hybrid_als_twotower_recommender_b200.scoring import label_lists_by_id  # noqa: E402
from tests import ranking_oracle  # noqa: E402

SAMPLE = 10_000
KERNEL_LAUNCHES = 20           # hals_ranking_metrics launches per graph replay (the time reported is per launch)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": line}


def pairs(rng, n_users, n_items, per_user):
    """per_user pairs of every user on average (1 + Poisson counts: every user has one), items uniform."""
    counts = 1 + rng.poisson(per_user - 1, n_users)
    users = np.repeat(np.arange(n_users, dtype=np.int64), counts)
    return pd.DataFrame({"userId": users, "itemId": rng.integers(0, n_items, len(users), dtype=np.int64)})


def timed(fn, n=1):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def metrics_graph(idx, labels, k, n):
    """A CUDA graph of n raw hals_ranking_metrics launches over every row of idx: replaying it times the kernel alone,
    without the Python checks, the output allocation and the ctypes call of ranking_metrics_batch."""
    rowptr, items = labels
    out = torch.empty((idx.shape[0], 5), dtype=torch.float64, device=idx.device)
    lib = nat.lib()

    def launch():
        nat.check(lib.hals_ranking_metrics(nat.ptr(idx), idx.stride(0), k, idx.shape[0], nat.ptr(rowptr),
                                           nat.ptr(items), nat.ptr(out), nat.current_stream()), "hals_ranking_metrics")

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        launch()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(n):
            launch()
    return graph, out


def stats(t):
    t = sorted(t)
    return {"ms_median": t[len(t) // 2], "ms_min": t[0], "ms_max": t[-1]}


def measure(name, als, train, test, k, reps, warmup, info):
    m = als.model
    n_u, n_i, rank = len(m.user_ids), len(m.item_ids), m.rank
    variants = {"evaluate_ranking": lambda: als.evaluate_ranking(test, k, exclude=train),
                "recommend_for_all_users": lambda: als.recommend_for_all_users(k, exclude=train, as_arrays=True)}
    times = {v: [] for v in variants}
    for rep in range(warmup + reps):
        for v, fn in variants.items():
            t = timed(fn)
            if rep >= warmup:
                times[v].append(t)
    result = als.evaluate_ranking(test, k, exclude=train)

    # the pieces on their own: the label CSR and one metrics launch over every user's lists
    dev = m.item_factors.device
    query_ids, cand_ids, slabs = als._topk_slabs(True, test["userId"].values, k, train, 65536)
    q_d, c_d = torch.from_numpy(query_ids).to(dev), torch.from_numpy(np.asarray(cand_ids, np.int64)).to(dev)
    tu, ti = (torch.from_numpy(np.ascontiguousarray(test[c].values)).to(dev) for c in ("userId", "itemId"))
    idx = torch.cat([s[2] for s in slabs])
    labels = label_lists_by_id(q_d, c_d, tu, ti)
    graph, graph_out = metrics_graph(idx, labels, k, KERNEL_LAUNCHES)
    t_csr, t_kernel = [], []
    for rep in range(warmup + reps):
        t1 = timed(lambda: label_lists_by_id(q_d, c_d, tu, ti))
        t2 = timed(graph.replay) / KERNEL_LAUNCHES
        if rep >= warmup:
            t_csr.append(t1)
            t_kernel.append(t2)

    # agreement on a sample of users: device rows against the numpy oracle on the same (raw-id) lists
    rng = np.random.default_rng(7)
    rows = np.sort(rng.choice(len(query_ids), min(SAMPLE, len(query_ids)), replace=False))
    full = ranking_metrics_batch(idx, labels, k)
    assert torch.equal(full, graph_out)                  # the graph computed what the Python entry point computes
    got = full[torch.from_numpy(rows).to(dev)].cpu().numpy()
    lists = idx[torch.from_numpy(rows).to(dev)].cpu().numpy()
    raw = np.where(lists >= 0, np.asarray(cand_ids)[np.maximum(lists, 0)], -1)
    sample = test[test["userId"].isin(query_ids[rows])]
    lab = sample.groupby("userId")["itemId"].apply(list).to_dict()
    want = ranking_oracle.metrics(raw, [lab[u] for u in query_ids[rows]], k)
    rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    rel[(got == 0) & (want == 0)] = 0.0

    res = {"shape": name, "n_users": n_u, "n_items": n_i, "rank": rank, "k": k, "train_pairs_excluded": len(train),
           "test_pairs": len(test), "reps": reps, "warmup": warmup, **info}
    for v in variants:
        res[v] = stats(times[v])
    res["evaluate_over_recommend"] = res["evaluate_ranking"]["ms_median"] / res["recommend_for_all_users"]["ms_median"]
    res["label_csr_build"] = stats(t_csr)
    res["hals_ranking_metrics_launch"] = stats(t_kernel)
    res["kernel_over_recommend"] = (res["hals_ranking_metrics_launch"]["ms_median"] /
                                    res["recommend_for_all_users"]["ms_median"])
    res["metrics"] = result
    res["agreement"] = {"rows": int(len(rows)), "max_rel_diff": float(rel.max()),
                        "rows_beyond_1e-12": int((rel > 1e-12).any(1).sum())}
    return res


def model(n_users, n_items, rank, g):
    uf = torch.randn(n_users, rank, device="cuda", generator=g) * rank ** -0.5
    itf = torch.randn(n_items, rank, device="cuda", generator=g)
    als = pkg.ALSModel(rank=rank)
    ones = torch.ones
    als.model = ALSFactors(rank, np.arange(n_users, dtype=np.int64), np.arange(n_items, dtype=np.int64), uf, itf,
                           ones(n_users, dtype=torch.bool, device="cuda"), ones(n_items, dtype=torch.bool, device="cuda"))
    return als


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
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
    rng = np.random.default_rng(1)
    if args.only in (None, "ml20m"):
        U, I, rank = 138_493, 26_744, 64
        als = model(U, I, rank, g)
        train, test = pairs(rng, U, I, 20_000_263 / U), pairs(rng, U, I, 10)
        for k in (10, 100):
            emit(measure("movielens20m", als, train, test, k, args.reps, args.warmup, info))
        del als, train, test
        torch.cuda.empty_cache()
    if args.only in (None, "c5"):
        U, I, rank = 1_000_000, 1_250_000, 128
        als = model(U, I, rank, g)
        train, test = pairs(rng, U, I, 10), pairs(rng, U, I, 10)
        emit(measure("config5_per_gpu", als, train, test, 100, args.reps, args.warmup, info))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
