"""numpy restatement of Spark 3.x RankingMetrics (countRelevantItemRatio, averagePrecision, ndcgAt; binary relevance),
the oracle of hals_ranking_metrics / ALSModel.evaluate_ranking.  Written loop by loop after Spark's Scala, one row at a
time; test_als_evaluate_cpu.py checks it against the values Spark's RankingMetricsSuite asserts."""
import math

import numpy as np


def row_metrics(pred, labels, k):
    """(precision@k, recall@k, NDCG@k, AP@k, AP) of one ranked list against one label collection.  `pred` is cut at its
    first negative entry (the -1 padding of a top-k list); `labels` may repeat (Spark builds lab.toSet)."""
    pred = [int(x) for x in pred]
    if any(x < 0 for x in pred):
        pred = pred[:next(i for i, x in enumerate(pred) if x < 0)]
    lab = set(int(x) for x in labels)
    if not lab:
        return (0.0, 0.0, 0.0, 0.0, 0.0)
    # countRelevantItemRatio(pred, lab, k, k) and (..., k, lab.size)
    n = min(len(pred), k)
    count = sum(1 for i in range(n) if pred[i] in lab)
    precision, recall = count / k, count / len(lab)
    # ndcgAt(k), binary relevance: Spark's natural log cancels in the ratio, log2 here as in the kernel
    n = min(max(len(pred), len(lab)), k)
    dcg = max_dcg = 0.0
    for i in range(n):
        gain = 1.0 / math.log2(i + 2)
        if i < len(pred) and pred[i] in lab:
            dcg += gain
        if i < len(lab):
            max_dcg += gain
    ndcg = dcg / max_dcg
    # averagePrecision(k) and meanAveragePrecision: the same sum over the (at most k long) list
    hits, prec_sum = 0, 0.0
    for i in range(min(len(pred), k)):
        if pred[i] in lab:
            hits += 1
            prec_sum += hits / (i + 1)
    return (precision, recall, ndcg, prec_sum / min(len(lab), k), prec_sum / len(lab))


def metrics(preds, labels, k):
    """float64 [n, 5], one row_metrics per (list, labels) pair."""
    return np.array([row_metrics(p, l, k) for p, l in zip(preds, labels)], np.float64).reshape(-1, 5)
