"""CPU ORACLE (test infrastructure, NOT product code) -- adaptive fusion + top-k.

Restates src/hybrid_system.py:57-75 (adaptive_fusion), :108 (stable descending sort,
first top_k) and src/als_model.py:171-177 (compute_f1_score, the weight selector used at
hybrid_system.py:47-48).  PINNED: oracle/ref_loader.py loads the reference's own,
unmodified hybrid_system.py in the build container and tests/golden/make_golden.py
commits its outputs as fixtures (tests/golden/hybrid_reference_cases.json);
tests/test_oracle_golden.py checks this restatement against them.

MinMaxScaler semantics (sklearn 1.2.2 pinned, requirements.txt:3; formula unchanged in
the installed 1.9.0): scale_ = 1/(max-min) with a zero range replaced by 1,
min_ = -min*scale_, out = x*scale_ + min_  => a constant vector maps to all 0.
"""
from __future__ import annotations

import numpy as np


def minmax(x):
    x = np.asarray(x, dtype=np.float64)
    mn, mx = x.min(), x.max()
    rng = mx - mn
    scale = 1.0 / rng if rng != 0.0 else 1.0
    return x * scale + (-mn * scale)


def fusion_weights(als_f1, tt_f1):
    """hybrid_system.py:69 -- strict '>' so equal scores (both start at 0.0, :26-27)
    favour the two-tower model."""
    return (0.8, 0.2) if als_f1 > tt_f1 else (0.2, 0.8)


def adaptive_fusion_dense(als_scores, tt_scores, als_f1=0.0, tt_f1=0.0):
    """Blend two aligned score vectors (same candidate items, same order)."""
    wa, wt = fusion_weights(als_f1, tt_f1)
    return wa * minmax(als_scores) + wt * minmax(tt_scores)


def topk_desc(scores, k, ids=None):
    """sorted(reverse=True)[:k] is stable, so ties keep candidate order; with
    candidates in ascending item order that is (score desc, item asc)."""
    scores = np.asarray(scores)
    order = np.argsort(-scores, kind="stable")[:k]
    if ids is None:
        return order, scores[order]
    return np.asarray(ids)[order], scores[order]


def compute_f1_score(actual, pred, k=10):
    """als_model.py:171-177 (identical copy at two_tower_model.py:238-245)."""
    actual_items = set(actual.keys())
    ranked = sorted(pred.items(), key=lambda x: x[1], reverse=True)[:k]
    pred_items = set(item for item, _ in ranked)
    tp = len(actual_items & pred_items)
    precision = tp / k
    recall = tp / len(actual_items) if actual_items else 0
    return 2 * (precision * recall) / (precision + recall) if (precision + recall) > 0 else 0


def hybrid_topk_dense(Ua, Ia, Ut, It, w_als, w_tt, k):
    """Batched restatement: all users x all items, fp32 sequential-equivalent dots
    (fp64 accumulate, cast fp32 like Spark's / Keras' fp32 outputs), fp64 blend."""
    Sa = (Ua.astype(np.float64) @ Ia.astype(np.float64).T).astype(np.float32).astype(np.float64)
    St = (Ut.astype(np.float64) @ It.astype(np.float64).T).astype(np.float32).astype(np.float64)

    def mm(S):
        mn = S.min(axis=1, keepdims=True)
        mx = S.max(axis=1, keepdims=True)
        rng = mx - mn
        scale = np.where(rng != 0.0, 1.0 / np.where(rng != 0.0, rng, 1.0), 1.0)
        return S * scale + (-mn * scale)

    B = w_als * mm(Sa) + w_tt * mm(St)
    idx = np.argsort(-B, axis=1, kind="stable")[:, :k]
    return idx.astype(np.int32), np.take_along_axis(B, idx, axis=1)


def find_similar_items(item_features, item_id, k=3):
    """als_model.py:93-104, literally: sklearn cosine_similarity per pair, stable descending sort over the dict order,
    first k, then the > 0.5 filter."""
    from sklearn.metrics.pairwise import cosine_similarity
    try:
        target = item_features[item_id]
    except KeyError:
        return []
    sims = []
    for other_id, feats in item_features.items():
        if other_id == item_id:
            continue
        sims.append((other_id, cosine_similarity([target["features"]], [feats["features"]])[0][0]))
    return [item for item, sim in sorted(sims, key=lambda x: x[1], reverse=True)[:k] if sim > 0.5]


def fallback_rating(item_features, item_id, global_mean):
    """als_model.py:83-85: mean rating of the similar items, else the global mean."""
    similar = find_similar_items(item_features, item_id)
    return float(np.mean([item_features[s]["rating"] for s in similar])) if similar else global_mean
