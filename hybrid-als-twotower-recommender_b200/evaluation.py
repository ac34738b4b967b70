"""`compute_f1_score` under the module name src/hybrid_system.py:15 imports it from (the
reference's evaluation.py does not define it; the only definitions are als_model.py:171-177
and the identical two_tower_model.py:238-245).  The rest of the reference's evaluation.py
(RecommenderEvaluator, plots) is out of scope (SURVEY.md 2.1 #4)."""
from .als_model import compute_f1_score  # noqa: F401


def f1_at_k_batch(pred_idx, actual_lists, k=10):
    """compute_f1_score (src/als_model.py:171-177) for many users in one launch (hals_f1_at_k).

    pred_idx: int32 device tensor [U, >=k] of score-sorted item ROW indices (-1 = no entry), e.g. from
    HybridScorer.recommend; actual_lists: per user, the row indices of the items the user rated.
    Returns a float32 device tensor [U]."""
    import numpy as np
    import torch
    from . import _native as nat
    U = int(pred_idx.shape[0])
    lens = np.fromiter((len(a) for a in actual_lists), dtype=np.int64, count=U)
    rowptr = np.zeros(U + 1, np.int64)
    np.cumsum(lens, out=rowptr[1:])
    flat = np.concatenate([np.sort(np.asarray(a, dtype=np.int32)) for a in actual_lists]) if rowptr[-1] else np.zeros(1, np.int32)
    dev = pred_idx.device
    rp, it = torch.from_numpy(rowptr).to(dev), torch.from_numpy(np.ascontiguousarray(flat, dtype=np.int32)).to(dev)
    pred_idx = pred_idx.contiguous()
    out = torch.empty(U, dtype=torch.float32, device=dev)
    nat.check(nat.lib().hals_f1_at_k(nat.ptr(pred_idx), pred_idx.stride(0), int(k), nat.ptr(rp), nat.ptr(it), U,
                                     nat.ptr(out), None, nat.current_stream()), "hals_f1_at_k")
    return out


RANKING_METRICS = ("precisionAtK", "recallAtK", "ndcgAtK", "meanAveragePrecisionAtK", "meanAveragePrecision")


def ranking_metrics_batch(pred_idx, labels, k):
    """Spark's RankingMetrics of every row in one launch (hals_ranking_metrics); the columns are RANKING_METRICS.

    pred_idx: int32 device tensor [n, >=k] of ranked ids, each list cut at its first negative entry (the -1 padding of
    the top-k kernels) and never repeating an id; labels: device CSR (rowptr int64 [n+1], items int32) of each row's
    relevant ids, ascending within a row, repeats allowed (scoring.label_lists_by_id builds it from raw id pairs).
    Returns a float64 device tensor [n, 5]."""
    import torch
    from . import _native as nat
    rowptr, items = labels
    n = int(pred_idx.shape[0])
    if pred_idx.dtype != torch.int32 or pred_idx.dim() != 2 or not 1 <= int(k) <= pred_idx.shape[1]:
        raise ValueError("pred_idx must be an int32 [n, >= k] tensor and k >= 1")
    if rowptr.dtype != torch.int64 or items.dtype != torch.int32 or rowptr.numel() != n + 1:
        raise ValueError("labels must be (rowptr int64 [n+1], items int32)")
    dev = pred_idx.device
    if rowptr.device != dev or items.device != dev:
        raise ValueError("pred_idx and labels must live on the same device")
    out = torch.empty((n, 5), dtype=torch.float64, device=dev)
    if n == 0:
        return out
    if pred_idx.stride(1) != 1:
        pred_idx = pred_idx.contiguous()
    rowptr = rowptr.contiguous()
    items = items.contiguous() if items.numel() else torch.zeros(1, dtype=torch.int32, device=dev)  # a valid pointer
    nat.check(nat.lib().hals_ranking_metrics(nat.ptr(pred_idx), pred_idx.stride(0), int(k), n, nat.ptr(rowptr),
                                             nat.ptr(items), nat.ptr(out), nat.current_stream()),
              "hals_ranking_metrics")
    return out
