"""CPU: host side of the batched per-user-list hybrid path (HybridRecommendationSystem.get_hybrid_recommendations_batch,
hals_score_blend_topk_lists) -- sticky F1 weights, candidate-list normalisation, and the C ABI's argument checks, which
all return before any CUDA call."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pandas as pd
import pytest
import torch

import hybrid_als_twotower_recommender_b200 as pkg
from hybrid_als_twotower_recommender_b200 import _native as nat
from hybrid_als_twotower_recommender_b200.scoring import candidate_lists, sticky_weights
from oracle import hybrid_oracle


def _loop_weights(actuals, preds, init):
    """The reference's loop: get_hybrid_recommendations re-evaluates the F1 pair only when actual_ratings is truthy
    (hybrid_system.py:104-105), and fusion_weights reads the sticky pair (:69)."""
    cur, out = init, []
    for act, (pa, pt) in zip(actuals, preds):
        if act:
            cur = (hybrid_oracle.compute_f1_score(act, pa), hybrid_oracle.compute_f1_score(act, pt))
        out.append(hybrid_oracle.fusion_weights(*cur))
    return np.asarray(out, np.float32), cur


@pytest.mark.parametrize("init", [(0.0, 0.0), (0.3, 0.1)])
def test_sticky_weights_match_the_reference_loop(init):
    rng = np.random.default_rng(0)
    # no ratings first, ratings, none between, an empty dict, the same user twice (rows 6 and 7), none at the end
    pattern = [None, None, "r", None, {}, "r", "r", "r", None, {}, "r", None, None]
    actuals, preds = [], []
    for p in pattern:
        items = rng.permutation(40)[:25]
        pa = {int(i): float(s) for i, s in zip(items, rng.integers(0, 4, 25))}    # coarse scores: many ties
        pt = {int(i): float(s) for i, s in zip(items, rng.normal(size=25))}
        preds.append((pa, pt))
        actuals.append({int(i): 5.0 for i in rng.choice(60, 8, replace=False)} if p == "r" else p)
    actuals[7], preds[7] = actuals[6], preds[6]
    want_w, want_last = _loop_weights(actuals, preds, init)
    rated = [j for j, a in enumerate(actuals) if a]
    fa = [hybrid_oracle.compute_f1_score(actuals[j], preds[j][0]) for j in rated]
    ft = [hybrid_oracle.compute_f1_score(actuals[j], preds[j][1]) for j in rated]
    w, last = sticky_weights(len(pattern), rated, fa, ft, init)
    assert w.dtype == np.float32 and (w == want_w).all()
    assert last == want_last


def test_sticky_weights_without_any_ratings_keep_the_current_pair():
    w, last = sticky_weights(3, [], [], [], (0.5, 0.25))
    assert (w == np.float32([0.8, 0.2])).all() and last == (0.5, 0.25)
    w, last = sticky_weights(0, [], [], [], (0.0, 0.0))
    assert w.shape == (0, 2) and last == (0.0, 0.0)


def test_candidate_lists_dedup_keeps_the_first_occurrence():
    universe = [10, 30, 20, 40]
    lists = [[20, 10, 20, 40, 10], [], [40], pd.DataFrame({"itemId": [30, 30, 10]})]
    rowptr, cand = candidate_lists(lists, universe, 4, "cpu")
    assert rowptr.tolist() == [0, 3, 3, 4, 6]
    assert cand.dtype == torch.int32 and cand.tolist() == [2, 0, 3, 3, 1, 0]


def test_candidate_lists_from_padded_arrays_and_none():
    universe = np.array([7, 5, 9])
    arr = np.array([[9, 5, -1, -1], [-1, -1, -1, -1], [5, 5, 7, 9]])
    rowptr, cand = candidate_lists(arr, universe, 3, "cpu")
    assert rowptr.tolist() == [0, 2, 2, 5] and cand.tolist() == [2, 1, 1, 0, 2]
    rowptr, cand = candidate_lists(torch.from_numpy(arr), universe, 3, "cpu")
    assert rowptr.tolist() == [0, 2, 2, 5] and cand.tolist() == [2, 1, 1, 0, 2]
    rowptr, cand = candidate_lists(None, universe, 2, "cpu")
    assert rowptr.tolist() == [0, 3, 6] and cand.tolist() == [0, 1, 2, 0, 1, 2]


def test_candidate_lists_reject_bad_input():
    with pytest.raises(ValueError, match="missing from item_features"):
        candidate_lists([[1, 2], [3]], [1, 2], 2, "cpu")
    with pytest.raises(ValueError, match="missing from item_features"):
        candidate_lists(np.array([[1, -2]]), [1, 2], 1, "cpu")
    with pytest.raises(ValueError, match="each itemId once"):
        candidate_lists([[1]], [1, 1], 1, "cpu")
    with pytest.raises(ValueError, match="lists for"):
        candidate_lists([[1]], [1], 2, "cpu")
    with pytest.raises(ValueError, match="rows for"):
        candidate_lists(np.ones((3, 2), np.int64), [1], 2, "cpu")


def test_unknown_candidate_raises_before_any_model_work():
    hrs = pkg.HybridRecommendationSystem()
    hrs.models_loaded = True
    # item_factors only names the device; a tower model of None fails on first touch
    hrs.als_model = SimpleNamespace(model=SimpleNamespace(item_factors=torch.zeros(1, 1)))
    items = pd.DataFrame({"itemId": [1, 2], "manufacturer_id": 0, "category_id": 0, "price": 1.0,
                          "average_review_rating": 3.0})
    with pytest.raises(ValueError, match="missing from item_features"):
        hrs.get_hybrid_recommendations_batch([0, 1], items, [[1], [3]])
    with pytest.raises(ValueError, match="top_k"):
        hrs.get_hybrid_recommendations_batch([0], items, top_k=0)
    with pytest.raises(ValueError, match="aligned"):
        hrs.get_hybrid_recommendations_batch([0, 1], items, actual_ratings_by_user=[None])


def _call(**kw):
    """hals_score_blend_topk_lists with valid host dummies, overridden by kw (nothing here reaches the device)."""
    buf = np.zeros(1 << 16, np.float32)
    p = nat.ptr(buf)
    a = dict(Ua=p, ua=4, Ia=p, ia=4, ka=4, Ut=p, ut=4, It=p, it=4, kt=4, n_rows=2, n_total=10, rowptr=p, cand=p,
             uk=None, ik=None, fb=None, rw=None, wa=0.8, wt=0.2, raw=0, topk=5, op=p, os=p, ws=p, wsb=1 << 40)
    a.update(kw)
    rc = nat.lib().hals_score_blend_topk_lists(a["Ua"], a["ua"], a["Ia"], a["ia"], a["ka"], a["Ut"], a["ut"], a["It"],
                                               a["it"], a["kt"], a["n_rows"], a["n_total"], a["rowptr"], a["cand"],
                                               a["uk"], a["ik"], a["fb"], a["rw"], a["wa"], a["wt"], a["raw"],
                                               a["topk"], a["op"], a["os"], a["ws"], a["wsb"], None)
    return rc, nat.lib().hals_last_error().decode()


@pytest.mark.parametrize("kw,msg", [
    (dict(topk=0), "topk"), (dict(topk=257), "topk"),
    (dict(ka=129), "ka must be"), (dict(kt=65), "ka must be"), (dict(ka=0, kt=0), "ka must be"),
    (dict(ka=-1), "ka must be"), (dict(Ia=None), "null operand"), (dict(Ut=None), "null operand"),
    (dict(n_rows=-1), "negative"), (dict(n_total=-1), "negative"), (dict(n_total=1 << 31), "int32"),
    (dict(rowptr=None), "null pointer"), (dict(op=None), "null pointer"), (dict(ws=None), "null pointer"),
    (dict(cand=None), "null pointer"), (dict(uk=ctypes.c_void_p(8)), "als_fallback"),
    (dict(ik=ctypes.c_void_p(8)), "als_fallback"),
])
def test_cabi_rejects_bad_arguments_before_cuda(kw, msg):
    rc, err = _call(**kw)
    assert rc == 1 and msg in err, (rc, err)


def test_cabi_workspace_and_empty_calls():
    L = nat.lib()
    need = int(L.hals_score_lists_workspace_bytes(10, 5))
    assert need > 0 and int(L.hals_score_lists_workspace_bytes(-1, 5)) == 0
    assert int(L.hals_score_lists_workspace_bytes(10, 0)) == 0 and int(L.hals_score_lists_workspace_bytes(10, 257)) == 0
    # lists longer than the split threshold need room for the partial extrema and lists
    assert int(L.hals_score_lists_workspace_bytes(100_000, 256)) > 8 * 100_000 + 256 * 8 * (100_000 // 8192)
    rc, err = _call(wsb=need - 1)
    assert rc == 3 and "workspace" in err
    assert _call(n_rows=0, wsb=need)[0] == 0                  # launches nothing
    assert _call(n_rows=0, n_total=0, cand=None, wsb=int(L.hals_score_lists_workspace_bytes(0, 5)))[0] == 0
    assert _call(ka=0, Ua=None, Ia=None, n_rows=0, wsb=need)[0] == 0
    assert _call(uk=ctypes.c_void_p(8), fb=ctypes.c_void_p(8), n_rows=0, wsb=need)[0] == 0
