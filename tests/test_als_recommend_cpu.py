"""CPU: hals_score_topk (the raw dot-product top-k behind ALSModel.recommend_for_*) and the ALSModel methods refuse bad
arguments before any CUDA call, so no GPU is needed."""
import numpy as np
import pandas as pd
import pytest

import hybrid_als_twotower_recommender_b200 as pkg
from hybrid_als_twotower_recommender_b200 import _native as nat

HALS_ERR_INVALID = 1


def _call(k=8, topk=10, xr=None, xi=None):
    """hals_score_topk on host buffers (never dereferenced: every call here fails its argument checks)."""
    Q, C = np.zeros((4, 128), np.float32), np.zeros((6, 128), np.float32)
    oi, os_ = np.zeros(4 * 256, np.int32), np.zeros(4 * 256, np.float32)
    ws = np.zeros(64, np.uint8)
    return nat.lib().hals_score_topk(nat.ptr(Q), 128, nat.ptr(C), 128, k, 4, 6, topk, 0, nat.ptr(xr), nat.ptr(xi),
                                     nat.ptr(oi), nat.ptr(os_), nat.ptr(ws), ws.nbytes, None)


@pytest.mark.parametrize("k", [0, 129, -1])
def test_rank_outside_1_128_is_rejected(k):
    assert _call(k=k) == HALS_ERR_INVALID
    assert b"hals_score_topk: k (the factor rank) must be in [1,128]" in nat.lib().hals_last_error()


@pytest.mark.parametrize("topk", [0, 257])
def test_topk_outside_1_256_is_rejected(topk):
    assert _call(topk=topk) == HALS_ERR_INVALID
    assert b"hals_score_topk: topk must be in [1,256]" in nat.lib().hals_last_error()


def test_exactly_one_exclusion_pointer_is_rejected():
    rowptr, items = np.zeros(5, np.int64), np.zeros(1, np.int32)
    for xr, xi in ((rowptr, None), (None, items)):
        assert _call(xr=xr, xi=xi) == HALS_ERR_INVALID
        assert b"excl_rowptr and excl_items must both be set or both NULL" in nat.lib().hals_last_error()


def test_null_operand_is_rejected():
    oi = np.zeros(40, np.int32)
    rc = nat.lib().hals_score_topk(None, 8, nat.ptr(oi), 8, 8, 4, 6, 10, 0, None, None, nat.ptr(oi), nat.ptr(oi),
                                   nat.ptr(oi), oi.nbytes, None)
    assert rc == HALS_ERR_INVALID and b"null pointer" in nat.lib().hals_last_error()


@pytest.mark.parametrize("num", [0, 257, -3, 2.0, True, "10"])
def test_recommend_rejects_a_bad_count(num):
    m = pkg.ALSModel()
    for call in (lambda: m.recommend_for_all_users(num), lambda: m.recommend_for_all_items(num),
                 lambda: m.recommend_for_user_subset(pd.DataFrame({"userId": [1]}), num),
                 lambda: m.recommend_for_item_subset(pd.DataFrame({"itemId": [1]}), num)):
        with pytest.raises(ValueError, match=r"int in \[1, 256\]"):
            call()


def test_recommend_without_a_model_raises():
    with pytest.raises(ValueError, match="no trained or loaded model"):
        pkg.ALSModel().recommend_for_all_users(10)
    with pytest.raises(ValueError, match="no trained or loaded model"):
        pkg.ALSModel().recommend_for_item_subset(pd.DataFrame({"itemId": [1]}), 256)
