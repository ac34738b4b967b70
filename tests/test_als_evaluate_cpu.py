"""CPU: the ranking-metrics oracle against the values of Spark's RankingMetricsSuite, and the argument checks of
hals_ranking_metrics, ALSModel.transform / evaluate_regression / evaluate_ranking, which all fail before any CUDA call
(no GPU is needed)."""
import numpy as np
import pandas as pd
import pytest

import hybrid_als_twotower_recommender_b200 as pkg
from hybrid_als_twotower_recommender_b200 import _native as nat
from tests import ranking_oracle

HALS_ERR_INVALID = 1

# RankingMetricsSuite: three ranked lists, their relevant items (the last row has none)
SUITE_PRED = [[1, 6, 2, 7, 8, 3, 9, 10, 4, 5], [4, 1, 5, 6, 2, 7, 3, 8, 9, 10], [1, 2, 3, 4, 5]]
SUITE_LABELS = [[1, 2, 3, 4, 5], [1, 2, 3], []]
PRECISION, RECALL, NDCG, MAP_AT_K, MAP = range(5)


def _mean(k):
    return ranking_oracle.metrics(SUITE_PRED, SUITE_LABELS, k).mean(0)


@pytest.mark.parametrize("k,col,want", [
    (1, PRECISION, 1 / 3), (2, PRECISION, 1 / 3), (3, PRECISION, 1 / 3), (4, PRECISION, 0.75 / 3),
    (5, PRECISION, 0.8 / 3), (10, PRECISION, 0.8 / 3), (15, PRECISION, 8 / 45),
    (1, RECALL, 1 / 15), (2, RECALL, 8 / 45),
    (1, MAP_AT_K, 1 / 3), (2, MAP_AT_K, 0.25),
    (3, NDCG, 1 / 3), (5, NDCG, 0.328788), (10, NDCG, 0.487913),
])
def test_oracle_reproduces_spark_ranking_metrics_suite(k, col, want):
    assert abs(_mean(k)[col] - want) < 1e-6


def test_oracle_map_and_ndcg_beyond_the_list():
    # meanAveragePrecision of the suite: AP over each whole list (every list here is at most 10 long)
    assert abs(_mean(10)[MAP] - 0.355026) < 1e-6
    assert _mean(15)[NDCG] == _mean(10)[NDCG]


def test_oracle_cuts_a_list_at_its_first_negative_entry_and_counts_repeated_labels_once():
    a = ranking_oracle.row_metrics([3, 1, -1, 2], [1, 1, 2, 2, 9], 4)
    b = ranking_oracle.row_metrics([3, 1], [1, 2, 9], 4)
    assert a == b and a[PRECISION] == 1 / 4 and a[RECALL] == 1 / 3


def _call(pred=True, rowptr=True, items=True, out=True, k=4, stride=4, n=2):
    """hals_ranking_metrics on host buffers (never dereferenced: every call here fails its argument checks)."""
    p, rp = np.zeros(8, np.int32), np.zeros(3, np.int64)
    it, o = np.zeros(1, np.int32), np.zeros(10, np.float64)
    return nat.lib().hals_ranking_metrics(nat.ptr(p) if pred else None, stride, k, n, nat.ptr(rp) if rowptr else None,
                                          nat.ptr(it) if items else None, nat.ptr(o) if out else None, None)


@pytest.mark.parametrize("kwargs,msg", [
    ({"pred": False}, b"pred_idx is null"), ({"rowptr": False}, b"label_rowptr is null"),
    ({"items": False}, b"label_items is null"), ({"out": False}, b"out is null"),
    ({"k": 0}, b"k must be >= 1"), ({"k": -3, "stride": 4}, b"k must be >= 1"),
    ({"k": 5, "stride": 4}, b"pred_stride must be >= k"), ({"n": -1}, b"n_rows must be >= 0"),
])
def test_ranking_metrics_rejects_a_bad_argument(kwargs, msg):
    assert _call(**kwargs) == HALS_ERR_INVALID
    err = nat.lib().hals_last_error()
    assert b"hals_ranking_metrics: " + msg in err, err


@pytest.mark.parametrize("k", [0, 257, -3, 2.0, True, "10"])
def test_evaluate_ranking_rejects_a_bad_count(k):
    with pytest.raises(ValueError, match=r"int in \[1, 256\]"):
        pkg.ALSModel().evaluate_ranking(pd.DataFrame({"userId": [1], "itemId": [2]}), k)


def test_evaluate_ranking_without_a_model_raises():
    with pytest.raises(ValueError, match="no trained or loaded model"):
        pkg.ALSModel().evaluate_ranking(pd.DataFrame({"userId": [1], "itemId": [2]}), 10)


@pytest.mark.parametrize("strategy", ["skip", "", None, 0])
def test_transform_rejects_an_unknown_cold_start_strategy(strategy):
    m = pkg.ALSModel(cold_start_strategy=strategy)          # construction accepts anything, as before
    frame = pd.DataFrame({"userId": [1], "itemId": [2], "average_review_rating": [3.0]})
    with pytest.raises(ValueError, match="cold_start_strategy must be 'drop' or 'nan'"):
        m.transform(frame)
    with pytest.raises(ValueError, match="cold_start_strategy must be 'drop' or 'nan'"):
        m.evaluate_regression(frame)


@pytest.mark.parametrize("metric", ["RMSE", "var", "", None])
def test_evaluate_regression_rejects_an_unknown_metric(metric):
    frame = pd.DataFrame({"userId": [1], "itemId": [2], "average_review_rating": [3.0]})
    with pytest.raises(ValueError, match="metric_name must be one of"):
        pkg.ALSModel().evaluate_regression(frame, metric)


def test_transform_without_a_model_raises():
    with pytest.raises(ValueError, match="no trained or loaded model"):
        pkg.ALSModel().transform(pd.DataFrame({"userId": [1], "itemId": [2]}))
