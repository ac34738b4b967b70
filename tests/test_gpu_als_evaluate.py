"""GPU: Spark-style evaluation of ALSModel -- hals_ranking_metrics against the numpy restatement of Spark's
RankingMetrics (tests/ranking_oracle.py), evaluate_ranking against that oracle on the model's own lists and against a
full numpy pipeline (fp64 top-k, then the metrics), and transform / evaluate_regression against numpy."""
import numpy as np
import pandas as pd
import pytest
import torch

from tests import ranking_oracle
from tests.test_gpu_als_recommend import route, train_frame
from tests.test_gpu_scoring import dev

pytestmark = pytest.mark.gpu

NAMES = ("precisionAtK", "recallAtK", "ndcgAtK", "meanAveragePrecisionAtK", "meanAveragePrecision")


def _pkg():
    import hybrid_als_twotower_recommender_b200 as pkg
    from hybrid_als_twotower_recommender_b200 import _native, evaluation
    return pkg, _native, evaluation


# ---- hals_ranking_metrics --------------------------------------------------------------------------------------------

def kernel_case(rng, k, stride, n_rows=600, n_items=5000):
    """Ranked lists (no repeated id; random length <= k; -1 after the end, and on some rows arbitrary ids after that -1;
    arbitrary ids in the stride padding beyond k) and label lists (sorted, with repeats; empty rows; rows of more than
    1000 labels).  Lists are drawn from a small universe around the labels so that hits are common."""
    preds = rng.integers(0, n_items, (n_rows, stride)).astype(np.int32)
    labels = []
    for r in range(n_rows):
        size = (0, 0, 1, 3, 1500)[r % 5] if r < 10 else int(rng.integers(0, 3 * k + 4))
        if r % 97 == 13:
            size = 1200
        lab = np.sort(rng.integers(0, n_items, size)).astype(np.int32)
        lab = np.sort(np.concatenate([lab, lab[: size // 4]]))           # repeats
        labels.append(lab)
        universe = np.unique(np.concatenate([lab, rng.integers(0, n_items, 2 * k + 8)]))
        n = min(k, len(universe)) if r % 3 else int(rng.integers(0, k + 1))
        preds[r, :n] = rng.permutation(universe)[:n]
        if n < k:
            preds[r, n] = -1
            if r % 2:
                preds[r, n + 1:k] = -1
    return preds, labels


def csr(labels):
    lens = np.array([len(x) for x in labels], np.int64)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    items = np.concatenate(labels).astype(np.int32) if rowptr[-1] else np.zeros(0, np.int32)
    return dev(rowptr), dev(items)


@pytest.mark.parametrize("k", [1, 10, 31, 32, 33, 100, 256])
def test_kernel_matches_the_oracle(k):
    _, _, evaluation = _pkg()
    rng = np.random.default_rng(k)
    stride = k + 7
    preds, labels = kernel_case(rng, k, stride)
    want = ranking_oracle.metrics([p[:k] for p in preds], labels, k)
    assert (want[:, 0] > 0).sum() > 50 and (want[:, 0] == 0).any()          # the case has hits and misses
    P, L = dev(preds), csr(labels)
    got = evaluation.ranking_metrics_batch(P, L, k)
    assert got.shape == (len(preds), 5) and got.dtype == torch.float64
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-12, atol=0)
    again = evaluation.ranking_metrics_batch(P, L, k)
    assert torch.equal(got.view(torch.int64), again.view(torch.int64))


def test_kernel_reads_row_slices_of_a_wider_label_csr_and_no_rows():
    """Slab by slab, evaluate_ranking passes rowptr[u0:u1+1] with the full items array: offsets are absolute."""
    _, _, evaluation = _pkg()
    rng = np.random.default_rng(5)
    preds, labels = kernel_case(rng, 20, 20, n_rows=300)
    rowptr, items = csr(labels)
    full = evaluation.ranking_metrics_batch(dev(preds), (rowptr, items), 20)
    part = evaluation.ranking_metrics_batch(dev(preds[100:230]), (rowptr[100:231], items), 20)
    assert torch.equal(part, full[100:230])
    empty = evaluation.ranking_metrics_batch(dev(preds[:0]), (rowptr[:1], items), 20)
    assert empty.shape == (0, 5)


# ---- ALSModel.evaluate_ranking -----------------------------------------------------------------------------------------

def own_lists_oracle(als, test, k, exclude=None):
    """The oracle applied to the lists recommend_for_user_subset returns: (means [5], numUsers, numColdUsers)."""
    q, rec, _ = als.recommend_for_user_subset(test, k, exclude=exclude, as_arrays=True)
    lab = test.groupby("userId")["itemId"].apply(list).to_dict()
    per = ranking_oracle.metrics(rec, [lab[u] for u in q], k)
    return per.mean(0), len(q), test["userId"].nunique() - len(q)


def check_ranking(got, want):
    means, n_users, n_cold = want
    assert got["numUsers"] == n_users and got["numColdUsers"] == n_cold
    np.testing.assert_allclose([got[n] for n in NAMES], means, rtol=1e-12, atol=0)


def test_evaluate_ranking_of_a_trained_model_against_its_own_lists():
    pkg, _, _ = _pkg()
    rng = np.random.default_rng(31)
    df = train_frame(rng)
    als = pkg.ALSModel(rank=10, max_iter=5, reg_param=0.1)
    assert als.train(df) is True
    m = als.model
    users, items = list(m.user_ids), list(m.item_ids)
    n = 700
    test = pd.DataFrame({"userId": np.concatenate([rng.choice(users, n), [-4, 10 ** 6, 10 ** 6 + 3]]),  # 3 unknown users
                         "itemId": np.concatenate([rng.choice(items, n), [items[0], 1, 77_777]])})
    unknown_items = pd.DataFrame({"userId": [users[1], users[2], users[2]], "itemId": [1, 77_777, 10 ** 9]})
    test = pd.concat([test, unknown_items], ignore_index=True)
    # a user whose relevant items are exactly the ones excluded (rated in training)
    seen = df[df["userId"] == users[0]]["itemId"].unique()
    test = pd.concat([test[test["userId"] != users[0]], pd.DataFrame({"userId": users[0], "itemId": seen})])
    train = df[["userId", "itemId"]]
    for k in (1, 10, 100):
        for exclude in (None, train):
            want = own_lists_oracle(als, test, k, exclude)
            assert want[2] == 3
            check_ranking(als.evaluate_ranking(test, k, exclude=exclude), want)
    # with the training pairs excluded, the user whose relevant items were all rated scores 0 everywhere
    one = als.evaluate_ranking(test[test["userId"] == users[0]], 10, exclude=train)
    assert one["numUsers"] == 1 and all(one[n] == 0.0 for n in NAMES)
    plain = als.evaluate_ranking(test[test["userId"] == users[0]], 100)
    assert plain["recallAtK"] > 0


def integer_model(pkg, rng, U, I, rank, absent=40):
    """ALSFactors with integer factors in [-3, 3]: every score is an exact integer on both routes (fp32 and bf16 hold
    the operands and the sums exactly), so the top-k lists are the fp64 ones with ties cut by ascending raw id."""
    from hybrid_als_twotower_recommender_b200.als_model import ALSFactors
    uid = np.sort(rng.choice(10 ** 7, U, replace=False)).astype(np.int64)
    iid = np.sort(rng.choice(10 ** 7, I, replace=False)).astype(np.int64)
    up, ip = np.ones(U, bool), np.ones(I, bool)
    up[rng.choice(U, absent, replace=False)] = False
    ip[rng.choice(I, absent, replace=False)] = False
    uf = rng.integers(-3, 4, (U, rank)).astype(np.float32)
    itf = rng.integers(-3, 4, (I, rank)).astype(np.float32)
    als = pkg.ALSModel(rank=rank)
    als.model = ALSFactors(rank, uid, iid, dev(uf), dev(itf), dev(up), dev(ip))
    return als, uid, iid, up, ip, uf, itf


def frames(rng, uid, iid, n_test, n_excl):
    """Test pairs (every user, plus two unknown users and a few unknown items) and exclusion pairs."""
    users = np.concatenate([uid, uid[rng.integers(0, len(uid), n_test - len(uid))], [-1, 10 ** 8]])
    items = iid[rng.integers(0, len(iid), len(users))]
    items[rng.choice(len(items), 30, replace=False)] = 10 ** 8 + rng.integers(0, 5, 30)
    test = pd.DataFrame({"userId": users, "itemId": items})
    excl = pd.DataFrame({"userId": uid[rng.integers(0, len(uid), n_excl)],
                         "itemId": iid[rng.integers(0, len(iid), n_excl)]})
    # some relevant items are excluded too
    pick = rng.choice(len(test), len(test) // 10, replace=False)
    return test, pd.concat([excl, test.iloc[pick]], ignore_index=True)


def numpy_pipeline(uid, iid, up, ip, uf, itf, test, exclude, k):
    """recommendForAllUsers(k) in fp64 (ties by ascending raw id), joined with the test pairs, then the oracle."""
    cand, C = iid[ip], itf[ip].astype(np.float64)
    lab = test.groupby("userId")["itemId"].apply(list).to_dict()
    ex = exclude.groupby("userId")["itemId"].apply(set).to_dict()
    warm = set(uid[up].tolist())
    q = [u for u in np.unique(test["userId"]) if u in warm]
    row = {u: r for r, u in enumerate(uid)}
    preds = []
    for u in q:
        s = C @ uf[row[u]].astype(np.float64)
        ranked = cand[np.lexsort((np.arange(len(cand)), -s))]
        keep = ranked[~np.isin(ranked, list(ex.get(u, ())))][:k].tolist()
        preds.append(keep + [-1] * (k - len(keep)))
    per = ranking_oracle.metrics(preds, [lab[u] for u in q], k)
    return per.mean(0), len(q), test["userId"].nunique() - len(q)


@pytest.mark.parametrize("want_route,U,I,rank,k", [("simt", 300, 1000, 16, 10), ("tc", 3072, 4096 + 40, 64, 100)])
def test_evaluate_ranking_equals_the_numpy_pipeline(want_route, U, I, rank, k):
    pkg, nat, _ = _pkg()
    rng = np.random.default_rng(U + k)
    als, uid, iid, up, ip, uf, itf = integer_model(pkg, rng, U, I, rank)
    test, excl = frames(rng, uid, iid, 4 * U, 20 * U)
    assert route(nat, int(up.sum()), int(ip.sum()), rank, k) == want_route
    for exclude in (None, excl):
        want = numpy_pipeline(uid, iid, up, ip, uf, itf, test, excl if exclude is not None else excl[:0], k)
        assert want[2] == 40 + 2                                   # absent users and unknown users
        check_ranking(als.evaluate_ranking(test, k, exclude=exclude), want)


@pytest.mark.parametrize("U,I,rank,k,slabs", [(300, 1000, 16, 10, (65536, 100, 7)),
                                              (3072 + 40, 4096 + 40, 64, 100, (65536, 1536, 1024))])
def test_evaluate_ranking_does_not_depend_on_the_slab_size(U, I, rank, k, slabs):
    pkg, _, _ = _pkg()
    rng = np.random.default_rng(U)
    als, uid, iid, *_ = integer_model(pkg, rng, U, I, rank)
    test, excl = frames(rng, uid, iid, 3 * U, 10 * U)
    got = [als._evaluate_ranking(test, k, excl, slab=s) for s in slabs]
    assert got[0]["numUsers"] > max(slabs[1:])                     # every other slab size splits the users
    for g in got[1:]:
        assert g == got[0]


# ---- ALSModel.transform / evaluate_regression --------------------------------------------------------------------------

def regression_case(pkg, rng):
    als, uid, iid, up, ip, uf, itf = integer_model(pkg, rng, 200, 300, 16, absent=10)
    als.model.user_factors = dev(rng.normal(0, 0.5, (200, 16)).astype(np.float32))
    als.model.item_factors = dev(rng.normal(0, 0.5, (300, 16)).astype(np.float32))
    n = 900
    users = rng.choice(np.concatenate([uid, [-1, 5 * 10 ** 7]]), n)
    items = rng.choice(np.concatenate([iid, [3, 6 * 10 ** 7]]), n)
    test = pd.DataFrame({"userId": users, "itemId": items, "average_review_rating": rng.integers(1, 6, n) * 1.0,
                         "other": np.arange(n)}, index=np.arange(n) * 3 + 5)
    return als, test


def expected_predictions(als, test):
    m = als.model
    X, Y = m.user_factors.cpu().numpy().astype(np.float64), m.item_factors.cpu().numpy().astype(np.float64)
    up, ip = m.user_present.cpu().numpy(), m.item_present.cpu().numpy()
    u = np.searchsorted(m.user_ids, test["userId"].values).clip(0, len(m.user_ids) - 1)
    i = np.searchsorted(m.item_ids, test["itemId"].values).clip(0, len(m.item_ids) - 1)
    cold = ((m.user_ids[u] != test["userId"].values) | (m.item_ids[i] != test["itemId"].values) | ~up[u] | ~ip[i])
    exact = (X[u] * Y[i]).sum(1)
    scale = (np.abs(X[u]) * np.abs(Y[i])).sum(1)
    return np.where(cold, np.nan, exact), scale, cold


def test_transform_under_both_cold_start_strategies():
    pkg, _, _ = _pkg()
    als, test = regression_case(pkg, np.random.default_rng(41))
    want, scale, cold = expected_predictions(als, test)
    assert 20 < cold.sum() < len(test) // 2
    als.cold_start_strategy = "nan"
    out = als.transform(test)
    assert list(out.index) == list(test.index) and out["prediction"].dtype == np.float32
    assert out.drop(columns="prediction").equals(test)
    p = out["prediction"].values.astype(np.float64)
    assert (np.isnan(p) == cold).all()
    assert (np.abs(p - want)[~cold] <= 1e-6 * scale[~cold]).all()
    als.cold_start_strategy = "drop"
    dropped = als.transform(test)
    assert list(dropped.index) == list(test.index[~cold])
    assert np.array_equal(dropped["prediction"].values, out["prediction"].values[~cold])
    assert "prediction" not in test.columns


def test_evaluate_regression_matches_numpy():
    pkg, _, _ = _pkg()
    als, test = regression_case(pkg, np.random.default_rng(42))
    out = als.transform(test)                                       # "drop", the default
    y, p = out["average_review_rating"].values.astype(np.float64), out["prediction"].values.astype(np.float64)
    err = y - p
    want = {"rmse": np.sqrt(np.mean(err ** 2)), "mse": np.mean(err ** 2), "mae": np.mean(np.abs(err)),
            "r2": 1.0 - np.sum(err ** 2) / np.sum((y - y.mean()) ** 2)}
    for name, w in want.items():
        assert abs(als.evaluate_regression(test, name) - w) <= 1e-12 * abs(w), name
    assert als.evaluate_regression(test) == als.evaluate_regression(test, "rmse")
    # "nan" keeps the cold rows, and a NaN prediction makes every metric NaN (Spark's evaluator does the same)
    als.cold_start_strategy = "nan"
    assert all(np.isnan(als.evaluate_regression(test, name)) for name in want)
    warm = test.loc[out.index]
    assert als.evaluate_regression(warm, "mae") == pytest.approx(want["mae"], rel=1e-12)
    # nothing left after dropping: NaN
    als.cold_start_strategy = "drop"
    cold = test[~test.index.isin(out.index)]
    assert len(cold) and all(np.isnan(als.evaluate_regression(cold, name)) for name in want)
