"""GPU: hybrid top-k over per-user candidate lists (hals_score_blend_topk_lists, scoring.blend_topk_lists and
HybridRecommendationSystem.get_hybrid_recommendations_batch) against the reference fixtures, the per-user path, an fp64
oracle on ragged shapes and the shared-candidate kernels."""
import json
import os

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import hybrid_oracle
from tests.util import assert_ran, check_topk_against_dense, launched_kernels

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
TOL = 2e-6


def _scoring():
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import scoring
    return scoring


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def csr(lens):
    rowptr = np.zeros(len(lens) + 1, np.int64)
    rowptr[1:] = np.cumsum(lens)
    return rowptr


def test_reference_fixtures_in_one_launch():
    """The ten golden per-user calls as the rows of one call: rank-1 operands (u = [1], item row = the score), each row
    with the weights its f1_after selects, topk = the largest top_k."""
    scoring = _scoring()
    cases = json.load(open(os.path.join(G, "hybrid_reference_cases.json")))["cases"]
    als = np.concatenate([np.array(c["als"], np.float32) for c in cases])[:, None]
    tt = np.concatenate([np.array(c["tt"], np.float32) for c in cases])[:, None]
    rowptr = csr([len(c["als"]) for c in cases])
    w = np.array([hybrid_oracle.fusion_weights(*c["f1_after"]) for c in cases], np.float32)
    k = max(c["top_k"] for c in cases)
    one = np.ones((len(cases), 1), np.float32)
    pos, s = scoring.blend_topk_lists(dev(one), dev(als), dev(one), dev(tt), dev(rowptr),
                                      dev(np.arange(len(als), dtype=np.int32)), k, row_weights=dev(w))
    pos, s = pos.cpu().numpy(), s.cpu().numpy()
    for r, c in enumerate(cases):
        n = len(c["out_items"])
        assert list(pos[r, :n] - rowptr[r]) == c["out_items"], c["name"]
        assert np.allclose(s[r, :n], c["out_scores"], atol=TOL), c["name"]
        got = pos[r][pos[r] >= 0]
        assert len(got) == min(k, len(c["als"])) and (got < rowptr[r + 1]).all()


def _models(tmp_path):
    import hybrid_als_twotower_recommender_b200 as pkg
    rng = np.random.default_rng(21)
    U, I, nnz = 120, 90, 1500
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    manu_of, cat_of = rng.integers(0, 11, I + 10), rng.integers(0, 6, I + 10)
    price_of = rng.uniform(2, 200, I + 10)
    df = pd.DataFrame({"userId": u, "itemId": i, "average_review_rating": rng.integers(1, 6, nnz).astype(float),
                       "manufacturer_id": manu_of[i], "category_id": cat_of[i], "price": price_of[i]})
    als = pkg.ALSModel(rank=10, max_iter=5, reg_param=0.1)
    assert als.train(df) is True
    als.save_model(str(tmp_path / "als"))
    tt = pkg.TwoTowerModel(U, I, 11, 6)
    tt.build_model(seed=1)
    tt._prepare_features(df)
    tt.save_model(str(tmp_path / "tt.keras"))
    systems = []
    for _ in range(2):
        hrs = pkg.HybridRecommendationSystem()
        assert hrs.load_models(str(tmp_path / "als"), str(tmp_path / "tt.keras")) is True
        systems.append(hrs)
    # the universe: every trained item plus three ids ALS has never seen (cold items)
    ids = np.concatenate([np.unique(i), [I + 1, I + 4, I + 7]])
    items = pd.DataFrame({"itemId": ids, "manufacturer_id": manu_of[ids], "category_id": cat_of[ids],
                          "price": price_of[ids], "average_review_rating": 3.0})
    return systems, items, np.unique(u), rng


def test_batch_equals_the_per_user_loop(tmp_path):
    (batch, loop), items, uid, rng = _models(tmp_path)
    ids = items["itemId"].values
    users = [int(x) for x in uid[:14]] + [99_999, int(uid[3])]          # one cold user, one user twice
    lens = [0, 1, 3, 40, 93, 25, 5, 60, 2, 17, 93, 8, 30, 70, 50, 12]
    lists = [list(rng.choice(ids, n, replace=True)) for n in lens]        # with repeats
    lists[4] = list(ids) + list(ids[:3])                                  # every item, cold ones included, repeated
    actual = [None, {int(ids[0]): 5.0}, None, {}, {int(x): 4.0 for x in rng.choice(ids, 12, replace=False)}, None,
              {int(x): 1.0 for x in lists[6][:2]} | {12345: 3.0}, None, None,
              {int(x): 5.0 for x in rng.choice(ids, 20, replace=False)}, {}, None,
              {int(x): 5.0 for x in lists[12][:10]}, None, {int(x): 5.0 for x in lists[14][5:9]}, None]
    actual[0] = {int(ids[1]): 5.0}                                        # ratings on an empty list change nothing
    batch.als_f1_score, batch.twotower_f1_score = 0.5, 0.1
    loop.als_f1_score, loop.twotower_f1_score = 0.5, 0.1
    top_k = 7
    got = batch.get_hybrid_recommendations_batch(users, items, lists, actual, top_k)
    pos_of = {int(x): n for n, x in enumerate(ids)}
    for n, (u, lst, act) in enumerate(zip(users, lists, actual)):
        want = loop.get_hybrid_recommendations(u, items.iloc[[pos_of[int(x)] for x in lst]], act, top_k)
        assert len(got[n]) == len(want) == min(top_k, len(set(lst))), n
        wd = dict((int(i), float(s)) for i, s in want)
        for i, s in got[n]:                                              # scores: bit for bit
            if i in wd:
                assert s == wd[i], (n, i, s, wd[i])
        ws = [float(s) for _, s in want]
        assert [s for _, s in got[n]] == ws, n
        # item lists: equal up to the order (and the cut) inside groups of exactly equal scores
        for sc in set(ws):
            g = {i for i, s in got[n] if s == sc}
            w = {int(i) for i, s in want if float(s) == sc}
            assert g == w or (sc == ws[-1] and len(g) == len(w)), (n, sc)
    assert (batch.als_f1_score, batch.twotower_f1_score) == (loop.als_f1_score, loop.twotower_f1_score)
    assert (batch.als_f1_score, batch.twotower_f1_score) != (0.5, 0.1)
    # the same call as arrays, and with a 2-D padded candidate array
    a_ids, a_sc = batch.get_hybrid_recommendations_batch(users, items, lists, None, top_k, as_arrays=True)
    arr = np.full((len(users), max(len(x) for x in lists)), -1, np.int64)
    for n, lst in enumerate(lists):
        arr[n, :len(lst)] = lst
    b_ids, b_sc = batch.get_hybrid_recommendations_batch(users, items, arr, None, top_k, as_arrays=True)
    assert (a_ids == b_ids).all() and (a_sc.view(np.int32) == b_sc.view(np.int32)).all()
    assert a_ids.shape == (len(users), top_k) and (a_ids[0] == -1).all() and np.isneginf(a_sc[0]).all()


def _oracle_rows(Ua, Ia, Ut, It, rowptr, cand, w, raw, uk=None, ik=None, fb=None):
    out = []
    for r in range(len(rowptr) - 1):
        c = cand[rowptr[r]:rowptr[r + 1]]
        sa = (Ia[c].astype(np.float64) @ Ua[r].astype(np.float64)) if Ua.shape[1] else np.zeros(len(c))
        if fb is not None:
            cold = (~ik[c]) | (not uk[r])
            sa = np.where(cold, fb[c], sa)
        st = (It[c].astype(np.float64) @ Ut[r].astype(np.float64)) if Ut.shape[1] else np.zeros(len(c))
        if raw:
            out.append(w[r, 0] * sa + w[r, 1] * st)
        else:
            out.append(w[r, 0] * hybrid_oracle.minmax(sa) + w[r, 1] * hybrid_oracle.minmax(st) if len(c) else sa)
    return out


@pytest.mark.parametrize("ka,kt,k,per_row,raw,cold,long_row", [
    (10, 50, 1, False, False, False, False), (128, 50, 64, True, False, True, False),
    (64, 64, 65, True, False, False, False), (128, 0, 128, False, True, False, False),
    (0, 64, 129, True, False, False, False), (33, 7, 256, True, True, True, False),
    (128, 64, 100, True, False, True, True), (16, 50, 256, False, False, False, True),
])
def test_ragged_lists_against_the_oracle(ka, kt, k, per_row, raw, cold, long_row):
    scoring = _scoring()
    rng = np.random.default_rng(ka * 1000 + kt * 10 + k)
    n_items = 5000
    lens = [0, 1, k - 1, k, k + 1, 2 * k + 3, 31, 32, 33] + list(rng.integers(0, 3000, 40))
    if long_row:
        lens.insert(5, 300_000)
    lens = [max(int(n), 0) for n in lens]
    R = len(lens)
    rowptr = csr(lens)
    cand = rng.integers(0, n_items, int(rowptr[-1])).astype(np.int32)
    Ua = rng.normal(0, max(ka, 1) ** -0.5, (R, ka)).astype(np.float32)
    Ia = rng.normal(0, 1, (n_items, ka)).astype(np.float32)
    Ut, It = rng.normal(0, 1, (R, kt)).astype(np.float32), rng.normal(0, 1, (n_items, kt)).astype(np.float32)
    Ia[7] = Ia[8]; It[7] = It[8]                                      # exact ties
    w = rng.choice([0.2, 0.8], (R, 1)).astype(np.float32)
    w = np.concatenate([w, 1 - w], 1) if per_row else np.tile(np.float32([0.8, 0.2]), (R, 1))
    kw = dict(row_weights=dev(w)) if per_row else dict(w_als=0.8, w_tt=0.2)
    uk = ik = fb = None
    if cold:
        uk, ik = rng.random(R) > 0.2, rng.random(n_items) > 0.1
        fb = rng.uniform(1, 5, n_items).astype(np.float32)
        kw.update(user_known=dev(uk), item_known=dev(ik), als_fallback=dev(fb))
    ops = [dev(Ua) if ka else None, dev(Ia) if ka else None, dev(Ut) if kt else None, dev(It) if kt else None]
    with launched_kernels() as names:
        pos, s = scoring.blend_topk_lists(*ops, dev(rowptr), dev(cand), k, raw=raw, **kw)
        torch.cuda.synchronize()
    if long_row:
        assert_ran(names, "lists_seg_kernel", "lists_merge_kernel")
    pos, s = pos.cpu().numpy(), s.cpu().numpy()
    B = _oracle_rows(Ua, Ia, Ut, It, rowptr, cand, w, raw, uk, ik, fb)
    tol = 1e-4 if raw else 5 * TOL
    for r in range(R):
        if lens[r] == 0:
            assert (pos[r] == -1).all() and np.isneginf(s[r]).all()
            continue
        check_topk_against_dense(B[r][None], pos[r:r + 1] - np.where(pos[r:r + 1] >= 0, rowptr[r], 0),
                                 s[r:r + 1], k, tol)
    # determinism: the same call again, bit for bit
    pos2, s2 = scoring.blend_topk_lists(*ops, dev(rowptr), dev(cand), k, raw=raw, **kw)
    assert (pos2.cpu().numpy() == pos).all() and (s2.cpu().numpy().view(np.int32) == s.view(np.int32)).all()


def test_repeated_item_is_returned_at_each_position():
    scoring = _scoring()
    Ia = np.float32([[1.0], [3.0], [2.0]])
    cand = np.int32([1, 0, 1, 2, 1])
    one = np.ones((1, 1), np.float32)
    pos, s = scoring.blend_topk_lists(dev(one), dev(Ia), None, None, dev(csr([5])), dev(cand), 4, w_als=1.0, raw=True)
    assert pos.cpu().tolist() == [[0, 2, 4, 3]] and s.cpu().tolist() == [[3.0, 3.0, 3.0, 2.0]]


def test_shared_list_equals_the_shared_candidate_kernels():
    """Every user given the same list: the shared-candidate path (HybridScorer.recommend, behind recommend_batch) and
    the list path agree within the tie band (their dot products are summed in different orders)."""
    scoring = _scoring()
    rng = np.random.default_rng(5)
    U, I, ka, kt, k = 300, 3000, 128, 50, 100
    Ua, Ia = rng.normal(0, ka ** -0.5, (U, ka)).astype(np.float32), rng.normal(0, 1, (I, ka)).astype(np.float32)
    Ut, It = rng.normal(0, 1, (U, kt)).astype(np.float32), rng.normal(0, 1, (I, kt)).astype(np.float32)
    ref_i, ref_s = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It)).recommend(k, 0.2, 0.8)
    rowptr, cand = scoring.candidate_lists(None, np.arange(I), U, "cuda")
    pos, s = scoring.blend_topk_lists(dev(Ua), dev(Ia), dev(Ut), dev(It), rowptr, cand, k, w_als=0.2, w_tt=0.8)
    item = torch.where(pos >= 0, cand[pos.clamp(min=0).long()], -1)
    ref_i, ref_s, item, s = ref_i.cpu().numpy(), ref_s.cpu().numpy(), item.cpu().numpy(), s.cpu().numpy()
    assert np.abs(ref_s - s).max() <= 5 * TOL
    B = 0.2 * np.stack([hybrid_oracle.minmax(x) for x in Ua.astype(np.float64) @ Ia.astype(np.float64).T]) + \
        0.8 * np.stack([hybrid_oracle.minmax(x) for x in Ut.astype(np.float64) @ It.astype(np.float64).T])
    check_topk_against_dense(B, item, s, k, 5 * TOL)
    check_topk_against_dense(B, ref_i, ref_s, k, 5 * TOL)
