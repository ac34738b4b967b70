"""GPU parity: towers, extrema, fused blend + top-k, merge, list fusion -- against the CPU
oracle and against fixtures produced by the reference's own src/hybrid_system.py.

Tolerance: blended scores are in [0,1]; kernels blend in fp32, the reference in fp64 ->
|score diff| <= 2e-6, and top-k index sets must be identical except for items whose oracle
score is within 2e-6 of the k-th score (ties)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import hybrid_oracle, towers_oracle
from tests.util import check_topk_against_dense

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
TOL = 2e-6


def _pkg():
    import hybrid_als_twotower_recommender_b200 as pkg
    from hybrid_als_twotower_recommender_b200 import _native, scoring
    return pkg, _native, scoring


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def dense_blend(Ua, Ia, Ut, It, wa, wt):
    Sa = (Ua.astype(np.float64) @ Ia.astype(np.float64).T)
    St = (Ut.astype(np.float64) @ It.astype(np.float64).T)

    def mm(S):
        mn, mx = S.min(1, keepdims=True), S.max(1, keepdims=True)
        rg = mx - mn
        sc = np.where(rg != 0, 1.0 / np.where(rg != 0, rg, 1.0), 1.0)
        return (S - mn) * sc
    return wa * mm(Sa) + wt * mm(St), Sa, St


@pytest.mark.parametrize("U,I,ka,kt,k", [(130, 1000, 10, 50, 5), (64, 257, 128, 50, 100), (3, 5000, 64, 50, 10),
                                         (1, 20000, 128, 50, 100), (200, 90, 16, 8, 200), (77, 640, 10, 50, 64)] +
                         # either side of each candidate-capacity switch (topk_capacity: 64/65, 128/129), item-split
                         [(150, 1800, 32, 16, k) for k in (64, 65, 128, 129, 256)])
def test_blend_topk_matches_oracle(U, I, ka, kt, k):
    _, nat, scoring = _pkg()
    assert int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k)) < 0, "expected the CUDA-core path"
    rng = np.random.default_rng(U + I)
    Ua, Ia = rng.normal(0, ka ** -0.5, (U, ka)).astype(np.float32), rng.normal(0, 1, (I, ka)).astype(np.float32)
    Ut, It = rng.normal(0, 1, (U, kt)).astype(np.float32), rng.normal(0, 1, (I, kt)).astype(np.float32)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    ex = sc.extrema().cpu().numpy()
    B, Sa, St = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    want_ex = np.stack([Sa.min(1), Sa.max(1), St.min(1), St.max(1)], 1)
    assert np.allclose(ex, want_ex, rtol=1e-5, atol=1e-5)
    idx, s = sc.recommend(k, 0.8, 0.2)
    check_topk_against_dense(B, idx.cpu().numpy(), s.cpu().numpy(), k, TOL * 5)


@pytest.mark.parametrize("U,I,ka,kt,k", [(300, 20000, 128, 50, 100), (1000, 5000, 10, 50, 5), (130, 40000, 64, 50, 10),
                                         (2000, 3000, 128, 50, 100), (5, 900000, 128, 50, 100), (257, 16500, 20, 50, 30)] +
                         # either side of make_plan's candidate-capacity switches (56/57: 128 -> 256 keys per stream;
                         # 24/25 only differ in a two-part build), of the exact re-scoring's sort width (64/65,
                         # 128/129, 256) and of topk_capacity in the merge; one user tile against 512 item tiles:
                         # 64 splits, 512 columns per candidate stream
                         [(64, 131072, 64, 50, k) for k in (1, 24, 25, 56, 57, 64, 65, 128, 129, 256)])
def test_tensor_core_path_matches_oracle(U, I, ka, kt, k):
    """Shapes large enough for the tcgen05 path (TMA-staged bf16 operands, fused selection epilogue, exact
    fp32 re-scoring): the result must still be the exact fp32 answer."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(U * 7 + I)
    Ua, Ia = rng.normal(0, ka ** -0.5, (U, ka)).astype(np.float32), rng.normal(0, 1, (I, ka)).astype(np.float32)
    Ut, It = rng.normal(0, 1, (U, kt)).astype(np.float32), rng.normal(0, 1, (I, kt)).astype(np.float32)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k)) >= 0, "expected the tensor-core path"
    ex = sc.extrema().cpu().numpy()
    B, Sa, St = dense_blend(Ua, Ia, Ut, It, 0.2, 0.8)
    want_ex = np.stack([Sa.min(1), Sa.max(1), St.min(1), St.max(1)], 1)
    assert np.allclose(ex, want_ex, rtol=1e-5, atol=2e-5)
    idx, s = sc.recommend(k, 0.2, 0.8)
    check_topk_against_dense(B, idx.cpu().numpy(), s.cpu().numpy(), k, TOL * 5)
    assert sc.flagged_users(U, k) <= max(2, U // 20), "the candidate margin should make exact re-runs rare"


@pytest.mark.parametrize("mode", ["few_distinct_items", "duplicated_rows", "zero_als_items"])
def test_tensor_core_path_with_mass_score_ties(mode):
    """Many items with EXACTLY equal scores (duplicate feature rows, items without ALS factors): the streaming
    candidate filter must trim tie groups by item index and never run past a user's candidate buffer."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(11)
    U, I, ka, kt, k = 600, 8192, 64, 50, 100
    Ua, Ut = rng.normal(0, ka ** -0.5, (U, ka)).astype(np.float32), rng.normal(0, 1, (U, kt)).astype(np.float32)
    if mode == "few_distinct_items":
        base_a, base_t = rng.normal(0, 1, (7, ka)).astype(np.float32), rng.normal(0, 1, (7, kt)).astype(np.float32)
        Ia, It = base_a[np.arange(I) % 7], base_t[np.arange(I) % 7]          # 7 distinct scores, ~1170 ties each
    elif mode == "duplicated_rows":
        Ia, It = rng.normal(0, 1, (I, ka)).astype(np.float32), rng.normal(0, 1, (I, kt)).astype(np.float32)
        Ia[1000:1400], It[1000:1400] = Ia[999], It[999]                       # one item repeated 400 times
        Ia[5000:5300], It[5000:5300] = Ia[4999], It[4999]
    else:
        Ia, It = rng.normal(0, 1, (I, ka)).astype(np.float32), np.zeros((I, kt), np.float32)
        Ia[::3] = 0.0                                                         # a third of the items score exactly 0
    Ia, It = np.ascontiguousarray(Ia), np.ascontiguousarray(It)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k)) >= 0, "expected the tensor-core path"
    sc.extrema()
    idx, s = sc.recommend(k, 0.8, 0.2)
    idx, s = idx.cpu().numpy(), s.cpu().numpy()
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    check_topk_against_dense(B, idx, s, k, TOL * 5)
    assert (idx >= 0).all() and (idx < I).all()
    for u in range(0, U, 37):                          # no item twice in a list (a buffer overrun would corrupt neighbours)
        assert len(set(idx[u].tolist())) == k


def test_tensor_core_path_falls_back_exactly_when_bf16_cannot_separate():
    """Items that differ by less than bf16 resolution: the verification must refuse the tensor-core
    candidates and the exact re-run must still produce the oracle answer (incl. a constant model)."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(3)
    U, I, ka, kt, k = 40, 6000, 16, 8, 10
    base_a, base_t = rng.normal(0, 1, (1, ka)), rng.normal(0, 1, (1, kt))
    Ia = (base_a + 3e-3 * rng.normal(0, 1, (I, ka))).astype(np.float32)
    It = (base_t + 3e-3 * rng.normal(0, 1, (I, kt))).astype(np.float32)
    Ua, Ut = rng.normal(0, 1, (U, ka)).astype(np.float32), rng.normal(0, 1, (U, kt)).astype(np.float32)
    Ut[:5] = 0.0                                     # tower score constant (0) for these users: zero range
    # enough pairs for the tensor-core path
    reps = 20
    Ua, Ut = np.tile(Ua, (reps, 1)), np.tile(Ut, (reps, 1))
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U * reps, I, ka, kt, k)) >= 0
    ex = sc.extrema().cpu().numpy()
    B, Sa, St = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    assert np.allclose(ex, np.stack([Sa.min(1), Sa.max(1), St.min(1), St.max(1)], 1), rtol=1e-5, atol=1e-5)
    idx, s = sc.recommend(k, 0.8, 0.2)
    assert sc.flagged_users(U * reps, k) > 0, "this input must trigger the exact re-run"
    # score ranges are ~1e-2 here, so fp32 cancellation in (s - min)/(max - min) costs ~1e-5 of the [0,1] range
    check_topk_against_dense(B, idx.cpu().numpy(), s.cpu().numpy(), k, 2e-4)


def test_tower_ids_outside_the_tables_are_safe():
    """An id outside an embedding table must not read out of bounds: it contributes a zero vector (Keras' GPU
    Embedding behaviour), i.e. the user tower outputs LayerNorm(0) = beta."""
    pkg, nat, scoring = _pkg()
    from hybrid_als_twotower_recommender_b200.two_tower_model import TowerParams
    tp = TowerParams.keras_init(20, 30, 5, 4, 50, "cuda", seed=1)
    tp.t["user_ln_b"] += 0.25                            # a non-trivial beta to recognise
    w = tp.struct(None)
    ids = torch.tensor([0, 19, 20, 10**6, -3], dtype=torch.int32, device="cuda")
    out = torch.full((5, 50), 7.0, device="cuda")
    nat.check(nat.lib().hals_tower_user(w, nat.ptr(ids), 5, nat.ptr(out), 50, nat.current_stream()))
    o = out.cpu().numpy()
    assert np.isfinite(o).all()
    beta = tp.t["user_ln_b"].cpu().numpy()
    for r in (2, 3, 4):
        assert np.allclose(o[r], beta, atol=1e-6)
    assert not np.allclose(o[0], beta, atol=1e-3)
    # item tower: every table checked separately
    n = 4
    iid = torch.tensor([0, 30, 1, 2], dtype=torch.int32, device="cuda")
    mid = torch.tensor([0, 0, 5, 1], dtype=torch.int32, device="cuda")
    cid = torch.tensor([0, 0, 0, -1], dtype=torch.int32, device="cuda")
    num = torch.rand((n, 2), device="cuda")
    io = torch.empty((n, 50), device="cuda")
    nat.check(nat.lib().hals_tower_item(w, nat.ptr(iid), nat.ptr(mid), nat.ptr(cid), nat.ptr(num), n, nat.ptr(io), 50,
                                        nat.current_stream()))
    assert torch.isfinite(io).all()


def test_reference_fixtures_through_fused_kernels():
    """Score lists from the reference fixtures are fed as rank-1 'factors' (u=[1], item=[score]) so
    the fused extrema + blend + top-k kernels see exactly the reference's inputs."""
    _, nat, scoring = _pkg()
    for c in json.load(open(os.path.join(G, "hybrid_reference_cases.json")))["cases"]:
        als, tt = np.array(c["als"], np.float32), np.array(c["tt"], np.float32)
        one = np.ones((1, 1), np.float32)
        sc = scoring.HybridScorer(dev(one), dev(als[:, None]), dev(one), dev(tt[:, None]))
        wa, wt = hybrid_oracle.fusion_weights(*c["f1_after"])
        k = c["top_k"]
        idx, s = sc.recommend(k, wa, wt)
        idx, s = idx.cpu().numpy()[0], s.cpu().numpy()[0]
        n = len(c["out_items"])
        assert list(idx[:n]) == c["out_items"], c["name"]
        assert (idx[n:] == -1).all()
        assert np.allclose(s[:n], c["out_scores"], atol=TOL), c["name"]


def test_reference_fixtures_through_adaptive_fusion_api():
    pkg, _, _ = _pkg()
    for c in json.load(open(os.path.join(G, "hybrid_reference_cases.json")))["cases"]:
        hrs = pkg.HybridRecommendationSystem()
        hrs.als_f1_score, hrs.twotower_f1_score = c["f1_after"]
        a = [(i, float(x)) for i, x in enumerate(c["als"])]
        t = [(i, np.float32(x)) for i, x in enumerate(c["tt"])]
        combined = hrs.adaptive_fusion(a, t)
        top = sorted(combined, key=lambda x: x[1], reverse=True)[: c["top_k"]]
        got_items = [i for i, _ in top]
        if got_items != c["out_items"]:   # only fp32-level near-ties may reorder
            sc = dict(combined)
            for gi, wi in zip(got_items, c["out_items"]):
                assert abs(sc[gi] - sc[wi]) <= TOL, c["name"]
        assert np.allclose([s for _, s in top], c["out_scores"], atol=TOL), c["name"]


def test_zero_range_model_contributes_nothing_and_ties_prefer_low_index():
    _, nat, scoring = _pkg()
    I = 300
    Ua = np.ones((2, 4), np.float32); Ia = np.ones((I, 4), np.float32)          # constant ALS scores
    Ut = np.ones((2, 1), np.float32); It = (np.arange(I) % 7).astype(np.float32)[:, None]
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    idx, s = sc.recommend(10, 0.8, 0.2)
    idx, s = idx.cpu().numpy(), s.cpu().numpy()
    want = [6 + 7 * j for j in range(10)]       # the items with the max tower score, ascending index
    assert list(idx[0]) == want and list(idx[1]) == want
    assert np.allclose(s, 0.2, atol=1e-7)


def test_topk_merge_equals_global_topk():
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(8)
    U, I, k, P = 50, 4000, 100, 8
    S = rng.normal(size=(U, I)).astype(np.float32)
    S[:, 100:140] = S[:, 50:90]                                    # exact ties across shards
    per = I // P
    pidx = np.zeros((P, U, k), np.int32); psc = np.zeros((P, U, k), np.float32)
    for p in range(P):
        blk = S[:, p * per:(p + 1) * per]
        o = np.argsort(-blk, axis=1, kind="stable")[:, :k]
        pidx[p] = o + p * per; psc[p] = np.take_along_axis(blk, o, 1)
    pidx[3, :, 90:] = -1; psc[3, :, 90:] = -np.inf                 # a short list
    S2 = S.copy(); 
    for u in range(U):
        drop = np.argsort(-S[u, 3 * per:4 * per], kind="stable")[90:100] + 3 * per
        S2[u, drop] = -np.inf
    oi, os_ = scoring.merge_lists(dev(pidx), dev(psc))
    want = np.argsort(-S2, axis=1, kind="stable")[:, :k]
    assert np.array_equal(oi.cpu().numpy(), want)
    assert np.array_equal(os_.cpu().numpy(), np.take_along_axis(S2, want, 1))


def test_towers_match_oracle_fixture():
    pkg, nat, _ = _pkg()
    z = np.load(os.path.join(G, "tower_oracle_case.npz"))
    from hybrid_als_twotower_recommender_b200.two_tower_model import TowerParams
    import pandas as pd
    from sklearn.preprocessing import MinMaxScaler
    m = pkg.TwoTowerModel(60, 80, 17, 9)
    m.model = TowerParams.from_numpy({k[2:]: z[k] for k in z.files if k.startswith("w_")}, torch.device("cuda"))
    sc = MinMaxScaler(); sc.scale_, sc.min_ = z["scale"], z["offset"]
    m.scaler = sc
    df = pd.DataFrame({"itemId": z["ids"], "manufacturer_id": z["manu"], "category_id": z["cat"],
                       "price": z["raw"][:, 0], "average_review_rating": z["raw"][:, 1]})
    iv = m.item_vectors(df).cpu().numpy()
    uv = m.user_vectors(np.arange(60)).cpu().numpy()
    assert np.abs(iv - z["item_vecs"]).max() <= 2e-5
    assert np.abs(uv - z["user_vecs"]).max() <= 2e-5
    preds = m.predict_for_user(11, df)
    assert [p[0] for p in preds] == list(z["ids"])
    assert np.allclose([p[1] for p in preds], z["scores_user11"], atol=1e-4)
    assert isinstance(preds[0][1], np.float32)


def test_end_to_end_api_against_reference_semantics(tmp_path):
    """ALSModel.train -> save/load -> HybridRecommendationSystem.get_hybrid_recommendations and
    recommend_batch, compared with the oracle pipeline (Spark-restated ALS + Keras-restated towers +
    the reference's fusion semantics)."""
    import pandas as pd
    from oracle import als_oracle
    pkg, nat, _ = _pkg()
    rng = np.random.default_rng(21)
    U, I, nnz = 120, 90, 1500
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    manu_of, cat_of = rng.integers(0, 11, I), rng.integers(0, 6, I)
    price_of = rng.uniform(2, 200, I)
    df = pd.DataFrame({"userId": u, "itemId": i, "average_review_rating": rng.integers(1, 6, nnz).astype(float),
                       "manufacturer_id": manu_of[i], "category_id": cat_of[i], "price": price_of[i]})
    als = pkg.ALSModel(rank=10, max_iter=10, reg_param=0.1)
    uid, uinv = np.unique(u, return_inverse=True); iid, iinv = np.unique(i, return_inverse=True)
    X0 = als_oracle.init_factors(len(uid), 10, 5)
    assert als.train(df, init_user_factors=X0) is True
    Xo, Yo = als_oracle.als_fit(uinv, iinv, df["average_review_rating"].values.astype(np.float32), len(uid), len(iid),
                                10, 10, 0.1, X0)
    assert np.abs(als.model.user_factors.cpu().numpy() - Xo).max() <= 2e-3
    als.save_model(str(tmp_path / "als"))
    tt = pkg.TwoTowerModel(U, I, 11, 6)
    tt.build_model(seed=1)
    tt._prepare_features(df)
    tt.save_model(str(tmp_path / "tt.keras"))
    hrs = pkg.HybridRecommendationSystem()
    with pytest.raises(ValueError):
        hrs.get_hybrid_recommendations(0, [1, 2])
    assert hrs.load_models(str(tmp_path / "als"), str(tt_path := tmp_path / "tt.keras")) is True
    items = pd.DataFrame({"itemId": iid, "manufacturer_id": manu_of[iid], "category_id": cat_of[iid],
                          "price": price_of[iid], "average_review_rating": 3.0})
    user = int(uid[7])
    # oracle pipeline for this user
    w = {k: v for k, v in tt.model.to_numpy().items()}
    num = towers_oracle.scale_numeric(items[["price", "average_review_rating"]].values, tt.scaler.scale_, tt.scaler.min_)
    iv = towers_oracle.item_tower(w, iid, manu_of[iid], cat_of[iid], num)
    s_t = towers_oracle.score(towers_oracle.user_tower(w, [user])[0], iv)
    s_a = als_oracle.als_predict(Xo, Yo, np.full(len(iid), 7), np.arange(len(iid)))
    blend = hybrid_oracle.adaptive_fusion_dense(s_a, s_t)
    want_idx, want_sc = hybrid_oracle.topk_desc(blend, 5, ids=iid)
    top = hrs.get_hybrid_recommendations(user, items, top_k=5)
    assert [t[0] for t in top] == list(want_idx)
    assert np.allclose([t[1] for t in top], want_sc, atol=5e-4)
    ids_b, sc_b = hrs.recommend_batch([user, int(uid[0])], items, top_k=5)
    assert list(ids_b[0]) == list(want_idx) and np.allclose(sc_b[0], want_sc, atol=5e-4)
    # F1-driven weight switch (hybrid_system.py:104-105,69)
    actual = {int(want_idx[0]): 5.0}
    hrs.get_hybrid_recommendations(user, items, actual_ratings=actual, top_k=5)
    assert hrs.fusion_weights() in ((0.8, 0.2), (0.2, 0.8))
    # batched weight selector == the per-user one (hybrid_system.py:42-55), user by user
    users_b = [user, int(uid[0]), int(uid[3])]
    actuals = [{int(x): 5.0 for x in iid[rng.choice(len(iid), 12, replace=False)]} for _ in users_b]
    fa, ft = hrs.evaluate_models_batch(users_b, actuals, items)
    for n, (uu, act) in enumerate(zip(users_b, actuals)):
        a1, t1 = hrs.evaluate_individual_models(uu, act, items)
        assert fa[n] == pytest.approx(a1, abs=1e-6) and ft[n] == pytest.approx(t1, abs=1e-6)
    # cold item -> fallback value, cold user -> every item falls back (als_model.py:82-86)
    preds = als.predict_for_user(user, [int(iid[0]), 10_000])
    assert preds[1][0] == 10_000 and preds[1][1] == pytest.approx(als.global_mean)
    cold = als.predict_for_user(99_999, [int(iid[0])])
    assert len(cold) == 1 and np.isfinite(cold[0][1])
    hrs.cleanup()


def test_batched_f1_matches_the_reference_function():
    """hals_f1_at_k against compute_f1_score (src/als_model.py:171-177) user by user: integer arithmetic, exact."""
    _pkg()
    from hybrid_als_twotower_recommender_b200.evaluation import f1_at_k_batch
    rng = np.random.default_rng(8)
    U, I, k = 300, 500, 10
    scores = rng.normal(size=(U, I))
    order = np.argsort(-scores, axis=1, kind="stable")[:, :25].astype(np.int32)
    order[5, 7:] = -1                                                      # a list shorter than k
    actual = [rng.choice(I, rng.integers(0, 40), replace=True) for _ in range(U)]   # duplicates and empty sets
    actual[3] = np.array([], dtype=np.int64)
    got = f1_at_k_batch(dev(order), actual, k).cpu().numpy()
    for u in range(U):
        pred = {int(i): float(scores[u, i]) for i in order[u] if i >= 0} if u == 5 else {int(i): float(scores[u, i]) for i in range(I)}
        want = hybrid_oracle.compute_f1_score({int(a): 1.0 for a in actual[u]}, pred, k)
        assert got[u] == pytest.approx(want, abs=1e-7), u
    assert got[3] == 0.0


def test_batched_cold_start_fallback_matches_the_reference_loop():
    """hals_similar_items against the reference's per-item loop (als_model.py:79-104) restated with sklearn:
    ties, zero feature rows, items without a neighbour above 0.5, unknown ids."""
    pkg, nat, _ = _pkg()
    rng = np.random.default_rng(9)
    n = 400
    F = rng.integers(-2, 4, (n, 4)).astype(np.float64)                    # many exact ties and opposite directions
    F[10] = 0.0
    F[::7] *= -1.0
    R = rng.uniform(1, 5, n)
    feats = {1000 + j * 3: {"features": F[j], "rating": float(R[j])} for j in range(n)}
    als = pkg.ALSModel()
    als.item_features = feats
    als.global_mean = 3.21
    q = [1000, 1003 + 27, 1000 + 3 * 10, 1000 + 3 * 399, 1000 + 3 * 7, 5, 1000 + 3 * 123]   # incl. unknown ids
    got = als._fallback_scores(q)
    for item, g in zip(q, got):
        assert g == pytest.approx(hybrid_oracle.fallback_rating(feats, item, 3.21), abs=1e-12), item
    more = [1000 + 3 * j for j in range(0, n, 5)]
    got = als._fallback_scores(more)
    want = [hybrid_oracle.fallback_rating(feats, item, 3.21) for item in more]
    assert np.allclose(got, want, atol=1e-12)


def test_train_compacts_raw_ids_on_the_device(tmp_path):
    """ALSModel.train with sparse, unsorted raw ids: the id compaction runs on the GPU (no host np.unique); the
    factor tables must be keyed by the sorted raw ids exactly as before."""
    import pandas as pd
    from oracle import als_oracle, c_oracle
    pkg, _, _ = _pkg()
    rng = np.random.default_rng(31)
    U, I, nnz = 300, 200, 6000
    raw_u = rng.choice(10**9, U, replace=False); raw_i = rng.choice(10**6, I, replace=False)
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    r = rng.integers(1, 6, nnz).astype(np.float32)
    df = pd.DataFrame({"userId": raw_u[u], "itemId": raw_i[i], "average_review_rating": r.astype(float)})
    als = pkg.ALSModel(rank=64, max_iter=3, reg_param=0.1)
    uid, uinv = np.unique(raw_u[u], return_inverse=True); iid, iinv = np.unique(raw_i[i], return_inverse=True)
    X0 = als_oracle.init_factors(len(uid), 64, 4)
    assert als.train(df, init_user_factors=X0) is True
    assert np.array_equal(als.model.user_ids, uid) and np.array_equal(als.model.item_ids, iid)
    Xo, Yo = als_oracle.als_fit(uinv, iinv, r, len(uid), len(iid), 64, 3, 0.1, X0, half_step=c_oracle.als_half_step)
    assert np.abs(als.model.user_factors.cpu().numpy() - Xo).max() <= 1e-3
    assert np.abs(als.model.item_factors.cpu().numpy() - Yo).max() <= 1e-3
    assert als.global_mean == pytest.approx(float(r.mean()), abs=1e-6)
    assert set(als.item_features.keys()) == set(iid.tolist())             # built lazily from the training frame


@pytest.mark.gpu
def test_hyperparameter_tuning_grid_search():
    """two_tower_model.hyperparameter_tuning (src/two_tower_model.py:169-236): returns one of the grid entries (a copy),
    trains on the users that are not held out and scores the held-out users through predict_for_user."""
    import pandas as pd
    from hybrid_als_twotower_recommender_b200 import two_tower_model as ttm
    rng = np.random.default_rng(5)
    U, I, nnz = 40, 30, 900
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    # the function sizes the embedding tables by nunique() of the TRAINING part, so ids must be compact there: give the
    # users it will hold out (same draw as the function) the highest ids
    seen = pd.unique(u)                                  # order of first appearance, what the function draws from
    held = np.random.RandomState(7).choice(seen, size=int(len(seen) * 0.25), replace=False)
    order = np.concatenate([np.setdiff1d(np.arange(U), held), held])
    relabel = np.empty(U, np.int64); relabel[order] = np.arange(len(order))
    u = relabel[u]
    manu_of, cat_of, price_of = rng.integers(0, 4, I), rng.integers(0, 3, I), rng.uniform(5, 50, I)
    rating_of = rng.integers(1, 6, I).astype(float)     # ratings follow the item: some grid entry reaches F1@10 > 0
    df = pd.DataFrame({"userId": u, "itemId": i, "average_review_rating": rating_of[i],
                       "manufacturer_id": manu_of[i], "category_id": cat_of[i], "price": price_of[i]})
    grid = [{"batch_size": 64, "epochs": 1}, {"batch_size": 128, "epochs": 2}]
    import contextlib, io
    log = io.StringIO()
    with contextlib.redirect_stdout(log):
        best = ttm.hyperparameter_tuning(df, grid, val_size=0.25, random_state=7)
    assert "Error with params" not in log.getvalue(), log.getvalue()
    assert best in grid and all(best is not g for g in grid)
    # an entry that raises (missing key; ids outside the tables) is reported and skipped, like the reference
    assert ttm.hyperparameter_tuning(df, [{"batch_size": 64}], val_size=0.25, random_state=7) is None
    bad = df.copy(); bad["userId"] = bad["userId"] + 1000
    with contextlib.redirect_stdout(log):
        assert ttm.hyperparameter_tuning(bad, grid, val_size=0.25, random_state=7) is None
    assert "ids must lie in" in log.getvalue()


@pytest.mark.gpu
def test_load_model_reads_a_checkpoint_written_by_the_reference(tmp_path):
    """ALSModel.load_model on what the reference's save_model leaves behind: a Spark ALSModel directory (parquet factors)
    plus `<path>_metadata.pkl` (src/als_model.py:116-136).  Predictions must be the dot products of the stored factors."""
    import json
    import pickle
    import pyarrow as pa
    import pyarrow.parquet as pq
    pkg, nat, _ = _pkg()
    rng = np.random.default_rng(3)
    rank, uid, iid = 10, np.array([4, 9, 17, 30]), np.arange(100, 140)
    UF, IF = rng.standard_normal((len(uid), rank)).astype(np.float32), rng.standard_normal((len(iid), rank)).astype(np.float32)
    root = tmp_path / "als"
    (root / "metadata").mkdir(parents=True)
    (root / "metadata" / "part-00000").write_text(json.dumps({"class": "org.apache.spark.ml.recommendation.ALSModel", "rank": rank}) + "\n")
    for name, ids, f in (("userFactors", uid, UF), ("itemFactors", iid, IF)):
        (root / name).mkdir()
        perm = rng.permutation(len(ids))
        pq.write_table(pa.table({"id": pa.array(ids[perm].astype(np.int32)),
                                 "features": pa.array([r.tolist() for r in f[perm]], type=pa.list_(pa.float32()))}),
                       root / name / "part-00000.snappy.parquet")
    with open(f"{root}_metadata.pkl", "wb") as f:
        pickle.dump({"rank": rank, "max_iter": 10, "reg_param": 0.1, "global_mean": 3.5, "item_features": {}}, f)
    m = pkg.ALSModel().load_model(str(root))
    assert m is not None and m.rank == rank and m.global_mean == 3.5
    preds = dict(m.predict_for_user(17, list(iid[:7])))
    want = IF[:7] @ UF[2]
    assert np.allclose([preds[i] for i in iid[:7]], want, atol=1e-5)
