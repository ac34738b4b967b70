"""GPU: hals_score_blend_topk_excluding (per-user exclusion lists) on both scoring paths, against the dense fp64 blend
with the excluded items set to -inf, and through the public API (recommend_batch / evaluate_models_batch with
exclude=...).  Tolerances as in test_gpu_scoring.py."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import hybrid_oracle
from tests.test_gpu_scoring import G, TOL, dense_blend, dev

pytestmark = pytest.mark.gpu


def _pkg():
    import hybrid_als_twotower_recommender_b200 as pkg
    from hybrid_als_twotower_recommender_b200 import _native, scoring
    return pkg, _native, scoring


def to_csr(lists):
    """Python lists of global item ids -> device (rowptr int64, items int32), rows sorted ascending."""
    lens = np.array([len(x) for x in lists], np.int64)
    rowptr = np.zeros(len(lists) + 1, np.int64)
    np.cumsum(lens, out=rowptr[1:])
    flat = np.concatenate([np.sort(np.asarray(x, np.int64)) for x in lists]) if rowptr[-1] else np.zeros(0, np.int64)
    return dev(rowptr), dev(flat.astype(np.int32))


def make_lists(U, I, k, rng, item_offset=0):
    """Row 0: random; 1: empty; 2: every item (all -1); 3: all but k // 2 items (a padded list); further rows random.
    Random rows hold duplicates and ids outside [item_offset, item_offset + I)."""
    lists = []
    for u in range(U):
        r = u if u < 4 else 0
        if r == 1:
            x = np.zeros(0, np.int64)
        elif r == 2:
            x = np.arange(I)
        elif r == 3:
            x = np.setdiff1d(np.arange(I), rng.choice(I, max(1, min(k // 2, I // 2)), replace=False))
        else:
            x = rng.choice(I, int(rng.integers(1, min(I, 3 * k) + 1)), replace=True)     # duplicates
            x = np.concatenate([x, x[: len(x) // 4]])
        x = x + item_offset
        if r == 0:
            x = np.concatenate([x, [item_offset - 1, item_offset - 1000, item_offset + I, item_offset + I + 77]])
        lists.append(x)
    return lists


def check_excluding(B, lists, idx, score, k, tol, item_offset=0):
    """B: fp64 blend [U, I] over all items.  The list of user u must be the top-k of B[u] with lists[u] removed
    (index sets identical outside the tie band `tol`), padded with -1 / -inf, no excluded item, no item twice."""
    U, I = B.shape
    for u in range(U):
        x = np.asarray(lists[u], np.int64) - item_offset
        x = x[(x >= 0) & (x < I)]
        Bm = B[u].copy()
        Bm[x] = -np.inf
        n_allowed = int(np.isfinite(Bm).sum())
        kk = min(k, n_allowed)
        got = idx[u]
        valid = got[:kk] - item_offset
        assert (got[:kk] >= 0).all() and (got[kk:] == -1).all(), (u, kk, got)
        assert np.isneginf(score[u, kk:]).all()
        assert len(set(valid.tolist())) == kk
        assert not (set(valid.tolist()) & set(x.tolist())), (u, "an excluded item was returned")
        if kk == 0:
            continue
        s = score[u, :kk].astype(np.float64)
        assert np.all(np.diff(s) <= 0)
        assert np.allclose(s, B[u, valid], rtol=0, atol=tol), np.abs(s - B[u, valid]).max()
        kth = np.sort(Bm)[::-1][kk - 1]
        must = set(np.nonzero(Bm > kth + tol)[0].tolist())
        assert must <= set(valid.tolist()), (u, must - set(valid.tolist()))
        assert np.all(B[u, valid] >= kth - tol)
        for a in range(kk - 1):
            if score[u, a] == score[u, a + 1]:
                assert got[a] < got[a + 1]


def random_operands(U, I, ka, kt, seed):
    rng = np.random.default_rng(seed)
    Ua, Ia = rng.normal(0, ka ** -0.5, (U, ka)).astype(np.float32), rng.normal(0, 1, (I, ka)).astype(np.float32)
    Ut, It = rng.normal(0, 1, (U, kt)).astype(np.float32), rng.normal(0, 1, (I, kt)).astype(np.float32)
    return rng, Ua, Ia, Ut, It


@pytest.mark.parametrize("U,I,ka,kt,k", [(130, 1000, 10, 50, 5), (64, 257, 128, 50, 100), (3, 5000, 64, 50, 10),
                                         (1, 20000, 128, 50, 100), (200, 90, 16, 8, 200), (77, 640, 10, 50, 64)])
def test_simt_path_excluding_matches_oracle(U, I, ka, kt, k):
    _, nat, scoring = _pkg()
    rng, Ua, Ia, Ut, It = random_operands(U, I, ka, kt, U + I)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k)) < 0, "expected the CUDA-core path"
    lists = make_lists(U, I, k, rng)
    idx, s = sc.recommend(k, 0.8, 0.2, exclude=to_csr(lists))
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    check_excluding(B, lists, idx.cpu().numpy(), s.cpu().numpy(), k, TOL * 5)


@pytest.mark.parametrize("U,I,ka,kt,k", [(300, 20000, 128, 50, 100), (1000, 5000, 10, 50, 5), (130, 40000, 64, 50, 10),
                                         (2000, 3000, 128, 50, 100), (5, 900000, 128, 50, 100), (257, 16500, 20, 50, 30)])
def test_tensor_core_path_excluding_matches_oracle(U, I, ka, kt, k):
    _, nat, scoring = _pkg()
    rng, Ua, Ia, Ut, It = random_operands(U, I, ka, kt, U * 7 + I)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k)) >= 0, "expected the tensor-core path"
    lists = make_lists(U, I, k, rng)
    idx, s = sc.recommend(k, 0.2, 0.8, exclude=to_csr(lists))
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.2, 0.8)
    check_excluding(B, lists, idx.cpu().numpy(), s.cpu().numpy(), k, TOL * 5)
    # the bound of test_tensor_core_path_matches_oracle, plus rows 2 and 3 of make_lists: a user left with fewer than
    # k items has kth = -inf and is re-run exactly whenever one of its streams raised its threshold
    assert sc.flagged_users(U, k) <= max(2, U // 20) + 2, "exclusion must not make exact re-runs common"


def test_tensor_core_path_long_lists_at_large_k():
    """k = 256 (streams compact above 224 candidates) with lists that exclude most of the items: the cursor walks long
    runs of excluded ids, users left with fewer than k items are padded (and re-run exactly when a stream compacted),
    users with a few hundred items left still get the exact answer."""
    _, nat, scoring = _pkg()
    U, I, ka, kt, k = 512, 16384, 64, 50, 256
    rng, Ua, Ia, Ut, It = random_operands(U, I, ka, kt, 1234)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k)) >= 0, "expected the tensor-core path"
    lists = []
    for u in range(U):
        left = (100, 200, 300, 600, 2000, I // 2)[u % 6]                 # allowed items left for this user
        lists.append(np.setdiff1d(np.arange(I), rng.choice(I, left, replace=False)))
    idx, s = sc.recommend(k, 0.8, 0.2, exclude=to_csr(lists))
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    check_excluding(B, lists, idx.cpu().numpy(), s.cpu().numpy(), k, TOL * 5)


def test_own_top_excluded_equals_the_tail_of_a_longer_list():
    """1.25 M items, each user's own top-156 excluded: the top-100 of what remains is entries 156..255 of the
    unexcluded top-256 (up to exact ties at either boundary)."""
    _, nat, scoring = _pkg()
    U, I, ka, kt = 4096, 1_250_000, 128, 50
    g = torch.Generator(device="cuda").manual_seed(7)
    Ua = torch.randn(U, ka, device="cuda", generator=g) * ka ** -0.5
    Ia = torch.randn(I, ka, device="cuda", generator=g)
    Ut = torch.nn.functional.layer_norm(torch.randn(U, kt, device="cuda", generator=g), (kt,))
    It = torch.nn.functional.layer_norm(torch.randn(I, kt, device="cuda", generator=g), (kt,))
    sc = scoring.HybridScorer(Ua, Ia, Ut, It)
    ex = sc.extrema()
    top156, _ = sc.topk_local(ex, 156, 0.8, 0.2)
    i256, s256 = sc.topk_local(ex, 256, 0.8, 0.2)
    rows = torch.arange(U, device="cuda").repeat_interleave(156)
    excl = scoring.exclusion_lists(rows, top156.reshape(-1).long(), U)
    idx, s = sc.topk_local(ex, 100, 0.8, 0.2, exclude=excl)
    f = sc.flagged_users(U, 100)
    assert f <= U // 20, f
    idx, s, i256, s256 = idx.cpu().numpy(), s.cpu().numpy(), i256.cpu().numpy(), s256.cpu().numpy()
    assert (idx >= 0).all()
    assert np.allclose(s, s256[:, 156:], rtol=0, atol=1e-6), np.abs(s - s256[:, 156:]).max()
    mism = 0
    for u in range(U):
        a, b = set(idx[u].tolist()), set(i256[u, 156:].tolist())
        if a != b:
            mism += 1
            score_of = dict(zip(i256[u].tolist(), s256[u].tolist()))
            score_of.update(zip(idx[u].tolist(), s[u].tolist()))
            bounds = (s256[u, 155], s256[u, 255])
            for it in a ^ b:         # only items tied with a boundary score may differ
                assert min(abs(score_of[it] - x) for x in bounds) <= 1e-6, (u, it)
    assert mism <= U // 100, mism


def test_adversarial_bf16_input_excluding_reruns_exactly():
    """The input of test_tensor_core_path_falls_back_exactly_when_bf16_cannot_separate with exclusions: the exact
    list-mode re-run (users indexed through the flagged list) must filter too."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(3)
    U, I, ka, kt, k = 40, 6000, 16, 8, 10
    base_a, base_t = rng.normal(0, 1, (1, ka)), rng.normal(0, 1, (1, kt))
    Ia = (base_a + 3e-3 * rng.normal(0, 1, (I, ka))).astype(np.float32)
    It = (base_t + 3e-3 * rng.normal(0, 1, (I, kt))).astype(np.float32)
    Ua, Ut = rng.normal(0, 1, (U, ka)).astype(np.float32), rng.normal(0, 1, (U, kt)).astype(np.float32)
    Ut[:5] = 0.0
    reps = 20
    Ua, Ut = np.tile(Ua, (reps, 1)), np.tile(Ut, (reps, 1))
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U * reps, I, ka, kt, k)) >= 0
    sc.extrema()
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    # each user loses its own oracle top-15 (so the answer lies entirely behind the excluded items) + random ids
    lists = [np.concatenate([np.argsort(-B[u], kind="stable")[:15], rng.choice(I, 40)]) for u in range(U * reps)]
    lists[3] = np.zeros(0, np.int64)
    idx, s = sc.recommend(k, 0.8, 0.2, exclude=to_csr(lists))
    assert sc.flagged_users(U * reps, k) > 0, "this input must trigger the exact re-run"
    check_excluding(B, lists, idx.cpu().numpy(), s.cpu().numpy(), k, 2e-4)


def test_mass_ties_excluding_part_of_a_tie_group():
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(11)
    U, I, ka, kt, k = 600, 8192, 64, 50, 100
    Ua, Ut = rng.normal(0, ka ** -0.5, (U, ka)).astype(np.float32), rng.normal(0, 1, (U, kt)).astype(np.float32)
    base_a, base_t = rng.normal(0, 1, (7, ka)).astype(np.float32), rng.normal(0, 1, (7, kt)).astype(np.float32)
    Ia, It = np.ascontiguousarray(base_a[np.arange(I) % 7]), np.ascontiguousarray(base_t[np.arange(I) % 7])
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    assert int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k)) >= 0
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    lists = []
    for u in range(U):
        group = np.nonzero(B[u] == B[u].max())[0]             # the user's top tie group, ascending
        lists.append(np.concatenate([group[: 150: 2], group[200:230], rng.choice(I, 20)]))
    idx, s = sc.recommend(k, 0.8, 0.2, exclude=to_csr(lists))
    idx, s = idx.cpu().numpy(), s.cpu().numpy()
    check_excluding(B, lists, idx, s, k, TOL * 5)
    for u in range(U):
        assert len(set(idx[u].tolist())) == k
        gone = set(lists[u].tolist())
        for g in set((idx[u] % 7).tolist()):                  # item i has feature row i % 7: one tie group per residue
            chosen = sorted(x for x in idx[u].tolist() if x % 7 == g)
            allowed = [x for x in range(g, I, 7) if x not in gone]
            assert chosen == allowed[: len(chosen)], (u, g)    # the lowest allowed indices of the group


def test_item_sharded_lists_merge_to_the_single_call():
    """Two item halves scored with item_offset and the SAME global lists, merged, equal one call over all items."""
    _, nat, scoring = _pkg()
    U, I, ka, kt, k = 600, 20000, 128, 50, 100
    rng, Ua, Ia, Ut, It = random_operands(U, I, ka, kt, 99)
    h = I // 2
    full = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    ex = full.extrema()
    lists = make_lists(U, I, k, rng)
    excl = to_csr(lists)
    want_i, want_s = full.topk_local(ex, k, 0.8, 0.2, exclude=excl)
    parts_i, parts_s = [], []
    for lo, hi in ((0, h), (h, I)):
        part = scoring.HybridScorer(dev(Ua), dev(Ia[lo:hi]), dev(Ut), dev(It[lo:hi]), item_offset=lo)
        assert int(nat.lib().hals_score_flag_counter_offset(U, hi - lo, ka, kt, k)) >= 0
        pi, ps = part.topk_local(ex, k, 0.8, 0.2, exclude=excl)
        parts_i.append(pi); parts_s.append(ps)
    got_i, got_s = scoring.merge_lists(torch.stack(parts_i), torch.stack(parts_s))
    assert torch.equal(got_i, want_i)
    assert torch.allclose(got_s, want_s, rtol=0, atol=1e-6)
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    check_excluding(B, lists, got_i.cpu().numpy(), got_s.cpu().numpy(), k, TOL * 5)


@pytest.mark.parametrize("U,I,ka,kt,k", [(130, 1000, 10, 50, 5), (300, 20000, 128, 50, 100)])
def test_empty_lists_are_bit_identical_to_the_plain_call(U, I, ka, kt, k):
    _, nat, scoring = _pkg()
    _, Ua, Ia, Ut, It = random_operands(U, I, ka, kt, 5)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    ex = sc.extrema()
    pi, ps = sc.topk_local(ex, k, 0.8, 0.2)
    empty = (torch.zeros(U + 1, dtype=torch.int64, device="cuda"), torch.zeros(0, dtype=torch.int32, device="cuda"))
    ei, es = sc.topk_local(ex, k, 0.8, 0.2, exclude=empty)
    assert torch.equal(pi, ei)
    assert torch.equal(ps.view(torch.int32), es.view(torch.int32))


def test_null_and_half_null_lists():
    """Both pointers NULL: the plain call; exactly one NULL: HALS_ERR_INVALID."""
    _, nat, scoring = _pkg()
    U, I, ka, kt, k = 20, 500, 8, 8, 5
    _, Ua, Ia, Ut, It = random_operands(U, I, ka, kt, 6)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    ex = sc.extrema()
    pi, ps = sc.topk_local(ex, k, 0.8, 0.2)
    L = nat.lib()
    ws = sc._workspace(U, k)
    rowptr = torch.zeros(U + 1, dtype=torch.int64, device="cuda")
    for rp, it, want_rc in ((None, None, 0), (rowptr, None, 1), (None, rowptr, 1)):
        oi = torch.full((U, k), 7, dtype=torch.int32, device="cuda")
        os_ = torch.empty((U, k), dtype=torch.float32, device="cuda")
        rc = L.hals_score_blend_topk_excluding(*sc._ops(0, U), U, I, nat.ptr(ex), 0.8, 0.2, k, 0, nat.ptr(oi),
                                               nat.ptr(os_), nat.ptr(rp), nat.ptr(it), nat.ptr(ws), ws.numel(),
                                               nat.current_stream())
        assert rc == want_rc
        if rc == 0:
            assert torch.equal(oi, pi) and torch.equal(os_, ps)


def test_reference_fixtures_with_exclusions_through_fused_kernels():
    """The reference fixtures through the rank-1 trick of test_reference_fixtures_through_fused_kernels, a few items
    excluded: adaptive_fusion_dense over ALL items, the excluded ones removed, then topk_desc."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(17)
    for c in json.load(open(os.path.join(G, "hybrid_reference_cases.json")))["cases"]:
        als, tt = np.array(c["als"], np.float32), np.array(c["tt"], np.float32)
        n = len(als)
        one = np.ones((1, 1), np.float32)
        sc = scoring.HybridScorer(dev(one), dev(als[:, None]), dev(one), dev(tt[:, None]))
        wa, wt = hybrid_oracle.fusion_weights(*c["f1_after"])
        k = c["top_k"]
        x = np.unique(np.concatenate([c["out_items"][:2], rng.choice(n, min(n, 3))]))
        idx, s = sc.recommend(k, wa, wt, exclude=to_csr([x]))
        idx, s = idx.cpu().numpy()[0], s.cpu().numpy()[0]
        blend = hybrid_oracle.adaptive_fusion_dense(als, tt, *c["f1_after"])
        keep = np.setdiff1d(np.arange(n), x)
        want_i, want_s = hybrid_oracle.topk_desc(blend[keep], k, ids=keep)
        m = len(want_i)
        assert list(idx[:m]) == list(want_i), c["name"]
        assert (idx[m:] == -1).all()
        assert np.allclose(s[:m], want_s, atol=TOL), c["name"]


def test_public_api_excludes_training_pairs(tmp_path):
    import pandas as pd
    pkg, nat, _ = _pkg()
    rng = np.random.default_rng(21)
    U, I, nnz = 120, 90, 1500
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    manu_of, cat_of = rng.integers(0, 11, I), rng.integers(0, 6, I)
    price_of = rng.uniform(2, 200, I)
    df = pd.DataFrame({"userId": u, "itemId": i, "average_review_rating": rng.integers(1, 6, nnz).astype(float),
                       "manufacturer_id": manu_of[i], "category_id": cat_of[i], "price": price_of[i]})
    als = pkg.ALSModel(rank=10, max_iter=5, reg_param=0.1)
    assert als.train(df) is True
    als.save_model(str(tmp_path / "als"))
    tt = pkg.TwoTowerModel(U, I, 11, 6)
    tt.build_model(seed=1)
    tt._prepare_features(df)
    tt.save_model(str(tmp_path / "tt.keras"))
    hrs = pkg.HybridRecommendationSystem()
    assert hrs.load_models(str(tmp_path / "als"), str(tmp_path / "tt.keras")) is True
    iid = np.unique(i)
    items = pd.DataFrame({"itemId": iid, "manufacturer_id": manu_of[iid], "category_id": cat_of[iid],
                          "price": price_of[iid], "average_review_rating": 3.0})
    uid = np.unique(u)
    users = [int(x) for x in uid[:40]] + [int(uid[0])]            # a repeated user
    train = df[["userId", "itemId"]]
    seen = {uu: set(df.itemId[df.userId == uu].tolist()) for uu in uid}
    top_k = 10
    ids_b, sc_b = hrs.recommend_batch(users, items, top_k=top_k, exclude=train)
    for r, uu in enumerate(users):
        row = [x for x in ids_b[r].tolist() if x >= 0]
        assert not (set(row) & seen[uu]), (uu, set(row) & seen[uu])
        assert len(row) == min(top_k, len(iid) - len(seen[uu] & set(iid.tolist())))
    assert list(ids_b[0]) == list(ids_b[-1])
    # the per-user reference path, filtered on the host
    for r in (0, 3, 7, 12):
        uu = users[r]
        combined = hrs.adaptive_fusion(hrs.als_model.predict_for_user(uu, items),
                                       hrs.twotower_model.predict_for_user(uu, items))
        ranked = sorted([(it, sc) for it, sc in combined if it not in seen[uu]], key=lambda p: p[1], reverse=True)[:top_k]
        assert np.allclose(sc_b[r][: len(ranked)], [p[1] for p in ranked], atol=5e-4)
        score_of = dict(combined)
        for a, b in zip(ids_b[r], [p[0] for p in ranked]):
            assert a == b or abs(score_of[a] - score_of[b]) <= 1e-3, (uu, a, b)
    # evaluate_models_batch: F1 of each model's own top-10 after the exclusion
    actuals = [{int(x): 5.0 for x in iid[rng.choice(len(iid), 12, replace=False)]} for _ in users]
    fa, ft = hrs.evaluate_models_batch(users, actuals, items, exclude=train)
    for r, (uu, act) in enumerate(zip(users, actuals)):
        for model, got in ((hrs.als_model, fa[r]), (hrs.twotower_model, ft[r])):
            preds = {it: float(sc) for it, sc in model.predict_for_user(uu, items) if it not in seen[uu]}
            assert got == pytest.approx(hybrid_oracle.compute_f1_score(act, preds, 10), abs=1e-6), (r, uu)
    hrs.cleanup()
