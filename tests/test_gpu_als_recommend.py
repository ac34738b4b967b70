"""GPU: the ALS top-k by raw dot product (hals_score_topk, HybridScorer.topk_dot) and Spark's recommendFor* API on
ALSModel, against numpy fp64 Q @ C.T on both routes (CUDA-core and tensor-core).  Raw scores are not in [0, 1], so
every row of the oracle and of the kernel scores is divided by s_q = |q| * max_c |c| before the comparison (the same
positive factor on both sides keeps the order and the ties); the tolerance is then relative to that scale."""
import json
import pickle

import numpy as np
import pandas as pd
import pytest
import torch

from tests.test_gpu_exclude import check_excluding, make_lists, to_csr
from tests.test_gpu_scoring import dev
from tests.util import assert_ran, check_topk_against_dense, launched_kernels

pytestmark = pytest.mark.gpu

TOL = 1e-5                                    # of s_q: fp32 dot products of up to 128 terms
KS = (1, 10, 24, 25, 56, 57, 64, 65, 100, 128, 129, 256)   # either side of every capacity switch of make_plan


def _pkg():
    import hybrid_als_twotower_recommender_b200 as pkg
    from hybrid_als_twotower_recommender_b200 import _native, scoring
    return pkg, _native, scoring


def oracle(Q, C):
    """(normalised fp64 scores [n_q, n_c], s_q [n_q])."""
    S = Q.astype(np.float64) @ C.astype(np.float64).T
    cmax = np.linalg.norm(C.astype(np.float64), axis=1).max() if len(C) else 1.0
    s = np.linalg.norm(Q.astype(np.float64), axis=1) * cmax
    s = np.where(s > 0, s, 1.0)
    return S / s[:, None], s


def check(Q, C, idx, score, k, c_offset=0, tol=TOL):
    idx, score = idx.cpu().numpy(), score.cpu().numpy()
    B, s = oracle(Q, C)
    kk = min(k, C.shape[0])
    assert np.isneginf(score[:, kk:]).all()
    check_topk_against_dense(B, idx, score / s[:, None], k, tol, item_offset=c_offset)


def route(nat, n_q, n_c, rank, k):
    return "tc" if int(nat.lib().hals_score_flag_counter_offset(n_q, n_c, rank, 0, k)) >= 0 else "simt"


def factors(n, rank, rng, scale=1.0):
    return (rng.normal(0, scale, (n, rank))).astype(np.float32)


@pytest.mark.parametrize("rank", [10, 64, 128])
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("want_route,U,I", [("simt", 100, 1500), ("tc", 1024, 4096)])
def test_topk_dot_matches_numpy(want_route, U, I, rank, k):
    _, nat, scoring = _pkg()
    assert route(nat, U, I, rank, k) == want_route
    rng = np.random.default_rng(U + I + rank + k)
    Q, C = factors(U, rank, rng, rank ** -0.5), factors(I, rank, rng)
    sc = scoring.HybridScorer(dev(Q), dev(C), None, None)
    idx, s = sc.topk_dot(k)
    check(Q, C, idx, s, k)
    f = sc.flagged_users(U, k, dot=True)
    assert (f < 0) == (want_route == "simt") and f <= U // 20, f


def test_more_columns_asked_than_exist_are_padded():
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(1)
    Q, C = factors(50, 32, rng), factors(30, 32, rng)
    idx, s = scoring.HybridScorer(dev(Q), dev(C), None, None).topk_dot(100)
    assert (idx[:, 30:] == -1).all() and torch.isneginf(s[:, 30:]).all()
    check(Q, C, idx, s, 100)


def _raw_call(nat, Q, q_stride, C, c_stride, rank, n_q, n_c, k, c_offset, excl=(None, None)):
    L = nat.lib()
    ws = torch.empty(int(L.hals_score_workspace_bytes(n_q, n_c, rank, 0, k)), dtype=torch.uint8, device="cuda")
    oi = torch.full((n_q, k), 7, dtype=torch.int32, device="cuda")
    os_ = torch.zeros((n_q, k), dtype=torch.float32, device="cuda")
    rc = L.hals_score_topk(nat.ptr(Q), q_stride, nat.ptr(C), c_stride, rank, n_q, n_c, k, c_offset, nat.ptr(excl[0]),
                           nat.ptr(excl[1]), nat.ptr(oi), nat.ptr(os_), nat.ptr(ws), ws.numel(), nat.current_stream())
    nat.check(rc, "hals_score_topk")
    return oi, os_, ws


def test_no_columns_gives_padded_lists():
    _, nat, _ = _pkg()
    Q, C = torch.randn(40, 16, device="cuda"), torch.randn(1, 16, device="cuda")
    oi, os_, _ = _raw_call(nat, Q, 16, C, 16, 16, 40, 0, 10, 0)
    assert (oi == -1).all() and torch.isneginf(os_).all()


@pytest.mark.parametrize("U,I,rank,k", [(70, 900, 24, 10), (1100, 4000, 64, 100), (600, 8192, 128, 30)])
def test_strided_row_views_with_a_column_offset(U, I, rank, k):
    """Q and C are column slices of wider tables (row stride > rank, not 16-byte aligned); indices come back + c_offset."""
    _, nat, _ = _pkg()
    rng = np.random.default_rng(U)
    Qw, Cw = factors(U, rank + 7, rng), factors(I, rank + 5, rng)
    Q, C = Qw[:, 3:3 + rank], Cw[:, 1:1 + rank]
    Qd, Cd = dev(Qw), dev(Cw)
    oi, os_, ws = _raw_call(nat, Qd[:, 3:], rank + 7, Cd[:, 1:], rank + 5, rank, U, I, k, 5000)
    check(Q, C, oi, os_, k, c_offset=5000)
    off = int(nat.lib().hals_score_flag_counter_offset(U, I, rank, 0, k))
    if I >= 2048:
        assert off >= 0 and int(ws[off:off + 4].view(torch.int32).item()) <= U // 20


@pytest.mark.parametrize("mode", ["few_distinct_items", "duplicated_rows", "zero_items"])
def test_tensor_core_route_with_mass_score_ties(mode):
    """Many columns with EXACTLY equal scores: tie groups are cut by column index and the result stays exact."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(11)
    U, I, rank, k = 600, 8192, 64, 100
    Q = factors(U, rank, rng, rank ** -0.5)
    if mode == "few_distinct_items":
        C = factors(7, rank, rng)[np.arange(I) % 7]
    elif mode == "duplicated_rows":
        C = factors(I, rank, rng)
        C[1000:1400], C[5000:5300] = C[999], C[4999]
    else:
        C = factors(I, rank, rng)
        C[::3] = 0.0
    C = np.ascontiguousarray(C)
    assert route(nat, U, I, rank, k) == "tc"
    idx, s = scoring.HybridScorer(dev(Q), dev(C), None, None).topk_dot(k)
    check(Q, C, idx, s, k)
    idx = idx.cpu().numpy()
    assert (idx >= 0).all() and all(len(set(r.tolist())) == k for r in idx)


def test_tensor_core_route_reruns_exactly_when_bf16_cannot_separate():
    """Columns that differ by less than bf16 resolution: the verification (gamma = 0) must refuse the candidates, and the
    exact CUDA-core re-run still gives the numpy answer."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(3)
    U, I, rank, k = 800, 6000, 16, 10
    C = (rng.normal(0, 1, (1, rank)) + 3e-3 * rng.normal(0, 1, (I, rank))).astype(np.float32)
    Q = factors(U, rank, rng)
    assert route(nat, U, I, rank, k) == "tc"
    sc = scoring.HybridScorer(dev(Q), dev(C), None, None)
    idx, s = sc.topk_dot(k)
    assert sc.flagged_users(U, k, dot=True) > 0, "this input must trigger the exact re-run"
    check(Q, C, idx, s, k, tol=1e-6)


@pytest.mark.parametrize("U,I,rank,k", [(130, 1000, 10, 5), (64, 257, 128, 100), (1024, 4096, 64, 10),
                                        (1100, 5000, 128, 100), (512, 16384, 64, 256)])
def test_exclusion_lists(U, I, rank, k):
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(U * 3 + I)
    Q, C = factors(U, rank, rng, rank ** -0.5), factors(I, rank, rng)
    sc = scoring.HybridScorer(dev(Q), dev(C), None, None)
    lists = make_lists(U, I, k, rng)          # incl. an empty row, a row excluding everything and a padded row
    idx, s = sc.topk_dot(k, exclude=to_csr(lists))
    B, sq = oracle(Q, C)
    check_excluding(B, lists, idx.cpu().numpy(), s.cpu().numpy() / sq[:, None], k, TOL)


@pytest.mark.parametrize("U,I,rank,k", [(130, 1000, 10, 5), (1024, 4096, 64, 100)])
def test_kept_scores_are_bit_identical_to_the_unexcluded_call(U, I, rank, k):
    """Random lists (no row runs out of columns): every column kept in both calls has the same fp32 bits.  The kernels
    re-score a column the same way whichever candidate stream it came from; on the tensor-core route this holds for rows
    neither call re-ran exactly, so the test asserts there are none."""
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(U + k)
    Q, C = factors(U, rank, rng, rank ** -0.5), factors(I, rank, rng)
    sc = scoring.HybridScorer(dev(Q), dev(C), None, None)
    lists = [rng.choice(I, int(rng.integers(0, 3 * k)), replace=True) for _ in range(U)]
    k2 = min(256, k + max(len(x) for x in lists))
    pi, ps = sc.topk_dot(k2)
    assert sc.flagged_users(U, k2, dot=True) <= 0
    ei, es = sc.topk_dot(k, exclude=to_csr(lists))
    assert sc.flagged_users(U, k, dot=True) <= 0
    pi, ps, ei, es = pi.cpu().numpy(), ps.cpu().numpy(), ei.cpu().numpy(), es.cpu().numpy()
    compared = 0
    for u in range(U):
        bits = dict(zip(pi[u].tolist(), ps[u].view(np.int32).tolist()))
        for i, b in zip(ei[u].tolist(), es[u].view(np.int32).tolist()):
            assert i not in set(lists[u].tolist())
            if i in bits:
                assert b == bits[i], (u, i)
                compared += 1
    assert compared >= U * k * 0.9


def test_one_pass_launches_no_extrema_kernel():
    _, nat, scoring = _pkg()
    rng = np.random.default_rng(2)
    U, I, rank, k = 1024, 4096, 64, 100
    sc = scoring.HybridScorer(dev(factors(U, rank, rng)), dev(factors(I, rank, rng)), None, None)
    assert route(nat, U, I, rank, k) == "tc"
    sc.topk_dot(k)
    with launched_kernels() as names:
        sc.topk_dot(k)
    assert_ran(names, "score_tc_kernel<2,", "score_exact_blend_kernel",
               absent=("score_tc_kernel<1,", "score_exact_extrema_kernel", "score_simt_kernel<true"))


def test_topk_dot_needs_the_als_operands():
    _, _, scoring = _pkg()
    t = torch.randn(4, 8, device="cuda")
    with pytest.raises(ValueError, match="ALS operands"):
        scoring.HybridScorer(None, None, t, t).topk_dot(3)


# ---- ALSModel.recommend_for_* -----------------------------------------------------------------------------------------

def numpy_recs(m, for_users, query_ids, exclude=None):
    """Oracle for the present rows: (normalised scores [Q, n_c], s_q, candidate raw ids (ascending), per query row the
    candidate positions `exclude` removes)."""
    uf, itf = m.user_factors.cpu().numpy(), m.item_factors.cpu().numpy()
    up, ip = m.user_present.cpu().numpy(), m.item_present.cpu().numpy()
    qi, qf, cids, cf, cp = (m.user_ids, uf, m.item_ids, itf, ip) if for_users else (m.item_ids, itf, m.user_ids, uf, up)
    B, s = oracle(qf[np.searchsorted(qi, query_ids)], cf[cp])
    cand = cids[cp]
    lists = [[] for _ in query_ids]
    if exclude is not None:
        qcol, ccol = ("userId", "itemId") if for_users else ("itemId", "userId")
        pos = {int(c): j for j, c in enumerate(cand)}
        row_of = {int(q): r for r, q in enumerate(query_ids)}
        for a, b in zip(exclude[qcol].values, exclude[ccol].values):
            if int(a) in row_of and int(b) in pos:
                lists[row_of[int(a)]].append(pos[int(b)])
    return B, s, cand, [np.asarray(x, np.int64) for x in lists]


def check_recs(m, for_users, out, arrays, num, want_ids, exclude=None):
    """The DataFrame `out` and the arrays form agree with each other and with the oracle (ties: ascending raw id)."""
    qcol = "userId" if for_users else "itemId"
    q_ids, rec, rat = arrays
    assert q_ids.dtype == np.int64 and rec.dtype == np.int64 and rat.dtype == np.float32
    assert list(q_ids) == sorted(want_ids) and rec.shape == rat.shape == (len(want_ids), num)
    assert list(out.columns) == [qcol, "recommendations"] and list(out[qcol]) == list(q_ids)
    for r, lst in enumerate(out["recommendations"]):
        n = int((rec[r] >= 0).sum())
        assert (rec[r, n:] == -1).all() and np.isneginf(rat[r, n:]).all()
        assert [a for a, _ in lst] == rec[r, :n].tolist()
        assert [b for _, b in lst] == rat[r, :n].astype(np.float64).tolist()
    B, s, cand, lists = numpy_recs(m, for_users, q_ids, exclude)
    assert (np.diff(cand) > 0).all()           # candidate positions ascend with the raw id
    pos = np.where(rec >= 0, np.searchsorted(cand, rec), -1)
    check_excluding(B, lists, pos, rat / s[:, None], num, TOL)


def train_frame(rng, U=120, I=90, nnz=1500):
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    return pd.DataFrame({"userId": u * 3 + 7, "itemId": i * 5 + 1000,
                         "average_review_rating": rng.integers(1, 6, nnz).astype(float)})


def test_als_model_trained_all_four_methods():
    pkg, _, _ = _pkg()
    rng = np.random.default_rng(21)
    df = train_frame(rng)
    als = pkg.ALSModel(rank=10, max_iter=5, reg_param=0.1)
    assert als.train(df) is True
    m = als.model
    for for_users, num in ((True, 10), (False, 7), (True, 256)):
        q_ids = m.user_ids if for_users else m.item_ids
        f_all = als.recommend_for_all_users if for_users else als.recommend_for_all_items
        check_recs(m, for_users, f_all(num), f_all(num, as_arrays=True), num, q_ids)
        # subset: duplicates collapse, unknown ids are dropped, output ascending
        col = "userId" if for_users else "itemId"
        pick = list(rng.choice(q_ids, 9, replace=False))
        ds = pd.DataFrame({col: pick + pick[:4] + [-5, 10 ** 9]})
        f_sub = als.recommend_for_user_subset if for_users else als.recommend_for_item_subset
        check_recs(m, for_users, f_sub(ds, num), f_sub(ds, num, as_arrays=True), num, np.unique(pick))
    empty = als.recommend_for_user_subset(pd.DataFrame({"userId": [-1]}), 5)
    assert len(empty) == 0 and list(empty.columns) == ["userId", "recommendations"]


def test_als_model_exclude_the_training_pairs():
    pkg, _, _ = _pkg()
    rng = np.random.default_rng(22)
    df = train_frame(rng)
    als = pkg.ALSModel(rank=10, max_iter=5, reg_param=0.1)
    assert als.train(df) is True
    m = als.model
    train = df[["userId", "itemId"]]
    seen_by_user = df.groupby("userId")["itemId"].apply(set).to_dict()
    seen_by_item = df.groupby("itemId")["userId"].apply(set).to_dict()
    for for_users, num, seen, q_ids in ((True, 10, seen_by_user, m.user_ids), (False, 60, seen_by_item, m.item_ids)):
        f_all = als.recommend_for_all_users if for_users else als.recommend_for_all_items
        arrays = f_all(num, exclude=train, as_arrays=True)
        out = f_all(num, exclude=train)
        n_cand = len(m.item_ids) if for_users else len(m.user_ids)
        for q, row in zip(arrays[0], arrays[1]):
            got = [x for x in row.tolist() if x >= 0]
            assert not (set(got) & seen[q]), q
            assert len(got) == min(num, n_cand - len(seen[q]))
        check_recs(m, for_users, out, arrays, num, q_ids, exclude=train)
        # a kept rating equals the unexcluded one (same route: these calls are small)
        plain = f_all(256, as_arrays=True)
        for r in range(len(arrays[0])):
            score_of = dict(zip(plain[1][r].tolist(), plain[2][r].view(np.int32).tolist()))
            for x, b in zip(arrays[1][r].tolist(), arrays[2][r].view(np.int32).tolist()):
                if x >= 0 and x in score_of:
                    assert b == score_of[x]


def test_als_model_factors_at_tensor_core_size_with_absent_rows():
    """ALSFactors built directly (2048 users x 4096 items, rank 64: both directions take the tensor-core route), a few
    rows marked absent: they are neither queries nor candidates."""
    pkg, nat, _ = _pkg()
    from hybrid_als_twotower_recommender_b200.als_model import ALSFactors
    rng = np.random.default_rng(23)
    U, I, rank = 2048 + 40, 4096 + 40, 64
    uid = np.sort(rng.choice(10 ** 7, U, replace=False)).astype(np.int64)
    iid = np.sort(rng.choice(10 ** 7, I, replace=False)).astype(np.int64)
    up, ip = np.ones(U, bool), np.ones(I, bool)
    up[rng.choice(U, 40, replace=False)] = False
    ip[rng.choice(I, 40, replace=False)] = False
    uf, itf = factors(U, rank, rng, rank ** -0.5), factors(I, rank, rng)
    als = pkg.ALSModel(rank=rank)
    als.model = ALSFactors(rank, uid, iid, dev(uf), dev(itf), dev(up), dev(ip))
    for for_users, num in ((True, 100), (False, 25)):
        nq, nc = (up.sum(), ip.sum()) if for_users else (ip.sum(), up.sum())
        assert route(nat, int(nq), int(nc), rank, num) == "tc"
        f_all = als.recommend_for_all_users if for_users else als.recommend_for_all_items
        q_ids = uid[up] if for_users else iid[ip]
        arrays = f_all(num, as_arrays=True)
        check_recs(als.model, for_users, f_all(num), arrays, num, q_ids)
        absent = set((iid[~ip] if for_users else uid[~up]).tolist())
        assert not (set(arrays[1].ravel().tolist()) & absent)
    sub = als.recommend_for_user_subset(pd.DataFrame({"userId": uid[~up][:3].tolist() + uid[up][:2].tolist()}), 5)
    assert list(sub["userId"]) == sorted(uid[up][:2].tolist())


def test_als_model_loaded_from_a_spark_directory(tmp_path):
    """A Spark ALSModel directory read with load_model recommends what its factors give."""
    import pyarrow as pa
    import pyarrow.parquet as pq
    pkg, _, _ = _pkg()
    from hybrid_als_twotower_recommender_b200.als_model import ALSFactors
    rng = np.random.default_rng(24)
    rank, uid, iid = 12, np.arange(5, 305, 3), np.arange(1000, 1150)
    UF, IF = factors(len(uid), rank, rng), factors(len(iid), rank, rng)
    root = tmp_path / "als"
    (root / "metadata").mkdir(parents=True)
    (root / "metadata" / "part-00000").write_text(json.dumps({"class": "org.apache.spark.ml.recommendation.ALSModel",
                                                               "rank": rank}) + "\n")
    for name, ids, f in (("userFactors", uid, UF), ("itemFactors", iid, IF)):
        (root / name).mkdir()
        perm = rng.permutation(len(ids))
        pq.write_table(pa.table({"id": pa.array(ids[perm].astype(np.int32)),
                                 "features": pa.array([r.tolist() for r in f[perm]], type=pa.list_(pa.float32()))}),
                       root / name / "part-00000.snappy.parquet")
    with open(f"{root}_metadata.pkl", "wb") as fh:
        pickle.dump({"rank": rank, "max_iter": 10, "reg_param": 0.1, "global_mean": 3.5, "item_features": {}}, fh)
    loaded = pkg.ALSModel().load_model(str(root))
    assert loaded is not None
    direct = pkg.ALSModel(rank=rank)
    ones = torch.ones
    direct.model = ALSFactors(rank, uid, iid, dev(UF), dev(IF), ones(len(uid), dtype=torch.bool, device="cuda"),
                              ones(len(iid), dtype=torch.bool, device="cuda"))
    for a, b in ((loaded.recommend_for_all_users(20, as_arrays=True), direct.recommend_for_all_users(20, as_arrays=True)),
                 (loaded.recommend_for_all_items(30, as_arrays=True), direct.recommend_for_all_items(30, as_arrays=True))):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    check_recs(loaded.model, True, loaded.recommend_for_all_users(20), loaded.recommend_for_all_users(20, as_arrays=True),
               20, uid)
