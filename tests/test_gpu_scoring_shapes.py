"""Hybrid top-k at the edges of what the C ABI accepts, on both paths (CUDA-core and tensor-core), against a dense
fp64 reference: operand widths from 1 to 128 + 64 and single-model calls, strided and unaligned operand views, the
degenerate and one-sided blend weights, an item order that puts the whole answer into one candidate stream, an exact
re-run of more than 2048 users, user slabs and repeated calls.

Tolerances are those of test_gpu_scoring.py (1e-5 on blended scores, 1e-5 / 2e-5 on the extrema) unless a test says
why its input needs more."""
import numpy as np
import pytest
import torch

from tests.test_gpu_exclude import check_excluding, to_csr
from tests.test_gpu_scoring import dense_blend, dev
from tests.util import check_topk_against_dense

pytestmark = pytest.mark.gpu
TOL = 1e-5

# One shape per path: SIMT takes calls with fewer than 2048 items; the tensor-core path needs >= 2048 items and
# >= 2^22 (user, item) pairs.
SIMT_SHAPE = (70, 1500)
TC_SHAPE = (256, 16384)
SHAPES = {"simt": SIMT_SHAPE, "tc": TC_SHAPE}


def _pkg():
    from hybrid_als_twotower_recommender_b200 import _native, scoring
    return _native, scoring


def operands(U, I, ka, kt, seed):
    rng = np.random.default_rng(seed)
    Ua = rng.normal(0, max(ka, 1) ** -0.5, (U, ka)).astype(np.float32)
    Ia = rng.normal(0, 1, (I, ka)).astype(np.float32)
    Ut, It = rng.normal(0, 1, (U, kt)).astype(np.float32), rng.normal(0, 1, (I, kt)).astype(np.float32)
    return Ua, Ia, Ut, It


def assert_path(nat, path, U, I, ka, kt, k):
    off = int(nat.lib().hals_score_flag_counter_offset(U, I, ka, kt, k))
    if path == "tc":
        assert off >= 0, "expected the tensor-core path"
    else:
        assert off < 0, "expected the CUDA-core path"


def want_extrema(Sa, St):
    return np.stack([Sa.min(1), Sa.max(1), St.min(1), St.max(1)], 1)


def extrema_tol(path):
    return 2e-5 if path == "tc" else 1e-5


# ---------------------------------------------------------------------------------------------- 1. operand widths
@pytest.mark.parametrize("path", ["simt", "tc"])
@pytest.mark.parametrize("ka,kt", [(ka, kt) for ka in (1, 63, 65, 100, 127, 128) for kt in (1, 33, 64)])
def test_operand_widths(path, ka, kt):
    """Every ALS width class (one and two 64-wide K blocks, padded and full) against every tower width class,
    kt = 64 with ka = 128 being the widest operand the kernels take (Kp = 192)."""
    nat, scoring = _pkg()
    U, I = SHAPES[path]
    k = 10
    assert_path(nat, path, U, I, ka, kt, k)
    Ua, Ia, Ut, It = operands(U, I, ka, kt, 1000 * ka + kt)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    ex = sc.extrema().cpu().numpy()
    B, Sa, St = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    assert np.allclose(ex, want_extrema(Sa, St), rtol=1e-5, atol=extrema_tol(path))
    idx, s = sc.recommend(k, 0.8, 0.2)
    check_topk_against_dense(B, idx.cpu().numpy(), s.cpu().numpy(), k, TOL)


@pytest.mark.parametrize("path", ["simt", "tc"])
@pytest.mark.parametrize("missing", ["als", "tower"])
def test_single_model_call(path, missing):
    """HybridScorer with None for one model: ka = 0 or kt = 0.  The missing model's extrema are exactly (0, 0)
    and the blend is the min-max of the other model times its weight."""
    nat, scoring = _pkg()
    U, I = SHAPES[path]
    ka, kt = (0, 50) if missing == "als" else (64, 0)
    k = 10
    assert_path(nat, path, U, I, ka, kt, k)
    Ua, Ia, Ut, It = operands(U, I, ka, kt, 7 + ka)
    if missing == "als":
        sc = scoring.HybridScorer(None, None, dev(Ut), dev(It))
    else:
        sc = scoring.HybridScorer(dev(Ua), dev(Ia), None, None)
    ex = sc.extrema().cpu().numpy()
    B, Sa, St = dense_blend(Ua, Ia, Ut, It, 0.3, 0.7)
    gone = slice(0, 2) if missing == "als" else slice(2, 4)
    assert (ex[:, gone] == 0).all(), "a missing model's extrema must be exactly (0, 0)"
    assert np.allclose(ex, want_extrema(Sa, St), rtol=1e-5, atol=extrema_tol(path))
    idx, s = sc.recommend(k, 0.3, 0.7)
    check_topk_against_dense(B, idx.cpu().numpy(), s.cpu().numpy(), k, TOL)
    assert s.cpu().numpy()[:, 0].max() <= (0.7 if missing == "als" else 0.3) + 1e-6


# -------------------------------------------------------------------------------- 2. row strides, unaligned views
def _abi_call(nat, Ua, Ia, Ut, It, ka, kt, k, w, excl=None):
    """hals_score_extrema + hals_score_blend_topk(_excluding) on the given (possibly strided) 2-D views."""
    L = nat.lib()
    U, I = Ua.shape[0], Ia.shape[0]
    ws = torch.empty(int(L.hals_score_workspace_bytes(U, I, ka, kt, k)), dtype=torch.uint8, device="cuda")
    ex = torch.empty((U, 4), dtype=torch.float32, device="cuda")
    ops = (nat.ptr(Ua), Ua.stride(0), nat.ptr(Ia), Ia.stride(0), ka, nat.ptr(Ut), Ut.stride(0), nat.ptr(It),
           It.stride(0), kt, U, I)
    tail = (nat.ptr(ws), ws.numel(), nat.current_stream())
    nat.check(L.hals_score_extrema(*ops, nat.ptr(ex), *tail), "hals_score_extrema")
    idx = torch.empty((U, k), dtype=torch.int32, device="cuda")
    sc = torch.empty((U, k), dtype=torch.float32, device="cuda")
    head = (*ops, nat.ptr(ex), w[0], w[1], k, 0, nat.ptr(idx), nat.ptr(sc))
    if excl is None:
        nat.check(L.hals_score_blend_topk(*head, *tail), "hals_score_blend_topk")
    else:
        nat.check(L.hals_score_blend_topk_excluding(*head, nat.ptr(excl[0]), nat.ptr(excl[1]), *tail),
                  "hals_score_blend_topk_excluding")
    torch.cuda.synchronize()
    return ex.cpu().numpy(), idx.cpu().numpy(), sc.cpu().numpy()


@pytest.mark.parametrize("path", ["simt", "tc"])
@pytest.mark.parametrize("ka,kt,pad,excluding", [(63, 33, 5, False), (100, 50, 3, False), (65, 64, 1, True)])
def test_strided_unaligned_operands_are_bit_identical(path, ka, kt, pad, excluding):
    """Operands as column slices M[:, :ka] and M[:, ka:ka+kt] of wider fp32 tables: row stride != width, and with
    ka % 4 != 0 the tower operand's base is not 16-byte aligned.  Same arithmetic, other addresses: extrema, indices
    and scores must equal those of the same call on contiguous copies bit for bit."""
    nat, _ = _pkg()
    U, I = SHAPES[path]
    k = 20
    assert_path(nat, path, U, I, ka, kt, k)
    rng = np.random.default_rng(ka + pad)
    Mu = torch.from_numpy(rng.normal(0, 0.15, (U, ka + kt + pad)).astype(np.float32)).cuda()
    Mi = torch.from_numpy(rng.normal(0, 1, (I, ka + kt + pad)).astype(np.float32)).cuda()
    Ua, Ut, Ia, It = Mu[:, :ka], Mu[:, ka:ka + kt], Mi[:, :ka], Mi[:, ka:ka + kt]
    assert Ua.stride(0) == ka + kt + pad and not Ut.is_contiguous()
    excl = None
    if excluding:
        lists = [rng.choice(I, 30, replace=False) for _ in range(U)]
        excl = to_csr(lists)
    got = _abi_call(nat, Ua, Ia, Ut, It, ka, kt, k, (0.8, 0.2), excl)
    want = _abi_call(nat, Ua.contiguous(), Ia.contiguous(), Ut.contiguous(), It.contiguous(), ka, kt, k, (0.8, 0.2),
                     excl)
    for g, w_, what in zip(got, want, ("extrema", "indices", "scores")):
        assert np.array_equal(g, w_), what
    B, Sa, St = dense_blend(*(t.cpu().numpy() for t in (Ua, Ia, Ut, It)), 0.8, 0.2)
    assert np.allclose(got[0], want_extrema(Sa, St), rtol=1e-5, atol=extrema_tol(path))
    if excluding:
        check_excluding(B, lists, got[1], got[2], k, TOL)
    else:
        check_topk_against_dense(B, got[1], got[2], k, TOL)


# ------------------------------------------------------------------------------------------------------ 3. weights
@pytest.mark.parametrize("path", ["simt", "tc"])
@pytest.mark.parametrize("w", [(1.0, 0.0), (0.0, 1.0), (0.5, 0.5), (0.0, 0.0)])
def test_blend_weights(path, w):
    """(1, 0) and (0, 1) are what evaluate_models_batch passes: one half of the folded user operand is zero, and so is
    its share of eps.  Items come in exact duplicates (ALS rows in pairs, tower rows in triples), so the weighted
    model's scores tie exactly and ties must resolve by index, also at the k-th place.  (0, 0): every blend is 0 and
    the answer is items 0..k-1."""
    nat, scoring = _pkg()
    U, I = SHAPES[path]
    ka, kt, k = 32, 16, 25
    assert_path(nat, path, U, I, ka, kt, k)
    Ua, Ia, Ut, It = operands(U, I, ka, kt, 5)
    Ia, It = np.ascontiguousarray(Ia[np.arange(I) // 2]), np.ascontiguousarray(It[np.arange(I) // 3])
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    sc.extrema()
    idx, s = sc.recommend(k, *w)
    idx, s = idx.cpu().numpy(), s.cpu().numpy()
    if w == (0.0, 0.0):
        assert (idx == np.arange(k)).all() and (s == 0).all()
        print(f"\n{path} (0, 0): {sc.flagged_users(U, k)} users re-run exactly")
        return
    B, _, _ = dense_blend(Ua, Ia, Ut, It, *w)
    check_topk_against_dense(B, idx, s, k, TOL)
    group = {(1.0, 0.0): 2, (0.0, 1.0): 3}.get(w)
    if group:                                   # a listed item's lower-indexed twins (same score) are listed too
        for u in range(U):
            listed = set(idx[u].tolist())
            for i in idx[u]:
                assert all(j in listed for j in range(i - i % group, i)), (u, i)


# ----------------------------------------------------------------------------- 4. top-k sizes, adversarial order
def test_answer_concentrated_in_one_candidate_stream():
    """16 users x 262144 items: one user tile and 1024 item tiles, so make_plan takes 64 splits of 16 tiles (on any
    GPU with >= 64 SMs) and candidate stream (split 0, part 0) owns the first quarter (64 columns) of each of the
    first 16 tiles.  The 256 best items of every user are placed there; at k = 256 a stream keeps only 128, so the
    verification must flag the users and the exact re-run must produce the answer.  This geometry is that of the
    default four-part build (HALS_SCORE_PARTS=4): a two-part build keeps 256 per stream, the answer then fits in one
    stream and nothing needs flagging."""
    nat, scoring = _pkg()
    U, I, ka, kt, k = 16, 262144, 32, 16, 256
    assert_path(nat, "tc", U, I, ka, kt, k)
    rng = np.random.default_rng(4)
    da, dt = np.ones(ka) / ka ** 0.5, np.ones(kt) / kt ** 0.5
    Ua = (da + 0.2 * rng.normal(0, ka ** -0.5, (U, ka))).astype(np.float32)
    Ut = (dt + 0.2 * rng.normal(0, kt ** -0.5, (U, kt))).astype(np.float32)
    Ia, It = rng.normal(0, 1, (I, ka)).astype(np.float32), rng.normal(0, 1, (I, kt)).astype(np.float32)
    stream00 = (256 * np.arange(16)[:, None] + np.arange(64)[None, :]).reshape(-1)     # 1024 columns
    best = np.sort(rng.choice(stream00, k, replace=False))
    Ia[best] = (8 * da + rng.normal(0, 0.3, (k, ka))).astype(np.float32)
    It[best] = (8 * dt + rng.normal(0, 0.3, (k, kt))).astype(np.float32)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    sc.extrema()
    idx, s = sc.recommend(k, 0.5, 0.5)
    idx, s = idx.cpu().numpy(), s.cpu().numpy()
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.5, 0.5)
    assert all(set(np.argsort(-B[u])[:k].tolist()) == set(best.tolist()) for u in range(U)), "input construction"
    assert sc.flagged_users(U, k) > 0, "one stream cannot hold the answer: the verification must flag"
    check_topk_against_dense(B, idx, s, k, TOL)


# ------------------------------------------------------------------------------- 5. exact re-run past 2048 users
def bf16_inseparable(U, I, ka, kt, seed):
    """Items that differ by less than bf16 resolution (test_gpu_scoring's fallback construction)."""
    rng = np.random.default_rng(seed)
    base_a, base_t = rng.normal(0, 1, (1, ka)), rng.normal(0, 1, (1, kt))
    Ia = (base_a + 3e-3 * rng.normal(0, 1, (I, ka))).astype(np.float32)
    It = (base_t + 3e-3 * rng.normal(0, 1, (I, kt))).astype(np.float32)
    Ua, Ut = rng.normal(0, 1, (U, ka)).astype(np.float32), rng.normal(0, 1, (U, kt)).astype(np.float32)
    return Ua, Ia, Ut, It


def test_exact_rerun_of_more_than_2048_users():
    """The SIMT re-run item-splits the first 2048 flagged users and runs the rest in a separate unsplit launch whose
    candidate rows follow the list region.  Score ranges are ~1e-2 here, so fp32 cancellation in
    (s - min) / (max - min) costs ~1e-5 of the [0, 1] range: scores are checked to 2e-4, as in test_gpu_scoring."""
    nat, scoring = _pkg()
    U, I, ka, kt, k = 3000, 6000, 16, 8, 10
    assert_path(nat, "tc", U, I, ka, kt, k)
    Ua, Ia, Ut, It = bf16_inseparable(U, I, ka, kt, 3)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    ex = sc.extrema().cpu().numpy()
    n_ex = sc.flagged_users(U, 0)
    B, Sa, St = dense_blend(Ua, Ia, Ut, It, 0.8, 0.2)
    assert n_ex > 0, "pass 1 must re-run some users exactly"
    assert np.allclose(ex, want_extrema(Sa, St), rtol=1e-5, atol=1e-5)
    idx, s = sc.recommend(k, 0.8, 0.2)
    n_top = sc.flagged_users(U, k)
    print(f"\nflagged: extrema {n_ex}, top-k {n_top} of {U}")
    assert n_top > 2048, "the re-run must overflow the item-split region"
    check_topk_against_dense(B, idx.cpu().numpy(), s.cpu().numpy(), k, 2e-4)


# ----------------------------------------------------------------------------------------- 6. slabs, determinism
@pytest.mark.parametrize("excluding", [False, True])
def test_user_slabs_match_the_whole_call(excluding):
    """recommend(k, w, u0, u1) over three slabs (operand pointers and the exclusion rowptr offset by u0) against one
    whole call and the oracle.  Split plans differ with the slab size and flagged users are rescored by the SIMT
    kernel, so last bits may differ: same items except near-ties, scores within 1e-6."""
    nat, scoring = _pkg()
    U, I, ka, kt, k = 600, 24576, 64, 50, 30
    bounds = [0, 200, 400, 600]
    for a, b in zip(bounds, bounds[1:]):
        assert_path(nat, "tc", b - a, I, ka, kt, k)
    Ua, Ia, Ut, It = operands(U, I, ka, kt, 17)
    rng = np.random.default_rng(17)
    lists = excl = None
    if excluding:
        B0, _, _ = dense_blend(Ua, Ia, Ut, It, 0.2, 0.8)
        top = np.argsort(-B0, axis=1)[:, :k]
        # part of each user's own answer plus random items
        lists = [np.concatenate([top[u, rng.choice(k, 10, replace=False)], rng.choice(I, 40)]) for u in range(U)]
        excl = to_csr(lists)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    whole_i, whole_s = (t.cpu().numpy() for t in sc.recommend(k, 0.2, 0.8, exclude=excl))
    parts = [sc.recommend(k, 0.2, 0.8, a, b, exclude=excl) for a, b in zip(bounds, bounds[1:])]
    slab_i = np.concatenate([p[0].cpu().numpy() for p in parts])
    slab_s = np.concatenate([p[1].cpu().numpy() for p in parts])
    B, _, _ = dense_blend(Ua, Ia, Ut, It, 0.2, 0.8)
    assert np.abs(slab_s - whole_s).max() <= 1e-6
    diff = slab_i != whole_i
    for u, p in zip(*np.nonzero(diff)):
        assert abs(B[u, slab_i[u, p]] - B[u, whole_i[u, p]]) <= TOL, (u, p)
    if excluding:
        check_excluding(B, lists, slab_i, slab_s, k, TOL)
    else:
        check_topk_against_dense(B, slab_i, slab_s, k, TOL)


def test_repeated_tensor_core_call_is_bit_identical():
    """An input that flags users (the bf16 construction): extrema, flag counts, indices and scores of three repeated
    calls are bit-identical -- the atomics are order-independent and every list is ordered by (score, index)."""
    nat, scoring = _pkg()
    U, I, ka, kt, k = 800, 6000, 16, 8, 50
    assert_path(nat, "tc", U, I, ka, kt, k)
    Ua, Ia, Ut, It = bf16_inseparable(U, I, ka, kt, 9)
    sc = scoring.HybridScorer(dev(Ua), dev(Ia), dev(Ut), dev(It))
    runs = []
    for _ in range(3):
        ex = sc.extrema()
        n_ex = sc.flagged_users(U, 0)
        idx, s = sc.recommend(k, 0.8, 0.2)
        runs.append((ex.cpu().numpy(), idx.cpu().numpy(), s.cpu().numpy(), n_ex, sc.flagged_users(U, k)))
    assert runs[0][4] > 0, "the input must trigger the exact re-run"
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert np.array_equal(a, b)
