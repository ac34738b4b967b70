"""GPU: nonnegative ALS half-steps (hals_als_half_step_nonnegative, the *_nnls_kernel instantiations) against the fp64
NNLS oracle from identical inputs.

Tolerances: the CUDA-core tolerances of the Cholesky route (DESIGN.md section 4): rel-L2 <= 2e-5 explicit, 5e-5 implicit;
per row the KKT conditions in fp64 on the kernel's x with tau_i = 1e-4 (|A| |x| + |b|)_i; 10 sweeps: rel-L2 <= 1e-3 on
both factor matrices and |RMSE difference| <= 1e-4.
"""
import numpy as np
import pytest
import torch

from oracle import als_oracle
from tests import nnls_oracle
from tests.util import assert_ran, draw_ratings, launched_kernels, rel_l2

pytestmark = pytest.mark.gpu
REL = {False: 2e-5, True: 5e-5}
ALPHA = 15.0
TC_KERNELS = ("als_ws64_kernel", "als_ws128_kernel", "als_tc64_kernel", "als_tc128_kernel", "als_build_solve_kernel<",
              "als_reduce_solve_kernel<")


def _mods():
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import _native, als_engine, csr
    return _native, als_engine, csr


def padded(k):
    return 16 if k <= 16 else 32 if k <= 32 else 64 if k <= 64 else 128


def nonneg_case(k, kind, implicit, seed, U=700, I=260, nnz=7000):
    """(item rows, user cols, ratings, X, U, I).  Source rows 0-49 are nonnegative, 50-99 nonpositive.  Items 0-19 only
    have positive ratings of nonpositive sources (b <= 0: all-zero rows); items 20-39 have one positive rating of a
    nonnegative source (an unconstrained solution that is already nonnegative); items I-10.. have no ratings.
    Implicit mode: ratings of both signs and zeros, and the other source rows have orthonormal columns, so that the
    Gram does not mix signs into the rows 20-39."""
    rng = np.random.default_rng(seed)
    X = als_oracle.init_factors(U, k, seed)
    if implicit:
        X[:50] = 0.1 * (1 + 0.2 * rng.random((50, k))) / np.sqrt(k)
        X[50:100] = -0.1 * np.abs(X[50:100])
        X[100:] = np.linalg.qr(rng.standard_normal((U - 100, k)))[0]
        r = (rng.gamma(1.5, 2.0, nnz) * rng.choice([1, 1, 1, -1, 0], nnz)).astype(np.float32)
    else:
        X[:50] = np.abs(X[:50])
        X[50:100] = -np.abs(X[50:100])
        r = draw_ratings(kind, nnz, rng)
    X = np.ascontiguousarray(X, np.float32)
    u, i = rng.integers(0, U, nnz), rng.integers(0, I - 10, nnz)
    m = i < 20
    u[m] = rng.integers(50, 100, m.sum())
    r[m] = np.abs(r[m]) + (r[m] == 0)
    keep = np.ones(nnz, bool)
    seen = set()
    for p in np.flatnonzero((i >= 20) & (i < 40)):
        keep[p] = i[p] not in seen
        seen.add(i[p])
    u, i, r = u[keep], i[keep], r[keep]
    m = (i >= 20) & (i < 40)
    u[m] = rng.integers(0, 50, m.sum())
    r[m] = np.abs(r[m]) + (r[m] == 0)
    return i, u, r.astype(np.float32), X, U, I


def gpu_nonneg(rows, cols, vals, n_rows, src, reg, implicit=False, alpha=ALPHA, seg_len=None, src_offset=0,
               counter=True):
    """One hals_als_half_step_nonnegative through als_engine.native_half_step.  The plan is built as the engine builds
    it (at ranks 64 / 128 it carries the tensor-core operands).  Returns (dst, plan, n_capped or None)."""
    _, als_engine, csr = _mods()
    dev = torch.device("cuda")
    shard = csr.build_csr(torch.as_tensor(rows).to(dev), torch.as_tensor(cols).to(dev), torch.as_tensor(vals).to(dev),
                          n_rows)
    k = src.shape[1]
    plan = csr.AlsPlanHandle(shard, k, seg_len, n_src=src.shape[0], implicit=implicit, alpha=alpha)
    buf = torch.empty(src.size + src_offset, dtype=torch.float32, device=dev)
    s = buf[src_offset:].view(src.shape)
    s.copy_(torch.from_numpy(np.ascontiguousarray(src)))
    dst = torch.full((n_rows, k), 7.0, dtype=torch.float32, device=dev)
    gram = None
    if implicit:
        gram = torch.empty((k, k), dtype=torch.float32, device=dev)
        ws = torch.empty(int(_mods()[0].lib().hals_gram_workspace_bytes(k)), dtype=torch.uint8, device=dev)
        als_engine.native_gram(s, gram, ws)
    capped = torch.zeros(1, dtype=torch.int32, device=dev) if counter else None
    als_engine.native_half_step(shard, plan, s, dst, k, reg, implicit, alpha, gram, nonnegative=True, n_capped=capped)
    torch.cuda.synchronize()
    return dst.cpu().numpy(), plan, (None if capped is None else int(capped.item()))


def check_case(got, rows, cols, vals, n_rows, src, reg, implicit, alpha=ALPHA, coverage=True, forward=True):
    """The KKT conditions per row, nonnegativity, zero empty rows; the rel-L2 forward tolerance unless forward=False
    (ill-conditioned cases, where fp32 rounding alone moves x by ~kappa u: the KKT check is then the criterion)."""
    rp, ci, v = als_oracle.coo_to_csr(rows, cols, vals, n_rows)
    ids, A, b = nnls_oracle.normal_equations(rp, ci, v, src, reg, implicit, alpha)
    x, _ = nnls_oracle.nnls_batched(A, b)
    want = np.zeros((n_rows, src.shape[1]))
    want[ids] = x
    if coverage:   # the case exercises the constraint
        assert (x == 0).mean() >= 0.2
        assert (~x.any(1)).sum() > 0
        unc = np.linalg.solve(A, b[..., None])[..., 0]
        assert ((unc >= 0).all(1) & x.any(1)).sum() > 0
    assert not np.isnan(got).any() and (got >= 0).all()
    empty = np.setdiff1d(np.arange(n_rows), ids)
    assert not got[empty].any(), "rows without ratings are zero"
    if forward:
        assert rel_l2(got, want) <= REL[implicit], rel_l2(got, want)
    g64 = got[ids].astype(np.float64)
    grad = np.einsum("rij,rj->ri", A, g64) - b
    tau = 1e-4 * (np.einsum("rij,rj->ri", np.abs(A), np.abs(g64)) + np.abs(b))
    pos = g64 > 0
    assert (np.abs(grad[pos]) <= tau[pos]).all(), np.max(np.abs(grad[pos]) / tau[pos])
    assert (grad[~pos] >= -tau[~pos]).all()
    return want


@pytest.mark.parametrize("kind", ["int", "decimal", "centred"])
@pytest.mark.parametrize("k", [1, 3, 10, 16, 33, 64, 100, 128])
def test_explicit_matches_nnls_oracle(k, kind):
    rows, cols, vals, X, U, I = nonneg_case(k, kind, False, k)
    with launched_kernels() as names:
        got, _, capped = gpu_nonneg(rows, cols, vals, I, X, 0.1)
    vec = k % 4 == 0
    assert_ran(names, f"als_build_solve_nnls_kernel<{padded(k)},false,{str(vec).lower()}>", absent=TC_KERNELS)
    check_case(got, rows, cols, vals, I, X, 0.1, False)
    assert capped == 0


@pytest.mark.parametrize("k", [10, 64, 128])
def test_implicit_matches_nnls_oracle(k):
    rows, cols, vals, X, U, I = nonneg_case(k, "mixed", True, 50 + k)
    assert (vals < 0).any() and (vals == 0).any()
    with launched_kernels() as names:
        got, plan, capped = gpu_nonneg(rows, cols, vals, I, X, 0.05, implicit=True)
    if k in (64, 128):
        assert plan.packed_alpha > 0, "the plan carries the tensor-core operands; they must not be used"
    assert_ran(names, f"als_build_solve_nnls_kernel<{padded(k)},true,{str(k % 4 == 0).lower()}>", absent=TC_KERNELS)
    check_case(got, rows, cols, vals, I, X, 0.05, True)
    assert capped == 0


@pytest.mark.parametrize("implicit", [False, True])
@pytest.mark.parametrize("k", [10, 64, 128])
def test_long_rows_go_through_the_nonnegative_reduce(k, implicit):
    """Rows cut into slices (seg_len 64): the partial sums meet in als_reduce_solve_nnls_kernel; bit-identical twice."""
    rows, cols, vals, X, U, I = nonneg_case(k, "decimal", implicit, 7 + k, U=2000, I=80, nnz=24000)
    reg = 0.05 if implicit else 0.1
    with launched_kernels() as names:
        got, plan, capped = gpu_nonneg(rows, cols, vals, I, X, reg, implicit=implicit, seg_len=64)
    assert plan.n_long > 0
    assert_ran(names, f"als_reduce_solve_nnls_kernel<{padded(k)}>", absent=TC_KERNELS)
    check_case(got, rows, cols, vals, I, X, reg, implicit, coverage=False)
    assert capped == 0
    again, _, _ = gpu_nonneg(rows, cols, vals, I, X, reg, implicit=implicit, seg_len=64)
    assert np.array_equal(got, again)


@pytest.mark.parametrize("implicit", [False, True])
@pytest.mark.parametrize("kp", [16, 32, 64, 128])
def test_every_instantiation_runs(kp, implicit):
    """Each padded rank, both modes, the vector gather (aligned source) and the scalar gather (source one float off
    16-byte alignment), and the reduce kernel.  At 64 / 128 the plan carries the packed operands and still no
    tensor-core kernel runs."""
    k = kp
    rows, cols, vals, X, U, I = nonneg_case(k, "decimal", implicit, 300 + kp, U=900, I=60, nnz=9000)
    reg = 0.05 if implicit else 0.1
    for off, vec in ((0, "true"), (1, "false")):
        with launched_kernels() as names:
            got, _, capped = gpu_nonneg(rows, cols, vals, I, X, reg, implicit=implicit, seg_len=96, src_offset=off)
        assert_ran(names, f"als_build_solve_nnls_kernel<{kp},{str(implicit).lower()},{vec}>",
                   f"als_reduce_solve_nnls_kernel<{kp}>", absent=TC_KERNELS)
        check_case(got, rows, cols, vals, I, X, reg, implicit, coverage=False)
        assert capped == 0


def test_argument_checks():
    nat, als_engine, csr = _mods()
    rows, cols, vals, X, U, I = nonneg_case(10, "int", False, 1)
    dev = torch.device("cuda")
    shard = csr.build_csr(torch.as_tensor(rows).to(dev), torch.as_tensor(cols).to(dev), torch.as_tensor(vals).to(dev), I)
    plan = csr.AlsPlanHandle(shard, 10, None, n_src=U)
    src = torch.from_numpy(X).to(dev)
    dst = torch.zeros((I, 10), device=dev)
    L = nat.lib()
    for reg in (0.0, -0.1):
        rc = L.hals_als_half_step_nonnegative(nat.ptr(shard.rowptr), nat.ptr(shard.colidx), nat.ptr(shard.vals), I,
                                              nat.ptr(src), U, nat.ptr(dst), 10, reg, 0, 1.0, None, plan.struct,
                                              nat.ptr(plan.workspace), plan.workspace_bytes, nat.current_stream(), None)
        assert rc == 1, "reg <= 0 must be HALS_ERR_INVALID"
    # n_capped = NULL is accepted and changes nothing
    a, _, _ = gpu_nonneg(rows, cols, vals, I, X, 0.1, counter=False)
    b, _, capped = gpu_nonneg(rows, cols, vals, I, X, 0.1)
    assert np.array_equal(a, b) and capped == 0


def _fit_data(k, kind, U, I, nnz, seed):
    rng = np.random.default_rng(seed)
    p = 1.0 / np.arange(1, I + 1) ** 0.7; p /= p.sum()
    u, i = rng.integers(0, U, nnz), rng.choice(I, nnz, p=p)
    u[:U] = np.arange(U)            # every id occurs: ALSModel's id compaction is the identity
    i[:I] = np.arange(I)
    r = draw_ratings(kind, nnz, rng)
    return u, i, r


@pytest.mark.parametrize("kind", ["int", "decimal"])
@pytest.mark.parametrize("k", [10, 64, 128])
def test_als_model_nonnegative_fit_matches_oracle(k, kind):
    import pandas as pd
    from hybrid_als_twotower_recommender_b200.als_model import ALSModel
    U, I, nnz = (1200, 400, 24000) if k == 10 else (700, 250, 14000)
    u, i, r = _fit_data(k, kind, U, I, nnz, 40 + k)
    X0 = als_oracle.init_factors(U, k, 5)
    Xo, Yo = nnls_oracle.als_fit_nnls(u, i, r, U, I, k, 10, 0.1, X0)
    m = ALSModel(rank=k, max_iter=10, reg_param=0.1, nonnegative=True)
    df = pd.DataFrame({"userId": u, "itemId": i, "average_review_rating": r})
    with launched_kernels() as names:
        assert m.train(df, init_user_factors=X0)
    assert_ran(names, f"als_build_solve_nnls_kernel<{padded(k)},false,", absent=TC_KERNELS)
    X, Y = m.model.user_factors.cpu().numpy(), m.model.item_factors.cpu().numpy()
    assert (X >= 0).all() and (Y >= 0).all() and (Xo == 0).any()
    assert rel_l2(X, Xo) <= 1e-3, rel_l2(X, Xo)
    assert rel_l2(Y, Yo) <= 1e-3, rel_l2(Y, Yo)
    assert abs(als_oracle.rmse(X, Y, u, i, r) - als_oracle.rmse(Xo, Yo, u, i, r)) <= 1e-4


@pytest.mark.parametrize("k", [10, 64])
def test_graphs_replay_the_nonnegative_half_steps(k):
    _, als_engine, _ = _mods()
    U, I, nnz = 900, 300, 15000
    u, i, r = _fit_data(k, "decimal", U, I, nnz, 3)
    X0 = als_oracle.init_factors(U, k, 2)
    eager = als_engine.AlsEngine(u, i, r, U, I, k, 0.1, nonnegative=True, seg_len=256)
    assert eager.split is None and eager.plan_Rt.n_long > 0
    eager.set_user_factors(X0)
    Xe, Ye = (t.cpu().numpy() for t in eager.fit(4))
    eng = als_engine.AlsEngine(u, i, r, U, I, k, 0.1, nonnegative=True, seg_len=256)
    eng.set_user_factors(X0)
    assert eng.enable_graphs()
    Xg, Yg = (t.cpu().numpy() for t in eng.fit(4))
    assert eng.graph_launches > 0
    assert np.array_equal(Xe, Xg) and np.array_equal(Ye, Yg)
    assert (Xg >= 0).all() and (Yg >= 0).all()
    assert eager.nonneg_capped_rows() == 0 and eng.nonneg_capped_rows() == 0


def test_hyperparameter_tuning_with_nonnegative():
    import pandas as pd
    from hybrid_als_twotower_recommender_b200.als_model import hyperparameter_tuning
    rng = np.random.default_rng(8)
    U, I, nnz = 40, 15, 400
    u, i, r = _fit_data(10, "int", U, I, nnz, 8)
    df = pd.DataFrame({"userId": u, "itemId": i, "average_review_rating": r})
    grid = [{"rank": 4, "max_iter": 3, "nonnegative": True}, {"rank": 6, "max_iter": 3, "reg_param": 0.2, "nonnegative": True}]
    best = hyperparameter_tuning(df, df.sample(120, random_state=int(rng.integers(100))), grid)
    assert best in grid
