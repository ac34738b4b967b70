"""CPU: the fp64 NNLS oracle of the nonnegative ALS half-step (KKT conditions, known answers, scipy), the sharded
nonnegative fit with that oracle injected, and ALSModel(nonnegative=True) without a GPU."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from scipy.optimize import nnls as scipy_nnls

from oracle import als_oracle
from tests import nnls_oracle

KKT_TOL = 1e-10


def _spd(k, rng, cond=None):
    if cond is None:
        Y = rng.standard_normal((3 * k + 2, k))
        return Y.T @ Y + 0.1 * np.eye(k)
    Q, _ = np.linalg.qr(rng.standard_normal((k, k)))
    return (Q * np.logspace(0, np.log10(cond), k)) @ Q.T


@pytest.mark.parametrize("k", [1, 2, 3, 10, 33, 64, 128])
def test_oracle_meets_kkt_on_random_problems(k):
    rng = np.random.default_rng(k)
    for trial in range(6):
        A = _spd(k, rng)
        b = rng.standard_normal(k) * 10 ** rng.uniform(-3, 3)
        x = nnls_oracle.nnls(A, b)
        assert (x >= 0).all()
        assert nnls_oracle.kkt_residual(A, b, x) <= KKT_TOL


@pytest.mark.parametrize("cond", [1e4, 1e8])
def test_oracle_meets_kkt_on_ill_conditioned_problems(cond):
    rng = np.random.default_rng(int(np.log10(cond)))
    for k in (5, 40, 128):
        A = _spd(k, rng, cond)
        A = (A + A.T) / 2
        b = rng.standard_normal(k)
        x = nnls_oracle.nnls(A, b)
        assert (x >= 0).all() and 0 < (x > 0).sum() < k
        assert nnls_oracle.kkt_residual(A, b, x) <= KKT_TOL


def test_oracle_degenerate_problems():
    rng = np.random.default_rng(3)
    for k in (1, 7, 64):
        A = _spd(k, rng)
        # b <= 0: x = 0 (g = -b >= 0), including exact zeros in b
        b = -np.abs(rng.standard_normal(k)); b[::3] = 0.0
        assert not nnls_oracle.nnls(A, b).any()
        # an unconstrained solution that is already nonnegative: the Cholesky solution itself
        xt = np.abs(rng.standard_normal(k)) + 0.1
        b = A @ xt
        x = nnls_oracle.nnls(A, b)
        assert np.allclose(x, als_oracle.solve_packed_cholesky(A, b), rtol=1e-12, atol=0)
        assert np.allclose(x, xt, rtol=1e-9)
    # k = 1: max(0, b / a)
    for a, b in ((2.0, 3.0), (2.0, -3.0), (0.5, 0.0), (1e-3, 7.0)):
        assert nnls_oracle.nnls(np.array([[a]]), np.array([b]))[0] == max(0.0, b / a)


@pytest.mark.parametrize("k", [3, 16, 50, 128])
def test_oracle_agrees_with_scipy_nnls(k):
    """With A = L L^T, 1/2 x^T A x - b^T x = 1/2 |L^T x - L^-1 b|^2 + const: scipy's Lawson-Hanson on (L^T, L^-1 b)
    has the same minimiser."""
    rng = np.random.default_rng(100 + k)
    for _ in range(4):
        A = _spd(k, rng)
        b = rng.standard_normal(k)
        L = np.linalg.cholesky(A)
        want, _ = scipy_nnls(L.T, np.linalg.solve(L, b), maxiter=50 * k)
        got = nnls_oracle.nnls(A, b)
        assert np.abs(got - want).max() <= 1e-9 * max(1.0, np.abs(want).max())
        assert np.array_equal(got == 0, want == 0) or np.abs(got - want).max() <= 1e-12


def test_oracle_half_step_rows_are_independent_and_constrained():
    """The batched half-step equals a row-by-row solve (a row's result does not depend on its batch) and its rows with
    ratings meet the KKT conditions of their normal equations; rows without ratings stay zero."""
    rng = np.random.default_rng(7)
    U, I, k, nnz = 60, 45, 8, 700
    u, i = rng.integers(0, U, nnz), rng.integers(0, I - 5, nnz)      # items 40..44 have no ratings
    r = ((rng.integers(10, 51, nnz) - 30) / 10).astype(np.float32)
    X = als_oracle.init_factors(U, k, 1)
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    x64 = nnls_oracle.als_half_step_nnls(rp, ci, v, X, 0.1, out64=True, batch=7)
    ids, A, b = nnls_oracle.normal_equations(rp, ci, v, X, 0.1)
    for n, j in enumerate(ids):
        assert np.array_equal(x64[j], nnls_oracle.nnls(A[n], b[n]))
        assert nnls_oracle.kkt_residual(A[n], b[n], x64[j]) <= KKT_TOL
    empty = np.setdiff1d(np.arange(I), ids)
    assert empty.size and not x64[empty].any()
    assert (x64 == 0).mean() > 0.2


# --- two ranks, gloo: the sharded nonnegative fit with the oracle injected ------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _oracle_half_step(shard, plan, src, dst_full, k, reg, implicit, alpha, gram, nonnegative=False):
    assert nonnegative, "the engine must pass nonnegative=True"
    out = nnls_oracle.als_half_step_nnls(shard.rowptr_host, shard.colidx.numpy(), shard.vals.numpy(), src.numpy(), reg,
                                         implicit, alpha)
    dst_full[shard.row_begin: shard.row_end] = torch.from_numpy(out)


def _worker(rank, world, port, case, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import als_engine
    z = np.load(case)
    U, I, k = int(z["U"]), int(z["I"]), int(z["k"])
    eng = als_engine.AlsEngine(z["u"], z["i"], z["r"], U, I, k, 0.1, implicit=bool(z["implicit"]), alpha=4.0,
                               device="cpu", dist_rank=rank, world=world, half_step=_oracle_half_step, make_plans=False,
                               nonnegative=True)
    assert eng.split is None and eng.nonneg_capped_rows() == 0
    eng.set_user_factors(z["X0"])
    X, Y = eng.fit(3)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), X=X.numpy(), Y=Y.numpy())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("implicit", [False, True])
def test_two_rank_nonnegative_fit_equals_single_process(tmp_path, implicit):
    rng = np.random.default_rng(6)
    U, I, k, nnz = 91, 57, 6, 1400
    p = 1.0 / np.arange(1, I + 1); p /= p.sum()
    u, i = rng.integers(0, U, nnz), rng.choice(I, nnz, p=p)
    r = ((rng.integers(10, 51, nnz) - 30) / 10).astype(np.float32)
    X0 = als_oracle.init_factors(U, k, 3)
    case = str(tmp_path / "case.npz")
    np.savez(case, u=u, i=i, r=r, U=U, I=I, k=k, X0=X0, implicit=implicit)
    mp.spawn(_worker, args=(2, _free_port(), case, str(tmp_path)), nprocs=2, join=True)
    Xo, Yo = nnls_oracle.als_fit_nnls(u, i, r, U, I, k, 3, 0.1, X0, implicit=implicit, alpha=4.0)
    assert (Xo >= 0).all() and (Yo >= 0).all() and (Xo == 0).mean() > 0.1
    for q in range(2):
        o = np.load(tmp_path / f"rank{q}.npz")
        assert np.array_equal(o["X"], Xo) and np.array_equal(o["Y"], Yo)


def test_als_model_nonnegative_train_without_gpu(capsys):
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the GPU tests cover ALSModel(nonnegative=True)")
    import pandas as pd
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200.als_model import ALSModel
    m = ALSModel(rank=4, max_iter=2, nonnegative=True)
    assert m.nonnegative is True
    df = pd.DataFrame({"userId": [1, 2, 2], "itemId": [10, 10, 11], "average_review_rating": [4.0, 3.5, 2.0]})
    assert m.train(df) is False
    assert "error" in capsys.readouterr().out.lower()
    with pytest.raises(TypeError):
        ALSModel(4, 2, 0.1, "drop", False)      # keyword-only, like implicit_prefs / alpha / seed
