"""GPU parity: the CUDA ALS path (through the C ABI) against the CPU oracle.

Tolerances (fp32 kernels vs Spark-faithful fp64 accumulation, stated per SURVEY.md 8c):
  one half-step from identical inputs : rel-L2 <= 2e-5, max-abs <= 1e-4 * max|x|
  10 sweeps from identical init       : rel-L2 <= 1e-3 on both factor matrices, |RMSE diff| <= 1e-4
"""
import os

import numpy as np
import pytest
import torch

from oracle import als_oracle, c_oracle
from tests.util import assert_ran, draw_ratings, launched_kernels, rel_l2

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
HS_REL, HS_ABS = 2e-5, 1e-4
# Implicit feedback: the weights c = alpha |r| (up to several hundred) worsen the conditioning of the normal equations.
# fp32 CUDA-core build: 5e-5.  Ranks 64 / 128 on the tensor cores: the rows rescaled by sqrt(c) are re-split into bf16 hi/lo
# (16-17 significant bits, twice the representation error of the explicit build): 2e-4.
IMPL_TOL = {False: dict(rel=5e-5, ab=3e-4), True: dict(rel=2e-4, ab=1e-3)}


def _mods():
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import als_engine, csr
    return als_engine, csr


def gpu_half_step(rows, cols, vals, n_rows, src, reg, implicit=False, alpha=1.0, seg_len=None, packed=True,
                  plan_implicit=None, src_offset=0):
    """One hals_als_half_step.  packed=False clears the plan's packed ratings (ranks 64 / 128: the round-1 kernels
    that split the fp32 ratings themselves); plan_implicit=False with implicit=True calls implicit mode with a plan
    built for explicit feedback (the CUDA-core kernel at every rank); src_offset > 0 places the source factors that
    many floats into a larger buffer (not 16-byte aligned: the CUDA-core kernel's scalar gather; CUDA-core ranks only,
    the tensor-core kernels and the rank-64 / 128 Gram assume aligned rows)."""
    als_engine, csr = _mods()
    dev = torch.device("cuda")
    shard = csr.build_csr(torch.as_tensor(rows).to(dev), torch.as_tensor(cols).to(dev),
                          torch.as_tensor(vals).to(dev), n_rows)
    k = src.shape[1]
    plan_implicit = implicit if plan_implicit is None else plan_implicit
    plan = csr.AlsPlanHandle(shard, k, seg_len, n_src=src.shape[0], implicit=plan_implicit, alpha=alpha)
    if not packed:
        plan.struct.vals_hl = None
    buf = torch.empty(src.size + src_offset, dtype=torch.float32, device=dev)
    s = buf[src_offset:].view(src.shape)
    s.copy_(torch.from_numpy(np.ascontiguousarray(src)))
    dst = torch.full((n_rows, k), 7.0, dtype=torch.float32, device=dev)   # poison: rows must be overwritten
    gram = None
    if implicit:
        gram = torch.empty((k, k), dtype=torch.float32, device=dev)
        ws = torch.empty(int(_nat().lib().hals_gram_workspace_bytes(k)), dtype=torch.uint8, device=dev)
        als_engine.native_gram(s, gram, ws)
    als_engine.native_half_step(shard, plan, s, dst, k, reg, implicit, alpha, gram)
    torch.cuda.synchronize()
    return dst.cpu().numpy(), plan


def _nat():
    from hybrid_als_twotower_recommender_b200 import _native
    return _native


def synth(U, I, nnz, seed, skew=False):
    rng = np.random.default_rng(seed)
    if skew:
        p = 1.0 / np.arange(1, I + 1); p /= p.sum()
        i = rng.choice(I, nnz, p=p)
    else:
        i = rng.integers(0, I, nnz)
    u = rng.integers(0, U, nnz)
    r = rng.integers(1, 6, nnz).astype(np.float32)
    return u, i, r


def assert_close(got, want, rel=HS_REL, ab=HS_ABS, floor=1.0):
    """rel-L2 <= rel and max-abs <= ab * max(floor, max|want|); floor=0 makes both bounds purely relative."""
    assert np.isfinite(got).all()
    assert rel_l2(got, want) <= rel, rel_l2(got, want)
    assert np.abs(got - want).max() <= ab * max(floor, np.abs(want).max()), np.abs(got - want).max()


def half_step_kernel(k, implicit, aligned=True):
    """Name (as launched_kernels reports it) of the main kernel hals_als_half_step runs for a default plan."""
    if k in (64, 128):
        return f"als_ws{k}_kernel"
    kp = 16 if k <= 16 else 32 if k <= 32 else 64 if k <= 64 else 128
    vec = k % 4 == 0 and aligned
    return f"als_build_solve_kernel<{kp},{str(implicit).lower()},{str(vec).lower()}>"


# odd ranks take the scalar gather; 33 / 127 sit one past / one below a padded-rank bucket
@pytest.mark.parametrize("k", [1, 2, 3, 10, 16, 20, 32, 33, 50, 64, 100, 127, 128])
def test_half_step_explicit_matches_oracle(k):
    U, I, nnz = 700, 300, 9000
    u, i, r = synth(U, I, nnz, k)
    X = als_oracle.init_factors(U, k, 1)
    with launched_kernels() as names:
        got, _ = gpu_half_step(i, u, r, I, X, 0.1)
    assert_ran(names, half_step_kernel(k, False))
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    assert_close(got, c_oracle.als_half_step(rp, ci, v, X, 0.1))


# 16 / 32 / 100: the vectorised-gather implicit instantiations at padded ranks 16, 32 and 128
@pytest.mark.parametrize("k", [10, 16, 32, 64, 100, 128])
def test_half_step_implicit_matches_oracle(k):
    U, I, nnz = 500, 260, 6000
    rng = np.random.default_rng(k)
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    r = (rng.geometric(0.4, nnz) * rng.choice([1, 1, 1, -1, 0], nnz)).astype(np.float32)
    X = als_oracle.init_factors(U, k, 3)
    with launched_kernels() as names:
        got, _ = gpu_half_step(i, u, r, I, X, 0.05, implicit=True, alpha=40.0)
    assert_ran(names, half_step_kernel(k, True))
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    want = c_oracle.als_half_step(rp, ci, v, X, 0.05, implicit=True, alpha=40.0)
    assert_close(got, want, **IMPL_TOL[k in (64, 128)])


@pytest.mark.parametrize("k", [10, 20, 64, 100, 128])
def test_implicit_long_rows_and_mixed_signs(k):
    """Implicit feedback with sliced rows, ratings of both signs, zeros and non-integer weights.  Ranks 64 / 128: the
    tensor-core build with rows rescaled by sqrt(c), the Gram added in the solver / the long-row reduce; other ranks:
    the CUDA-core kernel, whose long-row reduce (als_reduce_solve_kernel) adds the Gram."""
    U, I, nnz = 2500, 60, 24000
    rng = np.random.default_rng(11)
    p = 1.0 / np.arange(1, I + 1); p /= p.sum()
    i, u = rng.choice(I, nnz, p=p), rng.integers(0, U, nnz)
    r = (rng.gamma(1.5, 2.0, nnz) * rng.choice([1, 1, 1, -1, 0], nnz)).astype(np.float32)
    X = als_oracle.init_factors(U, k, 4)
    with launched_kernels() as names:
        got, plan = gpu_half_step(i, u, r, I, X, 0.05, implicit=True, alpha=15.0, seg_len=96)
    assert plan.n_long > 0
    assert_ran(names, half_step_kernel(k, True), *(() if k in (64, 128) else ("als_reduce_solve_kernel<",)))
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    want = c_oracle.als_half_step(rp, ci, v, X, 0.05, implicit=True, alpha=15.0)
    assert_close(got, want, **IMPL_TOL[k in (64, 128)])
    again, _ = gpu_half_step(i, u, r, I, X, 0.05, implicit=True, alpha=15.0, seg_len=96)
    assert np.array_equal(got, again)


@pytest.mark.parametrize("k,seg", [(10, 64), (64, 64), (128, 96), (64, 4096)])
def test_long_rows_are_sliced_deterministically(k, seg):
    U, I, nnz = 3000, 40, 30000            # ~750 ratings per item row, Zipf-skewed
    u, i, r = synth(U, I, nnz, 5, skew=True)
    X = als_oracle.init_factors(U, k, 2)
    got, plan = gpu_half_step(i, u, r, I, X, 0.1, seg_len=seg)
    if seg < 4096:
        assert plan.n_long > 0 and plan.n_slots > plan.n_long
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    assert_close(got, c_oracle.als_half_step(rp, ci, v, X, 0.1))
    again, _ = gpu_half_step(i, u, r, I, X, 0.1, seg_len=seg)
    assert np.array_equal(got, again), "bitwise reproducible (no float atomics)"


@pytest.mark.parametrize("k", [64, 128])
def test_many_slices_use_the_two_level_slot_reduction(k):
    """A row cut into more than 256 slices (seg_len 32): slot sums go through both pre-sum levels."""
    U, I, nnz = 4000, 6, 60000             # ~10k ratings per item row -> ~310 slices each
    u, i, r = synth(U, I, nnz, 11, skew=False)
    X = als_oracle.init_factors(U, k, 3)
    got, plan = gpu_half_step(i, u, r, I, X, 0.1, seg_len=32)
    assert plan.n_long > 0 and int(plan.host["long_nseg"][: plan.n_long].max()) > 256
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    assert_close(got, c_oracle.als_half_step(rp, ci, v, X, 0.1))
    again, _ = gpu_half_step(i, u, r, I, X, 0.1, seg_len=32)
    assert np.array_equal(got, again)


def test_empty_rows_duplicates_and_single_rating():
    k = 10
    X = als_oracle.init_factors(50, k, 0)
    u = np.array([3, 3, 3, 7, 7, 49, 12, 12]); i = np.array([0, 0, 0, 2, 5, 5, 9, 9])   # duplicates (3,0) x3, (12,9) x2
    r = np.array([5, 5, 1, 2, 3, 4, 1, 1], np.float32)
    got, _ = gpu_half_step(i, u, r, 12, X, 0.1)
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, 12)
    want = als_oracle.als_half_step_loops(rp, ci, v, X, 0.1)
    assert_close(got, want)
    for j in (1, 3, 4, 6, 7, 8, 10, 11):
        assert not got[j].any(), "rows without ratings are zero"
    y = X[7].astype(np.float64)
    assert np.allclose(got[2], 2.0 * y / (y @ y + 0.1), atol=1e-6)    # closed form, one rating


def test_fit_10_sweeps_matches_oracle_fixture():
    als_engine, _ = _mods()
    z = np.load(os.path.join(G, "als_oracle_cases.npz"))
    eng = als_engine.AlsEngine(z["mid_u"], z["mid_i"], z["mid_r"], 200, 150, 10, 0.1)
    eng.set_user_factors(z["mid_X0"])
    X, Y = eng.fit(10)
    assert rel_l2(X.cpu().numpy(), z["mid_X"]) <= 1e-3
    assert rel_l2(Y.cpu().numpy(), z["mid_Y"]) <= 1e-3
    assert abs(eng.rmse(z["mid_u"], z["mid_i"], z["mid_r"]) - float(z["mid_rmse"])) <= 1e-4
    eng2 = als_engine.AlsEngine(z["mid_u"], z["mid_i"], z["mid_r_implicit"], 200, 150, 10, 0.05, implicit=True, alpha=40.0)
    eng2.set_user_factors(z["mid_X0"])
    Xi, Yi = eng2.fit(5)
    assert rel_l2(Xi.cpu().numpy(), z["mid_Xi"]) <= 1e-3 and rel_l2(Yi.cpu().numpy(), z["mid_Yi"]) <= 1e-3


def test_config1_amazon_shape_rank10_10_iters():
    """BASELINE config 1: 10k x 10k, ~10k ratings, rank 10, maxIter 10, regParam 0.1."""
    als_engine, _ = _mods()
    rng = np.random.default_rng(1)
    pairs = rng.choice(10_000 * 10_000, 10_000, replace=False)
    u, i = pairs // 10_000, pairs % 10_000
    r = rng.integers(1, 6, 10_000).astype(np.float32)
    X0 = als_oracle.init_factors(10_000, 10, 1)
    Xo, Yo = als_oracle.als_fit(u, i, r, 10_000, 10_000, 10, 10, 0.1, X0, half_step=c_oracle.als_half_step)
    eng = als_engine.AlsEngine(u, i, r, 10_000, 10_000, 10, 0.1)
    eng.set_user_factors(X0)
    X, Y = eng.fit(10)
    assert rel_l2(X.cpu().numpy(), Xo) <= 1e-3 and rel_l2(Y.cpu().numpy(), Yo) <= 1e-3
    assert abs(eng.rmse(u, i, r) - als_oracle.rmse(Xo, Yo, u, i, r)) <= 1e-4


@pytest.mark.parametrize("kind", ["int", "decimal"])
@pytest.mark.parametrize("k", [64, 128])
def test_fit_10_sweeps_on_the_tensor_core_ranks(k, kind):
    """Ten full sweeps through the tcgen05 kernels (rank 64: warp-specialised kernel; rank 128) on a Zipf-skewed shape
    with sliced long rows, against the fp64-accumulating C oracle from identical initial factors.  Decimal ratings are
    mostly not bf16 numbers: they exercise the low rating part of the engine's split-form half-steps and the RMSE.
    Tolerance (north star: "factors and RMSE within a stated fp32 tolerance"): rel-L2 <= 1e-3 on both factor
    matrices, |RMSE difference| <= 1e-4.  (Parity unpinned: the oracle restates Spark MLlib 3.5.1, SURVEY App. A.)"""
    als_engine, _ = _mods()
    U, I, nnz = 6000, 900, 240_000
    u, i, r = synth(U, I, nnz, 21 + k, skew=True)
    if kind != "int":
        r = draw_ratings(kind, nnz, np.random.default_rng(k))
    X0 = als_oracle.init_factors(U, k, 5)
    Xo, Yo = als_oracle.als_fit(u, i, r, U, I, k, 10, 0.1, X0, half_step=c_oracle.als_half_step)
    eng = als_engine.AlsEngine(u, i, r, U, I, k, 0.1, seg_len=1024)
    assert eng.plan_Rt.n_long > 0, "the item half must exercise the slot reduction"
    eng.set_user_factors(X0)
    X, Y = eng.fit(10)
    X, Y = X.cpu().numpy(), Y.cpu().numpy()
    assert np.isfinite(X).all() and np.isfinite(Y).all()
    assert rel_l2(X, Xo) <= 1e-3, rel_l2(X, Xo)
    assert rel_l2(Y, Yo) <= 1e-3, rel_l2(Y, Yo)
    assert abs(eng.rmse(u, i, r) - als_oracle.rmse(Xo, Yo, u, i, r)) <= 1e-4
    # a second fit from the same start is bit-identical (static work split, slot sums in a fixed order)
    eng.set_user_factors(X0)
    X2, Y2 = eng.fit(10)
    assert np.array_equal(X2.cpu().numpy(), X) and np.array_equal(Y2.cpu().numpy(), Y)


def test_rank64_kernels_agree():
    """The warp-specialised rank-64 kernel (default) and the round-1 kernel (plan without chunk table / packed ratings)
    build the same normal equations and must agree to solver rounding."""
    U, I, nnz = 3000, 500, 90_000
    u, i, r = synth(U, I, nnz, 77, skew=True)
    X = als_oracle.init_factors(U, 64, 2)
    got, _ = gpu_half_step(i, u, r, I, X, 0.1, seg_len=512)
    old, _ = gpu_half_step(i, u, r, I, X, 0.1, seg_len=512, packed=False)     # -> als_tc64_kernel
    assert rel_l2(old, got) <= 5e-6


@pytest.mark.parametrize("k", [64, 128])
def test_full_size_half_step_property(k):
    """MovieLens-20M-like shape (scaled rows, full skew): sampled rows against the oracle and the
    normal-equation residual on those rows (size-independent property)."""
    U, I, nnz = 138_493, 26_744, 4_000_000 if k == 64 else 2_000_000
    u, i, r = synth(U, I, nnz, 9, skew=True)
    X = als_oracle.init_factors(U, k, 4)
    got, plan = gpu_half_step(i, u, r, I, X, 0.1)
    assert plan.n_long > 0
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    cnt = np.diff(rp)
    rows = np.concatenate([np.argsort(-cnt)[:6], np.random.default_rng(0).choice(I, 150, replace=False)])
    for j in rows:
        lo, hi = rp[j], rp[j + 1]
        if hi == lo:
            assert not got[j].any()
            continue
        Gm = X[ci[lo:hi]].astype(np.float64)
        A = Gm.T @ Gm + 0.1 * (hi - lo) * np.eye(k)
        b = v[lo:hi].astype(np.float64) @ Gm
        want = np.linalg.solve(A, b)
        assert np.abs(got[j] - want).max() <= 2e-4 * max(1.0, np.abs(want).max()), (j, hi - lo)
        assert np.linalg.norm(A @ got[j] - b) <= 1e-4 * np.linalg.norm(b) + 1e-3
    # the tensor-core path reduces long rows through fixed slots in a fixed order: a second run is bit-identical
    again, _ = gpu_half_step(i, u, r, I, X, 0.1)
    assert np.array_equal(got, again)


def test_gram_and_predict():
    als_engine, _ = _mods()
    nat = _nat()
    dev = torch.device("cuda")
    rng = np.random.default_rng(2)
    for n, k in ((1000, 10), (5000, 64), (70000, 128), (3, 20)):
        Y = rng.standard_normal((n, k)).astype(np.float32)
        out = torch.empty((k, k), dtype=torch.float32, device=dev)
        ws = torch.empty(int(nat.lib().hals_gram_workspace_bytes(k)), dtype=torch.uint8, device=dev)
        als_engine.native_gram(torch.from_numpy(Y).to(dev), out, ws)
        want = als_oracle.gram_f64(Y)
        assert np.abs(out.cpu().numpy() - want).max() <= 2e-5 * np.abs(want).max() + 1e-4
    X = rng.standard_normal((40, 10)).astype(np.float32); Y = rng.standard_normal((30, 10)).astype(np.float32)
    uu, ii = rng.integers(0, 40, 500).astype(np.int32), rng.integers(0, 30, 500).astype(np.int32)
    up = np.ones(40, np.uint8); up[5] = 0
    out = torch.empty(500, dtype=torch.float32, device=dev)
    t = lambda a: torch.from_numpy(a).to(dev)
    tx, ty, tu, ti, tp = t(X), t(Y), t(uu), t(ii), t(up)
    nat.check(nat.lib().hals_als_predict(nat.ptr(tx), nat.ptr(ty), 10, nat.ptr(tu), nat.ptr(ti), 500, nat.ptr(tp),
                                         None, nat.ptr(out), nat.current_stream()))
    got = out.cpu().numpy()
    want = als_oracle.als_predict(X, Y, uu, ii, user_present=up.astype(bool))
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.isnan(got).sum() > 0
    assert np.allclose(got[~np.isnan(got)], want[~np.isnan(want)], atol=2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [64, 128])
def test_device_chunk_table_equals_the_host_planner(k):
    """AlsPlanHandle derives the chunk table on the device; hals_als_plan_chunks_host (the C-ABI planner a C caller
    uses) must give exactly the same arrays."""
    als_engine, csr = _mods()
    nat = _nat()
    rng = np.random.default_rng(9)
    counts = rng.integers(0, 300, 4000); counts[[7, 900]] = [9000, 70000]
    rows = np.repeat(np.arange(len(counts)), counts)
    cols = rng.integers(0, 500, rows.size)
    vals = rng.integers(1, 6, rows.size).astype(np.float32)
    dev = torch.device("cuda")
    shard = csr.build_csr(torch.as_tensor(rows).to(dev), torch.as_tensor(cols).to(dev), torch.as_tensor(vals).to(dev), len(counts))
    plan = csr.AlsPlanHandle(shard, k, 1024, n_src=500)
    n, h = plan.n_items, plan.host
    L = nat.lib()
    nch = int(L.hals_als_plan_chunk_count_host(nat.ptr(h["item_len"]), n))
    assert nch == plan.n_chunks
    c0, cost0 = np.empty(n + 1, np.int64), np.empty(n + 1, np.int64)
    pos, cnt = np.empty(nch, np.int64), np.empty(nch, np.int32)
    nat.check(L.hals_als_plan_chunks_host(nat.ptr(h["item_len"]), nat.ptr(h["item_begin"]), nat.ptr(h["item_slot"]), n, k,
                                          nat.ptr(c0), nat.ptr(cost0), nat.ptr(pos), nat.ptr(cnt)))
    for name, want in (("item_chunk0", c0), ("item_cost0", cost0), ("chunk_pos", pos), ("chunk_cnt", cnt)):
        got = plan.dev[name].cpu().numpy()
        assert got.dtype == want.dtype and np.array_equal(got, want), name
