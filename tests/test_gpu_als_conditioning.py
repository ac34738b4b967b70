"""GPU: the ALS half-step on ill-conditioned normal equations (trained-like source factors, reg down to 1e-4, kappa up to
1e4), through every solver route, against the componentwise backward-error thresholds of tests/conditioning.py (which
tests/test_als_conditioning_cpu.py shows to pass fp32-accurate builds and fail TF32 / plain bf16 ones).  A forward
tolerance cannot be used there: the forward error of a correct fp32 solve grows with kappa.

Each case checks with torch.profiler which kernels ran.  HALS_FORCE_SIMT is read once per process, so the CUDA-core
kernels at ranks 64 / 128 run in a child process (this module run as a script)."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import als_oracle, c_oracle
from tests import conditioning as C
from tests.test_gpu_als import _mods, gpu_half_step, synth
from tests.test_gpu_als_inputs import (EMPTY, EXPLICIT_ROUTES, IMPLICIT_ROUTES, N_ROWS, ROOT, ROW_LENS, SEG, check_main_kernel,
                                       check_plan)
from tests.test_gpu_als_nonneg import check_case, gpu_nonneg, padded
from tests.util import assert_ran, launched_kernels, rel_l2

pytestmark = pytest.mark.gpu
KINDS = ("int", "decimal", "centred")
IMPLICIT_LAMBDAS = (1e-2, 1e-3)


def simt_kernels(k, implicit):
    vec = str(k % 4 == 0).lower()
    return f"als_build_solve_kernel<{padded(k)},{str(implicit).lower()},{vec}>", f"als_reduce_solve_kernel<{padded(k)}>"


# route -> (rank, plan with packed ratings, kernels that must run; the first is the main kernel)
EXPLICIT = dict(EXPLICIT_ROUTES)
EXPLICIT.update({f"simt{k}": (k, True, simt_kernels(k, False)) for k in (10, 33, 100)})
# route -> (rank, plan packed for implicit feedback, kernels that must run)
IMPLICIT = dict(IMPLICIT_ROUTES)
IMPLICIT["simt10"] = (10, False, simt_kernels(10, True))


def check_eta(got, rows, cols, r, X, reg, implicit, alpha, kind, label):
    """Every solved row has eta <= conditioning.eta_max; the line printed is the measured maximum (run pytest with -s to see it)."""
    assert np.isfinite(got).all(), f"{label}: non-finite rows {np.flatnonzero(~np.isfinite(got).all(1))}"
    assert not got[EMPTY].any(), "rows without ratings are zero"
    ids, eta, kappa = C.backward_error(*C.csr(rows, cols, r), X, got, reg, implicit, alpha)
    w = int(eta.argmax())
    limit = C.eta_max(kind, implicit)
    msg = (f"{label}: max eta {eta.max() / C.U:.1f} u (threshold {limit / C.U:.0f} u) at row {ids[w]} "
           f"({ROW_LENS[ids[w]]} ratings, kappa {kappa[w]:.1e}); median kappa {np.median(kappa):.1e}")
    print("ETA", msg)
    assert eta.max() <= limit, msg


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("reg", C.LAMBDAS)
@pytest.mark.parametrize("route", list(EXPLICIT))
def test_explicit_route_backward_error(route, reg, kind):
    """ws64 / ws128: the default plan; tc64 / tc128: no packed ratings (the round-1 kernels); simt*: the CUDA-core
    kernel at ranks 10, 33, 100.  Sliced long rows go through the slot pre-sums and the reduce-solve kernels.
    Tensor-core routes: a second call is bit-identical."""
    k, packed, kernels = EXPLICIT[route]
    rows, cols, r, X, _ = C.conditioned_case(kind, k, reg)
    run = lambda: gpu_half_step(rows, cols, r, N_ROWS, X, reg, seg_len=SEG, packed=packed)
    with launched_kernels() as names:
        got, plan = run()
    check_main_kernel(names, kernels)
    check_plan(plan)
    check_eta(got, rows, cols, r, X, reg, False, 1.0, kind, f"{route} reg={reg:g} {kind}")
    if not route.startswith("simt"):
        assert np.array_equal(got, run()[0])


@pytest.mark.parametrize("reg", IMPLICIT_LAMBDAS)
@pytest.mark.parametrize("route", list(IMPLICIT))
def test_implicit_route_backward_error(route, reg):
    """Ratings of both signs and zeros; the rows conditioning.NONPOS_ROWS (1 rating, 33 ratings, 300 ratings in four
    slices) have only ratings <= 0: n+ = 0, so no ridge and b = 0, and A = Y^T Y + sum c y y^T has kappa near 1/u.
    Spark's fp64 solve gives exactly 0 there; so must every route (no NaN from a pivot that rounds to <= 0)."""
    k, tc, kernels = IMPLICIT[route]
    rows, cols, r, X, alpha = C.conditioned_case(C.IMPLICIT_KIND, k, reg, implicit=True)
    run = lambda: gpu_half_step(rows, cols, r, N_ROWS, X, reg, implicit=True, alpha=alpha, seg_len=SEG,
                                plan_implicit=tc)
    with launched_kernels() as names:
        got, plan = run()
    check_main_kernel(names, kernels)
    check_plan(plan)
    nonpos = got[list(C.NONPOS_ROWS)]
    assert np.isfinite(nonpos).all() and not nonpos.any(), f"rows of ratings <= 0: {nonpos[:, :4]}"
    check_eta(got, rows, cols, r, X, reg, True, alpha, C.IMPLICIT_KIND, f"implicit {route} reg={reg:g}")
    if tc:
        assert np.array_equal(got, run()[0])


@pytest.mark.parametrize("reg", IMPLICIT_LAMBDAS)
@pytest.mark.parametrize("k", [10, 64, 128])
def test_nonnegative_half_step(k, reg):
    """hals_als_half_step_nonnegative on the ill-conditioned boundary case: the KKT conditions per row (the forward
    tolerance does not apply at this kappa) and no row at the iteration cap."""
    rows, cols, r, X, _ = C.conditioned_case("decimal", k, reg)
    with launched_kernels() as names:
        got, plan, capped = gpu_nonneg(rows, cols, r, N_ROWS, X, reg, seg_len=SEG)
    check_plan(plan)
    vec = str(k % 4 == 0).lower()
    assert_ran(names, f"als_build_solve_nnls_kernel<{padded(k)},false,{vec}>",
               f"als_reduce_solve_nnls_kernel<{padded(k)}>", absent=("als_ws64_kernel", "als_ws128_kernel"))
    check_case(got, rows, cols, r, N_ROWS, X, reg, False, coverage=False, forward=False)
    assert capped == 0


# --- ten sweeps at reg 0.01 ------------------------------------------------------------------------------------------

FIT_REG = 0.01


def fit_data(k):
    """The Zipf shape of test_gpu_als.test_fit_10_sweeps_on_the_tensor_core_ranks."""
    U, I, nnz = 6000, 900, 240_000
    u, i, r = synth(U, I, nnz, 21 + k, skew=True)
    return u, i, r, U, I, als_oracle.init_factors(U, k, 5)


def gpu_fit(k):
    als_engine, _ = _mods()
    u, i, r, U, I, X0 = fit_data(k)
    eng = als_engine.AlsEngine(u, i, r, U, I, k, FIT_REG, seg_len=1024)
    assert eng.plan_Rt.n_long > 0
    eng.set_user_factors(X0)
    with launched_kernels() as names:
        X, Y = eng.fit(10)
    return X.cpu().numpy(), Y.cpu().numpy(), names


def gpu_fit_stateless(k):
    """The same ten sweeps through the stateless hals_als_half_step (the oracle's sweep loop, each half-step on the
    GPU): the engine keeps ranks 64 / 128 in split form on the tensor-core kernels whatever HALS_FORCE_SIMT says, the
    stateless call honours it."""
    u, i, r, U, I, X0 = fit_data(k)

    def half_step(rp, ci, v, src, reg, implicit, alpha):
        got, _ = gpu_half_step(np.repeat(np.arange(len(rp) - 1), np.diff(rp)), ci, v, len(rp) - 1, src, reg,
                               seg_len=1024)
        return got

    with launched_kernels() as names:
        X, Y = als_oracle.als_fit(u, i, r, U, I, k, 10, FIT_REG, X0, half_step=half_step)
    return X, Y, names


@functools.lru_cache(maxsize=None)
def oracle_fit(k):
    u, i, r, U, I, X0 = fit_data(k)
    return als_oracle.als_fit(u, i, r, U, I, k, 10, FIT_REG, X0, half_step=c_oracle.als_half_step)


def check_fit(k, X, Y, label):
    """What ill-conditioning leaves well-determined: the RMSE and the predictions on the rated pairs.  The factors
    themselves are reported, not asserted."""
    u, i, r, *_ = fit_data(k)
    Xo, Yo = oracle_fit(k)
    assert np.isfinite(X).all() and np.isfinite(Y).all()
    pred, pred_o = (np.einsum("nk,nk->n", A[u].astype(np.float64), B[i].astype(np.float64)) for A, B in ((X, Y), (Xo, Yo)))
    d_rmse = abs(als_oracle.rmse(X, Y, u, i, r) - als_oracle.rmse(Xo, Yo, u, i, r))
    msg = (f"{label}: |dRMSE| {d_rmse:.1e}, predictions rel-L2 {rel_l2(pred, pred_o):.1e}; factors rel-L2 "
           f"X {rel_l2(X, Xo):.1e} Y {rel_l2(Y, Yo):.1e}")
    print("FIT", msg)
    assert d_rmse <= 1e-4, msg
    assert rel_l2(pred, pred_o) <= 1e-3, msg


@pytest.mark.parametrize("k", [64, 128])
def test_ten_sweeps_at_small_reg_tensor_core(k):
    X, Y, names = gpu_fit(k)
    assert_ran(names, f"als_ws{k}_kernel", absent=("als_build_solve_kernel",))
    check_fit(k, X, Y, f"ws{k}")


# --- HALS_FORCE_SIMT=1: the CUDA-core kernels at ranks 64 / 128, in a child process ---------------------------------

def _force_simt_child(out):
    res = {}
    for k in (64, 128):
        for kind in KINDS:
            for reg in C.LAMBDAS:
                rows, cols, r, X, _ = C.conditioned_case(kind, k, reg)
                with launched_kernels() as names:
                    res[f"x_{k}_{kind}_{reg}"], _ = gpu_half_step(rows, cols, r, N_ROWS, X, reg, seg_len=SEG)
                res[f"names_x_{k}_{kind}_{reg}"] = np.array(names)
        res[f"fit_X_{k}"], res[f"fit_Y_{k}"], names = gpu_fit_stateless(k)
        res[f"names_fit_{k}"] = np.array(names)
    np.savez(out, **res)


@pytest.fixture(scope="module")
def force_simt(tmp_path_factory):
    out = tmp_path_factory.mktemp("force_simt_cond") / "out.npz"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-m", "tests.test_gpu_als_conditioning", str(out)]
    p = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, HALS_FORCE_SIMT="1"), capture_output=True, text=True,
                       timeout=1800)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    with np.load(out) as z:
        return {n: z[n] for n in z.files}


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("reg", C.LAMBDAS)
@pytest.mark.parametrize("k", [64, 128])
def test_explicit_cuda_core_route_backward_error(force_simt, k, reg, kind):
    check_main_kernel(list(force_simt[f"names_x_{k}_{kind}_{reg}"]), simt_kernels(k, False))
    rows, cols, r, X, _ = C.conditioned_case(kind, k, reg)
    check_eta(force_simt[f"x_{k}_{kind}_{reg}"], rows, cols, r, X, reg, False, 1.0, kind,
              f"simt{k} (forced) reg={reg:g} {kind}")


@pytest.mark.parametrize("k", [64, 128])
def test_ten_sweeps_at_small_reg_cuda_core(force_simt, k):
    assert_ran(list(force_simt[f"names_fit_{k}"]), *simt_kernels(k, False),
               absent=("als_ws64_kernel", "als_ws128_kernel", "als_tc64_kernel", "als_tc128_kernel"))
    check_fit(k, force_simt[f"fit_X_{k}"], force_simt[f"fit_Y_{k}"], f"simt{k} (forced)")


if __name__ == "__main__":
    _force_simt_child(sys.argv[1])
