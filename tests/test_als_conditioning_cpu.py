"""CPU: the backward-error criterion of tests/conditioning.py can fail.  On the ill-conditioned cases the GPU tests use
(every reg of conditioning.LAMBDAS, ranks 64 and 128), CPU emulations of the routes' arithmetic show that the
thresholds (conditioning.eta_max) pass every fp32-accurate build (fp32 products and sums; the tensor-core bf16 hi/lo
build) with a margin of 3, and fail builds from TF32 or plain bf16 operands on the rows of at most conditioning.SHORT ratings --
while the forward error of the accurate builds grows with kappa and would fail a fixed forward tolerance."""
import functools

import numpy as np
import pytest

from oracle import als_oracle
from tests import conditioning as C
from tests import nnls_oracle
from tests.util import rel_l2

EXPLICIT_KINDS = ("int", "decimal", "centred")
ACCURATE = {False: ("fp32", "bf16x3"), True: ("fp32", "tc")}
INACCURATE = {False: ("tf32", "bf16"), True: ("tf32",)}


def case(kind, k, reg, implicit):
    return C.conditioned_case(kind, k, reg, implicit)


@functools.lru_cache(maxsize=None)
def system(build, kind, k, implicit):
    # the builds do not depend on reg: one system per build, the ridge is added per reg
    rows, cols, r, X, alpha = case(kind, k, C.LAMBDAS[0], implicit)
    builds = C.IMPLICIT_BUILDS if implicit else C.EXPLICIT_BUILDS
    return C.emulated_systems(builds[build], rows, cols, r, X, implicit, alpha)


def emulated_eta(build, kind, k, reg, implicit):
    """(eta of every row with ratings, the rows' ids, the emulated half-step)."""
    rows, cols, r, X, alpha = case(kind, k, reg, implicit)
    x = C.emulated_half_step(system(build, kind, k, implicit), reg)
    ids, eta, _ = C.backward_error(*C.csr(rows, cols, r), X, x, reg, implicit, alpha)
    return eta, ids, x


def oracle(kind, k, reg, implicit):
    rows, cols, r, X, alpha = case(kind, k, reg, implicit)
    rp, ci, v = C.csr(rows, cols, r)
    ids, A, b = nnls_oracle.normal_equations(rp, ci, v, X, reg, implicit, alpha)
    x = np.zeros((C.N_ROWS, k))
    x[ids] = np.linalg.solve(A, b[..., None])[..., 0]
    return x


CASES = [(False, kind) for kind in EXPLICIT_KINDS] + [(True, C.IMPLICIT_KIND)]


@pytest.mark.parametrize("reg", C.LAMBDAS)
@pytest.mark.parametrize("k", [64, 128])
@pytest.mark.parametrize("implicit,kind", CASES)
def test_accurate_builds_pass_with_margin(implicit, kind, k, reg):
    want = oracle(kind, k, reg, implicit)
    for build in ACCURATE[implicit]:
        eta, _, x = emulated_eta(build, kind, k, reg, implicit)
        assert np.isfinite(x).all()
        assert eta.max() * 3 <= C.eta_max(kind, implicit), (build, eta.max() / C.U)
        # what a forward tolerance would see: at kappa ~ 1e4 every fp32-accurate solve, the CUDA-core fp32 one too, is
        # farther from the oracle than the 2e-5 the well-conditioned tests allow (at 1e3 some are still inside)
        if reg <= 1e-4:
            assert rel_l2(x, want) > 2e-5, (build, rel_l2(x, want))


@pytest.mark.parametrize("reg", C.LAMBDAS)
@pytest.mark.parametrize("k", [64, 128])
@pytest.mark.parametrize("implicit,kind", CASES)
def test_inaccurate_builds_fail_on_short_rows(implicit, kind, k, reg):
    for build in INACCURATE[implicit]:
        eta, ids, _ = emulated_eta(build, kind, k, reg, implicit)
        short = C.short_rows()[ids]
        # integer ratings and implicit feedback: >= 3x above the threshold; non-integer explicit: above it
        margin = 1.0 if kind != "int" and not implicit else 3.0
        assert eta[short].max() >= margin * C.eta_max(kind, implicit), (build, eta[short].max() / C.U)


@pytest.mark.parametrize("k", [64, 128])
@pytest.mark.parametrize("implicit,kind", CASES)
def test_criterion_on_the_oracle_and_the_cases(implicit, kind, k):
    """The fp64 solution rounded to fp32 has eta <= u at every reg; kappa grows as ~1/reg (median over the solved
    rows within a factor 2 of 1/reg explicit, above it implicit); the implicit case holds rows with only ratings <= 0
    (b = 0: the solution is exactly 0), one of them sliced."""
    for reg in C.LAMBDAS:
        rows, cols, r, X, alpha = case(kind, k, reg, implicit)
        rp, ci, v = C.csr(rows, cols, r)
        x = oracle(kind, k, reg, implicit).astype(np.float32)
        _, eta, _ = C.backward_error(rp, ci, v, X, x, reg, implicit, alpha)
        assert eta.max() <= C.U, eta.max() / C.U
        _, kappa = C.solved_kappa(rows, cols, r, X, reg, implicit, alpha)
        assert 0.5 / reg <= np.median(kappa) <= (np.inf if implicit else 2.0 / reg), (reg, np.median(kappa))
    npos = C.positive_counts(rp, v, implicit)
    if implicit:
        rows_le0 = np.flatnonzero((npos == 0) & (np.diff(rp) > 0))
        assert set(C.NONPOS_ROWS) <= set(rows_le0)
        assert max(np.diff(rp)[list(C.NONPOS_ROWS)]) > 96, "one of them is a sliced long row"
        assert not oracle(kind, k, C.LAMBDAS[0], implicit)[list(C.NONPOS_ROWS)].any()


def test_trained_factors_shape():
    """A common direction carries most of every row; the noise spans `spread` (1e-3) of the leading singular value."""
    X = C.trained_factors(3000, 64, seed=1)
    assert X.dtype == np.float32 and X.shape == (3000, 64)
    mu = X.mean(0) / np.linalg.norm(X.mean(0))
    assert np.median(np.abs(X @ mu) / np.linalg.norm(X, axis=1)) > 0.8
    s = np.linalg.svd(X - X.mean(0), compute_uv=False)
    assert 0.5e-3 <= s[-1] / s[0] <= 2e-3, s[-1] / s[0]
    # and a fixed tolerance would not separate anything on init_factors-like cases: kappa ~ 10 there
    rows, cols, r, _ = C.boundary_case("int", 64)
    rp, ci, v = C.csr(rows, cols, r)
    _, A, _ = nnls_oracle.normal_equations(rp, ci, v, als_oracle.init_factors(C.N_SRC, 64, 7), 0.1)
    assert np.median(np.linalg.cond(A)) < 100
