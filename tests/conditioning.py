"""CPU helpers (test infrastructure): ill-conditioned ALS half-steps and a criterion that holds for any fp32-accurate
solver whatever the conditioning.  tests/test_als_conditioning_cpu.py checks the criterion itself,
tests/test_gpu_als_conditioning.py applies it to every solver route on the same cases.

Every other ALS accuracy test draws its source factors with als_oracle.init_factors (unit-norm rows in random
directions) at reg 0.05 / 0.1: the per-row normal matrix A_j = sum y y^T + reg n_j I has kappa ~ 10 there.  Factors of
a real fit share one dominant direction (the mean rating) and a grid search tries small regParam; kappa(A_j) then grows
as ~1/reg and the forward error of even a correct fp32 solve grows with it (~1e-3 at kappa = 1e4), so a forward
tolerance cannot tell an accurate solver from an inaccurate one there.  The componentwise backward error can:

    eta_j = max_i |A_j x_j - b_j|_i / ((|Y_j|^T |Y_j| + reg n_j I) |x_j| + |Y_j|^T |r_j|)_i

(fp64, from the fp32 inputs; x_j the solver's output, Y_j the gathered source rows).  Implicit feedback: the magnitudes
are |Y|^T |Y| + sum c |y| |y|^T + reg n+ I and sum_{r>0} (1 + c) |y|.  An fp32 build and an fp32 Cholesky keep eta at a
few u = 2^-24 at every kappa; a build with TF32 or plain bf16 operands lands one to two orders of magnitude higher.
The emulations below reproduce the routes' arithmetic on the CPU, so that test_als_conditioning_cpu.py shows the
thresholds pass every accurate build with a margin and fail every inaccurate one.
"""
import numpy as np

from oracle import als_oracle
from tests import nnls_oracle
from tests.test_gpu_als_inputs import N_ROWS, N_SRC, ROW_LENS, boundary_case, implicit_alpha

U = 2.0 ** -24
LAMBDAS = (1e-1, 1e-2, 1e-3, 1e-4)
SPREAD = 1e-3
# eta thresholds, per rating kind.  Set by the accurate builds of the CPU emulations below, with a margin of 3
# (tests/test_als_conditioning_cpu.py; DESIGN.md section 4).  Explicit, non-integer ratings: the tensor-core build drops
# l r_lo and l l^T (each up to 2^-18 = 64 u of |y| |r| and |y| |y|^T), which puts rows of a few ratings at up to ~90 u.
# Explicit, integer ratings (r_lo = 0) and implicit: every accurate build stays below 20 u.  Builds from TF32 or plain
# bf16 operands reach >= 330 u (explicit, every kind) and >= 400 u (implicit) on the rows of at most SHORT ratings.
ETA_MAX_INT = 64 * U
ETA_MAX_NONINT = 280 * U
ETA_MAX_IMPLICIT = 64 * U


def eta_max(kind, implicit=False):
    if implicit:
        return ETA_MAX_IMPLICIT
    return ETA_MAX_INT if kind == "int" else ETA_MAX_NONINT
# implicit cases: ratings of both signs and zeros; these rows get only ratings <= 0 (n+ = 0, b = 0: the solution is
# exactly 0): the 1-rating row, a 33-rating row and the 300-rating row (sliced into 4)
IMPLICIT_KIND = "centred"
NONPOS_ROWS = (1, 8, 16)
SHORT = 300      # rows of at most this many ratings: where TF32 / plain bf16 builds must fail the thresholds


def trained_factors(n, k, spread=SPREAD, seed=0):
    """Source factors that look like those of a fit after a sweep: a common unit direction mu plus 0.3 x noise whose
    singular values fall geometrically from 1 to `spread` in a random basis.  fp32 [n, k]."""
    rng = np.random.default_rng(seed)
    mu = rng.standard_normal(k)
    mu /= np.linalg.norm(mu)
    basis = np.linalg.qr(rng.standard_normal((k, k)))[0]
    noise = (rng.standard_normal((n, k)) * np.geomspace(1.0, spread, k)) @ basis.T
    return (mu + 0.3 * noise).astype(np.float32)


def conditioned_case(kind, k, reg, implicit=False):
    """(dst rows, src cols, ratings, source factors, alpha) of the boundary matrix of test_gpu_als_inputs (empty rows,
    duplicate pairs, rows around the MMA / chunk steps, sliced long rows) with trained-like source factors.  Implicit:
    the rows NONPOS_ROWS get only ratings <= 0.  Asserts that the case is as ill-conditioned as it claims: the median
    kappa(A_j) over the solved rows is >= 0.3 / reg."""
    rows, cols, r, _ = boundary_case(kind, k)
    X = trained_factors(N_SRC, k, seed=k)
    alpha = implicit_alpha(kind) if implicit else 1.0
    if implicit:
        r = r.copy()
        nonpos = np.isin(rows, NONPOS_ROWS)
        r[nonpos] = -np.abs(r[nonpos])
    _, kappa = solved_kappa(rows, cols, r, X, reg, implicit, alpha)
    assert np.median(kappa) >= 0.3 / reg, (np.median(kappa), reg)
    return rows, cols, r, X, alpha


def csr(rows, cols, r):
    return als_oracle.coo_to_csr(rows, cols, r, N_ROWS)


def solved_kappa(rows, cols, r, X, reg, implicit=False, alpha=1.0):
    """(row ids, kappa) of the rows with a ridge (n > 0; implicit: n+ > 0)."""
    rp, ci, v = csr(rows, cols, r)
    ids, A, _ = nnls_oracle.normal_equations(rp, ci, v, X, reg, implicit, alpha)
    keep = positive_counts(rp, v, implicit)[ids] > 0
    return ids[keep], np.linalg.cond(A[keep])


def positive_counts(rowptr, vals, implicit):
    """n (explicit) or n+ (implicit) per row."""
    vals = np.asarray(vals)
    return np.array([(vals[lo:hi] > 0).sum() if implicit else hi - lo for lo, hi in zip(rowptr[:-1], rowptr[1:])])


def backward_error(rowptr, colidx, vals, src, x, reg, implicit=False, alpha=1.0):
    """(row ids, eta, kappa) of every row with ratings: eta_j as in the module docstring (0 where the residual is 0,
    e.g. a row of implicit ratings <= 0 solved as exactly 0), kappa_j = kappa_2(A_j) in fp64."""
    ids, A, b = nnls_oracle.normal_equations(rowptr, colidx, vals, src, reg, implicit, alpha)
    absv = vals if implicit else np.abs(vals)      # implicit: c = alpha |r| and the signs of r define the magnitudes
    _, Am, bm = nnls_oracle.normal_equations(rowptr, colidx, absv, np.abs(src), reg, implicit, alpha)
    xd = np.asarray(x, np.float64)[ids]
    res = np.abs(np.einsum("rij,rj->ri", A, xd) - b)
    den = np.einsum("rij,rj->ri", Am, np.abs(xd)) + np.abs(bm)
    with np.errstate(divide="ignore", invalid="ignore"):
        eta = np.where(res == 0, 0.0, res / den).max(1)
    return ids, eta, np.linalg.cond(A)


# --- CPU emulations of the routes' arithmetic (used by the self-test only) -------------------------------------------

def bf16(x):
    """Round fp32 to bfloat16 (nearest even), returned as fp32."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000).astype(np.uint32).view(np.float32)


def tf32(x):
    """Round fp32 to TF32 (10 explicit mantissa bits, nearest even), returned as fp32."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0xFFF + ((u >> 13) & 1)) & 0xFFFFE000).astype(np.uint32).view(np.float32)


def split(x):
    h = bf16(x)
    return h, bf16(np.float32(x) - h)


def _accumulate(a, b, step=1):
    """sum_t a_t b_t^T accumulated in fp32: `step` products are added exactly (fp64) and then rounded
    into the fp32 sum (1: an FMA chain, the CUDA-core build; 16: one tensor-core K step)."""
    A = np.zeros((a.shape[1], b.shape[1]), np.float32)
    for t in range(0, a.shape[0], step):
        A = (A + a[t:t + step].astype(np.float64).T @ b[t:t + step].astype(np.float64)).astype(np.float32)
    return A


def _vec(w, b, step=1):
    return _accumulate(np.asarray(w, np.float32)[:, None], b, step=step)[0]


def build_fp32(G, r):
    return _accumulate(G, G), _vec(r, G)


def build_bf16x3(G, r):
    """DESIGN section 3.0: A = D_hh + D_hl + D_hl^T (l l^T dropped), b = (h + l) r_hi + h r_lo."""
    h, l = split(G)
    rh, rl = split(r)
    Dhh, Dhl = _accumulate(h, h, step=16), _accumulate(l, h, step=16)
    A = Dhh + Dhl + Dhl.T
    b = _vec(rh, h, 16) + _vec(rh, l, 16) + _vec(rl, h, 16)
    return A, b


def build_rounded(G, r, rnd):
    g, q = rnd(G), rnd(r)
    return _accumulate(g, g, step=16), _vec(q, g, 16)


def build_fp32_implicit(G, r, alpha):
    c = np.float32(alpha) * np.abs(r)
    wb = np.where(r > 0, np.float32(1) + c, np.float32(0)).astype(np.float32)
    return _accumulate((G * c[:, None]).astype(np.float32), G), _vec(wb, G)


def build_tc_implicit(G, r, alpha):
    """DESIGN section 3.1c: the split row (h + l) is rescaled by sqrt(c) in fp32 and split again; the rating column
    (1 + c) / sqrt(c) (0 unless r > 0) is split; then the explicit bf16x3 build on the rescaled rows."""
    h, l = split(G)
    c = np.float32(alpha) * np.abs(r)
    sc = np.sqrt(c).astype(np.float32)
    rho = np.where((r > 0) & (c > 0), (np.float32(1) + c) / np.where(sc > 0, sc, 1), 0).astype(np.float32)
    return build_bf16x3((sc[:, None] * (h + l)).astype(np.float32), rho)


def build_rounded_implicit(G, r, alpha, rnd):
    c = np.float32(alpha) * np.abs(r)
    sc = np.sqrt(c).astype(np.float32)
    rho = np.where((r > 0) & (c > 0), (np.float32(1) + c) / np.where(sc > 0, sc, 1), 0).astype(np.float32)
    return build_rounded((sc[:, None] * G).astype(np.float32), rho, rnd)


def cholesky_solve_f32(A, b):
    """Batched A [m,k,k], b [m,k] fp32: Cholesky and both substitutions, every operation rounded to fp32."""
    A = np.array(A, np.float32)
    y = np.array(b, np.float32)
    m, k = y.shape
    L = np.zeros_like(A)
    with np.errstate(invalid="ignore", divide="ignore"):
        for j in range(k):
            d = np.sqrt(A[:, j, j])
            L[:, j:, j] = A[:, j:, j] / d[:, None]
            L[:, j, j] = d
            col = L[:, j + 1:, j]
            A[:, j + 1:, j + 1:] -= col[:, :, None] * col[:, None, :]
        for j in range(k):
            y[:, j] = (y[:, j] - np.einsum("ri,ri->r", L[:, j, :j], y[:, :j])) / L[:, j, j]
        x = np.zeros_like(y)
        for j in reversed(range(k)):
            x[:, j] = (y[:, j] - np.einsum("ri,ri->r", L[:, j + 1:, j], x[:, j + 1:])) / L[:, j, j]
    return x


EXPLICIT_BUILDS = {
    "fp32": build_fp32,
    "bf16x3": build_bf16x3,
    "tf32": lambda G, r: build_rounded(G, r, tf32),
    "bf16": lambda G, r: build_rounded(G, r, bf16),
}
# implicit build -> (build of sum c y y^T and b, build of the Gram Y^T Y).  The Gram of the routes is fp32-accurate
# (gram_partial_kernel in fp32 below 2048 source rows, gram_tc_kernel in bf16x3 above).
IMPLICIT_BUILDS = {
    "fp32": (build_fp32_implicit, build_fp32),
    "tc": (build_tc_implicit, build_fp32),
    "tf32": (lambda G, r, a: build_rounded_implicit(G, r, a, tf32), EXPLICIT_BUILDS["tf32"]),
}


def emulated_systems(build, rows, cols, r, X, implicit=False, alpha=1.0):
    """(row ids, ridge counts, A without ridge [m,k,k] fp32, b [m,k] fp32) of the rows with a ridge (n > 0 / n+ > 0),
    built per row with `build` (implicit: a pair of IMPLICIT_BUILDS, the second one builds the Gram)."""
    rp, ci, v = csr(rows, cols, r)
    n = positive_counts(rp, v, implicit)
    ids = np.flatnonzero(n > 0)
    As, bs = [], []
    for j in ids:
        G = X[ci[rp[j]:rp[j + 1]]]
        rr = np.asarray(v[rp[j]:rp[j + 1]], np.float32)
        A, b = build[0](G, rr, alpha) if implicit else build(G, rr)
        As.append(A)
        bs.append(b)
    A, b = np.stack(As), np.stack(bs)
    if implicit:
        gram, _ = build[1](X, np.ones(len(X), np.float32))
        A = (A + gram).astype(np.float32)
    return ids, n[ids], A, b


def emulated_half_step(system, reg):
    """The fp32 solve of an emulated build at one reg: x [N_ROWS, k] (rows without a ridge stay 0)."""
    ids, n, A, b = system
    A = A.copy()
    k = A.shape[1]
    A[:, np.arange(k), np.arange(k)] += (np.float32(reg) * n.astype(np.float32))[:, None]
    x = np.zeros((N_ROWS, k), np.float32)
    x[ids] = cholesky_solve_f32(A, b)
    return x


def short_rows():
    return np.asarray(ROW_LENS) <= SHORT
