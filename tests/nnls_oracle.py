"""CPU ORACLE (test infrastructure, not product code): the nonnegative ALS half-step in fp64.

Spark's ALS with nonnegative=True hands the normal equations of every row (the same A, with regParam * n on the
diagonal, and b as the Cholesky route) to NNLSSolver.  Its iterates are an approximation; what this oracle computes
is the exact minimiser of

    1/2 x^T A x - b^T x   subject to x >= 0

(unique: A is positive definite), by block principal pivoting (Kim & Park 2011, Judice-Pires backup rule) in fp64:
x_F = A_FF^-1 b_F on the free set, x = 0 elsewhere, until the KKT conditions x >= 0, g = A x - b >= 0, x g = 0 hold.
The rows of a batch are solved together but independently: a row's result does not depend on the batch it is in.
"""
from __future__ import annotations

import numpy as np

from oracle import als_oracle


def nnls_batched(A, b, max_iter=None):
    """A [m,k,k] symmetric positive definite, b [m,k] -> (x [m,k] fp64, iterations [m]).  Raises when a row does not
    converge (the backup rule makes the exact method finite; the bound is far above what any test problem needs)."""
    A = np.asarray(A, np.float64)
    b = np.asarray(b, np.float64)
    m, k = b.shape
    cap = max_iter if max_iter is not None else 50 * k + 50
    x = np.zeros((m, k))
    g = -b.copy()
    F = np.zeros((m, k), bool)
    best = np.full(m, k + 1)
    left = np.full(m, 3)
    iters = np.zeros(m, np.int64)
    eye = np.eye(k)
    todo = np.arange(m)
    for _ in range(cap + 1):
        if todo.size == 0:
            break
        xs, gs, Fs = x[todo], g[todo], F[todo]
        # relative level of exact zero in fp64: a gradient entry this close to 0 is 0
        scale = np.abs(A[todo]) @ np.abs(xs)[..., None]
        tol = 1e-13 * (scale[..., 0] + np.abs(b[todo]))
        bad = (Fs & (xs < 0)) | (~Fs & (gs < -tol))
        nv = bad.sum(1)
        done = nv == 0
        todo, bad, nv, Fs = todo[~done], bad[~done], nv[~done], Fs[~done]
        if todo.size == 0:
            break
        improve = nv < best[todo]
        best[todo[improve]] = nv[improve]
        left[todo[improve]] = 3
        keep_full = ~improve & (left[todo] > 0)
        left[todo[keep_full]] -= 1
        full = improve | keep_full
        flip = np.where(full[:, None], bad, False)
        single = np.flatnonzero(~full)
        if single.size:
            last = k - 1 - np.argmax(bad[single][:, ::-1], axis=1)      # largest violating index
            flip[single, last] = True
        Fs = Fs ^ flip
        F[todo] = Fs
        # free subsystem: identity on the bound set, so one batched solve covers every row
        M = np.where(Fs[:, :, None] & Fs[:, None, :], A[todo], 0.0) + np.where(Fs, 0.0, 1.0)[:, :, None] * eye
        rhs = np.where(Fs, b[todo], 0.0)
        xn = np.linalg.solve(M, rhs[..., None])[..., 0]
        x[todo] = xn
        g[todo] = np.where(Fs, 0.0, (A[todo] @ xn[..., None])[..., 0] - b[todo])
        iters[todo] += 1
    else:
        if todo.size:
            raise RuntimeError(f"NNLS oracle: {todo.size} rows did not converge in {cap} iterations")
    return x, iters


def nnls(A, b):
    """One problem: A [k,k], b [k] -> x [k] fp64."""
    x, _ = nnls_batched(np.asarray(A)[None], np.asarray(b)[None])
    return x[0]


def kkt_residual(A, b, x):
    """max over i of the KKT violations relative to (|A| |x| + |b|)_i: -x_i, -g_i, and |g_i| where x_i > 0."""
    A = np.asarray(A, np.float64); b = np.asarray(b, np.float64); x = np.asarray(x, np.float64)
    g = A @ x - b
    s = np.abs(A) @ np.abs(x) + np.abs(b)
    s = np.where(s > 0, s, 1.0)
    viol = np.maximum(np.maximum(-x, -g), np.where(x > 0, np.abs(g), 0.0))
    return float(np.max(np.maximum(viol, 0.0) / s)) if x.size else 0.0


def normal_equations(rowptr, colidx, vals, src, reg, implicit=False, alpha=1.0, rows=None):
    """(row ids, A [r,k,k], b [r,k]) of the rows with ratings, built in fp64 exactly as the Cholesky oracle builds them
    (oracle.als_oracle.als_half_step)."""
    rowptr = np.asarray(rowptr)
    srcd = np.asarray(src, np.float64)
    k = srcd.shape[1]
    yty = srcd.T @ srcd if implicit else None
    ids, As, bs = [], [], []
    for j in (range(len(rowptr) - 1) if rows is None else rows):
        lo, hi = int(rowptr[j]), int(rowptr[j + 1])
        if hi == lo:
            continue
        G = srcd[colidx[lo:hi]]
        r = np.asarray(vals[lo:hi], np.float64)
        if implicit:
            c1 = alpha * np.abs(r)
            A = yty + (G * c1[:, None]).T @ G
            pos = r > 0.0
            b = ((1.0 + c1) * pos) @ G
            n = int(pos.sum())
        else:
            A = G.T @ G
            b = r @ G
            n = hi - lo
        A[np.diag_indices(k)] += reg * n
        ids.append(j); As.append(A); bs.append(b)
    if not ids:
        return np.zeros(0, np.int64), np.zeros((0, k, k)), np.zeros((0, k))
    return np.asarray(ids), np.stack(As), np.stack(bs)


def als_half_step_nnls(rowptr, colidx, vals, src, reg, implicit=False, alpha=1.0, out64=False, batch=256):
    """The nonnegative half-step: fp32 [m,k] (fp64 with out64=True); rows without ratings stay zero."""
    m = len(rowptr) - 1
    k = np.asarray(src).shape[1]
    out = np.zeros((m, k), np.float64 if out64 else np.float32)
    for r0 in range(0, m, batch):
        ids, A, b = normal_equations(rowptr, colidx, vals, src, reg, implicit, alpha, rows=range(r0, min(m, r0 + batch)))
        if len(ids):
            x, _ = nnls_batched(A, b)
            out[ids] = x
    return out


def als_fit_nnls(users, items, ratings, n_users, n_items, rank, max_iter, reg, init_user_factors, implicit=False,
                 alpha=1.0):
    """oracle.als_oracle.als_fit with the nonnegative half-step."""
    return als_oracle.als_fit(users, items, ratings, n_users, n_items, rank, max_iter, reg, init_user_factors,
                              implicit=implicit, alpha=alpha, half_step=als_half_step_nnls)
