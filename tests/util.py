import contextlib

import numpy as np


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# Ratings by kind.  "int" is exact in bf16; every other kind is mostly not, so the tensor-core kernels' low rating part
# (r - bf16(r)) carries weight.  decimal: one decimal place in [1, 5] (the reference trains on average_review_rating);
# centred: decimal - 3 (both signs, exact zeros); scaled_up / scaled_down: decimal x 1e3 / x 1e-3 (an explicit
# half-step is linear in the ratings, so only a relative tolerance applies).
RATING_KINDS = ("int", "decimal", "centred", "scaled_up", "scaled_down")
RATING_SCALE = {"scaled_up": 1e3, "scaled_down": 1e-3}


def draw_ratings(kind, n, rng):
    if kind == "int":
        return rng.integers(1, 6, n).astype(np.float32)
    tenths = rng.integers(10, 51, n)
    if kind == "centred":
        return ((tenths - 30) / 10).astype(np.float32)
    return (tenths / 10 * RATING_SCALE.get(kind, 1.0)).astype(np.float32)


def bf16_exact(x):
    """True where a float32 value is exactly a bfloat16 (its low 16 bits are zero)."""
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) & 0xFFFF) == 0


@contextlib.contextmanager
def launched_kernels():
    """Yields a list that, on exit, holds the names (whitespace removed, so "kern<64,true,true>") of the events
    torch.profiler recorded inside the block: the CUDA kernels launched there and the host calls around them."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    names = []
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], acc_events=True) as prof:
        # open the window with a kernel of its own: late in a long test session the profiler was seen to miss the
        # first device activity of a window
        torch.zeros(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        yield names
        torch.cuda.synchronize()
    names.extend(sorted({"".join(e.name.split()) for e in prof.events()}))


def assert_ran(names, *kernels, absent=()):
    for k in kernels:
        assert any(k in n for n in names), f"{k} did not run; launched: {names}"
    for k in absent:
        assert not any(k in n for n in names), f"{k} ran; launched: {names}"


def check_topk_against_dense(B, idx, score, k, tol, item_offset=0):
    """B: oracle blend [U,I] fp64.  idx/score: [U,k] from the kernels.  Top-k index sets must be
    identical except for items whose oracle score lies within `tol` of the k-th score (ties)."""
    U, I = B.shape
    kk = min(k, I)
    for u in range(U):
        got = idx[u]
        valid = got[got >= 0] - item_offset
        assert len(valid) == kk, (u, len(valid), kk)
        assert len(set(valid.tolist())) == kk
        assert (got[kk:] == -1).all()
        s = score[u, :kk].astype(np.float64)
        assert np.all(np.diff(s) <= 0), "scores must be sorted descending"
        assert np.allclose(s, B[u, valid], rtol=0, atol=tol), np.abs(s - B[u, valid]).max()
        order = np.sort(B[u])[::-1]
        kth = order[kk - 1]
        must = set(np.nonzero(B[u] > kth + tol)[0].tolist())
        assert must <= set(valid.tolist()), (u, must - set(valid.tolist()))
        assert np.all(B[u, valid] >= kth - tol)
        # equal scores: lower item index first
        for a in range(kk - 1):
            if score[u, a] == score[u, a + 1]:
                assert got[a] < got[a + 1]
