"""CPU: the C-ABI library loads, exports every symbol include/hals_b200.h declares, and the
host-side planner is correct.  No compute entry point is called here (no GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

import hybrid_als_twotower_recommender_b200  # noqa: F401  (import shim)
from hybrid_als_twotower_recommender_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "hals_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hals_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    L = nat.lib()
    names = header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/hals_b200.h but not exported"
    assert set(names) == set(nat.SIGNATURES), "ctypes table and header disagree"
    assert L.hals_abi_version() == 1


def _plan(rowptr, seg):
    L = nat.lib()
    rp = np.asarray(rowptr, np.int64)
    a, b, c = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
    nat.check(L.hals_als_plan_count_host(nat.ptr(rp), len(rp) - 1, seg, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
    ni, nl = a.value, b.value
    row, beg, ln, slot = np.empty(ni, np.int32), np.empty(ni, np.int64), np.empty(ni, np.int32), np.empty(ni, np.int32)
    lr, ls, ln2 = np.empty(max(nl, 1), np.int32), np.empty(max(nl, 1), np.int32), np.empty(max(nl, 1), np.int32)
    nat.check(L.hals_als_plan_fill_host(nat.ptr(rp), len(rp) - 1, seg, nat.ptr(row), nat.ptr(beg), nat.ptr(ln),
                                        nat.ptr(slot), nat.ptr(lr), nat.ptr(ls), nat.ptr(ln2)))
    return (ni, nl, c.value), row, beg, ln, slot, lr[:nl], ls[:nl], ln2[:nl]


def test_planner_covers_every_rating_exactly_once():
    rng = np.random.default_rng(0)
    counts = rng.integers(0, 50, 300)
    counts[[3, 77, 150]] = [1000, 64, 257]     # long rows
    counts[[0, 10]] = 0                        # empty rows
    rowptr = np.concatenate([[0], np.cumsum(counts)])
    (ni, nl, nslots), row, beg, ln, slot, lr, ls, ln2 = _plan(rowptr, 64)
    covered = np.zeros(rowptr[-1], np.int32)
    for r, b, l, s in zip(row, beg, ln, slot):
        assert rowptr[r] <= b and b + l <= rowptr[r + 1] and 0 < l <= 64
        covered[b:b + l] += 1
        assert (s >= 0) == (counts[r] > 64)
    assert (covered == 1).all()
    assert sorted(lr) == [3, 150] and nl == 2
    assert nslots == sum(ln2) and sorted(slot[slot >= 0]) == list(range(nslots))
    assert set(row) == set(np.nonzero(counts)[0])
    # slices are spread evenly among the whole rows: every prefix holds its proportional share (+-1) of the slices
    sliced = np.cumsum(slot >= 0)
    want = np.arange(1, ni + 1) * nslots / ni
    assert np.abs(sliced - want).max() <= 1.0
    # slot ids keep the order of the ratings inside a row (the slot reduction sums them in slot order)
    for r in (3, 150):
        sel = row == r
        assert list(slot[sel]) == sorted(slot[sel]) and list(beg[sel]) == sorted(beg[sel])


def test_chunk_table_matches_the_items():
    L = nat.lib()
    rng = np.random.default_rng(1)
    counts = rng.integers(0, 200, 100)
    counts[[5, 50]] = [3000, 129]
    rowptr = np.concatenate([[0], np.cumsum(counts)])
    (ni, nl, nslots), row, beg, ln, slot, lr, ls, ln2 = _plan(rowptr, 96)
    nch = L.hals_als_plan_chunk_count_host(nat.ptr(ln), ni)
    assert nch == int(((ln + 31) // 32).sum())
    c0, cost0 = np.empty(ni + 1, np.int64), np.empty(ni + 1, np.int64)
    pos, cnt = np.empty(nch, np.int64), np.empty(nch, np.int32)
    nat.check(L.hals_als_plan_chunks_host(nat.ptr(ln), nat.ptr(beg), nat.ptr(slot), ni, 64, nat.ptr(c0), nat.ptr(cost0),
                                          nat.ptr(pos), nat.ptr(cnt)))
    assert c0[0] == 0 and c0[-1] == nch and (np.diff(c0) == (ln + 31) // 32).all()
    assert cost0[0] == 0 and (np.diff(cost0) > 0).all()
    for i in range(ni):
        ks = np.arange(c0[i], c0[i + 1])
        assert (pos[ks] == beg[i] + 32 * np.arange(len(ks))).all()
        assert (cnt[ks] == ln[i] - 32 * np.arange(len(ks))).all() and cnt[ks[-1]] <= 32 < cnt[ks[-1]] + 32
    assert L.hals_als_plan_chunk_count_host(None, 3) == -1


def test_planner_rejects_bad_input():
    L = nat.lib()
    rp = np.array([0, 5, 3], np.int64)
    a = ctypes.c_int64()
    assert L.hals_als_plan_count_host(nat.ptr(rp), 2, 64, ctypes.byref(a), ctypes.byref(a), ctypes.byref(a)) != 0
    assert b"monotone" in L.hals_last_error()
    assert L.hals_als_plan_count_host(None, 2, 64, ctypes.byref(a), ctypes.byref(a), ctypes.byref(a)) != 0


def test_workspace_queries():
    L = nat.lib()
    assert L.hals_als_workspace_bytes(0, 10, 0) <= 1024      # slack only (holds the all-zero row of the split buffer)
    assert L.hals_als_workspace_bytes(0, 64, 0) <= 1024 + 32 * 72 * 4    # + Gram tiles (implicit, rank 64)
    assert L.hals_als_workspace_bytes(0, 128, 0) <= 1024 + 128 * 72 * 4   # + Gram tiles (implicit, rank 128)
    assert L.hals_als_sse_workspace_bytes() >= 1024 * 8
    assert L.hals_als_workspace_bytes(3, 64, 0) >= 3 * (64 * 64 + 64) * 4
    assert L.hals_als_workspace_bytes(3, 10, 0) >= 3 * (16 * 16 + 16) * 4
    assert L.hals_als_workspace_bytes(0, 64, 1000) >= 1000 * 64 * 4
    assert L.hals_gram_workspace_bytes(128) >= 128 * 128 * 4
    assert L.hals_max_rank() == 128


def test_compute_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import hybrid_als_twotower_recommender_b200 as pkg
    with pytest.raises(nat.NativeError):
        nat.require_cuda()
    assert pkg.ALSModel().initialize_spark() is False      # print + sentinel, like the reference
    with pytest.raises(nat.NativeError):
        pkg.TwoTowerModel(3, 3, 2, 2).build_model()


def test_half_steps_reject_a_negative_or_non_finite_reg():
    """Spark's regParam is >= 0: a negative reg can make A indefinite (silent NaN factors), a NaN one poisons every row.
    Both entry points refuse them before any CUDA call (a zeroed plan, null pointers, no GPU needed); reg = 0 is
    accepted as in Spark (here with no rows, so nothing runs)."""
    L = nat.lib()
    plan = nat.AlsPlan()
    for reg in (-0.1, float("nan"), float("inf")):
        for name, call in (
            ("hals_als_half_step", lambda: L.hals_als_half_step(None, None, None, 0, None, 0, None, 64, reg, 0, 1.0,
                                                                None, ctypes.byref(plan), None, 0, None)),
            ("hals_als_half_step_split", lambda: L.hals_als_half_step_split(None, 0, None, 0, None, None, 64, reg,
                                                                            ctypes.byref(plan), None, 0, None)),
        ):
            assert call() == 1, (name, reg)          # HALS_ERR_INVALID
            assert b"reg must be finite and >= 0" in L.hals_last_error(), (name, reg, L.hals_last_error())
    assert L.hals_als_half_step(None, None, None, 0, None, 0, None, 64, 0.0, 0, 1.0, None, ctypes.byref(plan), None, 0,
                                None) == 0
    assert L.hals_als_half_step_split(None, 0, None, 0, None, None, 64, 0.0, ctypes.byref(plan), None, 0, None) == 0
