"""CPU: building the per-user exclusion lists of hals_score_blend_topk_excluding (scoring.exclusion_lists and the
(userId, itemId) -> CSR mapping behind recommend_batch(exclude=...)) on CPU tensors."""
import numpy as np
import torch

import hybrid_als_twotower_recommender_b200  # noqa: F401  (import shim)
from hybrid_als_twotower_recommender_b200 import scoring


def rows_of(rowptr, items):
    rp, it = rowptr.numpy(), items.numpy()
    return [it[rp[r]:rp[r + 1]].tolist() for r in range(len(rp) - 1)]


def test_exclusion_lists_sorted_rows_with_duplicates():
    rng = np.random.default_rng(0)
    U, n = 37, 2000
    u = rng.integers(0, U, n)
    i = rng.integers(0, 500, n)
    u[:5], i[:5] = 3, 42                              # the same pair five times
    u = np.concatenate([u, [11]]); i = np.concatenate([i, [7]])
    rowptr, items = scoring.exclusion_lists(torch.from_numpy(u), torch.from_numpy(i), U)
    assert rowptr.dtype == torch.int64 and items.dtype == torch.int32
    assert rowptr.shape == (U + 1,) and int(rowptr[0]) == 0 and int(rowptr[-1]) == len(u)
    got = rows_of(rowptr, items)
    for r in range(U):
        assert got[r] == sorted(i[u == r].tolist()), r          # ascending, duplicates kept
    assert got[3].count(42) >= 5


def test_exclusion_lists_empty_and_unused_rows():
    rowptr, items = scoring.exclusion_lists(torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64), 4)
    assert rowptr.tolist() == [0, 0, 0, 0, 0] and items.numel() == 0
    rowptr, items = scoring.exclusion_lists(torch.tensor([2, 2, 0]), torch.tensor([9, 1, 5]), 4)
    assert rows_of(rowptr, items) == [[5], [], [1, 9], []]


def test_exclusion_by_id_maps_users_and_candidates():
    user_ids = torch.tensor([100, 7, 55, 7, 300])          # user 7 listed twice: rows 1 and 3
    cand_ids = torch.tensor([40, 10, 30, 20, 50])           # candidate order is not sorted
    pu = torch.tensor([7, 7, 100, 55, 999, 55, 100, 7, 300])
    pi = torch.tensor([20, 40, 50, 30, 10, 12345, 50, 20, 10])   # 999: unknown user; 12345: not a candidate
    rowptr, items = scoring.exclusion_lists_by_id(user_ids, cand_ids, pu, pi)
    got = rows_of(rowptr, items)
    # positions among the candidates: 40 -> 0, 10 -> 1, 30 -> 2, 20 -> 3, 50 -> 4
    assert got == [[4, 4], [0, 3, 3], [2], [0, 3, 3], [1]]


def test_exclusion_by_id_random_against_a_python_loop():
    rng = np.random.default_rng(5)
    user_ids = rng.integers(0, 60, 80)                      # repeats
    cand_ids = rng.permutation(400)[:300] * 3 + 1
    pu = rng.integers(0, 70, 3000)
    pi = rng.integers(0, 1300, 3000)
    rowptr, items = scoring.exclusion_lists_by_id(*(torch.from_numpy(np.asarray(a, np.int64))
                                                    for a in (user_ids, cand_ids, pu, pi)))
    pos = {int(c): p for p, c in enumerate(cand_ids)}
    want = [sorted(pos[int(b)] for a, b in zip(pu, pi) if a == uid and int(b) in pos) for uid in user_ids]
    assert rows_of(rowptr, items) == want
