"""Batched hybrid scoring on B200: replaces the reference's per-user loop of
ALSModel.predict_for_user + TwoTowerModel.predict_for_user + adaptive_fusion + sorted()[:k]
(src/hybrid_system.py:95-116) with two fused passes over an item shard:

  pass 1  hals_score_extrema     per-user (min,max) of both models      [+ min/max all-reduce]
  pass 2  hals_score_blend_topk  blend + per-user top-k, scores never stored
          [+ all-to-all of the per-shard lists and hals_topk_merge when item-sharded]

ALS-only top-k by raw dot product (HybridScorer.topk_dot, behind ALSModel.recommend_for_*) needs no extrema: it is
pass 2 alone, hals_score_topk.
"""
from __future__ import annotations

import torch

from . import _native as nat


def _dist():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized()) else None


def fusion_weights(als_f1: float, tt_f1: float):
    """src/hybrid_system.py:69 -- strict '>'."""
    return (0.8, 0.2) if als_f1 > tt_f1 else (0.2, 0.8)


def sticky_weights(n_users: int, rated, als_f1, tt_f1, f1_init):
    """The weights a loop of get_hybrid_recommendations gives each of n_users users: users `rated` (ascending) have
    their own F1 pair (als_f1[j], tt_f1[j] for rated[j]) and set the sticky F1 scalars; every other user keeps the pair
    of the nearest earlier rated user, or f1_init before the first.  Returns (float32 [n_users, 2] of fusion_weights,
    the F1 pair the loop leaves)."""
    import numpy as np
    fa = np.full(n_users, f1_init[0], np.float64)
    ft = np.full(n_users, f1_init[1], np.float64)
    if len(rated):
        src = np.full(n_users, -1, np.int64)
        src[list(rated)] = np.arange(len(rated))
        src = np.maximum.accumulate(src)
        have = src >= 0
        fa[have] = np.asarray(als_f1, np.float64)[src[have]]
        ft[have] = np.asarray(tt_f1, np.float64)[src[have]]
    better = fa > ft
    hi, lo = fusion_weights(1.0, 0.0)
    w = np.stack([np.where(better, hi, lo), np.where(better, lo, hi)], 1).astype(np.float32).reshape(n_users, 2)
    last = (float(als_f1[-1]), float(tt_f1[-1])) if len(rated) else (float(f1_init[0]), float(f1_init[1]))
    return w, last


def merge_lists(part_idx: torch.Tensor, part_score: torch.Tensor):
    """[P, U, k] partial lists -> [U, k] (score desc, index asc)."""
    L = nat.lib()
    P, U, k = part_idx.shape
    out_idx = torch.empty((U, k), dtype=torch.int32, device=part_idx.device)
    out_score = torch.empty((U, k), dtype=torch.float32, device=part_idx.device)
    nat.check(L.hals_topk_merge(nat.ptr(part_idx.contiguous()), nat.ptr(part_score.contiguous()), P, U, k,
                                nat.ptr(out_idx), nat.ptr(out_score), nat.current_stream()), "hals_topk_merge")
    return out_idx, out_score


def exchange_topk(idx, sc, rank: int, world: int, merge_fn):
    """Cross-shard merge of per-shard top-k lists ([U,k] on every rank, global item numbering).

    All-to-all: rank j receives, from every rank, the lists of ITS equal chunk of the users
    ([world, ceil(U/world), k]) and merges them with `merge_fn` -- each rank ends up owning the final
    top-k of U/world users (0.8 GB received per GPU at config 5 instead of 6.4 GB for an all-gather).
    Single-rank: returns the inputs unchanged."""
    dist = _dist()
    if dist is None or world == 1:
        return idx, sc
    n, k = idx.shape
    per = (n + world - 1) // world
    pad = per * world - n
    if pad:
        idx = torch.cat([idx, torch.full((pad, k), -1, dtype=idx.dtype, device=idx.device)])
        sc = torch.cat([sc, torch.full((pad, k), float("-inf"), dtype=sc.dtype, device=sc.device)])
    ridx, rsc = torch.empty_like(idx), torch.empty_like(sc)
    dist.all_to_all_single(ridx, idx.contiguous())     # chunk j of my lists -> rank j
    dist.all_to_all_single(rsc, sc.contiguous())
    return merge_fn(ridx.view(world, per, k), rsc.view(world, per, k))


def reduce_extrema(ex, world: int):
    """(min_a, max_a, min_t, max_t) per user -> global over all item shards: one MAX all-reduce
    on the sign-flipped minima."""
    dist = _dist()
    if dist is None or world == 1:
        return ex
    sign = torch.tensor([-1.0, 1.0, -1.0, 1.0], device=ex.device, dtype=ex.dtype)
    ex = ex * sign
    dist.all_reduce(ex, op=dist.ReduceOp.MAX)
    return ex * sign


def exclusion_lists(user_pos: torch.Tensor, item_pos: torch.Tensor, n_users: int):
    """(call row, global item index) pairs -> the exclusion CSR of hals_score_blend_topk_excluding:
    (rowptr int64 [n_users+1], items int32, ascending within a row; duplicates kept), on the pairs' device.
    Sorting by item first (stably) makes build_csr's stable grouping by row yield ascending rows."""
    from .csr import build_csr
    user_pos, item_pos = user_pos.reshape(-1).to(torch.int64), item_pos.reshape(-1).to(torch.int64)
    order = torch.sort(item_pos, stable=True).indices
    sh = build_csr(user_pos[order], item_pos[order], None, int(n_users))
    return sh.rowptr, sh.colidx


def _matches(ids: torch.Tensor, query: torch.Tensor):
    """Every (q, p) with ids[p] == query[q] (ids may repeat), by a sort of `ids` and two binary searches."""
    s, order = torch.sort(ids, stable=True)
    lo = torch.searchsorted(s, query, side="left")
    n = torch.searchsorted(s, query, side="right") - lo
    q = torch.repeat_interleave(torch.arange(query.numel(), device=query.device), n)
    first = torch.cumsum(n, 0) - n
    p = order[lo[q] + torch.arange(q.numel(), device=query.device) - first[q]]
    return q, p


def exclusion_lists_by_id(user_ids: torch.Tensor, item_ids: torch.Tensor, pair_users: torch.Tensor,
                          pair_items: torch.Tensor):
    """Exclusion CSR over the rows of a call from (raw user id, raw item id) pairs: row r = the call's r-th user
    (user_ids[r]), item = the position of the item among the call's candidates (item_ids).  A pair whose user is not
    a row or whose item is not a candidate is ignored; a user id listed twice gets its exclusions in both rows (and a
    candidate id listed twice is excluded at both positions)."""
    q, rows = _matches(user_ids.reshape(-1), pair_users.reshape(-1))
    q2, cols = _matches(item_ids.reshape(-1), pair_items.reshape(-1)[q])
    return exclusion_lists(rows[q2], cols, user_ids.numel())


def label_lists_by_id(user_ids: torch.Tensor, item_ids: torch.Tensor, pair_users: torch.Tensor,
                      pair_items: torch.Tensor):
    """Label CSR of a ranking evaluation (hals_ranking_metrics) from (raw user id, raw item id) pairs, in the format of
    exclusion_lists_by_id: row r = user_ids[r], items = positions among the candidates item_ids, ascending within a row,
    duplicates kept.  An item that is not a candidate (unknown to the model, or not present) still belongs to the
    label set: it gets the position len(item_ids) + its rank among the distinct such ids, which no prediction matches.
    Pairs whose user is not a row are ignored."""
    distinct = torch.unique(pair_items.reshape(-1))
    extra = distinct[~torch.isin(distinct, item_ids.reshape(-1))]
    return exclusion_lists_by_id(user_ids, torch.cat([item_ids.reshape(-1), extra]), pair_users, pair_items)


def candidate_lists(candidates, universe_ids, n_rows: int, device):
    """Per-row candidate lists -> the CSR of hals_score_blend_topk_lists: (rowptr int64 [n_rows+1], cand int32), cand
    holding ROWS of the universe (positions in `universe_ids`, which must not repeat an id).

    candidates: None (every universe item, in universe order, for every row); a 2-D integer array [n_rows, L] whose -1
    entries are padding (what ALSModel.recommend_for_all_users(..., as_arrays=True) returns); or a sequence of n_rows
    id sequences (a DataFrame stands for its itemId column).  Each list keeps the first occurrence of a repeated id.
    An id that is not in the universe raises ValueError.  The join and the deduplication run on `device`."""
    import numpy as np
    univ_h = np.array(universe_ids, dtype=np.int64)
    n_univ = len(univ_h)
    if len(np.unique(univ_h)) != n_univ:
        raise ValueError("item_features must list each itemId once")
    if candidates is None:
        rowptr = torch.arange(n_rows + 1, dtype=torch.int64, device=device) * n_univ
        return rowptr, torch.arange(n_univ, dtype=torch.int32, device=device).repeat(n_rows)
    if isinstance(candidates, (np.ndarray, torch.Tensor)) and candidates.ndim == 2:
        if candidates.shape[0] != n_rows:
            raise ValueError(f"candidates has {candidates.shape[0]} rows for {n_rows} users")
        ids = torch.as_tensor(np.asarray(candidates) if isinstance(candidates, np.ndarray) else candidates,
                              device=device).to(torch.int64)
        rows = torch.arange(n_rows, device=device).repeat_interleave(ids.shape[1])
        ids = ids.reshape(-1)
        real = ids != -1
        ids, rows = ids[real], rows[real]
    else:
        lists = list(candidates)
        if len(lists) != n_rows:
            raise ValueError(f"candidates has {len(lists)} lists for {n_rows} users")
        lists = [np.asarray(c["itemId"].values if hasattr(c, "columns") else list(c), dtype=np.int64).reshape(-1)
                 for c in lists]
        lens = np.fromiter((len(c) for c in lists), dtype=np.int64, count=n_rows)
        flat = np.concatenate(lists) if lens.sum() else np.zeros(0, np.int64)
        ids = torch.from_numpy(flat).to(device)
        rows = torch.repeat_interleave(torch.arange(n_rows, device=device), torch.from_numpy(lens).to(device))
    univ = torch.from_numpy(univ_h).to(device)
    srt, order = torch.sort(univ)
    pos = torch.searchsorted(srt, ids).clamp(max=max(n_univ - 1, 0))
    ok = srt[pos] == ids if n_univ else torch.zeros_like(ids, dtype=torch.bool)
    if not bool(ok.all()):
        raise ValueError(f"candidate ids missing from item_features: {ids[~ok][:5].tolist()}")
    urow = order[pos]
    # first occurrence of each (row, item): a stable sort keeps equal keys in list order
    sk, so = torch.sort(rows * max(n_univ, 1) + urow, stable=True)
    first = torch.ones_like(sk, dtype=torch.bool)
    first[1:] = sk[1:] != sk[:-1]
    keep = torch.empty_like(first)
    keep[so] = first
    rows, urow = rows[keep], urow[keep]
    rowptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=device)
    rowptr[1:] = torch.cumsum(torch.bincount(rows, minlength=n_rows), 0)
    return rowptr, urow.to(torch.int32)


def blend_topk_lists(Ua, Ia, Ut, It, rowptr, cand, topk: int, *, w_als: float = 0.0, w_tt: float = 0.0,
                     row_weights=None, raw: bool = False, user_known=None, item_known=None, als_fallback=None):
    """hals_score_blend_topk_lists: per-row candidate lists (see candidate_lists), each row min-max blended over its
    own list (raw=True: w_als*s_als + w_tt*s_tt) and cut to its best `topk`.  Ua [n_rows, ka] / Ut [n_rows, kt] are the
    rows' user operands, Ia [n, ka] / It [n, kt] the candidate rows' (one model may be None); user_known [n_rows] /
    item_known [n] (bool or uint8) mark ids known to ALS, the others take als_fallback [n] as their ALS score;
    row_weights [n_rows, 2] overrides (w_als, w_tt) row by row.  Returns (positions into cand int32, scores float32),
    both [n_rows, topk], padded with -1 / -inf; ties go to the lower position."""
    L = nat.lib()
    ref_u = Ua if Ua is not None else Ut
    ref_i = Ia if Ia is not None else It
    if ref_u is None or ref_i is None:
        raise ValueError("need the operands of at least one model")
    Ua, Ia, Ut, It = (None if t is None else t.contiguous() for t in (Ua, Ia, Ut, It))
    n_rows, n_cand_rows = int(ref_u.shape[0]), int(ref_i.shape[0])
    ka = 0 if Ua is None else int(Ua.shape[1])
    kt = 0 if Ut is None else int(Ut.shape[1])
    dev = ref_u.device
    if (Ua is None) != (Ia is None) or (Ut is None) != (It is None):
        raise ValueError("each model needs both its user and its item operand")
    for t, rows, k in ((Ua, n_rows, ka), (Ut, n_rows, kt), (Ia, n_cand_rows, ka), (It, n_cand_rows, kt)):
        if t is not None and (t.dtype != torch.float32 or t.dim() != 2 or tuple(t.shape) != (rows, k) or t.device != dev):
            raise ValueError("operands must be float32 [n_rows, k] (users) and [n, k] (items) on one device")
    if rowptr.dtype != torch.int64 or rowptr.numel() != n_rows + 1 or cand.dtype != torch.int32:
        raise ValueError("candidate lists must be (rowptr int64 [n_rows+1], cand int32)")

    def vec(t, n, dtype, what):
        if t is None:
            return None
        t = t.to(dtype) if t.dtype == torch.bool else t
        if t.dtype != dtype or t.numel() != n or t.device != dev:
            raise ValueError(f"{what} must be {dtype} [{n}] on the operands' device")
        return t.contiguous()
    user_known = vec(user_known, n_rows, torch.uint8, "user_known")
    item_known = vec(item_known, n_cand_rows, torch.uint8, "item_known")
    als_fallback = vec(als_fallback, n_cand_rows, torch.float32, "als_fallback")
    row_weights = vec(row_weights, 2 * n_rows, torch.float32, "row_weights")
    rowptr, cand = rowptr.contiguous(), cand.contiguous()
    if cand.numel() == 0:                   # a valid pointer for an empty list set
        cand = torch.zeros(1, dtype=torch.int32, device=dev)
    n_total = int(rowptr[-1].item()) if n_rows else 0
    ws = torch.empty(int(L.hals_score_lists_workspace_bytes(n_total, int(topk))), dtype=torch.uint8, device=dev)
    pos = torch.empty((n_rows, int(topk)), dtype=torch.int32, device=dev)
    score = torch.empty((n_rows, int(topk)), dtype=torch.float32, device=dev)

    def op(t):
        return (None, 0) if t is None else (nat.ptr(t), t.stride(0))
    nat.check(L.hals_score_blend_topk_lists(*op(Ua), *op(Ia), ka, *op(Ut), *op(It), kt, n_rows, n_total,
                                            nat.ptr(rowptr), nat.ptr(cand), nat.ptr(user_known), nat.ptr(item_known),
                                            nat.ptr(als_fallback), nat.ptr(row_weights), float(w_als), float(w_tt),
                                            int(bool(raw)), int(topk), nat.ptr(pos), nat.ptr(score), nat.ptr(ws),
                                            ws.numel(), nat.current_stream()), "hals_score_blend_topk_lists")
    return pos, score


def shard_items(n_items: int, rank: int, world: int):
    """Contiguous equal item shards (item-sharded scoring): [begin, end) of this rank."""
    per = (n_items + world - 1) // world
    return min(n_items, rank * per), min(n_items, (rank + 1) * per)


class HybridScorer:
    """Holds the four operand matrices of one item shard in HBM (fp32, row-major)."""

    def __init__(self, Ua, Ia, Ut, It, item_offset: int = 0, dist_rank: int = 0, world: int = 1):
        self.Ua, self.Ia, self.Ut, self.It = (None if t is None else t.contiguous() for t in (Ua, Ia, Ut, It))
        ref_u = self.Ua if self.Ua is not None else self.Ut
        ref_i = self.Ia if self.Ia is not None else self.It
        self.n_users, self.n_items = int(ref_u.shape[0]), int(ref_i.shape[0])
        self.ka = 0 if self.Ua is None else int(self.Ua.shape[1])
        self.kt = 0 if self.Ut is None else int(self.Ut.shape[1])
        self.device = ref_u.device
        self.item_offset, self.rank, self.world = int(item_offset), dist_rank, world
        self._ws = None

    def _ops(self, u0, u1):
        def sl(t):
            return (None, 0) if t is None else (nat.ptr(t[u0:u1]), t.stride(0))
        (ua, uas), (ut, uts) = sl(self.Ua), sl(self.Ut)
        ia = (None, 0) if self.Ia is None else (nat.ptr(self.Ia), self.Ia.stride(0))
        it = (None, 0) if self.It is None else (nat.ptr(self.It), self.It.stride(0))
        return ua, uas, ia[0], ia[1], self.ka, ut, uts, it[0], it[1], self.kt

    def _workspace(self, n_users: int, k: int, kt: int | None = None) -> torch.Tensor:
        kt = self.kt if kt is None else kt
        need = int(nat.lib().hals_score_workspace_bytes(n_users, self.n_items, self.ka, kt, k))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    def flagged_users(self, n_users: int, k: int, dot: bool = False) -> int:
        """Users of the last call (same n_users, k) that the tensor-core path re-ran exactly; -1 if the call
        took the CUDA-core path.  dot=True: the last call was topk_dot."""
        off = int(nat.lib().hals_score_flag_counter_offset(n_users, self.n_items, self.ka, 0 if dot else self.kt, k))
        if off < 0 or self._ws is None:
            return -1
        return int(self._ws[off:off + 4].view(torch.int32).item())

    def extrema(self, u0: int = 0, u1: int | None = None) -> torch.Tensor:
        """[U,4] = (min_als, max_als, min_tt, max_tt) per user over ALL items (all shards)."""
        L = nat.lib()
        u1 = self.n_users if u1 is None else u1
        ex = torch.empty((u1 - u0, 4), dtype=torch.float32, device=self.device)
        ws = self._workspace(u1 - u0, 0)
        nat.check(L.hals_score_extrema(*self._ops(u0, u1), u1 - u0, self.n_items, nat.ptr(ex), nat.ptr(ws),
                                       ws.numel(), nat.current_stream()), "hals_score_extrema")
        ex = reduce_extrema(ex, self.world)
        return ex

    def topk_local(self, extrema, k, w_als, w_tt, u0=0, u1=None, exclude=None):
        """Top-k of this item shard only (global item numbering via item_offset).  exclude: optional (rowptr, items)
        exclusion CSR over ALL of the scorer's users (see exclusion_lists; global item numbering, so every shard takes
        the same lists): the items of a user's row are left out of its list (hals_score_blend_topk_excluding)."""
        L = nat.lib()
        u1 = self.n_users if u1 is None else u1
        n = u1 - u0
        self._workspace(n, k)
        idx = torch.empty((n, k), dtype=torch.int32, device=self.device)
        sc = torch.empty((n, k), dtype=torch.float32, device=self.device)
        head = (*self._ops(u0, u1), n, self.n_items, nat.ptr(extrema), float(w_als), float(w_tt), int(k),
                self.item_offset, nat.ptr(idx), nat.ptr(sc))
        tail = (nat.ptr(self._ws), self._ws.numel(), nat.current_stream())
        if exclude is None:
            nat.check(L.hals_score_blend_topk(*head, *tail), "hals_score_blend_topk")
        else:
            rowptr, items = self._check_exclude(exclude)
            nat.check(L.hals_score_blend_topk_excluding(*head, nat.ptr(rowptr[u0:]), nat.ptr(items), *tail),
                      "hals_score_blend_topk_excluding")
        return idx, sc

    def _check_exclude(self, exclude):
        rowptr, items = exclude
        if rowptr.dtype != torch.int64 or items.dtype != torch.int32 or rowptr.numel() != self.n_users + 1:
            raise ValueError("exclude must be (rowptr int64 [n_users+1], items int32) over the scorer's users")
        if rowptr.device != self.device or items.device != self.device:
            raise ValueError("exclude must live on the scorer's device")
        rowptr, items = rowptr.contiguous(), items.contiguous()
        if items.numel() == 0:            # a valid pointer for an empty list set
            items = torch.zeros(1, dtype=torch.int32, device=self.device)
        return rowptr, items

    def recommend(self, k: int, w_als: float, w_tt: float, u0: int = 0, u1: int | None = None, exclude=None):
        """Final top-k for users [u0,u1).  Item-sharded runs return, on every rank, the merged
        lists of ITS slice of those users (rank r owns the r-th equal chunk) -- see
        `user_slice`.  exclude: as for topk_local."""
        u1 = self.n_users if u1 is None else u1
        ex = self.extrema(u0, u1)
        idx, sc = self.topk_local(ex, k, w_als, w_tt, u0, u1, exclude=exclude)
        return exchange_topk(idx, sc, self.rank, self.world, merge_lists)

    def topk_dot(self, k: int, u0: int = 0, u1: int | None = None, exclude=None):
        """The raw counterpart of `recommend`: for users [u0,u1) the k items with the largest ALS dot product
        <Ua[u], Ia[i]> (fp32; score descending, then lower item index; padded with -1 / -inf), in one pass over the
        items (hals_score_topk: no extrema, no scaling).  The tower operands are ignored.  exclude and the item-sharded
        result: as for `recommend`."""
        if self.Ua is None or self.Ia is None:
            raise ValueError("topk_dot needs the ALS operands (Ua, Ia)")
        L = nat.lib()
        u1 = self.n_users if u1 is None else u1
        n = u1 - u0
        self._workspace(n, k, kt=0)
        idx = torch.empty((n, k), dtype=torch.int32, device=self.device)
        sc = torch.empty((n, k), dtype=torch.float32, device=self.device)
        xr = xi = None
        if exclude is not None:
            xr, xi = self._check_exclude(exclude)
            xr = xr[u0:]
        nat.check(L.hals_score_topk(nat.ptr(self.Ua[u0:u1]), self.Ua.stride(0), nat.ptr(self.Ia), self.Ia.stride(0),
                                    self.ka, n, self.n_items, int(k), self.item_offset, nat.ptr(xr), nat.ptr(xi),
                                    nat.ptr(idx), nat.ptr(sc), nat.ptr(self._ws), self._ws.numel(),
                                    nat.current_stream()), "hals_score_topk")
        return exchange_topk(idx, sc, self.rank, self.world, merge_lists)

    def user_slice(self, u0, u1):
        n = u1 - u0
        per = (n + self.world - 1) // self.world
        return u0 + self.rank * per, min(u1, u0 + (self.rank + 1) * per)
