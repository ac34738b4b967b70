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
