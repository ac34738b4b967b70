"""ALS sweeps on B200: the replacement for `ALS(...).fit(df)` (src/als_model.py:52-62).

One process per GPU.  Rank r owns an nnz-balanced contiguous range of user rows of R and
of item rows of R^T (CSR shards resident in HBM) plus full replicas of both factor
matrices.  A sweep is   item half-step -> all-gather(Y) -> user half-step -> all-gather(X)
(Spark's loop order; ALS.scala train).  The half-step itself is one C-ABI call
(hals_als_half_step, or hals_als_half_step_nonnegative for Spark's nonnegative=True); the all-gather is NCCL through
torch.distributed.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as nat
from .csr import AlsPlanHandle, CsrShard, balanced_row_bounds, build_csr


def _dist():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized()) else None


def all_gather_rows(full: torch.Tensor, bounds, rank: int, world: int, group=None, cache: dict | None = None):
    """All-gather of uneven contiguous row shards of `full` ([n,k], every rank holds the whole
    buffer, its own rows freshly written).  Shards are padded to the largest one so a single
    equal-size all-gather moves them (NCCL ring/NVLS over NVLink), then one row gather unpacks
    them in place.  `cache` (a dict owned by the caller) keeps the staging buffers and the unpack
    index between calls: three launches per call instead of a dozen, no allocation."""
    dist = _dist()
    if dist is None or world == 1:
        return
    k = full.shape[1]
    key = (full.data_ptr(), tuple(int(b) for b in bounds), k)
    st = cache.get(key) if cache is not None else None
    if st is None:
        sizes = [int(bounds[r + 1] - bounds[r]) for r in range(world)]
        mx = max(sizes)
        if mx == 0:
            return
        # row n of `full` lives at recv[(owner, n - bounds[owner])]
        idx = torch.cat([torch.arange(sizes[r], dtype=torch.int64) + r * mx for r in range(world)]).to(full.device)
        st = {"sizes": sizes, "mx": mx, "idx": idx,
              "send": torch.zeros((mx, k), dtype=full.dtype, device=full.device),
              "recv": torch.empty((world * mx, k), dtype=full.dtype, device=full.device)}
        if cache is not None:
            cache[key] = st
    sizes, mx, send, recv = st["sizes"], st["mx"], st["send"], st["recv"]
    send[: sizes[rank]].copy_(full[int(bounds[rank]): int(bounds[rank + 1])])
    if full.is_cuda:
        dist.all_gather_into_tensor(recv, send, group=group)
    else:  # gloo (CPU tests)
        parts = list(recv.view(world, mx, k).unbind(0))
        dist.all_gather(parts, send, group=group)
    torch.index_select(recv, 0, st["idx"], out=full)


def route_to_owners(users, items, ratings, key, bounds, world: int):
    """All-to-all of rating triples to the rank that owns row `key` (bounds: [world+1] row ranges).  Triples arrive
    grouped by source rank, each group in its original order, so contiguous input slices reproduce the single-process
    rating order inside every row."""
    dist = _dist()
    dev = key.device
    cuts = torch.as_tensor(np.asarray(bounds[1:-1]), device=dev, dtype=key.dtype)
    owner = torch.bucketize(key, cuts, right=True)
    order = torch.sort(owner, stable=True).indices
    send_counts = torch.bincount(owner, minlength=world)
    recv_counts = torch.empty_like(send_counts)
    dist.all_to_all_single(recv_counts, send_counts)
    sc, rc = send_counts.tolist(), recv_counts.tolist()
    out = []
    for t in (users, items, ratings):
        src = t[order].contiguous()
        dst = torch.empty(int(sum(rc)), dtype=t.dtype, device=dev)
        dist.all_to_all_single(dst, src, output_split_sizes=rc, input_split_sizes=sc)
        out.append(dst)
    return out


def native_half_step(shard: CsrShard, plan: AlsPlanHandle, src: torch.Tensor, dst_full: torch.Tensor,
                     k: int, reg: float, implicit: bool, alpha: float, gram: torch.Tensor | None,
                     nonnegative: bool = False, n_capped: torch.Tensor | None = None):
    """dst_full[row_begin:row_end] = solve(shard, src).  The only compute path (CUDA).  nonnegative=True: the
    bound-constrained solve (x >= 0); rows that reach its iteration cap are added to n_capped (int32 [1], optional)."""
    L = nat.lib()
    dst = dst_full[shard.row_begin: shard.row_end]
    assert src.is_contiguous() and dst.is_contiguous() and src.dtype == torch.float32
    if nonnegative:
        assert n_capped is None or (n_capped.dtype == torch.int32 and n_capped.device == dst.device)
        nat.check(L.hals_als_half_step_nonnegative(
            nat.ptr(shard.rowptr), nat.ptr(shard.colidx), nat.ptr(shard.vals), shard.n_rows,
            nat.ptr(src), src.shape[0], nat.ptr(dst), k, float(reg), int(bool(implicit)), float(alpha),
            nat.ptr(gram) if gram is not None else None, plan.struct, nat.ptr(plan.workspace),
            plan.workspace_bytes, nat.current_stream(), nat.ptr(n_capped)), "hals_als_half_step_nonnegative")
        return
    nat.check(L.hals_als_half_step(
        nat.ptr(shard.rowptr), nat.ptr(shard.colidx), nat.ptr(shard.vals), shard.n_rows,
        nat.ptr(src), src.shape[0], nat.ptr(dst), k, float(reg), int(bool(implicit)), float(alpha),
        nat.ptr(gram) if gram is not None else None, plan.struct, nat.ptr(plan.workspace),
        plan.workspace_bytes, nat.current_stream()), "hals_als_half_step")


class SplitFactors:
    """Rank-64 / rank-128 factors in the form the tensor-core kernels gather: bf16 [rows + 1, 2k] = [hi(k) | lo(k)], stored
    PADDED BY OWNER RANK -- rank q's rows [bounds[q], bounds[q+1]) live at [q * mx, q * mx + n_q) -- so that the
    all-gather of the freshly solved rows is one in-place equal-size NCCL all-gather (no pack, no unpack, no
    re-split of the whole matrix on every rank).  The last row (index world * mx) is all zero: the ragged tail of a
    32-rating chunk gathers it."""

    def __init__(self, bounds, world: int, device, k: int = 64):
        self.bounds = np.asarray(bounds, dtype=np.int64)
        self.world = world
        self.k = int(k)
        self.sizes = np.diff(self.bounds)
        self.mx = int(max(1, self.sizes.max()))
        self.n_rows = world * self.mx                      # index of the zero row
        self.hl = torch.zeros((self.n_rows + 1, 2 * self.k), dtype=torch.bfloat16, device=device)
        # natural row -> padded row
        owner = np.searchsorted(self.bounds, np.arange(int(self.bounds[-1])), side="right") - 1
        self.pad_of_h = (owner * self.mx + np.arange(int(self.bounds[-1])) - self.bounds[owner]).astype(np.int64)
        self.pad_of = torch.from_numpy(self.pad_of_h).to(device)

    def segment(self, rank: int) -> torch.Tensor:
        return self.hl[rank * self.mx: (rank + 1) * self.mx]

    def load(self, full_fp32: torch.Tensor):
        """Split a complete natural-order fp32 factor matrix into the padded layout (once, at initialisation)."""
        L = nat.lib()
        tmp = torch.empty((full_fp32.shape[0], 2 * self.k), dtype=torch.bfloat16, device=full_fp32.device)
        nat.check(L.hals_als_split_factors(nat.ptr(full_fp32), full_fp32.shape[0], self.k, nat.ptr(tmp), nat.current_stream()),
                  "hals_als_split_factors")
        self.hl[: self.n_rows].zero_()
        self.hl.index_copy_(0, self.pad_of, tmp)

    def all_gather(self, rank: int, group=None):
        dist = _dist()
        if dist is None or self.world == 1:
            return
        dist.all_gather_into_tensor(self.hl[: self.n_rows], self.segment(rank), group=group)   # in place


def native_half_step_split(shard: CsrShard, plan: AlsPlanHandle, colidx_pad: torch.Tensor, src: SplitFactors,
                           dst_full: torch.Tensor, dst: SplitFactors, rank: int, reg: float):
    """Ranks 64 and 128, explicit: gathers from `src` (split, padded), writes this rank's rows of dst_full (fp32, natural order)
    and of `dst` (split, padded)."""
    L = nat.lib()
    out = dst_full[shard.row_begin: shard.row_end]
    nat.check(L.hals_als_half_step_split(
        nat.ptr(colidx_pad), shard.n_rows, nat.ptr(src.hl), src.n_rows, nat.ptr(out), nat.ptr(dst.segment(rank)), src.k,
        float(reg), plan.struct, nat.ptr(plan.workspace), plan.workspace_bytes, nat.current_stream()), "hals_als_half_step_split")


def native_gram(src: torch.Tensor, out: torch.Tensor, workspace: torch.Tensor):
    L = nat.lib()
    nat.check(L.hals_gram(nat.ptr(src), src.shape[0], src.shape[1], nat.ptr(out), nat.ptr(workspace),
                          workspace.numel(), nat.current_stream()), "hals_gram")


class AlsEngine:
    """Device-resident state of one ALS fit on this rank."""

    def __init__(self, users, items, ratings, n_users: int, n_items: int, rank: int, reg: float,
                 implicit: bool = False, alpha: float = 1.0, device=None, seg_len: int | None = None,
                 dist_rank: int = 0, world: int = 1, half_step=None, make_plans: bool = True,
                 partitioned: bool = False, nonnegative: bool = False):
        """users / items / ratings: the COO triples.  partitioned=False: every rank passes the WHOLE matrix and keeps
        its row shards.  partitioned=True (world > 1): every rank passes only ITS slice of the triples (rank q the q-th
        contiguous chunk, so that the concatenation over ranks is the original order); row counts are all-reduced
        and the triples are routed to the owner of their user row (for R) and of their item row (for R^T) with one
        all-to-all each -- 1/N of the upload and of the sort per rank.
        nonnegative=True: Spark's nonnegative=True, every factor row is the nonnegative least-squares solution of its
        normal equations (hals_als_half_step_nonnegative, fp32 factors only -- no split form).  An injected half_step
        then receives nonnegative=True as a keyword."""
        import os
        import time
        _t = [time.perf_counter()]
        _timing = os.environ.get("HALS_ENGINE_TIMING") == "1"

        def _mark(what):
            if _timing:
                torch.cuda.synchronize()
                now = time.perf_counter()
                if dist_rank == 0:
                    print(f"[als_engine] {what}: {(now - _t[0]) * 1e3:.2f} ms", flush=True)
                _t[0] = now
        self.k, self.reg, self.implicit, self.alpha = int(rank), float(reg), bool(implicit), float(alpha)
        self.nonnegative = bool(nonnegative)
        self.n_users, self.n_items = int(n_users), int(n_items)
        self.rank, self.world = dist_rank, world
        self.device = torch.device(device) if device is not None else torch.device("cuda")
        self._half_step = half_step or native_half_step
        users = torch.as_tensor(users).to(self.device)
        items = torch.as_tensor(items).to(self.device)
        ratings = torch.as_tensor(ratings).to(self.device, torch.float32)
        self.nnz_total = int(users.numel())
        # cost-balanced contiguous row ranges (identical on every rank: computed from global counts)
        ucnt_d = torch.bincount(users.to(torch.int64), minlength=n_users)
        icnt_d = torch.bincount(items.to(torch.int64), minlength=n_items)
        partitioned = bool(partitioned) and world > 1
        if partitioned:
            dist = _dist()
            dist.all_reduce(ucnt_d)
            dist.all_reduce(icnt_d)
            self.nnz_total = int(ucnt_d.sum().item())
        ucnt, icnt = ucnt_d.cpu().numpy(), icnt_d.cpu().numpy()
        _mark("upload + row counts")
        self.user_bounds = balanced_row_bounds(ucnt, world, k=self.k)
        self.item_bounds = balanced_row_bounds(icnt, world, k=self.k)
        self.user_present = torch.from_numpy(ucnt > 0).to(self.device)
        self.item_present = torch.from_numpy(icnt > 0).to(self.device)
        ub, ue = int(self.user_bounds[dist_rank]), int(self.user_bounds[dist_rank + 1])
        ib, ie = int(self.item_bounds[dist_rank]), int(self.item_bounds[dist_rank + 1])
        if partitioned:
            ru, ri, rr = route_to_owners(users, items, ratings, users, self.user_bounds, world)
            self.R = build_csr(ru, ri, rr, n_users, ub, ue, counts=ucnt_d)
            ru, ri, rr = route_to_owners(users, items, ratings, items, self.item_bounds, world)
            self.Rt = build_csr(ri, ru, rr, n_items, ib, ie, counts=icnt_d)
            del ru, ri, rr
        else:
            self.R = build_csr(users, items, ratings, n_users, ub, ue, counts=ucnt_d)    # user rows -> item columns
            self.Rt = build_csr(items, users, ratings, n_items, ib, ie, counts=icnt_d)   # item rows -> user columns
        _mark("routing + CSR build")
        self.plan_R = self.plan_Rt = None
        if make_plans:
            self.plan_R = AlsPlanHandle(self.R, self.k, seg_len, n_src=n_items, implicit=self.implicit, alpha=self.alpha)
            self.plan_Rt = AlsPlanHandle(self.Rt, self.k, seg_len, n_src=n_users, implicit=self.implicit, alpha=self.alpha)
        _mark("work plans")
        self.X = torch.zeros((n_users, self.k), dtype=torch.float32, device=self.device)
        self.Y = torch.zeros((n_items, self.k), dtype=torch.float32, device=self.device)
        self.gram = None
        self.gram_ws = None
        # ranks 64 and 128, explicit, native kernels: factors also live in split (bf16 hi|lo), owner-padded form; half-steps
        # exchange the split rows in place and the fp32 replicas of the OTHER ranks' rows are refreshed lazily
        self.split = None
        self._fp32_stale = False
        if (self.k in (64, 128) and not self.implicit and not self.nonnegative and self.device.type == "cuda"
                and self._half_step is native_half_step and make_plans):
            self.split = {"X": SplitFactors(self.user_bounds, world, self.device, self.k),
                          "Y": SplitFactors(self.item_bounds, world, self.device, self.k)}
            self.colidx_pad_R = self.split["Y"].pad_of[self.R.colidx.long()].to(torch.int32) if world > 1 else self.R.colidx
            self.colidx_pad_Rt = self.split["X"].pad_of[self.Rt.colidx.long()].to(torch.int32) if world > 1 else self.Rt.colidx
        _mark("factor buffers + column remap")
        # rows of nonnegative half-steps that reached the solver's iteration cap, summed by the kernels
        self._n_capped = None
        if self.nonnegative and self.device.type == "cuda" and self._half_step is native_half_step:
            self._n_capped = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._gather_cache = {}
        self._graphs = None                # (item, user) CUDA graphs after enable_graphs()
        self._graph_launch_counts = (0, 0)
        self.graph_launches = 0            # kernels of this library launched through graph replays
        if self.implicit:
            self.gram = torch.zeros((self.k, self.k), dtype=torch.float32, device=self.device)
            if self.device.type == "cuda":
                self.gram_ws = torch.empty(int(nat.lib().hals_gram_workspace_bytes(self.k)), dtype=torch.uint8,
                                           device=self.device)

    # -- factors ---------------------------------------------------------------------------
    def set_user_factors(self, X0):
        self.X.copy_(torch.as_tensor(X0, dtype=torch.float32).to(self.device))
        self._after_user_init()

    def _after_user_init(self):
        if self.split is not None:
            # users without ratings are absent from a Spark model; the stateless half-step zeroes their rows on every
            # call, the split-form path never touches them: zero them once
            self.X[~self.user_present] = 0
            self.split["X"].load(self.X)
            self._fp32_stale = False

    def init_user_factors(self, seed: int = 0):
        """Spark's `initialize` distribution: N(0,1) rows scaled to unit L2 norm.  Drawn on the device the engine runs on
        (CUDA: Philox, the same values on every rank and run for a given seed; drawing 9 M normals on the host and
        uploading them cost more than a whole sweep on the MovieLens-20M shape)."""
        g = torch.Generator(device=self.device).manual_seed(int(seed))
        f = torch.randn((self.n_users, self.k), generator=g, dtype=torch.float32, device=self.device)
        f = f / f.norm(dim=1, keepdim=True).clamp_min(1e-30)
        self.X.copy_(f)
        self._after_user_init()

    def nonneg_capped_rows(self) -> int:
        """Rows, over every nonnegative half-step this engine ran, whose NNLS solve reached its iteration cap (each
        keeps its last iterate with x >= 0).  0 when nonnegative=False."""
        return 0 if self._n_capped is None else int(self._n_capped.item())

    def _solve(self, shard, plan, src, dst, gram):
        if not self.nonnegative:
            self._half_step(shard, plan, src, dst, self.k, self.reg, self.implicit, self.alpha, gram)
        elif self._half_step is native_half_step:
            native_half_step(shard, plan, src, dst, self.k, self.reg, self.implicit, self.alpha, gram,
                             nonnegative=True, n_capped=self._n_capped)
        else:   # injected half-step (CPU tests): told only when the option is set, so plain callables keep working
            self._half_step(shard, plan, src, dst, self.k, self.reg, self.implicit, self.alpha, gram, nonnegative=True)

    def _gram_of(self, src):
        if not self.implicit:
            return None
        if self._half_step is native_half_step:
            native_gram(src, self.gram, self.gram_ws)
        else:  # injected half-step (CPU tests): it computes its own Gram
            return None
        return self.gram

    # -- one sweep = item half-step, then user half-step (Spark's order) ---------------------
    def _item_half_eager(self):
        if self.split is not None:
            native_half_step_split(self.Rt, self.plan_Rt, self.colidx_pad_Rt, self.split["X"], self.Y, self.split["Y"],
                                   self.rank, self.reg)
            self.split["Y"].all_gather(self.rank)
            self._fp32_stale = self.world > 1
            return
        self._solve(self.Rt, self.plan_Rt, self.X, self.Y, self._gram_of(self.X))
        all_gather_rows(self.Y, self.item_bounds, self.rank, self.world, cache=self._gather_cache)

    def _user_half_eager(self):
        if self.split is not None:
            native_half_step_split(self.R, self.plan_R, self.colidx_pad_R, self.split["Y"], self.X, self.split["X"],
                                   self.rank, self.reg)
            self.split["X"].all_gather(self.rank)
            self._fp32_stale = self.world > 1
            return
        self._solve(self.R, self.plan_R, self.Y, self.X, self._gram_of(self.Y))
        all_gather_rows(self.X, self.user_bounds, self.rank, self.world, cache=self._gather_cache)

    def sync_factors(self):
        """Sharded split-form runs exchange only the split rows during the sweeps: bring the fp32 replicas of the other
        ranks' rows up to date (one all-gather per matrix; called by fit() and rmse())."""
        if self.split is not None and self.world > 1 and self._fp32_stale:
            all_gather_rows(self.Y, self.item_bounds, self.rank, self.world, cache=self._gather_cache)
            all_gather_rows(self.X, self.user_bounds, self.rank, self.world, cache=self._gather_cache)
        self._fp32_stale = False

    def item_half_step(self):
        if self._graphs is not None:
            self._graphs[0].replay()
            self.graph_launches += self._graph_launch_counts[0]
            self._fp32_stale = self.split is not None and self.world > 1
        else:
            self._item_half_eager()

    def user_half_step(self):
        if self._graphs is not None:
            self._graphs[1].replay()
            self.graph_launches += self._graph_launch_counts[1]
            self._fp32_stale = self.split is not None and self.world > 1
        else:
            self._user_half_eager()

    def enable_graphs(self) -> bool:
        """Captures each half-step (its kernels and, when sharded, the NCCL all-gather) into a CUDA graph: a sweep
        becomes two graph launches, which matters once a rank's share of the sweep is shorter than the host's
        launch latency (c2 on 8 GPUs).  Factors are left untouched.  Returns False -- and stays on plain launches --
        if anything about the capture fails; every rank must call it (the capture includes collectives)."""
        if self._graphs is not None:
            return True
        if self.device.type != "cuda" or self._half_step is not native_half_step or self.plan_R is None:
            return False
        keep = (self.X.clone(), self.Y.clone(), None if self._n_capped is None else self._n_capped.clone())
        keep_split = None if self.split is None else (self.split["X"].hl.clone(), self.split["Y"].hl.clone(), self._fp32_stale)
        try:
            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):          # warm-up off the default stream (staging buffers, lazy inits)
                self._item_half_eager()
                self._user_half_eager()
            torch.cuda.current_stream(self.device).wait_stream(side)
            torch.cuda.synchronize(self.device)
            graphs, counts = [], []
            for fn in (self._item_half_eager, self._user_half_eager):
                g = torch.cuda.CUDAGraph()
                l0 = nat.launch_count()
                with torch.cuda.graph(g, capture_error_mode="thread_local"):
                    fn()
                counts.append(nat.launch_count() - l0)
                graphs.append(g)
            self._graphs, self._graph_launch_counts = tuple(graphs), tuple(counts)
            ok = True
        except Exception as exc:  # noqa: BLE001 - any capture problem means: keep launching eagerly
            print(f"[als_engine] CUDA graph capture unavailable ({type(exc).__name__}: {exc}); using plain launches")
            self._graphs, ok = None, False
            torch.cuda.synchronize(self.device)
        self.X.copy_(keep[0])
        self.Y.copy_(keep[1])
        if keep[2] is not None:          # the warm-up half-steps do not count
            self._n_capped.copy_(keep[2])
        if keep_split is not None:
            self.split["X"].hl.copy_(keep_split[0])
            self.split["Y"].hl.copy_(keep_split[1])
            self._fp32_stale = keep_split[2]
        return ok

    def sweep(self):
        self.item_half_step()
        self.user_half_step()

    def fit(self, max_iter: int):
        for _ in range(int(max_iter)):
            self.sweep()
        self.sync_factors()
        return self.X, self.Y

    # -- evaluation helpers -------------------------------------------------------------------
    def rmse(self, users, items, ratings) -> float:
        L = nat.lib()
        self.sync_factors()
        users = torch.as_tensor(users).to(self.device, torch.int32).contiguous()
        items = torch.as_tensor(items).to(self.device, torch.int32).contiguous()
        ratings = torch.as_tensor(ratings).to(self.device, torch.float32).contiguous()
        sse = torch.zeros(1, dtype=torch.float64, device=self.device)
        cnt = torch.zeros(1, dtype=torch.int64, device=self.device)
        ws = torch.empty(int(L.hals_als_sse_workspace_bytes()), dtype=torch.uint8, device=self.device)
        nat.check(L.hals_als_sse(nat.ptr(self.X), nat.ptr(self.Y), self.k, nat.ptr(users), nat.ptr(items),
                                 nat.ptr(ratings), users.numel(), nat.ptr(sse), nat.ptr(cnt), nat.ptr(ws), ws.numel(),
                                 nat.current_stream()), "hals_als_sse")
        return float(torch.sqrt(sse / cnt.clamp_min(1)).item())

    def algorithmic_bytes_per_sweep(self) -> int:
        """SURVEY.md 8(d): per half-step nnz*(8+4k) + m_dst*(4k+4); item + user half-steps."""
        k = self.k
        return int(2 * self.nnz_total * (8 + 4 * k) + (self.n_users + self.n_items) * (4 * k + 4))
