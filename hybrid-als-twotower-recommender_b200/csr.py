"""Host-side plumbing around the ALS kernels: COO -> CSR, row sharding, work plans.

Stands where the reference hands its pandas frame to Spark (src/als_model.py:51) and
Spark partitions ratings into in-blocks (ALS.scala makeBlocks, behind als_model.py:62).
torch is used for device memory and sorting only; the arithmetic is in csrc/.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import _native as nat


@dataclass
class CsrShard:
    """Rows [row_begin, row_end) of a ratings matrix in CSR form on one device."""
    row_begin: int
    row_end: int
    n_rows_total: int
    rowptr: torch.Tensor        # int64 [rows+1], local offsets (device)
    colidx: torch.Tensor        # int32 [nnz_local]
    vals: torch.Tensor          # fp32  [nnz_local]
    rowptr_host: np.ndarray     # int64 [rows+1]

    @property
    def n_rows(self):
        return self.row_end - self.row_begin

    @property
    def nnz(self):
        return int(self.colidx.numel())


def row_cost(counts: np.ndarray, k: int = 64) -> np.ndarray:
    """Cost of a row in the unit the kernels' work plan uses (csrc/api.cu, hals_als_plan_chunks_host): its 32-rating
    chunks plus the solve of its normal equations (~6 chunk times at rank <= 64, ~32 at rank 128).  A half-step costs per rating AND per row: the
    user side of a MovieLens-shaped matrix is dominated by the solves, so shards balanced on ratings alone leave the
    rank with the most rows ~15 % behind."""
    counts = np.asarray(counts, dtype=np.int64)
    return (counts + 31) // 32 + (32 if k > 64 else 6) * (counts > 0)


def balanced_row_bounds(counts: np.ndarray, world: int, by_cost: bool = True, k: int = 64) -> np.ndarray:
    """Contiguous row ranges of ~equal cost (see row_cost; by_cost=False: equal rating counts), one per rank.
    Returns int64 [world+1]."""
    n = len(counts)
    csum = np.concatenate([[0], np.cumsum(row_cost(counts, k) if by_cost else counts, dtype=np.int64)])
    total = csum[-1]
    bounds = np.zeros(world + 1, dtype=np.int64)
    for r in range(1, world):
        bounds[r] = np.searchsorted(csum, total * r / world, side="left")
    bounds[world] = n
    return np.maximum.accumulate(np.minimum(bounds, n))


def build_csr(rows: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, n_rows: int,
              row_begin: int = 0, row_end: int | None = None, counts: torch.Tensor | None = None) -> CsrShard:
    """Stable COO -> CSR for rows in [row_begin, row_end): the ratings of a row keep their
    input order, duplicates are kept (Spark does not merge them).  `counts` (int64 [n_rows], device) may pass
    the per-row rating counts of the WHOLE matrix when the caller already has them.  `vals` may be None (a pattern
    without values; the shard's `vals` is then None)."""
    if row_end is None:
        row_end = n_rows
    dev = rows.device
    whole = row_begin == 0 and row_end == n_rows
    if not whole:
        keep = (rows >= row_begin) & (rows < row_end)
        rows, cols = rows[keep], cols[keep]
        vals = vals[keep] if vals is not None else None
    # 32-bit sort keys: the radix sort moves half the bytes of an int64 sort
    local = (rows - row_begin).to(torch.int32) if not whole else rows.to(torch.int32)
    order = torch.sort(local, stable=True).indices
    if counts is not None:
        cnt = counts[row_begin:row_end]
    else:
        cnt = torch.bincount(local.to(torch.int64), minlength=row_end - row_begin)
    rowptr = torch.zeros(row_end - row_begin + 1, dtype=torch.int64, device=dev)
    torch.cumsum(cnt, 0, out=rowptr[1:])
    return CsrShard(row_begin, row_end, n_rows, rowptr, cols[order].to(torch.int32).contiguous(),
                    vals[order].to(torch.float32).contiguous() if vals is not None else None, rowptr.cpu().numpy())


class AlsPlanHandle:
    """Owns the device arrays of a hals_als_plan and the matching workspace."""

    def __init__(self, shard: CsrShard, k: int, seg_len: int | None = None, device=None, n_src: int = 0,
                 implicit: bool = False, alpha: float = 1.0):
        L = nat.lib()
        self.k = k
        rp = np.ascontiguousarray(shard.rowptr_host, dtype=np.int64)
        if seg_len:
            self.seg_len = int(seg_len)
        else:
            # Long rows are cut into slices of at most seg_len ratings; slices are what the persistent CTAs
            # round-robin over.  A small shard (one of 8 ranks on the MovieLens-20M shape) with the default 4096
            # would hand each CTA one or two slices and lose up to a slice time to quantisation, so the slice
            # shrinks until a CTA sees ~8 of them (bounded below: every slice costs a workspace slot).
            default = int(L.hals_als_default_seg_len(k))
            ctas = 4 * 148
            dev0 = torch.device(device) if device is not None else shard.colidx.device
            if dev0.type == "cuda":
                ctas = 4 * torch.cuda.get_device_properties(dev0).multi_processor_count
            lens = np.diff(rp)
            nnz = int(rp[-1])
            want = nnz // (8 * ctas) // 32 * 32
            # only shards whose ratings sit mostly in long rows (a Zipf head of items) are made of slices; where
            # long rows are the exception (users) finer slices just add slot traffic (measured: slower)
            heavy = nnz > 0 and float(lens[lens > default].sum()) > 0.25 * nnz
            seg = max(512, min(default, want)) if (want > 0 and heavy) else default
            # ... but every sliced row goes through the slot reduction (one small CTA per row): shrinking must not
            # turn thousands of mid-sized rows (active users) into long rows
            while seg < default and int((lens > seg).sum()) > 2 * ctas:
                seg = min(default, seg * 2)
            self.seg_len = seg
        m = len(rp) - 1
        n_items, n_long, n_slots = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        nat.check(L.hals_als_plan_count_host(nat.ptr(rp), m, self.seg_len, ctypes.byref(n_items),
                                             ctypes.byref(n_long), ctypes.byref(n_slots)), "plan_count")
        self.n_items, self.n_long, self.n_slots = n_items.value, n_long.value, n_slots.value
        h = {
            "item_row": np.empty(max(self.n_items, 1), np.int32),
            "item_begin": np.empty(max(self.n_items, 1), np.int64),
            "item_len": np.empty(max(self.n_items, 1), np.int32),
            "item_slot": np.empty(max(self.n_items, 1), np.int32),
            "long_row": np.empty(max(self.n_long, 1), np.int32),
            "long_slot0": np.empty(max(self.n_long, 1), np.int32),
            "long_nseg": np.empty(max(self.n_long, 1), np.int32),
        }
        nat.check(L.hals_als_plan_fill_host(nat.ptr(rp), m, self.seg_len, *(nat.ptr(h[n]) for n in (
            "item_row", "item_begin", "item_len", "item_slot", "long_row", "long_slot0", "long_nseg"))), "plan_fill")
        # long rows by slice count, descending: the slot pre-sum launches only cover the rows that need them
        n_gt16 = n_gt256 = 0
        if self.n_long:
            order = np.argsort(-h["long_nseg"][: self.n_long], kind="stable")
            for name in ("long_row", "long_slot0", "long_nseg"):
                h[name][: self.n_long] = h[name][: self.n_long][order]
            n_gt16 = int((h["long_nseg"][: self.n_long] > 16).sum())
            n_gt256 = int((h["long_nseg"][: self.n_long] > 256).sum())
        # chunk table (pieces of 32 ratings) + cost prefix: what the persistent rank-64 / rank-128 kernels stream.
        # On a CUDA device the table is derived there from the item arrays (a few torch ops on ~1 M entries); the host
        # planner entry point hals_als_plan_chunks_host computes the same thing for C callers and CPU tests
        # (tests/test_gpu_als.py checks the two against each other).  Building it on the host and uploading ~20 MB of
        # pageable memory was a third of the engine's set-up time on the MovieLens-20M shape.
        self.n_chunks = 0
        dev = device if device is not None else shard.colidx.device
        on_cuda = torch.device(dev).type == "cuda"
        want_chunks = k in (64, 128) and self.n_items > 0
        if want_chunks:
            self.n_chunks = int(((h["item_len"][: self.n_items].astype(np.int64) + 31) // 32).sum())
        if want_chunks and not on_cuda:
            h["item_chunk0"] = np.empty(self.n_items + 1, np.int64)
            h["item_cost0"] = np.empty(self.n_items + 1, np.int64)
            h["chunk_pos"] = np.empty(max(self.n_chunks, 1), np.int64)
            h["chunk_cnt"] = np.empty(max(self.n_chunks, 1), np.int32)
            nat.check(L.hals_als_plan_chunks_host(nat.ptr(h["item_len"]), nat.ptr(h["item_begin"]), nat.ptr(h["item_slot"]),
                                                  self.n_items, int(k), nat.ptr(h["item_chunk0"]), nat.ptr(h["item_cost0"]),
                                                  nat.ptr(h["chunk_pos"]), nat.ptr(h["chunk_cnt"])), "plan_chunks")
        self.host = h
        self.dev = {n: torch.from_numpy(a).to(dev) for n, a in h.items()}
        if want_chunks and on_cuda:
            n = self.n_items
            il, ib, isl = self.dev["item_len"][:n].long(), self.dev["item_begin"][:n], self.dev["item_slot"][:n]
            nch = (il + 31) // 32
            solve, park = (32, 6) if k > 64 else (6, 2)                 # == kSolveCost / kParkCost of csrc/api.cu
            c0 = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            torch.cumsum(nch, 0, out=c0[1:])
            cost0 = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            torch.cumsum(nch + torch.where(isl < 0, solve, park), 0, out=cost0[1:])
            item_of = torch.repeat_interleave(torch.arange(n, device=dev), nch, output_size=self.n_chunks)
            k_in = torch.arange(self.n_chunks, device=dev) - c0[item_of]
            self.dev["item_chunk0"], self.dev["item_cost0"] = c0, cost0
            self.dev["chunk_pos"] = ib[item_of] + 32 * k_in
            self.dev["chunk_cnt"] = (il[item_of] - 32 * k_in).to(torch.int32)
        # ratings as bf16 hi|lo pairs, packed once: the tensor-core kernels copy them into its operand
        # (implicit feedback, ranks 64 / 128: the Hu-Koren operands -- see hals_als_plan.vals_scale in include/hals_b200.h)
        self.vals_hl = self.vals_scale = self.item_npos = None
        self.packed_alpha = 0.0
        on_gpu = torch.device(dev).type == "cuda" and shard.vals.numel() > 0
        if implicit and k in (64, 128) and on_gpu and alpha > 0 and self.n_items > 0:
            nnz = shard.vals.numel()
            self.vals_hl = torch.empty(nnz, dtype=torch.int32, device=dev)
            self.vals_scale = torch.empty(nnz, dtype=torch.float32, device=dev)
            self.item_npos = torch.empty(self.n_items, dtype=torch.int32, device=dev)
            nat.check(L.hals_als_pack_ratings_implicit(nat.ptr(shard.vals), nnz, float(alpha), nat.ptr(self.vals_hl),
                                                       nat.ptr(self.vals_scale), nat.current_stream()), "pack_ratings_implicit")
            nat.check(L.hals_als_plan_count_positive(nat.ptr(shard.vals), nat.ptr(self.dev["item_begin"]),
                                                     nat.ptr(self.dev["item_len"]), self.n_items, nat.ptr(self.item_npos),
                                                     nat.current_stream()), "plan_count_positive")
            self.packed_alpha = float(np.float32(alpha))
        elif not implicit and k in (64, 128) and on_gpu:
            self.vals_hl = torch.empty(shard.vals.numel(), dtype=torch.int32, device=dev)
            nat.check(L.hals_als_pack_ratings(nat.ptr(shard.vals), shard.vals.numel(), nat.ptr(self.vals_hl),
                                              nat.current_stream()), "hals_als_pack_ratings")
        self.struct = nat.AlsPlan(
            n_items=self.n_items, n_long_rows=self.n_long, n_slots=self.n_slots, seg_len=self.seg_len,
            max_nseg=int(h["long_nseg"][: self.n_long].max()) if self.n_long else 0,
            vals_hl=self.vals_hl.data_ptr() if self.vals_hl is not None else None, n_chunks=self.n_chunks,
            vals_scale=self.vals_scale.data_ptr() if self.vals_scale is not None else None,
            item_npos=self.item_npos.data_ptr() if self.item_npos is not None else None, packed_alpha=self.packed_alpha,
            n_long_gt16=n_gt16 if self.n_long else 0, n_long_gt256=n_gt256 if self.n_long else 0,
            **{n: t.data_ptr() for n, t in self.dev.items()})
        self.workspace_bytes = int(L.hals_als_workspace_bytes(self.n_slots, k, int(n_src)))
        self.workspace = torch.empty(max(self.workspace_bytes, 16), dtype=torch.uint8, device=dev)
