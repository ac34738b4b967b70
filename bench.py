#!/usr/bin/env python
"""bench.py -- ALS ratings/s per sweep (headline) on synthetic data of the BASELINE.json shapes.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c1] [--impl ours|reference] [--dump-outputs DIR]

One step = one ALS sweep (item half-step, all-gather, user half-step, all-gather) over the
whole ratings matrix, factors and CSR shards resident in HBM.  `value` = nnz / (time per sweep),
whole job, max over ranks.  `e2e` = the same metric through the public `train()`-shaped path
with HOST inputs: pinned COO triples -> H2D -> CSR build + plan -> `e2e_sweeps` sweeps -> factors
D2H, all inside the timed region.  `roofline` is the half-step kernel sequence against the
measured HBM peak with SURVEY.md 8(d) algorithmic bytes; `cpu_baseline` is the CPU oracle port
(Spark local[N] cannot run in this image) on a bounded row sample.  Prints ONE JSON line.
`--dump-outputs DIR` writes the factor matrices of the last timed sweep as DIR/<name>.npy, so that two builds
can be compared output for output (same arguments -> same inputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (users, items, nnz, rank, reg, rating grid)
    "c1": dict(users=10_000, items=10_000, nnz=10_000, rank=10, reg=0.1, half=False,
               desc="synthetic Amazon-sample shape 10k x 10k, ~10k ratings, rank 10"),
    "c2": dict(users=138_493, items=26_744, nnz=20_000_263, rank=64, reg=0.1, half=True,
               desc="MovieLens-20M shape 138,493 x 26,744, 20,000,263 ratings, explicit ALS rank 64"),
    "c3": dict(users=480_189, items=17_770, nnz=100_480_507, rank=128, reg=0.1, half=False,
               desc="Netflix-prize shape 480,189 x 17,770, 100,480,507 ratings, explicit ALS rank 128"),
    # config 4 is quoted on 8 GPUs (10M users x 1M items, 1e9 interactions): one GPU's share of it -- 1/8 of the users
    # and interactions against the full item catalogue; N GPUs run N shares (weak scaling up to the full shape at 8)
    "c4s": dict(users=1_250_000, items=1_000_000, nnz=125_000_000, rank=128, reg=0.1, half=False, implicit=True, alpha=40.0,
                desc="1/8 slice per GPU of the implicit-feedback shape 10M x 1M, 1e9 interactions, Hu-Koren ALS rank 128"),
}
METRIC = "als_ratings_per_sec_per_sweep"
UNIT = "ratings/s"


_M64 = (1 << 64) - 1


def _s64(x):
    """Python int -> the signed 64-bit value torch.int64 arithmetic wraps to."""
    x &= _M64
    return x - (1 << 64) if x >= (1 << 63) else x


def _splitmix64(x):
    """SplitMix64 finaliser on torch.int64 (two's-complement wrap-around; logical shifts emulated with masks)."""
    z = x + _s64(0x9E3779B97F4A7C15)
    z = (z ^ ((z >> 30) & ((1 << 34) - 1))) * _s64(0xBF58476D1CE4E5B9)
    z = (z ^ ((z >> 27) & ((1 << 37) - 1))) * _s64(0x94D049BB133111EB)
    return z ^ ((z >> 31) & ((1 << 33) - 1))


def _uniform01(n, stream, seed, device):
    """n doubles in [0,1): a counter-based hash of (seed, stream, index) -- integer arithmetic only, so every rank,
    every run and the CPU reference arm draw bit-identical numbers (torch.multinomial on CUDA did not: round 1's
    train RMSE moved by 4e-5 between two identical runs)."""
    import torch
    idx = torch.arange(n, dtype=torch.int64, device=device)
    z = _splitmix64(idx + _s64(seed * 0x632BE59BD9B4E019 + stream * 0xD1342543DE82EF95))
    return ((z >> 11) & ((1 << 53) - 1)).to(torch.float64) * (1.0 / (1 << 53))


def synth_coo(w, device, seed=1234):
    """Zipf item popularity (exponent 1, popularity not sorted by id), log-normal user activity, duplicates kept (Spark
    does not merge them).  The two CDFs (138k / 27k entries) are built in numpy on the host; the draws are inverse-CDF
    lookups of hashed uniforms: deterministic across ranks, runs and devices."""
    import torch
    U, I, nnz = w["users"], w["items"], w["nnz"]
    rng = np.random.default_rng(seed)
    item_p = 1.0 / np.arange(1, I + 1, dtype=np.float64)
    item_w = np.empty(I)
    item_w[rng.permutation(I)] = item_p
    user_w = np.exp(rng.standard_normal(U))

    def draw(weights, stream):
        cdf = np.cumsum(weights)
        cdf /= cdf[-1]
        cdf_d = torch.from_numpy(cdf).to(device)
        out = torch.empty(nnz, dtype=torch.int32, device=device)
        for lo in range(0, nnz, 1 << 24):                    # bounded temporaries
            n = min(nnz - lo, 1 << 24)
            x = _uniform01(n, stream, seed + lo, device)
            out[lo:lo + n] = torch.searchsorted(cdf_d, x, right=True).clamp_(max=len(weights) - 1).to(torch.int32)
        return out

    u = draw(user_w, 1)
    i = draw(item_w, 2)
    r = torch.empty(nnz, dtype=torch.float32, device=device)
    for lo in range(0, nnz, 1 << 24):
        n = min(nnz - lo, 1 << 24)
        x = _uniform01(n, 3, seed + lo, device)
        r[lo:lo + n] = ((x * 10).floor() + 1).float() * 0.5 if w["half"] else ((x * 5).floor() + 1).float()
    return u, i, r


def coo_checksum(u, i, r):
    """Order-sensitive 63-bit checksum of the rating triples (wrap-around int64 arithmetic)."""
    import torch
    n = u.numel()
    k = torch.arange(n, dtype=torch.int64, device=u.device)
    h = (u.to(torch.int64) * 1000003 + i.to(torch.int64)) * 31 + (r * 2).to(torch.int64)
    return int((_splitmix64(h ^ (k * 0x9E3779B1)).sum().item()) & ((1 << 62) - 1))


def assert_same_on_all_ranks(values, what, dev, world):
    """Every rank must hold the same integers (inputs, shard bounds): max == min over ranks, or the run aborts."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return
    t = torch.tensor([int(v) for v in values], dtype=torch.int64, device=dev)
    hi, lo = t.clone(), t.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    if not torch.equal(hi, lo):
        raise RuntimeError(f"ranks disagree on {what}: max {hi.tolist()} min {lo.tolist()}")


DUMP_BUDGET = 60 << 20      # bytes of .npy payload: under 64 MB (10^6 bytes each) with the headers


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy.  When they hold more than DUMP_BUDGET bytes in all, every array keeps
    the same fixed, seeded sample of its rows (in row order), so dumps of two runs stay comparable row for row."""
    os.makedirs(out_dir, exist_ok=True)
    keep = min(1.0, DUMP_BUDGET / sum(a.nbytes for a in arrays.values()))
    for name, a in arrays.items():
        if keep < 1.0:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * keep), replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def algorithmic_bytes(w):
    k, nnz = w["rank"], w["nnz"]
    item_half = nnz * (8 + 4 * k) + w["items"] * (4 * k + 4)
    user_half = nnz * (8 + 4 * k) + w["users"] * (4 * k + 4)
    return item_half, user_half


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
# CPU baseline: the oracle port on a bounded row sample
# ------------------------------------------------------------------------------------------
class CpuBaseline:
    """The CPU oracle port timed on a bounded row sample of the workload (CSR built once, outside the timing)."""

    def __init__(self, w, u, i, r, target_nnz, seed=3):
        from oracle import als_oracle
        self.w = w
        U, I, k = w["users"], w["items"], w["rank"]
        t0 = time.time()
        self.X = als_oracle.init_factors(U, k, seed)
        self.Yfull = als_oracle.init_factors(I, k, seed + 1)
        self.item_csr = als_oracle.coo_to_csr(i, u, r, I)
        self.user_csr = als_oracle.coo_to_csr(u, i, r, U)

        def sample_rows(rowptr, n):
            if target_nnz >= rowptr[-1]:
                return 0, n, int(rowptr[-1])
            mid = n // 3
            end = int(np.searchsorted(rowptr, rowptr[mid] + min(target_nnz, rowptr[-1] - rowptr[mid])))
            end = max(min(end, n), mid + 1)
            return mid, end, int(rowptr[end] - rowptr[mid])

        self.isel = sample_rows(self.item_csr[0], I)
        self.usel = sample_rows(self.user_csr[0], U)
        self.prep_s = time.time() - t0

    def run(self, reps=3):
        from oracle import c_oracle
        w = self.w
        (ib, ie, inz), (ub, ue, unz) = self.isel, self.usel
        Y = np.zeros((w["items"], w["rank"]), np.float32)
        ti = tu = 0.0
        for _ in range(reps):      # ~10 s of CPU work on the box's host cores for c2
            t0 = time.time()
            c_oracle.als_half_step(*self.item_csr, self.X, w["reg"], row_begin=ib, row_end=ie, out=Y)
            ti += (time.time() - t0) / reps
            t0 = time.time()
            c_oracle.als_half_step(*self.user_csr, self.Yfull, w["reg"], row_begin=ub, row_end=ue)
            tu += (time.time() - t0) / reps
        per_rating = ti / max(inz, 1) + tu / max(unz, 1)          # seconds per rating per sweep
        return {"value": 1.0 / per_rating, "unit": UNIT, "cores": c_oracle.num_threads(), "kind": "port",
                "sample": f"item rows [{ib},{ie}) = {inz} ratings in {ti:.2f}s + user rows [{ub},{ue}) = {unz} ratings "
                          f"in {tu:.2f}s of the {w['nnz']}-rating workload (C oracle, fp64 packed dspr + dppsv, OpenMP); "
                          f"Spark local[N] unavailable offline", "prep_s": round(self.prep_s, 2)}


def cpu_baseline_run(w, u, i, r, target_nnz=25_000_000, seed=3):
    return CpuBaseline(w, u, i, r, target_nnz, seed).run()


def run_reference(args, w):
    """--impl reference: the reference's CPU path restated (oracle port; pyspark/JVM absent)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import c_oracle
    # torch.distributed.run exports OMP_NUM_THREADS=1 to its children: round 1's N>1 reference arm ran on one core
    c_oracle.set_num_threads(os.cpu_count() or 1)
    torch.set_num_threads(os.cpu_count() or 1)
    u, i, r = synth_coo(w, "cpu")
    u, i, r = u.numpy(), i.numpy(), r.numpy()
    vals = []
    res = None
    cb = CpuBaseline(w, u, i, r, args.cpu_sample)
    for s in range(args.warmup + args.steps):
        res = cb.run(reps=1)
        if s >= args.warmup:
            vals.append(res["value"])
    v = float(np.mean(vals))
    res["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * w["nnz"] / v, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {w['desc']}", "note": "CPU oracle port of Spark ALS on host cores; "
                       "ms_per_step extrapolated from the bounded sample to a full sweep"},
            "cpu_baseline": res, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def scoring_cpu_baseline(Ua, Ia, Ut, It, k, n_users=128):
    """Restated CPU baseline of the scoring path on the host cores (SURVEY 8d-ii): torch-CPU fp32 matmul of both
    models over a slice of users, per-user min-max, 0.8/0.2 blend, top-k.  The reference itself loops over users in
    Python around Keras predict + sklearn + sorted(); TensorFlow is not in the image, so this is the generous form."""
    import torch
    n = min(n_users, Ua.shape[0])
    ua, ut, ia, it = Ua[:n].cpu(), Ut[:n].cpu(), Ia.cpu(), It.cpu()
    torch.set_num_threads(os.cpu_count() or 1)

    def once():
        sa, st = ua @ ia.T, ut @ it.T
        na = (sa - sa.amin(1, keepdim=True)) / (sa.amax(1, keepdim=True) - sa.amin(1, keepdim=True)).clamp_min(1e-30)
        nt = (st - st.amin(1, keepdim=True)) / (st.amax(1, keepdim=True) - st.amin(1, keepdim=True)).clamp_min(1e-30)
        return torch.topk(0.8 * na + 0.2 * nt, k, dim=1)

    once()
    t0 = time.perf_counter()
    once()
    dt = time.perf_counter() - t0
    return {"value": n * float(Ia.shape[0]) / dt, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} users x {Ia.shape[0]} items in {dt:.2f}s: torch-CPU fp32 matmul (128-d + 50-d), per-user "
                      "min-max, 0.8/0.2 blend, topk; TF/Keras unavailable offline"}


def scoring_leg(args, dev, rank, world, barrier):
    """Second headline metric: hybrid scored user-item pairs/s at the BASELINE config-5 scale: 1,000,000 users against
    1.25M items per GPU (10M at 8 GPUs, item-sharded), 128-d ALS + 50-d tower, top-100, users in slabs of 65,536.
    `value`: operands resident in HBM, CUDA events over the whole pass, max over ranks.  `e2e`: pinned host user ids ->
    H2D -> gather of the users' rows -> two fused passes (+ extrema all-reduce, all-to-all + merge when sharded) ->
    D2H of this rank's [U/N, 100] indices and scores, wall clock between barriers.  A 64-user fp64 spot check of the
    local top-k runs on every rank."""
    import torch
    import torch.distributed as dist
    from hybrid_als_twotower_recommender_b200.scoring import HybridScorer, exchange_topk, merge_lists
    U, I, k, ka, kt, slab = args.score_users, args.score_items_per_gpu, args.score_topk, 128, 50, args.score_slab
    g = torch.Generator(device=dev).manual_seed(99)
    Ua = torch.randn(U, ka, device=dev, generator=g) * ka ** -0.5
    Ut = torch.nn.functional.layer_norm(torch.randn(U, kt, device=dev, generator=g), (kt,))
    gi = torch.Generator(device=dev).manual_seed(100 + rank)
    Ia = torch.randn(I, ka, device=dev, generator=gi)
    It = torch.nn.functional.layer_norm(torch.randn(I, kt, device=dev, generator=gi), (kt,))
    sc = HybridScorer(Ua, Ia, Ut, It, item_offset=rank * I, dist_rank=rank, world=world)
    slabs = [(a, min(U, a + slab)) for a in range(0, U, slab)]

    def one_pass(timed):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        t1 = t2 = 0.0
        for (a, b) in slabs:
            ev[0].record(); ex = sc.extrema(a, b); ev[1].record()
            idx, s = sc.topk_local(ex, k, 0.8, 0.2, a, b)
            fi, fs = exchange_topk(idx, s, rank, world, merge_lists)
            ev[2].record()
            if timed:
                torch.cuda.synchronize()
                t1 += ev[0].elapsed_time(ev[1]); t2 += ev[1].elapsed_time(ev[2])
        return t1, t2

    sc.extrema(*slabs[0]); sc.recommend(k, 0.8, 0.2, *slabs[0])      # warm-up (workspace, tensor maps)
    barrier()
    t1, t2 = one_pass(True)
    barrier()
    t = torch.tensor([t1, t2], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t1, t2 = (float(x) for x in t.tolist())
    flagged = 0
    # ---- spot check: 64 users of the first slab, local top-k against a dense fp64 blend over this rank's items
    a, b = slabs[0]
    ex = sc.extrema(a, b)
    idx, s = sc.topk_local(ex, k, 0.8, 0.2, a, b)
    flagged = sc.flagged_users(b - a, k)
    pick = torch.arange(0, b - a, max(1, (b - a) // 64), device=dev)[:64]
    exd = ex[pick].double()
    Sa = Ua[a:b][pick].double() @ Ia.double().T
    St = Ut[a:b][pick].double() @ It.double().T

    def mm(S, lo, hi):
        rg = hi - lo
        return (S - lo[:, None]) * torch.where(rg != 0, 1.0 / torch.where(rg != 0, rg, torch.ones_like(rg)), torch.ones_like(rg))[:, None]
    B = 0.8 * mm(Sa, exd[:, 0], exd[:, 1]) + 0.2 * mm(St, exd[:, 2], exd[:, 3])
    wv, wi = torch.topk(B, k, dim=1)
    got_i, got_s = idx[pick].long() - rank * I, s[pick].double()
    score_err = float((got_s - wv).abs().max())
    same = float((got_i == wi).double().mean())
    kth_gap_ok = bool((torch.gather(B, 1, got_i.clamp(0, I - 1)) >= wv[:, -1:] - 1e-5).all())
    spot = {"users": int(pick.numel()), "max_abs_score_err": score_err, "index_match": same, "all_within_tie_band": kth_gap_ok,
            "ok": bool(score_err <= 1e-5 and same >= 0.99 and kth_gap_ok)}
    del Sa, St, B
    # ---- end to end: host ids -> top-k lists on the host
    ids_h = torch.randperm(U, generator=torch.Generator().manual_seed(5)).to(torch.int32).pin_memory()
    per = [((b - a) + world - 1) // world for (a, b) in slabs]
    out_i = torch.empty((sum(per), k), dtype=torch.int32).pin_memory()
    out_s = torch.empty((sum(per), k), dtype=torch.float32).pin_memory()
    sl = HybridScorer(torch.empty((slab, ka), device=dev), Ia, torch.empty((slab, kt), device=dev), It,
                      item_offset=rank * I, dist_rank=rank, world=world)
    barrier()
    t0 = time.perf_counter()
    o = 0
    for j, (a, b) in enumerate(slabs):
        ids = ids_h[a:b].to(dev, non_blocking=True).long()
        torch.index_select(Ua, 0, ids, out=sl.Ua[: b - a]); torch.index_select(Ut, 0, ids, out=sl.Ut[: b - a])
        fi, fs = sl.recommend(k, 0.8, 0.2, 0, b - a)
        out_i[o:o + fi.shape[0]].copy_(fi, non_blocking=True); out_s[o:o + fi.shape[0]].copy_(fs, non_blocking=True)
        o += fi.shape[0]
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te)
    pairs = float(U) * float(I) * world
    flops = pairs * 2 * (ka + kt)
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:
        peak = 1590.0
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = scoring_cpu_baseline(Ua, Ia, Ut, It, k)
    return {"metric": "hybrid_scored_pairs_per_sec", "value": pairs / ((t1 + t2) * 1e-3), "unit": "pairs/s",
            "e2e": {"value": pairs / e2e_s, "unit": "pairs/s", "h2d_bytes": int(U * 4), "d2h_bytes": int(sum(per) * k * 8),
                    "seconds": e2e_s, "what": "pinned host user ids -> H2D -> row gather -> extrema pass -> blend + top-k pass "
                    "(+ all-reduce / all-to-all + merge) -> D2H of this rank's top-100 lists"},
            "cpu_baseline": cpu, "spot_check_fp64": spot,
            "config": {"users": U, "user_slab": slab, "items_per_gpu": I, "items_total": I * world, "k_als": ka, "k_tower": kt,
                       "topk": k, "weights": [0.8, 0.2], "sharding": "item-sharded, users replicated"},
            "ms_extrema_pass": t1, "ms_blend_topk_pass": t2,
            "tensor": {"bound": "tensor", "unit": "TFLOP/s", "peak": peak,
                       "achieved_pass2": flops / world / (t2 * 1e-3) / 1e12, "frac_pass2": flops / world / (t2 * 1e-3) / 1e12 / peak,
                       "achieved_both_passes": 2 * flops / world / ((t1 + t2) * 1e-3) / 1e12,
                       "note": "algorithmic flops 2*(128+50) per scored pair per pass, per GPU; pass times include operand "
                               "prep, exact re-scoring and (N>1) the extrema all-reduce / top-k all-to-all + merge"},
            "users_rerun_exactly_first_slab": flagged}


def c3_leg(args, dev, rank, world, barrier, name="c3"):
    """BASELINE config 3 (Netflix-prize shape, rank 128) or the config-4 slice (name="c4s": implicit feedback, users and
    interactions grow with N) at every N the driver runs: sweep time only (device events, max over ranks), same
    synthetic generator, same sharding as the headline workload."""
    import torch
    import torch.distributed as dist
    from hybrid_als_twotower_recommender_b200.als_engine import AlsEngine
    w = dict(WORKLOADS[name])
    if name == "c4s":
        w["users"], w["nnz"] = w["users"] * world, w["nnz"] * world
    u, i, r = synth_coo(w, dev)
    data_sum = coo_checksum(u, i, r)
    eng = AlsEngine(u, i, r, w["users"], w["items"], w["rank"], w["reg"], implicit=bool(w.get("implicit")),
                    alpha=float(w.get("alpha", 1.0)), device=dev, dist_rank=rank, world=world)
    assert_same_on_all_ranks([data_sum] + list(eng.user_bounds) + list(eng.item_bounds), f"{name} inputs / shard bounds", dev, world)
    del u, i, r
    eng.init_user_factors(1)
    eng.enable_graphs()
    for _ in range(3):
        eng.sweep()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.c3_steps):
        eng.sweep()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1) / args.c3_steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    b_item, b_user = algorithmic_bytes(w)
    peak, _ = measured_peaks()
    out = {"metric": METRIC, "value": w["nnz"] / (ms * 1e-3), "unit": UNIT, "ms_per_sweep": ms, "steps": args.c3_steps,
           "workload": f"{name}: {w['desc']}", "n_gpus": world, "inputs_checksum": data_sum,
           "users": w["users"], "items": w["items"], "nnz": w["nnz"], "scaling": "weak" if name == "c4s" else "strong",
           "roofline_frac": (b_item + b_user) / world / (ms * 1e-3) / 1e9 / peak,
           "algorithmic_bytes_per_sweep": b_item + b_user}
    del eng
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-sweeps", type=int, default=10, help="sweeps per end-to-end train()-shaped call")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-sample", type=int, default=25_000_000, help="ratings per half-step in the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel / collective individually in the timed sweeps")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (profiling runs only)")
    ap.add_argument("--no-scoring", action="store_true", help="skip the hybrid top-k scoring leg (extra.hybrid_topk)")
    ap.add_argument("--no-c3", action="store_true", help="skip the config-3 sweep timing (extra.als_c3)")
    ap.add_argument("--c3-steps", type=int, default=3)
    ap.add_argument("--no-c4", action="store_true", help="skip the config-4 slice (implicit feedback) sweep timing (extra.als_c4_slice)")
    ap.add_argument("--score-users", type=int, default=1_000_000)
    ap.add_argument("--score-slab", type=int, default=65536)
    ap.add_argument("--score-items-per-gpu", type=int, default=1_250_000)
    ap.add_argument("--score-topk", type=int, default=100)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the user / item factors of the last timed sweep as "
                    "DIR/als_user_factors.npy and DIR/als_item_factors.npy (fp32; a seeded sample of rows above 60 MiB)")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        return run_reference(args, w)

    import torch
    import torch.distributed as dist
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import _native as nat
    from hybrid_als_twotower_recommender_b200.als_engine import AlsEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    nat.lib()
    nat.require_cuda()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"

    u, i, r = synth_coo(w, dev)
    data_sum = coo_checksum(u, i, r)
    eng = AlsEngine(u, i, r, w["users"], w["items"], w["rank"], w["reg"], implicit=bool(w.get("implicit")),
                    alpha=float(w.get("alpha", 1.0)), device=dev, dist_rank=rank, world=world)
    # every rank generated the SAME matrix and derived the SAME shard bounds (the all-gathers rely on it)
    assert_same_on_all_ranks([data_sum] + list(eng.user_bounds) + list(eng.item_bounds), "inputs / shard bounds", dev, world)
    eng.init_user_factors(1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    graphs_on = (not args.no_graphs) and eng.enable_graphs()
    for _ in range(max(args.warmup, 3)):
        eng.sweep()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    l0 = nat.launch_count()
    g0 = eng.graph_launches
    barrier()
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for s in range(args.steps):
        ev[s][0].record(); eng.item_half_step(); ev[s][1].record()
        ev[s][2].record(); eng.user_half_step(); ev[s][3].record()
    t_end.record()
    barrier()
    launches = nat.launch_count() - l0 + (eng.graph_launches - g0)
    clocks = sampler.stop() if rank == 0 else None
    total_ms = t_start.elapsed_time(t_end)
    t_item = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
    t_user = float(np.mean([e[2].elapsed_time(e[3]) for e in ev]))
    tm = torch.tensor([total_ms, t_item, t_user], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    total_ms, t_item, t_user = (float(x) for x in tm.tolist())
    ms_per_step = total_ms / args.steps
    value = w["nnz"] / (ms_per_step * 1e-3)
    if args.dump_outputs:
        eng.sync_factors()          # what fit() returns: the full fp32 factors on every rank (a collective when sharded)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"als_user_factors": eng.X.cpu().numpy(), "als_item_factors": eng.Y.cpu().numpy()})
    rmse_train = eng.rmse(u[:1_000_000], i[:1_000_000], r[:1_000_000])

    # ---- end-to-end: host COO in pinned memory -> H2D -> CSR + plan -> sweeps -> factors D2H ----------
    hu, hi, hr = (t.cpu().pin_memory() for t in (u, i, r))
    X0 = eng.X.clone()
    del eng
    torch.cuda.empty_cache()
    e2e_ms = []
    hX = torch.empty((w["users"], w["rank"]), dtype=torch.float32).pin_memory()
    hY = torch.empty((w["items"], w["rank"]), dtype=torch.float32).pin_memory()
    for s in range(0 if args.no_e2e else 1 + args.e2e_steps):
        barrier()
        t0 = time.perf_counter()
        # every rank uploads ITS contiguous 1/N of the triples; the engine routes them to the row owners over NVLink
        c0, c1 = (w["nnz"] * rank) // world, (w["nnz"] * (rank + 1)) // world
        du, di, dr = (t[c0:c1].to(dev, non_blocking=True) for t in (hu, hi, hr))
        e = AlsEngine(du, di, dr, w["users"], w["items"], w["rank"], w["reg"], device=dev, dist_rank=rank, world=world,
                      partitioned=True)
        e.set_user_factors(X0)
        e.fit(args.e2e_sweeps)
        hX.copy_(e.X, non_blocking=True); hY.copy_(e.Y, non_blocking=True)
        barrier()
        if s > 0:
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
        del e
    te = torch.tensor([float(np.mean(e2e_ms)) if e2e_ms else 0.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms_call = float(te) if e2e_ms else None                      # None (JSON null) when the leg was skipped
    e2e_value = args.e2e_sweeps * w["nnz"] / (e2e_ms_call * 1e-3) if e2e_ms_call else None

    # ---- the same through the drop-in class: ALSModel.train(DataFrame) with raw 64-bit ids (device-side id
    # compaction + CSR build + sweeps) and the factors read back; single process only (the class drives one GPU)
    e2e_api = None
    if world == 1 and not args.no_e2e:
        import pandas as pd
        from hybrid_als_twotower_recommender_b200 import ALSModel
        df = pd.DataFrame({"userId": hu.numpy().astype(np.int64) * 7 + 3, "itemId": hi.numpy().astype(np.int64) * 5 + 1,
                           "average_review_rating": hr.numpy().astype(np.float64)})
        m = ALSModel(rank=w["rank"], max_iter=args.e2e_sweeps, reg_param=w["reg"])
        m.train(df.iloc[:200_000])                                   # warm-up: lazy initialisation ...
        m.train(df)                                                  # ... and the allocator at the full size
        api_ms = []
        for _ in range(args.e2e_steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ok = m.train(df)
            hXa, hYa = m.model.user_factors.cpu(), m.model.item_factors.cpu()
            api_ms.append((time.perf_counter() - t0) * 1e3)
            assert ok and hXa.shape[0] > 0 and torch.isfinite(hYa).all()
        e2e_api = {"value": args.e2e_sweeps * w["nnz"] / (float(np.mean(api_ms)) * 1e-3), "unit": UNIT,
                   "ms_per_call": float(np.mean(api_ms)), "sweeps_per_call": args.e2e_sweeps,
                   "h2d_bytes_per_step": int(w["nnz"] * 20), "d2h_bytes_per_step": int((w["users"] + w["items"]) * w["rank"] * 4),
                   "what": "ALSModel(rank, max_iter).train(pandas DataFrame with raw int64 ids, float64 ratings) -> factors on the host"}
        del m, df

    c3_extra = None
    if not args.no_c3:
        c3_extra = c3_leg(args, dev, rank, world, barrier)
    c4_extra = None
    if not args.no_c4:
        c4_extra = c3_leg(args, dev, rank, world, barrier, name="c4s")

    scoring_extra = None
    if not args.no_scoring:
        scoring_extra = scoring_leg(args, dev, rank, world, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peaks()
    b_item, b_user = algorithmic_bytes(w)
    # DRAM bytes per sweep (both half-step launches) cannot be measured outside a profiler: they come from the committed
    # `ncu --set full` capture of this workload, stamped with the commit the capture was taken at (stale once the
    # kernel changes: the note below carries the stamp)
    traffic, traffic_src = None, "no capture for this workload"
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            trj = json.load(f)
        tr = trj.get(args.workload)
        if tr and world == 1:
            traffic = sum(tr[h][k] for h in ("item_half", "user_half") for k in ("dram_read_bytes", "dram_write_bytes"))
            traffic_src = f"profiles/r02_traffic.json, captured at commit {trj.get('captured_at_commit', '?')} ({trj.get('kernel', '?')})"
    except (OSError, ValueError, KeyError):
        traffic = None
    # per-rank share of the algorithmic bytes (rows are cost-balanced across ranks)
    ach = (b_item + b_user) / world / ((t_item + t_user) * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {w['desc']}", "step": "one ALS sweep = item half-step + user half-step "
                   "(+ factor all-gathers when sharded)", "launch": "one CUDA graph per half-step" if graphs_on else "plain launches", "rows": "cost-balanced (chunks + solve per row) contiguous row shards per rank",
                   "l2": "per-step inputs (2 CSR orientations + factors) exceed the 126 MB L2; no flush between steps",
                   "train_rmse_after_run": rmse_train},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(w["nnz"] * 12 // world),
                "d2h_bytes_per_step": int((w["users"] + w["items"]) * w["rank"] * 4), "sweeps_per_call": args.e2e_sweeps,
                "ms_per_call": e2e_ms_call, "what": "pinned host COO (1/N of the triples per rank) -> H2D -> [all-to-all to the row owners] -> CSR build + plan -> "
                        "sweeps -> factors D2H on every rank"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                     "traffic_note": f"DRAM bytes per sweep (item + user launch), ncu --set full: {traffic_src}; far below the "
                                     "algorithmic bytes because the gathered factor rows are served by the 126 MB L2",
                     "kernel": "als half-step (build normal equations + Cholesky solve), item + user launches",
                     "algorithmic_bytes_per_sweep": b_item + b_user, "ms_item_half": t_item, "ms_user_half": t_user,
                     "peak_source": peak_src},
    }
    extra = {}
    if e2e_api is not None:
        line["e2e_api"] = e2e_api
    if scoring_extra is not None:
        extra["hybrid_topk"] = scoring_extra
    if c3_extra is not None:
        extra["als_c3"] = c3_extra
    if c4_extra is not None:
        extra["als_c4_slice"] = c4_extra
    if extra:
        line["extra"] = extra
    line["config"]["inputs_checksum"] = data_sum
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_run(w, hu.numpy(), hi.numpy(), hr.numpy(), target_nnz=args.cpu_sample)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
