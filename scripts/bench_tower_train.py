"""TwoTowerModel.train on the GPU trainer (hals_tower_train_step + hals_tower_adam_step) against the torch loop it
replaced (oracle/tower_train_oracle.py:train_reference on CUDA, fp32), embedding_size 50, batch 256 and 1024.

Workloads (features generated from a seed; ratings 1..5 also feed the numeric input, as in the reference):
  c1  the synthetic Amazon-sample shape: 10,000 users x 10,000 items, 10,000 rows, 100 manufacturers, 20 categories.
  c2  the MovieLens-20M shape: 138,493 users x 26,744 items, 20,000,263 rows, 1,000 manufacturers, 50 categories.
Timed:
  train    one epoch of train() (no validation), host clock around a synchronised call after one warm-up epoch:
           ms per step and examples/s.  c1: median of --reps epochs; c2: one epoch.
  torch    train_reference(device="cuda", dtype=float32) on a prefix of the same rows (--torch-steps steps, or the whole
           c1 epoch), after one warm-up step of the same batch size.
  kernels  CUDA events around --kernel-reps back-to-back launches of the step kernel alone and of the Adam kernel
           alone on one batch of the workload: the split of a step.  Adam moves >= 24 bytes per parameter (p, m, v
           read and written); that rate is reported against the 7.7 TB/s HBM data-sheet figure.  At c2 p, m and v take
           99 MB, under the 126 MB L2: back-to-back Adam launches can be served partly from L2 (no flush between them).
  check    (--check) c2's first 2,000,000 rows, one epoch at batch 1024 through train() and train_reference in fp32 on
           the GPU and fp64 on the CPU: the largest deviations from fp64 of both (the test's relative criterion).
Prints one JSON line per measurement and the GPU name and power limit; --out also writes them as a JSON list.
Usage: python scripts/bench_tower_train.py [--reps 5] [--torch-steps 200] [--check] [--out FILE] [--only c1|c2]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import pandas as pd
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hybrid_als_twotower_recommender_b200 as pkg  # noqa: E402
from hybrid_als_twotower_recommender_b200 import _native as nat, two_tower_model as ttm  # noqa: E402
from oracle import tower_train_oracle  # noqa: E402

HBM_TBS = 7.7
E = 50
SHAPES = {"c1": dict(users=10_000, items=10_000, rows=10_000, manu=100, cat=20),
          "c2": dict(users=138_493, items=26_744, rows=20_000_263, manu=1_000, cat=50)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": line}


def make_data(s, seed=0):
    rng = np.random.default_rng(seed)
    n, I = s["rows"], s["items"]
    item = rng.integers(0, I, n)
    manu_of, cat_of = rng.integers(0, s["manu"], I), rng.integers(0, s["cat"], I)
    price_of = rng.uniform(2, 250, I)
    return pd.DataFrame({"userId": rng.integers(0, s["users"], n), "itemId": item,
                         "manufacturer_id": manu_of[item], "category_id": cat_of[item], "price": price_of[item],
                         "average_review_rating": rng.integers(1, 6, n).astype(float)})


def model(s):
    m = pkg.TwoTowerModel(s["users"], s["items"], s["manu"], s["cat"], embedding_size=E, learning_rate=1e-3)
    m.build_model(seed=0)
    return m, {k: v.clone() for k, v in m.model.t.items()}


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def time_train(s, df, bs, reps):
    m, w0 = model(s)
    n = len(df)
    steps = -(-n // bs)

    def epoch():
        m.model = ttm.TowerParams({k: v.clone() for k, v in w0.items()}, E)
        m.train(df, None, batch_size=bs, epochs=1)
    epoch()                                          # warm-up: the allocator at this size, module load
    ts = [wall(epoch) for _ in range(reps)]
    sec = float(np.median(ts))
    return {"variant": "train", "batch": bs, "rows": n, "steps": steps, "ms_per_epoch": sec * 1e3,
            "ms_per_step": sec * 1e3 / steps, "examples_per_s": n / sec, "epochs_timed": reps}


def time_torch(s, df, bs, max_steps):
    _, w0 = model(s)
    rows = min(len(df), max_steps * bs)
    sub = df.iloc[:rows]
    tower_train_oracle.train_reference(w0, df.iloc[:bs], None, bs, 1, 1e-3, device="cuda", dtype=torch.float32)
    sec = wall(lambda: tower_train_oracle.train_reference(w0, sub, None, bs, 1, 1e-3, device="cuda", dtype=torch.float32))
    steps = -(-rows // bs)
    return {"variant": "torch_loop_fp32", "batch": bs, "rows_timed": rows, "steps_timed": steps,
            "ms_per_step": sec * 1e3 / steps, "examples_per_s": rows / sec,
            "note": "includes the host feature slicing and per-step loss read-back of the loop"}


def time_kernels(s, df, bs, reps):
    """The step kernel alone and the Adam kernel alone, back to back on one batch (CUDA events)."""
    m, _ = model(s)
    L = nat.lib()
    p = m.model
    mom = [ttm.TowerParams({k: torch.zeros_like(v) for k, v in p.t.items()}, E) for _ in range(2)]
    P, M, V = (ttm.nat_params(x) for x in (p, *mom))
    b = df.iloc[:bs]
    ids = [torch.tensor(b[c].values.astype(np.int32), device="cuda") for c, _ in ttm.TRAIN_IDS]
    order = [torch.argsort(x.long(), stable=True).to(torch.int32) for x in ids]
    num = torch.rand(bs, 2, device="cuda")
    y = torch.tensor(b["average_review_rating"].values.astype(np.float32), device="cuda")
    batch = nat.TowerBatch()
    batch.n = bs
    batch.user_ids, batch.item_ids, batch.manufacturer_ids, batch.category_ids = (x.data_ptr() for x in ids)
    batch.numeric, batch.labels = num.data_ptr(), y.data_ptr()
    batch.order_user, batch.order_item, batch.order_manufacturer, batch.order_category = (x.data_ptr() for x in order)
    wsb = int(L.hals_tower_train_workspace_bytes(P, bs))
    ws = torch.zeros(wsb, dtype=torch.uint8, device="cuda")
    loss = torch.zeros(1, device="cuda")
    st = nat.current_stream()

    def step(t):
        nat.check(L.hals_tower_train_step(P, batch, t, nat.ptr(ws), wsb, nat.ptr(loss), st))

    def adam(t):
        nat.check(L.hals_tower_adam_step(P, M, V, batch, t, nat.ptr(ws), wsb, 1e-3, 0.9, 0.999, 1e-7, st))

    def events(fn):
        fn(1)
        torch.cuda.synchronize()
        a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn(1)
        z.record()
        torch.cuda.synchronize()
        return a.elapsed_time(z) / reps
    step(1)
    ms_step, ms_adam = events(step), events(adam)
    n_params = sum(v.numel() for v in p.t.values())
    adam_bytes = 24 * n_params
    return {"variant": "kernels", "batch": bs, "launches_timed": reps, "step_kernel_us": ms_step * 1e3,
            "adam_kernel_us": ms_adam * 1e3, "params": n_params, "p_m_v_MB": 12 * n_params / 1e6,
            "adam_bytes_per_step": adam_bytes, "adam_TB_per_s": adam_bytes / (ms_adam * 1e-3) / 1e12,
            "adam_share_of_hbm_7.7TBs": adam_bytes / (ms_adam * 1e-3) / 1e12 / HBM_TBS}


def check(s, df):
    """One epoch on the first 2M rows at batch 1024: deviations from fp64 of the GPU trainer and the fp32 loop."""
    sub = df.iloc[:2_000_000]
    m, w0 = model(s)
    h = m.train(sub, None, batch_size=1024, epochs=1)
    pg = {k: v.double().cpu() for k, v in m.model.t.items()}
    p32, h32 = tower_train_oracle.train_reference(w0, sub, None, 1024, 1, 1e-3, device="cuda", dtype=torch.float32)
    p64, h64 = tower_train_oracle.train_reference(w0, sub, None, 1024, 1, 1e-3, device="cpu", dtype=torch.float64)
    out = {"variant": "check_2M_rows_batch1024", "loss": [h["loss"][0], h32["loss"][0], h64["loss"][0]]}
    ok = True
    for k in p64:
        dg = float((pg[k] - p64[k]).abs().max())
        d32 = float((p32[k].double().cpu() - p64[k]).abs().max())
        out[k] = [dg, d32]
        ok &= dg <= 2 * d32 + 1e-5
    dl = [abs(h["loss"][0] - h64["loss"][0]), abs(h32["loss"][0] - h64["loss"][0])]
    ok &= dl[0] <= 2 * dl[1] + 1e-5
    out.update({"loss_dev": dl, "within_test_criterion": bool(ok),
                "fields": "per tensor: [max |hals - fp64|, max |torch fp32 - fp64|]"})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--torch-steps", type=int, default=200)
    ap.add_argument("--kernel-reps", type=int, default=200)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--out")
    ap.add_argument("--only", choices=["c1", "c2"])
    a = ap.parse_args()
    nat.require_cuda()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    res = [info]
    for name, s in SHAPES.items():
        if a.only and a.only != name:
            continue
        df = make_data(s)
        rows = []
        for bs in (256, 1024):
            rows.append(time_train(s, df, bs, a.reps if name == "c1" else 1))
            rows.append(time_torch(s, df, bs, a.torch_steps if name == "c2" else 10 ** 9))
            rows.append(time_kernels(s, df, bs, a.kernel_reps))
            rows.append({"variant": "speedup_train_over_torch_loop", "batch": bs,
                         "ratio": rows[-3]["examples_per_s"] / rows[-2]["examples_per_s"]})
        if a.check and name == "c2":
            rows.append(check(s, df))
        for r in rows:
            r["workload"] = name
            print(json.dumps(r), flush=True)
            res.append(r)
        del df
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
