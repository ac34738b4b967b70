"""CPU/GPU ORACLE (test infrastructure, NOT product code) -- two-tower training.

train_reference is the torch Adam/MSE loop TwoTowerModel.train ran before it moved onto the CUDA trainer
(csrc/tower_train.cu), unchanged except that the device and dtype are parameters.  fp64 on the CPU it is the oracle of
tests/test_gpu_tower_train.py; fp32 on the GPU it is the baseline of scripts/bench_tower_train.py.  The forward graph
is the one oracle/towers_oracle.py restates (Keras LayerNormalization defaults, ids outside a table read as zero rows).
"""
from __future__ import annotations

import numpy as np

from .towers_oracle import LN_EPS

TRAIN_IDS = (("userId", "user_emb"), ("itemId", "item_emb"), ("manufacturer_id", "manu_emb"),
             ("category_id", "cat_emb"))


def prepare_features(scaler, data):
    """TwoTowerModel._prepare_features: the scaler is re-fitted on `data` (fit_transform)."""
    return {
        "user_in": data["userId"].values,
        "item_id_in": data["itemId"].values,
        "manufacturer_in": data["manufacturer_id"].values,
        "category_in": data["category_id"].values,
        "numeric_in": scaler.fit_transform(data[["price", "average_review_rating"]]),
    }


def torch_forward(p, f, dev, E, dtype):
    import torch
    import torch.nn.functional as F

    def rows(table, ids):
        # an id outside its table reads as a zero embedding row (what the tower kernels do)
        ids = torch.as_tensor(np.asarray(ids), device=dev).long()
        ok = (ids >= 0) & (ids < table.shape[0])
        return table[torch.where(ok, ids, torch.zeros_like(ids))] * ok.unsqueeze(1).to(table.dtype)

    u = F.layer_norm(rows(p["user_emb"], f["user_in"]), (E,), p["user_ln_g"], p["user_ln_b"], LN_EPS)
    num = torch.as_tensor(np.asarray(f["numeric_in"], dtype=np.float32), device=dev).to(dtype)
    h = torch.relu(num @ p["num_w"] + p["num_b"])
    cat = torch.cat([rows(p["item_emb"], f["item_id_in"]), rows(p["manu_emb"], f["manufacturer_in"]),
                     rows(p["cat_emb"], f["category_in"]), h], dim=1)
    i = F.layer_norm(cat @ p["out_w"] + p["out_b"], (E,), p["item_ln_g"], p["item_ln_b"], LN_EPS)
    return (u * i).sum(dim=1)


def train_reference(weights, train_frame, val_frame, batch_size, epochs, lr, *, device, dtype):
    """Adam(lr, eps=1e-7) on MSE, EarlyStopping(patience=3, best weights restored) when val_frame has rows.
    weights: name -> array or tensor (the initial parameters, cloned); frames: DataFrames with the columns train takes.
    Returns (name -> tensor on `device` in `dtype`, history)."""
    import torch
    from sklearn.preprocessing import MinMaxScaler
    dev = torch.device(device)
    params = {k: torch.as_tensor(np.asarray(v.detach().cpu()) if hasattr(v, "detach") else np.asarray(v))
              .to(device=dev, dtype=dtype).clone().requires_grad_(True) for k, v in weights.items()}
    E = int(params["user_emb"].shape[1])
    opt = torch.optim.Adam(list(params.values()), lr=lr, eps=1e-7)
    has_val = val_frame is not None and len(val_frame) > 0
    for col, table in TRAIN_IDS:
        ids = train_frame[col].values
        n_rows = int(params[table].shape[0])
        if len(ids) and (ids.min() < 0 or ids.max() >= n_rows):
            raise IndexError(f"{col}: ids must lie in [0, {n_rows}) (found {int(ids.min())}..{int(ids.max())})")
    scaler = MinMaxScaler()
    tf = prepare_features(scaler, train_frame)
    y = torch.as_tensor(train_frame["average_review_rating"].values.astype(np.float32), device=dev).to(dtype)
    vf = prepare_features(scaler, val_frame) if has_val else None
    vy = (torch.as_tensor(val_frame["average_review_rating"].values.astype(np.float32), device=dev).to(dtype)
          if has_val else None)
    n = len(train_frame)
    history = {"loss": [], "val_loss": []}
    best, best_state, bad = float("inf"), None, 0
    g = torch.Generator(device="cpu").manual_seed(0)
    for _ in range(int(epochs)):
        perm = torch.randperm(n, generator=g).numpy()
        tot = 0.0
        for s in range(0, n, batch_size):
            b = perm[s:s + batch_size]
            fb = {k: np.asarray(v)[b] for k, v in tf.items()}
            loss = ((torch_forward(params, fb, dev, E, dtype) - y[torch.as_tensor(b, device=dev)]) ** 2).mean()
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            tot += float(loss.detach()) * len(b)
        history["loss"].append(tot / max(n, 1))
        if has_val:
            with torch.no_grad():
                vl = float(((torch_forward(params, vf, dev, E, dtype) - vy) ** 2).mean())
            history["val_loss"].append(vl)
            if vl < best:
                best, bad = vl, 0
                best_state = {k: v.detach().clone() for k, v in params.items()}
            else:
                bad += 1
                if bad >= 3:
                    break
    final = best_state if best_state is not None else {k: v.detach() for k, v in params.items()}
    return {k: v.contiguous() for k, v in final.items()}, history
