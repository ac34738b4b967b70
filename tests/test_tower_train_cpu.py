"""CPU: oracle/tower_train_oracle.py:train_reference, the torch loop the GPU trainer is tested against and timed against.
  - in fp64 it applies torch.optim.Adam's update exactly as restated in csrc/tower_train.cu (lerp, addcmul, bias
    corrections in double);
  - in fp32 on the CPU its first epoch is bit-identical to the loop TwoTowerModel.train ran before the GPU trainer
    (inlined below as it was)."""
import numpy as np
import pandas as pd
import torch
import torch.nn.functional as F
from sklearn.preprocessing import MinMaxScaler

from oracle import tower_train_oracle, towers_oracle

TABLES = (40, 60, 5, 4)


def frame(rng, n):
    U, I, M, C = TABLES
    return pd.DataFrame({"userId": rng.integers(0, U, n), "itemId": rng.integers(0, I, n),
                         "manufacturer_id": rng.integers(0, M, n), "category_id": rng.integers(0, C, n),
                         "price": rng.uniform(2, 250, n), "average_review_rating": rng.integers(1, 6, n).astype(float)})


def weights(E=16, seed=0):
    w = towers_oracle.init_weights(*TABLES, embedding_size=E, seed=seed)
    return w


def test_fp64_step_is_the_restated_adam_update():
    rng = np.random.default_rng(0)
    w, tr = weights(), frame(rng, 50)
    lr = 3e-3
    got, _ = tower_train_oracle.train_reference(w, tr, None, 64, 1, lr, device="cpu", dtype=torch.float64)   # one step
    p = {k: torch.from_numpy(v).double().requires_grad_(True) for k, v in w.items()}
    f = tower_train_oracle.prepare_features(MinMaxScaler(), tr)
    perm = torch.randperm(len(tr), generator=torch.Generator("cpu").manual_seed(0)).numpy()
    fb = {k: np.asarray(v)[perm] for k, v in f.items()}
    y = torch.tensor(tr["average_review_rating"].values.astype(np.float32)[perm]).double()
    loss = ((tower_train_oracle.torch_forward(p, fb, torch.device("cpu"), 16, torch.float64) - y) ** 2).mean()
    loss.backward()
    b1, b2, eps, t = 0.9, 0.999, 1e-7, 1
    for k, v in p.items():
        g = v.grad.detach()
        m = torch.zeros_like(g).lerp_(g, 1 - b1)
        vv = torch.zeros_like(g).mul_(b2).addcmul_(g, g, value=1 - b2)
        bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
        want = v.detach() - (lr / bc1) * m / (vv.sqrt() / bc2 ** 0.5 + eps)
        assert torch.allclose(got[k], want, rtol=1e-14, atol=1e-17), k


def parent_train(model_t, E, lr, train_data, val_data, batch_size, epochs):
    """TwoTowerModel.train as it was before the GPU trainer (self.* made arguments)."""
    LN_EPS = 1e-3
    scaler = MinMaxScaler()

    def prep(data):
        return {"user_in": data["userId"].values, "item_id_in": data["itemId"].values,
                "manufacturer_in": data["manufacturer_id"].values, "category_in": data["category_id"].values,
                "numeric_in": scaler.fit_transform(data[["price", "average_review_rating"]])}

    def fwd(p, f, dev):
        def rows(table, ids):
            ids = torch.as_tensor(np.asarray(ids), device=dev).long()
            ok = (ids >= 0) & (ids < table.shape[0])
            return table[torch.where(ok, ids, torch.zeros_like(ids))] * ok.unsqueeze(1).to(table.dtype)
        u = F.layer_norm(rows(p["user_emb"], f["user_in"]), (E,), p["user_ln_g"], p["user_ln_b"], LN_EPS)
        num = torch.as_tensor(np.asarray(f["numeric_in"], dtype=np.float32), device=dev)
        h = torch.relu(num @ p["num_w"] + p["num_b"])
        cat = torch.cat([rows(p["item_emb"], f["item_id_in"]), rows(p["manu_emb"], f["manufacturer_in"]),
                         rows(p["cat_emb"], f["category_in"]), h], dim=1)
        i = F.layer_norm(cat @ p["out_w"] + p["out_b"], (E,), p["item_ln_g"], p["item_ln_b"], LN_EPS)
        return (u * i).sum(dim=1)

    dev = model_t["user_emb"].device
    params = {k: v.clone().requires_grad_(True) for k, v in model_t.items()}
    opt = torch.optim.Adam(list(params.values()), lr=lr, eps=1e-7)
    has_val = val_data is not None and len(val_data) > 0
    tf = prep(train_data)
    y = torch.as_tensor(train_data["average_review_rating"].values.astype(np.float32), device=dev)
    vf = prep(val_data) if has_val else None
    vy = torch.as_tensor(val_data["average_review_rating"].values.astype(np.float32), device=dev) if has_val else None
    if has_val:
        tf = prep(train_data)
    n = len(train_data)
    history = {"loss": [], "val_loss": []}
    g = torch.Generator(device="cpu").manual_seed(0)
    for _ in range(int(epochs)):
        perm = torch.randperm(n, generator=g).numpy()
        tot = 0.0
        for s in range(0, n, batch_size):
            b = perm[s:s + batch_size]
            fb = {k: np.asarray(v)[b] for k, v in tf.items()}
            loss = ((fwd(params, fb, dev) - y[torch.as_tensor(b, device=dev)]) ** 2).mean()
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            tot += float(loss.detach()) * len(b)
        history["loss"].append(tot / max(n, 1))
        if has_val:
            with torch.no_grad():
                history["val_loss"].append(float(((fwd(params, vf, dev) - vy) ** 2).mean()))
    return {k: v.detach() for k, v in params.items()}, history


def test_fp32_first_epoch_is_bit_identical_to_the_previous_loop():
    rng = np.random.default_rng(1)
    w = weights(E=24, seed=1)
    tr, va = frame(rng, 300), frame(rng, 80)
    va.loc[:5, "userId"] = TABLES[0] + 3                     # validation ids outside the table read as zero rows
    want_p, want_h = parent_train({k: torch.from_numpy(v.copy()) for k, v in w.items()}, 24, 1e-3, tr, va, 64, 1)
    got_p, got_h = tower_train_oracle.train_reference(w, tr, va, 64, 1, 1e-3, device="cpu", dtype=torch.float32)
    assert got_h == want_h
    for k in w:
        assert torch.equal(got_p[k], want_p[k]), k
