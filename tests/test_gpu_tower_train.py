"""TwoTowerModel.train on the GPU trainer (hals_tower_train_step + hals_tower_adam_step, csrc/tower_train.cu) against
the fp64 torch oracle, oracle/tower_train_oracle.py:train_reference, at four levels:
  1. the gradients of one step (read back through an Adam step with beta1 = 0, lr = 0, which leaves m = g exactly);
  2. one Adam step against torch's update evaluated in fp64, stage by stage from the kernel's own fp32 inputs;
  3. whole train() runs: the CUDA trainer's deviation from fp64 is at most twice that of the fp32 torch loop on the
     same GPU, plus a small absolute floor (Adam amplifies rounding on near-zero gradients in both);
  4. early stopping on an overfitting case: the same epochs as the oracle and the best epoch's weights.
Plus determinism (bitwise) and a constant number of launches per step."""
import numpy as np
import pandas as pd
import pytest
import torch

from oracle import tower_train_oracle

pytestmark = pytest.mark.gpu
TABLES = {"user": 300, "item": 500, "manu": 13, "cat": 7}
# level 1: max |g - g_fp64| / max(max |g_fp64|, GRAD_FLOOR) per tensor.  Measured on a B200: at most 8.2e-7 over the
# uncrowded cases and 2.1e-6 for the crowded B = 4096 batch (one user and one item in 80 % of the rows), so 1e-5 keeps
# >= 4.7x headroom.  The floor covers E = 1, where the LayerNorm of one value is constant: every gradient into the
# embeddings and the LN gain is zero in exact arithmetic, and the fp64 values are rounding noise (~1e-17).
GRAD_TOL = 1e-5
GRAD_FLOOR = 1e-6
# level 2, in ulps of the largest magnitude entering the stage.  m = lerp(m, g, 1 - b1) and v = v b2 + (1 - b2) g^2 are
# one or two rounded operations (bounds 2.5 and 2 ulp); the update m / (sqrt(v) / sqrt(bc2) + eps) passes through four
# rounded operations before p - step * u, so p is held to 4 ulp of max(|p|, |p_new|, |step * u|).  CPU emulation of the
# kernel's arithmetic over 4M random elements reaches 2.07, 1.48 and 3.1; measured on a B200 here: 1.28, 1.43, 1.90.
ULP_TOL = {"m": 2.5, "v": 2.0, "p": 4.0}


def _pkg():
    import hybrid_als_twotower_recommender_b200 as pkg
    from hybrid_als_twotower_recommender_b200 import _native as nat
    from hybrid_als_twotower_recommender_b200 import two_tower_model as ttm
    return pkg, nat, ttm


def make_weights(E, MD, CD, H, seed, tables=TABLES):
    """As tests/test_gpu_towers.py: Keras-like ranges, nonzero LayerNorm gains / biases and Dense biases."""
    rng = np.random.default_rng(seed)

    def u(*shape, lim=0.05):
        return rng.uniform(-lim, lim, shape).astype(np.float32)

    def n(size, mean=0.0):
        return (mean + 0.1 * rng.standard_normal(size)).astype(np.float32)

    C = E + MD + CD + H
    return {"user_emb": u(tables["user"], E), "item_emb": u(tables["item"], E), "manu_emb": u(tables["manu"], MD),
            "cat_emb": u(tables["cat"], CD), "num_w": u(2, H, lim=np.sqrt(6 / (2 + H))), "num_b": n(H),
            "out_w": u(C, E, lim=np.sqrt(6 / (C + E))), "out_b": n(E), "user_ln_g": n(E, 1.0), "user_ln_b": n(E),
            "item_ln_g": n(E, 1.0), "item_ln_b": n(E)}


def make_batch(rng, B, crowded=False, tables=TABLES):
    ids = {k: rng.integers(0, tables[k], B).astype(np.int32) for k in ("user", "item", "manu", "cat")}
    if crowded:                               # one user and one item fill most rows
        hot = rng.random(B) < 0.8
        ids["user"][hot] = 7
        ids["item"][rng.random(B) < 0.8] = 11
    num = np.stack([rng.uniform(0, 1, B), rng.uniform(0, 1, B)], 1).astype(np.float32)   # already scaled
    y = rng.uniform(1, 5, B).astype(np.float32)
    return ids, num, y


class Step:
    """One hals_tower_train_step + hals_tower_adam_step on device copies of fp32 numpy weights."""

    def __init__(self, w, B):
        _, nat, ttm = _pkg()
        self.nat, self.L = nat, nat.lib()
        E = w["user_emb"].shape[1]
        self.p = ttm.TowerParams.from_numpy(w, torch.device("cuda"))
        self.m = ttm.TowerParams({k: torch.zeros_like(v) for k, v in self.p.t.items()}, E)
        self.v = ttm.TowerParams({k: torch.zeros_like(v) for k, v in self.p.t.items()}, E)
        self.P, self.M, self.V = (ttm.nat_params(x) for x in (self.p, self.m, self.v))
        self.ws_bytes = int(self.L.hals_tower_train_workspace_bytes(self.P, B))
        self.ws = torch.zeros(self.ws_bytes, dtype=torch.uint8, device="cuda")
        self.loss = torch.zeros(1, device="cuda")

    def set_state(self, p=None, m=None, v=None):
        for src, dst in ((p, self.p), (m, self.m), (v, self.v)):
            if src is not None:
                for k in dst.t:
                    dst.t[k].copy_(torch.as_tensor(src[k]))

    def run(self, ids, num, y, t, lr=0.0, b1=0.0, b2=0.0, eps=1e-7):
        nat = self.nat
        d = {k: torch.from_numpy(np.ascontiguousarray(a)).cuda() for k, a in ids.items()}
        order = {k: torch.from_numpy(np.argsort(a, kind="stable").astype(np.int32)).cuda() for k, a in ids.items()}
        numd, yd = torch.from_numpy(num).cuda(), torch.from_numpy(y).cuda()
        b = nat.TowerBatch()
        b.n = len(y)
        b.user_ids, b.item_ids, b.manufacturer_ids, b.category_ids = (d[k].data_ptr() for k in ("user", "item", "manu", "cat"))
        b.numeric, b.labels = numd.data_ptr(), yd.data_ptr()
        b.order_user, b.order_item, b.order_manufacturer, b.order_category = (
            order[k].data_ptr() for k in ("user", "item", "manu", "cat"))
        st = nat.current_stream()
        nat.check(self.L.hals_tower_train_step(self.P, b, t, nat.ptr(self.ws), self.ws_bytes, nat.ptr(self.loss), st))
        nat.check(self.L.hals_tower_adam_step(self.P, self.M, self.V, b, t, nat.ptr(self.ws), self.ws_bytes, lr, b1, b2,
                                              eps, st))
        torch.cuda.synchronize()
        return float(self.loss.item())

    def state(self):
        return tuple({k: x.cpu().numpy().copy() for k, x in s.t.items()} for s in (self.p, self.m, self.v))


def hals_grads(w, ids, num, y):
    """The kernel's gradients: one Adam step with beta1 = 0 and lr = 0 leaves m = lerp(0, g, 1) = g exactly."""
    s = Step(w, len(y))
    loss = s.run(ids, num, y, 1)
    return s.state()[1], loss


def fp64_grads(w, ids, num, y):
    p = {k: torch.from_numpy(v).double().requires_grad_(True) for k, v in w.items()}
    f = {"user_in": ids["user"], "item_id_in": ids["item"], "manufacturer_in": ids["manu"], "category_in": ids["cat"],
         "numeric_in": num}
    pred = tower_train_oracle.torch_forward(p, f, torch.device("cpu"), w["user_emb"].shape[1], torch.float64)
    loss = ((pred - torch.from_numpy(y).double()) ** 2).mean()
    loss.backward()
    return {k: v.grad.numpy() for k, v in p.items()}, float(loss)


GRAD_CASES = [(E, (8, 8, 16), B, False) for E in (1, 32, 33, 50, 64) for B in (1, 7, 256, 4096)] + [
    (50, (4, 12, 32), 256, False), (20, (1, 1, 1), 256, False), (50, (8, 8, 16), 256, True),
    (33, (8, 8, 16), 4096, True)]


@pytest.mark.parametrize("E,dims,B,crowded", GRAD_CASES)
def test_step_gradients_match_fp64_autograd(E, dims, B, crowded):
    w = make_weights(E, *dims, seed=E * 7 + B)
    rng = np.random.default_rng(B + E)
    ids, num, y = make_batch(rng, B, crowded)
    got, loss = hals_grads(w, ids, num, y)
    want, wloss = fp64_grads(w, ids, num, y)
    assert loss == pytest.approx(wloss, rel=1e-5)
    worst = {}
    for k in w:
        scale = np.abs(want[k]).max()
        err = np.abs(got[k].astype(np.float64) - want[k]).max()
        worst[k] = err / max(scale, GRAD_FLOOR)
    # untouched embedding rows have an exactly zero gradient
    for k, tbl, key in (("user_emb", "user", "user"), ("item_emb", "item", "item")):
        untouched = np.setdiff1d(np.arange(TABLES[tbl]), ids[key])
        assert (got[k][untouched] == 0).all()
    print("grad rel err", E, dims, B, crowded, {k: f"{v:.1e}" for k, v in worst.items()})
    assert max(worst.values()) <= GRAD_TOL, worst


def ulps(got, want, scale):
    """|got - want| in units of the fp32 spacing at |scale| (elementwise)."""
    sp = np.spacing(np.abs(scale).astype(np.float32)).astype(np.float64)
    sp = np.maximum(sp, np.float64(np.finfo(np.float32).smallest_subnormal))
    return np.abs(got.astype(np.float64) - want) / sp


def check_adam(before, after, g, t, lr, b1, b2, eps):
    """torch's update in fp64 with the fp32 scalars torch applies to fp32 tensors (1 - b1, b2, 1 - b2, lr / bc1 and
    sqrt(bc2), each computed in double and rounded once), stage by stage from the kernel's fp32 inputs of the stage."""
    f32 = lambda x: float(np.float32(x))    # noqa: E731
    bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
    w1, B2, o2, step, bs = f32(1 - b1), f32(b2), f32(1 - b2), f32(lr / bc1), f32(np.sqrt(bc2))
    p0, m0, v0 = ({k: x.astype(np.float64) for k, x in d.items()} for d in before)
    p1, m1, v1 = after
    for k in p0:
        gk = g[k].astype(np.float64)
        wm = m0[k] + w1 * (gk - m0[k])
        wv = v0[k] * B2 + o2 * gk * gk
        u = step * m1[k].astype(np.float64) / (np.sqrt(v1[k].astype(np.float64)) / bs + eps)
        wp = p0[k] - u
        for name, got, want, scale in (
                ("m", m1[k], wm, np.maximum.reduce([np.abs(m0[k]), np.abs(wm), np.abs(w1 * gk)])),
                ("v", v1[k], wv, wv),
                ("p", p1[k], wp, np.maximum.reduce([np.abs(p0[k]), np.abs(wp), np.abs(u)]))):
            e = float(ulps(got, want, scale).max())
            print("adam ulps", k, name, t, e)
            assert e <= ULP_TOL[name], (k, name, t, e)


def test_adam_step_matches_the_fp64_update():
    """t = 1 from zero moments; t = 2 on a batch that leaves the step-1 rows alone (their g = 0: moments decay, the
    parameter still moves); t = 10**6 from random moments."""
    w = make_weights(50, 8, 8, 16, seed=3)
    rng = np.random.default_rng(4)
    lr, b1, b2, eps = 1e-3, 0.9, 0.999, 1e-7
    ids1, num1, y1 = make_batch(rng, 256)
    ids2, num2, y2 = make_batch(rng, 256)
    ids2["user"] = rng.integers(150, 300, 256).astype(np.int32)       # disjoint from step 1's users ...
    ids1["user"] = rng.integers(0, 150, 256).astype(np.int32)
    s = Step(w, 256)
    before = s.state()
    g1, _ = hals_grads(before[0], ids1, num1, y1)
    s.run(ids1, num1, y1, 1, lr, b1, b2, eps)
    after1 = s.state()
    check_adam(before, after1, g1, 1, lr, b1, b2, eps)
    g2, _ = hals_grads(after1[0], ids2, num2, y2)
    assert (g2["user_emb"][:150] == 0).all() and (after1[1]["user_emb"][np.unique(ids1["user"])] != 0).any()
    s.run(ids2, num2, y2, 2, lr, b1, b2, eps)
    after2 = s.state()
    check_adam(after1, after2, g2, 2, lr, b1, b2, eps)
    touched1 = np.unique(ids1["user"])
    assert (after2[0]["user_emb"][touched1] != after1[0]["user_emb"][touched1]).any()
    # a large t from random moments
    m0 = {k: (rng.standard_normal(v.shape) * 1e-3).astype(np.float32) for k, v in w.items()}
    v0 = {k: (rng.random(v.shape) * 1e-5).astype(np.float32) for k, v in w.items()}
    s2 = Step(w, 256)
    s2.set_state(m=m0, v=v0)
    before = s2.state()
    g3, _ = hals_grads(w, ids1, num1, y1)
    s2.run(ids1, num1, y1, 10 ** 6, lr, b1, b2, eps)
    check_adam(before, s2.state(), g3, 10 ** 6, lr, b1, b2, eps)


# ------------------------------------------------------------------------------------------------------------------
def make_frame(rng, n, tables=TABLES, strays=0):
    df = pd.DataFrame({"userId": rng.integers(0, tables["user"], n), "itemId": rng.integers(0, tables["item"], n),
                       "manufacturer_id": rng.integers(0, tables["manu"], n),
                       "category_id": rng.integers(0, tables["cat"], n), "price": rng.uniform(2, 250, n),
                       "average_review_rating": rng.integers(1, 6, n).astype(float)})
    if strays:                                # validation ids outside the tables read as zero rows
        idx = rng.choice(n, strays, replace=False)
        df.loc[idx[: strays // 2], "userId"] = tables["user"] + 5
        df.loc[idx[strays // 2:], "itemId"] = tables["item"] + 10 ** 6
    return df


def run_all(w, tr, va, bs, epochs, lr):
    """(hals trainer, fp32 torch on the GPU, fp64 torch on the CPU): (weights, history) each."""
    pkg, nat, ttm = _pkg()
    m = pkg.TwoTowerModel(TABLES["user"], TABLES["item"], TABLES["manu"], TABLES["cat"],
                          embedding_size=w["user_emb"].shape[1], learning_rate=lr)
    m.model = ttm.TowerParams.from_numpy(w, torch.device("cuda"))
    h = m.train(tr, va, batch_size=bs, epochs=epochs)
    got = ({k: v.cpu().numpy() for k, v in m.model.t.items()}, h)
    p32, h32 = tower_train_oracle.train_reference(w, tr, va, bs, epochs, lr, device="cuda", dtype=torch.float32)
    p64, h64 = tower_train_oracle.train_reference(w, tr, va, bs, epochs, lr, device="cpu", dtype=torch.float64)
    return got, ({k: v.cpu().numpy() for k, v in p32.items()}, h32), ({k: v.numpy() for k, v in p64.items()}, h64), m


def relative_check(got, ref32, ref64, floor):
    (pg, hg), (p32, h32), (p64, h64) = got, ref32, ref64
    assert len(hg["loss"]) == len(h64["loss"]) and len(hg["val_loss"]) == len(h64["val_loss"])
    report = {}
    for k in p64:
        dg, d32 = np.abs(pg[k] - p64[k]).max(), np.abs(p32[k] - p64[k]).max()
        report[k] = (float(dg), float(d32))
        assert dg <= 2 * d32 + floor, (k, dg, d32)
    for key in ("loss", "val_loss"):
        dg = np.abs(np.array(hg[key]) - np.array(h64[key])).max(initial=0.0)
        d32 = np.abs(np.array(h32[key]) - np.array(h64[key])).max(initial=0.0)
        report[key] = (float(dg), float(d32))
        assert dg <= 2 * d32 + floor, (key, dg, d32)
    print("deviation from fp64 (hals, torch fp32):", {k: f"{a:.1e}/{b:.1e}" for k, (a, b) in report.items()})


@pytest.mark.parametrize("n,bs,epochs", [(300, 512, 4), (1000, 96, 3)])
def test_train_matches_the_fp64_oracle(n, bs, epochs):
    """batch_size > n (one short batch per epoch) and n % batch_size != 0; validation ids outside the tables."""
    rng = np.random.default_rng(n)
    w = make_weights(50, 8, 8, 16, seed=n)
    tr, va = make_frame(rng, n), make_frame(rng, 200, strays=20)
    got, r32, r64, _ = run_all(w, tr, va, bs, epochs, 1e-3)
    relative_check(got, r32, r64, floor=1e-5)


def test_early_stopping_restores_the_best_epoch():
    """lr 0.05 on 120 rows with noise labels: the validation loss (fp64 oracle: 1.155, 1.275, 1.597, 1.489) rises
    from the first epoch on, so training stops after four epochs with the first epoch's weights."""
    rng = np.random.default_rng(11)
    tables = {"user": 20, "item": 30, "manu": 4, "cat": 3}
    w = make_weights(50, 8, 8, 16, seed=5, tables=tables)
    for k in ("user_ln_g", "item_ln_g"):
        w[k] = (w[k] * 0.3).astype(np.float32)
    tr, va = make_frame(rng, 120, tables), make_frame(rng, 100, tables)
    tr["average_review_rating"], va["average_review_rating"] = rng.normal(0, 1, 120), rng.normal(0, 1, 100)
    pkg, nat, ttm = _pkg()
    m = pkg.TwoTowerModel(20, 30, 4, 3, embedding_size=50, learning_rate=0.05)
    m.model = ttm.TowerParams.from_numpy(w, torch.device("cuda"))
    h = m.train(tr, va, batch_size=16, epochs=12)
    _, h64 = tower_train_oracle.train_reference(w, tr, va, 16, 12, 0.05, device="cpu", dtype=torch.float64)
    assert len(h["val_loss"]) == len(h64["val_loss"]) < 12, (h, h64)
    assert max(h["val_loss"][int(np.argmin(h["val_loss"])):]) > min(h["val_loss"]) * 1.05    # it clearly rose
    # the returned weights are the best epoch's: their validation loss (val-fitted scaling, as train computes it)
    from sklearn.preprocessing import MinMaxScaler
    vf = tower_train_oracle.prepare_features(MinMaxScaler(), va)
    p = {k: v.double() for k, v in m.model.t.items()}
    pred = tower_train_oracle.torch_forward(p, vf, torch.device("cuda"), 50, torch.float64)
    vl = float(((pred - torch.tensor(va["average_review_rating"].values, device="cuda")) ** 2).mean())
    assert vl == pytest.approx(min(h["val_loss"]), rel=1e-5)


def test_train_is_bitwise_deterministic():
    rng = np.random.default_rng(21)
    w = make_weights(50, 8, 8, 16, seed=21)
    tr, va = make_frame(rng, 2000), make_frame(rng, 300, strays=10)
    pkg, nat, ttm = _pkg()
    outs = []
    for _ in range(2):
        m = pkg.TwoTowerModel(TABLES["user"], TABLES["item"], TABLES["manu"], TABLES["cat"], embedding_size=50)
        m.model = ttm.TowerParams.from_numpy(w, torch.device("cuda"))
        h = m.train(tr, va, batch_size=64, epochs=2)
        outs.append(({k: v.cpu().numpy() for k, v in m.model.t.items()}, h))
    assert outs[0][1] == outs[1][1]
    for k in outs[0][0]:
        assert np.array_equal(outs[0][0][k], outs[1][0][k]), k


def test_launches_per_step_are_constant():
    rng = np.random.default_rng(22)
    w = make_weights(50, 8, 8, 16, seed=22)
    tr = make_frame(rng, 3000)
    pkg, nat, ttm = _pkg()
    per_step = []
    for bs in (64, 1000):
        m = pkg.TwoTowerModel(TABLES["user"], TABLES["item"], TABLES["manu"], TABLES["cat"], embedding_size=50)
        m.model = ttm.TowerParams.from_numpy(w, torch.device("cuda"))
        for epochs in (1, 2):
            c0 = nat.launch_count()
            m.train(tr, None, batch_size=bs, epochs=epochs)
            per_step.append((nat.launch_count() - c0) / (epochs * -(-3000 // bs)))
    assert per_step == [2.0] * 4, per_step


def test_train_rejects_wide_embeddings_and_bad_ids_before_device_work():
    pkg, nat, ttm = _pkg()
    rng = np.random.default_rng(23)
    tr = make_frame(rng, 50)
    m = pkg.TwoTowerModel(TABLES["user"], TABLES["item"], TABLES["manu"], TABLES["cat"], embedding_size=65)
    with pytest.raises(ValueError, match=r"\[1, 64\]"):
        m.train(tr, None)
    assert m.model is None
    m = pkg.TwoTowerModel(10, TABLES["item"], TABLES["manu"], TABLES["cat"], embedding_size=16)
    c0 = nat.launch_count()
    with pytest.raises(IndexError, match="ids must lie in"):
        m.train(tr, None)
    with pytest.raises(ValueError):
        pkg.TwoTowerModel(*TABLES.values(), embedding_size=16).train(tr, None, batch_size=0)
    with pytest.raises(TypeError):
        pkg.TwoTowerModel(*TABLES.values(), embedding_size=16).train(tr, None, batch_size=2.5)
    assert nat.launch_count() == c0


def test_c_abi_rejects_bad_arguments():
    pkg, nat, ttm = _pkg()
    L = nat.lib()
    w = make_weights(16, 8, 8, 16, seed=1)
    s = Step(w, 8)
    b = nat.TowerBatch()
    b.n = 8
    assert L.hals_tower_train_step(s.P, b, 1, nat.ptr(s.ws), s.ws_bytes, nat.ptr(s.loss), None) == 1   # null ids
    P = ttm.nat_params(s.p)
    P.embedding_size = 65
    assert L.hals_tower_train_workspace_bytes(s.P, 0) == 0
    assert L.hals_tower_train_step(P, b, 1, nat.ptr(s.ws), s.ws_bytes, nat.ptr(s.loss), None) == 1
    assert b"embedding_size" in L.hals_last_error()
