"""hals_tower_user / hals_tower_item against oracle/towers_oracle.py at the widths, strides and row counts the C ABI
accepts: embedding sizes on either side of one warp (E <= 32 uses one value per lane, E > 32 two), non-reference
manufacturer / category / hidden widths, a column slice of a wider output buffer, more rows than one grid pass covers,
and ids outside every table (a zero embedding).  Weights carry non-trivial LayerNorm gains and biases and nonzero
Dense biases so that every term shows.  Tolerance: 2e-5 on tower outputs, as for the reference fixture."""
import types

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import towers_oracle

pytestmark = pytest.mark.gpu
TOL = 2e-5
N_ROWS = 20000          # > 8 blocks x 8 warps x 148 SMs = 9472: the grid-stride loops wrap
TABLES = {"user": 300, "item": 500, "manu": 13, "cat": 7}
SCALER = types.SimpleNamespace(scale_=np.array([0.004, 0.25]), min_=np.array([-0.01, -0.25]))


def _pkg():
    import hybrid_als_twotower_recommender_b200 as pkg
    from hybrid_als_twotower_recommender_b200 import _native
    from hybrid_als_twotower_recommender_b200.two_tower_model import TowerParams
    return pkg, _native, TowerParams


def make_weights(E, MD, CD, H, seed):
    rng = np.random.default_rng(seed)

    def u(*shape, lim=0.05):
        return rng.uniform(-lim, lim, shape).astype(np.float32)

    def n(size, mean=0.0):
        return (mean + 0.1 * rng.standard_normal(size)).astype(np.float32)

    C = E + MD + CD + H
    return {"user_emb": u(TABLES["user"], E), "item_emb": u(TABLES["item"], E), "manu_emb": u(TABLES["manu"], MD),
            "cat_emb": u(TABLES["cat"], CD), "num_w": u(2, H, lim=np.sqrt(6 / (2 + H))), "num_b": n(H),
            "out_w": u(C, E, lim=np.sqrt(6 / (C + E))), "out_b": n(E), "user_ln_g": n(E, 1.0), "user_ln_b": n(E),
            "item_ln_g": n(E, 1.0), "item_ln_b": n(E)}


def with_zero_rows(w):
    """The oracle's tables with one zero row appended: an out-of-range id maps there (Keras' GPU Embedding)."""
    w = dict(w)
    for k in ("user_emb", "item_emb", "manu_emb", "cat_emb"):
        w[k] = np.vstack([w[k], np.zeros((1, w[k].shape[1]), np.float32)])
    return w


def ids_with_strays(rng, rows, n):
    """Random ids in [0, rows) with a few outside: -1, -rows, rows, 10**6."""
    ids = rng.integers(0, rows, n).astype(np.int32)
    ids[rng.choice(n, 40, replace=False)] = rng.choice([-1, -rows, rows, 10 ** 6], 40)
    return ids


def oracle_ids(ids, rows):
    return np.where((ids >= 0) & (ids < rows), ids, rows)


def run_towers(nat, TowerParams, w, uid, iid, mid, cid, num, col0, pad):
    """Both towers written into columns [col0, col0 + E) of poisoned [n, E + pad] buffers."""
    E = w["user_emb"].shape[1]
    tp = TowerParams.from_numpy(w, torch.device("cuda"))
    s = tp.struct(SCALER)
    assert (s.manu_dim, s.cat_dim, s.num_hidden) == (w["manu_emb"].shape[1], w["cat_emb"].shape[1], w["num_b"].size)
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in
         (("uid", uid), ("iid", iid), ("mid", mid), ("cid", cid), ("num", num))}
    outs = []
    for tower in ("user", "item"):
        buf = torch.full((len(uid), E + pad), -777.0, device="cuda")
        view = buf[:, col0:col0 + E]
        if tower == "user":
            rc = nat.lib().hals_tower_user(s, nat.ptr(d["uid"]), len(uid), nat.ptr(view), buf.stride(0),
                                           nat.current_stream())
        else:
            rc = nat.lib().hals_tower_item(s, nat.ptr(d["iid"]), nat.ptr(d["mid"]), nat.ptr(d["cid"]), nat.ptr(d["num"]),
                                           len(iid), nat.ptr(view), buf.stride(0), nat.current_stream())
        nat.check(rc, f"hals_tower_{tower}")
        b = buf.cpu().numpy()
        outside = np.ones(E + pad, bool)
        outside[col0:col0 + E] = False
        assert (b[:, outside] == -777.0).all(), f"{tower} tower wrote outside its columns"
        outs.append(b[:, col0:col0 + E])
    return outs


@pytest.mark.parametrize("E,dims,col0,pad", [(1, (8, 8, 16), 0, 0), (16, (8, 8, 16), 0, 0), (31, (8, 8, 16), 2, 5),
                                             (32, (8, 8, 16), 0, 0), (33, (8, 8, 16), 3, 4), (50, (8, 8, 16), 0, 0),
                                             (63, (8, 8, 16), 1, 1), (64, (8, 8, 16), 0, 0),
                                             (33, (4, 12, 32), 0, 0), (64, (4, 12, 32), 5, 7),
                                             (20, (1, 1, 1), 0, 0), (50, (1, 1, 1), 3, 3)])
def test_towers_match_oracle(E, dims, col0, pad):
    _, nat, TowerParams = _pkg()
    MD, CD, H = dims
    w = make_weights(E, MD, CD, H, seed=E * 100 + MD)
    rng = np.random.default_rng(E)
    n = N_ROWS
    uid, iid = ids_with_strays(rng, TABLES["user"], n), ids_with_strays(rng, TABLES["item"], n)
    mid, cid = ids_with_strays(rng, TABLES["manu"], n), ids_with_strays(rng, TABLES["cat"], n)
    num = np.stack([rng.uniform(2, 250, n), rng.uniform(1, 5, n)], 1).astype(np.float32)
    got_u, got_i = run_towers(nat, TowerParams, w, uid, iid, mid, cid, num, col0, pad)
    wz = with_zero_rows(w)
    want_u = towers_oracle.user_tower(wz, oracle_ids(uid, TABLES["user"]))
    scaled = towers_oracle.scale_numeric(num, SCALER.scale_, SCALER.min_)
    want_i = towers_oracle.item_tower(wz, oracle_ids(iid, TABLES["item"]), oracle_ids(mid, TABLES["manu"]),
                                      oracle_ids(cid, TABLES["cat"]), scaled)
    assert np.abs(got_u - want_u).max() <= TOL
    assert np.abs(got_i - want_i).max() <= TOL
    stray = (uid < 0) | (uid >= TABLES["user"])
    assert np.array_equal(got_u[stray], np.broadcast_to(w["user_ln_b"], got_u[stray].shape))


@pytest.mark.parametrize("E", [16, 33, 64])
def test_predict_for_user_matches_oracle(E):
    """TwoTowerModel(embedding_size=E).predict_for_user: both towers plus hals_score_one_user at v_stride = E."""
    pkg, nat, TowerParams = _pkg()
    w = make_weights(E, 8, 8, 16, seed=E)
    m = pkg.TwoTowerModel(TABLES["user"], TABLES["item"], TABLES["manu"], TABLES["cat"], embedding_size=E)
    m.model = TowerParams.from_numpy(w, torch.device("cuda"))
    m.scaler = SCALER
    rng = np.random.default_rng(E + 1)
    n = 3000
    df = pd.DataFrame({"itemId": rng.integers(0, TABLES["item"], n), "manufacturer_id": rng.integers(0, TABLES["manu"], n),
                       "category_id": rng.integers(0, TABLES["cat"], n), "price": rng.uniform(2, 250, n),
                       "average_review_rating": rng.uniform(1, 5, n)})
    preds = m.predict_for_user(123, df)
    num = df[["price", "average_review_rating"]].values
    iv = towers_oracle.item_tower(w, df["itemId"].values, df["manufacturer_id"].values, df["category_id"].values,
                                  towers_oracle.scale_numeric(num, SCALER.scale_, SCALER.min_))
    want = towers_oracle.score(towers_oracle.user_tower(w, [123])[0], iv)
    assert [p[0] for p in preds] == list(df["itemId"])
    assert np.allclose([p[1] for p in preds], want, atol=1e-4)
