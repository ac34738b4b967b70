"""TwoTowerModel -- drop-in for the reference's src/two_tower_model.py (class at :17-167).

Same constructor, attributes and method names.  The forward pass that the reference runs
through Keras `Model.predict` (two_tower_model.py:145) is evaluated by the tower kernels of
libhals_b200.so: hals_tower_item / hals_tower_user precompute the tower outputs once per id
(the reference recomputes the item tower for every user) and hals_score_one_user takes the
dot products.  `self.model` is a TowerWeights holder instead of a keras.Model.

Training (two_tower_model.py:91-121) runs on the GPU as well: `train` drives the fused training step and the
multi-tensor Adam step of csrc/tower_train.cu (hals_tower_train_step / hals_tower_adam_step) behind the reference's
signature.  The torch loop it replaced is kept as the test oracle, oracle/tower_train_oracle.py:train_reference.
"""
from __future__ import annotations

import os
import pickle

import numpy as np
from sklearn.preprocessing import MinMaxScaler

LN_EPS = 1e-3  # Keras LayerNormalization default epsilon


class TowerParams:
    """Weights of the graph built at two_tower_model.py:38-89, as fp32 device tensors."""
    NAMES = ("user_emb", "item_emb", "manu_emb", "cat_emb", "num_w", "num_b", "out_w", "out_b",
             "user_ln_g", "user_ln_b", "item_ln_g", "item_ln_b")

    def __init__(self, tensors: dict, embedding_size: int):
        self.t = tensors
        self.embedding_size = int(embedding_size)

    @classmethod
    def keras_init(cls, num_users, num_items, num_manufacturers, num_categories, embedding_size, device, seed=0):
        """Keras default initialisers: Embedding U(-0.05,0.05); Dense Glorot-uniform, zero bias;
        LayerNormalization gamma=1, beta=0."""
        import torch
        g = torch.Generator(device="cpu").manual_seed(seed)
        E = embedding_size

        def emb(n, d):
            return (torch.rand((n, d), generator=g) * 0.1 - 0.05)

        def glorot(i, o):
            lim = (6.0 / (i + o)) ** 0.5
            return (torch.rand((i, o), generator=g) * 2 - 1) * lim

        t = {
            "user_emb": emb(num_users, E), "item_emb": emb(num_items, E),
            "manu_emb": emb(num_manufacturers, 8), "cat_emb": emb(num_categories, 8),
            "num_w": glorot(2, 16), "num_b": torch.zeros(16),
            "out_w": glorot(E + 8 + 8 + 16, E), "out_b": torch.zeros(E),
            "user_ln_g": torch.ones(E), "user_ln_b": torch.zeros(E),
            "item_ln_g": torch.ones(E), "item_ln_b": torch.zeros(E),
        }
        return cls({k: v.float().contiguous().to(device) for k, v in t.items()}, E)

    @classmethod
    def from_numpy(cls, arrays: dict, device):
        import torch
        t = {k: torch.from_numpy(np.ascontiguousarray(arrays[k], dtype=np.float32)).to(device) for k in cls.NAMES}
        return cls(t, t["user_emb"].shape[1])

    def to_numpy(self):
        return {k: v.detach().cpu().numpy() for k, v in self.t.items()}

    def struct(self, scaler):
        from . import _native as nat
        w = nat.TowerWeights()
        w.embedding_size = self.embedding_size
        w.manu_dim = int(self.t["manu_emb"].shape[1])
        w.cat_dim = int(self.t["cat_emb"].shape[1])
        w.num_hidden = int(self.t["num_b"].shape[0])
        for k in self.NAMES:
            setattr(w, k, self.t[k].data_ptr())
        w.ln_eps = LN_EPS
        if scaler is not None and hasattr(scaler, "scale_"):
            sc, mn = scaler.scale_, scaler.min_
        else:
            sc, mn = (1.0, 1.0), (0.0, 0.0)
        w.num_scale[0], w.num_scale[1] = float(sc[0]), float(sc[1])
        w.num_offset[0], w.num_offset[1] = float(mn[0]), float(mn[1])
        # table sizes: ids outside a table get a zero embedding in the kernels instead of an out-of-bounds read
        w.num_users, w.num_items = int(self.t["user_emb"].shape[0]), int(self.t["item_emb"].shape[0])
        w.num_manufacturers, w.num_categories = int(self.t["manu_emb"].shape[0]), int(self.t["cat_emb"].shape[0])
        return w


TRAIN_IDS = (("userId", "user_emb"), ("itemId", "item_emb"), ("manufacturer_id", "manu_emb"),
             ("category_id", "cat_emb"))


def nat_params(p: TowerParams):
    """struct hals_tower_params over the tensors of `p` (the training step and Adam mutate them in place)."""
    from . import _native as nat
    s = nat.TowerParams()
    s.embedding_size = p.embedding_size
    s.manu_dim, s.cat_dim = int(p.t["manu_emb"].shape[1]), int(p.t["cat_emb"].shape[1])
    s.num_hidden = int(p.t["num_b"].shape[0])
    for k in TowerParams.NAMES:
        setattr(s, k, p.t[k].data_ptr())
    s.ln_eps = LN_EPS
    s.num_users, s.num_items = int(p.t["user_emb"].shape[0]), int(p.t["item_emb"].shape[0])
    s.num_manufacturers, s.num_categories = int(p.t["manu_emb"].shape[0]), int(p.t["cat_emb"].shape[0])
    return s


class TwoTowerModel:
    """
    Two-Tower Model Architecture (reference docstring, two_tower_model.py:18-23)
    - User Tower: userId embedding
    - Item Tower: itemId + manufacturer + category + numeric features
    - Dot product similarity with layer normalization
    """

    def __init__(self, num_users, num_items, num_manufacturers, num_categories,
                 embedding_size=50, learning_rate=0.001):
        self.num_users = num_users
        self.num_items = num_items
        self.num_manufacturers = num_manufacturers
        self.num_categories = num_categories
        self.embedding_size = embedding_size
        self.learning_rate = learning_rate
        self.model = None
        self.scaler = MinMaxScaler()
        self.is_trained = False

    # -- graph --------------------------------------------------------------------------------
    def build_model(self, seed=0):
        import torch
        from . import _native as nat
        nat.lib()
        nat.require_cuda()
        self.model = TowerParams.keras_init(self.num_users, self.num_items, self.num_manufacturers,
                                            self.num_categories, self.embedding_size, torch.device("cuda"), seed)
        return self.model

    def _prepare_features(self, data):
        """Feature preprocessing (two_tower_model.py:123-134); the scaler is re-fitted here, as in
        the reference (`fit_transform`, :133)."""
        if data is None:
            return None
        return {
            "user_in": data["userId"].values,
            "item_id_in": data["itemId"].values,
            "manufacturer_in": data["manufacturer_id"].values,
            "category_in": data["category_id"].values,
            "numeric_in": self.scaler.fit_transform(data[["price", "average_review_rating"]]),
        }

    # -- forward (the hot path) -----------------------------------------------------------------
    def item_vectors(self, item_features, out=None):
        """Item tower outputs [n, E] (device) for the rows of a DataFrame with the columns
        itemId, manufacturer_id, category_id, price, average_review_rating."""
        import torch
        from . import _native as nat
        dev = self.model.t["item_emb"].device
        n = len(item_features)

        def col(name):
            return torch.from_numpy(np.ascontiguousarray(item_features[name].values, dtype=np.int32)).to(dev)

        ids, manu, cat = col("itemId"), col("manufacturer_id"), col("category_id")
        num = torch.from_numpy(np.ascontiguousarray(
            item_features[["price", "average_review_rating"]].values, dtype=np.float32)).to(dev)
        if out is None:
            out = torch.empty((n, self.embedding_size), dtype=torch.float32, device=dev)
        w = self.model.struct(self.scaler)
        nat.check(nat.lib().hals_tower_item(w, nat.ptr(ids), nat.ptr(manu), nat.ptr(cat), nat.ptr(num), n,
                                            nat.ptr(out), out.stride(0), nat.current_stream()), "hals_tower_item")
        return out

    def user_vectors(self, user_ids, out=None):
        import torch
        from . import _native as nat
        dev = self.model.t["user_emb"].device
        ids = torch.from_numpy(np.ascontiguousarray(np.asarray(user_ids), dtype=np.int32)).to(dev)
        if out is None:
            out = torch.empty((ids.numel(), self.embedding_size), dtype=torch.float32, device=dev)
        w = self.model.struct(self.scaler)
        nat.check(nat.lib().hals_tower_user(w, nat.ptr(ids), ids.numel(), nat.ptr(out), out.stride(0),
                                            nat.current_stream()), "hals_tower_user")
        return out

    def predict_for_user(self, user_id, item_features):
        """Scores of one user against every row of `item_features` (two_tower_model.py:136-146)."""
        import torch
        from . import _native as nat
        iv = self.item_vectors(item_features)
        uv = self.user_vectors([user_id])
        out = torch.empty(iv.shape[0], dtype=torch.float32, device=iv.device)
        nat.check(nat.lib().hals_score_one_user(nat.ptr(uv), nat.ptr(iv), iv.stride(0), self.embedding_size, None,
                                                iv.shape[0], nat.ptr(out), nat.current_stream()),
                  "hals_score_one_user")
        predictions = out.cpu().numpy()
        return list(zip(item_features["itemId"], predictions.flatten()))

    # -- training (csrc/tower_train.cu) -----------------------------------------------------------------
    def train(self, train_data, val_data=None, batch_size=256, epochs=10):
        """Adam(lr, eps=1e-7) on MSE with EarlyStopping(patience=3, restore_best_weights) when validation data is
        given (two_tower_model.py:91-121).  Returns a dict of per-epoch losses.

        Every step runs on the GPU: hals_tower_train_step (fused forward and backward of the batch) and
        hals_tower_adam_step (one Adam step over every parameter, dense moments).  Per epoch the host draws the
        permutation (torch.randperm, seeded 0), uploads it once and reads the per-step losses and the validation loss
        once; there is no host synchronisation per step.  Steps are bitwise reproducible.  The validation loss runs
        the tower kernels on the pre-scaled features and reduces in fp64.

        Supported widths are those of the tower kernels: embedding_size in [1, 64] (ValueError otherwise, before any
        device work; predict_for_user and item_vectors reject wider models too), and manufacturer / category / hidden
        widths whose training step fits in shared memory (the reference widths 8 / 8 / 16 at E = 50 use 38 KB of 200 KB)."""
        import torch
        from . import _native as nat
        E = int(self.model.embedding_size if self.model is not None else self.embedding_size)
        if not 1 <= E <= 64:
            raise ValueError(f"embedding_size must be in [1, 64] for the GPU trainer (got {E})")
        if self.model is None:
            self.build_model()
        dev = self.model.t["user_emb"].device
        has_val = val_data is not None and len(val_data) > 0
        # Embedding ids are table rows (two_tower_model.py:47-62).  Keras on the CPU raises InvalidArgumentError for a
        # TRAINING id outside its table: checked here on the host.  (Validation rows may name users / items the tables
        # do not have -- the reference's own hyperparameter_tuning holds out whole users -- they read as zero rows.)
        for col, table in TRAIN_IDS:
            ids = train_data[col].values
            n_rows = int(self.model.t[table].shape[0])
            if len(ids) and (ids.min() < 0 or ids.max() >= n_rows):
                raise IndexError(f"{col}: ids must lie in [0, {n_rows}) (found {int(ids.min())}..{int(ids.max())})")
        n = len(train_data)
        starts = range(0, n, batch_size)   # TypeError / ValueError for a batch size range() rejects, as before
        tf = self._prepare_features(train_data)
        vf = self._prepare_features(val_data) if has_val else None
        if has_val:  # _prepare_features re-fits the scaler (reference behaviour); keep the train fit for predict
            tf = self._prepare_features(train_data)

        def ids32(a):  # ids beyond int32 stay outside every table
            return torch.from_numpy(np.clip(np.asarray(a, dtype=np.int64), -1, 2 ** 31 - 1).astype(np.int32)).to(dev)

        def floats(a):
            return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)

        feats = [ids32(tf[k]) for k in ("user_in", "item_id_in", "manufacturer_in", "category_in")]
        num, y = floats(tf["numeric_in"]), floats(train_data["average_review_rating"].values)
        rows = [int(self.model.t[t].shape[0]) for _, t in TRAIN_IDS]
        params = TowerParams({k: v.detach().clone().contiguous() for k, v in self.model.t.items()}, E)
        moments = [TowerParams({k: torch.zeros_like(v) for k, v in params.t.items()}, E) for _ in range(2)]
        P, M, V = (nat_params(x) for x in (params, *moments))
        L = nat.lib()
        stream = nat.current_stream()
        ws_bytes = int(L.hals_tower_train_workspace_bytes(P, max(1, min(batch_size, n)) if len(starts) else 1))
        ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=dev)
        losses = torch.empty(max(len(starts), 1), dtype=torch.float32, device=dev)
        if has_val:
            nv = len(val_data)
            vw = params.struct(None)      # identity scaler: the validation numerics are scaled on the host
            v_ids = [ids32(vf[k]) for k in ("user_in", "item_id_in", "manufacturer_in", "category_in")]
            v_num, v_y = floats(vf["numeric_in"]), floats(val_data["average_review_rating"].values)
            v_rows = torch.arange(nv, dtype=torch.int32, device=dev)
            uv, iv = (torch.empty((nv, E), dtype=torch.float32, device=dev) for _ in range(2))
            sse, cnt = torch.empty(1, dtype=torch.float64, device=dev), torch.empty(1, dtype=torch.int64, device=dev)
            sse_ws = torch.empty(int(L.hals_als_sse_workspace_bytes()), dtype=torch.uint8, device=dev)
            best_t = {k: torch.empty_like(v) for k, v in params.t.items()}
        batch = nat.TowerBatch()
        history = {"loss": [], "val_loss": []}
        best, have_best, bad, t = float("inf"), False, 0, 0
        g = torch.Generator(device="cpu").manual_seed(0)
        for _ in range(int(epochs)):
            perm = torch.randperm(n, generator=g).to(dev)
            if len(starts):
                ep_ids = [f[perm] for f in feats]
                ep_num, ep_y = num[perm].contiguous(), y[perm]
                # each batch's ids sorted stably (key: batch index, then id): the order the Adam step sums rows in
                b_of = torch.arange(n, device=dev) // batch_size
                orders = [(torch.sort(b_of * r + e.long(), stable=True).indices - b_of * batch_size).to(torch.int32)
                          for e, r in zip(ep_ids, rows)]
                for si, s in enumerate(starts):
                    t += 1
                    batch.n = min(batch_size, n - s)
                    batch.user_ids, batch.item_ids, batch.manufacturer_ids, batch.category_ids = (
                        a.data_ptr() + 4 * s for a in ep_ids)
                    batch.numeric, batch.labels = ep_num.data_ptr() + 8 * s, ep_y.data_ptr() + 4 * s
                    batch.order_user, batch.order_item, batch.order_manufacturer, batch.order_category = (
                        a.data_ptr() + 4 * s for a in orders)
                    nat.check(L.hals_tower_train_step(P, batch, t, nat.ptr(ws), ws_bytes,
                                                      losses.data_ptr() + 4 * si, stream), "hals_tower_train_step")
                    nat.check(L.hals_tower_adam_step(P, M, V, batch, t, nat.ptr(ws), ws_bytes, self.learning_rate,
                                                     0.9, 0.999, 1e-7, stream), "hals_tower_adam_step")
            if has_val:
                nat.check(L.hals_tower_user(vw, nat.ptr(v_ids[0]), nv, nat.ptr(uv), E, stream), "hals_tower_user")
                nat.check(L.hals_tower_item(vw, nat.ptr(v_ids[1]), nat.ptr(v_ids[2]), nat.ptr(v_ids[3]), nat.ptr(v_num),
                                            nv, nat.ptr(iv), E, stream), "hals_tower_item")
                nat.check(L.hals_als_sse(nat.ptr(uv), nat.ptr(iv), E, nat.ptr(v_rows), nat.ptr(v_rows), nat.ptr(v_y),
                                         nv, nat.ptr(sse), nat.ptr(cnt), nat.ptr(sse_ws), sse_ws.numel(), stream),
                          "hals_als_sse")
            step_losses = losses[:len(starts)].cpu().numpy()     # the epoch's one read-back
            tot = 0.0
            for s, ls in zip(starts, step_losses):
                tot += float(ls) * min(batch_size, n - s)
            history["loss"].append(tot / max(n, 1))
            if has_val:
                vl = float(sse.item()) / nv
                history["val_loss"].append(vl)
                if vl < best:
                    best, bad, have_best = vl, 0, True
                    for k, v in params.t.items():
                        best_t[k].copy_(v)
                else:
                    bad += 1
                    if bad >= 3:
                        break
        final = best_t if has_val and have_best else params.t
        self.model = TowerParams(final, E)
        self.is_trained = True
        return history

    # -- persistence ------------------------------------------------------------------------------
    def save_model(self, model_path="models/twotower.keras"):
        os.makedirs(os.path.dirname(model_path) or ".", exist_ok=True)
        with open(model_path, "wb") as f:
            np.savez(f, embedding_size=self.embedding_size, **self.model.to_numpy())
        with open(f"{model_path}_scaler.pkl", "wb") as f:
            pickle.dump(self.scaler, f)

    @classmethod
    def load_model(cls, model_path="models/twotower.keras"):
        import torch
        from . import _native as nat
        nat.lib()
        nat.require_cuda()
        try:
            z = np.load(model_path)
            missing = [k for k in TowerParams.NAMES if k not in z.files]
        except Exception as e:       # a Keras v3 archive (what the reference's save_model writes) is a zip of config + h5
            raise ValueError(f"{model_path} is not a tower checkpoint of this package (numpy .npz written by "
                             f"TwoTowerModel.save_model); a Keras archive has to be exported layer by layer, see "
                             f"INTEGRATION.md ({e})") from e
        if missing:
            raise ValueError(f"{model_path}: not a tower checkpoint of this package (missing arrays {missing[:3]}...); "
                             "Keras archives have to be exported layer by layer, see INTEGRATION.md")
        with open(f"{model_path}_scaler.pkl", "rb") as f:
            scaler = pickle.load(f)
        params = TowerParams.from_numpy({k: z[k] for k in TowerParams.NAMES}, torch.device("cuda"))
        loaded_model = cls(params.t["user_emb"].shape[0], params.t["item_emb"].shape[0],
                           params.t["manu_emb"].shape[0], params.t["cat_emb"].shape[0],
                           embedding_size=params.embedding_size)
        loaded_model.model = params
        loaded_model.scaler = scaler
        loaded_model.is_trained = True
        return loaded_model


def hyperparameter_tuning(train_data, param_grid, val_size=0.2, random_state=42):
    """F1@10-based grid search over {batch_size, epochs} (src/two_tower_model.py:169-236): hold out `val_size` of the
    users, train one TwoTowerModel(embedding_size=50, learning_rate=0.001) per grid entry on the rest, score the first 50
    held-out users against the held-out items with predict_for_user (the GPU tower kernels) and keep the entry with the
    best mean F1@10.  Returns the best entry (a copy) or None; an entry that raises is reported and skipped, like the
    reference.  One deviation: the reference passes `random_state` to np.random.choice, which has no such argument (its
    call raises TypeError before anything runs); the held-out users are drawn from np.random.RandomState(random_state)."""
    best_params = None
    best_f1 = 0.0
    train_users = train_data['userId'].unique()
    rng = np.random.RandomState(random_state)
    val_users = rng.choice(train_users, size=int(len(train_users) * val_size), replace=False)
    train_sub = train_data[~train_data['userId'].isin(val_users)]
    val_sub = train_data[train_data['userId'].isin(val_users)]
    num_users = train_sub['userId'].nunique()
    num_items = train_sub['itemId'].nunique()
    num_manufacturers = train_sub['manufacturer_id'].nunique()
    num_categories = train_sub['category_id'].nunique()
    for params in param_grid:
        print(f"\nTesting parameters: {params}")
        try:
            model = TwoTowerModel(num_users=num_users, num_items=num_items, num_manufacturers=num_manufacturers,
                                  num_categories=num_categories, embedding_size=50, learning_rate=0.001)
            model.train(train_sub, val_sub, batch_size=params['batch_size'], epochs=params['epochs'])
            f1_scores = []
            sample_users = val_sub['userId'].unique()[:50]
            items = val_sub[['itemId', 'manufacturer_id', 'category_id', 'price',
                             'average_review_rating']].drop_duplicates()
            for user_id in sample_users:
                rows = val_sub[val_sub['userId'] == user_id]
                actual = dict(zip(rows['itemId'], rows['average_review_rating']))
                preds = model.predict_for_user(user_id, items)
                f1_scores.append(compute_f1_score(actual, dict(preds), k=10))
            avg_f1 = np.mean(f1_scores)
            print(f"  Avg F1@10: {avg_f1:.4f}")
            if avg_f1 > best_f1:
                best_f1 = avg_f1
                best_params = params.copy()
                print(f"  New best F1@10: {best_f1:.4f}")
        except Exception as e:
            print(f"  Error with params {params}: {str(e)}")
            continue
    return best_params


def compute_f1_score(actual, pred, k=10):
    """two_tower_model.py:238-245 (same function as als_model.compute_f1_score)."""
    from .als_model import compute_f1_score as f
    return f(actual, pred, k)
