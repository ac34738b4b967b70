"""ALSModel -- drop-in for the reference's src/als_model.py (class at :21-140).

Same constructor, attributes, method names, return conventions (print + sentinel on error,
als_model.py:64-66,89-91,120-121,134-136).  What changed is what sits behind `train` and
`predict_for_user`: instead of pyspark.ml ALS.fit / ALSModel.transform over Py4J
(als_model.py:52-62,75) the factors are solved and scored by the sm_100a kernels of
libhals_b200.so (csrc/), driven by als_engine.AlsEngine.

Additive (keyword-only) extensions, none of which changes the reference behaviour:
  ALSModel(..., implicit_prefs=False, alpha=1.0, seed=0)   Spark's implicitPrefs / alpha / seed
  ALSModel(..., nonnegative=False)                         Spark's nonnegative: factors >= 0 (NNLS half-steps)
  train(data, init_user_factors=None)                      explicit initial factors for parity runs
  predict_for_users(user_ids, item_ids)                    dense [U,I] block of scores (device)
"""
from __future__ import annotations

import os
import pickle
import warnings

import numpy as np
import pandas as pd

from .data_preprocessing import get_item_features

warnings.filterwarnings("ignore")


class _Backend:
    """Stands where the reference keeps its SparkSession (`self.spark`, als_model.py:28,34-37)."""

    def __init__(self):
        from . import _native as nat
        nat.lib()
        nat.require_cuda()
        self.active = True

    def stop(self):
        self.active = False


class ALSFactors:
    """The fitted model (what pyspark's ALSModel holds): factor tables keyed by raw id."""

    def __init__(self, rank, user_ids, item_ids, user_factors, item_factors, user_present, item_present):
        self.rank = rank
        self.user_ids = np.asarray(user_ids)          # sorted raw ids; row i of the table <-> user_ids[i]
        self.item_ids = np.asarray(item_ids)
        self.user_factors = user_factors              # torch fp32 [U,k] on the device
        self.item_factors = item_factors              # torch fp32 [I,k]
        self.user_present = user_present
        self.item_present = item_present

    def user_row(self, user_id):
        i = int(np.searchsorted(self.user_ids, user_id))
        return i if i < len(self.user_ids) and self.user_ids[i] == user_id else -1

    def item_rows(self, items):
        items = np.asarray(items)
        pos = np.searchsorted(self.item_ids, items)
        pos = np.clip(pos, 0, max(len(self.item_ids) - 1, 0))
        ok = (self.item_ids[pos] == items) if len(self.item_ids) else np.zeros(len(items), bool)
        return np.where(ok, pos, -1)


def read_spark_als_dir(model_path):
    """Factors of a Spark `ALSModel` directory, i.e. what the reference's save_model writes (als_model.py:116-127 ->
    pyspark ALSModel.save): `metadata/part-00000` (one JSON line), `userFactors/*.parquet` and `itemFactors/*.parquet`
    with the columns `id: int` and `features: array<float>`.  Returns (rank, user_ids, user_factors, item_ids,
    item_factors) with ids sorted ascending and factors as fp32 [n, rank].  Pure host code (pyarrow)."""
    import json
    import pyarrow.parquet as pq

    def table(name):
        t = pq.read_table(os.path.join(model_path, name), columns=["id", "features"])
        ids = t["id"].combine_chunks().to_numpy(zero_copy_only=False).astype(np.int64)
        feats = t["features"].combine_chunks()
        flat = feats.flatten().to_numpy(zero_copy_only=False).astype(np.float32)
        if len(ids) == 0:
            return ids, flat.reshape(0, 0)
        k = len(flat) // len(ids)
        if k * len(ids) != len(flat):
            raise ValueError(f"{model_path}/{name}: feature vectors of unequal length")
        order = np.argsort(ids, kind="stable")
        return ids[order], np.ascontiguousarray(flat.reshape(len(ids), k)[order])

    uid, uf = table("userFactors")
    iid, itf = table("itemFactors")
    rank = uf.shape[1] if len(uid) else itf.shape[1]
    meta = os.path.join(model_path, "metadata", "part-00000")
    if os.path.exists(meta):
        with open(meta) as f:
            md = json.loads(f.readline())
        rank_md = md.get("rank", md.get("paramMap", {}).get("rank", rank))
        if int(rank_md) != rank:
            raise ValueError(f"{model_path}: metadata rank {rank_md} != stored feature length {rank}")
    if len(uid) and len(iid) and uf.shape[1] != itf.shape[1]:
        raise ValueError(f"{model_path}: user and item factors have different ranks")
    return int(rank), uid, uf, iid, itf


def _as_item_ids(all_items):
    """The reference hands the same `all_items` to both predictors (hybrid_system.py:101-102)
    although ALS wants ids and the two-tower model wants a DataFrame: accept both."""
    if isinstance(all_items, pd.DataFrame):
        return list(all_items["itemId"].values)
    return list(all_items)


class ALSModel:
    def __init__(self, rank=10, max_iter=10, reg_param=0.1, cold_start_strategy="drop", *,
                 implicit_prefs=False, alpha=1.0, seed=0, nonnegative=False):
        self.rank = rank
        self.max_iter = max_iter
        self.reg_param = reg_param
        self.cold_start_strategy = cold_start_strategy
        self.model = None
        self.spark = None
        self.global_mean = 3.0
        self._item_features = None
        self._train_frame = None
        self._fallback_table = None
        self.implicit_prefs = implicit_prefs
        self.alpha = alpha
        self.seed = seed
        self.nonnegative = nonnegative

    @property
    def item_features(self):
        """itemId -> {'features', 'rating'} (als_model.py:48), built on first use from the training frame."""
        if self._item_features is None and self._train_frame is not None:
            self._item_features = get_item_features(self._train_frame)
        return self._item_features

    @item_features.setter
    def item_features(self, value):
        self._item_features = value
        self._fallback_table = None

    def initialize_spark(self):
        try:
            if self.spark is None or not getattr(self.spark, "active", False):
                self.spark = _Backend()
            return True
        except Exception as e:
            print(f"Spark init error: {str(e)}")
            return False

    def train(self, data, init_user_factors=None):
        try:
            if not self.initialize_spark():
                return False
            import torch
            from .als_engine import AlsEngine

            # The raw columns go to the device as they are; id compaction (what Spark's makeBlocks does with the raw
            # ids, behind als_model.py:62) and the CSR build both run there.  The item-feature table the cold-id
            # fallback needs (als_model.py:48) is derived lazily, on first use.
            self._train_frame = data
            self._item_features = None
            dev = torch.device("cuda")
            uid = torch.from_numpy(np.ascontiguousarray(data["userId"].values)).to(dev)
            iid = torch.from_numpy(np.ascontiguousarray(data["itemId"].values)).to(dev)
            r = torch.from_numpy(np.ascontiguousarray(data["average_review_rating"].values, dtype=np.float32)).to(dev)
            self.global_mean = float(r.double().mean().item())
            user_ids_d, u = torch.unique(uid, sorted=True, return_inverse=True)
            item_ids_d, i = torch.unique(iid, sorted=True, return_inverse=True)
            user_ids, item_ids = user_ids_d.cpu().numpy(), item_ids_d.cpu().numpy()
            eng = AlsEngine(u, i, r, len(user_ids), len(item_ids), self.rank, self.reg_param,
                            implicit=self.implicit_prefs, alpha=self.alpha, nonnegative=self.nonnegative)
            if init_user_factors is not None:
                eng.set_user_factors(init_user_factors)
            else:
                eng.init_user_factors(self.seed)
            eng.fit(self.max_iter)
            torch.cuda.synchronize()
            self.model = ALSFactors(self.rank, user_ids, item_ids, eng.X, eng.Y, eng.user_present, eng.item_present)
            return True
        except Exception as e:
            print(f"Training error: {str(e)}")
            return False

    def predict_for_user(self, user_id, all_items):
        try:
            import torch
            from . import _native as nat
            items = _as_item_ids(all_items)
            m = self.model
            urow = m.user_row(user_id)
            rows = m.item_rows(items) if len(items) else np.zeros(0, np.int64)
            known = rows >= 0
            scores = np.full(len(items), np.nan, dtype=np.float32)
            if urow >= 0 and known.any():
                dev = m.item_factors.device
                ids = torch.from_numpy(rows[known].astype(np.int32)).to(dev)
                out = torch.empty(ids.numel(), dtype=torch.float32, device=dev)
                nat.check(nat.lib().hals_score_one_user(
                    nat.ptr(m.user_factors[urow]), nat.ptr(m.item_factors), m.item_factors.stride(0), m.rank,
                    nat.ptr(ids), ids.numel(), nat.ptr(out), nat.current_stream()), "hals_score_one_user")
                scores[known] = out.cpu().numpy()
            # cold user / cold item: content-similar fallback (als_model.py:82-86), all cold items in one launch
            cold = np.flatnonzero(np.isnan(scores))
            placeholders = self._fallback_scores([items[j] for j in cold]) if len(cold) else []
            final_preds = [(item, float(s)) for item, s in zip(items, scores)]
            for j, ph in zip(cold, placeholders):
                final_preds[j] = (items[j], ph)
            return final_preds
        except Exception as e:
            print(f"Prediction error: {str(e)}")
            return []

    def predict_for_users(self, user_ids, item_ids):
        """Additive batched entry point: [len(user_ids), len(item_ids)] fp32 scores on the device
        (NaN where the user or item is unknown, Spark's coldStartStrategy='nan' view)."""
        import torch
        from . import _native as nat
        m = self.model
        urows = np.array([m.user_row(u) for u in user_ids], dtype=np.int64)
        irows = m.item_rows(item_ids)
        dev = m.item_factors.device
        uu = torch.from_numpy(np.repeat(np.maximum(urows, 0), len(irows)).astype(np.int32)).to(dev)
        ii = torch.from_numpy(np.tile(np.maximum(irows, 0), len(urows)).astype(np.int32)).to(dev)
        out = torch.empty(uu.numel(), dtype=torch.float32, device=dev)
        nat.check(nat.lib().hals_als_predict(nat.ptr(m.user_factors), nat.ptr(m.item_factors), m.rank, nat.ptr(uu),
                                             nat.ptr(ii), uu.numel(), None, None, nat.ptr(out),
                                             nat.current_stream()), "hals_als_predict")
        out = out.view(len(urows), len(irows))
        bad = torch.from_numpy((urows < 0)[:, None] | (irows < 0)[None, :]).to(dev)
        return out.masked_fill(bad, float("nan"))

    def _fallback_scores(self, items):
        """Placeholder rating of every item in `items` (als_model.py:83-86): mean rating of its <= 3 cosine neighbours
        with similarity > 0.5, else the global mean -- hals_similar_items, one warp per item."""
        import torch
        from . import _native as nat
        feats = self.item_features or {}
        if self._fallback_table is None:
            ids = list(feats.keys())
            F = np.asarray([feats[i]["features"] for i in ids], dtype=np.float64).reshape(len(ids), -1)
            R = np.asarray([feats[i]["rating"] for i in ids], dtype=np.float64)
            dev = torch.device("cuda")
            self._fallback_table = ({item: n for n, item in enumerate(ids)}, torch.from_numpy(np.ascontiguousarray(F)).to(dev),
                                    torch.from_numpy(R).to(dev))
        pos, F, R = self._fallback_table
        if F.shape[0] == 0 or F.shape[1] > 8:
            return [self.global_mean] * len(items) if F.shape[0] == 0 else [
                (np.mean([feats[s]["rating"] for s in self._find_similar_items(it)]) if self._find_similar_items(it)
                 else self.global_mean) for it in items]
        q = torch.tensor([pos.get(it, -1) for it in items], dtype=torch.int32, device=F.device)
        out = torch.empty(len(items), dtype=torch.float64, device=F.device)
        nat.check(nat.lib().hals_similar_items(nat.ptr(F), int(F.shape[1]), nat.ptr(R), int(F.shape[0]), nat.ptr(q), len(items),
                                               float(self.global_mean), nat.ptr(out), None, nat.current_stream()),
                  "hals_similar_items")
        return out.cpu().numpy().tolist()

    def _find_similar_items(self, item_id, k=3):
        """Top-k cosine-similar items with similarity > 0.5 (als_model.py:93-104), vectorised."""
        try:
            target = self.item_features[item_id]
            ids = [i for i in self.item_features if i != item_id]
            if not ids:
                return []
            F = np.asarray([self.item_features[i]["features"] for i in ids], dtype=np.float64)
            t = np.asarray(target["features"], dtype=np.float64)
            denom = np.linalg.norm(F, axis=1) * np.linalg.norm(t)
            sim = np.divide(F @ t, denom, out=np.zeros(len(ids)), where=denom > 0)
            order = np.argsort(-sim, kind="stable")[:k]
            return [ids[j] for j in order if sim[j] > 0.5]
        except (KeyError, TypeError):
            return []

    def save_model(self, model_path="models/als"):
        try:
            os.makedirs(os.path.dirname(model_path) or ".", exist_ok=True)
            m = self.model
            np.savez(f"{model_path}.npz", rank=m.rank, user_ids=m.user_ids, item_ids=m.item_ids,
                     user_factors=m.user_factors.cpu().numpy(), item_factors=m.item_factors.cpu().numpy(),
                     user_present=m.user_present.cpu().numpy(), item_present=m.item_present.cpu().numpy())
            metadata = {
                "rank": self.rank,
                "max_iter": self.max_iter,
                "reg_param": self.reg_param,
                "global_mean": self.global_mean,
                "item_features": self.item_features,
            }
            with open(f"{model_path}_metadata.pkl", "wb") as f:
                pickle.dump(metadata, f)
            print(f"Model saved to {model_path}")
        except Exception as e:
            print(f"Saving error: {str(e)}")

    def load_model(self, model_path="models/als"):
        try:
            import torch
            if not self.initialize_spark():
                return None
            dev = torch.device("cuda")
            if os.path.isdir(model_path) and not os.path.exists(f"{model_path}.npz"):
                # a model trained and saved by the reference: a Spark ALSModel directory next to the same metadata pickle
                rank, uid, uf, iid, itf = read_spark_als_dir(model_path)
                self.model = ALSFactors(rank, uid, iid, torch.from_numpy(uf).to(dev), torch.from_numpy(itf).to(dev),
                                        torch.ones(len(uid), dtype=torch.bool, device=dev),
                                        torch.ones(len(iid), dtype=torch.bool, device=dev))
            else:
                z = np.load(f"{model_path}.npz")
                self.model = ALSFactors(int(z["rank"]), z["user_ids"], z["item_ids"],
                                        torch.from_numpy(z["user_factors"]).to(dev),
                                        torch.from_numpy(z["item_factors"]).to(dev),
                                        torch.from_numpy(z["user_present"]).to(dev),
                                        torch.from_numpy(z["item_present"]).to(dev))
            with open(f"{model_path}_metadata.pkl", "rb") as f:
                metadata = pickle.load(f)
                self.rank = metadata["rank"]
                self.max_iter = metadata["max_iter"]
                self.reg_param = metadata["reg_param"]
                self.global_mean = metadata["global_mean"]
                self.item_features = metadata["item_features"]
            return self
        except Exception as e:
            print(f"Loading error: {str(e)}")
            return None

    def stop_spark(self):
        if self.spark:
            self.spark.stop()


def hyperparameter_tuning(train_data, val_data, param_grid):
    """F1 grid search, as als_model.py:142-169."""
    best_params = None
    best_f1 = 0.0
    for params in param_grid:
        model = ALSModel(**params)
        if not model.train(train_data):
            continue
        f1_scores = []
        for user_id in val_data["userId"].sample(min(50, len(val_data))).unique():
            sel = val_data[val_data["userId"] == user_id]
            actual = dict(zip(sel["itemId"], sel["average_review_rating"]))
            preds = model.predict_for_user(user_id, val_data["itemId"].unique())
            f1_scores.append(compute_f1_score(actual, {item: score for item, score in preds}))
        avg_f1 = np.mean(f1_scores)
        if avg_f1 > best_f1:
            best_f1 = avg_f1
            best_params = params.copy()
        model.stop_spark()
    return best_params


def compute_f1_score(actual, pred, k=10):
    """F1@k of the top-k predicted ids against the rated ids (als_model.py:171-177)."""
    actual_items = set(actual.keys())
    ranked = sorted(pred.items(), key=lambda x: x[1], reverse=True)[:k]
    pred_items = set(item for item, _ in ranked)
    tp = len(actual_items & pred_items)
    precision = tp / k
    recall = tp / len(actual_items) if actual_items else 0
    return 2 * (precision * recall) / (precision + recall) if (precision + recall) > 0 else 0
