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
  recommend_for_all_users(num_items, *, exclude=None, as_arrays=False)            Spark's recommendForAllUsers
  recommend_for_all_items(num_users, *, exclude=None, as_arrays=False)            Spark's recommendForAllItems
  recommend_for_user_subset(dataset, num_items, *, exclude=None, as_arrays=False) Spark's recommendForUserSubset
  recommend_for_item_subset(dataset, num_users, *, exclude=None, as_arrays=False) Spark's recommendForItemSubset
  transform(dataset)                                       Spark's transform, honouring cold_start_strategy
  evaluate_regression(dataset, metric_name="rmse")         RegressionEvaluator on transform(dataset)
  evaluate_ranking(dataset, k=10, *, exclude=None)         RankingEvaluator on recommendForAllUsers(k) (hals_ranking_metrics)
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
        return _rows_of(self.item_ids, items)


def _rows_of(sorted_ids, ids):
    """Row of each id in a sorted id table, -1 where it is absent."""
    ids = np.asarray(ids)
    pos = np.searchsorted(sorted_ids, ids)
    pos = np.clip(pos, 0, max(len(sorted_ids) - 1, 0))
    ok = (sorted_ids[pos] == ids) if len(sorted_ids) else np.zeros(len(ids), bool)
    return np.where(ok, pos, -1)


def _on(values, dev, dtype=np.int64):
    """Host values (numpy / pandas column) as a contiguous torch tensor of `dtype` on `dev`."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(np.asarray(values, dtype=dtype))).to(dev)


MAX_RECOMMENDATIONS = 256   # longest list recommend_for_* returns (the top-k limit of hals_score_topk; Spark has none)


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

    # -- Spark's ALSModel.recommendFor* (additive) ------------------------------------------------------------------
    # rating = the fp32 dot product of the two factor rows (it agrees with predict_for_users to fp32 rounding; the
    # summation orders differ).  A list is ordered by rating descending, then ascending raw id (Spark leaves the order
    # of ties unspecified), and is min(num, candidates) long.  Only rows whose user_present / item_present is set take
    # part, as queries or as candidates.  num must be an int in [1, MAX_RECOMMENDATIONS].
    # exclude: optional DataFrame of userId / itemId pairs (e.g. the training frame): each list leaves its pairs out
    # and fills up with the next best (the item direction applies the same pairs transposed); a kept rating is the
    # one it has without `exclude`.
    # Returns a pandas DataFrame, one row per query id in ascending order: (<query id column>, recommendations = list
    # of (id, rating)); as_arrays=True returns numpy (query_ids int64 [Q], rec_ids int64 [Q, num] (-1 padded),
    # ratings float32 [Q, num] (-inf padded)) instead -- a frame of 1e6 x 100 tuples costs more on the host than the
    # GPU work.

    def recommend_for_all_users(self, num_items, *, exclude=None, as_arrays=False):
        """Top num_items items of every user: Spark's recommendForAllUsers (see the notes above)."""
        return self._recommend(True, None, num_items, exclude, as_arrays)

    def recommend_for_all_items(self, num_users, *, exclude=None, as_arrays=False):
        """Top num_users users of every item: Spark's recommendForAllItems."""
        return self._recommend(False, None, num_users, exclude, as_arrays)

    def recommend_for_user_subset(self, dataset, num_items, *, exclude=None, as_arrays=False):
        """recommend_for_all_users for the distinct dataset["userId"] known to the model (unknown ids are dropped, as
        in Spark's inner join): Spark's recommendForUserSubset."""
        return self._recommend(True, dataset["userId"].values, num_items, exclude, as_arrays)

    def recommend_for_item_subset(self, dataset, num_users, *, exclude=None, as_arrays=False):
        """recommend_for_all_items for the distinct dataset["itemId"] known to the model: Spark's recommendForItemSubset."""
        return self._recommend(False, dataset["itemId"].values, num_users, exclude, as_arrays)

    def _recommend(self, for_users, subset, num, exclude, as_arrays, slab=65536):
        q_col = "userId" if for_users else "itemId"
        query_ids, cand_ids, slabs = self._topk_slabs(for_users, subset, num, exclude, slab)
        rec = np.full((len(query_ids), num), -1, np.int64)
        ratings = np.full((len(query_ids), num), -np.inf, np.float32)
        for u0, u1, idx, s in slabs:
            idx = idx.cpu().numpy()
            rec[u0:u1] = np.where(idx >= 0, cand_ids[np.maximum(idx, 0)], -1)
            ratings[u0:u1] = s.cpu().numpy()
        if as_arrays:
            return query_ids, rec, ratings
        lens = (rec >= 0).sum(1)
        lists = [list(zip(r[:n].tolist(), s[:n].tolist())) for r, s, n in zip(rec, ratings, lens)]
        return pd.DataFrame({q_col: query_ids, "recommendations": pd.Series(lists, dtype=object)})

    def _topk_slabs(self, for_users, subset, num, exclude, slab):
        """What recommend_for_* and evaluate_ranking share: check num and the model, select the query rows (present;
        the distinct known ids of `subset` when it is given) and the candidate rows (present).  Returns (query raw ids
        int64 [n_q] ascending, candidate raw ids [n_c] ascending, slabs); iterating `slabs` runs the top-k slab by slab
        and yields (u0, u1, idx, scores): device tensors [u1-u0, num] of candidate positions (-1 padded) and fp32
        ratings (-inf padded) of query rows [u0, u1)."""
        self._check_topk(num)
        import torch
        from .scoring import HybridScorer, exclusion_lists_by_id
        m, num = self.model, int(num)
        q_col, c_col = ("userId", "itemId") if for_users else ("itemId", "userId")
        q_ids, q_fac, q_present = (m.user_ids, m.user_factors, m.user_present) if for_users else \
            (m.item_ids, m.item_factors, m.item_present)
        c_ids, c_fac, c_present = (m.item_ids, m.item_factors, m.item_present) if for_users else \
            (m.user_ids, m.user_factors, m.user_present)
        q_ok = q_present.cpu().numpy()
        if subset is None:
            q_rows = np.flatnonzero(q_ok)
        else:
            q_rows = _rows_of(q_ids, np.unique(np.asarray(subset)))
            q_rows = q_rows[q_rows >= 0]
            q_rows = q_rows[q_ok[q_rows]]
        c_rows = np.flatnonzero(c_present.cpu().numpy())
        dev = c_fac.device

        def take(fac, rows):      # the whole table when every row takes part (no copy)
            return fac if len(rows) == fac.shape[0] else fac[torch.from_numpy(rows).to(dev)]

        def slabs():
            n_q, n_c = len(q_rows), len(c_rows)
            if not (n_q and n_c):
                return
            sc = HybridScorer(take(q_fac, q_rows), take(c_fac, c_rows), None, None)
            excl = None
            if exclude is not None:
                excl = exclusion_lists_by_id(_on(q_ids[q_rows], dev), _on(c_ids[c_rows], dev),
                                             _on(exclude[q_col].values, dev), _on(exclude[c_col].values, dev))
            for u0 in range(0, n_q, slab):      # one scorer (candidates, workspace) for every slab of queries
                u1 = min(n_q, u0 + slab)
                yield (u0, u1, *sc.topk_dot(num, u0, u1, exclude=excl))

        return np.asarray(q_ids[q_rows], np.int64), c_ids[c_rows], slabs()

    # -- Spark's ALSModel.transform, RegressionEvaluator and RankingEvaluator (additive) --------------------------------

    def transform(self, dataset):
        """Spark's ALSModel.transform: a copy of `dataset` with a float32 "prediction" column, the fp32 dot product of
        the user's and the item's factors (hals_als_predict), NaN where the user or the item is unknown or not present.
        cold_start_strategy "drop" (the default) removes the NaN rows and keeps the index of the others; "nan" keeps
        them.  Any other strategy raises ValueError."""
        pred = self._predict_frame(dataset).cpu().numpy()
        out = dataset.copy()
        out["prediction"] = pred
        return out[~np.isnan(pred)] if self._drop_cold() else out

    def evaluate_regression(self, dataset, metric_name="rmse"):
        """Spark's RegressionEvaluator(metricName=...).evaluate(model.transform(dataset)), label column
        "average_review_rating": "rmse", "mse", "mae" or "r2" (1 - SS_res / SS_tot).  Sums in fp64 on the device.
        NaN when a NaN prediction remains (cold_start_strategy "nan") or when no row is left."""
        if metric_name not in ("rmse", "mse", "mae", "r2"):
            raise ValueError(f"metric_name must be one of 'rmse', 'mse', 'mae', 'r2', got {metric_name!r}")
        import torch
        p = self._predict_frame(dataset)
        y = _on(dataset["average_review_rating"].values, p.device, np.float64)
        p = p.double()
        if self._drop_cold():
            keep = ~torch.isnan(p)
            p, y = p[keep], y[keep]
        if p.numel() == 0:
            return float("nan")
        err = y - p
        if metric_name == "mae":
            v = err.abs().mean()
        elif metric_name == "r2":
            v = 1.0 - (err * err).sum() / ((y - y.mean()) ** 2).sum()
        else:
            v = (err * err).mean()
            v = v.sqrt() if metric_name == "rmse" else v
        return float(v.item())

    def evaluate_ranking(self, dataset, k=10, *, exclude=None):
        """recommendForAllUsers(k) joined with `dataset`'s (userId, itemId) pairs as each user's relevant items, then
        Spark's RankingEvaluator: a dict of the means over the users of precisionAtK, recallAtK, ndcgAtK,
        meanAveragePrecisionAtK and meanAveragePrecision (see hals_ranking_metrics), plus numUsers (the users
        evaluated) and numColdUsers (distinct users of `dataset` that are unknown or not present: like Spark's inner
        join, they are not in the means).  Every pair counts as relevant; a rating threshold is the caller's filter on
        `dataset`.  A relevant item the model cannot recommend still counts in the user's label set.
        k: an int in [1, MAX_RECOMMENDATIONS]; exclude: as for recommend_for_all_users (e.g. the training frame).
        The lists and per-user metrics stay on the device and are reduced once; of the results only the five means come
        back.  The id joins (test users, label and exclusion lists) still synchronise with the host for their sizes."""
        return self._evaluate_ranking(dataset, k, exclude)

    def _evaluate_ranking(self, dataset, k, exclude, slab=65536):
        self._check_topk(k)
        import torch
        from .evaluation import RANKING_METRICS, ranking_metrics_batch
        from .scoring import label_lists_by_id
        dev = self.model.item_factors.device
        users, items = _on(dataset["userId"].values, dev), _on(dataset["itemId"].values, dev)
        distinct = torch.unique(users).cpu().numpy()   # the test users, deduplicated on the device
        query_ids, cand_ids, slabs = self._topk_slabs(True, distinct, k, exclude, slab)
        n_q = len(query_ids)
        per_row = torch.zeros((n_q, 5), dtype=torch.float64, device=dev)
        if n_q:
            rowptr, labels = label_lists_by_id(_on(query_ids, dev), _on(cand_ids, dev), users, items)
            for u0, u1, idx, _ in slabs:
                per_row[u0:u1] = ranking_metrics_batch(idx, (rowptr[u0:u1 + 1], labels), k)
        means = per_row.mean(0).cpu().tolist()          # NaN when no user is left, as Spark's mean of nothing
        res = dict(zip(RANKING_METRICS, means))
        res["numUsers"] = n_q
        res["numColdUsers"] = len(distinct) - n_q
        return res

    def _check_topk(self, num):
        """The argument checks of recommend_for_* and evaluate_ranking, made before any device work."""
        if isinstance(num, bool) or not isinstance(num, (int, np.integer)) or not 1 <= num <= MAX_RECOMMENDATIONS:
            raise ValueError(f"the number of recommendations must be an int in [1, {MAX_RECOMMENDATIONS}], got {num!r}")
        if self.model is None:
            raise ValueError("no trained or loaded model: call train() or load_model() first")

    def _drop_cold(self):
        s = self.cold_start_strategy
        if not isinstance(s, str) or s.lower() not in ("drop", "nan"):
            raise ValueError(f"cold_start_strategy must be 'drop' or 'nan', got {s!r}")
        return s.lower() == "drop"

    def _predict_frame(self, dataset):
        """fp32 device tensor of the predictions of dataset's (userId, itemId) rows, NaN for unknown / absent ids."""
        self._drop_cold()
        if self.model is None:
            raise ValueError("no trained or loaded model: call train() or load_model() first")
        import torch
        from . import _native as nat
        m = self.model
        dev = m.item_factors.device
        urows = _on(_rows_of(m.user_ids, dataset["userId"].values), dev)
        irows = _on(_rows_of(m.item_ids, dataset["itemId"].values), dev)
        out = torch.empty(urows.numel(), dtype=torch.float32, device=dev)
        if out.numel():
            X, Y = m.user_factors.contiguous(), m.item_factors.contiguous()
            uu, ii = urows.clamp(min=0).to(torch.int32), irows.clamp(min=0).to(torch.int32)
            nat.check(nat.lib().hals_als_predict(nat.ptr(X), nat.ptr(Y), m.rank, nat.ptr(uu), nat.ptr(ii), out.numel(),
                                                 nat.ptr(m.user_present), nat.ptr(m.item_present), nat.ptr(out),
                                                 nat.current_stream()), "hals_als_predict")
        return out.masked_fill((urows < 0) | (irows < 0), float("nan"))

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
