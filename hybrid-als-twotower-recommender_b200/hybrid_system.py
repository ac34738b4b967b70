"""HybridRecommendationSystem -- drop-in for the reference's src/hybrid_system.py (:20-120).

Per-user API (same signatures and return conventions as the reference):
  get_hybrid_recommendations -> predict_for_user x2 -> adaptive_fusion -> sorted()[:top_k]
with the arithmetic of adaptive_fusion (MinMaxScaler x2 + 0.8/0.2 blend, :66-72) done by
hals_fuse_lists on the device.

Batched API (additive): `recommend_batch` scores every requested user against every
candidate item in two fused passes (hals_score_extrema, hals_score_blend_topk) -- the
replacement for the `for user_id in users:` loop of reproduce_results.sh:85-89.
"""
from __future__ import annotations

import os
import warnings

import numpy as np
import pandas as pd
from sklearn.preprocessing import MinMaxScaler

from .als_model import ALSModel
from .evaluation import compute_f1_score
from .two_tower_model import TwoTowerModel

warnings.filterwarnings("ignore")


class HybridRecommendationSystem:
    def __init__(self):
        self.als_model = None
        self.twotower_model = None
        self.als_scaler = MinMaxScaler()        # kept for attribute parity (hybrid_system.py:24-25);
        self.twotower_scaler = MinMaxScaler()   # the scaling itself runs in hals_fuse_lists
        self.als_f1_score = 0.0
        self.twotower_f1_score = 0.0
        self.models_loaded = False

    def load_models(self, als_model_path, twotower_model_path):
        try:
            print("=== Loading Pre-trained Models ===")
            self.als_model = ALSModel().load_model(als_model_path)
            self.twotower_model = TwoTowerModel.load_model(twotower_model_path)
            if self.als_model is None:
                raise RuntimeError("ALS model could not be loaded")
            self.models_loaded = True
            print("\n=== Models loaded successfully ===")
            return True
        except Exception as e:
            print(f"Error loading models: {str(e)}")
            return False

    def evaluate_individual_models(self, test_user_id, actual_ratings, all_items, k=10):
        try:
            als_preds = self.als_model.predict_for_user(test_user_id, all_items)
            tt_preds = self.twotower_model.predict_for_user(test_user_id, all_items)
            # `k` is accepted and ignored, as in the reference (hybrid_system.py:42,47-48)
            self.als_f1_score = compute_f1_score(actual_ratings, dict(als_preds))
            self.twotower_f1_score = compute_f1_score(actual_ratings, dict(tt_preds))
            print(f"Model F1 Scores - ALS: {self.als_f1_score:.4f}, "
                  f"Two-Tower: {self.twotower_f1_score:.4f}")
            return self.als_f1_score, self.twotower_f1_score
        except Exception as e:
            print(f"Error evaluating models: {str(e)}")
            return 0.0, 0.0

    def fusion_weights(self):
        """(w_als, w_tt) -- strict '>' and sticky F1 scalars, hybrid_system.py:69."""
        return (0.8, 0.2) if self.als_f1_score > self.twotower_f1_score else (0.2, 0.8)

    def adaptive_fusion(self, als_predictions, twotower_predictions):
        try:
            import torch
            from . import _native as nat
            als_dict = dict(als_predictions)
            tt_dict = dict(twotower_predictions)
            all_items = set(als_dict.keys()).union(set(tt_dict.keys()))   # set order, as the reference
            if not all_items:
                return []
            als_scores = np.asarray([als_dict.get(item, 0) for item in all_items], dtype=np.float32)
            tt_scores = np.asarray([tt_dict.get(item, 0) for item in all_items], dtype=np.float32)
            dev = torch.device("cuda")
            a = torch.from_numpy(als_scores).to(dev)
            t = torch.from_numpy(tt_scores).to(dev)
            out = torch.empty_like(a)
            scratch = torch.empty(4, dtype=torch.float32, device=dev)
            weights = self.fusion_weights()
            nat.check(nat.lib().hals_fuse_lists(nat.ptr(a), nat.ptr(t), a.numel(), weights[0], weights[1],
                                                nat.ptr(out), nat.ptr(scratch), nat.current_stream()),
                      "hals_fuse_lists")
            fused = out.cpu().numpy().astype(np.float64)
            return [(item, fused[i]) for i, item in enumerate(all_items)]
        except Exception as e:
            print(f"Error in adaptive fusion: {str(e)}")
            return []

    def save_predictions(self, user_id, predictions, save_dir="results/predictions"):
        os.makedirs(save_dir, exist_ok=True)
        file_path = os.path.join(save_dir, f"user_{user_id}_predictions.csv")
        df = pd.DataFrame(predictions, columns=["itemId", "hybrid_score"])
        df["userId"] = user_id
        df["prediction_rank"] = range(1, len(df) + 1)
        df["timestamp"] = pd.Timestamp.now()
        df.to_csv(file_path, index=False)
        print(f"Predictions saved to {file_path}")
        return file_path

    def load_predictions(self, user_id, save_dir="results/predictions"):
        file_path = os.path.join(save_dir, f"user_{user_id}_predictions.csv")
        if not os.path.exists(file_path):
            raise FileNotFoundError(f"No predictions found for user {user_id}")
        df = pd.read_csv(file_path)
        return list(zip(df["itemId"], df["hybrid_score"]))

    def get_hybrid_recommendations(self, user_id, all_items, actual_ratings=None,
                                   top_k=5, save_predictions=False):
        if not self.models_loaded:
            raise ValueError("Models not loaded. Call load_models() first.")
        try:
            als_preds = self.als_model.predict_for_user(user_id, all_items)
            tt_preds = self.twotower_model.predict_for_user(user_id, all_items)
            if actual_ratings:
                self.evaluate_individual_models(user_id, actual_ratings, all_items)
            combined = self.adaptive_fusion(als_preds, tt_preds)
            top_recommendations = sorted(combined, key=lambda x: x[1], reverse=True)[:top_k]
            if save_predictions:
                self.save_predictions(user_id, combined)
            return top_recommendations
        except Exception as e:
            print(f"Error generating recommendations: {str(e)}")
            return []

    # -- additive batched path ------------------------------------------------------------------
    @staticmethod
    def _exclusion(exclude, user_ids, cand_ids, dev):
        """DataFrame of (userId, itemId) pairs -> exclusion CSR over the rows of a batched call (None -> None).
        The id matching runs on the device (sorted ids + searchsorted)."""
        if exclude is None:
            return None
        import torch
        from .scoring import exclusion_lists_by_id

        def t(a):
            return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.int64))).to(dev)
        return exclusion_lists_by_id(t(user_ids), t(cand_ids), t(exclude["userId"].values), t(exclude["itemId"].values))

    def recommend_batch(self, user_ids, item_features, top_k=5, user_chunk=65536, *, exclude=None):
        """Top-k hybrid recommendations for many users at once.

        user_ids: raw user ids known to both models; item_features: DataFrame of candidates
        (itemId, manufacturer_id, category_id, price, average_review_rating), items known to the
        ALS model.  Returns (item_ids [U,top_k] int64 numpy, scores [U,top_k] float32 numpy); ties
        are broken by candidate order (the order of `item_features`), as a stable sort would.
        Uses the current F1-selected weights (fusion_weights()).

        exclude: optional DataFrame with userId / itemId columns (e.g. the training ratings): each user's list
        leaves those items out and is filled with the next best (padded with -1 / -inf when fewer than top_k
        candidates remain).  The min-max scaling still spans all candidates, so a kept item's score is the one it
        has without `exclude`.  Pairs whose user is not in user_ids or whose item is not a candidate are ignored."""
        import torch
        from .scoring import HybridScorer
        if not self.models_loaded:
            raise ValueError("Models not loaded. Call load_models() first.")
        m = self.als_model.model
        urows = np.array([m.user_row(u) for u in user_ids], dtype=np.int64)
        irows = m.item_rows(item_features["itemId"].values)
        if (urows < 0).any() or (irows < 0).any():
            raise ValueError("recommend_batch needs users and items known to the ALS model")
        dev = m.item_factors.device
        Ua = m.user_factors[torch.from_numpy(urows).to(dev)]
        Ia = m.item_factors[torch.from_numpy(irows).to(dev)]
        Ut = self.twotower_model.user_vectors(user_ids)
        It = self.twotower_model.item_vectors(item_features)
        w_als, w_tt = self.fusion_weights()
        item_ids = np.asarray(item_features["itemId"].values)
        excl = self._exclusion(exclude, user_ids, item_ids, dev)
        out_i, out_s = [], []
        sc = HybridScorer(Ua, Ia, Ut, It)       # one scorer (items, workspace) for every slab of users
        for u0 in range(0, len(urows), user_chunk):
            u1 = min(len(urows), u0 + user_chunk)
            idx, s = sc.recommend(top_k, w_als, w_tt, u0, u1, exclude=excl)
            out_i.append(idx.cpu().numpy())
            out_s.append(s.cpu().numpy())
        idx = np.concatenate(out_i)
        return np.where(idx >= 0, item_ids[np.maximum(idx, 0)], -1), np.concatenate(out_s)

    def evaluate_models_batch(self, user_ids, actual_ratings_by_user, item_features, k=10, user_chunk=65536, *,
                              exclude=None):
        """evaluate_individual_models (hybrid_system.py:42-55) for many users at once: each model's top-k by its own
        score (the fused scoring kernels with weights (1,0) / (0,1): min-max scaling does not change a model's order)
        and F1@k against the users' rated items (hals_f1_at_k).  actual_ratings_by_user: per user a dict / iterable of
        rated item ids (the keys of the reference's `actual_ratings`).  Returns (als_f1, tt_f1) float32 numpy [U];
        the sticky scalars als_f1_score / twotower_f1_score are set to the LAST user's values, which is what a loop
        over evaluate_individual_models leaves behind.  exclude: as for recommend_batch (e.g. the training ratings,
        so that held-out items are scored against lists without the items the models were fitted on)."""
        import torch
        from .evaluation import f1_at_k_batch
        from .scoring import HybridScorer
        if not self.models_loaded:
            raise ValueError("Models not loaded. Call load_models() first.")
        m = self.als_model.model
        urows = np.array([m.user_row(u) for u in user_ids], dtype=np.int64)
        cand_ids = np.asarray(item_features["itemId"].values)
        irows = m.item_rows(cand_ids)
        if (urows < 0).any() or (irows < 0).any():
            raise ValueError("evaluate_models_batch needs users and items known to the ALS model")
        dev = m.item_factors.device
        sc = HybridScorer(m.user_factors[torch.from_numpy(urows).to(dev)], m.item_factors[torch.from_numpy(irows).to(dev)],
                          self.twotower_model.user_vectors(user_ids), self.twotower_model.item_vectors(item_features))
        order = np.argsort(cand_ids, kind="stable")
        sorted_ids = cand_ids[order]

        def cand_rows(items):      # rated item ids -> positions in the candidate list (unknown ids cannot be predicted:
            items = np.asarray(list(items))   # they stay in |actual| through a position past the end)
            pos = np.searchsorted(sorted_ids, items)
            pos = np.clip(pos, 0, len(sorted_ids) - 1)
            ok = sorted_ids[pos] == items
            extra = len(cand_ids) + np.arange(int((~ok).sum()))
            return np.concatenate([order[pos[ok]], extra]).astype(np.int32)

        actual = [cand_rows(a.keys() if hasattr(a, "keys") else a) for a in actual_ratings_by_user]
        excl = self._exclusion(exclude, user_ids, cand_ids, dev)
        f_als, f_tt = [], []
        for u0 in range(0, len(urows), user_chunk):
            u1 = min(len(urows), u0 + user_chunk)
            ia, _ = sc.recommend(k, 1.0, 0.0, u0, u1, exclude=excl)
            it, _ = sc.recommend(k, 0.0, 1.0, u0, u1, exclude=excl)
            f_als.append(f1_at_k_batch(ia, actual[u0:u1], k).cpu().numpy())
            f_tt.append(f1_at_k_batch(it, actual[u0:u1], k).cpu().numpy())
        f_als, f_tt = np.concatenate(f_als), np.concatenate(f_tt)
        if len(f_als):
            self.als_f1_score, self.twotower_f1_score = float(f_als[-1]), float(f_tt[-1])
        return f_als, f_tt

    def cleanup(self):
        if self.als_model:
            self.als_model.stop_spark()
