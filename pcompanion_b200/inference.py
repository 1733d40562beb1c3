"""Complementary recommendation entry point (SURVEY 8f rank 3).

A working counterpart of /root/reference/inference.py ``PCompanionInference``: same constructor
idea (a trained P-Companion + a BPG), same ``recommend(query_id, num_recommendations=10)`` result
layout ({'complementary_types', 'recommendations', 'scores'}), same semantics as its loop at
:93-118 (for each predicted complementary type: products of that type, score = projected . item
features, top-k) - but the shipped file cannot be imported (:7-8, :17) and feeds a batch whose keys
do not match ``PCompanion.forward``; here the batch is built with the keys forward() consumes and the
per-type scoring runs on the type-segmented catalog kernel (exact fp64, ties -> lowest index).
``recommend_batch`` answers many queries in one launch.  ``rank_targets`` / ``evaluate`` score held-out
(query, complementary product) pairs against the whole catalog: the exact position of the true product in
``recommend``'s ranking, and hit@k / NDCG@k / MRR from those positions for any k.
"""
from __future__ import annotations

import os
from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch

from .bpg import BehaviorProductGraph
from .ops import TOPK_MAX_K
from .p_companion import PCompanion
from .retrieval import CatalogIndex, Metrics


class PCompanionInference:
    def __init__(self, model_path: Optional[str], config, bpg: BehaviorProductGraph, model: Optional[PCompanion] = None,
                 type_to_idx: Optional[Dict[Any, int]] = None):
        self.config = config
        self.device = config.DEVICE
        self.bpg = bpg.finalize()
        if model is None:
            raise ValueError("PCompanionInference needs a constructed PCompanion (its embedding table defines the catalog)")
        self.model = model.to(self.device)
        if model_path is not None:
            self._load_model(model_path)
        self.model.eval()
        # type name -> index used by the model's type embeddings (ComplementaryDataset.type_to_idx order by default)
        names = self.bpg._type_names or []
        self.type_to_idx = type_to_idx if type_to_idx is not None else {t: i for i, t in enumerate(names)}
        ids = self.bpg._ids
        self._ids = ids
        # catalog = raw product features, typed by the *model's* type index (inference.py:95-104)
        type_idx = torch.tensor([self.type_to_idx[self.bpg.nodes[p]["type"]] for p in ids], dtype=torch.int32)
        self.catalog = CatalogIndex(self.bpg.features.to(self.device), type_idx.to(self.device),
                                    num_types=max(self.type_to_idx.values()) + 1 if self.type_to_idx else None)
        self._type_of = type_idx

    def _load_model(self, model_path: str) -> None:
        if not os.path.exists(model_path):
            raise FileNotFoundError(f"Model file not found: {model_path}")
        checkpoint = torch.load(model_path, map_location=self.device)
        self.model.load_state_dict(checkpoint["model_state_dict"])

    def _prepare_input(self, query_ids: Sequence[str]) -> Dict[str, Any]:
        for q in query_ids:
            if q not in self.bpg.nodes:
                raise ValueError(f"Product ID {q} not found in BPG")
        types = torch.tensor([self.type_to_idx[self.bpg.nodes[q]["type"]] for q in query_ids], dtype=torch.int64,
                             device=self.device)
        return {"query_ids": list(query_ids), "query_types": types}

    def recommend_batch(self, query_ids: Sequence[str], num_recommendations: int = 10) -> List[Dict[str, Any]]:
        """Up to num_recommendations (1 .. TOPK_MAX_K = 1024) products per predicted complementary type; a type with
        fewer products returns all of them, as the reference's min(k, len(type_products))."""
        if not 1 <= num_recommendations <= TOPK_MAX_K:
            raise ValueError(f"num_recommendations={num_recommendations} outside [1, {TOPK_MAX_K}]")
        with torch.no_grad():
            outputs = self.model(self._prepare_input(query_ids))
            comp_types = outputs["complementary_types"]                      # [B, Kt]
            scores, idx = self.catalog.recommend(outputs["projected_embeddings"], comp_types, num_recommendations)
        comp_types, scores, idx = comp_types.cpu(), scores.cpu(), idx.cpu()
        results = []
        for b in range(len(query_ids)):
            recs, scs = [], []
            for t in range(comp_types.shape[1]):
                valid = idx[b, t] >= 0
                if not bool(valid.any()):
                    continue                                               # `if not type_products: continue`, :97-98
                recs.append([self._ids[j] for j in idx[b, t][valid].tolist()])
                scs.append(scores[b, t][valid].numpy())
            results.append({"complementary_types": comp_types[b].tolist(), "recommendations": recs, "scores": scs})
        return results

    def recommend(self, query_id: str, num_recommendations: int = 10) -> Dict[str, Any]:
        return self.recommend_batch([query_id], num_recommendations)[0]

    def rank_targets(self, query_ids: Sequence[str], target_ids: Sequence[str]) -> Tuple[torch.Tensor, torch.Tensor]:
        """Where each held-out complementary product would land in ``recommend(query)``: (ranks int64 [B], slots int64
        [B]).  slots[b] is the position among the predicted complementary types of the one equal to the target's type
        (-1 when the model did not predict it); ranks[b] is the target's 0-based position in that type's full ranking
        (CatalogIndex.rank), -1 without a slot.  recommend(query_ids[b], k) lists target_ids[b] exactly when
        0 <= ranks[b] < k, at position ranks[b] of slot slots[b].  One batched model forward."""
        if len(query_ids) != len(target_ids):
            raise ValueError(f"rank_targets: {len(query_ids)} queries but {len(target_ids)} targets")
        for t in target_ids:
            if t not in self.bpg.nodes:
                raise ValueError(f"Product ID {t} not found in BPG")
        batch = self._prepare_input(query_ids)
        tgt = torch.tensor([self.bpg._index[t] for t in target_ids], dtype=torch.int64)
        tgt_type = self._type_of[tgt].to(self.device, torch.int64)
        tgt = tgt.to(self.device)
        ranks = torch.full((len(query_ids),), -1, dtype=torch.int64, device=self.device)
        if not len(query_ids):
            return ranks, ranks.clone()
        with torch.no_grad():
            outputs = self.model(batch)
            match = outputs["complementary_types"].to(torch.int64) == tgt_type[:, None]          # [B, Kt]
            slots = torch.where(match.any(1), match.int().argmax(1).to(torch.int64), torch.full_like(tgt, -1))
            sel = torch.nonzero(slots >= 0).squeeze(1)
            if sel.numel():
                queries = outputs["projected_embeddings"][sel, slots[sel]]
                ranks[sel] = self.catalog.rank(queries, tgt[sel], tgt_type[sel])
        return ranks, slots

    def evaluate(self, query_ids: Sequence[str], target_ids: Sequence[str],
                 ks: Sequence[int] = (1, 3, 10, 50, 100)) -> Dict[str, float]:
        """Full-catalog retrieval quality on held-out (query, complementary product) pairs: Metrics.rank_metrics of
        rank_targets (hit@k, ndcg@k, mrr, num_rows; a pair whose target type was not predicted is a miss) and
        type_recall, the fraction of pairs whose target type is among the predicted complementary types.  hit@k is
        the fraction of pairs for which recommend(query, k) lists the target."""
        ranks, slots = self.rank_targets(query_ids, target_ids)
        metrics = Metrics.rank_metrics(ranks, ks)
        metrics["type_recall"] = (slots >= 0).double().mean().item() if slots.numel() else 0.0
        return metrics
