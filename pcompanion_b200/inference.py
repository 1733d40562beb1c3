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
``recommend``'s ranking, and hit@k / NDCG@k / MRR from those positions for any k.  ``exclude_ids`` leaves given
products out of a query's recommendations (the query itself, a cart, past purchases); ``filter_edges`` gives the
"filtered" evaluation rank, which does not count the query's other known complements (its neighbours in the graph).
"""
from __future__ import annotations

import os
from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch

from .bpg import EDGE_TYPES, BehaviorProductGraph
from .ops import TOPK_MAX_K
from .p_companion import PCompanion
from .retrieval import CatalogIndex, Exclusions, Metrics


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
        self._edge_lists: Dict[str, Exclusions] = {}

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

    def _node_index(self, product_id: str) -> int:
        i = self.bpg._index.get(product_id)
        if i is None:
            raise ValueError(f"Product ID {product_id} not found in BPG")
        return i

    def _id_lists(self, exclude_ids: Sequence[Sequence[str]], n: int, what: str) -> Exclusions:
        """One exclusion list of catalog indices per query from lists of product ids."""
        if len(exclude_ids) != n:
            raise ValueError(f"{what}: {len(exclude_ids)} exclusion lists for {n} queries")
        return Exclusions.from_lists([[self._node_index(p) for p in ids] for ids in exclude_ids], self.device)

    def _edge_exclusions(self, edge_type: str, query_nodes: torch.Tensor) -> Exclusions:
        """The graph's neighbour lists of `edge_type` as exclusion lists (its device CSR, ascending per node; the
        int64 copy of the columns is made once per edge type), row b using query_nodes[b]'s list."""
        if edge_type not in EDGE_TYPES:
            raise ValueError(f"filter_edges={edge_type!r} is not one of {EDGE_TYPES}")
        lists = self._edge_lists.get(edge_type)
        if lists is None:
            csr = self.bpg.csr(edge_type)
            lists = Exclusions(csr.rowptr.to(self.device, torch.int64), csr.col.to(self.device, torch.int64), sorted=True)
            self._edge_lists[edge_type] = lists
        return lists.for_rows(query_nodes)

    def recommend_batch(self, query_ids: Sequence[str], num_recommendations: int = 10,
                        exclude_ids: Optional[Sequence[Sequence[str]]] = None) -> List[Dict[str, Any]]:
        """Up to num_recommendations (1 .. TOPK_MAX_K = 1024) products per predicted complementary type; a type with
        fewer products returns all of them, as the reference's min(k, len(type_products)).  exclude_ids[b]: product
        ids that query b's recommendations leave out (its own id removes the query itself); the lists are exact: the
        next-best products take the freed places."""
        if not 1 <= num_recommendations <= TOPK_MAX_K:
            raise ValueError(f"num_recommendations={num_recommendations} outside [1, {TOPK_MAX_K}]")
        exclude = None if exclude_ids is None else self._id_lists(exclude_ids, len(query_ids), "recommend_batch")
        with torch.no_grad():
            outputs = self.model(self._prepare_input(query_ids))
            comp_types = outputs["complementary_types"]                      # [B, Kt]
            scores, idx = self.catalog.recommend(outputs["projected_embeddings"], comp_types, num_recommendations,
                                                 exclude=exclude)
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

    def recommend(self, query_id: str, num_recommendations: int = 10,
                  exclude_ids: Optional[Sequence[str]] = None) -> Dict[str, Any]:
        return self.recommend_batch([query_id], num_recommendations,
                                    None if exclude_ids is None else [exclude_ids])[0]

    def _pair_exclusions(self, query_ids: Sequence[str], exclude_ids: Optional[Sequence[Sequence[str]]],
                         filter_edges: Optional[str]) -> Optional[Exclusions]:
        """One exclusion list per (query, target) pair: exclude_ids[b], the query's filter_edges neighbours, or the
        union of both."""
        by_id = None if exclude_ids is None else self._id_lists(exclude_ids, len(query_ids), "rank_targets")
        if filter_edges is None:
            return by_id
        nodes = torch.tensor([self._node_index(q) for q in query_ids], dtype=torch.int64, device=self.device)
        by_edge = self._edge_exclusions(filter_edges, nodes)
        return by_edge if by_id is None else by_edge.union(by_id, len(query_ids))

    def rank_targets(self, query_ids: Sequence[str], target_ids: Sequence[str],
                     exclude_ids: Optional[Sequence[Sequence[str]]] = None,
                     filter_edges: Optional[str] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Where each held-out complementary product would land in ``recommend(query)``: (ranks int64 [B], slots int64
        [B]).  slots[b] is the position among the predicted complementary types of the one equal to the target's type
        (-1 when the model did not predict it); ranks[b] is the target's 0-based position in that type's full ranking
        (CatalogIndex.rank), -1 without a slot.  recommend(query_ids[b], k) lists target_ids[b] exactly when
        0 <= ranks[b] < k, at position ranks[b] of slot slots[b].  One batched model forward.

        Filtered rank: exclude_ids[b] (product ids) and / or filter_edges (one of EDGE_TYPES: the query's neighbours of
        that edge type, e.g. its other co-purchases) are not counted; with both, their union.  The target is never
        removed, so recommend(query_ids[b], k, exclude_ids=E_b - {target}) lists it exactly when 0 <= ranks[b] < k,
        at position ranks[b]."""
        if len(query_ids) != len(target_ids):
            raise ValueError(f"rank_targets: {len(query_ids)} queries but {len(target_ids)} targets")
        for t in target_ids:
            if t not in self.bpg.nodes:
                raise ValueError(f"Product ID {t} not found in BPG")
        batch = self._prepare_input(query_ids)
        exclude = self._pair_exclusions(query_ids, exclude_ids, filter_edges)
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
                ranks[sel] = self.catalog.rank(queries, tgt[sel], tgt_type[sel],
                                               exclude=None if exclude is None else exclude.for_rows(sel))
        return ranks, slots

    def evaluate(self, query_ids: Sequence[str], target_ids: Sequence[str],
                 ks: Sequence[int] = (1, 3, 10, 50, 100), exclude_ids: Optional[Sequence[Sequence[str]]] = None,
                 filter_edges: Optional[str] = None) -> Dict[str, float]:
        """Full-catalog retrieval quality on held-out (query, complementary product) pairs: Metrics.rank_metrics of
        rank_targets (hit@k, ndcg@k, mrr, num_rows; a pair whose target type was not predicted is a miss) and
        type_recall, the fraction of pairs whose target type is among the predicted complementary types.  hit@k is
        the fraction of pairs for which recommend(query, k) lists the target.  exclude_ids / filter_edges: the
        filtered metrics of rank_targets' filtered ranks."""
        ranks, slots = self.rank_targets(query_ids, target_ids, exclude_ids, filter_edges)
        metrics = Metrics.rank_metrics(ranks, ks)
        metrics["type_recall"] = (slots >= 0).double().mean().item() if slots.numel() else 0.0
        return metrics
