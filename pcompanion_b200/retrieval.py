"""Complementary retrieval and Hit@K metrics on the B200 kernels.

* ``Metrics`` mirrors /root/reference/src/utils/metrics.py (hit_at_k, type_diversity,
  mean_relevance, evaluate_model) with top-k done by pcompanion_b200/csrc/retrieval.cu.
* ``CatalogIndex`` is the catalog-wide retrieval the reference's inference.py:93-113 intends:
  for every (projected embedding, complementary type) row, rank the products of that type by
  dot product and return the top-k.  The catalog is kept with a type-sorted permutation
  (``BehaviorProductGraph.type_members``), so a row touches only its type's run of products.
* ``ShardedCatalog`` shards the catalog rows over the ranks of a process group; each rank ranks
  its shard and the per-shard lists are all-gathered and merged (ties -> lowest global index).
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import ops


def _score_matrix(rows: torch.Tensor, targets: torch.Tensor) -> torch.Tensor:
    """rows . targets^T (metrics.py:89) on the tcgen05 scoring kernel; shapes it is not instantiated for (a last batch
    whose size is not a multiple of 4, odd embedding widths) go to the library GEMM."""
    rows, targets = rows.float(), targets.float()
    if ops.type_scores_topk_supported(rows, targets, 1):
        return ops.type_scores_topk(rows, targets, 1, materialize=True)[0]
    return torch.matmul(rows, targets.T)


class Metrics:
    @staticmethod
    def hit_at_k(predictions: torch.Tensor, ground_truth: torch.Tensor, k: int) -> float:
        """metrics.py:7-26.  k is clipped to the number of columns as torch.topk requires; after that, k may be up to
        ops.TOPK_MAX_K (ValueError beyond)."""
        k = min(k, predictions.size(1))
        _, top_k = ops.topk_rows(predictions.float(), k)
        hits = torch.any(top_k == ground_truth.unsqueeze(1), dim=1)
        return hits.float().mean().item()

    @staticmethod
    def type_diversity(predicted_types: torch.Tensor) -> float:
        """metrics.py:29-41."""
        if predicted_types.numel() == 0:
            return 0.0
        unique_types = torch.unique(predicted_types, dim=1)
        return unique_types.size(1) / predicted_types.size(1)

    @staticmethod
    def mean_relevance(predictions: torch.Tensor, ground_truth: torch.Tensor) -> float:
        """metrics.py:44-59."""
        return torch.cosine_similarity(predictions, ground_truth.unsqueeze(1), dim=-1).mean().item()

    @staticmethod
    def evaluate_model(model: torch.nn.Module, data_loader, device: torch.device) -> Dict[str, float]:
        """metrics.py:62-117 (in-batch scoring of [3B, D] projections against the B targets)."""
        model.eval()
        metrics = {"hit@1": 0.0, "hit@3": 0.0, "hit@10": 0.0, "type_diversity": 0.0, "mean_relevance": 0.0}
        num_batches = 0
        with torch.no_grad():
            for batch in data_loader:
                batch = {k: v.to(device) if torch.is_tensor(v) else v for k, v in batch.items()}
                outputs = model(batch)
                proj = outputs["projected_embeddings"]
                similarities = _score_matrix(proj.reshape(-1, proj.size(-1)), batch["target_features"])
                gt = torch.arange(similarities.size(0), device=device)
                for k in [1, 3, min(10, similarities.size(1))]:
                    metrics[f"hit@{k}"] += Metrics.hit_at_k(similarities, gt, k=k)
                metrics["type_diversity"] += Metrics.type_diversity(outputs["complementary_types"])
                metrics["mean_relevance"] += Metrics.mean_relevance(proj, batch["positive_items"])
                num_batches += 1
        for key in metrics:
            metrics[key] /= max(num_batches, 1)
        return metrics


class CatalogIndex:
    """Type-segmented catalog on one GPU.

    catalog [P, D] fp32 (D % 128 == 0), type_id int32 [P].  ``index_base`` is the global id of
    local row 0 (sharded catalogs)."""

    def __init__(self, catalog: torch.Tensor, type_id: Optional[torch.Tensor] = None, index_base: int = 0,
                 num_types: Optional[int] = None):
        if not catalog.is_cuda:
            raise RuntimeError("CatalogIndex: catalog must live on the GPU (no CPU fallback)")
        self.catalog = catalog.contiguous().float()
        self.index_base = int(index_base)
        self.num_products = catalog.shape[0]
        self.type_id = None
        self.members = None
        self.offsets = None
        self._max_norm = None
        self._all = None
        if type_id is not None:
            self.type_id = type_id.to(catalog.device, torch.int32).contiguous()
            n_types = int(num_types) if num_types is not None else (int(self.type_id.max().item()) + 1 if self.num_products else 0)
            node = torch.arange(self.num_products, dtype=torch.int32, device=catalog.device)
            csr, _ = ops.build_csr(self.type_id, node, n_types, max(self.num_products, 1))
            self.members, self.offsets = csr.col, csr.rowptr
            self.num_types = n_types

    def topk(self, queries: torch.Tensor, k: int, row_type: Optional[torch.Tensor] = None,
             splits: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-k per query row, 1 <= k <= ops.TOPK_MAX_K (1024; ValueError otherwise); row_type[r] restricts row r
        to products of that type (all products when row_type is None).  Returns (scores float64 [R, k], global
        indices int64 [R, k]), padded with (-inf, -1) when a type has fewer than k products."""
        queries = queries.contiguous().float()
        if row_type is None:
            if self._all is None:
                self._all = torch.tensor([0, self.num_products], dtype=torch.int64, device=queries.device)
            return ops.topk_by_type(queries, self.catalog, self._all, 1, None, k, None, self.index_base, splits)
        if self.offsets is None:
            raise ValueError("CatalogIndex.topk: the catalog was built without type ids")
        rt = row_type.to(queries.device, torch.int32).contiguous()
        return ops.topk_by_type(queries, self.catalog, self.offsets, self.num_types, rt, k, self.members, self.index_base, splits)

    def topk_dense(self, queries: torch.Tensor, k: int, row_type: Optional[torch.Tensor] = None):
        """Same result as ``topk`` through the dense tensor-core path (BASELINE north_star part 4): single-pass TF32 scoring
        GEMM over the whole catalog, per-type mask and candidate selection in the epilogue, exact fp64 re-scoring.
        Rows whose guard band fails are re-run on the exact segmented kernel, so the output is always exact."""
        queries = queries.contiguous().float()
        if self._max_norm is None:
            self._max_norm = float(self.catalog.norm(dim=1).max().item())
        rt = None if row_type is None else row_type.to(queries.device, torch.int32).contiguous()
        s, i, flags = ops.score_topk_dense(queries, self.catalog, k, self.type_id, rt, self.index_base, self._max_norm)
        bad = torch.nonzero(flags).squeeze(1)
        if bad.numel():
            fs, fi = self.topk(queries[bad], k, None if rt is None else rt[bad])
            s[bad], i[bad] = fs, fi
        return s, i

    def recommend(self, projected_embeddings: torch.Tensor, complementary_types: torch.Tensor, k: int = 10):
        """The loop of inference.py:93-113 for a whole batch: projected [B, Kt, D], types [B, Kt] ->
        (scores [B, Kt, k], product indices [B, Kt, k]), 1 <= k <= ops.TOPK_MAX_K; a type with fewer than k products
        pads its rows with (-inf, -1)."""
        b, kt, d = projected_embeddings.shape
        s, i = self.topk(projected_embeddings.reshape(b * kt, d), k, complementary_types.reshape(-1))
        return s.reshape(b, kt, k), i.reshape(b, kt, k)


class ShardedCatalog:
    """Catalog rows sharded contiguously over a process group (SURVEY 8e): rank g owns rows
    [bounds[g], bounds[g+1]); queries are replicated; per-shard top-k lists are all-gathered and
    merged.  Works with NCCL (CUDA tensors) and gloo; the only collective is one [R, 2k] all-gather."""

    def __init__(self, local_catalog: torch.Tensor, local_type_id: Optional[torch.Tensor], index_base: int,
                 num_types: Optional[int] = None, group=None):
        self.group = group
        self.local = CatalogIndex(local_catalog, local_type_id, index_base, num_types)

    def topk(self, queries: torch.Tensor, k: int, row_type: Optional[torch.Tensor] = None):
        import torch.distributed as dist
        s, i = self.local.topk(queries, k, row_type)
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if world == 1:
            return s, i
        # ONE collective: the int64 indices travel as their float64 bit patterns next to the scores ([R, 2k] per rank)
        packed = torch.cat([s, i.view(torch.float64)], dim=1).contiguous()
        gathered = torch.empty(world, *packed.shape, dtype=torch.float64, device=s.device)
        dist.all_gather_into_tensor(gathered, packed, group=self.group)
        cat_s = gathered[:, :, :k].permute(1, 0, 2).reshape(s.shape[0], world * k)
        cat_i = gathered[:, :, k:].permute(1, 0, 2).reshape(s.shape[0], world * k).contiguous().view(torch.int64)
        return ops.topk_merge(cat_s, cat_i, k)
