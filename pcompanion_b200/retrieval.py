"""Complementary retrieval and Hit@K metrics on the B200 kernels.

* ``Metrics`` mirrors /root/reference/src/utils/metrics.py (hit_at_k, type_diversity,
  mean_relevance, evaluate_model) with top-k done by pcompanion_b200/csrc/retrieval.cu.
* ``CatalogIndex`` is the catalog-wide retrieval the reference's inference.py:93-113 intends:
  for every (projected embedding, complementary type) row, rank the products of that type by
  dot product and return the top-k.  The catalog is kept with a type-sorted permutation
  (``BehaviorProductGraph.type_members``), so a row touches only its type's run of products.
  ``CatalogIndex.rank`` gives the exact position of a target product in that ranking, and
  ``Metrics.rank_metrics`` turns such ranks into full-catalog hit@k / NDCG@k / MRR.
* ``ShardedCatalog`` shards the catalog rows over the ranks of a process group; each rank ranks
  its shard and the per-shard lists are all-gathered and merged (ties -> lowest global index);
  per-shard target ranks are added.
* ``Exclusions`` are per-row lists of products a ranking leaves out (products a user already has, the query itself,
  the other known positives of a filtered evaluation rank); they apply inside the top-K and rank kernels.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

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
    def rank_metrics(ranks: torch.Tensor, ks: Sequence[int] = (1, 3, 10, 50, 100)) -> Dict[str, float]:
        """Full-catalog retrieval metrics from target ranks (``CatalogIndex.rank``: 0-based, -1 = the target can never
        be listed), one relevant product per row; every mean is over all rows and a -1 counts as a miss.
        hit@k = mean(0 <= rank < k), ndcg@k = mean(1 / log2(rank + 2) if 0 <= rank < k else 0),
        mrr = mean(1 / (rank + 1), 0 for -1), num_rows.  Any k >= 1."""
        r = ranks.reshape(-1).to(torch.float64)
        n = r.numel()
        found = r >= 0
        out: Dict[str, float] = {}
        for k in ks:
            if k < 1:
                raise ValueError(f"rank_metrics: k={k} must be >= 1")
            hit = found & (r < k)
            out[f"hit@{k}"] = hit.double().mean().item() if n else 0.0
            gain = torch.where(hit, 1.0 / torch.log2(r + 2.0), torch.zeros_like(r))
            out[f"ndcg@{k}"] = gain.mean().item() if n else 0.0
        rr = torch.where(found, 1.0 / (r + 1.0), torch.zeros_like(r))
        out["mrr"] = rr.mean().item() if n else 0.0
        out["num_rows"] = n
        return out

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


class Exclusions:
    """Per-row exclusion lists for ``CatalogIndex.topk`` / ``rank`` / ``recommend`` and ``ShardedCatalog``: score row r
    ignores the products of list E_r.

    Lists hold GLOBAL product indices (int64) in CSR form: ``offsets`` [L + 1] and ``indices`` [offsets[L]], ascending
    within each list (the constructor sorts them), duplicates allowed.  ``row_list`` [R] maps score row r to its list;
    a value outside [0, L) means no exclusions; without row_list, row r uses list r.  Entries outside the catalog (or
    shard) and entries of another type have no effect, so one set of lists serves every shard unchanged.

    The input is validated once here (one host synchronisation, none per query): offsets[0] == 0, non-decreasing,
    offsets[-1] == indices.numel(), row_list 1-D; anything else raises ValueError.  ``sorted=True`` skips the sort for
    lists that are already ascending (a graph's CSR neighbour lists)."""

    def __init__(self, offsets: torch.Tensor, indices: torch.Tensor, row_list: Optional[torch.Tensor] = None,
                 sorted: bool = False):
        offsets = torch.as_tensor(offsets)
        indices = torch.as_tensor(indices, device=offsets.device)
        if offsets.dim() != 1 or offsets.numel() < 1 or indices.dim() != 1:
            raise ValueError(f"Exclusions: offsets {tuple(offsets.shape)} and indices {tuple(indices.shape)} must be 1-D, "
                             "offsets with at least one entry")
        if offsets.dtype.is_floating_point or indices.dtype.is_floating_point:
            raise ValueError("Exclusions: offsets and indices must be integer tensors")
        if offsets.numel() - 1 >= 2 ** 31:
            raise ValueError(f"Exclusions: {offsets.numel() - 1} lists (at most 2^31 - 1)")
        offsets = offsets.to(torch.int64).contiguous()
        indices = indices.to(torch.int64).contiguous()
        n = indices.numel()
        ok = (offsets[0] == 0) & (offsets[-1] == n) & (offsets.diff() >= 0).all()
        if not bool(ok):
            raise ValueError("Exclusions: offsets must start at 0, be non-decreasing and end at indices.numel()")
        if row_list is not None:
            row_list = torch.as_tensor(row_list, device=offsets.device)
            if row_list.dim() != 1 or row_list.dtype.is_floating_point:
                raise ValueError(f"Exclusions: row_list {tuple(row_list.shape)} must be a 1-D integer tensor")
        self.offsets = offsets
        self.indices = indices if sorted else self._sort_lists(offsets, indices)
        self.row_list = None if row_list is None else self._list_ids(row_list, self.num_lists)

    @property
    def num_lists(self) -> int:
        return self.offsets.numel() - 1

    @staticmethod
    def _list_ids(row_list: torch.Tensor, n_lists: int) -> torch.Tensor:
        """int32 list ids; anything outside [0, n_lists) becomes -1 (no exclusions) before the narrowing."""
        rl = row_list.to(torch.int64)
        return torch.where((rl >= 0) & (rl < n_lists), rl, torch.full_like(rl, -1)).to(torch.int32).contiguous()

    @staticmethod
    def _sort_lists(offsets: torch.Tensor, indices: torch.Tensor) -> torch.Tensor:
        """Sort every list on the device: a stable sort by value, then a stable sort by list id."""
        n = indices.numel()
        if n == 0:
            return indices
        lid = torch.repeat_interleave(torch.arange(offsets.numel() - 1, device=offsets.device), offsets.diff(),
                                      output_size=n)
        by_value = torch.argsort(indices, stable=True)
        by_list = torch.argsort(lid[by_value], stable=True)
        return indices[by_value][by_list].contiguous()

    @classmethod
    def _trusted(cls, offsets: torch.Tensor, indices: torch.Tensor, row_list: Optional[torch.Tensor]) -> "Exclusions":
        """Lists built by this module (valid offsets, ascending lists, int32 row_list): no validation, no sort."""
        ex = cls.__new__(cls)
        ex.offsets, ex.indices, ex.row_list = offsets, indices, row_list
        return ex

    @classmethod
    def from_lists(cls, lists: Sequence[Sequence[int]], device, row_list: Optional[torch.Tensor] = None) -> "Exclusions":
        """Lists of global product indices in any order (sorted on the device)."""
        lens = torch.tensor([len(x) for x in lists], dtype=torch.int64)
        offsets = torch.zeros(len(lists) + 1, dtype=torch.int64)
        torch.cumsum(lens, 0, out=offsets[1:])
        flat = torch.tensor([int(v) for x in lists for v in x], dtype=torch.int64)
        return cls(offsets.to(device), flat.to(device), row_list)

    def for_rows(self, row_of: torch.Tensor) -> "Exclusions":
        """The same lists for new score rows, row i using the list of this object's row row_of[i] (no list is
        copied)."""
        row_of = row_of.to(self.offsets.device, torch.int64)
        rl = self._list_ids(row_of, self.num_lists) if self.row_list is None else self.row_list[row_of].contiguous()
        return Exclusions._trusted(self.offsets, self.indices, rl)

    def union(self, other: "Exclusions", rows: int) -> "Exclusions":
        """One list per score row r < rows: the union (with duplicates) of r's lists in self and in other."""
        dev_ = self.offsets.device
        beg_a, len_a = self._spans(rows)
        beg_b, len_b = other._spans(rows)
        lens = len_a + len_b
        offsets = torch.zeros(rows + 1, dtype=torch.int64, device=dev_)
        torch.cumsum(lens, 0, out=offsets[1:])
        total = int(offsets[-1].item())
        row = torch.repeat_interleave(torch.arange(rows, device=dev_), lens, output_size=total)
        pos = torch.arange(total, device=dev_) - offsets[row]
        src = torch.where(pos < len_a[row], beg_a[row] + pos, self.indices.numel() + beg_b[row] + pos - len_a[row])
        values = torch.cat([self.indices, other.indices])[src]
        return Exclusions._trusted(offsets, self._sort_lists(offsets, values), None)

    def _spans(self, rows: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(first entry, length) of the list of every score row r < rows (length 0 without a list)."""
        dev_ = self.offsets.device
        lid = self.row_list.to(torch.int64) if self.row_list is not None else torch.arange(rows, device=dev_)
        if lid.numel() != rows:
            raise ValueError(f"Exclusions: row_list has {lid.numel()} rows, expected {rows}")
        ok = (lid >= 0) & (lid < self.num_lists)
        safe = torch.where(ok, lid, torch.zeros_like(lid))
        beg = self.offsets[safe]
        return beg, torch.where(ok, self.offsets[safe + 1] - beg, torch.zeros_like(beg))


def _check_exclusions(exclude: Optional[Exclusions], rows: int, what: str) -> None:
    if exclude is not None and exclude.row_list is not None and exclude.row_list.numel() != rows:
        raise ValueError(f"{what}: exclusion row_list has {exclude.row_list.numel()} entries for {rows} score rows")


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

    def _whole_run(self) -> torch.Tensor:
        """type_offsets {0, P} of one type holding the whole catalog: the run of rows without a row type."""
        if self._all is None:
            self._all = torch.tensor([0, self.num_products], dtype=torch.int64, device=self.catalog.device)
        return self._all

    def topk(self, queries: torch.Tensor, k: int, row_type: Optional[torch.Tensor] = None,
             splits: Optional[int] = None, exclude: Optional[Exclusions] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-k per query row, 1 <= k <= ops.TOPK_MAX_K (1024; ValueError otherwise); row_type[r] restricts row r
        to products of that type (all products when row_type is None).  Returns (scores float64 [R, k], global
        indices int64 [R, k]), padded with (-inf, -1) when a type has fewer than k products.  exclude: row r ranks
        its products without those of its exclusion list (the exact top-k of what remains)."""
        queries = queries.contiguous().float()
        _check_exclusions(exclude, queries.shape[0], "CatalogIndex.topk")
        if row_type is None:
            return ops.topk_by_type(queries, self.catalog, self._whole_run(), 1, None, k, None, self.index_base, splits,
                                    exclude)
        if self.offsets is None:
            raise ValueError("CatalogIndex.topk: the catalog was built without type ids")
        rt = row_type.to(queries.device, torch.int32).contiguous()
        return ops.topk_by_type(queries, self.catalog, self.offsets, self.num_types, rt, k, self.members, self.index_base,
                                splits, exclude)

    def topk_dense(self, queries: torch.Tensor, k: int, row_type: Optional[torch.Tensor] = None):
        """Same result as ``topk`` (bit for bit, every row type) through the dense tensor-core path (BASELINE north_star
        part 4): single-pass TF32 scoring GEMM over the whole catalog, per-type mask and candidate selection in the
        epilogue, exact fp64 re-scoring.  Rows whose guard band fails are re-run on the exact segmented kernel, so the
        output is always exact.  1 <= k <= 16 and D in {32, 64, 96, 128} (RuntimeError otherwise).  As in ``topk``, a
        row type outside [0, num_types) gives (-inf, -1) padding, and row types on a catalog built without type ids
        raise ValueError."""
        queries = queries.contiguous().float()
        if row_type is not None and self.type_id is None:
            raise ValueError("CatalogIndex.topk_dense: the catalog was built without type ids")
        if self._max_norm is None:
            self._max_norm = float(self.catalog.norm(dim=1).max().item())
        rt = None if row_type is None else row_type.to(queries.device, torch.int32).contiguous()
        s, i, flags = ops.score_topk_dense(queries, self.catalog, k, self.type_id, rt, self.index_base, self._max_norm)
        if rt is not None:
            # the kernel reads a negative row type as "no restriction"; topk lists nothing outside [0, num_types)
            out = ((rt < 0) | (rt >= self.num_types)).unsqueeze(1)
            s.masked_fill_(out, float("-inf"))
            i.masked_fill_(out, -1)
            flags.masked_fill_(out.squeeze(1), 0)
        bad = torch.nonzero(flags).squeeze(1)
        if bad.numel():
            fs, fi = self.topk(queries[bad], k, None if rt is None else rt[bad])
            s[bad], i[bad] = fs, fi
        return s, i

    def _owned_targets(self, queries: torch.Tensor, targets: torch.Tensor, row_type: Optional[torch.Tensor]):
        """(row types int32 or None, member bool [R], target rows fp32 [R, D]) for global target indices: member[r] when
        this catalog holds targets[r] and, with row types, the target has row r's type.  Rows that are not members get
        catalog row 0 as a stand-in (an out-of-range index is never gathered)."""
        rows = queries.shape[0]
        if tuple(targets.shape) != (rows,):
            raise ValueError(f"CatalogIndex.rank: targets {tuple(targets.shape)} != ({rows},)")
        if row_type is not None and self.offsets is None:
            raise ValueError("CatalogIndex.rank: the catalog was built without type ids")
        local = targets.to(queries.device, torch.int64) - self.index_base
        member = (local >= 0) & (local < self.num_products)
        safe = torch.where(member, local, torch.zeros_like(local))
        rt = None
        if row_type is not None:
            rt = row_type.to(queries.device, torch.int32).reshape(-1).contiguous()
            if self.num_products:
                member &= self.type_id[safe] == rt
        if self.num_products == 0:
            return rt, member, torch.zeros(rows, queries.shape[1], dtype=torch.float32, device=queries.device)
        return rt, member, ops.gather_rows(self.catalog, safe)

    def _rank_counts(self, queries: torch.Tensor, target_rows: torch.Tensor, targets: torch.Tensor,
                     row_type: Optional[torch.Tensor], splits: Optional[int] = None,
                     exclude: Optional[Exclusions] = None) -> torch.Tensor:
        """Products of this catalog that rank before each target and are not excluded (pc_rank_by_type, then
        pc_rank_remove_excluded; -1 for a row type out of range)."""
        targets = targets.to(queries.device, torch.int64).contiguous()
        if self.num_products == 0:
            return torch.zeros(queries.shape[0], dtype=torch.int64, device=queries.device)
        if row_type is None:
            return ops.rank_by_type(queries, self.catalog, self._whole_run(), 1, None, target_rows, targets, None,
                                    self.index_base, splits, exclude)
        return ops.rank_by_type(queries, self.catalog, self.offsets, self.num_types, row_type, target_rows, targets,
                                self.members, self.index_base, splits, exclude, self.type_id)

    def rank(self, queries: torch.Tensor, targets: torch.Tensor, row_type: Optional[torch.Tensor] = None,
             splits: Optional[int] = None, exclude: Optional[Exclusions] = None) -> torch.Tensor:
        """Exact rank of the product targets[r] (int64 global index) in row r's ranking: the number of products of the
        row's type (all products when row_type is None) that rank strictly before it, by score descending, then lower
        index.  -1 when the target can never be listed for the row: it is not in the catalog, or row_type[r] is not its
        type.  For every k, 0 <= rank < k exactly when ``topk(queries, k, row_type)`` lists the target, and it is then at
        position rank.  Returns int64 [R].

        exclude: the "filtered" rank, which does not count the products of row r's exclusion list.  The target itself
        is never removed, so a list of known positives can be passed as it is: 0 <= rank < k exactly when
        ``topk(queries, k, row_type, exclude=E - {target})`` lists the target, at position rank."""
        queries = queries.contiguous().float()
        _check_exclusions(exclude, queries.shape[0], "CatalogIndex.rank")
        rt, member, target_rows = self._owned_targets(queries, targets, row_type)
        counts = self._rank_counts(queries, target_rows, targets, rt, splits, exclude)
        return torch.where(member, counts, torch.full_like(counts, -1))

    def recommend(self, projected_embeddings: torch.Tensor, complementary_types: torch.Tensor, k: int = 10,
                  exclude: Optional[Exclusions] = None):
        """The loop of inference.py:93-113 for a whole batch: projected [B, Kt, D], types [B, Kt] ->
        (scores [B, Kt, k], product indices [B, Kt, k]), 1 <= k <= ops.TOPK_MAX_K; a type with fewer than k products
        pads its rows with (-inf, -1).  exclude: lists per QUERY (row b of the batch, or exclude.row_list[b]); every
        type row of query b leaves out query b's list."""
        b, kt, d = projected_embeddings.shape
        if exclude is not None:
            _check_exclusions(exclude, b, "CatalogIndex.recommend")
            exclude = exclude.for_rows(torch.arange(b, device=projected_embeddings.device).repeat_interleave(kt))
        s, i = self.topk(projected_embeddings.reshape(b * kt, d), k, complementary_types.reshape(-1), exclude=exclude)
        return s.reshape(b, kt, k), i.reshape(b, kt, k)


class ShardedCatalog:
    """Catalog rows sharded contiguously over a process group (SURVEY 8e): rank g owns rows
    [bounds[g], bounds[g+1]); queries are replicated; per-shard top-k lists are all-gathered and
    merged.  Works with NCCL (CUDA tensors) and gloo; the only collective of topk is one [R, 2k] all-gather (rank: two
    all-reduces, [R, D + 1] fp32 and [R] int64)."""

    def __init__(self, local_catalog: torch.Tensor, local_type_id: Optional[torch.Tensor], index_base: int,
                 num_types: Optional[int] = None, group=None):
        self.group = group
        self.local = CatalogIndex(local_catalog, local_type_id, index_base, num_types)

    def topk(self, queries: torch.Tensor, k: int, row_type: Optional[torch.Tensor] = None,
             exclude: Optional[Exclusions] = None):
        """CatalogIndex.topk over the whole sharded catalog; exclude holds global indices and every shard applies
        the same lists."""
        import torch.distributed as dist
        s, i = self.local.topk(queries, k, row_type, exclude=exclude)
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

    def rank(self, queries: torch.Tensor, targets: torch.Tensor, row_type: Optional[torch.Tensor] = None,
             exclude: Optional[Exclusions] = None) -> torch.Tensor:
        """CatalogIndex.rank over the whole sharded catalog (queries, targets and row types replicated on every rank);
        equal to the rank on the unsharded catalog.  The shard that owns a target supplies its row and membership (one
        all-reduce: the other shards add zeros, which change no bit of the row), every shard counts its own products that
        rank before it (less its own excluded products), and one all-reduce adds the counts."""
        import torch.distributed as dist
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if world == 1:
            return self.local.rank(queries, targets, row_type, exclude=exclude)
        _check_exclusions(exclude, queries.shape[0], "ShardedCatalog.rank")
        queries = queries.contiguous().float()
        rt, member, target_rows = self.local._owned_targets(queries, targets, row_type)
        packed = torch.cat([torch.where(member[:, None], target_rows, torch.zeros_like(target_rows)),
                            member[:, None].float()], dim=1).contiguous()
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=self.group)
        member = packed[:, -1] > 0
        counts = self.local._rank_counts(queries, packed[:, :-1].contiguous(), targets, rt, exclude=exclude)
        counts = counts.clamp_min(0)               # a row type past this shard's type count: none of its products
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=self.group)
        return torch.where(member, counts, torch.full_like(counts, -1))
