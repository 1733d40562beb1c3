"""Data path on top of the device CSR (SURVEY 8f rank 1).

Two layers:

* Drop-ins for /root/reference/src/data/data_loader.py - ``SimilarityDataset``, ``ComplementaryDataset``,
  ``collate_fn`` - with the same constructor signatures, sample / batch dict keys, padding rule and
  error behaviour, so ``scripts/pretrain_product2vec.py`` and ``train.py`` run unchanged.  The O(E)
  per-sample neighbour scan (bpg.py:24-38) and the per-sample rebuild of the anchor's similar set
  (data_loader.py:31) - 78 % of the reference's epoch time - become CSR row slices.
* ``GraphTripletSampler``: the CSR-native path.  A batch is a few index tensors on the device
  (anchor, positive, negatives) into the full-graph embedding table; negatives come from
  pcompanion_b200/csrc/sample.cu (same rejection rule as data_loader.py:27-40).  No feature copies,
  no padding, no Python per sample.  ``neighborhood_batches`` / ``TripletBatch`` add each anchor's co-view
  neighbour offsets for the reference's mini-batch step (Product2Vec.triplet_loss_graph).
"""
from __future__ import annotations

import logging
import random
from collections import defaultdict
from typing import Dict, List, NamedTuple, Optional, Tuple

import torch
from torch.utils.data import Dataset

from . import ops
from ._lib import call, dev, stream
from .bpg import BehaviorProductGraph


class SimilarityDataset(Dataset):
    """data_loader.py:11-88 (anchor, positive, 5 negatives, co-view neighbour features)."""

    def __init__(self, bpg: BehaviorProductGraph, config):
        self.bpg = bpg
        self.config = config
        self.logger = logging.getLogger(__name__)
        self.similar_pairs = bpg.similarity_pairs
        if len(self.similar_pairs) == 0:
            raise ValueError("No similarity pairs found in BPG")
        self._all_products = list(bpg.nodes.keys())
        self._similar_of: Dict[str, set] = defaultdict(set)
        for a, b in self.similar_pairs:
            self._similar_of[a].add(b)
        self._host_csr = None
        self.logger.info(f"Created similarity dataset with {len(self.similar_pairs)} pairs")

    def _get_negative_samples(self, anchor_id: str, k: int = 5) -> List[str]:
        neg_ids: List[str] = []
        similar = self._similar_of.get(anchor_id, ())
        while len(neg_ids) < k:
            neg_id = random.choice(self._all_products)
            if neg_id != anchor_id and neg_id not in similar and neg_id not in neg_ids:
                neg_ids.append(neg_id)
        return neg_ids

    def __len__(self) -> int:
        return len(self.similar_pairs)

    def _neighbors(self, product_id: str) -> List[str]:
        """co-view out-neighbours from a host copy of the CSR (DataLoader workers must not touch CUDA)."""
        if self._host_csr is None:
            g = self.bpg.csr("co_view")
            self._host_csr = (g.rowptr.cpu(), g.col.cpu(), {p: i for i, p in enumerate(self._all_products)})
        rowptr, col, index = self._host_csr
        i = index[product_id]
        return [self._all_products[j] for j in col[rowptr[i]: rowptr[i + 1]].tolist()]

    def _get_neighbor_features(self, product_id: str) -> Optional[torch.Tensor]:
        feats = [self.bpg.nodes[n]["features"].clone().detach() for n in self._neighbors(product_id) if n in self.bpg.nodes]
        return torch.stack(feats) if feats else None

    def __getitem__(self, idx: int) -> Dict[str, torch.Tensor]:
        anchor_id, positive_id = self.similar_pairs[idx]
        negative_ids = self._get_negative_samples(anchor_id)
        nodes = self.bpg.nodes
        sample = {
            "anchor_ids": anchor_id,
            "anchor": nodes[anchor_id]["features"].clone().detach(),
            "positive": nodes[positive_id]["features"].clone().detach(),
            "negative": torch.stack([nodes[n]["features"].clone().detach() for n in negative_ids]),
            "positive_id": positive_id,
            "negative_ids": negative_ids,
        }
        anchor_neighbors = self._get_neighbor_features(anchor_id)
        if anchor_neighbors is not None:
            sample["anchor_neighbors"] = anchor_neighbors
        return sample


class ComplementaryDataset(Dataset):
    """data_loader.py:90-157: comp(+1) u sim(-1) pairs, shuffled, 80/10/10 split."""

    def __init__(self, bpg: BehaviorProductGraph, config, mode: str = "train"):
        self.bpg = bpg
        self.config = config
        self.mode = mode
        self.logger = logging.getLogger(__name__)
        self.pairs = self._create_product_pairs()
        self.type_to_idx = {t: i for i, t in enumerate(bpg.get_all_types())}
        self.idx_to_type = {i: t for t, i in self.type_to_idx.items()}
        self.logger.info(f"Created {mode} complementary dataset with {len(self.pairs)} pairs")

    def _create_product_pairs(self) -> List[Tuple[str, str, int]]:
        all_pairs = [(s, t, 1) for s, t in self.bpg.complementary_pairs]
        all_pairs.extend((s, t, -1) for s, t in self.bpg.similarity_pairs)
        random.shuffle(all_pairs)
        total = len(all_pairs)
        if self.mode == "train":
            return all_pairs[: int(0.8 * total)]
        if self.mode == "val":
            return all_pairs[int(0.8 * total): int(0.9 * total)]
        return all_pairs[int(0.9 * total):]

    def __len__(self) -> int:
        return len(self.pairs)

    def __getitem__(self, idx: int) -> Dict[str, torch.Tensor]:
        query_id, target_id, label = self.pairs[idx]
        nodes = self.bpg.nodes
        query_type = self.type_to_idx[nodes[query_id]["type"]]
        target_type = self.type_to_idx[nodes[target_id]["type"]]
        query_features = nodes[query_id]["features"].clone().detach()
        target_features = nodes[target_id]["features"].clone().detach()
        return {
            "query_ids": query_id,
            "query_features": query_features,
            "target_features": target_features,
            "query_types": torch.tensor(query_type),
            "positive_types": torch.tensor([target_type if label == 1 else 0]),
            "negative_types": torch.tensor([target_type if label == -1 else (target_type + 1) % len(self.type_to_idx)]),
            "positive_items": target_features if label == 1 else torch.randn_like(target_features),
            "negative_items": target_features if label == -1 else torch.randn_like(target_features),
            "label": torch.tensor(label),
        }


def collate_fn(batch: List[Dict]) -> Dict:
    """data_loader.py:171-206: id lists stay lists, neighbour features are zero-padded to the batch
    maximum (samples without neighbours get one zero row), other tensors are stacked."""
    batch_dict = defaultdict(list)
    for sample in batch:
        for key, value in sample.items():
            batch_dict[key].append(value)
    if "anchor_neighbors" in batch_dict and len(batch_dict["anchor_neighbors"]) != len(batch):
        # samples without the key were skipped by the loop above; restore alignment with explicit Nones
        batch_dict["anchor_neighbors"] = [s.get("anchor_neighbors") for s in batch]
    result = {}
    for key, values in batch_dict.items():
        if key in ("anchor_ids", "positive_id", "negative_ids", "query_ids"):
            result[key] = values
        elif key == "anchor_neighbors" and any(v is not None for v in values):
            width = next(v for v in values if v is not None).size(1)
            max_neighbors = max(v.size(0) for v in values if v is not None)
            padded = []
            for v in values:
                if v is None:
                    v = torch.zeros(1, width)
                if v.size(0) < max_neighbors:
                    v = torch.cat([v, torch.zeros(max_neighbors - v.size(0), v.size(1))], dim=0)
                padded.append(v)
            result[key] = torch.stack(padded)
        elif isinstance(values[0], torch.Tensor):
            result[key] = torch.stack(values)
        else:
            result[key] = values
    return result


class GraphTripletSampler:
    """CSR-native triplet batches on the device.

    Built from a finalized BehaviorProductGraph: similarity pairs (Bcv n Bpv) - Bcp come from the set
    kernels as sorted keys, so the anchor's similar set is one CSR row.  ``sample(batch, seed)`` returns
    (anchor [B], positive [B], negatives [B, K]) int64 index tensors into the node table."""

    def __init__(self, bpg: BehaviorProductGraph, k_neg: int = 5):
        bpg.finalize()
        self.num_nodes = bpg.num_nodes
        self.k_neg = k_neg
        keys = bpg.similarity_keys()
        if keys.numel() == 0:
            raise ValueError("No similarity pairs found in BPG")
        self.anchor, self.positive = ops.unpack_keys(keys)          # int32, sorted by (anchor, positive)
        self.sim_rowptr, self.sim_col = ops.csr_from_sorted_keys(keys, self.num_nodes)
        self.device = keys.device
        # pc_sample_negatives pads with -1 when an anchor has fewer than k_neg eligible products; sample() / epoch() hand
        # their negatives to the indexed triplet loss, which would read table[-1]: refuse such graphs there (checked once)
        max_similar = int((self.sim_rowptr[1:] - self.sim_rowptr[:-1]).max().item())
        self.always_k = self.num_nodes - 1 - max_similar >= k_neg

    def __len__(self) -> int:
        return self.anchor.numel()

    def negatives_for(self, anchors: torch.Tensor, seed: int) -> torch.Tensor:
        anchors = anchors.to(self.device, torch.int32).contiguous()
        out = torch.empty(anchors.numel(), self.k_neg, dtype=torch.int32, device=self.device)
        call("pc_sample_negatives", dev(anchors, torch.int32, "anchor"), dev(self.sim_rowptr, torch.int64, "sim_rowptr"),
             dev(self.sim_col, torch.int32, "sim_col"), anchors.numel(), self.num_nodes, self.k_neg, int(seed) & (2 ** 64 - 1),
             dev(out, torch.int32, "out"), stream())
        return out

    def _require_k(self) -> None:
        if not self.always_k:
            raise ValueError(f"GraphTripletSampler: some anchor has fewer than {self.k_neg} eligible negatives "
                             f"({self.num_nodes} products); use negatives_for() and mask the -1 padding")

    def sample(self, batch_size: int, seed: int):
        self._require_k()
        g = torch.Generator(device=self.device).manual_seed(int(seed))
        pick = torch.randint(0, len(self), (batch_size,), generator=g, device=self.device)
        a, p = self.anchor[pick], self.positive[pick]
        n = self.negatives_for(a, seed)
        return a.to(torch.int64), p.to(torch.int64), n.to(torch.int64)

    def epoch(self, batch_size: int, seed: int):
        """One pass over all similarity pairs in a seeded random order (the reference's shuffle=True loader)."""
        self._require_k()
        g = torch.Generator(device=self.device).manual_seed(int(seed))
        perm = torch.randperm(len(self), generator=g, device=self.device)
        for i in range(0, len(self), batch_size):
            pick = perm[i: i + batch_size]
            a, p = self.anchor[pick], self.positive[pick]
            yield a.to(torch.int64), p.to(torch.int64), self.negatives_for(a, seed * 1_000_003 + i).to(torch.int64)

    def neighborhood_batches(self, batch_size: int, seed: int, csr: ops.CSRGraph):
        """epoch(batch_size, seed)'s triplets (same order, same negatives) as TripletBatch with each anchor's co-view
        neighbour offsets into `csr` (Product2Vec.triplet_loss_graph).  The anchors' degrees are taken in permutation order
        and summed once for the whole epoch; every batch's neighbour total comes back to the host in ONE read, before the
        first batch, so no batch of a graph without hub rows synchronises (ops.triplet_batch_rows)."""
        self._require_k()
        if csr.n_rows != self.num_nodes:
            raise ValueError(f"neighborhood_batches: the CSR has {csr.n_rows} rows for {self.num_nodes} products")
        g = torch.Generator(device=self.device).manual_seed(int(seed))
        perm = torch.randperm(len(self), generator=g, device=self.device)
        anchors = self.anchor[perm].to(torch.int64)
        cum = torch.zeros(len(self) + 1, dtype=torch.int64, device=self.device)
        cum[1:] = torch.cumsum(csr.rowptr[anchors + 1] - csr.rowptr[anchors], 0)
        starts = range(0, len(self), batch_size)
        bounds = torch.cat([cum[:-1:batch_size], cum[-1:]])
        totals = (bounds[1:] - bounds[:-1]).tolist()                       # the epoch's one host read
        csr.hub_split()               # whether batch graphs split hub rows: one read per graph, cached on the CSR
        for i, n_nbr in zip(starts, totals):
            a = anchors[i: i + batch_size]
            yield TripletBatch(a, self.positive[perm[i: i + batch_size]].to(torch.int64),
                               self.negatives_for(a, seed * 1_000_003 + i).to(torch.int64),
                               cum[i: i + a.numel() + 1] - cum[i], n_nbr)


class TripletBatch(NamedTuple):
    """One graph-native triplet batch: int64 index tensors on the device - anchor [B], positive [B], negatives [B, K] -
    and nbr_ptr int64 [B + 1], the prefix sum of the anchors' co-view degrees, with n_nbr = nbr_ptr[B] on the host."""
    anchor: torch.Tensor
    positive: torch.Tensor
    negatives: torch.Tensor
    nbr_ptr: torch.Tensor
    n_nbr: int

    @classmethod
    def build(cls, csr: ops.CSRGraph, anchor: torch.Tensor, positive: torch.Tensor, negatives: torch.Tensor) -> "TripletBatch":
        """A batch of caller-chosen triplets (one host read: the neighbour total)."""
        anchor = anchor.reshape(-1).to(csr.rowptr.device, torch.int64).contiguous()
        positive = positive.reshape(-1).to(anchor.device, torch.int64).contiguous()
        negatives = negatives.reshape(anchor.numel(), -1).to(anchor.device, torch.int64).contiguous()
        nbr_ptr = torch.zeros(anchor.numel() + 1, dtype=torch.int64, device=anchor.device)
        nbr_ptr[1:] = torch.cumsum(csr.rowptr[anchor + 1] - csr.rowptr[anchor], 0)
        return cls(anchor, positive, negatives, nbr_ptr, int(nbr_ptr[-1].item()))
