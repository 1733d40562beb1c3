"""Product2Vec on the B200 kernels.

Drop-in for /root/reference/src/models/product2vec.py: same constructor, method names,
argument meaning, error behaviour and ``state_dict`` layout (``ffn.{0,1,3,5}.*``,
``attention.in_proj_weight/bias``, ``attention.out_proj.*``), so ``scripts/pretrain_product2vec.py``
and shipped ``product2vec.pth`` checkpoints work unchanged.  ``nn.MultiheadAttention`` is kept
only as the parameter container (identical initialisation and key names); its forward is never
called - the attention core runs in pcompanion_b200/csrc/gat.cu over a CSR:

* dense drop-in ``forward(features, neighbors[B, N, D])``: the padded neighbour tensor is viewed
  as a regular CSR (row i -> rows i*N..(i+1)*N), so zero-padded rows are attended exactly as the
  reference does (no key_padding_mask, SURVEY fact 3) and BatchNorm sees the same B*N rows;
* graph API ``forward_graph(x, csr)``: FFN and K|V projection once per node, attention over the
  BPG's co-view CSR (the formulation that scales to 200 M edges, SURVEY H2);
* graph-native training ``triplet_loss_graph`` / ``train_model_graph``: the reference's mini-batch step
  (four FFN calls with their own BatchNorm statistics, attention for the anchors only) on rows gathered
  on the device from index tensors - no host feature copies, no padding, no Python per sample.
"""
from __future__ import annotations

import logging
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import ops
from .dense import ffn_forward, linear
from .fused import fused_supported, p2v_graph_layer


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"Product2Vec.{what}: input is on {t.device}; pcompanion_b200 runs on CUDA only "
                           "(no CPU fallback) - move the module and its inputs to the GPU")


class Product2Vec(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        d, hid = config.PRODUCT_EMB_DIM, config.HIDDEN_SIZE
        # same layer order / indices as product2vec.py:14-21 -> same state_dict keys and init order
        self.ffn = nn.Sequential(
            nn.Linear(d, hid), nn.BatchNorm1d(hid), nn.Tanh(),
            nn.Linear(hid, hid), nn.Tanh(),
            nn.Linear(hid, d),
        )
        # parameter container only (product2vec.py:24-29)
        self.attention = nn.MultiheadAttention(embed_dim=d, num_heads=config.NUM_ATTENTION_HEADS,
                                               dropout=config.DROPOUT, batch_first=True)
        self.heads = config.NUM_ATTENTION_HEADS
        self.attn_dropout = float(config.DROPOUT)

    # ------------------------------------------------------------------ pieces
    def _ffn_rows(self, rows: torch.Tensor) -> torch.Tensor:
        return ffn_forward(self.ffn, rows, self.training)

    def _dropout_args(self):
        if self.training and self.attn_dropout > 0.0:
            return self.attn_dropout, int(torch.randint(0, 2 ** 62, (1,)).item())
        return 0.0, 0

    def _attend(self, h_query: torch.Tensor, h_kv: torch.Tensor, graph: ops.CSRGraph) -> torch.Tensor:
        """in-proj (Q from the query rows, K|V from the source rows) -> CSR attention -> out-proj."""
        w, b = self.attention.in_proj_weight, self.attention.in_proj_bias
        e = w.shape[1]
        q = linear(h_query, w[:e], b[:e])
        kv = linear(h_kv, w[e:], b[e:])
        p, seed = self._dropout_args()
        o = ops.gat_attention(q, kv, graph, self.heads, p, seed)
        return linear(o, self.attention.out_proj.weight, self.attention.out_proj.bias)

    # ------------------------------------------------------------------ reference API
    def get_initial_embedding(self, features: torch.Tensor) -> torch.Tensor:
        """FFN embedding; 1-D / 2-D / 3-D inputs as product2vec.py:31-46."""
        _require_cuda(features, "get_initial_embedding")
        if features.dim() == 1:
            return self._ffn_rows(features.unsqueeze(0)).squeeze(0)
        if features.dim() == 2:
            return self._ffn_rows(features)
        if features.dim() == 3:
            b, n, d = features.shape
            return self._ffn_rows(features.reshape(-1, d)).reshape(b, n, -1)
        raise ValueError(f"Unexpected input dimension: {features.dim()}")

    def apply_attention(self, query: torch.Tensor, key_value: torch.Tensor) -> torch.Tensor:
        """Multi-head attention of every query row over its own neighbour rows (product2vec.py:48-68)."""
        _require_cuda(query, "apply_attention")
        q = query
        if q.dim() == 1:
            q = q.unsqueeze(0)
        elif q.dim() == 3:
            if q.size(1) != 1:
                raise ValueError("apply_attention: only one query position per row is supported")
            q = q.squeeze(1)
        kv = key_value.unsqueeze(0) if key_value.dim() == 2 else key_value
        b, n, d = kv.shape
        if q.size(0) != b:
            raise ValueError(f"apply_attention: {q.size(0)} query rows vs {b} neighbour lists")
        out = self._attend(q, kv.reshape(b * n, d), ops.regular_graph(b, n, q.device))
        if query.dim() == 1:
            return out.squeeze(0)
        if query.dim() == 3:
            return out.unsqueeze(1)
        return out

    def forward(self, features: torch.Tensor, neighbors: Optional[torch.Tensor] = None) -> torch.Tensor:
        embeddings = self.get_initial_embedding(features)
        if neighbors is not None and neighbors.size(0) > 0:
            neighbor_embeddings = self.get_initial_embedding(neighbors)
            embeddings = self.apply_attention(embeddings, neighbor_embeddings)
        return embeddings

    # ------------------------------------------------------------------ graph API
    def forward_graph(self, x: torch.Tensor, graph: ops.CSRGraph, double_ffn_query: bool = False) -> torch.Tensor:
        """Embeddings of all nodes from node features x [N, D] and a CSR: FFN per node, K|V per node,
        attention over the CSR, out-proj; nodes without out-neighbours keep ffn(x)
        (product2vec.py:76 / :98).  double_ffn_query=True is generate_all_embeddings' ffn(ffn(x)) query."""
        _require_cuda(x, "forward_graph")
        if not double_ffn_query and fused_supported(self, x):
            return p2v_graph_layer(self, x, graph)          # one autograd node, every row-sized op in a C-ABI kernel
        h = self._ffn_rows(x)
        hq = self._ffn_rows(h) if double_ffn_query else h
        if not torch.is_grad_enabled() and fused_supported(self, x):
            # inference (generate_all_embeddings): raw kernels, the "rows without neighbours keep ffn(x)" select in the
            # out-projection's epilogue
            w, b = self.attention.in_proj_weight, self.attention.in_proj_bias
            q = ops.linear_tc(hq, w[:128].contiguous(), b[:128].contiguous())
            kv = ops.linear_tc(h, w[128:].contiguous(), b[128:].contiguous())
            p, seed = self._dropout_args()
            o, _ = ops.gat_fwd_raw(q, kv, graph, self.heads, p, seed)
            return ops.linear_tc(o, self.attention.out_proj.weight.contiguous(), self.attention.out_proj.bias,
                                 ops.EPI_BIAS_SELECT, aux=h, rowptr=graph.rowptr)
        out = self._attend(hq, h, graph)
        has_nbr = (graph.rowptr[1:] > graph.rowptr[:-1]).unsqueeze(1)
        return torch.where(has_nbr, out, h)

    def embed_graph(self, bpg) -> torch.Tensor:
        """Batched generate_all_embeddings: one full-graph pass -> dense [P, D] table on the device."""
        was_training = self.training
        self.eval()
        try:
            with torch.no_grad():
                dev = next(self.parameters()).device
                return self.forward_graph(bpg.features.to(dev), bpg.csr("co_view"), double_ffn_query=True)
        finally:
            self.train(was_training)

    def generate_all_embeddings(self, bpg) -> Dict[str, torch.Tensor]:
        """product2vec.py:83-111 - same result (Dict[product_id, CPU tensor] in bpg.nodes order),
        computed in one graph pass instead of per-node launches and O(E) neighbour scans."""
        self.eval()
        bpg.finalize()
        table = self.embed_graph(bpg).cpu()
        return {pid: table[i] for i, pid in enumerate(bpg.nodes.keys())}

    def triplet_loss(self, anchor_emb, positive_emb, negative_emb) -> torch.Tensor:
        """The loss block of product2vec.py:137-154 as one fused kernel."""
        return ops.triplet_hinge(anchor_emb, positive_emb, negative_emb, self.config.MARGIN)

    def triplet_loss_indexed(self, table, anchor_idx, positive_idx, negative_idx) -> torch.Tensor:
        """Same loss on rows of a full-graph embedding table picked by index (graph training: the batch is index
        tensors into forward_graph's output instead of padded feature copies, SURVEY 8f.1)."""
        return ops.triplet_hinge_indexed(table, anchor_idx, positive_idx, negative_idx, self.config.MARGIN)

    def triplet_loss_graph(self, x: torch.Tensor, csr: ops.CSRGraph, batch) -> torch.Tensor:
        """The loss of one training batch of product2vec.py:132-154 from index tensors (a data.TripletBatch) into the
        feature table x [N, D] and its co-view CSR.  The rows are gathered on the device in one launch, then the four FFN
        calls run in the reference's order - anchors, neighbour rows, positives, negatives - each with the batch statistics
        of its own rows and its own running-statistics update.  Anchors attend over exactly their co-view neighbours;
        anchors without any keep ffn(x) (forward_graph, generate_all_embeddings), and a batch without neighbour rows
        skips the neighbour FFN and the attention.  Unlike the drop-in path there are no zero-padding rows: the two agree
        bit for bit when every anchor of the batch has the same degree >= 1.  x is not differentiated."""
        _require_cuda(x, "triplet_loss_graph")
        a_rows, nbr_rows, p_rows, n_rows, graph = ops.triplet_batch_rows(
            x, csr, batch.anchor, batch.positive, batch.negatives, batch.nbr_ptr, batch.n_nbr)
        anchor_emb = self._ffn_rows(a_rows)
        if batch.n_nbr > 0:
            out = self._attend(anchor_emb, self._ffn_rows(nbr_rows), graph)
            has_nbr = (batch.nbr_ptr[1:] > batch.nbr_ptr[:-1]).unsqueeze(1)
            anchor_emb = torch.where(has_nbr, out, anchor_emb)
        positive_emb = self._ffn_rows(p_rows)
        negative_emb = self._ffn_rows(n_rows).view(batch.negatives.shape[0], batch.negatives.shape[1], -1)
        return self.triplet_loss(anchor_emb, positive_emb, negative_emb)

    def train_model_graph(self, bpg, optimizer, num_epochs=10, batch_size=None, seed=0, k_neg=5) -> Dict[str, torch.Tensor]:
        """train_model's loop without the host data path: batches come from GraphTripletSampler.neighborhood_batches
        over the BPG's similarity pairs (epoch e uses seed * 100_003 + e), each step is triplet_loss_graph, and the loss is
        summed on the device (one host read per epoch for the log line, one for the epoch's plan).  Same log line and
        return value as train_model.  batch_size defaults to config.BATCH_SIZE."""
        from .data import GraphTripletSampler
        device = self.config.DEVICE
        logger = logging.getLogger(__name__)
        self.to(device)
        bpg.finalize()
        sampler = GraphTripletSampler(bpg, k_neg=k_neg)
        csr = bpg.csr("co_view")
        x = bpg.features.to(device)
        batch_size = self.config.BATCH_SIZE if batch_size is None else int(batch_size)
        for epoch in range(num_epochs):
            self.train()
            total_loss = torch.zeros((), dtype=torch.float32, device=device)
            num_batches = 0
            for batch in sampler.neighborhood_batches(batch_size, seed * 100_003 + epoch, csr):
                loss = self.triplet_loss_graph(x, csr, batch)
                optimizer.zero_grad()
                loss.backward()
                optimizer.step()
                total_loss += loss.detach()
                num_batches += 1
            logger.info(f"Epoch {epoch + 1}/{num_epochs}, Loss: {total_loss.item() / max(num_batches, 1):.4f}")
        self.eval()
        return self.generate_all_embeddings(bpg)

    def train_model(self, train_loader, optimizer, num_epochs=10) -> Dict[str, torch.Tensor]:
        """Training loop of product2vec.py:113-170 (same batch keys, same return value)."""
        device = self.config.DEVICE
        logger = logging.getLogger(__name__)
        self.to(device)
        for epoch in range(num_epochs):
            self.train()
            total_loss, num_batches = 0.0, 0
            for batch in train_loader:
                batch = {k: v.to(device) if isinstance(v, torch.Tensor) else v for k, v in batch.items()}
                anchor_emb = self(batch["anchor"], batch.get("anchor_neighbors"))
                positive_emb = self(batch["positive"])
                negative_emb = self(batch["negative"])
                loss = self.triplet_loss(anchor_emb, positive_emb, negative_emb)
                optimizer.zero_grad()
                loss.backward()
                optimizer.step()
                total_loss += loss.item()
                num_batches += 1
            logger.info(f"Epoch {epoch + 1}/{num_epochs}, Loss: {total_loss / max(num_batches, 1):.4f}")
        self.eval()
        return self.generate_all_embeddings(train_loader.dataset.bpg)
