#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ by running the REAL reference.

Needs a checkout of the reference project:

    python tests/golden/make_golden.py <path to the reference checkout>

The reference is imported from a throw-away temporary copy (its Config() mkdirs next to its
own sources, and Python would write __pycache__ there).  Config() is never instantiated; a
duck-typed namespace with the same attributes is used instead.  Seeds: random.seed(0),
torch.manual_seed(0), PYTHONHASHSEED irrelevant (every set is sorted before it is stored).

Fixtures (all float32 / int, a few hundred KB in total):
  p2v_module.npz  Product2Vec state_dict + inputs -> eval / train forward, BN running stats,
                  triplet loss and every parameter gradient (DROPOUT=0); weight-matrix gradients
                  as every GRAD_STRIDE-th element of the flattened matrix (tests/conftest.py golden_grad).
  p2v_graph.npz   small BPG + features -> generate_all_embeddings().
  bpg_c1.npz      the default synthetic BPG (config C1): edge sets, similarity /
                  complementary pairs, set helpers, neighbour samples, types.
  pcomp.npz       PCompanion (NUM_TYPES=40) forward outputs, loss, gradients.
  metrics.npz     Metrics.hit_at_k / evaluate_model-style in-batch scoring.
"""
import os
import random
import shutil
import sys
import tempfile
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GRAD_STRIDE = 7   # coprime with every row length (128, 256): the sample covers every row and column


def import_reference(ref_src):
    tmp = tempfile.mkdtemp(prefix="pc_ref_")
    dst = os.path.join(tmp, "ref")
    def skip(d, names):  # top-level models/ holds only checkpoints; src/models is needed
        return [n for n in names if n in (".git", "__pycache__") or (d == ref_src and n == "models")]
    shutil.copytree(ref_src, dst, ignore=skip)
    sys.path.insert(0, dst)
    sys.dont_write_bytecode = True
    return dst


def make_cfg(**over):
    cfg = SimpleNamespace(PRODUCT_EMB_DIM=128, TYPE_EMB_DIM=64, HIDDEN_SIZE=256, NUM_ATTENTION_HEADS=4,
                          DROPOUT=0.0, MARGIN=1.0, ALPHA=0.8, NUM_COMP_TYPES=3, NUM_TYPES=40,
                          DEVICE=torch.device("cpu"))
    for k, v in over.items():
        setattr(cfg, k, v)
    return cfg


def sd_to_np(sd, prefix="sd/"):
    return {prefix + k: v.detach().cpu().numpy().copy() for k, v in sd.items()}


def golden_p2v_module():
    from src.models.product2vec import Product2Vec
    import torch.nn.functional as F
    torch.manual_seed(0)
    cfg = make_cfg()
    m = Product2Vec(cfg)
    with torch.no_grad():  # non-trivial BN affine + running stats
        m.ffn[1].weight.uniform_(0.5, 1.5)
        m.ffn[1].bias.uniform_(-0.3, 0.3)
        m.ffn[1].running_mean.uniform_(-0.2, 0.2)
        m.ffn[1].running_var.uniform_(0.6, 1.4)
    out = sd_to_np(m.state_dict())
    B, N, K = 6, 5, 5
    anchor, positive = torch.randn(B, 128), torch.randn(B, 128)
    negative, nbrs = torch.randn(B, K, 128), torch.randn(B, N, 128)
    nbrs[1, 3:] = 0.0  # collate_fn-style zero padding is attended (SURVEY fact 3)
    out.update(anchor=anchor.numpy(), positive=positive.numpy(), negative=negative.numpy(), neighbors=nbrs.numpy())
    m.eval()
    with torch.no_grad():
        out["eval_forward_nbrs"] = m(anchor, nbrs).numpy()
        out["eval_forward_plain"] = m(anchor).numpy()
        out["eval_forward_neg3d"] = m(negative).numpy()
        out["eval_forward_1d"] = m(anchor[0], nbrs[0]).numpy()        # generate_all_embeddings shape
        out["eval_initial_1d"] = m.get_initial_embedding(anchor[0]).numpy()
    # one training step's forward/backward exactly as product2vec.py:132-158 (dropout 0)
    m.train()
    a = m(anchor, nbrs)
    p = m(positive)
    n = m(negative)
    dpos = F.pairwise_distance(a, p)
    dneg = torch.mean(F.pairwise_distance(a.unsqueeze(1).expand(-1, n.size(1), -1), n, p=2), dim=1)
    loss = F.relu(cfg.MARGIN - dpos + dneg).mean()
    loss.backward()
    out["train_anchor_emb"] = a.detach().numpy()
    out["train_positive_emb"] = p.detach().numpy()
    out["train_negative_emb"] = n.detach().numpy()
    out["train_loss"] = loss.detach().numpy()
    for k, v in m.named_parameters():
        gk = v.grad.numpy()
        out["grad/" + k] = gk.reshape(-1)[::GRAD_STRIDE].copy() if gk.ndim > 1 else gk.copy()
    out["grad_stride"] = np.array(GRAD_STRIDE, np.int64)
    out["train_running_mean"] = m.ffn[1].running_mean.numpy().copy()
    out["train_running_var"] = m.ffn[1].running_var.numpy().copy()
    out["train_num_batches_tracked"] = m.ffn[1].num_batches_tracked.numpy().copy()
    # attention-only gradient check: d(out)/d(query, key_value) through nn.MultiheadAttention
    m.eval()
    q = torch.randn(4, 128, requires_grad=True)
    kv = torch.randn(4, 7, 128, requires_grad=True)
    w = torch.randn(4, 128)
    o = m.apply_attention(q, kv)
    (o * w).sum().backward()
    out.update(attn_q=q.detach().numpy(), attn_kv=kv.detach().numpy(), attn_w=w.numpy(),
               attn_out=o.detach().numpy(), attn_dq=q.grad.numpy().copy(), attn_dkv=kv.grad.numpy().copy())
    np.savez_compressed(os.path.join(HERE, "p2v_module.npz"), **out)


def golden_p2v_graph():
    from src.models.product2vec import Product2Vec
    from src.data.bpg import BehaviorProductGraph
    torch.manual_seed(1)
    random.seed(1)
    cfg = make_cfg()
    m = Product2Vec(cfg)
    with torch.no_grad():
        m.ffn[1].running_mean.uniform_(-0.2, 0.2)
        m.ffn[1].running_var.uniform_(0.6, 1.4)
    n = 48
    bpg = BehaviorProductGraph()
    feats = torch.randn(n, 128)
    ids = [f"P{str(i).zfill(6)}" for i in range(n)]
    for i, pid in enumerate(ids):
        bpg.add_node(pid, {"features": feats[i], "type": f"type_{i % 5}"})
    src, dst = [], []
    for i in range(n):
        for j in range(i + 1, n):
            if random.random() < 0.15 and i % 7 != 3:      # nodes with i%7==3 keep ffn(x)
                bpg.add_edge(ids[i], ids[j], "co_view")
                src.append(i); dst.append(j)
    bpg.add_edge(ids[0], ids[1], "co_view"); src.append(0); dst.append(1)   # duplicate insert
    bpg.add_edge(ids[0], ids[2], "no_such_type")                            # silently dropped
    emb = m.generate_all_embeddings(bpg)
    out = sd_to_np(m.state_dict())
    out.update(features=feats.numpy(), src=np.array(src, np.int32), dst=np.array(dst, np.int32),
               embeddings=torch.stack([emb[p] for p in ids]).numpy())
    np.savez_compressed(os.path.join(HERE, "p2v_graph.npz"), **out)


def golden_bpg_c1():
    from src.data.synthetic_data import SyntheticDataGenerator
    random.seed(0)
    torch.manual_seed(0)
    cfg = make_cfg()
    gen = SyntheticDataGenerator(cfg)
    bpg = gen.generate_unified_bpg()
    ids = list(bpg.nodes.keys())
    idx = {p: i for i, p in enumerate(ids)}
    out = {}
    for t, es in bpg.edges.items():
        arr = np.array(sorted((idx[s], idx[d]) for s, d in es), dtype=np.int32).reshape(-1, 2)
        out["edges/" + t] = arr
        # insertion-like order with duplicates re-added, to exercise dedup on the device
    out["similarity_pairs"] = np.array(sorted((idx[s], idx[d]) for s, d in bpg.similarity_pairs), np.int32)
    out["complementary_pairs"] = np.array(sorted((idx[s], idx[d]) for s, d in bpg.complementary_pairs), np.int32)
    out["exclusive_co_purchase"] = np.array(sorted((idx[s], idx[d]) for s, d, _ in bpg.get_exclusive_co_purchase_pairs()), np.int32)
    out["co_view_intersection"] = np.array(sorted((idx[s], idx[d]) for s, d, _ in bpg.get_co_view_intersection_pairs()), np.int32)
    types = sorted(bpg.get_all_types())
    tix = {t: i for i, t in enumerate(types)}
    out["type_names"] = np.array(types)
    out["type_id"] = np.array([tix[bpg.nodes[p]["type"]] for p in ids], np.int32)
    cats = ['electronics', 'clothing', 'sports', 'home', 'office']
    out["category"] = np.array([cats.index(bpg.nodes[p]["category"]) for p in ids], np.int32)
    probe = [0, 1, 17, 500, 998, 999]
    out["probe_nodes"] = np.array(probe, np.int32)
    for p in probe:
        out[f"nbr_cv/{p}"] = np.array(sorted(idx[x] for x in bpg.get_neighbors(ids[p], "co_view")), np.int32)
        out[f"nbr_all/{p}"] = np.array(sorted(idx[x] for x in bpg.get_neighbors(ids[p])), np.int32)
    out["products_of_type0"] = np.array([idx[p] for p in bpg.get_products_by_type(types[0])], np.int32)
    np.savez_compressed(os.path.join(HERE, "bpg_c1.npz"), **out)


def golden_pcomp():
    from src.models.p_companion import PCompanion
    torch.manual_seed(2)
    cfg = make_cfg(NUM_TYPES=40)
    P, B = 64, 12
    table = {f"P{str(i).zfill(6)}": torch.randn(128) for i in range(P)}
    m = PCompanion(cfg, table)
    qidx = torch.randint(0, P, (B,))
    batch = {
        "query_ids": [f"P{str(int(i)).zfill(6)}" for i in qidx],
        "query_types": torch.randint(0, cfg.NUM_TYPES, (B,)),
        "positive_types": torch.randint(0, cfg.NUM_TYPES, (B, 1)),
        "negative_types": torch.randint(0, cfg.NUM_TYPES, (B, 1)),
        "positive_items": torch.randn(B, 128),
        "negative_items": torch.randn(B, 128),
        "target_features": torch.randn(B, 128),
    }
    m.train()  # DROPOUT = 0 -> identical to eval, but exercises the grad path
    o = m(batch)
    loss = m.compute_loss(batch, o)
    loss.backward()
    out = sd_to_np(m.state_dict())
    out["query_idx"] = qidx.numpy()
    for k in ("query_types", "positive_types", "negative_types", "positive_items", "negative_items", "target_features"):
        out["batch/" + k] = batch[k].numpy()
    out["projected_embeddings"] = o["projected_embeddings"].detach().numpy()
    out["complementary_types"] = o["complementary_types"].numpy()
    out["type_similarities"] = o["type_similarities"].detach().numpy()
    out["loss"] = loss.detach().numpy()
    out["type_loss"] = m._compute_type_loss(o["type_similarities"], batch["positive_types"].squeeze(-1),
                                            batch["negative_types"].squeeze(-1)).detach().numpy()
    out["item_loss"] = m._compute_item_loss(o["projected_embeddings"], batch["positive_items"],
                                            batch["negative_items"]).detach().numpy()
    for k, v in m.named_parameters():
        if v.grad is not None:
            out["grad/" + k] = v.grad.numpy().copy()
    # evaluate_model-style in-batch scoring, metrics.py:89-100
    from src.utils.metrics import Metrics
    sims = torch.matmul(o["projected_embeddings"].detach().view(-1, 128), batch["target_features"].T)
    out["eval_sims"] = sims.numpy()
    for k in (1, 3, 10):
        out[f"hit@{k}"] = np.array(Metrics.hit_at_k(sims, torch.arange(sims.size(0)), k))
    out["type_diversity"] = np.array(Metrics.type_diversity(o["complementary_types"]))
    out["mean_relevance"] = np.array(Metrics.mean_relevance(o["projected_embeddings"].detach(), batch["positive_items"]))
    np.savez_compressed(os.path.join(HERE, "pcomp.npz"), **out)


def golden_metrics():
    from src.utils.metrics import Metrics
    torch.manual_seed(3)
    pred = torch.randn(50, 37)
    gt = torch.randint(0, 37, (50,))
    out = {"pred": pred.numpy(), "gt": gt.numpy()}
    for k in (1, 3, 10, 60):
        out[f"hit@{k}"] = np.array(Metrics.hit_at_k(pred, gt, k))
    # retrieval as inference.py:93-113 does it: per-type filter, matmul, topk
    P, T, R, K = 400, 7, 9, 10
    catalog = torch.randn(P, 128)
    type_id = torch.randint(0, T, (P,))
    q = torch.randn(R, 128)
    row_type = torch.randint(0, T, (R,))
    idx = np.full((R, K), -1, np.int64)
    sc = np.full((R, K), -np.inf, np.float32)
    for r in range(R):
        members = [p for p in range(P) if int(type_id[p]) == int(row_type[r])]     # get_products_by_type
        emb = torch.stack([catalog[p] for p in members])
        s = torch.matmul(q[r].unsqueeze(0), emb.T)[0]
        ts, ti = torch.topk(s, k=min(K, len(members)))
        idx[r, :len(ti)] = [members[i] for i in ti.numpy()]
        sc[r, :len(ti)] = ts.numpy()
    # collate_fn (data_loader.py:171-206) on samples with ragged neighbour lists
    from src.data.data_loader import collate_fn
    samples = []
    for i, nn in enumerate((2, 5, 1, 3)):
        samples.append({"anchor_ids": f"A{i}", "anchor": torch.randn(8), "positive": torch.randn(8), "negative": torch.randn(5, 8),
                        "positive_id": f"P{i}", "negative_ids": [f"N{i}{j}" for j in range(5)], "anchor_neighbors": torch.randn(nn, 8)})
    col = collate_fn(samples)
    for i, smp in enumerate(samples):
        for k in ("anchor", "positive", "negative", "anchor_neighbors"):
            out[f"collate_in/{i}/{k}"] = smp[k].numpy()
    for k in ("anchor", "positive", "negative", "anchor_neighbors"):
        out["collate_out/" + k] = col[k].numpy()
    out["collate_out/anchor_ids"] = np.array(col["anchor_ids"])
    out.update(catalog=catalog.numpy(), type_id=type_id.numpy().astype(np.int32), q=q.numpy(),
               row_type=row_type.numpy().astype(np.int32), topk_idx=idx, topk_score=sc)
    np.savez_compressed(os.path.join(HERE, "metrics.npz"), **out)


if __name__ == "__main__":
    import_reference(os.path.abspath(sys.argv[1]))
    golden_p2v_module()
    golden_p2v_graph()
    golden_bpg_c1()
    golden_pcomp()
    golden_metrics()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))
