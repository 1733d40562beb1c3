"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares, the
ctypes prototypes cover the header, the host classes keep the reference's surface and refuse to
run without CUDA (no compute is launched here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, state_dict_from

HEADER = os.path.join(ROOT, "include", "pcompanion_b200.h")


def header_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pc_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol():
    from pcompanion_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = header_functions()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/pcompanion_b200.h but not exported"
    assert lib.pc_abi_version() == 1


def test_ctypes_prototypes_cover_the_header_exactly():
    from pcompanion_b200 import _lib
    assert sorted(_lib.PROTOTYPES) == header_functions()
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name, (_, args) in _lib.PROTOTYPES.items():
        m = re.search(r"\b" + name + r"\s*\(([^;]*)\)\s*;", src, flags=re.S)
        params = [p for p in m.group(1).split(",") if p.strip() and p.strip() != "void"]
        assert len(params) == len(args), f"{name}: header has {len(params)} parameters, ctypes binding {len(args)}"


def test_workspace_queries_need_no_gpu():
    from pcompanion_b200 import _lib
    assert _lib.LIB.pc_sort_keys_workspace_bytes(0) == 0
    assert _lib.LIB.pc_sort_keys_workspace_bytes(1_000_000) >= 8_000_000
    assert _lib.LIB.pc_compact_workspace_bytes(1_000_000) >= 8_000_000
    assert _lib.LIB.pc_topk_groups_workspace_bytes(10, 10, 1) == 0
    assert _lib.LIB.pc_topk_groups_workspace_bytes(10, 10, 4) == 10 * 4 * 10 * 16


def test_argument_errors_are_reported_without_a_gpu():
    from pcompanion_b200 import _lib
    rc = _lib.LIB.pc_gat_fwd(None, 128, None, None, None, 5, 3, 0.0, 0, None, None, None, None)
    assert rc != 0 and b"gat" in _lib.LIB.pc_last_error()
    with pytest.raises(RuntimeError, match="native call failed"):
        _lib.check(rc)
    assert _lib.LIB.pc_topk_merge(None, None, 4, 2, 64, None, None, None) != 0


def make_cfg(**over):
    from types import SimpleNamespace
    cfg = SimpleNamespace(PRODUCT_EMB_DIM=128, TYPE_EMB_DIM=64, HIDDEN_SIZE=256, NUM_ATTENTION_HEADS=4, DROPOUT=0.1,
                          MARGIN=1.0, ALPHA=0.8, NUM_COMP_TYPES=3, NUM_TYPES=40, DEVICE=torch.device("cpu"))
    for k, v in over.items():
        setattr(cfg, k, v)
    return cfg


def test_state_dict_layout_equals_the_reference():
    """Keys and shapes of the reference checkpoints (golden state_dicts come from the real modules)."""
    from pcompanion_b200 import PCompanion, Product2Vec
    g = load_golden("p2v_module.npz")
    ref = state_dict_from(g)
    m = Product2Vec(make_cfg())
    sd = m.state_dict()
    assert list(sd.keys()) == list(ref.keys())
    assert all(tuple(sd[k].shape) == ref[k].shape for k in ref)
    m.load_state_dict({k: torch.tensor(v) for k, v in ref.items()})
    gp = load_golden("pcomp.npz")
    refp = state_dict_from(gp)
    pm = PCompanion(make_cfg(), {f"P{i}": torch.zeros(128) for i in range(refp["product_embeddings.weight"].shape[0])})
    assert set(pm.state_dict().keys()) == set(refp.keys())
    assert all(tuple(pm.state_dict()[k].shape) == refp[k].shape for k in refp)
    assert not pm.product_embeddings.weight.requires_grad          # frozen, p_companion.py:26-29
    assert pm.product_to_idx["P3"] == 3


def test_same_seed_gives_the_reference_initialisation():
    """Same construction order as product2vec.py:14-29 -> torch.manual_seed(s) reproduces the
    reference's initial weights (the golden state_dict was drawn with seed 0 before BN edits)."""
    from pcompanion_b200 import Product2Vec
    g = load_golden("p2v_module.npz")
    torch.manual_seed(0)
    m = Product2Vec(make_cfg())
    for k in ("ffn.0.weight", "ffn.5.bias", "attention.in_proj_weight", "attention.out_proj.weight"):
        assert np.array_equal(m.state_dict()[k].numpy(), g["sd/" + k]), k


def test_cpu_inputs_are_refused_not_silently_computed():
    from pcompanion_b200 import PCompanion, Product2Vec, ops
    m = Product2Vec(make_cfg())
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(4, 128))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.get_initial_embedding(torch.zeros(128))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.pack_keys(torch.zeros(3, dtype=torch.int32), torch.zeros(3, dtype=torch.int32))
    pm = PCompanion(make_cfg(), torch.zeros(10, 128))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm({"query_ids": torch.zeros(2, dtype=torch.int64), "query_types": torch.zeros(2, dtype=torch.int64)})


def test_digit_mask_and_bpg_surface_without_device_work():
    from pcompanion_b200 import BehaviorProductGraph, ops
    assert ops.digit_mask_for(2) == 0x11 and ops.digit_mask_for(256) == 0x11 and ops.digit_mask_for(257) == 0x33
    assert ops.digit_mask_for(1_000_000) == 0x77 and ops.digit_mask_for(1 << 31) == 0xFF
    b = BehaviorProductGraph()
    b.add_node("a", {"type": "t0"}); b.add_node("b", {"type": "t1"})
    b.add_edge("a", "b", "co_view"); b.add_edge("a", "b", "co_view"); b.add_edge("a", "b", "nonsense")
    assert b.edges["co_view"] == {("a", "b")} and set(b.edges) == {"co_purchase", "co_view", "purchase_after_view"}
    assert b.get_all_types() == {"t0", "t1"}


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from pcompanion_b200 import _lib
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.NativeLibraryError, match="no CPU or PyTorch fallback"):
        _lib._load()


def test_collate_fn_matches_reference_golden():
    """collate_fn drop-in vs the real reference's output on ragged neighbour lists (data_loader.py:171-206)."""
    from pcompanion_b200 import collate_fn
    g = load_golden("metrics.npz")
    samples = []
    for i in range(4):
        samples.append({"anchor_ids": f"A{i}", "positive_id": f"P{i}", "negative_ids": [f"N{i}{j}" for j in range(5)],
                        **{k: torch.tensor(g[f"collate_in/{i}/{k}"]) for k in ("anchor", "positive", "negative", "anchor_neighbors")}})
    out = collate_fn(samples)
    for k in ("anchor", "positive", "negative", "anchor_neighbors"):
        assert np.array_equal(out[k].numpy(), g["collate_out/" + k]), k
    assert out["anchor_ids"] == g["collate_out/anchor_ids"].tolist()
    assert out["anchor_neighbors"].shape == (4, 5, 8) and float(out["anchor_neighbors"][2, 1:].abs().sum()) == 0.0
    assert out["negative_ids"][1] == [f"N1{j}" for j in range(5)]


def test_similarity_dataset_requires_pairs_like_reference():
    from pcompanion_b200 import BehaviorProductGraph, SimilarityDataset
    b = BehaviorProductGraph()
    b.similarity_pairs = []
    with pytest.raises(ValueError, match="No similarity pairs found in BPG"):
        SimilarityDataset(b, make_cfg())


def test_checkpoint_in_reference_layout_loads_into_the_drop_in_modules(tmp_path):
    """A checkpoint written in the layout of the reference's product2vec.pth (scripts/pretrain_product2vec.py:44-49:
    {'model_state_dict', 'embeddings', 'type_to_idx'}), filled from p2v_graph.npz: the real reference's state_dict, the
    embedding dict its generate_all_embeddings() returned for that model, and the graph's product types.  The
    state_dict loads strictly into Product2Vec, the embedding dict feeds PCompanion.__init__ as train.py:42-43 does."""
    from pcompanion_b200 import PCompanion, Product2Vec
    g = load_golden("p2v_graph.npz")
    n = g["embeddings"].shape[0]
    ids = [f"P{str(i).zfill(6)}" for i in range(n)]
    types = sorted({f"type_{i % 5}" for i in range(n)})                 # node types of the golden graph (make_golden.py)
    path = tmp_path / "product2vec.pth"
    torch.save({"model_state_dict": {k: torch.tensor(v) for k, v in state_dict_from(g).items()},
                "embeddings": {p: torch.tensor(e) for p, e in zip(ids, g["embeddings"])},
                "type_to_idx": {t: i for i, t in enumerate(types)}}, path)
    ck = torch.load(path, map_location="cpu", weights_only=True)
    m = Product2Vec(make_cfg())
    missing = m.load_state_dict(ck["model_state_dict"], strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    for k, v in m.state_dict().items():
        assert torch.equal(v, ck["model_state_dict"][k]), k
    emb = ck["embeddings"]
    pcm = PCompanion(make_cfg(), emb)
    ids = list(emb.keys())
    assert pcm.product_embeddings.weight.shape == (len(ids), 128) and not pcm.product_embeddings.weight.requires_grad
    assert pcm.product_to_idx[ids[0]] == 0 and pcm.product_to_idx[ids[-1]] == len(ids) - 1
    assert torch.equal(pcm.product_embeddings.weight[7], emb[ids[7]].float())


def test_scalable_generator_chain_equals_the_oracle_chain_on_shared_uniforms():
    """pcompanion_b200.synthetic.edge_chain (torch, O(E)) against oracle.bpg.edge_chain (numpy restatement of
    synthetic_data.py:101-128) on the same candidate pairs and the same uniforms: identical edge lists per type."""
    from oracle import bpg as obpg
    from pcompanion_b200.synthetic import edge_chain
    rng = np.random.default_rng(0)
    n, pairs = 5000, 200_000
    category = rng.integers(0, 5, n).astype(np.int32)
    a, b = rng.integers(0, n, pairs), rng.integers(0, n, pairs)
    keep = a != b
    src, dst = np.minimum(a, b)[keep].astype(np.int32), np.maximum(a, b)[keep].astype(np.int32)
    u = rng.random((3, src.size)).astype(np.float32)
    ours = edge_chain(torch.tensor(category), torch.tensor(src), torch.tensor(dst), torch.tensor(u[0]), torch.tensor(u[1]), torch.tensor(u[2]))
    ref = obpg.edge_chain(n, category, src, dst, u[0], u[1], u[2])
    for t in ("co_view", "purchase_after_view", "co_purchase"):
        s, d = ours[t]
        keys = (s.numpy().astype(np.int64) << 32) | d.numpy().astype(np.int64)
        assert np.array_equal(keys, np.asarray(ref[t]).astype(np.int64)), t
    assert 0.30 < ours["co_view"][0].numel() / src.size < 0.36          # 0.3 (x1.5 inside a category, 1/5 of the pairs)


def test_bench_reference_arm_prints_the_contract_line():
    """bench.py --impl reference: one JSON line with the contract's keys, timed on the host cores through the oracle port
    (the one place besides tests / smoke where oracle/ may be executed)."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "retrieval",
                          "--steps", "1", "--warmup", "0"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "topk_queries_per_sec" and line["unit"] == "queries/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["steps"] == 1
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
