"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden fixtures.

Integer / index results are compared bit-exactly; fp32 results within 1e-5 relative (stated per
test).  Run on the B200 box with ``pytest -m gpu``.
"""
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import golden_grad, load_golden, state_dict_from

pytestmark = pytest.mark.gpu

REL = 1e-5  # BASELINE.json north_star: "within 1e-5 relative in fp32"
# Gradients compared with the reference's OWN float32 gradients (golden fixtures written by the real reference): two fp32
# computations that are each within 1e-5 of the exact value can be 2e-5 apart.  profiles/r2_grad_error_probe.json
# (profiles/grad_error_probe.py) measures both sides against float64 autograd: CUDA path <= 5.1e-6, the reference's own
# float32 arithmetic <= 5.6e-6 on every tensor except the bias in front of BatchNorm (mathematically zero gradient).
REL_VS_FP32 = 2e-5


def dev():
    return torch.device("cuda:0")


def close(actual, ref, rel=REL, what="", atol=0.0):
    """|a - ref| <= rel * (|ref| + rms(ref)) + atol: 1e-5 relative, with the tensor's own scale as the
    floor for elements that cancel to ~0.  atol is only used for gradients that are mathematically
    zero (e.g. the bias in front of BatchNorm), where reference and CUDA path both hold rounding noise."""
    a = np.asarray(actual.detach().cpu().numpy() if torch.is_tensor(actual) else actual, np.float64)
    r = np.asarray(ref, np.float64)
    assert a.shape == r.shape, (what, a.shape, r.shape)
    scale = math.sqrt(float((r * r).mean())) if r.size else 0.0
    err = np.abs(a - r)
    bound = rel * (np.abs(r) + scale) + atol + 1e-30
    worst = float((err / bound).max()) if r.size else 0.0
    assert worst <= 1.0, f"{what}: error {worst:.2f}x the {rel:g} relative bound (max abs err {err.max():.3e}, scale {scale:.3e})"


def make_cfg(**over):
    cfg = SimpleNamespace(PRODUCT_EMB_DIM=128, TYPE_EMB_DIM=64, HIDDEN_SIZE=256, NUM_ATTENTION_HEADS=4, DROPOUT=0.0,
                          MARGIN=1.0, ALPHA=0.8, NUM_COMP_TYPES=3, NUM_TYPES=40, DEVICE=dev())
    for k, v in over.items():
        setattr(cfg, k, v)
    return cfg


def load_p2v(golden_name, **cfg_over):
    from pcompanion_b200 import Product2Vec
    g = load_golden(golden_name)
    m = Product2Vec(make_cfg(**cfg_over))
    m.load_state_dict({k: torch.tensor(v) for k, v in state_dict_from(g).items()})   # reference key names / shapes
    return g, m.to(dev())


def random_csr(n_dst, n_src, mean_deg, rng, hub=None, empty_every=7):
    deg = rng.poisson(mean_deg, n_dst)
    deg[::empty_every] = 0
    if hub is not None:
        deg[1] = hub
    deg = np.minimum(deg, n_src)
    rowptr = np.zeros(n_dst + 1, np.int64)
    np.cumsum(deg, out=rowptr[1:])
    col = np.concatenate([np.sort(rng.choice(n_src, d, replace=False)) for d in deg]).astype(np.int32) if deg.sum() else np.zeros(0, np.int32)
    return rowptr, col


# ----------------------------------------------------------------------------- (1) BPG / CSR / sets
@pytest.mark.parametrize("n", [0, 1, 2, 33, 4096, 4097, 100_003])
def test_radix_sort_matches_numpy(n):
    from pcompanion_b200 import ops
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 2 ** 63 - 1, n, dtype=np.int64)
    if n > 10:
        keys[: n // 3] = keys[n // 3: 2 * (n // 3)]           # duplicates
    t = torch.tensor(keys, device=dev())
    ops.sort_keys_(t, 0xFF)
    assert np.array_equal(t.cpu().numpy(), np.sort(keys))


def test_radix_sort_digit_mask_and_stability_of_low_ids():
    from pcompanion_b200 import ops
    rng = np.random.default_rng(5)
    n_ids = 70_000                                             # 17 bits -> 3 bytes per half
    src = rng.integers(0, n_ids, 300_000).astype(np.int32)
    dst = rng.integers(0, n_ids, 300_000).astype(np.int32)
    keys = ops.pack_keys(torch.tensor(src, device=dev()), torch.tensor(dst, device=dev()))
    assert ops.digit_mask_for(n_ids) == 0x77
    ops.sort_keys_(keys, ops.digit_mask_for(n_ids))
    from oracle import bpg as obpg
    assert np.array_equal(keys.cpu().numpy().astype(np.uint64), np.sort(obpg.pack_keys(src, dst)))
    s2, d2 = ops.unpack_keys(keys)
    assert np.array_equal(obpg.pack_keys(s2.cpu().numpy(), d2.cpu().numpy()), np.sort(obpg.pack_keys(src, dst)))


def test_bpg_c1_csr_neighbours_and_set_logic_bit_exact():
    """Config C1 (the reference's default synthetic BPG): device CSR, neighbour sets and the
    (Bcv n Bpv) - Bcp / Bcp - (Bpv u Bcv) sets equal the reference's Python sets."""
    from pcompanion_b200 import BehaviorProductGraph
    from oracle import bpg as obpg
    g = load_golden("bpg_c1.npz")
    n = len(g["type_id"])
    rng = np.random.default_rng(0)
    edges = {}
    for t in obpg.EDGE_TYPES:
        e = g["edges/" + t]
        e = np.concatenate([e, e[rng.integers(0, len(e), len(e) // 5)]])     # re-insert duplicates
        e = e[rng.permutation(len(e))]                                          # arbitrary insertion order
        edges[t] = (torch.tensor(e[:, 0].copy()), torch.tensor(e[:, 1].copy()))
    edges["not_an_edge_type"] = edges["co_view"]                                # silently dropped, bpg.py:21
    bpg = BehaviorProductGraph.from_arrays(n, edges, None, torch.tensor(g["type_id"]), dev())
    pk = lambda a: obpg.pack_keys(a[:, 0], a[:, 1]).astype(np.int64)
    for t in obpg.EDGE_TYPES:
        assert np.array_equal(bpg.keys(t).cpu().numpy(), pk(g["edges/" + t])), t
        rowptr, col = obpg.csr_from_keys(pk(g["edges/" + t]).astype(np.uint64), n)
        assert np.array_equal(bpg.csr(t).rowptr.cpu().numpy(), rowptr)
        assert np.array_equal(bpg.csr(t).col.cpu().numpy(), col)
        colptr, row, _ = obpg.csc_from_csr(rowptr, col, n)
        cp_dev, row_dev = bpg.csr(t).transposed()
        assert np.array_equal(cp_dev.cpu().numpy(), colptr) and np.array_equal(row_dev.cpu().numpy(), row)
    assert np.array_equal(bpg.similarity_keys().cpu().numpy(), pk(g["similarity_pairs"]))
    assert np.array_equal(bpg.complementary_keys().cpu().numpy(), pk(g["complementary_pairs"]))
    for p in g["probe_nodes"]:
        assert np.array_equal(bpg.neighbor_indices(int(p), "co_view").cpu().numpy(), g[f"nbr_cv/{p}"])
    members, offsets = bpg.type_members()
    lo, hi = offsets[0].item(), offsets[1].item()
    assert np.array_equal(members[lo:hi].cpu().numpy(), g["products_of_type0"])
    bpg.derive_pair_sets()
    assert bpg.similarity_pairs == [tuple(x) for x in g["similarity_pairs"].tolist()]


def test_bpg_reference_api_surface_on_strings():
    """dict/set surface of bpg.py with string ids: add_node/add_edge/get_neighbors/get_* helpers."""
    from pcompanion_b200 import BehaviorProductGraph
    g = load_golden("bpg_c1.npz")
    ids = [f"P{str(i).zfill(6)}" for i in range(len(g["type_id"]))]
    bpg = BehaviorProductGraph(dev())
    for i, pid in enumerate(ids):
        bpg.add_node(pid, {"type": str(g["type_names"][g["type_id"][i]]), "features": torch.zeros(128)})
    for t in ("co_view", "purchase_after_view", "co_purchase"):
        for s, d in g["edges/" + t]:
            bpg.add_edge(ids[s], ids[d], t)
    bpg.add_edge(ids[0], ids[1], "bogus")
    for p in g["probe_nodes"]:
        assert bpg.get_neighbors(ids[p], "co_view") == {ids[j] for j in g[f"nbr_cv/{p}"]}
        assert bpg.get_neighbors(ids[p]) == {ids[j] for j in g[f"nbr_all/{p}"]}
    assert bpg.get_neighbors("no-such-product") == set()
    assert bpg.get_all_types() == set(g["type_names"].tolist())
    t0 = str(sorted(g["type_names"].tolist())[0])
    assert bpg.get_products_by_type(t0) == [ids[j] for j in g["products_of_type0"]]
    assert sorted(bpg.get_exclusive_co_purchase_pairs()) == [(ids[a], ids[b], 1) for a, b in g["exclusive_co_purchase"].tolist()]
    assert sorted(bpg.get_co_view_intersection_pairs()) == [(ids[a], ids[b], -1) for a, b in g["co_view_intersection"].tolist()]


def test_empty_graph_and_empty_sets():
    from pcompanion_b200 import BehaviorProductGraph, ops
    z = torch.zeros(0, dtype=torch.int32)
    bpg = BehaviorProductGraph.from_arrays(5, {"co_view": (z, z)}, None, None, dev())
    assert bpg.csr("co_view").rowptr.tolist() == [0] * 6 and bpg.csr("co_view").num_edges == 0
    assert bpg.similarity_keys().numel() == 0
    a = torch.tensor([1, 5, 9], device=dev())
    e = torch.zeros(0, dtype=torch.int64, device=dev())
    assert ops.set_difference(a, e).tolist() == [1, 5, 9] and ops.set_intersection(a, e).tolist() == []
    assert ops.set_intersection(e, a).tolist() == []


# ----------------------------------------------------------------------------- (2) GAT kernels
@pytest.mark.parametrize("heads", [1, 2, 4, 8])
def test_gat_forward_backward_matches_oracle(heads):
    from pcompanion_b200 import ops
    from oracle import p2v
    rng = np.random.default_rng(heads)
    n_dst, n_src = 257, 301
    rowptr, col = random_csr(n_dst, n_src, 9, rng, hub=300)
    q = rng.normal(size=(n_dst, 128)).astype(np.float32)
    kv = rng.normal(size=(n_src, 256)).astype(np.float32)
    d_o = rng.normal(size=(n_dst, 128)).astype(np.float32)
    graph = ops.CSRGraph(torch.tensor(rowptr, device=dev()), torch.tensor(col, device=dev()), n_dst, n_src)
    qt = torch.tensor(q, device=dev(), requires_grad=True)
    kvt = torch.tensor(kv, device=dev(), requires_grad=True)
    o = ops.gat_attention(qt, kvt, graph, heads)
    o.backward(torch.tensor(d_o, device=dev()))
    ro, _ = p2v.gat_csr_forward(q.astype(np.float64), kv.astype(np.float64), rowptr, col, heads)
    rdq, rdkv = p2v.gat_csr_backward(q.astype(np.float64), kv.astype(np.float64), rowptr, col, heads, d_o.astype(np.float64))
    close(o, ro, what="o")
    close(qt.grad, rdq, what="dq")
    close(kvt.grad, rdkv, what="dkv")
    assert (o[::7] == 0).all()                                   # empty rows


@pytest.mark.parametrize("n_dst", [1, 3, 4, 5, 9, 64])
def test_gat_ring_edge_cases_degrees_and_chunk_tails(n_dst):
    """The kernels prefetch 8 rows ahead across the rows of a 4-row chunk: degrees 0, 1, around the ring depth,
    around the 32-entry id window, and far beyond both; row counts around the chunk size; separate (unpacked) Q / dO."""
    from pcompanion_b200 import ops
    from oracle import p2v
    rng = np.random.default_rng(100 + n_dst)
    n_src = 1500
    degs = [0, 1, 7, 8, 9, 31, 32, 33, 100, 1000, 2, 0, 0, 17]
    deg = np.array([degs[(i * 5 + n_dst) % len(degs)] for i in range(n_dst)])
    rowptr = np.zeros(n_dst + 1, np.int64); np.cumsum(deg, out=rowptr[1:])
    col = np.concatenate([np.sort(rng.choice(n_src, d, replace=False)) for d in deg] + [np.zeros(0, np.int64)]).astype(np.int32)
    q = rng.normal(size=(n_dst, 128)).astype(np.float32)
    kv = rng.normal(size=(n_src, 256)).astype(np.float32)
    d_o = rng.normal(size=(n_dst, 128)).astype(np.float32)
    graph = ops.CSRGraph(torch.tensor(rowptr, device=dev()), torch.tensor(col, device=dev()), n_dst, n_src)
    for heads in (1, 4):
        qt = torch.tensor(q, device=dev(), requires_grad=True)
        kvt = torch.tensor(kv, device=dev(), requires_grad=True)
        o = ops.gat_attention(qt, kvt, graph, heads)
        o.backward(torch.tensor(d_o, device=dev()))
        ro, _ = p2v.gat_csr_forward(q.astype(np.float64), kv.astype(np.float64), rowptr, col, heads)
        rdq, rdkv = p2v.gat_csr_backward(q.astype(np.float64), kv.astype(np.float64), rowptr, col, heads, d_o.astype(np.float64))
        # atol: a row with one neighbour has softmax weight 1 and a mathematically zero dq (rounding noise on both sides)
        close(o, ro, what=f"o h{heads}", atol=1e-6)
        close(qt.grad, rdq, what=f"dq h{heads}", atol=1e-6)
        close(kvt.grad, rdkv, what=f"dkv h{heads}", atol=1e-6)
        a = ops.gat_attention(qt.detach(), kvt.detach(), graph, heads, 0.3, 5)
        b = ops.gat_attention(qt.detach(), kvt.detach(), graph, heads, 0.3, 5)
        assert torch.equal(a, b)


def test_halo_push_and_peer_reduction_kernels_on_one_gpu():
    """pc_halo_push with two 'peers' that are both buffers of this GPU (gather + strided store semantics, cyclic start),
    and pc_rows_reduce_peers against index_add in the same peer order."""
    import ctypes
    from pcompanion_b200 import ops
    from pcompanion_b200._lib import call, dev as dptr, stream
    g = torch.Generator(device=dev()).manual_seed(9)
    table = torch.randn(500, 256, generator=g, device=dev())
    idx = torch.randperm(500, generator=g, device=dev())[:300]
    peers = [torch.zeros(400, 256, device=dev()), torch.zeros(400, 256, device=dev())]
    off = (ctypes.c_int64 * 3)(0, 120, 300)
    base = (ctypes.c_void_p * 2)(peers[0].data_ptr(), peers[1].data_ptr())
    dst0 = (ctypes.c_int64 * 2)(10, 200)
    for first in (0, 120, 299, 300):
        for pbuf in peers:
            pbuf.zero_()
        call("pc_halo_push", dptr(table, torch.float32, "t"), 256, dptr(idx, torch.int64, "i"), 2, off, base, None, dst0, first,
             256, stream())
        assert torch.equal(peers[0][10:130], table[idx[:120]]) and torch.equal(peers[1][200:380], table[idx[120:]])
        assert peers[0][:10].abs().sum() == 0 and peers[0][130:].abs().sum() == 0 and peers[1][:200].abs().sum() == 0
    # contiguous runs (index = NULL), strided source
    wide = torch.randn(500, 384, generator=g, device=dev())
    src0 = (ctypes.c_int64 * 2)(5, 250)
    for pbuf in peers:
        pbuf.zero_()
    call("pc_halo_push", ctypes.c_void_p(wide[:, 128:].data_ptr()), 384, None, 2, off, base, src0, dst0, 0, 256, stream())
    assert torch.equal(peers[0][10:130], wide[5:125, 128:]) and torch.equal(peers[1][200:380], wide[250:430, 128:])
    # owner-side reduction
    n, world = 700, 3
    tbl = torch.randn(n, 256, generator=g, device=dev())
    ref = tbl.clone()
    slot = torch.full((world, n), -1, dtype=torch.int32, device=dev())
    chunks, o = [], 0
    for p_ in range(world):
        ids = torch.randperm(n, generator=g, device=dev())[: 100 + 150 * p_]
        slot[p_, ids] = torch.arange(o, o + ids.numel(), dtype=torch.int32, device=dev())
        chunks.append(ids); o += ids.numel()
    rows = torch.randn(o, 256, generator=g, device=dev())
    o = 0
    for ids in chunks:                                   # same peer order => same rounding
        ref[ids] += rows[o: o + ids.numel()]; o += ids.numel()
    ops.rows_reduce_peers_(tbl, rows, slot)
    assert torch.equal(tbl, ref)



def test_gat_is_deterministic_and_dropout_is_consistent():
    from pcompanion_b200 import ops
    rng = np.random.default_rng(3)
    n = 2000
    rowptr, col = random_csr(n, n, 20, rng)
    graph = ops.CSRGraph(torch.tensor(rowptr, device=dev()), torch.tensor(col, device=dev()), n, n)
    q = torch.randn(n, 128, device=dev())
    kv = torch.randn(n, 256, device=dev())
    d_o = torch.randn(n, 128, device=dev())

    def run(p, seed):
        qt, kvt = q.clone().requires_grad_(True), kv.clone().requires_grad_(True)
        o = ops.gat_attention(qt, kvt, graph, 4, p, seed)
        o.backward(d_o)
        return o.detach(), qt.grad, kvt.grad

    a, b = run(0.0, 0), run(0.0, 0)
    assert all(torch.equal(x, y) for x, y in zip(a, b))          # bit-reproducible, no float atomics
    d1, d2, d3 = run(0.1, 7), run(0.1, 7), run(0.1, 8)
    assert all(torch.equal(x, y) for x, y in zip(d1, d2))
    assert not torch.equal(d1[0], d3[0])
    # E[dropout output] == no-dropout output: average over seeds approaches it
    acc = torch.zeros_like(a[0])
    for s in range(64):
        acc += ops.gat_attention(q, kv, graph, 4, 0.1, 1000 + s)
    rel = ((acc / 64 - a[0]).norm() / a[0].norm()).item()
    assert rel < 0.06, rel
    # gradient of the dropout forward agrees with a finite difference along a random direction
    qt = q[:64].clone().double()
    g64 = ops.CSRGraph(graph.rowptr[:65].contiguous(), graph.col[: int(graph.rowptr[64])].contiguous(), 64, n)
    dirn = torch.randn(64, 128, device=dev())
    f = lambda t: (ops.gat_attention(t.float(), kv, g64, 4, 0.1, 11).double() * d_o[:64].double()).sum().item()
    eps = 1e-2
    fd = (f(qt + eps * dirn) - f(qt - eps * dirn)) / (2 * eps)
    qg = q[:64].clone().requires_grad_(True)
    (ops.gat_attention(qg, kv, g64, 4, 0.1, 11) * d_o[:64]).sum().backward()
    an = (qg.grad.double() * dirn.double()).sum().item()
    assert abs(fd - an) <= 1e-2 * max(1.0, abs(an)), (fd, an)


def test_attention_matches_reference_multihead_attention_golden():
    """Dense drop-in path vs nn.MultiheadAttention as the reference calls it (incl. autograd)."""
    g, m = load_p2v("p2v_module.npz")
    m.eval()
    q = torch.tensor(g["attn_q"], device=dev(), requires_grad=True)
    kv = torch.tensor(g["attn_kv"], device=dev(), requires_grad=True)
    out = m.apply_attention(q, kv)
    (out * torch.tensor(g["attn_w"], device=dev())).sum().backward()
    close(out, g["attn_out"], what="attn_out")
    close(q.grad, g["attn_dq"], what="attn_dq")
    close(kv.grad, g["attn_dkv"], what="attn_dkv")


# ----------------------------------------------------------------------------- Product2Vec module
def test_product2vec_eval_forward_matches_reference_golden():
    g, m = load_p2v("p2v_module.npz")
    m.eval()
    t = lambda k: torch.tensor(g[k], device=dev())
    with torch.no_grad():
        close(m(t("anchor"), t("neighbors")), g["eval_forward_nbrs"], what="nbrs")      # zero pads attended
        close(m(t("anchor")), g["eval_forward_plain"], what="plain")
        close(m(t("negative")), g["eval_forward_neg3d"], what="3d")
        close(m(t("anchor")[0], t("neighbors")[0]), g["eval_forward_1d"], what="1d")
        close(m.get_initial_embedding(t("anchor")[0]), g["eval_initial_1d"], what="init1d")
    with pytest.raises(ValueError, match="Unexpected input dimension"):
        m.get_initial_embedding(torch.zeros(1, 1, 1, 128, device=dev()))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(2, 128))


def test_product2vec_train_step_matches_reference_golden():
    """One step of product2vec.py:132-158: embeddings, loss, every parameter gradient and the
    BatchNorm running statistics after three FFN calls."""
    g, m = load_p2v("p2v_module.npz")
    m.train()
    t = lambda k: torch.tensor(g[k], device=dev())
    a = m(t("anchor"), t("neighbors"))
    p = m(t("positive"))
    n = m(t("negative"))
    loss = m.triplet_loss(a, p, n)
    loss.backward()
    close(a, g["train_anchor_emb"], what="anchor")
    close(p, g["train_positive_emb"], what="positive")
    close(n, g["train_negative_emb"], what="negative")
    close(loss, g["train_loss"], what="loss")
    for k, v in m.named_parameters():
        close(*golden_grad(g, k, v.grad), rel=REL_VS_FP32, atol=1e-7, what="grad " + k)   # reference grads are themselves fp32
    close(m.ffn[1].running_mean, g["train_running_mean"], what="running_mean")
    close(m.ffn[1].running_var, g["train_running_var"], what="running_var")
    assert int(m.ffn[1].num_batches_tracked) == int(g["train_num_batches_tracked"])


def test_generate_all_embeddings_matches_reference_golden():
    from pcompanion_b200 import BehaviorProductGraph
    g, m = load_p2v("p2v_graph.npz")
    n = g["features"].shape[0]
    ids = [f"P{str(i).zfill(6)}" for i in range(n)]
    bpg = BehaviorProductGraph(dev())
    for i, pid in enumerate(ids):
        bpg.add_node(pid, {"features": torch.tensor(g["features"][i]), "type": f"type_{i % 5}"})
    for s, d in zip(g["src"], g["dst"]):
        bpg.add_edge(ids[s], ids[d], "co_view")
    emb = m.generate_all_embeddings(bpg)
    assert list(emb.keys()) == ids and all(v.device.type == "cpu" for v in emb.values())
    close(torch.stack([emb[p] for p in ids]), g["embeddings"], what="embeddings")


def test_forward_graph_train_matches_oracle_and_torch_port_grads():
    """Graph formulation (BN over node rows, SURVEY H2): forward vs the numpy oracle, parameter and
    input gradients vs float64 autograd of the torch port fed per-destination neighbour lists."""
    from pcompanion_b200 import ops
    from oracle import p2v, torch_port
    g, m = load_p2v("p2v_module.npz")
    rng = np.random.default_rng(11)
    n = 150
    rowptr, col = random_csr(n, n, 6, rng)
    x = rng.normal(size=(n, 128)).astype(np.float32)
    w = rng.normal(size=(n, 128)).astype(np.float32)
    graph = ops.CSRGraph(torch.tensor(rowptr, device=dev()), torch.tensor(col, device=dev()), n, n)
    m.train()
    xt = torch.tensor(x, device=dev(), requires_grad=True)
    out = m.forward_graph(xt, graph)
    (out * torch.tensor(w, device=dev())).sum().backward()
    sd = state_dict_from(g, dtype=np.float64)
    ref, _ = p2v.forward_graph(sd, x.astype(np.float64), rowptr, col, 4, training=True)
    close(out, ref, what="forward_graph")
    # float64 torch-port autograd as the gradient oracle
    pm = torch_port.PortProduct2Vec(torch_port.default_config(DROPOUT=0.0)).double()
    pm.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    pm.train()
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    h = pm.ffn(x64)
    rows = []
    for i in range(n):
        nb = col[rowptr[i]:rowptr[i + 1]]
        rows.append(pm.attend(h[i:i + 1], h[nb].unsqueeze(0))[0] if len(nb) else h[i])
    (torch.stack(rows) * torch.tensor(w, dtype=torch.float64)).sum().backward()
    close(xt.grad, x64.grad.numpy(), what="dx")
    for (k, v), (_, v64) in zip(m.named_parameters(), pm.named_parameters()):
        # ffn.0.bias sits in front of BatchNorm: its gradient is mathematically zero (sum of 150 terms that
        # cancel), both sides hold fp32 summation noise of ~1e-6 there
        close(v.grad, v64.grad.numpy(), atol=3e-6 if k == "ffn.0.bias" else 1e-7, what="grad " + k)


# ----------------------------------------------------------------------------- (3) losses / PCompanion
def test_triplet_and_item_hinge_match_oracle():
    from pcompanion_b200 import ops
    from oracle import p2v, pcomp
    rng = np.random.default_rng(2)
    b, k, d = 37, 5, 128
    a, p, n = (rng.normal(size=s).astype(np.float32) * 0.4 for s in ((b, d), (b, d), (b, k, d)))
    ta, tp, tn = (torch.tensor(x, device=dev(), requires_grad=True) for x in (a, p, n))
    loss = ops.triplet_hinge(ta, tp, tn, 1.0)
    loss.backward()
    rl, _ = p2v.triplet_hinge(a.astype(np.float64), p.astype(np.float64), n.astype(np.float64), 1.0)
    ga, gp, gn = p2v.triplet_hinge_backward(a.astype(np.float64), p.astype(np.float64), n.astype(np.float64), 1.0)
    close(loss, rl, what="triplet loss")
    close(ta.grad, ga, what="d anchor"); close(tp.grad, gp, what="d positive"); close(tn.grad, gn, what="d negative")
    proj = rng.normal(size=(b, 3, d)).astype(np.float32) * 0.3
    tpj = torch.tensor(proj, device=dev(), requires_grad=True)
    il = ops.item_hinge(tpj, torch.tensor(p, device=dev()), torch.tensor(a, device=dev()), 1.0)
    il.backward()
    close(il, pcomp.item_hinge(proj.astype(np.float64), p.astype(np.float64), a.astype(np.float64), 1.0), what="item loss")
    close(tpj.grad, pcomp.item_hinge_backward(proj.astype(np.float64), p.astype(np.float64), a.astype(np.float64), 1.0), what="d proj")
    # second evaluation is bit-identical (fixed-order reductions)
    assert torch.equal(ops.triplet_hinge(ta, tp, tn, 1.0), loss)


def test_pcompanion_matches_reference_golden():
    from pcompanion_b200 import PCompanion
    g = load_golden("pcomp.npz")
    cfg = make_cfg(NUM_TYPES=40)
    sd = {k: torch.tensor(v) for k, v in state_dict_from(g).items()}
    table = {f"P{str(i).zfill(6)}": sd["product_embeddings.weight"][i] for i in range(sd["product_embeddings.weight"].shape[0])}
    m = PCompanion(cfg, table)
    assert set(m.state_dict().keys()) == set(sd.keys())
    m.load_state_dict(sd)
    m = m.to(dev()).train()
    batch = {"query_ids": [f"P{str(int(i)).zfill(6)}" for i in g["query_idx"]]}
    for k in ("query_types", "positive_types", "negative_types", "positive_items", "negative_items", "target_features"):
        batch[k] = torch.tensor(g["batch/" + k], device=dev())
    out = m(batch)
    loss = m.compute_loss(batch, out)
    loss.backward()
    close(out["type_similarities"], g["type_similarities"], what="type_similarities")
    assert np.array_equal(out["complementary_types"].cpu().numpy(), g["complementary_types"])
    assert out["complementary_types"].dtype == torch.int64
    close(out["projected_embeddings"], g["projected_embeddings"], what="projected")
    close(loss, g["loss"], what="loss")
    for k, v in m.named_parameters():
        if v.grad is not None:
            close(v.grad, g["grad/" + k], rel=REL_VS_FP32, atol=1e-7, what="grad " + k)
    with pytest.raises(KeyError):
        m({**batch, "query_ids": ["nope"] * len(batch["query_ids"])})
    # dense-table constructor + index tensor ids give the same numbers
    m2 = PCompanion(cfg, sd["product_embeddings.weight"])
    m2.load_state_dict(sd)
    m2 = m2.to(dev()).eval()
    out2 = m2({**batch, "query_ids": torch.tensor(g["query_idx"], device=dev())})
    assert torch.equal(out2["complementary_types"], out["complementary_types"])


def test_metrics_match_reference_golden():
    from pcompanion_b200 import Metrics
    g = load_golden("metrics.npz")
    pred, gt = torch.tensor(g["pred"], device=dev()), torch.tensor(g["gt"], device=dev())
    for k in (1, 3, 10):
        assert abs(Metrics.hit_at_k(pred, gt, k) - float(g[f"hit@{k}"])) < 1e-6
    gp = load_golden("pcomp.npz")
    sims = torch.tensor(gp["eval_sims"], device=dev())
    for k in (1, 3, 10):
        assert abs(Metrics.hit_at_k(sims, torch.arange(sims.size(0), device=dev()), k) - float(gp[f"hit@{k}"])) < 1e-6
    assert abs(Metrics.type_diversity(torch.tensor(gp["complementary_types"], device=dev())) - float(gp["type_diversity"])) < 1e-6
    assert abs(Metrics.mean_relevance(torch.tensor(gp["projected_embeddings"], device=dev()),
                                      torch.tensor(gp["batch/positive_items"], device=dev())) - float(gp["mean_relevance"])) < 1e-5


# ----------------------------------------------------------------------------- (4) retrieval
def test_retrieval_matches_reference_golden_and_oracle_bit_exact():
    from pcompanion_b200 import CatalogIndex
    from oracle import retrieval as oret
    g = load_golden("metrics.npz")
    cat = CatalogIndex(torch.tensor(g["catalog"], device=dev()), torch.tensor(g["type_id"], device=dev()))
    q, rt = torch.tensor(g["q"], device=dev()), torch.tensor(g["row_type"], device=dev())
    s, i = cat.topk(q, 10, rt)
    assert np.array_equal(i.cpu().numpy(), g["topk_idx"])               # the reference's own per-type topk
    os_, oi = oret.masked_topk(g["q"], g["catalog"], 10, g["row_type"], g["type_id"])
    assert np.array_equal(i.cpu().numpy(), oi) and np.array_equal(s.cpu().numpy(), os_)
    for splits in (1, 2, 5):
        s2, i2 = cat.topk(q, 10, rt, splits=splits)
        assert torch.equal(i2, i) and torch.equal(s2, s)
    # unmasked (metrics.py-style) scoring over the whole catalog
    s3, i3 = cat.topk(q, 7)
    os3, oi3 = oret.masked_topk(g["q"], g["catalog"], 7)
    assert np.array_equal(i3.cpu().numpy(), oi3) and np.array_equal(s3.cpu().numpy(), os3)


def test_retrieval_ties_padding_and_shard_merge():
    from pcompanion_b200 import CatalogIndex, ops
    from oracle import retrieval as oret
    rng = np.random.default_rng(4)
    p, t, r, k = 5000, 11, 40, 10
    cat = rng.normal(size=(p, 128)).astype(np.float32)
    cat[rng.integers(0, p, 1500)] = cat[17]                            # many exact duplicates -> ties
    type_id = rng.integers(0, t, p).astype(np.int32)
    type_id[type_id == 3] = 4                                          # type 3 is empty
    type_id[type_id == 10] = 9
    type_id[:4] = 10                                                   # type 10 has 4 products < k
    q = rng.normal(size=(r, 128)).astype(np.float32)
    q[:5] = cat[17] * 0.5
    row_type = rng.integers(0, t, r).astype(np.int32)
    row_type[0], row_type[1] = 3, 10
    os_, oi = oret.masked_topk(q, cat, k, row_type, type_id)
    full = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=t)
    s, i = full.topk(torch.tensor(q, device=dev()), k, torch.tensor(row_type, device=dev()))
    assert np.array_equal(i.cpu().numpy(), oi) and np.array_equal(s.cpu().numpy(), os_)
    assert (i[0] == -1).all() and torch.isinf(s[0]).all()
    # 3 shards + merge == unsharded (SURVEY 8e), ties -> lowest global index
    bounds = [0, 1700, 3400, p]
    parts = []
    for a, b in zip(bounds[:-1], bounds[1:]):
        sh = CatalogIndex(torch.tensor(cat[a:b], device=dev()), torch.tensor(type_id[a:b], device=dev()), index_base=a, num_types=t)
        parts.append(sh.topk(torch.tensor(q, device=dev()), k, torch.tensor(row_type, device=dev())))
    ms, mi = ops.topk_merge(torch.cat([x[0] for x in parts], 1), torch.cat([x[1] for x in parts], 1), k)
    assert torch.equal(mi, i) and torch.equal(ms, s)


def test_topk_rows_is_a_stable_sort():
    from pcompanion_b200 import ops
    rng = np.random.default_rng(6)
    v = rng.integers(-5, 5, size=(33, 1000)).astype(np.float32)       # heavy ties
    for k in (1, 3, 10, 32):
        s, i = ops.topk_rows(torch.tensor(v, device=dev()), k)
        ref = np.argsort(-v, axis=1, kind="stable")[:, :k]
        assert np.array_equal(i.cpu().numpy(), ref)
        assert np.array_equal(s.cpu().numpy(), np.take_along_axis(v, ref, 1).astype(np.float64))
    s, i = ops.topk_rows(torch.tensor(v[:, :5].copy(), device=dev()), 8)
    assert (i[:, 5:] == -1).all()


# ----------------------------------------------------------------------------- full-size properties (C2)
def test_full_size_c2_properties():
    """Config C2 scale (1 M products / ~20 M co-view edges): size-independent properties.
    CSR sortedness + dedup, transpose involution, softmax weights sum to one (V = 1 -> O = 1),
    linearity of the output in V and of dKV in dO, determinism."""
    from pcompanion_b200 import ops
    from pcompanion_b200.synthetic import synthetic_bpg
    n = 1_000_000
    bpg = synthetic_bpg(n, 20_000_000, device=dev())
    g = bpg.csr("co_view")
    e = g.num_edges
    assert 18_000_000 < e < 22_000_000
    assert int(g.rowptr[0]) == 0 and int(g.rowptr[-1]) == e and bool((g.rowptr[1:] >= g.rowptr[:-1]).all())
    keys = bpg.keys("co_view")
    assert bool((keys[1:] > keys[:-1]).all())                         # strictly ascending == sorted + unique
    src, dst = ops.unpack_keys(keys)
    assert bool((src < dst).all()) and torch.equal(dst, g.col)
    colptr, row = g.transposed()
    assert int(colptr[-1]) == e and bool((colptr[1:] >= colptr[:-1]).all())
    back = ops.CSRGraph(colptr, row, n, n).transposed()                 # transpose twice == identity
    assert torch.equal(back[0], g.rowptr) and torch.equal(back[1], g.col)
    sim = bpg.similarity_keys()
    assert bool((sim[1:] > sim[:-1]).all()) and ops.set_intersection(sim, bpg.keys("co_purchase")).numel() == 0
    assert ops.set_difference(sim, bpg.keys("co_view")).numel() == 0

    q = torch.randn(n, 128, device=dev())
    kv = torch.randn(n, 256, device=dev())
    has = (g.rowptr[1:] > g.rowptr[:-1])
    kv1 = kv.clone(); kv1[:, 128:] = 1.0
    o1 = ops.gat_attention(q, kv1, g, 4)
    assert torch.allclose(o1[has], torch.ones_like(o1[has]), rtol=0, atol=2e-6) and bool((o1[~has] == 0).all())
    o = ops.gat_attention(q, kv, g, 4)
    kv2 = kv.clone(); kv2[:, 128:] *= 2.0
    assert torch.equal(ops.gat_attention(q, kv2, g, 4), o * 2.0)        # exact: scaling by 2 commutes with rounding
    assert torch.equal(ops.gat_attention(q, kv, g, 4), o)               # deterministic
    d_o = torch.randn(n, 128, device=dev())
    qt, kvt = q.clone().requires_grad_(True), kv.clone().requires_grad_(True)
    ops.gat_attention(qt, kvt, g, 4).backward(d_o)
    qt2, kvt2 = q.clone().requires_grad_(True), kv.clone().requires_grad_(True)
    ops.gat_attention(qt2, kvt2, g, 4).backward(d_o * 2.0)
    assert torch.equal(qt2.grad, qt.grad * 2.0) and torch.equal(kvt2.grad, kvt.grad * 2.0)
    # sum_j dV_j == sum_i dO_i over rows with neighbours (attention weights sum to one), per column
    lhs = kvt.grad[:, 128:].double().sum(0)
    rhs = d_o[has].double().sum(0)
    assert torch.allclose(lhs, rhs, rtol=1e-6, atol=1e-3 * math.sqrt(n))


def test_fused_graph_layer_equals_unfused_path_and_single_rank_partition():
    """fused.py (one autograd node) vs the op-by-op path, train and eval, plus the world-size-1 halo plan."""
    from pcompanion_b200 import ops
    from pcompanion_b200.distributed import HaloPlan, forward_graph_partitioned
    from pcompanion_b200.fused import p2v_graph_layer
    g, m = load_p2v("p2v_module.npz")
    rng = np.random.default_rng(21)
    n = 700
    rowptr, col = random_csr(n, n, 8, rng)
    graph = ops.CSRGraph(torch.tensor(rowptr, device=dev()), torch.tensor(col, device=dev()), n, n)
    x = torch.randn(n, 128, device=dev())
    w = torch.randn(n, 128, device=dev())
    bn = m.ffn[1]
    saved = (bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone())

    def run(fn, train):
        bn.running_mean.copy_(saved[0]); bn.running_var.copy_(saved[1]); bn.num_batches_tracked.copy_(saved[2])
        m.train(train)
        m.zero_grad()
        xt = x.clone().requires_grad_(True)
        out = fn(xt)
        (out * w).sum().backward()
        return out.detach(), xt.grad, [p.grad.clone() for p in m.parameters()], bn.running_mean.clone(), bn.running_var.clone()

    def unfused(xt):
        h = m._ffn_rows(xt)
        out = m._attend(h, h, graph)
        return torch.where((graph.rowptr[1:] > graph.rowptr[:-1]).unsqueeze(1), out, h)

    plan = HaloPlan(graph.rowptr, graph.col, [0, n], 0)
    for train in (True, False):
        ref = run(unfused, train)
        for name, fn in (("fused", lambda xt: p2v_graph_layer(m, xt, graph)),
                         ("partitioned", lambda xt: forward_graph_partitioned(m, xt, plan))):
            got = run(fn, train)
            close(got[0], ref[0].double().cpu().numpy(), what=f"{name} out train={train}")
            close(got[1], ref[1].double().cpu().numpy(), rel=REL_VS_FP32, what=f"{name} dx train={train}")   # two fp32 paths
            for (k, _), a, r in zip(m.named_parameters(), got[2], ref[2]):
                close(a, r.double().cpu().numpy(), rel=REL_VS_FP32, atol=3e-6 if k == "ffn.0.bias" else 1e-7, what=f"{name} grad {k} train={train}")
            close(got[3], ref[3].double().cpu().numpy(), what="running_mean")
            close(got[4], ref[4].double().cpu().numpy(), what="running_var")


def test_indexed_triplet_loss_equals_gathered_loss_and_is_deterministic():
    from pcompanion_b200 import ops
    g = torch.Generator(device=dev()).manual_seed(8)
    n, b, k = 5000, 3000, 5
    table = torch.randn(n, 128, generator=g, device=dev()) * 0.3
    ai, pi = (torch.randint(0, n, (b,), generator=g, device=dev()) for _ in range(2))
    ni = torch.randint(0, 40, (b, k), generator=g, device=dev())              # hot rows: many slots per node
    t1 = table.clone().requires_grad_(True)
    l1 = ops.triplet_hinge_indexed(t1, ai, pi, ni, 1.0)
    l1.backward()
    t2 = table.clone().double().requires_grad_(True)
    a, p, nn = t2[ai], t2[pi], t2[ni.reshape(-1)].reshape(b, k, 128)
    dpos = torch.nn.functional.pairwise_distance(a, p)
    dneg = torch.nn.functional.pairwise_distance(a.unsqueeze(1).expand(-1, k, -1), nn).mean(1)
    l2 = torch.relu(1.0 - dpos + dneg).mean()
    l2.backward()
    close(l1, l2.item(), what="indexed loss")
    close(t1.grad, t2.grad.cpu().numpy(), what="d table")
    t3 = table.clone().requires_grad_(True)
    ops.triplet_hinge_indexed(t3, ai, pi, ni, 1.0).backward()
    assert torch.equal(t3.grad, t1.grad)                                       # no atomics: bit-reproducible
    # a non-unit upstream gradient (the loss is scaled / is one term of a sum) reaches the table gradient
    t4 = table.clone().requires_grad_(True)
    (ops.triplet_hinge_indexed(t4, ai, pi, ni, 1.0) * -2.5).backward()
    close(t4.grad, -2.5 * t2.grad.cpu().numpy(), what="d table, upstream gradient -2.5")
    with torch.no_grad():
        assert torch.equal(ops.triplet_hinge_indexed(table, ai, pi, ni, 1.0), l1.detach())   # forward only: no gradient rows


def test_dense_tensor_core_retrieval_equals_exact_segmented_path():
    """north_star part 4 as worded: tcgen05 scoring GEMM + per-type mask + top-K over the whole catalog, then exact
    fp64 re-scoring.  Must agree bit for bit (indices and scores) with the exact type-segmented kernel, including
    rows whose guard band fails (many exact duplicates) and unmasked rows."""
    from pcompanion_b200 import CatalogIndex, ops
    from oracle import retrieval as oret
    rng = np.random.default_rng(12)
    p, t, r, k = 70_001, 37, 300, 10
    cat = rng.normal(size=(p, 128)).astype(np.float32)
    cat[rng.integers(0, p, 400)] = cat[123]                            # 400 exact duplicates -> ties
    tid = rng.integers(0, t, p).astype(np.int32)
    cat[1000:1040] = cat[123]                                          # 40 adjacent duplicates of one type: more equal
    tid[1000:1040] = tid[123]                                          # top scores than one candidate list holds
    q = rng.normal(size=(r, 128)).astype(np.float32)
    q[:8] = cat[123] * 0.7                                             # rows whose best products are the duplicates
    rt = rng.integers(0, t, r).astype(np.int32)
    rt[:4] = tid[123]
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(tid, device=dev()), num_types=t)
    qt, rtt = torch.tensor(q, device=dev()), torch.tensor(rt, device=dev())
    es, ei = index.topk(qt, k, rtt)
    ds, di = index.topk_dense(qt, k, rtt)
    assert torch.equal(di, ei) and torch.equal(ds, es)
    os_, oi = oret.masked_topk(q[:16], cat, k, rt[:16], tid)
    assert np.array_equal(di[:16].cpu().numpy(), oi) and np.array_equal(ds[:16].cpu().numpy(), os_)
    # unmasked: every row ranks the whole catalog (metrics.py-style scoring)
    eu = index.topk(qt[:130], k)
    du = index.topk_dense(qt[:130], k)
    assert torch.equal(du[1], eu[1]) and torch.equal(du[0], eu[0])
    # the raw kernel flags exactly the rows it cannot prove, and proves the generic ones
    _, _, flags = ops.score_topk_dense(qt, index.catalog, k, index.type_id, rtt, 0, None)
    assert int(flags[8:].sum()) == 0 and int(flags[:4].sum()) >= 1
