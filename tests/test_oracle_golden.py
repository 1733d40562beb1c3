"""Pin the oracle against fixtures produced by the REAL reference (tests/golden/make_golden.py).

The reference computes in float32; the oracle is evaluated in float64 on the same float32
inputs, so agreement is limited by the reference's own rounding (~1e-6 relative).
"""
import numpy as np
import torch

from conftest import golden_grad, load_golden, state_dict_from
from oracle import bpg as obpg
from oracle import p2v, pcomp, retrieval, torch_port

RTOL, ATOL = 2e-5, 2e-6


def close(a, b, rtol=RTOL, atol=ATOL):
    np.testing.assert_allclose(np.asarray(a, np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol)


def test_p2v_eval_forward_matches_reference():
    g = load_golden("p2v_module.npz")
    sd = state_dict_from(g, dtype=np.float64)
    f64 = lambda k: g[k].astype(np.float64)
    out, _ = p2v.forward(sd, f64("anchor"), f64("neighbors"), heads=4)
    close(out, g["eval_forward_nbrs"])
    out, _ = p2v.forward(sd, f64("anchor"), None, heads=4)
    close(out, g["eval_forward_plain"])
    out, _ = p2v.forward(sd, f64("negative"), None, heads=4)
    close(out, g["eval_forward_neg3d"])
    out, _ = p2v.forward(sd, f64("anchor")[0], f64("neighbors")[0], heads=4)
    close(out, g["eval_forward_1d"])
    out, _ = p2v.get_initial_embedding(sd, f64("anchor")[0])
    close(out, g["eval_initial_1d"])


def test_p2v_bad_rank_raises_like_reference():
    g = load_golden("p2v_module.npz")
    sd = state_dict_from(g, dtype=np.float64)
    try:
        p2v.get_initial_embedding(sd, np.zeros((1, 1, 1, 128)))
    except ValueError as e:
        assert "Unexpected input dimension" in str(e)
    else:
        raise AssertionError("expected ValueError")


def test_p2v_train_step_matches_reference():
    """Train-mode forward (BN batch statistics per call, running-stat updates in call order),
    triplet hinge with the reference's sign, product2vec.py:132-154."""
    g = load_golden("p2v_module.npz")
    sd = state_dict_from(g, dtype=np.float64)
    f64 = lambda k: g[k].astype(np.float64)
    a, (rm, rv) = p2v.forward(sd, f64("anchor"), f64("neighbors"), heads=4, training=True)
    close(a, g["train_anchor_emb"])
    sd["ffn.1.running_mean"], sd["ffn.1.running_var"] = rm, rv
    p, (rm, rv) = p2v.forward(sd, f64("positive"), None, heads=4, training=True)
    close(p, g["train_positive_emb"])
    sd["ffn.1.running_mean"], sd["ffn.1.running_var"] = rm, rv
    n, (rm, rv) = p2v.forward(sd, f64("negative"), None, heads=4, training=True)
    close(n, g["train_negative_emb"])
    close(rm, g["train_running_mean"])
    close(rv, g["train_running_var"])
    loss, _ = p2v.triplet_hinge(a, p, n, 1.0)
    close(loss, g["train_loss"])


def test_attention_backward_matches_reference_autograd():
    g = load_golden("p2v_module.npz")
    sd = state_dict_from(g, dtype=np.float64)
    q_in, kv_in, w = (g[k].astype(np.float64) for k in ("attn_q", "attn_kv", "attn_w"))
    b, n, e = kv_in.shape
    q, kv = p2v.in_projection(sd, q_in, kv_in.reshape(-1, e))
    rowptr = np.arange(b + 1, dtype=np.int64) * n
    col = np.arange(b * n, dtype=np.int32)
    o, _ = p2v.gat_csr_forward(q, kv, rowptr, col, 4)
    out = p2v.linear(o, sd["attention.out_proj.weight"], sd["attention.out_proj.bias"])
    close(out, g["attn_out"])
    d_o = w @ sd["attention.out_proj.weight"]                 # d(out*w).sum / d o
    dq, dkv = p2v.gat_csr_backward(q, kv, rowptr, col, 4, d_o)
    wi = sd["attention.in_proj_weight"]
    close(dq @ wi[:e], g["attn_dq"], rtol=1e-4, atol=1e-6)
    close((dkv @ wi[e:]).reshape(b, n, e), g["attn_dkv"], rtol=1e-4, atol=1e-6)


def test_triplet_backward_matches_finite_difference():
    rng = np.random.default_rng(0)
    a, p, n = rng.normal(size=(5, 16)), rng.normal(size=(5, 16)), rng.normal(size=(5, 3, 16))
    ga, gp, gn = p2v.triplet_hinge_backward(a, p, n, 1.0)
    eps = 1e-6
    for arr, grad in ((a, ga), (p, gp), (n, gn)):
        it = np.nditer(arr, flags=["multi_index"])
        for _ in range(20):
            idx = tuple(rng.integers(0, s) for s in arr.shape)
            old = arr[idx]
            arr[idx] = old + eps
            lp, _ = p2v.triplet_hinge(a, p, n, 1.0)
            arr[idx] = old - eps
            lm, _ = p2v.triplet_hinge(a, p, n, 1.0)
            arr[idx] = old
            assert abs((lp - lm) / (2 * eps) - grad[idx]) < 1e-6


def test_generate_all_embeddings_matches_reference():
    """generate_all_embeddings (product2vec.py:83-111): double FFN on the query, nodes
    without co-view out-neighbours keep ffn(x), duplicate / unknown-type inserts ignored."""
    g = load_golden("p2v_graph.npz")
    sd = state_dict_from(g, dtype=np.float64)
    n = g["features"].shape[0]
    keys = obpg.unique_sorted_keys(g["src"], g["dst"])
    assert len(keys) == len(g["src"]) - 1                      # the duplicate collapsed
    rowptr, col = obpg.csr_from_keys(keys, n)
    emb, _ = p2v.forward_graph(sd, g["features"].astype(np.float64), rowptr, col, 4, double_ffn_query=True)
    close(emb, g["embeddings"])
    assert (np.diff(rowptr) == 0).sum() >= 6


def test_bpg_c1_set_logic_bit_exact():
    g = load_golden("bpg_c1.npz")
    n = len(g["type_id"])
    keys = {t: obpg.unique_sorted_keys(g["edges/" + t][:, 0], g["edges/" + t][:, 1])
            for t in obpg.EDGE_TYPES}
    cv, pav, cp = keys["co_view"], keys["purchase_after_view"], keys["co_purchase"]
    pk = lambda a: obpg.pack_keys(a[:, 0], a[:, 1])
    assert np.array_equal(obpg.similarity_pairs(cv, pav, cp), pk(g["similarity_pairs"]))
    assert np.array_equal(obpg.complementary_pairs(cv, pav, cp), pk(g["complementary_pairs"]))
    assert np.array_equal(obpg.exclusive_co_purchase_pairs(cv, cp), pk(g["exclusive_co_purchase"]))
    assert np.array_equal(obpg.co_view_intersection_pairs(cv, pav), pk(g["co_view_intersection"]))
    rowptr, col = obpg.csr_from_keys(cv, n)
    all_keys = np.unique(np.concatenate([cv, pav, cp]))
    rp_all, col_all = obpg.csr_from_keys(all_keys, n)
    for p in g["probe_nodes"]:
        assert np.array_equal(obpg.neighbors(rowptr, col, p), g[f"nbr_cv/{p}"])
        assert np.array_equal(obpg.neighbors(rp_all, col_all, p), g[f"nbr_all/{p}"])
    assert np.array_equal(np.nonzero(g["type_id"] == 0)[0], g["products_of_type0"])
    colptr, row, perm = obpg.csc_from_csr(rowptr, col, n)
    src_of = np.repeat(np.arange(n), np.diff(rowptr))
    assert np.array_equal(src_of[perm], row) and np.array_equal(col[perm], np.repeat(np.arange(n), np.diff(colptr)))


def test_set_bpg_python_restatement_agrees_with_numpy():
    g = load_golden("bpg_c1.npz")
    b = obpg.SetBPG()
    for i in range(len(g["type_id"])):
        b.add_node(i, {"type": int(g["type_id"][i])})
    for t in obpg.EDGE_TYPES:
        for s, d in g["edges/" + t][:3000]:
            b.add_edge(int(s), int(d), t)
    b.add_edge(0, 1, "bogus")
    assert sum(len(v) for v in b.edges.values()) == sum(min(3000, len(g["edges/" + t])) for t in obpg.EDGE_TYPES)
    e = g["edges/co_view"][:3000]
    rowptr, col = obpg.csr_from_keys(obpg.unique_sorted_keys(e[:, 0], e[:, 1]), len(g["type_id"]))
    for p in (0, 1, 5):
        assert sorted(b.get_neighbors(p, "co_view")) == list(obpg.neighbors(rowptr, col, p))


def test_pcompanion_forward_loss_match_reference():
    g = load_golden("pcomp.npz")
    sd = state_dict_from(g, dtype=np.float64)
    out = pcomp.pcompanion_forward(sd, g["query_idx"], g["batch/query_types"], 3)
    close(out["type_similarities"], g["type_similarities"])
    assert np.array_equal(out["complementary_types"], g["complementary_types"])
    close(out["projected_embeddings"], g["projected_embeddings"])
    pos_t, neg_t = g["batch/positive_types"][:, 0], g["batch/negative_types"][:, 0]
    close(pcomp.type_hinge(out["type_similarities"], pos_t, neg_t, 1.0), g["type_loss"])
    pi, ni = g["batch/positive_items"].astype(np.float64), g["batch/negative_items"].astype(np.float64)
    close(pcomp.item_hinge(out["projected_embeddings"], pi, ni, 1.0), g["item_loss"])
    close(pcomp.compute_loss(out, pos_t, neg_t, pi, ni, 0.8, 1.0), g["loss"])
    for k in (1, 3, 10):
        assert abs(pcomp.hit_at_k(g["eval_sims"].astype(np.float64), np.arange(g["eval_sims"].shape[0]), k) - float(g[f"hit@{k}"])) < 1e-6


def test_item_hinge_backward_matches_torch_port_autograd():
    g = load_golden("pcomp.npz")
    proj = torch.tensor(g["projected_embeddings"], dtype=torch.float64, requires_grad=True)
    pi, ni = torch.tensor(g["batch/positive_items"], dtype=torch.float64), torch.tensor(g["batch/negative_items"], dtype=torch.float64)
    dp = torch.norm(proj - pi.unsqueeze(1), dim=-1)
    dn = torch.norm(proj - ni.unsqueeze(1), dim=-1)
    torch.clamp(1.0 - dp + dn, min=0).mean().backward()
    close(pcomp.item_hinge_backward(proj.detach().numpy(), pi.numpy(), ni.numpy(), 1.0), proj.grad.numpy())


def test_hit_at_k_and_retrieval_match_reference():
    g = load_golden("metrics.npz")
    for k in (1, 3, 10, 60):
        assert abs(pcomp.hit_at_k(g["pred"].astype(np.float64), g["gt"], k) - float(g[f"hit@{k}"])) < 1e-6
    s, i = retrieval.masked_topk(g["q"], g["catalog"], 10, g["row_type"], g["type_id"], chunk=128)
    assert np.array_equal(i, g["topk_idx"])           # no ties in random data -> same order as torch.topk
    fin = np.isfinite(g["topk_score"])
    close(s[fin], g["topk_score"][fin], rtol=1e-5, atol=1e-5)
    # sharded merge == unsharded (SURVEY 8e)
    parts = [retrieval.masked_topk(g["q"], g["catalog"][a:b], 10, g["row_type"], g["type_id"][a:b], index_base=a)
             for a, b in ((0, 150), (150, 400))]
    ms, mi = retrieval.merge_topk(np.concatenate([p[0] for p in parts], 1), np.concatenate([p[1] for p in parts], 1), 10)
    assert np.array_equal(mi, i) and np.array_equal(ms, s)


def test_retrieval_ties_break_to_lowest_index():
    rng = np.random.default_rng(1)
    cat = rng.normal(size=(40, 128)).astype(np.float32)
    cat[[3, 17, 29]] = cat[5]                           # four identical products
    q = cat[5:6] * 2
    _, i = retrieval.masked_topk(q, cat, 5)
    top = i[0].tolist()
    dup = [x for x in top if x in (3, 5, 17, 29)]
    assert dup == sorted(dup)


def test_torch_port_state_dict_and_numbers_match_reference():
    g = load_golden("p2v_module.npz")
    cfg = torch_port.default_config(DROPOUT=0.0)
    m = torch_port.PortProduct2Vec(cfg)
    sd = {k: torch.tensor(v) for k, v in state_dict_from(g).items()}
    assert set(sd) == set(m.state_dict())
    m.load_state_dict(sd)
    m.eval()
    with torch.no_grad():
        close(m(torch.tensor(g["anchor"]), torch.tensor(g["neighbors"])).numpy(), g["eval_forward_nbrs"], 1e-5, 1e-6)
    m.train()
    batch = {"anchor": torch.tensor(g["anchor"]), "positive": torch.tensor(g["positive"]),
             "negative": torch.tensor(g["negative"]), "anchor_neighbors": torch.tensor(g["neighbors"])}
    loss = torch_port.port_triplet_loss(m, batch, 1.0)
    loss.backward()
    close(loss.item(), g["train_loss"], 1e-5, 1e-6)
    for k, v in m.named_parameters():
        close(*golden_grad(g, k, v.grad.numpy()), 1e-4, 1e-6)
    gp = load_golden("pcomp.npz")
    sdp = {k: torch.tensor(v) for k, v in state_dict_from(gp).items()}
    pm = torch_port.PortPCompanion(torch_port.default_config(DROPOUT=0.0, NUM_TYPES=40), sdp["product_embeddings.weight"])
    assert set(sdp) == set(pm.state_dict())
    pm.load_state_dict(sdp)
    out = pm(torch.tensor(gp["query_idx"]), torch.tensor(gp["batch/query_types"]))
    l = pm.loss(out, torch.tensor(gp["batch/positive_types"][:, 0]), torch.tensor(gp["batch/negative_types"][:, 0]),
                torch.tensor(gp["batch/positive_items"]), torch.tensor(gp["batch/negative_items"]))
    close(l.item(), gp["loss"], 1e-5, 1e-6)
