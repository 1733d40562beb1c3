"""Graph-native Product2Vec training: pc_triplet_batch_rows, ops.triplet_batch_rows, the epoch plan of
GraphTripletSampler.neighborhood_batches / TripletBatch.build, Product2Vec.triplet_loss_graph and train_model_graph."""
import copy
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from _graph_batch_oracle import batch_rows_reference, step_grads_f64, step_reference_f64

gpu = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _cfg(**over):
    from test_gpu_parity import make_cfg
    return make_cfg(**over)


def _csr(rowptr, col, n):
    from pcompanion_b200 import ops
    return ops.CSRGraph(torch.as_tensor(rowptr, device=_dev()), torch.as_tensor(col, device=_dev()), n, n)


def _ring_bpg(n, d, feats=None):
    """Every product i has the co-view neighbours i+1 .. i+d (mod n), all of them also purchase-after-view: every
    co-view edge is a similarity pair and every anchor has degree d."""
    from pcompanion_b200 import BehaviorProductGraph
    src = torch.arange(n, dtype=torch.int32).repeat_interleave(d)
    dst = ((src.long() + torch.arange(1, d + 1).repeat(n)) % n).to(torch.int32)
    if feats is None:
        feats = torch.randn(n, 128, generator=torch.Generator().manual_seed(n + d))
    return BehaviorProductGraph.from_arrays(n, {"co_view": (src, dst), "purchase_after_view": (src, dst)}, feats, None, _dev())


def _drop_in_step(model, x, csr, batch):
    """The drop-in step (forward(anchor, neighbours[B, d, D]), forward(positive), forward(negative), triplet_loss) for a
    batch whose anchors all have the same degree d >= 1: no padding rows."""
    b = batch.anchor.numel()
    d = batch.n_nbr // b
    starts = csr.rowptr[batch.anchor]
    nbrs = csr.col[(starts.unsqueeze(1) + torch.arange(d, device=x.device)).reshape(-1)].long()
    a = model(x[batch.anchor], x[nbrs].view(b, d, x.shape[1]))
    p = model(x[batch.positive])
    n = model(x[batch.negatives])
    return model.triplet_loss(a, p, n)


def _bn_state(m):
    bn = m.ffn[1]
    return bn.running_mean, bn.running_var, bn.num_batches_tracked


# ----------------------------------------------------------------------------- (a) kernel
def _random_graph(n, rng, hub_row=3, hub_deg=300):
    deg = rng.poisson(6, n)
    deg[::5] = 0
    deg[hub_row] = hub_deg
    rowptr = np.zeros(n + 1, np.int64)
    np.cumsum(deg, out=rowptr[1:])
    col = np.concatenate([np.sort(rng.choice(n, k, replace=False)) for k in deg]).astype(np.int32)
    return rowptr, col


@gpu
@pytest.mark.parametrize("dim,batch", [(128, 517), (4, 300), (1024, 64), (128, 1), (128, 70_000)])
def test_batch_rows_kernel_equals_torch_gather(dim, batch):
    from pcompanion_b200 import TripletBatch, ops
    rng = np.random.default_rng(dim + batch)
    n = 3000
    rowptr, col = _random_graph(n, rng)
    csr = _csr(rowptr, col, n)
    # a strided table (row stride dim + 8 floats) standing in for a column slice of a wider feature matrix
    buf = torch.randn(n, dim + 8, device=_dev())
    x = buf[:, 4:4 + dim]
    anchor = torch.as_tensor(rng.integers(0, n, batch), device=_dev())
    if batch > 4:
        anchor[:4] = torch.tensor([3, 0, 3, 5], device=_dev())          # the hub (twice) and two zero-degree anchors
    positive = torch.as_tensor(rng.integers(0, n, batch), device=_dev())
    negatives = torch.as_tensor(rng.integers(0, n, (batch, 5)), device=_dev())
    tb = TripletBatch.build(csr, anchor, positive, negatives)
    rows, nbr_ptr, edge_row = batch_rows_reference(x, csr.rowptr, csr.col, anchor, positive, negatives)
    assert torch.equal(tb.nbr_ptr, nbr_ptr) and tb.n_nbr == int(nbr_ptr[-1])
    a_rows, nbr_rows, p_rows, n_rows, g = ops.triplet_batch_rows(x, csr, *tb)
    got = torch.cat([a_rows, nbr_rows, p_rows, n_rows])
    assert all(t.is_contiguous() for t in (a_rows, nbr_rows, p_rows, n_rows))
    assert torch.equal(got, rows)
    colptr, row = g.transposed()
    assert torch.equal(row, edge_row) and torch.equal(colptr, torch.arange(tb.n_nbr + 1, device=_dev()))
    assert torch.equal(g.rowptr, nbr_ptr) and torch.equal(g.col, torch.arange(tb.n_nbr, dtype=torch.int32, device=_dev()))
    assert (g.n_rows, g.n_cols) == (batch, tb.n_nbr)
    assert g.split_hubs                                                  # row 3 is a hub of the full CSR


@gpu
def test_batch_rows_refuses_bad_arguments():
    from pcompanion_b200 import TripletBatch, _lib, ops
    rowptr, col = _random_graph(50, np.random.default_rng(0), hub_deg=7)
    csr = _csr(rowptr, col, 50)
    x = torch.randn(50, 132, device=_dev())
    idx = torch.arange(8, device=_dev())
    tb = TripletBatch.build(csr, idx, idx, idx.view(8, 1).repeat(1, 3))
    assert not ops.triplet_batch_rows(x[:, :128], csr, *tb)[4].split_hubs       # no hub rows: the batch graph never splits
    with pytest.raises(RuntimeError, match="bad dim"):
        ops.triplet_batch_rows(x[:, :6], csr, *tb)                               # dim % 4 != 0
    with pytest.raises(RuntimeError, match="bad dim"):
        ops.triplet_batch_rows(torch.randn(50, 1028, device=_dev()), csr, *tb)  # dim > 1024
    with pytest.raises(RuntimeError, match="aligned"):
        ops.triplet_batch_rows(x[:, 1:129], csr, *tb)
    with pytest.raises(RuntimeError, match="bad sizes"):
        ops.triplet_batch_rows(x[:, :128], csr, tb.anchor, tb.positive, tb.negatives[:, :0], tb.nbr_ptr, tb.n_nbr)
    with pytest.raises(ValueError, match="expected"):
        ops.triplet_batch_rows(x[:, :128], csr, tb.anchor, tb.positive[:4], tb.negatives, tb.nbr_ptr, tb.n_nbr)
    p = ctypes.c_void_p(x.data_ptr())
    lib = _lib.LIB
    assert lib.pc_triplet_batch_rows(None, 128, 128, p, p, p, 8, 3, p, p, p, 4, p, p, None) == 1     # null table
    assert lib.pc_triplet_batch_rows(p, 128, 128, p, p, p, 8, 3, p, None, p, 4, p, p, None) == 1     # null col
    assert lib.pc_triplet_batch_rows(p, 124, 128, p, p, p, 8, 3, p, p, p, 4, p, p, None) == 1        # ld < dim
    assert lib.pc_triplet_batch_rows(p, 128, 128, p, p, p, -1, 3, p, p, p, 4, p, p, None) == 1       # batch < 0
    assert lib.pc_triplet_batch_rows(p, 128, 128, p, p, p, 8, 3, p, p, p, 1 << 31, p, p, None) == 1  # n_nbr >= 2^31
    assert lib.pc_triplet_batch_rows(None, 128, 128, None, None, None, 0, 3, None, None, None, 0, None, None, None) == 0


# ----------------------------------------------------------------------------- (b) parity with the drop-in step
@gpu
def test_equal_degree_batch_is_bit_identical_to_the_drop_in_step():
    from pcompanion_b200 import GraphTripletSampler, Product2Vec
    bpg = _ring_bpg(200, 7)
    csr, x = bpg.csr("co_view"), bpg.features
    torch.manual_seed(0)
    m1 = Product2Vec(_cfg()).to(_dev()).train()
    m2 = copy.deepcopy(m1)
    smp = GraphTripletSampler(bpg)
    batches = list(smp.neighborhood_batches(64, seed=5, csr=csr))
    assert len(batches) == 22 and all(b.n_nbr == 7 * b.anchor.numel() for b in batches)
    for batch in batches[:2]:                                                   # two steps: running statistics accumulate
        l1 = m1.triplet_loss_graph(x, csr, batch)
        l2 = _drop_in_step(m2, x, csr, batch)
        m1.zero_grad(); m2.zero_grad()
        l1.backward(); l2.backward()
        assert torch.equal(l1, l2)
        for (k, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
            assert torch.equal(p1.grad, p2.grad), k
        for s1, s2 in zip(_bn_state(m1), _bn_state(m2)):
            assert torch.equal(s1, s2)
    assert int(m1.ffn[1].num_batches_tracked) == 8                              # four FFN calls per step


# ----------------------------------------------------------------------------- (c) ragged degrees vs float64
@gpu
def test_ragged_batch_matches_float64_oracle_and_autograd():
    from pcompanion_b200 import GraphTripletSampler, Product2Vec, TripletBatch
    from oracle import torch_port
    from test_gpu_datapath import c1_bpg
    from test_gpu_parity import close
    _, _, bpg = c1_bpg()
    csr, x = bpg.csr("co_view"), bpg.features
    rowptr, col = csr.rowptr.cpu().numpy(), csr.col.cpu().numpy()
    deg = np.diff(rowptr)
    smp = GraphTripletSampler(bpg)
    a, p, n, _, _ = next(smp.neighborhood_batches(256, seed=2, csr=csr))
    zero = torch.as_tensor(np.flatnonzero(deg == 0)[:16], device=_dev())
    assert zero.numel() == 16
    a = a.clone()
    a[::16] = zero                                                              # 16 anchors without co-view neighbours
    batch = TripletBatch.build(csr, a, p, n)
    a_, p_, n_ = a.cpu().numpy(), p.cpu().numpy(), n.cpu().numpy()
    assert (deg[a_] == 0).sum() >= 16 and len(set(deg[a_].tolist())) > 5
    torch.manual_seed(3)
    m = Product2Vec(_cfg()).to(_dev()).train()
    sd = {k: v.detach().double().cpu().numpy() for k, v in m.state_dict().items()}
    port = torch_port.PortProduct2Vec(torch_port.default_config(DROPOUT=0.0)).double().train()
    port.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    loss = m.triplet_loss_graph(x, csr, batch)
    loss.backward()
    x64 = x.double().cpu().numpy()
    ref_loss, ref_rm, ref_rv = step_reference_f64(sd, x64, rowptr, col, a_, p_, n_, 4, 1.0)
    close(loss, ref_loss, what="loss")
    close(m.ffn[1].running_mean, ref_rm, what="running_mean")
    close(m.ffn[1].running_var, ref_rv, what="running_var")
    grads = step_grads_f64(port, x64, rowptr, col, a_, p_, n_, 1.0)
    for k, v in m.named_parameters():
        # ffn.0.bias sits in front of BatchNorm: its gradient is mathematically zero, both sides hold summation noise there
        close(v.grad, grads[k], atol=3e-6 if k == "ffn.0.bias" else 1e-7, what="grad " + k)


# ----------------------------------------------------------------------------- (d) edge cases
@gpu
def test_batch_without_neighbour_rows_is_ffn_only():
    from pcompanion_b200 import Product2Vec, TripletBatch
    from test_gpu_datapath import c1_bpg
    _, _, bpg = c1_bpg()
    csr, x = bpg.csr("co_view"), bpg.features
    zero = torch.nonzero(csr.rowptr[1:] == csr.rowptr[:-1]).squeeze(1)[:32]
    p = torch.arange(32, device=_dev())
    n = torch.arange(160, device=_dev()).view(32, 5)
    batch = TripletBatch.build(csr, zero, p, n)
    assert batch.n_nbr == 0
    torch.manual_seed(0)
    m1 = Product2Vec(_cfg()).to(_dev()).train()
    m2 = copy.deepcopy(m1)
    l1 = m1.triplet_loss_graph(x, csr, batch)
    l2 = m2.triplet_loss(m2(x[zero]), m2(x[p]), m2(x[n]))
    l1.backward(); l2.backward()
    assert torch.equal(l1, l2)
    for (k, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        assert (p1.grad is None and p2.grad is None) or torch.equal(p1.grad, p2.grad), k
    for s1, s2 in zip(_bn_state(m1), _bn_state(m2)):
        assert torch.equal(s1, s2)
    assert int(m1.ffn[1].num_batches_tracked) == 3                              # no neighbour FFN call


@gpu
def test_single_row_ffn_call_raises_batchnorm_value_error():
    from pcompanion_b200 import Product2Vec, TripletBatch
    from test_gpu_datapath import c1_bpg
    _, _, bpg = c1_bpg()
    csr, x = bpg.csr("co_view"), bpg.features
    deg = csr.rowptr[1:] - csr.rowptr[:-1]
    m = Product2Vec(_cfg()).to(_dev()).train()
    one = torch.tensor([3], device=_dev())
    with pytest.raises(ValueError, match="Expected more than 1 value per channel"):      # one anchor
        m.triplet_loss_graph(x, csr, TripletBatch.build(csr, one, one + 1, torch.arange(5, device=_dev()).view(1, 5)))
    a = torch.cat([torch.nonzero(deg == 1).squeeze(1)[:1], torch.nonzero(deg == 0).squeeze(1)[:3]])
    batch = TripletBatch.build(csr, a, a + 1, torch.arange(20, device=_dev()).view(4, 5))
    assert batch.n_nbr == 1
    with pytest.raises(ValueError, match="Expected more than 1 value per channel"):      # one neighbour row in the batch
        m.triplet_loss_graph(x, csr, batch)


@gpu
def test_hub_anchors_split_match_the_unsplit_drop_in_step():
    from pcompanion_b200 import GraphTripletSampler, Product2Vec, ops
    from test_gpu_parity import close
    bpg = _ring_bpg(400, 300)                                                   # every anchor is a hub (degree 300 > 256)
    csr, x = bpg.csr("co_view"), bpg.features
    assert csr.hub_split() is not None
    batch = next(GraphTripletSampler(bpg, k_neg=5).neighborhood_batches(16, seed=1, csr=csr))
    assert ops.triplet_batch_rows(x, csr, *batch)[4].hub_split() is not None
    torch.manual_seed(0)
    m1 = Product2Vec(_cfg()).to(_dev()).train()
    m2 = copy.deepcopy(m1)
    l1 = m1.triplet_loss_graph(x, csr, batch)
    l2 = _drop_in_step(m2, x, csr, batch)                                      # regular graph: never split
    l1.backward(); l2.backward()
    close(l1, l2.item(), what="loss")
    for (k, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        close(p1.grad, p2.grad.cpu().numpy(), atol=3e-6 if k == "ffn.0.bias" else 1e-7, what="grad " + k)
    for s1, s2 in zip(_bn_state(m1), _bn_state(m2)):
        assert torch.equal(s1, s2)                                              # the FFN calls see the same rows


@gpu
def test_degenerate_graphs_raise_the_sampler_value_error():
    from pcompanion_b200 import BehaviorProductGraph, Product2Vec
    m = Product2Vec(_cfg(BATCH_SIZE=4)).to(_dev())
    opt = torch.optim.Adam(m.parameters())
    src = torch.tensor([0, 1, 2], dtype=torch.int32)
    dst = torch.tensor([1, 2, 3], dtype=torch.int32)
    no_pairs = BehaviorProductGraph.from_arrays(8, {"co_view": (src, dst)}, torch.randn(8, 128), None, _dev())
    with pytest.raises(ValueError, match="No similarity pairs"):
        m.train_model_graph(no_pairs, opt, num_epochs=1)
    k = 6                                                                       # every other product is similar to 0
    s, d = torch.zeros(k - 1, dtype=torch.int32), torch.arange(1, k, dtype=torch.int32)
    tiny = BehaviorProductGraph.from_arrays(k, {"co_view": (s, d), "purchase_after_view": (s[:-2], d[:-2])},
                                            torch.randn(k, 128), None, _dev())
    with pytest.raises(ValueError, match="fewer than 5 eligible negatives"):
        m.train_model_graph(tiny, opt, num_epochs=1)


# ----------------------------------------------------------------------------- (e) the loop
@gpu
def test_neighborhood_batches_follow_epoch():
    from pcompanion_b200 import GraphTripletSampler
    from test_gpu_datapath import c1_bpg
    _, _, bpg = c1_bpg()
    csr = bpg.csr("co_view")
    smp = GraphTripletSampler(bpg)
    ref = list(smp.epoch(100, seed=9))
    got = list(smp.neighborhood_batches(100, seed=9, csr=csr))
    assert len(ref) == len(got) == -(-len(smp) // 100)
    for (a, p, n), b in zip(ref, got):
        assert torch.equal(a, b.anchor) and torch.equal(p, b.positive) and torch.equal(n, b.negatives)
        deg = csr.rowptr[a + 1] - csr.rowptr[a]
        assert b.nbr_ptr[0] == 0 and torch.equal(b.nbr_ptr[1:] - b.nbr_ptr[:-1], deg) and b.n_nbr == int(deg.sum())


@gpu
def test_train_model_graph_returns_train_model_embeddings_and_is_reproducible():
    from pcompanion_b200 import Product2Vec
    from test_gpu_datapath import c1_bpg
    _, ids, bpg = c1_bpg()

    def run(dropout):
        torch.manual_seed(0)
        m = Product2Vec(_cfg(DROPOUT=dropout, BATCH_SIZE=256)).to(_dev())
        before = [q.detach().clone() for q in m.parameters()]
        emb = m.train_model_graph(bpg, torch.optim.Adam(m.parameters(), lr=1e-3), num_epochs=2, seed=4)
        return m, before, emb

    m, before, emb = run(0.0)
    assert list(emb.keys()) == ids == list(bpg.nodes.keys())                   # train_model's return: bpg.nodes order
    assert all(v.shape == (128,) and v.device.type == "cpu" and torch.isfinite(v).all() for v in emb.values())
    assert any(not torch.equal(a, b) for a, b in zip(before, m.parameters()))
    assert not m.training
    for dropout in (0.0, 0.1):
        m1, _, _ = run(dropout)
        m2, _, _ = run(dropout)
        for (k, p1), (_, p2) in zip(m1.state_dict().items(), m2.state_dict().items()):
            assert torch.equal(p1, p2), (dropout, k)


@gpu
def test_batch_loop_does_not_synchronise():
    from pcompanion_b200 import GraphTripletSampler, Product2Vec
    from test_gpu_datapath import c1_bpg
    _, _, bpg = c1_bpg()
    csr, x = bpg.csr("co_view"), bpg.features
    torch.manual_seed(0)
    m = Product2Vec(_cfg(DROPOUT=0.1)).to(_dev()).train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    smp = GraphTripletSampler(bpg)
    batches = smp.neighborhood_batches(256, seed=0, csr=csr)
    first = next(batches)                                                       # the epoch's one planning read
    total = torch.zeros((), device=_dev())
    steps = 0
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for batch in [first, *batches]:
            loss = m.triplet_loss_graph(x, csr, batch)
            opt.zero_grad()
            loss.backward()
            opt.step()
            total += loss.detach()
            steps += 1
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert steps == -(-len(smp) // 256) and torch.isfinite(total)


# ----------------------------------------------------------------------------- (f) build
def test_batch_rows_kernel_compiles_for_sm100a_without_spills():
    import __graft_entry__ as ge
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([ge.NVCC, *ge.NVCC_FLAGS, "-Xptxas", "-v", "-c", os.path.join(ge.CSRC, "sample.cu"), "-o",
                            os.path.join(tmp, "sample.o")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    m = re.search(r"Compiling entry function '\S*triplet_batch_rows_kernel\S*' for 'sm_100a'.*?\n.*?\n\s*(\d+) bytes stack "
                  r"frame, (\d+) bytes spill stores, (\d+) bytes spill loads", r.stdout)
    assert m, r.stdout
    assert m.groups() == ("0", "0", "0")
