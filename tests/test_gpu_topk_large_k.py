"""GPU tests of the large-k top-K selection (32 < k <= 1024): CatalogIndex.topk / pc_topk_by_type, ops.topk_segments /
pc_topk_groups, ops.topk_rows, ops.topk_merge and the public recommend / hit_at_k, compared bit-exactly (scores and
indices) with the oracle or a stable sort."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import retrieval as oret
from test_gpu_parity import dev

pytestmark = pytest.mark.gpu

KS = (33, 64, 100, 257, 1000, 1024)
KMAX = 1024
N_TYPES = 6


def _data():
    """200 k products in 6 types (type 2 empty, type 5 with 20 products), 40 score rows: 12 rows of type 0 (two
    groups), rows asking for the empty type, the small type, a type past n_types and a negative type."""
    rng = np.random.default_rng(11)
    p, r = 200_000, 40
    cat = rng.normal(size=(p, 128)).astype(np.float32)
    type_id = rng.choice(np.array([0, 1, 3, 4], dtype=np.int32), p)
    type_id[rng.choice(p, 20, replace=False)] = 5
    q = rng.normal(size=(r, 128)).astype(np.float32)
    row_type = rng.integers(0, N_TYPES, r).astype(np.int32)
    row_type[row_type == 2] = 1
    row_type[:12] = 0
    row_type[12], row_type[13], row_type[14], row_type[15] = 2, 5, N_TYPES + 1, -1
    return cat, type_id, q, row_type


@pytest.fixture(scope="module")
def data():
    cat, type_id, q, row_type = _data()
    # the oracle's restriction treats row_type < 0 as "no restriction": give such rows a type no product has
    masked_rt = np.where((row_type < 0) | (row_type >= N_TYPES), N_TYPES + 1, row_type).astype(np.int32)
    os_, oi = oret.masked_topk(q, cat, KMAX, masked_rt, type_id)
    us, ui = oret.masked_topk(q[:9], cat, KMAX)          # row_type=None: the whole catalog
    from pcompanion_b200 import CatalogIndex
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=N_TYPES)
    return dict(cat=cat, type_id=type_id, q=q, row_type=row_type, os=os_, oi=oi, us=us, ui=ui, index=index,
                qt=torch.tensor(q, device=dev()), rtt=torch.tensor(row_type, device=dev()))


def _equal(s, i, ref_s, ref_i, what):
    assert np.array_equal(i.cpu().numpy(), ref_i), f"{what}: indices differ"
    assert np.array_equal(s.cpu().numpy(), ref_s), f"{what}: scores differ"


def test_catalog_topk_by_type_matches_the_oracle(data):
    index, qt, rtt = data["index"], data["qt"], data["rtt"]
    for k in KS:
        for splits in (None, 1, 2, 5, 37):
            s, i = index.topk(qt, k, rtt, splits=splits)
            _equal(s, i, data["os"][:, :k], data["oi"][:, :k], f"by_type k={k} splits={splits}")
        assert (i[12] == -1).all() and torch.isinf(s[12]).all()                 # empty type
        assert (i[13, :20] >= 0).all() and (i[13, 20:] == -1).all()             # 20 products < k: padding
        assert (i[14] == -1).all() and (i[15] == -1).all()                      # type outside [0, n_types)
        s2, i2 = index.topk(qt, k, rtt)
        assert torch.equal(s2, s) and torch.equal(i2, i)                        # repeatable
        su, iu = index.topk(qt[:9], k)                                           # row_type=None
        _equal(su, iu, data["us"][:, :k], data["ui"][:, :k], f"unrestricted k={k}")


def test_topk_segments_matches_the_oracle(data):
    from pcompanion_b200 import ops
    index, qt, rt = data["index"], data["qt"], data["row_type"]
    off = index.offsets.cpu().numpy()
    ok = (rt >= 0) & (rt < N_TYPES)
    t = np.where(ok, rt, 0)
    seg_b = torch.tensor(np.where(ok, off[t], 0), dtype=torch.int64, device=dev())
    seg_e = torch.tensor(np.where(ok, off[t + 1], 0), dtype=torch.int64, device=dev())
    for k in (33, 100, 257, 1000):
        for splits in (None, 3):
            s, i = ops.topk_segments(qt, index.catalog, seg_b, seg_e, k, index.members, 0, splits)
            _equal(s, i, data["os"][:, :k], data["oi"][:, :k], f"segments k={k} splits={splits}")


def test_prefix_of_k1024_equals_the_k10_and_k32_paths(data):
    index, qt, rtt = data["index"], data["qt"], data["rtt"]
    s, i = index.topk(qt, 1024, rtt)
    for k in (10, 32):
        sk, ik = index.topk(qt, k, rtt)
        assert torch.equal(s[:, :k], sk) and torch.equal(i[:, :k], ik), k


def test_shard_merge_equals_the_unsharded_result(data):
    from pcompanion_b200 import CatalogIndex, ops
    cat, type_id, qt, rtt = data["cat"], data["type_id"], data["qt"], data["rtt"]
    bounds = [0, 61_000, 140_000, cat.shape[0]]
    shards = [CatalogIndex(torch.tensor(cat[a:b], device=dev()), torch.tensor(type_id[a:b], device=dev()), index_base=a,
                           num_types=N_TYPES) for a, b in zip(bounds[:-1], bounds[1:])]
    for k in (100, 1000):
        parts = [sh.topk(qt, k, rtt) for sh in shards]
        ms, mi = ops.topk_merge(torch.cat([x[0] for x in parts], 1), torch.cat([x[1] for x in parts], 1), k)
        _equal(ms, mi, data["os"][:, :k], data["oi"][:, :k], f"merge k={k}")


def _stream_catalog(p, kind):
    """'rising': score of product p against e0 is p, so every product enters the running list (compaction at its
    highest rate).  'tied': identical rows, so only the index orders the products."""
    if kind == "rising":
        cat = np.zeros((p, 128), np.float32)
        cat[:, 0] = np.arange(p, dtype=np.float32)
        cat[:, 1:] = np.random.default_rng(0).normal(size=(p, 127)).astype(np.float32)
        q = np.zeros((10, 128), np.float32)
        q[:, 0] = np.arange(1, 11, dtype=np.float32)
        return cat, q
    row = np.random.default_rng(1).normal(size=128).astype(np.float32)
    return np.broadcast_to(row, (p, 128)).copy(), np.random.default_rng(2).normal(size=(10, 128)).astype(np.float32)


@pytest.mark.parametrize("kind", ["rising", "tied"])
def test_adversarial_streams(kind):
    from pcompanion_b200 import CatalogIndex, ops
    p = 100_000
    cat, q = _stream_catalog(p, kind)
    type_id = (np.arange(p) % 2).astype(np.int32)                     # two interleaved types of 50 k products
    rt = np.array([0, 1] * 5, np.int32)
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=2)
    qt, rtt = torch.tensor(q, device=dev()), torch.tensor(rt, device=dev())
    os_, oi = oret.masked_topk(q, cat, KMAX, rt, type_id)
    if kind == "rising":
        assert np.array_equal(oi[0, :3], [p - 2, p - 4, p - 6])
    else:
        assert np.array_equal(oi[1, :3], [1, 3, 5])
    off = index.offsets.cpu().numpy()
    seg_b = torch.tensor(off[rt], dtype=torch.int64, device=dev())
    seg_e = torch.tensor(off[rt + 1], dtype=torch.int64, device=dev())
    for k in (33, 100, 1000, 1024):
        for splits in (None, 1, 4):
            s, i = index.topk(qt, k, rtt, splits=splits)
            _equal(s, i, os_[:, :k], oi[:, :k], f"{kind} by_type k={k} splits={splits}")
        s, i = ops.topk_segments(qt, index.catalog, seg_b, seg_e, k, index.members)
        _equal(s, i, os_[:, :k], oi[:, :k], f"{kind} segments k={k}")


def test_topk_rows_is_a_stable_sort_for_large_k():
    from pcompanion_b200 import ops
    rng = np.random.default_rng(6)
    v = rng.integers(-5, 5, size=(33, 3000)).astype(np.float32)       # heavy ties
    ref = np.argsort(-v, axis=1, kind="stable")
    for k in (33, 100, 1000):
        for splits in (None, 4):
            s, i = ops.topk_rows(torch.tensor(v, device=dev()), k, splits)
            assert np.array_equal(i.cpu().numpy(), ref[:, :k]), (k, splits)
            assert np.array_equal(s.cpu().numpy(), np.take_along_axis(v, ref[:, :k], 1).astype(np.float64)), (k, splits)
    s, i = ops.topk_rows(torch.tensor(v[:, :50].copy(), device=dev()), 100)   # cols < k: padding
    assert np.array_equal(i[:, :50].cpu().numpy(), np.argsort(-v[:, :50], axis=1, kind="stable"))
    assert (i[:, 50:] == -1).all() and torch.isinf(s[:, 50:]).all()


def test_hit_at_k_50_equals_torch_topk():
    from pcompanion_b200 import Metrics
    g = torch.Generator(device=dev()).manual_seed(3)
    preds = torch.randn(256, 400, generator=g, device=dev())           # continuous values: no ties
    gt = torch.randint(0, 400, (256,), generator=g, device=dev())
    want = torch.any(torch.topk(preds, 50).indices == gt.unsqueeze(1), dim=1).float().mean().item()
    assert Metrics.hit_at_k(preds, gt, 50) == want
    assert Metrics.hit_at_k(preds, gt, 5000) == 1.0                      # k clipped to the 400 columns


def test_recommend_batch_with_100_recommendations_matches_brute_force():
    """As tests/test_gpu_datapath.py's k=10 check: every type of the C1 graph has fewer than 100 products, so each list
    is the whole type (min(k, len(type_products)) of the reference); every type has at least 37, so 33 fills them."""
    from test_gpu_datapath import c1_bpg, make_cfg
    from pcompanion_b200 import PCompanion, PCompanionInference
    _, ids, bpg = c1_bpg()
    cfg = make_cfg(NUM_TYPES=20)
    torch.manual_seed(0)
    model = PCompanion(cfg, {pid: torch.randn(128) for pid in ids})
    inf = PCompanionInference(None, cfg, bpg, model=model)
    queries = [ids[3], ids[500], ids[999]]
    with torch.no_grad():
        out = inf.model(inf._prepare_input(queries))
    feats = bpg.features.double().cpu().numpy()
    tidx = inf._type_of.numpy()
    lengths = set()
    for n in (100, 33):
        res = inf.recommend_batch(queries, num_recommendations=n)
        for b, r in enumerate(res):
            assert r["complementary_types"] == out["complementary_types"][b].tolist() and len(r["recommendations"]) == 3
            for t, (recs, scs) in enumerate(zip(r["recommendations"], r["scores"])):
                members = np.nonzero(tidx == r["complementary_types"][t])[0]
                proj = out["projected_embeddings"][b, t].double().cpu().numpy()
                sc = feats[members] @ proj
                order = np.lexsort((members, -sc))[:n]
                assert recs == [ids[j] for j in members[order]]
                np.testing.assert_allclose(scs, sc[order], rtol=1e-12)
                lengths.add((n, len(recs) == n))
    assert lengths == {(100, False), (33, True)}
    assert inf.recommend(ids[3], num_recommendations=100)["recommendations"] == \
        inf.recommend_batch([ids[3]], num_recommendations=100)[0]["recommendations"]
    with pytest.raises(ValueError, match="1024"):
        inf.recommend(ids[3], num_recommendations=1025)


def test_k_above_1024_is_refused(data):
    from pcompanion_b200 import ops
    index, qt, rtt = data["index"], data["qt"], data["rtt"]
    with pytest.raises(ValueError, match="1024"):
        index.topk(qt, 1025, rtt)
    with pytest.raises(ValueError, match="1024"):
        ops.topk_by_type(qt, index.catalog, index.offsets, N_TYPES, rtt, 1025, index.members)
    with pytest.raises(ValueError, match="1024"):
        ops.topk_rows(qt, 1025)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _sharded_worker(rank, world, port, results):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    d = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=d)
    try:
        from pcompanion_b200 import CatalogIndex, ShardedCatalog
        cat, type_id, q, row_type = _data()
        bounds = [0, 90_000, cat.shape[0]]
        a, b = bounds[rank], bounds[rank + 1]
        sh = ShardedCatalog(torch.tensor(cat[a:b], device=d), torch.tensor(type_id[a:b], device=d), a, N_TYPES)
        qt, rtt = torch.tensor(q, device=d), torch.tensor(row_type, device=d)
        s, i = sh.topk(qt, 100, rtt)
        fs, fi = CatalogIndex(torch.tensor(cat, device=d), torch.tensor(type_id, device=d), num_types=N_TYPES).topk(qt, 100, rtt)
        results[rank] = "ok" if torch.equal(s, fs) and torch.equal(i, fi) else "FAILED: sharded != unsharded"
    except Exception:  # pragma: no cover
        import traceback
        results[rank] = traceback.format_exc()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_sharded_catalog_k100_equals_single_gpu():
    import torch.multiprocessing as mp
    world = 2
    results = mp.Manager().dict()
    mp.spawn(_sharded_worker, args=(world, _free_port(), results), nprocs=world, join=True)
    assert all(results.get(r) == "ok" for r in range(world)), dict(results)
