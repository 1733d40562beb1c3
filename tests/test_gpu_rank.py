"""GPU tests of the exact target rank (pc_rank_by_type): CatalogIndex.rank against the reference rank, its agreement with
the top-K lists for k up to 1024, adversarial catalogs, launch chunking, shard sums, ShardedCatalog on two GPUs, and
PCompanionInference.rank_targets / evaluate end to end.  Ranks are integers and are compared exactly."""
import os

import numpy as np
import pytest
import torch

from _rank_oracle import masked_rank
from oracle.retrieval import scores_fp64
from test_gpu_parity import dev
from test_gpu_topk_large_k import N_TYPES, _data, _free_port, _stream_catalog

pytestmark = pytest.mark.gpu

# row -> position in its top-1024 list whose product becomes the row's target (row 13 ranks the 20-product type)
PICKS = {0: 0, 1: 1, 2: 9, 3: 10, 4: 31, 5: 32, 6: 99, 7: 100, 8: 1023, 9: 500, 13: 7}


def _targets(cat, type_id, row_type, top):
    """A random member of each row's type (any product for rows without products of their type), the products at the
    PICKS positions of the row's top list, three targets outside the catalog and two of another type."""
    rng = np.random.default_rng(5)
    p = cat.shape[0]
    t = np.empty(len(row_type), np.int64)
    for r, rt in enumerate(row_type):
        m = np.nonzero(type_id == rt)[0]
        t[r] = rng.choice(m) if m.size else rng.integers(0, p)
    for r, j in PICKS.items():
        t[r] = top[r, j]
    t[20], t[21], t[22] = -3, p, p + 1000
    for r in (23, 24):
        t[r] = rng.choice(np.nonzero(type_id != row_type[r])[0])
    return t


@pytest.fixture(scope="module")
def data():
    from pcompanion_b200 import CatalogIndex
    cat, type_id, q, row_type = _data()
    assert all(0 <= row_type[r] < N_TYPES and row_type[r] != 2 for r in range(16, 40))
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=N_TYPES)
    qt, rtt = torch.tensor(q, device=dev()), torch.tensor(row_type, device=dev())
    top = index.topk(qt, 1024, rtt)[1].cpu().numpy()          # only picks targets near the top of each list
    targets = _targets(cat, type_id, row_type, top)
    plain = np.random.default_rng(6).integers(0, cat.shape[0], 9)
    plain[0] = index.topk(qt[:1], 3)[1][0, 2].item()          # third of the unrestricted list
    return dict(cat=cat, type_id=type_id, q=q, row_type=row_type, index=index, qt=qt, rtt=rtt, targets=targets,
                tt=torch.tensor(targets, device=dev()), oracle=masked_rank(q, cat, targets, row_type, type_id),
                plain=plain, oracle_plain=masked_rank(q[:9], cat, plain))


def test_rank_matches_the_oracle(data):
    index, qt, rtt, tt, want = data["index"], data["qt"], data["rtt"], data["tt"], data["oracle"]
    for r, j in PICKS.items():
        assert want[r] == j, (r, j)                            # the reference agrees with the top-K list it was picked from
    assert (want[[12, 14, 15, 20, 21, 22, 23, 24]] == -1).all()
    assert (want[16:20] >= 0).all() and (want[25:] >= 0).all()
    for splits in (None, 1, 4, 37):
        got = index.rank(qt, tt, rtt, splits=splits)
        assert np.array_equal(got.cpu().numpy(), want), f"splits={splits}"
        assert torch.equal(index.rank(qt, tt, rtt, splits=splits), got), f"splits={splits}: repeated call differs"
    plain = torch.tensor(data["plain"], device=dev())
    for splits in (None, 1, 4, 37):
        whole = index.rank(qt[:9], plain, splits=splits)              # row_type=None: the whole catalog
        assert np.array_equal(whole.cpu().numpy(), data["oracle_plain"]) and whole[0].item() == 2, f"splits={splits}"


def test_kernel_gives_minus_one_only_for_rows_without_a_valid_type(data):
    """pc_rank_by_type does not check membership: it counts for every row of a valid type, and -1 is the row type's."""
    from pcompanion_b200 import ops
    index, qt, rtt, tt, want = data["index"], data["qt"], data["rtt"], data["tt"], data["oracle"]
    rows = index.catalog[tt.clamp(0, data["cat"].shape[0] - 1)]
    for splits in (1, 5):
        counts = ops.rank_by_type(qt, index.catalog, index.offsets, N_TYPES, rtt, rows, tt, index.members, 0, splits).cpu().numpy()
        member = want >= 0
        assert np.array_equal(counts[member], want[member]), f"splits={splits}"
        assert (counts[[12, 14, 15]] == [0, -1, -1]).all(), f"splits={splits}"   # empty type: nothing ranks before
        assert (counts[[20, 21, 22, 23, 24]] >= 0).all(), f"splits={splits}"


@pytest.mark.parametrize("k", [1, 10, 32, 33, 100, 1024])
def test_rank_agrees_with_topk(data, k):
    index, qt, rtt, tt = data["index"], data["qt"], data["rtt"], data["tt"]
    for rows, targets, row_type in ((slice(None), tt, rtt), (slice(0, 9), torch.tensor(data["plain"], device=dev()), None)):
        ranks = index.rank(qt[rows], targets, row_type).cpu()
        _, idx = index.topk(qt[rows], k, row_type)
        hit = (idx.cpu() == targets.cpu()[:, None])
        listed = hit.any(1)
        assert torch.equal(listed, (ranks >= 0) & (ranks < k)), f"k={k}"
        assert torch.equal(hit.int().argmax(1)[listed], ranks[listed]), f"k={k}: position"
        if row_type is not None:
            assert int(listed[list(PICKS)].sum()) == sum(j < k for j in PICKS.values()), f"k={k}"


def test_rank_without_type_ids_is_refused_for_typed_rows(data):
    from pcompanion_b200 import CatalogIndex
    plain = CatalogIndex(data["index"].catalog)
    with pytest.raises(ValueError, match="without type ids"):
        plain.rank(data["qt"], data["tt"], data["rtt"])
    with pytest.raises(ValueError, match="targets"):
        data["index"].rank(data["qt"], data["tt"][:5], data["rtt"])
    empty = CatalogIndex(torch.empty(0, 128, device=dev()))             # an empty shard holds no target
    assert (empty.rank(data["qt"], data["tt"]) == -1).all()


@pytest.mark.parametrize("kind", ["rising", "tied"])
def test_adversarial_catalogs(kind):
    from pcompanion_b200 import CatalogIndex, ops
    p = 100_000
    cat, q = _stream_catalog(p, kind)
    type_id = (np.arange(p) % 2).astype(np.int32)                     # two interleaved types of 50 k products
    rt = np.array([0, 1] * 5, np.int32)
    position = np.array([0, 1, 17, 31, 32, 1000, 1023, 20_000, 49_998, 49_999])
    targets = rt + 2 * position                                         # the position-th member of the row's type
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=2)
    qt, rtt, tt = torch.tensor(q, device=dev()), torch.tensor(rt, device=dev()), torch.tensor(targets, device=dev())
    want = position if kind == "tied" else masked_rank(q, cat, targets, rt, type_id)
    if kind == "tied":
        assert np.array_equal(masked_rank(q, cat, targets, rt, type_id), want)
    for splits in (None, 1, 4):
        got = ops.rank_by_type(qt, index.catalog, index.offsets, 2, rtt, index.catalog[tt], tt, index.members, 0, splits)
        assert np.array_equal(got.cpu().numpy(), want), f"{kind} splits={splits}"
    assert np.array_equal(index.rank(qt, tt, rtt).cpu().numpy(), want)


def test_more_than_65535_score_rows():
    from pcompanion_b200 import CatalogIndex
    rng = np.random.default_rng(8)
    p, r = 1500, 70_000
    cat = rng.normal(size=(p, 16)).astype(np.float32)
    type_id = rng.integers(0, 3, p).astype(np.int32)
    q = rng.normal(size=(r, 16)).astype(np.float32)
    row_type = rng.integers(0, 3, r).astype(np.int32)
    row_type[::1000] = 3                                               # past n_types
    members = [np.nonzero(type_id == t)[0] for t in range(3)]
    targets = np.array([rng.choice(members[t]) if t < 3 else 0 for t in row_type])
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=3)
    got = index.rank(torch.tensor(q, device=dev()), torch.tensor(targets, device=dev()), torch.tensor(row_type, device=dev()))
    want = np.concatenate([masked_rank(q[a:a + 10_000], cat, targets[a:a + 10_000], row_type[a:a + 10_000], type_id)
                           for a in range(0, r, 10_000)])
    assert np.array_equal(got.cpu().numpy(), want)
    assert (want[::1000] == -1).all() and (want[1:1000] >= 0).all()


def test_shard_counts_add_up_to_the_unsharded_rank(data):
    from pcompanion_b200 import CatalogIndex, ops
    cat, type_id, qt, rtt, tt = data["cat"], data["type_id"], data["qt"], data["rtt"], data["tt"]
    want = data["oracle"]
    bounds = [0, 61_000, 140_000, cat.shape[0]]
    shards = [CatalogIndex(torch.tensor(cat[a:b], device=dev()), torch.tensor(type_id[a:b], device=dev()), index_base=a,
                           num_types=N_TYPES) for a, b in zip(bounds[:-1], bounds[1:])]
    rows = data["index"].catalog[tt.clamp(0, cat.shape[0] - 1)]       # the owner's row of every target
    total = sum(ops.rank_by_type(qt, sh.catalog, sh.offsets, N_TYPES, rtt, rows, tt, sh.members, sh.index_base).clamp_min(0)
                for sh in shards)
    member = want >= 0
    assert np.array_equal(total.cpu().numpy()[member], want[member])
    owned = torch.stack([sh.rank(qt, tt, rtt) for sh in shards])       # each target belongs to at most one shard
    assert ((owned >= 0).sum(0) == torch.tensor(member.astype(np.int64), device=dev())).all()


def _sharded_rank_worker(rank, world, port, results):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    d = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=d)
    try:
        from pcompanion_b200 import CatalogIndex, ShardedCatalog
        cat, type_id, q, row_type = _data()
        targets = np.random.default_rng(9).integers(-10, cat.shape[0] + 10, len(row_type))
        targets[:12] = [np.random.default_rng(r).choice(np.nonzero(type_id == 0)[0]) for r in range(12)]
        bounds = [0, 90_000, cat.shape[0]]
        a, b = bounds[rank], bounds[rank + 1]
        sh = ShardedCatalog(torch.tensor(cat[a:b], device=d), torch.tensor(type_id[a:b], device=d), a, N_TYPES)
        qt, rtt, tt = torch.tensor(q, device=d), torch.tensor(row_type, device=d), torch.tensor(targets, device=d)
        full = CatalogIndex(torch.tensor(cat, device=d), torch.tensor(type_id, device=d), num_types=N_TYPES)
        ok = torch.equal(sh.rank(qt, tt, rtt), full.rank(qt, tt, rtt)) and torch.equal(sh.rank(qt, tt), full.rank(qt, tt))
        ok = ok and bool((full.rank(qt, tt, rtt)[:12] >= 0).all())
        results[rank] = "ok" if ok else "FAILED: sharded != unsharded"
    except Exception:  # pragma: no cover
        import traceback
        results[rank] = traceback.format_exc()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_sharded_rank_equals_single_gpu():
    import torch.multiprocessing as mp
    world = 2
    results = mp.Manager().dict()
    mp.spawn(_sharded_rank_worker, args=(world, _free_port(), results), nprocs=world, join=True)
    assert all(results.get(r) == "ok" for r in range(world)), dict(results)


def test_inference_rank_targets_and_evaluate():
    """C1 graph: ranks equal a brute force over the predicted type's members, a rank below 100 is the target's position
    in recommend(query, 100), and evaluate() is rank_metrics of those ranks plus the type recall."""
    from test_gpu_datapath import c1_bpg, make_cfg
    from pcompanion_b200 import Metrics, PCompanion, PCompanionInference
    _, ids, bpg = c1_bpg()
    cfg = make_cfg(NUM_TYPES=20)
    torch.manual_seed(0)
    model = PCompanion(cfg, {pid: torch.randn(128) for pid in ids})
    inf = PCompanionInference(None, cfg, bpg, model=model)
    rng = np.random.default_rng(10)
    q_idx = rng.choice(len(ids), 48, replace=False)
    queries = [ids[i] for i in q_idx]
    with torch.no_grad():
        out = inf.model(inf._prepare_input(queries))
    comp = out["complementary_types"].cpu().numpy()
    proj = out["projected_embeddings"].cpu().numpy()
    feats = bpg.features.float().cpu().numpy()
    tidx = inf._type_of.numpy()
    t_idx = []
    for b in range(len(queries)):
        if b % 4 == 3:
            t_idx.append(int(rng.integers(0, len(ids))))               # any product: its type may not be predicted
        else:
            m = np.nonzero(tidx == comp[b, b % 3])[0]                  # a member of a predicted type
            t_idx.append(int(m[0]) if b % 8 == 0 else int(rng.choice(m)))
    targets = [ids[j] for j in t_idx]
    ranks, slots = inf.rank_targets(queries, targets)
    ranks, slots = ranks.cpu().numpy(), slots.cpu().numpy()
    for b, g in enumerate(t_idx):
        hits = np.nonzero(comp[b] == tidx[g])[0]
        assert slots[b] == (hits[0] if hits.size else -1), b
        if not hits.size:
            assert ranks[b] == -1
            continue
        members = np.nonzero(tidx == tidx[g])[0]
        sc = scores_fp64(proj[b, hits[0]][None, :], feats[members])[0]
        s_t = sc[members == g][0]
        assert ranks[b] == int(((sc > s_t) | ((sc == s_t) & (members < g))).sum()), b
    assert (slots >= 0).sum() >= 36 and ((ranks >= 0) & (ranks < 100)).sum() > 0
    res = inf.recommend_batch(queries, num_recommendations=100)
    for b in np.nonzero((ranks >= 0) & (ranks < 100))[0]:
        assert res[b]["recommendations"][slots[b]][ranks[b]] == targets[b], b
    m = inf.evaluate(queries, targets)
    want = Metrics.rank_metrics(torch.tensor(ranks))
    want["type_recall"] = float((slots >= 0).mean())
    assert m == pytest.approx(want, abs=0, rel=1e-15)
    with pytest.raises(ValueError, match="not found"):
        inf.rank_targets([queries[0]], ["no-such-product"])
    with pytest.raises(ValueError, match="not found"):
        inf.evaluate(["no-such-product"], [targets[0]])


def test_rank_metrics_has_no_k_limit(data):
    from pcompanion_b200 import Metrics
    ranks = data["index"].rank(data["qt"], data["tt"], data["rtt"])
    want = float(((ranks >= 0) & (ranks < 5000)).double().mean().item())
    assert 0 < want < 1
    assert Metrics.rank_metrics(ranks, ks=(5000,))["hit@5000"] == want
