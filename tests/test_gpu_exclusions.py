"""GPU tests of exclusion lists (pc_topk_by_type_excluding, pc_rank_remove_excluded): filtered top-K and filtered rank
against the references, the rank / top-K property, an over-fetch cross-check, adversarial catalogs, launch chunking,
shards, and PCompanionInference end to end.  Indices and scores are compared bit-exactly, ranks exactly."""
import os

import numpy as np
import pytest
import torch

from _exclusion_oracle import masked_rank_excluding, masked_topk_excluding
from _rank_oracle import masked_rank
from oracle.retrieval import scores_fp64
from test_gpu_parity import dev
from test_gpu_topk_large_k import N_TYPES, _data, _free_port, _stream_catalog

pytestmark = pytest.mark.gpu

KS = (1, 10, 32, 33, 100, 1024)
M_TOP = {1: 1, 2: 31, 3: 32, 4: 33, 5: 500}        # row -> exclude its own true top-m


def _lists(cat, type_id, row_type, top, targets=None):
    """One list per row (plus a shared list 40) and a row_list: empty lists, own top-m, random same-type products,
    other-type / outside indices, duplicates, a whole type (row 13 ranks the 20-product type), many rows sharing
    list 40, row_list entries past the lists and negative.  With targets, most lists also name the row's target."""
    rng = np.random.default_rng(21)
    p = cat.shape[0]
    lists = []
    for r, rt in enumerate(row_type):
        same = np.nonzero(type_id == rt)[0]
        if r == 0:
            e = []
        elif r in M_TOP:
            e = list(top[r, :M_TOP[r]])
        elif r == 7:
            e = [-5, p, p + 100] + list(np.nonzero(type_id != rt)[0][:50])    # nothing of the row's run
        elif r == 8:
            e = list(top[r, :10]) * 2                                         # every entry twice
        elif r == 13:
            e = list(same)
        else:
            e = list(rng.choice(same, 16, replace=False)) + list(top[r, :3]) if same.size else [1, 2, 3]
        if targets is not None and r % 3 == 0:
            e = e + [targets[r], targets[r]]
        lists.append([int(x) for x in rng.permutation(np.array(e, dtype=np.int64))])
    shared = [int(x) for x in rng.choice(p, 3000, replace=False)] + [int(x) for x in top[30, :5]]
    lists.append(shared)
    row_list = np.arange(len(row_type))
    row_list[30:] = len(row_type)                                             # rows 30..39 share list 40
    row_list[28], row_list[29] = len(lists) + 5, -1                           # no exclusions
    return lists, row_list


def _per_row(lists, row_list):
    return [lists[l] if 0 <= l < len(lists) else None for l in row_list]


@pytest.fixture(scope="module")
def data():
    from pcompanion_b200 import CatalogIndex, Exclusions
    cat, type_id, q, row_type = _data()
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=N_TYPES)
    qt, rtt = torch.tensor(q, device=dev()), torch.tensor(row_type, device=dev())
    top = index.topk(qt, 1024, rtt)[1].cpu().numpy()
    lists, row_list = _lists(cat, type_id, row_type, top)
    per_row = _per_row(lists, row_list)
    ex = Exclusions.from_lists(lists, dev(), torch.tensor(row_list, device=dev()))
    ref_s, ref_i = masked_topk_excluding(q, cat, 1024, per_row, row_type, type_id)
    plain_top = index.topk(qt[:9], 1024)[1].cpu().numpy()                    # row_type=None: the whole catalog
    plain_lists = [list(map(int, plain_top[r, :M_TOP.get(r, 0)])) + [int(r * 7)] for r in range(9)]
    pl_s, pl_i = masked_topk_excluding(q[:9], cat, 1024, plain_lists)
    return dict(cat=cat, type_id=type_id, q=q, row_type=row_type, index=index, qt=qt, rtt=rtt, top=top, lists=lists,
                row_list=row_list, per_row=per_row, ex=ex, ref_s=ref_s, ref_i=ref_i, plain_lists=plain_lists,
                plain_ex=Exclusions.from_lists(plain_lists, dev()), pl_s=pl_s, pl_i=pl_i)


def _equal(s, i, ref_s, ref_i, what):
    assert np.array_equal(i.cpu().numpy(), ref_i), f"{what}: indices differ"
    assert np.array_equal(s.cpu().numpy(), ref_s), f"{what}: scores differ"


@pytest.mark.parametrize("k", KS)
def test_filtered_topk_matches_the_reference(data, k):
    index, qt, rtt, ex = data["index"], data["qt"], data["rtt"], data["ex"]
    for splits in (None, 1, 4, 37):
        s, i = index.topk(qt, k, rtt, splits=splits, exclude=ex)
        _equal(s, i, data["ref_s"][:, :k], data["ref_i"][:, :k], f"k={k} splits={splits}")
        s2, i2 = index.topk(qt, k, rtt, splits=splits, exclude=ex)
        assert torch.equal(s2, s) and torch.equal(i2, i), f"k={k} splits={splits}: repeated call differs"
        su, iu = index.topk(qt[:9], k, splits=splits, exclude=data["plain_ex"])
        _equal(su, iu, data["pl_s"][:, :k], data["pl_i"][:, :k], f"unrestricted k={k} splits={splits}")
    assert (i[13] == -1).all() and torch.isinf(s[13]).all()                 # the whole type is excluded
    got = i.cpu().numpy()
    for r, e in enumerate(data["per_row"]):
        if e is not None:
            assert not np.isin(got[r], e).any(), f"k={k}: row {r} lists an excluded product"
    # rows whose lists name nothing of their run, or that have no list, rank as without exclusions
    s0, i0 = index.topk(qt, k, rtt)
    for r in (0, 7, 28, 29):
        assert torch.equal(i[r], i0[r]) and torch.equal(s[r], s0[r]), f"k={k} row {r}"


@pytest.mark.parametrize("k", KS)
def test_all_empty_lists_equal_the_plain_topk(data, k):
    from pcompanion_b200 import Exclusions
    index, qt, rtt = data["index"], data["qt"], data["rtt"]
    empty = Exclusions(torch.zeros(41, dtype=torch.int64, device=dev()), torch.empty(0, dtype=torch.int64, device=dev()))
    no_effect = Exclusions.from_lists([[-1, 10 ** 12]] * 40, dev())
    for splits in (None, 1, 4):
        s0, i0 = index.topk(qt, k, rtt, splits=splits)
        for ex in (empty, no_effect):
            s, i = index.topk(qt, k, rtt, splits=splits, exclude=ex)
            assert torch.equal(s, s0) and torch.equal(i, i0), f"k={k} splits={splits}"


def test_over_fetch_cross_check(data):
    """Filtered top-k == unfiltered top-(k + |E_r|) without the excluded entries, truncated to k."""
    index, qt, rtt, ex = data["index"], data["qt"], data["rtt"], data["ex"]
    checked = 0
    for k in (1, 10, 32, 33, 100):
        s, i = index.topk(qt, k, rtt, exclude=ex)
        for r, e in enumerate(data["per_row"]):
            n_e = 0 if e is None else len(e)
            if k + n_e > 1024:
                continue
            fs, fi = index.topk(qt[r:r + 1], k + n_e, rtt[r:r + 1])
            keep = ~np.isin(fi[0].cpu().numpy(), [] if e is None else e)
            want_i, want_s = fi[0].cpu().numpy()[keep][:k], fs[0].cpu().numpy()[keep][:k]
            pad = k - want_i.size
            want_i = np.concatenate([want_i, np.full(pad, -1)])
            want_s = np.concatenate([want_s, np.full(pad, -np.inf)])
            assert np.array_equal(i[r].cpu().numpy(), want_i) and np.array_equal(s[r].cpu().numpy(), want_s), (k, r)
            checked += 1
    assert checked >= 100


def _targets(type_id, row_type, top, p):
    rng = np.random.default_rng(23)
    t = np.empty(len(row_type), np.int64)
    for r, rt in enumerate(row_type):
        m = np.nonzero(type_id == rt)[0]
        t[r] = rng.choice(m) if m.size else rng.integers(0, p)
    for r, j in {1: 1, 2: 31, 3: 40, 4: 33, 5: 600, 6: 20, 8: 12, 9: 1023, 10: 0, 11: 100, 13: 7}.items():
        t[r] = top[r, j]
    t[20], t[21] = -3, p + 1000
    t[23] = rng.choice(np.nonzero(type_id != row_type[23])[0])
    return t


@pytest.fixture(scope="module")
def rank_data(data):
    from pcompanion_b200 import Exclusions
    cat, type_id, q, row_type, top = data["cat"], data["type_id"], data["q"], data["row_type"], data["top"]
    targets = _targets(type_id, row_type, top, cat.shape[0])
    lists, row_list = _lists(cat, type_id, row_type, top, targets)
    per_row = _per_row(lists, row_list)
    assert sum(e is not None and int(targets[r]) in e for r, e in enumerate(per_row)) >= 10
    # per row, the list without the row's own target: the top-K side of the rank / top-K property
    minus = [[x for x in (e or []) if x != targets[r]] for r, e in enumerate(per_row)]
    return dict(targets=targets, tt=torch.tensor(targets, device=dev()), per_row=per_row,
                ex=Exclusions.from_lists(lists, dev(), torch.tensor(row_list, device=dev())),
                minus=Exclusions.from_lists(minus, dev()),
                want=masked_rank_excluding(q, cat, targets, per_row, row_type, type_id),
                plain=masked_rank(q, cat, targets, row_type, type_id))


def test_filtered_rank_matches_the_reference(data, rank_data):
    index, qt, rtt, tt, want = data["index"], data["qt"], data["rtt"], rank_data["tt"], rank_data["want"]
    assert (want[[12, 14, 15, 20, 21, 23]] == -1).all() and (want[:12] >= 0).all()
    assert (want <= rank_data["plain"]).all() and (want < rank_data["plain"]).sum() >= 10
    for splits in (None, 1, 4, 37):
        got = index.rank(qt, tt, rtt, splits=splits, exclude=rank_data["ex"])
        assert np.array_equal(got.cpu().numpy(), want), f"splits={splits}"
    assert np.array_equal(index.rank(qt, tt, rtt).cpu().numpy(), rank_data["plain"])       # exclude=None: unchanged


@pytest.mark.parametrize("k", KS)
def test_filtered_rank_agrees_with_filtered_topk(data, rank_data, k):
    index, qt, rtt, tt = data["index"], data["qt"], data["rtt"], rank_data["tt"]
    ranks = index.rank(qt, tt, rtt, exclude=rank_data["ex"]).cpu()
    _, idx = index.topk(qt, k, rtt, exclude=rank_data["minus"])
    hit = idx.cpu() == tt.cpu()[:, None]
    listed = hit.any(1)
    assert torch.equal(listed, (ranks >= 0) & (ranks < k)), f"k={k}"
    assert torch.equal(hit.int().argmax(1)[listed], ranks[listed]), f"k={k}: position"
    assert int(listed.sum()) >= (3 if k == 1 else 6), f"k={k}"


@pytest.mark.parametrize("kind", ["rising", "tied"])
def test_adversarial_catalogs(kind):
    from pcompanion_b200 import CatalogIndex, Exclusions
    p = 100_000
    cat, q = _stream_catalog(p, kind)
    type_id = (np.arange(p) % 2).astype(np.int32)
    rt = np.array([0, 1] * 5, np.int32)
    position = np.array([0, 1, 17, 31, 32, 1000, 1023, 20_000, 49_998, 49_999])
    targets = rt + 2 * position
    rng = np.random.default_rng(31)
    lists = [[int(t)] + [int(rt[r] + 2 * x) for x in rng.integers(0, 50_000, 40)] + [int(x) for x in range(rt[r], 2000, 2)]
             for r, t in enumerate(targets)]                                   # the row's first 1000 members, more
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=2)
    qt, rtt, tt = torch.tensor(q, device=dev()), torch.tensor(rt, device=dev()), torch.tensor(targets, device=dev())
    ex = Exclusions.from_lists(lists, dev())
    want = masked_rank_excluding(q, cat, targets, lists, rt, type_id)
    if kind == "tied":                                                         # only indices order the products
        assert np.array_equal(want, [position[r] - len({x for x in lists[r] if x < targets[r]}) for r in range(10)])
    for splits in (None, 1, 4):
        assert np.array_equal(index.rank(qt, tt, rtt, splits=splits, exclude=ex).cpu().numpy(), want), splits
    ref_s, ref_i = masked_topk_excluding(q, cat, 1024, lists, rt, type_id)
    for k in (10, 33, 1024):
        s, i = index.topk(qt, k, rtt, exclude=ex)
        _equal(s, i, ref_s[:, :k], ref_i[:, :k], f"{kind} k={k}")


def test_more_than_65535_score_rows():
    from pcompanion_b200 import CatalogIndex, Exclusions
    rng = np.random.default_rng(33)
    p, r = 1500, 70_000
    cat = rng.normal(size=(p, 16)).astype(np.float32)
    type_id = rng.integers(0, 3, p).astype(np.int32)
    q = rng.normal(size=(r, 16)).astype(np.float32)
    row_type = rng.integers(0, 3, r).astype(np.int32)
    members = [np.nonzero(type_id == t)[0] for t in range(3)]
    targets = np.array([rng.choice(members[t]) for t in row_type])
    lists = [[int(targets[i])] + [int(x) for x in rng.choice(members[row_type[i]], 6)] for i in range(r)]
    index = CatalogIndex(torch.tensor(cat, device=dev()), torch.tensor(type_id, device=dev()), num_types=3)
    qt, rtt = torch.tensor(q, device=dev()), torch.tensor(row_type, device=dev())
    ex = Exclusions.from_lists(lists, dev())
    got = index.rank(qt, torch.tensor(targets, device=dev()), rtt, exclude=ex).cpu().numpy()
    s, i = index.topk(qt, 5, rtt, exclude=ex)
    for a in range(0, r, 10_000):
        sl = slice(a, a + 10_000)
        assert np.array_equal(got[sl], masked_rank_excluding(q[sl], cat, targets[sl], lists[sl], row_type[sl], type_id))
        ref_s, ref_i = masked_topk_excluding(q[sl], cat, 5, lists[sl], row_type[sl], type_id)
        _equal(s[sl], i[sl], ref_s, ref_i, f"rows {a}..")


def test_three_shards_on_one_gpu(data, rank_data):
    from pcompanion_b200 import CatalogIndex, ops
    cat, type_id, qt, rtt, ex = data["cat"], data["type_id"], data["qt"], data["rtt"], data["ex"]
    bounds = [0, 61_000, 140_000, cat.shape[0]]
    shards = [CatalogIndex(torch.tensor(cat[a:b], device=dev()), torch.tensor(type_id[a:b], device=dev()), index_base=a,
                           num_types=N_TYPES) for a, b in zip(bounds[:-1], bounds[1:])]
    for k in (10, 100):
        parts = [sh.topk(qt, k, rtt, exclude=ex) for sh in shards]             # the same global lists on every shard
        s, i = ops.topk_merge(torch.cat([p[0] for p in parts], 1), torch.cat([p[1] for p in parts], 1), k)
        _equal(s, i, data["ref_s"][:, :k], data["ref_i"][:, :k], f"merged shards k={k}")
    tt, want, rex = rank_data["tt"], rank_data["want"], rank_data["ex"]
    rows = data["index"].catalog[tt.clamp(0, cat.shape[0] - 1)]
    total = sum(ops.rank_by_type(qt, sh.catalog, sh.offsets, N_TYPES, rtt, rows, tt, sh.members, sh.index_base,
                                 exclude=rex, type_id=sh.type_id).clamp_min(0) for sh in shards)
    member = want >= 0
    assert np.array_equal(total.cpu().numpy()[member], want[member])


def _sharded_worker(rank, world, port, results):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    d = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=d)
    try:
        from pcompanion_b200 import CatalogIndex, Exclusions, ShardedCatalog
        cat, type_id, q, row_type = _data()
        rng = np.random.default_rng(35)
        targets = np.array([rng.choice(np.nonzero(type_id == t)[0]) if (type_id == t).any() else 0 for t in row_type])
        lists = [[int(targets[r])] + [int(x) for x in rng.integers(0, cat.shape[0], 400)] for r in range(len(row_type))]
        bounds = [0, 90_000, cat.shape[0]]
        a, b = bounds[rank], bounds[rank + 1]
        sh = ShardedCatalog(torch.tensor(cat[a:b], device=d), torch.tensor(type_id[a:b], device=d), a, N_TYPES)
        full = CatalogIndex(torch.tensor(cat, device=d), torch.tensor(type_id, device=d), num_types=N_TYPES)
        qt, rtt, tt = torch.tensor(q, device=d), torch.tensor(row_type, device=d), torch.tensor(targets, device=d)
        ex = Exclusions.from_lists(lists, d)
        ok = torch.equal(sh.rank(qt, tt, rtt, exclude=ex), full.rank(qt, tt, rtt, exclude=ex))
        for k in (10, 100):
            ok = ok and all(torch.equal(x, y) for x, y in zip(sh.topk(qt, k, rtt, exclude=ex), full.topk(qt, k, rtt, exclude=ex)))
        results[rank] = "ok" if ok else "FAILED: sharded != unsharded"
    except Exception:  # pragma: no cover
        import traceback
        results[rank] = traceback.format_exc()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_sharded_exclusions_equal_single_gpu():
    import torch.multiprocessing as mp
    world = 2
    results = mp.Manager().dict()
    mp.spawn(_sharded_worker, args=(world, _free_port(), results), nprocs=world, join=True)
    assert all(results.get(r) == "ok" for r in range(world)), dict(results)


@pytest.fixture(scope="module")
def c1():
    from test_gpu_datapath import c1_bpg, make_cfg
    from pcompanion_b200 import PCompanion, PCompanionInference
    _, ids, bpg = c1_bpg()
    cfg = make_cfg(NUM_TYPES=20)
    torch.manual_seed(0)
    model = PCompanion(cfg, {pid: torch.randn(128) for pid in ids})
    inf = PCompanionInference(None, cfg, bpg, model=model)
    return dict(ids=ids, bpg=bpg, inf=inf, feats=bpg.features.float().cpu().numpy(), tidx=inf._type_of.numpy())


def _brute_top(proj_row, members, feats, k, excluded):
    members = members[~np.isin(members, list(excluded))]
    sc = scores_fp64(proj_row[None, :], feats[members])[0]
    order = np.lexsort((members, -sc))[:k]
    return members[order], sc[order]


def test_recommend_batch_excluding_ids(c1):
    inf, ids, feats, tidx = c1["inf"], c1["ids"], c1["feats"], c1["tidx"]
    rng = np.random.default_rng(40)
    q_idx = rng.choice(len(ids), 24, replace=False)
    queries = [ids[i] for i in q_idx]
    with torch.no_grad():
        out = inf.model(inf._prepare_input(queries))
    comp, proj = out["complementary_types"].cpu().numpy(), out["projected_embeddings"].cpu().numpy()
    excl = []
    for b, qi in enumerate(q_idx):
        same = np.nonzero(tidx == comp[b, 0])[0]
        top = _brute_top(proj[b, 0], same, feats, 5, set())[0]
        excl.append([ids[qi]] + [ids[j] for j in top[:3]] + [ids[j] for j in rng.choice(len(ids), 20)])
    res = inf.recommend_batch(queries, 10, exclude_ids=excl)
    plain = inf.recommend_batch(queries, 10)
    for b in range(len(queries)):
        ex_idx = {inf.bpg._index[p] for p in excl[b]}
        for t in range(comp.shape[1]):
            members = np.nonzero(tidx == comp[b, t])[0]
            want_i, want_s = _brute_top(proj[b, t], members, feats, 10, ex_idx)
            got = res[b]["recommendations"][t]
            assert got == [ids[j] for j in want_i], (b, t)
            assert np.array_equal(res[b]["scores"][t], want_s), (b, t)
            assert not set(got) & set(excl[b]), (b, t)
        assert res[b]["recommendations"] != plain[b]["recommendations"]
    one = inf.recommend(queries[0], 10, exclude_ids=excl[0])
    assert one["recommendations"] == res[0]["recommendations"]
    assert inf.recommend(queries[0], 10)["recommendations"] == plain[0]["recommendations"]     # exclude_ids=None


def test_filtered_rank_targets_and_evaluate(c1):
    from pcompanion_b200 import Metrics
    inf, ids, bpg, feats, tidx = c1["inf"], c1["ids"], c1["bpg"], c1["feats"], c1["tidx"]
    csr = bpg.csr("co_purchase")
    rowptr, col = csr.rowptr.cpu().numpy(), csr.col.cpu().numpy()
    rng = np.random.default_rng(41)
    q_idx = [i for i in rng.permutation(len(ids)) if rowptr[i + 1] - rowptr[i] >= 2][:48]
    assert len(q_idx) >= 24
    queries = [ids[i] for i in q_idx]
    with torch.no_grad():
        out = inf.model(inf._prepare_input(queries))
    comp, proj = out["complementary_types"].cpu().numpy(), out["projected_embeddings"].cpu().numpy()
    t_idx = []
    for b, qi in enumerate(q_idx):
        nb = col[rowptr[qi]:rowptr[qi + 1]]
        m = np.nonzero(tidx == comp[b, b % 3])[0]
        t_idx.append(int(nb[0]) if b % 4 == 0 else int(rng.choice(m)))     # a co-purchase neighbour, or any member
    targets = [ids[j] for j in t_idx]
    extra = [[ids[j] for j in rng.choice(len(ids), 30)] for _ in q_idx]
    for mode in ("edges", "ids", "both"):
        kw = dict(filter_edges="co_purchase" if mode != "ids" else None, exclude_ids=extra if mode != "edges" else None)
        ranks, slots = inf.rank_targets(queries, targets, **kw)
        ranks, slots = ranks.cpu().numpy(), slots.cpu().numpy()
        for b, (qi, g) in enumerate(zip(q_idx, t_idx)):
            hits = np.nonzero(comp[b] == tidx[g])[0]
            if not hits.size:
                assert ranks[b] == -1
                continue
            ex = set()
            if mode != "ids":
                ex |= set(col[rowptr[qi]:rowptr[qi + 1]].tolist())
            if mode != "edges":
                ex |= {bpg._index[p] for p in extra[b]}
            ex.discard(g)
            members = np.nonzero(tidx == tidx[g])[0]
            members = members[~np.isin(members, list(ex))]
            sc = scores_fp64(proj[b, hits[0]][None, :], feats[members])[0]
            s_t = sc[members == g][0]
            assert ranks[b] == int(((sc > s_t) | ((sc == s_t) & (members < g))).sum()), (mode, b)
        m = inf.evaluate(queries, targets, **kw)
        want = Metrics.rank_metrics(torch.tensor(ranks))
        want["type_recall"] = float((slots >= 0).mean())
        assert m == pytest.approx(want, abs=0, rel=1e-15)
    # a filtered rank below 100 is the target's position in recommend(query, 100, exclude_ids=neighbours - {target})
    ranks, slots = inf.rank_targets(queries, targets, filter_edges="co_purchase")
    ranks, slots = ranks.cpu().numpy(), slots.cpu().numpy()
    plain, _ = inf.rank_targets(queries, targets)
    assert (ranks <= plain.cpu().numpy()).all()
    checked = 0
    for b in np.nonzero((ranks >= 0) & (ranks < 100))[0]:
        nb = [ids[j] for j in col[rowptr[q_idx[b]]:rowptr[q_idx[b] + 1]] if j != t_idx[b]]
        rec = inf.recommend(queries[b], 100, exclude_ids=nb)
        assert rec["recommendations"][slots[b]][ranks[b]] == targets[b], b
        checked += 1
    assert checked >= 5


def test_errors(data, c1):
    from pcompanion_b200 import Exclusions
    index, qt, rtt = data["index"], data["qt"], data["rtt"]
    with pytest.raises(ValueError, match="Exclusions"):
        Exclusions(torch.tensor([0, 3, 2], device=dev()), torch.arange(2, device=dev()))
    bad_rows = Exclusions.from_lists([[1]], dev(), torch.zeros(5, dtype=torch.int64, device=dev()))
    with pytest.raises(ValueError, match="row_list"):
        index.topk(qt, 10, rtt, exclude=bad_rows)
    with pytest.raises(ValueError, match="row_list"):
        index.rank(qt, torch.zeros(40, dtype=torch.int64, device=dev()), rtt, exclude=bad_rows)
    inf, ids = c1["inf"], c1["ids"]
    with pytest.raises(ValueError, match="not found"):
        inf.recommend(ids[0], 10, exclude_ids=["no-such-product"])
    with pytest.raises(ValueError, match="not found"):
        inf.rank_targets([ids[0]], [ids[1]], exclude_ids=[["no-such-product"]])
    with pytest.raises(ValueError, match="filter_edges"):
        inf.evaluate([ids[0]], [ids[1]], filter_edges="bought_together")
