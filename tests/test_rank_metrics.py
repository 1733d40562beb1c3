"""CPU-side checks of the target-rank evaluation: Metrics.rank_metrics on hand-computed values, the reference rank
against a stable sort, and the argument checks of pc_rank_by_type / ops.rank_by_type, which run before any device
work."""
import math
from ctypes import c_void_p

import numpy as np
import pytest
import torch

from _rank_oracle import masked_rank


def test_rank_metrics_on_hand_computed_values():
    from pcompanion_b200 import Metrics
    ranks = torch.tensor([0, 2, -1, 9, 100, 1])
    m = Metrics.rank_metrics(ranks, ks=(1, 3, 10, 101))
    assert m["num_rows"] == 6
    assert m["hit@1"] == pytest.approx(1 / 6)
    assert m["hit@3"] == pytest.approx(3 / 6)              # ranks 0, 2, 1
    assert m["hit@10"] == pytest.approx(4 / 6)             # + 9
    assert m["hit@101"] == pytest.approx(5 / 6)            # + 100; the -1 is a miss for every k
    assert m["ndcg@1"] == pytest.approx(1 / 6)
    assert m["ndcg@3"] == pytest.approx((1 + 1 / math.log2(4) + 1 / math.log2(3)) / 6)
    assert m["ndcg@10"] == pytest.approx((1 + 1 / math.log2(4) + 1 / math.log2(3) + 1 / math.log2(11)) / 6)
    assert m["ndcg@101"] == pytest.approx((1 + 1 / math.log2(4) + 1 / math.log2(3) + 1 / math.log2(11) + 1 / math.log2(102)) / 6)
    assert m["mrr"] == pytest.approx((1 + 1 / 3 + 0 + 1 / 10 + 1 / 101 + 1 / 2) / 6)
    assert set(m) == {"hit@1", "hit@3", "hit@10", "hit@101", "ndcg@1", "ndcg@3", "ndcg@10", "ndcg@101", "mrr", "num_rows"}


def test_rank_metrics_defaults_and_limits():
    from pcompanion_b200 import Metrics
    ranks = torch.tensor([-1, -1, 4999, 5000, 0])
    m = Metrics.rank_metrics(ranks)
    assert {f"hit@{k}" for k in (1, 3, 10, 50, 100)} <= set(m) and m["hit@1"] == pytest.approx(1 / 5)
    assert Metrics.rank_metrics(ranks, ks=(5000,))["hit@5000"] == pytest.approx(2 / 5)     # no 1,024 limit here
    assert Metrics.rank_metrics(torch.full((3,), -1), ks=(1,)) == {"hit@1": 0.0, "ndcg@1": 0.0, "mrr": 0.0, "num_rows": 3}
    with pytest.raises(ValueError):
        Metrics.rank_metrics(ranks, ks=(0,))


def test_reference_rank_is_the_position_in_a_stable_sort():
    from oracle.retrieval import scores_fp64
    rng = np.random.default_rng(4)
    cat = rng.integers(-2, 3, size=(300, 16)).astype(np.float32)     # small integers: many tied scores
    type_id = rng.integers(0, 3, 300).astype(np.int32)
    q = rng.integers(-2, 3, size=(12, 16)).astype(np.float32)
    row_type = rng.integers(0, 3, 12).astype(np.int32)
    targets = np.array([rng.choice(np.nonzero(type_id == t)[0]) for t in row_type]) + 1000
    targets[0], targets[1] = 999, 1300                                 # outside the catalog (index_base 1000)
    targets[2] = 1000 + np.nonzero(type_id != row_type[2])[0][0]      # another type
    got = masked_rank(q, cat, targets, row_type, type_id, index_base=1000, chunk=64)
    s = scores_fp64(q, cat)
    for r in range(12):
        members = np.nonzero(type_id == row_type[r])[0]
        order = members[np.lexsort((members, -s[r, members]))] + 1000
        want = int(np.nonzero(order == targets[r])[0][0]) if targets[r] in order else -1
        assert got[r] == want, r
    assert list(got[:3]) == [-1, -1, -1]
    plain = rng.integers(0, 300, 12)                                   # no row types: the whole catalog
    plain[0], plain[1] = 300, -1
    whole = masked_rank(q, cat, plain)
    for r in range(12):
        order = np.lexsort((np.arange(300), -s[r]))
        want = int(np.nonzero(order == plain[r])[0][0]) if 0 <= plain[r] < 300 else -1
        assert whole[r] == want, r


def test_rank_workspace_bytes():
    from pcompanion_b200 import _lib
    assert _lib.LIB.pc_rank_by_type_workspace_bytes(0) == 0
    assert _lib.LIB.pc_rank_by_type_workspace_bytes(-5) == 0
    assert _lib.LIB.pc_rank_by_type_workspace_bytes(1) > 0
    assert _lib.LIB.pc_rank_by_type_workspace_bytes(100_000) > _lib.LIB.pc_rank_by_type_workspace_bytes(1000) > 0


def _call(rows=4, dim=128, ptr=c_void_p(256), n_types=1, splits=1, ws_bytes=1 << 40):
    """pc_rank_by_type with every device pointer set to `ptr` (never dereferenced: the arguments are refused first)."""
    from pcompanion_b200 import _lib
    return _lib.LIB.pc_rank_by_type(ptr, rows, dim, ptr, ptr, ptr, n_types, ptr, ptr, ptr, splits, 0, ptr, ptr, ws_bytes,
                                    None)


def test_rank_by_type_refuses_bad_arguments_without_a_device():
    from pcompanion_b200 import _lib
    assert _call(rows=0, ptr=None) == 0                                # nothing to do
    assert _call(ptr=None) == 1                                        # PC_ERR_INVALID: null pointer
    assert b"null pointer" in _lib.LIB.pc_last_error()
    assert _call(rows=-1) == 1
    assert _call(rows=1 << 31) == 1
    assert _call(n_types=0) == 1
    assert _call(dim=24) == 4                                          # PC_ERR_UNSUPPORTED
    assert b"dim=24" in _lib.LIB.pc_last_error()
    assert _call(dim=2048) == 4
    assert _call(splits=0) == 4
    assert _call(ws_bytes=16) == 3                                     # PC_ERR_WORKSPACE


def test_ops_rank_by_type_checks_shapes():
    from pcompanion_b200 import ops
    q = torch.zeros(4, 128)
    off = torch.tensor([0, 8])
    good_t, good_i = torch.zeros(4, 128), torch.zeros(4, dtype=torch.int64)
    with pytest.raises(ValueError, match="target_rows"):
        ops.rank_by_type(q, q, off, 1, None, torch.zeros(3, 128), good_i)
    with pytest.raises(ValueError, match="target_rows"):
        ops.rank_by_type(q, q, off, 1, None, torch.zeros(4, 64), good_i)
    with pytest.raises(ValueError, match="target_idx"):
        ops.rank_by_type(q, q, off, 1, None, good_t, torch.zeros(5, dtype=torch.int64))
    with pytest.raises(ValueError, match="row_type"):
        ops.rank_by_type(q, q, off, 1, torch.zeros(2, dtype=torch.int32), good_t, good_i)
