"""Exclusion lists without a GPU: Exclusions construction (device-side sort, duplicates kept, validation of outside
input) on CPU tensors, and the filtered top-K / rank references against hand-computed cases."""
import numpy as np
import pytest
import torch

from _exclusion_oracle import masked_rank_excluding, masked_topk_excluding
from _rank_oracle import masked_rank


def test_from_lists_sorts_each_list_and_keeps_duplicates():
    from pcompanion_b200 import Exclusions
    ex = Exclusions.from_lists([[9, 3, 3, -1], [], [7], [5, 2, 8, 2]], "cpu")
    assert ex.offsets.tolist() == [0, 4, 4, 5, 9] and ex.num_lists == 4
    assert ex.indices.tolist() == [-1, 3, 3, 9, 7, 2, 2, 5, 8]
    assert ex.indices.dtype == torch.int64 and ex.row_list is None
    ex = Exclusions(torch.tensor([0, 2, 3]), torch.tensor([4, 1, 0], dtype=torch.int32), torch.tensor([1, 5, -3, 0]))
    assert ex.indices.tolist() == [1, 4, 0]
    assert ex.row_list.dtype == torch.int32 and ex.row_list.tolist() == [1, -1, -1, 0]   # out of range: no list
    kept = Exclusions(torch.tensor([0, 2]), torch.tensor([8, 1]), sorted=True)           # trusted order: no sort
    assert kept.indices.tolist() == [8, 1]


def test_for_rows_and_union_share_and_merge_lists():
    from pcompanion_b200 import Exclusions
    a = Exclusions.from_lists([[4, 1], [6]], "cpu")
    view = a.for_rows(torch.tensor([0, 0, 1, 1, 7]))
    assert view.indices is a.indices and view.row_list.tolist() == [0, 0, 1, 1, -1]
    b = Exclusions.from_lists([[2], [], [3, 1]], "cpu")
    u = a.for_rows(torch.tensor([1, 0, 5])).union(b, 3)
    assert u.offsets.tolist() == [0, 2, 4, 6] and u.indices.tolist() == [2, 6, 1, 4, 1, 3]


@pytest.mark.parametrize("offsets, indices", [
    ([1, 2], [5, 6]),             # does not start at 0
    ([0, 2, 1, 3], [1, 2, 3]),    # decreasing
    ([0, 2], [1, 2, 3]),          # does not end at indices.numel()
    ([0, 4], [1, 2, 3]),
    ([], []),                     # no offsets at all
])
def test_malformed_offsets_are_refused(offsets, indices):
    from pcompanion_b200 import Exclusions
    with pytest.raises(ValueError, match="Exclusions"):
        Exclusions(torch.tensor(offsets, dtype=torch.int64), torch.tensor(indices, dtype=torch.int64))


def test_bad_shapes_and_dtypes_are_refused():
    from pcompanion_b200 import Exclusions
    with pytest.raises(ValueError, match="row_list"):
        Exclusions(torch.tensor([0, 1]), torch.tensor([3]), torch.zeros(2, 2, dtype=torch.int64))
    with pytest.raises(ValueError, match="1-D"):
        Exclusions(torch.tensor([[0, 1]]), torch.tensor([3]))
    with pytest.raises(ValueError, match="integer"):
        Exclusions(torch.tensor([0.0, 1.0]), torch.tensor([3]))


def _hand_case():
    """6 products, two types; row 0 ranks type 0, row 1 type 1; scores are q . c = c[:, 0] (dim 16)."""
    cat = np.zeros((6, 16), np.float32)
    cat[:, 0] = [5, 3, 9, 3, 7, 1]                      # type:  0 1 0 0 1 0
    type_id = np.array([0, 1, 0, 0, 1, 0], np.int32)
    q = np.zeros((2, 16), np.float32)
    q[:, 0] = 1
    return cat, type_id, q, np.array([0, 1], np.int32)


def test_filtered_topk_reference_on_a_hand_case():
    cat, type_id, q, rt = _hand_case()
    # row 0 ranks type 0 = products 2 (9), 0 (5), 3 (3), 5 (1); excluding 2 (twice), 4 (other type) and 77 (no product)
    s, i = masked_topk_excluding(q, cat, 3, [[2, 4, 77, 2], None], rt, type_id)
    assert i.tolist() == [[0, 3, 5], [4, 1, -1]]
    assert s[0].tolist() == [5, 3, 1] and s[1, :2].tolist() == [7, 3] and np.isneginf(s[1, 2])
    s, i = masked_topk_excluding(q, cat, 2, [[0, 2, 3, 5], [1, 4]], rt, type_id)     # whole types: padding
    assert (i == -1).all() and np.isneginf(s).all()


def test_filtered_rank_reference_on_a_hand_case():
    cat, type_id, q, rt = _hand_case()
    targets = np.array([3, 1])
    assert masked_rank(q, cat, targets, rt, type_id).tolist() == [2, 1]              # 2 and 0 before 3; 4 before 1
    # the target in its own list is not removed; duplicates count once; other-type / outside entries do nothing
    assert masked_rank_excluding(q, cat, targets, [[3, 2, 2, 4, -8], [1]], rt, type_id).tolist() == [1, 1]
    assert masked_rank_excluding(q, cat, targets, [[0, 2], [4]], rt, type_id).tolist() == [0, 0]
    assert masked_rank_excluding(q, cat, np.array([5, 0]), [[0], None], rt, type_id).tolist() == [2, -1]
    # global indices with an index base: list entries are global too
    assert masked_rank_excluding(q, cat, targets + 100, [[102], [104]], rt, type_id, index_base=100).tolist() == [1, 0]
