"""CPU-side checks of the top-K size limit (1 <= k <= 1024) and of the automatic split count for large k: both are
decided before any device work, so they need no GPU."""
import os
import re

import pytest
import torch

from conftest import ROOT


def test_python_limit_matches_the_header():
    from pcompanion_b200 import ops
    src = open(os.path.join(ROOT, "include", "pcompanion_b200.h")).read()
    assert int(re.search(r"#define PC_TOPK_MAX_K (\d+)", src).group(1)) == ops.TOPK_MAX_K == 1024


@pytest.mark.parametrize("k", [0, 1025])
def test_k_outside_the_limit_raises_before_the_library_is_called(k):
    from pcompanion_b200 import ops
    x = torch.zeros(4, 128)
    with pytest.raises(ValueError, match=r"\[1, 1024\]"):
        ops.topk_rows(x, k)
    with pytest.raises(ValueError, match=r"\[1, 1024\]"):
        ops.topk_by_type(x, x, torch.tensor([0, 4]), 1, None, k)
    with pytest.raises(ValueError, match=r"\[1, 1024\]"):
        ops.topk_segments(x, x, torch.zeros(4, dtype=torch.int64), torch.zeros(4, dtype=torch.int64), k)
    with pytest.raises(ValueError, match=r"\[1, 1024\]"):
        ops.topk_merge(torch.zeros(4, 2048, dtype=torch.float64), torch.zeros(4, 2048, dtype=torch.int64), k)


def test_split_workspace_grows_with_k():
    from pcompanion_b200 import _lib
    assert _lib.LIB.pc_topk_groups_workspace_bytes(10, 1024, 4) == 10 * 4 * 1024 * 16
    assert _lib.LIB.pc_topk_by_type_workspace_bytes(10, 1024, 4) - _lib.LIB.pc_topk_by_type_workspace_bytes(10, 1024, 1) \
        == 10 * 4 * 1024 * 16


def test_auto_splits_bound_the_workspace_and_keep_splits_long_for_large_k():
    from pcompanion_b200 import ops
    for units, avg_len, rows in ((1, 10_000_000, 4096), (3, 10_000_000, 3), (40, 200_000, 40), (1, 5_000, 1)):
        assert ops._auto_splits(units, avg_len, 10, rows) == ops._auto_splits(units, avg_len)   # k <= 32: unchanged
        for k in (33, 100, 1024):
            s = ops._auto_splits(units, avg_len, k, rows)
            assert s == 1 or (rows * s * k * 16 <= ops.SPLIT_WS_BYTES and avg_len / s >= 16 * k), (units, avg_len, rows, k, s)
    assert ops._auto_splits(1, 10_000_000, 1024, 4096) == 4           # 256 MiB = 4 x [4096, 1024] (f64, i64) lists
