"""Reference filtered top-K and filtered rank (test infrastructure only), on the score definition of
oracle/retrieval.py: row r's exclusion list (global product indices, any order, duplicates allowed; None = no list)
is left out of its ranking.  The filtered rank never removes the row's own target.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

from oracle.retrieval import merge_topk, scores_fp64


def _excluded(lists, r: int, index_base: int, lo: int, hi: int) -> np.ndarray:
    """Local catalog rows in [lo, hi) that row r's exclusion list names (global indices, any order, duplicates)."""
    e = np.asarray(lists[r], dtype=np.int64) - index_base
    return np.unique(e[(e >= lo) & (e < hi)])


def masked_topk_excluding(q: np.ndarray, catalog: np.ndarray, k: int, lists, row_type: Optional[np.ndarray] = None,
                          type_id: Optional[np.ndarray] = None, index_base: int = 0,
                          chunk: int = 1 << 16) -> Tuple[np.ndarray, np.ndarray]:
    """oracle.retrieval.masked_topk with row r's products lists[r] (global indices; None = no list) left out."""
    r = q.shape[0]
    best_s = np.full((r, k), -np.inf)
    best_i = np.full((r, k), -1, dtype=np.int64)
    for beg in range(0, catalog.shape[0], chunk):
        end = min(beg + chunk, catalog.shape[0])
        s = scores_fp64(q, catalog[beg:end])
        if row_type is not None:
            s = np.where(type_id[None, beg:end] == row_type[:, None], s, -np.inf)
        for i in range(r):
            if lists[i] is not None:
                s[i, _excluded(lists, i, index_base, beg, end) - beg] = -np.inf
        idx = np.broadcast_to(np.arange(beg, end, dtype=np.int64) + index_base, s.shape)
        cat_s = np.concatenate([best_s, s], axis=1)
        cat_i = np.where(np.isneginf(cat_s), -1, np.concatenate([best_i, idx], axis=1))
        best_s, best_i = merge_topk(cat_s, cat_i, k)
    return best_s, best_i


def masked_rank_excluding(q: np.ndarray, catalog: np.ndarray, targets: np.ndarray, lists,
                          row_type: Optional[np.ndarray] = None, type_id: Optional[np.ndarray] = None,
                          index_base: int = 0, chunk: int = 1 << 16) -> np.ndarray:
    """masked_rank counting only the products that are not in lists[r] (the target itself always counts as not
    excluded, so it never matters whether a list names it)."""
    r = q.shape[0]
    targets = np.asarray(targets, dtype=np.int64)
    local = targets - index_base
    member = (local >= 0) & (local < catalog.shape[0])
    safe = np.where(member, local, 0)
    if row_type is not None:
        member &= type_id[safe] == row_type
    t_score = np.array([scores_fp64(q[i:i + 1], catalog[safe[i]:safe[i] + 1])[0, 0] for i in range(r)])
    count = np.zeros(r, dtype=np.int64)
    for beg in range(0, catalog.shape[0], chunk):
        end = min(beg + chunk, catalog.shape[0])
        s = scores_fp64(q, catalog[beg:end])
        idx = np.arange(beg, end, dtype=np.int64)[None, :] + index_base
        before = (s > t_score[:, None]) | ((s == t_score[:, None]) & (idx < targets[:, None]))
        if row_type is not None:
            before &= type_id[None, beg:end] == row_type[:, None]
        for i in range(r):
            if lists[i] is not None:
                before[i, _excluded(lists, i, index_base, beg, end) - beg] = False
        count += before.sum(axis=1)
    return np.where(member, count, -1)
