"""Reference target rank (test infrastructure only), on the score definition of oracle/retrieval.py.

The rank of row r's target g is the number of products p of the row's type (of the whole catalog without row types)
with (score[r, p], p) before (score[r, g], g) under the ranking rule (score descending, then lower index).  It is -1
when the target can never appear in the row's list: g outside the catalog, or type_id[g] != row_type[r].
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from oracle.retrieval import scores_fp64


def masked_rank(q: np.ndarray, catalog: np.ndarray, targets: np.ndarray, row_type: Optional[np.ndarray] = None,
                type_id: Optional[np.ndarray] = None, index_base: int = 0, chunk: int = 1 << 16) -> np.ndarray:
    """int64 [R] ranks of the global indices `targets` against `catalog` (global ids index_base .. + P - 1)."""
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
        count += before.sum(axis=1)
    return np.where(member, count, -1)
