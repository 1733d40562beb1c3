"""Cost of the exact target rank (pc_rank_by_type) against the top-K call it replaces for evaluation (pc_topk_by_type
at k = 10 and k = 100), at the C4 shape of bench.py --workload retrieval: 10 M x 128 fp32 catalog (5.12 GB, larger
than the 126 MB L2), 1 K types, 4,096 queries x 3 type rows, each row's target a random member of its type.

Before timing, the rank / top-K property is asserted at k = 10 on the timed inputs: a row's target is in its top-10
list exactly when its rank is below 10, and then at that position.  After a warm-up of every call, the three calls are
alternated round by round so that clock and co-tenant drift spreads over all of them.  A sample is the device time of
one native call (CUDA events around it, as bench.py's abi_ms_per_step): type keys, sort, plan, scoring kernel, and for
top-K the split merge when the automatic split count is above 1.  The GPU name and power limit are read in the same run.

    python profiles/rank_by_type.py [--out profiles/rank_by_type.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from topk_large_k import gpu_info  # noqa: E402

CALLS = ("rank", "topk_k10", "topk_k100")


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rank_by_type.json"))
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=10, help="timed calls per kind per round")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank_by_type.py: no CUDA device (this is a GPU measurement)")
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib

    dev = torch.device("cuda:0")
    p, n_types, q_n = 10_000_000, 1000, 4096
    g = torch.Generator(device=dev).manual_seed(1234)           # bench.py's SEED: the same catalog and queries
    catalog = torch.randn(p, 128, generator=g, device=dev)
    type_id = torch.randint(0, n_types, (p,), generator=g, device=dev, dtype=torch.int32)
    index = pc.CatalogIndex(catalog, type_id, num_types=n_types)
    gq = torch.Generator(device=dev).manual_seed(1234)
    queries = torch.randn(q_n * 3, 128, generator=gq, device=dev)
    row_type = torch.randint(0, n_types, (q_n * 3,), generator=gq, device=dev, dtype=torch.int32)
    # target of row r: a uniformly drawn member of its type's run of the type-sorted permutation
    lo, hi = index.offsets[row_type.long()], index.offsets[row_type.long() + 1]
    n = hi - lo
    assert bool((n > 0).all()), "every type has products at this shape"
    u = torch.rand(q_n * 3, generator=torch.Generator(device=dev).manual_seed(99), device=dev, dtype=torch.float64)
    targets = index.members[lo + torch.minimum((u * n.double()).long(), n - 1)].long()
    assert bool((type_id[targets] == row_type).all()), "every target is a member of its row's type"

    ranks = index.rank(queries, targets, row_type)
    _, top10 = index.topk(queries, 10, row_type)
    hit = top10 == targets[:, None]
    listed = hit.any(1)
    assert torch.equal(listed, (ranks >= 0) & (ranks < 10)), "rank < 10 <=> target in the top-10 list"
    assert torch.equal(hit.int().argmax(1)[listed], ranks[listed]), "rank == position in the top-10 list"
    assert bool((ranks >= 0).all())

    run = {"rank": lambda: index.rank(queries, targets, row_type),
           "topk_k10": lambda: index.topk(queries, 10, row_type),
           "topk_k100": lambda: index.topk(queries, 100, row_type)}
    native = {"rank": "pc_rank_by_type", "topk_k10": "pc_topk_by_type", "topk_k100": "pc_topk_by_type"}

    def timed(kind: str, calls: int) -> list:
        _lib.PROFILE = []
        for _ in range(calls):
            run[kind]()
        torch.cuda.synchronize()
        prof, _lib.PROFILE = _lib.PROFILE, None
        return [s0.elapsed_time(s1) for name, s0, s1 in prof if name == native[kind]]

    for kind in CALLS:                                          # warm-up: module load, workspace sizes, clocks
        timed(kind, 3)
    samples = {kind: [] for kind in CALLS}
    for rnd in range(args.rounds):
        for kind in (CALLS if rnd % 2 == 0 else CALLS[::-1]):
            samples[kind] += timed(kind, args.calls)
    s10 = statistics.median(samples["topk_k10"])
    results = {}
    for kind in CALLS:
        med = statistics.median(samples[kind])
        results[kind] = {"native": native[kind], "median_ms": round(med, 4), "min_ms": round(min(samples[kind]), 4),
                         "max_ms": round(max(samples[kind]), 4), "samples": len(samples[kind]),
                         "vs_topk_k10": round(med / s10, 3)}
    line = {"what": "pc_rank_by_type vs pc_topk_by_type device time per call (C4 shape)", "gpu": gpu_info(0),
            "shape": {"catalog": [p, 128], "types": n_types, "score_rows": q_n * 3, "queries": q_n},
            "rank_topk_consistency_k10": "asserted", "rows_with_rank_below_10": int(((ranks < 10)).sum().item()),
            "rounds": args.rounds, "calls_per_round": args.calls, "l2": "catalog 5.12 GB > 126 MB L2; no flush",
            "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
