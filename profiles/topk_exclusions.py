"""Cost of exclusion lists in the retrieval kernels at the C4 shape of profiles/rank_by_type.py: 10 M x 128 fp32
catalog (5.12 GB, larger than the 126 MB L2), 1 K types, 4,096 queries x 3 type rows, the same seeds.

Timed calls (device time of one native call, CUDA events around it, as bench.py's abi_ms_per_step):
  topk_k10            pc_topk_by_type, k = 10, no exclusions
  topk_k10_excl16     pc_topk_by_type_excluding, k = 10, 16 random products of the row's type excluded per row
  topk_k10_excl_top64 pc_topk_by_type_excluding, k = 10, the row's true top-64 excluded (adversarial: every product
                      that would be listed is tested and rejected)
  topk_k74            pc_topk_by_type, k = 74: the over-fetch alternative (k + 64 entries, drop on the host)
  rank                pc_rank_by_type
  rank_excl256        pc_rank_by_type + pc_rank_remove_excluded, 256 random products of the row's type per row
                      (the correction is also reported alone)

Before timing, on the timed inputs: filtered top-10 equals the over-fetched top-74 with the excluded entries removed
(both lists), and the filtered rank agrees with the filtered top-10 (rank < 10 <=> listed, at that position; the
top-K side excludes each row's list without its target).  After a warm-up of every call, the calls alternate round by
round.  The GPU name and power limit are read in the same run.

    python profiles/topk_exclusions.py [--out profiles/topk_exclusions.json]
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

CALLS = ("topk_k10", "topk_k10_excl16", "topk_k10_excl_top64", "topk_k74", "rank", "rank_excl256")


def _same_type_draw(index, row_type, n, seed):
    """[R, n] uniformly drawn members (with repetition) of each row's type, as global indices."""
    lo, hi = index.offsets[row_type.long()], index.offsets[row_type.long() + 1]
    u = torch.rand(row_type.numel(), n, generator=torch.Generator(device=row_type.device).manual_seed(seed),
                   device=row_type.device, dtype=torch.float64)
    cnt = (hi - lo)[:, None]
    return index.members[lo[:, None] + torch.minimum((u * cnt.double()).long(), cnt - 1)].long()


def _csr(rows_of_lists):
    r, n = rows_of_lists.shape
    return torch.arange(r + 1, device=rows_of_lists.device, dtype=torch.int64) * n, rows_of_lists.reshape(-1)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "topk_exclusions.json"))
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=10, help="timed calls per kind per round")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_exclusions.py: no CUDA device (this is a GPU measurement)")
    import pcompanion_b200 as pc
    from pcompanion_b200 import Exclusions, _lib

    dev = torch.device("cuda:0")
    p, n_types, q_n = 10_000_000, 1000, 4096
    rows = q_n * 3
    g = torch.Generator(device=dev).manual_seed(1234)           # bench.py's SEED: the same catalog and queries
    catalog = torch.randn(p, 128, generator=g, device=dev)
    type_id = torch.randint(0, n_types, (p,), generator=g, device=dev, dtype=torch.int32)
    index = pc.CatalogIndex(catalog, type_id, num_types=n_types)
    gq = torch.Generator(device=dev).manual_seed(1234)
    queries = torch.randn(rows, 128, generator=gq, device=dev)
    row_type = torch.randint(0, n_types, (rows,), generator=gq, device=dev, dtype=torch.int32)
    targets = _same_type_draw(index, row_type, 1, 99)[:, 0]     # as rank_by_type.py: one random member per row
    assert bool((type_id[targets] == row_type).all())

    top74_s, top74 = index.topk(queries, 74, row_type)
    ex16 = Exclusions(*_csr(_same_type_draw(index, row_type, 16, 7)))
    ex64 = Exclusions(*_csr(top74[:, :64].contiguous()))
    e256 = _same_type_draw(index, row_type, 256, 11)
    e256[::4, 0] = targets[::4]                                 # a quarter of the rows also list their own target
    ex256 = Exclusions(*_csr(e256))

    # filtered top-10 == over-fetched top-74 less the excluded entries, truncated to 10 (16 and 64 entries <= 64)
    for ex, e in ((ex16, ex16.indices.view(rows, 16)), (ex64, top74[:, :64])):
        s, i = index.topk(queries, 10, row_type, exclude=ex)
        keep = ~(top74[:, :, None] == e[:, None, :]).any(2)
        order = torch.sort((~keep).to(torch.int8), dim=1, stable=True).indices[:, :10]
        assert bool((keep.sum(1) >= 10).all())
        assert torch.equal(i, top74.gather(1, order)) and torch.equal(s, top74_s.gather(1, order)), "over-fetch check"
    # filtered rank vs filtered top-10 with each row's list minus its own target
    ranks = index.rank(queries, targets, row_type, exclude=ex256)
    minus = torch.where(e256 == targets[:, None], torch.full_like(e256, -1), e256)
    _, top10 = index.topk(queries, 10, row_type, exclude=Exclusions(*_csr(minus)))
    hit = top10 == targets[:, None]
    listed = hit.any(1)
    assert torch.equal(listed, (ranks >= 0) & (ranks < 10)), "filtered rank < 10 <=> target in the filtered top-10"
    assert torch.equal(hit.int().argmax(1)[listed], ranks[listed]), "filtered rank == position in the filtered top-10"
    plain_ranks = index.rank(queries, targets, row_type)
    assert bool((ranks >= 0).all() and (ranks <= plain_ranks).all())

    run = {"topk_k10": lambda: index.topk(queries, 10, row_type),
           "topk_k10_excl16": lambda: index.topk(queries, 10, row_type, exclude=ex16),
           "topk_k10_excl_top64": lambda: index.topk(queries, 10, row_type, exclude=ex64),
           "topk_k74": lambda: index.topk(queries, 74, row_type),
           "rank": lambda: index.rank(queries, targets, row_type),
           "rank_excl256": lambda: index.rank(queries, targets, row_type, exclude=ex256)}
    native = {"topk_k10": ("pc_topk_by_type",), "topk_k10_excl16": ("pc_topk_by_type_excluding",),
              "topk_k10_excl_top64": ("pc_topk_by_type_excluding",), "topk_k74": ("pc_topk_by_type",),
              "rank": ("pc_rank_by_type",), "rank_excl256": ("pc_rank_by_type", "pc_rank_remove_excluded")}

    def timed(kind: str, calls: int) -> dict:
        _lib.PROFILE = []
        for _ in range(calls):
            run[kind]()
        torch.cuda.synchronize()
        prof, _lib.PROFILE = _lib.PROFILE, None
        return {name: [s0.elapsed_time(s1) for n, s0, s1 in prof if n == name] for name in native[kind]}

    for kind in CALLS:                                          # warm-up: module load, workspace sizes, clocks
        timed(kind, 3)
    samples = {kind: {name: [] for name in native[kind]} for kind in CALLS}
    for rnd in range(args.rounds):
        for kind in (CALLS if rnd % 2 == 0 else CALLS[::-1]):
            for name, v in timed(kind, args.calls).items():
                samples[kind][name] += v
    results = {}
    for kind in CALLS:
        per_call = [sum(x) for x in zip(*samples[kind].values())]
        results[kind] = {"native": "+".join(native[kind]), "median_ms": round(statistics.median(per_call), 4),
                         "min_ms": round(min(per_call), 4), "max_ms": round(max(per_call), 4), "samples": len(per_call)}
        if len(native[kind]) > 1:
            results[kind]["median_ms_each"] = {n: round(statistics.median(v), 4) for n, v in samples[kind].items()}
    base = {"topk": results["topk_k10"]["median_ms"], "rank": results["rank"]["median_ms"]}
    for kind in CALLS:
        results[kind]["vs_unfiltered"] = round(results[kind]["median_ms"] / base["rank" if kind.startswith("rank") else "topk"], 3)
    line = {"what": "exclusion lists in pc_topk_by_type / pc_rank_by_type: device time per call (C4 shape)",
            "gpu": gpu_info(0), "shape": {"catalog": [p, 128], "types": n_types, "score_rows": rows, "queries": q_n},
            "checks": "over-fetch equality (16 and top-64 excluded) and filtered rank / filtered top-10 property asserted",
            "rows_with_filtered_rank_below_10": int((ranks < 10).sum().item()),
            "rows_with_rank_below_10": int((plain_ranks < 10).sum().item()),
            "rounds": args.rounds, "calls_per_round": args.calls, "l2": "catalog 5.12 GB > 126 MB L2; no flush",
            "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
