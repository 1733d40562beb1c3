"""Cost of k for the type-segmented exact top-K (pc_topk_by_type) at the C4 shape of bench.py --workload retrieval:
10 M x 128 fp32 catalog (5.12 GB, larger than the 126 MB L2), 1 K types, 4,096 queries x 3 type rows.

Every k runs in the same process on the same inputs.  After a warm-up of every k, the k values are alternated round by
round so that clock and co-tenant drift spreads over all of them.  A sample is the device time of one pc_topk_by_type
call (CUDA events around the native call, as bench.py's abi_ms_per_step): type keys, sort, plan, ranking kernel, and
the split merge when the automatic split count is above 1.  The GPU name and power limit are read in the same run.

    python profiles/topk_large_k.py [--out profiles/topk_large_k.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KS = (10, 32, 33, 100, 256, 1000, 1024)


def gpu_info(index: int) -> dict:
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit,clocks.max.sm,driver_version",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=60).stdout.strip()
        power, clock, driver = [x.strip() for x in out.split(",")]
        info.update(power_limit_w=float(power), sm_max_mhz=float(clock), driver=driver)
    except Exception as e:  # the measurement stands without it, but say so
        info["nvidia_smi_error"] = repr(e)
    return info


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "topk_large_k.json"))
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=10, help="timed calls per k per round")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_large_k.py: no CUDA device (this is a GPU measurement)")
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

    def timed(k: int, calls: int) -> list:
        _lib.PROFILE = []
        for _ in range(calls):
            index.topk(queries, k, row_type)
        torch.cuda.synchronize()
        prof, _lib.PROFILE = _lib.PROFILE, None
        return [s0.elapsed_time(s1) for name, s0, s1 in prof if name == "pc_topk_by_type"]

    for k in KS:                                                # warm-up: module load, workspace sizes, clocks
        timed(k, 3)
    samples = {k: [] for k in KS}
    for rnd in range(args.rounds):
        for k in (KS if rnd % 2 == 0 else KS[::-1]):
            samples[k] += timed(k, args.calls)
    s10 = statistics.median(samples[10])
    results = {}
    for k in KS:
        med = statistics.median(samples[k])
        results[str(k)] = {"median_ms": round(med, 4), "min_ms": round(min(samples[k]), 4), "max_ms": round(max(samples[k]), 4),
                           "samples": len(samples[k]), "vs_k10": round(med / s10, 3)}
    line = {"what": "pc_topk_by_type device time per call vs k (C4 shape)", "gpu": gpu_info(0),
            "shape": {"catalog": [p, 128], "types": n_types, "score_rows": q_n * 3, "queries": q_n},
            "rounds": args.rounds, "calls_per_round": args.calls, "l2": "catalog 5.12 GB > 126 MB L2; no flush",
            "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
