"""Graph-native Product2Vec training (Product2Vec.train_model_graph's loop) against the drop-in loop.

C1 (the reference's default synthetic BPG, 1,000 products, B = 256, DROPOUT 0.1, fused Adam): one epoch of
  dropin  bench.py's c1_leg loop as it runs there: SimilarityDataset + DataLoader(shuffle) + collate_fn, per batch
          .to(device), forward(anchor, neighbours) / forward(positive) / forward(negative), triplet_loss, Adam step and
          a device synchronise (c1_leg's data / compute split);
  graph   train_model_graph's loop over the same similarity pairs: GraphTripletSampler.neighborhood_batches ->
          triplet_loss_graph -> zero_grad / backward / step, loss summed on the device, read once at the end.
  Both epochs are wall clock including the data path.  The two alternate, epoch by epoch, after one warm-up epoch each.
  Reported per path: seconds per epoch (median and all rounds), samples/s, C-ABI launches per step, and host reads per
  epoch (synchronising calls flagged by torch.cuda.set_sync_debug_mode in one extra un-timed epoch; the drop-in loop's
  per-batch timing synchronise is left out of that epoch).
C2-sized synthetic graph (1 M products, 20 M co-view edges, synthetic_bpg): steps/s and samples/s of the graph loop at
  B = 256, 4,096 and 65,536 with the neighbour rows per step.  The epoch's plan (permutation, degree prefix sum, one
  host read) together with the first batch's negatives is timed on its own; the first step then runs untimed, and
  each timed step after it includes drawing its batch's negatives.  Warm-up steps first; the batch sizes alternate
  round by round.

The GPU name and power limit are read in the same run.

    python profiles/p2v_graph_training.py [--out profiles/p2v_graph_training.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from topk_large_k import gpu_info  # noqa: E402

C2_BATCHES = (256, 4096, 65536)
C2_STEPS = {256: 200, 4096: 50, 65536: 8}


def count_syncs(fn) -> int:
    """Synchronising CUDA calls made by fn() (torch.cuda.set_sync_debug_mode('warn'))."""
    torch.cuda.synchronize()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            fn()
        finally:
            torch.cuda.set_sync_debug_mode("default")
    return sum("synchronizing" in str(w.message).lower() for w in caught)


def c1(dev, rounds: int) -> dict:
    import bench
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib
    from torch.utils.data import DataLoader
    cfg = bench.make_cfg(dev)
    bpg = bench.c1_bpg(dev)
    ds = pc.SimilarityDataset(bpg, cfg)
    loader = DataLoader(ds, batch_size=256, shuffle=True, collate_fn=pc.collate_fn, num_workers=0)
    smp = pc.GraphTripletSampler(bpg)
    csr, x = bpg.csr("co_view"), bpg.features
    assert len(smp) == len(ds)
    torch.manual_seed(bench.SEED)
    m_drop = pc.Product2Vec(cfg).to(dev)
    m_graph = pc.Product2Vec(cfg).to(dev)
    m_graph.load_state_dict(m_drop.state_dict())
    o_drop = torch.optim.Adam(m_drop.parameters(), lr=cfg.LEARNING_RATE, fused=True)
    o_graph = torch.optim.Adam(m_graph.parameters(), lr=cfg.LEARNING_RATE, fused=True)
    epoch_no = [0]

    def dropin(timing_sync=True):
        m_drop.train()
        steps = 0
        for batch in loader:
            batch = {k: v.to(dev) if isinstance(v, torch.Tensor) else v for k, v in batch.items()}
            a = m_drop(batch["anchor"], batch.get("anchor_neighbors"))
            p = m_drop(batch["positive"])
            n = m_drop(batch["negative"])
            loss = m_drop.triplet_loss(a, p, n)
            o_drop.zero_grad(); loss.backward(); o_drop.step()
            steps += 1
            if timing_sync:
                torch.cuda.synchronize()
        return steps, float(loss.item())

    def graph():
        m_graph.train()
        total = torch.zeros((), device=dev)
        steps = 0
        epoch_no[0] += 1
        for batch in smp.neighborhood_batches(256, bench.SEED * 100_003 + epoch_no[0], csr):
            loss = m_graph.triplet_loss_graph(x, csr, batch)
            o_graph.zero_grad(); loss.backward(); o_graph.step()
            total += loss.detach()
            steps += 1
        return steps, float(total.item()) / steps

    def timed(fn):
        torch.cuda.synchronize()
        l0 = _lib.LAUNCHES
        t0 = time.perf_counter()
        steps, loss = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, (_lib.LAUNCHES - l0) / steps, steps, loss

    dropin(); graph()                                                          # warm-up
    res = {"dropin": [], "graph": []}
    for _ in range(rounds):
        res["dropin"].append(timed(dropin))
        res["graph"].append(timed(graph))
    syncs = {"dropin": count_syncs(lambda: dropin(timing_sync=False)), "graph": count_syncs(graph)}
    out = {}
    for k, runs in res.items():
        secs = [r[0] for r in runs]
        med = statistics.median(secs)
        out[k] = {"epoch_s_median": med, "epoch_s": secs, "samples_per_s": len(ds) / med, "steps_per_epoch": runs[0][2],
                  "c_abi_launches_per_step": runs[0][1], "host_reads_per_epoch": syncs[k], "last_loss": runs[-1][3]}
    out["speedup"] = out["dropin"]["epoch_s_median"] / out["graph"]["epoch_s_median"]
    out["samples_per_epoch"] = len(ds)
    return out


def c2(dev, rounds: int) -> dict:
    import pcompanion_b200 as pc
    from pcompanion_b200.synthetic import synthetic_bpg
    import bench
    t0 = time.perf_counter()
    bpg = synthetic_bpg(1_000_000, 20_000_000, seed=bench.SEED, device=dev)
    smp = pc.GraphTripletSampler(bpg)
    csr, x = bpg.csr("co_view"), bpg.features
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    deg = csr.rowptr[1:] - csr.rowptr[:-1]
    torch.manual_seed(bench.SEED)
    model = pc.Product2Vec(bench.make_cfg(dev)).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, fused=True)
    res = {b: {"steps_s": [], "nbr_rows": [], "plan_s": []} for b in C2_BATCHES}

    def run(b, steps, seed):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        it = smp.neighborhood_batches(b, seed, csr)
        batch = next(it)                                     # the epoch's plan, its one read, the first batch's negatives
        torch.cuda.synchronize()
        plan_s = time.perf_counter() - t0
        loss = model.triplet_loss_graph(x, csr, batch)                         # untimed first step
        opt.zero_grad(); loss.backward(); opt.step()
        torch.cuda.synchronize()
        nbr = []
        t0 = time.perf_counter()
        for _ in range(steps):
            batch = next(it)
            loss = model.triplet_loss_graph(x, csr, batch)
            opt.zero_grad(); loss.backward(); opt.step()
            nbr.append(batch.n_nbr)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, plan_s, nbr

    for b in C2_BATCHES:
        run(b, 3, seed=0)                                                      # warm-up
    for r in range(rounds):
        for b in C2_BATCHES:
            dt, plan_s, nbr = run(b, C2_STEPS[b], seed=r + 1)
            res[b]["steps_s"].append(C2_STEPS[b] / dt)
            res[b]["plan_s"].append(plan_s)
            res[b]["nbr_rows"].extend(nbr)
    out = {"products": bpg.num_nodes, "co_view_edges": csr.num_edges, "similarity_pairs": len(smp),
           "max_co_view_degree": int(deg.max()), "graph_build_s": build_s, "batches": {}}
    for b, v in res.items():
        med = statistics.median(v["steps_s"])
        out["batches"][str(b)] = {"steps_per_s_median": med, "steps_per_s": v["steps_s"], "samples_per_s": med * b,
                                  "neighbour_rows_per_step_mean": statistics.mean(v["nbr_rows"]),
                                  "timed_steps_per_round": C2_STEPS[b],
                                  "plan_and_first_negatives_s_median": statistics.median(v["plan_s"])}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "p2v_graph_training.json"))
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("p2v_graph_training.py needs a CUDA device")
    dev = torch.device("cuda:0")
    result = {"what": __doc__.strip().splitlines()[0], "gpu": gpu_info(0), "rounds": args.rounds,
              "c1": c1(dev, args.rounds), "c2": c2(dev, args.rounds)}
    result["gpu_after"] = gpu_info(0)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
