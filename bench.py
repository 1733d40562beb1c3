#!/usr/bin/env python
"""Benchmark of the P-Companion hot path on B200 (contract: see the task statement / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload all|gat|gat_skewed|retrieval|retrieval_dense|pcompanion|c1|c5] [--dump-outputs DIR]

Every timed region is exactly K steps.  With the same arguments every run draws the same inputs, so two builds can be
compared output for output with --dump-outputs.

BASELINE.json's metric has two halves - "GAT edges/sec fwd+bwd (Product2Vec) & top-K queries/sec at 1/2/4/8 B200" -
so the default run (`--workload all`) measures both and prints ONE JSON line on rank 0:

* the line itself is configs[1] (C2): synthetic BPG with 1 M products / ~20 M co-view edges per GPU, one step = full-graph
  Product2Vec GAT forward + triplet hinge + backward + Adam (every destination, every edge, per-node FFN / QKV /
  out-proj included); `value` = co-view edges per second, whole job; at N > 1 the graph is node-partitioned with a halo
  exchange and the line carries the multi-GPU parity check that ran before the timing;
* `retrieval` (C4: masked top-10 over a 10 M-product catalog, 1 K types, sharded over the ranks) and, at N = 1,
  `retrieval_dense` (the north-star's tensor-core wording of the same query) - `topk_queries_per_sec` repeats the value;
* `pcompanion` (C3: joint P-Companion step on a 1 M-product table, 34,800 types, batch 256 and 65,536);
* at N = 1 also `gat_skewed` (the same step on a power-law graph, hub splitting on / off) and `c1` (configs[0]).

Every sub-record has its own value / ms_per_step / roofline / e2e (/ cpu_baseline at N = 1).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NODES_PER_GPU = 1_000_000
EDGES_PER_GPU = 20_000_000
TRIPLETS = 131_072
KNEG = 5
SEED = 1234
FP64_TFLOPS_NOMINAL = 37.0   # B200 vector fp64 (HGX B200: 296 TFLOP/s per 8 GPUs); no measured figure in MEASURED_PEAKS.json

# SURVEY.md 8(d): algorithmic bytes of the three sparse kernels (fp32, per edge / per node)
ALGO_BYTES = {
    "pc_gat_fwd": (1028, 1060),
    "pc_gat_bwd_dst": (1060, 1588),
    "pc_gat_bwd_src": (1064, 1028),
}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["bf16_tflops_sustained"]), "measured bf16 sustained (MEASURED_PEAKS.json); kind::tf32 runs at half the bf16 rate"
    return 1400.0, "fallback (B200_PROFILING.md); kind::tf32 runs at half the bf16 rate"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms.  The process is started BEFORE the warm-up (its start-up
    takes driver locks that stall kernel launches for tens of ms - enough to halve a 40 ms timed region); `mark()` is
    called when the timed region starts and only samples taken after it are reported (all of them if the region was
    shorter than one sampling period)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.proc = None
        self.t_mark = None
        if int(os.environ.get("RANK", 0)) != 0:
            return          # one sampler per job (rank 0's GPU): eight nvidia-smi pollers perturb millisecond-scale steps
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def mark(self):
        self.t_mark = time.time()
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        import datetime
        time.sleep(0.15)
        self.proc.terminate()
        out = self.proc.communicate()[0]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), [n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [r for r in rows if self.t_mark is None or r[0] >= self.t_mark - 0.05]
        use = inside if inside else rows[-1:]
        sm = sorted(r[1] for r in use)
        reasons = sorted({n for r in use for n in r[3]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((r[2] for r in use), default=None),
                "samples": len(use), "reasons": reasons}


def make_cfg(device):
    # reference config.py:8-24 defaults (DROPOUT = 0.1 stays on: attention dropout is part of a training step)
    return SimpleNamespace(PRODUCT_EMB_DIM=128, TYPE_EMB_DIM=64, HIDDEN_SIZE=256, NUM_ATTENTION_HEADS=4, DROPOUT=0.1,
                           MARGIN=1.0, ALPHA=0.8, NUM_COMP_TYPES=3, NUM_TYPES=34800, LEARNING_RATE=1e-3, DEVICE=device)


def _dist():
    import torch.distributed as dist
    return dist


def max_over_ranks(values, dev, world):
    t = torch.tensor(list(values), dtype=torch.float64, device=dev)
    if world > 1:
        _dist().all_reduce(t, op=_dist().ReduceOp.MAX)
    return t.tolist()


class L2Flush:
    """Between timed iterations of a leg whose working set fits the 126 MB L2: overwrite a 256 MB buffer (not timed)."""

    def __init__(self, dev):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def __call__(self):
        self.buf.zero_()


def warm_up(fn, min_steps, min_seconds, dev, world):
    """At least `min_steps` untimed calls AND about `min_seconds` of them (short steps must not be timed on a GPU that is
    still ramping its clocks).  The number of extra calls is derived from the max-over-ranks elapsed time, so every rank
    runs the SAME count - fn may contain collectives."""
    t0 = time.perf_counter()
    for _ in range(min_steps):
        fn()
    torch.cuda.synchronize()
    elapsed = max_over_ranks([time.perf_counter() - t0], dev, world)[0]
    if elapsed < min_seconds:
        extra = min(int(math.ceil((min_seconds - elapsed) / max(elapsed / max(min_steps, 1), 1e-5))), 2000)
        for _ in range(extra):
            fn()
        torch.cuda.synchronize()


class TrainingState:
    """A copy of what a training step reads and changes - parameters and buffers, optimiser state and torch's CPU generator
    (it draws the dropout seeds) - that restore() writes back in place.  Taken after exactly --warmup steps and restored
    after the time-based part of the warm-up, so the timed steps compute the same numbers in every run with the same
    arguments, however many steps the clocks needed."""

    def __init__(self, model, opt):
        self.live = list(model.state_dict().values()) + [v for s in opt.state.values() for v in s.values() if torch.is_tensor(v)]
        self.saved = [t.clone() for t in self.live]
        self.rng = torch.get_rng_state()

    def restore(self):
        with torch.no_grad():
            for t, s in zip(self.live, self.saved):
                t.copy_(s)
        torch.set_rng_state(self.rng)
        torch.cuda.synchronize()


def dump_outputs(args, prefix, arrays):
    """--dump-outputs DIR: every array as DIR/<prefix>.<name>.npy; floating point keeps float64 or becomes float32,
    integers become float64 (exact for indices below 2**53)."""
    import numpy as np
    os.makedirs(args.dump_outputs, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        a = a.astype(np.float32 if a.dtype.kind == "f" and a.dtype != np.float64 else np.float64)
        np.save(os.path.join(args.dump_outputs, f"{prefix}.{name}.npy"), a)


def timed_steps(fn, steps, dev, world, flush=None):
    """Average device time of exactly `steps` calls of fn (CUDA events on the current stream, barrier + synchronize on both
    sides, max over ranks) and fn's result of the last call.  With `flush` every step is timed on its own and the L2 flush
    between the steps is not."""
    torch.cuda.synchronize()
    if world > 1:
        _dist().barrier()
    out = None
    if flush is None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            out = fn()
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / steps
    else:
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            flush()
            a.record()
            out = fn()
            b.record()
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in evs) / steps
    if world > 1:
        _dist().barrier()
    return max_over_ranks([ms], dev, world)[0], out


# ============================================================================= GAT leg, one GPU (C2)
def gat_single(args, dev):
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib
    from pcompanion_b200.synthetic import synthetic_bpg
    # started before the graph is built: nvidia-smi's start-up takes driver locks that stall kernel launches for tens of ms,
    # it must be over long before the timed region (a 3-step warm-up alone is only ~70 ms)
    sampler = ClockSampler(dev.index)
    torch.manual_seed(SEED)
    t0 = time.perf_counter()
    bpg = synthetic_bpg(NODES_PER_GPU, EDGES_PER_GPU, seed=SEED, device=dev)
    graph = bpg.csr("co_view")
    graph.transposed()
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    n, e = graph.n_rows, graph.num_edges
    cfg = make_cfg(dev)
    model = pc.Product2Vec(cfg).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=cfg.LEARNING_RATE, fused=True)   # same Adam, one kernel for the 13 tensors
    g = torch.Generator(device=dev).manual_seed(SEED + 2)
    trip = torch.randint(0, n, (TRIPLETS, 2 + KNEG), generator=g, device=dev)
    x_dev = bpg.features
    # host copies for the end-to-end leg (pinned)
    x_host = x_dev.cpu().pin_memory()
    trip_host = trip.cpu().pin_memory()
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def step(x, tr, keep=None):
        emb = model.forward_graph(x, graph)
        loss = model.triplet_loss_indexed(emb, tr[:, 0], tr[:, 1], tr[:, 2:])
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        if keep is not None:
            keep["embeddings"] = emb.detach()
        return loss

    # end-to-end leg: every step's inputs come from pinned host memory.  The copy of step i+1 is issued on a
    # side stream while step i computes (double-buffered device staging), as a production input pipeline would.
    copy_stream = torch.cuda.Stream()
    stage = [(torch.empty_like(x_dev), torch.empty_like(trip), torch.cuda.Event()) for _ in range(2)]

    def prefetch(slot):
        xs, ts, ev = stage[slot]
        with torch.cuda.stream(copy_stream):
            xs.copy_(x_host, non_blocking=True)
            ts.copy_(trip_host, non_blocking=True)
            ev.record(copy_stream)

    def run_e2e(steps):
        prefetch(0)
        for i in range(steps):
            xs, ts, ev = stage[i % 2]
            torch.cuda.current_stream().wait_event(ev)
            if i + 1 < steps:
                copy_stream.wait_stream(torch.cuda.current_stream())   # slot (i+1)%2 was last read by step i-1
                prefetch((i + 1) % 2)
            loss = step(xs, ts)
            loss_host.copy_(loss.detach(), non_blocking=True)

    for _ in range(args.warmup):
        step(x_dev, trip)
    start = TrainingState(model, opt)
    warm_up(lambda: step(x_dev, trip), 1, 0.5, dev, 1)
    start.restore()

    # ---- device-resident timed region (per-kernel events on the launching stream)
    sampler.mark()
    _lib.PROFILE = []
    launches0 = _lib.LAUNCHES
    last = {} if args.dump_outputs else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for i in range(args.steps):
        loss = step(x_dev, trip, last if i == args.steps - 1 else None)
    ev1.record()
    torch.cuda.synchronize()
    total_ms = ev0.elapsed_time(ev1)
    prof, _lib.PROFILE = _lib.PROFILE, None
    launches = _lib.LAUNCHES - launches0
    clocks = sampler.stop()
    ms_per_step = total_ms / args.steps
    if args.dump_outputs:
        # the step's loss, the updated parameters / BatchNorm statistics, the gradients, and a fixed sample of the
        # embedding rows (all n x 128 of them would be 512 MB)
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(SEED))[:8192].sort().values
        dump_outputs(args, "gat", {"loss": loss, "embedding_rows": rows, "embeddings": last["embeddings"][rows.to(dev)],
                                   **{"state." + k: v for k, v in model.state_dict().items()},
                                   **{"grad." + k: p.grad for k, p in model.named_parameters() if p.grad is not None}})
        del last

    per_kernel = {}
    for name, s, t in prof:
        per_kernel.setdefault(name, []).append(s.elapsed_time(t))
    peak, peak_src = measured_peaks()
    kernels = {}
    for name, (be, bn) in ALGO_BYTES.items():
        if name in per_kernel:
            ms = sum(per_kernel[name]) / len(per_kernel[name])
            gbs = (be * e + bn * n) / (ms * 1e-3) / 1e9
            kernels[name] = {"ms": round(ms, 4), "algo_gbs": round(gbs, 1), "frac": round(gbs / peak, 4)}
    abi_ms = {name: round(sum(v) / args.steps, 4) for name, v in sorted(per_kernel.items(), key=lambda kv: -sum(kv[1]))}
    abi_calls = {name: len(v) // args.steps for name, v in per_kernel.items()}
    sparse_ms = sum(k["ms"] for k in kernels.values())
    dom = max(kernels, key=lambda k: kernels[k]["ms"])
    traffic, traffic_src = None, None
    for tname in ("r2_gat_dram_traffic.json", "r1_gat_dram_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath):   # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
            with open(tpath) as f:
                tj = json.load(f)
            if dom in tj["kernels"]:
                traffic, traffic_src = tj["kernels"][dom]["dram_bytes"], f"profiles/{tname} (ncu --set full, same workload)"
                break
    whole = (3152 * e + 3676 * n) / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["algo_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": ALGO_BYTES[dom][0] * e + ALGO_BYTES[dom][1] * n, "peak_source": peak_src,
                "sparse_fwd_bwd": {"ms": round(sparse_ms, 4),
                                   "algo_gbs": round((3152 * e + 3676 * n) / (sparse_ms * 1e-3) / 1e9, 1),
                                   "frac": round((3152 * e + 3676 * n) / (sparse_ms * 1e-3) / 1e9 / peak, 4)},
                "whole_step": {"ms": round(ms_per_step, 4), "algo_gbs": round(whole, 1), "frac": round(whole / peak, 4),
                               "note": "SURVEY 8(d) unit: the sparse kernels' algorithmic bytes against the WHOLE step "
                                       "(projections, BatchNorm, loss and Adam included)"},
                "kernels": kernels,
                "abi_ms_per_step": abi_ms, "abi_calls_per_step": abi_calls,
                "abi_total_ms_per_step": round(sum(abi_ms.values()), 3)}

    # ---- end-to-end leg: host buffers, H2D + D2H inside the timed region
    run_e2e(2)
    torch.cuda.synchronize()
    ev0.record()
    run_e2e(args.steps)
    ev1.record()
    torch.cuda.synchronize()
    e2e_ms = ev0.elapsed_time(ev1) / args.steps

    csr_build = time_csr_build(graph, peak)
    cpu = None if args.skip_cpu else cpu_baseline_gat(bpg, graph, cfg, seconds=12.0)
    return {
        "metric": "gat_edges_per_sec_fwd_bwd", "value": e / (ms_per_step * 1e-3), "unit": "edges/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2: synthetic BPG 1M products / 20M co-view edges, Product2Vec full-graph GAT fwd+bwd "
                               "(FFN+QKV+out-proj per node, triplet hinge on 131072 triplets, Adam), 1xB200",
                   "nodes": n, "edges": e, "heads": 4, "dropout": cfg.DROPOUT, "triplets": TRIPLETS,
                   "l2": "working set (K|V 1 GB, Q 0.5 GB) exceeds the 126 MB L2; no flush needed",
                   "bpg_build_s": round(build_s, 3)},
        "csr_build": csr_build,
        "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
        "e2e": {"value": e / (e2e_ms * 1e-3), "unit": "edges/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": x_host.numel() * 4 + trip_host.numel() * 8, "d2h_bytes_per_step": 4},
        "gpu_launches": launches, "loss": float(loss.item()),
    }


# ============================================================================= GAT leg on a skewed-degree graph (SURVEY H8)
def gat_skewed_leg(args, dev):
    """Same Product2Vec step on a power-law graph: 1 M products, ~20 M co-view edges, out-degrees and in-degrees Pareto
    (alpha 1.5) - a handful of products with 10^4..10^5 neighbours.  Timed with hub splitting (ops.HUB_THRESHOLD) and with
    one warp per row regardless of its degree."""
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib, ops
    n = NODES_PER_GPU
    g = torch.Generator(device=dev).manual_seed(SEED + 11)
    alpha, xm = 1.5, EDGES_PER_GPU / NODES_PER_GPU / 3.0
    deg = (xm * torch.rand(n, generator=g, device=dev).clamp_(min=1e-7).pow(-1.0 / alpha)).long().clamp_(max=n // 8)
    src = torch.repeat_interleave(torch.arange(n, device=dev, dtype=torch.int32), deg)
    wcol = torch.rand(n, generator=g, device=dev).clamp_(min=1e-7).pow(-1.0 / alpha)
    cdf = torch.cumsum(wcol.double(), 0)
    dst = torch.searchsorted(cdf, torch.rand(src.numel(), generator=g, device=dev, dtype=torch.float64) * cdf[-1]).clamp_(max=n - 1).to(torch.int32)
    base, _ = ops.build_csr(src, dst, n)
    del src, dst, cdf
    base.transposed()
    e = base.num_edges
    out_deg = base.rowptr[1:] - base.rowptr[:-1]
    colptr, _ = base.transposed()
    in_deg = colptr[1:] - colptr[:-1]
    cfg = make_cfg(dev)
    x = torch.randn(n, 128, generator=g, device=dev)
    trip = torch.randint(0, n, (TRIPLETS, 2 + KNEG), generator=g, device=dev)
    res = {}
    for name, split in (("hub_split", True), ("one_warp_per_row", False)):
        graph = ops.CSRGraph(base.rowptr, base.col, n, n, base._t, split_hubs=split)
        torch.manual_seed(SEED)
        model = pc.Product2Vec(cfg).to(dev).train()
        opt = torch.optim.Adam(model.parameters(), lr=cfg.LEARNING_RATE, fused=True)   # same Adam, one kernel for the 13 tensors

        def step():
            emb = model.forward_graph(x, graph)
            loss = model.triplet_loss_indexed(emb, trip[:, 0], trip[:, 1], trip[:, 2:])
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            return loss
        for _ in range(args.warmup):
            step()
        _lib.PROFILE = []
        ms, loss = timed_steps(step, args.steps, dev, 1)
        prof, _lib.PROFILE = _lib.PROFILE, None
        per = {}
        for nm, s0, s1 in prof:
            per[nm] = per.get(nm, 0.0) + s0.elapsed_time(s1) / args.steps
        res[name] = {"ms_per_step": ms, "edges_per_s": e / (ms * 1e-3), "loss": float(loss.item()),
                     "gat_ms": {k: round(v, 3) for k, v in per.items() if k.startswith("pc_gat") or k == "pc_rows_segment_sum"}}
    hs, hst = ops.CSRGraph(base.rowptr, base.col, n, n, base._t).hub_split(), ops.CSRGraph(base.rowptr, base.col, n, n, base._t).hub_split_t()
    return {"metric": "gat_edges_per_sec_fwd_bwd_skewed", "value": res["hub_split"]["edges_per_s"], "unit": "edges/s", "n_gpus": 1,
            "ms_per_step": res["hub_split"]["ms_per_step"],
            "config": {"workload": "power-law BPG: 1M products, Pareto(1.5) out- and in-degrees, Product2Vec full-graph GAT fwd+bwd + "
                                   "triplet hinge + Adam", "nodes": n, "edges": e, "max_out_degree": int(out_deg.max().item()),
                       "max_in_degree": int(in_deg.max().item()), "hub_threshold": ops.HUB_THRESHOLD, "hub_segment": ops.HUB_SEGMENT,
                       "hub_rows": 0 if hs is None else int(hs.hub_rows.numel()), "hub_columns": 0 if hst is None else int(hst.hub_rows.numel()),
                       "virtual_rows": 0 if hs is None else hs.n_virtual, "virtual_columns": 0 if hst is None else hst.n_virtual},
            "variants": res, "speedup_from_hub_split": res["one_warp_per_row"]["ms_per_step"] / res["hub_split"]["ms_per_step"]}


# ============================================================================= GAT leg, node-partitioned (N > 1)
def gat_partitioned(args, rank, world, dev, nodes_per_gpu=NODES_PER_GPU, edges_per_gpu=EDGES_PER_GPU, label="C5-style weak scaling"):
    """Node-partitioned Product2Vec step: `nodes_per_gpu` products / ~`edges_per_gpu` co-view edges per GPU, columns uniform over
    the global node range, so (N-1)/N of every rank's edges point at halo rows.  Runs the multi-GPU parity check first."""
    dist = _dist()
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib
    from pcompanion_b200.distributed import (HaloPlan, allreduce_gradients, forward_graph_partitioned, halo_gather,
                                              partition_edges)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _partition_check import check_partitioned
    sampler = ClockSampler(dev.index)                   # started long before the timed region (see gat_single)
    parity = check_partitioned(rank, world, dev)        # also warms NCCL (communicator, all-to-all, symmetric memory)
    if not parity["ok"]:
        if rank == 0:
            print(json.dumps({"metric": "gat_edges_per_sec_fwd_bwd", "error": "multi-GPU parity check failed", "parity": parity}))
        dist.barrier()
        dist.destroy_process_group()
        sys.exit(3)
    n_loc, e_loc = nodes_per_gpu, edges_per_gpu
    n_total = n_loc * world
    bounds = [i * n_loc for i in range(world + 1)]
    g = torch.Generator(device=dev).manual_seed(SEED + 100 + rank)
    # every rank draws its share of the GLOBAL edge list; the owners of the rows get them through the distributed
    # CSR build (one all-to-all of keys, then local sort / unique) - timed separately, outside the step
    rows = torch.randint(0, n_total, (e_loc,), generator=g, device=dev, dtype=torch.int32)
    cols = torch.randint(0, n_total, (e_loc,), generator=g, device=dev, dtype=torch.int32)
    partition_edges(rows[:4096], cols[:4096], bounds, rank)             # untimed warm-up of the exchange
    torch.cuda.synchronize(); dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    rowptr, col_global = partition_edges(rows, cols, bounds, rank)
    ev1.record()
    torch.cuda.synchronize(); dist.barrier()
    build_ms = max_over_ranks([ev0.elapsed_time(ev1)], dev, world)[0]
    del rows, cols
    plan = HaloPlan(rowptr, col_global, bounds, rank)
    plan.graph.transposed()
    dense_ok = plan.enable_dense_halo()
    peer_ok = (not dense_ok) and plan.enable_peer_memory()
    if dense_ok:
        transport = (f"dense (halo = {plan.halo_fraction():.0%} of the remote rows): h blocks (512 B/row) on the copy engines, one peer "
                     "per round, K|V projected at the receiver while the next round is in flight; dK|dV blocks returned on the "
                     "copy engines while the next owner's column range is computed")
    elif peer_ok:
        transport = "pc_halo_push: gather + NVLink stores into the peers' symmetric-memory tables, one launch per direction"
    else:
        transport = "NCCL all_to_all_single (" + getattr(plan, "peer_error", "peer memory disabled") + ")"
    e_local = col_global.numel()
    x = torch.randn(n_loc, 128, generator=g, device=dev)
    cfg = make_cfg(dev)
    torch.manual_seed(SEED)                      # identical replicated weights on every rank
    model = pc.Product2Vec(cfg).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=cfg.LEARNING_RATE, fused=True)   # same Adam, one kernel for the 13 tensors
    # triplets: anchors are local, positives / negatives are any product of the global graph; their rows come from
    # the owners through a row-fetch plan (built once: the index batch is fixed, as in the 1-GPU leg)
    trip_global = torch.cat([torch.randint(0, n_loc, (TRIPLETS, 1), generator=g, device=dev) + bounds[rank],
                             torch.randint(0, n_total, (TRIPLETS, 1 + KNEG), generator=g, device=dev)], dim=1)
    fetch = HaloPlan(None, trip_global.reshape(-1), bounds, rank)
    fetch.enable_peer_memory(width=128)
    trip = fetch.col_ext.view_as(trip_global).contiguous()
    x_host, trip_host = x.cpu().pin_memory(), trip.cpu().pin_memory()
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def step(xd, tr):
        emb = halo_gather(forward_graph_partitioned(model, xd, plan), fetch)
        loss = model.triplet_loss_indexed(emb, tr[:, 0], tr[:, 1], tr[:, 2:])
        opt.zero_grad(set_to_none=True)
        loss.backward()
        allreduce_gradients(model)
        opt.step()
        return loss

    # end-to-end leg: the next step's inputs are copied from pinned host memory on a side stream while this step
    # computes (double-buffered staging, as in the 1-GPU leg)
    copy_stream = torch.cuda.Stream()
    stage = [(torch.empty_like(x), torch.empty_like(trip), torch.cuda.Event()) for _ in range(2)]
    e2e_state = {"i": 0}

    def prefetch(slot):
        xs, ts, ev = stage[slot]
        with torch.cuda.stream(copy_stream):
            xs.copy_(x_host, non_blocking=True)
            ts.copy_(trip_host, non_blocking=True)
            ev.record(copy_stream)

    def step_e2e():
        i = e2e_state["i"]
        if i == 0:
            prefetch(0)
        xs, ts, ev = stage[i % 2]
        torch.cuda.current_stream().wait_event(ev)
        copy_stream.wait_stream(torch.cuda.current_stream())       # the other slot was last read by the previous step
        prefetch((i + 1) % 2)
        e2e_state["i"] = i + 1
        loss_host.copy_(step(xs, ts).detach(), non_blocking=True)

    warm_up(lambda: step(x, trip), args.warmup, 0.5, dev, world)
    sampler.mark()
    launches0 = _lib.LAUNCHES
    ms, loss = timed_steps(lambda: step(x, trip), args.steps, dev, world)
    launches = _lib.LAUNCHES - launches0
    clocks = sampler.stop()
    # where the step goes: CUDA events around every C-ABI call of two more steps (the difference to ms_per_step is
    # exchange time that compute did not hide, plus the optimiser and index plumbing)
    _lib.PROFILE = []
    for _ in range(2):
        step(x, trip)
    torch.cuda.synchronize()
    prof, _lib.PROFILE = _lib.PROFILE, None
    per = {}
    for name, s0, s1 in prof:
        per[name] = per.get(name, 0.0) + s0.elapsed_time(s1) / 2
    abi_ms = {k: round(v, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}
    # timeline of the second profiled step on rank 0: start offset and duration of every native call / copy-engine copy /
    # cross-rank wait, in issue order (calls on the side stream overlap the ones on the main stream)
    last = prof[len(prof) // 2:]
    timeline = [[name, round(last[0][1].elapsed_time(s0), 3), round(s0.elapsed_time(s1), 3)] for name, s0, s1 in last]
    for _ in range(2):
        step_e2e()
    e2e_ms, _ = timed_steps(step_e2e, args.steps, dev, world)
    tot = torch.tensor([e_local, plan.n_halo, fetch.n_halo], dtype=torch.float64, device=dev)
    dist.all_reduce(tot)
    e_total, halo_total, fetch_total = tot.tolist()
    if rank != 0:
        return None
    peak, peak_src = measured_peaks()
    algo = (3152 * e_local + 3676 * n_loc)
    halo_bytes = int(halo_total / world) * 1024
    if dense_ok:
        halo_bytes = {"forward_h_blocks": (n_total - n_loc) * 512, "backward_dkv_blocks": (n_total - n_loc) * 1024}
    push_ms = per.get("pc_halo_push")
    return {
        "metric": "gat_edges_per_sec_fwd_bwd", "value": e_total / (ms * 1e-3), "unit": "edges/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{label}: node-partitioned synthetic BPG, {n_loc} products / ~{e_loc} co-view edges per GPU x {world} GPUs, "
                               "columns uniform over the global range, Product2Vec GAT fwd+bwd with a halo exchange of K|V rows "
                               "(fwd) and dK|dV partials (bwd) over NVLink (transport: see halo_transport), triplet positives / "
                               "negatives fetched from their owners, gradient all-reduce, Adam",
                   "nodes_total": n_total, "edges_total": int(e_total), "halo_rows_per_gpu": int(halo_total / world),
                   "halo_bytes_per_gpu_per_direction": halo_bytes,
                   "triplet_rows_fetched_per_gpu": int(fetch_total / world), "halo_transport": transport,
                   "halo_push_gbs": round(halo_bytes / (push_ms * 1e-3) / 1e9, 1) if push_ms and peer_ok else None,
                   "csr_build": {"what": "distributed: all-to-all of edge keys by row owner + local radix sort / unique / CSR "
                                         "(device time, max over ranks, exchange warmed up)",
                                 "ms": build_ms, "edges_per_s": e_total / (build_ms * 1e-3)},
                   "batchnorm": "synchronised (all-reduce of the [2,256] column sums)",
                   "l2": "working set exceeds the 126 MB L2; no flush needed"},
        "parity": parity,
        "roofline": {"bound": "hbm", "achieved": algo / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": algo / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                     "note": "whole step per GPU against the sparse-kernel algorithmic bytes (3152 B/edge + 3676 B/node); "
                             "the halo exchange moves halo_bytes over NVLink each way on top"},
        "abi_ms_per_step": abi_ms, "abi_total_ms_per_step": round(sum(abi_ms.values()), 3),
        "timeline_rank0": {"columns": ["call", "start_ms", "duration_ms"], "rows": timeline},
        "clocks": clocks,
        "e2e": {"value": e_total / (e2e_ms * 1e-3), "unit": "edges/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": (x_host.numel() * 4 + trip_host.numel() * 8) * world, "d2h_bytes_per_step": 4 * world},
        "gpu_launches": launches, "loss": float(loss.item()),
    }


# ============================================================================= C3: P-Companion joint step
def pcompanion_leg(args, rank, world, dev, batch, cpu=False):
    """C3: P-Companion joint training step (type transition + item prediction, 0.8 item + 0.2 type hinge, Adam) on a
    frozen 1 M-product table, NUM_TYPES = 34,800 (reference default); data parallel over samples (replicated model,
    gradient all-reduce)."""
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib
    from pcompanion_b200.distributed import allreduce_gradients
    p, b = 1_000_000, batch
    cfg = make_cfg(dev)
    t = cfg.NUM_TYPES
    g = torch.Generator(device=dev).manual_seed(SEED + rank)
    table = torch.randn(p, 128, generator=g, device=dev)
    torch.manual_seed(SEED)
    model = pc.PCompanion(cfg, table).to(dev).train()
    opt = torch.optim.Adam([q for q in model.parameters() if q.requires_grad], lr=cfg.LEARNING_RATE)
    hg = torch.Generator().manual_seed(SEED + 7 + rank)
    host = {"query_ids": torch.randint(0, p, (b,), generator=hg), "query_types": torch.randint(0, t, (b,), generator=hg),
            "positive_types": torch.randint(0, t, (b, 1), generator=hg), "negative_types": torch.randint(0, t, (b, 1), generator=hg),
            "positive_items": torch.randn(b, 128, generator=hg), "negative_items": torch.randn(b, 128, generator=hg)}
    host = {k: v.pin_memory() for k, v in host.items()}
    bt_dev = {k: v.to(dev) for k, v in host.items()}
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def step(bt):
        out = model(bt)
        loss = model.compute_loss(bt, out)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if world > 1:
            allreduce_gradients(model)
        opt.step()
        return loss

    def step_e2e():
        loss_host.copy_(step({k: v.to(dev, non_blocking=True) for k, v in host.items()}).detach(), non_blocking=True)

    # the per-step working set (two [T,64] type tables + Adam state + [B,T] scores) fits the L2 at small batches
    small = b * t * 4 < (512 << 20)
    flush = L2Flush(dev) if small else None
    sampler = ClockSampler(dev.index)
    warm_up(lambda: step(bt_dev), args.warmup, 1.0, dev, world)
    sampler.mark()
    l0 = _lib.LAUNCHES
    ms, _ = timed_steps(lambda: step(bt_dev), args.steps, dev, world, flush)
    launches = _lib.LAUNCHES - l0
    clocks = sampler.stop()
    step_e2e()
    e2e_ms, _ = timed_steps(step_e2e, args.steps, dev, world, flush)
    eager = None
    if small and world == 1:
        # launch-bound regime: the whole step (forward + loss + backward + Adam) captured once in a CUDA graph and replayed
        eager = {"ms_per_step": ms, "samples_per_s": b / (ms * 1e-3), "e2e_ms_per_step": e2e_ms, "c_abi_calls_per_step": launches // args.steps}
        gopt = torch.optim.Adam([q for q in model.parameters() if q.requires_grad], lr=cfg.LEARNING_RATE, capturable=True)
        l1 = _lib.LAUNCHES
        gstep = pc.GraphedTrainStep(model, gopt, bt_dev)                 # 3 warm-up steps + 1 captured step
        launches = (_lib.LAUNCHES - l1) // 4 * args.steps                # C-ABI calls inside one replay x timed replays
        for _ in range(args.warmup):
            gstep(bt_dev)
        ms, _ = timed_steps(lambda: gstep(bt_dev), args.steps, dev, world, flush)

        def gstep_e2e():
            loss_host.copy_(gstep(host).detach(), non_blocking=True)
        gstep_e2e()
        e2e_ms, _ = timed_steps(gstep_e2e, args.steps, dev, world, flush)
    if rank != 0:
        return None
    peak, peak_src = measured_peaks()
    # bytes that must move per step: the [B, T] similarity matrix is written once (it is part of forward()'s contract; the
    # type loss reads two entries per row and its gradient goes to the factors), the two [T, 64] type tables are read,
    # their dense gradients written and read, and Adam reads / writes p, m, v of both
    algo = b * t * 4 + 2 * t * 64 * 4 * (1 + 2 + 6) + b * (128 * 4 * 3 + 3 * 128 * 4 * 2)
    line = {"metric": "pcompanion_samples_per_sec_fwd_loss_bwd", "value": b * world / (ms * 1e-3), "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C3: P-Companion joint step, 1M-product frozen table, {t} types, batch {b} per GPU, "
                                   "K_t=3, alpha 0.8, Adam" + (" (whole step replayed as one CUDA graph; `eager` = the same step launched "
                                   "call by call)" if eager is not None else ""), "batch": b, "types": t,
                       "l2": ("working set fits the L2: a 256 MB buffer is overwritten between timed steps (each step timed on "
                              "its own)") if small else "similarity matrix [B,T] fp32 = %.1f GB per step; no flush needed" % (b * t * 4 / 1e9)},
            "roofline": {"bound": "hbm", "achieved": algo / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": algo,
                         "note": "whole step against the [B,T] similarity write, the type-table read / gradient / Adam traffic "
                                 "and the per-sample rows; small batches are launch-latency bound, not bandwidth bound"},
            "cpu_baseline": cpu_baseline_pcompanion(cfg, b) if cpu else None, "clocks": clocks,
            "cuda_graph": eager is not None, "eager": eager,
            "e2e": {"value": b * world / (e2e_ms * 1e-3), "unit": "samples/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in host.values()) * world,
                    "d2h_bytes_per_step": 4 * world},
            "gpu_launches": launches}
    return line


def cpu_baseline_pcompanion(cfg, batch, seconds=6.0):
    from oracle import torch_port
    torch.set_num_threads(os.cpu_count() or 1)
    p = 1_000_000 if batch <= 4096 else 100_000
    g = torch.Generator().manual_seed(SEED)
    ccfg = torch_port.default_config(NUM_TYPES=cfg.NUM_TYPES)
    model = torch_port.PortPCompanion(ccfg, torch.randn(p, 128, generator=g)).train()
    opt = torch.optim.Adam([q for q in model.parameters() if q.requires_grad], lr=1e-3)
    b = min(batch, 4096)
    t = cfg.NUM_TYPES
    qi, qt = torch.randint(0, p, (b,), generator=g), torch.randint(0, t, (b,), generator=g)
    pt, nt = torch.randint(0, t, (b,), generator=g), torch.randint(0, t, (b,), generator=g)
    pi, ni = torch.randn(b, 128, generator=g), torch.randn(b, 128, generator=g)

    def one():
        out = model(qi, qt)
        loss = model.loss(out, pt, nt, pi, ni)
        opt.zero_grad(); loss.backward(); opt.step()
    one()
    t0, n = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds and n < 200:
        one(); n += 1
    dt = time.perf_counter() - t0
    return {"value": b * n / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": "port",
            "sample": f"{n} steps of batch {b} through the torch-CPU port of the reference PCompanion (forward + compute_loss + "
                      f"backward + Adam, {t} types, {p}-product table); {dt:.1f} s"}


# ============================================================================= C4: complementary retrieval
def retrieval_leg(args, rank, world, dev, dense=False, cpu=False):
    """C4: masked top-10 over a 10 M-product catalog (sharded over the ranks), 1 K types, Q queries x 3 type rows."""
    dist = _dist()
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib
    p_total, n_types, q_n, k = 10_000_000, 1000, args.queries, 10
    per = p_total // world
    base = rank * per
    g = torch.Generator(device=dev).manual_seed(SEED + rank)
    catalog = torch.randn(per, 128, generator=g, device=dev)
    type_id = torch.randint(0, n_types, (per,), generator=g, device=dev, dtype=torch.int32)
    cat = pc.ShardedCatalog(catalog, type_id, base, n_types)
    gq = torch.Generator(device=dev).manual_seed(SEED)
    queries = torch.randn(q_n * 3, 128, generator=gq, device=dev)
    row_type = torch.randint(0, n_types, (q_n * 3,), generator=gq, device=dev, dtype=torch.int32)
    q_host, t_host = queries.cpu().pin_memory(), row_type.cpu().pin_memory()
    i_host = torch.empty(q_n * 3, k, dtype=torch.int64).pin_memory()
    s_host = torch.empty(q_n * 3, k, dtype=torch.float64).pin_memory()
    if dense:   # north_star wording: dense tensor-core scoring GEMM + mask + top-K (exact after fp64 re-scoring)
        assert world == 1, "retrieval_dense is a single-GPU measurement"
        cat.local.topk_dense(queries[:128], k, row_type[:128])      # max-norm of the catalog is computed once, outside the timing
        topk = lambda qq, kk, tt: cat.local.topk_dense(qq, kk, tt)
    else:
        topk = cat.topk

    def step():
        return topk(queries, k, row_type)

    def step_e2e():
        qd = torch.empty_like(queries); qd.copy_(q_host, non_blocking=True)
        td = torch.empty_like(row_type); td.copy_(t_host, non_blocking=True)
        s, i = topk(qd, k, td)
        i_host.copy_(i, non_blocking=True)
        s_host.copy_(s, non_blocking=True)

    # a step is only a few ms: warm up for at least W steps AND ~0.5 s, so that the timed region does not start on a GPU
    # that is still ramping its clocks after the host-side setup
    sampler = ClockSampler(dev.index)
    warm_up(step, args.warmup, 1.5, dev, world)
    sampler.mark()
    launches0 = _lib.LAUNCHES
    ms, (scores, idx) = timed_steps(step, args.steps, dev, world)
    launches = _lib.LAUNCHES - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args, "retrieval_dense" if dense else "retrieval", {"scores": scores, "indices": idx})
    step_e2e()
    e2e_ms, _ = timed_steps(step_e2e, args.steps, dev, world)
    # per-kernel device time from a separate profiled pass (CUDA events around every C-ABI call)
    _lib.PROFILE = []
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    prof, _lib.PROFILE = _lib.PROFILE, None
    per_call = {}
    for name, s0, s1 in prof:
        per_call[name] = per_call.get(name, 0.0) + s0.elapsed_time(s1) / args.steps
    # algorithmic traffic of the segmented kernel on THIS rank's shard: rows that rank the same type are grouped eight at
    # a time and a group streams its type's run of catalog rows once
    counts = torch.bincount(row_type.long().cpu(), minlength=n_types)
    seg_len = (cat.local.offsets[1:] - cat.local.offsets[:-1]).cpu()
    groups = (counts + 7) // 8
    stream_bytes = int((groups * seg_len).sum().item()) * 512 + q_n * 3 * 512 + q_n * 3 * k * 16
    pair_flop = int((counts * seg_len).sum().item()) * 256                        # fp64 FMAs x 2 on this shard
    if rank != 0:
        return None
    peak, peak_src = measured_peaks()
    if dense:
        kms = per_call.get("pc_score_topk_dense", ms)
        tpeak, tsrc = measured_tensor_peak()
        tflops = q_n * 3 * per * 256 / (kms * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": "pc_score_topk_dense (score_topk_tf32_kernel + rescore_topk_kernel)",
                    "achieved": tflops, "peak": tpeak, "unit": "TFLOP/s", "frac": tflops / tpeak, "traffic": None,
                    "kernel_ms": kms, "peak_source": tsrc,
                    "algorithmic_flop_per_launch": q_n * 3 * per * 256,
                    "note": "256 flop per (score row, product) over the WHOLE catalog (SURVEY 8d); 99.9 % of the pairs are then "
                            "masked out by the per-type filter, which is why the type-segmented kernel is the default"}
    else:
        kms = per_call.get("pc_topk_by_type", ms)
        gbs = stream_bytes / (kms * 1e-3) / 1e9
        f64 = pair_flop / (kms * 1e-3) / 1e12
        roofline = {"bound": "hbm", "kernel": "pc_topk_by_type (topk_planned_kernel)", "achieved": gbs, "peak": peak, "unit": "GB/s",
                    "frac": gbs / peak, "traffic": None, "kernel_ms": kms, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": stream_bytes,
                    "fp64": {"achieved_tflops": f64, "peak_tflops_nominal": FP64_TFLOPS_NOMINAL, "frac": f64 / FP64_TFLOPS_NOMINAL,
                             "note": "exact scores: one fp64 FMA per (row, product of its type, dim)"},
                    "note": "bytes = catalog rows streamed once per group of <= 8 same-type score rows on rank 0's shard + queries "
                            "+ results; neither HBM nor the fp64 pipe is saturated: the kernel is bound by the fp32->fp64 "
                            "conversions and the sequential fp64 chains that make the scores order-independent"}
    line = {"metric": "topk_queries_per_sec", "value": q_n / (ms * 1e-3), "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C4: top-10 over 10M-product catalog, 1K types, {q_n} queries x 3 type rows, "
                                   f"catalog sharded over {world} GPU(s), " + ("dense tcgen05 TF32 scoring GEMM + per-type mask + "
                                   "fused candidate top-K + exact fp64 re-scoring" if dense else "type-segmented exact fp64 scoring "
                                   "(device-side grouping), per-shard lists all-gathered and merged"),
                       "l2": "the catalog (5.12 GB per 10M rows) exceeds the 126 MB L2; no flush needed"},
            "roofline": roofline, "abi_ms_per_step": {n_: round(v, 4) for n_, v in sorted(per_call.items(), key=lambda kv: -kv[1])},
            "cpu_baseline": cpu_baseline_retrieval() if cpu else None,
            "clocks": clocks,
            "e2e": {"value": q_n / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": q_host.numel() * 4 + t_host.numel() * 4, "d2h_bytes_per_step": q_n * 3 * k * 16},
            "gpu_launches": launches}
    return line


def cpu_baseline_retrieval(steps=5, warmup=1):
    """inference.py:93-113 semantics on the host cores: dense fp32 matmul + type mask + topk(10) on a 1 M-product sample of
    the catalog, scaled linearly to 10 M (BASELINE.md section 3)."""
    from oracle import torch_port
    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(SEED)
    p_sample, n_types, k, rows = 1_000_000, 1000, 10, 96
    catalog = torch.randn(p_sample, 128, generator=g)
    type_id = torch.randint(0, n_types, (p_sample,), generator=g)
    q = torch.randn(rows, 128, generator=g)
    rt = torch.randint(0, n_types, (rows,), generator=g)
    for _ in range(warmup):
        torch_port.port_dense_topk(q, catalog, rt, type_id, k)
    t0 = time.perf_counter()
    for _ in range(steps):
        torch_port.port_dense_topk(q, catalog, rt, type_id, k)
    dt = (time.perf_counter() - t0) / steps
    qps = rows / 3 / dt / 10.0
    return {"value": qps, "unit": "queries/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": "port",
            "ms_per_step": dt * 1e3,
            "sample": f"{steps} x (96 score rows x 1M-product sample): dense fp32 matmul + type mask + topk(10), scaled x1/10 to the 10M catalog"}


# ============================================================================= C1: the reference's own training flow
def c1_leg(args, dev, cpu=False):
    """configs[0]: the `python train.py` flow on the default synthetic BPG (1000 products, 20 types, B = 256) through the
    drop-in classes: SimilarityDataset + collate_fn + Product2Vec.train_model-style epochs (forward(features, neighbors),
    triplet loss, Adam), then generate_all_embeddings.  Reported as Product2Vec epoch time and padded edges/s."""
    import pcompanion_b200 as pc
    from pcompanion_b200 import _lib
    from torch.utils.data import DataLoader
    cfg = make_cfg(dev)
    bpg = c1_bpg(dev)
    ds = pc.SimilarityDataset(bpg, cfg)
    loader = DataLoader(ds, batch_size=256, shuffle=True, collate_fn=pc.collate_fn, num_workers=0)
    torch.manual_seed(SEED)
    model = pc.Product2Vec(cfg).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=cfg.LEARNING_RATE, fused=True)   # same Adam, one kernel for the 13 tensors

    def epoch():
        model.train()
        edges = 0
        t_data = t_compute = 0.0
        t0 = time.perf_counter()
        for batch in loader:
            t1 = time.perf_counter(); t_data += t1 - t0
            batch = {k: v.to(dev) if isinstance(v, torch.Tensor) else v for k, v in batch.items()}
            nb = batch.get("anchor_neighbors")
            a = model(batch["anchor"], nb)
            p_ = model(batch["positive"])
            n_ = model(batch["negative"])
            loss = model.triplet_loss(a, p_, n_)
            opt.zero_grad(); loss.backward(); opt.step()
            if nb is not None:
                edges += nb.shape[0] * nb.shape[1]
            torch.cuda.synchronize()
            t0 = time.perf_counter(); t_compute += t0 - t1
        return edges, t_data, t_compute, float(loss.item())

    epoch()
    l0 = _lib.LAUNCHES
    t0 = time.perf_counter()
    edges, t_data, t_compute, loss = epoch()
    dt = time.perf_counter() - t0
    launches = _lib.LAUNCHES - l0
    t0 = time.perf_counter()
    emb = model.generate_all_embeddings(bpg)
    gen_s = time.perf_counter() - t0
    line = {"metric": "c1_product2vec_epoch_padded_edges_per_sec", "value": edges / dt, "unit": "edges/s", "n_gpus": 1,
            "epoch_s": dt, "data_s": t_data, "compute_s": t_compute, "samples": len(ds), "padded_edges": edges, "loss": loss,
            "generate_all_embeddings_s": gen_s, "embeddings": len(emb), "gpu_launches": launches,
            "config": {"workload": "C1: train.py flow on the default synthetic BPG (1000 products, 20 types), B=256, drop-in "
                                   "SimilarityDataset / collate_fn / Product2Vec.forward(features, neighbors) / Adam; wall clock "
                                   "including the host-side data path, as the reference's own epoch"},
            "cpu_baseline": None}
    if cpu:
        line["cpu_baseline"] = cpu_baseline_c1(bpg, ds, cfg)
    return line


def c1_bpg(dev):
    """The reference's default synthetic BPG: edge sets produced by the real generator (src/data/synthetic_data.py:78-153,
    written by tests/golden/make_golden.py into tests/golden/bpg_c1.npz), rebuilt through the reference's string API."""
    import numpy as np
    import pcompanion_b200 as pc
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "bpg_c1.npz"), allow_pickle=False))
    n = len(g["type_id"])
    ids = [f"P{str(i).zfill(6)}" for i in range(n)]
    gen = torch.Generator().manual_seed(0)
    bpg = pc.BehaviorProductGraph(dev)
    for i, pid in enumerate(ids):
        bpg.add_node(pid, {"type": str(g["type_names"][g["type_id"][i]]), "features": torch.randn(128, generator=gen)})
    for t in ("co_view", "purchase_after_view", "co_purchase"):
        for s_, d_ in g["edges/" + t]:
            bpg.add_edge(ids[s_], ids[d_], t)
    bpg.finalize()
    bpg.derive_pair_sets()
    return bpg


def cpu_baseline_c1(bpg, ds, cfg):
    """The same epoch through the torch-CPU port of the reference modules (same batches: our datasets are drop-ins)."""
    import pcompanion_b200 as pc
    from oracle import torch_port
    from torch.utils.data import DataLoader
    torch.set_num_threads(os.cpu_count() or 1)
    loader = DataLoader(ds, batch_size=256, shuffle=True, collate_fn=pc.collate_fn, num_workers=0)
    torch.manual_seed(SEED)
    model = torch_port.PortProduct2Vec(torch_port.default_config(DROPOUT=cfg.DROPOUT)).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    edges = 0
    t0 = time.perf_counter()
    for batch in loader:
        loss = torch_port.port_triplet_loss(model, batch, cfg.MARGIN)
        opt.zero_grad(); loss.backward(); opt.step()
        nb = batch.get("anchor_neighbors")
        if nb is not None:
            edges += nb.shape[0] * nb.shape[1]
    dt = time.perf_counter() - t0
    return {"value": edges / dt, "unit": "edges/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": "port",
            "epoch_s": dt, "sample": "one epoch of the same C1 batches through the torch-CPU port of the reference Product2Vec"}


# ============================================================================= CSR build / CPU baselines of the GAT leg
def time_csr_build(graph, peak, reps: int = 3):
    """Part (1) of the path on its own: shuffled (src, dst) edge list -> pack, radix sort, unique, CSR, then the
    transposed lists (CSC) - device time from CUDA events.  SURVEY 8(d): ~100 algorithmic bytes per edge for the CSR
    (4 radix passes x 8 B read + write, + unique + scan); the CSC build costs about the same again."""
    from pcompanion_b200 import ops
    e = graph.num_edges
    rows = torch.repeat_interleave(torch.arange(graph.n_rows, device=graph.col.device, dtype=torch.int32),
                                   (graph.rowptr[1:] - graph.rowptr[:-1]))
    perm = torch.randperm(e, device=rows.device)
    src, dst = rows[perm].contiguous(), graph.col[perm].contiguous()
    del rows, perm
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    csr_ms, csc_ms = [], []
    for _ in range(reps + 1):
        ev[0].record()
        g2, _ = ops.build_csr(src, dst, graph.n_rows, graph.n_cols)
        ev[1].record()
        g2.transposed()
        ev[2].record()
        torch.cuda.synchronize()
        csr_ms.append(ev[0].elapsed_time(ev[1])); csc_ms.append(ev[1].elapsed_time(ev[2]))
    ok = bool(torch.equal(g2.col, graph.col) and torch.equal(g2.rowptr, graph.rowptr))
    a, b = min(csr_ms[1:]), min(csc_ms[1:])
    return {"edges": e, "csr_ms": round(a, 3), "csc_ms": round(b, 3), "edges_per_s": e / ((a + b) * 1e-3),
            "csr_edges_per_s": e / (a * 1e-3), "csr_algo_gbs": round(100 * e / (a * 1e-3) / 1e9, 1),
            "csr_frac_of_hbm": round(100 * e / (a * 1e-3) / 1e9 / peak, 4), "rebuilt_equals_original": ok,
            "note": "includes one host sync for the data-dependent unique count"}


def padded_batches(graph_rowptr, graph_col, feats, n_batches, batch, gen):
    """Index-based collate (no Python sets): dense zero-padded neighbour tensors exactly as
    data_loader.py:171-206 would build them for `batch` destinations."""
    n = graph_rowptr.numel() - 1
    for _ in range(n_batches):
        rows = torch.randint(0, n, (batch,), generator=gen)
        lo, hi = graph_rowptr[rows], graph_rowptr[rows + 1]
        deg = hi - lo
        nmax = int(deg.max().item())
        ar = torch.arange(max(nmax, 1)).unsqueeze(0)
        mask = ar < deg.unsqueeze(1)
        idx = (lo.unsqueeze(1) + ar).clamp_(max=graph_col.numel() - 1)
        nbr_ids = graph_col[idx].long()
        nbrs = feats[nbr_ids] * mask.unsqueeze(-1)
        yield {"anchor": feats[rows], "positive": feats[torch.randint(0, n, (batch,), generator=gen)],
               "negative": feats[torch.randint(0, n, (batch * KNEG,), generator=gen)].reshape(batch, KNEG, -1),
               "anchor_neighbors": nbrs}, int(deg.sum().item()), batch * max(nmax, 1)


def cpu_gat_sample(feats, rowptr, col, cfg, seconds, batch=4096, max_batches=64):
    from oracle import torch_port
    torch.manual_seed(SEED)
    model = torch_port.PortProduct2Vec(torch_port.default_config(DROPOUT=cfg.DROPOUT)).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    gen = torch.Generator().manual_seed(SEED)
    real = padded = nb = 0
    # one untimed batch to warm the allocator / thread pool
    for b, _, _ in padded_batches(rowptr, col, feats, 1, batch, gen):
        torch_port.port_triplet_loss(model, b, cfg.MARGIN).backward()
    t0 = time.perf_counter()
    for b, r, p in padded_batches(rowptr, col, feats, max_batches, batch, gen):
        loss = torch_port.port_triplet_loss(model, b, cfg.MARGIN)
        opt.zero_grad()
        loss.backward()
        opt.step()
        real += r; padded += p; nb += 1
        if time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    return real, padded, nb, dt


def cpu_baseline_gat(bpg, graph, cfg, seconds):
    torch.set_num_threads(os.cpu_count() or 1)
    feats = bpg.features.cpu()
    rowptr, col = graph.rowptr.cpu(), graph.col.cpu()
    real, padded, nb, dt = cpu_gat_sample(feats, rowptr, col, cfg, seconds)
    return {"value": padded / dt, "unit": "edges/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(),
            "kind": "port",
            "sample": f"{nb} batches x 4096 destinations of the same C2 graph through the torch-CPU port of the reference "
                      f"Product2Vec (zero-padded neighbour lists, FFN per edge row, fwd+bwd+Adam); value counts padded "
                      f"edges ({padded}), real edges {real} -> {real / dt:.0f} real edges/s; {dt:.1f} s"}


# ============================================================================= our arm
def run_ours(args):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        _dist().init_process_group("nccl", device_id=dev)
    import pcompanion_b200  # noqa: F401  (fails loudly without the CUDA library)
    cpu = (world == 1) and not args.skip_cpu
    wl = args.workload

    def free():
        import gc
        gc.collect()
        torch.cuda.empty_cache()

    line = None
    if wl in ("all", "gat"):
        line = gat_single(args, dev) if world == 1 else gat_partitioned(args, rank, world, dev)
        free()
    if wl == "c5":     # BASELINE configs[4] as specified: the fixed 10 M-product / 200 M-edge graph over the ranks (strong scaling)
        assert world > 1, "c5 is a multi-GPU configuration"
        line = gat_partitioned(args, rank, world, dev, 10_000_000 // world, 200_000_000 // world,
                               "C5 (fixed 10M products / 200M edges, strong scaling)")
        if line is not None:
            line["scaling"] = "strong"
    if wl in ("all", "retrieval"):
        r = retrieval_leg(args, rank, world, dev, dense=False, cpu=cpu)
        free()
        if wl == "retrieval":
            line = r
        elif line is not None:
            line["retrieval"] = r
            line["topk_queries_per_sec"] = r["value"]
    if wl in ("all", "retrieval_dense") and world == 1:
        r = retrieval_leg(args, rank, world, dev, dense=True, cpu=False)
        free()
        if wl == "retrieval_dense":
            line = r
        elif line is not None:
            line["retrieval_dense"] = r
    if wl in ("all", "pcompanion"):
        batches = [256, 65536] if wl == "all" else [args.batch]
        recs = {}
        for b in batches:
            recs[f"b{b}"] = pcompanion_leg(args, rank, world, dev, b, cpu=cpu and b <= 4096)
            free()
        if wl == "pcompanion":
            line = recs[f"b{args.batch}"]
        elif line is not None:
            line["pcompanion"] = recs
    if wl in ("all", "gat_skewed") and world == 1:
        r = gat_skewed_leg(args, dev)
        free()
        if wl == "gat_skewed":
            line = r
        elif line is not None:
            line["gat_skewed"] = r
    if wl in ("all", "c1") and world == 1:
        r = c1_leg(args, dev, cpu=cpu)
        free()
        if wl == "c1":
            line = r
        elif line is not None:
            line["c1"] = r
    if rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        _dist().barrier()
        _dist().destroy_process_group()


# ============================================================================= reference arm
def run_reference(args):
    """The reference's own CPU path (torch-CPU port in oracle/torch_port.py; the reference is pure
    Python/PyTorch and cannot travel to the GPU box) on the host cores, same workload.  Under torchrun the launcher
    exports OMP_NUM_THREADS=1: the thread count is reset to all host cores here."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = make_cfg(torch.device("cpu"))
    if args.workload in ("retrieval", "retrieval_dense"):
        cb = cpu_baseline_retrieval(steps=args.steps, warmup=args.warmup)
        line = {"impl": "reference", "metric": "topk_queries_per_sec", "value": cb["value"], "unit": "queries/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "C4 sample: torch matmul + type mask + topk(10), 96 rows x 1M-product sample, scaled x1/10 to 10M"},
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    # GAT: destinations of a C2-like graph (uniform random neighbours, Poisson(20) degrees); the CPU sample only
    # needs the local structure of the graph, not the 20 M-edge CSR
    gen = torch.Generator().manual_seed(SEED)
    n = NODES_PER_GPU
    per_step_batches = 2
    feats = torch.randn(n, 128, generator=gen)
    from oracle import torch_port
    model = torch_port.PortProduct2Vec(torch_port.default_config(DROPOUT=cfg.DROPOUT)).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    # neighbour lists are drawn at the C2 degree (mean 20): repeat-sample columns per destination
    def batches(k):
        for _ in range(k):
            rows = torch.randint(0, n, (4096,), generator=gen)
            deg = torch.poisson(torch.full((4096,), EDGES_PER_GPU / NODES_PER_GPU), generator=gen).long().clamp_(min=0)
            nmax = int(deg.max().item())
            nbr = torch.randint(0, n, (4096, nmax), generator=gen)
            mask = torch.arange(nmax).unsqueeze(0) < deg.unsqueeze(1)
            yield {"anchor": feats[rows], "positive": feats[torch.randint(0, n, (4096,), generator=gen)],
                   "negative": feats[torch.randint(0, n, (4096 * KNEG,), generator=gen)].reshape(4096, KNEG, -1),
                   "anchor_neighbors": feats[nbr] * mask.unsqueeze(-1)}, int(deg.sum()), 4096 * nmax

    def one_step():
        real = padded = 0
        for bt, r, p in batches(per_step_batches):
            loss = torch_port.port_triplet_loss(model, bt, cfg.MARGIN)
            opt.zero_grad(); loss.backward(); opt.step()
            real += r; padded += p
        return real, padded
    for _ in range(args.warmup):
        one_step()
    t0 = time.perf_counter()
    real = padded = 0
    for _ in range(args.steps):
        r, p = one_step()
        real += r; padded += p
    dt = time.perf_counter() - t0
    val = padded / dt
    line = {"impl": "reference", "metric": "gat_edges_per_sec_fwd_bwd", "value": val, "unit": "edges/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C2 sample: reference Product2Vec (torch-CPU port) fwd+bwd+Adam on 2 x 4096-destination padded "
                                   "batches per step, neighbour lists at the C2 degree distribution (Poisson mean 20)"},
            "cpu_baseline": {"value": val, "unit": "edges/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(),
                             "kind": "port", "sample": f"{args.steps} steps x 2 batches x 4096 destinations; padded edges {padded}, "
                                                       f"real edges {real} ({real / dt:.0f} real edges/s)"},
            "e2e": {"value": val, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.workload == "all":      # second half of the metric on the host cores (bounded sample)
        cb = cpu_baseline_retrieval(steps=3, warmup=1)
        line["retrieval"] = {"metric": "topk_queries_per_sec", "value": cb["value"], "unit": "queries/s", "cpu_baseline": cb}
        line["topk_queries_per_sec"] = cb["value"]
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "gat", "gat_skewed", "retrieval", "retrieval_dense", "pcompanion", "c1", "c5"])
    ap.add_argument("--batch", type=int, default=4096, help="pcompanion: samples per GPU per step")
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--skip-cpu", action="store_true", help="skip the CPU-baseline legs (profiling runs)")
    ap.add_argument("--dense", action="store_true", help="(compat) with --workload retrieval: same as --workload retrieval_dense")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy: the C2 training "
                         "step (gat.*: loss, updated parameters and BatchNorm statistics, gradients, a fixed sample of the "
                         "embedding rows) and the top-K results (retrieval.*, retrieval_dense.*); one GPU only.  The "
                         "P-Companion, skewed-graph and C1 legs of --workload all are timed but not dumped")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dense and args.workload == "retrieval":
        args.workload = "retrieval_dense"
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", 1)) != 1
                              or args.workload not in ("all", "gat", "retrieval", "retrieval_dense")):
        ap.error("--dump-outputs needs --impl ours on one GPU and --workload all, gat, retrieval or retrieval_dense")
    if args.impl == "ours":
        args.warmup = max(args.warmup, 3)      # timing rule: at least 3 untimed warm-up steps (reported as run)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
