"""Tensor-level wrappers and autograd Functions over the C ABI (include/pcompanion_b200.h).

Everything here is thin: argument checks, output allocation (torch owns device memory), the
current CUDA stream, one or a few native calls.  No arithmetic is done in PyTorch on this
layer and nothing falls back to it.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import call, dev, stream

I32, I64, F32, F64 = torch.int32, torch.int64, torch.float32, torch.float64
EMB = 128  # embed dim the GAT kernels are instantiated for (reference config.py:8)


# --------------------------------------------------------------------------- edge keys / sets
def pack_keys(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """(src, dst) int32 -> int64 keys src<<32|dst (pc_edge_keys_pack; bpg.py:19-22)."""
    if src.shape != dst.shape or src.dim() != 1:
        raise ValueError("src and dst must be 1-D tensors of equal length")
    keys = torch.empty(src.numel(), dtype=I64, device=src.device)
    call("pc_edge_keys_pack", dev(src, I32, "src"), dev(dst, I32, "dst"), src.numel(), dev(keys, I64, "keys"), stream())
    return keys


def unpack_keys(keys: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    src = torch.empty(keys.numel(), dtype=I32, device=keys.device)
    dst = torch.empty_like(src)
    call("pc_edge_keys_unpack", dev(keys, I64, "keys"), keys.numel(), dev(src, I32, "src"), dev(dst, I32, "dst"), stream())
    return src, dst


def digit_mask_for(num_ids: int) -> int:
    """Bytes of a src<<32|dst key that can be non-zero when ids < num_ids."""
    nbytes = max(1, ((max(int(num_ids), 2) - 1).bit_length() + 7) // 8)
    low = (1 << nbytes) - 1
    return low | (low << 4)


def sort_keys_(keys: torch.Tensor, digit_mask: int = 0xFF) -> torch.Tensor:
    """In-place ascending LSD radix sort (pc_sort_keys)."""
    n = keys.numel()
    ws = _lib.workspace(_lib.LIB.pc_sort_keys_workspace_bytes(n), keys.device)
    call("pc_sort_keys", dev(keys, I64, "keys"), n, digit_mask, dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return keys


def _compacted(out: torch.Tensor, n_out: torch.Tensor) -> torch.Tensor:
    return out[: int(n_out.item())]  # one host sync: the output size is data dependent


def unique_sorted(keys: torch.Tensor) -> torch.Tensor:
    """Set semantics of edges[type].add (bpg.py:21) on a sorted key array."""
    n = keys.numel()
    out = torch.empty_like(keys)
    n_out = torch.zeros(1, dtype=I64, device=keys.device)
    ws = _lib.workspace(_lib.LIB.pc_compact_workspace_bytes(n), keys.device)
    call("pc_unique_sorted_keys", dev(keys, I64, "keys"), n, dev(out, I64, "out"), dev(n_out, I64, "n_out"),
         dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return _compacted(out, n_out)


def set_filter(a: torch.Tensor, b: torch.Tensor, keep_if_present: bool) -> torch.Tensor:
    """a n b (keep_if_present) or a - b on sorted-unique key arrays (pc_set_filter_sorted)."""
    out = torch.empty_like(a)
    n_out = torch.zeros(1, dtype=I64, device=a.device)
    ws = _lib.workspace(_lib.LIB.pc_compact_workspace_bytes(a.numel()), a.device)
    call("pc_set_filter_sorted", dev(a, I64, "a"), a.numel(), dev(b, I64, "b"), b.numel(), int(keep_if_present),
         dev(out, I64, "out"), dev(n_out, I64, "n_out"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return _compacted(out, n_out)


def set_intersection(a, b):
    return set_filter(a, b, True)


def set_difference(a, b):
    return set_filter(a, b, False)


def set_union(a: torch.Tensor, b: torch.Tensor, num_ids: int) -> torch.Tensor:
    keys = torch.cat([a, b])
    return unique_sorted(sort_keys_(keys, digit_mask_for(num_ids)))


# --------------------------------------------------------------------------- CSR
# Rows (or transposed columns) with more neighbours than HUB_THRESHOLD are split into virtual rows of HUB_SEGMENT neighbours
# (SURVEY H8, include/pcompanion_b200.h "hub nodes").  A CTA keeps its slot until its slowest warp is done, so even rows of
# a few hundred neighbours cost occupancy: on the power-law graph of bench.py --workload gat_skewed thresholds of 4096 / 1024
# left the attention kernels at 8 ms (3.4 ms on a uniform graph of the same size); virtual rows all have the same length,
# so their launch is perfectly balanced.
HUB_THRESHOLD = 256
HUB_SEGMENT = 128


@dataclass
class HubSplit:
    """A CSR whose hub rows were emptied (`ptr`, `idx`) plus a second small CSR over the hubs' neighbour lists cut into
    virtual rows (`seg_rowptr`, `seg_idx`): virtual rows [seg_ptr[h], seg_ptr[h+1]) are consecutive slices of row
    hub_rows[h]; seg_row[v] is the real row of virtual row v."""
    ptr: torch.Tensor          # int64 [n + 1]
    idx: torch.Tensor          # int32 [E - E_hub]
    hub_rows: torch.Tensor     # int64 [H]
    seg_ptr: torch.Tensor      # int64 [H + 1]
    seg_row: torch.Tensor      # int64 [V]
    seg_row32: torch.Tensor    # int32 [V]
    seg_rowptr: torch.Tensor   # int64 [V + 1]
    seg_idx: torch.Tensor      # int32 [E_hub]
    seg_ids: torch.Tensor      # int32 [V] = arange(V): pc_rows_segment_sum's column list

    @property
    def n_virtual(self) -> int:
        return self.seg_row.numel()


def build_hub_split(ptr: torch.Tensor, idx: torch.Tensor, threshold: int, segment: int) -> Optional[HubSplit]:
    """None when no row has more than `threshold` neighbours (one host read of the maximum degree, once per graph)."""
    n = ptr.numel() - 1
    if n <= 0 or idx.numel() == 0:
        return None
    deg = ptr[1:] - ptr[:-1]
    if int(deg.max().item()) <= threshold:
        return None
    dev_ = ptr.device
    is_hub = deg > threshold
    hub_rows = torch.nonzero(is_hub).squeeze(1)
    hub_deg = deg[hub_rows]
    nseg = (hub_deg + segment - 1) // segment
    seg_ptr = torch.zeros(hub_rows.numel() + 1, dtype=I64, device=dev_)
    seg_ptr[1:] = torch.cumsum(nseg, 0)
    seg_row = torch.repeat_interleave(hub_rows, nseg)
    v = seg_row.numel()
    k_in_hub = torch.arange(v, device=dev_) - torch.repeat_interleave(seg_ptr[:-1], nseg)
    seg_len = torch.clamp(torch.repeat_interleave(hub_deg, nseg) - k_in_hub * segment, max=segment)
    seg_rowptr = torch.zeros(v + 1, dtype=I64, device=dev_)
    seg_rowptr[1:] = torch.cumsum(seg_len, 0)
    edge_is_hub = torch.repeat_interleave(is_hub, deg)
    main_deg = torch.where(is_hub, torch.zeros_like(deg), deg)
    main_ptr = torch.zeros(n + 1, dtype=I64, device=dev_)
    main_ptr[1:] = torch.cumsum(main_deg, 0)
    return HubSplit(main_ptr, idx[~edge_is_hub].contiguous(), hub_rows.contiguous(), seg_ptr, seg_row.contiguous(),
                    seg_row.to(I32).contiguous(), seg_rowptr, idx[edge_is_hub].contiguous(),
                    torch.arange(v, dtype=I32, device=dev_))


@dataclass
class CSRGraph:
    """Device CSR of one edge type: row i lists the ascending out-neighbours of node i
    (== sorted(get_neighbors(i, edge_type)), bpg.py:24-31).  The transposed lists (CSC) needed
    by the deterministic backward are built on first use, and so are the hub splits (rows / transposed columns with more
    than HUB_THRESHOLD neighbours)."""
    rowptr: torch.Tensor              # int64 [n_rows + 1]
    col: torch.Tensor                 # int32 [E]
    n_rows: int
    n_cols: int
    _t: Optional[Tuple[torch.Tensor, torch.Tensor]] = field(default=None, repr=False)
    split_hubs: bool = True           # False: never split (regular graphs of the dense drop-in path, halo partitions)
    _hub: Optional[Tuple] = field(default=None, repr=False)      # (HubSplit | None,) once computed
    _hub_t: Optional[Tuple] = field(default=None, repr=False)

    @property
    def num_edges(self) -> int:
        return self.col.numel()

    def transposed(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """(colptr int64 [n_cols+1], row int32 [E]): for every source j the ascending destinations."""
        if self._t is None:
            e = self.num_edges
            keys_t = torch.empty(e, dtype=I64, device=self.col.device)
            call("pc_csr_transpose_keys", dev(self.rowptr, I64, "rowptr"), dev(self.col, I32, "col"), self.n_rows, e,
                 dev(keys_t, I64, "keys_t"), stream())
            sort_keys_(keys_t, digit_mask_for(max(self.n_rows, self.n_cols)))
            colptr, row = csr_from_sorted_keys(keys_t, self.n_cols)
            self._t = (colptr, row)
        return self._t

    def hub_split(self) -> Optional[HubSplit]:
        if not self.split_hubs:
            return None
        if self._hub is None:
            self._hub = (build_hub_split(self.rowptr, self.col, HUB_THRESHOLD, HUB_SEGMENT),)
        return self._hub[0]

    def hub_split_t(self) -> Optional[HubSplit]:
        if not self.split_hubs:
            return None
        if self._hub_t is None:
            colptr, row = self.transposed()
            self._hub_t = (build_hub_split(colptr, row, HUB_THRESHOLD, HUB_SEGMENT),)
        return self._hub_t[0]


def csr_from_sorted_keys(keys: torch.Tensor, n_rows: int) -> Tuple[torch.Tensor, torch.Tensor]:
    e = keys.numel()
    rowptr = torch.empty(n_rows + 1, dtype=I64, device=keys.device)
    col = torch.empty(e, dtype=I32, device=keys.device)
    call("pc_csr_from_sorted_keys", dev(keys, I64, "keys"), e, n_rows, dev(rowptr, I64, "rowptr"), dev(col, I32, "col"), stream())
    return rowptr, col


def build_csr(src: torch.Tensor, dst: torch.Tensor, n_rows: int, n_cols: Optional[int] = None) -> Tuple[CSRGraph, torch.Tensor]:
    """Edge list (duplicates allowed) -> (deduplicated CSRGraph, its sorted-unique keys)."""
    n_cols = n_rows if n_cols is None else n_cols
    keys = pack_keys(src, dst)
    sort_keys_(keys, digit_mask_for(max(n_rows, n_cols)))
    keys = unique_sorted(keys)
    rowptr, col = csr_from_sorted_keys(keys, n_rows)
    return CSRGraph(rowptr, col, n_rows, n_cols), keys


_REGULAR_CACHE = {}


def regular_graph(batch: int, n_nbr: int, device) -> CSRGraph:
    """CSR of the dense drop-in path: row i attends to rows [i*n, (i+1)*n) of a [B*n, .] table -
    the zero-padded [B, N, D] neighbour tensor of data_loader.py:186-198 viewed as a graph."""
    key = (batch, n_nbr, str(device))
    g = _REGULAR_CACHE.get(key)
    if g is None:
        e = batch * n_nbr
        rowptr = torch.arange(batch + 1, dtype=I64, device=device) * n_nbr
        col = torch.arange(e, dtype=I32, device=device)
        colptr = torch.arange(e + 1, dtype=I64, device=device)
        row = (torch.arange(e, dtype=I64, device=device) // max(n_nbr, 1)).to(I32)
        g = CSRGraph(rowptr, col, batch, e, (colptr, row), split_hubs=False)
        if len(_REGULAR_CACHE) > 64:
            _REGULAR_CACHE.clear()
        _REGULAR_CACHE[key] = g
    return g


def triplet_batch_rows(table: torch.Tensor, csr: CSRGraph, anchor: torch.Tensor, positive: torch.Tensor,
                       negatives: torch.Tensor, nbr_ptr: torch.Tensor, n_nbr: int):
    """Feature rows of one triplet batch in one launch (pc_triplet_batch_rows): returns (anchor_rows [B, D],
    neighbour_rows [n_nbr, D], positive_rows [B, D], negative_rows [B * kneg, D]), contiguous views of one buffer, and
    the batch graph: row b attends to neighbour rows nbr_ptr[b] .. nbr_ptr[b + 1] (anchor b's co-view neighbours in CSR
    order), with its transpose filled in.  nbr_ptr int64 [B + 1] is the prefix sum of the anchors' co-view degrees and
    n_nbr == nbr_ptr[B] its host copy (GraphTripletSampler.neighborhood_batches / TripletBatch.build).

    The batch graph splits hub rows only when the full CSR has any (csr.hub_split(), one host read per graph); it then
    takes one host read per batch to find its own hub rows.  A graph without hubs reads nothing back per batch."""
    b = anchor.numel()
    if table.dim() != 2 or positive.numel() != b or negatives.dim() != 2 or negatives.shape[0] != b or nbr_ptr.numel() != b + 1:
        raise ValueError(f"triplet_batch_rows: table [N, D], anchor [B], positive [B], negatives [B, K] and nbr_ptr [B + 1] "
                         f"expected, got {tuple(table.shape)}, {tuple(anchor.shape)}, {tuple(positive.shape)}, "
                         f"{tuple(negatives.shape)}, {tuple(nbr_ptr.shape)}")
    kneg, d, n_nbr = negatives.shape[1], table.shape[1], int(n_nbr)
    rows = torch.empty(2 * b + n_nbr + b * kneg, d, dtype=F32, device=table.device)
    edge_row = torch.empty(n_nbr, dtype=I32, device=table.device)
    call("pc_triplet_batch_rows", _f32_cuda(table, "table"), table.stride(0), d, dev(anchor, I64, "anchor"),
         dev(positive, I64, "positive"), dev(negatives, I64, "negatives"), b, kneg, dev(csr.rowptr, I64, "rowptr"),
         dev(csr.col, I32, "col"), dev(nbr_ptr, I64, "nbr_ptr"), n_nbr, dev(rows, F32, "rows"), dev(edge_row, I32, "edge_row"),
         stream())
    a_rows, nbr_rows, p_rows, n_rows = rows.split([b, n_nbr, b, b * kneg])
    graph = CSRGraph(nbr_ptr, torch.arange(n_nbr, dtype=I32, device=table.device), b, n_nbr,
                     (torch.arange(n_nbr + 1, dtype=I64, device=table.device), edge_row),
                     split_hubs=csr.hub_split() is not None, _hub_t=(None,))   # every neighbour row has one edge: no hub columns
    return a_rows, nbr_rows, p_rows, n_rows, graph


# --------------------------------------------------------------------------- GAT
def _f32_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda or t.dtype != F32 or t.stride(-1) != 1:
        raise RuntimeError(f"{what}: expected a float32 CUDA tensor with unit column stride, got {t.dtype} on {t.device} "
                           "(no CPU fallback)")
    return _lib.c_void_p(t.data_ptr())


def _gat_fwd_call(q, kv, rowptr, col, n_rows, heads, dropout_p, seed, o, stats, dst_ids=None):
    call("pc_gat_fwd", _f32_cuda(q, "q"), q.stride(0), dev(kv, F32, "kv"), dev(rowptr, I64, "rowptr"), dev(col, I32, "col"), n_rows,
         heads, float(dropout_p), int(seed), dev(dst_ids, I32, "dst_ids"), dev(o, F32, "o"), dev(stats, F32, "stats"), stream())


def gat_fwd_raw(q: torch.Tensor, kv: torch.Tensor, graph: "CSRGraph", heads: int, dropout_p: float, seed: int):
    """pc_gat_fwd; q may be a strided [n, 128] view.  Returns (o [n,128], stats [n,2,heads]).  Hub rows are attended slice
    by slice (virtual rows) and merged (pc_gat_merge_segments)."""
    o = torch.empty(graph.n_rows, EMB, dtype=F32, device=q.device)
    stats = torch.empty(graph.n_rows, 2, heads, dtype=F32, device=q.device)
    hs = graph.hub_split()
    if hs is None:
        _gat_fwd_call(q, kv, graph.rowptr, graph.col, graph.n_rows, heads, dropout_p, seed, o, stats)
        return o, stats
    _gat_fwd_call(q, kv, hs.ptr, hs.idx, graph.n_rows, heads, dropout_p, seed, o, stats)        # hub rows: empty here
    v = hs.n_virtual
    qh = q.index_select(0, hs.seg_row).contiguous()
    oh = torch.empty(v, EMB, dtype=F32, device=q.device)
    sh = torch.empty(v, 2, heads, dtype=F32, device=q.device)
    _gat_fwd_call(qh, kv, hs.seg_rowptr, hs.seg_idx, v, heads, dropout_p, seed, oh, sh, hs.seg_row32)
    call("pc_gat_merge_segments", dev(oh, F32, "o_seg"), dev(sh, F32, "stats_seg"), dev(hs.seg_ptr, I64, "seg_ptr"),
         dev(hs.hub_rows, I64, "hub_rows"), hs.hub_rows.numel(), heads, dev(o, F32, "o"), dev(stats, F32, "stats"), stream())
    return o, stats


def gat_delta_raw(o, d_o, heads, stats) -> None:
    call("pc_gat_delta", dev(o, F32, "o"), _f32_cuda(d_o, "d_o"), d_o.stride(0), o.shape[0], heads, dev(stats, F32, "stats"), stream())


def _gat_bwd_dst_call(q, kv, rowptr, col, n_rows, heads, dropout_p, seed, o, d_o, stats, dq, dst_ids=None):
    call("pc_gat_bwd_dst", _f32_cuda(q, "q"), q.stride(0), dev(kv, F32, "kv"), dev(rowptr, I64, "rowptr"), dev(col, I32, "col"),
         n_rows, heads, float(dropout_p), int(seed), dev(dst_ids, I32, "dst_ids"), dev(o, F32, "o"), _f32_cuda(d_o, "d_o"),
         d_o.stride(0), dev(stats, F32, "stats"), _f32_cuda(dq, "dq"), dq.stride(0), stream())


def _segment_sums(rows: torch.Tensor, hs: HubSplit) -> torch.Tensor:
    """[H, W]: per hub, the sum of its virtual rows' partial gradients in ascending slice order."""
    out = torch.empty(hs.hub_rows.numel(), rows.shape[1], dtype=F32, device=rows.device)
    call("pc_rows_segment_sum", dev(rows, F32, "rows"), dev(hs.seg_ptr, I64, "rowptr"), dev(hs.seg_ids, I32, "col"),
         hs.hub_rows.numel(), rows.shape[1], dev(out, F32, "out"), stream())
    return out


def gat_bwd_dst_raw(q, kv, graph: "CSRGraph", heads, dropout_p, seed, o, d_o, stats, dq) -> None:
    hs = graph.hub_split()
    if hs is None:
        _gat_bwd_dst_call(q, kv, graph.rowptr, graph.col, graph.n_rows, heads, dropout_p, seed, o, d_o, stats, dq)
        return
    _gat_bwd_dst_call(q, kv, hs.ptr, hs.idx, graph.n_rows, heads, dropout_p, seed, o, d_o, stats, dq)   # also writes delta of every row
    v = hs.n_virtual
    qh, doh = q.index_select(0, hs.seg_row).contiguous(), d_o.index_select(0, hs.seg_row).contiguous()
    oh, sh = o.index_select(0, hs.seg_row), stats.index_select(0, hs.seg_row).contiguous()       # the ROW's final O and lse
    dqh = torch.empty(v, EMB, dtype=F32, device=q.device)
    _gat_bwd_dst_call(qh, kv, hs.seg_rowptr, hs.seg_idx, v, heads, dropout_p, seed, oh, doh, sh, dqh, hs.seg_row32)
    dq.index_copy_(0, hs.hub_rows, _segment_sums(dqh, hs))


def _gat_bwd_src_call(q, kv, colptr, row, n_cols, heads, dropout_p, seed, d_o, stats, dkv, src_base=0, src_ids=None):
    call("pc_gat_bwd_src", _f32_cuda(q, "q"), q.stride(0), dev(kv, F32, "kv"), dev(colptr, I64, "colptr"), dev(row, I32, "row"),
         n_cols, heads, float(dropout_p), int(seed), _f32_cuda(d_o, "d_o"), d_o.stride(0), dev(stats, F32, "stats"),
         _f32_cuda(dkv, "dkv"), dkv.stride(0), int(src_base), dev(src_ids, I32, "src_ids"), stream())


def gat_bwd_src_raw(q, kv, graph: "CSRGraph", heads, dropout_p, seed, d_o, stats, dkv, col_begin: int = 0,
                    col_count: Optional[int] = None) -> None:
    """needs stats[:,1,:] (delta) from pc_gat_bwd_dst or pc_gat_delta.  (col_begin, col_count) restricts the pass to a
    range of source columns (rows col_begin.. of kv / dkv); hub columns (whole-graph call only) are split like hub rows."""
    colptr, row = graph.transposed()
    whole = col_begin == 0 and (col_count is None or col_count == graph.n_cols)
    if col_count is None:
        col_count = graph.n_cols - col_begin
    if col_count <= 0:
        return
    hs = graph.hub_split_t() if whole else None
    if hs is None:
        kv_r, dkv_r = kv[col_begin: col_begin + col_count], dkv[col_begin: col_begin + col_count]
        _gat_bwd_src_call(q, kv_r, colptr[col_begin: col_begin + col_count + 1], row, col_count, heads, dropout_p, seed, d_o, stats,
                          dkv_r, col_begin)
        return
    _gat_bwd_src_call(q, kv, hs.ptr, hs.idx, graph.n_cols, heads, dropout_p, seed, d_o, stats, dkv)   # hub columns: zeros
    v = hs.n_virtual
    kvh = kv.index_select(0, hs.seg_row).contiguous()
    dkvh = torch.empty(v, 2 * EMB, dtype=F32, device=q.device)
    _gat_bwd_src_call(q, kvh, hs.seg_rowptr, hs.seg_idx, v, heads, dropout_p, seed, d_o, stats, dkvh, 0, hs.seg_row32)
    dkv.index_copy_(0, hs.hub_rows, _segment_sums(dkvh, hs))


def gat_bwd_raw(q, kv, graph: "CSRGraph", heads, dropout_p, seed, o, d_o, stats, dq, dkv) -> None:
    """pc_gat_bwd_dst + pc_gat_bwd_src; q, d_o, dq, dkv may be strided views (row strides are passed down)."""
    gat_bwd_dst_raw(q, kv, graph, heads, dropout_p, seed, o, d_o, stats, dq)
    gat_bwd_src_raw(q, kv, graph, heads, dropout_p, seed, d_o, stats, dkv)


class _GATAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, kv, graph: CSRGraph, heads: int, dropout_p: float, seed: int):
        q = q.contiguous()
        kv = kv.contiguous()
        if q.dim() != 2 or q.shape[1] != EMB or kv.dim() != 2 or kv.shape[1] != 2 * EMB:
            raise ValueError(f"gat: q must be [n_dst,{EMB}] and kv [n_src,{2 * EMB}], got {tuple(q.shape)}, {tuple(kv.shape)}")
        if q.shape[0] != graph.n_rows or kv.shape[0] != graph.n_cols:
            raise ValueError("gat: q / kv row counts do not match the graph")
        o, stats = gat_fwd_raw(q, kv, graph, heads, dropout_p, seed)
        ctx.save_for_backward(q, kv, o, stats)
        ctx.graph, ctx.heads, ctx.dropout_p, ctx.seed = graph, heads, float(dropout_p), int(seed)
        return o

    @staticmethod
    def backward(ctx, d_o):
        q, kv, o, stats = ctx.saved_tensors
        d_o = d_o.contiguous()
        dq = torch.empty_like(q)
        dkv = torch.empty_like(kv)
        gat_bwd_raw(q, kv, ctx.graph, ctx.heads, ctx.dropout_p, ctx.seed, o, d_o, stats, dq, dkv)
        return dq, dkv, None, None, None, None


def gat_attention(q: torch.Tensor, kv: torch.Tensor, graph: CSRGraph, heads: int, dropout_p: float = 0.0,
                  seed: int = 0) -> torch.Tensor:
    """o[i] = sum_j softmax_j(q_i.k_j / sqrt(dh)) v_j per head over the CSR (differentiable)."""
    return _GATAttention.apply(q, kv, graph, heads, dropout_p, seed)


# --------------------------------------------------------------------------- dense projections (tcgen05)
EPI_BIAS, EPI_BIAS_TANH, EPI_TANH_GRAD, EPI_BIAS_SELECT, EPI_BIAS_ADD, EPI_ROWMASK, EPI_ADD_UNSELECTED = 0, 1, 2, 3, 4, 5, 6


def linear_tc(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, epilogue: int = EPI_BIAS,
              aux: Optional[torch.Tensor] = None, rowptr: Optional[torch.Tensor] = None, split: Optional[int] = None,
              out0: Optional[torch.Tensor] = None, out1: Optional[torch.Tensor] = None, col_stats: bool = False):
    """epilogue(A . W^T + bias) on the tensor cores (pc_linear_tf32x3).  Returns one [m, n] tensor, or
    ([m, split], [m, n - split]) when `split` is given.  out0 / out1 may be preallocated (strided) views.
    col_stats=True (plain bias epilogue, n <= 256) also returns float64 [2, n]: column sums of the output and of its
    square, taken in the GEMM's epilogue."""
    m, k = a.shape
    n = w.shape[0]
    if a.stride(1) != 1 or w.stride() != (k, 1):
        raise ValueError("linear_tc: A must have unit column stride and W must be contiguous [n, k]")
    split_ = n if split is None else split
    if out0 is None:
        out0 = torch.empty(m, split_, dtype=F32, device=a.device)
    if out1 is None and split_ < n:
        out1 = torch.empty(m, n - split_, dtype=F32, device=a.device)
    ws = _lib.workspace(_lib.LIB.pc_linear_workspace_bytes(n, k), a.device)
    sums = torch.empty(2, n, dtype=F64, device=a.device) if col_stats else None
    call("pc_linear_tf32x3", _f32_cuda(a, "a"), m, k, a.stride(0), dev(w, F32, "w"), n, dev(bias, F32, "bias"), epilogue,
         _f32_cuda(aux, "aux") if aux is not None else None, aux.stride(0) if aux is not None else 0,
         dev(rowptr, I64, "rowptr"), _f32_cuda(out0, "out0"), out0.stride(0), split_,
         _f32_cuda(out1, "out1") if out1 is not None else None, out1.stride(0) if out1 is not None else 0,
         dev(sums, F64, "col_sums"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    if col_stats:
        return out0, sums
    return out0 if out1 is None else (out0, out1)


def wgrad_tc(dy: torch.Tensor, x: torch.Tensor, want_bias: bool = True):
    """(dW [n, k], db [n] | None) = (dY^T X, column sums of dY) on the tensor cores (pc_wgrad_tf32x3)."""
    m, n = dy.shape
    k = x.shape[1]
    if dy.stride(1) != 1 or x.stride(1) != 1 or x.shape[0] != m:
        raise ValueError("wgrad_tc: dY [m, n] and X [m, k] must have unit column stride and equal row counts")
    if not (dy.is_cuda and x.is_cuda and dy.dtype == F32 and x.dtype == F32):
        raise RuntimeError("wgrad_tc: float32 CUDA tensors required; no CPU fallback")
    dw = torch.empty(n, k, dtype=F32, device=dy.device)
    db = torch.empty(n, dtype=F32, device=dy.device) if want_bias else None
    ws = _lib.workspace(_lib.LIB.pc_wgrad_workspace_bytes(n, k), dy.device)
    call("pc_wgrad_tf32x3", _f32_cuda(dy, "dy"), m, n, dy.stride(0), _f32_cuda(x, "x"), k, x.stride(0),
         dev(dw, F32, "dw"), dev(db, F32, "db"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return dw, db


# --------------------------------------------------------------------------- BatchNorm / tanh / select kernels
def _col_reduce_ws(n: int, device):
    return _lib.workspace(_lib.LIB.pc_col_reduce_workspace_bytes(n), device)


def col_stats(x: torch.Tensor) -> torch.Tensor:
    """float64 [2, n]: column sums of x and of x^2 (fixed summation order)."""
    m, n = x.shape
    sums = torch.empty(2, n, dtype=F64, device=x.device)
    ws = _col_reduce_ws(n, x.device)
    call("pc_col_stats", _f32_cuda(x, "x"), m, n, x.stride(0), dev(sums, F64, "sums"), dev(ws, torch.uint8, "ws"),
         ws.numel(), stream())
    return sums


def col_sum_unselected(x: torch.Tensor, rowptr: torch.Tensor) -> torch.Tensor:
    """float64 [n]: column sums of x over the rows that have NO neighbours (rowptr[r+1] == rowptr[r])."""
    m, n = x.shape
    sums = torch.empty(2, n, dtype=F64, device=x.device)
    ws = _col_reduce_ws(n, x.device)
    call("pc_col_sum_unselected", _f32_cuda(x, "x"), m, n, x.stride(0), dev(rowptr, I64, "rowptr"), dev(sums, F64, "sums"),
         dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return sums[0]


def bn_bwd_reduce(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor) -> torch.Tensor:
    """float64 [2, n]: sum_r dy and sum_r dy * (x - mean) * rstd."""
    m, n = x.shape
    sums = torch.empty(2, n, dtype=F64, device=x.device)
    ws = _col_reduce_ws(n, x.device)
    call("pc_bn_bwd_reduce", _f32_cuda(dy, "dy"), dy.stride(0), _f32_cuda(x, "x"), x.stride(0), m, n, dev(mean, F32, "mean"),
         dev(rstd, F32, "rstd"), dev(sums, F64, "sums"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return sums


def scale_shift_tanh(x: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, tanh: bool = True) -> torch.Tensor:
    m, n = x.shape
    y = torch.empty(m, n, dtype=F32, device=x.device)
    call("pc_scale_shift_tanh", _f32_cuda(x, "x"), x.stride(0), m, n, dev(scale, F32, "scale"), dev(shift, F32, "shift"),
         int(tanh), dev(y, F32, "y"), n, stream())
    return y


def affine2(a: torch.Tensor, b: torch.Tensor, ca: torch.Tensor, cb: torch.Tensor, cc: torch.Tensor) -> torch.Tensor:
    """ca[c] * a + cb[c] * b + cc[c]."""
    m, n = a.shape
    out = torch.empty(m, n, dtype=F32, device=a.device)
    call("pc_affine2", _f32_cuda(a, "a"), a.stride(0), _f32_cuda(b, "b"), b.stride(0), m, n, dev(ca, F32, "ca"),
         dev(cb, F32, "cb"), dev(cc, F32, "cc"), dev(out, F32, "out"), n, stream())
    return out


def mask_split(g: torch.Tensor, rowptr: torch.Tensor):
    """(kept, rest): rows with neighbours keep g in `kept`, rows without in `rest` (zeros elsewhere)."""
    g = g.contiguous()
    kept, rest = torch.empty_like(g), torch.empty_like(g)
    call("pc_mask_split", dev(g, F32, "g"), g.shape[0], g.shape[1], dev(rowptr, I64, "rowptr"), dev(kept, F32, "kept"),
         dev(rest, F32, "rest"), stream())
    return kept, rest


# --------------------------------------------------------------------------- hinge losses
class _HingeRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, p, n, a_per_group: int, kneg: int, margin: float, eps: float):
        a, p, n = a.contiguous(), p.contiguous(), n.contiguous()
        rows, dim = a.shape
        per = torch.empty(rows, dtype=F32, device=a.device)
        loss = torch.empty((), dtype=F32, device=a.device)
        call("pc_hinge_rows_fwd", dev(a, F32, "a"), dev(p, F32, "p"), dev(n, F32, "n"), rows, a_per_group, kneg, dim,
             margin, eps, dev(per, F32, "per"), dev(loss, F32, "loss"), stream())
        ctx.save_for_backward(a, p, n)
        ctx.cfg = (a_per_group, kneg, margin, eps)
        return loss

    @staticmethod
    def backward(ctx, g):
        a, p, n = ctx.saved_tensors
        a_per_group, kneg, margin, eps = ctx.cfg
        rows, dim = a.shape
        g = g.contiguous().to(F32)
        da = torch.empty_like(a)
        need_pn = a_per_group == 1 and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        dp = torch.empty_like(p) if need_pn else None
        dn = torch.empty_like(n) if need_pn else None
        call("pc_hinge_rows_bwd", dev(a, F32, "a"), dev(p, F32, "p"), dev(n, F32, "n"), rows, a_per_group, kneg, dim,
             margin, eps, dev(g, F32, "grad"), dev(da, F32, "da"), dev(dp, F32, "dp"), dev(dn, F32, "dn"), stream())
        return da, dp, dn, None, None, None, None


def index_rows_grad(rows: torch.Tensor, index: torch.Tensor, n_rows: int, scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Dense [n_rows, W] gradient of table[index] from the gradient rows [S, W], no float atomics (pc_rows_index_grad:
    slots sorted stably by table row, summed per row in slot order, times the device scalar `scale` if given)."""
    rows = rows.contiguous()
    index = index.reshape(-1).to(I64).contiguous()
    slots, w = rows.shape
    out = torch.empty(n_rows, w, dtype=F32, device=rows.device)
    ws = _lib.workspace(_lib.LIB.pc_rows_index_grad_workspace_bytes(slots, n_rows), rows.device)
    call("pc_rows_index_grad", dev(rows, F32, "rows"), dev(index, I64, "index"), slots, n_rows, w,
         dev(None if scale is None else scale.reshape(1).contiguous().to(F32), F32, "scale"), dev(out, F32, "out"),
         dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return out


class _GatherRows(torch.autograd.Function):
    """table[index] (nn.Embedding / advanced-index gather, p_companion.py:49,54,66) with a deterministic dense gradient."""

    @staticmethod
    def forward(ctx, table, index):
        table = table.contiguous()
        index = index.reshape(-1).to(I64).contiguous()
        ctx.save_for_backward(index)
        ctx.n_rows = table.shape[0]
        return rows_gather(table, index)

    @staticmethod
    def backward(ctx, d_rows):
        (index,) = ctx.saved_tensors
        return index_rows_grad(d_rows, index, ctx.n_rows), None


def gather_rows(table: torch.Tensor, index: torch.Tensor) -> torch.Tensor:
    """[len(index), W] rows of `table` (differentiable with respect to the table when it requires grad)."""
    if table.requires_grad and torch.is_grad_enabled():
        return _GatherRows.apply(table, index)
    return rows_gather(table.detach().contiguous(), index.reshape(-1).to(I64).contiguous())


class _TripletFromTable(torch.autograd.Function):
    """Triplet hinge on rows of one embedding table selected by index (anchors | positives | negatives), ONE kernel for
    the loss and the gradient rows of all slots (pc_triplet_indexed reads the table through the index: no gathered copy,
    no second pass in backward).  Backward returns a dense d_table built without float atomics: the slot list is stably
    sorted by node, turned into a CSR and summed per node in slot order, times the upstream gradient (pc_rows_index_grad)."""

    @staticmethod
    def forward(ctx, table, slot_nodes, batch: int, kneg: int, margin: float, eps: float):
        table = table.contiguous()
        d = table.shape[1]
        per = torch.empty(batch, dtype=F32, device=table.device)
        loss = torch.empty((), dtype=F32, device=table.device)
        grads = torch.empty(slot_nodes.numel(), d, dtype=F32, device=table.device) if ctx.needs_input_grad[0] else None
        call("pc_triplet_indexed", dev(table, F32, "table"), dev(slot_nodes, I64, "slot_rows"), batch, kneg, d, margin, eps,
             dev(per, F32, "per"), dev(loss, F32, "loss"), dev(grads, F32, "slot_grads"), stream())
        ctx.save_for_backward(grads, slot_nodes)
        ctx.n_nodes = table.shape[0]
        return loss

    @staticmethod
    def backward(ctx, g):
        grads, slot_nodes = ctx.saved_tensors
        return index_rows_grad(grads, slot_nodes, ctx.n_nodes, scale=g), None, None, None, None, None


def triplet_hinge_indexed(table: torch.Tensor, anchor_idx: torch.Tensor, positive_idx: torch.Tensor,
                          negative_idx: torch.Tensor, margin: float, eps: float = 1e-6) -> torch.Tensor:
    """triplet_hinge(table[anchor], table[positive], table[negative [B, K]]) with a deterministic dense d_table."""
    b = anchor_idx.numel()
    k = negative_idx.numel() // b
    slot_nodes = torch.cat([anchor_idx.reshape(-1), positive_idx.reshape(-1), negative_idx.reshape(-1)]).to(I64).contiguous()
    return _TripletFromTable.apply(table, slot_nodes, b, k, float(margin), float(eps))


def triplet_hinge(anchor, positive, negative, margin: float, eps: float = 1e-6) -> torch.Tensor:
    """mean relu(margin - ||a-p+eps|| + mean_k ||a-n_k+eps||)  (product2vec.py:137-154)."""
    if negative.dim() == 2:
        negative = negative.unsqueeze(1)
    b, k, d = negative.shape
    return _HingeRows.apply(anchor, positive, negative.reshape(b * k, d), 1, k, float(margin), float(eps))


def item_hinge(projected, positive_items, negative_items, margin: float) -> torch.Tensor:
    """mean clamp(margin - ||proj-pos|| + ||proj-neg||, 0) over [B, K]  (p_companion.py:105-119)."""
    b, k, d = projected.shape
    return _HingeRows.apply(projected.reshape(b * k, d), positive_items, negative_items, k, 1, float(margin), 0.0)


class _HingeType(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sims, pos, neg, margin: float):
        sims = sims.contiguous()
        pos, neg = pos.contiguous().to(I64), neg.contiguous().to(I64)
        rows, nt = sims.shape
        per = torch.empty(rows, dtype=F32, device=sims.device)
        loss = torch.empty((), dtype=F32, device=sims.device)
        call("pc_hinge_type_fwd", dev(sims, F32, "sims"), dev(pos, I64, "pos"), dev(neg, I64, "neg"), rows, nt, margin,
             dev(per, F32, "per"), dev(loss, F32, "loss"), stream())
        ctx.save_for_backward(sims, pos, neg)
        ctx.margin = margin
        return loss

    @staticmethod
    def backward(ctx, g):
        sims, pos, neg = ctx.saved_tensors
        rows, nt = sims.shape
        d = torch.zeros_like(sims)
        g = g.contiguous().to(F32)
        call("pc_hinge_type_bwd", dev(sims, F32, "sims"), dev(pos, I64, "pos"), dev(neg, I64, "neg"), rows, nt,
             ctx.margin, dev(g, F32, "grad"), dev(d, F32, "d_sims"), stream())
        return d, None, None, None


class _HingeTypeFactored(torch.autograd.Function):
    """Same loss value as _HingeType on S = base . W^T, but the gradient goes straight to the factors: only two
    entries per row of S carry gradient, so d_base = c_i (W[neg_i] - W[pos_i]) and dW gets +-c_i base_i on two rows per
    sample - no dense [B, T] gradient and none of the two [B, T]-sized backward GEMMs (SURVEY 8 a13: they dominate C3).
    dW is accumulated without float atomics: slots sorted by type (pc_sort_keys), summed per type in slot order."""

    @staticmethod
    def forward(ctx, base, weight, sims, pos, neg, margin: float):
        sims = sims.contiguous()
        pos, neg = pos.contiguous().to(I64), neg.contiguous().to(I64)
        rows, nt = sims.shape
        per = torch.empty(rows, dtype=F32, device=sims.device)
        loss = torch.empty((), dtype=F32, device=sims.device)
        call("pc_hinge_type_fwd", dev(sims, F32, "sims"), dev(pos, I64, "pos"), dev(neg, I64, "neg"), rows, nt, margin,
             dev(per, F32, "per"), dev(loss, F32, "loss"), stream())
        ctx.save_for_backward(base, weight, per, pos, neg)
        return loss

    @staticmethod
    def backward(ctx, g):
        base, weight, per, pos, neg = ctx.saved_tensors
        rows, nt = base.shape[0], weight.shape[0]
        need_b, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        g = g.contiguous().to(F32)
        base_c, weight_c = base.contiguous(), weight.contiguous()
        d_base = torch.empty_like(base_c) if need_b else None
        vals = torch.empty(2 * rows, base.shape[1], dtype=F32, device=base.device) if need_w else None   # slot i: pos_i, B + i: neg_i
        call("pc_hinge_type_factored_bwd", dev(per, F32, "per"), dev(pos, I64, "pos"), dev(neg, I64, "neg"), dev(g, F32, "grad"),
             dev(base_c, F32, "base"), dev(weight_c, F32, "weight"), rows, base.shape[1], dev(d_base, F32, "d_base"),
             dev(vals, F32, "vals"), stream())
        d_w = index_rows_grad(vals, torch.cat([pos, neg]), nt) if need_w else None
        return d_base, d_w, None, None, None, None


def type_hinge(sims, pos, neg, margin: float) -> torch.Tensor:
    """mean clamp(margin - S[i,pos_i] + S[i,neg_i], 0)  (p_companion.py:95-103).  When `sims` was produced by
    PCompanion.forward it carries its factors (base [B, L], W [T, L]) and the gradient bypasses the [B, T] matrix."""
    factors = getattr(sims, "_pc_factors", None)
    if factors is not None and factors[0].shape[0] == sims.shape[0] and factors[1].shape[0] == sims.shape[1]:
        return _HingeTypeFactored.apply(factors[0], factors[1], sims.detach(), pos, neg, float(margin))
    return _HingeType.apply(sims, pos, neg, float(margin))


# --------------------------------------------------------------------------- P-Companion small layers
class _MLP2(torch.autograd.Function):
    """W2 . dropout(relu(W1 . x + b1)) + b2 on x = table[index] (or the rows of `table` when index is None):
    type_transition.py:15-20 (+ the nn.Embedding gather of p_companion.py:54) as one kernel each way."""

    @staticmethod
    def forward(ctx, table, index, w1, b1, w2, b2, p_drop: float, seed: int, seed_dev=None):
        table = table.contiguous()
        idx = None if index is None else index.reshape(-1).to(I64).contiguous()
        rows = table.shape[0] if idx is None else idx.numel()
        hid, d_in = w1.shape
        d_out = w2.shape[0]
        hidden = torch.empty(rows, hid, dtype=F32, device=table.device)
        out = torch.empty(rows, d_out, dtype=F32, device=table.device)
        w1c, w2c = w1.contiguous(), w2.contiguous()
        call("pc_mlp2_fwd", dev(table, F32, "table"), dev(idx, I64, "index"), rows, d_in, hid, d_out, dev(w1c, F32, "w1"),
             dev(b1, F32, "b1"), dev(w2c, F32, "w2"), dev(b2, F32, "b2"), float(p_drop), int(seed), dev(seed_dev, I64, "seed_dev"),
             dev(hidden, F32, "hidden"), dev(out, F32, "out"), stream())
        ctx.save_for_backward(table, idx, hidden, w1c, w2c)
        ctx.p_drop = float(p_drop)
        ctx.has_bias = (b1 is not None, b2 is not None)
        return out

    @staticmethod
    def backward(ctx, d_out):
        table, idx, hidden, w1, w2 = ctx.saved_tensors
        d_out = d_out.contiguous()
        rows = d_out.shape[0]
        hid, d_in = w1.shape
        n_out = w2.shape[0]
        need_x = ctx.needs_input_grad[0]
        d_x = torch.empty(rows, d_in, dtype=F32, device=d_out.device) if need_x else None
        d_w1, d_w2 = torch.empty_like(w1), torch.empty_like(w2)
        d_b1 = torch.empty(hid, dtype=F32, device=d_out.device) if ctx.has_bias[0] else None
        d_b2 = torch.empty(n_out, dtype=F32, device=d_out.device) if ctx.has_bias[1] else None
        if rows == 0:
            return (torch.zeros_like(table) if need_x else None, None, torch.zeros_like(w1), None if d_b1 is None else d_b1.zero_(),
                    torch.zeros_like(w2), None if d_b2 is None else d_b2.zero_(), None, None, None)
        ws = _lib.workspace(_lib.LIB.pc_mlp2_bwd_workspace_bytes(d_in, hid, n_out), d_out.device)
        call("pc_mlp2_bwd", dev(d_out, F32, "d_out"), dev(table, F32, "table"), dev(idx, I64, "index"), dev(hidden, F32, "hidden"),
             rows, d_in, hid, n_out, dev(w1, F32, "w1"), dev(w2, F32, "w2"), ctx.p_drop, dev(d_x, F32, "d_x"), dev(d_w1, F32, "d_w1"),
             dev(d_b1, F32, "d_b1"), dev(d_w2, F32, "d_w2"), dev(d_b2, F32, "d_b2"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
        d_table = None
        if need_x:
            d_table = d_x if idx is None else index_rows_grad(d_x, idx, table.shape[0])
        return d_table, None, d_w1, d_b1, d_w2, d_b2, None, None, None


def mlp2_supported(d_in: int, hid: int, d_out: int) -> bool:
    return 4 <= d_in <= 256 and 1 <= hid <= 128 and 1 <= d_out <= 256


def mlp2(table: torch.Tensor, index: Optional[torch.Tensor], w1, b1, w2, b2, p_drop: float = 0.0, seed: int = 0,
         seed_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """seed_dev: optional int64 device scalar added to `seed` when the kernel runs (CUDA-graph replays, see graphs.py)."""
    if not table.is_cuda:
        raise RuntimeError(f"pcompanion_b200.ops.mlp2: input on {table.device}; CUDA only (no CPU fallback)")
    return _MLP2.apply(table, index, w1, b1, w2, b2, float(p_drop), int(seed), seed_dev)


class _ItemCombine(torch.autograd.Function):
    """pi[:, None, :] * tp.view(B, Kt, D)   (item_prediction.py:38)."""

    @staticmethod
    def forward(ctx, pi, tp, kt: int):
        pi, tp = pi.contiguous(), tp.contiguous()
        b, d = pi.shape
        out = torch.empty(b, kt, d, dtype=F32, device=pi.device)
        call("pc_item_combine_fwd", dev(pi, F32, "pi"), dev(tp, F32, "tp"), b, kt, d, dev(out, F32, "out"), stream())
        ctx.save_for_backward(pi, tp)
        ctx.kt = kt
        return out

    @staticmethod
    def backward(ctx, d_out):
        pi, tp = ctx.saved_tensors
        d_out = d_out.contiguous()
        d_pi, d_tp = torch.empty_like(pi), torch.empty_like(tp)
        call("pc_item_combine_bwd", dev(d_out, F32, "d_out"), dev(pi, F32, "pi"), dev(tp, F32, "tp"), pi.shape[0], ctx.kt,
             pi.shape[1], dev(d_pi, F32, "d_pi"), dev(d_tp, F32, "d_tp"), stream())
        return d_pi, d_tp, None


def item_combine(pi: torch.Tensor, tp: torch.Tensor, kt: int) -> torch.Tensor:
    if tp.shape[0] != pi.shape[0] * kt or tp.shape[1] != pi.shape[1]:
        raise ValueError(f"item_combine: pi {tuple(pi.shape)} and tp {tuple(tp.shape)} do not match kt={kt}")
    return _ItemCombine.apply(pi, tp, int(kt))


def type_scores_topk_supported(base: torch.Tensor, weight: torch.Tensor, k: int) -> bool:
    return (base.is_cuda and base.dtype == F32 and base.dim() == 2 and base.shape[1] % 32 == 0 and 32 <= base.shape[1] <= 4096
            and weight.shape[0] % 4 == 0 and 1 <= k <= 4 and k <= weight.shape[0] and base.shape[0] > 0)


def type_scores_topk(base: torch.Tensor, weight: torch.Tensor, k: int, materialize: bool = True):
    """(S = base . W^T [B, T] or None, top scores f64 [B, k], top columns i64 [B, k]) - one tcgen05 GEMM whose epilogue keeps
    the row top-k (pc_type_scores_topk; p_companion.py:60-64).  Not differentiable here: see dense.type_scores."""
    base, weight = base.contiguous(), weight.contiguous()
    b, l = base.shape
    t = weight.shape[0]
    sims = torch.empty(b, t, dtype=F32, device=base.device) if materialize else None
    out_s = torch.empty(b, k, dtype=F64, device=base.device)
    out_i = torch.empty(b, k, dtype=I64, device=base.device)
    ws = _lib.workspace(_lib.LIB.pc_type_scores_topk_workspace_bytes(b, t, l, k), base.device)
    call("pc_type_scores_topk", dev(base, F32, "base"), b, l, l, dev(weight, F32, "weight"), t, dev(sims, F32, "sims"), t, k,
         dev(out_s, F64, "out_scores"), dev(out_i, I64, "out_idx"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return sims, out_s, out_i


# --------------------------------------------------------------------------- retrieval
TOPK_GROUP_ROWS = 8   # score rows the kernel ranks per pass over a segment (csrc/retrieval.cu RB)
TOPK_MAX_K = 1024     # PC_TOPK_MAX_K: the largest k the top-k kernels select
TOPK_WARP_K = 32      # k above this runs the buffered large-k selection (csrc/retrieval.cu WARP_K)
SPLIT_WS_BYTES = 256 << 20   # bound on the [rows, splits, k] (f64, i64) split lists chosen automatically for k > 32


def _check_k(k: int, what: str) -> None:
    if not 1 <= k <= TOPK_MAX_K:
        raise ValueError(f"{what}: k={k} outside [1, {TOPK_MAX_K}]")


def _auto_splits(units: int, avg_len: float, k: int = 1, rows: int = 0) -> int:
    sms = 148
    if units >= 2 * sms:
        return 1
    want = max(1, (2 * sms + units - 1) // max(units, 1))
    cap = max(1, int(avg_len // 256))
    if k > TOPK_WARP_K:
        # every split returns k entries per row: a split must rank many more than k products, and the lists stay bounded
        cap = min(cap, max(1, int(avg_len // (16 * k))), max(1, SPLIT_WS_BYTES // max(1, rows * k * 16)))
    return max(1, min(want, cap, 1024))


def topk_segments(q: torch.Tensor, catalog: torch.Tensor, seg_begin: torch.Tensor, seg_end: torch.Tensor, k: int,
                  members: Optional[torch.Tensor] = None, index_base: int = 0, splits: Optional[int] = None):
    """Exact top-k of every row over its run of catalog rows; returns (scores f64 [R,k], idx i64 [R,k]).
    Rows that rank the same run (same complementary type) are grouped, eight per pass (pc_topk_groups)."""
    _check_k(k, "topk_segments")
    rows, dim = q.shape
    dev_ = q.device
    out_s = torch.empty(rows, k, dtype=F64, device=dev_)
    out_i = torch.empty(rows, k, dtype=I64, device=dev_)
    if rows == 0:
        return out_s, out_i
    # index plumbing on [rows]-sized tensors: order rows by segment, cut runs into groups of <= 8
    key = seg_begin * (int(seg_end.max().item()) + 1) + seg_end
    order = torch.argsort(key, stable=True)
    skey = key[order]
    ar = torch.arange(rows, device=dev_)
    change = torch.ones(rows, dtype=torch.bool, device=dev_)
    change[1:] = skey[1:] != skey[:-1]
    run_start = torch.cummax(torch.where(change, ar, torch.zeros_like(ar)), 0).values
    new_group = change | ((ar - run_start) % TOPK_GROUP_ROWS == 0)
    starts = torch.nonzero(new_group).squeeze(1)
    n_groups = starts.numel()
    grp_begin = torch.cat([starts, torch.tensor([rows], device=dev_)]).to(I32).contiguous()
    g_beg = seg_begin[order][starts].contiguous()
    g_end = seg_end[order][starts].contiguous()
    row_ids = order.to(I32).contiguous()
    if splits is None:
        splits = _auto_splits(n_groups, float((g_end - g_beg).float().mean().item()), k, rows)
    ws = _lib.workspace(_lib.LIB.pc_topk_groups_workspace_bytes(rows, k, splits), dev_)
    call("pc_topk_groups", dev(q.contiguous(), F32, "q"), rows, dim, dev(catalog, F32, "catalog"),
         dev(members, I32, "members"), dev(row_ids, I32, "row_ids"), dev(grp_begin, I32, "grp_begin"),
         dev(g_beg, I64, "seg_begin"), dev(g_end, I64, "seg_end"), n_groups, k, splits, int(index_base),
         dev(out_s, F64, "out_scores"), dev(out_i, I64, "out_idx"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return out_s, out_i


def _by_type_splits(rows: int, n_types: int, catalog: torch.Tensor, members: Optional[torch.Tensor], k: int = 1) -> int:
    """Automatic splits of the device-grouped calls (topk_by_type, rank_by_type)."""
    # expected number of groups without looking at the data: distinct types hit + one more group per 8 rows
    n_cat = members.numel() if members is not None else catalog.shape[0]
    distinct = n_types * (1.0 - math.exp(-rows / max(n_types, 1)))
    return _auto_splits(int(distinct + rows / TOPK_GROUP_ROWS) + 1, n_cat / max(n_types, 1), k, rows)


def _exclusion_args(exclude, rows: int, what: str):
    """(excl_offsets, excl_idx, n_lists, row_list) pointers of a retrieval.Exclusions for `rows` score rows."""
    if exclude.row_list is not None and tuple(exclude.row_list.shape) != (rows,):
        raise ValueError(f"{what}: exclusion row_list {tuple(exclude.row_list.shape)} != ({rows},)")
    idx = exclude.indices
    if idx.numel() == 0:                        # every list is empty; the kernel still wants a valid pointer
        idx = torch.zeros(1, dtype=I64, device=idx.device)
    return (dev(exclude.offsets, I64, "excl_offsets"), dev(idx, I64, "excl_idx"), exclude.num_lists,
            dev(exclude.row_list, I32, "row_list"))


def topk_by_type(q: torch.Tensor, catalog: torch.Tensor, type_offsets: torch.Tensor, n_types: int,
                 row_type: Optional[torch.Tensor], k: int, members: Optional[torch.Tensor] = None, index_base: int = 0,
                 splits: Optional[int] = None, exclude=None):
    """Exact top-k of every row over the catalog rows of its type, grouping done on the device (pc_topk_by_type): no
    host synchronisation between the inputs and the result.  Returns (scores f64 [R,k], idx i64 [R,k]).
    exclude (retrieval.Exclusions of global indices): row r's list is left out of its ranking
    (pc_topk_by_type_excluding)."""
    _check_k(k, "topk_by_type")
    q = q.contiguous()
    rows, dim = q.shape
    out_s = torch.empty(rows, k, dtype=F64, device=q.device)
    out_i = torch.empty(rows, k, dtype=I64, device=q.device)
    if rows == 0:
        return out_s, out_i
    if splits is None:
        splits = _by_type_splits(rows, n_types, catalog, members, k)
    ws = _lib.workspace(_lib.LIB.pc_topk_by_type_workspace_bytes(rows, k, splits), q.device)
    if exclude is not None:
        call("pc_topk_by_type_excluding", dev(q, F32, "q"), rows, dim, dev(catalog, F32, "catalog"),
             dev(members, I32, "members"), dev(type_offsets, I64, "type_offsets"), int(n_types), dev(row_type, I32, "row_type"),
             k, splits, int(index_base), *_exclusion_args(exclude, rows, "topk_by_type"), dev(out_s, F64, "out_scores"),
             dev(out_i, I64, "out_idx"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
        return out_s, out_i
    call("pc_topk_by_type", dev(q, F32, "q"), rows, dim, dev(catalog, F32, "catalog"), dev(members, I32, "members"),
         dev(type_offsets, I64, "type_offsets"), int(n_types), dev(row_type, I32, "row_type"), k, splits, int(index_base),
         dev(out_s, F64, "out_scores"), dev(out_i, I64, "out_idx"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return out_s, out_i


def rank_by_type(q: torch.Tensor, catalog: torch.Tensor, type_offsets: torch.Tensor, n_types: int,
                 row_type: Optional[torch.Tensor], target_rows: torch.Tensor, target_idx: torch.Tensor,
                 members: Optional[torch.Tensor] = None, index_base: int = 0, splits: Optional[int] = None,
                 exclude=None, type_id: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Rank of each row's target among the catalog rows of the row's type (pc_rank_by_type): the number of products
    whose (score, global index) ranks strictly before (q[r] . target_rows[r], target_idx[r]); -1 for a row_type
    outside [0, n_types).  Membership of the target is the caller's: the kernel does not check it.  Returns int64 [R].
    exclude (retrieval.Exclusions of global indices): products of row r's list are not counted, the target itself
    excepted (pc_rank_remove_excluded after the count; type_id int32 [P] is the catalog's local type of each row and
    is needed with row_type)."""
    q = q.contiguous()
    rows, dim = q.shape
    target_rows = target_rows.contiguous()
    target_idx = target_idx.contiguous()
    if tuple(target_rows.shape) != (rows, dim):
        raise ValueError(f"rank_by_type: target_rows {tuple(target_rows.shape)} != queries {(rows, dim)}")
    if tuple(target_idx.shape) != (rows,):
        raise ValueError(f"rank_by_type: target_idx {tuple(target_idx.shape)} != ({rows},)")
    if row_type is not None and tuple(row_type.shape) != (rows,):
        raise ValueError(f"rank_by_type: row_type {tuple(row_type.shape)} != ({rows},)")
    out = torch.empty(rows, dtype=I64, device=q.device)
    if rows == 0:
        return out
    if splits is None:
        splits = _by_type_splits(rows, n_types, catalog, members)   # as topk_by_type for k <= 32
    ws = _lib.workspace(_lib.LIB.pc_rank_by_type_workspace_bytes(rows), q.device)
    call("pc_rank_by_type", dev(q, F32, "q"), rows, dim, dev(catalog, F32, "catalog"), dev(members, I32, "members"),
         dev(type_offsets, I64, "type_offsets"), int(n_types), dev(row_type, I32, "row_type"),
         dev(target_rows, F32, "target_rows"), dev(target_idx, I64, "target_idx"), splits, int(index_base),
         dev(out, I64, "out_rank"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    if exclude is not None:
        if row_type is not None and type_id is None:
            raise ValueError("rank_by_type: exclusions with row types need the catalog's type_id")
        call("pc_rank_remove_excluded", dev(q, F32, "q"), rows, dim, dev(catalog, F32, "catalog"), catalog.shape[0],
             dev(type_id if row_type is not None else None, I32, "type_id"), dev(row_type, I32, "row_type"),
             dev(target_rows, F32, "target_rows"), dev(target_idx, I64, "target_idx"), int(index_base),
             *_exclusion_args(exclude, rows, "rank_by_type"), dev(out, I64, "inout_rank"), stream())
    return out


def score_topk_dense(q: torch.Tensor, catalog: torch.Tensor, k: int, type_id: Optional[torch.Tensor] = None,
                     row_type: Optional[torch.Tensor] = None, index_base: int = 0, max_norm: Optional[float] = None,
                     units: Optional[int] = None):
    """Dense tensor-core scoring + mask + top-k (pc_score_topk_dense).  Returns (scores f64 [R,k], idx i64 [R,k],
    flags i32 [R]); flagged rows must be re-run on the exact path (topk_by_type)."""
    q = q.contiguous()
    rows, dim = q.shape
    if max_norm is None:
        max_norm = float(catalog.norm(dim=1).max().item())
    if units is None:
        m_blocks = (rows + 127) // 128
        n_tiles = (catalog.shape[0] + 127) // 128
        # a unit is (128-row block, product range); ~2 units per SM.  More, smaller units balance better but every
        # unit adds KP candidates per row to the exact re-scoring pass (measured: 20 units/SM is 30 % slower)
        units = max(1, min((2 * 148 + m_blocks - 1) // m_blocks, n_tiles, 4096))
    out_s = torch.empty(rows, k, dtype=F64, device=q.device)
    out_i = torch.empty(rows, k, dtype=I64, device=q.device)
    flags = torch.empty(rows, dtype=I32, device=q.device)
    ws = _lib.workspace(_lib.LIB.pc_score_topk_workspace_bytes(rows, units), q.device)
    call("pc_score_topk_dense", dev(q, F32, "q"), rows, dim, dev(catalog, F32, "catalog"), catalog.shape[0],
         dev(type_id, I32, "type_id"), dev(row_type, I32, "row_type"), k, units, int(index_base), float(max_norm),
         dev(out_s, F64, "out_scores"), dev(out_i, I64, "out_idx"), dev(flags, I32, "flags"), dev(ws, torch.uint8, "ws"),
         ws.numel(), stream())
    return out_s, out_i, flags


def topk_rows(values: torch.Tensor, k: int, splits: Optional[int] = None):
    """Row-wise top-k of a materialised fp32 matrix, ties -> lowest index (torch.topk replacement).  Columns past the
    end pad with (-inf, -1) when cols < k."""
    _check_k(k, "topk_rows")
    values = values.contiguous()
    rows, cols = values.shape
    if splits is None:
        splits = _auto_splits(rows, float(cols), k, rows)
    out_s = torch.empty(rows, k, dtype=F64, device=values.device)
    out_i = torch.empty(rows, k, dtype=I64, device=values.device)
    ws = _lib.workspace(_lib.LIB.pc_topk_rows_workspace_bytes(rows, k, splits), values.device)
    call("pc_topk_rows", dev(values, F32, "values"), rows, cols, k, splits, dev(out_s, F64, "out_scores"),
         dev(out_i, I64, "out_idx"), dev(ws, torch.uint8, "ws"), ws.numel(), stream())
    return out_s, out_i


def topk_merge(scores: torch.Tensor, idx: torch.Tensor, k: int):
    """Merge [R, lists*k] candidates -> [R, k] (per-shard merge, SURVEY 8e)."""
    _check_k(k, "topk_merge")
    rows, total = scores.shape
    lists = total // k
    out_s = torch.empty(rows, k, dtype=F64, device=scores.device)
    out_i = torch.empty(rows, k, dtype=I64, device=scores.device)
    call("pc_topk_merge", dev(scores.contiguous(), F64, "scores"), dev(idx.contiguous(), I64, "idx"), rows, lists, k,
         dev(out_s, F64, "out_scores"), dev(out_i, I64, "out_idx"), stream())
    return out_s, out_i


# --------------------------------------------------------------------------- halo helpers
def rows_gather(table: torch.Tensor, index: torch.Tensor) -> torch.Tensor:
    out = torch.empty(index.numel(), table.shape[1], dtype=F32, device=table.device)
    call("pc_rows_gather", dev(table, F32, "table"), dev(index, I64, "index"), index.numel(), table.shape[1],
         dev(out, F32, "out"), stream())
    return out


def rows_scatter_add_(table: torch.Tensor, index: torch.Tensor, rows: torch.Tensor) -> torch.Tensor:
    """table[index] += rows; `index` must hold unique ids (deterministic, no atomics)."""
    call("pc_rows_scatter_add", dev(rows.contiguous(), F32, "rows"), dev(index, I64, "index"), index.numel(),
         table.shape[1], dev(table, F32, "table"), stream())
    return table


def rows_reduce_peers_(table: torch.Tensor, rows: torch.Tensor, slot: torch.Tensor) -> torch.Tensor:
    """table[r] += sum_p rows[slot[p, r]] over the peers p in ascending order (slot < 0: nothing from p)."""
    world, n = slot.shape
    if table.shape[0] != n or not table.is_contiguous():
        raise ValueError("rows_reduce_peers_: table must be a contiguous [n, width] tensor matching slot [world, n]")
    if rows.numel() == 0:
        return table
    call("pc_rows_reduce_peers", dev(rows.contiguous(), F32, "rows"), dev(slot, I32, "slot"), world, n, table.shape[1],
         dev(table, F32, "table"), stream())
    return table
