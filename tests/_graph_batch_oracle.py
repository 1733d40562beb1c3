"""Reference helpers for tests/test_gpu_graph_training.py: the triplet batch gathered with torch indexing, and the
graph-native training step restated in float64 (numpy oracle for the loss and the BatchNorm running statistics, torch
autograd of the reference port for the parameter gradients)."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import p2v


def batch_rows_reference(x, rowptr, col, anchor, positive, negatives):
    """(rows, nbr_ptr, edge_row) of pc_triplet_batch_rows by torch indexing: anchors | neighbours | positives | negatives."""
    deg = rowptr[anchor + 1] - rowptr[anchor]
    nbr_ptr = torch.zeros(anchor.numel() + 1, dtype=torch.int64, device=x.device)
    nbr_ptr[1:] = torch.cumsum(deg, 0)
    e = int(nbr_ptr[-1])
    edges = torch.repeat_interleave(rowptr[anchor] - nbr_ptr[:-1], deg, output_size=e) + torch.arange(e, device=x.device)
    nbr = col[edges].long()
    rows = torch.cat([x[anchor], x[nbr], x[positive], x[negatives.reshape(-1)]])
    edge_row = torch.repeat_interleave(torch.arange(anchor.numel(), device=x.device), deg).to(torch.int32)
    return rows, nbr_ptr, edge_row


def _neighbour_lists(rowptr, col, anchor):
    return [col[rowptr[a]:rowptr[a + 1]] for a in anchor]


def step_reference_f64(sd, x, rowptr, col, anchor, positive, negatives, heads, margin):
    """Loss and running statistics of one graph-native step in float64 with oracle/p2v.py: ffn(anchors),
    ffn(neighbour rows), ffn(positives), ffn(negatives) in that order, statistics threaded through the four calls,
    attention over each anchor's real neighbours (anchors without any keep ffn(x))."""
    p = {k: np.asarray(v, np.float64) for k, v in sd.items()}

    def ffn(rows):
        y, (rm, rv) = p2v.ffn(p, rows, training=True)
        p["ffn.1.running_mean"], p["ffn.1.running_var"] = rm, rv
        return y

    lists = _neighbour_lists(rowptr, col, anchor)
    h_a = ffn(x[anchor])
    nbr = np.concatenate(lists) if lists else np.zeros(0, np.int64)
    if nbr.size:
        h_n = ffn(x[nbr])
        ptr = np.zeros(len(anchor) + 1, np.int64)
        np.cumsum([len(l) for l in lists], out=ptr[1:])
        q, kv = p2v.in_projection(p, h_a, h_n)
        o, _ = p2v.gat_csr_forward(q, kv, ptr, np.arange(nbr.size), heads)
        out = p2v.linear(o, p["attention.out_proj.weight"], p["attention.out_proj.bias"])
        h_a = np.where((np.diff(ptr) > 0)[:, None], out, h_a)
    h_p = ffn(x[positive])
    h_n = ffn(x[negatives.reshape(-1)]).reshape(negatives.shape[0], negatives.shape[1], -1)
    loss, _ = p2v.triplet_hinge(h_a, h_p, h_n, margin)
    return loss, p["ffn.1.running_mean"], p["ffn.1.running_var"]


def step_grads_f64(port, x, rowptr, col, anchor, positive, negatives, margin):
    """Parameter gradients of the same step by float64 autograd of oracle.torch_port.PortProduct2Vec (train mode)."""
    xt = torch.as_tensor(x, dtype=torch.float64)
    lists = _neighbour_lists(rowptr, col, anchor)
    h_a = port.embed(xt[anchor])
    nbr = np.concatenate(lists) if lists else np.zeros(0, np.int64)
    if nbr.size:
        h_n = port.embed(xt[nbr])
        rows, s = [], 0
        for i, l in enumerate(lists):
            rows.append(port.attend(h_a[i:i + 1], h_n[s:s + len(l)].unsqueeze(0))[0] if len(l) else h_a[i])
            s += len(l)
        h_a = torch.stack(rows)
    h_p = port.embed(xt[positive])
    h_n = port.embed(xt[negatives.reshape(-1)]).reshape(negatives.shape[0], negatives.shape[1], -1)
    dpos = F.pairwise_distance(h_a, h_p)
    dneg = F.pairwise_distance(h_a.unsqueeze(1).expand(-1, h_n.size(1), -1), h_n).mean(dim=1)
    loss = F.relu(margin - dpos + dneg).mean()
    port.zero_grad()
    loss.backward()
    return {k: v.grad.numpy() for k, v in port.named_parameters()}
