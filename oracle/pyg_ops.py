"""Stock-PyTorch restatement of the torch-geometric 1.4.2 operators used by ``Net_1``
(oracle; test infrastructure only).

torch-geometric 1.4.2 / torch 1.4.0 (README.md:7-11 of the reference) are third-party,
not vendored under /root/reference and not installable here (no Python-3.12 build), so the
published algorithm of that release is restated (SURVEY.md Appendix A) and anchored on the
reference's call sites: construction src/classes.py:48-57, calls src/classes.py:62-80.
The restatement is PINNED by the shipped checkpoints + logs + case-study lists
(tests/test_oracle_kat.py): five confusion matrices and two name lists reproduce exactly.

Everything is differentiable by autograd, dtype-generic (fp32 / fp64).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def add_remaining_self_loops(edge_index, num_nodes):
    """PyG 1.4.2 ``add_remaining_self_loops`` with no edge weights: existing self loops are
    removed and one (i,i) per node is appended AFTER the real edges (Appendix A.2)."""
    row, col = edge_index[0], edge_index[1]
    keep = row != col
    loop = torch.arange(num_nodes, dtype=edge_index.dtype, device=edge_index.device)
    return torch.stack([torch.cat([row[keep], loop]), torch.cat([col[keep], loop])])


def scatter_mean(src, index, dim_size):
    out = torch.zeros((dim_size,) + src.shape[1:], dtype=src.dtype, device=src.device)
    out = out.index_add(0, index, src)
    cnt = torch.zeros(dim_size, dtype=src.dtype, device=src.device)
    cnt = cnt.index_add(0, index, torch.ones_like(index, dtype=src.dtype))
    cnt = cnt.clamp(min=1)
    return out / cnt.view(-1, *([1] * (src.dim() - 1)))


def sage_conv(x, edge_index, weight, bias):
    """SAGEConv of PyG 1.4.x (aggr='mean', concat=False, normalize=False): ONE weight
    [in,out] + bias; mean over (neighbours U self); flow source_to_target: x_j = x[edge_index[0]]
    aggregated at edge_index[1]  (Appendix A.2; src/classes.py:48,62)."""
    n = x.shape[0]
    ei = add_remaining_self_loops(edge_index, n)
    agg = scatter_mean(x[ei[0]], ei[1], n)
    out = agg @ weight
    if bias is not None:
        out = out + bias
    return out


def topk_perm(score, ratio, batch, num_graphs=None):
    """PyG 1.4.2 ``topk``: scores are scattered into a dense [B, max_n] matrix padded with -2
    (below any tanh score), each row is sorted descending and the first k = ceil(ratio*n)
    (float32 arithmetic) entries are kept; graphs concatenated in order.  torch 1.4's sort
    leaves tie order unspecified; this build fixes it as stable = lower node index first
    (Appendix A.3)."""
    if num_graphs is None:
        num_graphs = int(batch.max()) + 1 if batch.numel() else 0
    score = score.detach()
    num_nodes = torch.zeros(num_graphs, dtype=torch.long).index_add(0, batch, torch.ones_like(batch))
    max_n = int(num_nodes.max()) if num_graphs else 0
    cum = torch.cat([num_nodes.new_zeros(1), num_nodes.cumsum(0)[:-1]])
    index = torch.arange(batch.numel()) - cum[batch] + batch * max_n
    dense = score.new_full((num_graphs * max_n,), -2.0)
    dense[index] = score
    order = torch.sort(dense.view(num_graphs, max_n), dim=-1, descending=True, stable=True)[1]
    order = order + cum.view(-1, 1)
    k = (torch.tensor(ratio, dtype=torch.float32) * num_nodes.to(torch.float32)).ceil().to(torch.long)
    keep = torch.arange(max_n).view(1, -1) < k.view(-1, 1)
    return order[keep]


def filter_adj(edge_index, perm, num_nodes):
    """PyG 1.4.2 ``filter_adj``: relabel by perm, drop edges with a dropped endpoint, keep order."""
    mask = perm.new_full((num_nodes,), -1)
    mask[perm] = torch.arange(perm.numel(), dtype=perm.dtype)
    row, col = mask[edge_index[0]], mask[edge_index[1]]
    keep = (row >= 0) & (col >= 0)
    return torch.stack([row[keep], col[keep]])


def topk_pooling(x, edge_index, batch, weight, ratio=0.5, forced_perm=None):
    """TopKPooling(in, ratio) with min_score=None, multiplier=1, nonlinearity=tanh
    (Appendix A.3; src/classes.py:49,63).  Returns the reference's 6-tuple."""
    score = (x * weight).sum(dim=-1)
    score = torch.tanh(score / weight.norm(p=2, dim=-1))
    perm = topk_perm(score, ratio, batch) if forced_perm is None else forced_perm
    xo = x[perm] * score[perm].view(-1, 1)
    bo = batch[perm]
    eo = filter_adj(edge_index, perm, x.shape[0])
    return xo, eo, None, bo, perm, score[perm]


def global_max_pool(x, batch, num_graphs=None):
    """Segment max; a graph with no rows gives 0 (PyG's scatter_ replaces the empty max fill with 0)."""
    if num_graphs is None:
        num_graphs = int(batch.max()) + 1
    out = torch.full((num_graphs, x.shape[1]), float("-inf"), dtype=x.dtype)
    idx = batch.view(-1, 1).expand(-1, x.shape[1])
    out = out.scatter_reduce(0, idx, x, reduce="amax", include_self=True)
    empty = torch.bincount(batch, minlength=num_graphs) == 0
    return torch.where(empty.view(-1, 1), torch.zeros_like(out), out)


def global_mean_pool(x, batch, num_graphs=None):
    if num_graphs is None:
        num_graphs = int(batch.max()) + 1
    return scatter_mean(x, batch, num_graphs)


def adam_l2_step(params, grads, m, v, step, lr, wd=1e-3, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam(lr, weight_decay) of torch 1.4 (Appendix A.6;
    src/train_with_twoDataset.PY:130): L2 added to the gradient, bias-corrected moments,
    denom = sqrt(v)/sqrt(1-b2^t) + eps.  In place on lists of tensors; ``step`` is 1-based."""
    bc1 = 1 - b1 ** step
    bc2 = 1 - b2 ** step
    for p, g, mi, vi in zip(params, grads, m, v):
        g = g + wd * p
        mi.mul_(b1).add_(g, alpha=1 - b1)
        vi.mul_(b2).addcmul_(g, g, value=1 - b2)
        denom = (vi.sqrt() / math.sqrt(bc2)).add_(eps)
        p.addcdiv_(mi, denom, value=-lr / bc1)
