"""Drop-in operator / model API (the torch-geometric surface the reference uses).

Mirrors, name for name, what reference src/classes.py imports and calls:
    torch_geometric.nn: TopKPooling, SAGEConv, global_mean_pool (gap), global_max_pool (gmp)
                                                      # src/classes.py:1-2
    class Net_1(torch.nn.Module)                      # src/classes.py:45-82
Same constructor arguments, same state-dict keys and shapes (SURVEY 0.2: conv*.weight [in,128],
conv*.bias [128], pool*.weight [1,128], lin*.weight/bias), same forward signatures and return
tuples, Python exceptions on misuse.  Every forward/backward runs hand-written CUDA kernels
through libnpi; CPU tensors raise (there is no CPU fallback).
"""
from __future__ import annotations

import math

import torch
from torch import nn

from . import _lib as L
from . import ops
from .engine import Engine, FlatParams, param_spec

H = 128


def _i32(t):
    return t.to(torch.int32).contiguous()


def _csr_of(edge_index, N, check_symmetric=True):
    """CSR by destination of a PyG edge_index (self loops dropped, edge order kept per row).

    The backward kernels use this CSR as its own transpose (the reference's enclosing subgraphs list
    every edge in both directions, src/classes.py:697-704), so an edge_index whose multiset of edges
    is not symmetric would give a right forward pass and WRONG gradients: it is rejected here."""
    L.require_cuda(edge_index)
    E = edge_index.shape[1]
    ei = edge_index.to(torch.int64).contiguous()
    sums = ops.edge_symmetry_sums(ei) if (check_symmetric and E > 0) else None
    rowptr = torch.empty(N + 1, dtype=torch.int32, device=edge_index.device)
    col = torch.empty(max(E, 1), dtype=torch.int32, device=edge_index.device)
    ops.coo_to_csr(ei, N, rowptr, col)
    if sums is not None:
        a, b = sums.tolist()
        if a != b:
            raise L.NPIError("edge_index is not symmetric (some edge (i,j) lacks its reverse (j,i)): the NPI-GNN kernels "
                             "implement SAGEConv / TopKPooling for undirected graphs given in both directions, like the "
                             "reference's enclosing subgraphs")
    return rowptr, col


def _graph_ptr_of(batch, N, device, num_graphs=None, size=None):
    """graph_ptr from a sorted PyG batch vector (one host sync: B = batch.max()+1, like PyG -- skipped when the
    batch object carries ``num_graphs``, as PyG's ``Batch`` and this package's loaders do).  The kernels take each
    graph's rows as one contiguous range, so the same sync also checks that ``batch`` is sorted.  ``size``: number
    of graphs (PyG's ``size`` argument); graphs with no rows, in a gap of ``batch`` or past its end, are empty."""
    if batch is None:
        return torch.tensor([0, N], dtype=torch.int32, device=device)
    if num_graphs is not None:
        B = int(num_graphs)
    elif N > 0:
        top, unsorted = torch.stack([batch.max(), (batch[1:] < batch[:-1]).any().to(batch.dtype)]).tolist()
        if unsorted:
            raise L.NPIError("batch must be sorted (the rows of each graph contiguous, graphs in increasing order), "
                             "as PyG's Batch builds it")
        B = top + 1
    else:
        B = 0
    if size is not None:
        if size < B:
            raise L.NPIError("size=%d is smaller than batch.max()+1 = %d" % (size, B))
        B = int(size)
    counts = torch.bincount(batch, minlength=B)
    gp = torch.zeros(B + 1, dtype=torch.int32, device=device)
    gp[1:] = torch.cumsum(counts, 0).to(torch.int32)
    return gp


# =========================================================================================== SAGEConv
class _SAGEConvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, rowptr, col):
        L.require_cuda(x, weight)
        x = x.contiguous().float()
        N = x.shape[0]
        out = torch.empty(N, H, dtype=torch.float32, device=x.device)
        w = weight.contiguous()
        b = None if bias is None else bias.contiguous()
        ops.sage_fwd(L.features_dense(x), rowptr, col, None, N, w, b, False, None, out, None, None)
        ctx.save_for_backward(x, w, rowptr, col)
        ctx.has_bias = bias is not None
        return out

    @staticmethod
    def backward(ctx, g):
        x, w, rowptr, col = ctx.saved_tensors
        g = g.contiguous().float()
        N, Fin = x.shape
        dW = torch.empty_like(w)
        db = torch.empty(H, dtype=torch.float32, device=x.device)
        ws = torch.empty(ops.sage_bwd_weight_workspace_bytes(Fin), dtype=torch.uint8, device=x.device)
        ops.sage_bwd_weight(L.features_dense(x), rowptr, col, None, None, N, g, dW, db, ws)
        dx = None
        if ctx.needs_input_grad[0]:
            if Fin != H:
                raise L.NPIError("SAGEConv input gradient is implemented for in_channels == 128 only")
            dx = torch.empty(N, H, dtype=torch.float32, device=x.device)
            ops.sage_bwd_input(g, None, rowptr, col, None, N, w, dx)
        return dx, dW, (db if ctx.has_bias else None), None, None


class SAGEConv(nn.Module):
    """torch-geometric 1.4.x ``SAGEConv(in_channels, out_channels)`` (aggr='mean', bias=True):
    out = mean_{j in N(i) U {i}} x_j . weight + bias, ONE weight [in,out] (SURVEY 0.2, A.2)."""

    def __init__(self, in_channels, out_channels, normalize=False, concat=False, bias=True, **kwargs):
        super().__init__()
        if out_channels != H:
            raise L.NPIError("this build implements SAGEConv with out_channels == 128 (Net_1's width), got %d" % out_channels)
        if normalize or concat:
            raise L.NPIError("normalize/concat are not used by the reference and not implemented")
        if not (1 <= in_channels <= 256):
            raise L.NPIError("in_channels must be in [1,256]")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = nn.Parameter(torch.empty(out_channels)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        b = 1.0 / math.sqrt(self.in_channels)          # PyG uniform(size=in_channels, tensor)
        nn.init.uniform_(self.weight, -b, b)
        if self.bias is not None:
            nn.init.uniform_(self.bias, -b, b)

    def forward(self, x, edge_index, edge_weight=None, size=None):
        if edge_weight is not None:
            raise L.NPIError("edge_weight is not used by the reference and not implemented")
        rowptr, col = _csr_of(edge_index, x.shape[0])
        return _SAGEConvFn.apply(x, self.weight, self.bias, rowptr, col)

    def __repr__(self):
        return "SAGEConv(%d, %d)" % (self.in_channels, self.out_channels)


# =========================================================================================== TopKPooling
class _TopKFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, gptr_in, gptr_out, max_n):
        L.require_cuda(x, weight)
        x = x.contiguous().float()
        N, dev = x.shape[0], x.device
        B = gptr_in.numel() - 1
        Np = int(gptr_out[-1].item())
        w = weight.contiguous().view(-1)
        z = torch.empty(N, dtype=torch.float32, device=dev)
        s = torch.empty(N, dtype=torch.float32, device=dev)
        ops.topk_score(x, None, N, w, z, s)
        perm = torch.empty(Np, dtype=torch.int32, device=dev)
        new_id = torch.empty(N, dtype=torch.int32, device=dev)
        batch_out = torch.empty(Np, dtype=torch.int32, device=dev)
        ws = torch.empty(max(16, ops.topk_select_workspace_bytes(B, max_n)), dtype=torch.uint8, device=dev)
        ops.topk_select(s, gptr_in, gptr_out, B, max_n, perm, new_id, batch_out, ws)
        xp = torch.empty(Np, H, dtype=torch.float32, device=dev)
        ro = torch.empty(B, 2 * H, dtype=torch.float32, device=dev)
        ops.pool_gate_readout(x, s, perm, gptr_out, B, xp, ro, False, None)
        score_perm = s[perm.long()]
        ctx.save_for_backward(x, w, z, s, perm, batch_out, gptr_out)
        ctx.mark_non_differentiable(perm, new_id, batch_out)
        return xp, score_perm, perm, new_id, batch_out

    @staticmethod
    def backward(ctx, g_xp, g_score, *unused):
        x, w, z, s, perm, batch_out, gptr_out = ctx.saved_tensors
        dev = x.device
        N, Np, B = x.shape[0], perm.numel(), gptr_out.numel() - 1
        g_xp = torch.zeros(Np, H, device=dev) if g_xp is None else g_xp.contiguous().float()
        if g_score is not None and bool((g_score != 0).any()):
            raise L.NPIError("gradient through TopKPooling's returned score is not implemented (Net_1 discards it)")
        d_ro = torch.zeros(B, 2 * H, device=dev)
        argmax = torch.full((B, H), -1, dtype=torch.int32, device=dev)
        dpre = torch.empty(Np, H, device=dev)
        d_w = torch.empty(H, device=dev)
        ws = torch.empty(ops.pool_bwd_workspace_bytes(), dtype=torch.uint8, device=dev)
        ops.pool_bwd(g_xp, d_ro, x, z, s, perm, batch_out, argmax, gptr_out, None, Np, B, w, False, dpre, d_w, ws)
        dx = torch.zeros(N, H, device=dev)
        dx[perm.long()] = dpre                       # scatter of distinct rows (plumbing)
        return dx, d_w.view(1, H), None, None, None


class TopKPooling(nn.Module):
    """torch-geometric 1.4.2 ``TopKPooling(in_channels, ratio=0.5)`` (min_score=None, multiplier=1,
    nonlinearity=tanh; SURVEY A.3).  forward returns the reference's 6-tuple
    (x', edge_index', edge_attr', batch', perm, score[perm])  (src/classes.py:63)."""

    def __init__(self, in_channels, ratio=0.5, min_score=None, multiplier=1, nonlinearity=torch.tanh):
        super().__init__()
        if in_channels != H:
            raise L.NPIError("this build implements TopKPooling with in_channels == 128 (Net_1's width), got %d" % in_channels)
        if min_score is not None or multiplier != 1 or nonlinearity is not torch.tanh:
            raise L.NPIError("only the reference's TopKPooling configuration (tanh, multiplier 1, no min_score) is implemented")
        self.in_channels, self.ratio = in_channels, ratio
        self.weight = nn.Parameter(torch.empty(1, in_channels))
        self.reset_parameters()

    def reset_parameters(self):
        b = 1.0 / math.sqrt(self.in_channels)
        nn.init.uniform_(self.weight, -b, b)

    def forward(self, x, edge_index, edge_attr=None, batch=None, attn=None):
        if edge_attr is not None or attn is not None:
            raise L.NPIError("edge_attr/attn are not used by the reference and not implemented")
        L.require_cuda(x, edge_index)
        N, dev = x.shape[0], x.device
        gp_in = _graph_ptr_of(batch, N, dev)
        n = (gp_in[1:] - gp_in[:-1])
        k = torch.ceil(torch.tensor(self.ratio, dtype=torch.float32, device=dev) * n.to(torch.float32)).to(torch.int32)
        gp_out = torch.zeros_like(gp_in)
        gp_out[1:] = torch.cumsum(k, 0).to(torch.int32)
        max_n = int(n.max().item()) if n.numel() else 2
        xp, score_perm, perm, new_id, batch_out = _TopKFn.apply(x, self.weight, gp_in, gp_out, max(max_n, 2))
        E = edge_index.shape[1]
        ei = edge_index.to(torch.int64).contiguous()
        out = torch.empty(2, max(E, 1), dtype=torch.int64, device=dev)
        cnt = torch.zeros(1, dtype=torch.int32, device=dev)
        ops.filter_edges_coo(ei, new_id, out, cnt) if E > 0 else None
        Ep = int(cnt.item())
        bo = batch_out.long() if batch is not None else torch.zeros(perm.numel(), dtype=torch.long, device=dev)
        return xp, out[:, :Ep], None, bo, perm.long(), score_perm

    def __repr__(self):
        return "TopKPooling(%d, ratio=%s)" % (self.in_channels, self.ratio)


# =========================================================================================== global pools
class _GlobalPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gptr, batch32, use_max):
        L.require_cuda(x)
        x = x.contiguous().float()
        if x.shape[1] != H:
            raise L.NPIError("global pooling kernels are built for 128 channels")
        N, dev = x.shape[0], x.device
        B = gptr.numel() - 1
        ident = torch.arange(N, dtype=torch.int32, device=dev)
        ones = torch.ones(N, dtype=torch.float32, device=dev)
        scratch = torch.empty(N, H, dtype=torch.float32, device=dev)
        ro = torch.empty(B, 2 * H, dtype=torch.float32, device=dev)
        argmax = torch.empty(B, H, dtype=torch.int32, device=dev)
        ops.pool_gate_readout(x, ones, ident, gptr, B, scratch, ro, False, argmax)
        ctx.save_for_backward(gptr, batch32, argmax)
        ctx.use_max, ctx.N = use_max, N
        return ro[:, :H].clone() if use_max else ro[:, H:].clone()

    @staticmethod
    def backward(ctx, g):
        gptr, batch32, argmax = ctx.saved_tensors
        B = gptr.numel() - 1
        d_ro = torch.zeros(B, 2 * H, dtype=torch.float32, device=g.device)
        if ctx.use_max:
            d_ro[:, :H] = g
        else:
            d_ro[:, H:] = g
        dx = torch.empty(ctx.N, H, dtype=torch.float32, device=g.device)
        ops.readout_bwd(d_ro, argmax, gptr, batch32, ctx.N, ctx.use_max, not ctx.use_max, dx)
        return dx, None, None, None


def global_max_pool(x, batch, size=None):
    """PyG 1.4.2 ``global_max_pool``: [size or batch.max()+1, 128]; an empty graph gives 0.  ``batch`` must be sorted."""
    gp = _graph_ptr_of(batch, x.shape[0], x.device, size=size)
    return _GlobalPoolFn.apply(x, gp, _i32(batch), True)


def global_mean_pool(x, batch, size=None):
    """PyG 1.4.2 ``global_mean_pool``: [size or batch.max()+1, 128]; an empty graph gives 0.  ``batch`` must be sorted."""
    gp = _graph_ptr_of(batch, x.shape[0], x.device, size=size)
    return _GlobalPoolFn.apply(x, gp, _i32(batch), False)


# =========================================================================================== Net_1
class _Net1Fn(torch.autograd.Function):
    """Whole-network forward/backward on the fused engine; the autograd tape only sees one node."""

    @staticmethod
    def forward(ctx, flat, net, training):
        eng = net._engine
        params = FlatParams(net.num_node_features, flat.device, flat=flat.detach().contiguous())
        net._fwd_calls += 1
        logp = eng.forward(params, training=training, seed=net._seed, sample_id_base=net._fwd_calls * 1000003)
        ctx.net, ctx.params = net, params
        ctx.engine, ctx.generation = eng, net._fwd_calls      # the engine keeps ONE batch's activations
        return logp.clone()

    @staticmethod
    def backward(ctx, g):
        net, eng = ctx.net, ctx.net._engine
        if eng is not ctx.engine or net._fwd_calls != ctx.generation:
            raise L.NPIError("Net_1.backward: another forward ran on this model since the output being differentiated "
                             "(the fused engine keeps the activations of its LAST forward only); call loss.backward() "
                             "before the next model(data), as the reference's train() does (src/train_with_twoDataset.PY:52-56)")
        grads = FlatParams(net.num_node_features, g.device)
        eng.backward(ctx.params, grads, d_logp=g.contiguous().float())
        return grads.flat, None, None


class Net_1(nn.Module):
    """Drop-in for the reference's ``Net_1(num_node_features, num_of_classes=2)``
    (src/classes.py:45-82).  ``forward(data)`` reads data.x / data.edge_index / data.batch like the
    reference; batches produced by this package's DataLoader carry the GPU extractor's CSR and
    skip the dense x entirely.  The 15 parameters keep the reference's names and shapes, so
    ``model.load_state_dict(torch.load(path))`` works on the shipped checkpoints."""

    def __init__(self, num_node_features, num_of_classes=2):
        super().__init__()
        if num_of_classes != 2:
            raise L.NPIError("the fused head implements the reference's 2-class output")
        self.num_node_features = num_node_features
        self.conv1 = SAGEConv(num_node_features, 128)
        self.pool1 = TopKPooling(128, ratio=0.5)
        self.conv2 = SAGEConv(128, 128)
        self.pool2 = TopKPooling(128, ratio=0.5)
        self.conv3 = SAGEConv(128, 128)
        self.pool3 = TopKPooling(128, ratio=0.5)
        self.lin1 = nn.Linear(256, 128)
        self.lin2 = nn.Linear(128, 64)
        self.lin3 = nn.Linear(64, num_of_classes)
        self._engine = None
        self._seed = int(torch.initial_seed() & 0x7FFFFFFFFFFFFFFF)
        self._fwd_calls = 0

    def _flat(self):
        sd = dict(self.named_parameters())
        return torch.cat([sd[name].reshape(-1) for name, _ in param_spec(self.num_node_features)])

    def _ensure_engine(self, B, n0, e0, max_n, graph, device):
        e = self._engine
        if (e is None or e.B < B or e.n_cap[0] < n0 or e.e_cap < e0 or e.max_graph_nodes < max_n or e.device != device
                or (graph is not None and e.V != graph.num_nodes)):
            grow = lambda v: int(v * 1.25) + 16
            self._engine = Engine(self.num_node_features, max(B, e.B if e else 0), grow(n0), grow(e0), grow(max_n),
                                  device=device, graph=graph)
        return self._engine

    def forward(self, data):
        dev = self.conv1.weight.device
        if dev.type != "cuda":
            raise L.NPIError("Net_1 runs on CUDA only (model.to('cuda')); there is no CPU fallback")
        nb = getattr(data, "_npi", None)
        if nb is not None:                       # batch from this package's DataLoader: GPU extraction
            ps, idx = nb.pairset, nb.index_dev
            n0, e0, mx = nb.caps
            eng = self._ensure_engine(len(nb), n0, e0, mx, ps.graph, dev)
            eng.load_pairs(ps, count=len(nb), pair_index=idx)
        else:                                    # foreign PyG-style batch: dense x + COO edge_index
            x, ei = data.x, data.edge_index
            L.require_cuda(x, ei)
            if x.shape[1] != self.num_node_features:
                raise L.NPIError("data.x has %d features, model expects %d" % (x.shape[1], self.num_node_features))
            N = x.shape[0]
            batch = getattr(data, "batch", None)
            gp = _graph_ptr_of(batch, N, dev, getattr(data, "num_graphs", None))
            rowptr, col = _csr_of(ei, N)
            n = gp[1:] - gp[:-1]
            eng = self._ensure_engine(gp.numel() - 1, N, ei.shape[1], int(n.max().item()), None, dev)
            eng.set_csr_batch(x.float(), rowptr, col[:ei.shape[1]], gp, getattr(data, "y", None))
        return _Net1Fn.apply(self._flat(), self, self.training)
