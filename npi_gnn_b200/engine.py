"""Fused Net_1 engine: batch assembly + extraction + forward + backward + Adam on one stream.

The kernel sequence mirrors reference src/classes.py:59-82 (Net_1.forward) and the training step
of src/train_with_twoDataset.PY:46-57, with every data-dependent size kept on the device (no
``.item()``, no host sync), so a whole step can be captured in one CUDA graph and replayed.
PyTorch only provides memory, streams and (optionally) the autograd tape.
"""
from __future__ import annotations

import math
import os

import numpy as np
import torch

from . import _lib as L
from . import ops

# NVTX ranges per phase of a step (SURVEY 5: tracing).  Host-side annotations around the launches of a phase -- what an
# nsys / ncu --nvtx timeline groups by; enabled with NPI_NVTX=1 (a no-op context manager otherwise).
_NVTX = os.environ.get("NPI_NVTX", "0") == "1"
_STAMPS = os.environ.get("NPI_STAMPS", "0") == "1"
# hub queue / row order of the filtered CSRs inside filter_adj's kernels (three launches on the chain the next aggregation
# waits for instead of five) for batches of up to this many rows only -- 0.247 -> 0.240 ms on RPI2241 (3 k rows), but
# 0.677 -> 0.684 ms at 215 k rows, where the count kernel's hub rows write their segment lists inside the sweep
SMALL_BATCH_ROWS = 65536


class _Range:
    __slots__ = ("name",)

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if _NVTX:
            torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        if _NVTX:
            torch.cuda.nvtx.range_pop()
        return False


def nvtx_range(name):
    return _Range(name)


def _nvtx_push(name):
    if _NVTX:
        torch.cuda.nvtx.range_push(name)


def _nvtx_pop():
    if _NVTX:
        torch.cuda.nvtx.range_pop()

H = 128
RATIO = 0.5
# small-subgraph path (csrc/tiny.cu): ONE launch takes every subgraph of the batch through the three layers (a CTA per subgraph)
# when no subgraph has more than ops.tiny_max_nodes() nodes and the batch averages at most TINY_MEAN_NODES rows per subgraph
# (RPI2241: 15); NPI_TINY=0 / 1 forces the per-layer path / the per-subgraph path wherever it is applicable
TINY_MEAN_NODES = 64
TINY_W1_DIRECT_ROWS = 16384
SMALL_TABLE_ROWS = 32768      # feature tables up to this many rows take the two-launch SIMT weight gradient (ops.table_grad)

# flat parameter layout == state_dict order of the reference's Net_1 (SURVEY 0.2)
def param_spec(F):
    return [("conv1.weight", (F, H)), ("conv1.bias", (H,)), ("pool1.weight", (1, H)),
            ("conv2.weight", (H, H)), ("conv2.bias", (H,)), ("pool2.weight", (1, H)),
            ("conv3.weight", (H, H)), ("conv3.bias", (H,)), ("pool3.weight", (1, H)),
            ("lin1.weight", (128, 256)), ("lin1.bias", (128,)),
            ("lin2.weight", (64, 128)), ("lin2.bias", (64,)),
            ("lin3.weight", (2, 64)), ("lin3.bias", (2,))]


def param_offsets(F):
    offs, o = {}, 0
    for name, shp in param_spec(F):
        n = int(np.prod(shp))
        offs[name] = (o, n, shp)
        o += n
    return offs, o


class FlatParams:
    """One flat fp32 buffer for the 15 tensors (97,602 floats at F=178) + views."""

    def __init__(self, F, device, flat=None):
        self.F = F
        self.offsets, self.total = param_offsets(F)
        self.flat = torch.zeros(self.total, dtype=torch.float32, device=device) if flat is None else flat
        assert self.flat.numel() == self.total

    def view(self, name, flat=None):
        o, n, shp = self.offsets[name]
        return (self.flat if flat is None else flat)[o:o + n].view(shp)

    def views(self, flat=None):
        return {name: self.view(name, flat) for name in self.offsets}

    def init_reference(self, generator=None):
        """PyG-1.4.2 / torch.nn.Linear default initialisation (Appendix A.2/A.3/A.5)."""
        g = generator
        def uni(t, bound):
            t.copy_((torch.rand(t.shape, generator=g, dtype=torch.float32) * 2 - 1) * bound)
        cpu = torch.zeros(self.total, dtype=torch.float32)
        v = self.views(cpu)
        for l, fin in ((1, self.F), (2, H), (3, H)):
            uni(v["conv%d.weight" % l], 1.0 / math.sqrt(fin))
            uni(v["conv%d.bias" % l], 1.0 / math.sqrt(fin))
            uni(v["pool%d.weight" % l], 1.0 / math.sqrt(H))
        for nm, fin in (("lin1", 256), ("lin2", 128), ("lin3", 64)):
            uni(v[nm + ".weight"], 1.0 / math.sqrt(fin))      # kaiming_uniform(a=sqrt(5)) == U(+-1/sqrt(fan_in))
            uni(v[nm + ".bias"], 1.0 / math.sqrt(fin))
        self.flat.copy_(cpu)
        return self

    def load_state_dict(self, sd):
        cpu = torch.zeros(self.total, dtype=torch.float32)
        v = self.views(cpu)
        for name in self.offsets:
            t = sd[name]
            if tuple(t.shape) != tuple(v[name].shape):
                raise L.NPIError("state_dict[%s] has shape %s, expected %s" % (name, tuple(t.shape), tuple(v[name].shape)))
            v[name].copy_(t.detach().to("cpu", torch.float32))
        self.flat.copy_(cpu)
        return self

    def state_dict(self):
        return {k: v.detach().clone() for k, v in self.views().items()}


def probe_contexts(pairset, B, n0_cap, e0_cap, max_graph_nodes, device, pair_index=None, first=0):
    """How much of a batch of this workload repeats (one extraction of B pairs, synchronises): returns
    (unique rows / rows, (entries + rows of the representatives) / (entries + rows)).  conv1 per context pays off when
    rows repeat (NPInter2-shaped, 200 two-hop subgraphs: 0.21 / 0.43); its backward per context only when the
    representatives carry well under half of the elements (x100, 3-hop, 4,096 subgraphs: 0.31 / 0.60 -- there the
    index structures cost more than the per-row transposed aggregation saves; RPI2241: 0.8 / 0.9, nothing to gain)."""
    g = pairset.graph
    eng = Engine(g.F, B, n0_cap, e0_cap, max_graph_nodes, device=device, graph=g, need_backward=False, extract_only=True)
    if not eng.contexts:
        return 1.0, 1.0
    eng.load_pairs(pairset, first=first, count=B, pair_index=pair_index)
    U, EU = eng.ctx_counters()
    N, E = eng.counters()
    del eng
    return U / max(N[0], 1), (EU + U) / max(E[0] + N[0], 1)


CTX_MAX_UNIQUE_ROWS = 0.7        # above: conv1 per row
CTX_BWD_MAX_SHARE = 0.5          # above: forward per context, backward per row


def context_policy(pairset, B, n0_cap, e0_cap, max_graph_nodes, device, pair_index=None, first=0):
    """(contexts, ctx_bwd) for Engine(...) from one probed batch; NPI_CTX_AUTO=0 keeps both on."""
    if os.environ.get("NPI_CTX_AUTO", "1") == "0" or os.environ.get("NPI_CTX_DEDUP", "1") == "0":
        return None, None
    uniq, share = probe_contexts(pairset, B, n0_cap, e0_cap, max_graph_nodes, device, pair_index, first)
    return uniq < CTX_MAX_UNIQUE_ROWS, share < CTX_BWD_MAX_SHARE


def tiny_wanted(tiny, env, n0_cap, B):
    """Whether a batch shape asks for the per-subgraph kernels (csrc/tiny.cu): the caller's explicit choice first, then the
    environment (NPI_TINY = 1 / 0), else by size -- at most TINY_MEAN_NODES rows per subgraph on average.  (The engine also
    requires the virtual input layer, split mode and subgraphs of at most ops.tiny_max_nodes() nodes.)"""
    if tiny is not None:
        return bool(tiny)
    if env == "1":
        return True
    if env == "0":
        return False
    return int(n0_cap) <= TINY_MEAN_NODES * max(int(B), 1)


def layer_caps(n0_cap, B):
    caps = [int(n0_cap)]
    for _ in range(3):
        caps.append((caps[-1] + B) // 2 + 1)
    return caps


class BatchSlot:
    """Everything the extraction of one batch produces (device-resident): targets, labels, graph
    pointers of the input layer and of the three pooled layers, node ids / hop labels, the input
    CSR by destination and the by-serial occurrence lists.  The engine owns two slots so that the
    batch of step i+1 can be extracted (side stream) while step i computes on the other one."""

    def __init__(self, B, n0_cap, e_cap, V, need_backward, dev, contexts=False, ctx_bwd=False):
        i32 = dict(dtype=torch.int32, device=dev)
        self.pairs_b = torch.zeros(B, 2, **i32)
        self.y_b = torch.zeros(B, **i32)
        self.gptrs = torch.zeros(4, B + 1, **i32)
        self.edge_ptr = torch.zeros(B + 1, **i32)
        self.sizes = torch.zeros(8, **i32)
        self.gid = torch.zeros(n0_cap, **i32)
        self.dist = torch.zeros(n0_cap, dtype=torch.uint8, device=dev)
        self.rowptr0 = torch.zeros(n0_cap + 1, **i32)
        self.col0 = torch.zeros(e_cap, **i32)
        self.hubq0 = torch.zeros(ops.hub_rows_bytes(e_cap), dtype=torch.uint8, device=dev)    # hub-row segments of the input CSR
        self.ent0 = torch.zeros(e_cap, **i32)       # packed entries of the input CSR: gid | dist << 29 (ops.entry_pack_virt)
        self.rows0 = torch.zeros(n0_cap, 4, **i32)  # rows of the input CSR binned by length class (ops.hub_rows_build)
        # layer-1 contexts (csrc/ctx.cu): representative of every row, and the hub queue / binned row order of the
        # representatives only (what the forward aggregation of layer 1 walks)
        self.rep_of = torch.zeros(n0_cap, **i32) if contexts else None
        self.ctx_stats = torch.zeros(4, **i32) if contexts else None
        self.hubq0u = torch.zeros(ops.hub_rows_bytes(e_cap), dtype=torch.uint8, device=dev) if contexts else None
        self.rows0u = torch.zeros(n0_cap, 4, **i32) if contexts else None
        # per-context backward of conv1: label sums, rows sorted by representative, CSR by global id over the contexts
        self.lsum = torch.zeros(n0_cap, **i32) if ctx_bwd else None
        if ctx_bwd:
            self.ck = [torch.zeros(n0_cap, **i32) for _ in range(2)]
            self.cr = [torch.zeros(n0_cap, **i32) for _ in range(2)]
            k = 1 if ops.ctx_class_result_in_b(n0_cap) else 0
            self.class_keys, self.class_rows = self.ck[k], self.cr[k]
            self.cptr2 = torch.zeros(n0_cap + 1, **i32)       # class CSR: two entries per member row (ops.ctx_class_pack)
            self.crep = torch.zeros(n0_cap, **i32)
            self.n_ctx = self.ctx_stats[3:4]
            self.selC = torch.zeros(n0_cap, 4, **i32)
            self.hubqC = torch.zeros(ops.hub_rows_bytes(2 * n0_cap), dtype=torch.uint8, device=dev)
            self.rowsC = torch.zeros(n0_cap, 4, **i32)
            self.inv_ptr = torch.zeros(V + 1, **i32)
            self.inv_sel = torch.zeros(n0_cap + e_cap, 2, **i32)
            self.hubqG = torch.zeros(ops.hub_rows_bytes(n0_cap + e_cap), dtype=torch.uint8, device=dev)
            self.rowsG = torch.zeros(V, 4, **i32)
        self.occ_ptr = torch.zeros(V + 1, **i32) if need_backward else None
        self.occ_node = torch.zeros(n0_cap, **i32) if need_backward else None
        self.size_views = [self.sizes[i:i + 1] for i in range(8)]
        self.gp = self.gptrs
        self.cur_B = 0


class Engine:
    """Preallocated buffers for batches of up to (B, N0_cap, E0_cap) and the kernel sequences.

    ``graph`` (BipartiteGraph) provides the virtual layer-1 features; pass ``graph=None`` and
    call ``set_dense_input`` for a foreign PyG-style batch with a dense x."""

    def __init__(self, F, B, n0_cap, e0_cap, max_graph_nodes, device="cuda", graph=None, need_backward=True,
                 mode="split", contexts=None, ctx_bwd=None, extract_only=False, tiny=None):
        """mode "split": dense projections (gemm.cu) + CSR gather kernels (agg.cu) -- the fast path;
        mode "fused_v1": the single-kernel aggregate->project variants of sage.cu (kept as an
        independently validated GPU implementation and for A/B profiling)."""
        dev = torch.device(device)
        self.device, self.F, self.B = dev, F, B
        self.graph = graph
        self.mode = mode
        if mode not in ("split", "fused_v1"):
            raise L.NPIError("unknown engine mode %r" % (mode,))
        self.n_cap = layer_caps(n0_cap, B)
        self.e_cap = int(max(e0_cap, 1))
        self.max_graph_nodes = int(max(max_graph_nodes, 2))
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        u8 = dict(dtype=torch.uint8, device=dev)
        nc = self.n_cap
        # batch assembly / extraction outputs: two slots (compute on one, prefetch into the other)
        V = graph.num_nodes if graph is not None else 1
        self.V = V
        # software-pipelined aggregation kernels over packed entry streams (NPI_AGG_PIPE=0: the plain
        # dependent-chain kernels, kept for A/B runs; results are bit-identical)
        self.pipelined = mode == "split" and os.environ.get("NPI_AGG_PIPE", "1") != "0"
        # the three layers of a subgraph in one CTA (tiny: None = by size, True / False = forced where applicable)
        self.tiny = bool(tiny_wanted(tiny, os.environ.get("NPI_TINY", "auto"), n0_cap, B) and mode == "split" and graph is not None
                         and not extract_only and self.max_graph_nodes <= ops.tiny_max_nodes())
        # conv1 once per layer-1 context of the batch (virtual input layer only; NPI_CTX_DEDUP=0: every row)
        # contexts / ctx_bwd: None = on (the environment switches are the A/B partners), False = off (a caller that probed
        # the workload and found too few repeated contexts: probe_contexts)
        self.contexts = (self.pipelined and graph is not None and os.environ.get("NPI_CTX_DEDUP", "1") != "0"
                         and contexts is not False and not self.tiny)
        # ... and its backward per context too (NPI_CTX_BWD=0: transposed aggregation over all rows + by-id reduction)
        self.ctx_bwd = self.contexts and need_backward and os.environ.get("NPI_CTX_BWD", "1") != "0" and ctx_bwd is not False
        self.slots = [BatchSlot(B, nc[0], self.e_cap, V, need_backward, dev, contexts=self.contexts, ctx_bwd=self.ctx_bwd)
                      for _ in range(2)]
        self.ws_ctx = torch.empty(ops.ctx_workspace_bytes(nc[0]), **u8) if self.contexts else None
        self.ws_ctxidx = torch.empty(ops.ctx_index_workspace_bytes(nc[0], self.e_cap), **u8) if self.ctx_bwd else None
        self.perm_src0 = torch.empty(nc[1], **i32) if self.contexts else None
        self.slot = 0
        self.overflow = torch.zeros(1, **i32)      # sticky: a batch did not fit the extraction buffers (check_overflow)
        # filtered adjacency of the pooled layers (compute side only)
        self._rowptr12 = [torch.zeros(nc[1] + 1, **i32), torch.zeros(nc[2] + 1, **i32)]
        self._col12 = [torch.zeros(self.e_cap, **i32), torch.zeros(self.e_cap, **i32)]
        # extract_only (probe_contexts): the engine will only extract a batch -- the activation buffers are not needed
        self.extract_only = bool(extract_only)
        if extract_only:
            real_nc, nc = nc, [1, 1, 1, 1]
        # per layer l = 1..3 (index l-1)
        self.h = [torch.empty(nc[l], H, **f32) for l in range(3)]
        self.z = [torch.empty(nc[l], **f32) for l in range(3)]
        self.s = [torch.empty(nc[l], **f32) for l in range(3)]
        self.new_id = [torch.empty(nc[l], **i32) for l in range(3)]
        self.perm = [torch.empty(nc[l + 1], **i32) for l in range(3)]
        self.batch = [torch.empty(nc[l + 1], **i32) for l in range(3)]
        self.xp = [torch.empty(nc[l + 1], H, **f32) for l in range(3)]
        self.argmax = [torch.empty(B, H, **i32) for _ in range(3)]
        self.readout = torch.zeros(B, 2 * H, **f32)
        self.a1 = torch.zeros(B, 128, **f32)
        self.drop_mask = torch.ones(B, 128, **u8)
        self.a2 = torch.zeros(B, 64, **f32)
        self.logp = torch.zeros(B, 2, **f32)
        self.loss = torch.zeros(1, **f32)
        self.dense_x = None
        self._xpad = None
        # workspaces
        self.ws_select = torch.empty(max(16, ops.topk_select_workspace_bytes(B, self.max_graph_nodes)), **u8)
        self.ws_filter = torch.empty(ops.filter_adj_workspace_bytes(nc[1]) + 16, **u8)
        self.ws_readout = [torch.empty(ops.pool_gate_readout_workspace_bytes(B), **u8) for _ in range(3)]   # per layer: combined on the aux stream
        self._hubq12 = [torch.zeros(ops.hub_rows_bytes(16 if extract_only else self.e_cap), **u8) for _ in range(2)]
        self.need_backward = need_backward
        self.sel = ([torch.zeros(self.e_cap, 2, **i32) for _ in range(3)]
                    if (need_backward and self.pipelined) else None)     # {new_id[col], 1/(deg_col+1)} per entry and layer
        self._rows12 = [torch.zeros(nc[1], 4, **i32), torch.zeros(nc[2], 4, **i32)] if self.pipelined else [None, None]
        if need_backward:
            # the readout gradient [B, 256] lives right behind the rows of dxp[0] in ONE buffer: the per-context backward of
            # conv1 gathers gradient rows and mean-readout rows through the same base pointer (ops.ctx_class_pack)
            self._dxp0_ext = torch.zeros(nc[1] + 2 * B, H, **f32)
            self.d_readout = self._dxp0_ext[nc[1]:].view(B, 2 * H)
            self.dpre = [torch.empty(nc[l + 1], H, **f32) for l in range(3)]
            self.dxp = [self._dxp0_ext[:nc[1]], torch.empty(nc[2], H, **f32)]
            self.ws_pool = [torch.empty(ops.pool_bwd_workspace_bytes(), **u8) for _ in range(3)]   # per layer: reduced on the aux stream
            self.ws_sagew = torch.empty(ops.sage_bwd_weight_workspace_bytes(max(F, H)), **u8)
            self.ws_head = torch.empty(max(16, ops.head_bwd_workspace_bytes(B)), **u8)
        # split mode: projected operands / transposed aggregation / by-serial occurrence lists
        if extract_only:
            nc = real_nc
        self.ybuf = torch.empty(1 if extract_only else nc[1], H, **f32)                 # x'.W of layers 2-3
        self.big = torch.empty(1 if extract_only else nc[0], H, **f32)   # x.W of a dense layer-1 input (fwd) / dxa of layer 1 (bwd)
        # transposed aggregation of layers 2-3: own buffers, so the weight-gradient GEMMs of a layer
        # (auxiliary stream) may still read them while the main stream goes on to the layer below
        self.dxa12 = [torch.empty(nc[1], H, **f32), torch.empty(nc[2], H, **f32)] if need_backward else None
        if self.tiny:
            # per-subgraph filtered adjacency (n_g + 1 row pointers per subgraph), transposed conv2 / conv3 weights,
            # per-subgraph partials of d_pool_w / d_bias
            self._rowptr_f = [torch.zeros(nc[1] + B + 1, **i32), torch.zeros(nc[2] + B + 1, **i32)]
            self._wt = [torch.empty(H, H, **f32) for _ in range(2)] if need_backward else None
            self._ybuf2 = torch.empty(nc[2], H, **f32)       # projected rows of layer 3 (layer 2's live in ybuf: subgraphs are in different layers at the same time)
            self._tiny_part = torch.empty(ops.tiny_partials_bytes(B), **u8) if need_backward else None
            self.ws_tn_tc_main = torch.empty(ops.gemm_tn_tc_workspace_bytes(), **u8) if need_backward else None
        # the SAGEConv weight gradients summed over the batch rows directly in one launch (conv1: work ~ N0 * F instead of the
        # route through the feature table -- by-node reduction, then table^T . G: work ~ V * F but three dependent launches;
        # conv2 / conv3: instead of two tcgen05 launches each): small batches only
        self.tiny_w1_direct = self.tiny and int(n0_cap) <= TINY_W1_DIRECT_ROWS and os.environ.get("NPI_TINY_W1", "direct") == "direct"
        self.ws_w1 = ops.tiny_weight_grads_workspace(F, dev) if (self.tiny_w1_direct and need_backward) else None
        self._aux = None                                         # auxiliary stream for independent branches
        self.stamps, self.stamp_names = None, []
        self._idx, self._idx_forked = None, False                # stream of the backward's index structures (_fork_index)
        self.hooks = {}                                          # name -> callable run at that point of the step (trainer: where the
                                                                 # next batch's extraction is forked): fwd_agg0 | fwd_end | bwd_l1
        self.serial = False                                      # True: no branches (per-kernel timing passes)
        self.ws_tn_tc = torch.empty(ops.gemm_tn_tc_workspace_bytes(), **u8) if need_backward else None
        self.use_tn_tc = True                                    # tcgen05 weight-gradient GEMM (K = 128 layers)
        self.t_gemm_tc = os.environ.get("NPI_T_GEMM", "tc") != "simt"   # T = table . W1 on tcgen05 (A/B switch)
        self.T = torch.empty(V, H, **f32)                        # feature table . W1  (layer 1, virtual input)
        if need_backward:
            self.G = torch.empty(V, H, **f32)
            self.ws_gid = torch.empty(ops.gid_index_workspace_bytes(V, nc[0]), **u8)
            self.label_part = torch.zeros(ops.gid_reduce_partials(), H, **f32)
            self.ws_tn = torch.empty(ops.gemm_tn_workspace_bytes(max(F, H)), **u8)
            self.ws_tg = torch.empty(ops.table_grad_workspace_bytes(F), **u8)

    def check_overflow(self):
        """Raise if any extraction since the last check skipped a pair for lack of buffer space (the
        kernels never write out of bounds; a truncated batch must not pass silently).  Synchronises."""
        if int(self.overflow.item()):
            self.overflow.zero_()
            raise L.NPIError("a batch exceeded the engine's extraction buffers (N0 cap %d, E0 cap %d): its subgraphs were "
                             "truncated -- size the engine from PairSet.batch_caps of the batches actually used"
                             % (self.n_cap[0], self.e_cap))

    # ---- views of the CURRENT slot (what forward/backward and the tests read) --------------------
    @property
    def cur(self):
        return self.slots[self.slot]

    def use_slot(self, k):
        self.slot = int(k) & 1

    pairs_b = property(lambda self: self.cur.pairs_b)
    y_b = property(lambda self: self.cur.y_b)
    gptrs = property(lambda self: self.cur.gptrs)
    edge_ptr = property(lambda self: self.cur.edge_ptr)
    sizes = property(lambda self: self.cur.sizes)
    gid = property(lambda self: self.cur.gid)
    dist = property(lambda self: self.cur.dist)
    occ_ptr = property(lambda self: self.cur.occ_ptr)
    occ_node = property(lambda self: self.cur.occ_node)
    cur_B = property(lambda self: self.cur.cur_B)
    _gp = property(lambda self: self.cur.gp)
    _size_views = property(lambda self: self.cur.size_views)
    rowptr = property(lambda self: [self.cur.rowptr0] + self._rowptr12)
    col = property(lambda self: [self.cur.col0] + self._col12)
    hubq = property(lambda self: [self.cur.hubq0] + self._hubq12)
    rows = property(lambda self: [self.cur.rows0 if self.pipelined else None] + self._rows12)

    # ------------------------------------------------------------------ batch assembly
    def load_pairs(self, pairset, first=0, count=None, pair_index=None, slot=None):
        """Device-side batch assembly + GPU extraction of ``count`` pairs of ``pairset``
        (indices first..first+count-1, or pair_index[:count]) into batch slot ``slot`` (default:
        the current one), then everything derived from the extracted batch (packed entries, contexts, row lists).
        Enqueued on the current stream."""
        B = self.B if count is None else int(count)
        if B > self.B:
            raise L.NPIError("batch of %d exceeds engine capacity %d" % (B, self.B))
        g = pairset.graph
        sl = self.cur if slot is None else self.slots[int(slot) & 1]
        gp = sl.gptrs if B == self.B else torch.zeros(4, B + 1, dtype=torch.int32, device=self.device)
        ops.batch_prepare(pair_index, first, B, pairset.pairs, pairset.y, pairset.n_all, pairset.e_all, RATIO,
                          sl.pairs_b, sl.y_b, gp, sl.edge_ptr, sl.sizes)
        sl.gp = gp
        ops.khop_fill(g, sl.pairs_b, B, pairset.h, pairset.max_nodes, gp[0], sl.edge_ptr, sl.gid, sl.dist,
                      sl.rowptr0, sl.col0, pairset.khop_ws, pairset.num_ctas, overflow=self.overflow)
        lean = self.ctx_bwd or self.tiny   # forward and backward of layer 1 walk the contexts / the subgraphs: no per-row lists needed
        if not lean:
            if self.pipelined:
                ops.hub_rows_build(sl.rowptr0, sl.sizes[0:1], self.n_cap[0], self.e_cap, sl.hubq0, sl.gid, sl.dist, sl.rows0)
            else:
                ops.hub_rows_build(sl.rowptr0, sl.sizes[0:1], self.n_cap[0], self.e_cap, sl.hubq0)
        if self.pipelined and not self.tiny:
            ops.entry_pack_virt(sl.rowptr0, sl.col0, sl.gid, sl.dist, sl.sizes[0:1], self.n_cap[0], g.num_nodes, sl.ent0)
        if self.contexts:
            ops.ctx_build(sl.rowptr0, sl.ent0, sl.gid, sl.dist, sl.sizes[0:1], self.n_cap[0], sl.rep_of, sl.ctx_stats, self.ws_ctx,
                          label_sum=sl.lsum)
            ops.hub_rows_build(sl.rowptr0, sl.sizes[0:1], self.n_cap[0], self.e_cap, sl.hubq0u, sl.gid, sl.dist, sl.rows0u,
                               keep=sl.rep_of)
        if self.ctx_bwd:
            if g.num_nodes != self.V:
                raise L.NPIError("engine was sized for a graph of %d nodes, got %d" % (self.V, g.num_nodes))
            pass                         # the backward's index structures are built next to the forward pass (_backward_index)
        elif self.need_backward and self.mode == "split" and not self.tiny_w1_direct:
            if g.num_nodes != self.V:
                raise L.NPIError("engine was sized for a graph of %d nodes, got %d" % (self.V, g.num_nodes))
            ops.gid_index_build(sl.gid, sl.sizes[0:1], self.n_cap[0], g.num_nodes, sl.occ_ptr, sl.occ_node, self.ws_gid)
        sl.cur_B = B
        self.graph = g
        self.dense_x = None

    def set_csr_batch(self, x, rowptr, col, graph_ptr, y=None):
        """Foreign batch: dense x [N,F], CSR by destination, graph_ptr [B+1] (all on device)."""
        B = graph_ptr.numel() - 1
        N, E = x.shape[0], col.numel()
        if B > self.B or N > self.n_cap[0] or E > self.e_cap:
            raise L.NPIError("batch exceeds engine capacity")
        sl = self.cur
        n = (graph_ptr[1:] - graph_ptr[:-1]).to(torch.int32)
        gp = torch.zeros(4, B + 1, dtype=torch.int32, device=self.device)
        gp[0] = graph_ptr.to(torch.int32)
        for l in range(1, 4):
            n = torch.ceil(torch.tensor(RATIO, dtype=torch.float32, device=self.device) * n.to(torch.float32)).to(torch.int32)
            gp[l, 1:] = torch.cumsum(n, 0)
        sl.gp = gp
        sl.sizes[:4] = gp[:, B]
        sl.sizes[4] = E
        sl.rowptr0[:N + 1].copy_(rowptr)
        sl.col0[:E].copy_(col)
        ops.hub_rows_build(sl.rowptr0, sl.sizes[0:1], self.n_cap[0], self.e_cap, sl.hubq0, None, None,
                           sl.rows0 if self.pipelined else None)
        if y is not None:
            sl.y_b[:B].copy_(y.to(torch.int32))
        # dense features go through a row-padded staging buffer [n_cap, round_up(F, 4)] (padding columns stay zero):
        # 16-byte aligned rows are what the TMA-fed tcgen05 projection and the tensor-core weight gradient need --
        # a PyG x of 178 columns has a 712-byte row stride -- and the buffer has the full n_cap rows the tensor map
        # covers.  One copy of x (read + write) instead of two SIMT fp32 GEMMs over N0 x 178 x 128.
        if self._xpad is None:
            self._xpad = torch.zeros(self.n_cap[0], (self.F + 3) // 4 * 4, dtype=torch.float32, device=self.device)
        self._xpad[:N, :self.F].copy_(x)
        self.dense_x = self._xpad[:N, :self.F]
        sl.cur_B = B

    # ------------------------------------------------------------------ forward / backward
    def _table_grad(self, g, gv, ws_tc=None):
        """conv1.weight gradient through the feature table: table^T . G + label row, last link of the step's chain."""
        ws_tc = self.ws_tn_tc if ws_tc is None else ws_tc
        if g.num_nodes <= SMALL_TABLE_ROWS:
            ops.table_grad(g.table, self.G, g.num_nodes, self.label_part, gv["conv1.weight"], self.ws_tg, K=self.F)
        elif self.t_gemm_tc and self.F <= 256:     # tcgen05: one pass per 128 table columns
            ops.gemm_tn_tc(g.table, self.G, None, g.num_nodes, self.label_part, gv["conv1.weight"], ws_tc, K=self.F)
        else:
            ops.gemm_tn(g.table, self.G, None, g.num_nodes, self.F, self.label_part, gv["conv1.weight"], self.ws_tn)

    # ---- small-subgraph path (csrc/tiny.cu) ----------------------------------------------------------
    def _tiny_on(self):
        return self.tiny and self.dense_x is None

    def _tiny_args(self, v, gv=None):
        """npi_tiny_args_t over the current slot's batch and this engine's activation buffers."""
        sl, gp = self.cur, self._gp
        kw = dict(B=self.cur_B, max_graph_nodes=self.max_graph_nodes, graph_ptr=[gp[l] for l in range(4)],
                  T=self.T, w_label=v["conv1.weight"][0], gid=sl.gid, dist=sl.dist, rowptr0=sl.rowptr0, col0=sl.col0,
                  weight=[v["conv%d.weight" % (l + 1)] for l in range(3)], bias=[v["conv%d.bias" % (l + 1)] for l in range(3)],
                  pool_w=[v["pool%d.weight" % (l + 1)] for l in range(3)],
                  h=self.h, z=self.z, s=self.s, perm=self.perm, new_id=self.new_id, batch=self.batch, xp=self.xp, argmax=self.argmax,
                  rowptr_f=self._rowptr_f, col_f=self._col12, y=[None, self.ybuf, self._ybuf2], readout=self.readout)
        if self.need_backward:
            kw.update(weight_t=[None, self._wt[0], self._wt[1]], d_readout=self.d_readout, dpre=self.dpre,
                      dxa=[self.big, self.dxa12[0], self.dxa12[1]], dxp=self.dxp, partials=self._tiny_part)
        if gv is not None:
            kw.update(d_pool_w=[gv["pool%d.weight" % (l + 1)] for l in range(3)], d_bias=[gv["conv%d.bias" % (l + 1)] for l in range(3)])
        return ops.tiny_args(**kw)

    def _forward_tiny(self, v):
        """T = table . conv1.weight, then one launch for conv1..3 + pool1..3 + readout (a CTA per subgraph)."""
        g, W = self.graph, v["conv1.weight"]
        _nvtx_push("forward/per-subgraph")
        if self.F <= 192 and self.t_gemm_tc:
            ops.gemm_nn_tc(g.table, None, g.num_nodes, self.F, W, False, self.T)
        else:
            ops.gemm_nn(g.table, None, g.num_nodes, self.F, W, False, self.T)
        self._stamp("fwd_gemm0")
        self._hook("fwd_agg0")           # the trainer forks the extraction of the next batch here: it runs next to the whole step
        if self.need_backward:
            with self._branch():         # W^T of conv2 / conv3 for the backward's dX = DXA . W^T
                ops.tiny_transpose(v["conv2.weight"], v["conv3.weight"], self._wt[0], self._wt[1])
        ops.tiny_fwd(self._tiny_args(v))
        for name in ("fwd_topk0", "fwd_agg1", "fwd_topk1", "fwd_agg2", "fwd_topk2"):
            self._hook(name)
        _nvtx_pop()

    def _backward_tiny(self, v, gv):
        """One launch for the backward of pool3/conv3 .. pool1/conv1 down to DXA of every layer; the weight gradients stay
        dense GEMMs over the batch (conv2/conv3 on the auxiliary stream, conv1 through the feature table on the chain)."""
        sz, g = self._size_views, self.graph
        _nvtx_push("backward/per-subgraph")
        ta = self._tiny_args(v, gv)
        ops.tiny_bwd(ta, phases=1)
        self._stamp("bwd_tiny")
        self._hook("bwd_l1")
        with self._branch():
            ops.tiny_bwd(ta, phases=2)
            if not self.tiny_w1_direct:
                for l in (2, 1):
                    ops.gemm_tn_tc(self.xp[l - 1], self.dxa12[l - 1], sz[l], self.n_cap[l], None, gv["conv%d.weight" % (l + 1)], self.ws_tn_tc)
        if self.tiny_w1_direct:          # the three SAGEConv weight gradients straight from the batch rows: one launch instead of seven
            ops.tiny_weight_grads(g.table, self.F, self.gid, self.dist, self.big, sz[0], self.n_cap[0], gv["conv1.weight"], self.ws_w1,
                                  x1=self.xp[0], dxa2=self.dxa12[0], n1_dev=sz[1], n1_host=self.n_cap[1], d_w2=gv["conv2.weight"],
                                  x2=self.xp[1], dxa3=self.dxa12[1], n2_dev=sz[2], n2_host=self.n_cap[2], d_w3=gv["conv3.weight"])
        else:
            ops.gid_reduce(self.big, self.dist, self.occ_ptr, self.occ_node, g.num_nodes, self.G, self.label_part)
            self._table_grad(g, gv, ws_tc=self.ws_tn_tc_main)
        _nvtx_pop()

    def _dedup0(self):
        """conv1 evaluated on one representative row per layer-1 context (virtual input layer, split mode)."""
        return self.contexts and self.dense_x is None and self.mode == "split"

    def layer_rows(self, l, n=None):
        """(h, z, s) of layer ``l`` (0-based) for rows 0..n-1, expanded through the context map where layer 1 keeps
        one copy per context -- for tests and diagnostics (allocates)."""
        n = self.n_cap[l] if n is None else int(n)
        if l == 0 and self._dedup0():
            idx = self.cur.rep_of[:n].long()
            return self.h[0][idx], self.z[0][idx], self.s[0][idx]
        return self.h[l][:n], self.z[l][:n], self.s[l][:n]

    def _backward_index(self):
        """Index structures of the per-context backward of conv1 for the current slot (rows sorted by representative,
        contexts, CSR by node over the contexts, their hub queues): ~40 small integer kernels that only the END of the
        backward pass needs, so they run on a stream of their own next to the forward pass of the same step (joined in
        backward()) instead of lengthening the extraction of the next batch."""
        sl = self.cur
        ops.ctx_index_build(sl.rowptr0, sl.ent0, sl.gid, sl.rep_of, sl.sizes[0:1], self.n_cap[0], self.e_cap, self.V,
                            sl.ck[0], sl.cr[0], sl.ck[1], sl.cr[1], sl.cptr2, sl.crep, sl.n_ctx, sl.inv_ptr, sl.inv_sel,
                            self.ws_ctxidx)
        ops.hub_rows_build(sl.cptr2, sl.n_ctx, self.n_cap[0], 2 * self.n_cap[0], sl.hubqC, None, None, sl.rowsC)
        ops.hub_rows_build(sl.inv_ptr, None, self.V, self.n_cap[0] + self.e_cap, sl.hubqG, None, None, sl.rowsG)

    def _fork_index(self):
        if self.serial:
            self._backward_index()
            return
        if self._idx is None:
            self._idx = torch.cuda.Stream(device=self.device)
        self._idx.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self._idx):
            self._backward_index()
        self._idx_forked = True

    def _join_index(self):
        if self._idx_forked:
            torch.cuda.current_stream(self.device).wait_stream(self._idx)
            self._idx_forked = False

    def _feat0(self):
        if self.dense_x is not None:
            return L.features_dense(self.dense_x)
        return self.graph.features_for(self.gid, self.dist)

    def forward(self, params: FlatParams, training=False, drop_mask=None, seed=0, step_dev=None,
                sample_ids=None, sample_id_base=0, compute_loss=False, loss_scale=None, defer_loss=False,
                fuse_head_delta=False):
        """defer_loss: sum the scalar loss on the auxiliary stream (joined by backward(); for callers
        that always run backward() right after -- nothing on the device waits for the loss).
        fuse_head_delta: the head's forward also leaves the mean-NLL deltas and d_readout (one launch instead of two on the
        chain); backward() with the same loss_scale and no explicit d_logp then skips that phase."""
        if self.extract_only:
            raise L.NPIError("this engine was built with extract_only=True")
        B = self.cur_B
        v = params.views()
        sz = self._size_views
        gp = self._gp
        if self.ctx_bwd and self._dedup0():
            self._fork_index()
        self._stamp("fwd_start")
        if self._tiny_on():
            self._forward_tiny(v)
        for l in (() if self._tiny_on() else range(3)):
            _nvtx_push("forward/conv%d+pool%d" % (l + 1, l + 1))
            W, bias, pw = v["conv%d.weight" % (l + 1)], v["conv%d.bias" % (l + 1)], v["pool%d.weight" % (l + 1)]
            if self.mode == "fused_v1":
                feat = self._feat0() if l == 0 else L.features_dense(self.xp[l - 1])
                self._join()
                ops.sage_fwd(feat, self.rowptr[l], self.col[l], sz[l], self.n_cap[l], W, bias, True, pw,
                             self.h[l], self.z[l], self.s[l])
            elif l == 0 and self.dense_x is None:
                g = self.graph       # project the V-row feature table once, gather 128-wide rows of it
                if self.F <= 192 and self.t_gemm_tc:     # tcgen05 + TMA: the table is streamed once, K = F columns
                    ops.gemm_nn_tc(g.table, None, g.num_nodes, self.F, W, False, self.T)
                else:
                    ops.gemm_nn(g.table, None, g.num_nodes, self.F, W, False, self.T)
                self._stamp("fwd_gemm0")
                dd = self._dedup0()
                ops.sage_aggregate_fwd(self.T, self.gid, self.dist, W[0], self.rowptr[0], self.col[0], sz[0], self.n_cap[0],
                                       bias, True, pw, self.h[0], self.z[0], self.s[0], self.cur.hubq0u if dd else self.hubq[0],
                                       packed=self.cur.ent0 if self.pipelined else None,
                                       row_order=self.cur.rows0u if dd else self.rows[0], pipelined=self.pipelined)
            else:
                x = self.dense_x if l == 0 else self.xp[l - 1]
                y = self.big if l == 0 else self.ybuf
                if x.shape[1] == H and l > 0:      # 128-wide pooled features: tcgen05 (3xTF32) projection
                    ops.gemm_nn_tc(x, sz[l], self.n_cap[l], H, W, False, y)
                    self._stamp("fwd_gemm%d" % l)
                elif l == 0 and self.F <= 192 and self.t_gemm_tc:      # dense x, row-padded staging buffer
                    ops.gemm_nn_tc(self._xpad, sz[0], self.n_cap[0], self.F, W, False, y)
                else:
                    ops.gemm_nn(x, sz[l], self.n_cap[l], x.shape[1], W, False, y)
                self._join()             # the filtered adjacency of this layer (auxiliary stream)
                ops.sage_aggregate_fwd(y, None, None, None, self.rowptr[l], self.col[l], sz[l], self.n_cap[l],
                                       bias, True, pw, self.h[l], self.z[l], self.s[l], self.hubq[l], row_order=self.rows[l],
                                       pipelined=self.pipelined)
            self._hook("fwd_agg%d" % l)
            dd = l == 0 and self._dedup0()      # layer 1 evaluated per context: h/z/s live at the representative rows
            fused_hub = l < 2 and self.pipelined and self.n_cap[0] <= SMALL_BATCH_ROWS
            if fused_hub:
                with self._branch():     # header of the next CSR's hub queue: zeroed next to the top-k, off the chain
                    ops.hub_rows_reset(self.hubq[l + 1])
            ops.topk_select(self.s[l], gp[l], gp[l + 1], B, self.max_graph_nodes, self.perm[l], self.new_id[l],
                            self.batch[l], self.ws_select, row_map=self.cur.rep_of if dd else None,
                            perm_src=self.perm_src0 if dd else None)
            self._hook("fwd_topk%d" % l)
            if l < 2:
                # filter_adj only feeds the NEXT aggregation: it runs on the auxiliary stream next to
                # gating/readout and the next layer's projection (joined in the next iteration).  It chases col -> new_id
                # itself: packing the entries first lengthened the chain the next aggregation waits for (0.675 -> 0.705 ms)
                with self._branch():
                    if fused_hub:        # hub queue + row order of the filtered CSR come out of filter_adj's own kernels
                        ops.filter_adj(self.rowptr[l], self.col[l], self.perm[l], self.new_id[l], sz[l + 1], self.n_cap[l + 1],
                                       self.rowptr[l + 1], self.col[l + 1], self.ws_filter,
                                       hubq=self.hubq[l + 1], hub_e_max=self.e_cap, row_order=self.rows[l + 1])
                    else:
                        ops.filter_adj(self.rowptr[l], self.col[l], self.perm[l], self.new_id[l], sz[l + 1], self.n_cap[l + 1],
                                       self.rowptr[l + 1], self.col[l + 1], self.ws_filter)
                        ops.hub_rows_build(self.rowptr[l + 1], sz[l + 1], self.n_cap[l + 1], self.e_cap, self.hubq[l + 1],
                                           None, None, self.rows[l + 1])
            if self.sel is not None and not (dd and self.ctx_bwd):
                # packed entries for the transposed aggregation of this layer (backward): auxiliary stream
                with self._branch():
                    ops.entry_pack_sel(self.rowptr[l], self.col[l], self.new_id[l], sz[l], self.n_cap[l], self.sel[l])
            gr_args = (self.h[l], self.s[l], self.perm_src0 if dd else self.perm[l], gp[l + 1], B, self.xp[l], self.readout, l > 0, self.argmax[l],
                       self.ws_readout[l])
            ops.pool_gate_readout(*gr_args, phases=1)
            self._stamp("fwd_gate%d" % l)
            with self._branch():     # the readouts accumulate on the auxiliary stream, in layer order; the head waits for them
                ops.pool_gate_readout(*gr_args, phases=2)
            _nvtx_pop()
        self._join()
        self._hook("fwd_end")
        _nvtx_push("forward/head")
        if loss_scale is None:
            loss_scale = 1.0 / B
        hf_args = (self.readout, B, v["lin1.weight"], v["lin1.bias"], v["lin2.weight"], v["lin2.bias"],
                   v["lin3.weight"], v["lin3.bias"], training, drop_mask, seed, step_dev, sample_ids, sample_id_base,
                   self.y_b if compute_loss else None, loss_scale, self.a1, self.drop_mask, self.a2, self.logp,
                   self.loss if compute_loss else None)
        self._head_delta_scale = None
        if fuse_head_delta and compute_loss and self.need_backward:
            ops.head_fwd_delta(self.readout, B, v["lin1.weight"], v["lin1.bias"], v["lin2.weight"], v["lin2.bias"],
                               v["lin3.weight"], v["lin3.bias"], training, drop_mask, seed, step_dev, sample_ids, sample_id_base,
                               self.y_b, loss_scale, self.a1, self.drop_mask, self.a2, self.logp, self.d_readout, self.ws_head)
            self._head_delta_scale = float(loss_scale)
        else:
            ops.head_fwd(*hf_args, phases=1)
        self._stamp("head_fwd")
        if compute_loss:
            if defer_loss and self.need_backward:
                with self._branch():
                    ops.head_fwd(*hf_args, phases=2)
            else:
                ops.head_fwd(*hf_args, phases=2)
        self._last_training = training
        _nvtx_pop()
        return self.logp[:B]

    def backward(self, params: FlatParams, grads: FlatParams, d_logp=None, loss_scale=None):
        """Gradients of all 15 tensors into ``grads.flat`` (written, not accumulated)."""
        if not self.need_backward:
            raise L.NPIError("engine was created with need_backward=False")
        B = self.cur_B
        v, gv = params.views(), grads.views()
        sz = self._size_views
        gp = self._gp
        if loss_scale is None:
            loss_scale = 1.0 / B
        if self.ctx_bwd and self._dedup0():
            self._join_index()
            with self._branch():     # entries of the class CSR for this step's selection: auxiliary stream, needed at the very end
                ops.ctx_class_pack(self.cur.class_rows, sz[0], self.n_cap[0], self.new_id[0], self.batch[0], gp[1], self.n_cap[1],
                                   self.cur.selC)
        _nvtx_push("backward/head")
        fused = getattr(self, "_head_delta_scale", None)
        self._head_delta_scale = None
        fused = fused is not None and d_logp is None and fused == float(loss_scale)       # forward() left the deltas already
        if not fused:
            ops.head_bwd(self.readout, B, v["lin1.weight"], v["lin2.weight"], v["lin3.weight"], self.a1,
                         self.drop_mask if self._last_training else None, self.a2, self.logp, self.y_b, loss_scale, d_logp,
                         gv["lin1.weight"], gv["lin1.bias"], gv["lin2.weight"], gv["lin2.bias"], gv["lin3.weight"],
                         gv["lin3.bias"], self.d_readout, self.ws_head, phases=1)
        self._stamp("head_bwd")
        with self._branch():     # the head's weight gradients only feed the optimizer
            ops.head_bwd(self.readout, B, v["lin1.weight"], v["lin2.weight"], v["lin3.weight"], self.a1,
                         self.drop_mask if self._last_training else None, self.a2, self.logp, self.y_b, loss_scale, d_logp,
                         gv["lin1.weight"], gv["lin1.bias"], gv["lin2.weight"], gv["lin2.bias"], gv["lin3.weight"],
                         gv["lin3.bias"], self.d_readout, self.ws_head, phases=2)
        _nvtx_pop()
        d_xp = None
        if self._tiny_on():
            self._backward_tiny(v, gv)
        for l in (() if self._tiny_on() else (2, 1, 0)):
            _nvtx_push("backward/pool%d+conv%d" % (l + 1, l + 1))
            W = v["conv%d.weight" % (l + 1)]
            split = self.mode == "split"
            dd = l == 0 and self._dedup0()
            pb_args = (d_xp, self.d_readout, self.h[l], self.z[l], self.s[l], self.perm_src0 if dd else self.perm[l], self.batch[l],
                       self.argmax[l], gp[l + 1], sz[l + 1], self.n_cap[l + 1], B, v["pool%d.weight" % (l + 1)], True,
                       self.dpre[l], gv["pool%d.weight" % (l + 1)], self.ws_pool[l])
            pb_bias = gv["conv%d.bias" % (l + 1)] if split else None
            cb = l == 0 and dd and self.ctx_bwd      # conv1 backward per context
            if cb:
                sl = self.cur
                ops.ctx_scatter_max(self.d_readout, self.argmax[0], B, d_xp)
                self._stamp("bwd_scatter")
                ops.csr_gather_sum(self._dxp0_ext, sl.cptr2, sl.selC, self.n_cap[0], self.big, sl.hubqC, sl.rowsC)
                self._stamp("bwd_gather_class")
                ops.ctx_finish(self.big, sl.crep, sl.n_ctx, self.n_cap[0], self.h[0], self.z[0], self.s[0], v["pool1.weight"], True,
                               sl.rowptr0, sl.lsum, self.label_part, self.ws_pool[0])
                self._stamp("bwd_finish")
            else:
                ops.pool_bwd(*pb_args, d_bias=pb_bias, phases=1)
                self._stamp("bwd_pool%d" % l)
            with self._branch():     # d_pool_w / d_bias only feed the optimizer
                ops.pool_bwd(*pb_args, d_bias=pb_bias, phases=2)
            if cb:
                g = self.graph
                ops.csr_gather_sum(self.big, sl.inv_ptr, sl.inv_sel, g.num_nodes, self.G, sl.hubqG, sl.rowsG)
                self._stamp("bwd_gather_node")
                self._table_grad(g, gv)
                _nvtx_pop()
                continue
            if not split:
                feat = self._feat0() if l == 0 else L.features_dense(self.xp[l - 1])
                ops.sage_bwd_weight(feat, self.rowptr[l], self.col[l], self.perm[l], sz[l + 1], self.n_cap[l + 1],
                                    self.dpre[l], gv["conv%d.weight" % (l + 1)], gv["conv%d.bias" % (l + 1)], self.ws_sagew)
                if l > 0:
                    ops.sage_bwd_input(self.dpre[l], self.new_id[l], self.rowptr[l], self.col[l], sz[l], self.n_cap[l],
                                       W, self.dxp[l - 1])
                    d_xp = self.dxp[l - 1]
                continue
            # transposed aggregation once, shared by the weight and the input gradient; the weight
            # gradient (a split-over-rows GEMM whose result is only needed by the optimizer) runs on
            # the auxiliary stream while the main stream continues down the layers
            dxa = self.big if l == 0 else self.dxa12[l - 1]
            ops.sage_aggregate_bwd(self.dpre[l], self.new_id[l], self.rowptr[l], self.col[l], sz[l], self.n_cap[l], dxa,
                                   self.hubq[l], packed=self.sel[l] if self.sel is not None else None,
                                   row_order=self.rows[l] if self.sel is not None else None)
            self._stamp("bwd_agg%d" % l)
            if l == 1:
                self._hook("bwd_l1")
            if l > 0:
                with self._branch():
                    if self.use_tn_tc:
                        ops.gemm_tn_tc(self.xp[l - 1], dxa, sz[l], self.n_cap[l], None, gv["conv%d.weight" % (l + 1)], self.ws_tn_tc)
                    else:
                        ops.gemm_tn(self.xp[l - 1], dxa, sz[l], self.n_cap[l], H, None, gv["conv%d.weight" % (l + 1)], self.ws_tn)
                ops.gemm_nn_tc(dxa, sz[l], self.n_cap[l], H, W, True, self.dxp[l - 1])
                self._stamp("bwd_gemm%d" % l)
                d_xp = self.dxp[l - 1]
            elif self.dense_x is not None:
                with self._branch():
                    if self.t_gemm_tc and self.F <= 256:
                        ops.gemm_tn_tc(self._xpad, dxa, sz[0], self.n_cap[0], None, gv["conv1.weight"], self.ws_tn_tc, K=self.F)
                    else:
                        ops.gemm_tn(self.dense_x, dxa, sz[0], self.n_cap[0], self.F, None, gv["conv1.weight"], self.ws_tn)
            else:
                g = self.graph
                with self._branch():
                    ops.gid_reduce(dxa, self.dist, self.occ_ptr, self.occ_node, g.num_nodes, self.G, self.label_part)
                    self._table_grad(g, gv)
            _nvtx_pop()
        self._join()
        self._stamp("bwd_end")

    # ---- auxiliary stream: independent branches of the step (captured as parallel graph branches) ----
    class _Branch:
        def __init__(self, eng):
            self.eng = eng

        def __enter__(self):
            e = self.eng
            self.ctx = None
            if e.serial:                      # profiling: everything in order on one stream
                return
            if e._aux is None:
                e._aux = torch.cuda.Stream(device=e.device)
            e._aux.wait_stream(torch.cuda.current_stream(e.device))      # fork
            self.ctx = torch.cuda.stream(e._aux)
            self.ctx.__enter__()
            e._forked = True

        def __exit__(self, *a):
            if self.ctx is not None:
                self.ctx.__exit__(*a)

    def _branch(self):
        return Engine._Branch(self)

    def _hook(self, name):
        fn = self.hooks.get(name)
        if fn is not None:
            fn()
        self._stamp(name)

    def _stamp(self, name):
        """NPI_STAMPS=1: %globaltimer of the main stream at named points of the step (tools/step_timeline.py)."""
        if not _STAMPS:
            return
        if self.stamps is None:
            self.stamps = torch.zeros(64, dtype=torch.int64, device=self.device)
            self.stamp_names = []
        if name not in self.stamp_names:
            self.stamp_names.append(name)
        L.call("npi_debug_stamp", L.ptr(self.stamps), self.stamp_names.index(name), L.stream_ptr(self.device))

    def _join(self):
        if getattr(self, "_forked", False):
            torch.cuda.current_stream(self.device).wait_stream(self._aux)
            self._forked = False

    # ------------------------------------------------------------------ algorithmic bytes (SURVEY 8d)
    def ctx_counters(self):
        """(representative rows, CSR entries of the representative rows) of the current batch, or None when layer 1
        is evaluated per row (host ints; synchronises)."""
        if not self._dedup0():
            return None
        st = self.cur.ctx_stats.cpu().numpy()
        return int(st[0]), int(st[2])

    def counters(self):
        """Realised N_l / E_l of the current batch (host ints; synchronises)."""
        s = self.sizes.cpu().numpy()
        N = [int(s[i]) for i in range(4)]
        if self._tiny_on():          # per-subgraph row pointers: subgraph g's n_g + 1 pointers start at lo_g + g
            B, gp, E = self.cur_B, self._gp.cpu().numpy(), [int(s[4])]
            for l in (1, 2):
                rp = self._rowptr_f[l - 1].cpu().numpy()
                first = gp[l][:B] + np.arange(B)
                E.append(int((rp[first + (gp[l][1:B + 1] - gp[l][:B])] - rp[first]).sum()))
            return N, E
        E = [int(s[4]), int(self.rowptr[1][N[1]].item()), int(self.rowptr[2][N[2]].item())]
        return N, E


def algorithmic_bytes(N, E, F, B, s_adj, training=True):
    """Compulsory traffic of one step per SURVEY.md 8(d) from realised counters.
    N = [N0..N3], E = [E0, E1, E2] (E3 is never materialised and counted as 0)."""
    E = list(E) + [0]
    extract = 4 * s_adj + 9 * N[0] + 8 * E[0] + 8 * N[0] * F
    idx = 4 * sum(3 * E[l] + 2 * E[l + 1] + 2 * N[l] + 2 * N[l + 1] for l in range(3))
    fwd = 4 * (N[0] * F + sum(2 * N[l] * H + N[l + 1] * H for l in range(3)) + sum(N[l] * H for l in (1, 2))) + idx + 4 * B * 3 * 256
    if not training:
        return extract + fwd
    fin = [F, H, H]
    bwd = 4 * (sum(N[l + 1] * H + 3 * N[l] * H + N[l] * fin[l] for l in range(3)) + sum(N[l] * H for l in (1, 2))) + idx
    return extract + fwd + bwd
