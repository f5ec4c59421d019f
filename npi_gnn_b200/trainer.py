"""Training / evaluation / scoring loops on the fused engine.

Mirrors the reference's ``train()`` (src/train_with_twoDataset.PY:46-57: zero_grad, forward,
nll_loss, backward, optimizer.step per batch, batches in a fixed order with the last one
partial), the LR rule of :158-160 (x0.95 when the epoch loss rises), the evaluation sweep of
src/methods.py:87-127 and the scoring rule of src/case_study_negativeSample.py:235-253 -- with
the whole step (device-side batch assembly, GPU extraction, forward, backward, Adam) enqueued on
one stream and replayed from a CUDA graph.

Data parallelism (SURVEY 8e): one process per GPU; rank r takes the r-th contiguous slice of
every global batch, the loss gradient is pre-scaled by 1/B_global and ONE sum all-reduce of the
flat 97,602-float gradient buffer runs per step; Adam state is replicated.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import _lib as L
from . import ops
from .engine import Engine, FlatParams, context_policy


def shard_of_batch(order, per_rank_batch, world_size, rank, gb, cost=None):
    """Pair indices of ``rank`` for global batch ``gb``: the global batch is the gb-th run of
    per_rank_batch*world_size entries of the fixed ``order``; rank r takes its r-th contiguous
    slice (a short last batch is split as evenly as possible, trailing ranks may get nothing).
    Returns (indices, size of the global batch).

    ``cost`` (per pair, indexed like the pair set: e.g. cached nodes + edges of the subgraph): the
    SAME global batch is dealt out by size instead of by position -- pairs in descending cost, each to
    the rank with the smallest load that still has a free seat (every rank keeps the contiguous
    scheme's seat count, so buffers and captured graphs are unchanged).  A data-parallel step lasts as
    long as its slowest rank; subgraph sizes span 2 ... 3,400 nodes, so contiguous slices of 200 differ
    by +-10 % in work (bench.py dp_breakdown).  The loss is a sum over the global batch and dropout is
    keyed by the pair index, so the assignment changes nothing but the order of a floating-point sum."""
    GB = per_rank_batch * world_size
    idx = order[gb * GB:(gb + 1) * GB]
    per = (len(idx) + world_size - 1) // world_size
    if cost is None or world_size == 1:
        return idx[rank * per:(rank + 1) * per], len(idx)
    seats = [max(0, min(per, len(idx) - r * per)) for r in range(world_size)]
    c = np.asarray(cost, dtype=np.float64)[idx]
    load = [0.0] * world_size
    mine = []
    for j in np.argsort(-c, kind="stable"):
        r = min((r for r in range(world_size) if seats[r] > 0), key=lambda r: (load[r], r))
        seats[r] -= 1
        load[r] += c[j]
        if r == rank:
            mine.append(j)
    mine = np.sort(np.asarray(mine, dtype=np.int64))            # keep the global batch's order inside the shard
    return idx[mine], len(idx)


class Trainer:
    def __init__(self, pairset, batch_size=200, lr=1e-3, weight_decay=1e-3, seed=0, params=None,
                 world_size=1, rank=0, use_cuda_graph=True, allreduce=None, order=None, exchange=None, balance=True):
        """batch_size is the PER-RANK batch; the global batch is batch_size*world_size.
        Gradient exchange under DP: ``exchange`` (a peer.PeerExchange: sum over peer memory fused
        into the Adam kernel, whole step in one CUDA graph) or ``allreduce`` (a callable doing a
        sum all-reduce of a tensor, e.g. NCCL -- two graphs with the collective between them)."""
        self.ps = pairset
        g = pairset.graph
        self.device = g.device
        self.B = int(batch_size)
        self.world_size, self.rank = int(world_size), int(rank)
        self.allreduce = allreduce
        self.exchange = exchange
        if self.world_size > 1 and allreduce is None:
            raise L.NPIError("world_size > 1 needs an allreduce callable (see npi_gnn_b200.dist)")
        if exchange is not None and (exchange.world != self.world_size or exchange.rank != self.rank):
            raise L.NPIError("peer exchange was built for another world/rank")
        P = len(pairset)
        self.order = np.arange(P, dtype=np.int64) if order is None else np.asarray(order, dtype=np.int64)
        # data parallel: deal every global batch out by cached subgraph size (see shard_of_batch)
        self.cost = (np.asarray(pairset.n_h, dtype=np.float64) + np.asarray(pairset.e_h, dtype=np.float64)) \
            if (balance and self.world_size > 1 and os.environ.get("NPI_DP_BALANCE", "1") != "0") else None
        self._shards = {}
        n0, e0, mx = self._caps()
        # one probed batch decides whether conv1 (and its backward) runs per layer-1 context (engine.context_policy)
        idx0, _ = self._rank_indices(0)
        pi0 = torch.zeros(self.B, dtype=torch.int32)
        pi0[:len(idx0)] = torch.as_tensor(np.asarray(idx0, dtype=np.int32))
        self.ctx_policy = context_policy(pairset, min(self.B, max(len(idx0), 1)), n0, e0, mx, self.device, pair_index=pi0.to(self.device))
        self.engine = Engine(g.F, self.B, n0, e0, mx, device=self.device, graph=g, contexts=self.ctx_policy[0],
                             ctx_bwd=self.ctx_policy[1])
        self.params = params if params is not None else FlatParams(g.F, self.device).init_reference(
            torch.Generator().manual_seed(seed))
        # gradients: one flat buffer, or -- under the peer exchange -- one per batch slot inside the peer allocation
        # (alternating buffers make the exchange's closing handshake unnecessary, peer.py)
        if exchange is not None:
            self._grads_slot = [FlatParams(g.F, self.device, flat=exchange.grads2[b]) for b in range(2)]
        else:
            one = FlatParams(g.F, self.device)
            self._grads_slot = [one, one]
        self.grads = self._grads_slot[0]
        self.m = torch.zeros_like(self.params.flat)
        self.v = torch.zeros_like(self.params.flat)
        self.lr_dev = torch.tensor([lr], dtype=torch.float32, device=self.device)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.lr, self.wd, self.seed = float(lr), float(weight_decay), int(seed)
        self.loss_acc = torch.zeros(1, dtype=torch.float32, device=self.device)
        # the epoch plan (which pairs form which batch) is fixed, like the reference's un-reshuffled
        # DataLoader (src/train_with_twoDataset.PY:142); keep it resident: [num_batches, B]
        nb = self.num_batches()
        plan = np.zeros((max(nb, 1), self.B), dtype=np.int32)
        for gb in range(nb):
            idx, _ = self._rank_indices(gb)
            plan[gb, :len(idx)] = idx
        self.plan_h = torch.from_numpy(plan).pin_memory()
        self.plan_dev = self.plan_h.to(self.device)
        # pair indices of the batch held by each engine slot (start from a batch that is known to fit)
        self.pair_index = [self.plan_dev[0].clone() for _ in range(2)]
        self._loss_pin = torch.zeros(1, dtype=torch.float32).pin_memory()
        self.use_graph = bool(use_cuda_graph)
        self._graphs = {}                 # slot parity -> (fwd/bwd[/update] graph, update graph or None)
        self._side = None                 # side stream of the prefetching extraction
        self._slot_gb = [None, None]      # which global batch each engine slot currently holds
        self.kernel_launches_per_step = None

    # ------------------------------------------------------------------ batch plan
    def _rank_indices(self, gb):
        # cached: step() asks twice per step, and dealing a global batch out by size is O(batch * world) in Python
        # (uncached it put 4 ms of host time into every 8-GPU step -- gpurun_out/r2j)
        hit = self._shards.get(gb)
        if hit is None:
            hit = self._shards[gb] = shard_of_batch(self.order, self.B, self.world_size, self.rank, gb, self.cost)
        return hit

    def num_batches(self):
        GB = self.B * self.world_size
        return (len(self.order) + GB - 1) // GB

    def _caps(self):
        n0 = e0 = mx = 2
        for gb in range(self.num_batches()):
            idx, _ = self._rank_indices(gb)
            if len(idx):
                n0 = max(n0, int(self.ps.n_h[idx].sum())); e0 = max(e0, int(self.ps.e_h[idx].sum()))
                mx = max(mx, int(self.ps.n_h[idx].max()))
        return n0, e0, mx

    # ------------------------------------------------------------------ one step
    def _enqueue_extract(self, count, slot):
        """Batch assembly + GPU extraction (+ by-serial index) of the pairs in pair_index[slot]."""
        self.engine.load_pairs(self.ps, count=count, pair_index=self.pair_index[slot], slot=slot)

    def _enqueue_compute(self, global_count):
        """Forward + loss + backward on the engine's current slot; gradients (pre-scaled by
        1/B_global) land in grads.flat."""
        eng = self.engine
        scale = 1.0 / float(global_count)
        eng.forward(self.params, training=True, seed=self.seed, step_dev=self.step_dev,
                    sample_ids=self.pair_index[eng.slot], compute_loss=True, loss_scale=scale, defer_loss=True,
                    fuse_head_delta=True)
        self.grads = self._grads_slot[eng.slot]
        eng.backward(self.params, self.grads, loss_scale=scale)

    def _enqueue_fwd_bwd(self, count, global_count):
        """Sequential form (no prefetch): extraction into the current slot, then compute."""
        self._enqueue_extract(count, self.engine.slot)
        self._enqueue_compute(global_count)

    def _adam(self):
        if self.exchange is not None:        # gradient sum over peer memory inside the optimizer kernel
            self.exchange.allreduce_adam(self.params.flat, self.m, self.v, self.lr_dev, self.step_dev,
                                         0.9, 0.999, 1e-8, self.wd, 1.0, buf=self.engine.slot)
        else:
            ops.adam_l2_step(self.params.flat, self.grads.flat, self.m, self.v, self.lr_dev, self.step_dev,
                             0.9, 0.999, 1e-8, self.wd, 1.0)

    def _begin_grads(self, buf):
        """Before anything writes the gradient buffer of slot ``buf``: under the double-buffered peer exchange a
        buffer used twice in a row (capture warm-up then replay, the eager tail of an epoch) needs all ranks to have
        finished reading it (peer.PeerExchange.begin_step).  Every rank takes the same branch: slots follow the
        global batch sequence."""
        if self.exchange is not None:
            self.exchange.begin_step(buf)

    def _enqueue_update(self, global_count):
        # engine.loss holds this rank's share of the global mean loss; ranks are summed by the caller.  The accumulation
        # runs next to the optimizer (auxiliary stream), not behind it: nothing on the device waits for it
        with self.engine._branch():
            ops.scalar_axpy(self.loss_acc, self.engine.loss, float(global_count))
        self._adam()
        self.engine._join()

    def _enqueue(self, count, global_count):
        self._enqueue_fwd_bwd(count, global_count)
        if self.world_size > 1 and self.exchange is None:
            self.allreduce(self.grads.flat)
        self._enqueue_update(global_count)

    def _enqueue_overlapped(self, GB):
        """Compute on the current slot while the OTHER slot's batch is extracted on a side stream
        (the extraction is integer, latency-bound work that hides under the bandwidth-bound model
        kernels).  Fork/join with events so the pair can be captured in one CUDA graph."""
        main = torch.cuda.current_stream(self.device)
        nxt = 1 - self.engine.slot

        def fork():
            self._side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(self._side):
                self._enqueue_extract(self.B, nxt)
        # the extraction's 200 fat CTAs (1024 threads, 76 KB of shared memory) take whole SMs for ~100 us: forked behind the
        # first aggregation, the most bandwidth-hungry kernel of the step, they sit next to the latency-bound per-graph top-k
        # kernels (242 k subgraphs/s, against 234 k forked at the start of the step and 237-240 k later in the forward pass)
        self.engine.hooks = {"fwd_agg0": fork}
        try:
            self._enqueue_compute(GB)
        finally:
            self.engine.hooks = {}
        main.wait_stream(self._side)

    def _state(self):
        return (self.params.flat, self.m, self.v, self.step_dev, self.loss_acc)

    def _capture(self, slot):
        """Capture the step for engine slot ``slot`` as CUDA graph(s): [compute on slot || extract
        the next batch into the other slot] + optimizer in one graph on a single GPU; under DP two
        graphs (forward+backward, optimizer) with the NCCL all-reduce issued between them."""
        GB = self.B * self.world_size
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        # default priority: a high-priority chain only made the auxiliary stream's GEMMs delay later links (0.6915 vs 0.6834 ms)
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        keep = [t.clone() for t in self._state()]
        self.engine.use_slot(slot)
        with torch.cuda.stream(s):                       # warm-up outside capture (lazy kernel attributes)
            self._begin_grads(slot)
            self._enqueue_overlapped(GB)
            self._enqueue_update(GB)
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        g1 = torch.cuda.CUDAGraph()
        if self.world_size == 1 or self.exchange is not None:
            with torch.cuda.graph(g1, stream=s):
                self._enqueue_overlapped(GB)
                self._enqueue_update(GB)
            self._graphs[slot] = (g1, None)
        else:
            g2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1, stream=s):
                self._enqueue_overlapped(GB)
            with torch.cuda.graph(g2, stream=s):
                self._enqueue_update(GB)
            self._graphs[slot] = (g1, g2)
        for t, k in zip(self._state(), keep):
            t.copy_(k)

    def _stage_indices(self, gb, from_host, slot=None):
        # plan_h is pinned and immutable, so the async H2D copy needs no staging ring
        slot = self.engine.slot if slot is None else slot
        src = self.plan_h[gb] if from_host else self.plan_dev[gb]
        self.pair_index[slot].copy_(src, non_blocking=True)

    def _is_full(self, gb):
        idx, gcount = self._rank_indices(gb)
        return len(idx) == self.B and gcount == self.B * self.world_size

    def step(self, gb, sync_loss=False, from_host=False, next_gb=None):
        """Global batch ``gb`` of the epoch plan.  from_host: the batch's pair indices come from
        pinned host memory (4*B bytes H2D) instead of the resident plan.  sync_loss: read the
        step's loss back to the host (what the reference does with loss.item()).  next_gb: the
        batch the caller will ask for next; its enclosing subgraphs are extracted on a side stream
        while this step computes (software pipelining of the extraction)."""
        idx, gcount = self._rank_indices(gb)
        cnt = len(idx)
        eng = self.engine
        full = (cnt == self.B and gcount == self.B * self.world_size)
        if full and self.use_graph:
            # which slot holds (or will hold) this batch
            if self._slot_gb[1 - eng.slot] == gb:
                eng.use_slot(1 - eng.slot)
            cur = eng.slot
            if self._slot_gb[cur] != gb:                 # not prefetched: extract it now, in order
                self._stage_indices(gb, from_host, cur)
                self._enqueue_extract(self.B, cur)
                self._slot_gb[cur] = gb
            if cur not in self._graphs:
                # the capture's warm-up extracts the OTHER slot with count = B: its pair list must be a full
                # plan row (a zero-padded partial row there would extract B-cnt extra copies of pair 0 and
                # could exceed the extraction buffers)
                self._stage_indices(gb, False, 1 - cur)
                self._capture(cur)
                self._slot_gb[1 - cur] = None            # the capture warm-up extracted into the other slot
            nxt = next_gb if (next_gb is not None and self._is_full(next_gb)) else gb
            self._stage_indices(nxt, from_host, 1 - cur)
            self._slot_gb[1 - cur] = nxt
            g1, g2 = self._graphs[cur]
            self._begin_grads(cur)
            g1.replay()
            if self.exchange is not None:
                self.exchange.note_used(cur)
            if g2 is not None:
                self.allreduce(self.grads.flat)
                g2.replay()
        elif cnt > 0:
            self._stage_indices(gb, from_host)
            self._slot_gb[eng.slot] = None
            self._begin_grads(eng.slot)
            self._enqueue(cnt, gcount)
        elif self.world_size > 1:       # empty shard of a short last batch still joins the all-reduce
            self._begin_grads(eng.slot)
            self.grads = self._grads_slot[eng.slot]
            self.grads.flat.zero_()
            if self.exchange is None:
                self.allreduce(self.grads.flat)
            self._adam()
        if sync_loss:
            self._loss_pin.copy_(self.engine.loss, non_blocking=False)
            return float(self._loss_pin[0])
        return None

    def train_epoch(self):
        """One pass over the fixed order; returns loss_all / len(dataset) like the reference."""
        self.loss_acc.zero_()
        nb = self.num_batches()
        for gb in range(nb):
            self.step(gb, next_gb=gb + 1 if gb + 1 < nb else None)
        if self.world_size > 1:
            self.allreduce(self.loss_acc)
        if self.exchange is not None:
            self.exchange.check()
        self.engine.check_overflow()
        return float(self.loss_acc.item()) / max(len(self.order), 1)

    def set_lr(self, lr):
        self.lr = float(lr)
        self.lr_dev.fill_(self.lr)

    def fit(self, epochs, gamma=0.95, on_epoch=None):
        """src/train_with_twoDataset.PY:152-160: lr *= gamma whenever the epoch loss increased."""
        last = float("inf")
        hist = []
        for ep in range(epochs):
            loss = self.train_epoch()
            if loss > last:
                self.set_lr(self.lr * gamma)
            last = loss
            hist.append(loss)
            if on_epoch is not None:
                on_epoch(ep + 1, loss, self)
        return hist


class Scorer:
    """Eval-mode forward over a PairSet: confusion counts (src/methods.py:87-127) or positive-class
    probabilities p = exp(logp[:,1]) (src/case_study_negativeSample.py:235-253).  Pairs are
    processed in contiguous slices; under sharding rank r takes the r-th contiguous range, no
    communication (SURVEY 8e).  Full batches replay one CUDA graph per batch slot: [forward on this
    slot || extraction of the next batch into the other slot]; the short tail runs eagerly."""

    def __init__(self, pairset, params, batch_size=200, world_size=1, rank=0, use_cuda_graph=True, index=None):
        """``index`` (optional): score pairset[index] in that order instead of the whole pair set
        (a shuffled / sliced dataset view); positions reported by ``batches()`` then refer to it."""
        self.ps, self.params = pairset, params
        g = pairset.graph
        self.device = g.device
        self.index = None if index is None else np.ascontiguousarray(index, dtype=np.int64)
        P = len(pairset) if self.index is None else len(self.index)
        self.P, self.world_size = P, int(world_size)
        per = (P + world_size - 1) // world_size
        self.lo, self.hi = min(P, rank * per), min(P, (rank + 1) * per)
        self.B = int(batch_size)
        n0 = e0 = mx = 2
        if self.hi > self.lo:
            own = np.arange(self.lo, self.hi) if self.index is None else self.index[self.lo:self.hi]
            n0, e0, mx = (max(2, v) for v in pairset.batch_caps(self.B, own))
        self.ctx_policy = context_policy(pairset, self.B, n0, e0, mx, g.device, first=self.lo) \
            if (self.index is None and self.hi - self.lo >= self.B) else (None, None)
        self.engine = Engine(g.F, self.B, n0, e0, mx, device=g.device, graph=g, need_backward=False, contexts=self.ctx_policy[0])
        self.use_graph = bool(use_cuda_graph)
        self._arange = torch.arange(self.B, dtype=torch.int32, device=self.device)
        self.pair_index = [self._arange.clone() for _ in range(2)]
        self._graphs = {}
        self._side = None
        self.batches_scored = 0
        self._from_host = False
        self._host_index = None
        if self.index is not None:       # this rank's slice of the view
            self._host_index = _padded_host_index(self.index[self.lo:self.hi], self.B)

    def _set_index(self, slot, first):
        if self._from_host or self.index is not None:     # pair indices from pinned host memory (4*B bytes H2D)
            self.pair_index[slot].copy_(self._host_index[first - self.lo:first - self.lo + self.B], non_blocking=True)
        else:
            torch.add(self._arange, int(first), out=self.pair_index[slot])

    def _extract(self, slot):
        self.engine.load_pairs(self.ps, count=self.B, pair_index=self.pair_index[slot], slot=slot)

    def _overlapped(self):
        main = torch.cuda.current_stream(self.device)
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            self._extract(1 - self.engine.slot)
        self.engine.forward(self.params, training=False)
        main.wait_stream(self._side)

    def _capture(self, slot):
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        self.engine.use_slot(slot)
        with torch.cuda.stream(s):                       # warm-up outside capture (lazy kernel attributes)
            self._overlapped()
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            self._overlapped()
        self._graphs[slot] = (g, self.params.flat.data_ptr())

    def batches(self, from_host=False):
        """Yields (first, count, logp[:count]) over this rank's range; the consumer enqueues its
        reads on the current stream before asking for the next batch.  from_host: every batch's
        pair indices are copied from pinned host memory instead of being generated on the device."""
        self._from_host = bool(from_host)
        if from_host and self._host_index is None:
            self._host_index = torch.arange(self.lo, max(self.hi, self.lo + self.B), dtype=torch.int32).pin_memory()
        return self._batches()

    def _batches(self):
        eng, B = self.engine, self.B
        nfull = (self.hi - self.lo) // B
        done = self.lo
        if self.use_graph and nfull >= 2:
            eng.use_slot(0)
            self._set_index(0, self.lo)
            self._extract(0)
            for b in range(nfull):
                cur = b & 1
                first = self.lo + b * B
                eng.use_slot(cur)
                self._set_index(1 - cur, first + B if b + 1 < nfull else first)
                if cur not in self._graphs or self._graphs[cur][1] != self.params.flat.data_ptr():
                    self._capture(cur)
                self._graphs[cur][0].replay()
                self.batches_scored += 1
                yield first, B, eng.logp[:B]
            done = self.lo + nfull * B
        for first in range(done, self.hi, B):
            cnt = min(B, self.hi - first)
            if self.index is None:
                eng.load_pairs(self.ps, first=first, count=cnt)
            else:
                self._set_index(eng.slot, first)
                eng.load_pairs(self.ps, count=cnt, pair_index=self.pair_index[eng.slot])
            self.batches_scored += 1
            yield first, cnt, eng.forward(self.params, training=False)

    def confusion(self, threshold=-1.0):
        counts = torch.zeros(4, dtype=torch.int64, device=self.ps.graph.device)
        for first, cnt, logp in self.batches():
            ops.confusion_counts(logp, self.engine.y_b, cnt, threshold, counts)
        TP, FN, TN, FP = [int(v) for v in counts.cpu()]
        return TP, FN, TN, FP

    def probabilities(self, out=None):
        if out is None:
            out = torch.empty(self.hi - self.lo, dtype=torch.float32, device=self.ps.graph.device)
        for first, cnt, logp in self.batches():
            torch.exp(logp[:cnt, 1], out=out[first - self.lo:first - self.lo + cnt])
        return out

    def rank_metrics(self, curve=False):
        """ROC AUC, average precision and trapezoidal PR AUC (``rank_metrics``) of the probabilities that
        ``probabilities()`` returns against the pair labels, plus ``confusion`` = (TP, FN, TN, FP) of the argmax rule,
        all from ONE sweep.  With world_size > 1 every rank's shard is gathered (torch.distributed must be initialised)
        and every rank computes the same, bit-identical result over all pairs -- the confusion counts included."""
        self._require_process_group("rank_metrics")
        n = self.hi - self.lo
        scores = torch.empty(n, dtype=torch.float32, device=self.device)
        labels = torch.empty(n, dtype=torch.int32, device=self.device)
        counts = torch.zeros(4, dtype=torch.int64, device=self.device)
        for first, cnt, logp in self.batches():
            o = first - self.lo
            torch.exp(logp[:cnt, 1], out=scores[o:o + cnt])
            labels[o:o + cnt].copy_(self.engine.y_b[:cnt])
            ops.confusion_counts(logp, self.engine.y_b, cnt, -1.0, counts)
        if self.world_size > 1:
            from . import dist as D
            D.allreduce_sum(counts)
        out = rank_metrics(self._gathered(scores), self._gathered(labels), curve=curve)
        out["confusion"] = tuple(int(v) for v in counts.cpu())
        return out

    def top_partners(self, k):
        """The ``k`` most likely partners of every node, from ONE sweep of ``probabilities()``: the pairs grouped by their
        RNA and by their protein (``top_k_by_group`` with the node serial as group id, so row s belongs to node s; rows of
        nodes of the other type, or in no pair, have count 0).  Returns {"rna": ..., "protein": ...}, each
        dict(partner, prob, count) of device tensors: partner int32 [num_nodes, k] = serial of the other endpoint by
        descending probability (-1 past count), prob float32 [num_nodes, k] (NaN past count), count int32 [num_nodes].
        Ties break by position in the pair set (in ``index`` order when a view was given).  With world_size > 1 every
        rank's shard is gathered (torch.distributed must be initialised) and every rank computes the same,
        bit-identical result over all pairs."""
        _check_k(k, "top_partners")
        probs, pairs, _ = self._view_probabilities("top_partners")
        out = {}
        for name, own, other in (("rna", 0, 1), ("protein", 1, 0)):
            r = top_k_by_group(probs, pairs[:, own].contiguous(), self.ps.graph.num_nodes, k)
            hit = r["pos"] >= 0
            partner = torch.where(hit, pairs[:, other][r["pos"].clamp(min=0).long()], -1)
            out[name] = dict(partner=partner, prob=r["score"], count=r["count"])
        return out

    def partner_ranks(self, hits=(1, 3, 10)):
        """Where every held-out interaction ranks among its node's candidates, per RNA and per protein, from ONE sweep of
        ``probabilities()`` and the pair labels: ``group_rank_metrics`` with the pairs grouped by their RNA ("rna") and by
        their protein ("protein"), node serials as group ids.  Pairs with label 1 are the queries, pairs with label 0
        their competitors; returns {"rna": ..., "protein": ...} of group_rank_metrics dicts (MRR, Hits@K, per-node AUC).

        Intended use: build the graph with the test pairs masked, then score one pair set made of the test positives
        (label 1), the test negatives (label 0) and ``BipartiteGraph.candidate_pairs()`` (label 0)::

            cand = g.candidate_pairs()
            pairs = np.concatenate([test_pos, test_neg, cand])
            y = np.concatenate([np.ones(len(test_pos)), np.zeros(len(test_neg)), np.zeros(len(cand))])
            Scorer(PairSet(g, pairs, y), params).partner_ranks()

        Honours an ``index`` view.  The result does not depend on the order of the pairs.  With world_size > 1 every
        rank's shard is gathered (torch.distributed must be initialised) and every rank computes the same, bit-identical
        result over all pairs."""
        ks = _hits_cutoffs(hits, "partner_ranks")
        probs, pairs, labels = self._view_probabilities("partner_ranks")
        return {name: group_rank_metrics(probs, labels, pairs[:, own].contiguous(), self.ps.graph.num_nodes, ks)
                for name, own in (("rna", 0), ("protein", 1))}

    def _require_process_group(self, who):
        from . import dist as D
        if self.world_size > 1 and not D.dist.is_initialized():
            raise L.NPIError("Scorer.%s with world_size > 1 needs an initialised torch.distributed process group" % who)

    def _gathered(self, t):
        """This rank's shard ``t`` of a per-pair tensor -> the whole view's, gathered across ranks."""
        if self.world_size == 1:
            return t
        from . import dist as D
        return D.gather_shards(t, self.P)

    def _view_probabilities(self, who):
        """(probabilities, pairs, labels) of the whole view, from one sweep of ``probabilities()`` gathered across ranks;
        ``who`` names the calling method in the process-group error."""
        self._require_process_group(who)
        probs = self._gathered(self.probabilities())
        pairs, labels = self.ps.pairs, self.ps.y
        if self.index is not None:
            idx = torch.from_numpy(self.index).to(self.device)
            pairs, labels = pairs[idx], labels[idx]
        return probs, pairs, labels


def _padded_host_index(index, B):
    """The pair indices of a view as int32 host memory (pinned when CUDA is available), padded with ``B`` copies of the
    last entry so that a full-batch read never runs off the end."""
    own = np.asarray(index).astype(np.int32)
    host = torch.from_numpy(np.concatenate([own, np.full(B, own[-1] if len(own) else 0, dtype=np.int32)]))
    return host.pin_memory() if torch.cuda.is_available() else host


class Explainer:
    """Why the model scores a pair as it does: gradient x input attribution of every pair's target to the nodes and the
    input features of its enclosing subgraph (include/npi.h npi_input_attribution for the semantics).  One eager sweep
    on the fused engine: per batch the extraction, the evaluation-mode forward, a backward pass seeded on the target
    class and one call of npi_input_attribution.

    The engine runs with ``contexts=False``: the per-context backward of conv1 sums the gradient rows of identical
    layer-1 contexts across subgraphs, which would mix pairs.  The small-subgraph path stays where the engine's size
    rule selects it (its layer-1 gradient is per row).  The weight gradients the backward pass also computes go to a
    scratch buffer and are discarded.

    ``index`` (optional): explain pairset[index] in that order; positions of the result refer to the view, so a pair
    listed twice appears twice.  To explain the output of ``Scorer.top_partners``, build a PairSet of the (node,
    partner) pairs it lists on the same graph and pass it here; ``top_nodes`` then names the nodes behind each score."""

    def __init__(self, pairset, params, batch_size=200, index=None):
        self.ps, self.params = pairset, params
        self.B = int(batch_size)
        if self.B < 1:
            raise ValueError("Explainer: batch_size = %d, expected >= 1" % self.B)
        P = len(pairset)
        if index is not None:
            index = np.ascontiguousarray(index, dtype=np.int64).reshape(-1)
            if len(index) and (index.min() < 0 or index.max() >= P):
                raise ValueError("Explainer: index entries must lie in [0, %d)" % P)
        self.index = index
        self.P = P if index is None else len(index)
        if self.P == 0:
            raise ValueError("Explainer: nothing to explain (empty pair set or index view)")
        n = pairset.n_h if index is None else pairset.n_h[index]
        self.n_rows = np.asarray(n, dtype=np.int64)        # rows of every pair's subgraph, in view order
        n0, e0, mx = (max(2, v) for v in pairset.batch_caps(self.B, index))
        g = pairset.graph
        self.device = g.device
        self.engine = Engine(g.F, self.B, n0, e0, mx, device=self.device, graph=g, need_backward=True, contexts=False)
        self.scratch = FlatParams(g.F, self.device)
        self.ws = torch.empty(ops.input_attribution_workspace_bytes(self.engine.n_cap[0], self.B, g.F), dtype=torch.uint8,
                              device=self.device)
        self._seed = torch.zeros(self.B, 2, dtype=torch.float32, device=self.device)
        self._onehot = torch.zeros(self.B, 2, dtype=torch.float32, device=self.device)
        self._pair_index = None
        if index is not None:
            self._host_index = _padded_host_index(index, self.B)
            self._pair_index = torch.zeros(self.B, dtype=torch.int32, device=self.device)

    def explain(self, target=1, wrt="logp", full=False):
        """Attributions of every pair of the view.  ``target``: the class whose score is explained (1 = interacts);
        ``wrt``: "logp" explains logp[p, target], "prob" explains exp(logp[p, target]); ``full``: also return the input
        gradient of every row.  Returns a dict of device tensors:
          logp          float32 [P, 2]  the evaluation-mode log-probabilities
          node_ptr      int64 [P + 1]   rows node_ptr[p] .. node_ptr[p+1]-1 belong to pair p
          node, hop     int32 [R]       node serial and hop distance of every row, in extraction order (the target pair
                                        first)
          node_attr     float32 [R]     sum_c x_i[c] d target / d x_i[c]   (gradient x input per row)
          feature_attr  float32 [P, F]  sum over the pair's rows of x_i[c] d target / d x_i[c]; column 0 is the
                                        structural label, columns 1.. the feature table's
          grad_x        float32 [R, F]  d target / d x_i (full=True only)
        Runs eagerly; synchronises once, at the end (a batch that overflowed the extraction buffers raises NPIError).
        Bad arguments raise ValueError before the device is touched."""
        if target not in (0, 1):
            raise ValueError("explain: target = %r, expected class 0 or 1" % (target,))
        if wrt not in ("logp", "prob"):
            raise ValueError("explain: wrt = %r, expected \"logp\" or \"prob\"" % (wrt,))
        target = int(target)
        g, F, P, B = self.ps.graph, self.ps.graph.F, self.P, self.B
        node_ptr_h = np.zeros(P + 1, dtype=np.int64)
        np.cumsum(self.n_rows, out=node_ptr_h[1:])
        R = int(node_ptr_h[-1])
        if full:
            need = R * F * 4
            free = torch.cuda.mem_get_info(self.device)[0]
            if need > free:
                raise ValueError("explain: full=True needs %d bytes for grad_x [%d, %d], %d bytes of device memory are free"
                                 % (need, R, F, free))
        dev = self.device
        out = dict(logp=torch.empty(P, 2, dtype=torch.float32, device=dev),
                   node_ptr=torch.from_numpy(node_ptr_h).to(dev),
                   node=torch.empty(R, dtype=torch.int32, device=dev), hop=torch.empty(R, dtype=torch.int32, device=dev),
                   node_attr=torch.empty(R, dtype=torch.float32, device=dev),
                   feature_attr=torch.empty(P, F, dtype=torch.float32, device=dev))
        grad_x = torch.empty(R, F, dtype=torch.float32, device=dev) if full else None
        if full:
            out["grad_x"] = grad_x
        eng, w1 = self.engine, self.params.view("conv1.weight")
        self._onehot.zero_()
        self._onehot[:, target] = 1.0
        if wrt == "logp":
            self._seed.copy_(self._onehot)
        for first in range(0, P, B):
            cnt = min(B, P - first)
            if self.index is None:
                eng.load_pairs(self.ps, first=first, count=cnt)
            else:
                self._pair_index.copy_(self._host_index[first:first + B], non_blocking=True)
                eng.load_pairs(self.ps, count=cnt, pair_index=self._pair_index)
            logp = eng.forward(self.params, training=False)
            if wrt == "prob":            # d exp(logp_c) / d logp_c = p_c
                torch.mul(torch.exp(logp), self._onehot[:cnt], out=self._seed[:cnt])
            eng.backward(self.params, self.scratch, d_logp=self._seed[:cnt])
            r0, r1 = int(node_ptr_h[first]), int(node_ptr_h[first + cnt])
            out["logp"][first:first + cnt].copy_(logp)
            out["node"][r0:r1].copy_(eng.gid[:r1 - r0])
            out["hop"][r0:r1].copy_(eng.dist[:r1 - r0])
            ops.input_attribution(eng.big, eng.gid, eng.dist, eng._gp[0], cnt, r1 - r0, g.table, F, w1,
                                  out["node_attr"][r0:r1], out["feature_attr"][first:first + cnt], self.ws,
                                  grad_x=None if grad_x is None else grad_x[r0:r1])
        eng.check_overflow()
        return out

    @staticmethod
    def top_nodes(result, k):
        """The ``k`` rows of largest |node_attr| in every pair of an ``explain`` result (``top_k_by_group`` with the pair
        as the group; ties by ascending row, i.e. extraction order).  Returns dict of device tensors: node int32 [P, k]
        (the node serials, -1 past count), attr float32 [P, k] (the signed node_attr, NaN past count), count int32 [P] =
        min(k, rows of the pair)."""
        _check_k(k, "top_nodes")
        na, ptr = result["node_attr"], result["node_ptr"]
        P, R = ptr.numel() - 1, na.numel()
        pair = torch.repeat_interleave(torch.arange(P, dtype=torch.int32, device=na.device), ptr.diff(), output_size=R)
        r = top_k_by_group(na.abs(), pair, P, k)
        hit = r["pos"] >= 0
        row = r["pos"].clamp(min=0).long()
        return dict(node=torch.where(hit, result["node"][row], -1),
                    attr=torch.where(hit, na[row], float("nan")), count=r["count"])


def metrics(TP, FN, TN, FP):
    """Accuracy, Precision, Sensitivity, Specificity, MCC exactly as src/methods.py:107-127."""
    tot = TP + TN + FP + FN
    acc = (TP + TN) / tot if tot else 0
    pre = TP / (TP + FP) if (TP + FP) else 0
    sen = TP / (TP + FN) if (TP + FN) else 0
    den = ((TP + FP) * (TP + FN) * (TN + FP) * (TN + FN)) ** 0.5
    mcc = (TP * TN - FP * FN) / den if den else 0
    spe = TN / (FP + TN) if (FP + TN) else 0
    return acc, pre, sen, spe, mcc


def _check_k(k, who):
    if not 1 <= int(k) <= 1024:
        raise ValueError("%s: k = %d outside 1..1024" % (who, k))


def _inputs_and_workspace(tensors, workspace_bytes, *args):
    """The CUDA ``tensors`` flattened and contiguous, and a device workspace of workspace_bytes(n, *args) bytes for their
    n items (at least 1)."""
    L.require_cuda(*tensors)
    flat = [t.reshape(-1).contiguous() for t in tensors]
    ws = torch.empty(workspace_bytes(max(flat[0].numel(), 1), *args), dtype=torch.uint8, device=flat[0].device)
    return flat, ws


def _raise_status(st, *messages):
    """Raises NPIError with messages[b] for the lowest bit b set in the nonzero status word ``st`` of an entry point;
    ``messages`` lists the meanings of its status bits 0, 1, ...."""
    for b, msg in enumerate(messages):
        if st >> b & 1:
            raise L.NPIError(msg)


def rank_metrics(scores, labels, curve=False):
    """Threshold-free metrics of CUDA float32 ``scores`` against int32 0/1 ``labels`` in ONE call of npi_rank_curve and
    one synchronising read: dict(auroc, ap, pr_auc_trapz, n_pos, n_neg, twice_u) -- sklearn's roc_auc_score,
    average_precision_score and auc(recall, precision) over precision_recall_curve, the metrics of the reference's
    src/compare_withKmer_noKmer.py.  ``curve=True`` adds the device tensors thresholds (float32), fpr, tpr, precision
    and recall (float64), one entry per distinct score in descending order.  NaN scores or labels other than 0/1 raise
    NPIError; a single class raises ValueError (ROC AUC is undefined)."""
    (scores, labels), ws = _inputs_and_workspace((scores, labels), ops.rank_workspace_bytes)
    n = scores.numel()
    dev = scores.device
    res = torch.zeros(7, dtype=torch.int64, device=dev)     # summary[4] | areas[2] (fp64) | status (int32)
    summary, areas, status = res[:4], res[4:6].view(torch.float64), res[6:7].view(torch.int32)[:1]
    thr = tps = fps = None
    if curve:
        thr = torch.empty(n, dtype=torch.float32, device=dev)
        tps = torch.empty(n, dtype=torch.int32, device=dev)
        fps = torch.empty(n, dtype=torch.int32, device=dev)
    ops.rank_curve(scores, labels, summary, areas, status, ws, thr, tps, fps)
    h = res.cpu()
    st = int(h[6:7].view(torch.int32)[0])
    if st:
        _raise_status(st, "rank_metrics: NaN score", "rank_metrics: label other than 0 or 1")
    n_pos, n_neg, T, twice_u = (int(v) for v in h[:4])
    if n_pos == 0 or n_neg == 0:
        raise ValueError("Only one class present in the labels: ROC AUC is not defined in that case")
    a = h[4:6].view(torch.float64)
    out = dict(auroc=twice_u / (2.0 * n_pos * n_neg), ap=float(a[0]), pr_auc_trapz=float(a[1]),
               n_pos=n_pos, n_neg=n_neg, twice_u=twice_u)
    if curve:
        t, f = tps[:T].double(), fps[:T].double()
        # divided by device tensors (t[-1] = n_pos, f[-1] = n_neg): a host scalar divisor becomes a multiplication by
        # its reciprocal, which is not always the correctly rounded quotient sklearn's tps / tps[-1] gives
        tpr = t / t[-1]
        out.update(thresholds=thr[:T], fpr=f / f[-1], tpr=tpr, precision=t / (t + f), recall=tpr)
    return out


def top_k_by_group(scores, group, num_groups, k):
    """The ``k`` highest of CUDA float32 ``scores`` in every group of int32 ``group`` ids (0 <= id < num_groups), in ONE
    call of npi_group_topk and one synchronising read: dict(pos, score, count) of device tensors -- pos int32
    [num_groups, k], the positions of the group's items by descending score with ties by ascending position (-0.0 and
    +0.0 tie), -1 past count; score float32 [num_groups, k], those scores bit for bit, NaN past count; count int32
    [num_groups] = min(k, group size).  NaN scores or group ids out of range raise NPIError; k outside 1..1024 raises
    ValueError."""
    _check_k(k, "top_k_by_group")
    (scores, group), ws = _inputs_and_workspace((scores, group), ops.group_topk_workspace_bytes, int(num_groups))
    dev = scores.device
    G, k = int(num_groups), int(k)
    pos = torch.empty((G, k), dtype=torch.int32, device=dev)
    score = torch.empty((G, k), dtype=torch.float32, device=dev)
    count = torch.empty(G, dtype=torch.int32, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    ops.group_topk(scores, group, G, k, pos, score, count, status, ws)
    st = int(status.item())
    if st:
        _raise_status(st, "top_k_by_group: NaN score", "top_k_by_group: group id out of range [0, %d)" % G)
    return dict(pos=pos, score=score, count=count)


def _hits_cutoffs(hits, who):
    """The Hits@K cut-offs as a tuple of ints: 1..8 of them, every K in 1 .. 2^31 - 1 (ValueError otherwise)."""
    try:
        ks = tuple(int(k) for k in hits)
    except (TypeError, ValueError):
        raise ValueError("%s: hits must be a sequence of integer cut-offs K, got %r" % (who, hits)) from None
    if not 1 <= len(ks) <= 8 or any(not 1 <= k < 1 << 31 for k in ks):
        raise ValueError("%s: hits = %r, expected 1 to 8 cut-offs K >= 1" % (who, hits))
    return ks


def group_rank_metrics(scores, labels, group, num_groups, hits=(1, 3, 10), per_item=False):
    """Filtered ranking of CUDA float32 ``scores`` per group of int32 ``group`` ids (0 <= id < num_groups), in ONE call of
    npi_group_rank and one synchronising read.  Items with ``labels`` 1 are queries (held-out interactions), items with
    label 0 their competitors (sampled negatives, unlabelled candidates).  Each query is ranked among the competitors of
    its group only, the group's other queries left out: rank = above + tied / 2 + 1 (ties get half credit, -0.0 and +0.0
    tie).  Returns dict:
      mrr              mean of 1 / rank over the ranked queries (those whose group has a competitor)
      hits             {K: fraction of the ranked queries with rank <= K}
      n_queries, n_unranked, n_groups_scored   ranked queries, queries of groups without a competitor, groups with both
                       classes
      auc_macro        fp64 mean of the defined per-group ROC AUCs (NaN if there is none)
      n_pos, n_neg     int32 [num_groups] device tensors; twice_u int64 [num_groups], the exact 2 x Mann-Whitney U
      auc              float64 [num_groups] device tensor, twice_u / (2 n_pos n_neg), NaN without both classes
      above, tied      (per_item=True) int32 [n] device tensors in input order, -1 for competitors
    NaN scores, labels other than 0/1 or group ids out of range raise NPIError.  A bad ``hits`` (1 to 8 cut-offs K >= 1)
    or num_groups < 1 raises ValueError before the device is touched; no ranked query raises ValueError (MRR is
    undefined)."""
    ks = _hits_cutoffs(hits, "group_rank_metrics")
    G = int(num_groups)
    if G < 1:
        raise ValueError("group_rank_metrics: num_groups = %d, expected >= 1" % G)
    (scores, labels, group), ws = _inputs_and_workspace((scores, labels, group), ops.group_rank_workspace_bytes, G)
    n, nh, dev = scores.numel(), len(ks), scores.device
    res = torch.zeros(16, dtype=torch.int64, device=dev)    # summary[3 + nh] | sum_rr | sum of defined AUCs | status
    summary = res[:3 + nh]
    sum_rr, auc_sum = res[11:12].view(torch.float64), res[12:13].view(torch.float64)
    status = res[13:14].view(torch.int32)[:1]
    n_pos = torch.empty(G, dtype=torch.int32, device=dev)
    n_neg = torch.empty(G, dtype=torch.int32, device=dev)
    twice_u = torch.empty(G, dtype=torch.int64, device=dev)
    above = torch.empty(n, dtype=torch.int32, device=dev) if per_item else None
    tied = torch.empty(n, dtype=torch.int32, device=dev) if per_item else None
    ops.group_rank(scores, labels, group, G, ks, n_pos, n_neg, twice_u, summary, sum_rr, status, ws, above, tied)
    both = (n_pos > 0) & (n_neg > 0)
    auc = torch.where(both, twice_u.double() / (2.0 * n_pos.double() * n_neg.double()), float("nan"))
    auc_sum.copy_(torch.where(both, auc, 0.0).sum().reshape(1))
    h = res.cpu()
    st = int(h[13:14].view(torch.int32)[0])
    if st:
        _raise_status(st, "group_rank_metrics: NaN score", "group_rank_metrics: label other than 0 or 1",
                      "group_rank_metrics: group id out of range [0, %d)" % G)
    nq, nu, ng = (int(v) for v in h[:3])
    if nq == 0:
        raise ValueError("group_rank_metrics: no query has a competitor in its group: MRR is not defined in that case")
    f = h[11:13].view(torch.float64)
    out = dict(mrr=float(f[0]) / nq, hits={k: int(h[3 + i]) / nq for i, k in enumerate(ks)},
               n_queries=nq, n_unranked=nu, n_groups_scored=ng,
               auc_macro=float(f[1]) / ng if ng else float("nan"),
               n_pos=n_pos, n_neg=n_neg, twice_u=twice_u, auc=auc)
    if per_item:
        out.update(above=above, tied=tied)
    return out
