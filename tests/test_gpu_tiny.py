"""Small-subgraph path (csrc/tiny.cu: conv1..3 + pool1..3 + readout of one subgraph per CTA, forward and backward)
against the per-layer path and against the fp64 oracle (reference: src/classes.py:59-82 Net_1.forward,
src/train_with_twoDataset.PY:53-54).  The RPI2241-shaped workload of BASELINE.json config 3 is what selects this path by
itself (15 nodes per subgraph); here it is also forced on for odd batches: one subgraph, two-node subgraphs, a batch
shorter than the engine's capacity."""
import numpy as np
import pytest
import torch

from oracle import khop, khop_cwrap, net as onet
from tests.common import load_ckpt, synthetic_bipartite

pytestmark = pytest.mark.gpu

LOGP_ATOL_FORCED = 5e-4
GRAD_REL_FORCED = 1e-3


def _rpi(B, ckpt):
    from npi_gnn_b200 import synth
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    d = synth.rpi2241_shaped(no_kmer=True)
    pairs, ys = synth.train_pairs(d)
    pairs, ys = pairs[:B], ys[:B]
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(synth.masked_pairs(d))
    ps = PairSet(g, pairs, ys, h=2)
    if ckpt is None:
        params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(17))
    else:
        params = FlatParams(g.F, "cuda").load_state_dict(load_ckpt(ckpt))
    return d, g, ps, pairs, ys, params


def _run(ps, g, B, params, tiny, training=True, count=None):
    from npi_gnn_b200.engine import Engine, FlatParams
    n0, e0, mx = ps.batch_caps(B)
    eng = Engine(g.F, B, n0, e0, mx, device="cuda", graph=g, tiny=tiny, contexts=False)
    assert eng.tiny == bool(tiny)
    grads = FlatParams(g.F, "cuda")
    eng.load_pairs(ps, 0, B if count is None else count)
    logp = eng.forward(params, training=training, seed=99, compute_loss=True).clone()
    eng.backward(params, grads)
    torch.cuda.synchronize()
    return eng, logp, grads


def test_rpi2241_selects_the_per_subgraph_path():
    from npi_gnn_b200.engine import Engine
    d, g, ps, pairs, ys, params = _rpi(200, None)
    n0, e0, mx = ps.batch_caps(200)
    assert Engine(g.F, 200, n0, e0, mx, device="cuda", graph=g).tiny
    assert not Engine(g.F, 200, n0, e0, mx, device="cuda", graph=g, tiny=False).tiny


@pytest.mark.parametrize("ckpt", ["ckpt_1223_1_noKmer_20.npz", None])
def test_tiny_matches_per_layer_path(ckpt):
    """Layer 1's aggregation is the same arithmetic in the same order (bit-identical h); the scores and layers 2-3 differ by
    rounding (fp32 FMA here, 3xTF32 on tcgen05 there): log-probs and gradients agree to 1e-5 / 2e-4 where
    the selections agree, which they do unless a score gap is at rounding level."""
    torch.set_flush_denormal(True)
    B = 200
    d, g, ps, pairs, ys, params = _rpi(B, ckpt)
    et, lt, gt = _run(ps, g, B, params, True)
    el, ll, gl = _run(ps, g, B, params, False)
    Nt, Et = et.counters()
    Nl, El = el.counters()
    assert Nt == Nl and Et[0] == El[0]
    n0, n1 = Nt[0], Nt[1]
    assert torch.equal(et.h[0][:n0], el.h[0][:n0])
    # the score's dot product is reduced over 32 lanes here and over 8-lane groups there: rounding only
    assert float((et.z[0][:n0] - el.z[0][:n0]).abs().max()) < 1e-6 and float((et.s[0][:n0] - el.s[0][:n0]).abs().max()) < 1e-6
    assert torch.equal(et.batch[0][:n1], el.batch[0][:n1])
    assert torch.equal(et.drop_mask[:B], el.drop_mask[:B])
    same = all(torch.equal(et.perm[l][:Nt[l + 1]], el.perm[l][:Nt[l + 1]]) for l in range(3))
    print("selections equal:", same, " N", Nt, " E", Et, El)
    if same:
        assert Et == El
        assert torch.equal(et.argmax[0][:B], el.argmax[0][:B])
        assert float((lt - ll).abs().max()) < 1e-5
        for name in gt.views():
            a, b = gt.views()[name].double(), gl.views()[name].double()
            err = float((a - b).abs().max() / max(float(b.abs().max()), 1e-12))
            assert err < 2e-4, (name, err)
    else:
        assert float((lt - ll).abs().max()) < 2e-3


def test_tiny_rerun_bit_identical():
    d, g, ps, pairs, ys, params = _rpi(200, "ckpt_1223_1_noKmer_35.npz")
    e1, l1, g1 = _run(ps, g, 200, params, True)
    e2, l2, g2 = _run(ps, g, 200, params, True)
    assert torch.equal(l1, l2) and torch.equal(g1.flat, g2.flat)
    assert torch.equal(e1.readout, e2.readout)


def _oracle_check(d, pairs, ys, h, mask_keys, eng, logp, grads, params, B):
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    omask = khop.mask_from_keys(og, [tuple(e) for e in mask_keys])
    N, E = eng.counters()
    c = khop_cwrap.collate_batch(og, omask, pairs, ys, h, d["table"])
    assert N[0] == len(c["gid"]) and E[0] == len(c["col"])
    perms = [eng.perm[l][:N[l + 1]].cpu().long() for l in range(3)]
    F = d["table"].shape[1] + 1
    m = onet.Net_1(F).double()
    m.load_state_dict({k: v.double().cpu() for k, v in params.state_dict().items()})
    m.eval()
    bn = onet.batch_namespace(c)
    bn.x = bn.x.double()
    out = m(bn, forced_perms=perms)
    loss = torch.nn.functional.nll_loss(out, bn.y)
    loss.backward()
    err = float((logp[:B].cpu().double() - out.detach()).abs().max())
    assert err < LOGP_ATOL_FORCED, err
    assert abs(float(eng.loss[0]) - float(loss.detach())) < 1e-4
    gv = grads.views()
    for name, p in m.named_parameters():
        ref = p.grad.double()
        got = gv[name].cpu().double()
        e = float((got - ref).abs().max() / max(float(ref.abs().max()), 1e-6))
        assert e < GRAD_REL_FORCED, (name, e)
    for l in range(3):
        assert np.array_equal(eng.batch[l][:N[l + 1]].cpu().numpy(), m.trace.batch[l].numpy())
    for l in range(2):
        assert E[l + 1] == m.trace.edge_index[l].shape[1]
    return N, E


@pytest.mark.parametrize("h,B,count", [(1, 1, 1), (2, 1, 1), (2, 7, 7), (2, 16, 11), (3, 33, 33)])
def test_tiny_odd_batches_vs_oracle(h, B, count):
    """One-subgraph batches, a batch shorter than the engine's capacity, two-node subgraphs (candidate pairs whose only
    edge is the target edge), three hops -- extraction, forward, loss and all 15 gradients against the fp64 oracle forced to
    the CUDA selections (dropout off)."""
    from npi_gnn_b200.engine import Engine, FlatParams
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    torch.set_flush_denormal(True)
    d = synthetic_bipartite(seed=11 + B, n_rna=60, n_prot=25, n_pos=90, n_neg=0, F=8)
    rng = np.random.default_rng(5)
    V = len(d["is_rna"])
    rna = np.nonzero(d["is_rna"])[0]
    prot = np.nonzero(d["is_rna"] == 0)[0]
    edges = d["edges"]
    pick = rng.choice(len(edges), size=max(count - 2, 1), replace=False)
    pairs = [tuple(edges[i]) for i in pick]
    have = {tuple(e) for e in edges.tolist()}
    while len(pairs) < count:                       # candidate pairs without an edge of their own
        a, b = int(rng.choice(rna)), int(rng.choice(prot))
        if (a, b) not in have:
            pairs.append((a, b))
    pairs = np.asarray(pairs[:count], dtype=np.int32)
    ys = (np.arange(count) % 2).astype(np.int32)
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    mask_keys = [tuple(e) for e in edges[:3].tolist()]
    g.set_mask(np.asarray(mask_keys, dtype=np.int32))
    ps = PairSet(g, pairs, ys, h=h)
    n0, e0, mx = ps.batch_caps(count)
    eng = Engine(g.F, B, n0 + 4, e0 + 4, mx, device="cuda", graph=g, tiny=True)
    assert eng.tiny and V == g.num_nodes
    params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(5))
    grads = FlatParams(g.F, "cuda")
    eng.load_pairs(ps, 0, count)
    logp = eng.forward(params, training=False, compute_loss=True).clone()
    eng.backward(params, grads)
    torch.cuda.synchronize()
    N, E = _oracle_check(d, pairs, ys, h, mask_keys, eng, logp, grads, params, count)
    print("h=%d B=%d count=%d: N %s E %s" % (h, B, count, N, E))


def test_tiny_trainer_graph_matches_eager():
    """The captured step on the per-subgraph path (compute || extraction of the next batch) gives bit-identical parameters
    and losses to the eager step, with a partial last batch."""
    from npi_gnn_b200 import synth
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    from npi_gnn_b200.trainer import Trainer
    d = synth.rpi2241_shaped(no_kmer=True)
    pairs, ys = synth.train_pairs(d)
    pairs, ys = pairs[:5 * 64 + 9], ys[:5 * 64 + 9]
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(synth.masked_pairs(d))
    ps = PairSet(g, pairs, ys, h=2)
    res = []
    for use_graph in (False, True):
        p = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(4))
        tr = Trainer(ps, batch_size=64, params=p, seed=11, use_cuda_graph=use_graph)
        assert tr.engine.tiny
        losses = [tr.train_epoch(), tr.train_epoch()]
        losses.append(tr.step(3, sync_loss=True))
        losses.append(tr.step(1, sync_loss=True, next_gb=2))
        losses.append(tr.step(2, sync_loss=True))
        torch.cuda.synchronize()
        res.append((p.flat.clone().cpu(), losses))
    assert res[0][1] == res[1][1]
    assert torch.equal(res[0][0], res[1][0])
    assert all(np.isfinite(x) for x in res[0][1])


def test_tiny_scorer_matches_per_layer_scorer():
    """Scoring sweep (forward only) on the per-subgraph path: probabilities within 1e-5 of the per-layer path's."""
    import os
    from npi_gnn_b200.trainer import Scorer
    d, g, ps, pairs, ys, params = _rpi(600, "ckpt_1223_1_noKmer_50.npz")
    out = []
    for env in ("1", "0"):
        os.environ["NPI_TINY"] = env
        try:
            sc = Scorer(ps, params, batch_size=200)
            out.append(sc.probabilities().clone().cpu())
        finally:
            os.environ.pop("NPI_TINY", None)
    assert out[0].shape == out[1].shape
    assert float((out[0] - out[1]).abs().max()) < 1e-4


@pytest.mark.parametrize("tiny", [True, False])
def test_fused_head_delta_is_bit_identical(tiny):
    """forward(fuse_head_delta=True) followed by backward() gives the same bits as the separate calls: head forward +
    mean-NLL deltas in one launch (both engine paths)."""
    from npi_gnn_b200 import _lib
    from npi_gnn_b200.engine import Engine, FlatParams
    B = 200
    d, g, ps, pairs, ys, params = _rpi(B, "ckpt_1223_1_noKmer_20.npz")
    n0, e0, mx = ps.batch_caps(B)
    eng = Engine(g.F, B, n0, e0, mx, device="cuda", graph=g, tiny=tiny, contexts=False)
    eng.load_pairs(ps, 0, B)
    out = []
    for fuse in (False, True):
        grads = FlatParams(g.F, "cuda")
        before = _lib.CALL_COUNTS.get("npi_head_fwd_delta", 0)
        logp = eng.forward(params, training=True, seed=7, compute_loss=True, fuse_head_delta=fuse).clone()
        eng.backward(params, grads)
        torch.cuda.synchronize()
        used = _lib.CALL_COUNTS.get("npi_head_fwd_delta", 0) - before
        assert used == (1 if fuse else 0), used
        out.append((logp, grads.flat.clone(), eng.d_readout.clone(), float(eng.loss[0])))
    for o in out[1:]:
        assert torch.equal(out[0][0], o[0]) and torch.equal(out[0][2], o[2]) and torch.equal(out[0][1], o[1])
        assert out[0][3] == o[3]


def test_tiny_weight_grads_vs_table_and_tcgen05_routes():
    """The three SAGEConv weight gradients summed over the batch rows directly (one launch) against the per-layer routes
    (conv1: npi_gid_reduce + npi_table_grad through the feature table; conv2 / conv3: npi_gemm_tn_tc) and against fp64
    products of the operands; two calls give the same bits (the in-kernel reduction runs in a fixed order)."""
    import os
    from npi_gnn_b200.engine import Engine, FlatParams
    B = 200
    d, g, ps, pairs, ys, params = _rpi(B, "ckpt_1223_1_noKmer_35.npz")
    n0, e0, mx = ps.batch_caps(B)
    res = []
    for mode in ("direct", "table", "direct"):
        os.environ["NPI_TINY_W1"] = mode
        try:
            eng = Engine(g.F, B, n0, e0, mx, device="cuda", graph=g, tiny=True)
        finally:
            os.environ.pop("NPI_TINY_W1", None)
        assert eng.tiny_w1_direct == (mode == "direct")
        grads = FlatParams(g.F, "cuda")
        eng.load_pairs(ps, 0, B)
        for _ in range(2):                       # the second call reuses the rewound ticket counters
            eng.forward(params, training=True, seed=3, compute_loss=True)
            eng.backward(params, grads)
        torch.cuda.synchronize()
        res.append(({k: grads.views()[k].clone() for k in ("conv1.weight", "conv2.weight", "conv3.weight")}, eng))
    eng = res[0][1]
    N, _ = eng.counters()
    x = torch.zeros(N[0], g.F, dtype=torch.float64, device="cuda")
    x[:, 0] = eng.dist[:N[0]].double()
    x[:, 1:] = g.table[eng.gid[:N[0]].long(), 1:g.F].double()
    refs = {"conv1.weight": x.t() @ eng.big[:N[0]].double(),
            "conv2.weight": eng.xp[0][:N[1]].double().t() @ eng.dxa12[0][:N[1]].double(),
            "conv3.weight": eng.xp[1][:N[2]].double().t() @ eng.dxa12[1][:N[2]].double()}
    for k, ref in refs.items():
        a, b = res[0][0][k].double(), res[1][0][k].double()
        scale = float(ref.abs().max())
        assert float((a - ref).abs().max()) < 2e-6 * scale, (k, float((a - ref).abs().max()) / scale)
        assert float((a - b).abs().max()) < 1e-5 * scale, k
        assert torch.equal(res[0][0][k], res[2][0][k]), k


def _dense_bipartite(n_rna=30, n_prot=30, F=8, seed=9):
    """Complete bipartite graph: every 2-hop enclosing subgraph is the whole graph (60 nodes, 1,800 directed entries -- far more
    than the per-CTA shared-memory entry cache of a 64-node subgraph holds)."""
    rng = np.random.default_rng(seed)
    is_rna = np.asarray([1] * n_rna + [0] * n_prot, dtype=np.uint8)
    edges = np.asarray([(a, n_rna + b) for a in range(n_rna) for b in range(n_prot)], dtype=np.int32)
    rng.shuffle(edges)
    table = rng.standard_normal((n_rna + n_prot, F)).astype(np.float32)
    return dict(edges=edges, is_rna=is_rna, table=table)


@pytest.mark.parametrize("case", ["star_h2", "dense_h2"])
def test_tiny_large_and_dense_subgraphs_vs_oracle(case):
    """The branches small subgraphs do not reach: more than 256 nodes (bitonic top-k instead of the rank count; 300-entry hub
    rows, rows emptied by the pooling) and more entries than the shared-memory entry cache holds (global-memory fallback of the
    column lookup in aggregation, filter_adj and the transposed aggregation) -- against the fp64 oracle forced to the CUDA
    selections."""
    from npi_gnn_b200.engine import Engine, FlatParams
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    torch.set_flush_denormal(True)
    if case == "star_h2":
        from tests.test_gpu_parity import _degenerate_graph
        d, pairs = _degenerate_graph()
        h, mask_keys = 2, [tuple(d["edges"][3].tolist())]
    else:
        d = _dense_bipartite()
        pairs = d["edges"][[0, 17, 101, 500, 899]]
        h, mask_keys = 2, [tuple(e) for e in d["edges"][[5, 17]].tolist()]
    ys = (np.arange(len(pairs)) % 2).astype(np.int32)
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(np.asarray(mask_keys, dtype=np.int32))
    B = len(pairs)
    ps = PairSet(g, pairs, ys, h=h)
    n0, e0, mx = ps.batch_caps(B)
    eng = Engine(g.F, B, n0, e0, mx, device="cuda", graph=g, tiny=True)
    assert eng.tiny
    params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(5))
    grads = FlatParams(g.F, "cuda")
    eng.load_pairs(ps, 0, B)
    logp = eng.forward(params, training=False, compute_loss=True).clone()
    eng.backward(params, grads)
    torch.cuda.synchronize()
    N, E = _oracle_check(d, pairs, ys, h, mask_keys, eng, logp, grads, params, B)
    gp = eng._gp.cpu().numpy()
    sizes = gp[0][1:B + 1] - gp[0][:B]
    if case == "star_h2":
        assert sizes.max() > 256
    else:
        assert E[0] // B > 4 * 64
    print("%s: N %s E %s, largest subgraph %d nodes" % (case, N, E, sizes.max()))
