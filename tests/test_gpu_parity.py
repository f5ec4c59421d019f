"""Parity of the CUDA path (through the libnpi C ABI) against the CPU oracle -- GPU box only.

Integer work (extraction, selection, relabelling) must be bit-exact; floating point is compared
with the tolerances SURVEY.md 7.3 derives from fp32-vs-fp64 runs of the oracle itself.
"""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import khop, khop_cwrap, net as onet, pyg_ops
from tests.common import GOLD, load_ckpt, load_kat, npinter2_oracle_graph, synthetic_bipartite

pytestmark = pytest.mark.gpu

LOGP_ATOL_FORCED = 5e-4      # SURVEY 7.3: log-probs with the oracle forced to the CUDA selections
GRAD_REL_FORCED = 1e-3       # max-norm relative, per tensor


def _product_graph(d):
    from npi_gnn_b200.graph import BipartiteGraph
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(np.concatenate([d["test_pos"], d["test_neg"]]))
    return g


@pytest.fixture(scope="module")
def npi():
    d, og, omask = npinter2_oracle_graph()
    return d, og, omask, _product_graph(d)


def _sample_pairs(d, n, seed, include_hub=True):
    rng = np.random.default_rng(seed)
    allp = np.concatenate([d["train_pos"], d["train_neg"], d["test_pos"], d["test_neg"]])
    ally = np.concatenate([np.ones(len(d["train_pos"])), np.zeros(len(d["train_neg"])),
                           np.ones(len(d["test_pos"])), np.zeros(len(d["test_neg"]))]).astype(np.int32)
    pick = rng.choice(len(allp), n, replace=False)
    return allp[pick], ally[pick]


def _engine_for(ps, B, F, graph, mode="split"):
    from npi_gnn_b200.engine import Engine
    n0, e0, mx = ps.batch_caps(B)
    return Engine(F, B, n0, e0, mx, device="cuda", graph=graph, mode=mode)


# ----------------------------------------------------------------------------- extraction
@pytest.mark.parametrize("h", [1, 2, 3])
def test_khop_bit_exact_vs_oracle(npi, h):
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    n = {1: 600, 2: 300, 3: 64}[h]
    pairs, ys = _sample_pairs(d, n, seed=h)
    ps = PairSet(g, pairs, ys, h=h)
    ref = khop_cwrap.khop_batch(og, omask, pairs, h, fill=False)
    assert np.array_equal(ps.n_h, ref["n_per"])
    assert np.array_equal(ps.e_h, ref["e_per"])
    B = 50 if h < 3 else 16
    eng = _engine_for(ps, B, g.F, g)
    for first in range(0, len(pairs) - B + 1, B):
        eng.load_pairs(ps, first=first, count=B)
        torch.cuda.synchronize()
        c = khop_cwrap.collate_batch(og, omask, pairs[first:first + B], ys[first:first + B], h, d["table"])
        N, E = len(c["gid"]), len(c["col"])
        assert int(eng.sizes[0]) == N and int(eng.sizes[4]) == E
        assert np.array_equal(eng.gid[:N].cpu().numpy(), c["gid"])
        assert np.array_equal(eng.dist[:N].cpu().numpy().astype(np.int32), c["dist"])
        assert np.array_equal(eng.rowptr[0][:N + 1].cpu().numpy(), c["rowptr"])
        assert np.array_equal(eng.col[0][:E].cpu().numpy(), c["col"])
        assert np.array_equal(eng._gp[0].cpu().numpy(), c["graph_ptr"])
        assert np.array_equal(eng.y_b[:B].cpu().numpy(), ys[first:first + B])
        # COO in Appendix-B order and dense x, bit for bit
        from npi_gnn_b200 import ops
        ei = torch.zeros(2, E, dtype=torch.int64, device="cuda")
        ops.subgraph_coo(eng._gp[0], eng.edge_ptr, B, h, eng.gid, eng.dist, g.is_rna, eng.rowptr[0], eng.col[0], ei, False)
        x = torch.zeros(N, g.F, dtype=torch.float32, device="cuda")
        ops.gather_features(g.features_for(eng.gid, eng.dist), None, N, x)
        torch.cuda.synchronize()
        assert np.array_equal(ei.cpu().numpy(), c["edge_index"])
        assert np.array_equal(x.cpu().numpy(), c["x"])


def test_khop_vs_reference_golden_h1(npi):
    """Against outputs of the REFERENCE'S OWN local_subgraph_generation (tests/golden/ref_extract_h1.npz)."""
    from npi_gnn_b200 import ops
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    z = np.load(os.path.join(GOLD, "ref_extract_h1.npz"))
    pairs = z["pairs"]
    ps = PairSet(g, pairs, np.zeros(len(pairs), dtype=np.int32), h=1)
    assert np.array_equal(ps.n_h, z["n"])
    B = len(pairs)
    eng = _engine_for(ps, B, g.F, g)
    eng.load_pairs(ps, 0, B)
    N, E = int(ps.n_h.sum()), int(ps.e_h.sum())
    ei = torch.zeros(2, E, dtype=torch.int64, device="cuda")
    ops.subgraph_coo(eng._gp[0], eng.edge_ptr, B, 1, eng.gid, eng.dist, g.is_rna, eng.rowptr[0], eng.col[0], ei, True)
    x = torch.zeros(N, g.F, dtype=torch.float32, device="cuda")
    ops.gather_features(g.features_for(eng.gid, eng.dist), None, N, x)
    torch.cuda.synchronize()
    x, ei = x.cpu().numpy(), ei.cpu().numpy()
    gp, ep = eng._gp[0].cpu().numpy(), eng.edge_ptr.cpu().numpy()
    for i in range(B):
        xi = np.ascontiguousarray(x[gp[i]:gp[i + 1]])
        assert hashlib.sha256(xi.tobytes()).hexdigest() == str(z["x_sha256"][i])
        e = sorted(map(tuple, ei[:, ep[i]:ep[i + 1]].T.tolist()))
        exp = [tuple(t) for t in z["edges_sorted"][z["edge_ptr"][i]:z["edge_ptr"][i + 1]].tolist()]
        assert e == exp


def test_khop_synthetic_edge_cases():
    """Tiny graphs: isolated targets, candidate (non-edge) pairs, everything masked."""
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    s = synthetic_bipartite(5, 12, 7, 30, 0, F=7)
    og = khop.build_csr([tuple(e) for e in s["edges"].tolist()], s["is_rna"])
    g = BipartiteGraph(s["edges"], s["is_rna"], s["table"])
    rna = np.nonzero(s["is_rna"])[0]; prot = np.nonzero(s["is_rna"] == 0)[0]
    pairs = np.array([(a, b) for a in rna for b in prot], dtype=np.int32)       # all candidates
    for masked in (s["edges"][:0], s["edges"][::2], s["edges"]):
        g.set_mask(masked)
        omask = khop.mask_from_keys(og, [tuple(e) for e in masked.tolist()])
        for h in (1, 2, 4):
            ps = PairSet(g, pairs, np.zeros(len(pairs), dtype=np.int32), h=h)
            eng = _engine_for(ps, len(pairs), g.F, g)
            eng.load_pairs(ps, 0, len(pairs))
            torch.cuda.synchronize()
            c = khop_cwrap.collate_batch(og, omask, pairs, np.zeros(len(pairs)), h, s["table"])
            N, E = len(c["gid"]), len(c["col"])
            assert np.array_equal(eng.gid[:N].cpu().numpy(), c["gid"])
            assert np.array_equal(eng.dist[:N].cpu().numpy().astype(np.int32), c["dist"])
            assert np.array_equal(eng.rowptr[0][:N + 1].cpu().numpy(), c["rowptr"])
            assert np.array_equal(eng.col[0][:E].cpu().numpy(), c["col"])


def test_khop_large_graph_global_workspace():
    """Config-4 shape in small: a disjoint union of NPInter2-shaped blocks whose V (20 k) no longer
    fits the shared-memory map, so the extractor runs with its working set in the global
    workspace; h = 2 and 3, bit-exact against the C oracle."""
    from npi_gnn_b200 import ops, synth
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    d = synth.scaled_blocks(4, seed=5)
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    cannot = synth.masked_pairs(d)
    omask = khop.mask_from_keys(og, [tuple(e) for e in cannot.tolist()])
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"])
    g.set_mask(cannot)
    assert ops.khop_workspace_bytes(g.num_nodes, 1) > 4 * g.num_nodes      # i.e. not the shared-memory path
    pairs, ys = synth.train_pairs(d, seed=2)
    for h, n in ((2, 96), (3, 24)):
        ps = PairSet(g, pairs[:n], ys[:n], h=h)
        ref = khop_cwrap.khop_batch(og, omask, pairs[:n], h, fill=False)
        assert np.array_equal(ps.n_h, ref["n_per"]) and np.array_equal(ps.e_h, ref["e_per"])
        eng = _engine_for(ps, n, g.F, g)
        eng.load_pairs(ps, 0, n)
        torch.cuda.synchronize()
        c = khop_cwrap.collate_batch(og, omask, pairs[:n], ys[:n], h, d["table"])
        N, E = len(c["gid"]), len(c["col"])
        assert np.array_equal(eng.gid[:N].cpu().numpy(), c["gid"])
        assert np.array_equal(eng.dist[:N].cpu().numpy().astype(np.int32), c["dist"])
        assert np.array_equal(eng.rowptr[0][:N + 1].cpu().numpy(), c["rowptr"])
        assert np.array_equal(eng.col[0][:E].cpu().numpy(), c["col"])


# ----------------------------------------------------------------------------- single operators
def _real_batch(npi, B=40, h=1, seed=3):
    d, og, omask, g = npi
    pairs, ys = _sample_pairs(d, B, seed)
    c = khop_cwrap.collate_batch(og, omask, pairs, ys, h, d["table"])
    return pairs, ys, c


@pytest.mark.parametrize("F,aligned", [(178, False), (128, True), (65, False), (12, True)])
def test_sage_fwd_dense_vs_oracle(npi, F, aligned):
    from npi_gnn_b200 import ops, _lib as L
    _, _, c = _real_batch(npi, B=30, h=2, seed=F)
    N = len(c["gid"])
    rng = np.random.default_rng(F)
    ld = (F + 3) // 4 * 4 if aligned else F
    xfull = torch.from_numpy(rng.standard_normal((N, ld)).astype(np.float32))
    x = xfull[:, :F]
    W = torch.from_numpy((rng.standard_normal((F, 128)) / np.sqrt(F)).astype(np.float32))
    b = torch.from_numpy(rng.standard_normal(128).astype(np.float32) * 0.1)
    pw = torch.from_numpy(rng.standard_normal((1, 128)).astype(np.float32) * 0.1)
    ei = torch.from_numpy(c["edge_index"])
    ref = torch.relu(pyg_ops.sage_conv(x.double(), ei, W.double(), b.double()))
    zref = (ref * pw.double()).sum(-1) / pw.double().norm()
    xd = xfull.cuda()[:, :F]
    h = torch.empty(N, 128, device="cuda"); z = torch.empty(N, device="cuda"); s = torch.empty(N, device="cuda")
    ops.sage_fwd(L.features_dense(xd), torch.from_numpy(c["rowptr"]).cuda(), torch.from_numpy(c["col"]).cuda(), None, N,
                 W.cuda(), b.cuda(), True, pw.cuda(), h, z, s)
    torch.cuda.synchronize()
    assert torch.allclose(h.cpu().double(), ref, atol=2e-5, rtol=1e-5)
    assert torch.allclose(z.cpu().double(), zref, atol=2e-5, rtol=1e-5)
    assert torch.allclose(s.cpu().double(), torch.tanh(zref), atol=2e-6)


@pytest.mark.parametrize("M,K,aligned", [(1, 128, True), (127, 128, True), (128, 178, True), (1000, 178, False), (5085, 65, False), (3333, 12, True)])
def test_gemm_nn_tn_vs_torch(M, K, aligned):
    from npi_gnn_b200 import ops
    rng = np.random.default_rng(M + K)
    ld = (K + 3) // 4 * 4 if aligned else K
    Afull = torch.from_numpy(rng.standard_normal((M, ld)).astype(np.float32)).cuda()
    A = Afull[:, :K]
    B = torch.from_numpy(rng.standard_normal((K, 128)).astype(np.float32)).cuda()
    D = torch.from_numpy(rng.standard_normal((M, 128)).astype(np.float32)).cuda()
    C = torch.full((M, 128), float("nan"), device="cuda")
    ops.gemm_nn(A, None, M, K, B, False, C)
    ref = (A.double() @ B.double())
    assert torch.allclose(C.double(), ref, atol=1e-4, rtol=1e-5)
    if K == 128:                                     # transposed-B form used by the input gradient
        C2 = torch.empty(M, 128, device="cuda")
        ops.gemm_nn(A, None, M, K, B, True, C2)
        assert torch.allclose(C2.double(), A.double() @ B.double().t(), atol=1e-4, rtol=1e-5)
    ws = torch.empty(ops.gemm_tn_workspace_bytes(K), dtype=torch.uint8, device="cuda")
    out = torch.full((K, 128), float("nan"), device="cuda")
    row0 = torch.from_numpy(rng.standard_normal((5, 128)).astype(np.float32)).cuda()
    ops.gemm_tn(A, D, None, M, K, row0, out, ws)
    ref_tn = A.double().t() @ D.double()
    ref_tn[0] += row0.double().sum(0)
    assert torch.allclose(out.double(), ref_tn, atol=2e-4 * max(1, M ** 0.5 / 8), rtol=1e-5)
    out2 = torch.empty_like(out)
    ops.gemm_tn(A, D, None, M, K, row0, out2, ws)
    assert torch.equal(out, out2)


def test_topk_select_bit_exact_given_scores():
    """Ties, duplicates, signed zeros, graphs of 1..5000 nodes: perm / new_id identical to the
    oracle's stable descending sort (Appendix A.3)."""
    from npi_gnn_b200 import ops
    rng = np.random.default_rng(7)
    sizes = [1, 2, 3, 5, 31, 32, 33, 100, 256, 257, 1024, 1025, 2947, 5000, 8191, 8192, 8193, 9000, 2, 2, 7]
    B = len(sizes)
    gin = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    k = [int(np.ceil(np.float32(0.5) * np.float32(n))) for n in sizes]
    gout = np.concatenate([[0], np.cumsum(k)]).astype(np.int32)
    N = int(gin[-1])
    s = np.tanh(rng.standard_normal(N)).astype(np.float32)
    s[rng.choice(N, N // 3, replace=False)] = np.float32(0.25)         # heavy ties
    s[rng.choice(N, N // 10, replace=False)] = np.float32(0.0)
    s[rng.choice(N, N // 20, replace=False)] = np.float32(-0.0)
    s = np.round(s * 8) / 8 if False else s
    batch = torch.from_numpy(np.repeat(np.arange(B), sizes))
    ref = pyg_ops.topk_perm(torch.from_numpy(s), 0.5, batch, B).numpy()
    perm = torch.empty(int(gout[-1]), dtype=torch.int32, device="cuda")
    new_id = torch.empty(N, dtype=torch.int32, device="cuda")
    bo = torch.empty(int(gout[-1]), dtype=torch.int32, device="cuda")
    ws = torch.empty(max(16, ops.topk_select_workspace_bytes(B, max(sizes))), dtype=torch.uint8, device="cuda")
    ops.topk_select(torch.from_numpy(s).cuda(), torch.from_numpy(gin).cuda(), torch.from_numpy(gout).cuda(), B, max(sizes),
                    perm, new_id, bo, ws)
    torch.cuda.synchronize()
    assert np.array_equal(perm.cpu().numpy(), ref)
    exp_new = np.full(N, -1, dtype=np.int32); exp_new[ref] = np.arange(len(ref))
    assert np.array_equal(new_id.cpu().numpy(), exp_new)
    assert np.array_equal(bo.cpu().numpy(), batch.numpy()[ref])


def test_filter_adj_and_readout_vs_oracle(npi):
    from npi_gnn_b200 import ops
    _, _, c = _real_batch(npi, B=25, h=2, seed=11)
    N, E, B = len(c["gid"]), len(c["col"]), len(c["y"])
    rng = np.random.default_rng(0)
    hmat = torch.from_numpy(np.maximum(rng.standard_normal((N, 128)), 0).astype(np.float32))
    s = torch.from_numpy(np.tanh(rng.standard_normal(N)).astype(np.float32))
    batch = torch.from_numpy(c["batch"])
    perm_ref = pyg_ops.topk_perm(s, 0.5, batch, B)
    n = np.diff(c["graph_ptr"]); k = (n + 1) // 2
    gout = np.concatenate([[0], np.cumsum(k)]).astype(np.int32)
    dev = "cuda"
    perm = torch.empty(len(perm_ref), dtype=torch.int32, device=dev); new_id = torch.empty(N, dtype=torch.int32, device=dev)
    bo = torch.empty(len(perm_ref), dtype=torch.int32, device=dev)
    ws = torch.empty(max(16, ops.topk_select_workspace_bytes(B, int(n.max()))), dtype=torch.uint8, device=dev)
    gin_d, gout_d = torch.from_numpy(c["graph_ptr"]).to(dev), torch.from_numpy(gout).to(dev)
    ops.topk_select(s.to(dev), gin_d, gout_d, B, int(n.max()), perm, new_id, bo, ws)
    Np = len(perm_ref)
    xp = torch.empty(Np, 128, device=dev); ro = torch.zeros(B, 256, device=dev); am = torch.empty(B, 128, dtype=torch.int32, device=dev)
    ops.pool_gate_readout(hmat.to(dev), s.to(dev), perm, gout_d, B, xp, ro, False, am)
    rp2 = torch.empty(Np + 1, dtype=torch.int32, device=dev); col2 = torch.empty(E, dtype=torch.int32, device=dev)
    wsf = torch.empty(ops.filter_adj_workspace_bytes(Np) + 16, dtype=torch.uint8, device=dev)
    ops.filter_adj(torch.from_numpy(c["rowptr"]).to(dev), torch.from_numpy(c["col"]).to(dev), perm, new_id, None, Np, rp2, col2, wsf)
    torch.cuda.synchronize()
    assert np.array_equal(perm.cpu().numpy(), perm_ref.numpy())
    xo, eo, _, bo_ref, _, _ = pyg_ops.topk_pooling(hmat, torch.from_numpy(c["edge_index"]), batch,
                                                    torch.ones(1, 128), 0.5, forced_perm=perm_ref)
    xo = hmat[perm_ref] * s[perm_ref].view(-1, 1)
    assert torch.equal(xp.cpu(), xo)                                   # one multiply per element: exact
    ro_ref = torch.cat([pyg_ops.global_max_pool(xo, bo_ref, B), pyg_ops.global_mean_pool(xo.double(), bo_ref, B).float()], 1)
    assert torch.equal(ro.cpu()[:, :128], ro_ref[:, :128])
    assert torch.allclose(ro.cpu()[:, 128:], ro_ref[:, 128:], atol=1e-6, rtol=1e-5)
    # filtered CSR == filter_adj of the oracle (as per-destination ordered source lists)
    Ep = int(rp2[Np])
    rp2, col2 = rp2.cpu().numpy(), col2.cpu().numpy()[:Ep]
    assert Ep == eo.shape[1]
    got = {(int(col2[kk]), r) for r in range(Np) for kk in range(rp2[r], rp2[r + 1])}
    assert got == set(map(tuple, eo.t().tolist()))
    # order inside a row preserved: sources of row r appear in the order of the old row
    new_id_h = new_id.cpu().numpy()
    for r in range(0, Np, max(1, Np // 200)):
        o = int(perm_ref[r])
        exp_row = [int(new_id_h[j]) for j in c["col"][c["rowptr"][o]:c["rowptr"][o + 1]] if new_id_h[j] >= 0]
        assert list(col2[rp2[r]:rp2[r + 1]]) == exp_row


# ----------------------------------------------------------------------------- whole network
def _oracle_model(F, sd):
    m = onet.Net_1(F)
    m.load_state_dict(sd)
    return m


def _params_from_sd(F, sd):
    from npi_gnn_b200.engine import FlatParams
    return FlatParams(F, "cuda").load_state_dict(sd)


@pytest.mark.parametrize("mode", ["split", "fused_v1"])
@pytest.mark.parametrize("h,ckpt", [(1, "ckpt_1223_1_15.npz"), (2, "ckpt_1223_1_5.npz")])
def test_forward_backward_vs_oracle(npi, h, ckpt, mode):
    """Log-probs, loss and all 15 gradients on real batches; the oracle is forced to the CUDA
    path's discrete decisions -- top-k selections, dropout mask, ReLU masks of the three conv layers
    and the head, the rows global_max_pool routes to -- so that fp rounding cannot flip one
    (free-running disagreement is measured in test_selection_agreement; that the ReLU / argmax
    decisions differ from the oracle's own only at rounding level is asserted in
    tests/test_gpu_synth_parity.py)."""
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import PairSet
    torch.set_flush_denormal(True)
    d, og, omask, g = npi
    sd = load_ckpt(ckpt)
    B = 48
    pairs, ys = _sample_pairs(d, B, seed=21 + h)
    ps = PairSet(g, pairs, ys, h=h)
    eng = _engine_for(ps, B, g.F, g, mode)
    params = _params_from_sd(g.F, sd)
    grads = FlatParams(g.F, "cuda")
    eng.load_pairs(ps, 0, B)
    logp = eng.forward(params, training=True, seed=1234, compute_loss=True).clone()
    eng.backward(params, grads)
    torch.cuda.synchronize()
    N, E = eng.counters()
    perms = [eng.perm[l][:N[l + 1]].cpu().long() for l in range(3)]
    mask = eng.drop_mask[:B].cpu().float()
    assert 0.35 < mask.mean() < 0.65
    relu = [(eng.layer_rows(l, N[l])[0] > 0).cpu() for l in range(3)]
    amax = [eng.argmax[l][:B].cpu().long() for l in range(3)]
    head = ((eng.a1[:B] > 0).cpu(), (eng.a2[:B] > 0).cpu())
    c = khop_cwrap.collate_batch(og, omask, pairs, ys, h, d["table"])
    for dtype, tol_lp, tol_g in ((torch.float32, LOGP_ATOL_FORCED, GRAD_REL_FORCED), (torch.float64, LOGP_ATOL_FORCED, GRAD_REL_FORCED)):
        m = _oracle_model(g.F, sd).to(dtype)
        m.train()
        bn = onet.batch_namespace(c)
        bn.x = bn.x.to(dtype)
        out = m(bn, dropout_mask=mask.to(dtype), forced_perms=perms, forced_relu=relu, forced_argmax=amax, forced_head=head)
        loss = torch.nn.functional.nll_loss(out, bn.y)
        loss.backward()
        assert max(m.trace.max_gap) < 1e-5
        assert torch.allclose(logp.cpu().double(), out.detach().double(), atol=tol_lp), (logp.cpu().double() - out.detach().double()).abs().max()
        assert abs(float(eng.loss[0]) - float(loss)) < 1e-4
        gv = grads.views()
        for name, p in m.named_parameters():
            ref = p.grad.double()
            got = gv[name].cpu().double()
            err = (got - ref).abs().max() / max(ref.abs().max(), 1e-12)
            assert err < tol_g, (name, float(err))
    # intermediate integer structures of every layer agree with the oracle trace
    tr = m.trace
    for l in range(3):
        assert np.array_equal(eng.batch[l][:N[l + 1]].cpu().numpy(), tr.batch[l].numpy())
    for l in range(2):
        rp = eng.rowptr[l + 1][:N[l + 1] + 1].cpu().numpy(); cl = eng.col[l + 1][:E[l + 1]].cpu().numpy()
        got = {(int(cl[kk]), r) for r in range(N[l + 1]) for kk in range(rp[r], rp[r + 1])}
        assert got == set(map(tuple, tr.edge_index[l].t().tolist()))


def _degenerate_graph(seed=3, F=8):
    """Isolated pairs (2-node subgraphs, every row one entry), a star (one protein with 300 RNAs: a hub
    row cut into ten 32-entry segments, 300 one-entry rows), a second protein shared by 20 of the
    star's RNAs (a row of 17..128 entries), candidate pairs without an edge (only the target edge)."""
    rng = np.random.default_rng(seed)
    edges, is_rna = [], []

    def node(isr):
        is_rna.append(isr)
        return len(is_rna) - 1
    iso = []
    for _ in range(6):
        a, b = node(1), node(0)
        edges.append((a, b)); iso.append((a, b))
    hub = node(0)
    leaves = [node(1) for _ in range(300)]
    edges += [(r, hub) for r in leaves]
    p2 = node(0)
    edges += [(r, p2) for r in leaves[:20]]
    lone_r, lone_p = node(1), node(0)                       # never on an edge
    table = rng.standard_normal((len(is_rna), F)).astype(np.float32)
    d = dict(edges=np.asarray(edges, dtype=np.int32), is_rna=np.asarray(is_rna, dtype=np.uint8), table=table)
    pairs = iso + [(leaves[0], hub), (leaves[5], p2), (leaves[299], hub), (lone_r, lone_p), (leaves[1], lone_p), (iso[0][0], hub)]
    return d, np.asarray(pairs, dtype=np.int32)


@pytest.mark.parametrize("h", [1, 2])
@pytest.mark.parametrize("single", [False, True])
def test_degenerate_batches_vs_oracle(h, single):
    """One-entry rows, hub segments, rows emptied by the pooling and a one-graph batch through extraction, forward,
    loss and backward against the oracle (forced to the CUDA selections, dropout off)."""
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    torch.set_flush_denormal(True)
    d, pairs = _degenerate_graph()
    if single:
        pairs = pairs[6:7]                                  # the star seen from one leaf: 302 nodes at h = 2
    ys = (np.arange(len(pairs)) % 2).astype(np.int32)
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    omask = khop.mask_from_keys(og, [tuple(d["edges"][3].tolist())])
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(d["edges"][3:4])
    B = len(pairs)
    ps = PairSet(g, pairs, ys, h=h)
    eng = _engine_for(ps, B, g.F, g)
    params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(5))
    grads = FlatParams(g.F, "cuda")
    eng.load_pairs(ps, 0, B)
    logp = eng.forward(params, training=False, compute_loss=True).clone()
    eng.backward(params, grads)
    torch.cuda.synchronize()
    N, E = eng.counters()
    c = khop_cwrap.collate_batch(og, omask, pairs, ys, h, d["table"])
    assert N[0] == len(c["gid"]) and E[0] == len(c["col"])
    assert np.array_equal(eng.gid[:N[0]].cpu().numpy(), c["gid"])
    assert np.array_equal(eng.rowptr[0][:N[0] + 1].cpu().numpy(), c["rowptr"])
    assert np.array_equal(eng.col[0][:E[0]].cpu().numpy(), c["col"])
    deg = np.diff(c["rowptr"])
    if not single:
        assert deg.min() == 1 and deg.max() >= 300 and ((deg > 16) & (deg <= 128)).any()
    perms = [eng.perm[l][:N[l + 1]].cpu().long() for l in range(3)]
    m = onet.Net_1(g.F).double()
    m.load_state_dict({k: v.double() for k, v in params.state_dict().items()})
    m.eval()
    bn = onet.batch_namespace(c)
    bn.x = bn.x.double()
    out = m(bn, forced_perms=perms)
    loss = torch.nn.functional.nll_loss(out, bn.y)
    loss.backward()
    assert torch.allclose(logp.cpu().double(), out.detach(), atol=LOGP_ATOL_FORCED), (logp.cpu().double() - out.detach()).abs().max()
    assert abs(float(eng.loss[0]) - float(loss)) < 1e-4
    gv = grads.views()
    for name, p in m.named_parameters():
        ref = p.grad.double()
        got = gv[name].cpu().double()
        err = (got - ref).abs().max() / max(float(ref.abs().max()), 1e-6)
        assert err < GRAD_REL_FORCED, (name, float(err))
    for l in range(3):
        assert np.array_equal(eng.batch[l][:N[l + 1]].cpu().numpy(), m.trace.batch[l].numpy())


def test_selection_agreement_free_running(npi):
    """Free-running CUDA vs free-running fp32 oracle: selections may only differ where the score
    gap at the top-k boundary is within rounding (SURVEY 7.3); count and bound them."""
    from npi_gnn_b200.graph import PairSet
    torch.set_flush_denormal(True)
    d, og, omask, g = npi
    sd = load_ckpt("ckpt_1223_1_15.npz")
    B = 200
    pairs, ys = _sample_pairs(d, B, seed=99)
    ps = PairSet(g, pairs, ys, h=1)
    eng = _engine_for(ps, B, g.F, g)
    params = _params_from_sd(g.F, sd)
    eng.load_pairs(ps, 0, B)
    logp = eng.forward(params, training=False).clone()
    torch.cuda.synchronize()
    N, _ = eng.counters()
    m = _oracle_model(g.F, sd); m.eval()
    c = khop_cwrap.collate_batch(og, omask, pairs, ys, 1, d["table"])
    with torch.no_grad():
        out = m(onet.batch_namespace(c))
    differing = 0
    for l in range(3):
        a = eng.perm[l][:N[l + 1]].cpu().numpy(); b = m.trace.perm[l].numpy()
        if not np.array_equal(a, b):
            differing += 1
            break
    if differing == 0:
        assert torch.allclose(logp.cpu(), out, atol=LOGP_ATOL_FORCED)
    else:
        assert torch.allclose(logp.cpu(), out, atol=2e-3)       # free-running bound of SURVEY 7.3
    assert (logp.cpu().argmax(1) == out.argmax(1)).float().mean() > 0.99


@pytest.mark.parametrize("mode", ["split", "fused_v1"])
def test_rerun_bit_identical(npi, mode):
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    pairs, ys = _sample_pairs(d, 64, seed=5)
    ps = PairSet(g, pairs, ys, h=2)
    eng = _engine_for(ps, 64, g.F, g, mode)
    params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(0))
    outs = []
    for _ in range(2):
        grads = FlatParams(g.F, "cuda")
        eng.load_pairs(ps, 0, 64)
        lp = eng.forward(params, training=True, seed=7, compute_loss=True).clone()
        eng.backward(params, grads)
        torch.cuda.synchronize()
        outs.append((lp.cpu(), grads.flat.cpu().clone(), eng.loss.cpu().clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])


@pytest.mark.parametrize("h,B", [(1, 96), (2, 64), (3, 16)])
def test_pipelined_aggregation_bit_identical_to_plain(npi, h, B, monkeypatch):
    """The software-pipelined aggregation kernels over the packed entry streams (what the engine
    launches) sum in the order of the plain dependent-chain kernels: log-probabilities, every
    intermediate activation, the loss and all gradients must be BIT-identical between the two
    (short rows and hub segments both occur at h >= 2 on NPInter2; the whole-warp tier is empty at
    the shipped 16-entry hub threshold).  Neither kernel is checked against a reference here:
    tests/test_gpu_aggregation.py does that."""
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    pairs, ys = _sample_pairs(d, B, seed=31 + h)
    ps = PairSet(g, pairs, ys, h=h)
    params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(2))
    outs = []
    monkeypatch.setenv("NPI_CTX_DEDUP", "0")       # this test is about the per-row kernels (contexts: tests/test_gpu_ctx.py)
    for pipe in ("1", "0"):
        monkeypatch.setenv("NPI_AGG_PIPE", pipe)
        eng = _engine_for(ps, B, g.F, g)
        assert eng.pipelined == (pipe == "1")
        grads = FlatParams(g.F, "cuda")
        eng.load_pairs(ps, 0, B)
        lp = eng.forward(params, training=True, seed=9, compute_loss=True).clone()
        eng.backward(params, grads)
        torch.cuda.synchronize()
        Ns, Es = eng.counters()
        outs.append(dict(lp=lp.cpu(), grads=grads.flat.cpu().clone(), loss=eng.loss.cpu().clone(),
                         h=[eng.layer_rows(l, Ns[l])[0].cpu().clone() for l in range(3)],
                         s=[eng.layer_rows(l, Ns[l])[2].cpu().clone() for l in range(3)],
                         dxa=[eng.big[:Ns[0]].cpu().clone()] + [eng.dxa12[l][:Ns[l + 1]].cpu().clone() for l in range(2)],
                         N=Ns, E=Es))
    a, b = outs
    assert a["N"] == b["N"] and a["E"] == b["E"]
    if h >= 2:
        deg = (eng.rowptr[0][1:a["N"][0] + 1] - eng.rowptr[0][:a["N"][0]])
        assert int(deg.max()) > 128 and int(((deg > 16) & (deg <= 128)).sum()) > 0      # hub rows of 1-4 and of > 4 segments
    for l in range(3):
        assert torch.equal(a["h"][l], b["h"][l]), "forward aggregation layer %d" % (l + 1)
        assert torch.equal(a["s"][l], b["s"][l])
        assert torch.equal(a["dxa"][l], b["dxa"][l]), "transposed aggregation layer %d" % (l + 1)
    assert torch.equal(a["lp"], b["lp"]) and torch.equal(a["loss"], b["loss"]) and torch.equal(a["grads"], b["grads"])


def test_entry_pack_streams(npi, monkeypatch):
    """npi_entry_pack_virt / npi_entry_pack_sel against their definitions (integer: bit-exact)."""
    from npi_gnn_b200 import ops
    monkeypatch.setenv("NPI_CTX_DEDUP", "0")       # per-row lists of the input layer (the context path does not build them)
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    pairs, ys = _sample_pairs(d, 32, seed=77)
    ps = PairSet(g, pairs, ys, h=2)
    eng = _engine_for(ps, 32, g.F, g)
    params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(2))
    eng.load_pairs(ps, 0, 32)
    eng.forward(params, training=False)
    torch.cuda.synchronize()
    Ns, Es = eng.counters()
    col = eng.col[0][:Es[0]].long()
    want = eng.gid[:Ns[0]][col] | (eng.dist[:Ns[0]].int()[col] << 29)
    assert torch.equal(eng.cur.ent0[:Es[0]], want.int())
    for l in range(3):
        rp = eng.rowptr[l][:Ns[l] + 1]
        c = eng.col[l][:Es[l]].long()
        nid = eng.new_id[l][:Ns[l]]
        deg = (rp[1:] - rp[:-1])
        inv = torch.where(nid[c] >= 0, 1.0 / (deg[c] + 1).float(), torch.zeros((), device="cuda"))
        got = eng.sel[l][:Es[l]]
        assert torch.equal(got[:, 0], nid[c])
        assert torch.equal(got[:, 1].contiguous().view(torch.float32), inv)
    # rows binned by length class (npi_hub_rows_build): a permutation of the non-hub rows, classes ascending
    HUB = 16                                     # NPI_AG_HUB (agg.cu): longer rows are cut into segments
    bounds = torch.tensor([1, 3, 5, 7, 11, 16, HUB], device="cuda")
    for l in range(3):
        rp = eng.rowptr[l][:Ns[l] + 1]
        deg = (rp[1:] - rp[:-1])
        keep = torch.nonzero(deg <= HUB).flatten()
        R = eng.rows[l][:keep.numel()]
        assert torch.equal(torch.sort(R[:, 0]).values, keep.int())
        rows = R[:, 0].long()
        assert torch.equal(R[:, 1], rp[rows]) and torch.equal(R[:, 2], rp[rows + 1])
        cls = torch.bucketize(deg[rows], bounds)
        assert bool((cls[1:] >= cls[:-1]).all())
        hdr = eng.hubq[l].view(torch.int32)[:32]
        assert [int(v) for v in hdr[4:12]] == [int((torch.bucketize(deg, bounds) == c).sum()) for c in range(8)]
        if l == 0:
            assert torch.equal(R[:, 3], eng.gid[:Ns[0]][rows] | (eng.dist[:Ns[0]].int()[rows] << 29))
        else:
            assert torch.equal(R[:, 3], R[:, 0])
    # identity selection (new_id NULL) on the input CSR
    out = torch.zeros(Es[0], 2, dtype=torch.int32, device="cuda")
    ops.entry_pack_sel(eng.rowptr[0], eng.col[0], None, eng.sizes[0:1], eng.n_cap[0], out)
    assert torch.equal(out[:, 0], eng.col[0][:Es[0]])


def test_trainer_graph_prefetch_matches_eager(npi):
    """The captured step (compute on one batch slot || extraction of the next batch into the other
    slot on a side stream) must give bit-identical parameters and losses to the sequential eager
    step, over two epochs with a partial last batch and an out-of-order access."""
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import PairSet
    from npi_gnn_b200.trainer import Trainer
    d, og, omask, g = npi
    pairs, ys = _sample_pairs(d, 5 * 48 + 17, seed=21)
    ps = PairSet(g, pairs, ys, h=2)
    res = []
    for use_graph in (False, True):
        p = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(4))
        tr = Trainer(ps, batch_size=48, params=p, seed=11, use_cuda_graph=use_graph)
        losses = [tr.train_epoch(), tr.train_epoch()]
        losses.append(tr.step(3, sync_loss=True))              # not prefetched
        losses.append(tr.step(1, sync_loss=True, next_gb=2))
        losses.append(tr.step(2, sync_loss=True))              # prefetched by the previous call
        torch.cuda.synchronize()
        res.append((p.flat.clone().cpu(), losses))
    assert res[0][1] == res[1][1]
    assert torch.equal(res[0][0], res[1][0])


def test_adam_l2_vs_torch():
    from npi_gnn_b200 import ops
    torch.manual_seed(0)
    n = 97602
    p0 = torch.randn(n); steps = 5
    p_ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([p_ref], lr=1e-3, weight_decay=1e-3)
    p = p0.clone().cuda(); m = torch.zeros(n, device="cuda"); v = torch.zeros(n, device="cuda")
    lr = torch.tensor([1e-3], device="cuda"); step = torch.zeros(1, dtype=torch.int32, device="cuda")
    for t in range(steps):
        g = torch.randn(n) * (0.1 if t % 2 else 1e-4)
        p_ref.grad = g.clone()
        opt.step()
        ops.adam_l2_step(p, g.cuda(), m, v, lr, step, 0.9, 0.999, 1e-8, 1e-3, 1.0)
    torch.cuda.synchronize()
    assert int(step[0]) == steps
    assert torch.allclose(p.cpu(), p_ref.detach(), atol=2e-6, rtol=1e-5)


# ----------------------------------------------------------------------------- known answers on the GPU
@pytest.mark.parametrize("proj,ep", [("1223_1", 5), ("1223_1", 15), ("1223_1", 30), ("1223_1", 50), ("1223_1_noKmer", 20), ("1223_1_noKmer", 35), ("1223_1_noKmer", 50)])
def test_confusion_kat_on_gpu(proj, ep):
    """The shipped checkpoints reproduce the reference's logged confusion matrices through the
    CUDA path (GPU extraction -> fused forward -> npi_confusion_counts), SURVEY 0.5."""
    from npi_gnn_b200 import ops
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    d, og, omask = npinter2_oracle_graph()
    no_kmer = proj.endswith("noKmer")
    table = d["table"][:, :64] if no_kmer else d["table"]
    g = BipartiteGraph(d["edges"], d["is_rna"], table)
    g.set_mask(np.concatenate([d["test_pos"], d["test_neg"]]))
    pairs = np.concatenate([d["test_pos"], d["test_neg"]])
    ys = np.concatenate([np.ones(len(d["test_pos"])), np.zeros(len(d["test_neg"]))]).astype(np.int32)
    perm = np.random.default_rng(0).permutation(len(pairs))
    pairs, ys = pairs[perm], ys[perm]
    ps = PairSet(g, pairs, ys, h=1)
    B = 200
    eng = _engine_for(ps, B, g.F, g)
    params = _params_from_sd(g.F, load_ckpt("ckpt_%s_%d.npz" % (proj, ep)))
    counts = torch.zeros(4, dtype=torch.int64, device="cuda")
    for first in range(0, len(pairs), B):
        cnt = min(B, len(pairs) - first)
        eng.load_pairs(ps, first, cnt)
        logp = eng.forward(params, training=False)
        ops.confusion_counts(logp, eng.y_b, cnt, -1.0, counts)
    torch.cuda.synchronize()
    exp = load_kat()["confusion"][proj][str(ep)]
    TP, FN, TN, FP = [int(v) for v in counts.cpu()]
    got = dict(TP=TP, FN=FN, TN=TN, FP=FP)
    _record_kat("%s/%d" % (proj, ep), got, exp)
    # exact: the confusion matrix the authors' PyG-1.4.2 stack logged (README/DESIGN say "reproduced exactly")
    assert got == {k: exp[k] for k in ("TP", "FN", "TN", "FP")}, (got, exp)


def _record_kat(name, got, exp):
    """got/expected pairs of every GPU KAT are appended to gpurun_out/kat_gpu.jsonl (copied under profiles/)."""
    import json
    try:
        os.makedirs(os.path.join(os.path.dirname(GOLD), "..", "gpurun_out"), exist_ok=True)
        with open(os.path.join(os.path.dirname(GOLD), "..", "gpurun_out", "kat_gpu.jsonl"), "a") as f:
            f.write(json.dumps({"kat": name, "got": got, "expected": {k: exp[k] for k in ("TP", "FN", "TN", "FP")}}) + "\n")
    except OSError:
        pass


@pytest.mark.parametrize("thr", ["0.5", "0.95"])
def test_case_study_kat_on_gpu(thr):
    """src/case_study_negativeSample.py:235-253,339-355 through Scorer: the test negatives scored
    positive by checkpoint 15 are exactly the reference's shipped lists (SURVEY 0.5)."""
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    from npi_gnn_b200.trainer import Scorer
    d, og, omask = npinter2_oracle_graph()
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"])
    g.set_mask(np.concatenate([d["test_pos"], d["test_neg"]]))
    exp = load_kat()["case_study"][thr]
    pairs = d["test_neg"]
    ps = PairSet(g, pairs, np.zeros(len(pairs), dtype=np.int32), h=1)
    params = _params_from_sd(g.F, load_ckpt(exp["ckpt"]))
    sc = Scorer(ps, params, batch_size=256)
    p1 = sc.probabilities().cpu().numpy()
    got = sorted([list(map(int, pairs[i])) for i in np.nonzero(p1 > float(thr))[0]])
    # a pair whose probability sits within fp32 rounding of the threshold may flip; none does here
    assert got == exp["positives"]
    # sharded scoring (2 shards, no communication) covers the same pairs with the same values
    parts = [Scorer(ps, params, batch_size=256, world_size=2, rank=r).probabilities().cpu().numpy() for r in range(2)]
    assert np.array_equal(np.concatenate(parts), p1)
    TP, FN, TN, FP = sc.confusion(threshold=float(thr))
    assert (TP, FN) == (0, 0) and FP == len(exp["positives"]) and TN + FP == len(pairs)
