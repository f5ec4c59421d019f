"""Input attribution of scored pairs on the GPU (Explainer, npi_input_attribution) -- against the fp64 oracle under
autograd, forced to the CUDA path's discrete decisions, on real and degenerate batches; exact properties, internal
consistency, agreement with Scorer, determinism, the kernel in isolation and top_nodes."""
import numpy as np
import pytest
import torch

from oracle import khop, khop_cwrap, net as onet
from tests.common import load_ckpt, npinter2_oracle_graph

pytestmark = pytest.mark.gpu

LOGP_ATOL_FORCED = 5e-4      # SURVEY 7.3: log-probs with the oracle forced to the CUDA selections
GRAD_REL_FORCED = 1e-3       # max-norm relative, per tensor


def _rel(got, ref):
    got, ref = torch.as_tensor(got).double().cpu(), torch.as_tensor(ref).double().cpu()
    return float((got - ref).abs().max() / max(float(ref.abs().max()), 1e-12))


@pytest.fixture(scope="module")
def npi():
    from npi_gnn_b200.graph import BipartiteGraph
    d, og, omask = npinter2_oracle_graph()
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(np.concatenate([d["test_pos"], d["test_neg"]]))
    return d, og, omask, g


def _test_pairs(d, n=None):
    """NPInter2 fold-0 test pairs, positives and negatives interleaved."""
    k = min(len(d["test_pos"]), len(d["test_neg"]))
    pairs = np.stack([d["test_pos"][:k], d["test_neg"][:k]], 1).reshape(-1, 2)
    ys = np.tile(np.array([1, 0], dtype=np.int32), k)
    return (pairs, ys) if n is None else (pairs[:n], ys[:n])


def _params(F, ckpt=None, seed=5):
    from npi_gnn_b200.engine import FlatParams
    if ckpt is None:
        return FlatParams(F, "cuda").init_reference(torch.Generator().manual_seed(seed))
    return FlatParams(F, "cuda").load_state_dict(load_ckpt(ckpt))


def _oracle(ex, pairs, ys, h, table, og, omask, target, wrt):
    """fp64 oracle in eval mode on the ONE batch the explainer's engine holds, forced to its top-k selections, ReLU masks
    and max-pool rows, with x.requires_grad_().  The head's ReLUs run free (the oracle's forced_head encodes the
    training-mode dropout scale): their decisions are asserted equal to the CUDA path's."""
    eng = ex.engine
    B = len(pairs)
    N, _ = eng.counters()
    perms = [eng.perm[l][:N[l + 1]].cpu().long() for l in range(3)]
    relu = [(eng.layer_rows(l, N[l])[0] > 0).cpu() for l in range(3)]
    amax = [eng.argmax[l][:B].cpu().long() for l in range(3)]
    c = khop_cwrap.collate_batch(og, omask, pairs, ys, h, table)
    assert N[0] == len(c["gid"])
    m = onet.Net_1(ex.ps.graph.F).double()
    m.load_state_dict({k: v.cpu().double() for k, v in ex.params.state_dict().items()})
    m.eval()
    bn = onet.batch_namespace(c)
    x = bn.x.double().requires_grad_()
    bn.x = x
    out = m(bn, forced_perms=perms, forced_relu=relu, forced_argmax=amax)
    assert max(m.trace.max_gap) < 1e-5
    for pre, cuda in zip(m.trace.head_pre, (eng.a1[:B], eng.a2[:B])):
        diff = (cuda > 0).cpu() != (pre.detach() > 0)
        assert not diff.any(), "head ReLU decided differently at |pre| = %g" % float(pre.detach()[diff].abs().min())
    t = out[:, target]
    if wrt == "prob":
        t = t.exp()
    t.sum().backward()
    gx = x.grad
    xg = x.detach() * gx
    fa = torch.zeros(B, x.shape[1], dtype=torch.float64).index_add_(0, torch.from_numpy(c["batch"]).long(), xg)
    return dict(logp=out.detach(), grad_x=gx, node_attr=xg.sum(1), feature_attr=fa, c=c)


def _check_vs_oracle(res, ref, bar=GRAD_REL_FORCED):
    assert float((res["logp"].cpu().double() - ref["logp"]).abs().max()) < LOGP_ATOL_FORCED
    errs = {k: _rel(res[k], ref[k]) for k in ("grad_x", "node_attr", "feature_attr")}
    assert max(errs.values()) < bar, errs
    c = ref["c"]
    assert np.array_equal(res["node"].cpu().numpy(), c["gid"])
    assert np.array_equal(res["hop"].cpu().numpy(), c["dist"])
    assert np.array_equal(res["node_ptr"].cpu().numpy(), c["graph_ptr"].astype(np.int64))
    return errs


# ----------------------------------------------------------------------------- against the fp64 oracle
@pytest.mark.parametrize("target,wrt", [(1, "logp"), (1, "prob"), (0, "logp")])
@pytest.mark.parametrize("h,ckpt", [(1, "ckpt_1223_1_15.npz"), (2, "ckpt_1223_1_5.npz")])
def test_explain_vs_oracle(npi, h, ckpt, target, wrt):
    from npi_gnn_b200 import Explainer
    from npi_gnn_b200.graph import PairSet
    torch.set_flush_denormal(True)
    d, og, omask, g = npi
    pairs, ys = _test_pairs(d, 48)
    ps = PairSet(g, pairs, ys, h=h)
    ex = Explainer(ps, _params(g.F, ckpt), batch_size=len(pairs))
    res = ex.explain(target=target, wrt=wrt, full=True)
    torch.cuda.synchronize()
    ref = _oracle(ex, pairs, ys, h, d["table"], og, omask, target, wrt)
    errs = _check_vs_oracle(res, ref)
    print("h=%d target=%d wrt=%s tiny=%s: %s" % (h, target, wrt, ex.engine.tiny, errs))


@pytest.mark.parametrize("tiny", ["1", "0"])
def test_both_paths_vs_oracle_on_rpi2241_shaped(monkeypatch, tiny):
    """15-node subgraphs: the per-subgraph path (csrc/tiny.cu) and the per-layer path both meet the oracle bar."""
    from npi_gnn_b200 import Explainer, synth
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    torch.set_flush_denormal(True)
    monkeypatch.setenv("NPI_TINY", tiny)
    d = synth.rpi2241_shaped(no_kmer=True)
    pairs, ys = synth.train_pairs(d)
    pairs, ys = pairs[:200], ys[:200]
    cannot = synth.masked_pairs(d)
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    omask = khop.mask_from_keys(og, [tuple(e) for e in cannot.tolist()])
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(cannot)
    ps = PairSet(g, pairs, ys, h=2)
    ex = Explainer(ps, _params(g.F, "ckpt_1223_1_noKmer_20.npz"), batch_size=200)
    assert ex.engine.tiny == (tiny == "1")
    res = ex.explain(full=True)
    torch.cuda.synchronize()
    ref = _oracle(ex, pairs, ys, 2, d["table"], og, omask, 1, "logp")
    print("tiny=%s: %s" % (tiny, _check_vs_oracle(res, ref)))


# ----------------------------------------------------------------------------- degenerate batches
def _degenerate_graph(seed=3, F=8):
    """Isolated pairs (2-node subgraphs; the first one's two nodes have all-zero feature rows), a star (one protein with
    300 RNAs: 302 rows at h = 2, ten 32-row chunks), a second protein shared by 20 of the star's RNAs, and candidate
    pairs without an edge."""
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
    lone_r, lone_p = node(1), node(0)
    table = rng.standard_normal((len(is_rna), F)).astype(np.float32)
    table[list(iso[0])] = 0.0
    d = dict(edges=np.asarray(edges, dtype=np.int32), is_rna=np.asarray(is_rna, dtype=np.uint8), table=table)
    pairs = iso + [(leaves[0], hub), (leaves[5], p2), (leaves[299], hub), (lone_r, lone_p), (leaves[1], lone_p), (iso[0][0], hub)]
    return d, np.asarray(pairs, dtype=np.int32)


def _degenerate(h):
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    d, pairs = _degenerate_graph()
    ys = (np.arange(len(pairs)) % 2).astype(np.int32)
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    omask = khop.mask_from_keys(og, [tuple(d["edges"][3].tolist())])
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(d["edges"][3:4])
    return d, pairs, ys, og, omask, g, PairSet(g, pairs, ys, h=h)


@pytest.mark.parametrize("h", [1, 2])
@pytest.mark.parametrize("single", [False, True])
def test_degenerate_batches_vs_oracle(h, single):
    """2-node subgraphs, the star's hub subgraph over many chunks, and P = 1 (the star seen from one leaf)."""
    from npi_gnn_b200 import Explainer
    from npi_gnn_b200.graph import PairSet
    torch.set_flush_denormal(True)
    d, pairs, ys, og, omask, g, ps = _degenerate(h)
    if single:
        pairs, ys = pairs[6:7], ys[6:7]
        ps = PairSet(g, pairs, ys, h=h)
    ex = Explainer(ps, _params(g.F), batch_size=len(pairs))
    res = ex.explain(full=True)
    torch.cuda.synchronize()
    ref = _oracle(ex, pairs, ys, h, d["table"], og, omask, 1, "logp")
    _check_vs_oracle(res, ref)
    n = ps.n_h
    if not single:
        assert n.min() == 2 and (h == 1 or n.max() > 32 * 8)
        na = res["node_attr"].cpu()
        assert torch.equal(na[:2], torch.zeros(2))      # the all-zero rows (table rows 0, label 0) of the first pair


def test_tail_batch_and_repeated_pairs():
    """P not a multiple of B, and an index view that lists pairs twice -- in one batch and across batches: each copy gives
    the same bits, and every pair the same attributions as in one batch of all pairs."""
    from npi_gnn_b200 import Explainer
    d, pairs, ys, og, omask, g, ps = _degenerate(2)
    params = _params(g.F)
    whole = Explainer(ps, params, batch_size=len(pairs)).explain(full=True)
    tail = Explainer(ps, params, batch_size=5).explain(full=True)            # 5 + 5 + 2
    for k in ("logp", "node_attr", "feature_attr", "grad_x"):
        assert _rel(tail[k], whole[k]) < 1e-6, k
    for k in ("node_ptr", "node", "hop"):
        assert torch.equal(tail[k], whole[k]), k
    index = np.array([6, 0, 6, 3, 8, 6, 0, 11, 3], dtype=np.int64)
    view = Explainer(ps, params, batch_size=4, index=index).explain(full=True)
    wp, vp = whole["node_ptr"].cpu().numpy(), view["node_ptr"].cpu().numpy()
    assert np.array_equal(np.diff(vp), ps.n_h[index])
    for j, p in enumerate(index):
        for k in ("logp", "feature_attr"):
            assert _rel(view[k][j], whole[k][p]) < 1e-6, (k, j)
        for k in ("node_attr", "grad_x", "node", "hop"):
            assert _rel(view[k][vp[j]:vp[j + 1]], whole[k][wp[p]:wp[p + 1]]) < 1e-6, (k, j)
    for p in (6, 0, 3):                                                      # the copies of one pair: bit for bit
        js = np.nonzero(index == p)[0]
        for j in js[1:]:
            for k in ("logp", "feature_attr"):
                assert torch.equal(view[k][j], view[k][js[0]]), (k, p)
            for k in ("node_attr", "grad_x"):
                assert torch.equal(view[k][vp[j]:vp[j + 1]], view[k][vp[js[0]]:vp[js[0] + 1]]), (k, p)


# ----------------------------------------------------------------------------- exact properties, internal consistency
def _x_rows(g, res):
    x = g.table[res["node"].long(), :g.F].double()
    x[:, 0] = res["hop"].double()
    return x


def test_exact_properties_and_internal_consistency(npi):
    from npi_gnn_b200 import Explainer
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    pairs, ys = _test_pairs(d, 100)
    ps = PairSet(g, pairs, ys, h=2)
    params = _params(g.F, "ckpt_1223_1_5.npz")
    ex = Explainer(ps, params, batch_size=100)            # one batch: the engine keeps its dxa and projected table
    res = ex.explain(full=True)
    torch.cuda.synchronize()
    c = khop_cwrap.collate_batch(og, omask, pairs, ys, 2, d["table"])
    assert np.array_equal(res["node"].cpu().numpy(), c["gid"])
    assert np.array_equal(res["hop"].cpu().numpy(), c["dist"])
    assert np.array_equal(res["node_ptr"].cpu().numpy(), np.concatenate([[0], np.cumsum(ps.n_h)]))
    R = int(ps.n_h.sum())
    # node_attr = dxa . (T[gid] + dist W1[0]) with T = table . W1, the engine's projected table
    eng = ex.engine
    w1 = params.view("conv1.weight").double()
    proj = eng.T[eng.gid[:R].long()].double() + eng.dist[:R].double()[:, None] * w1[0]
    assert _rel(res["node_attr"], (eng.big[:R].double() * proj).sum(1)) < 1e-5
    # sum over features of feature_attr = sum over rows of node_attr, to 1e-5 of the sum of magnitudes
    x = _x_rows(g, res)
    mag = (x * res["grad_x"].double()).abs().sum(1)
    ptr = res["node_ptr"]
    pair = torch.repeat_interleave(torch.arange(len(pairs), device="cuda"), ptr.diff())
    na_sum = torch.zeros(len(pairs), dtype=torch.float64, device="cuda").index_add_(0, pair, res["node_attr"].double())
    mag_sum = torch.zeros(len(pairs), dtype=torch.float64, device="cuda").index_add_(0, pair, mag)
    assert ((res["feature_attr"].double().sum(1) - na_sum).abs() <= 1e-5 * mag_sum).all()
    # column 0 of feature_attr is the structural label's share, sum of dist_i * grad_x[i, 0] (rows with dist 0 add exactly
    # nothing: test_kernel_label_column_and_zero_rows)
    lab = torch.zeros(len(pairs), dtype=torch.float64, device="cuda").index_add_(0, pair, x[:, 0] * res["grad_x"][:, 0].double())
    assert _rel(res["feature_attr"][:, 0], lab) < 1e-5
    # wrt="prob" is p_1 times the logp result
    pr = ex.explain(wrt="prob", full=True)
    p1 = res["logp"][:, 1].double().exp()
    assert _rel(pr["feature_attr"], res["feature_attr"].double() * p1[:, None]) < 1e-5
    assert _rel(pr["node_attr"], res["node_attr"].double() * p1[pair]) < 1e-5
    assert _rel(pr["grad_x"], res["grad_x"].double() * p1[pair][:, None]) < 1e-5
    assert torch.equal(pr["logp"], res["logp"])


def test_logp_equals_scorer_bit_for_bit(npi):
    """exp(logp[:, 1]) of the explain sweep is Scorer.probabilities() bit for bit: the same forward, per row instead of
    per layer-1 context (documented bit-identical), with a tail batch."""
    from npi_gnn_b200 import Explainer, Scorer
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    pairs, ys = _test_pairs(d)
    ps = PairSet(g, pairs, ys, h=2)
    params = _params(g.F, "ckpt_1223_1_5.npz")
    res = Explainer(ps, params, batch_size=200).explain()
    prob = Scorer(ps, params, batch_size=200).probabilities()
    assert len(pairs) % 200 != 0
    assert torch.equal(torch.exp(res["logp"][:, 1]), prob)


# ----------------------------------------------------------------------------- determinism
def test_rerun_is_bit_identical_with_poisoned_buffers(npi):
    from npi_gnn_b200 import Explainer
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    pairs, ys = _test_pairs(d, 250)
    ps = PairSet(g, pairs, ys, h=2)
    ex = Explainer(ps, _params(g.F, "ckpt_1223_1_5.npz"), batch_size=100)
    a = ex.explain(full=True)
    torch.cuda.synchronize()
    junk = [torch.full((t.numel(),), float("nan"), device="cuda") for t in a.values() for _ in range(2)]
    del junk                                              # the caching allocator hands the NaN blocks out again
    ex.ws.fill_(0xFF)
    ex.engine.big.fill_(float("nan"))
    b = ex.explain(full=True)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_batch_size_does_not_change_a_pairs_attributions(npi, monkeypatch):
    """The same pair in batches of 1, 7 and 200 on the per-layer path: within 1e-6 relative per tensor.  Chunks of the
    attribution kernel start at each pair's first row, so its sums do not depend on the pair's place in the batch; what
    is asserted beyond that is whether the backward pass's layer-1 gradient is too (BITWISE below)."""
    from npi_gnn_b200 import Explainer
    from npi_gnn_b200.graph import PairSet
    monkeypatch.setenv("NPI_TINY", "0")
    d, og, omask, g = npi
    pairs, ys = _test_pairs(d, 200)
    ps = PairSet(g, pairs, ys, h=2)
    params = _params(g.F, "ckpt_1223_1_5.npz")
    out = {}
    for B in (1, 7, 200):
        ex = Explainer(ps, params, batch_size=B)
        assert not ex.engine.tiny
        out[B] = ex.explain(full=True)
    bitwise = {}
    for B in (1, 7):
        for k in ("logp", "node_attr", "feature_attr", "grad_x"):
            assert _rel(out[B][k], out[200][k]) < 1e-6, (B, k)
            bitwise[(B, k)] = torch.equal(out[B][k], out[200][k])
    print("bit-identical across batch sizes:", bitwise)
    assert all(bitwise.values()) == BITWISE_ACROSS_BATCH_SIZES, bitwise


# Measured on a B200: the per-layer path gives every pair the same bits in batches of 1, 7 and 200.
BITWISE_ACROSS_BATCH_SIZES = True


# ----------------------------------------------------------------------------- the kernel in isolation
def _kernel_case(rng, F, sizes, V=300, ld=None, dist_max=4):
    ld = ld or (F + 3) // 4 * 4
    N = int(sum(sizes))
    dxa = torch.from_numpy(rng.standard_normal((N, 128)).astype(np.float32)).cuda()
    table = torch.from_numpy(rng.standard_normal((V, ld)).astype(np.float32)).cuda()
    w1 = torch.from_numpy((rng.standard_normal((F, 128)) / np.sqrt(F)).astype(np.float32)).cuda()
    gid = torch.from_numpy(rng.integers(0, V, N).astype(np.int32)).cuda()
    dist = torch.from_numpy(rng.integers(0, dist_max, N).astype(np.uint8)).cuda()
    gptr = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).cuda()
    return dxa, gid, dist, gptr, table, w1


def _kernel_ref(dxa, gid, dist, gptr, table, w1, F):
    x = table[gid.long(), :F].double()
    x[:, 0] = dist.double()
    gx = dxa.double() @ w1.double().t()
    xg = x * gx
    mag = x.abs() * (dxa.double().abs() @ w1.double().abs().t())     # what fp32 rounding of the 128-term dots scales with
    B = gptr.numel() - 1
    pair = torch.repeat_interleave(torch.arange(B, device="cuda"), gptr.diff().long())
    fa = torch.zeros(B, F, dtype=torch.float64, device="cuda").index_add_(0, pair, xg)
    fmag = torch.zeros(B, F, dtype=torch.float64, device="cuda").index_add_(0, pair, mag)
    return gx, xg.sum(1), mag.sum(1), fa, fmag


def _run_kernel(case, F, full=True, poison=True):
    from npi_gnn_b200 import ops
    dxa, gid, dist, gptr, table, w1 = case
    N, B = dxa.shape[0], gptr.numel() - 1
    fill = float("nan") if poison else 0.0
    na = torch.full((N,), fill, device="cuda")
    fa = torch.full((B, F), fill, device="cuda")
    gx = torch.full((N, F), fill, device="cuda") if full else None
    ws = torch.full((ops.input_attribution_workspace_bytes(N, B, F),), 0xFF, dtype=torch.uint8, device="cuda")
    ops.input_attribution(dxa, gid, dist, gptr, B, N, table, F, w1, na, fa, ws, grad_x=gx)
    return na, fa, gx


@pytest.mark.parametrize("F", [1, 8, 65, 178, 256])
@pytest.mark.parametrize("shape", ["rows0", "rows1", "many"])
def test_kernel_vs_float64(F, shape):
    rng = np.random.default_rng(F * 7 + len(shape))
    sizes = {"rows0": [0, 0, 0], "rows1": [1],
             # one-row pairs, pairs of 31 / 32 / 33 rows, a hub of 3,001 rows (94 chunks), an empty pair, random sizes
             "many": [1, 1, 2, 31, 32, 33, 3001, 0, 1] + list(rng.integers(1, 80, 300)) + [64, 1]}[shape]
    case = _kernel_case(rng, F, sizes)
    na, fa, gx = _run_kernel(case, F)
    ref_gx, ref_na, mag_na, ref_fa, mag_fa = _kernel_ref(*case, F)
    if shape == "rows0":
        assert torch.equal(fa, torch.zeros_like(fa))
        return
    assert _rel(gx, ref_gx) < 1e-5
    assert ((na.double() - ref_na).abs() <= 1e-5 * mag_na + 1e-30).all()
    assert ((fa.double() - ref_fa).abs() <= 1e-5 * mag_fa + 1e-30).all()
    if shape == "many":
        assert torch.equal(fa[7], torch.zeros(F, device="cuda"))                        # the empty pair
    # bit-identical on rerun (fresh poisoned buffers), and without grad_x
    na2, fa2, gx2 = _run_kernel(case, F)
    na3, fa3, _ = _run_kernel(case, F, full=False)
    assert torch.equal(na, na2) and torch.equal(fa, fa2) and torch.equal(gx, gx2)
    assert torch.equal(na, na3) and torch.equal(fa, fa3)


def test_kernel_label_column_and_zero_rows():
    """Rows with dist 0 add exactly nothing to column 0; a row whose table row and label are zero has node_attr 0."""
    rng = np.random.default_rng(4)
    F = 65
    case = list(_kernel_case(rng, F, [40, 3, 70], V=50))
    case[1][:] = torch.arange(113, device="cuda", dtype=torch.int32) % 50
    case[2][:40] = 0                                                                     # pair 0: every label 0
    case[2][40:43] = 0
    case[4][7] = 0.0                                                                     # rows of node 7: zero features
    na, fa, gx = _run_kernel(case, F)
    assert float(fa[0, 0]) == 0.0 and float(fa[1, 0]) == 0.0
    zero = (case[1] == 7) & (case[2] == 0)
    assert zero.any() and torch.equal(na[zero], torch.zeros(int(zero.sum()), device="cuda"))
    assert torch.isfinite(gx).all()


def test_kernel_argument_errors_and_workspace_query():
    from npi_gnn_b200 import NPIError, ops, _lib as L
    import ctypes as C
    rng = np.random.default_rng(1)
    F = 8
    case = _kernel_case(rng, F, [5, 40])
    dxa, gid, dist, gptr, table, w1 = case
    N, B = 45, 2
    need = ops.input_attribution_workspace_bytes(N, B, F)
    assert need >= 4 * (B + 1) + 4 * F * 2                                              # chunk pointers + two chunk partials
    assert ops.input_attribution_workspace_bytes(N, B, 256) > need
    assert ops.input_attribution_workspace_bytes(10 * N, B, F) > need
    na = torch.empty(N, device="cuda"); fa = torch.empty(B, F, device="cuda")
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")

    def call(F_=F, B_=B, n=N, ld=table.stride(0), ws_bytes=need, gp=gptr, w=w1, feat=fa, d=dxa):
        L.call("npi_input_attribution", L.ptr(d), L.ptr(gid), L.ptr(dist), L.ptr(gp), C.c_int32(B_), C.c_int32(n), L.ptr(table),
               C.c_int32(ld), C.c_int32(F_), L.ptr(w), L.ptr(na), L.ptr(feat), None, L.ptr(ws), C.c_int64(ws_bytes),
               L.stream_ptr())
    call()
    for kw, msg in ((dict(F_=0), "F = 0"), (dict(F_=257), "F = 257"), (dict(B_=0), "B = 0"), (dict(n=-1), "n_rows"),
                    (dict(ld=F - 1), "row stride"), (dict(ws_bytes=need - 1), "workspace"), (dict(gp=None), "null"),
                    (dict(w=None), "null"), (dict(feat=None), "null"), (dict(d=None), "null"),
                    (dict(d=dxa.view(-1)[1:]), "aligned")):
        with pytest.raises(NPIError, match=msg):
            call(**kw)
    with pytest.raises(NPIError, match="input_attribution"):                           # the wrapper's own checks
        ops.input_attribution(dxa.double(), gid, dist, gptr, B, N, table, F, w1, na, fa, ws)
    with pytest.raises(NPIError, match="input_attribution"):
        ops.input_attribution(dxa, gid, dist, gptr, B, N, table, F, w1, na, fa[:1], ws)


# ----------------------------------------------------------------------------- top_nodes
def test_top_nodes_vs_host_argsort(npi):
    from npi_gnn_b200 import Explainer
    from npi_gnn_b200.graph import PairSet
    d, og, omask, g = npi
    pairs, ys = _test_pairs(d, 120)
    ps = PairSet(g, pairs, ys, h=2)
    res = Explainer(ps, _params(g.F, "ckpt_1223_1_5.npz"), batch_size=50).explain()
    na, node, ptr = res["node_attr"].cpu().numpy(), res["node"].cpu().numpy(), res["node_ptr"].cpu().numpy()
    for k in (1, 5, 1024):
        top = Explainer.top_nodes(res, k)
        tn, ta, tc = top["node"].cpu().numpy(), top["attr"].cpu().numpy(), top["count"].cpu().numpy()
        for p in range(len(pairs)):
            a = na[ptr[p]:ptr[p + 1]]
            order = np.argsort(-np.abs(a), kind="stable")[:k]          # ties by position
            cnt = len(order)
            assert tc[p] == cnt
            assert np.array_equal(tn[p, :cnt], node[ptr[p]:ptr[p + 1]][order])
            assert np.array_equal(ta[p, :cnt].view(np.uint32), a[order].view(np.uint32))
            assert (tn[p, cnt:] == -1).all() and np.isnan(ta[p, cnt:]).all()
