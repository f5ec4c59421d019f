"""The drop-in operator modules of npi_gnn_b200.nn (SAGEConv, TopKPooling, global_max_pool,
global_mean_pool) and the COO kernels behind them, one operator at a time, forward and backward,
against the fp64 restatement of torch-geometric 1.4.2 in oracle/pyg_ops.py run on the CPU.

Tolerance: element-wise  |got - ref| <= K * 2^-24 * ref_abs + TINY,  where ref_abs is the same fp64
reference evaluated on absolute values (|x|, |W|, |b|, |g|): it bounds the magnitude of every term
that enters a result, so the check follows the rounding an fp32 kernel can make, entry by entry,
instead of the size of the largest entry.  Integer outputs, the max readout and the gate x*s are
compared exactly.  Graphs are synthetic and sized from the SM count so that every persistent kernel
walks more than one tile per CTA.
"""
import math

import numpy as np
import pytest
import torch

from oracle import pyg_ops

pytestmark = pytest.mark.gpu

K = 64                 # rounding budget, in units of 2^-24 * ref_abs
U = 2.0 ** -24
TINY = 1e-30
H = 128
DEV = "cuda"

F_ALL = [1, 3, 4, 12, 31, 32, 33, 64, 127, 128, 129, 178, 180, 252, 255, 256]


# ------------------------------------------------------------------------------------------ helpers
def _check(got, ref, ref_abs, what):
    got = got.detach().double().cpu()
    ref, ref_abs = ref.detach().double().cpu(), ref_abs.detach().double().cpu()
    assert got.shape == ref.shape, (what, tuple(got.shape), tuple(ref.shape))
    err = (got - ref).abs()
    bad = ~(err <= K * U * ref_abs + TINY)                   # NaN fails too
    if bool(bad.any()):
        i = int(torch.nonzero(bad.reshape(-1))[0])
        worst = float((err / (U * ref_abs + TINY)).max())
        raise AssertionError("%s: %d of %d entries off by more than K*2^-24*ref_abs (K=%d; worst err/(2^-24 ref_abs) = %.1f); "
                             "first at flat index %d: got %r, ref %r, ref_abs %r"
                             % (what, int(bad.sum()), bad.numel(), K, worst, i, float(got.reshape(-1)[i]),
                                float(ref.reshape(-1)[i]), float(ref_abs.reshape(-1)[i])))


def _same_bits(a, b, what):
    a, b = a.detach(), b.detach()
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    assert torch.equal(a, b), "%s differs between two identical runs" % what


@pytest.fixture(scope="module")
def sms():
    from npi_gnn_b200 import _lib, ops
    _lib.load()
    return ops.sm_count()


def feature_graph(N, seed, avg_deg=4):
    """int64 [2,E] edge multiset over N >= 6000 nodes, symmetric (every (i,j) as often as (j,i)), with the
    structures the aggregation kernels branch on:
      node 0      hub of degree 5000 (100 neighbours, 50 parallel edges each)
      nodes 1-3   degree 31, 32, 33 (around the 32-wide neighbour-index preload)
      nodes 4, 5  joined by 3 parallel edges and nothing else (multi-edges count with multiplicity)
      node 6      two explicit self loops and two real edges; node 7 a self loop only (PyG drops both, re-adds one)
      nodes 8-19  isolated (the mean is the node itself)
      nodes >= 20 random edges, self loops and duplicates included; edge order shuffled."""
    rng = np.random.default_rng(seed)
    src, dst = [], []

    def both(a, b):
        src.extend([a, b]); dst.extend([b, a])

    for j in range(20, 120):
        for _ in range(50):
            both(0, j)
    nb = rng.choice(np.arange(20, N), 31 + 32 + 33, replace=False)
    for node, lo, hi in ((1, 0, 31), (2, 31, 63), (3, 63, 96)):
        for j in nb[lo:hi]:
            both(node, int(j))
    for _ in range(3):
        both(4, 5)
    src += [6, 6, 7]; dst += [6, 6, 7]
    both(6, 20); both(6, 21)
    m = avg_deg * N // 2
    a = rng.integers(20, N, m); b = rng.integers(20, N, m)
    b[:50] = a[:50]                                          # self loops among the random edges
    a[50:90] = a[100:140]; b[50:90] = b[100:140]             # duplicate edges
    s = np.concatenate([np.array(src), a, b]); d = np.concatenate([np.array(dst), b, a])
    order = rng.permutation(len(s))
    ei = np.stack([s[order], d[order]]).astype(np.int64)
    keep = ei[0] != ei[1]
    deg = np.bincount(ei[1][keep], minlength=N)
    assert list(deg[:8]) == [5000, 31, 32, 33, 3, 3, 2, 0] and not deg[8:20].any()
    return torch.from_numpy(ei)


@pytest.fixture(scope="module")
def small_graph():
    N = 6007
    return feature_graph(N, seed=1), N


@pytest.fixture(scope="module")
def big_graph(sms):
    # sage_fwd / sage_bwd_input run 2 CTAs per SM over 64-row tiles: N above twice one pass
    N = 2 * (2 * sms * 64) + 77
    return feature_graph(N, seed=2), N


# ------------------------------------------------------------------------------------------ SAGEConv
def sage_ref(x, ei, W, b, g, need_dx):
    """fp64 forward and autograd gradients of pyg_ops.sage_conv, and the same on absolute values."""
    res = []
    for f in (lambda t: t, torch.abs):
        xd = f(x.double()).requires_grad_(need_dx)
        Wd = f(W.double()).requires_grad_()
        bd = f(b.double()).requires_grad_()
        out = pyg_ops.sage_conv(xd, ei, Wd, bd)
        out.backward(f(g.double()))
        res.append(dict(out=out.detach(), dW=Wd.grad, db=bd.grad, dx=xd.grad))
    return res


def _x_layout(N, F, layout, gen):
    """x on the device as SAGEConv's kernels may see it.  'contig': [N,F] contiguous.  'slice4': a column slice
    of a wider buffer, 16-byte aligned with ld % 4 == 0 (the float4 path even for F % 4 != 0).  'slice1': a
    slice starting one float into the buffer (the scalar path).  Columns outside the slice are NaN: a kernel
    that reads them into a result fails."""
    x = torch.randn(N, F, generator=gen)
    if layout == "contig":
        return x, x.to(DEV)
    off = 4 if layout == "slice4" else 1
    buf = torch.full((N, (F + 3) // 4 * 4 + 8), float("nan"))
    buf[:, off:off + F] = x
    xv = buf.to(DEV)[:, off:off + F]
    aligned = xv.data_ptr() % 16 == 0 and xv.stride(0) % 4 == 0
    assert aligned == (layout == "slice4")
    return x, xv


def _sage_run(x_dev, ei_dev, N, W, b, g, layout):
    """(out, dW, db, dx) of one forward + backward: through the SAGEConv module for a contiguous x, through
    ops.sage_fwd / ops.sage_bwd_weight (which the module calls) for a strided view, which the module would copy."""
    F = W.shape[0]
    if layout == "contig":
        from npi_gnn_b200 import SAGEConv
        conv = SAGEConv(F, H).to(DEV)
        with torch.no_grad():
            conv.weight.copy_(W); conv.bias.copy_(b)
        x = x_dev.clone().requires_grad_(F == H)
        out = conv(x, ei_dev)
        out.backward(g)
        return out.detach(), conv.weight.grad, conv.bias.grad, x.grad
    from npi_gnn_b200 import _lib as L, ops
    from npi_gnn_b200.nn import _csr_of
    rowptr, col = _csr_of(ei_dev, N)
    out = torch.empty(N, H, device=DEV)
    ops.sage_fwd(L.features_dense(x_dev), rowptr, col, None, N, W, b, False, None, out, None, None)
    dW = torch.empty_like(W)
    db = torch.empty(H, device=DEV)
    ws = torch.empty(ops.sage_bwd_weight_workspace_bytes(F), dtype=torch.uint8, device=DEV)
    ops.sage_bwd_weight(L.features_dense(x_dev), rowptr, col, None, None, N, g, dW, db, ws)
    return out, dW, db, None


def _sage_case(ei, N, F, layout, seed):
    gen = torch.Generator().manual_seed(seed)
    x, x_dev = _x_layout(N, F, layout, gen)
    W = torch.randn(F, H, generator=gen) / math.sqrt(F)
    b = torch.randn(H, generator=gen)
    g = torch.randn(N, H, generator=gen)
    ei_dev = ei.to(DEV)
    dev = [t.to(DEV) for t in (W, b, g)]
    got = _sage_run(x_dev, ei_dev, N, *dev, layout)
    again = _sage_run(x_dev, ei_dev, N, *dev, layout)
    torch.cuda.synchronize()
    need_dx = layout == "contig" and F == H
    ref, ref_abs = sage_ref(x, ei, W, b, g, need_dx)
    for name, gt, gt2 in zip(("out", "dW", "db", "dx"), got, again):
        if name == "dx" and not need_dx:
            continue
        _check(gt, ref[name], ref_abs[name], "SAGEConv F=%d %s %s" % (F, layout, name))
        _same_bits(gt, gt2, "SAGEConv F=%d %s %s" % (F, layout, name))


@pytest.mark.parametrize("layout", ["contig", "slice4", "slice1"])
@pytest.mark.parametrize("F", F_ALL)
def test_sageconv_vs_fp64(small_graph, F, layout):
    """Forward, dW, db (and dx at F = 128) on a graph with a degree-5000 hub, rows of degree 31/32/33,
    multi-edges, self loops and isolated nodes."""
    ei, N = small_graph
    _sage_case(ei, N, F, layout, seed=F)


@pytest.mark.parametrize("F,layout", [(128, "contig"), (256, "slice4"), (255, "slice1"), (12, "contig")])
def test_sageconv_every_cta_loops(big_graph, F, layout):
    """N above twice the rows one pass of the persistent forward, weight-gradient and input-gradient grids covers."""
    ei, N = big_graph
    _sage_case(ei, N, F, layout, seed=1000 + F)


@pytest.mark.parametrize("case", ["single_node", "no_edges", "only_self_loops"])
@pytest.mark.parametrize("F", [3, 128])
def test_sageconv_degenerate_graphs(case, F):
    N = 1 if case == "single_node" else 37
    if case == "only_self_loops":
        v = torch.tensor([0, 3, 3, 5, 36, 36, 36])
        ei = torch.stack([v, v])
    else:
        ei = torch.empty(2, 0, dtype=torch.int64)
    _sage_case(ei, N, F, "contig", seed=7 + F)


# ------------------------------------------------------------------------------------------ TopKPooling
def topk_batch(sms, seed, extremes):
    """Graphs of 1, 2, 3, 255, 256, 257 (the shared-memory sorts) and 8193 nodes (the workspace sort) among
    random-size graphs, enough rows that at ratio 0.9 the backward's persistent grid loops: 3 CTAs per SM,
    8 warps, 8 rows a warp per pass.  With ``extremes``, some graphs are scaled so that tanh saturates to
    exactly +-1, some hold repeated rows (exact score ties) and all-zero rows (ties at 0)."""
    rng = np.random.default_rng(seed)
    target = math.ceil(2 * 3 * sms * 8 * 8 / 0.9) + 500
    special = [1, 2, 3, 255, 256, 257, 8193]
    sizes = []
    while sum(sizes) + sum(special) < target:
        sizes.append(int(rng.integers(1, 600)))
    for i, s in enumerate(special):
        sizes.insert((i * 7) % (len(sizes) + 1), s)
    sizes = np.array(sizes)
    gptr = np.concatenate([[0], np.cumsum(sizes)])
    N = int(gptr[-1])
    x = rng.standard_normal((N, H)).astype(np.float32)
    for gi, n in enumerate(sizes if extremes else []):
        lo, hi = gptr[gi], gptr[gi + 1]
        if n in (3, 256, 8193) or gi % 7 == 2:                  # exact ties: repeated rows and zero rows
            reps = rng.integers(lo, lo + max(1, n // 8), n)
            x[lo:hi] = x[reps]
            x[lo + n // 3:lo + n // 3 + n // 10] = 0.0
        if n in (257, 8193) or gi % 5 == 1:                     # saturated: |z| >> 9, s == +-1 exactly
            x[lo:lo + max(1, n // 2)] *= 60.0
    batch = np.repeat(np.arange(len(sizes)), sizes)
    E = 2 * N
    ei = np.stack([rng.integers(0, N, E), rng.integers(0, N, E)]).astype(np.int64)
    w = (rng.standard_normal((1, H)) * 0.1).astype(np.float32)
    return torch.from_numpy(x), torch.from_numpy(ei), torch.from_numpy(batch).long(), torch.from_numpy(w)


def topk_ref(x, w, ei, batch, perm, g):
    """fp64 TopKPooling with the kernel's perm forced, its gradients by autograd, and the abs pass: the same
    terms on absolute values, where tanh and 1 - s^2 also carry the rounding they pass on.  With t = 1 - s^2
    (= tanh'), an error of order 2^-24 z_abs in z moves s by t z_abs, and tanhf adds a few ulp of s:
    s_b = t z_abs + |s|.  The fp32 1 - s^2 is off by 2 t z_abs plus a few 2^-24 (a fraction of that where t
    itself is below 2^-24, as the fp32 score is then exactly +-1)."""
    x64 = x.double().requires_grad_()
    w64 = w.double().requires_grad_()
    xo, eo, _, bo, _, _ = pyg_ops.topk_pooling(x64, ei, batch, w64, forced_perm=perm)
    xo.backward(g.double())
    xa, wa, ga = x.double().abs(), w.double().abs(), g.double().abs()
    nrm = w.double().norm()
    z = (x.double() * w.double()).sum(-1) / nrm
    z_abs = (xa * wa).sum(-1) / nrm
    s = torch.tanh(z)
    t = 1 - s * s
    s_b = t * z_abs + s.abs()
    ds_abs = (ga * xa[perm]).sum(-1)
    tp = t[perm]
    dz_abs = ds_abs * (tp * (1 + 2 * z_abs[perm]) + 4 * torch.clamp(tp / U, max=1))
    dx_abs = torch.zeros_like(xa)
    dx_abs[perm] = ga * s_b[perm, None] + dz_abs[:, None] * wa / nrm
    dw_abs = (dz_abs[:, None] * xa[perm]).sum(0) / nrm + wa * (dz_abs * z_abs[perm]).sum() / nrm ** 2
    return dict(s=s, s_abs=s_b, xp=xo.detach(), xp_abs=xa[perm] * s_b[perm, None], eo=eo, bo=bo,
                dx=x64.grad, dx_abs=dx_abs, dw=w64.grad, dw_abs=dw_abs)


@pytest.fixture(scope="module")
def topk_data(sms):
    return {kind: topk_batch(sms, seed=5, extremes=kind == "extremes") for kind in ("extremes", "plain")}


def _topk_run(pool, x_dev, ei_dev, batch_dev, g_dev):
    x = x_dev.clone().requires_grad_()
    pool.weight.grad = None
    xp, eo, ea, bo, perm, sc = pool(x, ei_dev, None, batch_dev)
    assert ea is None
    xp.backward(g_dev)
    return xp.detach(), eo, bo, perm, sc.detach(), x.grad, pool.weight.grad.clone()


@pytest.mark.parametrize("ratio,kind", [(0.5, "extremes"), (0.3, "extremes"), (0.9, "extremes"), (1.0, "extremes"),
                                        (0.5, "plain"), (0.9, "plain")])
def test_topkpooling_vs_fp64(topk_data, ratio, kind):
    """Selection, x', batch', edge_index', dx and d weight.  The saturated rows of the "extremes" batch have a
    rounding allowance large enough to hide small errors in d weight (one sum over all rows); the "plain" batch
    keeps that check tight."""
    from npi_gnn_b200 import NPIError, TopKPooling, ops
    x, ei, batch, w = topk_data[kind]
    N = x.shape[0]
    pool = TopKPooling(H, ratio=ratio).to(DEV)
    with torch.no_grad():
        pool.weight.copy_(w)
    x_dev, ei_dev, batch_dev = x.to(DEV), ei.to(DEV), batch.to(DEV)
    # the kernel's own scores: the selection is checked against them (fp32 ties and saturation are its inputs)
    z_k = torch.empty(N, device=DEV)
    s_k = torch.empty(N, device=DEV)
    ops.topk_score(x_dev, None, N, w.to(DEV), z_k, s_k)
    s_k = s_k.cpu()
    perm_ref = pyg_ops.topk_perm(s_k, ratio, batch)
    k = torch.ceil(torch.tensor(ratio, dtype=torch.float32) * torch.bincount(batch).float()).long()
    assert perm_ref.numel() == int(k.sum())
    # upstream gradient partly aligned with sign(s) x: sum(dz z) then grows with the row count instead of
    # cancelling, so the w (dz.z) / |w|^2 term of d weight stands well above its rounding allowance
    g = torch.sign(s_k[perm_ref])[:, None] * x[perm_ref] + 0.5 * torch.randn(perm_ref.numel(), H,
                                                                             generator=torch.Generator().manual_seed(int(ratio * 10)))
    got = _topk_run(pool, x_dev, ei_dev, batch_dev, g.to(DEV))
    again = _topk_run(pool, x_dev, ei_dev, batch_dev, g.to(DEV))
    torch.cuda.synchronize()
    xp, eo, bo, perm, sc, dx, dw = got
    for name, a, b in zip(("x'", "edge_index'", "batch'", "perm", "score", "dx", "d weight"), got, again):
        _same_bits(a, b, "TopKPooling(ratio=%s) %s" % (ratio, name))
    perm = perm.cpu()
    assert torch.equal(perm, perm_ref), "perm differs from topk_perm of the kernel's own scores"
    ref = topk_ref(x, w, ei, batch, perm, g)
    _check(s_k, ref["s"], ref["s_abs"], "TopKPooling score")
    assert torch.equal(sc.cpu(), s_k[perm])
    assert torch.equal(xp.cpu(), x[perm] * s_k[perm, None]), "gate x*s is one fp32 product per element"
    _check(xp, ref["xp"], ref["xp_abs"], "TopKPooling x'")
    assert torch.equal(bo.cpu(), ref["bo"])
    assert torch.equal(eo.cpu(), ref["eo"]), "edge_index' differs from filter_adj (order kept)"
    _check(dx, ref["dx"], ref["dx_abs"], "TopKPooling dx")
    _check(dw, ref["dw"], ref["dw_abs"], "TopKPooling d weight")
    # a gradient through the returned score is not implemented: it must raise, not be dropped
    out = pool(x_dev.clone().requires_grad_(), ei_dev, None, batch_dev)
    with pytest.raises(NPIError):
        out[5].sum().backward()


# ------------------------------------------------------------------------------------------ global pools
def pool_batch(kind, seed):
    """(x, batch, size).  x has exact ties in columns 0-15 (small integers; -0.0 / +0.0 maxima in columns
    8-15), only negative values in columns 16-31 and random values elsewhere."""
    rng = np.random.default_rng(seed)
    if kind == "one_graph":
        sizes, extra = [20011], 0                                # splits over all GR_SPLIT row ranges
    elif kind == "empty_graphs":
        sizes, extra = [3, 0, 5, 0, 0, 1, 4], 2                  # empty in the middle and, via size, at the end
    else:
        sizes = list(rng.integers(1, 7, 5000))                   # B = 5000 ...
        sizes[2500] = 20000                                      # ... with one graph over the GR_SPLIT ranges
        sizes[1234] = 0
        extra = 3
    sizes = np.array(sizes)
    N = int(sizes.sum())
    x = rng.standard_normal((N, H)).astype(np.float32)
    x[:, 0:8] = rng.integers(-2, 3, (N, 8))
    v = -rng.integers(0, 3, (N, 8)).astype(np.float32)
    zero = np.where(rng.random((N, 8)) < 0.5, -0.0, 0.0).astype(np.float32)
    x[:, 8:16] = np.where(v == 0, zero, v)                       # maxima of 0 held by -0.0 and +0.0 rows
    x[:, 16:32] = -np.abs(x[:, 16:32]) - 1.0
    batch = np.repeat(np.arange(len(sizes)), sizes)
    return torch.from_numpy(x), torch.from_numpy(batch).long(), len(sizes) + extra


def max_pool_grad_ref(x, batch, B, mx, g):
    """dx of the max readout: the whole gradient to the LOWEST row attaining the maximum (the kernel's rule)."""
    N = x.shape[0]
    rows = torch.arange(N).view(-1, 1).expand(N, H)
    cand = torch.where(x.double() == mx[batch], rows, torch.full_like(rows, N))
    first = torch.full((B, H), N, dtype=torch.long).scatter_reduce(0, batch.view(-1, 1).expand(N, H), cand, "amin")
    dx = torch.zeros(N + 1, H, dtype=torch.float64)
    dx.scatter_(0, first, g.double())                            # empty graphs write into the spare row N
    return dx[:N]


def _pool_run(fn, x_dev, batch_dev, size, g_dev):
    x = x_dev.clone().requires_grad_()
    out = fn(x, batch_dev, size)
    out.backward(g_dev)
    return out.detach(), x.grad


@pytest.mark.parametrize("kind", ["one_graph", "empty_graphs", "many"])
def test_global_pools_vs_fp64(kind):
    from npi_gnn_b200 import global_max_pool, global_mean_pool
    x, batch, B = pool_batch(kind, seed=len(kind))
    g = torch.randn(B, H, generator=torch.Generator().manual_seed(3))
    x_dev, batch_dev, g_dev = x.to(DEV), batch.to(DEV), g.to(DEV)
    mx, dmx = _pool_run(global_max_pool, x_dev, batch_dev, B, g_dev)
    mn, dmn = _pool_run(global_mean_pool, x_dev, batch_dev, B, g_dev)
    for name, fn, got in (("max", global_max_pool, (mx, dmx)), ("mean", global_mean_pool, (mn, dmn))):
        again = _pool_run(fn, x_dev, batch_dev, B, g_dev)
        _same_bits(got[0], again[0], "global_%s_pool" % name)
        _same_bits(got[1], again[1], "global_%s_pool dx" % name)
    torch.cuda.synchronize()
    mx_ref = pyg_ops.global_max_pool(x.double(), batch, B)
    assert torch.equal(mx.cpu().double(), mx_ref), "global_max_pool must be exact"
    assert torch.equal(dmx.cpu().double(), max_pool_grad_ref(x, batch, B, mx_ref, g))
    res = []
    for f in (lambda t: t, torch.abs):
        xd = f(x.double()).requires_grad_()
        out = pyg_ops.global_mean_pool(xd, batch, B)
        out.backward(f(g.double()))
        res.append((out.detach(), xd.grad))
    (mn_ref, dmn_ref), (mn_abs, dmn_abs) = res
    _check(mn, mn_ref, mn_abs, "global_mean_pool")
    _check(dmn, dmn_ref, dmn_abs, "global_mean_pool dx")


def test_global_pool_empty_graph_reads_zero():
    """PyG returns 0 for a graph with no rows (scatter_mean clamps the count to 1, scatter_ zeroes the max fill)."""
    from npi_gnn_b200 import global_max_pool, global_mean_pool
    x = torch.randn(4, H, device=DEV) - 5.0
    batch = torch.tensor([0, 0, 2, 2], device=DEV)
    for fn in (global_max_pool, global_mean_pool):
        xg = x.clone().requires_grad_()
        out = fn(xg, batch)
        assert out.shape == (3, H)
        assert torch.equal(out[1], torch.zeros(H, device=DEV)), (fn.__name__, out[1, :4])
        out.backward(torch.ones_like(out))
        assert bool(torch.isfinite(xg.grad).all())


def test_global_pool_size_argument():
    from npi_gnn_b200 import NPIError, global_max_pool, global_mean_pool
    x = torch.randn(5, H, device=DEV)
    batch = torch.tensor([0, 0, 1, 1, 1], device=DEV)
    for fn in (global_max_pool, global_mean_pool):
        out = fn(x, batch, 4)
        assert out.shape == (4, H), fn.__name__
        assert torch.equal(out[2:], torch.zeros(2, H, device=DEV))
        assert torch.equal(out[:2], fn(x, batch))
        with pytest.raises(NPIError):
            fn(x, batch, 1)


def test_unsorted_batch_is_rejected():
    """The kernels take each graph's rows as one contiguous range; PyG accepts any order, so an unsorted batch
    would otherwise give wrong numbers silently."""
    from npi_gnn_b200 import NPIError, TopKPooling, global_max_pool, global_mean_pool
    x = torch.randn(6, H, device=DEV)
    batch = torch.tensor([0, 1, 0, 1, 2, 2], device=DEV)
    for fn in (global_max_pool, global_mean_pool):
        with pytest.raises(NPIError):
            fn(x, batch)
    ei = torch.tensor([[0, 1], [1, 0]], device=DEV)
    with pytest.raises(NPIError):
        TopKPooling(H).to(DEV)(x, ei, None, batch)


# ------------------------------------------------------------------------------------------ COO kernels
def test_coo_to_csr_vs_numpy():
    """npi_coo_to_csr at N + 1 > 256 * 1024 (the chunk-total scan past its first pass), with a 5000-entry row,
    duplicate edges and self loops: self loops dropped, edge order kept inside every row, bit-exact."""
    from npi_gnn_b200 import ops
    rng = np.random.default_rng(11)
    N = 300_000
    E0 = 400_000
    src = rng.integers(0, N, E0)
    dst = rng.integers(0, N, E0)
    src[:2000] = dst[:2000]                                       # self loops
    src[2000:4000], dst[2000:4000] = src[4000:6000], dst[4000:6000]   # duplicate edges
    hub = 6000 + rng.choice(E0 - 6000, 5000, replace=False)
    dst[hub] = 12345                                              # a 5000-entry row, with repeated sources
    src[hub] = rng.integers(0, 300, 5000)
    ei = np.stack([src, dst]).astype(np.int64)
    keep = ei[0] != ei[1]
    order = np.argsort(ei[1][keep], kind="stable")
    col_ref = ei[0][keep][order].astype(np.int32)
    rowptr_ref = np.concatenate([[0], np.cumsum(np.bincount(ei[1][keep], minlength=N))]).astype(np.int32)
    assert rowptr_ref[12346] - rowptr_ref[12345] >= 5000
    ei_dev = torch.from_numpy(ei).to(DEV)
    outs = []
    for _ in range(2):
        rowptr = torch.empty(N + 1, dtype=torch.int32, device=DEV)
        col = torch.full((E0 + 64,), -7, dtype=torch.int32, device=DEV)  # slack: a write past the end shows
        ops.coo_to_csr(ei_dev, N, rowptr, col)
        outs.append((rowptr.cpu().numpy(), col.cpu().numpy()))
    for rowptr, col in outs:
        assert np.array_equal(rowptr, rowptr_ref)
        assert np.array_equal(col[:len(col_ref)], col_ref)
        assert (col[len(col_ref):] == -7).all()


def test_filter_edges_coo_vs_filter_adj():
    """npi_filter_edges_coo against pyg_ops.filter_adj for E > 256 * 1024 (the chunk-total scan past its first
    pass), a shuffled perm, and with every edge dropped."""
    from npi_gnn_b200 import ops
    rng = np.random.default_rng(12)
    N, E = 60_000, 300_000
    ei = torch.from_numpy(np.stack([rng.integers(0, N, E), rng.integers(0, N, E)]).astype(np.int64))
    perm = torch.from_numpy(rng.permutation(N)[:N // 2].astype(np.int64))
    new_id = torch.full((N,), -1, dtype=torch.int32)
    new_id[perm] = torch.arange(perm.numel(), dtype=torch.int32)
    ref = pyg_ops.filter_adj(ei, perm, N)
    ei_dev = ei.to(DEV)
    for nid, want in ((new_id, ref), (torch.full((N,), -1, dtype=torch.int32), torch.empty(2, 0, dtype=torch.int64))):
        for _ in range(2):
            out = torch.full((2, E), -7, dtype=torch.int64, device=DEV)
            cnt = torch.full((1,), -1, dtype=torch.int32, device=DEV)
            ops.filter_edges_coo(ei_dev, nid.to(DEV), out, cnt)
            Ep = int(cnt.item())
            assert Ep == want.shape[1]
            assert torch.equal(out[:, :Ep].cpu(), want)
            assert bool((out[:, Ep:] == -7).all())


def test_edge_symmetry_sums():
    """Symmetric multigraphs give equal fingerprints whatever self loops are added; a missing reverse edge or a
    multiplicity that differs between (i,j) and (j,i) gives different ones, and SAGEConv refuses the edge set."""
    from npi_gnn_b200 import NPIError, SAGEConv, ops
    rng = np.random.default_rng(13)
    N, M = 5000, 40_000
    a, b = rng.integers(0, N, M), rng.integers(0, N, M)
    a[:500], b[:500] = a[500:1000], b[500:1000]                   # multiplicities > 1
    sym = np.stack([np.concatenate([a, b]), np.concatenate([b, a])])
    sym = sym[:, rng.permutation(sym.shape[1])]

    def sums(e):
        return tuple(ops.edge_symmetry_sums(torch.from_numpy(np.ascontiguousarray(e, dtype=np.int64)).to(DEV)).tolist())

    base = sums(sym)
    assert base[0] == base[1]
    loops = rng.integers(0, N, 300)
    for extra in (np.stack([loops[:1], loops[:1]]), np.stack([loops, loops]), np.stack([loops[:7].repeat(5)] * 2)):
        assert sums(np.concatenate([sym, extra], 1)) == base
    i, j = next((int(p), int(q)) for p, q in sym.T if p != q)
    drop = np.nonzero((sym[0] == j) & (sym[1] == i))[0][0]
    missing = np.delete(sym, drop, axis=1)                          # (i,j) loses one copy of its reverse
    extra = np.concatenate([sym, [[i], [j]]], 1)                    # (i,j) once more than (j,i)
    conv = SAGEConv(8, H).to(DEV)
    x = torch.randn(N, 8, device=DEV)
    for bad in (missing, extra):
        s = sums(bad)
        assert s[0] != s[1]
        with pytest.raises(NPIError):
            conv(x, torch.from_numpy(bad).to(DEV))
