"""The CSR aggregation kernels of csrc/agg.cu one entry point at a time -- npi_sage_aggregate_fwd,
npi_sage_aggregate_bwd, npi_csr_gather_sum and the queues that feed them (npi_hub_rows_build and
npi_filter_adj) -- against an fp64 restatement of each kernel's documented formula on the CPU.

Tolerance: element-wise  |got - ref| <= (K_i + C) * 2^-24 * ref_abs + TINY,  where ref_abs is the same
reference run on absolute values and K_i counts the sequential additions the documented summation
order makes in row i:
  short row (<= 16 entries)  L + 1           (entries in CSR order, then the self row)
  hub row                    32 + nseg + 1   (one 32-entry segment, the nseg partials, the self row)
  two-level (gather, > 16 segments)  32 + 8 + ngrp  (one segment, 8 partials of a group, the group sums)
and C covers the division, the bias, the label FMA and the rounded 1/(deg+1) weight.  The bound is
below the mean size of one term at every row length tested (0.8 of it at 20,000 entries, far less
below), so a dropped entry, segment or group fails.
Integer outputs (queue headers, segment lists, row records) are compared exactly, and the plain and
pipelined kernels must agree bit for bit.  The CSRs are synthetic and sized from the SM count so that
every persistent warp loops more than once over the short rows and over the hub segments.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
TINY = 1e-30
C_FIN = 6              # division, bias, label FMA, rounded 1/(deg+1), in units of 2^-24 * ref_abs
H = 128
DEV = "cuda"
SEG, HUB, GRP = 32, 16, 8          # AG_SEG, AG_HUB, HUB_GRP of csrc/hub.cuh
AG_CTAS, AG_WARPS = 3, 8           # CTAs per SM and warps per CTA of the aggregation kernels

SPECIAL = list(range(0, 41)) + [63, 64, 65, 127, 128, 129, 511, 512, 513, 544, 1024, 1025, 5000, 20000]


# ------------------------------------------------------------------------------------------ helpers
def _check(got, ref, ref_abs, K, what):
    """K: per-row rounding budget (tensor [n] or [n,1]) in units of 2^-24 * ref_abs."""
    got = got.detach().double().cpu()
    ref, ref_abs = ref.detach().double().cpu(), ref_abs.detach().double().cpu()
    assert got.shape == ref.shape, (what, tuple(got.shape), tuple(ref.shape))
    K = K.double().reshape(-1, *([1] * (ref.dim() - 1)))
    err = (got - ref).abs()
    tol = K * U * ref_abs + TINY
    bad = ~(err <= tol)                                      # NaN fails too
    if bool(bad.any()):
        i = int(torch.nonzero(bad.reshape(-1))[0])
        row = i // (ref[0].numel() if ref.dim() > 1 else 1)
        raise AssertionError("%s: %d of %d entries off by more than K_i*2^-24*ref_abs; first in row %d (K=%d): got %r, "
                             "ref %r, ref_abs %r" % (what, int(bad.sum()), bad.numel(), row, int(K.reshape(-1)[row]),
                                                     float(got.reshape(-1)[i]), float(ref.reshape(-1)[i]),
                                                     float(ref_abs.reshape(-1)[i])))


def _same_bits(a, b, what):
    a, b = a.detach(), b.detach()
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    if not torch.equal(a, b):
        d = (a != b).reshape(a.shape[0], -1).any(1).nonzero()
        raise AssertionError("%s: %d rows differ bitwise, first row %d" % (what, d.numel(), int(d[0])))


def _nan(*shape):
    return torch.full(shape, float("nan"), device=DEV)


def _k_rows(L, self_term=True, two_level=False):
    """Summation-order budget of each row (module docstring), before C_FIN."""
    L = torch.as_tensor(L, dtype=torch.int64)
    nseg = (L + SEG - 1) // SEG
    K = torch.where(L <= HUB, L, SEG + nseg)
    if two_level:
        K = torch.where(nseg > 2 * GRP, SEG + GRP + (nseg + GRP - 1) // GRP, K)
    return K + (1 if self_term else 0) + C_FIN


def row_class(L):
    L = np.asarray(L)
    return np.select([L <= 1, L <= 3, L <= 5, L <= 7, L <= 11, L <= 16], [0, 1, 2, 3, 4, 5], 7)


def seg_sum(rowptr, X, idx, w=None, chunk=1 << 16):
    """out[r] = sum_{k in row r} X[idx[k]] * w[k]  (fp64; rowptr/idx numpy, X a double tensor)."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    n = len(rowptr) - 1
    rows = torch.repeat_interleave(torch.arange(n), torch.from_numpy(np.diff(rowptr)))
    idx = torch.from_numpy(np.asarray(idx, dtype=np.int64))
    out = torch.zeros(n, *X.shape[1:], dtype=torch.float64)
    for k0 in range(0, len(idx), chunk):
        v = X[idx[k0:k0 + chunk]]
        if w is not None:
            v = v * w[k0:k0 + chunk].reshape(-1, *([1] * (X.dim() - 1)))
        out.index_add_(0, rows[k0:k0 + chunk], v)
    return out


def _nwarps(sms):
    return sms * AG_CTAS * AG_WARPS


# ------------------------------------------------------------------------------------------ synthetic CSRs
class Csr:
    """Host (numpy int32) and device copies of a CSR, with its row lengths."""

    def __init__(self, rowptr, col):
        self.rowptr_np = np.ascontiguousarray(rowptr, dtype=np.int32)
        self.col_np = np.ascontiguousarray(col, dtype=np.int32)
        self.n = len(rowptr) - 1
        self.E = int(rowptr[-1])
        self.L = np.diff(self.rowptr_np.astype(np.int64))
        self.rowptr = torch.from_numpy(self.rowptr_np).to(DEV)
        self.col = torch.from_numpy(self.col_np).to(DEV)


def gen_lengths(sms, rng, n_short=None):
    """Row lengths: every length 0..40, 63-65, 127-129, the hub lengths of SPECIAL, a bulk of short rows
    (62 % of one entry) and enough rows of 17..160 entries that the hub segments outnumber the
    persistent warps more than twice; shuffled, so that the length classes interleave."""
    nw = _nwarps(sms)
    n_short = 3 * nw * 4 if n_short is None else n_short          # > 2 passes of four rows per warp
    short = np.where(rng.random(n_short) < 0.62, 1, rng.integers(0, HUB + 1, n_short))
    segs = sum(-(-L // SEG) for L in SPECIAL if L > HUB)
    mid = []
    while segs <= 2.5 * nw:
        L = int(rng.integers(HUB + 1, 161))
        mid.append(L)
        segs += -(-L // SEG)
    lengths = np.concatenate([short, np.array(SPECIAL), np.array(mid, dtype=np.int64)])
    rng.shuffle(lengths)
    return lengths


def gen_csr(lengths, rng, n_cols=None):
    """Random entries; duplicate entries and rows that list themselves included."""
    n = len(lengths)
    n_cols = n if n_cols is None else n_cols
    rowptr = np.zeros(n + 1, dtype=np.int64)
    rowptr[1:] = np.cumsum(lengths)
    col = rng.integers(0, n_cols, int(rowptr[-1]))
    multi = np.nonzero(lengths >= 2)[0]
    dup = rng.choice(multi, len(multi) // 10, replace=False)
    col[rowptr[dup] + 1] = col[rowptr[dup]]                            # a duplicate entry
    one = np.nonzero(lengths >= 1)[0]
    me = rng.choice(one, len(one) // 20, replace=False)
    col[rowptr[me] + rng.integers(0, lengths[me])] = me % n_cols       # the row itself
    return Csr(rowptr, col)


def sym_csr(sms, rng):
    """A symmetric CSR (undirected multigraph, self loops once): hubs of 513..20000 neighbours at random
    row ids, a bulk with mostly one neighbour, duplicate edges."""
    n = 3 * _nwarps(sms) * 4
    perm = rng.permutation(n)
    hubs = perm[:8]
    a, b = [], []
    for hnode, d in zip(hubs, [17, 33, 64, 513, 1024, 1025, 5000, 20000]):
        a.append(np.full(d, hnode)); b.append(rng.choice(perm[8:], d))
    bulk = perm[8:]
    m = len(bulk) // 2
    a.append(bulk[:m]); b.append(bulk[m:2 * m])                       # one neighbour each
    x = rng.choice(bulk, n // 4); y = rng.choice(bulk, n // 4)
    a.append(x); b.append(y)
    a.append(x[:200]); b.append(y[:200])                              # duplicate edges
    a = np.concatenate(a); b = np.concatenate(b)
    loops = rng.choice(bulk, 300, replace=False)
    keep = a != b
    src = np.concatenate([a[keep], b[keep], loops]); dst = np.concatenate([b[keep], a[keep], loops])
    order = rng.permutation(len(src))
    src, dst = src[order], dst[order]
    order = np.argsort(src, kind="stable")
    rowptr = np.zeros(n + 1, dtype=np.int64)
    rowptr[1:] = np.cumsum(np.bincount(src, minlength=n))
    return Csr(rowptr, dst[order])


# ------------------------------------------------------------------------------------------ device wrappers
def _ops():
    from npi_gnn_b200 import _lib, ops
    _lib.load()
    return ops


def new_queue(csr, fill=0, n_dev=None, gid=None, dist=None, keep=None, e_max=None):
    """hub queue + row order of a CSR; ``fill`` is the byte the queue's memory holds before the build."""
    ops = _ops()
    e_max = csr.E if e_max is None else e_max
    q = torch.full((ops.hub_rows_bytes(e_max),), fill, dtype=torch.uint8, device=DEV)
    ro = torch.zeros((csr.n, 4), dtype=torch.int32, device=DEV)      # unlisted records would read as an in-bounds empty row
    ops.hub_rows_build(csr.rowptr, n_dev, csr.n, e_max, q, gid=gid, dist=dist, row_order=ro, keep=keep)
    return q, ro


def fwd(csr, lay, relu, pool, pipelined, q=None, ro=None, n_dev=None, bias=True):
    """One forward aggregation into NaN-filled h/z/s; ``pool``: None, 'zs', 'z' or 's'."""
    ops = _ops()
    if q is None:
        q, ro = new_queue(csr, n_dev=n_dev, gid=lay.get("gid"), dist=lay.get("dist"))
    h, z, s = _nan(csr.n, H), _nan(csr.n), _nan(csr.n)
    ops.sage_aggregate_fwd(lay["Y"], lay.get("gid"), lay.get("dist"), lay.get("w0"), csr.rowptr, csr.col, n_dev, csr.n,
                           lay["b"] if bias else None, relu, lay["p"] if pool else None, h,
                           z if pool in ("zs", "z", None) else None, s if pool in ("zs", "s", None) else None,
                           hubq=q, packed=lay.get("packed"), row_order=ro, pipelined=pipelined)
    return h, z, s


def bwd(csr, dpre, new_id, pipelined, q=None, ro=None):
    ops = _ops()
    if q is None:
        q, ro = new_queue(csr)
    packed = None
    if pipelined:
        packed = ops.entry_pack_sel(csr.rowptr, csr.col, new_id, None, csr.n,
                                    torch.empty((max(csr.E, 1), 2), dtype=torch.int32, device=DEV))
    dxa = _nan(csr.n, H)
    ops.sage_aggregate_bwd(dpre, new_id, csr.rowptr, csr.col, None, csr.n, dxa, hubq=q, packed=packed,
                           row_order=ro if pipelined else None)
    return dxa


# ------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def sms():
    return _ops().sm_count()


@pytest.fixture(scope="module")
def graph(sms):
    """The forward / backward CSR (square: entries index rows) with its layers and fp64 sums."""
    rng = np.random.default_rng(11)
    csr = gen_csr(gen_lengths(sms, rng), rng)
    assert csr.E < 2 ** 31 and (csr.L > HUB).sum() > 0
    g = torch.Generator().manual_seed(5)
    n = csr.n
    b = torch.randn(H, generator=g) * 0.1
    p = torch.randn(H, generator=g)
    # non-virtual layer: y_j = Y[j]
    Y = torch.randn(n, H, generator=g)
    # virtual layer: y_j = T[gid_j] + dist_j * w0 over a table whose unreferenced rows are NaN
    V = n // 2
    used = rng.choice(V, V // 2, replace=False)
    gid = used[rng.integers(0, len(used), n)].astype(np.int32)
    dist = rng.integers(0, 8, n).astype(np.uint8)
    T = torch.randn(V, H, generator=g)
    T[torch.from_numpy(np.setdiff1d(np.arange(V), used))] = float("nan")
    w0 = torch.randn(H, generator=g)
    ops = _ops()
    layers = {}
    Yd = Y.double()
    S = seg_sum(csr.rowptr_np, Yd, csr.col_np) + Yd
    Sa = seg_sum(csr.rowptr_np, Yd.abs(), csr.col_np) + Yd.abs()
    layers["plain"] = dict(Y=Y.to(DEV), b=b.to(DEV), p=p.to(DEV), S=S, Sa=Sa)
    Td = T.double()
    gcol = gid[csr.col_np]
    ds = seg_sum(csr.rowptr_np, torch.from_numpy(dist.astype(np.float64))[:, None], csr.col_np)[:, 0] + torch.from_numpy(
        dist.astype(np.float64))
    S = seg_sum(csr.rowptr_np, Td, gcol) + Td[torch.from_numpy(gid).long()] + ds[:, None] * w0.double()
    Sa = seg_sum(csr.rowptr_np, Td.abs(), gcol) + Td.abs()[torch.from_numpy(gid).long()] + ds[:, None] * w0.double().abs()
    gid_d = torch.from_numpy(gid).to(DEV)
    dist_d = torch.from_numpy(dist).to(DEV)
    packed = ops.entry_pack_virt(csr.rowptr, csr.col, gid_d, dist_d, None, n, V, torch.empty(csr.E, dtype=torch.int32, device=DEV))
    layers["virtual"] = dict(Y=T.to(DEV), gid=gid_d, dist=dist_d, w0=w0.to(DEV), packed=packed, b=b.to(DEV), p=p.to(DEV),
                             S=S, Sa=Sa)
    return csr, layers


def fwd_ref(csr, lay, relu, bias=True):
    """fp64 h, h on absolute values, and the per-row budget."""
    dv = torch.from_numpy(csr.L + 1).double()[:, None]
    b = lay["b"].double().cpu() if bias else torch.zeros(H, dtype=torch.float64)
    h = lay["S"] / dv + b
    ha = lay["Sa"] / dv + b.abs()
    if relu:
        h = h.clamp_min(0)
    return h, ha, _k_rows(csr.L)


def check_fwd(csr, lay, relu, pool, got, rows, what):
    """rows: the rows that must have been written (the others must still be NaN, bit for bit)."""
    h, z, s = got
    href, ha, K = fwd_ref(csr, lay, relu)
    r = torch.as_tensor(rows)
    _check(h.cpu()[r], href[r], ha[r], K[r], what + " h")
    untouched = torch.ones(csr.n, dtype=torch.bool)
    untouched[r] = False
    _same_bits(h.cpu()[untouched], _nan(int(untouched.sum()), H).cpu(), what + " h rows that must stay untouched")
    p = lay["p"].double().cpu()
    zref = href @ p / p.norm()
    za = ha @ p.abs() / p.norm()
    Kz = K + 24                                                         # the 128-wide dot and the norm
    if pool in ("zs", "z"):
        _check(z.cpu()[r], zref[r], za[r], Kz[r], what + " z")
    if pool in ("zs", "s"):
        sref = torch.tanh(zref)
        # |d tanh| <= |dz|, plus tanhf's own rounding (<= 2 ulp): a budget on za + |s|
        _check(s.cpu()[r], sref[r], za[r] + sref[r].abs() * 4 / Kz[r].double(), Kz[r], what + " s")
    for name, t in (("z", z), ("s", s)):
        if pool is None or (pool != "zs" and pool != name):
            _same_bits(t, _nan(csr.n), what + " %s must not be written" % name)
        else:
            _same_bits(t.cpu()[untouched], _nan(int(untouched.sum())).cpu(), what + " %s rows that must stay untouched" % name)


# ------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("pool", [None, "zs", "z", "s"])
@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("layer", ["plain", "virtual"])
def test_aggregate_fwd_vs_fp64(graph, layer, relu, pool):
    csr, layers = graph
    lay = layers[layer]
    outs = []
    for pipe in (False, True):
        got = fwd(csr, lay, relu, pool, pipe)
        check_fwd(csr, lay, relu, pool, got, np.arange(csr.n), "%s fwd (%s)" % (layer, "pipelined" if pipe else "plain"))
        outs.append(got)
    for name, a, b in zip("hzs", outs[0], outs[1]):
        _same_bits(a, b, "%s fwd: plain vs pipelined %s" % (layer, name))


@pytest.mark.parametrize("layer", ["plain", "virtual"])
def test_aggregate_fwd_n_dev_below_n_host(graph, layer):
    """n_dev < n_host: rows n_dev.. stay untouched (the queue is built with the same device count)."""
    csr, layers = graph
    lay = layers[layer]
    n = csr.n - 1237
    n_dev = torch.tensor([n], dtype=torch.int32, device=DEV)
    outs = []
    for pipe in (False, True):
        q, ro = new_queue(csr, n_dev=n_dev, gid=lay.get("gid"), dist=lay.get("dist"))
        got = fwd(csr, lay, 1, "zs", pipe, q=q, ro=ro, n_dev=n_dev)
        check_fwd(csr, lay, 1, "zs", got, np.arange(n), "%s fwd n_dev (%s)" % (layer, pipe))
        outs.append(got)
    for name, a, b in zip("hzs", outs[0], outs[1]):
        _same_bits(a, b, "plain vs pipelined %s" % name)


def test_aggregate_fwd_keep_representatives(graph):
    """keep: the pipelined kernel evaluates only rows with keep[i] == i and leaves every other row of h/z/s untouched."""
    csr, layers = graph
    lay = layers["virtual"]
    rng = np.random.default_rng(3)
    keep = np.arange(csr.n, dtype=np.int32)
    drop = rng.random(csr.n) < 0.5
    drop[0] = False
    keep[drop] = rng.integers(0, np.maximum(np.nonzero(drop)[0], 1))       # some earlier row
    q, ro = new_queue(csr, gid=lay["gid"], dist=lay["dist"], keep=torch.from_numpy(keep).to(DEV))
    got = fwd(csr, lay, 0, "zs", True, q=q, ro=ro)
    check_fwd(csr, lay, 0, "zs", got, np.nonzero(~drop)[0], "fwd keep")


# ------------------------------------------------------------------------------------------ backward
def make_sel(n, mode, rng):
    """new_id (None = identity), N'."""
    if mode == "identity":
        return None, n
    if mode == "none":
        return torch.full((n,), -1, dtype=torch.int32), 0
    kept = np.nonzero(rng.random(n) < 0.5)[0]
    nid = np.full(n, -1, dtype=np.int32)
    nid[kept] = rng.permutation(len(kept))
    return torch.from_numpy(nid), len(kept)


def bwd_ref(csr, dpre, new_id):
    """dxa_j = sum_{i in row(j) U {j}, new_id[i] >= 0} dpre[new_id[i]] / (deg_i+1), and on absolute values."""
    n = csr.n
    nid = np.arange(n) if new_id is None else new_id.numpy()
    D = dpre.double().cpu()
    Dz = torch.cat([D, torch.zeros(1, H, dtype=torch.float64)])          # row -1: dropped
    idx = np.where(nid >= 0, nid, len(D))
    inv = torch.from_numpy(1.0 / (csr.L + 1.0))[:, None]
    out = []
    for X in (Dz, Dz.abs()):
        P = X[torch.from_numpy(idx)] * inv                              # what row i contributes wherever it is listed
        out.append(seg_sum(csr.rowptr_np, P, csr.col_np) + P)
    return out[0], out[1], _k_rows(csr.L)


@pytest.mark.parametrize("mode", ["identity", "half", "none"])
def test_aggregate_bwd_vs_fp64(graph, mode):
    csr, _ = graph
    rng = np.random.default_rng(17)
    new_id, Np = make_sel(csr.n, mode, rng)
    dpre = torch.randn(Np + 1, H, generator=torch.Generator().manual_seed(8))
    dpre[Np] = float("nan")                                             # just past N': never read
    ref, refa, K = bwd_ref(csr, dpre[:Np], new_id)
    nid_d = None if new_id is None else new_id.to(DEV)
    outs = []
    for pipe in (False, True):
        dxa = bwd(csr, dpre.to(DEV), nid_d, pipe)
        _check(dxa, ref, refa, K, "bwd %s (%s)" % (mode, "pipelined" if pipe else "plain"))
        outs.append(dxa)
    _same_bits(outs[0], outs[1], "bwd %s: plain vs pipelined" % mode)


@pytest.mark.parametrize("mode", ["identity", "half"])
def test_aggregate_bwd_is_adjoint_of_mean(sms, mode):
    """On a symmetric CSR the backward is the adjoint of the forward mean (no bias, no ReLU) under the selection:
    dxa == d/dY sum_{i : new_id[i] >= 0} <mean_i(Y), dpre[new_id[i]]>, by fp64 autograd."""
    rng = np.random.default_rng(23)
    csr = sym_csr(sms, rng)
    new_id, Np = make_sel(csr.n, mode, rng)
    g = torch.Generator().manual_seed(4)
    dpre = torch.randn(Np + 1, H, generator=g)
    dpre[Np] = float("nan")
    nid = np.arange(csr.n) if new_id is None else new_id.numpy()
    sel = torch.from_numpy(np.nonzero(nid >= 0)[0])
    grads = []
    for f in (lambda t: t, torch.abs):
        Y = torch.zeros(csr.n, H, dtype=torch.float64, requires_grad=True)
        mean = (seg_sum(csr.rowptr_np, Y, csr.col_np) + Y) / torch.from_numpy(csr.L + 1.0)[:, None]
        loss = (mean[sel] * f(dpre[:Np].double())[torch.from_numpy(nid[sel.numpy()]).long()]).sum()
        loss.backward()
        grads.append(Y.grad)
    nid_d = None if new_id is None else new_id.to(DEV)
    for pipe in (False, True):
        dxa = bwd(csr, dpre.to(DEV), nid_d, pipe)
        _check(dxa, grads[0], grads[1], _k_rows(csr.L), "adjoint %s (%s)" % (mode, pipe))


# ------------------------------------------------------------------------------------------ gather
@pytest.fixture(scope="module")
def gather_case(sms):
    """csr_gather_sum input: packed {row, weight} entries, some with a negative row; rows of 0..16 segments
    (single level), 17, 18, 24, 25 and several hundred segments (two-level, full and partial last groups)."""
    rng = np.random.default_rng(29)
    nw = _nwarps(sms)
    lens = list(range(0, 41)) + [SEG * k + d for k in range(1, 17) for d in (-1, 0, 1)]
    lens += [SEG * 16 + 1, SEG * 17, SEG * 17 + 1, SEG * 24, SEG * 24 + 1, SEG * 25, SEG * 300, SEG * 301 - 7]
    segs = sum(-(-L // SEG) for L in lens)
    while segs <= 2.5 * nw:
        ns = int(rng.integers(17, 400))
        L = ns * SEG - int(rng.integers(0, SEG))
        lens.append(L)
        segs += ns
    short = np.where(rng.random(3 * nw * 4) < 0.62, 1, rng.integers(0, HUB + 1, 3 * nw * 4))
    lengths = np.concatenate([np.array(lens), short])
    rng.shuffle(lengths)
    n_src = 50000
    nan_rows = rng.choice(n_src, n_src // 10, replace=False)
    ok_rows = np.setdiff1d(np.arange(n_src), nan_rows)
    csr = gen_csr(lengths, rng, n_cols=1)
    E = csr.E
    ids = ok_rows[rng.integers(0, len(ok_rows), E)]
    skip = rng.random(E) < 0.1
    ids[skip] = -1 - nan_rows[rng.integers(0, len(nan_rows), int(skip.sum()))]     # rows with a NaN source row
    w = (rng.uniform(0.25, 2.0, E) * rng.choice([-1.0, 1.0], E)).astype(np.float32)
    packed = np.stack([ids.astype(np.int32), w.view(np.int32)], 1)
    src = torch.randn(n_src, H, generator=torch.Generator().manual_seed(6))
    src[torch.from_numpy(nan_rows)] = float("nan")
    srcz = torch.cat([src.double(), torch.zeros(1, H, dtype=torch.float64)])
    idx = np.where(ids >= 0, ids, n_src)
    wt = torch.from_numpy(w.astype(np.float64))
    ref = seg_sum(csr.rowptr_np, srcz, idx, wt)
    refa = seg_sum(csr.rowptr_np, srcz.abs(), idx, wt.abs())
    return csr, torch.from_numpy(packed).to(DEV), src.to(DEV), ref, refa, _k_rows(csr.L, self_term=False, two_level=True)


def gather(csr, packed, src, q, ro):
    out = _nan(csr.n, H)
    _ops().csr_gather_sum(src, csr.rowptr, packed, csr.n, out, q, ro)
    return out


def test_csr_gather_sum_vs_fp64(gather_case):
    csr, packed, src, ref, refa, K = gather_case
    nseg = -(-csr.L // SEG)
    assert {17, 18, 24, 25, 300, 301} <= set(nseg.tolist())
    q, ro = new_queue(csr)
    out = gather(csr, packed, src, q, ro)
    _check(out, ref, refa, K, "csr_gather_sum")


# ------------------------------------------------------------------------------------------ queue contents
def read_queue(q):
    """header, seg_row and seg_base of the listed segments (layout of csrc/hub.cuh)."""
    qi = q.view(torch.int32).cpu().numpy()
    hdr = qi[:32].copy()
    cap, nsegs = int(hdr[1]), min(int(hdr[0]), int(hdr[1]))
    return hdr, qi[32:32 + nsegs].copy(), qi[32 + cap:32 + cap + nsegs].copy()


def hub_cap(e):
    return (e // SEG + e // (HUB + 1) + 8 + 3) & ~3


def check_queue(csr, q, ro, listed, self_payload, what):
    """The queue and row order of the rows in ``listed`` (bool [n]) against their definitions, exactly."""
    hdr, seg_row, seg_base = read_queue(q)
    L = csr.L
    cls = row_class(L)
    hubrow = listed & (L > HUB)
    nseg = -(-L // SEG)
    assert hdr[0] == int(nseg[hubrow].sum()), (what, "segments listed", int(hdr[0]), int(nseg[hubrow].sum()))
    assert hdr[0] <= hdr[1], (what, "segments beyond capacity")
    assert list(hdr[4:12]) == list(np.bincount(cls[listed], minlength=8)), (what, "class totals", list(hdr[4:12]))
    # every hub row owns nseg consecutive slots, and seg_base of each is the row's first slot
    slots = {}
    for s, r in enumerate(seg_row.tolist()):
        slots.setdefault(r, []).append(s)
    assert sorted(slots) == np.nonzero(hubrow)[0].tolist(), (what, "hub rows listed")
    for r, sl in slots.items():
        b = sl[0]
        assert sl == list(range(b, b + int(nseg[r]))), (what, "row %d of %d segments owns slots %s.." % (r, nseg[r], sl[:4]))
        assert (seg_base[sl] == b).all(), (what, "seg_base of row %d" % r)
    if ro is None:
        return hdr
    # row order: the non-hub listed rows, classes ascending, records {row, beg, end, self payload}
    short = listed & (L <= HUB)
    rec = ro.cpu().numpy()[:int(short.sum())]
    assert np.array_equal(np.sort(rec[:, 0]), np.nonzero(short)[0]), (what, "row order is not a permutation of the short rows")
    assert (np.diff(cls[rec[:, 0]]) >= 0).all(), (what, "classes not ascending")
    r = rec[:, 0]
    assert np.array_equal(rec[:, 1], csr.rowptr_np[r]) and np.array_equal(rec[:, 2], csr.rowptr_np[r + 1]), (what, "extents")
    assert np.array_equal(rec[:, 3], self_payload[r]), (what, "self payload")
    return hdr


@pytest.mark.parametrize("keep", [False, True])
@pytest.mark.parametrize("layer", ["plain", "virtual"])
def test_hub_rows_build_contents(graph, layer, keep):
    csr, layers = graph
    lay = layers[layer]
    listed = np.ones(csr.n, dtype=bool)
    keep_d = None
    if keep:
        rng = np.random.default_rng(41)
        kp = np.arange(csr.n, dtype=np.int32)
        drop = rng.random(csr.n) < 0.4
        drop[0] = False
        kp[drop] = 0
        listed = ~drop
        keep_d = torch.from_numpy(kp).to(DEV)
    if layer == "virtual":
        payload = lay["gid"].cpu().numpy() | (lay["dist"].cpu().numpy().astype(np.int32) << 29)
    else:
        payload = np.arange(csr.n, dtype=np.int32)
    q, ro = new_queue(csr, gid=lay.get("gid"), dist=lay.get("dist"), keep=keep_d, fill=0xAB)
    hdr = check_queue(csr, q, ro, listed, payload, "hub_rows_build %s keep=%s" % (layer, keep))
    assert hdr[1] == hub_cap(csr.E)
    assert hdr[4 + 6] == 0                         # whole-warp rows: none at the shipped 16-entry hub threshold


def test_hub_queue_capacity_worst_case():
    """Every row of 33 entries (two segments per 33 entries: the most segments per entry) at e_max = E."""
    n = 20000
    rowptr = np.arange(n + 1, dtype=np.int64) * 33
    csr = Csr(rowptr, np.zeros(int(rowptr[-1]), dtype=np.int32))
    q, ro = new_queue(csr)
    hdr = read_queue(q)[0]
    assert hdr[0] == 2 * n and hdr[0] <= hdr[1] == hub_cap(csr.E)
    check_queue(csr, q, ro, np.ones(n, dtype=bool), np.arange(n, dtype=np.int32), "capacity")


# ------------------------------------------------------------------------------------------ second producer
def test_filter_adj_queue_matches_hub_rows_build(graph):
    """filter_adj lists the hub queue and row order of its output CSR on the way: same header, same segments per
    row, same row records as hub_rows_build of the finished CSR, and the aggregations over either queue agree bit for bit."""
    ops = _ops()
    csr, layers = graph
    rng = np.random.default_rng(43)
    kept = np.nonzero(rng.random(csr.n) < 0.7)[0]
    perm = rng.permutation(kept).astype(np.int32)
    new_id = np.full(csr.n, -1, dtype=np.int32)
    new_id[perm] = np.arange(len(perm), dtype=np.int32)
    Np = len(perm)
    rp_out = torch.empty(Np + 1, dtype=torch.int32, device=DEV)
    col_out = torch.empty(csr.E, dtype=torch.int32, device=DEV)
    qa = torch.full((ops.hub_rows_bytes(csr.E),), 0xFF, dtype=torch.uint8, device=DEV)
    roa = torch.zeros((Np, 4), dtype=torch.int32, device=DEV)
    ops.hub_rows_reset(qa)
    ws = torch.empty(ops.filter_adj_workspace_bytes(Np), dtype=torch.uint8, device=DEV)
    ops.filter_adj(csr.rowptr, csr.col, torch.from_numpy(perm).to(DEV), torch.from_numpy(new_id).to(DEV), None, Np,
                   rp_out, col_out, ws, hubq=qa, hub_e_max=csr.E, row_order=roa)
    # the output CSR on the host, from its definition
    rows = [csr.col_np[csr.rowptr_np[p]:csr.rowptr_np[p + 1]] for p in perm]
    rows = [new_id[r][new_id[r] >= 0] for r in rows]
    rp = np.zeros(Np + 1, dtype=np.int64)
    rp[1:] = np.cumsum([len(r) for r in rows])
    out = Csr(rp, np.concatenate(rows))
    assert np.array_equal(rp_out.cpu().numpy(), out.rowptr_np) and np.array_equal(col_out[:out.E].cpu().numpy(), out.col_np)
    assert (out.L > 40 * SEG).any()
    out.rowptr, out.col = rp_out, col_out[:out.E]
    hdr_a = check_queue(out, qa, roa, np.ones(Np, dtype=bool), np.arange(Np, dtype=np.int32), "filter_adj queue")
    qb, rob = new_queue(out, e_max=csr.E)
    hdr_b = check_queue(out, qb, rob, np.ones(Np, dtype=bool), np.arange(Np, dtype=np.int32), "hub_rows_build queue")
    assert list(hdr_a) == list(hdr_b)
    g = torch.Generator().manual_seed(12)
    lay = dict(Y=torch.randn(Np, H, generator=g).to(DEV), b=torch.randn(H, generator=g).to(DEV),
               p=torch.randn(H, generator=g).to(DEV))
    dpre = torch.randn(Np, H, generator=g).to(DEV)
    nid = torch.from_numpy(np.where(rng.random(Np) < 0.5, np.arange(Np), -1).astype(np.int32)).to(DEV)
    res = []
    for q, ro in ((qa, roa), (qb, rob)):
        res.append(fwd(out, lay, 1, "zs", True, q=q, ro=ro) + (bwd(out, dpre, nid, True, q=q, ro=ro),))
    for name, a, b in zip(["h", "z", "s", "dxa"], res[0], res[1]):
        _same_bits(a, b, "aggregation over the filter_adj vs hub_rows_build queue: %s" % name)


# ------------------------------------------------------------------------------------------ queue life cycle
def test_queue_reuse_is_bit_identical(graph, gather_case):
    """Two launches on one queue (the second into fresh NaN-filled outputs: a row the second launch fails to write
    shows), then forward / backward / forward on one queue, then the queue rebuilt for a CSR of another layout."""
    csr, layers = graph
    lay = layers["virtual"]
    q, ro = new_queue(csr, gid=lay["gid"], dist=lay["dist"])
    f1 = fwd(csr, lay, 1, "zs", True, q=q, ro=ro)
    f2 = fwd(csr, lay, 1, "zs", True, q=q, ro=ro)
    for name, a, b in zip("hzs", f1, f2):
        _same_bits(a, b, "fwd twice on one queue: %s" % name)
    dpre = torch.randn(csr.n, H, generator=torch.Generator().manual_seed(1)).to(DEV)
    q2, ro2 = new_queue(csr)
    b1 = bwd(csr, dpre, None, True, q=q2, ro=ro2)
    b2 = bwd(csr, dpre, None, True, q=q2, ro=ro2)
    _same_bits(b1, b2, "bwd twice on one queue")
    # forward, backward, forward on the queue of the non-virtual layer
    pl = layers["plain"]
    f3 = fwd(csr, pl, 0, "zs", True, q=q2, ro=ro2)
    b3 = bwd(csr, dpre, None, True, q=q2, ro=ro2)
    f4 = fwd(csr, pl, 0, "zs", True, q=q2, ro=ro2)
    for name, a, b in zip("hzs", f3, f4):
        _same_bits(a, b, "fwd / bwd / fwd on one queue: %s" % name)
    _same_bits(b1, b3, "bwd after a forward on its queue")
    # gather twice on one queue (two-level counters)
    gcsr, packed, src, *_ = gather_case
    gq, gro = new_queue(gcsr)
    g1 = gather(gcsr, packed, src, gq, gro)
    g2 = gather(gcsr, packed, src, gq, gro)
    _same_bits(g1, g2, "gather twice on one queue")
    # one buffer rebuilt for CSRs of different layouts, back and forth: results of a fresh queue
    ops = _ops()
    buf = torch.zeros(max(q.numel(), gq.numel()), dtype=torch.uint8, device=DEV)
    for _ in range(2):
        ops.hub_rows_build(csr.rowptr, None, csr.n, csr.E, buf, gid=lay["gid"], dist=lay["dist"], row_order=ro)
        for name, a, b in zip("hzs", f1, fwd(csr, lay, 1, "zs", True, q=buf, ro=ro)):
            _same_bits(a, b, "fwd on a rebuilt queue: %s" % name)
        ops.hub_rows_build(gcsr.rowptr, None, gcsr.n, gcsr.E, buf, row_order=gro)
        _same_bits(g1, gather(gcsr, packed, src, buf, gro), "gather on a rebuilt queue")


def test_queue_in_unzeroed_memory(graph, gather_case):
    """A queue whose memory holds 0xFF bytes before hub_rows_build gives the results of a zeroed one, for all three
    kernels (the two-level combine of the gather counts groups in arrival slots behind the row's own)."""
    csr, layers = graph
    lay = layers["virtual"]
    dpre = torch.randn(csr.n, H, generator=torch.Generator().manual_seed(2)).to(DEV)
    res = {}
    for fill in (0, 0xFF):
        q, ro = new_queue(csr, fill=fill, gid=lay["gid"], dist=lay["dist"])
        h, z, s = fwd(csr, lay, 1, "zs", True, q=q, ro=ro)
        q, ro = new_queue(csr, fill=fill)
        dxa = bwd(csr, dpre, None, True, q=q, ro=ro)
        gcsr, packed, src, *_ = gather_case
        q, ro = new_queue(gcsr, fill=fill)
        res[fill] = dict(h=h, z=z, s=s, dxa=dxa, gather=gather(gcsr, packed, src, q, ro))
    for k in ("h", "z", "s", "dxa", "gather"):
        _same_bits(res[0][k], res[0xFF][k], "queue in 0xFF memory: %s" % k)


# ------------------------------------------------------------------------------------------ independence of rows
def test_rows_are_independent_of_their_numbering(graph):
    """Renumbering the rows of a CSR (entries relabelled, order inside a row kept) permutes the outputs bit for bit:
    every row is summed in its own CSR order whatever warp or slot it lands in."""
    csr, layers = graph
    lay = layers["plain"]
    rng = np.random.default_rng(47)
    pi = rng.permutation(csr.n)                          # old row i -> new row pi[i]
    inv = np.argsort(pi)
    rows = [pi[csr.col_np[csr.rowptr_np[i]:csr.rowptr_np[i + 1]]] for i in inv]
    rp = np.zeros(csr.n + 1, dtype=np.int64)
    rp[1:] = np.cumsum(csr.L[inv])
    pc = Csr(rp, np.concatenate(rows))
    inv_t, pi_t = torch.from_numpy(inv).to(DEV), torch.from_numpy(pi).to(DEV)
    play = dict(lay, Y=lay["Y"][inv_t])
    dpre = torch.randn(csr.n, H, generator=torch.Generator().manual_seed(3)).to(DEV)
    for pipe in (False, True):
        a = fwd(csr, lay, 1, "zs", pipe)
        b = fwd(pc, play, 1, "zs", pipe)
        for name, x, y in zip("hzs", a, b):
            _same_bits(x, y[pi_t], "renumbered rows, fwd %s (%s)" % (name, pipe))
        _same_bits(bwd(csr, dpre, None, pipe), bwd(pc, dpre[inv_t], None, pipe)[pi_t], "renumbered rows, bwd (%s)" % pipe)


# ------------------------------------------------------------------------------------------ argument checks
def test_argument_checks(graph):
    from npi_gnn_b200._lib import NPIError
    ops = _ops()
    csr, layers = graph
    lay = layers["virtual"]
    q, ro = new_queue(csr, gid=lay["gid"], dist=lay["dist"])
    h = _nan(csr.n, H)
    with pytest.raises(NPIError):                      # pipelined without row_order
        ops.sage_aggregate_fwd(lay["Y"], lay["gid"], lay["dist"], lay["w0"], csr.rowptr, csr.col, None, csr.n, None, 0, None,
                               h, None, None, hubq=q, packed=lay["packed"], row_order=None, pipelined=True)
    with pytest.raises(NPIError):                      # gid without dist
        ops.sage_aggregate_fwd(lay["Y"], lay["gid"], None, lay["w0"], csr.rowptr, csr.col, None, csr.n, None, 0, None,
                               h, None, None, hubq=q)
    with pytest.raises(NPIError):
        ops.sage_aggregate_bwd(h, None, csr.rowptr, csr.col, None, csr.n, h, hubq=q,
                               packed=torch.empty((csr.E, 2), dtype=torch.int32, device=DEV), row_order=None)
    # misaligned row order / packed entries
    ro_bad = torch.empty(csr.n * 4 + 1, dtype=torch.int32, device=DEV)[1:].view(csr.n, 4)
    sel_bad = torch.empty(2 * csr.E + 1, dtype=torch.int32, device=DEV)[1:].view(csr.E, 2)
    sel_ok = torch.empty((csr.E, 2), dtype=torch.int32, device=DEV)
    with pytest.raises(NPIError):
        ops.hub_rows_build(csr.rowptr, None, csr.n, csr.E, torch.empty_like(q), row_order=ro_bad)
    with pytest.raises(NPIError):
        ops.sage_aggregate_fwd(lay["Y"], lay["gid"], lay["dist"], lay["w0"], csr.rowptr, csr.col, None, csr.n, None, 0, None,
                               h, None, None, hubq=q, packed=lay["packed"], row_order=ro_bad, pipelined=True)
    with pytest.raises(NPIError):
        ops.sage_aggregate_bwd(h, None, csr.rowptr, csr.col, None, csr.n, h, hubq=q, packed=sel_bad, row_order=ro)
    with pytest.raises(NPIError):
        ops.sage_aggregate_bwd(h, None, csr.rowptr, csr.col, None, csr.n, h, hubq=q, packed=sel_ok, row_order=ro_bad)
    with pytest.raises(NPIError):
        ops.csr_gather_sum(h, csr.rowptr, sel_bad, csr.n, h, q, ro)
    with pytest.raises(NPIError):
        ops.csr_gather_sum(h, csr.rowptr, sel_ok, csr.n, h, q, ro_bad)
    with pytest.raises(NPIError):
        ops.entry_pack_sel(csr.rowptr, csr.col, None, None, csr.n, sel_bad)
    # a queue smaller than hub_rows_bytes(e_max)
    with pytest.raises(NPIError):
        ops.hub_rows_build(csr.rowptr, None, csr.n, csr.E, torch.empty(ops.hub_rows_bytes(csr.E) - 4, dtype=torch.uint8, device=DEV))
    # entry_pack_virt: graph ids must fit the 29-bit field (checked by value)
    tiny = torch.zeros(2, dtype=torch.int32, device=DEV)
    with pytest.raises(NPIError):
        ops.entry_pack_virt(tiny, tiny, tiny, torch.zeros(2, dtype=torch.uint8, device=DEV), None, 1, 2 ** 29, tiny)
    ops.entry_pack_virt(tiny, tiny, tiny, torch.zeros(2, dtype=torch.uint8, device=DEV), None, 1, 2 ** 29 - 1, tiny)
    torch.cuda.synchronize()
    # nothing above was launched into h
    assert bool(torch.isnan(h).all())
