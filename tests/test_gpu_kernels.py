"""Isolated parity tests of the kernels that dominate the step (VERDICT r01 "the dominant kernels have
no test of their own"): the tcgen05 projections npi_gemm_nn_tc / npi_gemm_tn_tc against an fp64
product over the edge shapes (M = 1, tile boundaries, fewer tiles than SMs, device-side M, both
operand orientations, every accepted K), and the by-serial occurrence lists / reduction of the
layer-1 weight gradient (npi_gid_index_build / npi_gid_reduce) against a sorted index_add in fp64.
Reference semantics: the `@ weight` of PyG-1.4.2 SAGEConv and its backward (src/classes.py:62,66,70;
SURVEY Appendix A.2)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# 3xTF32 error-compensated split: measured 1.7e-6 of max|C| (tools/tc_probe.py); the bar of the verdict
TC_REL = 4e-6


def _ref_nn(A, B, transB):
    Bm = B.double().t() if transB else B.double()
    return A.double() @ Bm


@pytest.mark.parametrize("transB", [0, 1])
@pytest.mark.parametrize("K", [32, 64, 96, 128])
@pytest.mark.parametrize("M", [1, 31, 127, 128, 129, 4097, 107579])
def test_gemm_nn_tc_vs_fp64(M, K, transB):
    from npi_gnn_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M * 7 + K + transB)
    A = torch.randn(M, K, device="cuda", generator=g)
    B = torch.randn((128, K) if transB else (K, 128), device="cuda", generator=g)
    C = torch.full((M + 3, 128), float("nan"), device="cuda")
    ops.gemm_nn_tc(A, None, M, K, B, bool(transB), C)
    torch.cuda.synchronize()
    R = _ref_nn(A, B, transB)
    assert torch.isnan(C[M:]).all()                              # rows past M are never written
    err = float((C[:M].double() - R).abs().max()) / float(R.abs().max())
    assert err <= TC_REL, err
    C2 = torch.empty(M, 128, device="cuda")
    ops.gemm_nn_tc(A, None, M, K, B, bool(transB), C2)
    torch.cuda.synchronize()
    assert torch.equal(C[:M], C2)                                # rerun bit-identical


@pytest.mark.parametrize("F,ld", [(178, 180), (65, 68), (150, 152), (192, 192), (5, 8)])
@pytest.mark.parametrize("M", [300, 5085])
def test_gemm_nn_tc_feature_table_widths(M, F, ld):
    """T = table . W1 of layer 1 (reference src/classes.py:62 on the virtual features): K = F is not a multiple of
    32, the row stride is ld = round_up(F, 4) and the padding columns hold GARBAGE here -- the tensor map's inner
    extent is K, so the TMA zero-fills everything past column K, and weight rows past K are taken as zero.
    K > 128 runs with one TMEM accumulator (2 x 192 weight columns + 128)."""
    from npi_gnn_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + F)
    table = torch.randn(M, ld, device="cuda", generator=g)
    table[:, F:] = float("nan") if F < ld else 0.0
    W = torch.randn(F, 128, device="cuda", generator=g)
    C = torch.full((M + 2, 128), float("nan"), device="cuda")
    ops.gemm_nn_tc(table, None, M, F, W, False, C)
    torch.cuda.synchronize()
    R = table[:, :F].double() @ W.double()
    assert torch.isnan(C[M:]).all()
    err = float((C[:M].double() - R).abs().max()) / float(R.abs().max())
    assert err <= TC_REL, err
    C2 = torch.empty(M, 128, device="cuda")
    ops.gemm_nn_tc(table, None, M, F, W, False, C2)
    torch.cuda.synchronize()
    assert torch.equal(C[:M], C2)


def test_gemm_nn_tc_device_side_m_and_strided_operand():
    """M read from device memory (what the captured step does) and an A operand that is a column slice
    of a wider, padded buffer (lda > K)."""
    from npi_gnn_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    Afull = torch.randn(5000, 192, device="cuda", generator=g)
    B = torch.randn(128, 128, device="cuda", generator=g)
    md = torch.tensor([3333], dtype=torch.int32, device="cuda")
    for K in (64, 128):
        A = Afull[:, :K]
        Bk = B[:K].contiguous()
        C = torch.full((5000, 128), float("nan"), device="cuda")
        ops.gemm_nn_tc(A, md, 5000, K, Bk, False, C)
        torch.cuda.synchronize()
        R = _ref_nn(A[:3333], Bk, 0)
        assert float((C[:3333].double() - R).abs().max()) / float(R.abs().max()) <= TC_REL
        assert torch.isnan(C[3333:]).all()


def test_gemm_nn_tc_structured_layout():
    """One-hot rows pick single rows of B: any swizzle / descriptor slip shows as an exact mismatch."""
    from npi_gnn_b200 import ops
    for K in (32, 128):
        M = 384
        A = torch.zeros(M, K, device="cuda")
        A[torch.arange(M), torch.arange(M) % K] = 1.0
        B = (torch.arange(K, device="cuda").float()[:, None] * 128 + torch.arange(128, device="cuda").float()[None, :]).contiguous()
        for transB in (0, 1):
            Bin = B.t().contiguous() if transB else B
            C = torch.empty(M, 128, device="cuda")
            ops.gemm_nn_tc(A, None, M, K, Bin, bool(transB), C)
            torch.cuda.synchronize()
            assert torch.equal(C, _ref_nn(A, Bin, transB).float())


def test_gemm_nn_tc_rejects_bad_arguments():
    from npi_gnn_b200 import ops, _lib as L
    A = torch.zeros(8, 48, device="cuda"); B = torch.zeros(48, 128, device="cuda"); C = torch.zeros(8, 128, device="cuda")
    with pytest.raises(L.NPIError):
        ops.gemm_nn_tc(A, None, 8, 48, B.t().contiguous(), True, C)     # transposed weights: K must be a multiple of 32
    with pytest.raises(L.NPIError):
        ops.gemm_nn_tc(torch.zeros(8, 200, device="cuda"), None, 8, 200, torch.zeros(200, 128, device="cuda"), False, C)   # K > 192
    A = torch.zeros(8, 130, device="cuda")[:, 1:129]
    with pytest.raises(L.NPIError):
        ops.gemm_nn_tc(A, None, 8, 128, torch.zeros(128, 128, device="cuda"), False, C)      # misaligned operand


@pytest.mark.parametrize("with_row0", [False, True])
@pytest.mark.parametrize("M", [1, 31, 32, 33, 127, 129, 4097, 107579])
def test_gemm_tn_tc_vs_fp64(M, with_row0):
    """dW = X^T . DXA: reduction over the rows, split over the CTAs and summed in fixed order.  The
    bound scales with the magnitude actually summed (|A|^T |D|): fp32 accumulation over M terms."""
    from npi_gnn_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + 11)
    A = torch.randn(M, 128, device="cuda", generator=g)
    D = torch.randn(M, 128, device="cuda", generator=g)
    row0 = torch.randn(5, 128, device="cuda", generator=g) if with_row0 else None
    ws = torch.empty(ops.gemm_tn_tc_workspace_bytes(), dtype=torch.uint8, device="cuda")
    out = torch.full((128, 128), float("nan"), device="cuda")
    ops.gemm_tn_tc(A, D, None, M, row0, out, ws)
    torch.cuda.synchronize()
    R = A.double().t() @ D.double()
    if with_row0:
        R[0] += row0.double().sum(0)
    mag = A.double().abs().t() @ D.double().abs() + (row0.double().abs().sum(0)[None, :] if with_row0 else 0.0)
    assert bool(((out.double() - R).abs() <= 2e-6 * mag + 1e-30).all()), float(((out.double() - R).abs() / mag).max())
    assert float((out.double() - R).abs().max()) / float(R.abs().max()) <= 2e-5
    out2 = torch.empty_like(out)
    ops.gemm_tn_tc(A, D, None, M, row0, out2, ws)
    torch.cuda.synchronize()
    assert torch.equal(out, out2)


@pytest.mark.parametrize("F,ld", [(178, 180), (65, 68), (256, 256)])
def test_gemm_tn_tc_feature_table_widths(F, ld):
    """dW1 = table^T . G of the layer-1 weight gradient (reference: SAGEConv backward of src/classes.py:62 on the virtual
    features): K = F > 128 takes one pass per 128 table columns, the label-row partials land on row 0 only."""
    from npi_gnn_b200 import ops
    M = 5085
    g = torch.Generator(device="cuda").manual_seed(F)
    table = torch.zeros(M, ld, device="cuda")
    table[:, 1:F] = torch.randn(M, F - 1, device="cuda", generator=g)
    G = torch.randn(M, 128, device="cuda", generator=g)
    row0 = torch.randn(37, 128, device="cuda", generator=g)
    out = torch.full((F + 1, 128), float("nan"), device="cuda")
    ws = torch.empty(ops.gemm_tn_tc_workspace_bytes(), dtype=torch.uint8, device="cuda")
    ops.gemm_tn_tc(table, G, None, M, row0, out, ws, K=F)
    torch.cuda.synchronize()
    R = table[:, :F].double().t() @ G.double()
    R[0] += row0.double().sum(0)
    assert torch.isnan(out[F:]).all()
    err = float((out[:F].double() - R).abs().max()) / float(R.abs().max())
    assert err <= TC_REL, err
    out2 = torch.empty(F, 128, device="cuda")
    ops.gemm_tn_tc(table, G, None, M, row0, out2, ws, K=F)
    torch.cuda.synchronize()
    assert torch.equal(out[:F], out2)


@pytest.mark.parametrize("V", [1, 31, 33, 1000, 5085, 32768])
@pytest.mark.parametrize("F,ld", [(178, 180), (65, 68), (256, 256), (5, 5)])
def test_table_grad_small_table(V, F, ld):
    """ops.table_grad (two-launch SIMT weight gradient through a small feature table, the last link of the step) against an
    fp64 product: exact fp32 products, fixed-order sums -- plain fp32 accumulation error, rerun bit-identical."""
    from npi_gnn_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(V * 7 + F)
    table = torch.zeros(V, ld, device="cuda")
    table[:, 1:F] = torch.randn(V, F - 1, device="cuda", generator=g)
    G = torch.randn(V, 128, device="cuda", generator=g)
    row0 = torch.randn(444, 128, device="cuda", generator=g)
    out = torch.full((F + 1, 128), float("nan"), device="cuda")
    ws = torch.empty(ops.table_grad_workspace_bytes(F), dtype=torch.uint8, device="cuda")
    ops.table_grad(table, G, V, row0, out, ws, K=F)
    torch.cuda.synchronize()
    R = table[:, :F].double().t() @ G.double()
    R[0] += row0.double().sum(0)
    mag = table[:, :F].double().abs().t() @ G.double().abs()
    mag[0] += row0.double().abs().sum(0)
    assert torch.isnan(out[F:]).all()
    assert bool(((out[:F].double() - R).abs() <= 2e-6 * mag + 1e-30).all()), float(((out[:F].double() - R).abs() / (mag + 1e-30)).max())
    out2 = torch.empty(F, 128, device="cuda")
    ops.table_grad(table, G, V, row0, out2, ws, K=F)
    torch.cuda.synchronize()
    assert torch.equal(out[:F], out2)


def test_gemm_tn_tc_device_side_m():
    from npi_gnn_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    A = torch.randn(6000, 128, device="cuda", generator=g)
    D = torch.randn(6000, 128, device="cuda", generator=g)
    A[4097:] = float("nan")                                      # rows past m must not be read into the sum
    md = torch.tensor([4097], dtype=torch.int32, device="cuda")
    ws = torch.empty(ops.gemm_tn_tc_workspace_bytes(), dtype=torch.uint8, device="cuda")
    out = torch.empty(128, 128, device="cuda")
    ops.gemm_tn_tc(A, D, md, 6000, None, out, ws)
    torch.cuda.synchronize()
    R = A[:4097].double().t() @ D[:4097].double()
    assert float((out.double() - R).abs().max()) / float(R.abs().max()) <= 2e-5


# ----------------------------------------------------------------------------- by-serial lists
def _gid_case(seed, N, V, hub=None):
    rng = np.random.default_rng(seed)
    gid = rng.integers(0, V, size=N).astype(np.int32)
    if hub is not None:                                         # one serial occurring in a large share of the rows
        gid[rng.random(N) < 0.3] = hub
    dist = rng.integers(0, 4, size=N).astype(np.uint8)
    return gid, dist


@pytest.mark.parametrize("N,V,hub", [(1, 1, None), (5, 9, None), (1000, 37, 3), (50000, 5085, 17), (215000, 5085, 100),
                                     (120000, 70001, 11)])      # > 8192 buckets: the three-kernel scan inside gid_index_build
def test_gid_index_build_and_reduce(N, V, hub):
    """occ_ptr / occ_node = the rows of every serial in ascending row order (bit-exact: that order is
    what makes G deterministic); G[v] = sum of dxa over the list, label partials = sum_j dist_j dxa_j."""
    from npi_gnn_b200 import ops
    gid_h, dist_h = _gid_case(N + V, N, V, hub)
    gid = torch.from_numpy(gid_h).cuda(); dist = torch.from_numpy(dist_h).cuda()
    cap = N + 7
    gid_pad = torch.cat([gid, torch.zeros(7, dtype=torch.int32, device="cuda")])
    n_dev = torch.tensor([N], dtype=torch.int32, device="cuda")
    occ_ptr = torch.full((V + 1,), -1, dtype=torch.int32, device="cuda")
    occ_node = torch.full((cap,), -1, dtype=torch.int32, device="cuda")
    ws = torch.empty(ops.gid_index_workspace_bytes(V, cap), dtype=torch.uint8, device="cuda")
    ops.gid_index_build(gid_pad, n_dev, cap, V, occ_ptr, occ_node, ws)
    torch.cuda.synchronize()
    order = np.argsort(gid_h, kind="stable")
    cnt = np.bincount(gid_h, minlength=V)
    assert np.array_equal(occ_ptr.cpu().numpy(), np.concatenate([[0], np.cumsum(cnt)]))
    assert np.array_equal(occ_node[:N].cpu().numpy(), order.astype(np.int32))
    g = torch.Generator(device="cuda").manual_seed(N)
    dxa = torch.randn(cap, 128, device="cuda", generator=g)
    G = torch.full((V, 128), float("nan"), device="cuda")
    lab = torch.zeros(ops.gid_reduce_partials(), 128, device="cuda")
    ops.gid_reduce(dxa, torch.cat([dist, torch.zeros(7, dtype=torch.uint8, device="cuda")]), occ_ptr, occ_node, V, G, lab)
    torch.cuda.synchronize()
    ref = torch.zeros(V, 128, dtype=torch.float64, device="cuda").index_add_(0, gid.long(), dxa[:N].double())
    mag = torch.zeros(V, 128, dtype=torch.float64, device="cuda").index_add_(0, gid.long(), dxa[:N].double().abs())
    assert bool(((G.double() - ref).abs() <= 1e-6 * mag + 1e-30).all())
    lab_ref = (dist.double()[:, None] * dxa[:N].double()).sum(0)
    lab_mag = (dist.double()[:, None] * dxa[:N].double().abs()).sum(0)
    assert bool(((lab.double().sum(0) - lab_ref).abs() <= 1e-5 * lab_mag + 1e-30).all())
    G2 = torch.empty_like(G); lab2 = torch.zeros_like(lab)
    ops.gid_reduce(dxa, torch.cat([dist, torch.zeros(7, dtype=torch.uint8, device="cuda")]), occ_ptr, occ_node, V, G2, lab2)
    torch.cuda.synchronize()
    assert torch.equal(G, G2) and torch.equal(lab, lab2)         # no float atomics: rerun bit-identical


# ----------------------------------------------------------------------------- dropout stream
def test_philox_dropout_is_keyed_by_sample_id_not_by_position():
    """The dropout mask of a sample depends on (seed, step, global sample id, feature) only -- the same
    pair draws the same mask whatever its position in the batch and whatever the batch holds, which is
    what makes a 1-GPU and an N-GPU run of the same global batch draw identical masks (SURVEY 8e)."""
    from npi_gnn_b200 import ops
    B = 64
    g = torch.Generator(device="cuda").manual_seed(1)
    readout = torch.randn(B, 256, device="cuda", generator=g)
    w1 = torch.randn(128, 256, device="cuda", generator=g) * 0.05; b1 = torch.zeros(128, device="cuda")
    w2 = torch.randn(64, 128, device="cuda", generator=g) * 0.05; b2 = torch.zeros(64, device="cuda")
    w3 = torch.randn(2, 64, device="cuda", generator=g) * 0.05; b3 = torch.zeros(2, device="cuda")
    step = torch.tensor([7], dtype=torch.int32, device="cuda")

    def masks(ids, seed=99, step_dev=step):
        a1 = torch.empty(B, 128, device="cuda"); m = torch.empty(B, 128, dtype=torch.uint8, device="cuda")
        a2 = torch.empty(B, 64, device="cuda"); lp = torch.empty(B, 2, device="cuda")
        ops.head_fwd(readout, len(ids), w1, b1, w2, b2, w3, b3, True, None, seed, step_dev,
                     torch.tensor(ids, dtype=torch.int32, device="cuda"), 0, None, 1.0, a1, m, a2, lp, None)
        torch.cuda.synchronize()
        return m[:len(ids)].cpu()

    ids = list(range(1000, 1000 + B))
    full = masks(ids)
    assert 0.45 < float(full.float().mean()) < 0.55
    # two "ranks": each half of the batch alone draws the rows the full batch drew
    assert torch.equal(masks(ids[:B // 2]), full[:B // 2])
    assert torch.equal(masks(ids[B // 2:]), full[B // 2:])
    # a permuted batch draws the permuted masks
    perm = np.random.default_rng(0).permutation(B)
    assert torch.equal(masks([ids[i] for i in perm]), full[torch.from_numpy(perm)])
    # other seed / other step: different stream
    assert not torch.equal(masks(ids, seed=100), full)
    assert not torch.equal(masks(ids, step_dev=torch.tensor([8], dtype=torch.int32, device="cuda")), full)
    # rows are pairwise different (no accidental reuse of one stream for every sample)
    assert len({bytes(r.numpy().tobytes()) for r in full}) == B
