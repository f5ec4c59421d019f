"""Top-k per group on the GPU (npi_group_topk, trainer.top_k_by_group, Scorer.top_partners) against a numpy oracle:
per group, np.lexsort((positions, -score)) with -0.0 folded to +0.0.  Positions and scores must be equal exactly."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.common import config5_pairs, fold0, grouped, synthetic_bipartite, ties

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# members of a group whose score keys are staged once in shared memory; larger groups take the reread path
STAGE = int(re.search(r"constexpr int TK_STAGE = (\d+);",
                      open(os.path.join(ROOT, "npi_gnn_b200", "csrc", "topk.cu")).read()).group(1))


def oracle(s, grp, G, k):
    """(pos [G,k], score [G,k], count [G]): per group the items by descending score, ties by ascending position."""
    s = np.asarray(s, dtype=np.float32)
    grp = np.asarray(grp, dtype=np.int64)
    n = len(s)
    folded = s + np.float32(0.0)                                     # -0.0 -> +0.0
    order = np.lexsort((np.arange(n), -folded, grp))                 # group, then descending score, then position
    gs = grp[order]
    cnt = np.bincount(grp, minlength=G)
    rank = np.arange(n) - (np.cumsum(cnt) - cnt)[gs]
    keep = rank < k
    pos = np.full((G, k), -1, dtype=np.int32)
    sc = np.full((G, k), np.nan, dtype=np.float32)
    pos[gs[keep], rank[keep]] = order[keep]
    sc[gs[keep], rank[keep]] = s[order[keep]]
    return pos, sc, np.minimum(cnt, k).astype(np.int32)


def _gpu(s, grp, G, k):
    from npi_gnn_b200 import top_k_by_group
    r = top_k_by_group(torch.as_tensor(np.asarray(s, dtype=np.float32)).cuda(),
                       torch.as_tensor(np.asarray(grp, dtype=np.int32)).cuda(), G, k)
    return r["pos"].cpu().numpy(), r["score"].cpu().numpy(), r["count"].cpu().numpy()


def _assert_same(got, want):
    (gp, gs, gc), (wp, ws, wc) = got, want
    assert np.array_equal(gc, wc), np.nonzero(gc != wc)[0][:10]
    bad = np.argwhere(gp != wp)
    assert len(bad) == 0, ("positions differ", bad[:5], gp[tuple(bad[0])], wp[tuple(bad[0])])
    live = wp >= 0
    assert np.array_equal(gs[live].view(np.int32), ws[live].view(np.int32))      # bit for bit, signs of zeros included
    assert np.isnan(gs[~live]).all()


def _check(s, grp, G, k):
    _assert_same(_gpu(s, grp, G, k), oracle(s, grp, G, k))


# ----------------------------------------------------------------------------- hand cases
def test_k_larger_than_every_group():
    rng = np.random.default_rng(1)
    grp = grouped(rng, [3, 1, 5, 2, 4])
    s = ties(rng, len(grp))
    got = _gpu(s, grp, 5, 7)
    assert list(got[2]) == [3, 1, 5, 2, 4]
    _assert_same(got, oracle(s, grp, 5, 7))


def test_empty_groups_first_last_and_between():
    rng = np.random.default_rng(2)
    sizes = [0, 4, 0, 0, 9, 1, 0, 30, 0]
    grp = grouped(rng, sizes)
    s = ties(rng, len(grp))
    pos, sc, cnt = _gpu(s, grp, len(sizes), 8)
    assert list(cnt) == [min(c, 8) for c in sizes]
    for g in (0, 2, 3, 6, 8):
        assert (pos[g] == -1).all() and np.isnan(sc[g]).all()
    _assert_same((pos, sc, cnt), oracle(s, grp, len(sizes), 8))


def test_all_scores_tied_take_first_positions():
    grp = np.tile(np.array([0, 1], dtype=np.int32), 3000)           # two interleaved groups of 3,000 equal scores
    s = np.full(6000, 0.25, dtype=np.float32)
    pos, sc, cnt = _gpu(s, grp, 2, 100)
    assert list(pos[0]) == list(range(0, 200, 2)) and list(pos[1]) == list(range(1, 200, 2))
    assert (sc == 0.25).all() and list(cnt) == [100, 100]


def test_signed_zeros_are_one_value():
    s = np.array([-0.0, 0.0, -0.0, 1.0, 0.0, -0.0, -1.0, 0.0], dtype=np.float32)
    grp = np.zeros(8, dtype=np.int32)
    pos, sc, cnt = _gpu(s, grp, 1, 5)
    assert list(pos[0]) == [3, 0, 1, 2, 4]                          # the zeros in position order, whatever their sign
    assert list(np.signbit(sc[0])) == [False, True, False, True, False]
    _assert_same((pos, sc, cnt), oracle(s, grp, 1, 5))
    rng = np.random.default_rng(3)                                  # many zeros of both signs, k below their count
    s = np.where(rng.random(5000) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    s[rng.random(5000) < 0.01] = 2.0
    grp = (rng.random(5000) < 0.5).astype(np.int32)
    _check(s, grp, 2, 300)


def test_infinities_are_ordinary_scores():
    s = np.array([np.inf, 1.0, -np.inf, np.inf, 0.0, -np.inf, 3e38, -3e38], dtype=np.float32)
    grp = np.zeros(8, dtype=np.int32)
    pos, sc, cnt = _gpu(s, grp, 1, 8)
    assert list(pos[0]) == [0, 3, 6, 1, 4, 7, 2, 5]
    _assert_same((pos, sc, cnt), oracle(s, grp, 1, 8))


@pytest.mark.parametrize("k", [1, 1024])
def test_smallest_and_largest_k(k):
    rng = np.random.default_rng(k)
    sizes = [1, 2, 1023, 1024, 1025, 3000, 0, 20000]
    grp = grouped(rng, sizes)
    _check(ties(rng, len(grp)), grp, len(sizes), k)


def test_single_item():
    assert [list(a.ravel()) for a in _gpu([0.5], [0], 1, 3)[::2]] == [[0, -1, -1], [1]]
    _check(np.array([-0.0], dtype=np.float32), [2], 4, 1)


def test_nan_scores_and_group_ids_out_of_range_raise():
    from npi_gnn_b200 import NPIError, top_k_by_group
    s = torch.rand(9000, device="cuda")
    grp = (torch.arange(9000, device="cuda") % 7).to(torch.int32)
    s2 = s.clone(); s2[8999] = float("nan")
    with pytest.raises(NPIError, match="NaN"):
        top_k_by_group(s2, grp, 7, 5)
    for bad in (-1, 7, 1 << 30):
        g2 = grp.clone(); g2[4100] = bad
        with pytest.raises(NPIError, match="group id"):
            top_k_by_group(s, g2, 7, 5)
    assert int(top_k_by_group(s, grp, 7, 5)["count"].sum()) == 35


def test_argument_checks():
    import ctypes as C
    from npi_gnn_b200 import NPIError, ops, top_k_by_group
    from npi_gnn_b200 import _lib as L
    s = torch.rand(100, device="cuda")
    grp = torch.zeros(100, dtype=torch.int32, device="cuda")
    for k in (0, 1025, -3):
        with pytest.raises(ValueError):
            top_k_by_group(s, grp, 1, k)
    pos = torch.empty((4, 1025), dtype=torch.int32, device="cuda")
    sc = torch.empty((4, 1025), dtype=torch.float32, device="cuda")
    cnt = torch.empty(4, dtype=torch.int32, device="cuda")
    st = torch.empty(1, dtype=torch.int32, device="cuda")
    ws = torch.empty(ops.group_topk_workspace_bytes(100, 4), dtype=torch.uint8, device="cuda")
    for k in (0, 1025):
        with pytest.raises(NPIError, match="k = "):
            ops.group_topk(s, grp, 1, k, pos, sc, cnt, st, ws)

    def raw(n, G, k, wsb):
        L.call("npi_group_topk", L.ptr(s), L.ptr(grp), C.c_int64(n), C.c_int32(G), C.c_int32(k), L.ptr(pos), L.ptr(sc),
               L.ptr(cnt), L.ptr(st), L.ptr(ws), C.c_int64(wsb), L.stream_ptr())
    full = ws.numel()
    raw(100, 4, 8, full)
    for n in (-1, 0, -(1 << 40)):
        with pytest.raises(NPIError, match="n = "):
            raw(n, 4, 8, full)
    for G in (0, -2, 1 << 24):
        with pytest.raises(NPIError, match="num_groups"):
            raw(100, G, 8, full)
    with pytest.raises(NPIError, match="workspace"):
        raw(100, 4, 8, full - 1)
    with pytest.raises(NPIError, match="float32"):
        ops.group_topk(s.double(), grp, 1, 8, pos, sc, cnt, st, ws)
    with pytest.raises(NPIError, match="outputs"):
        ops.group_topk(s, grp, 5, 1025, pos, sc, cnt, st, ws)


# ----------------------------------------------------------------------------- random cases
@pytest.mark.parametrize("size", [STAGE - 1, STAGE, STAGE + 1])
@pytest.mark.parametrize("k", [10, 1024])
def test_group_sizes_across_the_stage(size, k):
    """Groups just below, at and one past the shared-memory stage next to small ones; the last member of every group
    holds its unique top score, so a group cut at the stage loses its first entry."""
    rng = np.random.default_rng(size * 7 + k)
    sizes = [size, 5, size, 0, size, 1500]
    grp = grouped(rng, sizes)
    s = ties(rng, len(grp))
    for g in range(len(sizes)):
        members = np.nonzero(grp == g)[0]
        if len(members):
            s[members[-1]] = 10.0 + g
    pos, sc, cnt = _gpu(s, grp, len(sizes), k)
    for g in range(len(sizes)):
        if sizes[g]:
            assert pos[g, 0] == np.nonzero(grp == g)[0][-1]
    _assert_same((pos, sc, cnt), oracle(s, grp, len(sizes), k))


@pytest.mark.parametrize("k", [7, 1024])
def test_one_group_of_2_20_items(k):
    rng = np.random.default_rng(20 + k)
    n = 1 << 20
    _check(ties(rng, n), np.zeros(n, dtype=np.int32), 1, k)
    grp = np.where(rng.random(n) < 0.001, 2, 1).astype(np.int32)    # one huge group between an empty and a small one
    _check(ties(rng, n), grp, 3, k)


def test_more_groups_than_eight_per_sm():
    from npi_gnn_b200 import ops
    rng = np.random.default_rng(4)
    G = 8 * ops.sm_count() + 37
    sizes = rng.integers(0, 60, G)
    sizes[rng.random(G) < 0.02] = 2000
    grp = grouped(rng, sizes)
    _check(ties(rng, len(grp)), grp, G, 16)


def test_shuffled_group_ids():
    """Group ids relabelled by a random permutation and items in random order: rows follow the labels."""
    rng = np.random.default_rng(5)
    sizes = rng.integers(0, 400, 1000)
    grp = grouped(rng, sizes)
    s = ties(rng, len(grp))
    relabel = rng.permutation(1000).astype(np.int32)
    _check(s, relabel[grp], 1000, 50)
    pos, sc, cnt = _gpu(s, relabel[grp], 1000, 50)
    p0, s0, c0 = _gpu(s, grp, 1000, 50)
    assert np.array_equal(pos[relabel], p0) and np.array_equal(cnt[relabel], c0)


@pytest.mark.parametrize("k", [10, 100])
def test_config5_groupings_full_size(k):
    """All 2,081,564 RNA x protein pairs of the NPInter2-shaped graph, probabilities on a 1/64 grid, grouped by RNA
    (449 members per group) and by protein (4,636 members), node serials as group ids (num_groups = all nodes)."""
    allp, _, V = config5_pairs()
    rng = np.random.default_rng(k)
    s = (rng.integers(0, 65, len(allp)) / 64.0).astype(np.float32)
    for col, members in ((0, 449), (1, 4636)):
        grp = allp[:, col]
        got = _gpu(s, grp, V, k)
        assert set(np.bincount(grp, minlength=V)) == {0, members}
        _assert_same(got, oracle(s, grp, V, k))


# ----------------------------------------------------------------------------- determinism, permutation, capture
def _bufs(n, G, k):
    from npi_gnn_b200 import ops
    return (torch.empty((G, k), dtype=torch.int32, device="cuda"), torch.empty((G, k), dtype=torch.float32, device="cuda"),
            torch.empty(G, dtype=torch.int32, device="cuda"), torch.empty(1, dtype=torch.int32, device="cuda"),
            torch.empty(ops.group_topk_workspace_bytes(n, G), dtype=torch.uint8, device="cuda"))


def _run(s, grp, G, k, bufs):
    from npi_gnn_b200 import ops
    ops.group_topk(s, grp, G, k, *bufs)


def _out(bufs):
    pos, sc, cnt, st, _ = bufs
    return [t.clone().view(torch.int32) for t in (pos, sc, cnt, st)]


def test_bit_identical_on_rerun():
    rng = np.random.default_rng(6)
    sizes = rng.integers(0, 3 * STAGE, 300)
    grp_np = grouped(rng, sizes)
    s, grp = torch.as_tensor(ties(rng, len(grp_np))).cuda(), torch.as_tensor(grp_np).cuda()
    bufs = _bufs(len(grp_np), 300, 200)
    _run(s, grp, 300, 200, bufs)
    first = _out(bufs)
    for t in bufs:
        t.view(torch.uint8).fill_(0xA5)                                # outputs and workspace
    _run(s, grp, 300, 200, bufs)
    assert all(torch.equal(a, b) for a, b in zip(first, _out(bufs)))
    assert int(first[3][0]) == 0


def test_permuted_input_gives_the_same_pairs():
    """Distinct scores: permuting the items and mapping the positions back gives the same pairs in the same order."""
    rng = np.random.default_rng(7)
    n, G = 300000, 70
    s = (rng.permutation(n) / n).astype(np.float32)
    grp = rng.integers(0, G, n).astype(np.int32)
    pos, sc, cnt = _gpu(s, grp, G, 500)
    perm = rng.permutation(n)
    pos2, sc2, cnt2 = _gpu(s[perm], grp[perm], G, 500)
    mapped = np.where(pos2 >= 0, perm[np.maximum(pos2, 0)], -1)
    assert np.array_equal(mapped, pos) and np.array_equal(sc2.view(np.int32), sc.view(np.int32))
    assert np.array_equal(cnt2, cnt)


def test_cuda_graph_capture_and_replay_on_new_scores():
    rng = np.random.default_rng(8)
    G, k = 500, 64
    sizes = rng.integers(0, 2 * STAGE // 50, G)
    sizes[:3] = (STAGE + 100, 0, 3 * STAGE)                           # the reread path inside the graph too
    grp_np = grouped(rng, sizes)
    n = len(grp_np)
    s0, s1 = ties(rng, n), ties(rng, n)
    s, grp = torch.as_tensor(s0).cuda(), torch.as_tensor(grp_np).cuda()
    bufs = _bufs(n, G, k)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _run(s, grp, G, k, bufs)                                     # warm-up outside capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _run(s, grp, G, k, bufs)
    s.copy_(torch.as_tensor(s1))
    bufs[0].fill_(-7)
    g.replay()
    torch.cuda.synchronize()
    pos, sc, cnt, st, _ = bufs
    assert int(st[0]) == 0
    _assert_same((pos.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()), oracle(s1, grp_np, G, k))


# ----------------------------------------------------------------------------- Scorer
def _check_partners(r, probs, pairs, V, k):
    for name, own, other in (("rna", 0, 1), ("protein", 1, 0)):
        pos, sc, cnt = oracle(probs, pairs[:, own], V, k)
        got = r[name]
        assert np.array_equal(got["count"].cpu().numpy(), cnt), name
        assert np.array_equal(got["partner"].cpu().numpy(), np.where(pos >= 0, pairs[np.maximum(pos, 0), other], -1)), name
        gp = got["prob"].cpu().numpy()
        live = pos >= 0
        assert np.array_equal(gp[live].view(np.int32), sc[live].view(np.int32)) and np.isnan(gp[~live]).all(), name


def test_scorer_top_partners_on_npinter2_fold0():
    from npi_gnn_b200.trainer import Scorer
    d, og, omask, pairs, ys, ps, params = fold0()
    sc = Scorer(ps, params, batch_size=200)
    r = sc.top_partners(5)
    probs = sc.probabilities().cpu().numpy()
    _check_partners(r, probs, pairs, ps.graph.num_nodes, 5)
    assert (r["rna"]["count"].cpu().numpy()[d["is_rna"] == 0] == 0).all()
    assert (r["protein"]["count"].cpu().numpy()[d["is_rna"] == 1] == 0).all()
    # a shuffled index view: ties break by position in the view, so compare against the view's own order
    perm = np.random.default_rng(3).permutation(len(pairs))
    sv = Scorer(ps, params, batch_size=200, index=perm)
    _check_partners(sv.top_partners(5), sv.probabilities().cpu().numpy(), pairs[perm], ps.graph.num_nodes, 5)


def test_scorer_top_partners_over_candidate_pairs():
    from npi_gnn_b200.engine import FlatParams
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    from npi_gnn_b200.trainer import Scorer
    d = synthetic_bipartite(11, 60, 40, 300, 300)
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"])
    cand = g.candidate_pairs()
    R, P = int(d["is_rna"].sum()), int((d["is_rna"] == 0).sum())
    assert len(cand) == R * P - len(d["edges"]) and (g.edge_ids(cand) < 0).all()
    ps = PairSet(g, cand, np.zeros(len(cand), dtype=np.int32), h=1)
    params = FlatParams(g.F, "cuda").init_reference(torch.Generator().manual_seed(2))
    sc = Scorer(ps, params, batch_size=200)
    _check_partners(sc.top_partners(7), sc.probabilities().cpu().numpy(), cand, g.num_nodes, 7)


def test_scorer_top_partners_needs_a_process_group_when_sharded():
    from npi_gnn_b200 import NPIError
    from npi_gnn_b200.trainer import Scorer
    d, og, omask, pairs, ys, ps, params = fold0()
    with pytest.raises(NPIError, match="process group"):
        Scorer(ps, params, batch_size=200, world_size=2, rank=0).top_partners(5)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_top_partners_two_gpus_match_one():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29641", os.path.join(ROOT, "tests", "scorer_dp_worker.py"),
           "top_partners"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stderr[-3000:]
    assert "TOPK_DP_OK" in out.stdout
