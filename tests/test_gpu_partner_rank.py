"""Filtered per-node ranking on the GPU (npi_group_rank, trainer.group_rank_metrics, Scorer.partner_ranks) against the fp64
numpy oracle of tests/test_partner_rank_host.py.  above / tied, n_pos / n_neg / twice_u and the hits counts must be equal
exactly; MRR and the macro AUC to 1e-12 relative."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.common import config5_pairs, fold0, grouped, ties
from tests.test_partner_rank_host import oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HITS = (1, 3, 10)
REL = 1e-12


def _t(a, dt):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=dt)).cuda()


def _gpu(s, y, grp, G, hits=HITS):
    from npi_gnn_b200 import group_rank_metrics
    return group_rank_metrics(_t(s, np.float32), _t(y, np.int32), _t(grp, np.int32), G, hits=hits, per_item=True)


def _close(a, b):
    return (np.isnan(a) and np.isnan(b)) or abs(a - b) <= REL * abs(b)


def _assert_same(r, o, hits=HITS):
    for k in ("above", "tied", "n_pos", "n_neg", "twice_u"):
        got = r[k].cpu().numpy()
        bad = np.nonzero(got != o[k])[0]
        assert len(bad) == 0, (k, bad[:5], got[bad[:5]], o[k][bad[:5]])
    for k in ("n_queries", "n_unranked", "n_groups_scored"):
        assert r[k] == o[k], (k, r[k], o[k])
    assert r["hits"] == {k: o["hits"][k] / o["n_queries"] for k in hits}
    assert _close(r["mrr"], o["mrr"]), (r["mrr"], o["mrr"])
    assert _close(r["auc_macro"], o["auc_macro"]), (r["auc_macro"], o["auc_macro"])
    np.testing.assert_array_equal(r["auc"].cpu().numpy(), o["auc"])


def _check(s, y, grp, G, hits=HITS):
    r = _gpu(s, y, grp, G, hits)
    _assert_same(r, oracle(s, y, grp, G, hits), hits)
    return r


def _labels(rng, n, p=0.2):
    return (rng.random(n) < p).astype(np.int32)


# ----------------------------------------------------------------------------- hand cases
def test_all_scores_tied():
    rng = np.random.default_rng(1)
    n = 6000
    grp = (np.arange(n) % 3).astype(np.int32)
    y = _labels(rng, n)
    r = _check(np.full(n, 0.25, dtype=np.float32), y, grp, 3)
    above, tied = r["above"].cpu().numpy(), r["tied"].cpu().numpy()
    n_neg = r["n_neg"].cpu().numpy()
    assert (above[y == 1] == 0).all() and (tied[y == 1] == n_neg[grp[y == 1]]).all()
    assert (above[y == 0] == -1).all() and (tied[y == 0] == -1).all()
    np.testing.assert_array_equal(r["auc"].cpu().numpy(), [0.5, 0.5, 0.5])


def test_signed_zeros_are_one_score():
    s = np.array([-0.0, 0.0, -0.0, 1.0, 0.0, -0.0, -1.0, 0.0], dtype=np.float32)
    y = np.array([1, 0, 0, 0, 1, 1, 0, 0], dtype=np.int32)
    r = _check(s, y, np.zeros(8, dtype=np.int32), 1)
    assert list(r["above"].cpu().numpy()[[0, 4, 5]]) == [1, 1, 1] and list(r["tied"].cpu().numpy()[[0, 4, 5]]) == [3, 3, 3]
    rng = np.random.default_rng(3)
    s = np.where(rng.random(5000) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    s[rng.random(5000) < 0.05] = 2.0
    _check(s, _labels(rng, 5000), (rng.random(5000) < 0.5).astype(np.int32), 2)


def test_infinities_are_ordinary_scores():
    s = np.array([np.inf, 1.0, -np.inf, np.inf, 0.0, -np.inf, 3e38, -3e38], dtype=np.float32)
    y = np.array([1, 0, 1, 0, 0, 0, 1, 0], dtype=np.int32)
    r = _check(s, y, np.zeros(8, dtype=np.int32), 1)
    assert list(r["above"].cpu().numpy()[[0, 2, 6]]) == [0, 4, 1] and list(r["tied"].cpu().numpy()[[0, 2, 6]]) == [1, 1, 0]


def test_empty_groups_first_last_and_between():
    rng = np.random.default_rng(2)
    sizes = [0, 4, 0, 0, 9, 1, 0, 30, 0, 300, 0]
    grp = grouped(rng, sizes)
    y = _labels(rng, len(grp), 0.4)
    r = _check(ties(rng, len(grp)), y, grp, len(sizes))
    for g in (0, 2, 3, 6, 8, 10):
        assert r["n_pos"][g] == 0 and r["n_neg"][g] == 0 and r["twice_u"][g] == 0 and torch.isnan(r["auc"][g])


def test_groups_of_queries_only_are_unranked_and_groups_of_competitors_only_unscored():
    rng = np.random.default_rng(4)
    grp = np.array([0] * 5 + [1] * 7 + [2] * 9 + [3] * 3, dtype=np.int32)
    y = np.array([1] * 5 + [0] * 7 + [1, 0] * 4 + [1] + [1, 1, 0], dtype=np.int32)
    r = _check(ties(rng, len(grp)), y, grp, 4)
    assert r["n_unranked"] == 5 and r["n_queries"] == 5 + 2 and r["n_groups_scored"] == 2
    assert (r["above"].cpu().numpy()[:5] == 0).all() and (r["tied"].cpu().numpy()[:5] == 0).all()
    assert torch.isnan(r["auc"][:2]).all()


def test_single_item():
    from npi_gnn_b200 import ops
    for y in (1, 0):                                                 # a lone query is unranked, a lone competitor no query
        with pytest.raises(ValueError, match="MRR"):
            _gpu([0.5], [y], [0], 1)
    n_pos, n_neg, twice_u, summary, sum_rr, status, ws, above, tied = _bufs(1, 3, 3)
    ops.group_rank(_t([-0.0], np.float32), _t([1], np.int32), _t([2], np.int32), 3, HITS, n_pos, n_neg, twice_u, summary,
                   sum_rr, status, ws, above, tied)
    assert summary.tolist() == [0, 1, 0, 0, 0, 0] and float(sum_rr) == 0.0 and int(status) == 0
    assert n_pos.tolist() == [0, 0, 1] and n_neg.tolist() == [0, 0, 0] and twice_u.tolist() == [0, 0, 0]
    assert above.tolist() == [0] and tied.tolist() == [0]
    n_pos, n_neg, twice_u, summary, sum_rr, status, ws, above, tied = _bufs(2, 1, 1)
    ops.group_rank(_t([0.5, 0.5], np.float32), _t([1, 0], np.int32), _t([0, 0], np.int32), 1, (1,), n_pos, n_neg, twice_u,
                   summary, sum_rr, status, ws, above, tied)
    assert summary[:4].tolist() == [1, 0, 1, 0] and float(sum_rr) == 1.0 / 1.5 and twice_u[0] == 1


def test_one_group_of_2_20_items():
    rng = np.random.default_rng(20)
    n = 1 << 20
    _check(ties(rng, n), _labels(rng, n, 0.01), np.zeros(n, dtype=np.int32), 1)
    grp = np.where(rng.random(n) < 0.001, 2, 1).astype(np.int32)     # one huge group between an empty and a small one
    _check(ties(rng, n), _labels(rng, n, 0.3), grp, 3, hits=(1, 2, 5, 10, 100, 1000, 10000, 100000))


def test_more_than_2_18_groups():
    """19 key bits: the three-pass sort of the group ids."""
    rng = np.random.default_rng(5)
    G = (1 << 18) + 4321
    sizes = rng.integers(0, 8, G)
    sizes[rng.random(G) < 0.001] = 700
    grp = grouped(rng, sizes)
    _check(ties(rng, len(grp)), _labels(rng, len(grp), 0.3), grp, G)


def test_shuffled_group_ids():
    """Group ids relabelled by a random permutation: the per-group outputs follow the labels, the summary stays."""
    rng = np.random.default_rng(6)
    sizes = rng.integers(0, 400, 1000)
    grp = grouped(rng, sizes)
    s, y = ties(rng, len(grp)), _labels(rng, len(grp))
    relabel = rng.permutation(1000).astype(np.int32)
    r = _check(s, y, relabel[grp], 1000)
    r0 = _gpu(s, y, grp, 1000)
    for k in ("n_pos", "n_neg", "twice_u", "auc"):
        assert torch.equal(r[k][torch.as_tensor(relabel).cuda().long()].view(torch.int32), r0[k].view(torch.int32)), k
    for k in ("hits", "n_queries", "n_unranked", "n_groups_scored"):
        assert r[k] == r0[k], k
    assert _close(r["mrr"], r0["mrr"])                                # the group order changes the order of the fp64 sum
    assert torch.equal(r["above"], r0["above"]) and torch.equal(r["tied"], r0["tied"])


def test_bad_scores_labels_and_group_ids_raise():
    from npi_gnn_b200 import NPIError, group_rank_metrics
    n = 9000
    s = torch.rand(n, device="cuda")
    y = (torch.arange(n, device="cuda") % 5 == 0).to(torch.int32)
    grp = (torch.arange(n, device="cuda") % 7).to(torch.int32)
    s2 = s.clone(); s2[8999] = float("nan")
    with pytest.raises(NPIError, match="NaN"):
        group_rank_metrics(s2, y, grp, 7)
    for bad in (2, -1):
        y2 = y.clone(); y2[4100] = bad
        with pytest.raises(NPIError, match="label"):
            group_rank_metrics(s, y2, grp, 7)
    for bad in (-1, 7, 1 << 30):
        g2 = grp.clone(); g2[4100] = bad
        with pytest.raises(NPIError, match="group id"):
            group_rank_metrics(s, y, g2, 7)
    assert group_rank_metrics(s, y, grp, 7)["n_queries"] == 1800


def _bufs(n, G, nh):
    from npi_gnn_b200 import ops
    i32 = dict(dtype=torch.int32, device="cuda")
    return (torch.empty(G, **i32), torch.empty(G, **i32), torch.empty(G, dtype=torch.int64, device="cuda"),
            torch.empty(3 + nh, dtype=torch.int64, device="cuda"), torch.empty(1, dtype=torch.float64, device="cuda"),
            torch.empty(1, **i32), torch.empty(ops.group_rank_workspace_bytes(n, G), dtype=torch.uint8, device="cuda"),
            torch.empty(n, **i32), torch.empty(n, **i32))


def test_argument_checks():
    import ctypes as C
    from npi_gnn_b200 import NPIError, ops
    from npi_gnn_b200 import _lib as L
    s = torch.rand(100, device="cuda")
    y = torch.zeros(100, dtype=torch.int32, device="cuda")
    grp = torch.zeros(100, dtype=torch.int32, device="cuda")
    b = _bufs(100, 4, 3)
    n_pos, n_neg, twice_u, summary, sum_rr, status, ws, above, tied = b

    def raw(n, G, ks, wsb):
        arr = (C.c_int32 * max(len(ks), 1))(*ks)
        L.call("npi_group_rank", L.ptr(s), L.ptr(y), L.ptr(grp), C.c_int64(n), C.c_int32(G), arr, C.c_int32(len(ks)),
               L.ptr(n_pos), L.ptr(n_neg), L.ptr(twice_u), L.ptr(summary), L.ptr(sum_rr), None, None, L.ptr(status), L.ptr(ws),
               C.c_int64(wsb), L.stream_ptr())
    full = ws.numel()
    raw(100, 4, (1, 3, 10), full)
    for n in (-1, 0, -(1 << 40)):
        with pytest.raises(NPIError, match="n = "):
            raw(n, 4, (1,), full)
    for G in (0, -2, 1 << 24):
        with pytest.raises(NPIError, match="num_groups"):
            raw(100, G, (1,), full)
    for ks in ((), tuple(range(1, 10))):
        with pytest.raises(NPIError, match="n_hits"):
            raw(100, 4, ks, full)
    for ks in ((0,), (3, -2)):
        with pytest.raises(NPIError, match="K = "):
            raw(100, 4, ks, full)
    with pytest.raises(NPIError, match="workspace"):
        raw(100, 4, (1,), full - 1)
    with pytest.raises(NPIError, match="float32"):
        ops.group_rank(s.double(), y, grp, 4, (1,), *b)
    with pytest.raises(NPIError, match="float32"):
        ops.group_rank(s, y[:99], grp, 4, (1,), *b)
    with pytest.raises(NPIError, match="outputs"):
        ops.group_rank(s, y, grp, 5, (1,), *b)                      # n_pos holds 4 groups
    with pytest.raises(NPIError, match="outputs"):
        ops.group_rank(s, y, grp, 4, (1, 2, 3, 4), *b)               # summary holds 3 hits
    with pytest.raises(NPIError, match="outputs"):
        ops.group_rank(s, y, grp, 4, (1,), n_pos, n_neg, twice_u.int(), summary, sum_rr, status, ws)


# ----------------------------------------------------------------------------- full size
def test_config5_groupings_full_size():
    """All 2,081,564 RNA x protein pairs of the NPInter2-shaped graph, the known interactions as queries, probabilities on
    a 1e-4 grid, grouped by RNA and by protein with node serials as group ids."""
    allp, y, V = config5_pairs()
    assert 5000 < y.sum() < 20000
    s = np.round(np.random.default_rng(7).random(len(allp)), 4).astype(np.float32)
    for col in (0, 1):
        _check(s, y, allp[:, col], V)


# ----------------------------------------------------------------------------- determinism, permutation, capture, launches
def _run(s, y, grp, G, bufs, hits=HITS):
    from npi_gnn_b200 import ops
    ops.group_rank(s, y, grp, G, hits, *bufs)


def _out(bufs):
    n_pos, n_neg, twice_u, summary, sum_rr, status, _, above, tied = bufs
    return [t.clone().view(torch.int32) for t in (n_pos, n_neg, twice_u, summary, sum_rr, status, above, tied)]


def test_bit_identical_on_rerun_and_under_permutation():
    rng = np.random.default_rng(8)
    G = 3000
    grp_np = grouped(rng, rng.integers(0, 300, G))
    n = len(grp_np)
    s_np, y_np = ties(rng, n), _labels(rng, n, 0.1)
    s, y, grp = _t(s_np, np.float32), _t(y_np, np.int32), _t(grp_np, np.int32)
    bufs = _bufs(n, G, 3)
    _run(s, y, grp, G, bufs)
    first = _out(bufs)
    for _ in range(2):
        for t in bufs:
            t.view(torch.uint8).fill_(0xA5)                            # outputs and workspace
        _run(s, y, grp, G, bufs)
        assert all(torch.equal(a, b) for a, b in zip(first, _out(bufs)))
    assert int(first[5][0]) == 0
    perm = rng.permutation(n)
    for t in bufs:
        t.view(torch.uint8).fill_(0xA5)
    _run(_t(s_np[perm], np.float32), _t(y_np[perm], np.int32), _t(grp_np[perm], np.int32), G, bufs)
    second = _out(bufs)
    for a, b in zip(first[:6], second[:6]):                           # per-group outputs, summary, sum_rr bits, status
        assert torch.equal(a, b)
    inv = torch.as_tensor(np.argsort(perm)).cuda()
    for a, b in zip(first[6:], second[6:]):                           # per-item outputs follow their items
        assert torch.equal(a, b[inv])


def test_cuda_graph_capture_and_replay_on_new_scores():
    rng = np.random.default_rng(9)
    G = 700
    grp_np = grouped(rng, rng.integers(0, 500, G))
    n = len(grp_np)
    s0, s1, y_np = ties(rng, n), ties(rng, n), _labels(rng, n)
    s, y, grp = _t(s0, np.float32), _t(y_np, np.int32), _t(grp_np, np.int32)
    bufs = _bufs(n, G, 3)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _run(s, y, grp, G, bufs)                                      # warm-up outside capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _run(s, y, grp, G, bufs)
    s.copy_(torch.as_tensor(s1))
    for t in bufs:
        t.view(torch.uint8).fill_(0xA5)
    g.replay()
    torch.cuda.synchronize()
    n_pos, n_neg, twice_u, summary, sum_rr, status, _, above, tied = bufs
    o = oracle(s1, y_np, grp_np, G)
    assert int(status[0]) == 0
    assert np.array_equal(above.cpu().numpy(), o["above"]) and np.array_equal(tied.cpu().numpy(), o["tied"])
    assert np.array_equal(twice_u.cpu().numpy(), o["twice_u"]) and np.array_equal(n_neg.cpu().numpy(), o["n_neg"])
    assert summary.tolist() == [o["n_queries"], o["n_unranked"], o["n_groups_scored"]] + [o["hits"][k] for k in HITS]
    assert _close(float(sum_rr[0]), o["sum_rr"])


@pytest.mark.parametrize("G", [5, 5000, (1 << 18) + 1])
def test_launch_count_matches_kernels_per_call(G):
    """The count booked in KERNELS_PER_CALL for each sort-pass variant is what one call launches (profiler trace)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    from npi_gnn_b200 import _lib as L
    rng = np.random.default_rng(G)
    n = 20000
    s, y, grp = _t(ties(rng, n), np.float32), _t(_labels(rng, n), np.int32), _t(rng.integers(0, G, n), np.int32)
    bufs = _bufs(n, G, 3)
    _run(s, y, grp, G, bufs)
    torch.cuda.synchronize()
    snap = dict(L.CALL_COUNTS)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        _run(s, y, grp, G, bufs)
        torch.cuda.synchronize()
    kernels = [e for e in prof.events() if e.device_type == DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset"))]
    booked = L.launches_since(snap)
    assert booked == {5: 24, 5000: 27, (1 << 18) + 1: 30}[G]
    assert len(kernels) == booked, sorted(e.name for e in kernels)


# ----------------------------------------------------------------------------- Scorer
def _fold0_with_candidates():
    """The NPInter2 fold-0 graph with the test pairs masked, the shipped checkpoint, and a pair set of the test positives
    (label 1), the test negatives and the candidate pairs of the first 100 RNAs with a test positive (label 0)."""
    from npi_gnn_b200.graph import PairSet
    d, og, omask, pairs, ys, ps, params = fold0()
    g = ps.graph
    cand = g.candidate_pairs()
    cand = cand[np.isin(cand[:, 0], np.unique(d["test_pos"][:, 0])[:100])]
    allp = np.concatenate([pairs, cand])
    y = np.concatenate([ys, np.zeros(len(cand), dtype=np.int32)])
    return allp, y, PairSet(g, allp, y, h=1), params


def test_scorer_partner_ranks_on_npinter2_fold0():
    from npi_gnn_b200.trainer import Scorer
    pairs, y, ps, params = _fold0_with_candidates()
    V = ps.graph.num_nodes
    sc = Scorer(ps, params, batch_size=200)
    r = sc.partner_ranks()
    probs = sc.probabilities().cpu().numpy()
    for name, own in (("rna", 0), ("protein", 1)):
        o = oracle(probs, y, pairs[:, own], V)
        for k in ("n_pos", "n_neg", "twice_u"):
            assert np.array_equal(r[name][k].cpu().numpy(), o[k]), (name, k)
        for k in ("n_queries", "n_unranked", "n_groups_scored"):
            assert r[name][k] == o[k], (name, k)
        assert r[name]["hits"] == {k: o["hits"][k] / o["n_queries"] for k in HITS}
        assert _close(r[name]["mrr"], o["mrr"]) and _close(r[name]["auc_macro"], o["auc_macro"])
        np.testing.assert_array_equal(r[name]["auc"].cpu().numpy(), o["auc"])
    assert r["rna"]["n_queries"] > 0 and r["protein"]["n_queries"] > 0
    perm = np.random.default_rng(3).permutation(len(pairs))
    r2 = Scorer(ps, params, batch_size=200, index=perm).partner_ranks()
    for name in ("rna", "protein"):
        for k in ("mrr", "hits", "n_queries", "n_unranked", "n_groups_scored"):
            assert r2[name][k] == r[name][k], (name, k)
        assert np.float64(r2[name]["auc_macro"]).view(np.int64) == np.float64(r[name]["auc_macro"]).view(np.int64)
        for k in ("n_pos", "n_neg", "twice_u", "auc"):
            assert torch.equal(r2[name][k].view(torch.int32), r[name][k].view(torch.int32)), (name, k)


def test_scorer_partner_ranks_needs_a_process_group_when_sharded():
    from npi_gnn_b200 import NPIError
    from npi_gnn_b200.trainer import Scorer
    d, og, omask, pairs, ys, ps, params = fold0()
    with pytest.raises(NPIError, match="process group"):
        Scorer(ps, params, batch_size=200, world_size=2, rank=0).partner_ranks()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_partner_ranks_two_gpus_match_one():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29643", os.path.join(ROOT, "tests", "scorer_dp_worker.py"),
           "partner_ranks"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stderr[-3000:]
    assert "PARTNER_RANK_DP_OK" in out.stdout
