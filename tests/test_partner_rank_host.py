"""Host side of the filtered per-node ranking (npi_group_rank): the fp64 numpy oracle that tests/test_gpu_partner_rank.py
compares against, checked here against a brute-force count from the definition and against sklearn, and the argument
checks of group_rank_metrics that run before the device is touched (no GPU)."""
import numpy as np
import pytest


def oracle(s, y, grp, G, hits=(1, 3, 10)):
    """include/npi.h npi_group_rank in numpy: each query (label 1) counted against the competitors (label 0) of its group,
    -0.0 folded to +0.0.  Returns dict of above / tied (int32 [n], -1 for competitors), n_pos / n_neg (int32 [G]),
    twice_u (int64 [G]), n_queries, n_unranked, n_groups_scored, hits {K: count}, sum_rr, mrr, auc (float64 [G], NaN
    without both classes) and auc_macro."""
    s = np.asarray(s, dtype=np.float32) + np.float32(0.0)
    y = np.asarray(y, dtype=np.int64)
    grp = np.asarray(grp, dtype=np.int64)
    n = len(s)
    vals = np.unique(s)
    M = len(vals) + 1
    key = grp * M + np.searchsorted(vals, s)                         # (group, score) as one ordered int64
    q, c = y == 1, y == 0
    ck = np.sort(key[c])
    qk, qg = key[q], grp[q]
    right = np.searchsorted(ck, qk, "right")
    tied_q = right - np.searchsorted(ck, qk, "left")
    above_q = np.searchsorted(ck, (qg + 1) * M, "left") - right
    above = np.full(n, -1, dtype=np.int32)
    tied = np.full(n, -1, dtype=np.int32)
    above[q], tied[q] = above_q, tied_q
    n_pos = np.bincount(grp[q], minlength=G).astype(np.int32)
    n_neg = np.bincount(grp[c], minlength=G).astype(np.int32)
    twice_u = np.zeros(G, dtype=np.int64)
    np.add.at(twice_u, qg, 2 * (n_neg[qg].astype(np.int64) - above_q - tied_q) + tied_q)
    ranked = n_neg[qg] > 0
    twice_rank = 2 * above_q[ranked] + tied_q[ranked] + 2
    sum_rr = float(np.sum(2.0 / twice_rank.astype(np.float64)))
    nq = int(ranked.sum())
    both = (n_pos > 0) & (n_neg > 0)
    with np.errstate(invalid="ignore", divide="ignore"):
        auc = np.where(both, twice_u / (2.0 * n_pos.astype(np.float64) * n_neg), np.nan)
    return dict(above=above, tied=tied, n_pos=n_pos, n_neg=n_neg, twice_u=twice_u, n_queries=nq,
                n_unranked=int(q.sum()) - nq, n_groups_scored=int(both.sum()),
                hits={k: int((twice_rank <= 2 * k).sum()) for k in hits}, sum_rr=sum_rr,
                mrr=sum_rr / nq if nq else float("nan"), auc=auc,
                auc_macro=float(np.mean(auc[both])) if both.any() else float("nan"))


def _brute(s, y, grp, G, hits):
    """O(n^2) restatement of the definition with Python floats (-0.0 == 0.0, inf ordinary)."""
    s = [float(v) for v in np.asarray(s, dtype=np.float32)]
    n = len(s)
    above, tied = [-1] * n, [-1] * n
    n_pos, n_neg = [0] * G, [0] * G
    for i in range(n):
        (n_pos if y[i] == 1 else n_neg)[grp[i]] += 1
    twice_u, hit, rr, nq = [0] * G, {k: 0 for k in hits}, [], 0
    for i in range(n):
        if y[i] != 1:
            continue
        comp = [s[j] for j in range(n) if y[j] == 0 and grp[j] == grp[i]]
        above[i] = sum(v > s[i] for v in comp)
        tied[i] = sum(v == s[i] for v in comp)
        twice_u[grp[i]] += 2 * (n_neg[grp[i]] - above[i] - tied[i]) + tied[i]
        if comp:
            nq += 1
            rr.append(1.0 / (above[i] + tied[i] / 2 + 1))
            for k in hits:
                hit[k] += above[i] + tied[i] / 2 + 1 <= k
    return above, tied, n_pos, n_neg, twice_u, hit, nq, sum(rr)


def _random_case(rng, n, G):
    s = (rng.integers(-6, 7, n) / 4.0).astype(np.float32)           # heavy ties
    s[rng.random(n) < 0.1] = -0.0
    s[rng.random(n) < 0.03] = np.inf
    s[rng.random(n) < 0.03] = -np.inf
    y = (rng.random(n) < 0.3).astype(np.int32)
    grp = rng.integers(0, G, n).astype(np.int32)
    return s, y, grp


@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_brute_force(seed):
    rng = np.random.default_rng(seed)
    n, G = [1, 7, 60, 150, 300, 400][seed], [1, 3, 5, 9, 12, 40][seed]
    s, y, grp = _random_case(rng, n, G)
    hits = (1, 2, 5)
    o = oracle(s, y, grp, G, hits)
    above, tied, n_pos, n_neg, twice_u, hit, nq, rr = _brute(s, y, grp, G, hits)
    assert list(o["above"]) == above and list(o["tied"]) == tied
    assert list(o["n_pos"]) == n_pos and list(o["n_neg"]) == n_neg and list(o["twice_u"]) == twice_u
    assert o["n_queries"] == nq and o["n_unranked"] == int((y == 1).sum()) - nq and o["hits"] == hit
    assert o["sum_rr"] == pytest.approx(rr, rel=1e-13, abs=0)


def test_oracle_signed_zeros_and_infinities():
    s = np.array([-0.0, 0.0, 0.0, np.inf, -np.inf, np.inf, 1.0], dtype=np.float32)
    y = np.array([1, 0, 0, 1, 1, 0, 0], dtype=np.int32)
    o = oracle(s, y, np.zeros(7, dtype=np.int32), 1)
    assert list(o["above"]) == [2, -1, -1, 0, 4, -1, -1] and list(o["tied"]) == [2, -1, -1, 1, 0, -1, -1]
    assert o["hits"] == {1: 0, 3: 1, 10: 3}                          # 2 ranks: 8, 3, 10


def test_oracle_auc_matches_sklearn():
    skm = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(9)
    s, y, grp = _random_case(rng, 3000, 17)
    s[np.isinf(s)] = 0.5                                              # sklearn rejects infinite scores
    o = oracle(s, y, grp, 17)
    for g in range(17):
        m = grp == g
        if o["n_pos"][g] and o["n_neg"][g]:
            assert o["auc"][g] == pytest.approx(skm.roc_auc_score(y[m], s[m]), rel=1e-12)
        else:
            assert np.isnan(o["auc"][g])


def test_group_rank_metrics_rejects_bad_arguments_before_touching_the_device():
    import torch
    from npi_gnn_b200 import group_rank_metrics
    s, y, grp = torch.zeros(4), torch.zeros(4, dtype=torch.int32), torch.zeros(4, dtype=torch.int32)
    for hits in ((), tuple(range(1, 10)), (0,), (3, -1), (1, 1 << 31), 5, ("a",)):
        with pytest.raises(ValueError, match="hits"):
            group_rank_metrics(s, y, grp, 1, hits=hits)
    for G in (0, -5):
        with pytest.raises(ValueError, match="num_groups"):
            group_rank_metrics(s, y, grp, G)
