"""torchrun worker for tests/test_gpu_partner_rank.py: Scorer(world_size=2).partner_ranks() on the NPInter2 fold-0 test
set plus the candidate pairs of 30 RNAs gives the same, bit-identical result on both ranks, equal to the single-GPU
result."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from npi_gnn_b200 import dist as D  # noqa: E402
from npi_gnn_b200.engine import FlatParams  # noqa: E402
from npi_gnn_b200.graph import BipartiteGraph, PairSet  # noqa: E402
from npi_gnn_b200.trainer import Scorer  # noqa: E402
from tests.common import load_ckpt, load_npinter2  # noqa: E402


def main():
    world, rank, local = D.init("nccl")
    dev = torch.device("cuda", local)
    d = load_npinter2()
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device=dev)
    g.set_mask(np.concatenate([d["test_pos"], d["test_neg"]]))
    cand = g.candidate_pairs()
    cand = cand[np.isin(cand[:, 0], np.unique(d["test_pos"][:, 0])[:30])]
    pairs = np.concatenate([d["test_pos"], d["test_neg"], cand])
    ys = np.concatenate([np.ones(len(d["test_pos"])), np.zeros(len(d["test_neg"]) + len(cand))]).astype(np.int32)
    perm = np.random.default_rng(0).permutation(len(pairs))
    ps = PairSet(g, pairs[perm], ys[perm], h=1)
    params = FlatParams(g.F, dev).load_state_dict(load_ckpt("ckpt_1223_1_15.npz"))
    dp = Scorer(ps, params, batch_size=200, world_size=world, rank=rank).partner_ranks()
    one = Scorer(ps, params, batch_size=200).partner_ranks()
    for side in ("rna", "protein"):
        for key in ("mrr", "hits", "n_queries", "n_unranked", "n_groups_scored"):
            assert dp[side][key] == one[side][key], (rank, side, key)
        assert np.float64(dp[side]["auc_macro"]).view(np.int64) == np.float64(one[side]["auc_macro"]).view(np.int64)
        for key in ("n_pos", "n_neg", "twice_u", "auc"):
            a, b = dp[side][key], one[side][key]
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (rank, side, key)
            other = a.clone()
            torch.distributed.broadcast(other, src=0)
            assert torch.equal(other.view(torch.int32), a.view(torch.int32)), (rank, side, key)
        summary = torch.tensor([dp[side]["mrr"], dp[side]["auc_macro"]], dtype=torch.float64, device=dev)
        other = summary.clone()
        torch.distributed.broadcast(other, src=0)
        assert torch.equal(other.view(torch.int64), summary.view(torch.int64)), (rank, side)
    D.barrier()
    if rank == 0:
        print("PARTNER_RANK_DP world=%d rna MRR %.5f (%d queries), protein MRR %.5f (%d queries)"
              % (world, dp["rna"]["mrr"], dp["rna"]["n_queries"], dp["protein"]["mrr"], dp["protein"]["n_queries"]))
        print("PARTNER_RANK_DP_OK")


if __name__ == "__main__":
    main()
