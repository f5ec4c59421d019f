"""torchrun worker for tests/test_gpu_rank.py: Scorer(world_size=2).rank_metrics() on the NPInter2 fold-0 test set gives
the same, bit-identical result on both ranks, equal to the single-GPU result."""
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

SCALARS = ("auroc", "ap", "pr_auc_trapz", "n_pos", "n_neg", "twice_u", "confusion")
CURVES = ("thresholds", "fpr", "tpr", "precision", "recall")


def main():
    world, rank, local = D.init("nccl")
    dev = torch.device("cuda", local)
    d = load_npinter2()
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device=dev)
    g.set_mask(np.concatenate([d["test_pos"], d["test_neg"]]))
    pairs = np.concatenate([d["test_pos"], d["test_neg"]])
    ys = np.concatenate([np.ones(len(d["test_pos"])), np.zeros(len(d["test_neg"]))]).astype(np.int32)
    perm = np.random.default_rng(0).permutation(len(pairs))
    ps = PairSet(g, pairs[perm], ys[perm], h=1)
    params = FlatParams(g.F, dev).load_state_dict(load_ckpt("ckpt_1223_1_15.npz"))
    dp = Scorer(ps, params, batch_size=200, world_size=world, rank=rank).rank_metrics(curve=True)
    one = Scorer(ps, params, batch_size=200).rank_metrics(curve=True)
    for k in SCALARS:
        assert dp[k] == one[k], (rank, k, dp[k], one[k])
    for k in CURVES:
        assert torch.equal(dp[k], one[k]), (rank, k)
        other = dp[k].clone()
        torch.distributed.broadcast(other, src=0)
        assert torch.equal(other, dp[k]), (rank, k)
    row = torch.tensor([dp["auroc"], dp["ap"], dp["pr_auc_trapz"], float(dp["twice_u"])], dtype=torch.float64, device=dev)
    rows = D.gather_rows(row, dev)
    assert torch.equal(rows[0], rows[1])
    D.barrier()
    if rank == 0:
        print("RANK_DP world=%d auroc=%.12f ap=%.12f pr_auc_trapz=%.12f" % (world, dp["auroc"], dp["ap"], dp["pr_auc_trapz"]))
        print("RANK_DP_OK")


if __name__ == "__main__":
    main()
