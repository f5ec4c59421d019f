"""torchrun worker for tests/test_gpu_topk.py: Scorer(world_size=2).top_partners() on the NPInter2 fold-0 test set gives
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
    dp = Scorer(ps, params, batch_size=200, world_size=world, rank=rank).top_partners(20)
    one = Scorer(ps, params, batch_size=200).top_partners(20)
    for side in ("rna", "protein"):
        for key in ("partner", "prob", "count"):
            a, b = dp[side][key], one[side][key]
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (rank, side, key)
            other = a.clone()
            torch.distributed.broadcast(other, src=0)
            assert torch.equal(other.view(torch.int32), a.view(torch.int32)), (rank, side, key)
    D.barrier()
    if rank == 0:
        print("TOPK_DP world=%d rna rows=%d protein rows=%d" % (world, int((dp["rna"]["count"] > 0).sum()),
                                                                int((dp["protein"]["count"] > 0).sum())))
        print("TOPK_DP_OK")


if __name__ == "__main__":
    main()
