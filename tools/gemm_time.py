#!/usr/bin/env python
"""Per-launch time of npi_gemm_nn_tc (CUDA events on the launching stream, L2 flushed between launches) over a
range of M: separates the fixed cost of a launch (allocation of tensor memory, weight staging, pipeline fill,
drain) from the streaming rate.   Usage (GPU box): python tools/gemm_time.py [out.json]"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from npi_gnn_b200 import _lib as L, ops  # noqa: E402

L.load()
dev = torch.device("cuda", 0)
peak = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))["hbm_gbs"] \
    if os.path.exists("MEASURED_PEAKS.json") else 6547.2
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
W = torch.randn(128, 128, device=dev)
res = []
for M in (128, 148 * 128, 53790, 107579, 4 * 107579):
    A = torch.randn(M, 128, device=dev)
    C = torch.empty(M, 128, device=dev)
    ts = []
    for i in range(12):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.gemm_nn_tc(A, None, M, 128, W, i & 1, C)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    us = float(np.median(ts[2:]))
    gbs = 2 * M * 512 / us / 1e3
    res.append(dict(M=M, us=us, alg_GBps=gbs, frac=gbs / peak))
    print(res[-1], flush=True)
if len(sys.argv) > 1:
    json.dump(res, open(sys.argv[1], "w"), indent=1)
