#!/usr/bin/env python
"""profiles/<tag>_traffic.json (tools/ncu_summary.py: DRAM bytes per captured launch, per kernel, in
launch order) -> profiles/roofline_traffic.json (what bench.py attaches as roofline.traffic), keyed
by "<C-ABI entry point>#<occurrence within the step>".

    python tools/traffic_map.py r01z "ncu --set full ... description"

A step launches every kernel a fixed number of times in a fixed order (forward layers 1,2,3, backward
layers 3,2,1), so occurrence k of an entry point is launch k of its kernel within the step; the FIRST
captured step is used."""
import json
import os
import sys

tag = sys.argv[1]
desc = sys.argv[2] if len(sys.argv) > 2 else ""
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = os.path.join(ROOT, "profiles")
t = json.load(open(os.path.join(P, "%s_traffic.json" % tag)))

# entry point -> [(kernel-name prefix, launches of that kernel per step, [index within the step per occurrence])]
MAP = {
    "npi_sage_aggregate_fwd": [("aggregate_fwd_pipe_kernel<1>", 1, {0: 0}), ("aggregate_fwd_pipe_kernel<0>", 2, {1: 0, 2: 1}),
                               ("aggregate_fwd_kernel<1>", 1, {0: 0}), ("aggregate_fwd_kernel<0>", 2, {1: 0, 2: 1})],
    # per-context backward of layer 1 (round 2): the transposed-aggregation kernel runs four times per step -- layers 3 and 2
    # (npi_sage_aggregate_bwd#0/#1), then the class gather and the by-node gather (npi_csr_gather_sum#0/#1)
    "npi_sage_aggregate_bwd": [("aggregate_bwd_pipe_kernel", 2, {0: 0, 1: 1}), ("aggregate_bwd_kernel", 3, {0: 0, 1: 1, 2: 2})],
    "npi_csr_gather_sum": [("aggregate_bwd_pipe_kernel", 4, {0: 2, 1: 3}), ("aggregate_bwd_pipe_kernel", 3, {0: 2})],
    "npi_ctx_finish": [("ctx_finish_kernel", 1, {0: 0})],
    "npi_pool_bwd": [("pool_bwd_kernel", 2, {0: 0, 2: 1}), ("pool_bwd_kernel", 3, {0: 0, 2: 1, 4: 2})],      # odd occurrences = the partial reduce (phase 2)
    "npi_pool_gate_readout": [("gate_readout_kernel", 3, {0: 0, 2: 1, 4: 2})],   # odd occurrences = the readout combine (phase 2)
    "npi_gemm_nn_tc": [("tc::gemm_tc_tma_kernel", 5, {0: 0, 1: 1, 2: 2, 3: 3, 4: 4})],
    "npi_gemm_tn_tc": [("tc::gemm_tn_tc_kernel", 2, {0: 0, 1: 1})],
    "npi_gid_reduce": [("gid_reduce_kernel", 1, {0: 0})],
    "npi_khop_fill": [("khop_kernel<1, 1>", 1, {0: 0})],
    "npi_topk_select": [("topk_select_kernel", 3, {0: 0, 1: 1, 2: 2})],
    "npi_gemm_nn": [("gemm_nn_kernel<1, 32>", 1, {0: 0})],
    "npi_gemm_tn": [("gemm_tn_kernel<1>", 1, {0: 0})],
}
entries = {}
for ep, alts in MAP.items():
    for kname, per_step, occ in alts:
        rec = t.get(kname)
        if not rec or len(rec["dram_bytes_per_launch"]) < per_step:
            continue
        v = rec["dram_bytes_per_launch"]
        for k, idx in occ.items():
            key = "%s#%d" % (ep, k)
            if key not in entries:
                entries[key] = {"dram_bytes_per_launch": float(v[idx]), "kernels": [kname]}
out = {"source": "profiles/%s_ncu.md (%s; dram__bytes_read.sum + dram__bytes_write.sum per launch, first captured step)" % (tag, desc),
       "entries": entries}
json.dump(out, open(os.path.join(P, "roofline_traffic.json"), "w"), indent=1)
print("wrote %d entries" % len(entries))
for k in sorted(entries):
    print("  %-28s %10.1f MB  %s" % (k, entries[k]["dram_bytes_per_launch"] / 1e6, entries[k]["kernels"][0]))
