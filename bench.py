#!/usr/bin/env python
"""Benchmark of the NPI-GNN hot path (BASELINE.json metric: enclosing subgraphs/sec of a
training step -- GPU extraction + gather + forward + backward + Adam -- at batch 200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N = 1 workload: BASELINE.json configs[1] -- synthetic bipartite graph of NPInter2 shape
(4,636 RNA + 449 protein, ~9.9 k positives + balanced negatives, fold 0 masked), 2-hop
enclosing subgraphs, node2vec+k-mer features (F = 178), batch 200.  N > 1: the same workload
data-parallel, 200 subgraphs per rank per step (weak scaling), one NCCL all-reduce per step.

One JSON line is printed by rank 0 (see DESIGN.md "Measurement" for every field).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "subgraphs/s"

# BASELINE.json configs: [1] is the bench line (the configuration the metric is quoted on); the others
# are selectable with --workload and recorded under profiles/ (they are parity-test cases first).
WORKLOADS = {
    "npinter2": dict(gen="npinter2_shaped", hops=2, batch=200, scaling="weak",
                     text="synthetic NPInter2-shaped bipartite graph (4636 RNA + 449 protein, fold 0 masked), "
                          "2-hop enclosing subgraphs, F=178 (node2vec+k-mer), batch 200 per GPU",
                     l2="every step streams a fresh batch whose working set (~1.9 GB) exceeds the 126 MB L2"),
    "rpi2241": dict(gen="rpi2241_shaped", hops=2, batch=200, scaling="weak",
                    text="synthetic RPI2241-shaped bipartite graph (838 RNA + 3752 protein, 2241+ / 2240- edges, fold 0 masked), "
                         "noKmer variant (F=65, node2vec only), 2-hop enclosing subgraphs, batch 200 per GPU",
                    l2="batches are smaller than L2: a 256 MB buffer is rewritten between timed steps"),
    "real_h1": dict(gen="real", hops=1, batch=200, scaling="weak",
                    text="REAL NPInter2 project 1223_1 fold 0 (tests/golden/npinter2_fold0.npz from the reference's shipped files: "
                         "5,085 nodes, 10,412+ / 10,412- edges, 16,658 training pairs, fold-0 test keys masked), 1-hop enclosing "
                         "subgraphs (what the reference ran), F=178, batch 200 per GPU, one epoch",
                    l2="every step streams a fresh batch; an epoch touches ~0.5 GB"),
    "real_h2": dict(gen="real", hops=2, batch=200, scaling="weak",
                    text="REAL NPInter2 project 1223_1 fold 0 (tests/golden/npinter2_fold0.npz), 2-hop enclosing subgraphs "
                         "(BASELINE.json configs[0]), F=178, batch 200 per GPU, one epoch",
                    l2="every step streams a fresh batch whose working set exceeds the 126 MB L2"),
    "x100": dict(gen="scaled_blocks", hops=3, global_batch=4096, scaling="strong",
                 text="100x scaled synthetic graph (disjoint union of 100 NPInter2-shaped blocks: 508,500 nodes, ~1.63 M edges), "
                      "3-hop enclosing subgraphs, F=178, GLOBAL batch 4096 split evenly over the ranks",
                 l2="every step streams a fresh batch whose working set (tens of GB) exceeds the 126 MB L2"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock + clock-event (throttle) reasons sampled while the timed region runs: NVML every
    5 ms when pynvml is importable, else one nvidia-smi query every 200 ms."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self._stop_ev = index, threading.Event()
        self.sm, self.mx, self.reasons, self.source = [], [], set(), "nvidia-smi"
        self.nv = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx.append(int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
            self.nv, self.source = pynvml, "nvml"
        except Exception:
            self.nv = None

    def _sample_nvml(self):
        nv = self.nv
        self.sm.append(int(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
        r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        for name, bit in (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                          ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                          ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                          ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if not out:
            return
        r = [c.strip() for c in out.split(",")]
        if r[0].isdigit():
            self.sm.append(int(r[0]))
        if r[1].isdigit():
            self.mx.append(int(r[1]))
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self._stop_ev.is_set():
            try:
                if self.nv is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop_ev.wait(0.005 if self.nv is not None else 0.2)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=6)
        return {"sm_mhz": int(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.source}


class KernelTimer:
    """CUDA-event pairs around every C-ABI call (on the launching stream); keys are
    (entry point, occurrence within the step)."""

    def __init__(self):
        self.events, self.occ, self.cur = [], {}, None

    def new_step(self):
        self.occ = {}

    def begin(self, name):
        k = self.occ.get(name, 0)
        self.occ[name] = k + 1
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        self.cur = ((name, k), s, e)

    def end(self, name):
        key, s, e = self.cur
        e.record()
        self.events.append((key, s, e))

    def summary(self):
        agg = {}
        for key, s, e in self.events:
            agg.setdefault(key, []).append(s.elapsed_time(e))
        return {k: (float(np.mean(v)), len(v)) for k, v in agg.items()}


TABLE_GEMM_ON_TC = os.environ.get("NPI_T_GEMM", "tc") != "simt"      # engine.t_gemm_tc: the V-row projection of layer 1 runs on tcgen05


# layer-1 contexts (csrc/ctx.cu): {"U": representative rows, "EU": their CSR entries, "bwd": conv1 backward per context}; set from
# Engine.ctx_counters() by the per-kernel pass.  None = layer 1 evaluated per row.
CTX = None


def note_ctx(engines_counters, bwd):
    global CTX
    cs = [c for c in engines_counters if c is not None]
    CTX = {"U": float(np.mean([c[0] for c in cs])), "EU": float(np.mean([c[1] for c in cs])), "bwd": bool(bwd)} if cs else None


def kernel_alg_bytes(key, N, E, F, B, V):
    """Algorithmic bytes of one launch (DESIGN.md 'Kernels'): every operand read once, every
    result written once, int32 = fp32 = 4 B; weights (<0.4 MB) ignored.  ``key`` = (entry point,
    occurrence within the step); forward calls come in layer order 0,1,2, backward calls 2,1,0."""
    name, k = key
    Hh = 128
    if name == "npi_gemm_nn":                        # T = table.W1 (SIMT fp32, K = F)
        return 4 * V * (F + Hh)
    if name == "npi_gemm_nn_tc":                     # tcgen05: [T = table.W1 (K = F)] | x'1.W2 | x'2.W3 | dxa3.W3^T | dxa2.W2^T
        if TABLE_GEMM_ON_TC:
            if k == 0:
                return 4 * V * (F + Hh)
            k -= 1
        M = [N[1], N[2], N[2], N[1]][k]
        return 4 * M * (Hh + Hh)
    if name == "npi_gemm_tn":                        # table^T.G (SIMT fp32, K = F)
        return 4 * V * (F + Hh)
    if name == "npi_table_grad":                     # table^T.G of a small feature table (SIMT, two launches)
        return 4 * V * (F + Hh)
    if name == "npi_gemm_tn_tc":                     # tcgen05: x'2^T.dxa3 | x'1^T.dxa2 | [table^T.G (K = F)]
        if k >= 2:
            return 4 * V * (F + Hh)
        M = [N[2], N[1]][k]
        return 4 * M * (Hh + Hh)
    if name == "npi_sage_aggregate_fwd":
        if k == 0 and CTX:                           # one row per context: table rows once, h/z/s of the representatives, their entries
            return 4 * (V * Hh + CTX["U"] * (Hh + 2)) + 4 * (CTX["EU"] + CTX["U"])
        return 4 * N[k] * (2 * Hh + 2) + 4 * (E[k] + N[k])
    if name == "npi_csr_gather_sum":                 # k = 0: class CSR (selected d_xp rows in, X out); k = 1: by node (dU in, G out)
        if k == 0:
            return 4 * (N[1] + CTX["U"]) * Hh + 16 * N[0]
        return 4 * (CTX["U"] + V) * Hh + 8 * (CTX["EU"] + CTX["U"])
    if name == "npi_ctx_finish":                     # X in, dU out, h of the representatives
        return 12 * CTX["U"] * Hh
    if name == "npi_ctx_class_pack":
        return 28 * N[0]
    if name == "npi_ctx_scatter_max":
        return 16 * B * Hh
    if name == "npi_ctx_build":                      # entries hashed and compared once, per-row records, hash table
        return 8 * E[0] + 40 * N[0]
    if name == "npi_ctx_index_build":                # two pair sorts of two passes each (read + write 8 B per item and pass), item emission
        return 40 * N[0] + 40 * (E[0] + N[0])
    if name == "npi_sage_aggregate_bwd":
        l = 2 - k
        return 4 * N[l + 1] * Hh + 4 * (E[l] + 2 * N[l]) + 4 * N[l] * Hh
    if name == "npi_entry_pack_virt":                # read col, write one packed int per entry (+ gid/dist of every node once)
        return 8 * E[0] + 5 * N[0]
    if name == "npi_entry_pack_sel":                 # read col, write {id, 1/deg} per entry (+ new_id/rowptr of every node once)
        return 12 * E[k] + 8 * N[k]
    if name == "npi_gid_reduce":
        return 4 * N[0] * Hh + 4 * V * Hh + 5 * N[0]
    if name == "npi_gid_index_build":
        return 12 * N[0]
    if name == "npi_hub_rows_build":                 # input CSR (next to the extraction), then the two filtered CSRs
        return 4 * N[min(k, 2)]
    if name == "npi_sage_fwd":                       # single-kernel variant (engine mode fused_v1)
        fin = F if k == 0 else Hh
        return 4 * N[k] * (fin + Hh + 2) + 4 * (E[k] + N[k])
    if name == "npi_sage_bwd_weight":
        l = 2 - k
        fin = F if l == 0 else Hh
        return 4 * N[l] * fin + 4 * (E[l] + N[l]) + 4 * N[l + 1] * (Hh + 1)
    if name == "npi_sage_bwd_input":
        l = 2 - k
        return 4 * N[l + 1] * Hh + 4 * (E[l] + 2 * N[l]) + 4 * N[l] * Hh
    if name == "npi_pool_gate_readout":              # per layer: gating kernel (even k), then the readout combine (odd k, aux stream)
        if k % 2:
            return 4 * B * 8 * 3 * Hh
        return 4 * N[k // 2 + 1] * (2 * Hh + 2)
    if name == "npi_pool_bwd":                       # per layer: main kernel (even k), then the partial reduce (odd k, aux stream)
        if k % 2 or (CTX and CTX["bwd"] and k == 4):  # (per-context conv1 backward: layer 1 only runs the reduce here)
            return 4 * 444 * 260
        l = 2 - k // 2
        return 4 * N[l + 1] * (3 * Hh + 4)
    if name == "npi_topk_select":
        return 4 * (2 * N[k] + 2 * N[k + 1])
    if name == "npi_filter_adj":
        return 4 * (2 * E[k] + 2 * N[k + 1] + E[k + 1])
    if name == "npi_khop_fill":
        return 4 * E[0] + 9 * N[0] + 8 * E[0]
    if name == "npi_tiny_fwd":                       # per-subgraph path: what the per-layer kernels it replaces move (projection,
        return (sum(4 * N[l] * (2 * Hh + 2) + 4 * (E[l] + N[l]) for l in range(3)) + sum(4 * N[l] * 2 * Hh for l in (1, 2))       # aggregation,
                + sum(4 * (2 * N[l] + 2 * N[l + 1]) + 4 * N[l + 1] * (2 * Hh + 2) for l in range(3))                           # top-k, gating,
                + sum(4 * (2 * E[l] + 2 * N[l + 1] + E[l + 1]) for l in range(2)))                                           # filter_adj)
    if name == "npi_tiny_weight_grads":              # x^T . dxa of the three layers over the batch rows (operands once, results once)
        return 4 * (N[0] * (F + Hh) + N[1] * 2 * Hh + N[2] * 2 * Hh) + 4 * (F + 2 * Hh) * Hh
    if name == "npi_tiny_bwd":                       # even k: the per-subgraph kernel; odd k: the partial reduce
        if k % 2:
            return 4 * 3 * B * 260
        return (sum(4 * N[l + 1] * (3 * Hh + 4) + 4 * N[l + 1] * Hh + 4 * (E[l] + 2 * N[l]) + 4 * N[l] * Hh for l in range(3))
                + sum(4 * N[l] * 2 * Hh for l in (1, 2)))
    return 0


_GEN_CACHE = {}


def generate(wl):
    from npi_gnn_b200 import synth
    key = wl["gen"]
    if key not in _GEN_CACHE:
        if key == "real":          # the reference's shipped NPInter2 fold 0, as committed under tests/golden (tools/make_golden.py)
            z = np.load(os.path.join(ROOT, "tests", "golden", "npinter2_fold0.npz"))
            _GEN_CACHE[key] = {k: z[k] for k in z.files}
        else:
            _GEN_CACHE[key] = getattr(synth, key)()
    return _GEN_CACHE[key]


def per_rank_batch(wl, world):
    if "global_batch" in wl and os.environ.get("NPI_BENCH_GLOBAL_BATCH"):      # tuning runs: e.g. one rank's share of the strong-scaling batch
        wl = dict(wl, global_batch=int(os.environ["NPI_BENCH_GLOBAL_BATCH"]))
    if "global_batch" in wl:
        if wl["global_batch"] % world:
            raise SystemExit("global batch %d does not split evenly over %d ranks" % (wl["global_batch"], world))
        return wl["global_batch"] // world
    return wl["batch"]


def build_workload(wl, device, world, rank, max_batches):
    from npi_gnn_b200 import synth
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    d = generate(wl)
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device=device)
    g.set_mask(synth.masked_pairs(d))
    pairs, y = synth.train_pairs(d)
    GB = per_rank_batch(wl, world) * world
    nb = min(len(pairs) // GB, max_batches)          # full global batches only inside the timed region
    if nb < 2:
        raise SystemExit("workload has fewer than two full global batches of %d" % GB)
    ps = PairSet(g, pairs[:nb * GB], y[:nb * GB], h=wl["hops"])
    return d, g, ps


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_run(wl, steps, warmup, batch):
    """The reference's CPU path restated (oracle/): C extraction + PyG-style collation on one core,
    stock-PyTorch fp32 forward/backward + torch.optim.Adam(L2) on all host threads."""
    from npi_gnn_b200 import synth
    from oracle import khop, khop_cwrap, net as onet
    torch.set_flush_denormal(True)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    d = generate(wl)
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    omask = khop.mask_from_keys(og, [tuple(e) for e in synth.masked_pairs(d).tolist()])
    pairs, y = synth.train_pairs(d)
    torch.manual_seed(0)
    m = onet.Net_1(d["table"].shape[1] + 1)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-3)
    m.train()

    nbat = max(1, len(pairs) // batch)

    t_extract = [0.0]

    def one(i):
        i = i % nbat                                       # small workloads: wrap around the epoch
        sl = slice(i * batch, (i + 1) * batch)
        ta = time.perf_counter()
        c = khop_cwrap.collate_batch(og, omask, pairs[sl], y[sl], wl["hops"], d["table"])
        b = onet.batch_namespace(c)
        t_extract[0] += time.perf_counter() - ta
        opt.zero_grad()
        loss = torch.nn.functional.nll_loss(m(b), b.y)
        loss.backward()
        opt.step()
        return float(loss.detach())

    for i in range(warmup):
        one(i)
    t_extract[0] = 0.0
    t0 = time.perf_counter()
    for i in range(steps):
        one(warmup + i)
    dt = time.perf_counter() - t0
    # the reference's train() iterates a dataset whose subgraphs were generated once in process(): the
    # extraction + collation share of the step is reported separately (ADVICE r01)
    return {"value": steps * batch / dt, "seconds": dt, "cores": cores, "steps": steps, "batch": batch,
            "extract_collate_seconds": t_extract[0], "value_precomputed_subgraphs": steps * batch / max(dt - t_extract[0], 1e-9)}


def cpu_scoring_run(steps, warmup, batch):
    """Eval-mode forward of the oracle on candidate pairs (src/case_study_negativeSample.py:339-355 restated)."""
    from npi_gnn_b200 import synth
    from oracle import khop, khop_cwrap, net as onet
    torch.set_flush_denormal(True)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    d = synth.npinter2_shaped()
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    omask = khop.mask_from_keys(og, [tuple(e) for e in synth.masked_pairs(d).tolist()])
    pairs = synth.all_candidate_pairs(d)
    torch.manual_seed(0)
    m = onet.Net_1(d["table"].shape[1] + 1)
    m.eval()

    def one(i):
        sl = slice(i * batch, (i + 1) * batch)
        c = khop_cwrap.collate_batch(og, omask, pairs[sl], np.zeros(batch, dtype=np.int32), 2, d["table"])
        with torch.no_grad():
            return torch.exp(m(onet.batch_namespace(c))[:, 1])

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    for i in range(steps):
        one(warmup + i)
    dt = time.perf_counter() - t0
    return {"value": steps * batch / dt, "seconds": dt, "cores": cores, "steps": steps, "batch": batch}


def load_traffic(entry_key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
    (profiles/roofline_traffic.json, written by tools/ncu_summary.py); None if it was not captured."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p))
    e = d.get("entries", {}).get(entry_key)
    return (e["dram_bytes_per_launch"], e.get("source") or d.get("source")) if e else (None, d.get("source"))


def dropin_e2e(ps, g, batch, steps, warmup, device):
    """End to end through the REFERENCE-FACING API with HOST buffers: the reference's train() loop
    (src/train_with_twoDataset.PY:46-57) with this package's drop-in classes -- a PyG-style batch
    (dense x, COO edge_index, batch, y) sits in pinned host memory, ``data.to(device)`` copies it,
    then Net_1.forward / F.nll_loss / backward / loss.item() / torch.optim.Adam.step()."""
    import torch.nn.functional as Fn
    from npi_gnn_b200.data import Batch, Data
    from npi_gnn_b200.nn import Net_1
    nbatch = 6
    host = []
    h2d = 0
    for b in range(nbatch):                      # untimed: what the reference's dataset cache holds
        bt = Batch(ps, np.arange(b * batch, (b + 1) * batch))
        t = dict(x=bt.x, edge_index=bt.edge_index, batch=bt.batch, y=bt.y)
        torch.cuda.synchronize(device)
        hb = {k: v.cpu().pin_memory() for k, v in t.items()}
        h2d = max(h2d, sum(v.numel() * v.element_size() for v in hb.values()))
        host.append(hb)
        del bt, t
    torch.manual_seed(0)
    model = Net_1(g.F).to(device)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-3)
    model.train()

    def one(i):
        hb = host[i % nbatch]
        data = Data(**{k: v.to(device, non_blocking=True) for k, v in hb.items()})
        data.num_graphs = batch
        opt.zero_grad()
        out = model(data)
        loss = Fn.nll_loss(out, data.y)
        loss.backward()
        lv = data.num_graphs * loss.item()
        opt.step()
        return lv

    for i in range(warmup):
        one(i)
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        one(warmup + i)
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1)

    # the same loop over this package's prefetching loader: the SAME pinned host batches, their copies one step ahead on
    # a copy stream (DataLoader(prefetch_device=) / PrefetchLoader); `data.to(device)` in the loop body is then a no-op
    from npi_gnn_b200.data import PrefetchLoader

    class HostLoader:
        def __init__(self, n):
            self.n = n

        def __len__(self):
            return self.n

        def __iter__(self):
            for i in range(self.n):
                hb = host[i % nbatch]
                yield Data(num_graphs=batch, **hb)

    def epoch(n):
        for data in PrefetchLoader(HostLoader(n), device):
            data = data.to(device)
            opt.zero_grad()
            out = model(data)
            loss = Fn.nll_loss(out, data.y)
            loss.backward()
            data.num_graphs * loss.item()
            opt.step()
    epoch(warmup)
    torch.cuda.synchronize(device)
    e0.record()
    epoch(steps)
    e1.record()
    torch.cuda.synchronize(device)
    ms_pf = e0.elapsed_time(e1)
    del model, opt, host
    torch.cuda.empty_cache()
    return {"value": steps * batch / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": 4, "steps": steps,
            "api": "reference train() loop on drop-in Net_1 / Data: dense x + COO edge_index + batch + y from pinned host memory "
                   "(data.to(device)), F.nll_loss, backward, loss.item(), torch.optim.Adam",
            "prefetch_value": steps * batch / (ms_pf * 1e-3), "prefetch_ms_per_step": ms_pf / steps,
            "prefetch_api": "the same loop and host batches through npi_gnn_b200.data.PrefetchLoader (what DataLoader(prefetch_device=) "
                            "uses): the H2D copy of the next batch overlaps the current step; still inside the timed region"}


def timed_steps(run_step, K, sync, flush=None):
    """K steps bracketed by barrier + synchronize; one event pair around the whole region, or
    (flush given: a buffer larger than L2 rewritten between steps) one pair per step, summed."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    if flush is None:
        e0.record()
        for i in range(K):
            run_step(i)
        e1.record()
        sync()
        return e0.elapsed_time(e1)
    pairs = []
    for i in range(K):
        flush.add_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run_step(i)
        b.record()
        pairs.append((a, b))
    sync()
    return float(sum(a.elapsed_time(b) for a, b in pairs))


def dump_outputs(dirname, arrays):
    """--dump-outputs: what the timed path computed in its last step, one float32 DIR/<name>.npy per array.  Every
    input is seeded, so two builds run with the same arguments can be compared output for output.  The arrays are
    batch-sized or the 97,602-float parameter buffer: a few MB in all."""
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), t.detach().float().cpu().numpy())


# The dominant kernel is ranked by KERNEL, as the ncu launch list groups launches: entry points that launch the same kernel
# are one family (the transposed aggregation runs under npi_sage_aggregate_bwd for layers 2-3 and under npi_csr_gather_sum
# for the two gathers of the per-context backward of layer 1).  Entry points that are a sequence of many small integer
# kernels (index building next to the extraction / on the index stream: up to 22 launches of 3-20 us each, whose CUDA-event
# time is mostly launch overhead) are listed in `kernels` but not ranked: none of their kernels is near the top of the
# launch list (profiles/r3*_launches.csv).
KERNEL_FAMILY = {"npi_sage_aggregate_bwd": "aggregate_bwd_pipe_kernel", "npi_csr_gather_sum": "aggregate_bwd_pipe_kernel"}
HELPER_ENTRY_POINTS = {"npi_ctx_index_build", "npi_ctx_build", "npi_gid_index_build", "npi_hub_rows_build", "npi_filter_adj"}


def roofline_block(summ, Nm, Em, F, B, V, peak, peak_src):
    """Roofline of the DOMINANT kernel = the C-ABI entry point with the largest summed duration over its
    launches of one step (the ncu launch list groups the same way: by kernel).  Figures are per
    launch: mean algorithmic bytes / mean duration over that entry point's launches of the step."""
    total_ms = sum(v[0] for v in summ.values())
    kernels = {"%s#%d" % k: {"ms": round(v[0], 4), "share": round(v[0] / total_ms, 4),
                              "alg_GBps": round(kernel_alg_bytes(k, Nm, Em, F, B, V) / (v[0] * 1e-3) / 1e9, 1)}
               for k, v in sorted(summ.items(), key=lambda kv: -kv[1][0])}
    by_ep = {}
    for (name, k), (ms, _) in summ.items():
        if name in HELPER_ENTRY_POINTS or (name == "npi_tiny_bwd" and k % 2):      # (odd calls of npi_tiny_bwd: the partial reduce, another kernel)
            continue
        e = by_ep.setdefault(KERNEL_FAMILY.get(name, name), {"ms": 0.0, "bytes": 0.0, "keys": []})
        e["ms"] += ms
        e["bytes"] += kernel_alg_bytes((name, k), Nm, Em, F, B, V)
        e["keys"].append("%s#%d" % (name, k))
    top, te = max(by_ep.items(), key=lambda kv: kv[1]["ms"])
    n = len(te["keys"])
    achieved = te["bytes"] / (te["ms"] * 1e-3) / 1e9
    traffic, traffic_src, got = 0.0, None, 0
    for key in te["keys"]:
        t, traffic_src = load_traffic(key)
        if t is not None:
            traffic += t
            got += 1
    roof = {"bound": "hbm", "kernel": top, "launches_per_step": n, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic / n if got == n else None, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": te["bytes"] / n, "peak_source": peak_src,
            "kernel_ms": te["ms"] / n, "kernel_share_of_step": te["ms"] / total_ms,
            "per_launch": {key: kernels[key] for key in sorted(te["keys"])}}
    return roof, kernels


# ------------------------------------------------------------------------------------------ scoring (config 5)
SCORE_METRIC = "candidate pairs scored/sec (eval forward, 2-hop enclosing subgraphs)"
SCORE_UNIT = "pairs/s"


def bench_scoring(args, world, rank, local):
    """BASELINE.json configs[4]: every RNA x protein candidate pair of the NPInter2-shaped graph
    (4,636 x 449 = 2,081,564, RNA-major), eval-mode forward with fixed random weights, contiguous
    1/N slice per GPU, no communication (src/case_study_negativeSample.py:339-355)."""
    from npi_gnn_b200 import _lib as L, dist as D, synth
    from npi_gnn_b200.engine import FlatParams, algorithmic_bytes
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    from npi_gnn_b200.trainer import Scorer
    SB = args.score_batch
    K, W = args.steps, args.warmup
    config = {"workload": "inference-only scoring of all 4636 x 449 = 2,081,564 candidate pairs of the synthetic NPInter2-shaped "
                          "graph (fold 0 masked), 2-hop, F=178, contiguous 1/N slice per GPU, %d pairs per forward" % SB,
              "hops": 2, "batch_per_gpu": SB, "parallelism": "shard%d (no communication)" % world,
              "l2": "every step streams a fresh batch whose working set exceeds the 126 MB L2"}
    if args.impl == "reference":
        if rank != 0:
            return
        steps = K
        r = cpu_scoring_run(steps, W, 200)
        print(json.dumps({"impl": "reference", "metric": SCORE_METRIC, "value": r["value"], "unit": SCORE_UNIT, "n_gpus": args.gpus,
                          "steps": steps, "warmup": W, "ms_per_step": 1e3 * r["seconds"] / steps, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": r["value"], "unit": SCORE_UNIT, "cores": r["cores"], "kind": "port",
                                           "sample": "%d eval forwards of 200 pairs (oracle)" % steps},
                          "e2e": {"value": r["value"], "unit": SCORE_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    L.load()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        D.init("nccl")
    d = synth.npinter2_shaped()
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device=device)
    g.set_mask(synth.masked_pairs(d))
    allp = synth.all_candidate_pairs(d)
    per = (len(allp) + world - 1) // world
    mine = allp[rank * per:(rank + 1) * per]
    need = (W + K) * SB
    if need > len(mine):
        raise SystemExit("--steps %d: this GPU's share of the sweep has %d batches of %d pairs, %d of them warm-up"
                         % (K, len(mine) // SB, SB, W))
    mine = mine[:need]                                        # this rank's slice, first (W+K) batches
    ps = PairSet(g, mine, np.zeros(len(mine), dtype=np.int32), h=2)
    params = FlatParams(g.F, device).init_reference(torch.Generator().manual_seed(0))
    sc = Scorer(ps, params, batch_size=SB)
    out = torch.empty(len(mine), dtype=torch.float32, device=device)
    out_h = torch.empty(len(mine), dtype=torch.float32).pin_memory()

    def sync():
        if world > 1:
            D.barrier()
        torch.cuda.synchronize(device)

    def sweep(host):
        """One pass over the (W+K) batches; returns ms of the last K (device events)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        it = sc.batches(from_host=host)
        for b, (first, cnt, logp) in enumerate(it):
            if b == W:
                sync()
                e0.record()
            torch.exp(logp[:cnt, 1], out=out[first:first + cnt])
            if host:
                out_h[first:first + cnt].copy_(out[first:first + cnt], non_blocking=True)
        e1.record()
        sync()
        return e0.elapsed_time(e1)

    sweep(False)                                             # graph capture + warm caches
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    snap = dict(L.CALL_COUNTS)
    ms = sweep(False)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        last = (W + K - 1) * SB
        dump_outputs(args.dump_outputs, {"prob": out[last:last + SB], "logp": sc.engine.logp[:SB]})
    ms = D.max_over_ranks(ms, device) if world > 1 else ms
    ms_e2e = sweep(True)
    ms_e2e = D.max_over_ranks(ms_e2e, device) if world > 1 else ms_e2e
    value = K * SB * world / (ms * 1e-3)
    if world > 1:
        D.barrier()
        import torch.distributed as tdist
        tdist.destroy_process_group()
    if rank != 0:
        return
    # per-kernel pass (eager, serialised) + launches per step
    peak, peak_src = load_peaks()
    timer = KernelTimer()
    counters, ctxc = [], []
    eng = sc.engine
    eng.serial = True
    per_step = None
    for i in range(min(args.profile_steps, W + K)):
        snap = dict(L.CALL_COUNTS)
        timer.new_step()
        L.TIMER = timer
        eng.load_pairs(ps, first=i * SB, count=SB)
        eng.forward(params, training=False)
        L.TIMER = None
        torch.cuda.synchronize(device)
        per_step = L.launches_since(snap)
        counters.append(eng.counters())
        ctxc.append(eng.ctx_counters())
    note_ctx(ctxc, False)
    summ = timer.summary()
    Nm = [float(np.mean([c[0][l] for c in counters])) for l in range(4)]
    Em = [float(np.mean([c[1][l] for c in counters])) for l in range(3)]
    roof, kernels = roofline_block(summ, Nm, Em, g.F, SB, g.num_nodes, peak, peak_src)
    step_bytes = algorithmic_bytes(Nm, Em, g.F, SB, Em[0], training=False)
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        r = cpu_scoring_run(args.cpu_steps, 1, 200)
        cpu = {"value": r["value"], "unit": SCORE_UNIT, "cores": r["cores"], "kind": "port",
               "sample": "%d eval forwards of 200 candidate pairs of the same sweep (oracle: C extraction 1 core + stock-PyTorch "
                         "fp32 forward on %d threads); %.1f s" % (args.cpu_steps, r["cores"], r["seconds"])}
    line = {"metric": SCORE_METRIC, "value": value, "unit": SCORE_UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": K * SB * world / (ms_e2e * 1e-3), "unit": SCORE_UNIT, "h2d_bytes_per_step": 4 * SB,
                    "d2h_bytes_per_step": 4 * SB, "ms_per_step": ms_e2e / K,
                    "api": "Scorer.batches(from_host=True): pair indices from pinned host memory, probabilities copied back to pinned host memory"},
            "gpu_launches": per_step * K,
            "roofline": roof,
            "step_roofline": {"algorithmic_bytes_per_step": step_bytes, "achieved_GBps": step_bytes / (ms / K * 1e-3) / 1e9,
                              "frac": step_bytes / (ms / K * 1e-3) / 1e9 / peak, "bytes_per_pair": step_bytes / SB,
                              "note": "SURVEY 8(d) extraction+gather and forward terms; the path never materialises x, so >100% is possible"},
            "batch_stats": {"N": Nm, "E": Em, "launches_per_step": per_step, "pairs_scored_per_rank": K * SB},
            "kernels": kernels, "cpu_baseline": cpu}
    print(json.dumps(line))


CPU_STEPS_DEFAULT = {"npinter2": 30, "rpi2241": 200, "x100": 3, "real_h1": 60, "real_h2": 20}


def reference_line(args, name):
    """`--impl reference`: the reference's CPU path restated (oracle/), all host threads, K timed steps after W
    warm-up steps of the same workload, config, metric and unit as our arm (a step of x100 is a 256-subgraph
    sample of the 4096-subgraph global batch -- said in `sample`; it takes seconds, so pass a small --steps)."""
    wl = WORKLOADS[name]
    BPR = per_rank_batch(wl, 1)
    cpu_batch = min(BPR, 256) if name == "x100" else BPR
    steps, warm = args.steps, args.warmup
    r = cpu_reference_run(wl, steps, warm, cpu_batch)
    world = args.gpus
    config = workload_config(wl, per_rank_batch(wl, world), world)
    return {"impl": "reference", "metric": metric_name(wl), "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": 1e3 * r["seconds"] / steps,
            "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32",
            "data": "real (shipped NPInter2)" if wl["gen"] == "real" else "synthetic", "config": config,
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                             "sample": "%d training steps of batch %d (oracle: C extraction + stock-PyTorch fp32 "
                                       "fwd/bwd/Adam, torch %s); %.1f s of %.1f s are extraction + collation"
                                       % (steps, cpu_batch, torch.__version__, r["extract_collate_seconds"], r["seconds"]),
                             "value_precomputed_subgraphs": r["value_precomputed_subgraphs"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def metric_name(wl):
    return "enclosing subgraphs/sec (train fwd+bwd, batch %d)" % (wl.get("global_batch") or wl["batch"])


def workload_config(wl, BPR, world):
    return {"workload": wl["text"], "hops": wl["hops"], "batch_per_gpu": BPR, "global_batch": BPR * world,
            "parallelism": "dp%d" % world, "l2": wl["l2"]}


def training_workload(name, args, world, rank, local, device, K, W, detail, D=None):
    """One training workload measured on this process's GPU (all ranks call it under torchrun).  detail: the
    per-kernel timing pass, the drop-in end-to-end loop and the full-size CPU sample (the bench line's own
    workload); otherwise value / e2e / step roofline / a small CPU sample (`other_workloads`)."""
    from npi_gnn_b200 import _lib as L
    from npi_gnn_b200.engine import algorithmic_bytes
    from npi_gnn_b200.trainer import Trainer
    wl = WORKLOADS[name]
    BPR = per_rank_batch(wl, world)
    GBATCH = BPR * world
    config = workload_config(wl, BPR, world)
    d, g, ps = build_workload(wl, device, world, rank, max_batches=12 if name == "x100" else 10 ** 9)
    exchange, exchange_note = None, "none (single GPU)"
    if world > 1:
        if args.exchange == "peer":
            from npi_gnn_b200 import peer
            from npi_gnn_b200.engine import param_offsets
            exchange, why = peer.make_exchange(param_offsets(g.F)[1], device)
            exchange_note = ("peer memory: rank-ordered sum over NVLink fused into the Adam kernel (npi_allreduce_adam_fused), "
                             "one CUDA graph per step") if exchange is not None else "nccl all_reduce (peer exchange unavailable: %s)" % why
        else:
            exchange_note = "nccl all_reduce between two CUDA graphs"
    tr = Trainer(ps, batch_size=BPR, world_size=world, rank=rank, allreduce=D.allreduce_sum if world > 1 else None, seed=0,
                 exchange=exchange)
    nb = tr.num_batches()
    small = name in ("rpi2241",)
    flush = torch.zeros(64 << 20, dtype=torch.float32, device=device) if small else None    # 256 MB > L2
    if flush is not None:
        config["l2"] = "a 256 MB buffer is rewritten between timed steps (L2 flush); steps timed individually and summed"

    def sync():
        if world > 1:
            D.barrier()
        torch.cuda.synchronize(device)

    for i in range(W):                                   # warm-up (includes CUDA-graph capture)
        tr.step(i % nb, next_gb=(i + 1) % nb)
    sync()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed_steps(lambda i: tr.step((W + i) % nb, next_gb=(W + i + 1) % nb), K, sync, flush)
    ms = D.max_over_ranks(ms, device) if world > 1 else ms
    clocks = sampler.stop() if rank == 0 else None
    value = K * GBATCH / (ms * 1e-3)
    if detail and rank == 0 and args.dump_outputs:       # before the end-to-end pass below trains further
        out = {"logp": tr.engine.logp[:BPR], "loss": tr.engine.loss, "params": tr.params.flat}
        if exchange is None:       # the gradient Adam applied (the peer exchange sums it inside Adam, it is never stored)
            out["grads"] = tr._grads_slot[tr.engine.slot].flat      # the slot of the last step, not of the last capture
        dump_outputs(args.dump_outputs, out)

    snap = dict(L.CALL_COUNTS)                           # launches per step, counted from an eager step
    tr._enqueue_fwd_bwd(BPR, GBATCH)
    tr._enqueue_update(GBATCH)
    per_step = L.launches_since(snap)
    sync()

    # end to end through the public API: pair indices from pinned host memory every step (H2D inside the
    # timed region) and the step's loss read back to the host (D2H)
    ms_e2e = timed_steps(lambda i: tr.step((W + i) % nb, sync_loss=True, from_host=True, next_gb=(W + i + 1) % nb), K, sync, flush)
    ms_e2e = D.max_over_ranks(ms_e2e, device) if world > 1 else ms_e2e
    e2e_value = K * GBATCH / (ms_e2e * 1e-3)
    tr.engine.check_overflow()
    if exchange is not None:
        exchange.check()
    dp_breakdown = None
    if world > 1:
        D.barrier()
        dp_breakdown = dp_breakdown_probe(ps, tr, BPR, world, rank, device, K, W, ms / K, D)
        D.barrier()
        tr.exchange = None            # the per-kernel pass below runs on rank 0 alone: local Adam
    res = {"metric": metric_name(wl), "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": ms / K, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
           "dtype": "f32", "data": "real (shipped NPInter2)" if wl["gen"] == "real" else "synthetic", "config": config,
           "gradient_exchange": exchange_note, "clocks": clocks,
           "sharding": None if world == 1 else ("every global batch dealt to the ranks by cached subgraph size (nodes + edges), equal counts"
                                                if tr.cost is not None else "contiguous slices of every global batch"),
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 4 * BPR, "d2h_bytes_per_step": 4,
                   "ms_per_step": ms_e2e / K,
                   "api": "Trainer.step(from_host=True, sync_loss=True): the batch's pair indices from pinned host memory, loss read back"},
           "gpu_launches": per_step * K}
    if dp_breakdown is not None:
        res["dp_breakdown"] = dp_breakdown
    if rank != 0:
        return None, tr, ps, g
    return res, tr, ps, g


def dp_breakdown_probe(ps, tr, BPR, world, rank, device, K, W, dp_ms_per_step, D):
    """Where the weak-scaling loss comes from (VERDICT r01 item 4): every rank re-runs ITS OWN shard of the same
    K global batches with no cross-rank exchange (a single-GPU Trainer over the rank's slices, same captured
    step), timing every step with its own CUDA-event pair.  With t[r][i] the local time of step i on rank r:
      mean_local   = mean_r mean_i t[r][i]        what a rank needs by itself
      skew_bound   = mean_i max_r t[r][i]          a perfectly cheap exchange still waits for the slowest rank
      rendezvous   = dp_ms - skew_bound            what the exchange itself (flags, peer reads, launch) costs."""
    from npi_gnn_b200.trainer import Trainer, shard_of_batch
    nb = tr.num_batches()
    mine = np.concatenate([shard_of_batch(tr.order, BPR, world, rank, gb, tr.cost)[0] for gb in range(nb)])
    loc = Trainer(ps, batch_size=BPR, seed=0, order=mine)
    nbl = loc.num_batches()
    for i in range(W):
        loc.step(i % nbl, next_gb=(i + 1) % nbl)
    torch.cuda.synchronize(device)
    D.barrier()
    ev = []
    for i in range(K):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        loc.step((W + i) % nbl, next_gb=(W + i + 1) % nbl)
        b.record()
        ev.append((a, b))
    torch.cuda.synchronize(device)
    t = np.array([a.elapsed_time(b) for a, b in ev])
    # per-step event pairs add the launch gap of a graph replay to every step: also time the K steps as one region
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        loc.step((W + i) % nbl, next_gb=(W + i + 1) % nbl)
    e1.record()
    torch.cuda.synchronize(device)
    region = e0.elapsed_time(e1) / K
    rows = D.gather_rows(t, device).numpy()                       # [world, K]
    regions = D.gather_rows([region], device).numpy()[:, 0]
    n0 = D.gather_rows(ps.n_h[mine[:(W + K) * BPR]].reshape(-1, BPR).sum(1)[W:W + K] if len(mine) >= (W + K) * BPR
                       else np.zeros(K), device).numpy()
    del loc
    torch.cuda.empty_cache()
    scale = float(regions.mean() / rows.mean())                   # per-step pairs -> back-to-back scale
    skew = float(rows.max(0).mean() * scale)
    return {"per_rank_local_ms_per_step": [float(v) for v in regions],
            "mean_local_ms": float(regions.mean()), "slowest_rank_local_ms": float(regions.max()),
            "skew_bound_ms": skew, "dp_ms_per_step": float(dp_ms_per_step),
            "rendezvous_ms": float(dp_ms_per_step - skew),
            "per_step_max_over_mean": float((rows.max(0) / rows.mean(0)).mean()),
            "n0_per_rank_mean": [float(v) for v in n0.mean(1)], "n0_max_over_mean_per_step": float((n0.max(0) / np.maximum(n0.mean(0), 1)).mean()),
            "how": "single-GPU Trainer over this rank's slices of the same global batches, no exchange; per-step CUDA-event pairs "
                   "scaled to the back-to-back region time"}


def finish_stats(res, counters, g, BPR, GBATCH, world, ms_per_step, per_step):
    from npi_gnn_b200.engine import algorithmic_bytes
    peak, _ = load_peaks()
    Nm = [float(np.mean([c[0][l] for c in counters])) for l in range(4)]
    Em = [float(np.mean([c[1][l] for c in counters])) for l in range(3)]
    step_bytes = algorithmic_bytes(Nm, Em, g.F, BPR, Em[0], training=True) * world      # whole job (rank 0's batch stats)
    res["step_roofline"] = {"algorithmic_bytes_per_step": step_bytes, "achieved_GBps": step_bytes / (ms_per_step * 1e-3) / 1e9,
                            "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / (peak * world),
                            "bytes_per_subgraph": step_bytes / GBATCH}
    res["batch_stats"] = {"N": Nm, "E": Em, "launches_per_step": per_step,
                          "nodes_per_subgraph": Nm[0] / BPR, "edges_per_subgraph": Em[0] / BPR}
    return Nm, Em


def other_training_workload(name, args, device, K, W, cpu_steps):
    """Short run of another BASELINE.json configuration on one GPU for the `other_workloads` block."""
    wl = WORKLOADS[name]
    BPR = per_rank_batch(wl, 1)
    t0 = time.perf_counter()
    res, tr, ps, g = training_workload(name, args, 1, 0, 0, device, K, W, False)
    tr.engine.serial = True
    counters = []
    for i in range(min(2, tr.num_batches())):
        tr._stage_indices(i, False)
        tr._enqueue_fwd_bwd(BPR, BPR)
        torch.cuda.synchronize(device)
        counters.append(tr.engine.counters())
    finish_stats(res, counters, g, BPR, BPR, 1, res["ms_per_step"], res["gpu_launches"] // K)
    out = {k: res[k] for k in ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "scaling", "data", "config", "e2e",
                               "gpu_launches", "step_roofline", "batch_stats")}
    if name.startswith("real"):                          # config 1 is quoted per EPOCH: time whole epochs incl. the partial batch
        tr.engine.serial = False
        tr.train_epoch()
        torch.cuda.synchronize(device)
        t1 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = tr.train_epoch()
        e1.record()
        torch.cuda.synchronize(device)
        out["epoch"] = {"pairs": len(ps), "batches": tr.num_batches(), "device_ms": e0.elapsed_time(e1),
                        "wall_ms": 1e3 * (time.perf_counter() - t1), "subgraphs_per_s": len(ps) / (e0.elapsed_time(e1) * 1e-3),
                        "loss": loss}
    if cpu_steps and not args.no_cpu_baseline:
        cpu_batch = min(BPR, 256) if name == "x100" else BPR
        r = cpu_reference_run(wl, cpu_steps, 1, cpu_batch)
        out["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                               "sample": "%d training steps of batch %d (oracle); %.1f s" % (cpu_steps, cpu_batch, r["seconds"])}
    out["seconds_total"] = round(time.perf_counter() - t0, 1)
    del tr, ps, g
    torch.cuda.empty_cache()
    return out


def train_shell_wallclock(device, epochs=50):
    """The reference's whole training script on the real NPInter2 fold 0 at h = 1 -- 50 epochs, 9 intermediate
    + 1 final evaluation of both datasets, 10 checkpoints -- next to the 1413.46 s the authors logged for it
    (reference result/1223_1/log_0.txt:29; their hardware, their stack: reported, not a same-box ratio)."""
    import tempfile
    from npi_gnn_b200 import LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory as DS, train_shell
    d = generate(WORKLOADS["real_h1"])
    cannot = set(map(tuple, np.concatenate([d["test_pos"], d["test_neg"]]).tolist()))

    def ds(pos, neg):
        pairs = np.concatenate([pos, neg])
        ys = np.concatenate([np.ones(len(pos), np.int32), np.zeros(len(neg), np.int32)])
        return DS(None, h=1, set_allInteractionKey_cannotUse=cannot,
                  arrays=dict(edges=d["edges"], is_rna=d["is_rna"], table=d["table"], pairs=pairs, y=ys))
    t0 = time.perf_counter()
    train_ds, test_ds = ds(d["train_pos"], d["train_neg"]), ds(d["test_pos"], d["test_neg"])
    t_build = time.perf_counter() - t0
    with tempfile.TemporaryDirectory() as tmp:
        a = train_shell.parse_args(["--trainingName", "bench", "--trainingDatasetName", "train", "--testingDatasetName", "test",
                                    "--fold", "0", "--epochNumber", str(epochs), "--seed", "0", "--resultRoot", tmp])
        r = train_shell.run(a, train_dataset=train_ds, test_dataset=test_ds, echo=False)
    acc, pre, sen, spe, mcc = r["final_test"]
    return {"what": "train_shell.run: %d epochs x 16,658 subgraphs (batch 200, h=1) + %d evaluations of the 16,658 training and "
                    "4,166 testing subgraphs + %d checkpoints" % (epochs, epochs // 5, epochs // 5),
            "seconds": r["seconds"], "dataset_build_seconds": t_build,
            "reference_seconds": 1413.46, "reference_source": "reference result/1223_1/log_0.txt:29 ('Time consuming', the authors' "
            "GPU machine, PyG 1.4.2; the dataset build is excluded there too)",
            "final_test": {"Accuracy": acc, "Precision": pre, "Sensitivity": sen, "Specificity": spe, "MCC": mcc},
            "reference_final_test_accuracy": 0.93519, "epoch_losses_first_last": [r["losses"][0], r["losses"][-1]]}


def node2vec_stage(args, device, reps=5):
    """SURVEY 8(f) N4 in short: the reference's node2vec stage for one fold (main.py defaults: p = q = 1, 10 walks x 80
    per node, window 5, 64 dimensions, one SGD epoch) on the real NPInter2 fold-0 training graph, phase by phase
    (CUDA events, median of `reps` after one warm-up), next to a CPU sample of the oracle restatement."""
    from npi_gnn_b200 import node2vec as n2v
    d = generate(WORKLOADS["real_h1"])
    edges = n2v.training_graph_edges(d["edges"], np.concatenate([d["test_pos"], d["test_neg"]]))
    G = n2v.Graph(edges, False, 1.0, 1.0, device=device)

    def timed(fn):
        ms, r = [], None
        for i in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(device)
            e0.record()
            r = fn()
            e1.record()
            torch.cuda.synchronize(device)
            ms.append(e0.elapsed_time(e1))
        return r, float(np.median(ms[1:]))
    _, ms_tab = timed(G.preprocess_transition_probs)
    walks, ms_walk = timed(lambda: G.simulate_walks(10, 80, seed=1))
    sg, ms_vocab = timed(lambda: n2v.SkipGram(walks, G.V, seed=1))
    _, ms_sg = timed(lambda: sg.train_epoch(0, 1, shuffle=True))
    tokens = int(sg.total)
    peak, _ = load_peaks()
    tab_bytes = 12 * (G.etab_total + G.E)                       # J (4 B) + q (8 B) per slot, written once
    res = {"what": "alias tables + 10 x 80 walks + one skip-gram epoch (negative 5, window 5, dim 64) on the real fold-0 training graph",
           "graph": {"nodes": len(G.nodes()), "csr_entries": G.E, "second_order_slots": G.etab_total},
           "alias_tables_ms": ms_tab, "alias_tables_gbs": tab_bytes / (ms_tab * 1e-3) / 1e9,
           "walks_ms": ms_walk, "value": len(walks) / (ms_walk * 1e-3), "unit": "walks/s", "walk_steps_per_s": len(walks) * 79 / (ms_walk * 1e-3),
           "vocabulary_ms": ms_vocab, "skipgram_ms": ms_sg, "skipgram_tokens_per_s": tokens / (ms_sg * 1e-3),
           "stage_ms": ms_tab + ms_walk + ms_vocab + ms_sg,
           "reference_cpu": "profiles/ref_node2vec_cpu.json (the reference's own code, build container, one core)"}
    if not args.no_cpu_baseline:
        from oracle import node2vec as on2v
        g = on2v.SortedGraph(edges)
        src_of = np.repeat(np.arange(g.V), np.diff(g.rowptr))
        rng = np.random.default_rng(0)
        es = rng.choice(len(g.col), size=400, replace=False)
        t0 = time.perf_counter()
        slots = 0
        for e in es.tolist():
            J, _q = on2v.alias_setup(on2v.edge_probs(g, int(src_of[e]), int(g.col[e]), 1.0, 1.0))
            slots += len(J)
        t_tab = time.perf_counter() - t0
        res["cpu_baseline"] = {"kind": "port", "cores": 1, "value": slots / t_tab, "unit": "alias slots/s",
                               "sample": "second-order tables of 400 random directed edges (oracle/node2vec.py, CPython like the reference); %.1f s" % t_tab,
                               "gpu_value": (G.etab_total + G.E) / (ms_tab * 1e-3)}
    return res


def scoring_sample(args, device, K, W):
    """Config 5 for `other_workloads`: the first (W+K) batches of the candidate-pair sweep on one GPU."""
    from npi_gnn_b200 import synth
    from npi_gnn_b200.engine import FlatParams, algorithmic_bytes
    from npi_gnn_b200.graph import BipartiteGraph, PairSet
    from npi_gnn_b200.trainer import Scorer
    SB = args.score_batch
    d = generate(WORKLOADS["npinter2"])
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device=device)
    g.set_mask(synth.masked_pairs(d))
    mine = synth.all_candidate_pairs(d)[:(W + K) * SB]
    if len(mine) < (W + K) * SB:
        raise ValueError("--steps %d: the sweep has only %d batches of %d pairs" % (K, len(mine) // SB, SB))
    ps = PairSet(g, mine, np.zeros(len(mine), dtype=np.int32), h=2)
    params = FlatParams(g.F, device).init_reference(torch.Generator().manual_seed(0))
    sc = Scorer(ps, params, batch_size=SB)
    out = torch.empty(len(mine), dtype=torch.float32, device=device)
    out_h = torch.empty(len(mine), dtype=torch.float32).pin_memory()

    def sweep(host):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for b, (first, cnt, logp) in enumerate(sc.batches(from_host=host)):
            if b == W:
                torch.cuda.synchronize(device)
                e0.record()
            torch.exp(logp[:cnt, 1], out=out[first:first + cnt])
            if host:
                out_h[first:first + cnt].copy_(out[first:first + cnt], non_blocking=True)
        e1.record()
        torch.cuda.synchronize(device)
        return e0.elapsed_time(e1)
    sweep(False)
    ms = sweep(False)
    ms_e2e = sweep(True)
    sc.engine.check_overflow()
    eng = sc.engine
    eng.serial = True
    eng.load_pairs(ps, first=0, count=SB)
    eng.forward(params, training=False)
    Nn, En = eng.counters()
    peak, _ = load_peaks()
    sb = algorithmic_bytes(Nn, En, g.F, SB, En[0], training=False)
    res = {"metric": SCORE_METRIC, "value": K * SB / (ms * 1e-3), "unit": SCORE_UNIT, "steps": K, "warmup": W, "ms_per_step": ms / K,
           "config": {"workload": "first %d of the 2,081,564 candidate pairs of the NPInter2-shaped graph, %d per forward, eval mode" % ((W + K) * SB, SB)},
           "e2e": {"value": K * SB / (ms_e2e * 1e-3), "unit": SCORE_UNIT, "h2d_bytes_per_step": 4 * SB, "d2h_bytes_per_step": 4 * SB},
           "step_roofline": {"algorithmic_bytes_per_step": sb, "frac": sb / (ms / K * 1e-3) / 1e9 / peak}}
    if not args.no_cpu_baseline:
        r = cpu_scoring_run(15, 1, 200)
        res["cpu_baseline"] = {"value": r["value"], "unit": SCORE_UNIT, "cores": r["cores"], "kind": "port",
                               "sample": "15 eval forwards of 200 candidate pairs (oracle); %.1f s" % r["seconds"]}
    del sc, ps, g
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="npinter2", choices=sorted(WORKLOADS) + ["scoring"],
                    help="npinter2 = BASELINE.json configs[1] (the bench line); real_h1 / real_h2 = configs[0] (shipped NPInter2 "
                         "fold 0); rpi2241 / x100 / scoring = configs[2] / [3] / [4]")
    ap.add_argument("--cpu-steps", type=int, default=None, help="CPU-baseline sample size in steps (default: ~10-30 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-steps", type=int, default=8)
    ap.add_argument("--no-dropin", action="store_true", help="skip the drop-in-API end-to-end measurement")
    ap.add_argument("--no-others", action="store_true", help="skip the short runs of the other BASELINE.json configurations")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: gradient sum over peer memory fused into Adam (default) or an NCCL all-reduce")
    ap.add_argument("--score-batch", type=int, default=2048, help="scoring workload: candidate pairs per forward")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32): the log-probabilities "
                         "of the batch, its loss, the gradient and the updated parameters (scoring: the batch's probabilities "
                         "and log-probabilities).  Under --gpus > 1: rank 0's share of the batch and loss, the summed gradient, "
                         "no gradient with the peer exchange")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "scoring":
        if args.cpu_steps is None:
            args.cpu_steps = 60
        return bench_scoring(args, world, rank, local)
    name = args.workload
    wl = WORKLOADS[name]
    if args.cpu_steps is None:
        args.cpu_steps = CPU_STEPS_DEFAULT[name]

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(reference_line(args, name)))
        return

    # ------------------------------------------------------------------ our arm
    from npi_gnn_b200 import _lib as L, dist as D
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    L.load()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        D.init("nccl")
    BPR = per_rank_batch(wl, world)
    GBATCH = BPR * world
    K, W = args.steps, args.warmup
    line, tr, ps, g = training_workload(name, args, world, rank, local, device, K, W, True, D)
    if world > 1:
        import torch.distributed as tdist
        tdist.destroy_process_group()
    if rank != 0:
        return
    nb = tr.num_batches()
    dropin = None
    if world == 1 and not args.no_dropin and name != "x100":
        dropin = dropin_e2e(ps, g, BPR, K, W, device)
    line["e2e"]["dropin_value"] = dropin["value"] if dropin else None
    line["e2e"]["dropin_prefetch_value"] = dropin["prefetch_value"] if dropin else None
    line["e2e"]["dropin"] = dropin

    # ---- per-kernel timing pass (eager, CUDA events on the launching stream) + roofline
    peak, peak_src = load_peaks()
    timer = KernelTimer()
    counters, ctxc = [], []
    tr.engine.serial = True          # isolated per-kernel times: no concurrent branches in this pass
    P = min(args.profile_steps, nb)
    for i in range(P):
        tr._stage_indices((W + i) % nb, False)
        timer.new_step()
        L.TIMER = timer
        tr._enqueue_fwd_bwd(BPR, GBATCH)
        tr._enqueue_update(GBATCH)
        L.TIMER = None
        torch.cuda.synchronize(device)
        counters.append(tr.engine.counters())
        ctxc.append(tr.engine.ctx_counters())
    note_ctx(ctxc, tr.engine.ctx_bwd)
    summ = timer.summary()
    Nm, Em = finish_stats(line, counters, g, BPR, GBATCH, world, line["ms_per_step"], line["gpu_launches"] // K)
    if CTX:
        line["batch_stats"]["layer1_contexts"] = {"rows": Nm[0], "unique": CTX["U"], "entries_in_unique": CTX["EU"], "entries": Em[0],
                                                  "backward_per_context": CTX["bwd"]}
    roof, kernels = roofline_block(summ, Nm, Em, g.F, BPR, g.num_nodes, peak, peak_src)
    line["roofline"] = roof
    line["kernels"] = kernels

    cpu = None
    cpu_batch = min(BPR, 256) if name == "x100" else BPR
    if not args.no_cpu_baseline and world == 1:
        r = cpu_reference_run(wl, args.cpu_steps, 1, cpu_batch)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
               "sample": "%d training steps of batch %d on the same workload (oracle: C extraction 1 core + stock-PyTorch "
                         "fp32 fwd/bwd/Adam on %d threads); %.1f s, of which %.1f s extraction + collation (1 core)"
                         % (args.cpu_steps, cpu_batch, r["cores"], r["seconds"], r["extract_collate_seconds"]),
               "value_precomputed_subgraphs": r["value_precomputed_subgraphs"],
               "note": "value includes per-step extraction + collation like our arm; value_precomputed_subgraphs is the model "
                       "step alone on pre-extracted subgraphs (what the reference's train() loop does after process())"}
    line["cpu_baseline"] = cpu

    # ---- the other BASELINE.json configurations in short (N = 1, the default bench line only)
    if world == 1 and name == "npinter2" and not args.no_others:
        del tr, ps
        torch.cuda.empty_cache()
        others = {}
        for nm, cs in (("real_h1", 40), ("real_h2", 10), ("rpi2241", 100), ("x100", 1)):     # cs: CPU-sample steps
            try:
                others[nm] = other_training_workload(nm, args, device, K, W, cs)
            except Exception as ex:                      # a failing side workload must not take the bench line down
                others[nm] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        try:
            others["scoring"] = scoring_sample(args, device, K, W)
        except Exception as ex:
            others["scoring"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        try:
            others["train_shell_real_h1"] = train_shell_wallclock(device)
        except Exception as ex:
            others["train_shell_real_h1"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        try:
            others["node2vec_stage"] = node2vec_stage(args, device)
        except Exception as ex:
            others["node2vec_stage"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        line["other_workloads"] = others
    print(json.dumps(line))


if __name__ == "__main__":
    main()
