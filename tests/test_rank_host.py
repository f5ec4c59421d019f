"""Host side of the ranking metrics: the trainer shell's --rankMetrics flag and rank line, and the shard gather that
Scorer.rank_metrics uses under data parallelism (gloo, no GPU)."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_rank_metrics_flag_and_line_format():
    from npi_gnn_b200 import train_shell as ts
    assert ts.parse_args([]).rankMetrics == 0
    assert ts.parse_args(["--rankMetrics", "1"]).rankMetrics == 1
    line = ts.rank_line("Epoch: 015, testing dataset", dict(auroc=0.987654321, ap=0.5, pr_auc_trapz=0.912345678))
    assert line == "Epoch: 015, testing dataset, AUROC: 0.98765, AP: 0.50000, PR-AUC(trapz): 0.91235"
    assert re.match(r"^result, testing dataset, AUROC: \d\.\d{5}, AP: \d\.\d{5}, PR-AUC\(trapz\): \d\.\d{5}$",
                    ts.rank_line("result, testing dataset", dict(auroc=1.0, ap=0.0, pr_auc_trapz=1.0)))


_GATHER_SCRIPT = r"""
import sys, torch
sys.path.insert(0, %r)
from npi_gnn_b200 import dist as D
world, rank, _ = D.init("gloo")
for total in (7, 8, 1, 0):
    per = (total + world - 1) // world
    lo, hi = min(total, rank * per), min(total, (rank + 1) * per)
    full = torch.arange(total, dtype=torch.int32) * 3 + 1
    got = D.gather_shards(full[lo:hi].clone(), total)
    assert torch.equal(got, full), (rank, total, got)
D.barrier()
if rank == 0:
    print("GATHER_OK")
"""


def test_gather_shards_gloo_world2(tmp_path):
    """Contiguous shards (the last one short or empty) come back as the whole vector, in order, on every rank."""
    script = tmp_path / "gather.py"
    script.write_text(_GATHER_SCRIPT % ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29633", str(script)],
                         capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "GATHER_OK" in out.stdout
