"""MRR3 / MRR3F row-sharded over two GPUs (one process per GPU under torch.distributed.run) against the one-GPU fit of the same
data and the oracle: fixed sweeps at k = 4 and k = 20, a run to convergence, updateMu / HCS / OneVarB / MRR3F, CNT(gen) through
the centred loader with a shard that lacks a column's smallest code, emRR on four systems, and the refusals every rank takes
together (tools/mrr_dist_check.py).  Skipped where fewer than two GPUs are visible."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_mrr3_row_sharded_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    # a rank left waiting in a collective ends the subprocess at the timeout instead of hanging the suite
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29581", os.path.join(ROOT, "tools", "mrr_dist_check.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "MRR DIST CHECK OK" in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]
