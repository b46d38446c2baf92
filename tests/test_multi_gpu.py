"""2-GPU data-parallel PPO update == single-GPU update on the concatenated batch (needs >= 2 GPUs)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_update_matches_single_gpu(lib):
    here = os.path.dirname(os.path.abspath(__file__))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29611", os.path.join(here, "_dp_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0
