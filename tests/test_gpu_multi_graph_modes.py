"""Two-GPU sharded solve of the whole-frame graph modes and the l1 RPCA vs the single-GPU solve (skipped on a one-GPU box; the
CPU-side choreography is covered by tests/test_dist_gloo_graph_modes.py, the frame blocks by tests/test_gpu_sharded_graph.py)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_two_rank_nccl_graph_modes_match_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29521", os.path.join(ROOT, "scripts", "check_sharded_modes.py")]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
