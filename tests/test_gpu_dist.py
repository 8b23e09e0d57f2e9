"""N>1 on real GPUs: launches tests/dist_gpu_check.py under torchrun (one rank per GPU, NCCL) when
the box has at least two GPUs; the CPU-side sharding logic is covered by test_dist_gloo.py."""
import json
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_multi_gpu_run_equals_single_gpu_union_batch(cuda):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (one rank per GPU)")
    world = 2 if n < 4 else 4
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node",
           str(world), "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "dist_gpu_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["ok"] and line["actions_bit_identical"] and line["replica_max_minus_min"] == 0.0
