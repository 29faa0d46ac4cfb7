"""2-GPU NCCL data-parallel equivalence (needs >= 2 CUDA devices: `python -m pytest tests/test_dp_nccl.py -m gpu` on a
machine with two; skipped on a 1-GPU machine).  The CPU-side arithmetic of the same sharding is covered by tests/test_dp_gloo.py."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dp_equivalence_two_gpus():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    with socket.socket() as s:            # a free port: a fixed one can be taken by another job on a shared host
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "dp_nccl_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stderr[-3000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("DP_NCCL_RESULT ")]
    assert line, out.stdout[-2000:]
    r = json.loads(line[-1][len("DP_NCCL_RESULT "):])
    print("DP NCCL equivalence:", r)
    # heads kernel with the GLOBAL completeness denominator: sharded + all-reduced == global batch (fp32 summation order only)
    for k, v in r["heads_64_videos"].items():
        assert v < 2e-5, (k, v)
    # whole step: per-frame work is identical on both sides; weight gradients differ by their pixel-reduction split only
    s = r["step_4_videos"]
    assert s["losses"] < 1e-5 and s["aggregate_grad"] < 1e-4 and s["worst_grad"] < 2e-3, s
