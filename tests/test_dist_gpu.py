"""Multi-GPU parity as a collected test: tests/dist_gpu_worker.py under torchrun on 2 GPUs (skipped on boxes with
fewer), for the peer-memory halo exchange (host-driven and as one CUDA graph per rank) and the NCCL all-gather path."""
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:                       # noqa: BLE001
        return 0


@pytest.mark.gpu
@pytest.mark.timeout(400)
@pytest.mark.parametrize("mode", [("peer",), ("peer", "graph"), ("allgather",)])
def test_two_gpu_cycle_matches_the_oracle(mode):
    if os.environ.get("AMGB_TEST_EMU") == "1" or _ngpus() < 2:
        pytest.skip("needs two CUDA devices")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "dist_gpu_worker.py"), *mode]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=360, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:])
    assert r.returncode == 0, (r.stdout + r.stderr)[-4000:]
    assert "FAIL" not in r.stdout
