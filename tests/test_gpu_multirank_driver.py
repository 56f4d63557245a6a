"""-m gpu, needs >= 2 GPUs (skipped otherwise): sampling and metrics through DDPM_model after enable_data_parallel(),
against the same model run on one GPU.  One process per GPU under torch.distributed.run; the worker is
tests/_multirank_driver_worker.py."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("world", [2])
def test_driver_sharded_sampling_and_metrics_match_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs (have {torch.cuda.device_count()})")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "_multirank_driver_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:])
    print(r.stderr[-4000:])
    assert r.returncode == 0
    assert "MULTIRANK_DRIVER" in r.stdout
