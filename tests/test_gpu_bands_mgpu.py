"""Row-band feature_adj under every measure and metric_pool_sharded (tests/mgpu_bands_check.py under torchrun): 3 ranks
sharing cuda:0 over gloo, and one rank per GPU over NCCL where there are several GPUs."""
import os
import socket
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu


def _torchrun(nproc, *extra):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(HERE, "mgpu_bands_check.py"), *extra], capture_output=True, text=True, timeout=1200)
    print(out.stdout[-6000:])
    assert out.returncode == 0 and "MGPU_BANDS_OK" in out.stdout, out.stdout[-4000:] + out.stderr[-3000:]


def test_row_bands_gloo_one_gpu():
    """3 ranks on one GPU: at n = 90 two ranks hold no tile rows and one no result band."""
    _torchrun(3, "--gloo")


def test_row_bands_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _torchrun(min(torch.cuda.device_count(), 4))
