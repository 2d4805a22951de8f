"""attack() with adjacency noise (--eps != 0) on tile-row shards (world > 1, MSELoss): the scope guard without a GPU, and
tests/mgpu_eps_check.py under torchrun -- over NCCL on two GPUs, and over gloo with every rank on one GPU."""
import os
import socket
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def test_eps_sharded_scope_guard():
    from mcgra_b200.engine import HostBands, check_noise_supported
    full = torch.zeros(4, 4)
    check_noise_supported("MSELoss", 2, full, "cuda")
    check_noise_supported("MSELoss", 8, full, torch.device("cuda", 1))
    with pytest.raises(NotImplementedError, match="eps"):
        check_noise_supported("MSELoss", 2, HostBands(4, {(0, 4): full}), "cuda")
    for measure in ("KL", "HSIC", "CKA", "DP", "KDE"):
        with pytest.raises(NotImplementedError, match="eps"):
            check_noise_supported(measure, 2, full, "cuda")
    with pytest.raises(NotImplementedError, match="eps"):
        check_noise_supported("MSELoss", 2, full, "cpu")


def _torchrun(nproc, *extra):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(HERE, "mgpu_eps_check.py"), *extra], capture_output=True, text=True, timeout=900)
    print(out.stdout[-4000:])
    assert out.returncode == 0 and "MGPU_EPS_OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


@pytest.mark.gpu
def test_two_gpu_sharded_noisy_attack():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _torchrun(2)


@pytest.mark.gpu
def test_sharded_noisy_attack_gloo_one_gpu():
    """The same checks with 3 ranks sharing cuda:0 over gloo (shards of 3, 2 and 1 tile rows)."""
    _torchrun(3, "--gloo")
