"""The GraphMI attacks on row bands: the band decode kernel (mcgra_decode_band) against the tiled decode and its
expansion, the sharded attacks (tests/mgpu_graphmi_check.py under torchrun: 3 ranks over gloo on one GPU, 2 over NCCL),
and `--mode baseline` on the command line, in one process and on 3 ranks."""
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
RUN = os.path.join(HERE, "cli_rank_run.py")


# ---- without a GPU: the command line's scope -------------------------------------------------------------------
def test_cli_baseline_with_noise_raises():
    from mcgra_b200.main import main
    with pytest.raises(NotImplementedError, match="baseline"):
        main(["--mode", "baseline", "--eps", "0.1", "--dataset", "synthetic:100:8:2"])


@pytest.mark.parametrize("argv", [["--mode", "search"], ["--mode", "tune"], ["--arch", "gat"],
                                  ["--arch", "sage", "--mode", "baseline"]])
def test_cli_other_modes_still_raise(argv):
    from mcgra_b200.main import main
    with pytest.raises(NotImplementedError, match="only --arch gcn"):
        main(argv + ["--dataset", "synthetic:100:8:2"])


# ---- the kernel ------------------------------------------------------------------------------------------------
def _decode_full(z):
    """mcgra_decode_to_tiles followed by mcgra_tiles_to_dense (raw): the single-GPU GraphMI modified_adj."""
    from mcgra_b200 import _native as N
    n = z.shape[0]
    T = (n + N.TILE - 1) // N.TILE
    st = N.stream_ptr()
    tiles = torch.empty(T * (T + 1) // 2 * N.TILE * N.TILE, dtype=torch.float32, device=z.device)
    N.call("mcgra_decode_to_tiles", N.ptr(z), n, 0, T, N.ptr(tiles), st)
    out = torch.zeros(n, n, dtype=torch.float32, device=z.device)
    N.call("mcgra_tiles_to_dense", N.ptr(tiles), n, 0, T, None, 1, N.ptr(out), n, st)
    del tiles
    return out


def _decode_band(z, b0, b1, ld=None):
    from mcgra_b200 import _native as N
    n = z.shape[0]
    ld = n if ld is None else ld
    out = torch.full((max(b1 - b0, 0), ld), 7.0, dtype=torch.float32, device=z.device)
    N.call("mcgra_decode_band", N.ptr(z), n, b0, b1, N.ptr(out), ld, N.stream_ptr())
    return out


def _embedding(n, normalised, seed):
    from mcgra_b200 import _native as N
    g = torch.Generator().manual_seed(seed)
    z = (torch.randn(n, 16, generator=g) + 0.3).cuda()      # shifted: both signs of z_i . z_j, so the relu matters
    if not normalised:
        return z
    zn = torch.empty_like(z)
    N.call("mcgra_row_normalize", N.ptr(z), n, 16, 2.0, N.ptr(zn), N.stream_ptr())
    return zn


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("normalised", [True, False], ids=["normalised", "raw"])
@pytest.mark.parametrize("n", [90, 700, 1000])
def test_decode_band_bit_equal_to_tiles_expansion(n, normalised):
    z = _embedding(n, normalised, n)
    full = _decode_full(z)
    bands = [(0, n), (0, 0), (n, n), (37, 37), (0, 1), (n - 1, n), (n // 2, n // 2 + 1), (5, min(n, 261)),
             (n // 3, n)]
    for b0, b1 in bands:
        got = _decode_band(z, b0, b1)
        assert got.shape == (b1 - b0, n)
        assert torch.equal(_bits(got), _bits(full[b0:b1])), (n, b0, b1)
    # a leading dimension wider than n (rows not 16-byte aligned): the columns past n are left alone
    got = _decode_band(z, 3, min(n, 200), ld=n + 3)
    assert torch.equal(_bits(got[:, :n]), _bits(full[3:min(n, 200)]))
    assert bool((got[:, n:] == 7.0).all())
    assert float(full.diagonal().abs().max()) == 0.0 and float(full.min()) == 0.0 and float(full.max()) > 0.0


@pytest.mark.gpu
def test_decode_band_n65536_matches_full_decode_rows():
    """One band of 8 192 rows at n = 65 536 (the 17 GB expansion of the 8.6 GB tiles as reference)."""
    n, b0, b1 = 65536, 20000, 28192
    z = _embedding(n, True, 5)
    ref = _decode_full(z)[b0:b1].clone()
    torch.cuda.empty_cache()
    got = _decode_band(z, b0, b1)
    assert torch.equal(_bits(got), _bits(ref))


# ---- the sharded attacks ---------------------------------------------------------------------------------------
def _torchrun(nproc, script, *extra, cwd=None, timeout=1500):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
                           "--master-addr", "127.0.0.1", "--master-port", str(port), script, *extra],
                          capture_output=True, text=True, timeout=timeout, cwd=cwd)


def _check(nproc, *extra):
    out = _torchrun(nproc, os.path.join(HERE, "mgpu_graphmi_check.py"), *extra)
    print(out.stdout[-8000:])
    assert out.returncode == 0 and "MGPU_GRAPHMI_OK" in out.stdout, out.stdout[-4000:] + out.stderr[-3000:]


@pytest.mark.gpu
def test_graphmi_sharded_gloo_one_gpu():
    """3 ranks sharing cuda:0 over gloo: at n = 90 / 150 some ranks hold no tile rows and one no result band."""
    _check(3, "--gloo")


@pytest.mark.gpu
def test_graphmi_sharded_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _check(2)


# ---- the command line ------------------------------------------------------------------------------------------
CLI = ["--mode", "baseline", "--dataset", "synthetic:2000:64:4", "--density", "1", "--topk", "100", "--lr", "-2",
       "--epochs", "20", "--log_name", "graphmi.log"]


def _logged(log):
    m = re.findall(r"In attack graph: AUC=(\S+)\tIn train graph: AUC=(\S+)\tIn Whole Graph: AUC=(\S+)", log)
    assert len(m) == 1, log
    d = re.findall(r"current density: (\S+)", log)
    assert len(d) == 1, log
    return [float(x) for x in m[0]], float(d[0])


@pytest.mark.gpu
def test_cli_baseline_one_gpu_and_three_ranks(tmp_path):
    single, multi = tmp_path / "single", tmp_path / "multi"
    single.mkdir()
    multi.mkdir()
    out = subprocess.run([sys.executable, RUN, str(single)] + CLI, cwd=single, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    log1 = (single / "results" / "graphmi.log").read_text()
    a1, d1 = _logged(log1)
    print(f"one GPU: AUCs {a1}, density {d1}")
    assert all(0.5 < a <= 1.0 for a in a1)
    top = np.load(single / "results" / "graphmi.log.topk.npz")
    assert len(top["rows"]) == 100 and bool(np.all(np.diff(top["scores"]) <= 0))
    assert "Top-K: precision=" in log1

    out = _torchrun(3, RUN, str(multi), *CLI, "--dist_backend", "gloo", cwd=multi, timeout=900)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    logn = (multi / "results" / "graphmi.log").read_text()
    for key in ("current parameter:", "current density:", "Top-K:"):
        assert logn.count(key) == 1, logn                     # rank 0 alone writes, one block
    an, dn = _logged(logn)
    print(f"3 ranks: AUCs {an}, density {dn}")
    # attack-graph and whole-graph AUC and the density: 1e-6.  The train-graph AUC (200 nodes, 102 positive entries of
    # 40 000) moves by 2.5e-7 per reordered near-tie, and two single-GPU runs of the same build already differ by
    # 3.4e-6 there after these 20 iterations (the loop's fp32 atomics have no fixed order;
    # profiles/graphmi_cli_run_to_run.txt): it is held to 2e-5, about 80 such pairs
    assert abs(a1[0] - an[0]) <= 1e-6 and abs(a1[2] - an[2]) <= 1e-6
    assert abs(a1[1] - an[1]) <= 2e-5
    assert abs(d1 - dn) <= 1e-6 * abs(d1)
    assert len(np.load(multi / "results" / "graphmi.log.topk.npz")["rows"]) == 100
