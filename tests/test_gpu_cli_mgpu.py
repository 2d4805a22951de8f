"""The command line on several ranks (`torchrun --nproc-per-node 3 -m mcgra_b200.main --dist_backend gloo ...`, every rank
on cuda:0) against the same command in one process: the logged AUCs agree, rank 0 alone writes one log block and the
top-k file, every rank returns the same AUC and top-k pairs, and no process outlives the run."""
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
RUN = os.path.join(HERE, "cli_rank_run.py")
pytestmark = pytest.mark.gpu

COMMON = ["--dataset", "synthetic:2000:64:4", "--w1", "0.01", "--w2", "0.01", "--w6", "10", "--w7", "10", "--w9", "10",
          "--w10", "1000", "--lr", "-2", "--useH_A", "--useY_A", "--useY", "--epochs", "20", "--topk", "200",
          "--log_name", "cli.log"]


def _aucs(log):
    m = re.findall(r"In attack graph: AUC=(\S+)\tIn train graph: AUC=(\S+)\tIn Whole Graph: AUC=(\S+)", log)
    assert len(m) == 1, log
    return [float(x) for x in m[0]]


def _alive(marker):
    """Processes whose command line names `marker`."""
    found = []
    for p in os.listdir("/proc"):
        if p.isdigit():
            try:
                with open(f"/proc/{p}/cmdline", "rb") as f:
                    if marker.encode() in f.read():
                        found.append(int(p))
            except OSError:
                pass
    return found


# (under noise Adam turns the reordered fp32 sums of the sharded path into full-size steps on entries whose gradient is
#  near zero, so the two runs drift apart with the number of steps: the noisy run is kept short)
@pytest.mark.parametrize("extra", [[], ["--measure", "MSELoss", "--eps", "0.01", "--epochs", "5"]],
                         ids=["HSIC", "MSELoss_eps"])
def test_cli_three_ranks_gloo_matches_one_process(tmp_path, extra):
    single, multi = tmp_path / "single", tmp_path / "multi"
    single.mkdir()
    multi.mkdir()
    args = COMMON + extra
    out = subprocess.run([sys.executable, RUN, str(single)] + args, cwd=single, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "3",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), RUN, str(multi)] + args
                         + ["--dist_backend", "gloo"], cwd=multi, capture_output=True, text=True, timeout=900)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert not _alive(str(multi)), "a process of the torchrun run is still alive"

    log1 = (single / "results" / "cli.log").read_text()
    logn = (multi / "results" / "cli.log").read_text()
    for key in ("current parameter:", "current density:", "Top-K:"):
        assert logn.count(key) == 1, logn                     # rank 0 alone writes, one block
    a1, an = _aucs(log1), _aucs(logn)
    print(f"AUCs one process {a1}, 3 ranks {an}")
    assert max(abs(x - y) for x, y in zip(a1, an)) <= 1e-3
    d1 = float(re.search(r"current density: (\S+)", log1).group(1))
    dn = float(re.search(r"current density: (\S+)", logn).group(1))
    assert abs(d1 - dn) <= 1e-3 * max(abs(d1), 1e-6)

    written = np.load(multi / "results" / "cli.log.topk.npz")
    ranks = [np.load(multi / f"rank{r}.npz") for r in range(3)]
    assert len(written["rows"]) == 200
    for r in ranks:
        assert float(r["auc_all"]) == float(ranks[0]["auc_all"]) == an[2]
        for k in ("rows", "cols", "scores"):
            assert np.array_equal(r[k], written[k])
