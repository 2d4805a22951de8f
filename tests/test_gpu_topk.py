"""Top-k recovered edges (metrics.topk_pairs / topk_pairs_sharded, PGDAttack.recovered_edges, main.py --topk) against a
stable numpy / torch oracle: exact indices and bit-equal scores, ties broken by the row-major index."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
KINDS = ("continuous", "quant8", "zeros", "mixed", "asym")


def scores_of(kind, n, seed=0):
    """n x n fp32 scores.  Every kind puts large values on the diagonal and, except `asym`, mirrors the upper triangle:
    a kernel that read the diagonal or the lower triangle would return them."""
    rng = np.random.RandomState(seed + n)
    if kind == "continuous":
        a = rng.standard_normal((n, n)).astype(np.float32)
    elif kind == "quant8":
        a = (rng.randint(0, 8, (n, n)) / 8.0).astype(np.float32)
    elif kind == "zeros":
        a = np.where(rng.random_sample((n, n)) < 0.9, 0.0, rng.random_sample((n, n))).astype(np.float32)
    elif kind == "mixed":
        a = rng.choice(np.array([-np.inf, -1.5, -0.0, 0.0, 0.25, 1.5, np.inf], np.float32), (n, n))
    else:
        a = rng.standard_normal((n, n)).astype(np.float32)
    if kind != "asym":
        iu, ju = np.triu_indices(n, 1)
        a[ju, iu] = a[iu, ju]                   # mirror without arithmetic: -0.0 stays -0.0
    else:
        a[np.tril_indices(n, -1)] = 1e30        # the lower triangle of an asymmetric matrix is never a candidate
    np.fill_diagonal(a, 1e30)
    return a


def oracle(a, k):
    """First k of the stable descending arg-sort of the upper-triangle values listed row-major."""
    n = a.shape[0]
    iu, ju = np.triu_indices(n, 1)
    v = a[iu, ju]
    o = np.argsort(-v, kind="stable")[:k]
    return iu[o], ju[o], v[o]


def ks_of(a):
    """k in {0, 1, a value inside a tie run, P - 1, P}."""
    n = a.shape[0]
    P = n * (n - 1) // 2
    v = np.sort(a[np.triu_indices(n, 1)])[::-1]
    inside = 1
    for q in range(1, P - 1):               # first k whose k-th and (k+1)-th values tie with the (k-1)-th
        if v[q - 1] == v[q] == v[q + 1]:
            inside = q + 1
            break
    return sorted({0, 1, inside, max(P - 1, 0), P})


def check_equal(got, a, k):
    r, c, s = (t.cpu().numpy() for t in got)
    ri, ci, si = oracle(a, k)
    assert r.dtype == np.int64 and c.dtype == np.int64 and s.dtype == np.float32 and len(r) == k
    np.testing.assert_array_equal(r, ri)
    np.testing.assert_array_equal(c, ci)
    np.testing.assert_array_equal(s.view(np.uint32), si.view(np.uint32))      # bit-equal, -0.0 included


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [2, 37, 300, 700])
def test_topk_matches_stable_oracle(n, kind):
    from mcgra_b200.metrics import topk_pairs
    a = scores_of(kind, n)
    S = torch.from_numpy(a).cuda()
    for k in ks_of(a):
        check_equal(topk_pairs(S, k), a, k)


def test_topk_unaligned_rows_and_strided_input():
    """n not a multiple of 4 (scalar loads) and a non-contiguous input (copied) give the same result."""
    from mcgra_b200.metrics import topk_pairs
    a = scores_of("quant8", 301)
    S = torch.from_numpy(a).cuda()
    check_equal(topk_pairs(S, 777), a, 777)
    big = torch.from_numpy(np.ascontiguousarray(np.pad(a, ((0, 0), (0, 3))))).cuda()
    check_equal(topk_pairs(big[:, :301], 777), a, 777)


def test_topk_rejects_bad_input():
    from mcgra_b200.metrics import topk_pairs
    a = scores_of("continuous", 50)
    S = torch.from_numpy(a).cuda()
    bad = S.clone()
    bad[3, 17] = float("nan")
    with pytest.raises(ValueError, match="NaN"):
        topk_pairs(bad, 5)
    ok = S.clone()
    ok[17, 3] = float("nan")                  # lower triangle and diagonal are not candidates
    ok[4, 4] = float("nan")
    check_equal(topk_pairs(ok, 5), a, 5)
    with pytest.raises(ValueError):
        topk_pairs(S, 50 * 49 // 2 + 1)
    with pytest.raises(ValueError):
        topk_pairs(S, -1)
    with pytest.raises(ValueError):
        topk_pairs(S[:, :49], 1)


def test_topk_at_scale_against_torch_stable_sort():
    """n = 32 768 (P = 5.4e8): quantised scores put the threshold inside a tie run of ~1.3e5 entries."""
    from mcgra_b200 import _native as N
    from mcgra_b200.metrics import topk_pairs
    n = 32768
    g = torch.Generator(device="cuda").manual_seed(7)
    S = torch.floor(torch.rand(n, n, device="cuda", generator=g) * 4096) / 4096
    mask = torch.ones(n, n, dtype=torch.bool, device="cuda").triu_(1)
    v = S[mask]
    vals, pos = torch.sort(v, descending=True, stable=True)
    del mask
    ar = torch.arange(n, device="cuda", dtype=torch.int64)
    row_start = ar * (n - 1) - ar * (ar - 1) // 2            # first triangle position of row i
    for k in (1_000_000, 5_000_000):
        p = pos[:k]
        i = torch.searchsorted(row_start, p, right=True) - 1
        j = p - row_start[i] + i + 1
        r, c, s = topk_pairs(S, k)
        assert vals[k - 1] == vals[k]                         # the threshold falls inside a tie run
        assert torch.equal(r, i) and torch.equal(c, j) and torch.equal(s, vals[:k])
        assert N.lib().mcgra_topk_workspace_bytes(n, n, k) < 0.01 * n * n * 4      # selection: O(n^2 / 8192 + bins)
        assert N.lib().mcgra_sort_workspace_bytes(k) < 24 * k + (1 << 20)           # final sort: O(k)


# ---- row bands ----------------------------------------------------------------------------------------------------------

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


BANDS = [(0, 100), (100, 100), (100, 300)]          # unequal, the middle one empty


def banded_case():
    a = scores_of("quant8", 300, seed=3)
    iu, ju = np.triu_indices(300, 1)
    v = a[iu, ju]
    tau = np.unique(v)[-2]                           # second-highest level: its ties lie in every non-empty band
    gt = int((v > tau).sum())
    ties0 = int(((v == tau) & (iu < 100)).sum())
    return a, [1, 777, gt + ties0 + 5, len(v)]        # gt + ties0 + 5: the tie run is cut inside the last band


def _band_worker(rank, world, port, backend, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank % torch.cuda.device_count() if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        from mcgra_b200.metrics import topk_pairs_sharded
        a, ks = banded_case()
        bands = BANDS if world == 3 else [(0, 150), (150, 300)]
        b0, b1 = bands[rank]
        band = torch.from_numpy(a[b0:b1]).to(dev)
        res = []
        for k in ks:
            r, c, s = topk_pairs_sharded(band, b0, 300, k)
            res.append((r.cpu().numpy(), c.cpu().numpy(), s.cpu().numpy()))
        out[rank] = res
    finally:
        dist.destroy_process_group()


def _run_bands(world, backend):
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_band_worker, args=(world, _free_port(), backend, out), nprocs=world, join=True)
    a, ks = banded_case()
    from mcgra_b200.metrics import topk_pairs
    S = torch.from_numpy(a).cuda()
    for q, k in enumerate(ks):
        want = [t.cpu().numpy() for t in topk_pairs(S, k)]
        ri, ci, si = oracle(a, k)
        np.testing.assert_array_equal(want[0], ri)
        for rank in range(world):
            got = out[rank][q]
            for g, w in zip(got, want):
                np.testing.assert_array_equal(g.view(np.uint32) if g.dtype == np.float32 else g,
                                              w.view(np.uint32) if w.dtype == np.float32 else w)


@pytest.mark.parametrize("world", [2, 3])
def test_topk_row_bands_gloo_match_whole_matrix(world):
    a, ks = banded_case()
    iu, _ = np.triu_indices(300, 1)
    v = a[np.triu_indices(300, 1)]
    tau = np.sort(v)[::-1][ks[2] - 1]
    sel_ties = np.flatnonzero(v == tau)[:ks[2] - int((v > tau).sum())]
    assert iu[sel_ties].min() < 100 <= iu[sel_ties].max()          # the selected tie run crosses a band boundary
    _run_bands(world, "gloo")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_topk_row_bands_nccl_two_gpus():
    _run_bands(2, "nccl")


# ---- end to end ---------------------------------------------------------------------------------------------------------

def test_recovered_edges_after_attack_and_precision_recall():
    from helpers import make_args, make_models, synthetic_case
    from mcgra_b200.metrics import precision_recall_at_k
    from mcgra_b200.topology_attack import PGDAttack
    d = synthetic_case(700, 32, 4, measure="KL", weights={1: 0.5, 2: 0.3, 6: 2.0, 7: 3.0, 9: 1.5, 10: 50.0}, epochs=2)
    dev = torch.device("cuda:0")
    n = 700
    victim, emb = make_models(d, dev)
    model = PGDAttack(model=victim, embedding=emb, H_A=torch.from_numpy(d["H_A2"]).to(dev),
                      Y_A=torch.from_numpy(d["Y_A"]).to(dev), nnodes=n, loss_type="CE", device=dev).to(dev)
    with pytest.raises(RuntimeError, match="attack"):
        model.recovered_edges(10)
    model.adj_changes.data = torch.from_numpy(d["x0"].copy()).to(dev)
    model.attack(make_args(d), None, 10 ** float(d["lr_exp"]), 0, float(d["weight_sup"]), tuple(d["weights"]),
                 torch.from_numpy(d["feature_adj"]), 0, 0, 0, None, None, np.arange(8),
                 torch.from_numpy(d["adj"].astype(np.float32)), d["X"], np.zeros((n, n), np.float32), d["labels"],
                 d["idx_attack"], int(d["num_edges"]), 0, epochs=2)
    a = model.modified_adj.cpu().numpy()
    A = d["adj"].astype(bool)
    true = {(i, j) for i, j in zip(*np.nonzero(np.triu(A, 1)))}
    for k in (1, 500, 2000, 20000):
        rows, cols, scores = model.recovered_edges(k)
        check_equal((rows, cols, scores), a, k)
        hits = sum((int(i), int(j)) in true for i, j in zip(rows.tolist(), cols.tolist()))
        p, r = precision_recall_at_k(rows, cols, np.argwhere(A), n)
        assert p == hits / k and r == hits / len(true)
        coo = torch.from_numpy(d["adj"].astype(np.float32)).to_sparse().cuda()
        assert precision_recall_at_k(rows, cols, coo, n) == (p, r)


def test_cli_topk_writes_pairs_and_log_line(tmp_path, monkeypatch):
    from mcgra_b200 import main as cli
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synthetic:600:48:3", "--measure", "MSELoss", "--w1", "0.01", "--w6", "10", "--w7", "10",
            "--w9", "10", "--w10", "1000", "--lr", "-2", "--useH_A", "--useY_A", "--useY", "--epochs", "5"]
    auc_off = cli.main(base + ["--log_name", "off.log"])
    auc_on = cli.main(base + ["--log_name", "on.log", "--topk", "300"])
    off = open(os.path.join("results", "off.log")).read().splitlines()
    on = open(os.path.join("results", "on.log")).read().splitlines()
    assert len(off) == 3 and not any(line.startswith("Top-K") for line in off)
    assert "topk" not in off[0]
    assert len(on) == 4 and on[3].startswith("Top-K: precision=") and " recall=" in on[3]
    assert abs(float(auc_on) - float(auc_off)) < 1e-6
    z = np.load(os.path.join("results", "on.log.topk.npz"))
    assert z["rows"].shape == (300,) and z["rows"].dtype == np.int64 and z["scores"].dtype == np.float32
    assert np.all(z["rows"] < z["cols"]) and np.all(np.diff(z["scores"]) <= 0)
    assert not os.path.exists(os.path.join("results", "off.log.topk.npz"))
