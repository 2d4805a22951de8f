"""The defended victim end to end: the CSR kernels of the defended training (mcgra_spmm_csr against fp64, mcgra_gram_auc_stage
bit-equal to the dense link AUROC, on one call and on row bands), `mcgpb_gcn.GCN.fit` on a sparse adjacency (reference
replay, agreement with the dense input, memory), and `main.py --defense` on one process and on three ranks."""
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch
from scipy.stats import rankdata

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
DEV = torch.device("cuda:0")


def _csr_tensors(A):
    A = sp.csr_matrix(A)
    A.sort_indices()
    return (torch.from_numpy(A.indptr.astype(np.int64)).to(DEV), torch.from_numpy(A.indices.astype(np.int32)).to(DEV),
            torch.from_numpy(A.data.astype(np.float32)).to(DEV))


def _random_sym(n, deg, rng, hub=None, isolated=0):
    """Symmetric 0/1 adjacency without self-loops; `hub`: a node joined to that many others; the last `isolated` nodes
    have no edges."""
    m = max(n - isolated, 1)
    e = rng.randint(0, m, size=(n * deg // 2, 2))
    if hub is not None:
        e = np.concatenate([e, np.stack([np.zeros(hub, np.int64), rng.choice(np.arange(1, m), hub, replace=False)], 1)])
    e = e[e[:, 0] != e[:, 1]]
    A = sp.coo_matrix((np.ones(len(e)), (e[:, 0], e[:, 1])), shape=(n, n)).tocsr()
    A = ((A + A.T) > 0).astype(np.float64)
    return sp.csr_matrix(A)


# ---- mcgra_spmm_csr --------------------------------------------------------------------------------------------------
def _spmm(rowptr, cols, vals, B):
    from mcgra_b200._native import call, ptr, stream_ptr
    Y = torch.empty_like(B)
    call("mcgra_spmm_csr", ptr(rowptr), ptr(cols), ptr(vals), rowptr.numel() - 1, ptr(B), B.shape[1], ptr(Y), stream_ptr())
    return Y


@pytest.mark.parametrize("K", [16, 32])
@pytest.mark.parametrize("n", [1, 31, 700, 20000])
def test_spmm_csr_against_fp64(n, K):
    rng = np.random.RandomState(n + K)
    if n == 1:
        A = sp.csr_matrix(np.array([[0.75]]))
    else:
        # self-loops as entries, empty rows, and at n = 20 000 a row of degree 1 500
        A = _random_sym(n, 6, rng, hub=1500 if n >= 20000 else None, isolated=n // 10)
        A = A + sp.diags(np.where(np.arange(n) % 3 == 0, 1.0, 0.0))
        A = sp.csr_matrix(A.multiply(rng.uniform(0.1, 1.0, size=A.shape[0])[:, None]))
        A.eliminate_zeros()
    assert n < 20000 or np.diff(A.indptr).max() > 1000
    assert n == 1 or (np.diff(A.indptr) == 0).any()
    rowptr, cols, vals = _csr_tensors(A)
    B = torch.from_numpy(rng.standard_normal((n, K)).astype(np.float32)).to(DEV)
    Y = _spmm(rowptr, cols, vals, B)
    A64 = sp.csr_matrix((vals.cpu().numpy().astype(np.float64), A.indices, A.indptr), shape=A.shape)
    ref = A64 @ B.cpu().numpy().astype(np.float64)
    got = Y.cpu().numpy().astype(np.float64)
    rel = np.linalg.norm(got - ref) / max(np.linalg.norm(ref), 1e-300)
    print(f"[spmm] n={n} K={K}: relative error {rel:.2e}")
    assert rel <= 1e-6
    absbound = abs(A64) @ np.abs(B.cpu().numpy().astype(np.float64))     # per entry: |A| |B| scale of the sum
    assert np.all(np.abs(got - ref) <= 1e-5 * absbound + 1e-30)
    assert torch.equal(Y, _spmm(rowptr, cols, vals, B))                  # fixed summation order: bit-identical rerun


# ---- mcgra_gram_auc_stage ---------------------------------------------------------------------------------------------
def _gram_auc_bands(Z, rowptr, cols, bands):
    """mcgra_gram_auc_stage on row bands combined as metrics._auc_ap_sharded combines ranks: the positives' keys
    gathered, the counts summed.  Returns (auc, ap, npos, nneg)."""
    from mcgra_b200 import _native as N
    from mcgra_b200._native import call, ptr, stream_ptr
    n, d = Z.shape
    npos = max(int(cols.numel()), 1)
    wsb = N.lib().mcgra_gram_auc_workspace_bytes(npos)
    ho = int(N.lib().mcgra_auc_hist_offset(npos))
    out = torch.zeros(4, dtype=torch.float64, device=DEV)
    st = stream_ptr()
    wss = [torch.zeros(wsb, dtype=torch.uint8, device=DEV) for _ in bands]
    keys = []
    for ws, (r0, r1) in zip(wss, bands):
        call("mcgra_gram_auc_stage", 0, ptr(Z), d, n, ptr(rowptr), ptr(cols), r0, r1, npos, ptr(ws), ptr(out), st)
        c = int(ws[:8].view(torch.int64).item())
        keys.append(ws[256:256 + 4 * c].clone())
    allk = torch.cat(keys)
    for ws in wss:
        ws[256:256 + allk.numel()] = allk
        ws[:8].view(torch.int64).fill_(allk.numel() // 4)
    hist = torch.zeros(npos + 2, dtype=torch.int64, device=DEV)
    sums = torch.zeros(2, dtype=torch.int64, device=DEV)
    for ws, (r0, r1) in zip(wss, bands):
        call("mcgra_gram_auc_stage", 1, ptr(Z), d, n, ptr(rowptr), ptr(cols), r0, r1, npos, ptr(ws), ptr(out), st)
        hist += ws[ho:ho + 8 * (npos + 2)].view(torch.int64)
        sums += ws[8:24].view(torch.int64)
    ws = wss[0]
    ws[ho:ho + 8 * (npos + 2)].view(torch.int64).copy_(hist)
    ws[8:24].view(torch.int64).copy_(sums)
    call("mcgra_gram_auc_stage", 2, ptr(Z), d, n, ptr(rowptr), ptr(cols), 0, n, npos, ptr(ws), ptr(out), st)
    return out.cpu().numpy()


def _auc_fp64(Z, A):
    """sklearn's roc_auc_score restated in fp64: the Mann-Whitney statistic with average ranks for ties, over the fp32
    scores relu(Z Z^T - I) as mcgra_gram_accumulate forms them."""
    from mcgra_b200._native import call, ptr, stream_ptr
    n, d = Z.shape
    S = torch.zeros(n, n, dtype=torch.float32, device=DEV)
    call("mcgra_gram_accumulate", ptr(Z), d, n, 1, None, ptr(S), n, 0, n, stream_ptr())
    s = S.cpu().numpy().reshape(-1).astype(np.float64)
    y = (A.toarray() != 0).reshape(-1)
    r = rankdata(s)
    P, Nn = int(y.sum()), int((~y).sum())
    return (r[y].sum() - P * (P + 1) / 2.0) / (P * Nn)


def _gram_cases():
    rng = np.random.RandomState(3)
    cases = []
    for n in (300, 2000):
        for d in (16, 7):           # 7: the width of a class-logit layer (scalar operand loads)
            cases.append((f"random_n{n}_d{d}", rng.standard_normal((n, d)) * 0.4, _random_sym(n, 5, rng)))
    Z = rng.standard_normal((40, 16)) * 0.5
    cases.append(("duplicate_rows", Z[rng.randint(0, 40, size=500)], _random_sym(500, 6, rng)))
    Z = rng.standard_normal((800, 16))
    Z[:, 0] = np.where(np.arange(800) % 2 == 0, 3.0, -3.0)        # half of all inner products far below 0: ties at 0
    cases.append(("negative_products", Z * 0.5, _random_sym(800, 5, rng)))
    cases.append(("isolated_nodes", rng.standard_normal((600, 16)) * 0.4, _random_sym(600, 5, rng, isolated=150)))
    return cases


@pytest.mark.parametrize("name,Z,A", _gram_cases(), ids=[c[0] for c in _gram_cases()])
def test_gram_auc_matches_link_auc(name, Z, A):
    from mcgra_b200 import mcgpb_gcn as G
    n = A.shape[0]
    Zt = torch.from_numpy(Z.astype(np.float32)).to(DEV).contiguous()
    rowptr, cols, _ = _csr_tensors(A)
    labels = torch.from_numpy((A.toarray() != 0).astype(np.uint8)).to(DEV)
    dense = G.link_auc(Zt, labels)
    coo = torch.from_numpy(np.vstack([A.tocoo().row, A.tocoo().col]).astype(np.int64))
    csr = G.Csr(torch.sparse_coo_tensor(coo, torch.ones(coo.shape[1]), (n, n)).to(DEV))
    sparse = G.link_auc(Zt, csr)
    ref = _auc_fp64(Zt, A)
    print(f"[gram-auc] {name}: dense {dense!r} csr {sparse!r} fp64 {ref!r}")
    assert sparse == dense
    assert abs(sparse - ref) <= 1e-12
    one = _gram_auc_bands(Zt, rowptr, cols, [(0, n)])
    bands = _gram_auc_bands(Zt, rowptr, cols, [(0, n // 3), (n // 3, n // 3 + 7), (n // 3 + 7, n)])
    assert one[0] == sparse
    assert np.array_equal(one, bands)
    assert int(one[2]) == A.nnz and int(one[3]) == n * n - A.nnz


# ---- defended training on a sparse adjacency --------------------------------------------------------------------------
def _fit(d, mi, adj, **kw):
    from mcgra_b200.mcgpb_gcn import GCN
    f, c = d["X"].shape[1], int(d["labels"].max()) + 1
    model = GCN(nfeat=f, nclass=c, nhid=16, nlayer=2, dropout=0.0, weight_decay=5e-4, device=DEV).to(DEV)
    for layer in model.gc:
        layer.to(DEV)
    model.load_state_dict({k[5:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("init_")})
    beta = {str(k): float(v) for k, v in zip(d["beta_keys"], d["beta_vals"])}
    res = model.fit(torch.from_numpy(d["X"]), adj, torch.from_numpy(d["labels"]), d["idx_train"], d["idx_val"],
                    d["idx_test"], train_iters=int(d["epochs"]), initialize=False, beta=beta, MI_type=mi, plain_acc=0.7,
                    pair_draws=d["pair_draws"], **kw)
    return model, res


@pytest.mark.parametrize("mi", ["linear_HSIC", "linear_CKA", "DP"])
def test_sparse_fit_replays_reference_and_dense(mi):
    from mcgra_b200.mcgpb_gcn import SparseAdjacency
    d = np.load(os.path.join(GOLDEN, f"mcgpb_fit_{mi}_n300.npz"))
    adj = torch.from_numpy(d["adj"].astype(np.float32))
    model, res = _fit(d, mi, adj.to_sparse())
    assert isinstance(model.adj_norm, SparseAdjacency)
    got, ref = np.array(res["full_losses"]), d["full_losses"]
    rel = np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-12))
    print(f"[mcgpb-fit sparse] {mi}: max rel err vs reference {rel:.3e}")
    assert rel < 2e-3                          # the bounds of test_gpu_mcgpb.test_defended_fit_replays_reference
    np.testing.assert_allclose(res["IAZ"].numpy(), d["IAZ"], atol=1e-4)
    np.testing.assert_allclose(res["IYZ"].numpy(), d["IYZ"], atol=1e-6)
    np.testing.assert_allclose(np.asarray(res["final_layer_aucs"], dtype=np.float64), d["final_layer_aucs"], atol=1e-4)
    for k in d.files:
        if k.startswith("final_") and k != "final_layer_aucs":
            w = model.state_dict()[k[6:]].cpu().numpy()
            bad = np.abs(w - d[k]) > 2e-4 * max(1.0, np.max(np.abs(d[k])))
            assert bad.mean() < 0.02 and np.max(np.abs(w - d[k])) <= 0.031, k
    smodel, sres = _fit(d, mi, sp.csr_matrix(d["adj"]))      # a scipy adjacency takes the same CSR path
    assert isinstance(smodel.adj_norm, SparseAdjacency)
    srel = np.max(np.abs(np.array(sres["full_losses"]) - got) / np.maximum(np.abs(got), 1e-12))
    assert srel < 1e-5
    np.testing.assert_allclose(sres["IAZ"].numpy(), res["IAZ"].numpy(), atol=1e-6)
    dmodel, dres = _fit(d, mi, adj)            # dense input: the tiled path
    drel = np.max(np.abs(got - np.array(dres["full_losses"])) / np.maximum(np.abs(np.array(dres["full_losses"])), 1e-12))
    print(f"[mcgpb-fit sparse] {mi}: max rel difference to the dense input {drel:.3e}")
    assert drel < 1e-4                         # the same computation up to fp32 summation order
    np.testing.assert_allclose(res["IAZ"].numpy(), dres["IAZ"].numpy(), atol=1e-5)
    np.testing.assert_allclose(res["IYZ"].numpy(), dres["IYZ"].numpy(), atol=1e-6)


def test_sparse_edge_drop_draws_match_dense():
    from mcgra_b200.mcgpb_gcn import GCN
    d = np.load(os.path.join(GOLDEN, "mcgpb_fit_linear_HSIC_n300.npz"))
    adj = torch.from_numpy(d["adj"].astype(np.float32))
    kept = []
    for a in (adj, adj.to_sparse()):
        m = GCN(nfeat=d["X"].shape[1], nclass=int(d["labels"].max()) + 1, nhid=16, device=DEV).to(DEV)
        torch.manual_seed(7)
        m.fit(torch.from_numpy(d["X"]), a, torch.from_numpy(d["labels"]), d["idx_train"], d["idx_val"], train_iters=1,
              stochastic=1, aug_pe=0.3)
        o = m.origin_adj
        kept.append((o.coalesce().indices().t() if o.is_sparse else o.nonzero()).cpu().numpy())
    assert 0 < len(kept[0]) < np.count_nonzero(d["adj"])
    assert np.array_equal(kept[0], kept[1])


def test_sparse_fit_memory_below_n_squared_bytes():
    from mcgra_b200 import synth
    from mcgra_b200.mcgpb_gcn import GCN
    n = 20000
    g = synth.make_graph(n, 64, 4)
    e = g["edges"]
    idx = torch.from_numpy(np.concatenate([e, e[:, ::-1]]).T.copy())
    adj = torch.sparse_coo_tensor(idx, torch.ones(idx.shape[1]), (n, n)).coalesce().to(DEV)
    X, y = torch.from_numpy(g["features"]).to(DEV), torch.from_numpy(g["labels"]).to(DEV)
    perm = np.random.RandomState(0).permutation(n)
    model = GCN(nfeat=64, nclass=4, nhid=16, device=DEV).to(DEV)
    for layer in model.gc:
        layer.to(DEV)
    beta = {"layer-0": 1e-3, "layer-1": 1e-3, "layer-2": 1e-3, "layer_inter-0": 1e-3, "layer_inter-1": 1e-3}
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    res = model.fit(X, adj, y, perm[:2000], perm[2000:4000], perm[4000:], train_iters=3, beta=beta,
                    MI_type="linear_HSIC", stochastic=1)
    peak = torch.cuda.max_memory_allocated() - base
    print(f"[mcgpb-fit sparse] n={n}: peak device memory of fit {peak / 1e6:.1f} MB (n^2 bytes = {n * n / 1e6:.0f} MB)")
    assert peak < n * n
    assert all(0.0 <= a <= 1.0 for a in res["final_layer_aucs"])


# ---- command line -----------------------------------------------------------------------------------------------------
CLI = ["--dataset", "synthetic:2000:64:4", "--w1", "0.01", "--w6", "10", "--w7", "10", "--w9", "10", "--w10", "1000",
       "--lr", "-2", "--useH_A", "--useY_A", "--useY", "--epochs", "20", "--log_name", "cli.log", "--defense",
       "--MI_type", "linear_HSIC", "--beta", "0.001,0.001,0.001,0.0001,0.0001"]
MODES = {"evaluate": ["--mode", "evaluate"], "baseline": ["--mode", "baseline", "--measure", "MSELoss"]}


def _aucs(log):
    m = re.findall(r"In attack graph: AUC=(\S+)\tIn train graph: AUC=(\S+)\tIn Whole Graph: AUC=(\S+)", log)
    assert len(m) == 1, log
    return [float(x) for x in m[0]]


def _check_defense_lines(log):
    lines = log.splitlines()
    acc = [i for i, l in enumerate(lines) if l.startswith("Defended victim: test accuracy=")]
    aucs = [i for i, l in enumerate(lines) if l.startswith("Defended victim: final layer AUROCs=")]
    auc_line = [i for i, l in enumerate(lines) if l.startswith("In attack graph: AUC=")]
    assert len(acc) == len(aucs) == 1 and acc[0] < aucs[0] < auc_line[0], log
    a = float(re.search(r"test accuracy=(\S+)", lines[acc[0]]).group(1))
    assert 0.0 < a <= 1.0
    layer = eval(lines[aucs[0]].split("=", 1)[1])
    assert len(layer) == 3 and all(0.0 <= x <= 1.0 for x in layer)


@pytest.mark.parametrize("mode", list(MODES))
def test_cli_defense_one_gpu(tmp_path, monkeypatch, mode):
    from mcgra_b200 import main as cli
    monkeypatch.chdir(tmp_path)
    seen = {}
    defend = cli._defend

    def spy(victim, *a, **k):
        seen["plain"] = {key: v.detach().clone() for key, v in victim.state_dict().items()}
        out = defend(victim, *a, **k)
        seen["defended"] = {key: v.detach().clone() for key, v in victim.state_dict().items()}
        return out
    monkeypatch.setattr(cli, "_defend", spy)
    auc = cli.main(CLI + MODES[mode])
    assert 0.5 < float(auc) <= 1.0
    log = (tmp_path / "results" / "cli.log").read_text()
    _check_defense_lines(log)
    assert 0.5 < _aucs(log)[2] <= 1.0
    assert set(seen["plain"]) == set(seen["defended"]) and any(k.startswith("gc2.") for k in seen["plain"])
    assert all(not torch.equal(seen["plain"][k], seen["defended"][k]) for k in seen["plain"])


@pytest.mark.parametrize("mode", list(MODES))
def test_cli_defense_three_ranks_gloo_matches_one_process(tmp_path, mode):
    single, multi = tmp_path / "single", tmp_path / "multi"
    single.mkdir()
    multi.mkdir()
    run = os.path.join(HERE, "cli_rank_run.py")
    args = CLI + MODES[mode]
    out = subprocess.run([sys.executable, run, str(single)] + args, cwd=single, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "3",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), run, str(multi)] + args
                         + ["--dist_backend", "gloo"], cwd=multi, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    log1 = (single / "results" / "cli.log").read_text()
    logn = (multi / "results" / "cli.log").read_text()
    _check_defense_lines(logn)
    a1, an = _aucs(log1), _aucs(logn)
    print(f"[cli --defense {mode}] AUCs one process {a1}, 3 ranks {an}")
    assert max(abs(x - y) for x, y in zip(a1, an)) <= 1e-3      # the tolerance of test_gpu_cli_mgpu
