"""Host-side parts of the top-k recovered edges that need no GPU: precision / recall at k against a numpy set computation,
the argument checks that run before any device work, and the command line's --topk flag."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch


def _numpy_pr(rows, cols, edges, n):
    true = {(min(a, b), max(a, b)) for a, b in edges if a != b}
    pred = [(min(a, b), max(a, b)) for a, b in zip(rows, cols)]
    hits = sum(p in true for p in pred)
    return hits / len(pred), hits / len(true)


def test_precision_recall_at_k_matches_sets():
    from mcgra_b200.metrics import precision_recall_at_k
    rng = np.random.RandomState(0)
    n = 60
    edges = rng.randint(0, n, (300, 2))                      # duplicates, both orientations and self-loops included
    iu, ju = np.triu_indices(n, 1)
    pick = rng.choice(len(iu), 150, replace=False)
    rows, cols = iu[pick], ju[pick]
    want = _numpy_pr(rows, cols, edges, n)
    assert precision_recall_at_k(torch.from_numpy(rows), torch.from_numpy(cols), edges, n) == want
    assert precision_recall_at_k(rows, cols, torch.from_numpy(edges), n) == want
    A = sp.coo_matrix((np.ones(len(edges)), (edges[:, 0], edges[:, 1])), shape=(n, n))
    assert precision_recall_at_k(rows, cols, A, n) == want
    coo = torch.sparse_coo_tensor(torch.from_numpy(edges.T.copy()), torch.ones(len(edges)), (n, n))
    assert precision_recall_at_k(rows, cols, coo, n) == want
    assert precision_recall_at_k(rows[:0], cols[:0], edges, n) == (0.0, 0.0)
    with pytest.raises(ValueError):
        precision_recall_at_k(rows, cols, np.array([[0, n]]), n)


def test_topk_argument_checks_before_device_work():
    from mcgra_b200.metrics import topk_pairs
    S = torch.zeros(5, 5)
    for k in (-1, 11):
        with pytest.raises(ValueError, match="outside"):
            topk_pairs(S, k)
    with pytest.raises(ValueError, match="square"):
        topk_pairs(torch.zeros(5, 4), 1)
    r, c, s = topk_pairs(S, 0)
    assert r.shape == c.shape == s.shape == (0,) and r.dtype == torch.int64 and s.dtype == torch.float32


def test_recovered_edges_needs_attack():
    from mcgra_b200.topology_attack import PGDAttack
    m = PGDAttack(model=None, nnodes=4, device="cpu")
    with pytest.raises(RuntimeError, match="attack"):
        m.recovered_edges(2)


def test_cli_topk_flag():
    from mcgra_b200.main import build_parser
    assert build_parser().parse_args([]).topk == 0
    assert build_parser().parse_args(["--topk", "1000"]).topk == 1000
