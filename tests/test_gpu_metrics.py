"""GPU AUC / AP / arg-sort against sklearn-semantics oracle and the reference-generated fixture."""
import os

import numpy as np
import pytest
import torch

import pgd_oracle as O
from helpers import engines

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_auc_ap_matches_sklearn_fixture_with_ties():
    from mcgra_b200 import metrics
    fn = np.load(os.path.join(GOLDEN, "functions.npz"))
    s = torch.from_numpy(fn["auc_scores"]).cuda()
    y = torch.from_numpy(fn["auc_labels"]).cuda()
    auc, ap = metrics.roc_auc_ap(s, y)
    assert abs(auc - float(fn["auc_value"])) < 1e-12
    assert abs(ap - float(fn["ap_value"])) < 1e-12


@pytest.mark.parametrize("engine", [1, 0])
@pytest.mark.parametrize("n,ties", [(1000, False), (300000, True), (1300003, False), (2000003, False), (2500001, True),
                                    (5000011, False), (7000003, False)])
def test_auc_ap_random(n, ties, engine):
    """engine 1: distinct positive keys in dynamic shared memory -- keys + start indices + private histogram (tied cases,
    n = 1000), sampled keys + one 32-byte block per segment of 1 / 2 / 3 distinct keys (~39 000 / ~60 000 / ~150 000
    positives: n = 1.3e6, 2e6, 5e6), sampled keys + search in global memory (~210 000: n = 7e6); engine 0: the
    1024-sample kernel over the sorted positives."""
    from mcgra_b200 import metrics
    rng = np.random.RandomState(n % 1000)
    y = (rng.random_sample(n) < 0.03).astype(np.uint8)
    s = (rng.standard_normal(n) + 0.8 * y).astype(np.float32)
    if ties:
        s = np.round(s * 20) / 20
    with engines({6: engine}):
        auc, ap = metrics.roc_auc_ap(torch.from_numpy(s).cuda(), torch.from_numpy(y).cuda())
    assert abs(auc - O.roc_auc(y, s)) < 1e-10
    assert abs(ap - O.average_precision(y, s)) < 1e-10


def test_auc_edge_cases():
    from mcgra_b200 import metrics
    # all scores equal -> AUC 0.5; negative scores / negative zero / huge values keep their order
    y = torch.tensor([1, 0, 0, 1, 0], dtype=torch.uint8).cuda()
    auc, ap = metrics.roc_auc_ap(torch.zeros(5).cuda(), y)
    assert auc == 0.5 and abs(ap - 0.4) < 1e-12
    s = torch.tensor([-1e30, -3.0, -0.0, 0.0, 5e30]).cuda()
    yy = np.array([0, 1, 0, 1, 1], dtype=np.uint8)
    auc, ap = metrics.roc_auc_ap(s, torch.from_numpy(yy).cuda())
    assert abs(auc - O.roc_auc(yy, s.cpu().numpy())) < 1e-12
    assert abs(ap - O.average_precision(yy, s.cpu().numpy())) < 1e-12


@pytest.mark.parametrize("n", [5, 4096, 100001])
def test_argsort_desc_is_stable_and_bit_exact(n):
    from mcgra_b200 import metrics
    rng = np.random.RandomState(n)
    s = rng.standard_normal(n).astype(np.float32)
    s[::7] = s[0]                                  # ties: stable order must keep the lower index first
    order = metrics.argsort_desc(torch.from_numpy(s).cuda()).cpu().numpy()
    ref = np.argsort(-s.astype(np.float64), kind="stable")
    assert np.array_equal(order, ref)


def test_metric_pool_api():
    from mcgra_b200 import metrics
    d = np.load(os.path.join(GOLDEN, "attack_mse_A_n150.npz"))
    adj = torch.from_numpy(d["adj"].astype(np.float32)).cuda()
    inf = torch.from_numpy(d["modified_adj"]).cuda()
    auc = metrics.metric_pool(adj, inf, np.arange(150), None)
    assert abs(auc - float(d["auc"])) < 1e-9
    idx = np.random.RandomState(0).permutation(150)[:70]
    sub = metrics.metric_pool(adj, inf, idx, None)
    real = d["adj"][idx][:, idx].reshape(-1)
    pred = d["modified_adj"][idx][:, idx].reshape(-1)
    assert abs(sub - O.roc_auc(real, pred)) < 1e-9


@pytest.mark.parametrize("engine", [1, 0])
@pytest.mark.parametrize("n", [97, 300, 515, 1024])
def test_fused_ensemble_is_bitwise_the_sequence_of_terms(n, engine):
    """mcgra_ensemble (one pass over the n x n result) == mcgra_tiles_to_dense followed by mcgra_gram_accumulate /
    mcgra_dense_add / mcgra_label_accumulate in the same order, bit for bit (topology_attack.py:300-322)."""
    import ctypes
    from mcgra_b200 import _native as N
    from mcgra_b200._native import call, ptr
    g = torch.Generator(device="cuda").manual_seed(n)
    T = (n + N.TILE - 1) // N.TILE
    st = N.stream_ptr()
    packed = torch.rand(n * (n - 1) // 2, device="cuda", generator=g)
    tiles = torch.zeros(T * (T + 1) // 2 * N.TILE * N.TILE, device="cuda")
    call("mcgra_tril_to_tiles", ptr(packed), n, 0, T, ptr(tiles), st)
    Z1 = torch.randn(n, 16, device="cuda", generator=g)
    Z2 = torch.randn(n, 7, device="cuda", generator=g)
    rown = torch.rand(n, device="cuda", generator=g) + 0.5
    D = torch.randn(n, n, device="cuda", generator=g)
    lab = torch.randint(0, 4, (n,), device="cuda", generator=g)
    seq = torch.zeros(n, n, device="cuda")
    call("mcgra_tiles_to_dense", ptr(tiles), n, 0, T, None, 1, ptr(seq), n, st)
    call("mcgra_gram_accumulate", ptr(Z1), 16, n, 0, None, ptr(seq), n, 0, n, st)
    call("mcgra_gram_accumulate", ptr(Z2), 7, n, 1, None, ptr(seq), n, 0, n, st)
    call("mcgra_dense_add", ptr(seq), ptr(D), n * n, st)
    call("mcgra_gram_accumulate", ptr(Z1), 16, n, 2, ptr(rown), ptr(seq), n, 0, n, st)
    call("mcgra_label_accumulate", ptr(lab), n, ptr(seq), n, 0, n, st)
    ea = N.EnsembleArgs()
    spec = [(N.TERM_GRAM, Z1, 0, None), (N.TERM_GRAM, Z2, 1, None), (N.TERM_DENSE, D, 0, None),
            (N.TERM_GRAM, Z1, 2, rown), (N.TERM_LABEL, lab, 0, None)]
    for k, (kind, t, variant, rn) in enumerate(spec):
        e = ea.t[k]
        e.kind, e.variant = kind, variant
        if kind == N.TERM_GRAM:
            e.d, e.Z, e.rownorm = t.shape[1], ptr(t), ptr(rn)
        elif kind == N.TERM_DENSE:
            e.dense = ptr(t)
        else:
            e.labels = ptr(t)
    ea.nterms = len(spec)
    fused = torch.full((n, n), float("nan"), device="cuda")
    with engines({5: engine}):      # 1: one CTA per block pair (symmetric terms once), 0: one CTA per block
        call("mcgra_ensemble", ptr(tiles), n, ctypes.byref(ea), ptr(fused), n, 0, n, st)
        torch.cuda.synchronize()
    assert torch.equal(fused, seq)
