"""Shared helpers for the GPU parity tests: run the native attack on a golden fixture, switch kernel engines."""
import contextlib
import os
import tempfile
from copy import deepcopy

import numpy as np
import torch


class Args:
    pass


@contextlib.contextmanager
def engines(values, caps=None):
    """Run the block with the kernel engines `values` ({stage: engine}, mcgra_set_engine in include/mcgra.h) and the
    persistent-grid caps `caps` ({stage: CTAs} for stages 1 and 4).  On exit, even on failure, every stage in `values`
    gets its previous engine back and the grid caps are off."""
    from mcgra_b200 import _native as N
    L = N.lib()
    saved = {which: L.mcgra_get_engine(which) for which in values}
    try:
        for which, value in values.items():
            assert L.mcgra_set_engine(which, value) == 0, (which, value)
        for which, cap in (caps or {}).items():
            assert L.mcgra_set_engine(which, 100 + cap) == 0, (which, cap)
        yield
    finally:
        for which, value in saved.items():
            assert L.mcgra_set_engine(which, value) == 0, (which, value)
        for which in (1, 4):
            assert L.mcgra_set_engine(which, 100) == 0


def make_models(d, device):
    from mcgra_b200.models.gcn import GCN, embedding_GCN
    f = d["X"].shape[1]
    c = int(d["Wl"].shape[0])
    victim = GCN(nfeat=f, nclass=c, nhid=16, nlayer=2, dropout=0.5, weight_decay=5e-4, device=device)
    with torch.no_grad():
        victim.gc[0].weight.copy_(torch.from_numpy(d["W1"]))
        victim.gc[0].bias.copy_(torch.from_numpy(d["b1"]))
        victim.gc[1].weight.copy_(torch.from_numpy(d["W2"]))
        victim.gc[1].bias.copy_(torch.from_numpy(d["b2"]))
        victim.linear1.weight.copy_(torch.from_numpy(d["Wl"]))
        victim.linear1.bias.copy_(torch.from_numpy(d["bl"]))
    victim = victim.to(device)
    for layer in victim.gc:
        layer.to(device)
    emb = embedding_GCN(nfeat=f, nhid=16, nlayer=2, device=device)
    emb.gc = deepcopy(victim.gc)
    victim.eval()
    emb.eval()
    return victim, emb


def make_args(d):
    a = Args()
    a.max_eval = 100
    a.lr = float(d["lr_exp"])
    a.eps = float(d["eps"])
    a.measure = str(d["measure"])
    a.dataset = str(d["dataset"])
    a.useH_A, a.useY_A, a.useY = [bool(u) for u in d["use"]]
    for k in range(1, 11):
        setattr(a, f"w{k}", float(d["weights"][k - 1]))
    return a


def run_native_case(d, device="cuda:0", epochs=None, trace=True, graph=True):
    """Drive mcgra_b200.topology_attack.PGDAttack.attack exactly like main.objective does (main.py:298-307)."""
    from mcgra_b200.topology_attack import PGDAttack
    dev = torch.device(device)
    n = int(d["labels"].shape[0])
    victim, emb = make_models(d, dev)
    args = make_args(d)
    H_A = torch.from_numpy(d["H_A2"]).to(dev)
    Y_A = torch.from_numpy(d["Y_A"]).to(dev)
    model = PGDAttack(model=victim, embedding=emb, H_A=H_A, Y_A=Y_A, nnodes=n, loss_type="CE", device=dev).to(dev)
    if np.any(d["x0"] != 0):
        model.adj_changes.data = torch.from_numpy(d["x0"].copy()).to(dev)
    epochs = int(d["epochs"]) if epochs is None else epochs
    adj = torch.from_numpy(d["adj"].astype(np.float32))
    feature_adj = torch.from_numpy(d["feature_adj"])
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)   # no ./saved_data here: label_adj comes from the labels (same matrix, main.py:440-450)
        try:
            model.attack(args, None, 10 ** float(d["lr_exp"]), 0, float(d["weight_sup"]), tuple(d["weights"]),
                         feature_adj, 0, 0, 0, None, None, np.arange(min(8, n)), adj, d["X"],
                         np.zeros((n, n), np.float32), d["labels"], d["idx_attack"], int(d["num_edges"]), 0,
                         epochs=epochs, _trace=trace, _graph=graph)
        finally:
            os.chdir(cwd)
    torch.cuda.synchronize()
    L = model.engine.losses()
    return dict(loss=L["loss"], terms=L, x_iters=[x.cpu().numpy() for x in model._trace],
                x_final=model.adj_changes.data.cpu().numpy(), modified_adj=model.gather_modified_adj().cpu().numpy(),
                model=model)


def synthetic_case(n, f, c, measure="MSELoss", weights=None, lr_exp=-2.0, epochs=3, dataset="cora", seed=15,
                   x0_scale=0.3, density=1e7, use=(True, True, True), weight_sup=1.0, gain=3.0, mean_deg=4.5):
    """A fixture-shaped dict (same keys as tests/golden/attack_*.npz) for any size, targets from the oracle."""
    import pgd_oracle as O
    from mcgra_b200 import synth
    g = synth.make_graph(n, f, c, seed=seed, mean_deg=mean_deg)
    W = synth.gcn_weights(f, 16, c, seed=seed, gain=gain)
    A = synth.dense_adj(n, g["edges"])
    X = g["features"]
    Wt = {k: torch.from_numpy(v) for k, v in W.items()}
    Xt, At = torch.from_numpy(X), torch.from_numpy(A)
    rng = np.random.RandomState(seed + 77)
    P = n * (n - 1) // 2
    x0 = (rng.random_sample(P) * x0_scale * (rng.random_sample(P) < 0.5)).astype(np.float32) if x0_scale > 0 \
        else np.zeros(P, np.float32)
    wts = np.zeros(10)
    for k, v in (weights or {1: 0.01, 6: 10, 7: 10, 9: 10, 10: 1000}).items():
        wts[k - 1] = v
    idx = np.random.RandomState(seed).permutation(n).astype(np.int64)
    num_edges = int(0.5 * density * A.sum() / n ** 2 * n ** 2)
    d = dict(X=X, adj=A.astype(np.uint8), labels=g["labels"], idx_attack=idx,
             feature_adj=O.feature_adj_of(Xt, dataset).numpy(), H_A2=O.embed(Xt, At, Wt, 2).numpy(),
             Y_A=O.victim(Xt, At, Wt).numpy(), num_edges=np.int64(num_edges), epochs=np.int64(epochs),
             lr_exp=np.float64(lr_exp), eps=np.float64(0.0), weight_sup=np.float64(weight_sup), weights=wts,
             measure=np.array(measure), dataset=np.array(dataset), use=np.array(use, dtype=np.bool_), x0=x0, **W)
    return d
