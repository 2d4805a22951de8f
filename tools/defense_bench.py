"""The defended training (mcgpb_gcn.GCN.fit with beta and MI_type) on the synthetic graphs of bench.py's shapes: ms per
epoch split into propagation, link AUROCs, penalties and the rest, and the peak device memory of the fit.  The sparse
(CSR) path runs at n = 19 717 and n = 65 536; at n = 19 717 the dense (tiled) path runs too, alternating with the sparse
one, for comparison.  Stage times are CUDA events around each native call; "rest" is the epoch time (host clock around
a synchronised fit) minus the stages.

    python tools/defense_bench.py [--epochs 200] [--rounds 2] [--out profiles/defense_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {19717: (500, 3), 65536: (512, 8)}           # bench.py workloads "pubmed" and "large": n -> (features, classes)
                                                      # (other n, the warm-up: 64 features, 4 classes)
STAGES = {"propagation": ("mcgra_spmm_csr", "mcgra_propagate"),
          "link_aurocs": ("mcgra_gram_auc_stage", "mcgra_gram_accumulate", "mcgra_auc_ap"),
          "penalties": ("mcgra_cross_moments", "mcgra_cross_moments_bwd")}
BETA = {"layer-0": 1e-3, "layer-1": 1e-3, "layer-2": 1e-3, "layer_inter-0": 1e-4, "layer_inter-1": 1e-4}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def graph(n, dev):
    from mcgra_b200 import synth
    f, c = SHAPES.get(n, (64, 4))
    g = synth.make_graph(n, f, c)
    e = g["edges"]
    idx = torch.from_numpy(np.concatenate([e, e[:, ::-1]]).T.copy())
    adj = torch.sparse_coo_tensor(idx, torch.ones(idx.shape[1]), (n, n)).coalesce().to(dev)
    return adj, torch.from_numpy(g["features"]).to(dev), torch.from_numpy(g["labels"]).to(dev), f, c


def run(n, path, epochs, dev):
    from mcgra_b200 import _native as N
    from mcgra_b200.mcgpb_gcn import GCN
    adj, X, y, f, c = graph(n, dev)
    if path == "dense":
        adj = adj.to_dense()
    perm = np.random.RandomState(0).permutation(n)
    torch.manual_seed(0)
    np.random.seed(0)
    model = GCN(nfeat=f, nclass=c, nhid=16, nlayer=2, device=dev).to(dev)
    for layer in model.gc:
        layer.to(dev)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    N.TIMERS["on"] = {}
    t0 = time.perf_counter()
    res = model.fit(X, adj, y, perm[:n // 10], perm[n // 10:n // 5], perm[n // 5:], train_iters=epochs, beta=BETA,
                    MI_type="linear_HSIC")
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    timers, N.TIMERS["on"] = N.TIMERS["on"], None
    peak = torch.cuda.max_memory_allocated() - base
    per = {}
    for stage, names in STAGES.items():
        per[stage] = sum(s.elapsed_time(e) for name in names for s, e in timers.get(name, [])) / epochs
    per["rest"] = wall / epochs - sum(per.values())
    out = {"n": n, "path": path, "epochs": epochs, "ms_per_epoch": wall / epochs,
           "ms_per_epoch_split": {k: round(v, 3) for k, v in per.items()},
           "peak_device_memory_MB_beyond_inputs": round(peak / 1e6, 1),
           "final_layer_aucs": None if res["final_layer_aucs"] is None else [float(a) for a in res["final_layer_aucs"]]}
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "defense_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("defense_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    run(2000, "sparse", 3, dev)                    # warm-up: module loads, cuBLAS / allocator set-up
    run(2000, "dense", 3, dev)
    res = {"card": card(), "note": "CUDA-event stage times per epoch; peak memory = torch.cuda.max_memory_allocated "
                                   "during fit minus what was allocated before it (graph, features)",
           "beta": BETA, "MI_type": "linear_HSIC", "runs": []}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    plan = [(19717, p) for _ in range(a.rounds) for p in ("sparse", "dense")] + [(65536, "sparse")]   # n = 19 717 alternates
    for n, path in plan:
        res["runs"].append(run(n, path, a.epochs, dev))
        with open(a.out, "w") as f:             # after every run: a cut-short session keeps what it measured
            json.dump(res, f, indent=1)
    print(f"[defense_bench] {res['card']} -> {a.out}")


if __name__ == "__main__":
    main()
