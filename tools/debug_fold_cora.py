"""Engine 2 vs engine 3 of the fold on the real-Cora 100-iteration run: AUC / AP and parameter differences."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import pgd_oracle as O
from helpers import engines, run_native_case
import test_gpu_parity_sizes as T

ds = sys.argv[1] if len(sys.argv) > 1 else "cora"
ep = int(sys.argv[2]) if len(sys.argv) > 2 else 100
r, d = T._real_case(ds, ep)
real = d["adj"].reshape(-1).astype(np.float32)
res = {}
for tag, eng in [("e2a", 2), ("e2b", 2), ("e3a", 3), ("e3b", 3)]:
    with engines({1: eng}):
        got = run_native_case(d, trace=False)
    sc = got["modified_adj"].reshape(-1)
    res[tag] = got
    print(tag, "AUC %.5f AP %.5f" % (O.roc_auc(real, sc), O.average_precision(real, sc)), "loss[-1] %.6e" % got["loss"][-1],
          "ref auc %.5f ap %.5f" % (float(r["auc_full"]), float(r["ap_full"])), flush=True)
for a, b in [("e2a", "e2b"), ("e3a", "e3b"), ("e2a", "e3a")]:
    xa, xb = res[a]["x_final"], res[b]["x_final"]
    dx = np.abs(xa - xb)
    la, lb = np.asarray(res[a]["loss"]), np.asarray(res[b]["loss"])
    print(a, b, "max|dx| %.3e  frac>1e-4 %.3e  max rel dloss %.3e at it %d" % (dx.max(), (dx > 1e-4).mean(), np.max(np.abs(la - lb) / np.abs(la)), int(np.argmax(np.abs(la - lb) / np.abs(la)))))
