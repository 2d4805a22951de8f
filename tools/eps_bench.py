"""attack() with adjacency noise (--eps != 0) against the noise-free loop on one GPU: device-event it/s, peak device memory,
per-kernel times of the noisy stages as fractions of the HBM peak, and a 3-iteration exact-FFMA vs default-engine
comparison at the largest size with injected noise.  bench.py's synthetic inputs; --measure MSELoss runs Profile A (README
Cora weights), --measure KDE the README's Cora K = {X, Y} KDE command (w1 = 1000, w6 = 0.01, lr = 1e-3).

    python tools/eps_bench.py [--measure MSELoss|KDE] [--sizes cora,large] [--steps 10] [--out FILE]
"""
import argparse
import gc
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (the benchmark's problem builder and kernel timers)

HBM_PEAK_GBS = 7700.0      # HGX B200 data sheet, one GPU
# measure -> (weights w1..w10, lr exponent, description, default output)
MEASURES = {"MSELoss": (bench.PROFILE_A, -2.0, bench.PROFILES["A"]["flags"], "eps_bench.json"),
            "KDE": ((1000, 0, 0, 0, 0, 0.01, 0, 0, 0, 0), -3.0, "README Cora K={X,Y} KDE: w1=1000 w6=.01 lr=1e-3",
                    "eps_kde_bench.json")}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def noisy_bytes(P, n, feat, nb):
    """Compulsory HBM bytes per launch of each noisy stage (P = stored entries; a noise block is read twice: once per
    orientation; feat: the terms and gradient passes read both orientations of feature_adj (c1 under MSELoss); the KDE
    gather reads nb columns of the L plane and updates an n x nb slab)."""
    f = 8 * P if feat else 0
    return {"mcgra_noise_stage": 20 * P, "propagate32_sel": 4 * P, "propagate16_sel": 4 * P, "mcgra_noisy_terms": 8 * P + f,
            "mcgra_noisy_grad": 16 * P + f, "mcgra_fold_adam": 28 * P, "randn": 8 * P, "mcgra_slab_ahat_noisy": 12 * n * nb}


def build(wl_name, eps, steps, noise=None, measure="MSELoss"):
    from mcgra_b200 import _native as N
    dev = torch.device("cuda", 0)
    prob = bench.build_problem(bench.WORKLOADS[wl_name], dev)
    weights, lr, _, _ = MEASURES[measure]
    args = bench.make_args("A")
    args.eps, args.measure, args.lr = eps, measure, lr
    for k, w in enumerate(weights, 1):
        setattr(args, f"w{k}", w)
    atk, adj = bench.make_attack(prob, dev)
    n = prob["n"]
    kw = {} if noise is None else {"_noise": noise}
    atk.attack(args, None, 10 ** args.lr, 0, 1.0, weights, prob["feature_adj"], 0, 0, 0, None, None, None, adj,
               prob["X"], torch.zeros(1), prob["labels"], prob["idx_attack"], int(1e7 * prob["nedges"]), 0, epochs=0,
               _engine_epochs=steps + 16, _skip_finalize=True, **kw)
    del prob
    N.lib()
    return atk


def time_loop(atk, warm, steps):
    eng = atk.engine
    for _ in range(warm):
        eng.iterate()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        eng.iterate()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def kernels(atk, steps=3):
    from mcgra_b200 import _native as N
    eng = atk.engine
    N.TIMERS["on"] = {}
    for _ in range(steps):
        eng.iterate()
    torch.cuda.synchronize()
    kt, kc = bench.kernel_times(N.TIMERS["on"], float(steps))
    N.TIMERS["on"] = None
    n = eng.n
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        torch.randn((n, n), dtype=torch.float32, device=eng.dev)
    e.record()
    torch.cuda.synchronize()
    kt["randn"], kc["randn"] = s.elapsed_time(e) / steps, 1.0
    return kt, kc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--measure", default="MSELoss", choices=list(MEASURES))
    ap.add_argument("--sizes", default="cora,large")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None, help="default: profiles/eps_bench.json (MSELoss), profiles/eps_kde_bench.json (KDE)")
    a = ap.parse_args()
    if a.out is None:
        a.out = os.path.join(ROOT, "profiles", MEASURES[a.measure][3])
    if not torch.cuda.is_available():
        raise SystemExit("eps_bench needs a CUDA device")
    from mcgra_b200 import _native as N
    out = {"card": card(), "profile": MEASURES[a.measure][2], "hbm_peak_gbs_datasheet": HBM_PEAK_GBS, "sizes": {}}
    print(out["card"], flush=True)
    for wl in a.sizes.split(","):
        rec = {}
        for eps in (0.0, 0.05):
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            atk = build(wl, eps, a.steps + 8, measure=a.measure)
            ms = time_loop(atk, 2, a.steps)
            r = {"ms_per_iter": ms, "it_s": 1000.0 / ms, "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9}
            if eps != 0.0:
                n = atk.engine.n
                P = n * (n - 1) // 2
                kt, kc = kernels(atk)
                eng = atk.engine
                by = noisy_bytes(P, n, eng.nn.FLt is not None, eng.nn.nb)
                r["kernels"] = {k: {"ms": kt[k], "launches_per_iter": kc[k],
                                    **({"hbm_frac": by[k] / (kt[k] * 1e-3) / (HBM_PEAK_GBS * 1e9)} if k in by else {})}
                                for k in kt}
                r["alg_bytes_per_iter_over_P"] = sum(by[k] * kc.get(k, 0) for k in by) / P
            rec[f"eps={eps}"] = r
            print(wl, eps, json.dumps(r), flush=True)
            atk.engine = None
            del atk
            gc.collect()
        out["sizes"][wl] = rec
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    # exact-FFMA engines vs defaults on the noisy path, 3 iterations, same injected draws
    wl = a.sizes.split(",")[-1]
    res = []
    for engines in ((5, 3), (0, 0)):
        N.lib().mcgra_set_engine(0, engines[0])
        N.lib().mcgra_set_engine(1, engines[1])
        torch.cuda.empty_cache()

        def noise(t, dev=torch.device("cuda", 0)):
            g = torch.Generator(device=dev)
            g.manual_seed(1000 + t)
            n = atk.engine.n
            return torch.randn((n, n), dtype=torch.float32, device=dev, generator=g)
        atk = build(wl, 0.05, 3, noise=noise, measure=a.measure)
        atk.engine.run(3)
        res.append((atk.engine.losses()["loss"], atk.engine.packed_parameter()[:1 << 22].cpu().numpy()))
        atk.engine = None
        del atk
        gc.collect()
    N.lib().mcgra_set_engine(0, 5)
    N.lib().mcgra_set_engine(1, 3)
    (la, xa), (lb, xb) = res
    out["exact_vs_default"] = {"size": wl, "iters": 3, "loss_default": list(map(float, la)), "loss_exact": list(map(float, lb)),
                               "rel_loss": float(np.max(np.abs(la - lb) / np.abs(lb))),
                               "max_dx_first_4M_entries": float(np.max(np.abs(xa - xb)))}
    print(json.dumps(out["exact_vs_default"]), flush=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
