#!/usr/bin/env python
"""bench.py -- PGD attack iterations/second of the native path (BASELINE.json metric).

    python bench.py --gpus 1 --steps 10 --warmup 3            # one JSON line on stdout
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...                      # the reference's CPU algorithm (oracle port)
    python bench.py --steps 10 --warmup 3 --dump-outputs DIR  # also write the timed path's outputs as DIR/<name>.npy

Workload (config.workload): synthetic planted-partition graph of BASELINE.json's shape, README-Cora flag
profile ("Profile A": --w1=0.01 --w6=10 --w7=10 --w9=10 --w10=1000 --lr=-2 --measure=MSELoss, all three priors,
MC-GRA/README.md:29).  One step = one full PGD iteration (forward, prior losses, backward, Adam, projection test),
SURVEY.md 3.2 steps 1-17.  `value` is timed with CUDA events with all inputs resident in HBM; `e2e` goes through
the public API (PGDAttack.attack + AUC) starting from pinned HOST tensors and ending with the AUC scalar on the host.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "large": dict(n=65536, f=512, c=8, name="synthetic n=65536 f=512 c=8 (BASELINE configs[4])"),
    "pubmed": dict(n=19717, f=500, c=3, name="synthetic PubMed-shape n=19717 f=500 c=3 (BASELINE configs[3])"),
    "cora": dict(n=2708, f=1433, c=7, name="synthetic Cora-shape n=2708 f=1433 c=7 (BASELINE configs[0] shape)"),
    "tiny": dict(n=1024, f=64, c=4, name="synthetic n=1024 (debug)"),
}
PROFILE_A = (0.01, 0, 0, 0, 0, 10, 10, 0, 10, 1000)
# SURVEY 8(d) Profile B = README Polblogs all-priors command (MC-GRA/README.md:90), measure HSIC, lr 10^-2.5
PROFILE_B = (0.01, 0.01, 0, 0, 0, 10000, 100, 0, 0.001, 1000)
PROFILES = {"A": dict(w=PROFILE_A, measure="MSELoss", lr=-2.0,
                      flags="Profile A: README Cora MSELoss w1=.01 w6=10 w7=10 w9=10 w10=1000 lr=1e-2"),
            "B": dict(w=PROFILE_B, measure="HSIC", lr=-2.5,
                      flags="Profile B: README Polblogs HSIC w1=.01 w2=.01 w6=1e4 w7=100 w9=.001 w10=1000 lr=10^-2.5 "
                            "(n x n HSIC stage on library GEMMs, DESIGN.md 1)")}
SAMPLE_N = int(os.environ.get("MCGRA_BENCH_SAMPLE_N", "3072"))   # CPU baseline sample size (the reference algorithm is O(n^3) per iteration)
DUMP_SAMPLE = 1 << 22     # --dump-outputs keeps at most this many entries of an array: two 16 MB samples + loss histories


class Args:
    pass


def make_args(profile="A"):
    pr = PROFILES[profile]
    a = Args()
    a.max_eval, a.lr, a.eps, a.measure, a.dataset = 100, pr["lr"], 0.0, pr["measure"], "cora"
    a.useH_A = a.useY_A = a.useY = True
    for k, w in enumerate(pr["w"], 1):
        setattr(a, f"w{k}", w)
    return a


def clocks_sampler(stop, out, index):
    """SM clock / power / throttle reasons sampled DURING the timed region (NVML, every 20 ms; falls back to
    nvidia-smi polling when pynvml is unavailable)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        R = pynvml
        names = [("hw_slowdown", R.nvmlClocksEventReasonHwSlowdown if hasattr(R, "nvmlClocksEventReasonHwSlowdown") else 0x8),
                 ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]
        while not stop.is_set():
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
            try:
                rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            flags = ["Active" if (rs & bit) else "Not Active" for _, bit in names]
            out.append(f"{sm}, {mx}, {pw:.1f}, " + ", ".join(flags))
            stop.wait(0.02)
        return
    except Exception:
        pass
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=5)
            out.append(r.stdout.strip())
        except Exception:
            pass
        stop.wait(0.2)


def summarise_clocks(samples):
    sm, mx, reasons = [], 0, set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for s in samples:
        p = [x.strip() for x in s.split(",")]
        if len(p) < 7:
            continue
        try:
            sm.append(float(p[0]))
            mx = max(mx, float(p[1]))
        except ValueError:
            continue
        for nme, v in zip(names, p[3:7]):
            if v.lower().startswith("active"):
                reasons.add(nme)
    pw = []
    for s_ in samples:
        try:
            pw.append(float(s_.split(",")[2]))
        except Exception:
            pass
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": float(np.min(sm)) if sm else None,
            "sm_max_mhz": mx or None, "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons),
            "samples": len(sm)}


def build_problem(wl, device, seed=15, host_feature_adj=True):
    """Synthetic inputs on the HOST (pinned) + victim weights.  SURVEY.md 8(d)."""
    import torch
    from mcgra_b200 import synth
    g = synth.make_graph(wl["n"], wl["f"], wl["c"], seed=seed)
    W = synth.gcn_weights(wl["f"], 16, wl["c"], seed=seed, gain=3.0)
    n = wl["n"]
    X = torch.from_numpy(g["features"])
    edges = torch.from_numpy(g["edges"])
    # feature_adj = sigmoid(relu(X X^T - I)) (main.dot_product_decode for cora, main.py:44-55); computed on the
    # device once (setup, untimed) and handed to the API as a host tensor like the reference driver does
    Xd = X.to(device)
    fa = Xd @ Xd.t()
    fa.diagonal().sub_(1.0)
    fa = torch.sigmoid_(torch.relu_(fa))
    if host_feature_adj:
        fa_host = torch.empty(n, n, dtype=torch.float32, pin_memory=True)
        fa_host.copy_(fa)
        del fa
    else:
        # N > 1: every rank keeps (pinned, on the host) exactly the row bands of feature_adj it touches -- the rows of its
        # tile-row shard for the loop and its band of the n x n result for the ensemble -- and copies them host -> device
        # inside the timed e2e call, so that e2e means the same thing at every N (all ranks together move >= the n x n
        # matrix once, like the single n x n copy at N = 1)
        from mcgra_b200.engine import HostBands, TILE, output_band, shard_tile_rows
        rank = int(os.environ.get("RANK", 0))
        world = int(os.environ.get("WORLD_SIZE", 1))
        T = (n + TILE - 1) // TILE
        tr0, tr1 = shard_tile_rows(T, world)[rank]
        bands = {}
        for r0, r1 in {(tr0 * TILE, min(n, tr1 * TILE)), output_band(n, rank, world)}:
            if r1 > r0:
                hb = torch.empty(r1 - r0, n, dtype=torch.float32, pin_memory=True)
                hb.copy_(fa[r0:r1])
                bands[(r0, r1)] = hb
        del fa
        fa_host = HostBands(n, bands)
    del Xd
    torch.cuda.empty_cache()
    rng = np.random.RandomState(seed)
    idx_attack = rng.permutation(n)
    return dict(n=n, X=X.pin_memory(), edges=edges, labels=torch.from_numpy(g["labels"]), W=W,
                feature_adj=fa_host, idx_attack=idx_attack, nedges=int(edges.shape[0]))


def sparse_adj(prob, device):
    import torch
    e = prob["edges"].to(device)
    idx = torch.cat([e.t(), e.t().flip(0)], 1)
    return torch.sparse_coo_tensor(idx, torch.ones(idx.shape[1], device=device), (prob["n"], prob["n"])).coalesce()


def make_attack(prob, device):
    import torch
    from copy import deepcopy
    from mcgra_b200.models.gcn import GCN, embedding_GCN
    from mcgra_b200.topology_attack import PGDAttack
    W = prob["W"]
    f, c, n = W["W1"].shape[0], W["Wl"].shape[0], prob["n"]
    victim = GCN(nfeat=f, nclass=c, nhid=16, nlayer=2, device=device)
    with torch.no_grad():
        victim.gc[0].weight.copy_(torch.from_numpy(W["W1"])); victim.gc[0].bias.copy_(torch.from_numpy(W["b1"]))
        victim.gc[1].weight.copy_(torch.from_numpy(W["W2"])); victim.gc[1].bias.copy_(torch.from_numpy(W["b2"]))
        victim.linear1.weight.copy_(torch.from_numpy(W["Wl"])); victim.linear1.bias.copy_(torch.from_numpy(W["bl"]))
    victim = victim.to(device)
    for layer in victim.gc:
        layer.to(device)
    emb = embedding_GCN(nfeat=f, nhid=16, nlayer=2, device=device)
    emb.gc = deepcopy(victim.gc)
    victim.eval(); emb.eval()
    adj = sparse_adj(prob, device)
    with torch.no_grad():
        Xd = prob["X"].to(device)
        H_A = emb(Xd, adj)
        Y_A = victim(Xd, adj)
    # .to(device) like the reference driver (main.py:300): adj_changes (P floats) lives on the device
    atk = PGDAttack(model=victim, embedding=emb, H_A=H_A, Y_A=Y_A, nnodes=n, loss_type="CE", device=device).to(device)
    return atk, adj


def w_active(w, k):
    return w[k] != 0


def large_parity(a, prob, args, PROFILE_W, num_edges, device, world, iters=5, rows=64):
    """Untimed precision evidence AT THE BENCH SIZE (the reference cannot run there): (1) the exact fp32 FFMA engines
    (mcgra_set_engine(*, 0)) against the default tensor-core engines for `iters` iterations from the same start: relative
    loss difference and max |dx|; (2) an fp64 evaluation of `rows` sampled rows of the first propagation
    Y = M [r*S1 | S1] against the tcgen05 result.  Collective at N > 1 (every rank runs it)."""
    import torch
    from mcgra_b200 import _native as N
    out = {}
    runs = {}
    try:
        for name, engines in (("exact", {0: 0, 1: 0, 2: 0}), ("default", {0: 5, 1: 3, 2: 2})):
            for w, v in engines.items():
                N.lib().mcgra_set_engine(w, v)
            atk, adj = make_attack(prob, device)
            n = prob["n"]
            atk.attack(args, None, 10 ** args.lr, 0, 1.0, PROFILE_W, prob["feature_adj"], 0, 0, 0, None, None, None, adj,
                       prob["X"], torch.zeros(1), prob["labels"], prob["idx_attack"], num_edges, 0, epochs=0,
                       _engine_epochs=iters + 2, _skip_finalize=True)
            eng = atk.engine
            if name == "default":       # fp64 check of sampled rows of the first propagation (before any update: x = 0
                eng.iterate()           # gives M = 0, so check after one iteration)
                rs = np.random.RandomState(0)
                ii = torch.from_numpy(rs.randint(0, n, rows)).to(device)
                xp = eng.packed_parameter()
                keep_row = eng._acc_row(eng.step).clone()
                eng.forward_stages(eng.step)             # re-runnable (node kernels re-zero their outputs) ...
                eng._acc_row(eng.step).copy_(keep_row)   # ... except for the loss accumulators of this iteration
                Y1 = eng.Y1[ii].double()
                B1 = eng.B1.double()
                jj = torch.arange(n, device=device)
                errs = []
                for q in range(rows):
                    i = int(ii[q])
                    lo = (i * (i - 1)) // 2 + jj[:i]
                    hi = (jj[i + 1:] * (jj[i + 1:] - 1)) // 2 + i
                    row = torch.zeros(n, dtype=torch.float64, device=device)
                    row[:i] = xp[lo].double().clamp(0, 1)
                    row[i + 1:] = xp[hi].double().clamp(0, 1)
                    y = row @ B1
                    errs.append(float(((Y1[q] - y).abs() / (row @ B1.abs() + 1e-30)).max()))
                out["fp64_rows_checked"] = rows
                out["propagate_max_rel_err_vs_fp64"] = max(errs)
                del xp
                for _ in range(iters - 1):
                    eng.iterate()
            else:
                for _ in range(iters):
                    eng.iterate()
            runs[name] = (eng.losses()["loss"], eng.packed_parameter())
            del eng, atk
            torch.cuda.empty_cache()
    finally:
        for w, v in {0: 5, 1: 3, 2: 2}.items():
            N.lib().mcgra_set_engine(w, v)
    le, xe = runs["exact"]
    ld, xd = runs["default"]
    out["iters"] = iters
    out["rel_loss"] = float(np.max(np.abs(le - ld) / np.abs(le)))
    out["max_dx"] = float((xe - xd).abs().max())
    out["what"] = ("exact fp32 FFMA engines vs default tcgen05 engines, same start, %d iterations at the bench size; "
                   "fp64 check of %d sampled rows of the first propagation" % (iters, rows))
    return out


def same_config_baseline(a, device, n=2708, f=1433, c=7, iters=3):
    """The SAME configuration on every arm, in the same run, at a size the reference's dense algorithm can run:
    synthetic Cora shape (BASELINE configs[0]), Profile A, `iters` iterations each -- native (device-resident),
    the oracle port on the host cores, and the oracle port on this GPU (fp32, allow_tf32=False: the reference's own
    PyTorch-GPU path, BASELINE.md 3).  At N = 1 only."""
    import torch
    res = {"n": n, "f": f, "c": c, "profile": "A", "iters": iters}
    wl = dict(n=n, f=f, c=c, name="same-config")
    prob = build_problem(wl, device)
    args = make_args("A")
    atk, adj = make_attack(prob, device)
    atk.attack(args, None, 10 ** args.lr, 0, 1.0, PROFILE_A, prob["feature_adj"], 0, 0, 0, None, None, None, adj,
               prob["X"], torch.zeros(1), prob["labels"], prob["idx_attack"], 10 ** 12, 0, epochs=0,
               _engine_epochs=iters + 8, _skip_finalize=True)
    eng = atk.engine
    for _ in range(3):
        eng.iterate()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        eng.iterate()
    e1.record()
    torch.cuda.synchronize()
    res["native_it_s"] = iters / (e0.elapsed_time(e1) * 1e-3)
    native_loss = eng.losses()["loss"][:iters]
    del eng, atk
    O, cprob, cfg = cpu_problem(n, f, c)
    torch.set_num_threads(os.cpu_count())
    O.attack(cprob, cfg, 1, bookkeeping=True)
    t0 = time.perf_counter()
    r = O.attack(cprob, cfg, iters, bookkeeping=True)
    res["oracle_cpu_it_s"] = iters / (time.perf_counter() - t0)
    res["oracle_cpu_cores"] = os.cpu_count()
    res["max_rel_loss_native_vs_oracle"] = float(np.max(np.abs(np.asarray(r["loss"]) - native_loss) / np.abs(np.asarray(r["loss"]))))
    res["oracle_cuda"] = oracle_on_cuda(O, cprob, cfg, device, iters)
    return res


def oracle_on_cuda(O, cprob, cfg, device, iters):
    """The reference's dense PyTorch algorithm (oracle port) on the GPU in fp32 with TF32 off."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        gprob = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in cprob.items()}
        gprob["W"] = {k: v.to(device) for k, v in cprob["W"].items()}
        with torch.device(device):
            O.attack(gprob, cfg, 1, bookkeeping=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            O.attack(gprob, cfg, iters, bookkeeping=True)
            torch.cuda.synchronize()
        return {"it_s": iters / (time.perf_counter() - t0), "dtype": "fp32, allow_tf32=False", "n": cprob["n"]}
    except Exception as e:          # the oracle is CPU test infrastructure; report instead of failing the bench
        return {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def kernel_times(timers, steps):
    """mean launch time and launches per step of every timed entry point.  Bisection passes that found the search finished
    return without reading anything (~0.07 ms): they are left out of the mean and of the count, so that the pass kernel's
    bandwidth is that of the passes that actually stream the parameter."""
    kt, kcount = {}, {}
    for k, v in timers.items():
        ms = [s.elapsed_time(e) for s, e in v]
        if k == "mcgra_bisect_pass" and ms:
            work = [m for m in ms if m > 0.2 * max(ms)]
            ms = work or ms
        kt[k] = float(np.mean(ms))
        kcount[k] = len(ms) / steps
    return kt, kcount


def roofline_report(kt, kcount, n, P, world, a, peaks, extra):
    """`roofline` of the DOMINANT kernel of the step (largest share of the iteration) + per-kernel fractions.
    Algorithmic bytes per launch (DESIGN.md 3): one read of the rank's shard of every streamed tile array + the node
    arrays; flops of the dense contraction: 2 n^3 / world per GEMM (row panel), issued = 3x (three kind::f16 MMAs)."""
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    bf16 = float(peaks.get("bf16_tflops", 1650.0))
    src = "MEASURED_PEAKS.json (measured)" if peaks else "fallback (B200_PROFILING.md)"
    w = PROFILES[a.profile]["w"]
    c1 = w[0] != 0
    Pw = P / world
    alg = {"elem_stats": (8.0 if c1 else 4.0) * Pw, "propagate32": 4.0 * Pw + 3 * n * 32 * 4, "propagate32_elem": 8.0 * Pw,
           "propagate16": 4.0 * Pw + 3 * n * 16 * 4, "mcgra_fold_adam": (28.0 if (c1 or a.profile == "B") else 24.0) * Pw,
           "mcgra_pairs": (12.0 * Pw if a.profile == "B" else 0.0), "mcgra_bisect_pass": 4.0 * Pw,
           "mcgra_bisect_finish": 4.0 * Pw, "mcgra_sym_to_tiles": 4.0 * n * n / world + 4.0 * Pw,
           "mcgra_image_ahat": 4.0 * P + 4.0 * n * n, "mcgra_image_m1": 4.0 * n * n,
           "mcgra_image_from_dense": 12.0 * n * n}
    flops = {k: 2.0 * n ** 3 / world for k in ("gemm_c1", "gemm_c2_T", "gemm_grad", "gemm_self")}
    per = []
    for k, ms in kt.items():
        cnt = kcount.get(k, 1.0)
        row = {"kernel": k, "ms": ms, "launches_per_step": cnt, "ms_per_step": ms * cnt}
        if k in flops:
            row.update(bound="tensor", useful_tflops=flops[k] / (ms * 1e-3) / 1e12,
                       issued_tflops=3 * flops[k] / (ms * 1e-3) / 1e12, frac=3 * flops[k] / (ms * 1e-3) / 1e12 / bf16)
        elif alg.get(k, 0.0) > 0:
            row.update(bound="hbm", alg_bytes=alg[k], gbs=alg[k] / (ms * 1e-3) / 1e9, frac=alg[k] / (ms * 1e-3) / 1e9 / hbm)
        per.append(row)
    per.sort(key=lambda r: -r["ms_per_step"])
    dom = next((r for r in per if "frac" in r), None)
    if dom is None:
        return None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    traffic = None
    if world == 1 and os.path.exists(tp):
        traffic = json.load(open(tp)).get(f"{a.workload}_{a.profile}", {}).get(dom["kernel"])
    if dom["bound"] == "tensor":
        roof = {"bound": "tensor", "kernel": dom["kernel"] + " (mcgra_gemm_nt / k_gemm3<2>: TMA-fed tcgen05 kind::f16 x3 from fp16x2 "
                "operand images, cta_group::2, fp32 accumulators in TMEM)",
                "achieved": dom["issued_tflops"], "peak": bf16, "unit": "TFLOP/s", "frac": dom["frac"], "traffic": traffic,
                "peak_source": src + ": bf16_tflops (the kernel issues kind::f16 MMAs)",
                "useful_tflops": dom["useful_tflops"], "tf32_peak_measured": extra.get("tf32_tflops"),
                "useful_over_tf32_peak": (dom["useful_tflops"] / extra["tf32_tflops"]) if extra.get("tf32_tflops") else None,
                "note": "useful = 2 n^3 / t (TF32-equivalent work of the reference's fp32 GEMM); a 3xTF32 kernel cannot exceed "
                        "1/3 of the TF32 peak in useful flops, the fp16x2 split reaches the same precision class at the "
                        "kind::f16 rate"}
    else:
        roof = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["gbs"], "peak": hbm, "unit": "GB/s",
                "frac": dom["frac"], "traffic": traffic, "peak_source": src + ": hbm_gbs",
                "launch_ms": dom["ms"], "algorithmic_bytes_per_launch": dom["alg_bytes"]}
    roof["share_of_step"] = dom["ms_per_step"] / max(1e-9, sum(r["ms_per_step"] for r in per))
    roof["per_kernel"] = per
    return roof


def measure_tf32_peak(device):
    """TF32 tensor peak measured the way MEASURED_PEAKS.json measures bf16 (torch.matmul 8192^3, best of 10), untimed setup."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        x = torch.randn(8192, 8192, device=device)
        y = torch.randn(8192, 8192, device=device)
        best = 1e9
        for _ in range(10):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            x @ y
            e.record()
            torch.cuda.synchronize()
            best = min(best, s.elapsed_time(e))
        return 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def sample_flat(t, seed):
    """Flattened float32 host copy of a device tensor: all of it up to DUMP_SAMPLE entries, else the entries at a fixed
    seeded set of sorted, distinct flat indices (np.unique of RandomState(seed).randint(0, numel, DUMP_SAMPLE)), so that
    two runs or two builds at the same size compare entry for entry."""
    import torch
    flat = t.reshape(-1)
    if flat.numel() > DUMP_SAMPLE:
        idx = np.unique(np.random.RandomState(seed).randint(0, flat.numel(), DUMP_SAMPLE, dtype=np.int64))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    return flat.float().cpu().numpy()


def write_outputs(path, arrays, rank):
    """--dump-outputs: rank 0 writes every array as <path>/<name>.npy, float32 arrays as they are, the rest as float64."""
    if rank != 0:
        return
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        v = np.asarray(v)
        np.save(os.path.join(path, name + ".npy"), v if v.dtype == np.float32 else v.astype(np.float64))


def run_native(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from mcgra_b200 import _native as N
    from mcgra_b200 import metrics
    N.lib()
    wl = WORKLOADS[a.workload]
    n = wl["n"]
    P = n * (n - 1) // 2
    extra = {}
    if rank == 0:
        extra["tf32_tflops"] = measure_tf32_peak(device)
    prob = build_problem(wl, device, host_feature_adj=(world == 1))
    args = make_args(a.profile)
    PROFILE_W = PROFILES[a.profile]["w"]
    K, Wm = a.steps, a.warmup

    # ------------------------------------------------------------------ device-resident steps (`value`)
    atk, adj = make_attack(prob, device)
    num_edges = int(0.5 * a.density * (2 * prob["nedges"]) / n ** 2 * n ** 2)    # main.py:247-248 (--density, default 1e7)
    # epochs=0: builds the engine (constants, tiled feature_adj) without iterating; then we drive iterate() here
    atk.attack(args, None, 10 ** args.lr, 0, 1.0, PROFILE_W, prob["feature_adj"], 0, 0, 0, None, None, None, adj,
               prob["X"], torch.zeros(1), prob["labels"], prob["idx_attack"], num_edges, 0, epochs=0,
               _engine_epochs=K + Wm + 16, _skip_finalize=True)
    eng = atk.engine
    for _ in range(Wm):
        eng.iterate()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    stop, samples = threading.Event(), []
    th = threading.Thread(target=clocks_sampler, args=(stop, samples, local), daemon=True)
    th.start()
    graphed = bool(eng.ring_mode) and K >= 8
    if graphed:
        # small graphs: the timed region replays two iterations per CUDA graph (engine.run), which cannot carry CUDA
        # events per kernel -- the per-kernel times come from three eager iterations just before it
        N.TIMERS['on'] = {}
        for _ in range(3):
            eng.iterate()
        torch.cuda.synchronize()
        kt, kcount = kernel_times(N.TIMERS['on'], 3.0)
        N.TIMERS['on'] = None
        eng.run(8, use_graph=True)  # captures the graph (one-off, cached on the engine) outside the timed region
        torch.cuda.synchronize()
    else:
        N.TIMERS['on'] = {}
    l0 = N.LAUNCHES["kernels"]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    if graphed:
        eng.run(K, use_graph=True)
    else:
        for _ in range(K):
            eng.iterate()
    ev1.record()
    torch.cuda.synchronize()
    launches = N.LAUNCHES["kernels"] - l0      # hand-written kernels launched inside the timed region
    stop.set()
    th.join()
    ms = ev0.elapsed_time(ev1)
    if not graphed:
        kt, kcount = kernel_times(N.TIMERS['on'], float(K))
        if os.environ.get("MCGRA_BENCH_DUMP_KERNEL") in N.TIMERS['on'] and rank == 0:     # per-launch times of one kernel
            v = N.TIMERS['on'][os.environ["MCGRA_BENCH_DUMP_KERNEL"]]
            print("[per-launch ms]", [round(s.elapsed_time(e), 3) for s, e in v][:40], file=sys.stderr)
        N.TIMERS['on'] = None
    if world > 1:
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    hist = eng.losses()
    losses = hist["loss"]
    if a.dump_outputs:      # the K timed iterations' loss terms and the parameter after the last one (collective at N > 1)
        dump = {("loss" if k == "loss" else "loss_" + k): v[-K:] for k, v in hist.items()}
        dump["adj_changes"] = sample_flat(eng.packed_parameter(), seed=0)
        write_outputs(a.dump_outputs, dump, rank)
    del eng, atk
    torch.cuda.empty_cache()
    parity_large = None
    if not a.no_parity:
        parity_large = large_parity(a, prob, args, PROFILE_W, num_edges, device, world)

    # ------------------------------------------------------------------ end to end through the public API
    e2e = None
    if not a.no_e2e:
        atk, adj = make_attack(prob, device)
        labels_pos = prob["edges"]
        # one warm call at 1 epoch so allocator / lazy init are not in the timed region
        def score(atk_):
            if world == 1:
                return metrics.auc_ap_from_edges(atk_.modified_adj, labels_pos)
            return metrics.auc_ap_from_edges_sharded(atk_.modified_adj, atk_.modified_adj_rows[0], n, labels_pos)
        atk.attack(args, None, 10 ** args.lr, 0, 1.0, PROFILE_W, prob["feature_adj"], 0, 0, 0, None, None, None, adj,
                   prob["X"], torch.zeros(1), prob["labels"], prob["idx_attack"], num_edges, 0, epochs=1, _gather_x=False)
        score(atk)
        atk.adj_changes.data.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        atk.attack(args, None, 10 ** args.lr, 0, 1.0, PROFILE_W, prob["feature_adj"], 0, 0, 0, None, None, None, adj,
                   prob["X"], torch.zeros(1), prob["labels"], prob["idx_attack"], num_edges, 0, epochs=K, _gather_x=False,
                   _timing=bool(os.environ.get("MCGRA_E2E_TIMING")))
        t_att = time.perf_counter() - t0
        loss_hist = atk.engine.losses()["loss"]            # D2H of the per-iteration loss history
        auc, ap = score(atk)                               # D2H of two scalars
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if os.environ.get("MCGRA_E2E_TIMING"):
            sys.stderr.write(f"[e2e rank {rank}] attack {t_att:.3f}s (phases {getattr(atk, '_timing', None)}), "
                             f"losses+AUC {dt - t_att:.3f}s, total {dt:.3f}s\n")
        if world > 1:
            t = torch.tensor([dt], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        if a.dump_outputs:      # what PGDAttack.attack + AUC hand back (gathering the row bands is collective at N > 1)
            write_outputs(a.dump_outputs, {"e2e_loss": loss_hist, "e2e_auc_ap": [auc, ap],
                                           "e2e_modified_adj": sample_flat(atk.gather_modified_adj(), seed=1)}, rank)
        if world == 1:
            fa_bytes = prob["feature_adj"].numel() * 4
        else:       # all ranks' row bands together
            t = torch.tensor([sum(b.numel() * 4 for b in prob["feature_adj"].bands.values())], device=device, dtype=torch.float64)
            dist.all_reduce(t)
            fa_bytes = int(t.item())
        h2d = fa_bytes + world * (prob["X"].numel() * 4 + prob["labels"].numel() * 8 + n * 8)
        e2e = {"value": K / dt, "unit": "iterations/s", "h2d_bytes_per_step": int(h2d / K),
               "d2h_bytes_per_step": int((len(loss_hist) * 32 * 8 + 16) / K),
               "includes": "PGDAttack.attack(epochs=K) from pinned host tensors (features, labels, idx, feature_adj"
                           + (" n x n" if world == 1 else " as per-rank row bands: shard rows + result band")
                           + ") + final ensemble + GPU AUC/AP" + ("" if world == 1 else " on row bands (counts all-reduced)")
                           + ", amortised over K",
               "auc": auc, "ap": ap}

    parity_mgpu = None
    if world > 1 and not a.no_parity:
        parity_mgpu = mgpu_parity(device, world)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    roof = roofline_report(kt, kcount, n, P, world, a, peaks, extra)
    clocks = summarise_clocks(samples)
    out = {"metric": "PGD attack iterations/s (fwd+bwd+prior losses+Adam+projection)", "value": K / (ms * 1e-3),
           "unit": "iterations/s", "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": wl["name"], "n": n, "flags": PROFILES[a.profile]["flags"] + f", density {a.density:g}"
                      + (" (budget binds: bisection every iteration)" if num_edges < P else ""), "l2": "inputs larger than L2 (tiled x/m/v/F >> 126 MB)"
                      if 4 * P > 4e8 else "flush: none (working set fits L2 at this size)",
                      "sharding": f"tile-row shards x{world}" if world > 1 else "single GPU",
                      "cuda_graph": graphed},
           "roofline": roof, "gpu_launches": launches, "clocks": clocks, "e2e": e2e,
           "iter_bytes_algorithmic": 52.0 * P, "hbm_frac_whole_iter": 52.0 * P / world / (ms / K * 1e-3) / 1e9 / hbm,
           "loss_first_last": [float(losses[0]), float(losses[-1])], "parity_large": parity_large,
           "tf32_tflops_measured": extra.get("tf32_tflops")}
    if parity_mgpu is not None:
        out["parity_mgpu"] = parity_mgpu
    if a.profile == "B":
        out["dense_flops_per_iter_useful"] = (8.0 if w_active(PROFILE_W, 0) else 6.0) * float(n) ** 3
    if world == 1 and not a.no_cpu:
        out["cpu_baseline"] = cpu_baseline(a, threads=os.cpu_count())
        out["same_config_baseline"] = same_config_baseline(a, device)
    print(json.dumps(out))


def mgpu_parity(device, world):
    """Untimed, N > 1: the sharded attack of THIS process group (tile-row shards, row-band finalisation, sharded AUC / AP)
    against single-GPU golden fixtures generated from the unmodified reference (tests/golden/attack_*.npz,
    tests/golden/make_golden.py): per-iteration loss, final n x n result, and the sharded AUC / AP against the
    single-process kernel on the gathered matrix.  The full list of cases is tests/mgpu_check.py."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    from mcgra_b200 import metrics
    out = {"world": world, "cases": {}}
    ok = True
    got = d = None
    for case in ("mse_all_n150", "mse_budget_n150", "hsic_B_n150"):
        d = np.load(os.path.join(ROOT, "tests", "golden", f"attack_{case}.npz"))
        got = helpers.run_native_case(d, device=str(device))
        e_loss = float(np.max(np.abs(got["loss"] - d["loss"]) / np.abs(d["loss"])))
        e_adj = float(np.max(np.abs(got["modified_adj"] - d["modified_adj"])))
        out["cases"][case] = {"rel_loss": e_loss, "max_dadj": e_adj}
        ok = ok and e_loss < 1e-4 and e_adj < 2e-3
    mdl = got["model"]
    n = int(d["labels"].shape[0])
    ee = np.argwhere(np.triu(d["adj"], 1) > 0)
    auc_s, ap_s = metrics.auc_ap_from_edges_sharded(mdl.modified_adj, mdl.modified_adj_rows[0], n, ee)
    auc_f, ap_f = metrics.auc_ap_from_edges(torch.from_numpy(got["modified_adj"]).to(device), ee)
    out["auc_ap_sharded"] = [auc_s, ap_s]
    out["auc_ap_gathered"] = [auc_f, ap_f]
    ok = ok and abs(auc_s - auc_f) < 1e-12 and abs(ap_s - ap_f) < 1e-12
    out["ok"] = bool(ok)
    out["tolerances"] = "rel_loss < 1e-4, max_dadj < 2e-3, sharded AUC / AP equal to the gathered value"
    return out


def cpu_problem(n, f, c, seed=15):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pgd_oracle as O
    from mcgra_b200 import synth
    g = synth.make_graph(n, f, c, seed=seed)
    W = {k: torch.from_numpy(v) for k, v in synth.gcn_weights(f, 16, c, seed=seed, gain=3.0).items()}
    X = torch.from_numpy(g["features"])
    A = torch.from_numpy(synth.dense_adj(n, g["edges"]))
    prob = dict(n=n, X=X, adj=A, labels=torch.from_numpy(g["labels"]), W=W,
                idx_attack=torch.from_numpy(np.random.RandomState(seed).permutation(n)),
                feature_adj=O.feature_adj_of(X, "cora"))
    prob["H_A"] = O.embed(X, A, W, 2)
    prob["Y_A"] = O.victim(X, A, W)
    cfg = dict(measure="MSELoss", weights=list(PROFILE_A), lr=1e-2, eps=0.0, weight_sup=1.0, dataset="cora",
               use=(True, True, True), num_edges=10 ** 12)
    return O, prob, cfg


def cpu_baseline(a, threads, iters=2):
    """The reference's algorithm (oracle port, dense n x n torch CPU autograd incl. its per-iteration bookkeeping)
    on the host cores, on a bounded sample of the workload."""
    import torch
    torch.set_num_threads(max(1, threads))
    wl = WORKLOADS[a.workload]
    n = min(SAMPLE_N, wl["n"])
    O, prob, cfg = cpu_problem(n, wl["f"], wl["c"])
    O.attack(prob, cfg, 1, bookkeeping=True)       # warm
    t0 = time.perf_counter()
    O.attack(prob, cfg, iters, bookkeeping=True)
    dt = time.perf_counter() - t0
    v = iters / dt
    scale = (wl["n"] / n) ** 3
    return {"value": v, "unit": "iterations/s", "cores": threads, "kind": "port", "sample_n": n,
            "value_scaled_to_workload": v / scale,       # n^3 extrapolation of the sample rate to the bench size
            "sample": f"oracle port of the reference loop at n={n} (f={wl['f']}, c={wl['c']}), {iters} iterations incl. "
                      f"the reference's in-loop bookkeeping; the reference algorithm is O(n^3)/iteration and needs "
                      f">0.9 TB at n={wl['n']} (not runnable) -- n^3 extrapolation to n={wl['n']}: {v / scale:.3e} it/s"}


def run_reference(a):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    wl = WORKLOADS[a.workload]
    threads = os.cpu_count()
    import torch
    torch.set_num_threads(threads)
    n = min(SAMPLE_N, wl["n"])
    O, prob, cfg = cpu_problem(n, wl["f"], wl["c"])
    for _ in range(a.warmup):
        O.attack(prob, cfg, 1, bookkeeping=True)
    K = a.steps
    t0 = time.perf_counter()
    O.attack(prob, cfg, K, bookkeeping=True)
    dt = time.perf_counter() - t0
    v = K / dt
    sample = (f"oracle port of the reference loop at n={n} (bounded sample; the reference needs >0.9 TB and "
              f"O(n^3) work per iteration at n={wl['n']}), {K} timed iterations")
    out = {"impl": "reference", "metric": "PGD attack iterations/s (fwd+bwd+prior losses+Adam+projection)", "value": v,
           "unit": "iterations/s", "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": K, "warmup": a.warmup,
           "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"bounded sample n={n} of: " + wl["name"], "n": n, "sample_n": n,
                      "same_config_as_native_arm": n == wl["n"],
                      "note": "the reference's dense algorithm is O(n^3) time / >0.9 TB at n=65536; the native arm reports a "
                              "same-size comparison in `same_config_baseline` (n=2708, all three arms in one run)"},
           "cpu_baseline": {"value": v, "unit": "iterations/s", "cores": threads, "kind": "port", "sample": sample, "sample_n": n,
                            "value_scaled_to_workload": v / (wl["n"] / n) ** 3},
           "e2e": {"value": v, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="large", choices=list(WORKLOADS))
    ap.add_argument("--profile", default="A", choices=list(PROFILES), help="flag profile of SURVEY 8(d)")
    ap.add_argument("--density", type=float, default=1e7, help="main.py --density (1e7: budget never binds; 1: it does)")
    ap.add_argument("--no-e2e", dest="no_e2e", action="store_true")
    ap.add_argument("--no-cpu", dest="no_cpu", action="store_true")
    ap.add_argument("--no-parity", dest="no_parity", action="store_true", help="skip the untimed large-size precision check")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps write what they computed as DIR/<name>.npy: the loss terms of the K timed "
                         "iterations and the parameter after the last one, and of the e2e run its loss history, AUC / AP "
                         f"and modified_adj (arrays over {DUMP_SAMPLE} entries as a fixed seeded sample).  The inputs are "
                         "the same in every run; fp32 atomics make two runs of one build differ in the last bits, so "
                         "compare with a tolerance")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "native":
        ap.error("--dump-outputs writes the native path's outputs (--impl native)")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)


if __name__ == "__main__":
    main()
