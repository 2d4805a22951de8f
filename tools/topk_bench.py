"""Top-k recovered edges (metrics.topk_pairs) at n = 65 536 on one GPU: CUDA-event time per call and per stage, the bytes
the streaming passes read over their time, and the peak device memory beyond the score matrix.

The scores are a seeded mix of ties and continuous values (60 % exact zeros, 20 % on 64 levels, 20 % uniform), 17 GB,
far beyond the 126 MB L2, so every pass streams from HBM.

    python tools/topk_bench.py [--n 65536] [--ks 100000,1000000,10000000] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK_GBS = 7700.0      # HGX B200 data sheet, one GPU
STAGES = {0: "hist0", 1: "select0", 2: "hist1", 3: "select1", 4: "hist2", 5: "select2", 6: "count+scan", 7: "write"}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def scores(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    S = torch.rand(n, n, device="cuda", generator=g)
    sel = torch.rand(n, n, device="cuda", generator=g)
    S[sel < 0.6] = 0.0
    lv = (sel >= 0.6) & (sel < 0.8)
    S[lv] = torch.floor(S[lv] * 64) / 64
    del sel, lv
    torch.cuda.empty_cache()
    return S


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--ks", default="100000,1000000,10000000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_bench needs a CUDA device")
    import __graft_entry__ as g
    g.build()
    from mcgra_b200 import _native as N
    from mcgra_b200.metrics import topk_pairs
    n = a.n
    P = n * (n - 1) // 2
    S = scores(n, a.seed)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    stream_bytes = 4 * 4 * P            # levels 0-2 and the count pass each read the upper triangle once
    res = dict(card=card(), n=n, P=P, scores_gb=n * n * 4 / 1e9, reps=a.reps,
               note="scores: 60% exact zeros, 20% on 64 levels, 20% uniform (seeded); ms = CUDA events around "
                    "topk_pairs, mean of reps after one warm-up call; stream = stages 0, 2, 4, 6 (4 reads of the "
                    "upper triangle); peak_extra = peak allocated beyond the score matrix", runs=[])
    for k in [int(x) for x in a.ks.split(",")]:
        topk_pairs(S, k)                                   # warm-up (module load, allocator)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            r, c, s = topk_pairs(S, k)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.reps
        peak = torch.cuda.max_memory_allocated() - base
        N.TIMERS["on"] = {}                                # one more call with per-stage events
        topk_pairs(S, k)
        torch.cuda.synchronize()
        tm, N.TIMERS["on"] = N.TIMERS["on"], None
        stages = {}
        for name, evs in tm.items():
            stages[name] = sum(s_.elapsed_time(e_) for s_, e_ in evs)
        per = {}
        for (s_, e_), st in zip(tm["mcgra_topk_stage"], [0, 1, 2, 3, 4, 5, 6, 7]):
            per[STAGES[st]] = s_.elapsed_time(e_)
        stream_ms = per["hist0"] + per["hist1"] + per["hist2"] + per["count+scan"]
        run = dict(k=k, ms=ms, algorithmic_bytes_min=stream_bytes + 12 * k,
                   gbs_over_call=(stream_bytes + 12 * k) / ms / 1e6, stream_ms=stream_ms,
                   stream_gbs=stream_bytes / stream_ms / 1e6, stream_frac_hbm_peak=stream_bytes / stream_ms / 1e6 / HBM_PEAK_GBS,
                   stages_ms=per, calls_ms=stages, peak_extra_mb=peak / 1e6,
                   ws_bytes=int(N.lib().mcgra_topk_workspace_bytes(n, n, k)),
                   last_score=float(s[-1]), first_score=float(s[0]))
        print(json.dumps(run), flush=True)
        res["runs"].append(run)
    txt = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
