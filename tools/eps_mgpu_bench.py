"""attack() with adjacency noise (--eps 0.05, MSELoss, Profile A) on N GPUs of one box, tile-row sharded: device-event
it/s of the loop, the time of the redundant full draw every rank makes, and peak device memory per rank (set-up
included).  Run once per N
(N = 1 also runs without torchrun); every run adds its record to the output file:

    torchrun --nproc-per-node N tools/eps_mgpu_bench.py [--sizes 65536,98304] [--steps 10] [--out FILE]

bench.py's synthetic inputs (bench.build_problem) at the given n, feature_adj passed as a full host tensor."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def card(index):
    r = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 and r.stdout.strip() else "unknown"


def one_size(n, steps, dev, world):
    prob = bench.build_problem(dict(n=n, f=512, c=8), dev)
    args = bench.make_args("A")
    args.eps = 0.05
    atk, adj = bench.make_attack(prob, dev)
    torch.cuda.manual_seed(1234)           # every rank draws the same matrices (PGDEngine.check_noise_agreement)
    atk.attack(args, None, 10 ** args.lr, 0, 1.0, bench.PROFILE_A, prob["feature_adj"], 0, 0, 0, None, None, None, adj,
               prob["X"], torch.zeros(1), prob["labels"], prob["idx_attack"], int(1e7 * prob["nedges"]), 0, epochs=0,
               _engine_epochs=steps + 4, _skip_finalize=True)
    del prob
    eng = atk.engine
    for _ in range(2):
        eng.iterate()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        eng.iterate()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    eng.check_noise_agreement()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(3):
        torch.randn((n, n), dtype=torch.float32, device=dev)
    e.record()
    torch.cuda.synchronize()
    draw_ms = s.elapsed_time(e) / 3
    peak = torch.tensor([torch.cuda.max_memory_allocated(dev) / 1e9], dtype=torch.float64, device=dev)
    peaks = [torch.zeros_like(peak) for _ in range(world)]
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)         # the slowest rank sets the pace
        dist.all_gather(peaks, peak)
    else:
        peaks = [peak]
    loss = eng.losses()["loss"]
    atk.engine = None
    return {"ms_per_iter": float(ms), "it_s": 1000.0 / float(ms), "draw_ms": draw_ms,
            "peak_mem_gb_per_rank": [round(float(p), 2) for p in peaks], "loss_last": float(loss[-1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="65536")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eps_mgpu_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eps_mgpu_bench needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank = dist.get_rank() if world > 1 else 0
    rec = {"card": card(local), "gpus": world, "profile": bench.PROFILES["A"]["flags"] + ", eps=0.05", "sizes": {}}
    for n in map(int, a.sizes.split(",")):
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        r = one_size(n, a.steps, dev, world)
        rec["sizes"][str(n)] = r
        if rank == 0:
            print(f"N={world} n={n}: {json.dumps(r)}", flush=True)
    if world > 1:
        dist.destroy_process_group()
    if rank == 0:
        out = {}
        if os.path.exists(a.out):
            with open(a.out) as f:
                out = json.load(f)
        out.setdefault("runs", {})[f"N={world}"] = rec
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
