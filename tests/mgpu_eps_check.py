"""Run under torchrun: attack() with adjacency noise (--eps != 0, MSELoss) on tile-row shards.

One rank per GPU over NCCL; with --gloo every rank runs on cuda:0 over gloo (the same code path and collectives on a
one-GPU box, used for the 8-rank run with empty shards).  Checks, at n = 700 with all six weights:
  * the sharded run against the CPU oracle fed with the same draws (the bounds of test_eps_multi_tile_matches_oracle),
  * against the single-GPU native run on the same draws (SINGLE_* bounds, DESIGN.md 3.7),
  * the sharded AUC / AP against the gathered matrix, recovered_edges(k) equal on every rank,
  * the default stream: ranks seeded alike reproduce the single-GPU default-stream run,
  * ranks seeded differently make attack() raise RuntimeError.
Prints MGPU_EPS_OK / MGPU_EPS_FAIL on rank 0."""
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

CASES = [(0.05, 1e7), (0.5, 1e7), (0.05, 1.0)]
# sharded vs single-GPU native run on the same draws (3 iterations, n = 700): the two differ only in the order of fp32
# sums (atomics of one GPU against per-shard partials + all-reduce).  Measured on a B200 with 3 and 8 ranks over gloo
# (profiles/eps_mgpu_check_gloo8.log, DESIGN.md 3.7): loss 8.7e-9 relative, |dx| 5.3e-6, |d modified_adj| 9.5e-7 at most;
# the bounds leave about 10x each and stay well inside the oracle's (1e-4, 2e-4)
SINGLE_LOSS_RTOL = 1e-7
SINGLE_DX = 5e-5
SINGLE_DADJ = 1e-5


def run_noisy(d, dev, noise=None, epochs=3):
    """PGDAttack.attack as main.objective drives it (tests/test_gpu_eps.py::run_noisy on a given device)."""
    from helpers import make_args, make_models
    from mcgra_b200.topology_attack import PGDAttack
    n = int(d["labels"].shape[0])
    victim, emb = make_models(d, dev)
    model = PGDAttack(model=victim, embedding=emb, H_A=torch.from_numpy(d["H_A2"]).to(dev),
                      Y_A=torch.from_numpy(d["Y_A"]).to(dev), nnodes=n, loss_type="CE", device=dev).to(dev)
    if np.any(d["x0"] != 0):
        model.adj_changes.data = torch.from_numpy(d["x0"].copy()).to(dev)
    kw = {} if noise is None else {"_noise": lambda t: noise[t]}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)
        try:
            model.attack(make_args(d), None, 10 ** float(d["lr_exp"]), 0, float(d["weight_sup"]), tuple(d["weights"]),
                         torch.from_numpy(d["feature_adj"]), 0, 0, 0, None, None, np.arange(min(8, n)),
                         torch.from_numpy(d["adj"].astype(np.float32)), d["X"], np.zeros((n, n), np.float32), d["labels"],
                         d["idx_attack"], int(d["num_edges"]), 0, epochs=epochs, _trace=True, **kw)
        finally:
            os.chdir(cwd)
    torch.cuda.synchronize(dev)
    return dict(loss=np.asarray(model.engine.losses()["loss"]), x_iters=[x.cpu().numpy() for x in model._trace],
                modified_adj=model.gather_modified_adj().cpu().numpy(), model=model)


def main():
    gloo = "--gloo" in sys.argv
    local = int(os.environ.get("LOCAL_RANK", 0))
    rank = int(os.environ.get("RANK", 0))
    dev = torch.device("cuda", 0 if gloo else local)
    torch.cuda.set_device(dev)
    from test_gpu_eps import draws, noisy_case, oracle_noisy
    noise = draws(31, 700, 3)
    # single-GPU references, run before the process group exists (attack() sees world = 1)
    single = [run_noisy(noisy_case(eps, density), dev, noise) for eps, density in CASES]
    torch.cuda.manual_seed(1234)
    single_default = run_noisy(noisy_case(0.05), dev)
    for s in single + [single_default]:
        s.pop("model")

    dist.init_process_group("gloo" if gloo else "nccl", **({} if gloo else {"device_id": dev}))
    world = dist.get_world_size()
    import pgd_oracle as O
    from mcgra_b200 import metrics
    from mcgra_b200.engine import shard_tile_rows
    tr0, tr1 = shard_tile_rows(6, world)[rank]
    tag = f"[mgpu-eps world={world} rank={rank} tile rows [{tr0}, {tr1})]"
    ok = True
    for (eps, density), ref1 in zip(CASES, single):
        d = noisy_case(eps, density)
        got = run_noisy(d, dev, noise)
        e_loss1 = float(np.max(np.abs(got["loss"] - ref1["loss"]) / np.abs(ref1["loss"])))
        e_x1 = max(float(np.max(np.abs(a - b))) for a, b in zip(got["x_iters"], ref1["x_iters"]))
        e_adj1 = float(np.max(np.abs(got["modified_adj"] - ref1["modified_adj"])))
        print(f"{tag} eps={eps} density={density:g} vs 1 GPU: rel loss {e_loss1:.2e} max|dx| {e_x1:.2e} "
              f"max|dadj| {e_adj1:.2e}", flush=True)
        ok &= e_loss1 <= SINGLE_LOSS_RTOL and e_x1 <= SINGLE_DX and e_adj1 <= SINGLE_DADJ
        if rank == 0:
            ref = oracle_noisy(d, noise, 3)
            e_loss = float(np.max(np.abs(got["loss"] - ref["loss"]) / np.abs(ref["loss"])))
            e_x = max(float(np.max(np.abs(a - b.numpy()))) for a, b in zip(got["x_iters"], ref["x_iters"]))
            adj_ok = np.allclose(got["modified_adj"], ref["modified_adj"].numpy(), rtol=1e-3, atol=1e-3)
            print(f"{tag} eps={eps} density={density:g} vs oracle: rel loss {e_loss:.2e} max|dx| {e_x:.2e} "
                  f"modified_adj within 1e-3: {adj_ok}", flush=True)
            ok &= e_loss <= 1e-4 and e_x < 2e-4 and adj_ok
        if (eps, density) == CASES[0]:
            # metrics on the row bands: AUC / AP in place, top-k through the sharded selection
            mdl, n = got["model"], 700
            full = torch.from_numpy(got["modified_adj"])
            ee = np.argwhere(np.triu(d["adj"], 1) > 0)
            auc_s, ap_s = metrics.auc_ap_from_edges_sharded(mdl.modified_adj, mdl.modified_adj_rows[0], n, ee)
            real = d["adj"].reshape(-1).astype(np.float32)
            auc_f, ap_f = O.roc_auc(real, full.reshape(-1).numpy()), O.average_precision(real, full.reshape(-1).numpy())
            k = 2000
            mine = [t.cpu() for t in mdl.recovered_edges(k)]
            want = [t.cpu() for t in metrics.topk_pairs(full.to(dev), k)]
            packed = torch.cat([mine[0].double(), mine[1].double(), mine[2].double()])
            lo, hi = packed.clone().to(dev), (-packed).to(dev)
            dist.all_reduce(lo, op=dist.ReduceOp.MAX)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            same = bool(torch.equal(lo, -hi)) and all(torch.equal(a, b) for a, b in zip(mine, want))
            print(f"{tag} sharded AUC {auc_s:.9f} / AP {ap_s:.9f} vs gathered {auc_f:.9f} / {ap_f:.9f}; "
                  f"recovered_edges({k}) equal on every rank and to the gathered matrix's: {same}", flush=True)
            ok &= abs(auc_s - auc_f) < 1e-9 and abs(ap_s - ap_f) < 1e-9 and same
        del got
    # the default stream: every rank draws torch.randn((n, n)) from its own generator, seeded alike
    torch.cuda.manual_seed(1234)
    got = run_noisy(noisy_case(0.05), dev)
    e_def = float(np.max(np.abs(got["loss"] - single_default["loss"]) / np.abs(single_default["loss"])))
    print(f"{tag} default stream, seeded alike, vs 1 GPU: rel loss {e_def:.2e}", flush=True)
    ok &= e_def <= 1e-4
    del got
    # ranks seeded differently draw different matrices: attack() must refuse the result on every rank
    torch.cuda.manual_seed(1234 + rank)
    try:
        run_noisy(noisy_case(0.05), dev, epochs=2)
        raised = False
    except RuntimeError as e:
        raised = "drew different noise" in str(e)
    print(f"{tag} seeds 1234 + rank: attack() raised RuntimeError: {raised}", flush=True)
    ok &= raised
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_EPS_OK" if flag.item() == 1.0 else "MGPU_EPS_FAIL", flush=True)
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
