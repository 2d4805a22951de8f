"""Run under torchrun: row-band feature_adj (engine.HostBands) under every measure, and metric_pool_sharded.

Every rank holds only the rows of feature_adj it touches (its tile-row shard and its result band).  Checks:
  * the single-GPU goldens of HSIC / CKA / DP / KL-c2 / KDE with row bands, to the tolerances tests/mgpu_check.py holds
    the full-tensor runs of the same cases to;
  * the same ranks with a full tensor: iteration 1's loss agrees to 1e-6 relative (the constants are bit-identical,
    only atomics reorder), and no rank copies more rows of feature_adj than its bands hold;
  * an n = 900 HSIC case with c1 and c2 on row bands against the oracle;
  * metric_pool_sharded equals metric_pool on the gathered matrix (some result bands are empty at n = 90 with 3 ranks).

One rank per GPU over NCCL; with --gloo every rank runs on cuda:0 over gloo."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

CASES = ["hsic_B_n150", "hsic_all_n90", "cka_n90", "dp_n90", "kl_all_n90", "kl_C_n150", "kde_n90", "kde_readme_n150"]


def main():
    gloo = "--gloo" in sys.argv
    dev = torch.device("cuda", 0 if gloo else int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo" if gloo else "nccl", **({} if gloo else {"device_id": dev}))
    import pgd_oracle as O
    from helpers import run_native_case, synthetic_case
    from mcgra_b200 import metrics
    from mcgra_b200.engine import HostBands, TILE, output_band, shard_tile_rows
    rank, world = dist.get_rank(), dist.get_world_size()
    ok = True

    def say(msg):
        if rank == 0:
            print(f"[bands world={world}] {msg}", flush=True)

    def run_row_bands(d):
        """run_native_case with feature_adj as this rank's row bands; returns (result, rows copied, rows held)."""
        n = int(d["labels"].shape[0])
        tr0, tr1 = shard_tile_rows((n + TILE - 1) // TILE, world)[rank]
        fa_full = torch.from_numpy(d["feature_adj"])
        bands = {(r0, r1): fa_full[r0:r1].clone().pin_memory()
                 for r0, r1 in {(tr0 * TILE, min(n, tr1 * TILE)), output_band(n, rank, world)} if r1 > r0}
        hb = HostBands(n, bands)
        copied = []
        rows = hb.rows
        hb.rows = lambda r0, r1, device: copied.append(max(r1 - r0, 0)) or rows(r0, r1, device)
        torch_from = torch.from_numpy            # run_native_case does torch.from_numpy(d["feature_adj"])
        torch.from_numpy = lambda a: hb if a is d["feature_adj"] else torch_from(a)
        try:
            got = run_native_case(d, device=dev)
        finally:
            torch.from_numpy = torch_from
        return got, sum(copied), sum(r1 - r0 for r0, r1 in bands)

    for case in CASES:
        d = dict(np.load(os.path.join(ROOT, "tests", "golden", f"attack_{case}.npz")))      # (one array per key)
        got, copied, held = run_row_bands(d)
        full = run_native_case(d, device=dev)
        e_loss = float(np.max(np.abs(got["loss"] - d["loss"]) / np.abs(d["loss"])))
        if case.startswith("kde"):          # as tests/mgpu_check.py: the fp64 oracle at the native parameter
            prob64, cfg64 = O.problem_from_npz(d, dtype=torch.float64)
            xs_prev = [d["x0"]] + got["x_iters"][:-1]
            forced = np.array([float(O.iteration_terms(torch.from_numpy(np.asarray(xp)).double(), prob64, cfg64)[0])
                               for xp in xs_prev])
            e_loss = float(np.max(np.abs(np.asarray(got["loss"]) - forced) / np.abs(forced)))
        frac = float(np.mean(np.abs(np.stack(got["x_iters"]) - d["x_iters"]) > 2e-4))
        e_first = abs(float(got["loss"][0]) - float(full["loss"][0])) / abs(float(full["loss"][0]))
        e_adj = float(np.max(np.abs(got["modified_adj"] - full["modified_adj"])) / np.max(np.abs(full["modified_adj"])))
        c = torch.tensor([copied, held], dtype=torch.int64, device=dev)
        allc = [torch.zeros_like(c) for _ in range(world)]
        dist.all_gather(allc, c)
        over = [tuple(x.tolist()) for x in allc if int(x[0]) > int(x[1])]
        say(f"{case}: rel loss err {e_loss:.2e} frac|dx|>2e-4 {frac:.2e}; vs full tensor: iteration-1 rel loss err "
            f"{e_first:.2e} max|dadj|/max|adj| {e_adj:.2e}; rows copied / held per rank {[tuple(x.tolist()) for x in allc]}")
        ok &= e_loss < (4e-4 if (case.startswith("kl") or case == "hsic_all_n90") else 1e-4) and frac < 0.01
        # (rank 0 always holds tile rows and a result band: the bands were read)
        ok &= e_first <= 1e-6 and e_adj < 1e-3 and not over and int(allc[0][0]) > 0

    # n = 900 (several tile rows per rank), HSIC with c1 and c2 on row bands, against the oracle
    d = synthetic_case(900, 40, 5, measure="HSIC", weights={1: 1e-4, 2: 1e-4, 6: 2.0, 7: 3.0, 9: 1e-3, 10: 5.0}, epochs=3,
                       mean_deg=8.0)
    prob, cfg = O.problem_from_npz(d)
    ref = O.attack(prob, cfg, 3, x0=torch.from_numpy(d["x0"]))
    got, _, _ = run_row_bands(d)
    e_loss = float(np.max(np.abs(got["loss"] - np.array(ref["loss"])) / np.abs(np.array(ref["loss"]))))
    frac = float(np.mean(np.abs(np.stack(got["x_iters"]) - np.stack([x.numpy() for x in ref["x_iters"]])) > 2e-4))
    say(f"n=900 HSIC c1 + c2, row-band feature_adj, vs oracle: rel loss err {e_loss:.2e} frac|dx|>2e-4 {frac:.2e}")
    ok &= e_loss < 1e-4 and frac < 0.01

    # metric_pool_sharded against metric_pool on the gathered matrix; n = 90 over 3 ranks leaves one result band empty
    for case in ["hsic_all_n90", "hsic_B_n150"]:
        d = dict(np.load(os.path.join(ROOT, "tests", "golden", f"attack_{case}.npz")))
        got, _, _ = run_row_bands(d)
        mdl = got["model"]
        n = int(d["labels"].shape[0])
        ij = np.argwhere(d["adj"] != 0).T
        adj = torch.sparse_coo_tensor(torch.from_numpy(ij.astype(np.int64)), torch.ones(ij.shape[1]), (n, n)).coalesce()
        gathered = torch.from_numpy(got["modified_adj"]).to(dev)
        b0, b1 = mdl.modified_adj_rows
        for name, idx in (("idx_attack", d["idx_attack"]), ("subset", np.arange(n)[(np.arange(n) % 7) == 3]),
                          ("first band only", np.arange(min(n, 40))), ("arange(n)", np.arange(n))):
            s = metrics.metric_pool_sharded(adj, mdl.modified_adj, b0, n, idx)
            f = metrics.metric_pool(adj, gathered, idx)
            both = torch.tensor([s, -s], dtype=torch.float64, device=dev)
            dist.all_reduce(both, op=dist.ReduceOp.MAX)            # the same value on every rank
            say(f"{case} metric_pool_sharded {name}: {s:.9f} vs metric_pool {f:.9f} (rank 0; result band "
                f"[{b0}, {b1}))")
            ok &= abs(s - f) <= 1e-9 and float(both[0]) == -float(both[1])

    flag = torch.tensor([0 if ok else 1], dtype=torch.int64, device=dev)
    dist.all_reduce(flag)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_BANDS_OK" if int(flag) == 0 else "MGPU_BANDS_FAIL")
    sys.exit(0 if int(flag) == 0 else 1)


if __name__ == "__main__":
    main()
