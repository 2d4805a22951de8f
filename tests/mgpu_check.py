"""Run under torchrun: the sharded attack must reproduce the single-GPU golden fixtures.

One rank per GPU over NCCL; with --gloo every rank runs on cuda:0 over gloo (the same code path and collectives on a
one-GPU box)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    gloo = "--gloo" in sys.argv
    dev = torch.device("cuda", 0 if gloo else int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo" if gloo else "nccl", **({} if gloo else {"device_id": dev}))
    import pgd_oracle as O
    from helpers import run_native_case, synthetic_case
    rank = dist.get_rank()
    ok = True
    for case in ["mse_A_n150", "mse_all_n150", "mse_budget_n150"]:
        d = np.load(os.path.join(ROOT, "tests", "golden", f"attack_{case}.npz"))
        got = run_native_case(d, device=dev)
        e_loss = float(np.max(np.abs(got["loss"] - d["loss"]) / np.abs(d["loss"])))
        e_x = float(np.max(np.abs(np.stack(got["x_iters"]) - d["x_iters"])))
        e_adj = float(np.max(np.abs(got["modified_adj"] - d["modified_adj"])))
        if rank == 0:
            print(f"[mgpu world={dist.get_world_size()}] {case}: rel loss err {e_loss:.2e} max|dx| {e_x:.2e} "
                  f"max|dadj| {e_adj:.2e}")
        ok &= e_loss < 1e-4 and e_x < 5e-5 and e_adj < 2e-3
    # the dense-contraction measures (row-panel GEMMs + all-gather) and the KL tile passes (row statistics all-reduced):
    # sharded loss against the single-GPU golden, robust x comparison as in tests/test_gpu_attack.py
    for case in ["hsic_B_n150", "hsic_all_n90", "cka_n90", "dp_n90", "kl_all_n90", "kl_C_n150", "kde_n90", "kde_readme_n150"]:
        d = np.load(os.path.join(ROOT, "tests", "golden", f"attack_{case}.npz"))
        got = run_native_case(d, device=dev)
        e_loss = float(np.max(np.abs(got["loss"] - d["loss"]) / np.abs(d["loss"])))
        if case.startswith("kde"):
            # the reference's fp32 MutualInformation is itself 1e-4 .. 1e-3 from its fp64 value (tests/test_oracle_golden.py::
            # test_kde_reference_fp32_is_off_its_fp64): hold the sharded run to the fp64 oracle at its own parameter
            prob64, cfg64 = O.problem_from_npz(d, dtype=torch.float64)
            xs_prev = [d["x0"]] + got["x_iters"][:-1]
            forced = np.array([float(O.iteration_terms(torch.from_numpy(np.asarray(xp)).double(), prob64, cfg64)[0]) for xp in xs_prev])
            e_loss = float(np.max(np.abs(np.asarray(got["loss"]) - forced) / np.abs(forced)))
        dx = np.abs(np.stack(got["x_iters"]) - d["x_iters"])
        frac = float(np.mean(dx > 2e-4))
        if rank == 0:
            print(f"[mgpu world={dist.get_world_size()}] {case}: rel loss err {e_loss:.2e} frac|dx|>2e-4 {frac:.2e}"
                  + (" (loss vs fp64 oracle at the native parameter)" if case.startswith("kde") else ""))
        # (kl_* and hsic_all_n90 are the listed tie-break cases of tests/test_gpu_attack.py: their free-running fp32
        #  trajectories are allowed to separate from the reference's by more than 1e-4)
        ok &= e_loss < (4e-4 if (case.startswith("kl") or case == "hsic_all_n90") else 1e-4) and frac < 0.01
    # row-band input (every rank holds only the rows of feature_adj it touches) + sharded AUC / AP against the
    # single-process values of the full matrix
    from mcgra_b200 import metrics
    from mcgra_b200.engine import HostBands, TILE, output_band, shard_tile_rows
    import helpers
    d = dict(np.load(os.path.join(ROOT, "tests", "golden", "attack_mse_all_n150.npz")))
    n = int(d["labels"].shape[0])
    world = dist.get_world_size()
    T = (n + TILE - 1) // TILE
    tr0, tr1 = shard_tile_rows(T, world)[rank]
    fa_full = torch.from_numpy(d["feature_adj"])
    bands = {}
    for r0, r1 in {(tr0 * TILE, min(n, tr1 * TILE)), output_band(n, rank, world)}:
        if r1 > r0:
            bands[(r0, r1)] = fa_full[r0:r1].clone().pin_memory()
    orig_from_numpy = torch.from_numpy
    d_b = dict(d)
    d_b["feature_adj"] = d["feature_adj"]
    _rn = helpers.run_native_case

    class _FA:       # run_native_case does torch.from_numpy(d["feature_adj"]): hand it the band object instead
        pass
    torch_from = torch.from_numpy
    hb = HostBands(n, bands)
    torch.from_numpy = lambda a: hb if a is d_b["feature_adj"] else torch_from(a)
    try:
        got = run_native_case(d_b, device=dev)
    finally:
        torch.from_numpy = torch_from
    e_loss = float(np.max(np.abs(got["loss"] - d["loss"]) / np.abs(d["loss"])))
    e_adj = float(np.max(np.abs(got["modified_adj"] - d["modified_adj"])))
    mdl = got["model"]
    ee = np.argwhere(np.triu(d["adj"], 1) > 0)
    auc_s, ap_s = metrics.auc_ap_from_edges_sharded(mdl.modified_adj, mdl.modified_adj_rows[0], n, ee)
    real = d["adj"].reshape(-1).astype(np.float32)
    auc_f, ap_f = O.roc_auc(real, got["modified_adj"].reshape(-1)), O.average_precision(real, got["modified_adj"].reshape(-1))
    if rank == 0:
        print(f"[mgpu] row-band feature_adj: rel loss err {e_loss:.2e} max|dadj| {e_adj:.2e}; sharded AUC {auc_s:.6f} / AP {ap_s:.6f} "
              f"vs full-matrix {auc_f:.6f} / {ap_f:.6f}")
    ok &= e_loss < 1e-4 and e_adj < 2e-3 and abs(auc_s - auc_f) < 1e-9 and abs(ap_s - ap_f) < 1e-9
    # a multi-tile case with an active budget against the oracle
    d = synthetic_case(900, 40, 5, weights={1: 0.5, 2: 0.3, 6: 2.0, 7: 3.0, 9: 1.5, 10: 50.0}, epochs=3, density=1.0,
                       mean_deg=8.0)
    prob, cfg = O.problem_from_npz(d)
    ref = O.attack(prob, cfg, 3, x0=torch.from_numpy(d["x0"]))
    got = run_native_case(d, device=dev)
    e_loss = float(np.max(np.abs(got["loss"] - np.array(ref["loss"])) / np.abs(np.array(ref["loss"]))))
    e_x = max(float(np.max(np.abs(a - b.numpy()))) for a, b in zip(got["x_iters"], ref["x_iters"]))
    if rank == 0:
        print(f"[mgpu] n=900 budget-active vs oracle: rel loss err {e_loss:.2e} max|dx| {e_x:.2e}")
    ok &= e_loss < 1e-4 and e_x < 2e-4
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_OK" if ok else "MGPU_FAIL")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
