"""Round-2 debug probes (GPU): dense HSIC stage at n=1490, pairs engine 2 vs 0, GraphMI baseline x trace."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import pgd_oracle as O
from helpers import engines, run_native_case, synthetic_case, make_models
from mcgra_b200 import _native as N
GOLDEN = os.path.join(ROOT, "tests", "golden")
dev = torch.device("cuda:0")


def nanstat(name, t):
    t = t.float()
    print(f"   {name}: nan {int(torch.isnan(t).sum())} inf {int(torch.isinf(t).sum())} absmax {float(t[torch.isfinite(t)].abs().max()) if torch.isfinite(t).any() else -1:.3e}")


def probe_polblogs():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_parity_sizes import _real_case
    r, d = _real_case("polblogs", 3)
    from mcgra_b200.topology_attack import PGDAttack
    print("== polblogs real, HSIC, c1 inactive")
    got = run_native_case(d, trace=True)
    print("   native loss", got["loss"], " reference", r["loss_short"][:3])
    eng = got["model"].engine
    for nm in ("Ft", "Ct", "Fdiag", "rho", "xt", "mt", "vt", "dzhat", "eps_row"):
        nanstat(nm, getattr(eng, nm))
    terms = got["terms"]
    print("   terms c1", terms["c1"], "c2", terms["c2"], "c6", terms["c6"], "c7", terms["c7"], "c9", terms["c9"], "c10", terms["c10"], "origin", terms["origin"])
    prob, cfg = O.problem_from_npz(d, dtype=torch.float64)
    l0, t0, _ = O.iteration_terms(torch.zeros(prob["n"] * (prob["n"] - 1) // 2, dtype=torch.float64), prob, cfg)
    print("   fp64 oracle at x=0: loss", float(l0), {k: float(v) for k, v in t0.items()})
    x1 = torch.from_numpy(got["x_iters"][0]).double()
    l1, t1, _ = O.iteration_terms(x1, prob, cfg)
    print("   fp64 oracle at native x1: loss", float(l1), {k: float(v) for k, v in t1.items()})
    ref = O.attack(O.problem_from_npz(d)[0], O.problem_from_npz(d)[1], 1)
    dx = np.abs(got["x_iters"][0] - ref["x_iters"][0].numpy())
    print("   x after iteration 0 vs fp32 oracle: max", dx.max(), "frac>2e-4", (dx > 2e-4).mean(), " native x1 stats", got["x_iters"][0].min(), got["x_iters"][0].max(), got["x_iters"][0].mean(), "oracle mean", float(ref["x_iters"][0].mean()))


def probe_pairs():
    print("== pairs engine 0 vs 2 (raw kernel call)")
    for n in (150, 1300, 4500):
        g = torch.Generator().manual_seed(n)
        z = torch.nn.functional.normalize(torch.relu(torch.randn(n, 16, generator=g)), dim=1).to(dev).contiguous()
        T = (n + 127) // 128
        k7 = -10.0 * 10 / n / n
        outs = {}
        for eng in (0, 2):
            dz = torch.zeros(n, 16, device=dev)
            acc = torch.zeros(32, dtype=torch.float64, device=dev)
            eps = torch.zeros(n, device=dev)
            r = torch.ones(n, device=dev)
            ws = torch.empty(int(N.lib().mcgra_pairs_ws_bytes(n)), dtype=torch.uint8, device=dev)
            tiles = torch.zeros(T * (T + 1) // 2 * 128 * 128, device=dev)
            with engines({2: eng}):
                N.call("mcgra_pairs", N.ptr(tiles), n, 0, T, None, 2, N.ptr(z), N.ptr(r), k7, 0.0, None, None, N.ptr(dz),
                       N.ptr(eps), N.ptr(acc), N.ptr(ws), N.stream_ptr())
                torch.cuda.synchronize()
            outs[eng] = (float(acc[4]), dz.clone())
        S = (z.double() @ z.double().t())
        q = S.clamp(min=0).clamp(1e-4, 1 - 1e-4)
        ref = float(k7 * (torch.tril(2 * q * torch.log2(q), -1)).sum())
        c0, c2 = outs[0][0], outs[2][0]
        ddz = (outs[0][1] - outs[2][1]).abs()
        per_row = ddz.max(1).values
        bad = torch.nonzero(per_row > 1e-3 * outs[0][1].abs().max()).flatten()
        print(f"   n={n}: c7 fp64 {ref:.9e} eng0 {c0:.9e} eng2 {c2:.9e} rel2 {(c2 - ref) / ref:.2e} rel0 {(c0 - ref) / ref:.2e}; "
              f"dz max diff {float(ddz.max()):.3e} of {float(outs[0][1].abs().max()):.3e}; bad rows {bad.numel()} first {bad[:12].tolist()}")


def probe_baseline():
    print("== GraphMI baseline free_n90")
    from mcgra_b200.baseline import PGDAttack
    d = np.load(os.path.join(GOLDEN, "baseline_free_n90.npz"))
    n = int(d["labels"].shape[0])
    victim, emb = make_models(d, dev)
    model = PGDAttack(model=victim, embedding=emb, nnodes=n, loss_type="CE", device=dev).to(dev)
    model.attack(None, float(d["lr"]), 0, 1.0, None, None, 0, 0, 0, None, None, None, torch.from_numpy(d["adj"].astype(np.float32)),
                 d["X"], np.zeros((n, n), np.float32), d["labels"], d["idx_attack"], int(d["num_edges"]), 0, epochs=3, _trace=True)
    loss = model.engine.losses()
    print("   native loss", loss["loss"], "golden", d["loss"][:3], "origin", loss["origin"])
    for k in range(3):
        a, b = model._trace[k].cpu().numpy(), d["x_iters"][k]
        dx = np.abs(a - b)
        print(f"   iter {k}: max|dx| {dx.max():.3e} frac>2e-4 {(dx > 2e-4).mean():.3e}; native nonzero {int((a != 0).sum())} golden nonzero {int((b != 0).sum())}; "
              f"where golden==0 native max {a[b == 0].max():.3e}; where native==0 golden max {b[a == 0].max() if (a == 0).any() else 0:.3e}")


if __name__ == "__main__":
    which = sys.argv[1:] or ["polblogs", "pairs", "baseline"]
    if "pairs" in which:
        probe_pairs()
    if "baseline" in which:
        probe_baseline()
    if "polblogs" in which:
        probe_polblogs()
