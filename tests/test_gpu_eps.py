"""attack() with adjacency noise (--eps != 0; MC-GRA/topology_attack.py:165, 474-478) on the native path: the reference's
golden fixture, multi-tile trajectories and the gradient itself against the CPU oracle fed with the same draws, engine
agreement, the default torch stream, and the scope guards."""
import os
import tempfile

import numpy as np
import pytest
import torch

import pgd_oracle as O
from helpers import engines, make_args, make_models, synthetic_case

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL_SIX = {1: 0.5, 2: 0.3, 6: 2.0, 7: 3.0, 9: 1.5, 10: 50.0}


def draws(seed, n, count, device="cpu"):
    """The reference's stream: manual_seed, then one n x n fp32 torch.randn per iteration (tests/golden/make_golden.py)."""
    if device == "cpu":
        torch.manual_seed(seed)
    else:
        torch.cuda.manual_seed(seed)
    return [torch.randn((n, n), dtype=torch.float32, device=device) for _ in range(count)]


def run_noisy(d, noise=None, epochs=None, measure=None, **kw):
    """PGDAttack.attack as main.objective drives it, with the test hook `_noise` (None: the default draw)."""
    from mcgra_b200.topology_attack import PGDAttack
    dev = torch.device("cuda:0")
    n = int(d["labels"].shape[0])
    victim, emb = make_models(d, dev)
    args = make_args(d)
    if measure is not None:
        args.measure = measure
    model = PGDAttack(model=victim, embedding=emb, H_A=torch.from_numpy(d["H_A2"]).to(dev),
                      Y_A=torch.from_numpy(d["Y_A"]).to(dev), nnodes=n, loss_type="CE", device=dev).to(dev)
    if np.any(d["x0"] != 0):
        model.adj_changes.data = torch.from_numpy(d["x0"].copy()).to(dev)
    epochs = int(d["epochs"]) if epochs is None else epochs
    if noise is not None:
        kw["_noise"] = lambda t: noise[t]
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)
        try:
            model.attack(args, None, 10 ** float(d["lr_exp"]), 0, float(d["weight_sup"]), tuple(d["weights"]),
                         torch.from_numpy(d["feature_adj"]), 0, 0, 0, None, None, np.arange(min(8, n)),
                         torch.from_numpy(d["adj"].astype(np.float32)), d["X"], np.zeros((n, n), np.float32), d["labels"],
                         d["idx_attack"], int(d["num_edges"]), 0, epochs=epochs, _trace=True, **kw)
        finally:
            os.chdir(cwd)
    torch.cuda.synchronize()
    return dict(loss=model.engine.losses()["loss"], x_iters=[x.cpu().numpy() for x in model._trace],
                x_final=model.adj_changes.data.cpu().numpy(), modified_adj=model.gather_modified_adj().cpu().numpy(),
                model=model)


def oracle_noisy(d, noise, epochs, dtype=torch.float32):
    """O.attack's loop with the draw of iteration t passed to iteration_terms (O.attack draws its own)."""
    prob, cfg = O.problem_from_npz(d, dtype=dtype)
    x = torch.from_numpy(d["x0"].copy()).to(dtype)
    m, v = torch.zeros_like(x), torch.zeros_like(x)
    losses, xs = [], []
    A_hat = None
    for t in range(epochs):
        xr = x.clone().requires_grad_(True)
        loss, _, A_hat = O.iteration_terms(xr, prob, cfg, noise=noise[t].cpu().to(dtype))
        loss.backward()
        losses.append(float(loss.detach().double()))
        O.adam_update(x, xr.grad, m, v, t + 1, cfg["lr"])
        x = torch.clamp(O.projection(x, cfg["num_edges"]), 0, 1)
        xs.append(x.clone())
        A_hat = A_hat.detach()
    x_final, cur = O.finalize(prob, cfg, A_hat)
    return dict(loss=np.array(losses), x_iters=xs, x_final=x_final, modified_adj=cur)


def noisy_case(eps, density=1e7, epochs=3):
    d = synthetic_case(700, 40, 5, weights=ALL_SIX, epochs=epochs, density=density, mean_deg=8.0, x0_scale=0.4)
    d["eps"] = np.float64(eps)
    return d


def test_eps_golden_matches_reference():
    d = np.load(os.path.join(GOLDEN, "attack_mse_eps_n37.npz"))
    n, T = int(d["labels"].shape[0]), int(d["epochs"])
    got = run_noisy(d, noise=draws(int(d["noise_seed"]), n, T))
    rel = np.max(np.abs(np.asarray(got["loss"]) - d["loss"]) / np.abs(d["loss"]))
    print(f"[eps] golden n37: max rel loss err {rel:.3e}")
    assert rel <= 1e-4
    assert np.max(np.abs(np.stack(got["x_iters"]) - d["x_iters"])) < 2e-4
    np.testing.assert_allclose(got["x_final"], d["x_final"], rtol=1e-3, atol=2e-4)
    np.testing.assert_allclose(got["modified_adj"], d["modified_adj"], rtol=1e-3, atol=1e-3)
    real = d["adj"].reshape(-1).astype(np.float32)
    tol = max(1e-3, 2.0 / float(real.sum()))
    assert abs(O.roc_auc(real, got["modified_adj"].reshape(-1)) - float(d["auc"])) < tol
    assert abs(O.average_precision(real, got["modified_adj"].reshape(-1)) - float(d["ap"])) < tol


@pytest.mark.parametrize("eps,density", [(0.05, 1e7), (0.5, 1e7), (0.05, 1.0)])
def test_eps_multi_tile_matches_oracle(eps, density):
    """n = 700 (ragged last tile row), all six weights; eps = 0.5 clamps heavily at both ends; density = 1 binds the
    budget every iteration (bisection on the lazily projected view)."""
    d = noisy_case(eps, density)
    noise = draws(31, 700, 3)
    ref = oracle_noisy(d, noise, 3)
    got = run_noisy(d, noise=noise)
    print(f"[eps] n700 eps={eps} density={density}: max rel loss err "
          f"{np.max(np.abs(np.asarray(got['loss']) - ref['loss']) / np.abs(ref['loss'])):.3e}")
    np.testing.assert_allclose(got["loss"], ref["loss"], rtol=1e-4)
    for a, b in zip(got["x_iters"], ref["x_iters"]):
        assert np.max(np.abs(a - b.numpy())) < 2e-4
    np.testing.assert_allclose(got["modified_adj"], ref["modified_adj"].numpy(), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("eps", [0.05, 0.5])
def test_eps_gradient_matches_autograd(eps):
    """After one iteration the first Adam moment is (1 - beta1) g: compared entry by entry with the oracle's autograd
    gradient at the same draw (fp64), which pins the masks, the orientation of every product and rho."""
    from mcgra_b200 import _native as N
    d = noisy_case(eps, epochs=1)
    n = 700
    noise = draws(7, n, 1)
    got = run_noisy(d, noise=noise, epochs=1)
    eng = got["model"].engine
    m = torch.zeros(n * (n - 1) // 2, dtype=torch.float32, device="cuda")
    N.call("mcgra_tiles_to_tril", N.ptr(eng.mt), n, 0, eng.T, None, 2, N.ptr(m), N.stream_ptr())
    g_native = (m.double() / 0.1).cpu().numpy()
    prob, cfg = O.problem_from_npz(d, dtype=torch.float64)
    xr = torch.from_numpy(d["x0"].copy()).double().requires_grad_(True)
    loss, _, _ = O.iteration_terms(xr, prob, cfg, noise=noise[0].double())
    loss.backward()
    g_ref = xr.grad.numpy()
    err = np.max(np.abs(g_native - g_ref)) / np.max(np.abs(g_ref))
    print(f"[eps] gradient eps={eps}: max |dg| / max |g| = {err:.3e}")
    assert err < 1e-4


@pytest.mark.parametrize("which", [0, 1])
def test_eps_exact_engines_agree(which):
    """exact-fp32 FFMA propagate (0) / fold (1) against the default tensor-core engines on the noisy path."""
    d = noisy_case(0.05)
    noise = draws(11, 700, 3)
    with engines({which: 0}):
        a = run_noisy(d, noise=noise)
    b = run_noisy(d, noise=noise)
    np.testing.assert_allclose(a["loss"], b["loss"], rtol=5e-6)
    assert np.max(np.abs(np.stack(a["x_iters"]) - np.stack(b["x_iters"]))) < 2e-5


def test_eps_default_stream_is_the_references():
    """No hook: the native path draws torch.randn((n, n)) on the attack's device, i.e. what the reference's
    torch.randn_like(M) draws there after the same seed."""
    d = noisy_case(0.05)
    torch.cuda.manual_seed(1234)
    got = run_noisy(d)
    ref = oracle_noisy(d, draws(1234, 700, 3, device="cuda"), 3)
    np.testing.assert_allclose(got["loss"], ref["loss"], rtol=1e-4)


@pytest.mark.parametrize("measure", ["KL", "HSIC"])
def test_eps_other_measures_raise(measure):
    d = np.load(os.path.join(GOLDEN, "attack_mse_eps_n37.npz"))
    with pytest.raises(NotImplementedError, match="eps"):
        run_noisy(d, measure=measure)


def test_eps_cli(tmp_path, monkeypatch):
    from mcgra_b200 import main as cli
    monkeypatch.chdir(tmp_path)
    auc = cli.main(["--dataset", "synthetic:2000:64:4", "--measure", "MSELoss", "--w1", "0.01", "--w6", "10", "--w7", "10",
                    "--w9", "10", "--w10", "1000", "--lr", "-2", "--useH_A", "--useY_A", "--useY", "--eps", "0.01",
                    "--epochs", "5", "--log_name", "eps_test.log"])
    assert 0.5 < float(auc) <= 1.0
