"""B200-native `baseline` -- the GraphMI baseline attack, same surface as the reference's MC-GRA/baseline.py.

`PGDAttack(model, embedding, nnodes, loss_type, device).attack(index_delete, lr_ori, ..., epochs)` keeps the reference's
signature (baseline.py:14-41) and side effects (`modified_adj`, `adj_changes.data`, returns the victim's last output).
The loop (baseline.py:52-86) is the supervised part of the MC-GRA loop -- expand, normalise, 2-layer GCN forward, nll +
0.001 ||x||, backward, Adam, budget projection -- so it runs on the same engine (engine.PGDEngine) with every prior
weight at zero; with `--density 1` the budget binds and the device bisection runs every iteration.
"""
import torch
from torch.nn import functional as F

from . import _native as N
from ._native import call, ptr
from .base_attack import RowBandResult
from .engine import HID, PGDEngine, output_band


class PGDAttack(RowBandResult):
    plain_gd = False            # the MC-GPB variant (mcgpb_attack.PGDAttack) steps with plain gradient descent
    decode_normalised = True    # ... and decodes without row normalisation

    def _run(self, lr, weight_sup, ori_features, ori_adj, labels, idx_attack, num_edges, epochs, trace=False,
             setup=None, pre_iter=None, gather_x=True):
        dev = torch.device(self.device)
        n = self.nnodes
        (W1, b1, W2, b2, Wl, bl), X, labels_t, (rank, world), x0 = self._prepare(ori_features, ori_adj, labels)
        with torch.no_grad():
            S1 = X @ W1
        if x0 is not None and bool(((x0 < 0) | (x0 > 1)).any()):
            raise NotImplementedError("a preset adj_changes must lie in [0, 1]: the reference does not clamp the forward "
                                      "of this attack (baseline.py:54)")
        zeros16 = torch.zeros(n, HID, device=dev)
        zerosc = torch.zeros(n, Wl.shape[0], device=dev)
        self.engine = eng = PGDEngine(n, S1, W2, b1, b2, Wl, bl, labels_t, idx_attack, zeros16, zerosc, None, "MSELoss",
                                      (0,) * 10, lr, weight_sup=weight_sup, num_edges=num_edges, x0=x0, device=dev,
                                      rank=rank, world=world, max_epochs=max(int(epochs), 1), plain_gd=self.plain_gd)
        if setup is not None:
            setup(eng, X)
        self._trace = []
        for t in range(int(epochs)):
            if pre_iter is not None:
                pre_iter(eng, t)
            eng.iterate()
            if trace:
                self._trace.append(eng.packed_parameter())
        if int(epochs) == 0:
            eng.forward_stages(0)
        self._finalize(eng, gather_x)
        return F.log_softmax(eng.H2 @ Wl.t() + bl, dim=1).detach()       # victim output of the last iteration

    def _finalize(self, eng, gather_x=True):
        """Final decode: adj_changes.data = tril(relu(zf zf^T)), modified_adj its symmetric expansion.  With world > 1 a
        rank decodes only its tile rows and keeps only its row band of modified_adj (`modified_adj_rows`,
        engine.output_band), `gather_modified_adj()` assembles the full matrix; one GPU's band is all n rows."""
        zf = self._decode_last(eng, gather_x, self.decode_normalised)[0]        # (:80-82); its tiles are freed here
        # mcgra_decode_band is the decoded tiles' symmetric expansion, bit for bit
        b0, b1 = output_band(eng.n, eng.rank, eng.world)
        out = torch.empty(max(b1 - b0, 0), eng.n, dtype=torch.float32, device=eng.dev)
        call("mcgra_decode_band", ptr(zf), eng.n, b0, b1, ptr(out), eng.n, N.stream_ptr())
        self.modified_adj = out.detach()
        self.modified_adj_rows = (b0, b1)

    def attack(self, index_delete, lr_ori, weight_aux, weight_supervised, weight_param, feature_adj,
               aux_adj, aux_feature, aux_num_edges, idx_train, idx_val, idx_test, adj,
               ori_features, ori_adj, labels, idx_attack, num_edges,
               dropout_rate, epochs=200, sample=False, **kwargs):
        """baseline.py:36-86.  (`sample=True` only changes an unused local `lr` in the reference, :72-74.)"""
        return self._run(lr_ori, 1.0, ori_features, ori_adj, labels, idx_attack, num_edges, epochs,
                         trace=bool(kwargs.get("_trace")), gather_x=kwargs.get("_gather_x", True))

    def get_modified_adj2(self):
        return self._expand(self.adj_changes.data, None)

    def feature_smoothing(self, adj, X):
        """tr(X^T L~ X), L~ = D~^-1/2 (D - A) D~^-1/2, D~ = D + 1e-3 (baseline.py:155-169) without the dense-diagonal
        products: sum_i r_i^2 d_i |x_i|^2 - sum_ij r_i A_ij r_j <x_i, x_j>.  Helper outside the loop (the reference's loop
        never reaches it: `if t > -1`, :56)."""
        d = adj.sum(1).flatten()
        r = (d + 1e-3).pow(-0.5)
        r = torch.where(torch.isinf(r), torch.zeros_like(r), r)
        Xr = r[:, None] * X
        return (d * (Xr * Xr).sum(1)).sum() - ((adj @ Xr) * Xr).sum()

    def filter(self, Z):
        return torch.where(Z > 0.9, Z, torch.zeros_like(Z))
