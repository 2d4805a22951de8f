"""B200-native `baseline` -- the GraphMI baseline attack, same surface as the reference's MC-GRA/baseline.py.

`PGDAttack(model, embedding, nnodes, loss_type, device).attack(index_delete, lr_ori, ..., epochs)` keeps the reference's
signature (baseline.py:14-41) and side effects (`modified_adj`, `adj_changes.data`, returns the victim's last output).
The loop (baseline.py:52-86) is the supervised part of the MC-GRA loop -- expand, normalise, 2-layer GCN forward, nll +
0.001 ||x||, backward, Adam, budget projection -- so it runs on the same engine (engine.PGDEngine) with every prior
weight at zero; with `--density 1` the budget binds and the device bisection runs every iteration.
"""
import numpy as np
import scipy.sparse as sp
import torch
from torch.nn import functional as F
from torch.nn.parameter import Parameter

from . import _native as N
from ._native import call, ptr
from .base_attack import BaseAttack, RowBandResult
from .engine import HID, PGDEngine, output_band
from .topology_attack import PGDAttack as _MCGRA, _dense


class PGDAttack(RowBandResult, BaseAttack):

    def __init__(self, model=None, embedding=None, nnodes=None, loss_type='CE', feature_shape=None,
                 attack_structure=True, attack_features=False, device='cpu'):
        super(PGDAttack, self).__init__(model, nnodes, attack_structure, attack_features, device)
        assert attack_features or attack_structure, 'attack_features or attack_structure cannot be both False'
        self.loss_type = loss_type
        self.modified_adj = None
        self.modified_features = None
        self.edge_select = None
        self.complementary = None
        self.embedding = embedding
        self.engine = None
        if attack_structure:
            assert nnodes is not None, 'Please give nnodes='
            self.adj_changes = Parameter(torch.zeros(int(nnodes * (nnodes - 1) / 2)))
        if attack_features:
            assert True, 'Topology Attack does not support attack feature'

    # shared with the MC-GRA class: weight extraction, packed <-> dense helpers, decode, device bisection
    _victim_weights = _MCGRA._victim_weights
    _expand = _MCGRA._expand
    dot_product_decode = _MCGRA.dot_product_decode
    projection = _MCGRA.projection
    bisection = _MCGRA.bisection
    _loss = _MCGRA._loss

    plain_gd = False            # the MC-GPB variant (mcgpb_attack.PGDAttack) steps with plain gradient descent
    decode_normalised = True    # ... and decodes without row normalisation

    def _run(self, lr, weight_sup, ori_features, ori_adj, labels, idx_attack, num_edges, epochs, trace=False,
             setup=None, pre_iter=None, gather_x=True):
        if self.loss_type != 'CE':
            raise NotImplementedError("native path implements loss_type='CE' (the reference driver's choice)")
        dev = torch.device(self.device)
        n = self.nnodes
        self.engine = None
        self.modified_adj = None
        self.surrogate.eval()
        if self.embedding is not None:
            self.embedding.eval()
        W1, b1, W2, b2, Wl, bl = self._victim_weights()
        X = _dense(ori_features, dev)
        labels_t = torch.as_tensor(np.asarray(labels) if not torch.is_tensor(labels) else labels).long().to(dev)
        if torch.is_tensor(ori_adj):
            assert not bool(ori_adj.any()), "reference driver passes init_adj = 0 (dataset.py:433-437)"
        elif sp.issparse(ori_adj):
            assert ori_adj.nnz == 0, "reference driver passes init_adj = 0"
        else:
            assert not np.any(ori_adj), "reference driver passes init_adj = 0"
        with torch.no_grad():
            S1 = X @ W1
        rank, world = 0, 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            rank, world = torch.distributed.get_rank(), torch.distributed.get_world_size()
        x0 = self.adj_changes.data
        if bool(((x0 < 0) | (x0 > 1)).any()):
            raise NotImplementedError("a preset adj_changes must lie in [0, 1]: the reference does not clamp the forward "
                                      "of this attack (baseline.py:54)")
        x0 = x0 if bool((x0 != 0).any()) else None
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
        """Final decode: adj_changes.data = tril(relu(zf zf^T)), modified_adj its symmetric expansion.  One GPU
        holds all of both; with world > 1 a rank decodes only its tile rows and keeps only its row band of modified_adj
        (`modified_adj_rows`, engine.output_band), `gather_modified_adj()` assembles the full matrix."""
        st = N.stream_ptr()
        n, dev = eng.n, eng.dev
        # em = embedding(features, adj_norm of the last iteration) = hidden state of the normalised branch (:80-82)
        zf = torch.empty_like(eng.H2)
        if self.decode_normalised:
            call("mcgra_row_normalize", ptr(eng.H2), n, HID, 2.0, ptr(zf), st)
        else:
            zf.copy_(eng.H2)
        if eng.world == 1:
            T = eng.T
            xf = torch.empty(T * (T + 1) // 2 * N.TILE * N.TILE, dtype=torch.float32, device=dev)
            call("mcgra_decode_to_tiles", ptr(zf), n, 0, T, ptr(xf), st)
            packed = torch.empty(n * (n - 1) // 2, dtype=torch.float32, device=dev)
            call("mcgra_tiles_to_tril", ptr(xf), n, 0, T, None, 1, ptr(packed), st)
            self.adj_changes.data = packed
            out = torch.zeros(n, n, dtype=torch.float32, device=dev)
            call("mcgra_tiles_to_dense", ptr(xf), n, 0, T, None, 1, ptr(out), n, st)
            self.modified_adj = out.detach()
            self.modified_adj_rows = (0, n)
            return
        # every value below equals the single-GPU one bit for bit (mcgra_decode_band is the tiles' symmetric expansion)
        if gather_x:        # the reference leaves the full packed vector in adj_changes.data (`_gather_x=False`: skip it)
            # every rank writes its tile rows' entries into a zeroed vector and the vectors are summed
            xf = torch.empty(max(eng.ntiles, 1) * N.TILE * N.TILE, dtype=torch.float32, device=dev)
            call("mcgra_decode_to_tiles", ptr(zf), n, eng.tr0, eng.tr1, ptr(xf), st)
            packed = torch.zeros(n * (n - 1) // 2, dtype=torch.float32, device=dev)
            call("mcgra_tiles_to_tril", ptr(xf), n, eng.tr0, eng.tr1, None, 1, ptr(packed), st)
            del xf
            eng._allreduce(packed)
            self.adj_changes.data = packed
        b0, b1 = output_band(n, eng.rank, eng.world)
        out = torch.empty(max(b1 - b0, 0), n, dtype=torch.float32, device=dev)
        call("mcgra_decode_band", ptr(zf), n, b0, b1, ptr(out), n, st)
        self.modified_adj = out.detach()
        self.modified_adj_rows = (b0, b1)

    def attack(self, index_delete, lr_ori, weight_aux, weight_supervised, weight_param, feature_adj,
               aux_adj, aux_feature, aux_num_edges, idx_train, idx_val, idx_test, adj,
               ori_features, ori_adj, labels, idx_attack, num_edges,
               dropout_rate, epochs=200, sample=False, **kwargs):
        """baseline.py:36-86.  (`sample=True` only changes an unused local `lr` in the reference, :72-74.)"""
        return self._run(lr_ori, 1.0, ori_features, ori_adj, labels, idx_attack, num_edges, epochs,
                         trace=bool(kwargs.get("_trace")), gather_x=kwargs.get("_gather_x", True))

    def get_modified_adj(self, ori_adj=None):
        return self._expand(self.adj_changes.data, ori_adj)

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
