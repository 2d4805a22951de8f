"""Attack base class -- same surface as the reference's `base_attack.BaseAttack`
(MC-GRA/base_attack.py:11-119): stores surrogate, nnodes, device, modified_adj; check_adj / save helpers."""
import os.path as osp

import numpy as np
import scipy.sparse as sp
import torch
from torch.nn.modules.module import Module


class BaseAttack(Module):
    def __init__(self, model, nnodes, attack_structure=True, attack_features=False, device='cpu'):
        super(BaseAttack, self).__init__()
        self.surrogate = model
        self.nnodes = nnodes
        self.attack_structure = attack_structure
        self.attack_features = attack_features
        self.device = device
        self.modified_adj = None
        self.modified_features = None
        if model is not None:
            self.nclass = model.nclass
            self.nfeat = model.nfeat
            self.hidden_sizes = model.hidden_sizes

    def attack(self, ori_adj, n_perturbations, **kwargs):
        pass

    def check_adj(self, adj):
        """Symmetric, unweighted, zero-diagonal check (base_attack.py:60-71)."""
        if type(adj) is torch.Tensor:
            adj = adj.cpu().numpy()
        assert np.abs(adj - adj.T).sum() == 0, "Input graph is not symmetric"
        if sp.issparse(adj):
            assert adj.tocsr().max() == 1, "Max value should be 1!"
            assert adj.tocsr().min() == 0, "Min value should be 0!"
        else:
            assert adj.max() == 1, "Max value should be 1!"
            assert adj.min() == 0, "Min value should be 0!"

    def save_adj(self, root=r'/tmp/', name='mod_adj'):
        assert self.modified_adj is not None, 'modified_adj is None! Please perturb the graph first.'
        name = name + '.npz'
        modified_adj = self.modified_adj
        if type(modified_adj) is torch.Tensor:
            modified_adj = sp.csr_matrix(modified_adj.detach().cpu().numpy())
        sp.save_npz(osp.join(root, name), modified_adj)

    def save_features(self, root=r'/tmp/', name='mod_features'):
        assert self.modified_features is not None, 'modified_features is None! Please perturb the graph first.'
        name = name + '.npz'
        modified_features = self.modified_features
        if type(modified_features) is torch.Tensor:
            modified_features = sp.csr_matrix(modified_features.detach().cpu().numpy())
        sp.save_npz(osp.join(root, name), modified_features)


class RowBandResult:
    """The n x n result of the native attacks on several GPUs: with world > 1 every rank holds only its row band
    `modified_adj` = rows [b0, b1) (`modified_adj_rows`, engine.output_band) of its PGDEngine `self.engine`."""

    def gather_modified_adj(self):
        """Full n x n result on every rank from the row bands (world > 1); identity otherwise."""
        eng = self.engine
        if eng is None or eng.world == 1:
            return self.modified_adj
        import torch.distributed as dist
        from .engine import output_band
        n = eng.n
        rb = output_band(n, 0, eng.world)[1]
        mine = torch.zeros(rb, n, dtype=torch.float32, device=eng.dev)
        mine[:self.modified_adj.shape[0]] = self.modified_adj
        full = torch.empty(eng.world * rb, n, dtype=torch.float32, device=eng.dev)
        dist.all_gather_into_tensor(full, mine, group=eng.group)
        return full[:n]

    def recovered_edges(self, k):
        """The reconstructed graph: the k highest-scoring node pairs (i < j) of `modified_adj`, as (rows, cols, scores)
        device tensors in (score desc, i * n + j asc) order (metrics.topk_pairs).  With world > 1 each rank passes its
        row band and every rank returns the same result (metrics.topk_pairs_sharded)."""
        if self.modified_adj is None:
            raise RuntimeError("recovered_edges() needs the scores of attack(): call attack() first")
        from .metrics import topk_pairs, topk_pairs_sharded
        eng = self.engine
        if eng is not None and eng.world > 1:
            return topk_pairs_sharded(self.modified_adj, self.modified_adj_rows[0], self.nnodes, k, group=eng.group)
        return topk_pairs(self.modified_adj, k)
