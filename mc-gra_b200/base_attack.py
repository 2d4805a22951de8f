"""Attack base classes -- `BaseAttack` has the surface of the reference's `base_attack.BaseAttack`
(MC-GRA/base_attack.py:11-119): stores surrogate, nnodes, device, modified_adj; check_adj / save helpers.
`RowBandResult` is what the native attacks (MC-GRA, GraphMI) share on top of it."""
import os.path as osp

import numpy as np
import scipy.sparse as sp
import torch
from torch.nn import functional as F
from torch.nn.modules.module import Module
from torch.nn.parameter import Parameter

from . import _native as N
from ._native import call, ptr
from .engine import BISECT_PASSES, HID, bisect, output_band, packed_to_tiles, tile_buffer, tiles_to_packed


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


def _dense(t, device):
    if sp.issparse(t):
        t = np.asarray(t.todense())
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(t))
    if t.is_sparse:
        t = t.to_dense()
    return t.to(device=device, dtype=torch.float32)


def _rank_world():
    """(rank, world size) of the default process group; (0, 1) without one."""
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        return torch.distributed.get_rank(), torch.distributed.get_world_size()
    return 0, 1


class RowBandResult(BaseAttack):
    """Base of the native attacks: the victim's weights and the inputs on the device, the decode of the last embedding
    into `adj_changes`, the reference's stand-alone helpers, and the n x n result on several GPUs: with world > 1 every
    rank holds only its row band `modified_adj` = rows [b0, b1) (`modified_adj_rows`, engine.output_band) of its
    PGDEngine `self.engine`."""

    def __init__(self, model=None, embedding=None, nnodes=None, loss_type='CE', feature_shape=None,
                 attack_structure=True, attack_features=False, device='cpu'):
        super().__init__(model, nnodes, attack_structure, attack_features, device)
        assert attack_features or attack_structure, 'attack_features or attack_structure cannot be both False'
        self.loss_type = loss_type
        self.edge_select = None
        self.complementary = None
        self.embedding = embedding
        self.engine = None
        if attack_structure:
            assert nnodes is not None, 'Please give nnodes='
            self.adj_changes = Parameter(torch.zeros(int(nnodes * (nnodes - 1) / 2)))
        if attack_features:
            assert True, 'Topology Attack does not support attack feature'

    def _victim_weights(self):
        victim, emb = self.surrogate, self.embedding
        if len(victim.gc) != 2:
            raise NotImplementedError("native path is built for the 2-layer GCN victim (main.py --nlayers 2)")
        W1, b1 = victim.gc[0].weight, victim.gc[0].bias
        W2, b2 = victim.gc[1].weight, victim.gc[1].bias
        Wl, bl = victim.linear1.weight, victim.linear1.bias
        if W1.shape[1] != HID or W2.shape != (HID, HID):
            raise NotImplementedError("native path is built for nhid=16 (hard-coded in the reference, main.py:175)")
        if b1 is None or b2 is None or bl is None:
            raise NotImplementedError("with_bias=False victims are not supported")
        if not getattr(victim, "with_relu", True):
            raise NotImplementedError("with_relu=False victims are not supported (the native path hard-codes the relu)")
        if emb is not None:
            for k in range(2):   # embedding.gc = deepcopy(victim.gc) in the reference driver (main.py:185-190)
                if not (torch.equal(emb.gc[k].weight.detach().cpu(), victim.gc[k].weight.detach().cpu())
                        and torch.equal(emb.gc[k].bias.detach().cpu(), victim.gc[k].bias.detach().cpu())):
                    raise NotImplementedError("embedding.gc must share the victim's GC weights (main.py:185-190)")
        return [t.detach().to(self.device, torch.float32).contiguous() for t in (W1, b1, W2, b2, Wl, bl)]

    def _prepare(self, ori_features, ori_adj, labels):
        """Start of attack(): releases the previous call's engine and result first, so that the allocator can recycle
        their blocks instead of growing (x', m, v, F tiles and the n x n result are tens of GB at n = 65 536; cudaMalloc of
        such blocks costs ~0.1 s each), and puts the victim and embedding in eval mode.  Returns the victim's weights
        (W1, b1, W2, b2, Wl, bl), the features X and the labels on the device, (rank, world) and the preset parameter x0
        (None when adj_changes is all zero)."""
        if self.loss_type != 'CE':
            raise NotImplementedError("native path implements loss_type='CE' (the reference driver's choice)")
        dev = torch.device(self.device)
        self.engine = None
        self.modified_adj = None
        self.surrogate.eval()
        if self.embedding is not None:
            self.embedding.eval()
        weights = self._victim_weights()
        X = _dense(ori_features, dev)
        labels_t = torch.as_tensor(np.asarray(labels) if not torch.is_tensor(labels) else labels).long().to(dev)
        if torch.is_tensor(ori_adj):
            assert not bool(ori_adj.any()), "reference driver passes init_adj = 0 (dataset.py:433-437)"
        elif sp.issparse(ori_adj):
            assert ori_adj.nnz == 0, "reference driver passes init_adj = 0"
        else:
            assert not np.any(ori_adj), "reference driver passes init_adj = 0"
        x0 = self.adj_changes.data
        return weights, X, labels_t, _rank_world(), (x0 if bool((x0 != 0).any()) else None)

    def _decode_last(self, eng, gather_x, normalise=True):
        """Decode the last iteration's embedding H2 (em = embedding(X, adj_norm), the hidden state of the normalised
        branch): returns zf (H2, row-normalised unless `normalise` is False) and the tiles of relu(zf zf^T) over this
        rank's tile rows.  adj_changes.data becomes their packed vector (the reference leaves it there) on one GPU, and
        with world > 1 unless `gather_x` is False; there every rank writes its tile rows' entries and the shards are
        summed."""
        st = N.stream_ptr()
        zf = torch.empty_like(eng.H2)
        if normalise:
            call("mcgra_row_normalize", ptr(eng.H2), eng.n, HID, 2.0, ptr(zf), st)
        else:
            zf.copy_(eng.H2)
        xf = tile_buffer(eng.tr0, eng.tr1, eng.dev, zero=False)
        call("mcgra_decode_to_tiles", ptr(zf), eng.n, eng.tr0, eng.tr1, ptr(xf), st)
        if gather_x or eng.world == 1:
            self.adj_changes.data = tiles_to_packed(xf, eng.n, eng.tr0, eng.tr1, None, 1, eng._allreduce)
        return zf, xf

    # ------------------------------------------------------------------------------------------------
    # stand-alone helpers of the reference classes, same names and semantics
    def get_modified_adj(self, ori_adj=None):
        """Symmetric zero-diagonal expansion of adj_changes (+ ori_adj) (topology_attack.py:365-379)."""
        return self._expand(self.adj_changes.data, ori_adj)

    def _on_device(self, x):
        return x.detach().to(torch.device(self.device), torch.float32).contiguous()

    def _expand(self, packed, ori_adj=None):
        n = self.nnodes
        T = (n + N.TILE - 1) // N.TILE
        tiles = packed_to_tiles(self._on_device(packed), n, 0, T)
        out = torch.zeros(n, n, dtype=torch.float32, device=tiles.device)
        call("mcgra_tiles_to_dense", ptr(tiles), n, 0, T, None, 1, ptr(out), n, N.stream_ptr())
        if ori_adj is not None and torch.is_tensor(ori_adj) and bool(ori_adj.any()):
            out = out + ori_adj.to(tiles.device)
        return out

    def dot_product_decode(self, Z):
        """tril(relu(Zn Zn^T)), Zn = F.normalize(Z) (topology_attack.py:414-419) -> packed P-vector."""
        n = Z.shape[0]
        if Z.shape[1] != HID:
            raise NotImplementedError("native decode is built for 16-wide embeddings")
        T = (n + N.TILE - 1) // N.TILE
        st = N.stream_ptr()
        Zc = self._on_device(Z)
        zn = torch.empty_like(Zc)
        call("mcgra_row_normalize", ptr(Zc), n, HID, 2.0, ptr(zn), st)
        tiles = tile_buffer(0, T, Zc.device, zero=False)
        call("mcgra_decode_to_tiles", ptr(zn), n, 0, T, ptr(tiles), st)
        return tiles_to_packed(tiles, n, 0, T, None, 1)

    def projection(self, num_edges):
        """Stand-alone projection of adj_changes (topology_attack.py:338-347) on the device bisection."""
        n = self.nnodes
        T = (n + N.TILE - 1) // N.TILE
        st = N.stream_ptr()
        x = self._on_device(self.adj_changes.data)
        tiles = packed_to_tiles(x, n, 0, T)
        acc = torch.zeros(N.ACC_N, dtype=torch.float64, device=x.device)
        acc[N.ACC["SUMCLAMP"]] = torch.clamp(x, 0, 1).double().sum()
        minmax = torch.stack([x.min(), x.max()]).contiguous()
        state = torch.zeros(8, dtype=torch.float32, device=x.device)
        mu = torch.zeros(1, dtype=torch.float32, device=x.device)
        cand = torch.zeros(8, dtype=torch.float64, device=x.device)
        call("mcgra_bisect_init", ptr(acc), ptr(minmax), float(num_edges), ptr(state), ptr(mu), st)
        bisect(tiles, n, 0, T, float(num_edges), 1e-5, BISECT_PASSES, state, cand, mu)
        self.adj_changes.data.copy_(tiles_to_packed(tiles, n, 0, T, mu, 0))

    def bisection(self, a, b, num_edges, epsilon):
        """Root of sum(clamp(adj_changes - mu, 0, 1)) = num_edges on [a, b] (topology_attack.py:397-412) on the device
        bisection kernels (same fp32 midpoints as the scalar loop, three halvings per pass over the parameter)."""
        n = self.nnodes
        T = (n + N.TILE - 1) // N.TILE
        tiles = packed_to_tiles(self._on_device(self.adj_changes.data), n, 0, T)
        a, b = float(a), float(b)
        state = torch.tensor([a, b, a, 0.0, 1.0, 0.0, 0.0, 0.0], dtype=torch.float32, device=tiles.device)
        mu = torch.full((1,), a, dtype=torch.float32, device=tiles.device)
        cand = torch.zeros(8, dtype=torch.float64, device=tiles.device)
        passes = max(1, int(np.ceil(np.log2(max(b - a, epsilon) / epsilon) / 3.0)) + 1)
        bisect(tiles, n, 0, T, float(num_edges), float(epsilon), passes, state, cand, mu)
        return mu[0]

    def _loss(self, output, labels):
        if self.loss_type == "CE":
            return F.nll_loss(output, labels)
        if self.loss_type == "CW":       # topology_attack.py:329-335 (stand-alone helper; the loop uses CE)
            onehot = torch.eye(int(labels.max()) + 1, device=output.device)[labels]
            best_second_class = (output - 1000 * onehot).argmax(1)
            ar = torch.arange(len(output), device=output.device)
            margin = output[ar, labels] - output[ar, best_second_class]
            return -torch.clamp(margin, min=0).mean()
        raise ValueError(self.loss_type)

    # ------------------------------------------------------------------------------------------------
    def gather_modified_adj(self):
        """Full n x n result on every rank from the row bands (world > 1); identity otherwise."""
        eng = self.engine
        if eng is None or eng.world == 1:
            return self.modified_adj
        import torch.distributed as dist
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
