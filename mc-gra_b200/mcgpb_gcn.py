"""B200-native defended GCN training of the defence repo -- same surface as the reference's MC-GPB/models/gcn.py `GCN`
(BASELINE.json configs[2], SURVEY 8(f) rank 1).

`GCN(...).fit(features, adj, labels, idx_train, idx_val, idx_test, beta=..., MI_type='linear_HSIC' | 'linear_CKA' | 'DP')`
runs `_train_with_MI_constrain` (MC-GPB/models/gcn.py:321-513): per epoch a forward returning the three layer embeddings,
the inter-layer penalties IAZ(next next^T, emb) and the node-pair penalties IAZ(right right^T, left) on 1000 sampled
edges (:382-417), the auxiliary nll terms, six n x n link-AUROCs (:348-357, 419, 433-434), Adam.

What runs natively (C ABI, include/mcgra.h):
  * the n x n products A_hat . (X W) of GraphConvolution (forward AND backward: A_hat is symmetric) on the tiled tcgen05
    propagation kernel (`mcgra_propagate` over the tiles of the fixed normalised adjacency);
  * every penalty: the reference forms the n x n (or 1000 x 1000) gram and calls CudaCKA.linear_HSIC / linear_CKA or DP on it
    (MC-GPB/utils.py:774-797, six n^3 GEMMs each); here all of them are functions of WEIGHTED SECOND MOMENTS of the n x d
    factors -- `mcgra_cross_moments` forward, `mcgra_cross_moments_bwd` backward, O(n d d'), no n x n object:
        linear_HSIC(N N^T, Z) = ||N N^T H Z||_F^2 = sum (Gs B) o B,     B = N^T H Z,  Gs = N^T N
        hsic(N N^T, N N^T)    = tr((C Gs)^2),  C = N^T H N;      hsic(Z, Z) = ||Z^T H Z||_F^2
        DP(N N^T, Z)          = ||Z Z^T N N^T||_F = sqrt(tr(Gs (N^T Z) (Z^T Z) (Z^T N)))
    (the d x d algebra on the moment matrices is a handful of torch ops on 16 x 16 tensors);
  * the link AUROCs: `mcgra_gram_accumulate` (relu(Z Z^T - I)) + `mcgra_auc_ap` (exact sklearn semantics, on device).
A sparse adjacency takes the CSR path instead, which holds no n x n object: `mcgra_spmm_csr` propagates, and
`mcgra_gram_auc_stage` ranks the gram scores against the CSR labels as it generates them (bit-equal AUCs).
PyTorch keeps the parameter tensors, autograd's tape between the native ops, the small dense X W products and Adam.
There is no CPU path: the model must live on a CUDA device.
"""
import math
from copy import deepcopy

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
import torch.optim as optim
from torch.nn.modules.module import Module
from torch.nn.parameter import Parameter

from . import _native as N
from . import utils
from ._native import call, ptr
from .engine import TILE, tile_buffer


# ----------------------------------------------------------------------------------------------------------------
# native autograd ops
# ----------------------------------------------------------------------------------------------------------------
class TiledAdjacency:
    """Fixed symmetric adjacency with entries in [0, 1] (the normalised A_hat) as tiles of its strict lower triangle plus
    its diagonal: the operand layout of mcgra_propagate."""

    def __init__(self, A):
        if not A.is_cuda:
            raise N.NativeError("mcgpb_gcn needs a CUDA device (no CPU fallback)")
        A = (A.to_dense() if A.is_sparse else A).to(torch.float32).contiguous()
        n = A.shape[0]
        self.n, self.T = n, (n + TILE - 1) // TILE
        self.tiles = tile_buffer(0, self.T, A.device)
        self.diag = torch.zeros(n, dtype=torch.float32, device=A.device)
        call("mcgra_dense_to_tiles", ptr(A), n, n, 0, self.T, 1, ptr(self.tiles), ptr(self.diag), N.stream_ptr())
        self.ws = torch.empty(int(N.lib().mcgra_propagate_ws_bytes(n, 32)), dtype=torch.uint8, device=A.device)

    def matmul(self, B):
        B = B.contiguous()
        K = B.shape[1]
        if K not in (16, 32):
            raise NotImplementedError("native propagation handles 16- or 32-wide operands (nhid = 16 in the reference)")
        Y = torch.zeros_like(B)
        call("mcgra_propagate", ptr(self.tiles), self.n, 0, self.T, None, 2, ptr(B), K, ptr(Y), ptr(self.ws),
             N.stream_ptr())
        return Y + self.diag[:, None] * B


class SparseAdjacency:
    """Fixed symmetric adjacency in CSR form (int64 row pointers, int32 sorted columns, fp32 values, the self-loop an
    ordinary entry): the operand of mcgra_spmm_csr, with the matmul interface of TiledAdjacency.  Holds O(n + |E|)."""

    def __init__(self, rowptr, cols, vals):
        if not vals.is_cuda:
            raise N.NativeError("mcgpb_gcn needs a CUDA device (no CPU fallback)")
        self.rowptr, self.cols, self.vals = rowptr.contiguous(), cols.contiguous(), vals.contiguous()
        self.n = rowptr.numel() - 1

    def matmul(self, B):
        B = B.contiguous()
        K = B.shape[1]
        if K not in (16, 32):
            raise NotImplementedError("native propagation handles 16- or 32-wide operands (nhid = 16 in the reference)")
        Y = torch.empty_like(B)
        call("mcgra_spmm_csr", ptr(self.rowptr), ptr(self.cols), ptr(self.vals), self.n, ptr(B), K, ptr(Y),
             N.stream_ptr())
        return Y


class Csr:
    """CSR of a sparse n x n matrix without explicit zeros: rowptr (int64, n + 1), rows / cols of the entries in row-major
    order (int64 / int32), vals (float32)."""

    def __init__(self, a):
        n = a.shape[0]
        if a.layout != torch.sparse_coo:
            a = a.to_sparse_coo()
        a = a.coalesce()                     # row-major, columns sorted within a row
        keep = a.values() != 0
        self.rows, cols = a.indices()[0][keep], a.indices()[1][keep]
        self.cols, self.vals = cols.to(torch.int32).contiguous(), a.values()[keep].to(torch.float32).contiguous()
        self.rowptr = torch.zeros(n + 1, dtype=torch.int64, device=a.device)
        self.rowptr[1:] = torch.cumsum(torch.bincount(self.rows, minlength=n), 0)
        self.n = n

    def coo(self):
        return torch.sparse_coo_tensor(torch.stack([self.rows, self.cols.long()]), self.vals, (self.n, self.n))


def normalize_csr(a):
    """utils.normalize_adj_tensor on a Csr: D^-1/2 (A + I) D^-1/2 with the same value order (r_i * m_ij) * r_j, where
    r = rowsum(A + I)^-1/2 (0 where the row sum is 0)."""
    n, dev = a.n, a.vals.device
    ar = torch.arange(n, device=dev)
    mx = Csr(torch.sparse_coo_tensor(torch.stack([torch.cat([a.rows, ar]), torch.cat([a.cols.long(), ar])]),
                                     torch.cat([a.vals, torch.ones(n, device=dev)]), (n, n)))
    r_inv = torch.segment_reduce(mx.vals, "sum", offsets=mx.rowptr).pow(-1 / 2)
    r_inv = torch.where(torch.isinf(r_inv), torch.zeros_like(r_inv), r_inv)
    return SparseAdjacency(mx.rowptr, mx.cols, (r_inv[mx.rows] * mx.vals) * r_inv[mx.cols.long()])


class _Propagate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, B, adj):
        ctx.adj = adj
        return adj.matmul(B.detach().to(torch.float32))

    @staticmethod
    def backward(ctx, g):
        return ctx.adj.matmul(g.contiguous()), None          # A_hat is symmetric


class _CrossMoments(torch.autograd.Function):
    """[sum x | sum y | sum x y^T | sum y y^T] in fp64 (mcgra_cross_moments), differentiable w.r.t. both factors."""

    @staticmethod
    def forward(ctx, X, Y):
        Xc, Yc = X.detach().to(torch.float32).contiguous(), Y.detach().to(torch.float32).contiguous()
        n, dx, dy = Xc.shape[0], Xc.shape[1], Yc.shape[1]
        out = torch.zeros(dx + dy + dx * dy + dy * dy, dtype=torch.float64, device=Xc.device)
        call("mcgra_cross_moments", ptr(Xc), dx, ptr(Yc), dy, None, n, ptr(out), N.stream_ptr())
        ctx.save_for_backward(Xc, Yc)
        return out

    @staticmethod
    def backward(ctx, g):
        Xc, Yc = ctx.saved_tensors
        n, dx, dy = Xc.shape[0], Xc.shape[1], Yc.shape[1]
        g = g.to(torch.float64).contiguous()
        dX, dY = torch.empty_like(Xc), torch.empty_like(Yc)
        call("mcgra_cross_moments_bwd", ptr(Xc), dx, ptr(Yc), dy, None, n, ptr(g), ptr(dX), ptr(dY), N.stream_ptr())
        return dX, dY


def _moments(Nf, Z):
    """S1 = sum n_i, S2 = sum z_i, Sxy = N^T Z, Syy = Z^T Z, Gs = N^T N (fp64, differentiable)."""
    dn, dz = Nf.shape[1], Z.shape[1]
    o = _CrossMoments.apply(Nf, Z)
    S1, S2 = o[:dn], o[dn:dn + dz]
    Sxy = o[dn + dz:dn + dz + dn * dz].view(dn, dz)
    Syy = o[dn + dz + dn * dz:].view(dz, dz)
    o2 = _CrossMoments.apply(Nf, Nf)
    Gs = o2[2 * dn + dn * dn:].view(dn, dn)
    return S1, S2, Sxy, Syy, Gs


def linear_HSIC(Nf, Z):
    """utils.linear_HSIC(Nf Nf^T, Z) (MC-GPB/utils.py:783-785) from the factors."""
    m = Nf.shape[0]
    S1, S2, Sxy, _, Gs = _moments(Nf, Z)
    B = Sxy - torch.outer(S1, S2) / m
    return ((Gs @ B) * B).sum().float()


def linear_CKA(Nf, Z):
    """utils.linear_CKA(Nf Nf^T, Z) (MC-GPB/utils.py:778-780)."""
    m = Nf.shape[0]
    S1, S2, Sxy, Syy, Gs = _moments(Nf, Z)
    B = Sxy - torch.outer(S1, S2) / m
    hxy = ((Gs @ B) * B).sum()
    Cn = Gs - torch.outer(S1, S1) / m
    hxx = ((Cn @ Gs) * (Cn @ Gs).t()).sum()                      # tr((C Gs)^2)
    Cz = Syy - torch.outer(S2, S2) / m
    hyy = (Cz * Cz).sum()
    return (hxy / (torch.sqrt(hxx) * torch.sqrt(hyy))).float()


def DP(Nf, Z):
    """utils.DP(Nf Nf^T, Z) = ||Z Z^T Nf Nf^T||_F (MC-GPB/utils.py:788-792)."""
    _, _, Sxy, Syy, Gs = _moments(Nf, Z)
    return torch.sqrt(torch.trace(Gs @ Sxy @ Syy @ Sxy.t())).float()


MI_FUNCS = {"linear_HSIC": linear_HSIC, "linear_CKA": linear_CKA, "DP": DP}


def link_auc(Z, adj_labels):
    """calculate_AUC (MC-GPB/models/gcn.py:348-357): AUROC of relu(Z Z^T - I) against the true adjacency over all n^2
    ordered pairs, on the device.  `adj_labels`: the n x n uint8 label matrix, or the Csr of the true adjacency (then
    mcgra_gram_auc_stage forms neither scores nor labels; the same AUC bit for bit)."""
    from .metrics import roc_auc_ap
    Zc = Z.detach().to(torch.float32).contiguous()
    n, d = Zc.shape
    if d > 32:
        raise NotImplementedError("embedding width > 32")
    if isinstance(adj_labels, Csr):
        npos = max(int(adj_labels.cols.numel()), 1)
        ws = torch.empty(N.lib().mcgra_gram_auc_workspace_bytes(npos), dtype=torch.uint8, device=Zc.device)
        out = torch.zeros(4, dtype=torch.float64, device=Zc.device)
        for stage in range(3):
            call("mcgra_gram_auc_stage", stage, ptr(Zc), d, n, ptr(adj_labels.rowptr), ptr(adj_labels.cols), 0, n, npos,
                 ptr(ws), ptr(out), N.stream_ptr())
        o = out.cpu().numpy()
        if int(o[2]) > npos:
            raise N.NativeError(f"positives {int(o[2])} exceed npos_max {npos}")
        return float(o[0])
    S = torch.zeros(n, n, dtype=torch.float32, device=Zc.device)
    call("mcgra_gram_accumulate", ptr(Zc), d, n, 1, None, ptr(S), n, 0, n, N.stream_ptr())
    return roc_auc_ap(S, adj_labels)[0]


# ----------------------------------------------------------------------------------------------------------------
# model (MC-GPB/models/gcn.py:16-176)
# ----------------------------------------------------------------------------------------------------------------
class GraphConvolution(Module):
    def __init__(self, in_features, out_features, with_bias=True):
        super(GraphConvolution, self).__init__()
        self.in_features, self.out_features = in_features, out_features
        self.weight = Parameter(torch.FloatTensor(in_features, out_features))
        self.bias = Parameter(torch.FloatTensor(out_features)) if with_bias else None
        if not with_bias:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        stdv = 1. / math.sqrt(self.weight.T.size(1))          # models/gcn.py:30-35 (uniform in +-1/sqrt(in_features))
        self.weight.data.uniform_(-stdv, stdv)
        if self.bias is not None:
            self.bias.data.uniform_(-stdv, stdv)

    def forward(self, input, adj):
        support = torch.mm(input, self.weight)
        if isinstance(adj, (TiledAdjacency, SparseAdjacency)):
            output = _Propagate.apply(support, adj)
        else:
            output = torch.spmm(adj, support)
        return output + self.bias if self.bias is not None else output


class embedding_GCN(nn.Module):
    def __init__(self, nfeat, nhid, nlayer=1, with_bias=True, device=None):
        super(embedding_GCN, self).__init__()
        assert device is not None, "Please specify 'device'!"
        self.device, self.nfeat, self.nlayer, self.hidden_sizes = device, nfeat, nlayer, [nhid]
        self.gc = [GraphConvolution(nfeat, nhid, with_bias=with_bias)]
        for _ in range(nlayer - 1):
            self.gc.append(GraphConvolution(nhid, nhid, with_bias=with_bias))
        self.gc1 = self.gc[0]
        self.with_bias = with_bias

    def forward(self, x, adj):
        for i in range(self.nlayer):
            x = F.relu(self.gc[i].to(self.device)(x, adj))
        return x

    def set_layers(self, nlayer):
        self.nlayer = nlayer


class GCN(nn.Module):
    def __init__(self, nfeat, nhid, nclass, nlayer=2, dropout=0.5, lr=0.01, weight_decay=5e-4, with_relu=True,
                 with_bias=True, device=None):
        super(GCN, self).__init__()
        assert device is not None, "Please specify 'device'!"
        self.device, self.nfeat, self.hidden_sizes, self.nclass, self.nlayer = device, nfeat, [nhid], nclass, nlayer
        self.gc = [GraphConvolution(nfeat, nhid, with_bias=with_bias)]
        for _ in range(nlayer - 1):
            self.gc.append(GraphConvolution(nhid, nhid, with_bias=with_bias))
        self.gc1 = self.gc[0]
        self.gc2 = self.gc[1]
        self.linear1 = nn.Linear(nhid, nclass, bias=with_bias)
        self.dropout, self.lr = dropout, lr
        self.weight_decay = weight_decay if with_relu else 0
        self.with_relu, self.with_bias = with_relu, with_bias
        self.output = self.best_model = self.best_output = self.adj_norm = self.features = self.origin_adj = None
        self.origin_csr = None
        self.initialize()

    def forward(self, x, adj):
        node_emb = []
        for i, layer in enumerate(self.gc):
            layer = layer.to(self.device)
            x = F.relu(layer(x, adj)) if self.with_relu else layer(x, adj)
            if i != len(self.gc) - 1:
                x = F.dropout(x, self.dropout, training=self.training)
            node_emb.append(x)
        x = self.linear1(x)
        node_emb.append(x)
        return F.log_softmax(x, dim=1), node_emb

    def initialize(self):
        for layer in self.gc:
            layer.reset_parameters()

    def fit(self, features, adj, labels, idx_train, idx_val=None, idx_test=None, train_iters=200, initialize=True,
            verbose=False, normalize=True, patience=500, beta=None, MI_type='linear_HSIC', stochastic=0, con=0, aug_pe=0.1,
            plain_acc=0.7, pair_draws=None, **kwargs):
        """models/gcn.py:184-277.  `pair_draws` (test hook): the node-pair index draws of every epoch instead of
        np.random.choice, so that a run can be replayed against a reference fixture.

        A sparse `adj` (torch sparse tensor or scipy matrix) is never densified: the normalised adjacency, the labels of
        the link AUROCs and the node pairs are held in CSR form (O(n + |E|) device memory), with the same node-pair and
        edge-drop draws as a dense `adj`.  A dense `adj` takes the tiled dense path."""
        self.device = self.gc1.weight.device
        if self.device.type != "cuda":
            raise N.NativeError("mcgpb_gcn needs a CUDA device (no CPU fallback)")
        if type(adj) is not torch.Tensor:
            features, adj, labels = utils.to_tensor(features, adj, labels, device=self.device)
        else:
            features, adj, labels = features.to(self.device), adj.to(self.device), labels.to(self.device)
        if adj.layout != torch.strided:
            self._set_sparse_adj(adj, stochastic, aug_pe, normalize)
        else:
            self._set_dense_adj(adj, stochastic, aug_pe, normalize)
        self.features, self.labels = features, labels
        if con:
            raise NotImplementedError("contrastive training (con=1) is not on the MC-GPB README path")
        if beta is None:
            return self._train_with_val(labels, idx_train, idx_val, train_iters, verbose)
        return self._train_with_MI_constrain(labels, idx_train, idx_val, idx_test, train_iters, beta, MI_type, plain_acc,
                                             verbose, pair_draws)

    def _set_sparse_adj(self, adj, stochastic, aug_pe, normalize):
        a = Csr(adj)
        if stochastic:        # the dense path's edge drop: one draw per upper-triangle entry, in row-major order
            up = a.cols.long() > a.rows
            keep = torch.rand(int(up.sum()), device=self.device) >= aug_pe
            i, j = a.rows[up][keep], a.cols.long()[up][keep]
            a = Csr(torch.sparse_coo_tensor(torch.stack([torch.cat([i, j]), torch.cat([j, i])]),
                                            torch.ones(2 * i.numel(), device=self.device), (a.n, a.n)))
        self.adj_norm = normalize_csr(a) if normalize else SparseAdjacency(a.rowptr, a.cols, a.vals)
        self.origin_adj, self.origin_csr = a.coo(), a

    def _set_dense_adj(self, adj, stochastic, aug_pe, normalize):
        if stochastic:        # utils.stochastic (PyGCL EdgeRemoving, MC-GPB/utils.py:799-805): drop each undirected edge with prob. pe
            iu = torch.triu(adj, 1).nonzero()
            keep = torch.rand(iu.shape[0], device=self.device) >= aug_pe
            new = torch.zeros_like(adj)
            new[iu[keep, 0], iu[keep, 1]] = 1.0
            adj = new + new.t()
        adj_norm = utils.normalize_adj_tensor(adj) if normalize else adj
        self.adj_norm = TiledAdjacency(adj_norm)
        self.origin_adj, self.origin_csr = adj, None

    def _train_with_val(self, labels, idx_train, idx_val, train_iters, verbose):
        """models/gcn.py:279-319."""
        optimizer = optim.Adam(self.parameters(), lr=self.lr, weight_decay=self.weight_decay)
        best_loss_val, best_acc_val = 100, 0
        weights = deepcopy(self.state_dict())
        for _ in range(train_iters):
            self.train()
            optimizer.zero_grad()
            output = self.forward(self.features, self.adj_norm)[0]
            F.nll_loss(output[idx_train], labels[idx_train]).backward()
            optimizer.step()
            self.eval()
            with torch.no_grad():
                output = self.forward(self.features, self.adj_norm)[0]
                loss_val = F.nll_loss(output[idx_val], labels[idx_val])
                acc_val = utils.accuracy(output[idx_val], labels[idx_val])
            if best_loss_val > loss_val:
                best_loss_val, self.output, weights = loss_val, output, deepcopy(self.state_dict())
            if acc_val > best_acc_val:
                best_acc_val, self.output, weights = acc_val, output, deepcopy(self.state_dict())
        self.load_state_dict(weights)

    def _train_with_MI_constrain(self, labels, idx_train, idx_val, idx_test, train_iters, beta, MI_type, plain_acc, verbose,
                                 pair_draws=None):
        """models/gcn.py:321-513."""
        if MI_type not in MI_FUNCS:
            raise NotImplementedError(f"MI_type {MI_type!r}: the native path implements linear_HSIC, linear_CKA and DP")
        IAZ_func = MI_FUNCS[MI_type]
        optimizer = optim.Adam(self.parameters(), lr=self.lr, weight_decay=self.weight_decay)
        best_loss_val, best_acc_val = 100, 0
        IAZ = torch.zeros((train_iters, self.nlayer + 1))
        IYZ = torch.zeros((train_iters, self.nlayer + 1))
        full_losses = [[] for _ in range(4)]
        if self.origin_csr is not None:          # row-major, as origin_adj.nonzero() lists them
            edge_index = torch.stack([self.origin_csr.rows, self.origin_csr.cols.long()], 1)
            adj_labels = self.origin_csr
        else:
            edge_index = self.origin_adj.nonzero()
            adj_labels = (self.origin_adj != 0).to(torch.uint8).contiguous()
        sample_size = min(1000, edge_index.size(0))
        best_layer_AUC, weights, final_layer_aucs, best_acc_test = 1e10, None, 1000, 0
        weights2 = final_layer_aucs_2 = None
        for epoch in range(train_iters):
            self.train()
            optimizer.zero_grad()
            output, node_embs = self.forward(self.features, self.adj_norm)
            draw = pair_draws[epoch] if pair_draws is not None else np.random.choice(edge_index.size(0), size=sample_size,
                                                                                      replace=True)
            draw = torch.as_tensor(np.asarray(draw), device=self.device).long()
            node_idx_1, node_idx_2 = edge_index[draw][:, 0], edge_index[draw][:, 1]
            loss_IAZ = loss_inter = loss_mission = 0
            layer_aucs = []
            for idx, node_emb in enumerate(node_embs):
                if (idx + 1) <= len(node_embs) - 1:                                        # complexity constraint (:398-406)
                    loss_inter = loss_inter + beta['layer_inter-{}'.format(idx)] * IAZ_func(node_embs[idx + 1], node_emb)
                loss_IAZ = loss_IAZ + beta['layer-{}'.format(idx)] * IAZ_func(node_emb[node_idx_2], node_emb[node_idx_1])
                layer_aucs.append(link_auc(node_emb, adj_labels))                          # :419
                if idx != len(node_embs) - 1:                                              # accuracy constraint (:422-427)
                    loss_mission = loss_mission + F.nll_loss(F.log_softmax(self.linear1(node_emb), dim=1)[idx_train],
                                                             labels[idx_train])
            with torch.no_grad():                                                          # GIP bookkeeping (:430-441)
                for l_idx, l_out in enumerate(node_embs):
                    IAZ[epoch, l_idx] = layer_aucs[l_idx]
                    lo = self.linear1(l_out) if l_idx < len(node_embs) - 1 else l_out
                    IYZ[epoch, l_idx] = utils.accuracy(F.log_softmax(lo, dim=1)[idx_test], labels[idx_test]).item()
            output = F.log_softmax(output, dim=1)
            loss_IYZ = F.nll_loss(output[idx_train], labels[idx_train])
            for li, lv in enumerate((loss_IYZ, loss_IAZ, loss_inter, loss_mission)):
                full_losses[li].append(float(lv))
            loss_train = loss_IYZ + loss_IAZ + loss_inter
            if plain_acc != 0.6303:                                                        # :452-453
                loss_train = loss_train + loss_mission
            loss_train.backward()
            optimizer.step()
            self.eval()
            with torch.no_grad():
                output = F.log_softmax(self.forward(self.features, self.adj_norm)[0], dim=1)
                loss_val = F.nll_loss(output[idx_val], labels[idx_val])
                acc_val = utils.accuracy(output[idx_val], labels[idx_val])
                acc_test = utils.accuracy(output[idx_test], labels[idx_test])
            weights2 = final_layer_aucs_2 = None
            if best_loss_val > loss_val:
                best_loss_val, self.output = loss_val, output
                weights2, final_layer_aucs_2 = deepcopy(self.state_dict()), layer_aucs
            if acc_val > best_acc_val:
                best_acc_val, self.output = acc_val, output
                weights2, final_layer_aucs_2 = deepcopy(self.state_dict()), layer_aucs
            if (sum(layer_aucs) < best_layer_AUC) and ((plain_acc - acc_test) < 0.05) and (acc_test > best_acc_test):
                best_acc_test, best_layer_AUC, self.output = acc_test, sum(layer_aucs), output
                weights, final_layer_aucs = deepcopy(self.state_dict()), layer_aucs
        if weights:
            self.load_state_dict(weights)
        elif weights2:
            self.load_state_dict(weights2)
        if final_layer_aucs == 1000:
            final_layer_aucs = final_layer_aucs_2
        return {'IAZ': IAZ, 'IYZ': IYZ, 'full_losses': full_losses, 'final_layer_aucs': final_layer_aucs}
