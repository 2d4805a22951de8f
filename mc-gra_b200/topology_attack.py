"""B200-native `topology_attack` -- same surface as the reference's MC-GRA/topology_attack.py.

`PGDAttack(model, embedding, H_A, Y_A, nnodes, loss_type, device)` and `.attack(args, ...)` keep the reference's
signatures (topology_attack.py:57-58, 95-98) and side effects (`self.modified_adj`, `self.adj_changes.data`);
the loop body runs as hand-written sm_100a kernels sequenced by `engine.PGDEngine` through the C ABI of
include/mcgra.h.  No CPU fallback: constructing the engine without a CUDA device raises.

Deliberately hoisted / dropped (results unchanged, SURVEY.md Appendix C):
  * iteration-invariant constants H_A, Y_A (true adjacency) and X W1 are computed once, not per iteration
    (reference recomputes them at :177-182, 241-243);
  * dead per-iteration work (:168-170, 285-296: unused decodes, the n x n `.cpu().mean()`, the accuracy of a
    second forward) is not executed; the per-iteration `.item()` syncs become one read of a device-side history.
"""
import os

import numpy as np
import torch
from torch.nn import functional as F

from . import _native as N
from ._native import call, ptr
from .base_attack import RowBandResult, _dense, _rank_world
from .dense_measure import DenseMeasure
from .engine import HID, HostBands, PGDEngine, check_noise_supported, output_band

Align_Parameter_Cora = {"c1": 100, "c2": 1000, "c3": 100, "c4": 10, "c5": 10, "c6": 10, "c7": 10, "c8": 0.01,
                        "c9": 1, "c10": 1}


def Info_entropy(prob):
    """Reference helper kept for API parity (topology_attack.py:44-47); torch ops, not on the hot path."""
    prob = torch.clamp(prob, 1e-4, 1 - 1e-4)
    return -torch.mean(prob * torch.log2(prob))


def _ident(t):
    """Cheap identity of an input for the cross-call constant cache: storage address + in-place version for tensors,
    object id otherwise."""
    if torch.is_tensor(t):
        return (t.data_ptr() if not t.is_sparse else id(t), t._version, tuple(t.shape), str(t.device))
    return (id(t), getattr(t, "shape", None))


class PGDAttack(RowBandResult):

    def __init__(self, model=None, embedding=None, H_A=None, Y_A=None, nnodes=None, loss_type='CE', feature_shape=None,
                 attack_structure=True, attack_features=False, device='cpu'):
        super().__init__(model, embedding, nnodes, loss_type, feature_shape, attack_structure, attack_features, device)
        self.complementary_after = None
        self.H_A = H_A
        self.Y_A = Y_A
        self._adj_changes_after = None
        self._const_cache = {}

    # the reference allocates a second P-vector eagerly on the host (:73-74); it is materialised on demand here
    @property
    def adj_changes_after(self):
        if self._adj_changes_after is None:
            self._adj_changes_after = torch.zeros(int(self.nnodes * (self.nnodes - 1) / 2))
        return self._adj_changes_after

    @adj_changes_after.setter
    def adj_changes_after(self, v):
        self._adj_changes_after = v

    # ------------------------------------------------------------------------------------------------
    @staticmethod
    def _mm_adj(adj, S):
        return torch.sparse.mm(adj, S) if adj.is_sparse else adj @ S

    def attack(self, args, index_delete, lr_ori, weight_aux, weight_supervised, weight_param, feature_adj,
               aux_adj, aux_feature, aux_num_edges, idx_train, idx_val, idx_test, adj,
               ori_features, ori_adj, labels, idx_attack, num_edges,
               dropout_rate, epochs=200, sample=False, **kwargs):
        """Same parameters and side effects as the reference (topology_attack.py:95-324).  Returns (0,0,0,0)."""
        if args.max_eval == 1:
            lr_ori = 10 ** args.lr
        self.args = args
        eps = float(getattr(args, "eps", 0) or 0)
        if eps != 0.0:        # scope of the noisy path, checked before any device work
            check_noise_supported(args.measure, _rank_world()[1], feature_adj, self.device)
        dev = torch.device(self.device)
        n = self.nnodes
        timing = {} if kwargs.get("_timing") else None      # bench hook: phase wall-clock (adds synchronisations)
        import time as _time

        def _mark(name, _t=[None]):
            if timing is None:
                return
            torch.cuda.synchronize(dev)
            now = _time.perf_counter()
            if _t[0] is not None:
                timing[name] = timing.get(name, 0.0) + now - _t[0]
            _t[0] = now
        _mark("start")
        (W1, b1, W2, b2, Wl, bl), X, labels_t, (rank, world), x0 = self._prepare(ori_features, ori_adj, labels)
        adj_d = adj.to(dev) if torch.is_tensor(adj) else _dense(adj, dev)
        if not adj_d.is_sparse:
            adj_d = adj_d.to(torch.float32)

        w1, w2, _, _, _, w6, w7, w8, w9, w10 = weight_param
        if args.max_eval == 1:          # (:152-159, including the reference's `w7 = args.w8` overwrite)
            w1, w2, w6, w7, w9, w10 = args.w1, args.w2, args.w6, args.w8, args.w9, args.w10
        weights = (w1, w2, 0, 0, 0, w6, w7, w8, w9, w10)

        # iteration-invariant constants (hoisted from :177-182): targets on the TRUE, un-normalised adjacency.  They are
        # also invariant ACROSS attack() calls on the same inputs (main.py's search mode calls objective() repeatedly):
        # cached on the object, keyed by the identity + version of the tensors they are built from.
        ckey = tuple(_ident(t) for t in (ori_features, adj, W1, b1, W2, b2, Wl, bl))
        if self._const_cache.get("key") == ckey:
            S1, HA_loop, YA_loop = self._const_cache["val"]
        else:
            with torch.no_grad():
                S1 = X @ W1
                E1 = torch.relu(self._mm_adj(adj_d, S1) + b1)
                HA_loop = torch.relu(self._mm_adj(adj_d, E1 @ W2) + b2)
                YA_loop = F.log_softmax(HA_loop @ Wl.t() + bl, dim=1)
            self._const_cache = {"key": ckey, "val": (S1, HA_loop, YA_loop)}
        _mark("inputs_and_constants")
        if isinstance(feature_adj, HostBands):     # multi-GPU: every rank copies only the row bands it touches
            fa = feature_adj
        else:
            fa = feature_adj.to(dev) if torch.is_tensor(feature_adj) else _dense(feature_adj, dev)
        _mark("feature_adj_h2d")

        self.engine = PGDEngine(n, S1, W2, b1, b2, Wl, bl, labels_t, idx_attack, HA_loop, YA_loop, fa,
                                args.measure, weights, lr_ori, weight_sup=weight_supervised, num_edges=num_edges,
                                x0=x0, device=dev, rank=rank, world=world,
                                max_epochs=max(int(epochs), int(kwargs.get('_engine_epochs', 1)), 1),
                                eps=eps, noise=kwargs.get("_noise"))
        eng = self.engine
        fa_on_host = not isinstance(feature_adj, HostBands) and not (torch.is_tensor(feature_adj) and feature_adj.is_cuda)
        if isinstance(eng.nn, DenseMeasure) and fa_on_host:
            fa = None          # the contraction stage keeps its own constant image; the dense copy returns for the ensemble
        _mark("engine_setup")
        self._trace = []
        self._timing = timing
        # test hook `_trace`: parameter after every iteration's projection; `_graph`: True / False force or forbid CUDA-graph replay (default: auto)
        # `_noise`: callable(t) -> n x n draw of iteration t for --eps != 0 (default: torch.randn on the attack's device)
        on_iter = (lambda: self._trace.append(eng.packed_parameter())) if kwargs.get("_trace") else None
        eng.run(int(epochs), on_iter=on_iter, use_graph=kwargs.get("_graph", "auto"))
        eng.check_noise_agreement()        # world > 1 with noise: raises if the ranks drew differently
        if kwargs.get("_skip_finalize"):         # bench hook: engine is driven by the caller
            return 0, 0, 0, 0
        if int(epochs) == 0:
            eng.forward_stages(0)
        _mark("iterations")
        if isinstance(eng.nn, DenseMeasure):     # n x n operand images / gradient buffers are not needed past the loop
            eng.nn = None
        if fa is None:
            fa = feature_adj.to(dev) if torch.is_tensor(feature_adj) else _dense(feature_adj, dev)
        self._finalize(eng, args, fa, labels_t, W2, b1, b2, Wl, bl, gather_x=kwargs.get("_gather_x", True))
        _mark("finalize")
        return 0, 0, 0, 0

    # ------------------------------------------------------------------------------------------------
    def _decode2_spec(self, Z):
        """dot_product_decode2's dataset / flag table (topology_attack.py:421-467) ->
        (Z', variant, rownorm) for mcgra_gram_accumulate."""
        a = self.args
        ds = a.dataset
        st = N.stream_ptr()
        Z = Z.contiguous()
        n, d = Z.shape

        def normed(p):
            out = torch.empty_like(Z)
            call("mcgra_row_normalize", ptr(Z), n, d, float(p), ptr(out), st)
            return out

        if ds in ('cora', 'AIDS'):
            return Z, 0, None
        if ds == 'citeseer':
            return normed(2), 0, None
        if ds == 'brazil':
            return Z, 1, None
        if ds in ('polblogs', 'usair'):
            if ds == 'polblogs' and a.useH_A and a.useY_A and a.useY:
                pass
            elif ds == 'usair' and a.useY and not a.useH_A and not a.useY_A:
                return normed(3), 1, None
            elif ds == 'usair' and not a.useY and a.useH_A and a.useY_A:
                return normed(2), 1, None
            elif ds == 'usair' and a.useY and a.useH_A and not a.useY_A:
                return normed(5), 1, None
            # row-normalised gram: ||row i of Z Z^T||_2 = sqrt(z_i^T (Z^T Z) z_i)
            Cm = Z.t() @ Z
            rown = ((Z @ Cm) * Z).sum(1).clamp_min(0).sqrt().contiguous()
            return Z, 2, rown
        raise UnboundLocalError(f"dataset {ds!r} has no dot_product_decode2 branch (topology_attack.py:421-467)")

    def _gram_add(self, out, Z):
        Zp, variant, rown = self._decode2_spec(Z.to(torch.float32))
        n, d = Zp.shape
        call("mcgra_gram_accumulate", ptr(Zp), d, n, variant, ptr(rown), ptr(out), n, 0, n, N.stream_ptr())

    def _finalize(self, eng, args, fa, labels_t, W2, b1, b2, Wl, bl, gather_x=True):
        """topology_attack.py:300-322.  The decoded parameter stays sharded by tile rows like the loop's (its two
        propagations are all-reduced), and every rank evaluates the ensemble for ITS ROW BAND of the n x n result only
        (`self.modified_adj` = rows [b0, b1), `self.modified_adj_rows`); with world > 1 `gather_modified_adj()` assembles
        the full matrix and `metrics.auc_ap_from_edges_sharded` scores the bands in place.  One GPU owns all rows."""
        import ctypes as _C
        st = N.stream_ptr()
        n, dev, world = eng.n, eng.dev, eng.world
        zf, xf = self._decode_last(eng, gather_x)        # adj_changes.data (:301)
        # embeddings / victim output on the raw decoded adjacency (:304-308): two propagations over xf
        Y = torch.zeros(n, HID, dtype=torch.float32, device=dev)
        call("mcgra_propagate", ptr(xf), n, eng.tr0, eng.tr1, None, 1, ptr(eng.S1), HID, ptr(Y), ptr(eng.prop_ws), st)
        eng._allreduce(Y)
        H1 = torch.relu(Y + b1)
        T2 = (H1 @ W2).contiguous()
        Y2 = torch.zeros(n, HID, dtype=torch.float32, device=dev)
        call("mcgra_propagate", ptr(xf), n, eng.tr0, eng.tr1, None, 1, ptr(T2), HID, ptr(Y2), ptr(eng.prop_ws), st)
        eng._allreduce(Y2)
        H2 = torch.relu(Y2 + b2)
        YA2 = F.log_softmax(H2 @ Wl.t() + bl, dim=1)
        # cur_adj = modified_adj (:302) + H_A1 + H_A2 + feature_adj + Y_A2 (+ ori_HA) (+ ori_YA) (+ label_adj), summed in
        # this order in ONE pass over the result band (mcgra_ensemble)
        b0, b1_ = output_band(n, eng.rank, world)
        ea = N.EnsembleArgs()
        keep = []                                   # operands must outlive the launch

        def gram(Z, variant=None):
            if variant is None:
                Zp, variant, rown = self._decode2_spec(Z.to(torch.float32))
            else:
                Zp, rown = Z.to(torch.float32).contiguous(), None
            keep.append((Zp, rown))
            t = ea.t[ea.nterms]
            t.kind, t.d, t.variant, t.Z, t.rownorm = N.TERM_GRAM, int(Zp.shape[1]), variant, ptr(Zp), ptr(rown)
            ea.nterms += 1

        def dense(band):            # rows [b0, b1) of an n x n operand: the global row index lands in the band
            band = band.to(device=dev, dtype=torch.float32).contiguous()
            keep.append(band)
            t = ea.t[ea.nterms]
            t.kind, t.dense = N.TERM_DENSE, band.data_ptr() - b0 * n * 4
            ea.nterms += 1

        # modified_adj: one GPU reads the decoded tiles (clamped to [0, 1] in the kernel); the row bands of several
        # GPUs need tiles of other ranks, so they re-expand relu(zf zf^T) with zero diagonal instead and free theirs
        if world > 1:
            xf = None
            gram(zf, 4)
        gram(H1)
        gram(H2)
        dense(HostBands.of(fa).rows(b0, b1_, dev))
        gram(YA2)
        if args.useH_A:
            gram(self.H_A.detach().to(dev))
        if args.useY_A:
            gram(self.Y_A.detach().to(dev))
        if args.useY:
            path = "./saved_data/" + args.dataset + ".npy"
            lab = np.load(path, mmap_mode="r") if os.path.exists(path) else None                # :133-134
            if lab is not None and lab.shape == (n, n):      # (a stale file of another graph size is ignored)
                dense(torch.from_numpy(np.ascontiguousarray(lab[b0:b1_])))
            else:    # same matrix built from the labels (main.prepare, main.py:440-450)
                t = ea.t[ea.nterms]
                t.kind, t.labels = N.TERM_LABEL, ptr(labels_t)
                ea.nterms += 1
        out = torch.empty(max(b1_ - b0, 0), n, dtype=torch.float32, device=dev)
        if b1_ > b0:
            call("mcgra_ensemble", ptr(xf), n, _C.byref(ea), out.data_ptr() - b0 * n * 4, n, b0, b1_, st)
        if world > 1:
            torch.cuda.current_stream().synchronize()       # `keep` holds the operands until the launch has consumed them
        del xf, keep
        self.modified_adj = out.detach()
        self.modified_adj_rows = (b0, b1_)

    # ------------------------------------------------------------------------------------------------
    # stand-alone helpers of the reference class, same names and semantics (more in base_attack.RowBandResult)
    def get_modified_adj2(self, ori_adj, adj_changes):
        return self._expand(adj_changes, ori_adj)

    def get_modified_adj_after(self, ori_adj=None):
        return self._expand(self.adj_changes_after, ori_adj)

    def dot_product_decode2(self, Z):
        n = Z.shape[0]
        out = torch.zeros(n, n, dtype=torch.float32, device=torch.device(self.device))
        self._gram_add(out, Z.detach().to(self.device))
        return out

    def adding_noise(self, modified_adj, eps=0):
        """clamp(M + eps * N(0,1), 0, 1) in place on M (topology_attack.py:474-478).  The draw comes from torch's CUDA
        generator (the reference's stream), the add + clamp is one native streaming pass."""
        M = modified_adj
        if not (M.is_cuda and M.dtype == torch.float32 and M.is_contiguous()):
            raise N.NativeError("adding_noise needs a contiguous fp32 CUDA tensor (no CPU fallback)")
        noise = torch.randn_like(M)
        call("mcgra_noise_clamp", ptr(M), ptr(noise), float(eps), M.numel(), N.stream_ptr())
        return M

    def delete_eye(self, A):
        """topology_attack.py:469-472 (the reference computes A * (1 - I) and returns None)."""
        A = A * (torch.ones_like(A) - torch.eye(self.nnodes, device=A.device, dtype=A.dtype))

    def dot_product(self, X, Y):
        """|| Y^T X ||_F (topology_attack.py:480-481): second moments for narrow operands, the tcgen05 contraction
        (mcgra_gemm_nt on transposed operand images) for wide ones."""
        from .dense_measure import cross_frobenius
        return cross_frobenius(X, Y, center=False).sqrt().float()

    def calc_kl(self, X, Y):
        """KLDivLoss(batchmean)(log_softmax(Y, 1), softmax(X, 1)) (topology_attack.py:483-487), forward value."""
        X = X.detach().to(torch.float32).contiguous()
        Y = Y.detach().to(torch.float32).contiguous()
        if not X.is_cuda:
            raise N.NativeError("calc_kl needs CUDA tensors (no CPU fallback)")
        out = torch.zeros(1, dtype=torch.float64, device=X.device)
        call("mcgra_row_kl", ptr(X), ptr(Y), X.shape[0], X.shape[1], X.stride(0), Y.stride(0), ptr(out), N.stream_ptr())
        return (out[0] / X.shape[0]).float()

    def test(self, idx_attack, idx_val, idx_test, adj, features, labels, victim_model):
        """Accuracy of the victim on the normalised adjacency (topology_attack.py:83-93)."""
        from . import utils
        adj, features, labels = utils.to_tensor(adj, features, labels, device=self.device)
        victim_model.eval()
        adj_norm = utils.normalize_adj_tensor(adj)
        output = victim_model(features, adj_norm)
        return utils.accuracy(output[idx_test], labels[idx_test]).item()
