"""PGDEngine: host-side sequencing of the native stages of one PGD iteration.

One PGD iteration of the reference (MC-GRA/topology_attack.py:161-283, SURVEY.md 3.2 steps 1-17) becomes a
fixed sequence of C-ABI calls on the current CUDA stream, with no host synchronisation:

    node_pre -> [row_sumexp] -> propagate#1(+element-wise c1/c6) -> node_mid -> propagate#2 -> node_head
    -> pairs(c7,c2) -> node_bwd2 -> propagate#3 -> node_bwd1 -> propagate#4 -> node_rho -> fold_adam
    -> [bisection passes]

The adjacency estimate lives only as the tiled lower triangle (x', Adam m, v); n x n matrices are never
materialised.  With world_size > 1 every rank owns a contiguous range of tile rows (equal tile counts) and the
n x K partial results are summed with torch.distributed.all_reduce (NCCL over NVLink) between stages.
PyTorch is used for device memory, streams and the collective only.
"""
import ctypes as C
import math
import os

import torch

from . import _native as N
from ._native import ACC, call, ptr

HID = N.HID
TILE = N.TILE
MEASURES = {"MSELoss": N.M_MSE, "KL": N.M_KL, "HSIC": N.M_HSIC, "CKA": N.M_CKA, "DP": N.M_DP, "KDE": N.M_KDE}
KDE_NB = 8      # columns of an n x n operand that reach utils.MutualInformation's kernel (bin_j ~ j, values in [0, 1]; csrc/kde.cu)
ALIGN = {"c1": 100, "c2": 1000, "c6": 10, "c7": 10, "c9": 1, "c10": 1}      # MC-GRA/utils.py:1100-1111


# largest n for which the iteration is replayed as a CUDA graph (0 disables); env override for A/B runs
BISECT_PASSES = 10
GRAPH_MAX_N = int(os.environ.get("MCGRA_GRAPH_MAX_N", "8192"))


def tri(i):
    return i * (i + 1) // 2


def shard_tile_rows(T, world):
    """Contiguous tile-row ranges with (nearly) equal tile counts: boundaries ~ T*sqrt(g/G) (SURVEY 8(e))."""
    total = tri(T)
    bounds = [0]
    for g in range(1, world):
        target = total * g / world
        I = int(round((math.sqrt(8 * target + 1) - 1) / 2))
        I = max(bounds[-1], min(T, I))
        bounds.append(I)
    bounds.append(T)
    return [(bounds[g], bounds[g + 1]) for g in range(world)]


class HostBands:
    """An n x n matrix given by row bands (multi-GPU: every rank holds, and copies host -> device, only the rows it
    touches).  `bands` maps (r0, r1) -> tensor [r1 - r0, n] (pinned host or device memory)."""

    def __init__(self, n, bands):
        self.n, self.bands = int(n), dict(bands)

    def rows(self, r0, r1, device):
        if r1 <= r0:                      # a rank without tile rows / without a result band (more ranks than tile rows)
            return torch.zeros(0, self.n, dtype=torch.float32, device=device)
        for (b0, b1), t in self.bands.items():
            if b0 <= r0 and r1 <= b1:
                return t[r0 - b0:r1 - b0].to(device=device, dtype=torch.float32, non_blocking=True).contiguous()
        raise KeyError(f"rows [{r0}, {r1}) are not covered by the bands {sorted(self.bands)}")

    @staticmethod
    def of(t):
        return t if isinstance(t, HostBands) else HostBands(t.shape[0], {(0, t.shape[0]): t})


def output_band(n, rank, world):
    """Row band [b0, b1) of the n x n result owned by `rank`: equal 64-aligned bands (mcgra_ensemble's block height)."""
    rb = ((n + world - 1) // world + 63) // 64 * 64
    return min(n, rank * rb), min(n, (rank + 1) * rb)


NOISE_MEASURES = ("MSELoss", "KDE")


def check_noise_supported(measure, world, feature_adj, device):
    """Scope of attack() with adjacency noise (--eps != 0): MSELoss or KDE on one CUDA device, MSELoss on tile-row shards
    (world > 1), feature_adj as a full tensor.  Raised before any device work."""
    if measure not in NOISE_MEASURES:
        raise NotImplementedError(f"--eps != 0 is implemented for --measure MSELoss and KDE only (got {measure!r}): the "
                                  "other measures' passes and closed forms assume a symmetric A_hat")
    if isinstance(feature_adj, HostBands):
        raise NotImplementedError("--eps != 0 needs feature_adj as a full tensor: the row-band noisy path is not built")
    if world > 1 and measure != "MSELoss":
        raise NotImplementedError(f"--eps != 0 with world > 1 is implemented for --measure MSELoss only (got {measure!r}): "
                                  "the sharded noisy KDE path is not built")
    if torch.device(device).type != "cuda":
        raise NotImplementedError(f"--eps != 0 needs a CUDA device (got {device!r}); there is no CPU fallback")


class PGDEngine:
    def __init__(self, n, S1, W2, b1, b2, Wl, bl, labels, idx_attack, HA, YA, feature_adj, measure, weights,
                 lr, weight_sup=1.0, num_edges=None, x0=None, device="cuda", rank=0, world=1, group=None,
                 max_epochs=1024, plain_gd=False, eps=0.0, noise=None):
        self.eps = float(eps)
        if self.eps != 0.0:
            check_noise_supported(measure, world, feature_adj, device)
        if not torch.cuda.is_available():
            raise N.NativeError("mcgra_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        N.lib()
        import time as _t
        _dbg = bool(os.environ.get("MCGRA_E2E_TIMING"))
        _t0 = [_t.perf_counter()]

        def _tick(name):
            if _dbg:
                torch.cuda.synchronize()
                now = _t.perf_counter()
                print(f"[engine-setup rank {rank}] {name}: {now - _t0[0]:.3f}s", flush=True)
                _t0[0] = now
        self._tick = _tick
        dev = torch.device(device)
        self.dev, self.n, self.rank, self.world, self.group = dev, int(n), rank, world, group
        n = self.n
        self.T = (n + TILE - 1) // TILE
        self.npad = self.T * TILE
        self.tr0, self.tr1 = shard_tile_rows(self.T, world)[rank]
        self.ntiles = tri(self.tr1) - tri(self.tr0)
        self.P = n * (n - 1) // 2
        f32 = dict(dtype=torch.float32, device=dev)

        def dv(t, dtype=torch.float32):
            return t.detach().to(device=dev, dtype=dtype).contiguous()

        self.S1 = dv(S1)
        self.W2, self.b1, self.b2, self.Wl, self.bl = dv(W2), dv(b1), dv(b2), dv(Wl), dv(bl)
        assert self.W2.shape == (HID, HID) and self.S1.shape == (n, HID), "hidden width must be 16 (main.py:175)"
        self.nclass = int(self.Wl.shape[0])
        if self.nclass > N.MAXC:
            raise N.NativeError(f"nclass {self.nclass} > {N.MAXC}")
        self.labels = dv(labels, torch.int64)
        idx = torch.as_tensor(idx_attack, dtype=torch.int64, device=dev)
        self.wmult = (torch.bincount(idx, minlength=n).to(torch.float32) / float(idx.numel())).contiguous()
        self.HA, self.YA = dv(HA), dv(YA)
        assert self.HA.shape == (n, HID) and self.YA.shape == (n, self.nclass)

        # ---- flags -> scaled constants (topology_attack.py:151, 211-272) ----
        self.measure_name = measure
        if measure not in MEASURES:
            raise NotImplementedError(f"measure {measure!r}")
        self.measure = MEASURES[measure]
        w1, w2, _, _, _, w6, w7, _w8, w9, w10 = [float(w) for w in weights]
        self.w = (w1, w2, w6, w7, w9, w10)
        self.weight_sup = float(weight_sup)
        self.lr = float(lr)
        nn2 = float(n) * float(n)
        sgn = -1.0 if measure == "HSIC" else 1.0
        self.c1_active = False
        self.Ft = self.Fdiag = self.lseF = self.Ct = None
        self.k1 = self.k2 = 0.0
        self.meas_nn = N.M_NONE       # measure code used by the element-wise n x n kernels
        self.idx = idx
        fa = None
        fa_row0 = 0           # first global row held by `fa` (row-band input: only this rank's tile rows are resident)
        if w1 != 0 and feature_adj is not None:
            if isinstance(feature_adj, HostBands):
                fa_row0 = self.tr0 * TILE
                fa = feature_adj.rows(fa_row0, min(n, self.tr1 * TILE), dev)
                mm = torch.stack([fa.max() if fa.numel() else torch.tensor(-math.inf, device=dev),
                                  -(fa.min() if fa.numel() else torch.tensor(math.inf, device=dev))])
                if world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(mm, op=dist.ReduceOp.MAX, group=group)
                self.c1_active = bool(mm[0] != -mm[1])
            else:
                fa = feature_adj.to(dev)
                # topology_attack.py:212: the term is skipped when feature_adj is constant
                if bool(fa.max() != fa.min()):
                    self.c1_active = True
                    fa = fa.to(torch.float32).contiguous()
        _tick("node constants + feature_adj rows on device")
        native_nn = (self.measure == N.M_MSE) or (self.measure == N.M_KL and w2 == 0)
        # Which engine evaluates the n x n terms c1 / c2:
        #   "native": fused element-wise kernels (MSELoss; KL when only c1 is on)
        #   "kl2"   : KL with c2 on -- row-softmax statistics of A_hat AND of the decode gram M1: three tile passes
        #             (csrc/kl2.cu) that hand the element-wise gradient tiles to the pipeline (MCGRA_M_PRE)
        #   "dense" : HSIC / CKA / DP -- n^3 contractions on tcgen05 (dense_measure.DenseMeasure, csrc/gemm.cu), gradient
        #             tiles handed over the same way
        #   "kde"   : utils.MutualInformation -- kernel-value slabs of the first KDE_NB columns, weighted second moments
        #             and their closed-form gradient (csrc/kde.cu), gradient tiles handed over the same way
        self.nn_mode = "native" if native_nn else ("kl2" if self.measure == N.M_KL else
                                                   "kde" if self.measure == N.M_KDE else "dense")
        if not (self.c1_active or w2 != 0):
            self.nn_mode = "off"
        self.w1, self.w2 = w1, w2
        self.dense = None
        ntl = max(self.ntiles, 1) * TILE * TILE
        if self.nn_mode == "native":
            if self.c1_active:
                self.Ft = torch.zeros(ntl, **f32)
                self.Fdiag = torch.zeros(n, **f32)
                # (row-band input: the pointer is shifted so that the kernel's global row index lands in the band; the
                #  mirrored entries live on other ranks, so the band is taken as is instead of (F_ij + F_ji) / 2)
                call("mcgra_dense_to_tiles", fa.data_ptr() - fa_row0 * n * 4, n, n, self.tr0, self.tr1,
                     0 if isinstance(feature_adj, HostBands) else 1, ptr(self.Ft), ptr(self.Fdiag), N.stream_ptr())
                if self.eps != 0.0:
                    # the noisy A_hat is not symmetric: c1 pairs A_hat_ij with F_ij and A_hat_ji with F_ji, so both
                    # orientations of feature_adj are tiled as they are (F, then F^T).  Only the rows of this rank's tile
                    # rows are read, so F^T is formed for that band alone (columns [r0, r1) of F): n x (r1 - r0) floats
                    # instead of n x n, with the pointer shifted as for row-band input
                    self.FLt = torch.zeros(ntl, **f32)
                    self.FUt = torch.zeros(ntl, **f32)
                    r0, r1 = self.tr0 * TILE, min(n, self.tr1 * TILE)
                    if r1 > r0:
                        call("mcgra_dense_to_tiles", ptr(fa), n, n, self.tr0, self.tr1, 0, ptr(self.FLt), None,
                             N.stream_ptr())
                        faT = fa[:, r0:r1].t().contiguous()
                        call("mcgra_dense_to_tiles", faT.data_ptr() - r0 * n * 4, n, n, self.tr0, self.tr1, 0,
                             ptr(self.FUt), None, N.stream_ptr())
                        del faT
                if world > 1:     # each rank wrote the diagonal of its own tile rows only
                    self._allreduce(self.Fdiag)
                self.meas_nn = self.measure
                if self.measure == N.M_MSE:
                    self.k1 = w1 * 1000 * ALIGN["c1"] / nn2
                else:
                    self.k1 = w1 * 1000 * ALIGN["c1"] / float(n)
                    if isinstance(feature_adj, HostBands):
                        self.lseF64 = torch.zeros(n, dtype=torch.float64, device=dev)
                        self.lseF64[fa_row0:fa_row0 + fa.shape[0]] = torch.logsumexp(fa.double(), dim=1)
                        self._allreduce(self.lseF64)
                    else:
                        self.lseF64 = torch.logsumexp(fa.double(), dim=1)
                    self.lseF = self.lseF64.float().contiguous()
            if w2 != 0:
                self.k2 = w2 * 100 * ALIGN["c2"] / nn2
        elif self.nn_mode in ("kl2", "dense", "kde"):
            if isinstance(feature_adj, HostBands):
                raise NotImplementedError("row-band feature_adj input is implemented for the element-wise measures (MSELoss, "
                                          "KL with w2 = 0); pass a full tensor for HSIC / CKA / DP / KL-c2")
            # dL/dA_ij + dL/dA_ji and dL/dM1_ij + dL/dM1_ji.  The noisy path (KDE) hands the A_hat gradient to its own
            # kernels as a column slab, and needs the M1 tiles only when c2 is on
            self.Ft = torch.zeros(ntl, **f32) if self.eps == 0.0 else None
            self.Ct = torch.zeros(ntl, **f32) if (self.eps == 0.0 or w2 != 0) else None
            self.Fdiag = torch.zeros(n, **f32)     # dL/dA_ii
            self.meas_nn = N.M_PRE
            self.sgn = sgn
            k1c = w1 * 1000 * ALIGN["c1"] if self.c1_active else 0.0
            k2c = w2 * 100 * ALIGN["c2"]
            if self.nn_mode == "dense":
                from .dense_measure import DenseMeasure
                self.dense = DenseMeasure(self, fa if self.c1_active else None, self.measure, k1c, k2c, sgn)
            elif self.nn_mode == "kde":
                nb = min(KDE_NB, n)
                hi = max(float(fa.max()), 1.0) if self.c1_active else 1.0
                if hi > 3.0:      # column j >= KDE_NB would no longer underflow: exp(-0.5 ((v - j) / 0.32)^2) > fp32 min
                    raise NotImplementedError("KDE: feature_adj values above 3 reach bins beyond the kept columns")
                self.kde = kd = dict(nb=nb, k1c=k1c, k2c=k2c, bin=float(n) / float(n - 1),
                                     w=torch.full((n,), 1.0 / n, **f32),
                                     slabA=torch.zeros(n, nb, **f32), slabM=torch.zeros(n, nb, **f32),
                                     kvA=torch.zeros(n, nb, **f32), kvM=torch.zeros(n, nb, **f32),
                                     gkvA=torch.zeros(n, nb, **f32), gkvM=torch.zeros(n, nb, **f32),
                                     gA=torch.zeros(n, nb, **f32), gM=torch.zeros(n, nb, **f32),
                                     mom=torch.zeros(2 * nb + 2 * nb * nb, dtype=torch.float64, device=dev),
                                     gmom=torch.zeros(2 * nb + 2 * nb * nb, dtype=torch.float64, device=dev))
                if self.c1_active and self.eps != 0.0:     # the noisy path's fp64 stage forms kernel values itself
                    kd["slabF"] = fa[:, :nb].contiguous()
                elif self.c1_active:
                    kd["kvF"] = torch.zeros(n, nb, **f32)
                    call("mcgra_kde_kv", ptr(fa), n, nb, n, kd["bin"], ptr(kd["kvF"]), N.stream_ptr())
            else:
                self.kl2 = k = N.Kl2Args()
                self._kl2_keep = keep = {}
                for name in ("seA", "seM", "lseA", "lseM", "klrow", "c1row"):
                    keep[name] = torch.zeros(n, **f32)
                    setattr(k, name, ptr(keep[name]))
                if self.c1_active:
                    keep["Ffeat"] = torch.zeros(ntl, **f32)
                    keep["Fdiag_feat"] = torch.zeros(n, **f32)
                    call("mcgra_dense_to_tiles", ptr(fa), n, n, self.tr0, self.tr1, 1, ptr(keep["Ffeat"]),
                         ptr(keep["Fdiag_feat"]), N.stream_ptr())
                    if world > 1:
                        self._allreduce(keep["Fdiag_feat"])
                    keep["lseF"] = torch.logsumexp(fa.double(), dim=1).float().contiguous()
                    k.Ftiles, k.Fdiag_feat, k.lseF = ptr(keep["Ffeat"]), ptr(keep["Fdiag_feat"]), ptr(keep["lseF"])
                k.tr0, k.tr1, k.n = self.tr0, self.tr1, n
                k.EAt, k.Ct = ptr(self.Ft), ptr(self.Ct)
                k.k1c, k.k2c = k1c, k2c
        del fa
        _tick("feature tiles / measure setup")
        self.k6 = -w6 * 100 * ALIGN["c6"] / nn2
        self.k7 = -w7 * ALIGN["c7"] / nn2
        self.nd_native = self.measure in (N.M_MSE, N.M_KL)
        self.w9 = sgn * w9 * ALIGN["c9"]
        self.w10 = sgn * w10 * ALIGN["c10"]
        self.plain_gd = bool(plain_gd)
        self.Gt = None                 # optional upstream dL/dM tiles (feature smoothing, mcgpb_attack)
        self.smooth = None
        self.smooth_on = False
        self.budget = float(num_edges) if num_edges is not None else float("inf")
        self.proj_possible = self.budget < float(self.P)

        # ---- state: tiled triangle of x', m, v ----
        nel = max(self.ntiles, 1) * TILE * TILE
        self.xt = torch.zeros(nel, **f32)
        self.mt = torch.zeros(nel, **f32)
        self.vt = torch.zeros(nel, **f32)
        self.mu = torch.zeros(1, **f32)
        self.raw = 0
        self.step = 0
        self.max_epochs = max_epochs
        self.acc_hist = torch.zeros(max_epochs + 2, N.ACC_N, dtype=torch.float64, device=dev)
        # Ring mode (small graphs, launch-bound): the accumulator rows are a fixed ring of two, the Adam step is a device
        # counter and a tiny kernel appends the finished row to acc_hist, so that no launch carries a per-iteration host
        # scalar and two consecutive iterations can be replayed as ONE CUDA graph (run()).  Large graphs keep the direct
        # history rows: launch overhead is < 1 % there and per-kernel CUDA-event timing stays possible.
        self.ring_mode = (GRAPH_MAX_N > 0 and n <= GRAPH_MAX_N and world == 1 and self.nn_mode in ("native", "off")
                          and self.measure == N.M_MSE and self.eps == 0.0)
        self.acc_ring = torch.zeros(2, N.ACC_N, dtype=torch.float64, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self._graph = None
        self.minmax = torch.zeros(2, **f32)
        self.bstate = torch.zeros(8, **f32)
        self.cand = torch.zeros(8, dtype=torch.float64, device=dev)
        self.d = torch.zeros(n, **f32)
        self.d_next = torch.zeros(n, **f32)

        # ---- node buffers ----
        z = lambda *s: torch.zeros(*s, **f32)
        self.r = z(n)
        self.B1, self.Y1, self.B2, self.Y2, self.B3, self.Y3 = (z(n, 32) for _ in range(6))
        # Y4 and eps_row are reduced across ranks at the same point of the iteration: one buffer, one collective
        self.Y4e = z(n * HID + n)
        self.B4, self.Y4 = z(n, HID), self.Y4e[:n * HID].view(n, HID)
        (self.S2, self.T2, self.H2, self.dZ2, self.dZ1, self.dQ1, self.dQ2, self.demd, self.zhat,
         self.dzhat) = (z(n, HID) for _ in range(10))
        self.inv_norm, self.eps_row, self.rho = z(n), self.Y4e[n * HID:], z(n)
        self.em = z(n, HID)
        self.masks = torch.zeros(n, dtype=torch.int32, device=dev)
        self.masks2 = torch.zeros(n, dtype=torch.int32, device=dev)
        self.Wt = z(128, self.npad)
        self.fold_ws = torch.empty(int(N.lib().mcgra_fold_ws_bytes(n)), dtype=torch.uint8, device=dev)
        self.prop_ws = torch.empty(int(N.lib().mcgra_propagate_ws_bytes(n, 32)), dtype=torch.uint8, device=dev)
        self.pairs_ws = torch.empty(int(N.lib().mcgra_pairs_ws_bytes(n)), dtype=torch.uint8, device=dev)
        kl_native = self.meas_nn == N.M_KL and self.nn_mode == "native"
        self.sumexp = z(n) if kl_native else None
        self.lseA = z(n) if kl_native else None
        self.dlse = z(n) if kl_native else None

        if self.measure == N.M_KDE and (self.w9 != 0.0 or self.w10 != 0.0):
            c = self.nclass
            md = max(HID, c)
            self.kde_nd = nd = dict(kvE=z(n, md), gkv=z(n, md), gV=z(n, md), p2=z(n, c),
                                    mom=torch.zeros(2 * md + 2 * md * md, dtype=torch.float64, device=dev),
                                    gmom=torch.zeros(2 * md + 2 * md * md, dtype=torch.float64, device=dev),
                                    m=float(idx.numel()))
            if self.w9 != 0.0:        # bins = linspace(0, 16, 16) (topology_attack.py:246-248)
                nd["kvH"] = z(n, HID)
                call("mcgra_kde_kv", ptr(self.HA), HID, HID, n, HID / (HID - 1.0), ptr(nd["kvH"]), N.stream_ptr())
            if self.w10 != 0.0:       # bins = linspace(0, c, c) (:261-263)
                nd["kvY"] = z(n, c)
                nd["binc"] = c / (c - 1.0) if c > 1 else 0.0
                call("mcgra_kde_kv", ptr(self.YA), c, c, n, nd["binc"], ptr(nd["kvY"]), N.stream_ptr())
        elif not self.nd_native and (self.w9 != 0.0 or self.w10 != 0.0):
            self.nd_p2 = z(n, self.nclass)
            self.nd_mom = torch.zeros(int(N.lib().mcgra_nd_scratch_doubles(self.nclass)), dtype=torch.float64, device=dev)
            self.nd_coef = z(int(N.lib().mcgra_nd_scratch_floats(self.nclass)))
            self.nd_m = float(idx.numel())
        _tick("state + node buffers")
        if self.eps != 0.0:
            # noisy path: the two orientations of M, its diagonal, the gradient tiles handed to the fold, and zero
            # factors / rho for that fold (its own product and degree terms are already inside the gradient tiles)
            self.Lt, self.Ut, self.Gn = (torch.zeros(nel, **f32) for _ in range(3))
            self.mdiag = z(n)
            self.Wt0, self.rho0 = z(128, self.npad), z(n)
            if not self.c1_active or self.nn_mode != "native":
                self.FLt = self.FUt = None
            # (the default draw captures no reference to the engine: a cycle would keep its device memory alive
            #  after attack() drops the engine)
            self._noise_fn = noise if noise is not None else (
                lambda t, n=n, dev=dev: torch.randn((n, n), dtype=torch.float32, device=dev))
            # world > 1: every rank draws the whole matrix and reads its tiles' blocks of it, so the ranks must draw
            # alike.  Per iteration, the fp64 sums of row 0 and of the diagonal (f) go through one MAX all-reduce as
            # (f, -f); the ranks agreed iff max f == min f (check_noise_agreement, once, after the loop)
            self.noise_fp = torch.zeros(max_epochs, 4, dtype=torch.float64, device=dev) if world > 1 else None
        self.set_parameter(x0)
        _tick("set_parameter")

    # ------------------------------------------------------------------------------------------------
    def _allreduce(self, t, op=None):
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=op or dist.ReduceOp.SUM, group=self.group)

    def set_parameter(self, x_packed):
        """Load a packed parameter vector (reference layout) -- zeros when None (topology_attack.py:77-78)."""
        st = N.stream_ptr()
        self.mt.zero_()
        self.vt.zero_()
        self.mu.zero_()
        self.step = 0
        self.acc_hist.zero_()
        self.acc_ring.zero_()
        self.step_dev.zero_()
        if x_packed is None:
            self.xt.zero_()
            self.raw = 0
            sumsq = 0.0
        else:
            xp = x_packed.detach().to(device=self.dev, dtype=torch.float32).contiguous()
            assert xp.numel() == self.P
            call("mcgra_tril_to_tiles", ptr(xp), self.n, self.tr0, self.tr1, ptr(self.xt), st)
            self.raw = 1
            sumsq = float((xp.double() ** 2).sum())
        self._acc_row(0)[ACC["SUMSQ"]] = sumsq
        self.d.fill_(1.0 if self.rank == 0 else 0.0)
        call("mcgra_degree", ptr(self.xt), self.n, self.tr0, self.tr1, ptr(self.mu), self.raw, ptr(self.d), st)
        self._allreduce(self.d)

    def _acc_row(self, t):
        """Accumulator row of iteration t (tensor view): a history row, or one of the two ring rows."""
        return self.acc_ring[t & 1] if self.ring_mode else self.acc_hist[t]

    def _node_args(self, t):
        a = N.NodeArgs()
        a.n, a.nclass = self.n, self.nclass
        a.W2, a.b1, a.b2, a.Wl, a.bl = ptr(self.W2), ptr(self.b1), ptr(self.b2), ptr(self.Wl), ptr(self.bl)
        a.S1, a.labels, a.wmult, a.HA, a.YA = ptr(self.S1), ptr(self.labels), ptr(self.wmult), ptr(self.HA), ptr(self.YA)
        a.d, a.r = ptr(self.d), ptr(self.r)
        a.B1, a.Y1, a.B2, a.Y2, a.B3, a.Y3 = (ptr(x) for x in (self.B1, self.Y1, self.B2, self.Y2, self.B3, self.Y3))
        a.B4, a.Y4 = ptr(self.B4), ptr(self.Y4)
        a.S2, a.T2, a.H2, a.dZ2, a.dZ1, a.dQ1 = (ptr(x) for x in (self.S2, self.T2, self.H2, self.dZ2, self.dZ1, self.dQ1))
        a.dQ2, a.demd, a.zhat, a.dzhat = ptr(self.dQ2), ptr(self.demd), ptr(self.zhat), ptr(self.dzhat)
        a.inv_norm, a.masks, a.masks2 = ptr(self.inv_norm), ptr(self.masks), ptr(self.masks2)
        a.eps_row, a.rho, a.Wt = ptr(self.eps_row), ptr(self.rho), ptr(self.Wt)
        a.Fdiag = ptr(self.Fdiag)
        a.acc = self._acc_row(t).data_ptr()
        a.measure = self.measure                      # n x d terms c9 / c10 (node kernel handles MSE / KL)
        a.measure_nn = self.meas_nn                   # n x n terms: diagonal part in node_rho
        a.weight_sup = self.weight_sup
        a.k1 = self.k1 if (self.c1_active and self.nn_mode == "native") else 0.0
        a.k2, a.k6, a.k7 = self.k2, self.k6, self.k7
        a.w9, a.w10 = (self.w9, self.w10) if self.nd_native else (0.0, 0.0)
        a.npad = self.npad
        a.d_next, a.d_fill = ptr(self.d_next), (1.0 if self.rank == 0 else 0.0)
        a.acc_next = self._acc_row(t + 1).data_ptr()
        a.minmax = ptr(self.minmax)
        a.lseA, a.lseF = ptr(self.lseA), ptr(self.lseF)
        a.em = ptr(self.em)
        a.dlse = ptr(self.dlse)
        return a

    def forward_stages(self, t):
        """Forward half of an iteration (through node_head); returns the node-args struct."""
        st = N.stream_ptr()
        n, tr0, tr1, mu, raw = self.n, self.tr0, self.tr1, ptr(self.mu), self.raw
        a = self._node_args(t)
        ap = C.byref(a)
        call("mcgra_node_pre", ap, st)
        if self.meas_nn == N.M_KL and self.nn_mode == "native":
            self.sumexp.zero_()
            call("mcgra_row_sumexp", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.r), ptr(self.sumexp), st)
            self._allreduce(self.sumexp)
            lseA64 = torch.log(self.sumexp.double() + torch.exp((self.r * self.r).double()))   # + diagonal r_i^2
            self.lseA.copy_(lseA64)
            self.dlse.copy_(self.lseF64 - lseA64)
        c1_native = self.c1_active and self.nn_mode == "native"
        if c1_native or self.k6 != 0.0:
            e = N.ElemArgs()
            e.r, e.Ftiles, e.lseA, e.lseF = ptr(self.r), (ptr(self.Ft) if c1_native else None), ptr(self.lseA), ptr(self.lseF)
            e.measure = self.meas_nn if c1_native else N.M_NONE
            e.k1, e.k6 = (self.k1 if c1_native else 0.0), self.k6
            e.acc, e.eps_row = self._acc_row(t).data_ptr(), ptr(self.eps_row)
            e.dlse = ptr(self.dlse)
            call("mcgra_elem_stats", ptr(self.xt), n, tr0, tr1, mu, raw, C.byref(e), st, tag="elem_stats")
        call("mcgra_propagate", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.B1), 32, ptr(self.Y1), ptr(self.prop_ws), st,
             tag="propagate32")
        self._allreduce(self.Y1)
        call("mcgra_node_mid", ap, st)
        call("mcgra_propagate", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.B2), 32, ptr(self.Y2), ptr(self.prop_ws), st, tag="propagate32")
        self._allreduce(self.Y2)
        call("mcgra_node_head", ap, st)
        return a

    def iterate(self):
        """One full PGD iteration (forward, backward, Adam, projection); no host synchronisation."""
        t = self.step
        if t >= self.max_epochs:
            raise RuntimeError("acc history exhausted; construct the engine with a larger max_epochs")
        if self.eps != 0.0:
            return self._iterate_noisy(t)
        st = N.stream_ptr()
        n, tr0, tr1, mu, raw = self.n, self.tr0, self.tr1, ptr(self.mu), self.raw
        a = self.forward_stages(t)
        ap = C.byref(a)
        dense = self.nn_mode in ("dense", "kl2", "kde")      # gradient tiles handed over as MCGRA_M_PRE
        if self.nn_mode == "dense":
            self.dense.step(t)
        elif self.nn_mode == "kl2":
            self._kl2_stage(t)
        elif self.nn_mode == "kde":
            self._kde_stage(t)
        if self.measure == N.M_KDE:
            if self.w9 != 0.0 or self.w10 != 0.0:
                self._kde_nd_stage(t)
        elif not self.nd_native and (self.w9 != 0.0 or self.w10 != 0.0):
            self._nd_stage(t)
        if self.k7 != 0.0 or self.k2 != 0.0 or dense:
            call("mcgra_pairs", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.zhat), ptr(self.r),
                 self.k7, self.k2, (ptr(self.Ft) if dense else None), (ptr(self.Ct) if dense else None),
                 ptr(self.dzhat), ptr(self.eps_row), self._acc_row(t).data_ptr(), ptr(self.pairs_ws), st)
            if self.k7 != 0.0 and self.k2 == 0.0 and not dense:
                N.LAUNCHES["kernels"] += 2      # tcgen05 engine: operand prep (2 kernels) + k_pairs_tc
            self._allreduce(self.dzhat)
        call("mcgra_node_bwd2", ap, st)
        call("mcgra_propagate", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.B3), 32, ptr(self.Y3), ptr(self.prop_ws), st, tag="propagate32")
        self._allreduce(self.Y3)
        call("mcgra_node_bwd1", ap, st)
        call("mcgra_propagate", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.B4), 16, ptr(self.Y4), ptr(self.prop_ws), st, tag="propagate16")
        self._allreduce(self.Y4e)          # Y4 and eps_row in one collective
        call("mcgra_node_rho", ap, st)
        if self.smooth is not None and self.smooth_on:
            self._smooth_stage(t)

        f = N.FoldArgs()
        f.n, f.npad, f.Wt, f.r, f.rho = n, self.npad, ptr(self.Wt), ptr(self.r), ptr(self.rho)
        use_f = dense or (self.c1_active and self.nn_mode == "native")
        f.Ftiles = ptr(self.Ft) if use_f else None
        f.lseA, f.lseF = ptr(self.lseA), ptr(self.lseF)
        f.zhat = ptr(self.zhat)
        f.measure = self.meas_nn if use_f else N.M_NONE
        f.k1, f.k6, f.k2 = (self.k1 if use_f else 0.0), self.k6, self.k2
        f.norm_coef = self.weight_sup * 0.001
        f.lr, f.beta1, f.beta2, f.adam_eps = self.lr, 0.9, 0.999, 1e-8
        f.step = t + 1
        f.acc_prev = self._acc_row(t).data_ptr()
        f.acc_next = self._acc_row(t + 1).data_ptr()
        f.step_ptr = ptr(self.step_dev) if self.ring_mode else None
        f.d_next = ptr(self.d_next)
        f.store_clamped = 0 if self.proj_possible else 1
        f.Wk = ptr(self.fold_ws)
        f.plain_gd = 1 if self.plain_gd else 0
        f.Gtiles = ptr(self.Gt) if (self.smooth is not None and self.smooth_on) else None
        call("mcgra_fold_adam", ptr(self.xt), ptr(self.mt), ptr(self.vt), tr0, tr1, mu, raw, C.byref(f),
             ptr(self.minmax), st)
        # the buffer now holds the un-projected Adam output x' (mu = 0), or the clamped parameter itself
        self.raw = 0 if self.proj_possible else 2
        self.mu.zero_()
        if self.world > 1:
            import torch.distributed as dist
            self._allreduce(self._acc_row(t + 1)[:16])
            if self.proj_possible:         # the bisection bracket is only read when the budget can bind
                self._allreduce(self.minmax[0:1], dist.ReduceOp.MIN)
                self._allreduce(self.minmax[1:2], dist.ReduceOp.MAX)
        if self.proj_possible:
            self._project(t)
        self._allreduce(self.d_next)
        self.d, self.d_next = self.d_next, self.d
        if self.ring_mode:       # hist[step_dev] = finished row; step_dev += 1
            call("mcgra_history_push", self._acc_row(t).data_ptr(), ptr(self.acc_hist), self.acc_hist.shape[0],
                 ptr(self.step_dev), st)
        self.step = t + 1

    def _propagate_noisy(self, B, K, Y, transpose, reduce=None):
        """Y += M B (transpose=False) or M^T B from the two orientation planes and the diagonal (mcgra.h).  With world > 1
        the shards' products are all-reduced (`reduce`: a buffer that holds Y, default Y itself) before the diagonal is
        added, once, on every rank."""
        st, n = N.stream_ptr(), self.n
        first, second = (self.Ut, self.Lt) if transpose else (self.Lt, self.Ut)
        for plane, sel in ((first, N.PROD_DIRECT), (second, N.PROD_MIRRORED)):
            call("mcgra_propagate_sel", ptr(plane), n, self.tr0, self.tr1, None, 2, ptr(B), K, ptr(Y), ptr(self.prop_ws),
                 sel, st, tag=f"propagate{K}_sel")
        self._allreduce(Y if reduce is None else reduce)
        call("mcgra_diag_axpy", ptr(self.mdiag), ptr(B), K, n, ptr(Y), st)

    def _record_noise(self, noise, t):
        """Fingerprint of this rank's draw, reduced across ranks without a host synchronisation (world > 1)."""
        import torch.distributed as dist
        f = torch.stack((noise[0].double().sum(), noise.diagonal().double().sum()))
        row = self.noise_fp[t]
        row[:2], row[2:] = f, -f
        self._allreduce(row, dist.ReduceOp.MAX)

    def check_noise_agreement(self):
        """Raise if the ranks drew different noise in any iteration so far (world > 1, --eps != 0).  One host read."""
        if self.eps == 0.0 or self.world == 1 or self.step == 0:
            return
        rec = self.noise_fp[:self.step].cpu()
        bad = torch.nonzero(rec[:, :2] != -rec[:, 2:])
        if bad.numel():
            raise RuntimeError(f"--eps != 0 with world = {self.world}: the ranks drew different noise (first in iteration "
                               f"{int(bad[0, 0])}).  Every rank draws the full n x n matrix from its default CUDA generator: "
                               "seed all ranks alike (torch.cuda.manual_seed) before attack()")

    def _iterate_noisy(self, t):
        """One iteration with adjacency noise (--eps != 0, topology_attack.py:165, 474-478): MSELoss or KDE on one GPU,
        MSELoss on tile-row shards.
        noise stage -> node_pre -> M B1 -> node_mid -> M B2 -> node_head -> [KDE: c1 / c2 slab stage, c9 / c10]
        -> pairs (c7, KDE: c2's M1 gradient) -> noisy terms (c1, c2, c6; KDE: the A_hat slab gradient) -> node_bwd2
        -> M^T B3 -> node_bwd1 -> M^T B4 -> node_rho_diag -> noisy gradient -> fold (Adam, clamp, sums).
        world > 1 adds the collectives of DESIGN.md 3.7: the draw's fingerprint, d between the two noise stages, each
        product before its diagonal, dzhat, Y4 with eps_row, and after the fold the statistics and the bracket."""
        st = N.stream_ptr()
        n, tr0, tr1, mu, raw = self.n, self.tr0, self.tr1, ptr(self.mu), self.raw
        noise = self._noise_fn(t)
        if tuple(noise.shape) != (n, n):
            raise ValueError(f"noise draw of shape {tuple(noise.shape)}, expected ({n}, {n})")
        noise = noise.to(device=self.dev, dtype=torch.float32).contiguous()
        if self.world == 1:
            call("mcgra_noise_stage", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(noise), self.eps, ptr(self.Lt),
                 ptr(self.Ut), ptr(self.mdiag), ptr(self.d), st)
        else:
            self._record_noise(noise, t)
            self.d.zero_()
            call("mcgra_noise_tiles", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(noise), self.eps, ptr(self.Lt),
                 ptr(self.Ut), ptr(self.d), st)
            self._allreduce(self.d)
            call("mcgra_noise_diag", n, ptr(noise), self.eps, ptr(self.mdiag), ptr(self.d), st)
        a = self._node_args(t)
        ap = C.byref(a)
        call("mcgra_node_pre", ap, st)
        self._propagate_noisy(self.B1, 32, self.Y1, False)
        call("mcgra_node_mid", ap, st)
        self._propagate_noisy(self.B2, 32, self.Y2, False)
        call("mcgra_node_head", ap, st)
        kde = self.nn_mode == "kde"
        if kde:
            self._kde_stage_noisy(t)
        if self.measure == N.M_KDE and (self.w9 != 0.0 or self.w10 != 0.0):
            self._kde_nd_stage(t)
        # c7 and the M1 side of KDE's c2 are functions of the symmetric decode M1 only: the existing pass, with no A_hat
        # tiles (EAt = NULL): the noisy kernels form A_hat's part of eps_row themselves
        if self.k7 != 0.0 or self.Ct is not None:
            call("mcgra_pairs", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.zhat), ptr(self.r), self.k7, 0.0, None,
                 ptr(self.Ct), ptr(self.dzhat), ptr(self.eps_row), self._acc_row(t).data_ptr(), ptr(self.pairs_ws), st)
        na = N.NoisyArgs()
        na.n, na.npad, na.tr0, na.tr1 = n, self.npad, tr0, tr1
        na.tiles, na.mu, na.raw, na.noise, na.eps = ptr(self.xt), mu, raw, ptr(noise), self.eps
        na.Lt, na.Ut, na.FLt, na.FUt = ptr(self.Lt), ptr(self.Ut), ptr(self.FLt), ptr(self.FUt)
        na.zhat, na.r, na.rho, na.Wt = ptr(self.zhat), ptr(self.r), ptr(self.rho), ptr(self.Wt)
        na.k1 = self.k1 if self.FLt is not None else 0.0
        na.k2, na.k6 = self.k2, self.k6
        na.acc, na.eps_row, na.dzhat, na.Gt = self._acc_row(t).data_ptr(), ptr(self.eps_row), ptr(self.dzhat), ptr(self.Gn)
        if kde:
            na.gslab, na.nb = ptr(self.kde["gA"]), self.kde["nb"]
        nap = C.byref(na)
        call("mcgra_noisy_terms", nap, st)
        self._allreduce(self.dzhat)
        call("mcgra_node_bwd2", ap, st)
        self._propagate_noisy(self.B3, 32, self.Y3, True)
        call("mcgra_node_bwd1", ap, st)
        self._propagate_noisy(self.B4, 16, self.Y4, True, reduce=self.Y4e)      # Y4 and eps_row in one collective
        call("mcgra_node_rho_diag", ap, ptr(self.mdiag), st)
        call("mcgra_noisy_grad", nap, st)

        f = N.FoldArgs()
        f.n, f.npad, f.Wt, f.r, f.rho = n, self.npad, ptr(self.Wt0), ptr(self.r), ptr(self.rho0)
        f.Ftiles, f.lseA, f.lseF, f.zhat = None, None, None, None
        f.measure = N.M_NONE
        f.k1, f.k6, f.k2 = 0.0, 0.0, 0.0
        f.norm_coef = self.weight_sup * 0.001
        f.lr, f.beta1, f.beta2, f.adam_eps = self.lr, 0.9, 0.999, 1e-8
        f.step = t + 1
        f.acc_prev = self._acc_row(t).data_ptr()
        f.acc_next = self._acc_row(t + 1).data_ptr()
        f.step_ptr = None
        f.d_next = ptr(self.d_next)
        f.store_clamped = 0 if self.proj_possible else 1
        f.Wk = ptr(self.fold_ws)
        f.plain_gd = 0
        f.Gtiles = ptr(self.Gn)
        call("mcgra_fold_adam", ptr(self.xt), ptr(self.mt), ptr(self.vt), tr0, tr1, mu, raw, C.byref(f),
             ptr(self.minmax), st)
        self.raw = 0 if self.proj_possible else 2
        self.mu.zero_()
        if self.world > 1:
            import torch.distributed as dist
            self._allreduce(self._acc_row(t + 1)[:16])
            if self.proj_possible:
                self._allreduce(self.minmax[0:1], dist.ReduceOp.MIN)
                self._allreduce(self.minmax[1:2], dist.ReduceOp.MAX)
        if self.proj_possible:
            self._project(t)
        self.step = t + 1     # (the degree of the next iteration comes from its own noise stage)

    def run(self, epochs, on_iter=None, use_graph="auto"):
        """`epochs` iterations.  In ring mode (small graphs) two consecutive iterations are captured once as a CUDA graph
        and replayed: the loop is launch-bound there (~40 launches of a few microseconds each per iteration).  Capture costs
        about as much as 100 iterations save at the Cora shape (0.60 vs 0.72 ms per iteration), so "auto" only does it for
        long runs or when the engine already holds a captured graph; True forces it (tests, bench)."""
        k = int(epochs)
        if use_graph == "auto":
            use_graph = self._graph is not None or k >= 128
        if on_iter is not None or not use_graph or not self.ring_mode or k < 8 or N.TIMERS["on"] is not None:
            for _ in range(k):
                self.iterate()
                if on_iter is not None:
                    on_iter()
            return
        # eager until the parameter view has settled (raw 1 -> 2 / 0, two iterations) and the step is even (the graph
        # holds an even + an odd iteration: ring rows and the d / d_next ping-pong return to their roles)
        while k > 0 and (self.step < 2 or (self.step & 1)):
            self.iterate()
            k -= 1
        if self._graph is None and k >= 2:
            torch.cuda.synchronize(self.dev)
            g = torch.cuda.CUDAGraph()
            l0, c0, step0 = N.LAUNCHES["kernels"], N.LAUNCHES["count"], self.step
            with torch.cuda.graph(g, capture_error_mode="relaxed"):
                self.iterate()
                self.iterate()
            self._graph_kernels = N.LAUNCHES["kernels"] - l0
            N.LAUNCHES["kernels"], N.LAUNCHES["count"] = l0, c0      # capture records, it does not execute
            self.step = step0
            self._graph = g      # cached: later run() calls on this engine replay it without re-capturing
        for _ in range(k // 2 if self._graph is not None else 0):
            self._graph.replay()
            self.step += 2
            N.LAUNCHES["kernels"] += self._graph_kernels
            k -= 2
        for _ in range(k):
            self.iterate()

    def _project(self, t):
        """projection + bisection (topology_attack.py:338-347, 397-412) without a host round trip."""
        st = N.stream_ptr()
        n, tr0, tr1 = self.n, self.tr0, self.tr1
        acc_next = self._acc_row(t + 1).data_ptr()
        self.cand.zero_()
        call("mcgra_bisect_init", acc_next, ptr(self.minmax), self.budget, ptr(self.bstate), ptr(self.mu), st)
        for _ in range(BISECT_PASSES):   # 10 passes x 3 halvings: brackets up to ~10^4 wide at eps = 1e-5; finished passes read nothing
            call("mcgra_bisect_pass", ptr(self.xt), n, tr0, tr1, 1e-5, ptr(self.bstate), ptr(self.cand), st)
            self._allreduce(self.cand)
            call("mcgra_bisect_update", self.budget, 1e-5, ptr(self.bstate), ptr(self.cand), ptr(self.mu), st)
        call("mcgra_bisect_finish", ptr(self.xt), n, tr0, tr1, ptr(self.bstate), ptr(self.mu), acc_next,
             ptr(self.d_next), 1, st)
        # (with world > 1 the reset writes d_next = 1 on every rank; keep rank 0's only)
        if self.world > 1 and self.rank != 0:
            self.d_next.sub_(self.bstate[4])
        if self.world > 1:
            # bisect_finish re-accumulated SUMSQ from this rank's shard only (when the projection was active): the
            # slot was all-reduced BEFORE the projection, so reduce the re-accumulated partial again.  bstate[4] = active.
            ssq = self._acc_row(t + 1)[ACC["SUMSQ"]:ACC["SUMSQ"] + 1]
            part = torch.where(self.bstate[4] != 0, ssq, ssq / self.world)
            self._allreduce(part)
            ssq.copy_(part)

    # ------------------------------------------------------------------------------------------------
    def enable_smoothing(self, X, coef):
        """coef * tr(X^T L~ X) (feature_smoothing, MC-GPB/topology_attack.py:163-177) as an extra loss term: G = X X^T is
        tiled once (constant); toggle per iteration with `smooth_on` (the reference adds the term for t >= 50, :57-61)."""
        n, dev, st = self.n, self.dev, N.stream_ptr()
        f32 = dict(dtype=torch.float32, device=dev)
        X = X.detach().to(dev, torch.float32).contiguous()
        G = torch.zeros(n, n, **f32)
        call("mcgra_gram_accumulate", ptr(X), X.shape[1], n, 3, None, ptr(G), n, 0, n, st) if X.shape[1] <= 32 else G.copy_(X @ X.t())
        ntl = max(self.ntiles, 1) * TILE * TILE
        Gfeat = torch.zeros(ntl, **f32)
        gdiag = torch.zeros(n, **f32)
        call("mcgra_dense_to_tiles", ptr(G), n, n, self.tr0, self.tr1, 1, ptr(Gfeat), ptr(gdiag), st)
        gdiag.copy_(G.diagonal())
        del G
        self.Gt = torch.zeros(ntl, **f32)
        self.smooth = dict(Gfeat=Gfeat, gdiag=gdiag, rt=torch.zeros(n, **f32), trow=torch.zeros(n, **f32), coef=float(coef))

    def _smooth_stage(self, t):
        sm, st = self.smooth, N.stream_ptr()
        call("mcgra_smooth", ptr(self.xt), ptr(sm["Gfeat"]), ptr(sm["gdiag"]), self.n, self.tr0, self.tr1, ptr(self.mu),
             self.raw, ptr(self.d), sm["coef"], ptr(sm["rt"]), ptr(sm["trow"]), ptr(self.Gt), st)
        self._allreduce(sm["trow"])
        call("mcgra_smooth_node", self.n, ptr(self.d), ptr(sm["rt"]), ptr(sm["trow"]), ptr(sm["gdiag"]), sm["coef"],
             ptr(self.rho), self._acc_row(t).data_ptr() + 8 * ACC["C1D"], st)

    def _kl2_stage(self, t):
        """c1 / c2 under --measure KL with c2 on (topology_attack.py:212-229, 483-487): three tile passes, row
        statistics all-reduced across ranks in between (csrc/kl2.cu)."""
        st = N.stream_ptr()
        k, keep = self.kl2, self._kl2_keep
        k.tiles, k.mu, k.raw = ptr(self.xt), ptr(self.mu), self.raw
        k.zhat, k.r = ptr(self.zhat), ptr(self.r)
        kp = C.byref(k)
        for name in ("seA", "seM", "klrow", "c1row"):
            keep[name].zero_()
        call("mcgra_kl2_pass", 0, kp, st)
        self._allreduce(keep["seA"])
        self._allreduce(keep["seM"])
        call("mcgra_kl2_node", 0, kp, None, None, st)
        call("mcgra_kl2_pass", 1, kp, st)
        self._allreduce(keep["klrow"])
        self._allreduce(keep["c1row"])
        call("mcgra_kl2_node", 1, kp, ptr(self.Fdiag), self._acc_row(t).data_ptr(), st)
        call("mcgra_kl2_pass", 2, kp, st)

    def _kde_mi(self, X, dx, Y, dy, w, m, weight, slot, mom, gmom, gX, gY):
        """weight * MutualInformation(X, Y) from the kernel-value matrices X [n x d], Y [n x d] (d = dx = dy): moments,
        entropies + d/d moments, gradient w.r.t. the kernel values (gX / gY may be None)."""
        st = N.stream_ptr()
        n = self.n
        mom.zero_()
        call("mcgra_cross_moments", ptr(X), dx, ptr(Y), dy, ptr(w), n, ptr(mom), st)
        call("mcgra_kde_scalars", ptr(mom), dx, m, weight, slot, ptr(gmom), st)
        call("mcgra_cross_moments_bwd", ptr(X), dx, ptr(Y), dy, ptr(w), n, ptr(gmom), ptr(gX), ptr(gY), st)

    def _kde_stage(self, t):
        """c1 / c2 under --measure KDE (topology_attack.py:199-201, 212-229; utils.py:980-1053): only the first KDE_NB
        columns of A_hat / M1 / feature_adj reach the Gaussian bins, so the n x n x n joint pdf is an NB x NB weighted
        second moment.  Slabs are assembled from every rank's tile rows (one all-reduce), the scalar work is replicated."""
        st = N.stream_ptr()
        kd, n = self.kde, self.n
        nb, bin_ = kd["nb"], kd["bin"]
        acc = self._acc_row(t).data_ptr()
        kd["slabA"].zero_()
        call("mcgra_slab_ahat", ptr(self.xt), n, self.tr0, self.tr1, ptr(self.mu), self.raw, ptr(self.r), nb,
             ptr(kd["slabA"]), st)
        self._allreduce(kd["slabA"])
        call("mcgra_kde_kv", ptr(kd["slabA"]), nb, nb, n, bin_, ptr(kd["kvA"]), st)
        first = True
        if self.c1_active:
            self._kde_mi(kd["kvF"], nb, kd["kvA"], nb, kd["w"], float(n), kd["k1c"], acc + 8 * ACC["C1D"], kd["mom"],
                         kd["gmom"], None, kd["gkvA"])
            call("mcgra_kde_chain", ptr(kd["slabA"]), nb, ptr(kd["kvA"]), ptr(kd["gkvA"]), nb, n, bin_, ptr(kd["gA"]), 0, st)
            first = False
        if self.w2 != 0:
            call("mcgra_slab_m1", ptr(self.zhat), n, nb, ptr(kd["slabM"]), st)
            call("mcgra_kde_kv", ptr(kd["slabM"]), nb, nb, n, bin_, ptr(kd["kvM"]), st)
            self._kde_mi(kd["kvA"], nb, kd["kvM"], nb, kd["w"], float(n), kd["k2c"], acc + 8 * ACC["C2D"], kd["mom"],
                         kd["gmom"], kd["gkvA"], kd["gkvM"])
            call("mcgra_kde_chain", ptr(kd["slabA"]), nb, ptr(kd["kvA"]), ptr(kd["gkvA"]), nb, n, bin_, ptr(kd["gA"]),
                 0 if first else 1, st)
            call("mcgra_kde_chain", ptr(kd["slabM"]), nb, ptr(kd["kvM"]), ptr(kd["gkvM"]), nb, n, bin_, ptr(kd["gM"]), 0, st)
            call("mcgra_slab_to_tiles", ptr(kd["gM"]), n, self.tr0, self.tr1, nb, ptr(self.Ct), None, st)
        call("mcgra_slab_to_tiles", ptr(kd["gA"]), n, self.tr0, self.tr1, nb, ptr(self.Ft), None, st)
        self.Fdiag.zero_()
        self.Fdiag[:nb].copy_(kd["gA"][:nb, :nb].diagonal())

    def _kde_stage_noisy(self, t):
        """c1 / c2 under --measure KDE with adjacency noise (single GPU).  The draw decorrelates A_hat from feature_adj
        and from M1, so each MI is ~1e-6 of the entropies it is the difference of: the kernel values and the moments are
        formed in fp64 from the value slabs (mcgra_kde_moments64 / _chain64).  A_hat is gathered from the noisy
        estimate's planes; its gradient stays the slab kd["gA"] (mcgra_noisy_terms / mcgra_noisy_grad read it as gslab),
        its diagonal goes to Fdiag, M1's gradient to the tiles Ct."""
        st = N.stream_ptr()
        kd, n = self.kde, self.n
        nb, bin_, wt = kd["nb"], float(n) / float(n - 1), 1.0 / n
        acc = self._acc_row(t).data_ptr()
        kd["slabA"].zero_()
        call("mcgra_slab_ahat_noisy", ptr(self.Lt), ptr(self.Ut), ptr(self.mdiag), n, self.tr0, self.tr1, ptr(self.r), nb,
             ptr(kd["slabA"]), st)
        kd["gA"].zero_()
        pairs = []
        if self.c1_active:
            pairs.append((kd["slabF"], kd["slabA"], kd["k1c"], ACC["C1D"], None, kd["gA"]))
        if self.w2 != 0:
            call("mcgra_slab_m1", ptr(self.zhat), n, nb, ptr(kd["slabM"]), st)
            kd["gM"].zero_()
            pairs.append((kd["slabA"], kd["slabM"], kd["k2c"], ACC["C2D"], kd["gA"], kd["gM"]))
        for X, Y, weight, slot, gX, gY in pairs:
            kd["mom"].zero_()
            call("mcgra_kde_moments64", ptr(X), ptr(Y), nb, n, bin_, wt, ptr(kd["mom"]), st)
            call("mcgra_kde_scalars", ptr(kd["mom"]), nb, float(n), weight, acc + 8 * slot, ptr(kd["gmom"]), st)
            call("mcgra_kde_chain64", ptr(X), ptr(Y), nb, n, bin_, wt, ptr(kd["gmom"]), ptr(gX), ptr(gY), st)
        if self.w2 != 0:
            call("mcgra_slab_to_tiles", ptr(kd["gM"]), n, self.tr0, self.tr1, nb, ptr(self.Ct), None, st)
        self.Fdiag.zero_()
        self.Fdiag[:nb].copy_(kd["gA"][:nb, :nb].diagonal())

    def _kde_nd_stage(self, t):
        """c9 / c10 under --measure KDE (topology_attack.py:246-269): bins = 16 / nclass; gradient added to demd."""
        st = N.stream_ptr()
        nd, n, c = self.kde_nd, self.n, self.nclass
        acc = self._acc_row(t).data_ptr()
        if self.w9 != 0.0:
            b16 = HID / (HID - 1.0)
            kv, gkv, gV = (nd[k].view(-1)[: n * HID].view(n, HID) for k in ("kvE", "gkv", "gV"))
            call("mcgra_kde_kv", ptr(self.em), HID, HID, n, b16, ptr(kv), st)
            self._kde_mi(nd["kvH"], HID, kv, HID, self.wmult, nd["m"], self.w9, acc + 8 * ACC["C9"], nd["mom"], nd["gmom"],
                         None, gkv)
            call("mcgra_kde_chain", ptr(self.em), HID, ptr(kv), ptr(gkv), HID, n, b16, ptr(gV), 0, st)
            self.demd.add_(gV)
        if self.w10 != 0.0:
            kv, gkv, gV = (nd[k].view(-1)[: n * c].view(n, c) for k in ("kvE", "gkv", "gV"))
            call("mcgra_softmax_rows", ptr(self.em), ptr(self.Wl), ptr(self.bl), n, c, ptr(nd["p2"]), st)
            call("mcgra_kde_kv", ptr(nd["p2"]), c, c, n, nd["binc"], ptr(kv), st)
            self._kde_mi(nd["kvY"], c, kv, c, self.wmult, nd["m"], self.w10, acc + 8 * ACC["C10"], nd["mom"], nd["gmom"],
                         None, gkv)
            call("mcgra_kde_chain", ptr(nd["p2"]), c, ptr(kv), ptr(gkv), c, n, nd["binc"], ptr(gV), 0, st)
            call("mcgra_softmax_chain", ptr(gV), ptr(nd["p2"]), ptr(self.Wl), n, c, ptr(self.demd), st)

    def _nd_stage(self, t):
        """c9 / c10 under HSIC / CKA / DP (n x 16 and n x c operands): weighted second moments + closed-form gradient,
        O(n d^2) (csrc/ndmeasure.cu); the gradient is added to the node-level demd buffer."""
        a = N.NdArgs()
        a.n, a.nclass, a.measure = self.n, self.nclass, self.measure
        a.em, a.HA, a.YA, a.Wl, a.bl, a.wmult = (ptr(x) for x in (self.em, self.HA, self.YA, self.Wl, self.bl, self.wmult))
        a.m, a.w9, a.w10 = self.nd_m, self.w9, self.w10
        a.p2, a.mom, a.coef, a.demd = ptr(self.nd_p2), ptr(self.nd_mom), ptr(self.nd_coef), ptr(self.demd)
        a.acc = self._acc_row(t).data_ptr()
        call("mcgra_nd_measure", C.byref(a), N.stream_ptr())

    # ------------------------------------------------------------------------------------------------
    def losses(self):
        """Per-iteration totals from the accumulator history (one device->host copy).  Returns dict of
        numpy arrays: loss (what loss.backward() is called on, :274), origin (:172-173), and each term.
        Collective when world > 1 (every rank must call it)."""
        hist = self.acc_hist[: self.step]
        if self.world > 1:       # slots 0-7 (tile-level loss terms) are per-shard partials: sum them once, here
            hist = hist.clone()
            part = hist[:, :8].contiguous()
            self._allreduce(part)
            hist[:, :8] = part
        h = hist.cpu().numpy()
        g = lambda k: h[:, ACC[k]]
        origin = g("NLL") + 0.001 * (g("SUMSQ") ** 0.5)
        c1, c2 = g("C1") + g("C1D"), g("C2") + g("C2D")
        c6, c7 = g("C6") + g("C6D"), g("C7") + g("C7D")
        sgn = -1.0 if self.measure_name == "HSIC" else 1.0
        loss = self.weight_sup * origin + sgn * (c1 + c2) + c6 + c7 + g("C9") + g("C10")
        return dict(loss=loss, origin=origin, c1=c1, c2=c2, c6=c6, c7=c7, c9=g("C9"), c10=g("C10"))

    def packed_parameter(self):
        """The optimised parameter in the reference's packed layout (all ranks' shards summed)."""
        out = torch.zeros(self.P, dtype=torch.float32, device=self.dev)
        call("mcgra_tiles_to_tril", ptr(self.xt), self.n, self.tr0, self.tr1, ptr(self.mu), self.raw, ptr(out),
             N.stream_ptr())
        self._allreduce(out)
        return out
