"""PGDEngine: host-side sequencing of the native stages of one PGD iteration.

One PGD iteration of the reference (MC-GRA/topology_attack.py:161-283, SURVEY.md 3.2 steps 1-17) becomes a
fixed sequence of C-ABI calls on the current CUDA stream, with no host synchronisation:

    node_pre -> [row_sumexp] -> elem_stats (c1/c6) -> propagate#1 -> node_mid -> propagate#2 -> node_head
    -> [n x n stage: HSIC/CKA/DP, KL-c2, KDE] -> [n x d stage: c9/c10] -> pairs (c7, c2) -> node_bwd2 -> propagate#3
    -> node_bwd1 -> propagate#4 -> node_rho -> [smoothing] -> fold_adam -> [bisection passes]

With adjacency noise (--eps != 0, topology_attack.py:165, 474-478) a noise stage forms the noisy estimate M first; the
four products run on M's two orientation planes plus its diagonal (M^T for #3 and #4); row_sumexp and elem_stats are
skipped and a noisy-terms pass before node_bwd2 carries c1/c2/c6 instead; KDE's n x n stage works on M's slabs; pairs
keeps c7 and KDE's M1 gradient only; node_rho_diag and a noisy-gradient pass replace node_rho.

The measure-specific stages and their buffers are the engine's terms objects `nn` (c1 / c2) and `nd` (c9 / c10).

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
from .dense_measure import DenseMeasure
from .terms import ElementwiseTerms, Kl2Terms, KdeNdTerms, KdeTerms, MomentNdTerms, NNTerms

HID = N.HID
TILE = N.TILE
MEASURES = {"MSELoss": N.M_MSE, "KL": N.M_KL, "HSIC": N.M_HSIC, "CKA": N.M_CKA, "DP": N.M_DP, "KDE": N.M_KDE}
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
        self.weight_sup = float(weight_sup)
        self.lr = float(lr)
        nn2 = float(n) * float(n)
        sgn = -1.0 if measure == "HSIC" else 1.0
        self.idx = idx
        fa = None             # feature_adj on the device when c1 is on (topology_attack.py:212: off when it is constant)
        banded = isinstance(feature_adj, HostBands)
        fa_row0 = self.tr0 * TILE if banded else 0    # first global row held by `fa` (row-band input: this rank's rows)
        fmax = None           # max of all of feature_adj (KDE's range check)
        if w1 != 0 and feature_adj is not None:
            if banded:
                fa = feature_adj.rows(fa_row0, min(n, self.tr1 * TILE), dev)
                mm = torch.stack([fa.max() if fa.numel() else torch.tensor(-math.inf, device=dev),
                                  -(fa.min() if fa.numel() else torch.tensor(math.inf, device=dev))])
                self._allreduce(mm, torch.distributed.ReduceOp.MAX)
                fmax = mm[0]
                fa = fa if bool(mm[0] != -mm[1]) else None
            else:
                fa = feature_adj.to(dev)
                fmax = fa.max()
                fa = fa.to(torch.float32).contiguous() if bool(fmax != fa.min()) else None
        c1 = fa is not None
        _tick("node constants + feature_adj rows on device")
        # c1 / c2: element-wise (MSELoss; KL with c2 off) or a stage handing over gradient tiles (terms.py)
        k1c = w1 * 1000 * ALIGN["c1"] if c1 else 0.0
        k2c = w2 * 100 * ALIGN["c2"]
        self.k2 = k2c / nn2 if self.measure == N.M_MSE else 0.0      # MSELoss's c2: element-wise in pairs / node kernels
        self.nn = NNTerms()
        if self.measure == N.M_MSE or (self.measure == N.M_KL and w2 == 0):
            if c1:
                self.nn = ElementwiseTerms(self, fa, fa_row0, banded, self.measure, k1c)
        elif c1 or w2 != 0:
            if self.measure == N.M_KL:
                self.nn = Kl2Terms(self, fa, fa_row0, banded, k1c, k2c)
            elif self.measure == N.M_KDE:
                self.nn = KdeTerms(self, fa, fa_row0, banded, fmax, k1c, k2c)
            else:       # Kf = Hc F F^T Hc needs all of F: row bands are assembled on the device for the setup only
                self.nn = DenseMeasure(self, self._full_rows(fa, fa_row0, banded), self.measure, k1c, k2c, sgn)
        del fa
        _tick("feature tiles / measure setup")
        self.k6 = -w6 * 100 * ALIGN["c6"] / nn2
        self.k7 = -w7 * ALIGN["c7"] / nn2
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
        # (MSELoss has element-wise n x n terms or none)
        self.ring_mode = (GRAPH_MAX_N > 0 and n <= GRAPH_MAX_N and world == 1 and self.measure == N.M_MSE
                          and self.eps == 0.0)
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
        self.nd = None         # c9 / c10 outside the node kernels (HSIC / CKA / DP, KDE)
        if (self.w9 != 0.0 or self.w10 != 0.0) and self.measure not in (N.M_MSE, N.M_KL):
            self.nd = KdeNdTerms(self) if self.measure == N.M_KDE else MomentNdTerms(self)
        _tick("state + node buffers")
        if self.eps != 0.0:
            # noisy path: the two orientations of M, its diagonal, the gradient tiles handed to the fold, and zero
            # factors / rho for that fold (its own product and degree terms are already inside the gradient tiles)
            self.Lt, self.Ut, self.Gn = (torch.zeros(nel, **f32) for _ in range(3))
            self.mdiag = z(n)
            self.Wt0, self.rho0 = z(128, self.npad), z(n)
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

    def _dense_tiles(self, dense, symmetrize, row0=0):
        """Tiles of this rank's tile rows of a dense n x n matrix (`row0`: first row of a band), all-reduced diagonal."""
        tiles = torch.zeros(max(self.ntiles, 1) * TILE * TILE, dtype=torch.float32, device=self.dev)
        diag = torch.zeros(self.n, dtype=torch.float32, device=self.dev)
        call("mcgra_dense_to_tiles", dense.data_ptr() - row0 * self.n * 4, self.n, self.n, self.tr0, self.tr1, symmetrize,
             ptr(tiles), ptr(diag), N.stream_ptr())
        self._allreduce(diag)
        return tiles, diag

    def _full_rows(self, fa, row0, banded, cols=None):
        """Columns [0, cols) of all n rows of feature_adj (None: c1 off).  Full input: a view of `fa`.  Row bands (`fa`:
        rows [row0, ...) of disjoint bands that cover [0, n)): placed in a zero-filled buffer summed across the ranks,
        which is exact because every entry has exactly one non-zero contributor."""
        if fa is None or not banded:
            return fa if fa is None else fa[:, :cols]
        cols = self.n if cols is None else cols
        full = torch.zeros(self.n, cols, dtype=torch.float32, device=self.dev)
        full[row0:row0 + fa.shape[0]] = fa[:, :cols]
        self._allreduce(full)
        return full

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
        a.Fdiag = ptr(self.nn.Fdiag)
        a.acc = self._acc_row(t).data_ptr()
        a.measure = self.measure                      # n x d terms c9 / c10 (node kernel handles MSE / KL)
        a.measure_nn = self.nn.measure                # n x n terms: diagonal part in node_rho
        a.weight_sup = self.weight_sup
        a.k1, a.k2, a.k6, a.k7 = self.nn.k1, self.k2, self.k6, self.k7
        a.w9, a.w10 = (0.0, 0.0) if self.nd is not None else (self.w9, self.w10)
        a.npad = self.npad
        a.d_next, a.d_fill = ptr(self.d_next), (1.0 if self.rank == 0 else 0.0)
        a.acc_next = self._acc_row(t + 1).data_ptr()
        a.minmax = ptr(self.minmax)
        a.lseA, a.lseF, a.dlse = ptr(self.nn.lseA), ptr(self.nn.lseF), ptr(self.nn.dlse)
        a.em = ptr(self.em)
        return a

    def forward_stages(self, t, noisy=False):
        """Forward half of an iteration (through node_head) on the noise-free operator, or on the noisy one (`noisy`: the
        noise stage of iteration t has run; its terms pass carries c1 / c6); returns the node-args struct."""
        st = N.stream_ptr()
        n, tr0, tr1, mu, raw = self.n, self.tr0, self.tr1, ptr(self.mu), self.raw
        a = self._node_args(t)
        ap = C.byref(a)
        call("mcgra_node_pre", ap, st)
        nn = self.nn
        elem = nn.measure in (N.M_MSE, N.M_KL)       # c1 evaluated element-wise
        if elem:
            nn.step(self, t, noisy)
        if not noisy and (elem or self.k6 != 0.0):
            e = N.ElemArgs()
            e.r, e.lseA, e.lseF, e.dlse = ptr(self.r), ptr(nn.lseA), ptr(nn.lseF), ptr(nn.dlse)
            e.Ftiles, e.measure, e.k1 = (ptr(nn.Ftiles), nn.measure, nn.k1) if elem else (None, N.M_NONE, 0.0)
            e.k6, e.acc, e.eps_row = self.k6, self._acc_row(t).data_ptr(), ptr(self.eps_row)
            call("mcgra_elem_stats", ptr(self.xt), n, tr0, tr1, mu, raw, C.byref(e), st, tag="elem_stats")
        self._product(self.B1, 32, self.Y1, False, noisy)
        call("mcgra_node_mid", ap, st)
        self._product(self.B2, 32, self.Y2, False, noisy)
        call("mcgra_node_head", ap, st)
        return a

    def _product(self, B, K, Y, transpose, noisy, reduce=None):
        """Y += A_hat B, or A_hat^T B (`transpose`), for the n x K operand B.  Noise-free: one pass over the symmetric x'.
        Noisy: the two orientation planes of M, then the diagonal (mcgra.h).  With world > 1 the shards' products are
        all-reduced (`reduce`: a buffer that holds Y, default Y itself) before the diagonal is added, once, on every rank."""
        st, n = N.stream_ptr(), self.n
        if noisy:
            first, second = (self.Ut, self.Lt) if transpose else (self.Lt, self.Ut)
            for plane, sel in ((first, N.PROD_DIRECT), (second, N.PROD_MIRRORED)):
                call("mcgra_propagate_sel", ptr(plane), n, self.tr0, self.tr1, None, 2, ptr(B), K, ptr(Y),
                     ptr(self.prop_ws), sel, st, tag=f"propagate{K}_sel")
        else:
            call("mcgra_propagate", ptr(self.xt), n, self.tr0, self.tr1, ptr(self.mu), self.raw, ptr(B), K, ptr(Y),
                 ptr(self.prop_ws), st, tag=f"propagate{K}")
        self._allreduce(Y if reduce is None else reduce)
        if noisy:
            call("mcgra_diag_axpy", ptr(self.mdiag), ptr(B), K, n, ptr(Y), st)

    def iterate(self):
        """One full PGD iteration (forward, backward, Adam, projection): the stage list of the module docstring, with its
        noisy variants when eps != 0.  No host synchronisation.  With world > 1 the n x K products, dzhat, and the fold's
        sums and bracket are all-reduced; under noise also d and the draw's fingerprint (DESIGN.md 3.7)."""
        t = self.step
        if t >= self.max_epochs:
            raise RuntimeError("acc history exhausted; construct the engine with a larger max_epochs")
        st = N.stream_ptr()
        n, tr0, tr1, mu, raw = self.n, self.tr0, self.tr1, ptr(self.mu), self.raw
        noisy = self.eps != 0.0
        noise = self._noise_stage(t) if noisy else None
        a = self.forward_stages(t, noisy)
        ap = C.byref(a)
        nn = self.nn
        pre = nn.measure == N.M_PRE          # gradient tiles handed over by the measure's own stage
        if pre:
            nn.step(self, t, noisy)
        if self.nd is not None:
            self.nd.step(self, t)
        # under noise c7 and the M1 side of KDE's c2 are functions of the symmetric decode M1 only: no A_hat tiles exist
        # (Ftiles = None), the noisy kernels form A_hat's part of eps_row themselves
        EAt, Ct = (nn.Ftiles, nn.Ct) if pre else (None, None)
        k2 = 0.0 if noisy else self.k2
        pairs = self.k7 != 0.0 or k2 != 0.0 or EAt is not None or Ct is not None
        if pairs:
            call("mcgra_pairs", ptr(self.xt), n, tr0, tr1, mu, raw, ptr(self.zhat), ptr(self.r), self.k7, k2, ptr(EAt),
                 ptr(Ct), ptr(self.dzhat), ptr(self.eps_row), self._acc_row(t).data_ptr(), ptr(self.pairs_ws), st)
            if self.k7 != 0.0 and k2 == 0.0 and EAt is None and Ct is None:
                N.LAUNCHES["kernels"] += 2      # tcgen05 engine: operand prep (2 kernels) + k_pairs_tc
        if noisy:
            na = N.NoisyArgs()
            na.n, na.npad, na.tr0, na.tr1 = n, self.npad, tr0, tr1
            na.tiles, na.mu, na.raw, na.noise, na.eps = ptr(self.xt), mu, raw, ptr(noise), self.eps
            na.Lt, na.Ut, na.FLt, na.FUt = ptr(self.Lt), ptr(self.Ut), ptr(nn.FLt), ptr(nn.FUt)
            na.zhat, na.r, na.rho, na.Wt = ptr(self.zhat), ptr(self.r), ptr(self.rho), ptr(self.Wt)
            na.k1, na.k2, na.k6 = nn.k1, self.k2, self.k6
            na.acc, na.eps_row, na.dzhat, na.Gt = self._acc_row(t).data_ptr(), ptr(self.eps_row), ptr(self.dzhat), ptr(self.Gn)
            na.gslab, na.nb = ptr(nn.gslab), nn.nb
            nap = C.byref(na)
            call("mcgra_noisy_terms", nap, st)
        if pairs or noisy:
            self._allreduce(self.dzhat)
        call("mcgra_node_bwd2", ap, st)
        self._product(self.B3, 32, self.Y3, True, noisy)
        call("mcgra_node_bwd1", ap, st)
        self._product(self.B4, 16, self.Y4, True, noisy, reduce=self.Y4e)      # Y4 and eps_row in one collective
        if noisy:
            call("mcgra_node_rho_diag", ap, ptr(self.mdiag), st)
            call("mcgra_noisy_grad", nap, st)
        else:
            call("mcgra_node_rho", ap, st)
            if self.smooth is not None and self.smooth_on:
                self._smooth_stage(t)
        self._fold(t, noisy)
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
        if not noisy:      # (under noise the degree of the next iteration comes from its own noise stage)
            self._allreduce(self.d_next)
            self.d, self.d_next = self.d_next, self.d
            if self.ring_mode:       # hist[step_dev] = finished row; step_dev += 1
                call("mcgra_history_push", self._acc_row(t).data_ptr(), ptr(self.acc_hist), self.acc_hist.shape[0],
                     ptr(self.step_dev), st)
        self.step = t + 1

    def _fold(self, t, noisy):
        """Adam step, clamp and the next iteration's sums (mcgra_fold_adam).  Under noise the product and degree terms
        are already inside the gradient tiles Gn: zero factors and rho, no n x n term."""
        f = N.FoldArgs()
        f.n, f.npad, f.r = self.n, self.npad, ptr(self.r)
        f.norm_coef = self.weight_sup * 0.001
        f.lr, f.beta1, f.beta2, f.adam_eps = self.lr, 0.9, 0.999, 1e-8
        f.step = t + 1
        f.acc_prev = self._acc_row(t).data_ptr()
        f.acc_next = self._acc_row(t + 1).data_ptr()
        f.d_next = ptr(self.d_next)
        f.store_clamped = 0 if self.proj_possible else 1
        f.Wk = ptr(self.fold_ws)
        if noisy:
            f.Wt, f.rho = ptr(self.Wt0), ptr(self.rho0)
            f.measure = N.M_NONE
            f.Gtiles = ptr(self.Gn)
        else:
            f.Wt, f.rho = ptr(self.Wt), ptr(self.rho)
            f.Ftiles, f.measure = ptr(self.nn.Ftiles), self.nn.measure
            f.lseA, f.lseF = ptr(self.nn.lseA), ptr(self.nn.lseF)
            f.zhat = ptr(self.zhat)
            f.k1, f.k6, f.k2 = self.nn.k1, self.k6, self.k2
            f.step_ptr = ptr(self.step_dev) if self.ring_mode else None
            f.plain_gd = 1 if self.plain_gd else 0
            f.Gtiles = ptr(self.Gt) if (self.smooth is not None and self.smooth_on) else None
        call("mcgra_fold_adam", ptr(self.xt), ptr(self.mt), ptr(self.vt), self.tr0, self.tr1, ptr(self.mu), self.raw,
             C.byref(f), ptr(self.minmax), N.stream_ptr())

    def _noise_stage(self, t):
        """Draw iteration t's noise and form M's two orientation planes, its diagonal and the degree d; returns the draw.
        With world > 1 the draw is fingerprinted and d is all-reduced before the diagonal is added, once."""
        st, n = N.stream_ptr(), self.n
        noise = self._noise_fn(t)
        if tuple(noise.shape) != (n, n):
            raise ValueError(f"noise draw of shape {tuple(noise.shape)}, expected ({n}, {n})")
        noise = noise.to(device=self.dev, dtype=torch.float32).contiguous()
        args = (ptr(self.xt), n, self.tr0, self.tr1, ptr(self.mu), self.raw, ptr(noise), self.eps, ptr(self.Lt), ptr(self.Ut))
        if self.world == 1:
            call("mcgra_noise_stage", *args, ptr(self.mdiag), ptr(self.d), st)
        else:
            self._record_noise(noise, t)
            self.d.zero_()
            call("mcgra_noise_tiles", *args, ptr(self.d), st)
            self._allreduce(self.d)
            call("mcgra_noise_diag", n, ptr(noise), self.eps, ptr(self.mdiag), ptr(self.d), st)
        return noise

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
        Gfeat, gdiag = self._dense_tiles(G, 1)
        del G
        self.Gt = torch.zeros(max(self.ntiles, 1) * TILE * TILE, **f32)
        self.smooth = dict(Gfeat=Gfeat, gdiag=gdiag, rt=torch.zeros(n, **f32), trow=torch.zeros(n, **f32), coef=float(coef))

    def _smooth_stage(self, t):
        sm, st = self.smooth, N.stream_ptr()
        call("mcgra_smooth", ptr(self.xt), ptr(sm["Gfeat"]), ptr(sm["gdiag"]), self.n, self.tr0, self.tr1, ptr(self.mu),
             self.raw, ptr(self.d), sm["coef"], ptr(sm["rt"]), ptr(sm["trow"]), ptr(self.Gt), st)
        self._allreduce(sm["trow"])
        call("mcgra_smooth_node", self.n, ptr(self.d), ptr(sm["rt"]), ptr(sm["trow"]), ptr(sm["gdiag"]), sm["coef"],
             ptr(self.rho), self._acc_row(t).data_ptr() + 8 * ACC["C1D"], st)

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
