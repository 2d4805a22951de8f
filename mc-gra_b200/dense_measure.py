"""c1 / c2 under the HSIC, CKA and DP measures: the n x n x n contractions of the reference
(CudaCKA.linear_HSIC / linear_CKA, utils.py:1060-1091; PGDAttack.dot_product, topology_attack.py:480-481; call sites
topology_attack.py:190-229) as a sequence of native tcgen05 GEMMs (`mcgra_gemm_nt`) with closed-form gradients --
no autograd, no library GEMM.

With A = A_hat and M = M1 (both symmetric), Hc = H (HSIC, CKA) or I (DP), a = A 1, m = M 1:

    c1:  S1  = sum (Kf A) o A,   Kf = Hc F F^T Hc (constant, built once)       d S1 / dA  = 2 Kf A
    c2:  hAM = ||T||_F^2,        T = A Hc M = A M - a (m/n)^T                   d hAM / dA = 2 (Hc M) T^T
                                                                                d hAM / dM = 2 (Hc A) T
    CKA additionally: hAA = ||A Hc A||^2 (d/dA = 4 Hc A S_A), hMM likewise.

    HSIC: c = k S;  DP: c = k sqrt(S);  CKA: c = k S / sqrt(h_xx h_yy)   (scalars on device: mcgra_dense_scalars).

The dense gradients GA = dL/dA_hat and GM = dL/dM1 are handed to the tiled pipeline as tiles of G_ij + G_ji
(`Ftiles`, `Ct`, measure code MCGRA_M_PRE) and the diagonal dL/dA_ii (`Fdiag`): terms.NNTerms.

Multi-GPU: every GEMM is computed by row panels (rank g owns rows [g*rp, (g+1)*rp)) and the panels are all-gathered
(NCCL); the operand images are rebuilt redundantly on every rank from the all-reduced tile triangle (O(n^2)).
"""
import ctypes as C

import torch

from . import _native as N
from ._native import ACC, call, ptr
from .terms import NNTerms

TILE = N.TILE


def _rup(x, m):
    return (x + m - 1) // m * m


class _Img:
    """An fp16x2 operand image (two fp16 planes + row scales) and its C struct."""

    def __init__(self, rows, cols, dev):
        self.rows, self.cols, self.ld = rows, cols, _rup(cols, 64)
        self.hi = torch.zeros(rows, self.ld, dtype=torch.float16, device=dev)
        self.lo = torch.zeros(rows, self.ld, dtype=torch.float16, device=dev)
        self.inv = torch.ones(rows, dtype=torch.float32, device=dev)
        self.c = N.Image(ptr(self.hi), ptr(self.lo), ptr(self.inv), rows, cols, self.ld)

    @property
    def ref(self):
        return C.byref(self.c)


class DenseMeasure(NNTerms):
    def __init__(self, eng, feature_adj, measure, k1c, k2c, sign):
        """eng: PGDEngine (n, dev, rank, world, group, tile rows); feature_adj: dense fp32 device tensor or None (c1
        inactive); k1c / k2c: fully scaled term weights (0 = off); sign: -1 for HSIC (:215-229)."""
        self._gradient_tiles(eng, k2c != 0.0)
        self.n, self.dev, self.rank, self.world, self.group = eng.n, eng.dev, eng.rank, eng.world, eng.group
        self.kind = measure
        self.k1c, self.k2c, self.sign = float(k1c), float(k2c), float(sign)
        self.c1 = feature_adj is not None and k1c != 0.0
        self.c2 = k2c != 0.0
        self.cka = measure == N.M_CKA
        self.cen = 0.0 if measure == N.M_DP else 1.0
        n, dev, world = self.n, self.dev, self.world
        self.ld = _rup(n, 64)
        self.rp = (n + world - 1) // world                  # rows per rank panel
        self.row0 = min(n, eng.rank * self.rp)
        self.row1 = min(n, self.row0 + self.rp)
        rows_alloc = self.rp * world
        f32 = dict(dtype=torch.float32, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        self.GA = torch.zeros(rows_alloc, self.ld, **f32)
        self.ws = torch.zeros(n + 8, dtype=torch.int32, device=dev)
        self.scal = torch.zeros(8, **f64)
        self.alpha = torch.zeros(8, **f32)
        self.rsA, self.rsM = torch.zeros(n, **f64), torch.zeros(n, **f64)
        self.a32, self.abar32, self.m32, self.mbar32 = (torch.zeros(n, **f32) for _ in range(4))
        self.vd = torch.zeros(n, **f64)
        self.v1, self.v2, self.v3, self.v4 = (torch.zeros(n, **f32) for _ in range(4))
        self.hFF = 0.0
        self.imgK = None
        if self.c1:                  # constant kernel image first: its temporaries (F image) are gone before the rest
            self._build_kernel_image(feature_adj)
        self.GM = torch.zeros(rows_alloc, self.ld, **f32) if (self.c2 or self.cka) else None
        self.imgA = _Img(n, n, dev)
        self.imgM = _Img(n, n, dev) if self.c2 else None
        self.imgT = _Img(n, n, dev) if self.c2 else None
        # the image of T^T is built after the last use of M1's image (HSIC / DP), so it can live in the same memory
        self.imgTt = (self.imgM if not self.cka else _Img(n, n, dev)) if self.c2 else None
        self.imgSA = _Img(n, n, dev) if self.cka else None
        self.imgSM = _Img(n, n, dev) if (self.cka and self.c2) else None
        self.tiles_full = None
        if world > 1:
            T = eng.T
            self.tiles_full = torch.zeros((T * (T + 1) // 2) * TILE * TILE, **f32)

    # ------------------------------------------------------------------------------------------------
    def _gemm(self, A, B, Cbuf=None, alpha=1.0, beta=0.0, alpha_dev=None, beta_dev=None, u=None, v=None, coef=0.0,
              sumsq=None, dot=None, dot_with=None, tag="gemm_nt"):
        """C[rows of this rank] = ...; then all-gather the row panels so every rank holds the full C."""
        e = N.GemmEpilogue()
        e.C, e.ldc = (ptr(Cbuf), self.ld) if Cbuf is not None else (None, 0)
        e.alpha, e.beta = float(alpha), float(beta)
        e.alpha_dev, e.beta_dev = alpha_dev, beta_dev
        e.u, e.v, e.coef = ptr(u), ptr(v), float(coef)
        e.sumsq, e.dot = sumsq, dot
        e.dot_with = C.pointer(dot_with.c) if dot_with is not None else None
        e.row0, e.row1 = self.row0, self.row1
        if self.row1 > self.row0:
            call("mcgra_gemm_nt", A.ref, B.ref, C.byref(e), N.stream_ptr(), tag=tag)
        if self.world > 1 and Cbuf is not None:
            import torch.distributed as dist
            panel = Cbuf[self.rank * self.rp:(self.rank + 1) * self.rp]
            dist.all_gather_into_tensor(Cbuf, panel, group=self.group)

    def _image(self, src, img, transpose=0):
        call("mcgra_image_from_dense", ptr(src), self.n, self.n, self.ld, transpose, img.ref, ptr(self.ws), N.stream_ptr())

    def _sptr(self, k):
        return self.scal.data_ptr() + 8 * k

    def _aptr(self, k):
        return self.alpha.data_ptr() + 4 * k

    def _build_kernel_image(self, fa):
        """Kf = Hc F F^T Hc once (F constant): one GEMM + closed-form centring; hFF = ||Kf||_F^2 for CKA."""
        n, st = self.n, N.stream_ptr()
        fa = fa.to(torch.float32).contiguous()
        imgF = _Img(n, n, self.dev)
        call("mcgra_image_from_dense", ptr(fa), n, n, n, 0, imgF.ref, ptr(self.ws), st)
        self._gemm(imgF, imgF, self.GA, tag="gemm_setup")
        del imgF
        if self.cen:
            wsd = torch.zeros(n + 1, dtype=torch.float64, device=self.dev)
            call("mcgra_center_dense", ptr(self.GA), n, self.ld, ptr(wsd), st)
        if self.cka:
            h = torch.zeros(1, dtype=torch.float64, device=self.dev)
            call("mcgra_dense_sumsq", ptr(self.GA), n, n, self.ld, ptr(h), st)
            self.hFF = h
        self.imgK = _Img(n, n, self.dev)
        self._image(self.GA, self.imgK)

    def _full_tiles(self, eng):
        if eng.world == 1:
            return eng.xt
        import torch.distributed as dist
        self.tiles_full.zero_()
        o = (eng.tr0 * (eng.tr0 + 1) // 2) * TILE * TILE
        self.tiles_full[o:o + eng.ntiles * TILE * TILE].copy_(eng.xt[:eng.ntiles * TILE * TILE])
        dist.all_reduce(self.tiles_full, group=eng.group)
        return self.tiles_full

    def _gemv(self, X, w, transpose, out32):
        self.vd.zero_()
        st = N.stream_ptr()
        call("mcgra_dense_gemv", ptr(X), self.n, self.n, self.ld, ptr(w), 1.0 / self.n, transpose, ptr(self.vd), st)
        call("mcgra_d2f", ptr(self.vd), self.n, 1.0, ptr(out32), st)

    # ------------------------------------------------------------------------------------------------
    def step(self, eng, t, noisy):
        """Evaluate c1 / c2 and their gradients at the current parameter; fills Ftiles / Fdiag / Ct."""
        n, st = self.n, N.stream_ptr()
        cen = self.cen
        tiles = self._full_tiles(eng)
        self.scal.zero_()
        self.rsA.zero_()
        call("mcgra_image_ahat", ptr(tiles), n, ptr(eng.mu), eng.raw, ptr(eng.r), self.imgA.ref, ptr(self.rsA), st)
        call("mcgra_d2f", ptr(self.rsA), n, 1.0, ptr(self.a32), st)
        call("mcgra_d2f", ptr(self.rsA), n, 1.0 / n, ptr(self.abar32), st)
        if self.imgM is not None:
            self.rsM.zero_()
            call("mcgra_image_m1", ptr(eng.zhat), n, self.imgM.ref, ptr(self.rsM), st)
            call("mcgra_d2f", ptr(self.rsM), n, 1.0, ptr(self.m32), st)
            call("mcgra_d2f", ptr(self.rsM), n, 1.0 / n, ptr(self.mbar32), st)
        rank1 = dict(coef=cen) if cen else {}

        # ---- values ----
        if self.c1:       # G1 = Kf A, S1 = sum G1 o A
            self._gemm(self.imgK, self.imgA, self.GA, dot=self._sptr(0), dot_with=self.imgA, tag="gemm_c1")
        if self.cka:      # S_A = A Hc A
            self._gemm(self.imgA, self.imgA, self.GM, u=self.a32, v=self.abar32 if cen else None, sumsq=self._sptr(2),
                       tag="gemm_self", **rank1)
            self._image(self.GM, self.imgSA)
            self._gemv(self.GM, self.rsA, 0, self.v3)            # abar^T S_A
        if self.c2:       # T = A Hc M
            self._gemm(self.imgA, self.imgM, self.GM, u=self.a32, v=self.mbar32 if cen else None, sumsq=self._sptr(1),
                       tag="gemm_c2_T", **rank1)
            self._image(self.GM, self.imgT)
            if self.cka:
                self._image(self.GM, self.imgTt, transpose=1)
            self._gemv(self.GM, self.rsM, 1, self.v1)            # T mbar
            self._gemv(self.GM, self.rsA, 0, self.v2)            # abar^T T
            if self.cka:  # S_M = M Hc M
                self._gemm(self.imgM, self.imgM, self.GM, u=self.m32, v=self.mbar32 if cen else None,
                           sumsq=self._sptr(3), tag="gemm_self", **rank1)
                self._image(self.GM, self.imgSM)
                self._gemv(self.GM, self.rsM, 0, self.v4)        # mbar^T S_M
        if eng.world > 1:
            import torch.distributed as dist
            dist.all_reduce(self.scal[:4], group=eng.group)
        if self.cka and self.c1:
            self.scal[4:5].copy_(self.hFF)
        call("mcgra_dense_scalars", self.kind, ptr(self.scal), self.k1c if self.c1 else 0.0, self.k2c, self.sign,
             eng._acc_row(t).data_ptr(), ptr(self.alpha), st)

        # ---- gradients: GA = dL/dA_hat, GM = dL/dM1 ----
        ga = "raw" if self.c1 else "empty"                       # GA holds G1 unscaled / nothing

        def acc_into_ga(A, B, k, v):
            nonlocal ga
            beta, beta_dev = (0.0, None) if ga == "empty" else ((1.0, self._aptr(0)) if ga == "raw" else (1.0, None))
            self._gemm(A, B, self.GA, alpha=1.0, alpha_dev=self._aptr(k), beta=beta, beta_dev=beta_dev,
                       v=v if cen else None, coef=cen, tag="gemm_grad")
            ga = "scaled"

        if self.c2:
            acc_into_ga(self.imgM, self.imgT, 1, self.v1)        # (Hc M) T^T
        if self.cka:
            acc_into_ga(self.imgA, self.imgSA, 2, self.v3)       # (Hc A) S_A
        gm = False
        if self.c2:
            if not self.cka:         # M1's image is dead now: T^T takes its place (T is still in the GM buffer)
                self._image(self.GM, self.imgTt, transpose=1)
            self._gemm(self.imgA, self.imgTt, self.GM, alpha=1.0, alpha_dev=self._aptr(3), v=self.v2 if cen else None,
                       coef=cen, tag="gemm_grad")                # (Hc A) T
            gm = True
            if self.cka:
                self._gemm(self.imgM, self.imgSM, self.GM, alpha=1.0, alpha_dev=self._aptr(4), beta=1.0,
                           v=self.v4 if cen else None, coef=cen, tag="gemm_grad")
        call("mcgra_sym_to_tiles", ptr(self.GA), self.ld, n, eng.tr0, eng.tr1, 1.0,
             self._aptr(0) if ga == "raw" else None, ptr(self.Ftiles), ptr(self.Fdiag), st)
        if gm:
            call("mcgra_sym_to_tiles", ptr(self.GM), self.ld, n, eng.tr0, eng.tr1, 1.0, None, ptr(self.Ct), None, st)


def cross_frobenius(X, Y, center):
    """|| Xc^T Yc ||_F^2 (center=True: linear_HSIC, utils.py:1080-1084) or || Y^T X ||_F^2 (center=False: dot_product,
    topology_attack.py:480-481) of two m-row operands, on the device.  Narrow operands: weighted second moments
    (mcgra_cross_moments); wide ones: one tcgen05 contraction X^T Y on transposed operand images with the centring as a
    rank-1 correction and the Frobenius norm as the fused epilogue reduction."""
    X = X.detach().to(torch.float32).contiguous()
    Y = Y.detach().to(torch.float32).contiguous()
    if not X.is_cuda:
        raise N.NativeError("needs CUDA tensors (no CPU fallback)")
    m, dx, dy = X.shape[0], X.shape[1], Y.shape[1]
    dev, st = X.device, N.stream_ptr()
    if dx <= 64 and dy <= 64:
        out = torch.zeros(dx + dy + dx * dy + dy * dy, dtype=torch.float64, device=dev)
        call("mcgra_cross_moments", ptr(X), dx, ptr(Y), dy, None, m, ptr(out), st)
        G = out[dx + dy:dx + dy + dx * dy].view(dx, dy)
        if center:
            G = G - torch.outer(out[:dx], out[dx:dx + dy]) / m
        return (G ** 2).sum()
    ws = torch.zeros(max(m, dx, dy) + 8, dtype=torch.int32, device=dev)
    ix, iy = _Img(dx, m, dev), _Img(dy, m, dev)
    call("mcgra_image_from_dense", ptr(X), m, dx, dx, 1, ix.ref, ptr(ws), st)
    call("mcgra_image_from_dense", ptr(Y), m, dy, dy, 1, iy.ref, ptr(ws), st)
    red = torch.zeros(1, dtype=torch.float64, device=dev)
    e = N.GemmEpilogue()
    e.alpha = 1.0
    e.sumsq = red.data_ptr()
    if center:       # Xc^T Yc = X^T Y - m xbar ybar^T
        u = (X.double().sum(0)).float().contiguous()
        v = (Y.double().mean(0)).float().contiguous()
        e.u, e.v, e.coef = ptr(u), ptr(v), 1.0
    call("mcgra_gemm_nt", ix.ref, iy.ref, C.byref(e), st)
    return red[0]
