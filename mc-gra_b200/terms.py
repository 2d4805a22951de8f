"""PGDEngine's per-measure terms (DESIGN.md 1).  No object keeps a reference to the engine or to the full feature_adj."""
import ctypes as C

import torch

from . import _native as N
from ._native import ACC, HID, TILE, call, ptr

KDE_NB = 8      # columns of an n x n operand that reach utils.MutualInformation's kernel (bin_j ~ j, values in [0, 1]; csrc/kde.cu)


class NNTerms:
    """No n x n terms; the fields are what every n x n terms object hands the kernels."""
    measure = N.M_NONE
    Ftiles = Fdiag = Ct = None
    k1 = 0.0
    lseA = lseF = dlse = None
    FLt = FUt = None
    gslab, nb = None, 0

    def step(self, eng, t, noisy):
        pass

    def _gradient_tiles(self, eng, c2):
        """Gradient tiles (MCGRA_M_PRE); under noise A_hat's gradient is a slab and M1's tiles exist only with c2."""
        from .engine import tile_buffer      # (engine imports this module)
        noisy = eng.eps != 0.0
        self.measure = N.M_PRE
        self.Ftiles = None if noisy else tile_buffer(eng.tr0, eng.tr1, eng.dev)
        self.Ct = tile_buffer(eng.tr0, eng.tr1, eng.dev) if (not noisy or c2) else None
        self.Fdiag = torch.zeros(eng.n, dtype=torch.float32, device=eng.dev)     # dL/dA_ii


def feature_lse(eng, fa, row0=0, banded=False):
    """fp64 log sum_j exp(F_ij) of every row of feature_adj (`banded`: `fa` holds rows [row0, ...), all-reduced)."""
    lse = torch.logsumexp(fa.double(), dim=1)
    if banded:
        lse, band = torch.zeros(eng.n, dtype=torch.float64, device=eng.dev), lse
        lse[row0:row0 + fa.shape[0]] = band
        eng._allreduce(lse)
    return lse


class ElementwiseTerms(NNTerms):
    """c1 under MSELoss or KL with c2 off (topology_attack.py:212-229), evaluated element-wise from the tiles of
    feature_adj.  `fa` holds rows [row0, ...) of feature_adj (`banded`: only this rank's tile rows)."""

    def __init__(self, eng, fa, row0, banded, measure, k1c):
        n, f32 = eng.n, dict(dtype=torch.float32, device=eng.dev)
        self.measure = measure
        if eng.eps == 0.0:
            # (row bands are tiled as they are: the mirrored entries F_ji live on other ranks)
            self.Ftiles, self.Fdiag = eng._dense_tiles(fa, 0 if banded else 1, row0)
        else:
            # the noisy A_hat is not symmetric: F and F^T are tiled as they are (on the diagonal F equals its
            # symmetrisation).  F^T is formed for this rank's rows alone (columns [r0, r1) of F), pointer shifted
            from .engine import tile_buffer
            self.FLt, self.FUt = tile_buffer(eng.tr0, eng.tr1, eng.dev), tile_buffer(eng.tr0, eng.tr1, eng.dev)
            self.Fdiag = torch.zeros(n, **f32)
            r0, r1 = eng.tr0 * TILE, min(n, eng.tr1 * TILE)
            if r1 > r0:
                call("mcgra_dense_to_tiles", ptr(fa), n, n, eng.tr0, eng.tr1, 0, ptr(self.FLt), ptr(self.Fdiag),
                     N.stream_ptr())
                faT = fa[:, r0:r1].t().contiguous()
                call("mcgra_dense_to_tiles", faT.data_ptr() - r0 * n * 4, n, n, eng.tr0, eng.tr1, 0, ptr(self.FUt), None,
                     N.stream_ptr())
            eng._allreduce(self.Fdiag)
        if measure == N.M_MSE:
            self.k1 = k1c / (float(n) * float(n))
        else:
            self.k1 = k1c / float(n)
            self.lseF64 = feature_lse(eng, fa, row0, banded)
            self.lseF = self.lseF64.float().contiguous()
            self.sumexp, self.lseA, self.dlse = (torch.zeros(n, **f32) for _ in range(3))

    def step(self, eng, t, noisy):
        """KL: the row log-sum-exp of A_hat, before elem_stats (the diagonal r_i^2 added here); noise-free only."""
        if noisy or self.measure != N.M_KL:
            return
        self.sumexp.zero_()
        call("mcgra_row_sumexp", ptr(eng.xt), eng.n, eng.tr0, eng.tr1, ptr(eng.mu), eng.raw, ptr(eng.r),
             ptr(self.sumexp), N.stream_ptr())
        eng._allreduce(self.sumexp)
        lseA64 = torch.log(self.sumexp.double() + torch.exp((eng.r * eng.r).double()))
        self.lseA.copy_(lseA64)
        self.dlse.copy_(self.lseF64 - lseA64)


class Kl2Terms(NNTerms):
    """c1 / c2 under --measure KL with c2 on (topology_attack.py:212-229, 483-487): three tile passes (csrc/kl2.cu).
    `fa` holds rows [row0, ...) of feature_adj (`banded`: only this rank's tile rows, tiled as they are)."""

    def __init__(self, eng, fa, row0, banded, k1c, k2c):
        self._gradient_tiles(eng, True)
        self.args = k = N.Kl2Args()
        self.bufs = b = {}
        for name in ("seA", "seM", "lseA", "lseM", "klrow", "c1row"):
            b[name] = torch.zeros(eng.n, dtype=torch.float32, device=eng.dev)
            setattr(k, name, ptr(b[name]))
        if fa is not None:
            b["Ffeat"], b["Fdiag_feat"] = eng._dense_tiles(fa, 0 if banded else 1, row0)
            b["lseF"] = feature_lse(eng, fa, row0, banded).float().contiguous()
            k.Ftiles, k.Fdiag_feat, k.lseF = ptr(b["Ffeat"]), ptr(b["Fdiag_feat"]), ptr(b["lseF"])
        k.tr0, k.tr1, k.n = eng.tr0, eng.tr1, eng.n
        k.EAt, k.Ct = ptr(self.Ftiles), ptr(self.Ct)
        k.k1c, k.k2c = k1c, k2c

    def step(self, eng, t, noisy):
        st, k, b = N.stream_ptr(), self.args, self.bufs
        k.tiles, k.mu, k.raw = ptr(eng.xt), ptr(eng.mu), eng.raw
        k.zhat, k.r = ptr(eng.zhat), ptr(eng.r)
        kp = C.byref(k)
        for name in ("seA", "seM", "klrow", "c1row"):
            b[name].zero_()
        call("mcgra_kl2_pass", 0, kp, st)
        eng._allreduce(b["seA"])
        eng._allreduce(b["seM"])
        call("mcgra_kl2_node", 0, kp, None, None, st)
        call("mcgra_kl2_pass", 1, kp, st)
        eng._allreduce(b["klrow"])
        eng._allreduce(b["c1row"])
        call("mcgra_kl2_node", 1, kp, ptr(self.Fdiag), eng._acc_row(t).data_ptr(), st)
        call("mcgra_kl2_pass", 2, kp, st)


def _kde_mi(n, X, dx, Y, dy, w, m, weight, slot, mom, gmom, gX, gY):
    """weight * MutualInformation(X, Y) of kernel-value matrices and its gradient w.r.t. them (gX / gY may be None)."""
    st = N.stream_ptr()
    mom.zero_()
    call("mcgra_cross_moments", ptr(X), dx, ptr(Y), dy, ptr(w), n, ptr(mom), st)
    call("mcgra_kde_scalars", ptr(mom), dx, m, weight, slot, ptr(gmom), st)
    call("mcgra_cross_moments_bwd", ptr(X), dx, ptr(Y), dy, ptr(w), n, ptr(gmom), ptr(gX), ptr(gY), st)


class KdeTerms(NNTerms):
    """c1 / c2 under --measure KDE (utils.py:980-1053): only the first KDE_NB columns of A_hat / M1 / feature_adj reach
    the Gaussian bins, so the joint pdf is an NB x NB weighted second moment.  `fa` holds rows [row0, ...) of
    feature_adj (`banded`: only this rank's tile rows); `fmax`: the maximum of all of feature_adj."""

    def __init__(self, eng, fa, row0, banded, fmax, k1c, k2c):
        n, f32 = eng.n, dict(dtype=torch.float32, device=eng.dev)
        self._gradient_tiles(eng, k2c != 0.0)
        self.nb = nb = min(KDE_NB, n)
        hi = max(float(fmax), 1.0) if fa is not None else 1.0
        if hi > 3.0:      # column j >= KDE_NB would no longer underflow: exp(-0.5 ((v - j) / 0.32)^2) > fp32 min
            raise NotImplementedError("KDE: feature_adj values above 3 reach bins beyond the kept columns")
        self.c1, self.c2 = fa is not None, k2c != 0.0
        self.k1c, self.k2c, self.bin = k1c, k2c, float(n) / float(n - 1)
        self.w = torch.full((n,), 1.0 / n, **f32)
        self.slabA, self.slabM, self.kvA, self.kvM, self.gkvA, self.gkvM, self.gA, self.gM = (
            torch.zeros(n, nb, **f32) for _ in range(8))
        self.mom, self.gmom = (torch.zeros(2 * nb + 2 * nb * nb, dtype=torch.float64, device=eng.dev) for _ in range(2))
        self.gslab = self.gA
        slabF = eng._full_rows(fa, row0, banded, nb).contiguous() if self.c1 else None      # F[:, :NB]
        if self.c1 and eng.eps != 0.0:     # the noisy path's fp64 stage forms kernel values itself
            self.slabF = slabF
        elif self.c1:
            self.kvF = torch.zeros(n, nb, **f32)
            call("mcgra_kde_kv", ptr(slabF), nb, nb, n, self.bin, ptr(self.kvF), N.stream_ptr())

    def step(self, eng, t, noisy):
        """Under noise each MI is ~1e-6 of the entropies it is the difference of: kernel values and moments are formed
        in fp64 from the value slabs, and A_hat's gradient stays the slab gA (gslab of the noisy kernels)."""
        st, n, nb, bin_ = N.stream_ptr(), eng.n, self.nb, self.bin
        acc = eng._acc_row(t).data_ptr()
        self.slabA.zero_()
        if not noisy:
            call("mcgra_slab_ahat", ptr(eng.xt), n, eng.tr0, eng.tr1, ptr(eng.mu), eng.raw, ptr(eng.r), nb,
                 ptr(self.slabA), st)
            eng._allreduce(self.slabA)
            call("mcgra_kde_kv", ptr(self.slabA), nb, nb, n, bin_, ptr(self.kvA), st)
            if self.c1:
                _kde_mi(n, self.kvF, nb, self.kvA, nb, self.w, float(n), self.k1c, acc + 8 * ACC["C1D"], self.mom,
                        self.gmom, None, self.gkvA)
                call("mcgra_kde_chain", ptr(self.slabA), nb, ptr(self.kvA), ptr(self.gkvA), nb, n, bin_, ptr(self.gA), 0,
                     st)
            if self.c2:
                call("mcgra_slab_m1", ptr(eng.zhat), n, nb, ptr(self.slabM), st)
                call("mcgra_kde_kv", ptr(self.slabM), nb, nb, n, bin_, ptr(self.kvM), st)
                _kde_mi(n, self.kvA, nb, self.kvM, nb, self.w, float(n), self.k2c, acc + 8 * ACC["C2D"], self.mom,
                        self.gmom, self.gkvA, self.gkvM)
                call("mcgra_kde_chain", ptr(self.slabA), nb, ptr(self.kvA), ptr(self.gkvA), nb, n, bin_, ptr(self.gA),
                     1 if self.c1 else 0, st)
                call("mcgra_kde_chain", ptr(self.slabM), nb, ptr(self.kvM), ptr(self.gkvM), nb, n, bin_, ptr(self.gM), 0,
                     st)
        else:
            call("mcgra_slab_ahat_noisy", ptr(eng.Lt), ptr(eng.Ut), ptr(eng.mdiag), n, eng.tr0, eng.tr1, ptr(eng.r), nb,
                 ptr(self.slabA), st)
            self.gA.zero_()
            pairs = [(self.slabF, self.slabA, self.k1c, ACC["C1D"], None, self.gA)] if self.c1 else []
            if self.c2:
                call("mcgra_slab_m1", ptr(eng.zhat), n, nb, ptr(self.slabM), st)
                self.gM.zero_()
                pairs.append((self.slabA, self.slabM, self.k2c, ACC["C2D"], self.gA, self.gM))
            for X, Y, weight, slot, gX, gY in pairs:
                self.mom.zero_()
                call("mcgra_kde_moments64", ptr(X), ptr(Y), nb, n, bin_, 1.0 / n, ptr(self.mom), st)
                call("mcgra_kde_scalars", ptr(self.mom), nb, float(n), weight, acc + 8 * slot, ptr(self.gmom), st)
                call("mcgra_kde_chain64", ptr(X), ptr(Y), nb, n, bin_, 1.0 / n, ptr(self.gmom), ptr(gX), ptr(gY), st)
        if self.c2:
            call("mcgra_slab_to_tiles", ptr(self.gM), n, eng.tr0, eng.tr1, nb, ptr(self.Ct), None, st)
        if not noisy:
            call("mcgra_slab_to_tiles", ptr(self.gA), n, eng.tr0, eng.tr1, nb, ptr(self.Ftiles), None, st)
        self.Fdiag.zero_()
        self.Fdiag[:nb].copy_(self.gA[:nb, :nb].diagonal())


class KdeNdTerms:
    """c9 / c10 under --measure KDE (topology_attack.py:246-269): bins = 16 / nclass; gradient added to demd."""

    def __init__(self, eng):
        n, c = eng.n, eng.nclass
        md = max(HID, c)
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=eng.dev)
        self.kvE, self.gkv, self.gV, self.p2 = z(n, md), z(n, md), z(n, md), z(n, c)
        self.mom, self.gmom = (torch.zeros(2 * md + 2 * md * md, dtype=torch.float64, device=eng.dev) for _ in range(2))
        self.m = float(eng.idx.numel())
        if eng.w9 != 0.0:        # bins = linspace(0, 16, 16) (topology_attack.py:246-248)
            self.kvH = z(n, HID)
            call("mcgra_kde_kv", ptr(eng.HA), HID, HID, n, HID / (HID - 1.0), ptr(self.kvH), N.stream_ptr())
        if eng.w10 != 0.0:       # bins = linspace(0, c, c) (:261-263)
            self.kvY = z(n, c)
            self.binc = c / (c - 1.0) if c > 1 else 0.0
            call("mcgra_kde_kv", ptr(eng.YA), c, c, n, self.binc, ptr(self.kvY), N.stream_ptr())

    def _mi_grad(self, eng, X, d, bin_, kvT, weight, slot):
        """weight * MI(kvT, kernel values of X [n x d]); returns its gradient w.r.t. X."""
        n, st = eng.n, N.stream_ptr()
        kv, gkv, gV = (x.view(-1)[: n * d].view(n, d) for x in (self.kvE, self.gkv, self.gV))
        call("mcgra_kde_kv", ptr(X), d, d, n, bin_, ptr(kv), st)
        _kde_mi(n, kvT, d, kv, d, eng.wmult, self.m, weight, slot, self.mom, self.gmom, None, gkv)
        call("mcgra_kde_chain", ptr(X), d, ptr(kv), ptr(gkv), d, n, bin_, ptr(gV), 0, st)
        return gV

    def step(self, eng, t):
        st, n, c = N.stream_ptr(), eng.n, eng.nclass
        acc = eng._acc_row(t).data_ptr()
        if eng.w9 != 0.0:
            eng.demd.add_(self._mi_grad(eng, eng.em, HID, HID / (HID - 1.0), self.kvH, eng.w9, acc + 8 * ACC["C9"]))
        if eng.w10 != 0.0:
            call("mcgra_softmax_rows", ptr(eng.em), ptr(eng.Wl), ptr(eng.bl), n, c, ptr(self.p2), st)
            gV = self._mi_grad(eng, self.p2, c, self.binc, self.kvY, eng.w10, acc + 8 * ACC["C10"])
            call("mcgra_softmax_chain", ptr(gV), ptr(self.p2), ptr(eng.Wl), n, c, ptr(eng.demd), st)


class MomentNdTerms:
    """c9 / c10 under HSIC / CKA / DP: weighted second moments + closed-form gradient into demd (csrc/ndmeasure.cu)."""

    def __init__(self, eng):
        self.p2 = torch.zeros(eng.n, eng.nclass, dtype=torch.float32, device=eng.dev)
        self.mom = torch.zeros(int(N.lib().mcgra_nd_scratch_doubles(eng.nclass)), dtype=torch.float64, device=eng.dev)
        self.coef = torch.zeros(int(N.lib().mcgra_nd_scratch_floats(eng.nclass)), dtype=torch.float32, device=eng.dev)
        self.args = a = N.NdArgs()
        a.n, a.nclass, a.measure = eng.n, eng.nclass, eng.measure
        a.em, a.HA, a.YA, a.Wl, a.bl, a.wmult = (ptr(x) for x in (eng.em, eng.HA, eng.YA, eng.Wl, eng.bl, eng.wmult))
        a.m, a.w9, a.w10 = float(eng.idx.numel()), eng.w9, eng.w10
        a.p2, a.mom, a.coef, a.demd = ptr(self.p2), ptr(self.mom), ptr(self.coef), ptr(eng.demd)

    def step(self, eng, t):
        self.args.acc = eng._acc_row(t).data_ptr()
        call("mcgra_nd_measure", C.byref(self.args), N.stream_ptr())
