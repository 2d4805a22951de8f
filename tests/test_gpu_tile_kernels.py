"""The tiled-triangle kernels of the PGD iteration, one C-ABI call at a time, against fp64 references of their header
contract (include/mcgra.h): layout converters, mcgra_degree, mcgra_propagate_sel, mcgra_elem_stats, mcgra_fold_adam and
the four bisection calls.

Every group runs over the same sizes (n = 2 .. 8321: one tile, exact multiples of 128, 128k + 1 where the last tile
row holds one row, and T = 66 tile rows, where tile rows 64 and 65 cross the H_RUN = 64 run split of k_propagate_h) and
the same tile-row shards (the whole range; a three-way split with unequal tile counts whose calls accumulate into the
same outputs; the single last tile row; an empty shard, which must return 0 and write nothing).

Where the data allow it the comparison is exact: tile values in {0, 1/4, 1/2, 3/4, 1} under every parameter view,
small-integer x power-of-two feature columns (the fp16 hi plane of the tensor-core image is exact and the lo plane 0),
dyadic feature_adj, every sum below 2^24 units.  Then a dropped, duplicated, mirrored-wrong or mis-masked entry fails
whatever n is.  Elsewhere the bounds are derived from the arithmetic; the constants fixed from the first B200 run are
stated next to each test.  The references are fp64 (torch on the same device, so that n = 8321 stays fast).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import engines

pytestmark = pytest.mark.gpu

TILE = 128
SIZES = [2, 127, 128, 129, 255, 256, 257, 1000, 8321]
SPLITS = ["whole", "split3", "last", "empty"]
U = 2.0 ** -24                     # unit roundoff of fp32
# parameter views (include/mcgra.h "PARAMETER VIEW"): (name, raw, mu); the random mu is dyadic so that x' - mu is exact
VIEWS = [("lazy_mu0", 0, 0.0), ("lazy_mu5/16", 0, 0.3125), ("lazy_murand", 0, 181.0 / 512.0), ("raw1", 1, 0.0),
         ("raw2", 2, 0.0)]


# ---------------------------------------------------------------------------------------------------------------------
# helpers: the tiled triangle of the header, tri(I), tile-row shards
# ---------------------------------------------------------------------------------------------------------------------
def tri(I):
    return I * (I + 1) // 2


def shards(kind, T):
    """Tile-row shards [tr0, tr1) of one call sequence over T tile rows."""
    if kind == "whole":
        return [(0, T)]
    if kind == "split3":           # unequal tile counts (a triangle); at T = 66 the last shard holds tile rows 44..65
        cuts = sorted({0, T // 3, (2 * T) // 3, T})
        return list(zip(cuts[:-1], cuts[1:]))
    if kind == "last":
        return [(T - 1, T)]
    if kind == "empty":
        return [(T // 2, T // 2)]
    raise ValueError(kind)


class Tri:
    """Tiled strict lower triangle of an n x n matrix, tile rows [0, T): tile (I, J), J <= I, at storage index
    tri(I) + J, entry (a, b) = element (128 I + a, 128 J + b), valid iff j < i < n."""

    def __init__(self, n, dev):
        self.n, self.dev = n, dev
        self.T = (n + TILE - 1) // TILE
        self.npad = self.T * TILE
        self.nt = tri(self.T)
        I = np.repeat(np.arange(self.T), np.arange(self.T) + 1)
        J = np.concatenate([np.arange(i + 1) for i in range(self.T)])
        self.I = torch.from_numpy(I).to(dev)
        self.J = torch.from_numpy(J).to(dev)
        ar = torch.arange(TILE, device=dev)
        self.gi = (self.I[:, None] * TILE + ar)[:, :, None]            # [nt, 128, 1]
        self.gj = (self.J[:, None] * TILE + ar)[:, None, :]            # [nt, 1, 128]
        self.valid = (self.gj < self.gi) & (self.gi < n)

    def zeros(self, dtype=torch.float32):
        return torch.zeros(self.nt, TILE, TILE, dtype=dtype, device=self.dev)

    def full(self, v, dtype=torch.float32):
        return torch.full((self.nt, TILE, TILE), v, dtype=dtype, device=self.dev)

    def rows_mask(self, shard_list):
        """Tiles of the tile rows covered by the shards."""
        m = torch.zeros(self.nt, dtype=torch.bool, device=self.dev)
        for tr0, tr1 in shard_list:
            m[tri(tr0):tri(tr1)] = True
        return m

    def from_dense(self, D):
        """Dense [n, >= n] -> tiles of its strict lower triangle (same dtype, invalid entries 0)."""
        P = torch.zeros(self.npad, self.npad, dtype=D.dtype, device=self.dev)
        P[:self.n, :self.n] = D[:self.n, :self.n]
        P4 = P.view(self.T, TILE, self.T, TILE).permute(0, 2, 1, 3)
        return torch.where(self.valid, P4[self.I, self.J], torch.zeros((), dtype=D.dtype, device=self.dev))

    def to_dense(self, tiles, sel=None):
        """Tiles -> dense [n, n] strict lower triangle (fp64); sel restricts to a subset of tiles."""
        P = torch.zeros(self.npad, self.npad, dtype=torch.float64, device=self.dev)
        P4 = P.view(self.T, TILE, self.T, TILE).permute(0, 2, 1, 3)
        t = torch.where(self.valid, tiles.double(), torch.zeros((), dtype=torch.float64, device=self.dev))
        if sel is None:
            P4[self.I, self.J] = t
        else:
            P4[self.I[sel], self.J[sel]] = t[sel]
        return P[:self.n, :self.n]

    def node(self, vec):
        """Per-tile views of a node vector [n]: (v_i [nt, 128, 1], v_j [nt, 1, 128]), 0 beyond n."""
        p = torch.zeros(self.npad, dtype=vec.dtype, device=self.dev)
        p[:self.n] = vec
        return p[self.gi], p[self.gj]

    def rowcol(self, row_vals, col_vals, sel):
        """out[i] = sum over the selected tiles of row_vals in row i + col_vals in column i (fp64, [n])."""
        out = torch.zeros(self.npad, dtype=torch.float64, device=self.dev)
        out.index_add_(0, self.gi[sel].reshape(-1), row_vals[sel].double().sum(2).reshape(-1))
        out.index_add_(0, self.gj[sel].reshape(-1), col_vals[sel].double().sum(1).reshape(-1))
        return out[:self.n]

    def block(self, X):
        """Rows of a node matrix [n, K] per tile row: [T, 128, K] (0 beyond n)."""
        P = torch.zeros(self.npad, X.shape[1], dtype=X.dtype, device=self.dev)
        P[:self.n] = X
        return P.view(self.T, TILE, X.shape[1])


def sl(buf, tr0, tr1):
    """The buffer of a shard's tile rows (contiguous part of the whole-range buffer)."""
    return buf[tri(tr0):tri(tr1)]


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def N():
    from mcgra_b200 import _native
    return _native


def P(t):
    return N().ptr(t)


def stream():
    return N().stream_ptr()


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    N().lib()
    return torch.device("cuda:0")


def gen(dev, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    return g


def dyadic_view_tiles(tr, raw, mu, g):
    """Stored x' of a view whose adjacency entries clamp(.) lie in {0, 1/4, 1/2, 3/4, 1}.  u in {-1/2, 0, .., 1, 3/2}
    (the clamp matters): raw 0 stores u + mu, raw 1 stores u, raw 2 stores clamp(u, 0, 1).  Returns (x', adj, param,
    mask) as fp32 tiles with invalid entries 0."""
    k = torch.randint(-2, 7, (tr.nt, TILE, TILE), generator=g, device=tr.dev).float()
    u = k * 0.25
    adj = u.clamp(0.0, 1.0)
    if raw == 0:
        x = u + mu
        param = adj
    elif raw == 1:
        x, param = u, u
    else:
        x, param = adj, adj
    mask = ((u >= 0) & (u <= 1)).float() if raw == 1 else torch.ones_like(u)
    z = torch.zeros((), device=tr.dev)
    return tuple(torch.where(tr.valid, t, z).contiguous() for t in (x, adj, param, mask))


def random_view_tiles(tr, raw, mu, g, lo=-0.25, hi=1.25):
    """Random stored x' and its view, evaluated in fp32 exactly as the kernels do (one subtraction, clamp)."""
    x = torch.rand(tr.nt, TILE, TILE, generator=g, device=tr.dev) * (hi - lo) + lo
    if raw == 2:
        x = x.clamp(0.0, 1.0)
    mu32 = torch.tensor(mu, dtype=torch.float32, device=tr.dev)
    if raw == 0:
        x = x + mu32
        param = (x - mu32).clamp(0.0, 1.0)
        adj = param
    else:
        param = x
        adj = x.clamp(0.0, 1.0)
    mask = ((x >= 0) & (x <= 1)).float() if raw == 1 else torch.ones_like(x)
    z = torch.zeros((), device=tr.dev)
    return tuple(torch.where(tr.valid, t, z).contiguous() for t in (x, adj, param, mask))


def mu_tensor(mu, dev):
    return torch.tensor([mu], dtype=torch.float32, device=dev)


# ---------------------------------------------------------------------------------------------------------------------
# 1. layout
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("split", SPLITS)
@pytest.mark.parametrize("n", SIZES)
def test_layout_exact(dev, n, split):
    tr = Tri(n, dev)
    sh = shards(split, tr.T)
    sel = tr.rows_mask(sh)
    g = gen(dev, 1000 + n)
    st = stream()
    nan = float("nan")
    ld = n + 3
    ri, ci = torch.tril_indices(n, n, -1, device=dev)          # packed order k = i (i - 1) / 2 + j
    prow_cov = torch.zeros(n, dtype=torch.bool, device=dev)          # rows of the shards' tile rows
    for tr0, tr1 in sh:
        prow_cov[tr0 * TILE:min(tr1 * TILE, n)] = True
    pk_cov = prow_cov[ri]

    # tril_to_tiles: NaN-prefilled destination, invalid entries come back +0.0, tile rows outside the shards untouched
    packed = (torch.rand(ri.numel(), generator=g, device=dev) * 2.0 - 0.5).contiguous()
    D = torch.zeros(n, n, device=dev)
    D[ri, ci] = packed
    exp_tiles = tr.from_dense(D)
    tiles = tr.full(nan)
    for tr0, tr1 in sh:
        assert N().lib().mcgra_tril_to_tiles(P(packed), n, tr0, tr1, P(sl(tiles, tr0, tr1)), st) == 0
    torch.cuda.synchronize()
    assert bits_equal(tiles[sel], exp_tiles[sel]), "tril_to_tiles: stored entries or the +0.0 padding differ"
    assert torch.isnan(tiles[~sel]).all(), "tril_to_tiles wrote outside its tile rows"

    for name, raw, mu in VIEWS:
        src = exp_tiles.clone()
        pk = packed.clone()
        if raw == 2:
            src = src.clamp(0.0, 1.0)
            pk = pk.clamp(0.0, 1.0)
        mu32 = torch.tensor(mu, dtype=torch.float32, device=dev)
        want = (pk - mu32).clamp(0.0, 1.0) if raw == 0 else pk
        mud = mu_tensor(mu, dev)
        # tiles_to_tril: round trip under the view
        out = torch.full_like(packed, nan)
        for tr0, tr1 in sh:
            N().call("mcgra_tiles_to_tril", P(sl(src, tr0, tr1)), n, tr0, tr1, P(mud), raw, P(out), st)
        torch.cuda.synchronize()
        assert torch.equal(out[pk_cov], want[pk_cov]), f"tiles_to_tril {name}"
        assert torch.isnan(out[~pk_cov]).all(), f"tiles_to_tril {name} wrote rows outside its shard"
        # tiles_to_dense: the symmetric zero-diagonal expansion of the owned rows and their mirrored columns, ld > n
        dense = torch.full((n, ld), nan, device=dev)
        for tr0, tr1 in sh:
            N().call("mcgra_tiles_to_dense", P(sl(src, tr0, tr1)), n, tr0, tr1, P(mud), raw, P(dense), ld, st)
        torch.cuda.synchronize()
        E = torch.full((n, ld), nan, device=dev)
        own = pk_cov
        E[ri[own], ci[own]] = want[own]
        E[ci[own], ri[own]] = want[own]
        assert bits_equal(dense, E), f"tiles_to_dense {name}: wrong entries, or entries written off the owned rows"

    # dense_to_tiles (plain / symmetrised, diag) and sym_to_tiles (scale, scale_dev): dyadic data, exact; the ld > n
    # padding columns are NaN, so a read through the wrong leading dimension shows
    F = torch.full((n, ld), nan, device=dev)
    F[:, :n] = torch.randint(-128, 129, (n, n), generator=g, device=dev).float() / 64.0
    for symm in (0, 1):
        want = F[:, :n] if not symm else 0.5 * (F[:, :n] + F[:, :n].t())
        exp = tr.from_dense(want)
        tiles = tr.full(nan)
        diag = torch.full((n,), nan, device=dev)
        for tr0, tr1 in sh:
            N().call("mcgra_dense_to_tiles", P(F), ld, n, tr0, tr1, symm, P(sl(tiles, tr0, tr1)), P(diag), st)
        torch.cuda.synchronize()
        assert bits_equal(tiles[sel], exp[sel]), f"dense_to_tiles symmetrize={symm}"
        assert torch.isnan(tiles[~sel]).all()
        dcov = prow_cov[:n]
        assert torch.equal(diag[dcov], torch.diagonal(F[:, :n])[dcov]) and torch.isnan(diag[~dcov]).all()
    for sdev in (None, torch.tensor([4.0], device=dev)):
        sc = 0.5 * (4.0 if sdev is not None else 1.0)
        exp = tr.from_dense((F[:, :n] + F[:, :n].t()) * sc)
        tiles = tr.full(nan)
        diag = torch.full((n,), nan, device=dev)
        for tr0, tr1 in sh:
            N().call("mcgra_sym_to_tiles", P(F), ld, n, tr0, tr1, 0.5, P(sdev), P(sl(tiles, tr0, tr1)), P(diag), st)
        torch.cuda.synchronize()
        assert bits_equal(tiles[sel], exp[sel]), f"sym_to_tiles scale_dev={sdev is not None}"
        assert torch.isnan(tiles[~sel]).all()
        assert torch.equal(diag, torch.diagonal(F[:, :n]) * sc), "sym_to_tiles: diag is written for every node"


# ---------------------------------------------------------------------------------------------------------------------
# 2. degree
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("split", SPLITS)
@pytest.mark.parametrize("n", SIZES)
def test_degree_exact(dev, n, split):
    tr = Tri(n, dev)
    sh = shards(split, tr.T)
    sel = tr.rows_mask(sh)
    g = gen(dev, 2000 + n)
    st = stream()
    for name, raw, mu in VIEWS:
        x, adj, _, _ = dyadic_view_tiles(tr, raw, mu, g)
        d0 = 1.0 + torch.randint(0, 8, (n,), generator=g, device=dev).float() * 0.25
        d = d0.clone()
        for tr0, tr1 in sh:
            assert N().lib().mcgra_degree(P(sl(x, tr0, tr1)), n, tr0, tr1, P(mu_tensor(mu, dev)), raw, P(d), st) == 0
        torch.cuda.synchronize()
        want = d0.double() + tr.rowcol(adj, adj, sel)
        assert torch.equal(d.double(), want), f"degree {name}: max |diff| {(d.double() - want).abs().max():.3e}"


# ---------------------------------------------------------------------------------------------------------------------
# 3. propagation
# ---------------------------------------------------------------------------------------------------------------------
PROP_ENGINES = [("ffma", 0, True), ("tc", 5, True), ("tc_ws_null", 5, False)]   # engine 5 without ws runs the FFMA kernel


def prop_ref(tr, adj, B, sel, products):
    """fp64 sum over the selected tiles: DIRECT adds L B (rows of I), MIRRORED adds L^T B (rows of J)."""
    Bt = tr.block(B.double())
    Y = torch.zeros(tr.npad, B.shape[1], dtype=torch.float64, device=tr.dev)
    A = adj.double()[sel]
    I, J = tr.I[sel], tr.J[sel]
    if products & 1:
        Y.index_add_(0, tr.gi[sel].reshape(-1), torch.bmm(A, Bt[J]).reshape(-1, B.shape[1]))
    if products & 2:
        Y.index_add_(0, tr.gj[sel].reshape(-1), torch.bmm(A.transpose(1, 2), Bt[I]).reshape(-1, B.shape[1]))
    return Y[:tr.n]


def run_prop(tr, x, mu, raw, B, K, Y, sh, products, use_ws):
    st = stream()
    ws = torch.empty(N().lib().mcgra_propagate_ws_bytes(tr.n, K), dtype=torch.uint8, device=tr.dev) if use_ws else None
    for tr0, tr1 in sh:
        N().call("mcgra_propagate_sel", P(sl(x, tr0, tr1)), tr.n, tr0, tr1, P(mu_tensor(mu, tr.dev)), raw, P(B), K,
                 P(Y), P(ws), products, st)


def dyadic_features(n, K, g, dev):
    """Small integers times a per-column power of two: the column-scaled fp16 hi plane is exact, the lo plane 0."""
    k = torch.randint(-8, 9, (n, K), generator=g, device=dev).float()
    return (k * torch.pow(2.0, (torch.arange(K, device=dev) % 5 - 2).float())).contiguous()


@pytest.mark.parametrize("K", [16, 32])
@pytest.mark.parametrize("split", SPLITS)
@pytest.mark.parametrize("n", SIZES)
def test_propagate_exact(dev, n, split, K):
    tr = Tri(n, dev)
    sh = shards(split, tr.T)
    sel = tr.rows_mask(sh)
    g = gen(dev, 3000 + n + K)
    for name, raw, mu in VIEWS:
        x, adj, _, _ = dyadic_view_tiles(tr, raw, mu, g)
        B = dyadic_features(n, K, g, dev)
        Y0 = (torch.randint(-16, 17, (n, K), generator=g, device=dev).float() * 0.25).contiguous()
        refs = {p: prop_ref(tr, adj, B, sel, p) for p in (1, 2)}
        for ename, eng, use_ws in PROP_ENGINES:
            with engines({0: eng}):
                for products in (1, 2, 3):
                    Y = Y0.clone()
                    run_prop(tr, x, mu, raw, B, K, Y, sh, products, use_ws)
                    torch.cuda.synchronize()
                    want = Y0.double() + (refs[1] if products & 1 else 0) + (refs[2] if products & 2 else 0)
                    assert torch.equal(Y.double(), want), \
                        f"{ename} {name} products={products}: max |diff| {(Y.double() - want).abs().max():.3e}"


@pytest.mark.parametrize("split", ["whole", "split3"])
@pytest.mark.parametrize("n", SIZES)
def test_propagate_two_planes(dev, n, split):
    """The noisy path's use: a non-symmetric M kept as Lt (M_ij at (i,j), i > j) and Ut (M_ji at (i,j)), raw = 2:
    DIRECT(Lt) + MIRRORED(Ut) = M B and DIRECT(Ut) + MIRRORED(Lt) = M^T B, against a dense M built independently."""
    tr = Tri(n, dev)
    sh = shards(split, tr.T)
    g = gen(dev, 3500 + n)
    K = 16
    _, Lt, _, _ = dyadic_view_tiles(tr, 2, 0.0, g)
    _, Ut, _, _ = dyadic_view_tiles(tr, 2, 0.0, g)
    M = tr.to_dense(Lt) + tr.to_dense(Ut).t()
    B = dyadic_features(n, K, g, dev)
    for ename, eng, use_ws in PROP_ENGINES:
        with engines({0: eng}):
            for first, second, Mx in ((Lt, Ut, M), (Ut, Lt, M.t())):
                Y = torch.zeros(n, K, device=dev)
                run_prop(tr, first, 0.0, 2, B, K, Y, sh, 1, use_ws)
                run_prop(tr, second, 0.0, 2, B, K, Y, sh, 2, use_ws)
                torch.cuda.synchronize()
                assert torch.equal(Y.double(), Mx @ B.double()), ename


@pytest.mark.parametrize("n", [257, 1000])
def test_propagate_rejects_bad_arguments(dev, n):
    tr = Tri(n, dev)
    x = tr.zeros()
    B = torch.zeros(n, 32, device=dev)
    Y = torch.full((n, 32), 3.0, device=dev)
    ws = torch.empty(N().lib().mcgra_propagate_ws_bytes(n, 32), dtype=torch.uint8, device=dev)
    L = N().lib()
    for _, eng, use_ws in PROP_ENGINES:
        with engines({0: eng}):
            w = P(ws) if use_ws else None
            for products in (0, 4, -1, 7):
                assert L.mcgra_propagate_sel(P(x), n, 0, tr.T, None, 2, P(B), 32, P(Y), w, products, stream()) < 0
            for K in (8, 24, 64):
                assert L.mcgra_propagate_sel(P(x), n, 0, tr.T, None, 2, P(B), K, P(Y), w, 3, stream()) < 0
    torch.cuda.synchronize()
    assert (Y == 3.0).all()


# Precision on random data.  Engine 5 (fp16 x 2 image of tile and column-scaled B, fp32 accumulation in tensor memory):
# |Y - Y64|_ic <= 2^-19 sum_j |M_ij| max_j |B_jc| (DESIGN 3.1: relative to the COLUMN maximum; column 0 has a 2^20
# dynamic range).  Engine 0 (fp32 FFMA, a 128-term chain per tile, one atomic per tile row): <= (128 + T) 2^-24
# sum_j |M_ij B_jc|.  Largest fraction of each bound seen on a B200 (printed as [prop-precision]): engine 5 0.85 (n = 8321,
# the all-positive column: fp32 accumulation over a 32-tile half run in tensor memory), engine 0 0.06.
@pytest.mark.parametrize("split", ["whole", "split3"])
@pytest.mark.parametrize("n", SIZES)
def test_propagate_precision(dev, n, split):
    tr = Tri(n, dev)
    sh = shards(split, tr.T)
    sel = tr.rows_mask(sh)
    g = gen(dev, 4000 + n)
    worst = {}
    for name, raw, mu in (VIEWS[2], VIEWS[3], VIEWS[4]):
        mu_r = float(np.float32(0.123456789)) if raw == 0 else 0.0
        x, adj, _, _ = random_view_tiles(tr, raw, mu_r, g)
        for K in (16, 32):
            B = torch.randn(n, K, generator=g, device=dev)
            B[:, 0] *= torch.pow(2.0, -20.0 * torch.rand(n, generator=g, device=dev))
            B[:, 1] = torch.pow(2.0, -20.0 * torch.rand(n, generator=g, device=dev))
            B = B.contiguous()
            ref = prop_ref(tr, adj, B, sel, 3)
            absref = prop_ref(tr, adj, B.abs(), sel, 3)
            rowM = prop_ref(tr, adj, torch.ones(n, 1, device=dev), sel, 3)
            bound5 = 2.0 ** -19 * rowM * B.abs().max(0).values.double()[None, :]
            bound0 = (128 + tr.T) * U * absref
            for ename, eng, use_ws in PROP_ENGINES:
                with engines({0: eng}):
                    Y = torch.zeros(n, K, device=dev)
                    run_prop(tr, x, mu_r, raw, B, K, Y, sh, 3, use_ws)
                    torch.cuda.synchronize()
                err = (Y.double() - ref).abs()
                bound = bound5 if (eng == 5 and use_ws) else bound0
                frac = float((err / bound.clamp_min(1e-300)).max())
                worst[ename] = max(worst.get(ename, 0.0), frac)
                assert (err <= bound).all(), f"{ename} {name} K={K}: {frac:.3f} of the bound"
    print(f"[prop-precision] n={n} {split}: largest error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


# ---------------------------------------------------------------------------------------------------------------------
# 4. element-wise terms
# ---------------------------------------------------------------------------------------------------------------------
ELEM_ENGINES = [("stats", 0, 0), ("rs_cap5", 1, 5), ("rs", 1, 0)]      # (name, engine, grid cap: 0 = none)
# Bounds (fp32 arithmetic of the kernels against fp64): acc[C1] / acc[C6] within C_VAL 2^-24 S, S the sum of the absolute
# values of the summed parts; eps_row[i] within C_ROW 2^-24 sum_j s_ij M_ij r_j, s_ij the absolute size of the parts of
# e'_ij + e'_ji (MSE: 4|k1|(A + F), KL: |k1|(A_ij + X_ij + A_ji + X_ji)(1 + |lse|), entropy: 2|k6|(|log2 q| + 2)).
# A per-thread fp32 chain covers 64 entries in k_elem_stats: C = 128 covers the chain, the two or three roundings
# of A_hat and the MUFU exp / log2 (2^-22 relative).  Largest fraction seen on a B200 ([elem-precision]): acc[C1] 0.003,
# acc[C6] 0.022, eps_row 0.051, engine 1 vs engine 0 0.024 (of twice the row bound).
C_VAL = 128.0
C_ROW = 128.0


def elem_reference(tr, adj, r, F, measure, k1, k6):
    """fp64: Â (diagonal r_i^2), the off-diagonal term values, e' = dL/dÂ of the full terms by autograd, lse's."""
    n, dev = tr.n, tr.dev
    Ms = tr.to_dense(adj)
    Ms = Ms + Ms.t()
    rd = r.double()
    Ah = (rd[:, None] * Ms * rd[None, :]).fill_diagonal_(0) + torch.diag(rd * rd)
    Ah.requires_grad_(True)
    off = ~torch.eye(n, dtype=torch.bool, device=dev)
    Fd = F.double()
    lseA = torch.logsumexp(Ah, 1)
    lseF = torch.logsumexp(Fd, 1)
    loss = torch.zeros((), dtype=torch.float64, device=dev)
    c1 = torch.zeros((), dtype=torch.float64, device=dev)
    mag1 = torch.zeros((), dtype=torch.float64, device=dev)
    if measure == 1:
        t = (Ah - Fd) ** 2
        loss = loss + k1 * t.sum()
        c1 = k1 * t[off].sum()
        mag1 = abs(k1) * (t[off].sum() + 2 * ((Ah.abs() + Fd.abs()) * (Ah - Fd).abs())[off].sum())
    elif measure == 2:
        X = torch.softmax(Fd, 1)
        lr_ = (Fd - lseF[:, None]) - (Ah - lseA[:, None])
        t = X * lr_
        loss = loss + k1 * t.sum()
        c1 = k1 * t[off].sum()
        mag1 = abs(k1) * (X * (Fd.abs() + Ah.abs() + (lseF - lseA).abs()[:, None]) * (1 + lseF.abs()[:, None]))[off].sum()
    q = Ah.clamp(1e-4, 1 - 1e-4)
    te = q * torch.log2(q)
    c6 = k6 * te[off].sum()
    mag6 = abs(k6) * (te.abs() + q)[off].sum()
    if k6 != 0.0:
        loss = loss + k6 * te[off].sum()
    if loss.requires_grad:
        loss.backward()
    ep = Ah.grad.detach() if Ah.grad is not None else torch.zeros_like(Ah.detach())
    esym = ep + ep.t()
    # absolute size of the parts of e'_ij + e'_ji
    A = Ah.detach()
    s = torch.zeros_like(A)
    if measure == 1:
        s = s + 4 * abs(k1) * (A + Fd.abs())
    elif measure == 2:
        Aso = torch.softmax(A, 1)
        X = torch.softmax(Fd, 1)
        s = s + abs(k1) * ((Aso + X) + (Aso + X).t()) * (1 + lseF.abs().max())
    if k6 != 0.0:
        s = s + 2 * abs(k6) * (torch.log2(q.detach()).abs() + 2)
    return dict(c1=float(c1.detach()), c6=float(c6.detach()), mag1=float(mag1.detach()), mag6=float(mag6.detach()),
                esym=esym, s=s,
                lseA=lseA.detach(), lseF=lseF.detach())


@pytest.mark.parametrize("k6", [0.0, -0.21])
@pytest.mark.parametrize("measure", [0, 1, 2], ids=["none", "mse", "kl"])
@pytest.mark.parametrize("n", SIZES)
def test_elem_stats(dev, n, measure, k6):
    tr = Tri(n, dev)
    g = gen(dev, 5000 + n + 7 * measure)
    k1 = 0.37
    st = stream()
    worst = {"c1": 0.0, "c6": 0.0, "row": 0.0, "eng": 0.0}
    for name, raw, mu in VIEWS:
        mu_r = float(np.float32(0.2718)) if name == "lazy_murand" else mu
        x, adj, _, _ = random_view_tiles(tr, raw, mu_r, g)
        r = (0.05 + 0.55 * torch.rand(n, generator=g, device=dev)).contiguous()
        Fh = torch.rand(n, n, generator=g, device=dev) * (0.3 if measure != 2 else 1.0)
        F = torch.triu(Fh, 1) + torch.triu(Fh, 1).t() + torch.diag(torch.diagonal(Fh))
        Ft = tr.from_dense(F).contiguous()
        ref = elem_reference(tr, adj, r, F, measure, k1, k6)
        lseA = ref["lseA"].float().contiguous()
        lseF = ref["lseF"].float().contiguous()
        dlse = (ref["lseF"] - ref["lseA"]).float().contiguous()
        es_t = tr.from_dense(ref["esym"])
        s_t = tr.from_dense(ref["s"])
        ri, rj = tr.node(r.double())
        out0 = None
        for split in SPLITS:
            sh = shards(split, tr.T)
            sel = tr.rows_mask(sh)
            a = adj.double()
            row_ref = tr.rowcol(es_t * a * rj, es_t * a * ri, sel)
            row_mag = tr.rowcol(s_t * a * rj, s_t * a * ri, sel)
            for ename, eng, cap in ELEM_ENGINES:
                if eng == 1 and not (measure == 1 and raw in (0, 2)):
                    continue                      # engine 1 only takes MSE on the clamped / lazily projected view
                acc = torch.zeros(32, dtype=torch.float64, device=dev)
                eps = torch.zeros(n, device=dev)
                ea = N().ElemArgs(r=P(r), Ftiles=None, lseA=P(lseA), lseF=P(lseF), measure=measure, k1=k1, k6=k6,
                                  acc=P(acc), eps_row=P(eps), dlse=P(dlse))
                with engines({4: eng}, caps={4: cap}):
                    for tr0, tr1 in sh:
                        ea.Ftiles = P(sl(Ft, tr0, tr1))
                        N().call("mcgra_elem_stats", P(sl(x, tr0, tr1)), n, tr0, tr1, P(mu_tensor(mu_r, dev)), raw,
                                 C.byref(ea), st)
                    torch.cuda.synchronize()
                tag = f"{ename} {name} {split}"
                others = torch.ones(32, dtype=torch.bool, device=dev)
                others[[1, 3]] = False
                assert (acc[others] == 0).all(), f"{tag}: slots other than C1 / C6 written"
                if split == "empty":
                    assert (acc == 0).all() and (eps == 0).all(), f"{tag}: the empty shard wrote"
                    continue
                if split == "whole":
                    for slot, key, mag in ((1, "c1", "mag1"), (3, "c6", "mag6")):
                        want = ref[key] if (key == "c6" and k6 != 0.0) or (key == "c1" and measure != 0) else 0.0
                        err = abs(float(acc[slot]) - want)
                        bnd = C_VAL * U * ref[mag] + 1e-300
                        worst[key] = max(worst[key], err / bnd)
                        assert err <= bnd, f"{tag}: acc[{key}] {float(acc[slot])!r} vs {want!r} ({err / bnd:.3f} of the bound)"
                err = (eps.double() - row_ref).abs()
                bnd = C_ROW * U * row_mag
                worst["row"] = max(worst["row"], float((err / bnd.clamp_min(1e-300)).max()))
                assert (err <= bnd).all(), f"{tag}: eps_row {float((err / bnd.clamp_min(1e-300)).max()):.3f} of the bound"
                if split == "whole":
                    if out0 is None:
                        out0 = eps.double()
                    else:
                        e2 = (eps.double() - out0).abs()
                        worst["eng"] = max(worst["eng"], float((e2 / (2 * bnd).clamp_min(1e-300)).max()))
                        assert (e2 <= 2 * bnd).all(), f"{tag}: engine disagreement beyond the rounding bound"
    print(f"[elem-precision] n={n} measure={measure} k6={k6}: largest error / bound " +
          ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


# ---------------------------------------------------------------------------------------------------------------------
# 5. gradient fold + Adam
# ---------------------------------------------------------------------------------------------------------------------
FOLD_ENGINES = [("ffma", 0, 0), ("tc", 2, 0), ("rs_cap1", 3, 1), ("rs_cap5", 3, 5), ("rs", 3, 0)]
# the kernels receive these as fp32: the reference uses the same fp32 values (1 - 0.999f is 1.3e-5 away from 0.001)
BETA1, BETA2, ADAM_EPS, LR = (float(np.float32(v)) for v in (0.9, 0.999, 1e-8, 0.01))
STEP = 5
NORM_COEF, SUMSQ_PREV = float(np.float32(0.0013)), 1234.5
# Configurations (measure, k6, k2, view, store_clamped, Gtiles, plain_gd, step_ptr).  Engine 3 takes the launches with
# the clamped store / the lazily projected view and MSE / PRE / no c1 term; every other one runs on engine 2.
FOLD_CFGS = {
    "mse_clamped": dict(measure=1, raw=2, store_clamped=1),
    "mse_ent_lazy": dict(measure=1, k6=-0.21, raw=0, mu=0.3125),
    "pre_ent_clamped": dict(measure=6, k6=-0.21, raw=2, store_clamped=1),
    "none_lazy": dict(measure=0, raw=0, mu=181.0 / 512.0),
    "none_ent_clamped": dict(measure=0, k6=-0.21, raw=2, store_clamped=1),
    "kl_ent_raw1": dict(measure=2, k6=-0.21, raw=1),
    "mse_k2_lazy": dict(measure=1, k2=0.29, raw=0, mu=0.0),
    "mse_gtiles_clamped": dict(measure=1, raw=2, store_clamped=1, G=True),
    "plain_gd_gtiles_raw1": dict(measure=0, raw=1, G=True, plain_gd=1),
    "mse_step_ptr_lazy": dict(measure=1, raw=0, mu=0.3125, step_ptr=True),
}


def fold_inputs(tr, cfg, g):
    n, dev = tr.n, tr.dev
    raw, mu = cfg["raw"], cfg.get("mu", 0.0)
    # every valid parameter in [0.3, 0.9] (raw 1: also above 1, where the clamp mask is 0): every returned x' > 0.1, so a
    # padding 0 leaking into the minimum shows
    base = 0.3 + 0.6 * torch.rand(tr.nt, TILE, TILE, generator=g, device=dev)
    if raw == 1:
        base = torch.where(torch.rand(base.shape, generator=g, device=dev) < 0.1, base + 0.8, base)
    x = base + torch.tensor(mu, dtype=torch.float32, device=dev) if raw == 0 else base
    z = torch.zeros((), device=dev)
    x = torch.where(tr.valid, x, z).contiguous()
    m = torch.where(tr.valid, 1e-3 * torch.randn(x.shape, generator=g, device=dev), z).contiguous()
    v = torch.where(tr.valid, 1e-6 + 9e-6 * torch.rand(x.shape, generator=g, device=dev), z).contiguous()
    meas = cfg["measure"]
    if meas == 6:
        Ft = 0.05 * torch.randn(x.shape, generator=g, device=dev)
    else:
        Ft = (0.3 if meas == 1 else 1.0) * torch.rand(x.shape, generator=g, device=dev)
    Ft = torch.where(tr.valid, Ft, z).contiguous()
    Gt = torch.where(tr.valid, 0.01 * torch.randn(x.shape, generator=g, device=dev), z).contiguous() \
        if cfg.get("G") else None
    Wt = torch.zeros(128, tr.npad, device=dev)
    Wt[:, :n] = 0.05 * torch.randn(128, n, generator=g, device=dev)
    r = (0.05 + 0.55 * torch.rand(n, generator=g, device=dev)).contiguous()
    rho = (0.01 * torch.randn(n, generator=g, device=dev)).contiguous()
    lse = float(np.log(max(n, 2)))
    lseA = (lse + torch.rand(n, generator=g, device=dev)).contiguous()
    lseF = (lse + torch.rand(n, generator=g, device=dev)).contiguous()
    zhat = (0.3 * torch.randn(n, 16, generator=g, device=dev)).contiguous()
    return dict(x=x, m=m, v=v, Ft=Ft, Gt=Gt, Wt=Wt.contiguous(), r=r, rho=rho, lseA=lseA, lseF=lseF, zhat=zhat)


def fold_reference(tr, cfg, d):
    """fp64 restatement of the header's gradient and torch.optim.Adam's update (or x - lr g) for every tile.  Returns
    x_new, m', v', g, and the absolute size S of the gradient's parts."""
    raw, mu = cfg["raw"], cfg.get("mu", 0.0)
    k1 = 0.37 if cfg["measure"] in (1, 2) else 0.0
    k6, k2 = cfg.get("k6", 0.0), cfg.get("k2", 0.0)
    x = d["x"].double()
    if raw == 0:
        par = (d["x"] - torch.tensor(mu, dtype=torch.float32, device=tr.dev)).clamp(0.0, 1.0).double()
        adj, mask = par, torch.ones_like(x)
    else:
        par, adj = x, x.clamp(0.0, 1.0)
        mask = ((x >= 0) & (x <= 1)).double() if raw == 1 else torch.ones_like(x)
    ri, rj = tr.node(d["r"].double())
    rhoi, rhoj = tr.node(d["rho"].double())
    Wb = d["Wt"].double().t().reshape(tr.T, TILE, 128)                      # [T, 128 nodes, 128 factors]
    Ui, Vi = Wb[tr.I][:, :, :64], Wb[tr.I][:, :, 64:]
    Uj, Vj = Wb[tr.J][:, :, :64], Wb[tr.J][:, :, 64:]
    prod = torch.bmm(Ui, Vj.transpose(1, 2)) + torch.bmm(Vi, Uj.transpose(1, 2))
    prod_abs = torch.bmm(Ui.abs(), Vj.abs().transpose(1, 2)) + torch.bmm(Vi.abs(), Uj.abs().transpose(1, 2))
    ah = ri * adj * rj
    F = d["Ft"].double()
    es = torch.zeros_like(x)
    es_abs = torch.zeros_like(x)
    if cfg["measure"] == 1:
        es, es_abs = 4 * k1 * (ah - F), 4 * abs(k1) * (ah + F.abs())
    elif cfg["measure"] == 6:
        es, es_abs = F, F.abs()
    elif cfg["measure"] == 2:
        lAi, lAj = tr.node(d["lseA"].double())
        lFi, lFj = tr.node(d["lseF"].double())
        parts = (torch.exp(ah - lAi), torch.exp(F - lFi), torch.exp(ah - lAj), torch.exp(F - lFj))
        es = k1 * ((parts[0] - parts[1]) + (parts[2] - parts[3]))
        es_abs = abs(k1) * sum(parts) * (2 + float(np.log(max(tr.n, 2))))
    if k6 != 0.0:
        inside = (ah >= 1e-4) & (ah <= 1 - 1e-4)
        lg = torch.log2(ah.clamp(1e-4, 1 - 1e-4)) + 1.0 / np.log(2.0)
        es = es + torch.where(inside, 2 * k6 * lg, torch.zeros_like(lg))
        es_abs = es_abs + 2 * abs(k6) * (lg.abs() + 1)
    if k2 != 0.0:
        Z = tr.block(d["zhat"].double())
        s = torch.bmm(Z[tr.I], Z[tr.J].transpose(1, 2))
        es = es + 4 * k2 * (ah - s.clamp_min(0.0))
        es_abs = es_abs + 4 * abs(k2) * (ah + torch.bmm(Z[tr.I].abs(), Z[tr.J].abs().transpose(1, 2)))
    G = d["Gt"].double() if d["Gt"] is not None else torch.zeros_like(x)
    inv_norm = 1.0 / np.sqrt(SUMSQ_PREV)
    g = mask * (ri * rj * es + rhoi + rhoj + prod + G) + NORM_COEF * inv_norm * par
    S = ri * rj * es_abs + rhoi.abs() + rhoj.abs() + prod_abs + G.abs() + NORM_COEF * inv_norm * par.abs()
    m1 = BETA1 * d["m"].double() + (1 - BETA1) * g
    v1 = BETA2 * d["v"].double() + (1 - BETA2) * g * g
    bc1, bc2 = 1 - BETA1 ** STEP, 1 - BETA2 ** STEP
    step_size = LR / bc1
    den = v1.sqrt() / np.sqrt(bc2) + ADAM_EPS
    xn = par - LR * g if cfg.get("plain_gd") else par - step_size * m1 / den
    return dict(xn=xn, m=m1, v=v1, g=g, S=S, par=par, den=den, step_size=step_size)


def fold_call(tr, cfg, d, sh, use_engine):
    """Run mcgra_fold_adam over the shards on copies of x, m, v; returns the outputs."""
    n, dev = tr.n, tr.dev
    x, m, v = d["x"].clone(), d["m"].clone(), d["v"].clone()
    d_next = d["d0"].clone()
    acc_prev = torch.zeros(32, dtype=torch.float64, device=dev)
    acc_prev[9] = SUMSQ_PREV
    acc_next = torch.zeros(32, dtype=torch.float64, device=dev)
    minmax = torch.tensor([float("inf"), float("-inf")], device=dev)
    wk = torch.empty(N().lib().mcgra_fold_ws_bytes(n), dtype=torch.uint8, device=dev)
    step_dev = torch.tensor([STEP - 1], dtype=torch.int32, device=dev)
    f = N().FoldArgs()
    f.n, f.npad, f.Wt, f.r, f.rho = n, tr.npad, P(d["Wt"]), P(d["r"]), P(d["rho"])
    f.lseA, f.lseF, f.zhat = P(d["lseA"]), P(d["lseF"]), P(d["zhat"])
    f.measure = cfg["measure"]
    f.k1 = 0.37 if cfg["measure"] in (1, 2) else 0.0
    f.k6, f.k2 = cfg.get("k6", 0.0), cfg.get("k2", 0.0)
    f.norm_coef, f.lr, f.beta1, f.beta2, f.adam_eps = NORM_COEF, LR, BETA1, BETA2, ADAM_EPS
    f.step = -100 if cfg.get("step_ptr") else STEP          # step_ptr overrides step
    f.step_ptr = P(step_dev) if cfg.get("step_ptr") else None
    f.acc_prev, f.acc_next, f.d_next = P(acc_prev), P(acc_next), P(d_next)
    f.store_clamped = cfg.get("store_clamped", 0)
    f.Wk = P(wk)
    f.plain_gd = cfg.get("plain_gd", 0)
    mu = mu_tensor(cfg.get("mu", 0.0), dev)
    _, eng, cap = use_engine
    with engines({1: eng}, caps={1: cap}):
        for tr0, tr1 in sh:
            f.Ftiles = P(sl(d["Ft"], tr0, tr1)) if cfg["measure"] != 0 else None
            f.Gtiles = P(sl(d["Gt"], tr0, tr1)) if d["Gt"] is not None else None
            N().call("mcgra_fold_adam", P(sl(x, tr0, tr1)), P(sl(m, tr0, tr1)), P(sl(v, tr0, tr1)), tr0, tr1, P(mu),
                     cfg["raw"], C.byref(f), P(minmax), stream())
        torch.cuda.synchronize()
    return dict(x=x, m=m, v=v, d_next=d_next, acc=acc_next, minmax=minmax)


# Bounds: the gradient g is formed in fp32 (engines 2 / 3: 3xTF32 factor product, ~2^-21 of sum |U_i V_j|) to within
# dg = 2^-19 S, S the sum of the absolute values of its parts.  m' is linear in g: |m' - m'64| <= (1 - beta1) dg + 2 u
# |m'|.  v' and x' follow from dg through Adam's formulas plus a few roundings of the MUFU sqrt / divide (2^-21 relative).
# The sums the kernel forms from its own x' are checked far tighter: d_next within (128 + 2 T) u of the row sums,
# SUMCLAMP / SUMSQ within 128 u (per-thread fp32 chains of at most 64 entries), min / max bit for bit.  Largest fraction
# of the bounds seen on a B200 ([fold-precision]): m' 0.35, v' 0.35, x' 0.25.
@pytest.mark.parametrize("cfg_name", list(FOLD_CFGS))
@pytest.mark.parametrize("n", SIZES)
def test_fold_adam(dev, n, cfg_name):
    cfg = FOLD_CFGS[cfg_name]
    tr = Tri(n, dev)
    g = gen(dev, 6000 + n + 31 * list(FOLD_CFGS).index(cfg_name))
    d = fold_inputs(tr, cfg, g)
    d["d0"] = (1.0 + 0.25 * torch.randint(0, 8, (n,), generator=g, device=dev).float()).contiguous()
    ref = fold_reference(tr, cfg, d)
    dg = 2.0 ** -19 * ref["S"]
    bm = (1 - BETA1) * dg + 2 * U * ref["m"].abs()
    bv = (1 - BETA2) * (2 * ref["g"].abs() * dg + dg * dg) + 4 * U * ref["v"]
    if cfg.get("plain_gd"):
        bx = LR * dg + 4 * U * (ref["par"].abs() + LR * ref["g"].abs())
    else:
        den, ss = ref["den"], ref["step_size"]
        dden = bv / (2 * ref["v"].sqrt() * np.sqrt(1 - BETA2 ** STEP)) + 4 * U * den
        bx = ss * (bm / den + ref["m"].abs() * dden / den ** 2) + 8 * U * (ref["par"].abs() + ss * ref["m"].abs() / den)
    sc = bool(cfg.get("store_clamped"))
    want_x = ref["xn"].clamp(0.0, 1.0) if sc else ref["xn"]
    worst = {"m": 0.0, "v": 0.0, "x": 0.0}
    for eng in FOLD_ENGINES:
        for split in SPLITS:
            sh = shards(split, tr.T)
            sel = tr.rows_mask(sh)
            out = fold_call(tr, cfg, d, sh, eng)
            tag = f"{eng[0]} {split}"
            # tiles outside the shards untouched; invalid entries of the shards' tiles +0.0
            for key in ("x", "m", "v"):
                assert bits_equal(out[key][~sel], d[key][~sel]), f"{tag}: {key} written outside the shard"
                inval = out[key][sel][~tr.valid[sel]]
                assert bits_equal(inval, torch.zeros_like(inval)), f"{tag}: invalid entries of {key} are not +0.0"
            if split == "empty":
                assert torch.equal(out["d_next"], d["d0"]) and (out["acc"] == 0).all(), f"{tag}: the empty shard wrote"
                assert out["minmax"][0] == float("inf") and out["minmax"][1] == float("-inf")
                continue
            vm = tr.valid & sel[:, None, None]
            for key, want, bnd in (("m", ref["m"], bm), ("v", ref["v"], bv), ("x", want_x, bx)):
                err = (out[key].double() - want).abs()[vm]
                frac = float((err / bnd[vm]).max()) if err.numel() else 0.0
                worst[key] = max(worst[key], frac)
                assert frac <= 1.0, f"{tag}: {key}' {frac:.3f} of the bound"
            # self-consistency with the kernel's own x'
            xr = out["x"].double()
            c = torch.where(vm, xr.clamp(0.0, 1.0), torch.zeros_like(xr))
            rs = tr.rowcol(c, c, sel)
            want_d = d["d0"].double() + rs
            bd = (128 + 2 * tr.T) * U * want_d
            assert ((out["d_next"].double() - want_d).abs() <= bd).all(), f"{tag}: d_next is not 1 + the row sums of x'"
            for slot, s in ((8, c.sum()), (9, (c * c).sum())):
                assert abs(float(out["acc"][slot]) - float(s)) <= 128 * U * float(s), f"{tag}: acc[{slot}]"
            others = torch.ones(32, dtype=torch.bool, device=dev)
            others[[8, 9]] = False
            assert (out["acc"][others] == 0).all()
            if not sc:
                xv = out["x"][vm]
                assert bits_equal(out["minmax"], torch.stack([xv.min(), xv.max()])), \
                    f"{tag}: minmax {out['minmax'].tolist()} vs {xv.min().item()!r}, {xv.max().item()!r}"
    print(f"[fold-precision] n={n} {cfg_name}: largest error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


# ---------------------------------------------------------------------------------------------------------------------
# 6. bisection
# ---------------------------------------------------------------------------------------------------------------------
EPS = np.float32(1e-5)
PASSES = 10                        # as the engine issues (engine.BISECT_PASSES)


def replay_bisection(xv, a, b, budget, eps):
    """oracle.pgd_oracle.bisection with fp32 midpoints (a + b) / 2 and func evaluated in fp64 (x' and the fp32
    midpoints are exact in fp64).  Returns (mu, [(midpoint, func)])."""
    a, b = np.float32(a), np.float32(b)

    def func(c):
        return float((xv - float(c)).clamp(0.0, 1.0).sum()) - budget

    miu, seen = a, []
    while np.float32(b - a) >= eps:
        miu = np.float32((a + b) / np.float32(2))
        f = func(miu)
        seen.append((miu, f))
        if f == 0.0:
            break
        if f * func(a) < 0:
            b = miu
        else:
            a = miu
    return miu, seen


def bisect_run(tr, x, sh, minmax, budget, eps, acc, passes=PASSES):
    dev, st = tr.dev, stream()
    state = torch.full((8,), float("nan"), device=dev)
    mu = torch.full((1,), float("nan"), device=dev)
    cand = torch.zeros(7, dtype=torch.float64, device=dev)
    N().call("mcgra_bisect_init", P(acc), P(minmax), budget, P(state), P(mu), st)
    for _ in range(passes):
        for tr0, tr1 in sh:
            N().call("mcgra_bisect_pass", P(sl(x, tr0, tr1)), tr.n, tr0, tr1, float(eps), P(state), P(cand), st)
        N().call("mcgra_bisect_update", budget, float(eps), P(state), P(cand), P(mu), st)
    torch.cuda.synchronize()
    return state, mu, cand


def bisect_finish_check(tr, x, state, mu, sh, exact, tag):
    """finish (reset 0 / 1) adds 1 + row and column sums and sum clamp^2 of clamp(x' - mu, 0, 1) (reset first sets
    d_next = 1, SUMSQ = 0)."""
    dev = tr.dev
    sel = tr.rows_mask(sh)
    c = torch.where(tr.valid, (x - mu).clamp(0.0, 1.0), torch.zeros((), device=dev)).double()
    rs = tr.rowcol(c, c, sel)
    ssq = float((c[sel] ** 2).sum())
    for reset in (0, 1):
        d0 = torch.full((tr.n,), 2.5, device=dev)
        acc = torch.zeros(32, dtype=torch.float64, device=dev)
        acc[9] = 7.5
        acc[8] = 11.0
        for k, (tr0, tr1) in enumerate(sh):       # the reset belongs to the first call of the sequence
            N().call("mcgra_bisect_finish", P(sl(x, tr0, tr1)), tr.n, tr0, tr1, P(state), P(mu), P(acc), P(d0),
                     reset if k == 0 else 0, stream())
        torch.cuda.synchronize()
        want_d = (1.0 if reset else 2.5) + rs
        want_s = (0.0 if reset else 7.5) + ssq
        if exact:
            assert torch.equal(d0.double(), want_d) and float(acc[9]) == want_s, f"{tag} reset={reset}"
        else:
            assert ((d0.double() - want_d).abs() <= (128 + 2 * tr.T) * U * want_d).all(), f"{tag} reset={reset}: d_next"
            assert abs(float(acc[9]) - want_s) <= 128 * U * want_s, f"{tag} reset={reset}: SUMSQ"
        assert float(acc[8]) == 11.0


@pytest.mark.parametrize("split", ["whole", "split3"])
@pytest.mark.parametrize("n", SIZES)
def test_bisect_matches_replay(dev, n, split):
    tr = Tri(n, dev)
    sh = shards(split, tr.T)
    g = gen(dev, 7000 + n)
    z = torch.zeros((), device=dev)
    # x' = k / 8 in [0, 1] with both ends present: the bracket [min - 1, max] is [-1, 1] ([0, 1] at n = 2), so every fp32
    # midpoint down to the 1e-5 stop is a multiple of 2^-18, x' - c is exact in fp32 and so is every per-thread sum of
    # clamp(x' - c) (at most 64 terms: < 2^6 in units of 2^-18 < 2^24): the kernel's func values are exact, and its
    # decisions are the replay's unless one is a tie (func = 0), which the data rule out.
    k = torch.randint(0, 9, (tr.nt, TILE, TILE), generator=g, device=dev).float()
    k[0, 1, 0], k[0, 2, 0] = (8.0, 0.0) if n > 2 else (8.0, 8.0)
    x = torch.where(tr.valid, k / 8.0, z).contiguous()
    xv = x[tr.valid].double()
    lo, hi = float(xv.min()), float(xv.max())
    assert (lo, hi) == ((0.0, 1.0) if n > 2 else (1.0, 1.0))
    minmax = torch.tensor([lo, hi], device=dev)
    a0, b0 = np.float32(np.float32(lo) - np.float32(1.0)), np.float32(hi)
    # the root at 2/3 of the bracket (binary 0.1010...): no midpoint of any depth is a root, so no decision is a tie
    croot = float(a0) + (float(b0) - float(a0)) * 2.0 / 3.0
    budget = float((xv - croot).clamp(0.0, 1.0).sum())
    acc = torch.zeros(32, dtype=torch.float64, device=dev)
    acc[8] = float(xv.clamp(0.0, 1.0).sum())
    assert acc[8] > budget
    mu_ref, seen = replay_bisection(xv, a0, b0, budget, EPS)
    assert len(seen) <= 3 * PASSES
    for c, f in seen:
        assert float(c) * 2 ** 18 == round(float(c) * 2 ** 18), f"midpoint {c!r} is not a multiple of 2^-18"
        assert f != 0.0, f"decision at {c!r} is a tie: choose other data"

    # the first pass over shards, accumulated into one cand_sums, equals the whole-range pass (dyadic: exact)
    state = torch.full((8,), float("nan"), device=dev)
    mu = torch.full((1,), float("nan"), device=dev)
    N().call("mcgra_bisect_init", P(acc), P(minmax), budget, P(state), P(mu), stream())
    cw = torch.zeros(7, dtype=torch.float64, device=dev)
    N().call("mcgra_bisect_pass", P(x), n, 0, tr.T, float(EPS), P(state), P(cw), stream())
    cs = torch.zeros(7, dtype=torch.float64, device=dev)
    for tr0, tr1 in sh + shards("empty", tr.T):
        N().call("mcgra_bisect_pass", P(sl(x, tr0, tr1)), n, tr0, tr1, float(EPS), P(state), P(cs), stream())
    torch.cuda.synchronize()
    assert torch.equal(cw, cs)
    lo_hi = [(a0, b0)]                               # the depth-3 midpoints of the first pass, heap order
    mids = []
    for k in range(7):
        a_, b_ = lo_hi[k]
        c_ = np.float32((a_ + b_) / np.float32(2))
        mids.append(c_)
        lo_hi += [(a_, c_), (c_, b_)]
    want = torch.tensor([float((xv - float(c_)).clamp(0.0, 1.0).sum()) for c_ in mids], dtype=torch.float64, device=dev)
    assert torch.equal(cw, want), "first pass: candidate sums"

    state, mu, cand = bisect_run(tr, x, sh, minmax, budget, EPS, acc)
    assert bits_equal(mu, torch.tensor([mu_ref], device=dev)), f"mu {mu.item()!r} vs replay {mu_ref!r}"
    assert state[3] == 1.0 and state[4] == 1.0 and (cand == 0).all()
    # extra pass / update pairs after convergence change nothing
    st = stream()
    s0 = state.clone()
    for _ in range(3):
        N().call("mcgra_bisect_pass", P(x), n, 0, tr.T, float(EPS), P(state), P(cand), st)
        N().call("mcgra_bisect_update", budget, float(EPS), P(state), P(cand), P(mu), st)
    torch.cuda.synchronize()
    assert bits_equal(mu, torch.tensor([mu_ref], device=dev)) and bits_equal(state, s0)
    bisect_finish_check(tr, x, state, mu, sh, False, f"n={n} {split}")


@pytest.mark.parametrize("n", SIZES)
def test_bisect_edges(dev, n):
    tr = Tri(n, dev)
    sh = shards("whole", tr.T)
    g = gen(dev, 8000 + n)
    z = torch.zeros((), device=dev)
    # exact hit: x' in {0, 1, 2}, the first midpoint of [min - 1, max] zeroes func
    x = torch.where(tr.valid, torch.randint(0, 3, (tr.nt, TILE, TILE), generator=g, device=dev).float(), z)
    if n == 2:
        x = torch.where(tr.valid, torch.ones_like(x), z)
    x = x.contiguous()
    xv = x[tr.valid].double()
    lo, hi = float(xv.min()), float(xv.max())
    minmax = torch.tensor([lo, hi], device=dev)
    c0 = np.float32((np.float32(lo - 1.0) + np.float32(hi)) / np.float32(2))
    budget = float((xv - float(c0)).clamp(0.0, 1.0).sum())
    acc = torch.zeros(32, dtype=torch.float64, device=dev)
    acc[8] = float(xv.clamp(0.0, 1.0).sum())
    assert acc[8] > budget
    state, mu, _ = bisect_run(tr, x, sh, minmax, budget, EPS, acc)
    assert float(mu) == float(c0) and state[3] == 1.0, f"exact hit: mu {mu.item()!r}, want {float(c0)!r}"
    bisect_finish_check(tr, x, state, mu, sh, True, f"n={n} exact hit")

    # inactive budget (sum clamp <= budget): mu = 0, finish leaves d_next and SUMSQ alone, even with reset
    state, mu, _ = bisect_run(tr, x, sh, minmax, float(acc[8]), EPS, acc)
    assert bits_equal(mu, torch.zeros(1, device=dev)) and state[4] == 0.0
    for reset in (0, 1):
        d0 = torch.full((n,), 2.5, device=dev)
        a2 = torch.zeros(32, dtype=torch.float64, device=dev)
        a2[9] = 7.5
        N().call("mcgra_bisect_finish", P(x), n, 0, tr.T, P(state), P(mu), P(a2), P(d0), reset, stream())
        torch.cuda.synchronize()
        assert (d0 == 2.5).all() and float(a2[9]) == 7.5

    # a bracket already narrower than epsilon: mu = a = min - 1
    state, mu, _ = bisect_run(tr, x, sh, minmax, budget, np.float32(8.0), acc)
    assert float(mu) == float(np.float32(lo - 1.0))

    # empty shard: finish with reset still resets d_next / SUMSQ of an active projection, and adds nothing
    state, mu, _ = bisect_run(tr, x, sh, minmax, budget, EPS, acc)
    e0, e1 = shards("empty", tr.T)[0]
    for reset in (0, 1):
        d0 = torch.full((n,), 2.5, device=dev)
        a2 = torch.zeros(32, dtype=torch.float64, device=dev)
        a2[9] = 7.5
        assert N().lib().mcgra_bisect_finish(P(x), n, e0, e1, P(state), P(mu), P(a2), P(d0), reset, stream()) == 0
        torch.cuda.synchronize()
        assert (d0 == (1.0 if reset else 2.5)).all() and float(a2[9]) == (0.0 if reset else 7.5)
