"""GPU parity of the dense contraction K6 (csrc/gemm.cu: TMA-fed tcgen05 kind::f16 x3 on CTA pairs) and of its
O(n^2) helpers (csrc/dense.cu) against fp64 torch, through the C ABI."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _N():
    from mcgra_b200 import _native as N
    N.lib()
    return N


def _img(N, rows, cols, dev):
    from mcgra_b200.dense_measure import _Img
    return _Img(rows, cols, dev)


def _image_of(N, X):
    """image of a dense fp32 matrix via the C ABI"""
    dev = X.device
    rows, cols = X.shape
    img = _img(N, rows, cols, dev)
    ws = torch.zeros(max(rows, cols) + 8, dtype=torch.int32, device=dev)
    N.call("mcgra_image_from_dense", N.ptr(X), rows, cols, X.stride(0), 0, img.ref, N.ptr(ws), N.stream_ptr())
    return img


def _recon(img):
    return (img.hi[:, :img.cols].double() + img.lo[:, :img.cols].double()) * img.inv.double()[:, None]


@pytest.mark.parametrize("transpose", [0, 1])
def test_image_from_dense(transpose):
    N = _N()
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(1)
    X = (torch.randn(301, 517, generator=g) * torch.exp(torch.randn(301, 1, generator=g) * 3)).to(dev)
    X[7] = 0.0                                                  # an all-zero row keeps scale 1
    src = X.t().contiguous() if transpose else X
    rows, cols = src.shape
    orows, ocols = (cols, rows) if transpose else (rows, cols)
    img = _img(N, orows, ocols, dev)
    ws = torch.zeros(max(rows, cols) + 8, dtype=torch.int32, device=dev)
    N.call("mcgra_image_from_dense", N.ptr(src), rows, cols, src.stride(0), transpose, img.ref, N.ptr(ws), N.stream_ptr())
    torch.cuda.synchronize()
    R = _recon(img)
    rowmax = X.abs().max(1, keepdim=True).values.double().clamp_min(1e-30)
    assert float(((R - X.double()).abs() / rowmax).max()) < 2.0 ** -22
    assert float((img.hi[:, :ocols].float() * 1.0).abs().max()) <= 16384.0


# the last five shapes put the end of K on and next to the boundaries of the 16-K-block accumulation chunks
@pytest.mark.parametrize("shape", [(256, 256, 64), (300, 200, 150), (1000, 700, 513), (130, 5, 37), (640, 1290, 2050),
                                   (256, 256, 1024), (300, 260, 1088), (257, 511, 2048), (200, 520, 3136), (512, 384, 4160)])
def test_gemm_nt(shape):
    N = _N()
    dev = torch.device("cuda:0")
    M, Nn, K = shape
    g = torch.Generator(device="cpu").manual_seed(M + K)
    A = (torch.randn(M, K, generator=g) * torch.exp(torch.randn(M, 1, generator=g))).to(dev)
    B = torch.rand(Nn, K, generator=g).to(dev)
    ia, ib = _image_of(N, A), _image_of(N, B)
    ldc = (Nn + 63) // 64 * 64
    Cbuf = torch.full((M, ldc), 7.0, dtype=torch.float32, device=dev)
    u, v = torch.randn(M, device=dev), torch.randn(Nn, device=dev)
    red = torch.zeros(2, dtype=torch.float64, device=dev)
    alpha_dev = torch.tensor([0.5], device=dev)
    e = N.GemmEpilogue()
    e.C, e.ldc, e.alpha, e.beta = N.ptr(Cbuf), ldc, 2.0, 0.25
    e.alpha_dev = N.ptr(alpha_dev)
    e.u, e.v, e.coef = N.ptr(u), N.ptr(v), 1.5
    e.sumsq = red.data_ptr()
    N.call("mcgra_gemm_nt", ia.ref, ib.ref, C.byref(e), N.stream_ptr())
    torch.cuda.synchronize()
    ref = A.double() @ B.double().t() - 1.5 * torch.outer(u.double(), v.double())
    scale = (A.double().abs() @ B.double().abs().t()) + 1.5 * torch.outer(u.double().abs(), v.double().abs())
    got = Cbuf[:, :Nn].double()
    want = 0.25 * 7.0 + 2.0 * 0.5 * ref
    err = float(((got - want).abs() / (scale + 1.0)).max())
    assert err < 2e-6, f"shape={shape}: max scaled err {err:.3e}"
    assert torch.all(Cbuf[:, Nn:] == 7.0), "padding columns must stay untouched"
    ssq = float(red[0])
    # (tensor-core fp32 accumulation truncates: a small systematic bias, see test_gemm_large_k)
    assert abs(ssq - float((ref ** 2).sum())) <= 2e-5 * float((ref ** 2).sum())
    # row panel: only rows [row0, row1) are written
    C2 = torch.zeros(M, ldc, dtype=torch.float32, device=dev)
    e2 = N.GemmEpilogue()
    e2.C, e2.ldc, e2.alpha, e2.beta = N.ptr(C2), ldc, 1.0, 0.0
    e2.row0, e2.row1 = M // 3, M // 3 + max(1, M // 2)
    N.call("mcgra_gemm_nt", ia.ref, ib.ref, C.byref(e2), N.stream_ptr())
    torch.cuda.synchronize()
    full = A.double() @ B.double().t()
    r0, r1 = e2.row0, e2.row1
    sc = A.double().abs() @ B.double().abs().t() + 1.0
    assert float(((C2[r0:r1, :Nn].double() - full[r0:r1]).abs() / sc[r0:r1]).max()) < 2e-6
    assert torch.all(C2[:r0] == 0) and torch.all(C2[r1:] == 0)


@pytest.mark.parametrize("K", [16384, 65536])
def test_gemm_large_k(K):
    """All-positive operands (the A_hat M1 product: no cancellation) at the K of the large configurations: the relative
    error of every entry, dominated by the accumulator's truncation bias, must stay far below the 1e-4 loss budget."""
    N = _N()
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(K)
    A = (torch.rand(384, K, generator=g) * 1e-3).to(dev)
    B = torch.rand(256, K, generator=g).to(dev)
    ia, ib = _image_of(N, A), _image_of(N, B)
    Cbuf = torch.zeros(384, 256, dtype=torch.float32, device=dev)
    e = N.GemmEpilogue()
    e.C, e.ldc, e.alpha = N.ptr(Cbuf), 256, 1.0
    N.call("mcgra_gemm_nt", ia.ref, ib.ref, C.byref(e), N.stream_ptr())
    torch.cuda.synchronize()
    ref = A.double() @ B.double().t()
    rel = (Cbuf.double() - ref) / ref
    print(f"K={K}: mean rel err {float(rel.mean()):.3e}, max |rel err| {float(rel.abs().max()):.3e}")
    assert float(rel.abs().max()) < 1.5e-5


def test_gemm_dot_epilogue():
    """sum (A B^T) o E with E an image (the c1 value sum (Kf A) o A)."""
    N = _N()
    dev = torch.device("cuda:0")
    n = 333
    g = torch.Generator(device="cpu").manual_seed(9)
    A = torch.randn(n, n, generator=g).to(dev)
    B = torch.rand(n, n, generator=g).to(dev)
    ia, ib = _image_of(N, A), _image_of(N, B)
    red = torch.zeros(1, dtype=torch.float64, device=dev)
    e = N.GemmEpilogue()
    e.alpha = 1.0
    e.dot = red.data_ptr()
    e.dot_with = C.pointer(ib.c)
    N.call("mcgra_gemm_nt", ia.ref, ib.ref, C.byref(e), N.stream_ptr())
    torch.cuda.synchronize()
    ref = float(((A.double() @ B.double().t()) * B.double()).sum())
    mag = float(((A.double().abs() @ B.double().abs().t()) * B.double().abs()).sum())
    assert abs(float(red[0]) - ref) <= 2e-6 * mag


def test_operand_images_and_helpers():
    """image_ahat / image_m1 / center / gemv / sym_to_tiles against torch."""
    N = _N()
    dev = torch.device("cuda:0")
    n = 300
    T = (n + 127) // 128
    g = torch.Generator(device="cpu").manual_seed(4)
    P = n * (n - 1) // 2
    x = torch.rand(P, generator=g).to(dev)
    tiles = torch.zeros(T * (T + 1) // 2 * 128 * 128, device=dev)
    st = N.stream_ptr()
    N.call("mcgra_tril_to_tiles", N.ptr(x), n, 0, T, N.ptr(tiles), st)
    Md = torch.zeros(n, n, device=dev)
    N.call("mcgra_tiles_to_dense", N.ptr(tiles), n, 0, T, None, 1, N.ptr(Md), n, st)
    d = Md.double().sum(1) + 1.0
    r = d.pow(-0.5).float().contiguous()
    img = _img(N, n, n, dev)
    rs = torch.zeros(n, dtype=torch.float64, device=dev)
    N.call("mcgra_image_ahat", N.ptr(tiles), n, None, 1, N.ptr(r), img.ref, N.ptr(rs), st)
    A = (r[:, None] * (Md + torch.eye(n, device=dev))) * r[None, :]
    torch.cuda.synchronize()
    assert float((_recon(img) - A.double()).abs().max()) < 1e-7
    assert float((rs - A.double().sum(1)).abs().max()) < 1e-5
    z = torch.nn.functional.normalize(torch.relu(torch.randn(n, 16, generator=g)), dim=1).to(dev).contiguous()
    im = _img(N, n, n, dev)
    rm = torch.zeros(n, dtype=torch.float64, device=dev)
    N.call("mcgra_image_m1", N.ptr(z), n, im.ref, N.ptr(rm), st)
    M1 = torch.relu(z @ z.t())
    M1.fill_diagonal_(0.0)
    torch.cuda.synchronize()
    assert float((_recon(im) - M1.double()).abs().max()) < 1e-6
    assert float((rm - M1.double().sum(1)).abs().max()) < 1e-4
    # centring
    ld = 320
    X = torch.zeros(n, ld, device=dev)
    S = torch.randn(n, n, generator=g).to(dev)
    S = S + S.t()
    X[:, :n] = S
    ws = torch.zeros(n + 1, dtype=torch.float64, device=dev)
    N.call("mcgra_center_dense", N.ptr(X), n, ld, N.ptr(ws), st)
    H = torch.eye(n, device=dev, dtype=torch.float64) - 1.0 / n
    assert float((X[:, :n].double() - H @ S.double() @ H).abs().max()) < 1e-5
    # gemv both orientations
    w = torch.rand(n, dtype=torch.float64, device=dev)
    out = torch.zeros(n, dtype=torch.float64, device=dev)
    N.call("mcgra_dense_gemv", N.ptr(X), n, n, ld, N.ptr(w), 0.5, 0, N.ptr(out), st)
    assert float((out - 0.5 * (w @ X[:, :n].double())).abs().max()) < 1e-9 * n
    out.zero_()
    N.call("mcgra_dense_gemv", N.ptr(X), n, n, ld, N.ptr(w), 0.5, 1, N.ptr(out), st)
    assert float((out - 0.5 * (X[:, :n].double() @ w)).abs().max()) < 1e-9 * n
    # sym_to_tiles
    G = torch.randn(n, ld, generator=g).to(dev)
    tl = torch.zeros_like(tiles)
    dg = torch.zeros(n, device=dev)
    sc = torch.tensor([3.0], device=dev)
    N.call("mcgra_sym_to_tiles", N.ptr(G), ld, n, 0, T, 0.5, N.ptr(sc), N.ptr(tl), N.ptr(dg), st)
    back = torch.zeros(n, n, device=dev)
    N.call("mcgra_tiles_to_dense", N.ptr(tl), n, 0, T, None, 1, N.ptr(back), n, st)
    want = 1.5 * (G[:, :n] + G[:, :n].t())
    want.fill_diagonal_(0.0)
    torch.cuda.synchronize()
    assert float((back - want).abs().max()) < 1e-5
    assert float((dg - 1.5 * G[:, :n].diagonal()).abs().max()) < 1e-6
