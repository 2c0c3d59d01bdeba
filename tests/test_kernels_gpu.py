"""Kernel-level parity (B200): every libmpnn_sm100 entry point, called through
the C ABI, against NumPy / PyTorch-CPU restatements on seeded inputs."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import np_ref
from util import Geo, from_planes, rel_err, to_planes

pytestmark = pytest.mark.gpu

F32, BF16 = 0, 1


def L():
    from lib import _cabi
    return _cabi.lib()


def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


_KEEP = []


def dev(a, dtype=None):
    """host array -> device tensor, kept alive until the module is torn down: the
    kernels are asynchronous and only see raw pointers, so a temporary freed
    right after vp() would be recycled by the caching allocator."""
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    t = t if dtype is None else t.to(dtype)
    _KEEP.append(t)
    if len(_KEEP) > 4096:
        torch.cuda.synchronize()
        del _KEEP[:2048]
    return t


def bf16_round(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).float().numpy()


def pack_w(w_hwio, Ktot, k_off, Ntot, n_off, packed, mode, dt):
    w = dev(w_hwio.astype(np.float32))
    kh, kw, I, O = w_hwio.shape
    L().pack_weights(vp(w), kh * kw, I, O, mode, k_off, Ktot, n_off, Ntot, vp(packed), dt, None)


# --------------------------------------------------------------------------- #
# tcgen05 bring-up: descriptor conventions
# --------------------------------------------------------------------------- #
def _blob_kmajor(M, K, rows_total, row_off, a):
    """planes layout [K/8][rows_total][8] bf16 holding a[M][K] from row row_off"""
    t = np.zeros((K // 8, rows_total, 8), np.float32)
    for kg in range(K // 8):
        t[kg, row_off:row_off + M] = a[:, kg * 8:(kg + 1) * 8]
    return t


@pytest.mark.parametrize('N,K,row_off', [(16, 16, 0), (32, 64, 0), (64, 32, 21), (128, 128, 7), (256, 16, 3)])
def test_umma_kmajor_descriptors(N, K, row_off):
    rng = np.random.default_rng(0)
    a = bf16_round(rng.standard_normal((128, K)))
    b = bf16_round(rng.standard_normal((N, K)))
    rows = 128 + 40
    A = dev(_blob_kmajor(128, K, rows, row_off, a), torch.bfloat16)
    Bm = dev(_blob_kmajor(N, K, N, 0, b), torch.bfloat16)
    D = torch.zeros((128, N), device='cuda')
    L().umma_selftest(vp(A), A.numel() * 2, row_off * 16, vp(Bm), Bm.numel() * 2, vp(D), N, K, 0, 0,
                      rows * 16, 128, N * 16, 128, None)
    torch.cuda.synchronize()
    ref = a.astype(np.float64) @ b.astype(np.float64).T
    assert rel_err(D.cpu().numpy(), ref) < 1e-5


@pytest.mark.parametrize('shift', [1, 5, 33])
def test_umma_mnmajor_group_stride_as_row_shift(shift):
    """MN-major B operand whose SBO (stride between 8-channel groups) is `shift` 16-byte rows instead of
    a plane: group j then reads the SAME 8-channel plane displaced by j*shift pixels -- how the weight-
    gradient kernel stacks the three kernel rows along N without staging copies."""
    rng = np.random.default_rng(2)
    K, N = 64, 32
    a = bf16_round(rng.standard_normal((128, K)))
    A = np.zeros((16, K, 8), np.float32)
    for mg in range(16):
        A[mg] = a[mg * 8:(mg + 1) * 8].T
    rows = K + 3 * shift
    plane = bf16_round(rng.standard_normal((rows, 8)))
    b = np.stack([plane[(n // 8) * shift:(n // 8) * shift + K, n % 8] for n in range(N)])     # B[n][k]
    A = dev(A, torch.bfloat16); Bm = dev(plane[None], torch.bfloat16)
    D = torch.zeros((128, N), device='cuda')
    L().umma_selftest(vp(A), A.numel() * 2, 0, vp(Bm), Bm.numel() * 2, vp(D), N, K, 1, 1,
                      128, K * 16, 128, shift * 16, None)
    torch.cuda.synchronize()
    assert rel_err(D.cpu().numpy(), a.astype(np.float64) @ b.astype(np.float64).T) < 1e-5


@pytest.mark.parametrize('N,K,row_off', [(16, 32, 0), (64, 128, 0), (144, 64, 0), (32, 64, 5), (16, 128, 35)])
def test_umma_mnmajor_descriptors(N, K, row_off):
    """MN-major operands (the wgrad orientation): element (m,k) of A lives at
    plane m/8, row k -- SBO = plane stride, LBO = 128 B per 8 rows of K.  row_off
    shifts the start address by whole 16-byte rows (a convolution tap)."""
    rng = np.random.default_rng(1)
    a = bf16_round(rng.standard_normal((128, K)))      # A[m][k]
    b = bf16_round(rng.standard_normal((N, K)))        # B[n][k]
    if row_off:
        rows = K + 48
        A = np.zeros((16, rows, 8), np.float32)
        for mg in range(16):
            A[mg, row_off:row_off + K] = a[mg * 8:(mg + 1) * 8].T
        Bm = np.zeros((N // 8, K, 8), np.float32)
        for ng in range(N // 8):
            Bm[ng] = b[ng * 8:(ng + 1) * 8].T
        A = dev(A, torch.bfloat16); Bm = dev(Bm, torch.bfloat16)
        D = torch.zeros((128, N), device='cuda')
        L().umma_selftest(vp(A), A.numel() * 2, row_off * 16, vp(Bm), Bm.numel() * 2, vp(D), N, K, 1, 1,
                          128, rows * 16, 128, K * 16, None)
        torch.cuda.synchronize()
        assert rel_err(D.cpu().numpy(), a.astype(np.float64) @ b.astype(np.float64).T) < 1e-5
        return
    A = np.zeros((16, K, 8), np.float32)
    for mg in range(16):
        A[mg] = a[mg * 8:(mg + 1) * 8].T
    Bm = np.zeros((N // 8, K, 8), np.float32)
    for ng in range(N // 8):
        Bm[ng] = b[ng * 8:(ng + 1) * 8].T
    A = dev(A, torch.bfloat16); Bm = dev(Bm, torch.bfloat16)
    D = torch.zeros((128, N), device='cuda')
    L().umma_selftest(vp(A), A.numel() * 2, 0, vp(Bm), Bm.numel() * 2, vp(D), N, K, 1, 1,
                      128, K * 16, 128, K * 16, None)
    torch.cuda.synchronize()
    ref = a.astype(np.float64) @ b.astype(np.float64).T
    assert rel_err(D.cpu().numpy(), ref) < 1e-5


# --------------------------------------------------------------------------- #
# stencil GEMM (conv forward), SIMT and tcgen05
# --------------------------------------------------------------------------- #
def _conv_case(B, H, Cin, Cp, Cout, seed=0):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, H, H, Cin)).astype(np.float32)
    xp = rng.standard_normal((B, H, H, Cp)).astype(np.float32) if Cp else None
    wh = (rng.standard_normal((3, 3, Cin, Cout)) / np.sqrt(9 * Cin)).astype(np.float32)
    wv = (rng.standard_normal((3, 3, Cp, Cout)) / np.sqrt(9 * Cp)).astype(np.float32) if Cp else None
    bias = rng.standard_normal(Cout).astype(np.float32)
    return x, xp, wh, wv, bias


def _run_gemm(x, xp, wh, wv, bias, dt, impl, want_stats=True):
    B, H, _, Cin = x.shape
    Cout = wh.shape[3]
    Cp = xp.shape[3] if xp is not None else 0
    geo = Geo(B, H, H)
    q = 16 if dt == BF16 else 8
    K0 = (Cin + q - 1) // q * q
    td = torch.float32 if dt == F32 else torch.bfloat16
    A0 = dev(to_planes(x, geo, K0), td)
    A1 = dev(to_planes(xp, geo), td) if xp is not None else None
    Wp = torch.zeros((9, (K0 + Cp) // 8, Cout, 8), dtype=td, device='cuda')
    pack_w(wh, K0 + Cp, 0, Cout, 0, Wp, 0, dt)
    if wv is not None:
        pack_w(wv, K0 + Cp, K0, Cout, 0, Wp, 0, dt)
    out = torch.zeros((Cout // 8, geo.P, 8), dtype=td, device='cuda')
    stats = torch.zeros(592 * 2 * Cout, device='cuda')
    cnt = ctypes.c_int(0)
    L().stencil_gemm(vp(A0), K0, vp(A1), Cp, vp(Wp), 9, vp(dev(bias)), vp(out), Cout, 0, None, 0, 0,
                     B, H, H, geo.G, geo.P, vp(stats) if want_stats else None, 592, ctypes.byref(cnt),
                     dt, dt, impl, None)
    torch.cuda.synchronize()
    y = from_planes(out.float().cpu().numpy(), geo, Cout)
    st = stats.cpu().numpy()[:cnt.value * 2 * Cout].reshape(cnt.value, 2, Cout).sum(0) if want_stats else None
    return y, st


def _ref_conv(x, xp, wh, wv, bias, rounder=lambda a: a):
    y = np_ref.conv3_same(np.float64(rounder(x)), np.float64(rounder(wh))) + bias
    if xp is not None:
        y = y + np_ref.conv3_same(np.float64(rounder(xp)), np.float64(rounder(wv)))
    return y


@pytest.mark.parametrize('B,H,Cin,Cp,Cout', [(3, 8, 3, 0, 16), (2, 16, 16, 16, 16), (5, 4, 32, 64, 64),
                                              (2, 32, 16, 0, 32), (7, 4, 128, 0, 128)])
def test_stencil_gemm_simt_fp32(B, H, Cin, Cp, Cout):
    x, xp, wh, wv, bias = _conv_case(B, H, Cin, Cp, Cout)
    y, st = _run_gemm(x, xp, wh, wv, bias, F32, 0)
    ref = _ref_conv(x, xp, wh, wv, bias)
    assert rel_err(y, ref) < 1e-5
    np.testing.assert_allclose(st[0], ref.sum((0, 1, 2)), rtol=1e-4, atol=1e-3)
    np.testing.assert_allclose(st[1], (ref ** 2).sum((0, 1, 2)), rtol=1e-4)


@pytest.mark.parametrize('impl', [0, 1])
@pytest.mark.parametrize('B,H,Cin,Cp,Cout', [(3, 8, 3, 0, 16), (2, 16, 16, 16, 16), (5, 4, 32, 64, 64),
                                              (2, 32, 16, 0, 32), (7, 4, 128, 0, 128), (40, 4, 64, 64, 64),
                                              (9, 8, 64, 0, 64), (130, 32, 16, 16, 16)])
def test_stencil_gemm_bf16(impl, B, H, Cin, Cp, Cout):
    x, xp, wh, wv, bias = _conv_case(B, H, Cin, Cp, Cout, seed=impl)
    y, st = _run_gemm(x, xp, wh, wv, bias, BF16, impl)
    ref = _ref_conv(x, xp, wh, wv, bias, bf16_round)     # exact products of bf16 operands
    # output itself is stored as bf16: 2^-9 relative rounding
    assert rel_err(y, ref) < 4e-3
    np.testing.assert_allclose(st[0], ref.sum((0, 1, 2)), rtol=2e-3, atol=0.05 * np.sqrt(ref.size / Cout))
    np.testing.assert_allclose(st[1], (ref ** 2).sum((0, 1, 2)), rtol=2e-3)


@pytest.mark.parametrize('dt,impl', [(F32, 0), (BF16, 0), (BF16, 1)])
def test_stencil_dgrad_split_outputs(dt, impl):
    """dgrad = same kernel with transposed/flipped weights, columns split over two outputs"""
    rng = np.random.default_rng(5)
    B, H, Cin, Cp, Cout = 4, 8, 32, 16, 32
    g = rng.standard_normal((B, H, H, Cout)).astype(np.float32)
    wh = rng.standard_normal((3, 3, Cin, Cout)).astype(np.float32) / 10
    wv = rng.standard_normal((3, 3, Cp, Cout)).astype(np.float32) / 10
    geo = Geo(B, H, H)
    td = torch.float32 if dt == F32 else torch.bfloat16
    rd = (lambda a: a) if dt == F32 else bf16_round
    G = dev(to_planes(g, geo), td)
    Wd = torch.zeros((9, Cout // 8, Cin + Cp, 8), dtype=td, device='cuda')
    pack_w(wh, Cout, 0, Cin + Cp, 0, Wd, 1, dt)
    pack_w(wv, Cout, 0, Cin + Cp, Cin, Wd, 1, dt)
    o0 = torch.zeros((Cin // 8, geo.P, 8), dtype=td, device='cuda')
    o1 = torch.zeros((Cp // 8, geo.P, 8), dtype=td, device='cuda')
    L().stencil_gemm(vp(G), Cout, None, 0, vp(Wd), 9, None, vp(o0), Cin, 0, vp(o1), Cp, 0,
                     B, H, H, geo.G, geo.P, None, 0, None, dt, dt, impl, None)
    torch.cuda.synchronize()
    gt = torch.tensor(rd(g), dtype=torch.float64).permute(0, 3, 1, 2)
    for w, o, C in ((wh, o0, Cin), (wv, o1, Cp)):
        wt = torch.tensor(rd(w), dtype=torch.float64).permute(3, 2, 0, 1)      # OIHW
        ref = torch.nn.functional.conv_transpose2d(gt, wt, padding=1).permute(0, 2, 3, 1).numpy()
        assert rel_err(from_planes(o.float().cpu().numpy(), geo, C), ref) < (1e-5 if dt == F32 else 4e-3)


@pytest.mark.parametrize('dt,impl', [(F32, 0), (BF16, 1)])
@pytest.mark.parametrize('B,H,K0,K1,N', [(3, 8, 16, 0, 16), (40, 16, 16, 16, 32), (7, 4, 64, 32, 64), (300, 8, 16, 0, 16)])
def test_deferred_bn_statistics_equal_the_last_cta_protocol(dt, impl, B, H, K0, K1, N):
    """bn.defer = 1: the conv only adds its partial sums into acc and mpnn_bn_relu_pool_fwd_acc derives scale / shift,
    mean / rstd and the running moments -- same numbers as the conv's last-CTA finalisation + mpnn_bn_relu_pool_fwd"""
    from lib.engine import _BN_FUSE, _host_struct
    rng = np.random.default_rng(23)
    td = torch.float32 if dt == F32 else torch.bfloat16
    geo, gp = Geo(B, H, H), Geo(B, H // 2, H // 2)
    mk = lambda C: dev(to_planes(rng.standard_normal((B, H, H, C)).astype(np.float32), geo), td)
    A0, A1 = mk(K0), (mk(K1) if K1 else None)
    Wp = dev(rng.standard_normal((9, (K0 + K1) // 8, N, 8)).astype(np.float32) * 0.1, td)
    bias = dev(rng.standard_normal(N).astype(np.float32))
    gamma, beta = dev(rng.standard_normal(N).astype(np.float32)), dev(rng.standard_normal(N).astype(np.float32))
    res = []
    for defer in (0, 1):
        acc = torch.zeros(2 * N + 2, dtype=torch.float64, device='cuda')
        ss, mr = torch.zeros((2, N), device='cuda'), torch.zeros((2, N), device='cuda')
        ma, va = torch.zeros(N, device='cuda'), torch.ones(N, device='cuda')
        lin = torch.zeros((N // 8, geo.P, 8), dtype=td, device='cuda')
        act = torch.zeros_like(lin)
        pooled = torch.zeros((N // 8, gp.P, 8), dtype=td, device='cuda')
        f = _host_struct(_BN_FUSE, acc=vp(acc), gamma=vp(gamma), beta=vp(beta), m_avg=vp(ma), v_avg=vp(va),
                         ss=vp(ss), mr=vp(mr), count=float(B * H * H), d=0.9, eps=1e-6, defer=defer)
        fp = ctypes.c_void_p(f.ctypes.data)
        L().conv_bn_stats(vp(A0), K0, vp(A1), K1, vp(Wp), vp(bias), vp(lin), N, B, H, H, geo.G, geo.P, fp, dt, impl, None)
        if defer:
            L().bn_relu_pool_fwd_acc(vp(lin), N, B, H, H, geo.G, geo.P, fp, vp(act), vp(pooled), gp.P, None, 0, dt, None)
        else:
            L().bn_relu_pool_fwd(vp(lin), N, B, H, H, geo.G, geo.P, vp(ss), vp(act), vp(pooled), gp.P, None, 0, dt, None)
        torch.cuda.synchronize()
        res.append([t.float().cpu().numpy() for t in (lin, act, pooled, ss, mr, ma, va)])
    for a, b, name in zip(res[0], res[1], ('lin', 'act', 'pooled', 'ss', 'mr', 'm_avg', 'v_avg')):
        if name in ('lin', 'pooled'):
            assert np.array_equal(a, b), name
        else:
            np.testing.assert_allclose(b, a, rtol=2e-5, atol=2e-6, err_msg=name)


@pytest.mark.parametrize('B,H,K,N0,N1', [(5, 8, 16, 16, 0), (40, 16, 16, 16, 16), (9, 8, 32, 32, 0), (130, 32, 16, 16, 0),
                                         (6, 8, 32, 16, 32), (7, 8, 64, 64, 0), (3, 4, 64, 32, 64), (300, 8, 16, 16, 16)])
def test_dgrad_with_fused_bn_backward_sums(B, H, K, N0, N1):
    """mpnn_conv_dgrad_bn_reduce: the data gradient is bit-identical to mpnn_stencil_gemm, and the sums /
    dgamma / dbeta the last CTA writes match the stand-alone mpnn_bn_bwd_reduce_fused pass over
    (lin, dAct).  Shapes cover the 16- / 32-wide fast epilogues, the generic one (N = 48, 64, 96) and a
    grid with more tiles than CTAs; run twice to check that the accumulator cleans itself."""
    from lib.engine import _BN_BWD_EPI, _BN_BWD_FUSE, _host_struct
    rng = np.random.default_rng(31)
    td = torch.bfloat16
    geo = Geo(B, H, H)
    mk = lambda C: dev(to_planes(rng.standard_normal((B, H, H, C)).astype(np.float32), geo), td)
    G, lin = mk(K), mk(N0)
    Wd = dev(rng.standard_normal((9, K // 8, N0 + N1, 8)).astype(np.float32) * 0.1, td)
    ss = dev(np.stack([rng.standard_normal(N0), 0.3 * rng.standard_normal(N0)]).astype(np.float32))
    mr = dev(np.stack([rng.standard_normal(N0), 0.5 + rng.random(N0)]).astype(np.float32))
    mko = lambda C: torch.zeros((max(C, 8) // 8, geo.P, 8), dtype=td, device='cuda')
    a0, a1, b0, b1 = mko(N0), mko(N1), mko(N0), mko(N1)
    L().stencil_gemm(vp(G), K, None, 0, vp(Wd), 9, None, vp(a0), N0, 0, vp(a1) if N1 else None, N1, 0,
                     B, H, H, geo.G, geo.P, None, 0, None, BF16, BF16, 1, None)
    acc = torch.zeros(2 * N0 + 1, dtype=torch.float64, device='cuda')
    sums_a = torch.zeros((2, N0), device='cuda'); dg_a = torch.zeros(N0, device='cuda'); db_a = torch.zeros(N0, device='cuda')
    fa = _host_struct(_BN_BWD_FUSE, acc=vp(acc), sums=vp(sums_a), dgamma=vp(dg_a), dbeta=vp(db_a))
    L().bn_bwd_reduce_fused(vp(lin), vp(a0), None, 0, vp(ss), vp(mr), N0, B, H, H, geo.G, geo.P,
                            ctypes.c_void_p(fa.ctypes.data), BF16, None)
    sums_b = torch.zeros((2, N0), device='cuda'); dg_b = torch.zeros(N0, device='cuda'); db_b = torch.zeros(N0, device='cuda')
    epi = _host_struct(_BN_BWD_EPI, lin=vp(lin), ss=vp(ss), mr=vp(mr), acc=vp(acc), sums=vp(sums_b),
                       dgamma=vp(dg_b), dbeta=vp(db_b))
    for rep in range(2):
        dg_b.zero_(); db_b.zero_(); b0.zero_(); b1.zero_()
        L().conv_dgrad_bn_reduce(vp(G), K, vp(Wd), vp(b0), N0, vp(b1) if N1 else None, N1, B, H, H, geo.G, geo.P,
                                 ctypes.c_void_p(epi.ctypes.data), BF16, 1, None)
        torch.cuda.synchronize()
        assert float(acc.abs().max()) == 0.0
        for a, b, C in ((a0, b0, N0), (a1, b1, N1)):
            if C:
                assert np.array_equal(from_planes(a.float().cpu().numpy(), geo, C), from_planes(b.float().cpu().numpy(), geo, C))
        scale = float(sums_a.abs().max())
        for a, b in ((sums_a, sums_b), (dg_a, dg_b), (db_a, db_b)):
            np.testing.assert_allclose(b.cpu().numpy(), a.cpu().numpy(), rtol=5e-5, atol=5e-6 * scale)


@pytest.mark.parametrize('B,H,Cin,Cp,Cout', [(3, 8, 16, 0, 16), (4, 16, 16, 16, 32), (5, 4, 64, 32, 64), (130, 32, 16, 16, 16),
                                              (6, 4, 128, 0, 128)])
def test_bf16x3_conv_reaches_fp32_accuracy_on_the_tensor_cores(B, H, Cin, Cp, Cout):
    """mpnn_split_planes + residual weight packing + mpnn_conv_acc_bn_stats: the conv of FP32 operands evaluated as
    a_hi*w_hi + a_lo*w_hi + a_hi*w_lo on tcgen05 (fp32 planes out, pooled predecessor accumulated by a second
    launch, BN moments of the final values) against the exact conv: 1e-4, where plain bf16 gives 4e-3."""
    from lib.engine import _BN_FUSE, _host_struct
    rng = np.random.default_rng(11)
    x = rng.standard_normal((B, H, H, Cin)).astype(np.float32)
    xp = rng.standard_normal((B, H, H, Cp)).astype(np.float32) if Cp else None
    wh = (rng.standard_normal((3, 3, Cin, Cout)) / np.sqrt(9 * Cin)).astype(np.float32)
    wv = (rng.standard_normal((3, 3, Cp, Cout)) / np.sqrt(9 * Cp)).astype(np.float32) if Cp else None
    bias = rng.standard_normal(Cout).astype(np.float32)
    geo = Geo(B, H, H)

    def split(a, C):
        src = dev(to_planes(a, geo, C))
        dst = torch.zeros((2 * C // 8, geo.P, 8), dtype=torch.bfloat16, device='cuda')
        L().split_planes(vp(src), C, geo.P, vp(dst), None)
        return src, dst

    def pack3(w, C):
        W3 = torch.zeros((9, 3 * C // 8, Cout, 8), dtype=torch.bfloat16, device='cuda')
        for k_off, mode in ((0, 0), (C, 0), (2 * C, 4)):
            pack_w(w, 3 * C, k_off, Cout, 0, W3, mode, BF16)
        return W3
    xs, xsp = split(x, Cin)
    hi = xsp[:Cin // 8].float().cpu().numpy(); lo = xsp[Cin // 8:].float().cpu().numpy()
    assert rel_err(hi + lo, xs.cpu().numpy()) < 2e-5                       # x = hi + lo up to 2^-17
    out = torch.zeros((Cout // 8, geo.P, 8), device='cuda')
    acc = torch.zeros(2 * Cout + 1, dtype=torch.float64, device='cuda')
    gm, bt = torch.ones(Cout, device='cuda'), torch.zeros(Cout, device='cuda')
    ss, mr = torch.zeros((2, Cout), device='cuda'), torch.zeros((2, Cout), device='cuda')
    f = _host_struct(_BN_FUSE, acc=vp(acc), gamma=vp(gm), beta=vp(bt), m_avg=None, v_avg=None, ss=vp(ss), mr=vp(mr),
                     count=float(B * H * H), d=0.9, eps=1e-6)
    fp = ctypes.c_void_p(f.ctypes.data)
    W3h = pack3(wh, Cin)
    L().conv_acc_bn_stats(vp(xsp), 2 * Cin, vp(xsp), Cin, vp(W3h), vp(dev(bias)), vp(out), Cout, 0,
                          B, H, H, geo.G, geo.P, None if Cp else fp, BF16, F32, 1, None)
    if Cp:
        _, psp = split(xp, Cp)
        W3v = pack3(wv, Cp)
        L().conv_acc_bn_stats(vp(psp), 2 * Cp, vp(psp), Cp, vp(W3v), None, vp(out), Cout, 1,
                              B, H, H, geo.G, geo.P, fp, BF16, F32, 1, None)
    torch.cuda.synchronize()
    ref = _ref_conv(x, xp, wh, wv, bias, lambda a: a)
    y = from_planes(out.cpu().numpy(), geo, Cout)
    assert rel_err(y, ref) < 1e-4, rel_err(y, ref)
    np.testing.assert_allclose(mr[0].cpu().numpy(), ref.mean((0, 1, 2)), rtol=1e-3, atol=1e-4)
    np.testing.assert_allclose(mr[1].cpu().numpy(), 1 / np.sqrt(ref.var((0, 1, 2)) + 1e-6), rtol=1e-3)


@pytest.mark.parametrize('B,H,Cin,Cp,Cout', [(3, 8, 16, 0, 16), (4, 16, 16, 16, 32), (5, 4, 64, 32, 64), (6, 4, 128, 0, 128)])
def test_bf16x6_conv_matches_fp32_arithmetic_on_the_tensor_cores(B, H, Cin, Cp, Cout):
    """mpnn_split_planes3 + first / second residual weight packing: the conv of FP32 operands as the six bf16
    products a_h*w_h + a_m*w_h + a_l*w_h + a_h*w_m + a_m*w_m + a_h*w_l (two accumulating launches of K = 3C per
    source) against the exact conv: 1e-5, i.e. fp32-accumulation level (the three-product mode is held to 1e-4, plain bf16 to 4e-3)."""
    rng = np.random.default_rng(12)
    x = rng.standard_normal((B, H, H, Cin)).astype(np.float32)
    xp = rng.standard_normal((B, H, H, Cp)).astype(np.float32) if Cp else None
    wh = (rng.standard_normal((3, 3, Cin, Cout)) / np.sqrt(9 * Cin)).astype(np.float32)
    wv = (rng.standard_normal((3, 3, Cp, Cout)) / np.sqrt(9 * Cp)).astype(np.float32) if Cp else None
    bias = rng.standard_normal(Cout).astype(np.float32)
    geo = Geo(B, H, H)

    def split(a, C):
        src = dev(to_planes(a, geo, C))
        dst = torch.zeros((3 * C // 8, geo.P, 8), dtype=torch.bfloat16, device='cuda')
        L().split_planes3(vp(src), C, geo.P, vp(dst), None)
        return src, dst

    def packs(w, C):
        out = []
        for modes in ((0, 0, 0), (4, 4, 8)):
            W3 = torch.zeros((9, 3 * C // 8, Cout, 8), dtype=torch.bfloat16, device='cuda')
            for j, mode in enumerate(modes):
                pack_w(w, 3 * C, j * C, Cout, 0, W3, mode, BF16)
            out.append(W3)
        return out
    xs, xsp = split(x, Cin)
    parts = [xsp[j * Cin // 8:(j + 1) * Cin // 8].double().cpu().numpy() for j in range(3)]
    assert rel_err(parts[0] + parts[1] + parts[2], xs.double().cpu().numpy()) < 1e-7      # x = hi + mid + lo to 2^-24
    W = packs(wh, Cin)
    w_parts = W[0][:, :Cin // 8].double() + W[1][:, :Cin // 8].double() + W[1][:, 2 * Cin // 8:].double()
    ref_w = torch.zeros((9, Cin // 8, Cout, 8), device='cuda')
    pack_w(wh, Cin, 0, Cout, 0, ref_w, 0, F32)
    assert rel_err(w_parts.cpu().numpy(), ref_w.double().cpu().numpy()) < 1e-7
    out = torch.zeros((Cout // 8, geo.P, 8), device='cuda')
    todo = [(xsp, Cin, Wk) for Wk in W]
    if Cp:
        _, psp = split(xp, Cp)
        todo += [(psp, Cp, Wk) for Wk in packs(wv, Cp)]
    for i, (src, C, Wk) in enumerate(todo):
        na0, na1 = (3, 0) if i % 2 == 0 else (2, 1)
        L().conv_acc_bn_stats(vp(src), na0 * C, vp(src) if na1 else None, na1 * C, vp(Wk), vp(dev(bias)) if i == 0 else None,
                              vp(out), Cout, 0 if i == 0 else 1, B, H, H, geo.G, geo.P, None, BF16, F32, 1, None)
    torch.cuda.synchronize()
    ref = _ref_conv(x, xp, wh, wv, bias, lambda a: a)
    y = from_planes(out.cpu().numpy(), geo, Cout)
    print('bf16x6 conv error', rel_err(y, ref))
    assert rel_err(y, ref) < 1e-5, rel_err(y, ref)


@pytest.mark.parametrize('dt,impl,shape', [
    (F32, 0, (6, 8, 3, 16, 32)), (BF16, 0, (6, 8, 3, 16, 32)), (BF16, 1, (6, 8, 3, 16, 32)),
    (BF16, 1, (3, 32, 16, 16, 16)), (BF16, 1, (50, 4, 64, 64, 64)), (BF16, 1, (33, 4, 128, 0, 128)),
    (BF16, 1, (9, 16, 32, 32, 32)), (BF16, 1, (700, 4, 32, 64, 64))])
def test_stencil_wgrad(dt, impl, shape):
    rng = np.random.default_rng(6)
    B, H, Cin, Cp, Cout = shape
    x = rng.standard_normal((B, H, H, Cin)).astype(np.float32)
    xp = rng.standard_normal((B, H, H, Cp)).astype(np.float32) if Cp else None
    g = rng.standard_normal((B, H, H, Cout)).astype(np.float32)
    geo = Geo(B, H, H)
    q = 16 if dt == BF16 else 8
    K0 = (Cin + q - 1) // q * q
    td = torch.float32 if dt == F32 else torch.bfloat16
    rd = (lambda a: a) if dt == F32 else bf16_round
    A0 = dev(to_planes(x, geo, K0), td); G = dev(to_planes(g, geo), td)
    A1 = dev(to_planes(xp, geo), td) if Cp else None
    dW0 = torch.zeros((9, Cin, Cout), device='cuda')
    dW1 = torch.zeros((9, Cp, Cout), device='cuda') if Cp else None
    db = torch.zeros(Cout, device='cuda')
    L().stencil_wgrad(vp(A0), K0, Cin, vp(dW0), vp(A1), Cp, Cp, vp(dW1), vp(G), Cout, Cout, vp(db), 9,
                      B, H, H, geo.G, geo.P, dt, impl, None)
    torch.cuda.synchronize()
    gt = torch.tensor(rd(g), dtype=torch.float64).permute(0, 3, 1, 2)
    for xin, dW, C in ((x, dW0, Cin), (xp, dW1, Cp)):
        if not C:
            continue
        xt = torch.tensor(rd(xin), dtype=torch.float64).permute(0, 3, 1, 2).requires_grad_(False)
        w = torch.zeros((Cout, C, 3, 3), dtype=torch.float64, requires_grad=True)
        (torch.nn.functional.conv2d(xt, w, padding=1) * gt).sum().backward()
        ref = w.grad.permute(2, 3, 1, 0).reshape(9, C, Cout).numpy()
        assert rel_err(dW.cpu().numpy(), ref) < 1e-4
    np.testing.assert_allclose(db.cpu().numpy(), rd(g).sum((0, 1, 2)), rtol=1e-4, atol=1e-3)


# --------------------------------------------------------------------------- #
# BN + ReLU + pool
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('pool', [True, False])
def test_bn_relu_pool_fwd_bwd(dt, pool):
    rng = np.random.default_rng(7)
    B, H, C = 5, 8 if pool else 4, 16
    td = torch.float32 if dt == F32 else torch.bfloat16
    rd = (lambda a: a) if dt == F32 else bf16_round
    lin = rd(rng.standard_normal((B, H, H, C)).astype(np.float32) * 2 + 0.5)
    gamma = rng.standard_normal(C).astype(np.float32); beta = rng.standard_normal(C).astype(np.float32) * 0.1
    geo = Geo(B, H, H); gp = Geo(B, H // 2, H // 2)
    LIN = dev(to_planes(lin, geo), td)
    # statistics from exact per-channel sums (finalize path)
    part = dev(np.stack([lin.sum((0, 1, 2)), (lin.astype(np.float64) ** 2).sum((0, 1, 2))]).astype(np.float32))
    ss = torch.zeros((2, C), device='cuda'); mr = torch.zeros((2, C), device='cuda')
    m_avg = torch.zeros(C, device='cuda'); v_avg = torch.ones(C, device='cuda')
    L().bn_finalize(vp(part), 1, C, float(B * H * H), vp(dev(gamma)), vp(dev(beta)), vp(m_avg), vp(v_avg),
                    0.9, 1e-6, 1, vp(ss), vp(mr), None)
    act = torch.zeros_like(LIN)
    pooled = torch.zeros((C // 8, gp.P, 8), dtype=td, device='cuda') if pool else None
    Balloc = 8
    feat = None if pool else torch.zeros((H * H * C // 8, Balloc, 8), dtype=td, device='cuda')
    L().bn_relu_pool_fwd(vp(LIN), C, B, H, H, geo.G, geo.P, vp(ss), vp(act), vp(pooled), gp.P if pool else 0,
                         vp(feat), Balloc, dt, None)
    torch.cuda.synchronize()
    xt = torch.tensor(lin, dtype=torch.float64, requires_grad=True)
    m = xt.mean((0, 1, 2)); v = ((xt - m) ** 2).mean((0, 1, 2))
    yt = torch.relu(torch.tensor(gamma, dtype=torch.float64) * (xt - m) / torch.sqrt(v + 1e-6)
                    + torch.tensor(beta, dtype=torch.float64))
    tol = 1e-4 if dt == F32 else 1e-2
    assert rel_err(from_planes(act.float().cpu().numpy(), geo, C), yt.detach().numpy()) < tol
    np.testing.assert_allclose(m_avg.cpu().numpy(), 0.1 * m.detach().numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(v_avg.cpu().numpy(), 0.9 + 0.1 * v.detach().numpy(), rtol=1e-4)
    if pool:
        pt = torch.nn.functional.max_pool2d(xt.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        np.testing.assert_array_equal(from_planes(pooled.float().cpu().numpy(), gp, C), pt.detach().numpy())
    else:
        f = feat.float().cpu().numpy()          # [F/8][Balloc][8] -> (B, F)
        flat = np.concatenate([f[i, :B] for i in range(f.shape[0])], 1)
        assert rel_err(flat, yt.detach().numpy().reshape(B, -1)) < tol
    # backward
    dy = rd(rng.standard_normal((B, H, H, C)).astype(np.float32))
    dp = rd(rng.standard_normal((B, H // 2, H // 2, C)).astype(np.float32)) if pool else None
    df = None if pool else rd(rng.standard_normal((B, H, H, C)).astype(np.float32))
    DY = dev(to_planes(dy, geo), td)
    DP = dev(to_planes(dp, gp), td) if pool else None
    DF = None
    if df is not None:
        t = np.zeros((H * H * C // 8, Balloc, 8), np.float32)
        flat = df.reshape(B, -1)
        for i in range(t.shape[0]):
            t[i, :B] = flat[:, i * 8:(i + 1) * 8]
        DF = dev(t, td)
    parts = torch.zeros(592 * 2 * C, device='cuda'); cnt = ctypes.c_int(0)
    L().bn_bwd_reduce(vp(LIN), vp(DY), vp(DF), Balloc, vp(ss), vp(mr), C, B, H, H, geo.G, geo.P,
                      vp(parts), 592, ctypes.byref(cnt), dt, None)
    sums = torch.zeros((2, C), device='cuda'); dg = torch.zeros(C, device='cuda'); dbt = torch.zeros(C, device='cuda')
    L().bn_bwd_finalize(vp(parts), cnt.value, C, vp(mr), vp(sums), vp(dg), vp(dbt), None)
    dlin = torch.zeros_like(LIN)
    dbias = torch.zeros(C, device='cuda')
    L().bn_relu_pool_bwd(vp(LIN), vp(DY), vp(DF), Balloc, vp(DP), gp.P if pool else 0, vp(ss), vp(mr), vp(sums),
                         float(B * H * H), C, B, H, H, geo.G, geo.P, vp(dlin), vp(dbias), dt, None)
    torch.cuda.synchronize()
    got_dlin = from_planes(dlin.float().cpu().numpy(), geo, C)
    np.testing.assert_allclose(dbias.cpu().numpy(), got_dlin.sum((0, 1, 2)), rtol=2e-2,
                               atol=2e-3 if dt == F32 else 0.2)     # dLin itself is bf16-rounded
    gtot = torch.tensor(dy, dtype=torch.float64) + (torch.tensor(df, dtype=torch.float64) if df is not None else 0)
    loss = (yt * gtot).sum()
    if pool:
        loss = loss + (pt * torch.tensor(dp, dtype=torch.float64)).sum()
    loss.backward()
    assert rel_err(from_planes(dlin.float().cpu().numpy(), geo, C), xt.grad.numpy()) < (1e-4 if dt == F32 else 2e-2)


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('B,H,C,with_act,with_feat', [(5, 4, 16, True, True), (128, 4, 64, True, True), (200, 4, 16, False, True),
                                                     (512, 4, 32, True, False), (31, 8, 8, True, False)])
def test_bn_fwd_small_matches_finalize_plus_bn_relu(dt, B, H, C, with_act, with_feat):
    """mpnn_bn_fwd_small (train-mode statistics + BN / ReLU / flatten in one cluster launch) against exact channel
    sums -> mpnn_bn_finalize -> mpnn_bn_relu_pool_fwd: constants, running moments, activations, features."""
    rng = np.random.default_rng(32)
    td = torch.float32 if dt == F32 else torch.bfloat16
    rd = (lambda a: a) if dt == F32 else bf16_round
    geo = Geo(B, H, H)
    Balloc = -(-B // 128) * 128
    lin = rd(rng.standard_normal((B, H, H, C)).astype(np.float32) * 2 + 0.5)
    LIN = dev(to_planes(lin, geo), td)
    gamma, beta = dev(rng.standard_normal(C).astype(np.float32)), dev(0.1 * rng.standard_normal(C).astype(np.float32))
    part = dev(np.stack([lin.astype(np.float64).sum((0, 1, 2)), (lin.astype(np.float64) ** 2).sum((0, 1, 2))]).astype(np.float32))
    mk = lambda: (torch.zeros((2, C), device='cuda'), torch.zeros((2, C), device='cuda'),
                  torch.full((C,), 0.3, device='cuda'), torch.full((C,), 1.7, device='cuda'),
                  torch.zeros_like(LIN) if with_act else None,
                  torch.zeros((H * H * C // 8, Balloc, 8), dtype=td, device='cuda') if with_feat else None)
    ss_a, mr_a, ma_a, va_a, act_a, feat_a = mk()
    L().bn_finalize(vp(part), 1, C, float(B * H * H), vp(gamma), vp(beta), vp(ma_a), vp(va_a), 0.9, 1e-6, 1,
                    vp(ss_a), vp(mr_a), None)
    L().bn_relu_pool_fwd(vp(LIN), C, B, H, H, geo.G, geo.P, vp(ss_a), vp(act_a), None, 0, vp(feat_a), Balloc, dt, None)
    ss_b, mr_b, ma_b, va_b, act_b, feat_b = mk()
    L().bn_fwd_small(vp(LIN), C, B, H, H, geo.G, geo.P, vp(gamma), vp(beta), vp(ma_b), vp(va_b), 0.9, 1e-6,
                     vp(ss_b), vp(mr_b), vp(act_b), vp(feat_b), Balloc, dt, None)
    torch.cuda.synchronize()
    for a, b in ((ss_a, ss_b), (mr_a, mr_b), (ma_a, ma_b), (va_a, va_b)):
        np.testing.assert_allclose(b.cpu().numpy(), a.cpu().numpy(), rtol=3e-5, atol=3e-6)
    tol = 1e-5 if dt == F32 else 4e-3
    if with_act:
        assert rel_err(from_planes(act_b.float().cpu().numpy(), geo, C), from_planes(act_a.float().cpu().numpy(), geo, C)) < tol
    if with_feat:
        assert rel_err(feat_b.float().cpu().numpy(), feat_a.float().cpu().numpy()) < tol
        assert float(feat_b.float().abs().sum()) > 0


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('B,H,C,with_act,with_feat', [(5, 4, 16, True, True), (128, 4, 64, True, True), (200, 4, 16, False, True),
                                                     (512, 4, 32, True, False), (31, 8, 8, True, False)])
def test_bn_bwd_small_matches_the_two_pass_pair(dt, B, H, C, with_act, with_feat):
    """mpnn_bn_bwd_small (one launch: 8-CTA cluster per plane, pixels in registers, sums through distributed shared
    memory) against mpnn_bn_bwd_reduce_fused + mpnn_bn_relu_pool_bwd on the same operands: 1 / 2 / 4 pixels per
    thread, with the head gradient on the flattened features, the data gradient, or both."""
    from lib.engine import _BN_BWD_FUSE, _host_struct
    rng = np.random.default_rng(31)
    td = torch.float32 if dt == F32 else torch.bfloat16
    geo = Geo(B, H, H)
    Balloc = -(-B // 128) * 128
    LIN = dev(to_planes(rng.standard_normal((B, H, H, C)).astype(np.float32) * 2 + 0.5, geo), td)
    DY = dev(to_planes(rng.standard_normal((B, H, H, C)).astype(np.float32), geo), td) if with_act else None
    DF = dev(rng.standard_normal((H * H * C // 8, Balloc, 8)).astype(np.float32), td) if with_feat else None
    ss = dev(np.stack([rng.standard_normal(C), 0.3 * rng.standard_normal(C)]).astype(np.float32))
    mr = dev(np.stack([0.5 + 0.2 * rng.standard_normal(C), 0.5 + rng.random(C)]).astype(np.float32))
    count = float(B * H * H)
    acc = torch.zeros(2 * C + 1, dtype=torch.float64, device='cuda')
    sums_a = torch.zeros((2, C), device='cuda'); dg_a = torch.zeros(C, device='cuda'); db_a = torch.zeros(C, device='cuda')
    f = _host_struct(_BN_BWD_FUSE, acc=vp(acc), sums=vp(sums_a), dgamma=vp(dg_a), dbeta=vp(db_a))
    L().bn_bwd_reduce_fused(vp(LIN), vp(DY), vp(DF), Balloc, vp(ss), vp(mr), C, B, H, H, geo.G, geo.P,
                            ctypes.c_void_p(f.ctypes.data), dt, None)
    dlin_a = torch.zeros_like(LIN); dbias_a = torch.zeros(C, device='cuda')
    L().bn_relu_pool_bwd(vp(LIN), vp(DY), vp(DF), Balloc, None, 0, vp(ss), vp(mr), vp(sums_a), count,
                         C, B, H, H, geo.G, geo.P, vp(dlin_a), vp(dbias_a), dt, None)
    sums_b = torch.zeros((2, C), device='cuda'); dg_b = torch.ones(C, device='cuda'); db_b = torch.ones(C, device='cuda')
    dlin_b = torch.zeros_like(LIN); dbias_b = torch.zeros(C, device='cuda')
    L().bn_bwd_small(vp(LIN), vp(DY), vp(DF), Balloc, vp(ss), vp(mr), C, B, H, H, geo.G, geo.P,
                     vp(sums_b), vp(dg_b), vp(db_b), count, vp(dlin_b), vp(dbias_b), dt, None)
    torch.cuda.synchronize()
    scale = float(sums_a.abs().max())
    np.testing.assert_allclose(sums_b.cpu().numpy(), sums_a.cpu().numpy(), rtol=2e-5, atol=2e-6 * scale)
    np.testing.assert_allclose(dg_b.cpu().numpy() - 1, dg_a.cpu().numpy(), rtol=2e-5, atol=2e-5 * scale)      # accumulates
    np.testing.assert_allclose(db_b.cpu().numpy() - 1, db_a.cpu().numpy(), rtol=2e-5, atol=2e-5 * scale)
    a, b = from_planes(dlin_a.float().cpu().numpy(), geo, C), from_planes(dlin_b.float().cpu().numpy(), geo, C)
    assert rel_err(b, a) < (1e-5 if dt == F32 else 4e-3), rel_err(b, a)
    np.testing.assert_allclose(dbias_b.cpu().numpy(), dbias_a.cpu().numpy(), rtol=1e-3, atol=1e-3 * float(dbias_a.abs().max()) + 1e-4)
    assert float(dlin_b.float().abs().sum()) > 0 and torch.equal(dlin_b[:, :geo.G], torch.zeros_like(dlin_b[:, :geo.G]))    # pads untouched


# --------------------------------------------------------------------------- #
# heads
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('dt,impl', [(F32, 0), (BF16, 0), (BF16, 1)])
@pytest.mark.parametrize('B,H,K0,K1,N', [(3, 8, 16, 0, 16), (40, 16, 16, 16, 32), (7, 4, 64, 32, 64), (300, 8, 16, 0, 16)])
def test_fused_bn_statistics_match_the_two_launch_path(dt, impl, B, H, K0, K1, N):
    """conv_bn_stats / bn_bwd_reduce_fused ("last CTA finalises", fp64 atomics) against
    stencil_gemm + bn_finalize and bn_bwd_reduce + bn_bwd_finalize; run twice to check that
    the accumulator cleans itself."""
    from lib.engine import _BN_BWD_FUSE, _BN_FUSE, _host_struct
    rng = np.random.default_rng(21)
    td = torch.float32 if dt == F32 else torch.bfloat16
    geo = Geo(B, H, H)
    mk = lambda C: dev(to_planes(rng.standard_normal((B, H, H, C)).astype(np.float32), geo), td)
    A0, A1 = mk(K0), (mk(K1) if K1 else None)
    Wp = dev(rng.standard_normal((9, (K0 + K1) // 8, N, 8)).astype(np.float32) * 0.1, td)
    bias = dev(rng.standard_normal(N).astype(np.float32))
    gamma, beta = dev(rng.standard_normal(N).astype(np.float32)), dev(rng.standard_normal(N).astype(np.float32))
    count = float(B * H * H)
    # two-launch path
    out_a = torch.zeros((N // 8, geo.P, 8), dtype=td, device='cuda')
    parts = torch.zeros(592 * 2 * N, device='cuda'); cnt = ctypes.c_int(0)
    L().stencil_gemm(vp(A0), K0, vp(A1), K1, vp(Wp), 9, vp(bias), vp(out_a), N, 0, None, 0, 0, B, H, H, geo.G, geo.P,
                     vp(parts), 592, ctypes.byref(cnt), dt, dt, impl, None)
    ss_a, mr_a = torch.zeros((2, N), device='cuda'), torch.zeros((2, N), device='cuda')
    ma_a, va_a = torch.zeros(N, device='cuda'), torch.ones(N, device='cuda')
    L().bn_finalize(vp(parts), cnt.value, N, count, vp(gamma), vp(beta), vp(ma_a), vp(va_a), 0.9, 1e-6, 1,
                    vp(ss_a), vp(mr_a), None)
    # fused path (twice)
    acc = torch.zeros(2 * N + 1, dtype=torch.float64, device='cuda')
    ss_b, mr_b = torch.zeros((2, N), device='cuda'), torch.zeros((2, N), device='cuda')
    ma_b, va_b = torch.zeros(N, device='cuda'), torch.ones(N, device='cuda')
    out_b = torch.zeros_like(out_a)
    f = _host_struct(_BN_FUSE, acc=vp(acc), gamma=vp(gamma), beta=vp(beta), m_avg=vp(ma_b), v_avg=vp(va_b),
                     ss=vp(ss_b), mr=vp(mr_b), count=count, d=0.9, eps=1e-6)
    for rep in range(2):
        ma_b.zero_(); va_b.fill_(1.0)
        L().conv_bn_stats(vp(A0), K0, vp(A1), K1, vp(Wp), vp(bias), vp(out_b), N, B, H, H, geo.G, geo.P,
                          ctypes.c_void_p(f.ctypes.data), dt, impl, None)
        torch.cuda.synchronize()
        assert torch.equal(out_a, out_b)
        assert float(acc.abs().max()) == 0.0                       # self-cleaned (ticket included)
        for a, b in ((ss_a, ss_b), (mr_a, mr_b), (ma_a, ma_b), (va_a, va_b)):
            np.testing.assert_allclose(b.cpu().numpy(), a.cpu().numpy(), rtol=2e-5, atol=2e-6)
    # backward reduction
    DY = mk(N)
    sums_a = torch.zeros((2, N), device='cuda'); dg_a = torch.zeros(N, device='cuda'); db_a = torch.zeros(N, device='cuda')
    L().bn_bwd_reduce(vp(out_a), vp(DY), None, 0, vp(ss_a), vp(mr_a), N, B, H, H, geo.G, geo.P,
                      vp(parts), 592, ctypes.byref(cnt), dt, None)
    L().bn_bwd_finalize(vp(parts), cnt.value, N, vp(mr_a), vp(sums_a), vp(dg_a), vp(db_a), None)
    sums_b = torch.zeros((2, N), device='cuda'); dg_b = torch.zeros(N, device='cuda'); db_b = torch.zeros(N, device='cuda')
    fb = _host_struct(_BN_BWD_FUSE, acc=vp(acc), sums=vp(sums_b), dgamma=vp(dg_b), dbeta=vp(db_b))
    for rep in range(2):
        dg_b.zero_(); db_b.zero_()
        L().bn_bwd_reduce_fused(vp(out_a), vp(DY), None, 0, vp(ss_a), vp(mr_a), N, B, H, H, geo.G, geo.P,
                                ctypes.c_void_p(fb.ctypes.data), dt, None)
        torch.cuda.synchronize()
        assert float(acc.abs().max()) == 0.0
        scale = float(sums_a.abs().max())
        for a, b in ((sums_a, sums_b), (dg_a, dg_b), (db_a, db_b)):
            np.testing.assert_allclose(b.cpu().numpy(), a.cpu().numpy(), rtol=2e-5, atol=2e-6 * scale)


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('B,H,C', [(3, 8, 16), (37, 4, 32), (20, 16, 8)])
def test_maxpool_and_global_maxpool(dt, B, H, C):
    """mpnn_maxpool2_fwd/bwd and mpnn_global_maxpool_fwd/bwd against numpy (layer_types.py:86-100; gradients to the
    first maximum)"""
    rng = np.random.default_rng(41)
    td = torch.float32 if dt == F32 else torch.bfloat16
    rd = (lambda a: a) if dt == F32 else bf16_round
    geo, gp = Geo(B, H, H), Geo(B, H // 2, H // 2)
    x = rd(rng.standard_normal((B, H, H, C)).astype(np.float32))
    X = dev(to_planes(x, geo), td)
    Balloc = (B + 7) // 8 * 8
    F = (H // 2) ** 2 * C
    out = torch.zeros((C // 8, gp.P, 8), dtype=td, device='cuda')
    feat = torch.zeros((F // 8, Balloc, 8), dtype=td, device='cuda')
    L().maxpool2_fwd(vp(X), C, B, H, H, geo.G, geo.P, vp(out), gp.P, vp(feat), Balloc, dt, None)
    torch.cuda.synchronize()
    blocks = x.reshape(B, H // 2, 2, H // 2, 2, C).transpose(0, 1, 3, 2, 4, 5).reshape(B, H // 2, H // 2, 4, C)
    ref = blocks.max(3)
    assert np.array_equal(from_planes(out.float().cpu().numpy(), gp, C), ref)
    f = feat.float().cpu().numpy()
    assert np.array_equal(np.concatenate([f[i, :B] for i in range(F // 8)], 1), ref.reshape(B, -1))
    # backward: pooled-tensor gradient + head gradient, routed to the first maximum of each block
    dout = rd(rng.standard_normal(ref.shape).astype(np.float32))
    dfe = rd(rng.standard_normal((B, F)).astype(np.float32))
    DF = np.zeros((F // 8, Balloc, 8), np.float32)
    for i in range(F // 8):
        DF[i, :B] = dfe[:, i * 8:(i + 1) * 8]
    dx = torch.zeros_like(X)
    L().maxpool2_bwd(vp(X), vp(dev(to_planes(dout, gp), td)), vp(dev(DF, td)), Balloc, C, B, H, H, geo.G, geo.P, gp.P,
                     vp(dx), dt, None)
    torch.cuda.synchronize()
    d = rd(dout + dfe.reshape(ref.shape)) if dt == F32 else dout + dfe.reshape(ref.shape)
    am = blocks.argmax(3)                                                  # first maximum
    refdx = np.zeros_like(blocks)
    np.put_along_axis(refdx, am[:, :, :, None, :], d[:, :, :, None, :], 3)
    refdx = refdx.reshape(B, H // 2, H // 2, 2, 2, C).transpose(0, 1, 3, 2, 4, 5).reshape(B, H, H, C)
    got = from_planes(dx.float().cpu().numpy(), geo, C)
    np.testing.assert_allclose(got, rd(refdx), rtol=0, atol=0 if dt == F32 else 2e-2)
    # global max pool
    gf = torch.zeros((C // 8, Balloc, 8), dtype=td, device='cuda')
    arg = torch.zeros((C // 8, Balloc, 8), dtype=torch.int32, device='cuda')
    L().global_maxpool_fwd(vp(X), C, B, H, H, geo.G, geo.P, vp(gf), vp(arg), Balloc, dt, None)
    torch.cuda.synchronize()
    g = gf.float().cpu().numpy()
    assert np.array_equal(np.concatenate([g[i, :B] for i in range(C // 8)], 1), x.reshape(B, -1, C).max(1))
    a = arg.cpu().numpy()
    assert np.array_equal(np.concatenate([a[i, :B] for i in range(C // 8)], 1), x.reshape(B, -1, C).argmax(1))
    dg = rd(rng.standard_normal((B, C)).astype(np.float32))
    DG = np.zeros((C // 8, Balloc, 8), np.float32)
    for i in range(C // 8):
        DG[i, :B] = dg[:, i * 8:(i + 1) * 8]
    dx2 = torch.zeros_like(X)
    L().global_maxpool_bwd(vp(dev(DG, td)), vp(arg), Balloc, C, B, H, H, geo.G, geo.P, vp(dx2), dt, None)
    torch.cuda.synchronize()
    ref2 = np.zeros((B, H * H, C), np.float32)
    np.put_along_axis(ref2, x.reshape(B, -1, C).argmax(1)[:, None, :], dg[:, None, :], 1)
    assert np.array_equal(from_planes(dx2.float().cpu().numpy(), geo, C), ref2.reshape(B, H, H, C))


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('B,F,n,extra', [(5, 256, 10, False), (37, 512, 16, True), (128, 2048, 2, False)])
def test_fc_fwd_bwd(dt, B, F, n, extra):
    rng = np.random.default_rng(8)
    td = torch.float32 if dt == F32 else torch.bfloat16
    rd = (lambda a: a) if dt == F32 else bf16_round
    x = rd(rng.standard_normal((B, F)).astype(np.float32))
    W = rng.standard_normal((F + (1 if extra else 0), n)).astype(np.float32) / 10
    bias = rng.standard_normal(n).astype(np.float32)
    ex = rng.standard_normal(B).astype(np.float32) if extra else None
    Balloc = (B + 7) // 8 * 8
    t = np.zeros((F // 8, Balloc, 8), np.float32)
    for i in range(F // 8):
        t[i, :B] = x[:, i * 8:(i + 1) * 8]
    X = dev(t, td)
    Z = torch.zeros((B, n), device='cuda')
    Wd, EX = dev(W), (dev(ex) if extra else None)
    L().fc_fwd(vp(X), F, Balloc, B, vp(Wd), vp(dev(bias)), vp(EX), n, vp(Z), dt, None)
    xf = np.concatenate([x, ex[:, None]], 1) if extra else x
    ref = xf.astype(np.float64) @ W + bias
    torch.cuda.synchronize()
    assert rel_err(Z.cpu().numpy(), ref) < 1e-5
    dZ = rng.standard_normal((B, n)).astype(np.float32)
    dZ2 = rng.standard_normal((B, 16)).astype(np.float32)
    W2 = rng.standard_normal((F, 16)).astype(np.float32) / 10
    dX = torch.zeros_like(X)
    L().fc_bwd_data(vp(dev(dZ)), vp(Wd), n, vp(dev(dZ2)), vp(dev(W2)), 16, F, Balloc, B, vp(dX), dt, None)
    torch.cuda.synchronize()
    f = dX.float().cpu().numpy()
    got = np.concatenate([f[i, :B] for i in range(F // 8)], 1)
    refx = dZ.astype(np.float64) @ W[:F].T + dZ2.astype(np.float64) @ W2.T
    assert rel_err(got, refx) < (1e-5 if dt == F32 else 4e-3)
    dW = torch.zeros_like(Wd); db = torch.zeros(n, device='cuda')
    L().fc_bwd_weight(vp(X), F, Balloc, B, vp(EX), vp(dev(dZ)), n, vp(dW), vp(db), dt, None)
    torch.cuda.synchronize()
    assert rel_err(dW.cpu().numpy(), xf.astype(np.float64).T @ dZ) < 1e-5
    np.testing.assert_allclose(db.cpu().numpy(), dZ.sum(0), rtol=1e-4, atol=1e-4)


def test_softmax_ce():
    rng = np.random.default_rng(9)
    B, n = 77, 10
    z = rng.standard_normal((B, n)).astype(np.float32) * 3
    z[0] = 0            # tie -> first index
    y = np.eye(n, dtype=np.float32)[rng.integers(0, n, B)]
    coef = rng.random(B).astype(np.float32)
    Z, Y = dev(z), dev(y)
    prob = torch.zeros_like(Z); ce = torch.zeros(B, device='cuda'); dc = torch.zeros(B, device='cuda')
    L().softmax_ce_fwd(vp(Z), n, vp(Y), B, n, 1e-6, vp(prob), vp(ce), vp(dc), None)
    dZ = torch.zeros_like(Z)
    Balloc = 128
    dZp = torch.zeros((2, Balloc, 8), dtype=torch.bfloat16, device='cuda')
    dbias = torch.zeros(n, device='cuda')
    L().softmax_ce_bwd(vp(prob), vp(Y), B, n, 1e-6, vp(dev(coef)), 1.0 / B, vp(dZ), vp(dZp), Balloc, vp(dbias), None)
    torch.cuda.synchronize()
    planes = dZp.float().cpu().numpy()
    got_p = np.concatenate([planes[0, :B], planes[1, :B]], 1)
    assert rel_err(got_p[:, :n], dZ.cpu().numpy()) < 4e-3 and np.all(got_p[:, n:] == 0) and np.all(planes[:, B:] == 0)
    np.testing.assert_allclose(dbias.cpu().numpy(), dZ.cpu().numpy().sum(0), rtol=1e-4, atol=1e-6)
    zt = torch.tensor(z, dtype=torch.float64, requires_grad=True)
    p = torch.softmax(zt, 1)
    c = -(torch.tensor(y, dtype=torch.float64) * torch.log(1e-6 / n + (1 - 1e-6) * p)).sum(1)
    (c * torch.tensor(coef, dtype=torch.float64) / B).sum().backward()
    np.testing.assert_allclose(ce.cpu().numpy(), c.detach().numpy(), rtol=1e-5, atol=1e-6)
    assert rel_err(dZ.cpu().numpy(), zt.grad.numpy()) < 1e-5
    from oracle.torch_ref import first_argmax
    exp = (first_argmax(p.detach(), 1) == first_argmax(torch.tensor(y), 1)).float().numpy()
    np.testing.assert_array_equal(dc.cpu().numpy(), exp)


@pytest.mark.parametrize('B,ns', [(9, 2), (700, 3)])
def test_router_tail(B, ns):
    rng = np.random.default_rng(10)
    C = 16
    z1 = rng.standard_normal((B, C)).astype(np.float32)
    P = {k: rng.standard_normal(s).astype(np.float32) * sc for k, s, sc in [
        ('g1', C, 1), ('b1', C, .3), ('W2', (C, C), .3), ('c2', C, .1), ('g2', C, 1), ('b2', C, .3),
        ('W3', (C, ns), .3), ('c3', ns, .1)]}
    D = {k: dev(v) for k, v in P.items()}
    m1 = torch.zeros(C, device='cuda'); v1 = torch.ones(C, device='cuda')
    m2 = torch.zeros(C, device='cuda'); v2 = torch.ones(C, device='cuda')
    Z1 = dev(z1); Z2 = torch.zeros((B, C), device='cuda'); R = torch.zeros((B, ns), device='cuda')
    save = torch.zeros(64, device='cuda')
    L().router_tail_fwd(vp(Z1), B, C, vp(D['g1']), vp(D['b1']), vp(m1), vp(v1), vp(D['W2']), vp(D['c2']),
                        vp(D['g2']), vp(D['b2']), vp(m2), vp(v2), vp(D['W3']), vp(D['c3']), ns, 0.9, 1e-6, 1,
                        vp(Z2), vp(R), vp(save), None)
    T = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in P.items()}
    zt = torch.tensor(z1, dtype=torch.float64, requires_grad=True)

    def bn(x, g, b):
        m = x.mean(0); v = ((x - m) ** 2).mean(0)
        return g * (x - m) / torch.sqrt(v + 1e-6) + b, m, v
    h1, mm1, vv1 = bn(zt, T['g1'], T['b1'])
    z2 = torch.relu(h1) @ T['W2'] + T['c2']
    h2, mm2, vv2 = bn(z2, T['g2'], T['b2'])
    r = torch.relu(h2) @ T['W3'] + T['c3']
    torch.cuda.synchronize()
    assert rel_err(R.cpu().numpy(), r.detach().numpy()) < 1e-4
    np.testing.assert_allclose(v2.cpu().numpy(), 0.9 + 0.1 * vv2.detach().numpy(), rtol=1e-4)
    dr = rng.standard_normal((B, ns)).astype(np.float32)
    (r * torch.tensor(dr, dtype=torch.float64)).sum().backward()
    G = {k: torch.zeros_like(D[k]) for k in P}
    dZ1 = torch.zeros((B, C), device='cuda'); scratch = torch.zeros(2 * B * C, device='cuda')
    L().router_tail_bwd(vp(Z1), vp(Z2), vp(dev(dr)), B, C, ns, vp(D['g1']), vp(D['b1']), vp(D['W2']),
                        vp(D['g2']), vp(D['b2']), vp(D['W3']), vp(save),
                        vp(G['g1']), vp(G['b1']), vp(G['W2']), vp(G['c2']), vp(G['g2']), vp(G['b2']),
                        vp(G['W3']), vp(G['c3']), vp(dZ1), vp(scratch), None)
    torch.cuda.synchronize()
    assert rel_err(dZ1.cpu().numpy(), zt.grad.numpy()) < 2e-4
    for k in P:
        if k == 'c2':       # a bias in front of train-mode BN has zero gradient
            assert np.abs(G[k].cpu().numpy()).max() < 1e-4 * np.abs(G['c3'].cpu().numpy()).max()
            continue
        assert rel_err(G[k].cpu().numpy(), T[k].grad.numpy()) < 2e-4, k


@pytest.mark.parametrize('train', [1, 0])
@pytest.mark.parametrize('B', [24, 128, 1000, 2048 + 77, 4096, 5000, 9000])
def test_router_tail_fwd_batched_matches_single(B, train):
    """cluster forward (8 CTAs per router, two-pass moments through DSMEM; rows resident in registers, 1 / 2 / 4 per
    thread, up to B = 8192, the re-reading kernel beyond) against the single-CTA kernel"""
    from lib.engine import _RT_FWD
    rng = np.random.default_rng(13)
    C = 16
    rows, cases = [], []
    for ns in (2, 5, 8):
        Z1 = dev(rng.standard_normal((B, C)).astype(np.float32) * 2 + 0.3)
        P = {k: dev(rng.standard_normal(sh).astype(np.float32) * sc) for k, sh, sc in [
            ('g1', C, 1), ('b1', C, .3), ('W2', (C, C), .3), ('c2', C, .1), ('g2', C, 1), ('b2', C, .3),
            ('W3', (C, ns), .3), ('c3', ns, .1)]}
        outs = []
        for which in range(2):
            st = [dev(rng.standard_normal(C).astype(np.float32) * 0 + 0.1), dev(np.full(C, 1.5, np.float32)),
                  dev(np.full(C, -0.2, np.float32)), dev(np.full(C, 0.7, np.float32))]
            outs.append(dict(st=st, Z2=torch.zeros((B, C), device='cuda'), R=torch.zeros((B, ns), device='cuda'),
                             save=torch.zeros(64, device='cuda')))
        o = outs[0]
        L().router_tail_fwd(vp(Z1), B, C, vp(P['g1']), vp(P['b1']), vp(o['st'][0]), vp(o['st'][1]), vp(P['W2']), vp(P['c2']),
                            vp(P['g2']), vp(P['b2']), vp(o['st'][2]), vp(o['st'][3]), vp(P['W3']), vp(P['c3']), ns,
                            0.9, 1e-6, train, vp(o['Z2']), vp(o['R']), vp(o['save']), None)
        o = outs[1]
        ptr = lambda t: t.data_ptr()
        rows.append((ptr(Z1), ptr(P['g1']), ptr(P['b1']), ptr(o['st'][0]), ptr(o['st'][1]), ptr(P['W2']), ptr(P['c2']),
                     ptr(P['g2']), ptr(P['b2']), ptr(o['st'][2]), ptr(o['st'][3]), ptr(P['W3']), ptr(P['c3']),
                     ptr(o['Z2']), ptr(o['R']), ptr(o['save']), ns, 0))
        cases.append(outs)
    table = dev(np.frombuffer(np.array(rows, dtype=_RT_FWD).tobytes(), np.uint8).copy(), torch.uint8)
    L().router_tail_fwd_batched(vp(table), len(rows), B, C, 0.9, 1e-6, train, None)
    torch.cuda.synchronize()
    for ref, got in cases:
        for k in ('Z2', 'R', 'save'):
            assert rel_err(got[k].cpu().numpy(), ref[k].cpu().numpy()) < 1e-5, k
        for a, b in zip(ref['st'], got['st']):
            np.testing.assert_allclose(b.cpu().numpy(), a.cpu().numpy(), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize('B', [24, 128, 1000, 2048 + 77, 4096, 5000])
def test_router_tail_bwd_batched_matches_single(B):
    """The one-launch cluster kernel (8 CTAs per router, DSMEM reductions) against the
    single-CTA kernel validated above; routers of different fan-out in the same launch."""
    from lib.engine import _RT_BWD
    rng = np.random.default_rng(12)
    C = 16
    Balloc = -(-B // 128) * 128
    cases, rows = [], []
    for ns in (2, 5, 8):
        z1 = rng.standard_normal((B, C)).astype(np.float32)
        P = {k: dev(rng.standard_normal(sh).astype(np.float32) * sc) for k, sh, sc in [
            ('g1', C, 1), ('b1', C, .3), ('W2', (C, C), .3), ('c2', C, .1), ('g2', C, 1), ('b2', C, .3),
            ('W3', (C, ns), .3), ('c3', ns, .1)]}
        st = [torch.zeros(C, device='cuda'), torch.ones(C, device='cuda'), torch.zeros(C, device='cuda'),
              torch.ones(C, device='cuda')]
        Z1 = dev(z1); Z2 = torch.zeros((B, C), device='cuda'); R = torch.zeros((B, ns), device='cuda')
        save = torch.zeros(64, device='cuda')
        L().router_tail_fwd(vp(Z1), B, C, vp(P['g1']), vp(P['b1']), vp(st[0]), vp(st[1]), vp(P['W2']), vp(P['c2']),
                            vp(P['g2']), vp(P['b2']), vp(st[2]), vp(st[3]), vp(P['W3']), vp(P['c3']), ns, 0.9, 1e-6, 1,
                            vp(Z2), vp(R), vp(save), None)
        dR = dev(rng.standard_normal((B, ns)).astype(np.float32))
        ref = {k: torch.zeros_like(P[k]) for k in P}
        ref['dZ1'] = torch.zeros((B, C), device='cuda')
        scratch = torch.zeros(2 * B * C, device='cuda')
        L().router_tail_bwd(vp(Z1), vp(Z2), vp(dR), B, C, ns, vp(P['g1']), vp(P['b1']), vp(P['W2']),
                            vp(P['g2']), vp(P['b2']), vp(P['W3']), vp(save),
                            vp(ref['g1']), vp(ref['b1']), vp(ref['W2']), vp(ref['c2']), vp(ref['g2']), vp(ref['b2']),
                            vp(ref['W3']), vp(ref['c3']), vp(ref['dZ1']), vp(scratch), None)
        got = {k: torch.zeros_like(P[k]) for k in P}
        got['dZ1'] = torch.zeros((B, C), device='cuda')
        got['dZ1p'] = torch.zeros((2, Balloc, 8), dtype=torch.bfloat16, device='cuda')
        got['c1'] = torch.zeros(C, device='cuda')
        ptr = lambda t: t.data_ptr()
        rows.append((ptr(Z1), ptr(Z2), ptr(dR), ptr(P['g1']), ptr(P['b1']), ptr(P['W2']), ptr(P['g2']), ptr(P['b2']),
                     ptr(P['W3']), ptr(save), ptr(got['g1']), ptr(got['b1']), ptr(got['W2']), ptr(got['c2']),
                     ptr(got['g2']), ptr(got['b2']), ptr(got['W3']), ptr(got['c3']), ptr(got['dZ1']), 0,
                     ptr(got['dZ1p']), ptr(got['c1']), ns, Balloc))
        cases.append((ref, got, (Z2, R, save, scratch, st)))     # keep every buffer alive until the batched launch
    table = dev(np.frombuffer(np.array(rows, dtype=_RT_BWD).tobytes(), np.uint8).copy(), torch.uint8)
    L().router_tail_bwd_batched(vp(table), len(rows), B, C, None)
    torch.cuda.synchronize()
    for ref, got, _ in cases:
        for k in ref:
            a, b = got[k].cpu().numpy(), ref[k].cpu().numpy()
            if k == 'c2':          # zero gradient (bias in front of train-mode BN): both are rounding noise
                assert np.abs(a).max() < 1e-4 * np.abs(ref['c3'].cpu().numpy()).max()
                continue
            assert rel_err(a, b) < 2e-5, (k, [(kk, float(rel_err(got[kk].cpu().numpy(), ref[kk].cpu().numpy()))) for kk in ref])
        planes = got['dZ1p'].float().cpu().numpy()
        flat = np.concatenate([planes[0, :B], planes[1, :B]], 1)
        assert rel_err(flat, ref['dZ1'].cpu().numpy()) < 4e-3 and np.all(planes[:, B:] == 0)
        assert np.abs(got['c1'].cpu().numpy()).max() < 1e-3      # column sums of dZ1 vanish under train-mode BN


# --------------------------------------------------------------------------- #
# compaction / gather / scatter / optimiser
# --------------------------------------------------------------------------- #
def test_compact_gather_scatter():
    rng = np.random.default_rng(11)
    nn, B = 5, 2500
    pe = (rng.random((nn, B)) < np.array([1.0, 0.5, 0.02, 0.0, 0.9])[:, None]).astype(np.float32)
    PE = dev(pe)
    idx = torch.full((nn, B), -1, dtype=torch.int32, device='cuda'); cnt = torch.zeros(nn, dtype=torch.int32, device='cuda')
    L().compact_paths(vp(PE), nn, B, vp(idx), vp(cnt), None)
    torch.cuda.synchronize()
    for i in range(nn):
        want = np.nonzero(pe[i])[0]
        assert int(cnt[i]) == len(want)
        np.testing.assert_array_equal(idx[i, :len(want)].cpu().numpy(), want)      # bit-exact, order preserving
    # gather images of node 1 and scatter them back
    Bs, H, C = 64, 4, 16
    x = rng.standard_normal((Bs, H, H, C)).astype(np.float32)
    sel = np.sort(rng.choice(Bs, 20, replace=False)).astype(np.int32)
    gs, gd = Geo(Bs, H, H), Geo(32, H, H)
    for dt, td in ((F32, torch.float32), (BF16, torch.bfloat16)):
        rd = (lambda a: a) if dt == F32 else bf16_round
        X = dev(to_planes(rd(x), gs), td)
        I = dev(sel); N = dev(np.array([len(sel)], np.int32))
        Y = torch.zeros((C // 8, gd.P, 8), dtype=td, device='cuda')
        L().gather_images(vp(X), Bs, gs.P, vp(I), vp(N), vp(Y), 32, gd.P, C, H, H, gs.G, dt, None)
        torch.cuda.synchronize()
        got = from_planes(Y.float().cpu().numpy(), gd, C)
        np.testing.assert_array_equal(got[:len(sel)], rd(x)[sel])
        Zt = torch.zeros_like(X)
        L().scatter_add_images(vp(Y), 32, gd.P, vp(I), vp(N), vp(Zt), Bs, gs.P, C, H, H, gs.G, dt, None)
        torch.cuda.synchronize()
        back = from_planes(Zt.float().cpu().numpy(), gs, C)
        exp = np.zeros_like(x); exp[sel] = rd(x)[sel]
        np.testing.assert_array_equal(back, exp)


def test_talr_momentum_step():
    rng = np.random.default_rng(12)
    sizes = [7, 100, 33, 1, 500]
    n = sum(sizes)
    th = rng.standard_normal(n).astype(np.float32); g = rng.standard_normal(n).astype(np.float32)
    a = rng.standard_normal(n).astype(np.float32)
    start = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    node = np.array([0, 1, 1, 2, 2], np.int32); mult = np.array([1, 1, 2, 1, .5], np.float32)
    l2 = np.array([0, 1e-4, 0, 1e-4, 0], np.float32)
    stats = np.array([[1.0, 1.0], [0.25, 0.4], [1e-6, 1e-3]], np.float32)
    hyp = np.zeros(8, np.float32); hyp[0] = 0.1; hyp[1] = 0.9; hyp[5] = 0.5
    TH, A = dev(th), dev(a)
    # moments ride in the all-reduced tail: kernel multiplies them by gscale too
    L().talr_momentum_step(vp(TH), vp(dev(g)), vp(A), n, vp(dev(start)), vp(dev(node)), vp(dev(mult)), vp(dev(l2)),
                           5, vp(dev(stats / 0.5)), 1, vp(dev(hyp)), None)
    torch.cuda.synchronize()
    exp_th, exp_a = th.astype(np.float64).copy(), a.astype(np.float64).copy()
    for s in range(5):
        sl = slice(start[s], start[s + 1])
        gg = g[sl] * 0.5 + 2 * l2[s] * stats[node[s], 1] * th[sl]
        gg = gg * mult[s] / np.sqrt(stats[node[s], 0])
        exp_a[sl] = 0.9 * a[sl] + gg
        exp_th[sl] = th[sl] - 0.1 * exp_a[sl]
    np.testing.assert_allclose(A.cpu().numpy(), exp_a, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(TH.cpu().numpy(), exp_th, rtol=1e-5, atol=1e-6)


# --------------------------------------------------------------------------- #
# routing walk: forward products and backward (actor / critic) vs autograd
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('kind,hy', [('ac', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=1e-7)),
                                     ('cr', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9, optimistic=True))])
def test_route_fwd_bwd(kind, hy):
    from util import tiny_net
    B, tau, eps = 50, 0.6, 1e-6
    net = tiny_net(kind, **hy).configure(precision='fp32')
    eng = net._get_engine()
    plan = eng._plan(B, True, True)
    rng = np.random.default_rng(13)
    critic = kind == 'cr'
    nodes = eng.nodes
    Rs = {}
    for nd in eng.switches:
        r = rng.standard_normal((B, len(nd.kids))).astype(np.float32)
        plan.rtr[nd.idx].R.copy_(torch.from_numpy(r)); Rs[nd.idx] = r
    ce = {}
    for nd in eng.regs:
        c = (rng.random(B) * 3).astype(np.float32)
        plan.reg[nd.idx].c_err.copy_(torch.from_numpy(c)); ce[nd.idx] = c
    hyp = np.zeros(8, np.float32); hyp[2] = tau; hyp[3] = eps; hyp[4] = hy['k_cpt']
    eng.hyp.copy_(torch.from_numpy(hyp))
    eng.stream = None
    plan.fwd_ops[-1]()          # route_fwd
    plan.bwd_ops[0]()           # route_bwd
    torch.cuda.synchronize()
    # ---- float64 reference from the plan's tables (actor dR by autograd)
    from util import route_ref, tree_tables
    ref = route_ref(tree_tables(plan), [torch.from_numpy(Rs[nd.idx]) for nd in eng.switches], tau, eps,
                    c_err=[torch.from_numpy(ce[nd.idx]) for nd in eng.regs], k_cpt=hy['k_cpt'], critic=critic,
                    k_dec=0.0 if critic else 0.01, k_cre=1e-3 if critic else 0.0,
                    optimistic=bool(hy.get('optimistic')))
    got_ptr = plan.p_tr.cpu().numpy()
    for nd in nodes:
        np.testing.assert_allclose(got_ptr[nd.idx], ref['p_tr'][nd.idx].numpy(), rtol=2e-5, atol=1e-9)
        np.testing.assert_array_equal(plan.p_ev.cpu().numpy()[nd.idx], ref['p_ev'][nd.idx].numpy())
    np.testing.assert_allclose(plan.c_data.cpu().numpy(), ref['c_data'].numpy(), rtol=2e-5)
    for s, nd in enumerate(eng.switches):
        got = plan.rtr[nd.idx].dR.cpu().numpy()
        assert rel_err(got, ref['dR'][s].numpy()) < 1e-4, nd.idx


# --------------------------------------------------------------------------- #
# fully-connected heads on the tensor cores (ntaps = 1, K streamed in slices)
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('B,F,n_cls,dyn', [(40, 256, 10, False), (300, 2048, 10, True), (129, 512, 2, False)])
def test_fc_heads_umma(B, F, n_cls, dyn):
    rng = np.random.default_rng(14)
    Balloc = (B + 127) // 128 * 128
    Fext = F + (16 if dyn else 0)
    x = bf16_round(rng.standard_normal((B, F)).astype(np.float32))
    kx = bf16_round(rng.random(B).astype(np.float32)) if dyn else None
    Wl = (rng.standard_normal((F, n_cls)) / 10).astype(np.float32)
    Wr = (rng.standard_normal((F + (1 if dyn else 0), 16)) / 10).astype(np.float32)
    bl = rng.standard_normal(n_cls).astype(np.float32); br = rng.standard_normal(16).astype(np.float32)
    X = np.zeros((Fext // 8, Balloc, 8), np.float32)
    for i in range(F // 8):
        X[i, :B] = x[:, i * 8:(i + 1) * 8]
    if dyn:
        X[F // 8, :B, 0] = kx
    X = dev(X, torch.bfloat16)
    # pack [W_leaf | W_r1] and the bias vector with the batched packer
    Wfc = torch.zeros((1, Fext // 8, 32, 8), dtype=torch.bfloat16, device='cuda')
    bias = torch.zeros(32, device='cuda')
    dWl, dWr, dbl, dbr = dev(Wl), dev(Wr), dev(bl), dev(br)
    desc = np.zeros(4, dtype=np.dtype([('w', '<u8'), ('packed', '<u8')] + [(k, '<i4') for k in (
        'ntaps', 'I', 'O', 'mode', 'k_off', 'Ktot', 'n_off', 'Ntot')], align=True))
    desc[0] = (dWl.data_ptr(), Wfc.data_ptr(), 1, F, n_cls, 0, 0, Fext, 0, 32)
    desc[1] = (dWr.data_ptr(), Wfc.data_ptr(), 1, Wr.shape[0], 16, 0, 0, Fext, 16, 32)
    desc[2] = (dbl.data_ptr(), bias.data_ptr(), 1, 1, n_cls, 2, 0, 8, 0, 32)
    desc[3] = (dbr.data_ptr(), bias.data_ptr(), 1, 1, 16, 2, 0, 8, 16, 32)
    D = dev(desc.view(np.uint8))
    L().pack_weights_batched(vp(D), 4, 8, BF16, None)
    Z16 = torch.zeros((B, 16), device='cuda'); Z1 = torch.zeros((B, 16), device='cuda')
    L().stencil_gemm(vp(X), Fext, None, 0, vp(Wfc), 1, vp(bias), vp(Z16), 16, 0, vp(Z1), 16, 0,
                     B, 0, 0, 0, Balloc, None, 0, None, BF16, 2, 1, None)
    torch.cuda.synchronize()
    xf = np.concatenate([x, kx[:, None]], 1) if dyn else x
    ref_l = x.astype(np.float64) @ bf16_round(Wl) + bl
    ref_r = xf.astype(np.float64) @ bf16_round(Wr) + br
    assert rel_err(Z16.cpu().numpy()[:, :n_cls], ref_l) < 1e-4
    assert rel_err(Z1.cpu().numpy(), ref_r) < 1e-4
    # backward: dZ planes [4][Balloc][8]
    dz = bf16_round(rng.standard_normal((B, 32)).astype(np.float32))
    dz[:, n_cls:16] = 0
    P = np.zeros((4, Balloc, 8), np.float32)
    for i in range(4):
        P[i, :B] = dz[:, i * 8:(i + 1) * 8]
    P = dev(P, torch.bfloat16)
    gWl = torch.zeros_like(dWl); gWr = torch.zeros_like(dWr)
    L().fc_wgrad(vp(X), Fext, Balloc, B, vp(P), 32, 16, vp(gWl), F, n_cls, vp(gWr), Wr.shape[0], 16, None)
    torch.cuda.synchronize()
    assert rel_err(gWl.cpu().numpy(), x.astype(np.float64).T @ dz[:, :n_cls]) < 1e-4
    assert rel_err(gWr.cpu().numpy(), xf.astype(np.float64).T @ dz[:, 16:]) < 1e-4
    Wfd = torch.zeros((1, 4, F, 8), dtype=torch.bfloat16, device='cuda')
    desc2 = desc[:2].copy()
    desc2[0] = (dWl.data_ptr(), Wfd.data_ptr(), 1, F, n_cls, 1, 0, 32, 0, F)
    desc2[1] = (dWr.data_ptr(), Wfd.data_ptr(), 1, F, 16, 1, 16, 32, 0, F)
    D2 = dev(desc2.view(np.uint8))
    L().pack_weights_batched(vp(D2), 2, 8, BF16, None)
    dX = torch.zeros((F // 8, Balloc, 8), dtype=torch.bfloat16, device='cuda')
    L().stencil_gemm(vp(P), 32, None, 0, vp(Wfd), 1, None, vp(dX), F, 0, None, 0, 0,
                     B, 0, 0, 0, Balloc, None, 0, None, BF16, BF16, 1, None)
    torch.cuda.synchronize()
    f = dX.float().cpu().numpy()
    got = np.concatenate([f[i, :B] for i in range(F // 8)], 1)
    ref = dz[:, :n_cls].astype(np.float64) @ bf16_round(Wl).T + dz[:, 16:].astype(np.float64) @ bf16_round(Wr[:F]).T
    assert rel_err(got, ref) < 4e-3


def test_gpu_augmentation_reproduces_the_numpy_batches():
    """csrc/augment.cu against lib/data.py (itself a restatement of scripts/lib/data.py:24-34) with the
    same seeded sampler: copied pixels bit-exact, mean fill to fp32 rounding, labels exact."""
    from lib.data import Dataset, synthetic_archive
    arch = synthetic_archive(300, 10, (32, 32, 3), 10)
    arch['m_sym'] = np.array([True, False] * 5)
    arch['x0_tr'] = arch['x0_tr'].astype(np.float32).astype(np.float64)    # fp32-representable pixels, as in the real archives
    a, b = Dataset(archive=arch, seed=11), Dataset(archive=arch, seed=11)
    for n in (1, 37, 256):
        xc, yc = a.augmented_training_batch(n)
        xg, yg = b.augmented_training_batch_gpu(n)
        torch.cuda.synchronize()
        xg, yg = xg.cpu().numpy(), yg.cpu().numpy()
        np.testing.assert_array_equal(yg, yc.astype(np.float32))
        xc32 = xc.astype(np.float32)
        same = xg == xc32
        assert same.mean() > 0.9999                             # everything but (possibly) a fill value on a rounding tie
        np.testing.assert_allclose(xg, xc32, rtol=2e-7, atol=0)
