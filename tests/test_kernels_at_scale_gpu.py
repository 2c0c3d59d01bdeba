"""Kernel parity at the benchmark's batch (B200): libmpnn_sm100 entry points, called through the C ABI at
B = 4096 and the ragged 4095 / 4097 on the real architecture's stages (32x32x16 .. 4x4x128), against float64
references computed on the device with plain torch.

At these sizes the grid-stride loops run their second and later passes, the BN statistics are the two-pass
(not the one-launch) kernels, the head GEMMs see a partly-filled 128-row tile, and every reduction is thousands
of times longer than in test_kernels_gpu.py.  Tolerances are derived in each docstring; u = 2^-24 is the fp32
unit roundoff.  Run with -s to see the measured errors."""
import ctypes
import functools
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from util import (Geo, dropout_mask_t, from_feat_t, from_planes_t, pad_tree, random_tree, route_ref, to_feat_t,
                  to_planes_t, tree_tables)

pytestmark = pytest.mark.gpu

F32, BF16 = 0, 1
TD = {F32: torch.float32, BF16: torch.bfloat16}
U = 2.0 ** -24
EPS = 1e-6                      # the BatchNorm epsilon of lib/layer_types.py
BATCHES = (4095, 4096, 4097)


def L():
    from lib import _cabi
    return _cabi.lib()


def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def ru(a, b):
    return -(-a // b) * b


def gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def rnd(g, shape, dt, scale=1.0, shift=0.0):
    """fp32 normal samples on the device, rounded to the operand type (so an fp64 reference of them is exact)"""
    x = torch.randn(shape, generator=g, device='cuda') * scale + shift
    return x if dt == F32 else x.to(torch.bfloat16).float()


def ints(g, shape, lo, hi):
    """small integers as fp32: exact in bf16, and ties in every max-pool window"""
    return torch.randint(lo, hi, shape, generator=g, device='cuda').float()


def err(got, ref):
    return float(rel_err_t(got, ref))


def rel_err_t(a, b):
    a, b = a.double(), b.double()
    n = torch.linalg.vector_norm(b)
    d = torch.linalg.vector_norm(a - b)
    return d / n if n > 0 else d


def conv3_ref(x, w):
    """3x3 'same' cross-correlation in float64 on the device, as nine shifted matmuls: x (B,H,W,C), w (3,3,C,O)"""
    B, H, W, C = x.shape
    xp = Fn.pad(x.double(), (0, 0, 1, 1, 1, 1))
    y = torch.zeros((B * H * W, w.shape[3]), dtype=torch.float64, device='cuda')
    w = w.double()
    for t in range(9):
        y += xp[:, t // 3:t // 3 + H, t % 3:t % 3 + W].reshape(-1, C) @ w[t // 3, t % 3]
    return y.view(B, H, W, -1)


def pack(w, Ktot, k_off, Ntot, packed, dt):
    """(3,3,I,O) fp32 device weights -> packed [9][Ktot/8][Ntot][8] (mode 0)"""
    w = w.contiguous()
    L().pack_weights(vp(w), 9, w.shape[2], w.shape[3], 0, k_off, Ktot, 0, Ntot, vp(packed), dt, None)


def conv_operands(x, xp, w, wv, dt):
    B, H, W, Cin = x.shape
    Cp, Cout = (xp.shape[3] if xp is not None else 0), w.shape[3]
    geo = Geo(B, H, W)
    K0 = ru(Cin, 16 if dt == BF16 else 8)
    A0 = to_planes_t(x, geo, K0).to(TD[dt])
    A1 = to_planes_t(xp, geo).to(TD[dt]) if Cp else None
    Wp = torch.zeros((9, (K0 + Cp) // 8, Cout, 8), dtype=TD[dt], device='cuda')
    pack(w, K0 + Cp, 0, Cout, Wp, dt)
    if Cp:
        pack(wv, K0 + Cp, K0, Cout, Wp, dt)
    return geo, K0, Cp, A0, A1, Wp


def bn_fuse(N, count, defer=0, gamma=None, beta=None):
    """mpnn_bn_fuse host struct + the device buffers it points to (kept in the returned dict)"""
    from lib.engine import _BN_FUSE, _host_struct
    b = dict(acc=torch.zeros(2 * N + 2, dtype=torch.float64, device='cuda'),
             gamma=gamma if gamma is not None else torch.ones(N, device='cuda'),
             beta=beta if beta is not None else torch.zeros(N, device='cuda'),
             m_avg=torch.zeros(N, device='cuda'), v_avg=torch.ones(N, device='cuda'),
             ss=torch.zeros((2, N), device='cuda'), mr=torch.zeros((2, N), device='cuda'))
    f = _host_struct(_BN_FUSE, **{k: vp(v) for k, v in b.items()}, count=float(count), d=0.9, eps=EPS, defer=defer)
    b['f'] = f
    return b, ctypes.c_void_p(f.ctypes.data)


def moments_ref(y):
    """two-pass float64 mean and variance over all but the channel axis"""
    y = y.reshape(-1, y.shape[-1]).double()
    m = y.mean(0)
    return m, ((y - m) ** 2).mean(0)


# --------------------------------------------------------------------------- #
# conv forward: outputs and BN sums
# --------------------------------------------------------------------------- #
CONV_SHAPES = [(32, 16, 16, 16), (16, 32, 32, 32), (8, 64, 64, 64), (4, 128, 0, 128)]


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('dt,impl', [(F32, 0), (BF16, 1)])
@pytest.mark.parametrize('H,Cin,Cp,Cout', CONV_SHAPES)
def test_conv_forward_and_statistics_at_scale(B, dt, impl, H, Cin, Cp, Cout):
    """mpnn_stencil_gemm (pooled second input, per-CTA sums) and mpnn_conv_bn_stats (fused "last CTA finalises")
    against the float64 conv of the same operands.  Outputs: fp32 1e-5 (dot products of 9(Cin+Cp) <= 1152 terms,
    probabilistic fp32 error ~ sqrt(1152) u = 2e-6), bf16 4e-3 (stored in bf16: 2^-9 per element).  Sums: each
    is an fp32 sum whose longest chain is the tiles of one CTA (<= ceil(tiles / 148)) plus the warp / CTA trees
    (16), fed by conv values that carry 9(Cin+Cp) fp32 additions each: the recursive-summation bound gamma_n with
    n = that depth, |d sum y| <= n u sum|y| and |d sum y^2| <= 2 n u sum y^2.  The fused path's mean and rstd are
    held to the same bound, carried through var = E[y^2] - mean^2."""
    g = gen(1000 + H + B + 7 * impl)
    x = rnd(g, (B, H, H, Cin), dt)
    xp = rnd(g, (B, H, H, Cp), dt) if Cp else None
    w = rnd(g, (3, 3, Cin, Cout), dt, 1 / math.sqrt(9 * Cin))
    wv = rnd(g, (3, 3, Cp, Cout), dt, 1 / math.sqrt(9 * Cp)) if Cp else None
    bias = torch.randn(Cout, generator=g, device='cuda')
    geo, K0, Cp, A0, A1, Wp = conv_operands(x, xp, w, wv, dt)
    out = torch.zeros((Cout // 8, geo.P, 8), dtype=TD[dt], device='cuda')
    stats = torch.zeros(592 * 2 * Cout, device='cuda')
    cnt = ctypes.c_int(0)
    L().stencil_gemm(vp(A0), K0, vp(A1), Cp, vp(Wp), 9, vp(bias), vp(out), Cout, 0, None, 0, 0,
                     B, H, H, geo.G, geo.P, vp(stats), 592, ctypes.byref(cnt), dt, dt, impl, None)
    count = B * H * H
    b, fp = bn_fuse(Cout, count)
    out2 = torch.zeros_like(out)
    L().conv_bn_stats(vp(A0), K0, vp(A1), Cp, vp(Wp), vp(bias), vp(out2), Cout, B, H, H, geo.G, geo.P, fp, dt, impl, None)
    torch.cuda.synchronize()
    ref = conv3_ref(x, w) + bias.double()
    if Cp:
        ref += conv3_ref(xp, wv)
    e = err(from_planes_t(out, geo, Cout), ref)
    assert torch.equal(out, out2)
    st = stats[:cnt.value * 2 * Cout].view(cnt.value, 2, Cout).double().sum(0)
    n = -(-ru(geo.rows, 128) // 128 // 148) + 16 + 9 * (Cin + Cp)
    r2 = ref.reshape(-1, Cout)
    e1 = ((st[0] - r2.sum(0)).abs() / (r2.abs().sum(0))).max().item()
    e2 = ((st[1] - (r2 ** 2).sum(0)).abs() / (r2 ** 2).sum(0)).max().item()
    m, v = moments_ref(r2)
    em = ((b['mr'][0].double() - m).abs() / r2.abs().mean(0)).max().item()
    rstd = 1 / torch.sqrt(v + EPS)
    er = ((b['mr'][1].double() - rstd).abs() / rstd).max().item()
    tol_r = 3 * n * U * ((r2 ** 2).mean(0) / (v + EPS)).max().item() + 4 * U
    tol_o = 1e-5 if dt == F32 else 4e-3
    print('conv B=%d H=%d %s: out %.2e (tol %.0e), sum %.2e (tol %.1e), sum sq %.2e (tol %.1e), '
          'fused mean %.2e (tol %.1e), rstd %.2e (tol %.1e)'
          % (B, H, 'fp32' if dt == F32 else 'bf16', e, tol_o, e1, n * U, e2, 2 * n * U, em, n * U + U, er, tol_r))
    assert e < tol_o
    assert e1 <= n * U and e2 <= 2 * n * U
    assert em <= n * U + U and er <= tol_r
    assert float(b['acc'].abs().max()) == 0.0                 # self-cleaned for the next launch


# --------------------------------------------------------------------------- #
# BN -> ReLU -> (pool | flatten), forward and backward, two-pass kernels
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('H,C,pool', [(32, 16, True), (8, 64, True), (16, 32, False), (4, 128, False)])
def test_bn_relu_pool_fwd_bwd_at_scale(B, dt, H, C, pool):
    """mpnn_bn_finalize (592 partial rows, as many as a conv writes) + mpnn_bn_relu_pool_fwd with pooled or
    flattened-feature output, then mpnn_bn_bwd_reduce + mpnn_bn_bwd_finalize, mpnn_bn_bwd_reduce_fused and
    mpnn_bn_relu_pool_bwd, against float64 autograd of BN -> ReLU -> max-pool (as test_bn_relu_pool_fwd_bwd).
    Activations and dLin: fp32 1e-4 (the per-channel sums are fp32 chains of <= ~40 terms per thread plus the
    trees, ~1e-6 relative; the rest is elementwise), bf16 4e-3 (stored in bf16, 2^-9).  Pooled values: exact.
    Two-pass vs fused backward sums: the bounds of test_fused_bn_statistics_match_the_two_launch_path.  dbias
    (column sums of dLin): |d| <= 1e-5 sum|dLin| in fp32, 2^-9 sum|dLin| in bf16 (each summand is the stored value).
    dLin is compared away from the ReLU kink: where the float64 pre-activation is within 1e-5 of zero, the kernel's
    fp32 gate (the reference network's own arithmetic) may fall on the other side and pass or drop an O(1)
    gradient; at 67 M elements that happens a few times per tensor."""
    g = gen(2000 + B + H + dt)
    geo, gp = Geo(B, H, H), Geo(B, H // 2, H // 2)
    Balloc = ru(B, 128)
    lin = rnd(g, (B, H, H, C), dt, 2.0, 0.5)
    gamma = torch.randn(C, generator=g, device='cuda')
    beta = 0.1 * torch.randn(C, generator=g, device='cuda')
    LIN = to_planes_t(lin, geo).to(TD[dt])
    parts = torch.stack([torch.stack([p.double().sum((0, 1, 2)), (p.double() ** 2).sum((0, 1, 2))])
                         for p in torch.tensor_split(lin, 592)]).float().contiguous()
    ss = torch.zeros((2, C), device='cuda'); mr = torch.zeros((2, C), device='cuda')
    m_avg = torch.zeros(C, device='cuda'); v_avg = torch.ones(C, device='cuda')
    count = float(B * H * H)
    L().bn_finalize(vp(parts), 592, C, count, vp(gamma), vp(beta), vp(m_avg), vp(v_avg), 0.9, EPS, 1, vp(ss), vp(mr), None)
    act = torch.zeros_like(LIN)
    pooled = torch.zeros((C // 8, gp.P, 8), dtype=TD[dt], device='cuda') if pool else None
    feat = None if pool else torch.zeros((H * H * C // 8, Balloc, 8), dtype=TD[dt], device='cuda')
    L().bn_relu_pool_fwd(vp(LIN), C, B, H, H, geo.G, geo.P, vp(ss), vp(act), vp(pooled), gp.P if pool else 0,
                         vp(feat), Balloc, dt, None)
    xt = lin.double().requires_grad_(True)
    m = xt.mean((0, 1, 2)); v = ((xt - m) ** 2).mean((0, 1, 2))
    yt = torch.relu(gamma.double() * (xt - m) / torch.sqrt(v + EPS) + beta.double())
    tol = 1e-4 if dt == F32 else 4e-3
    torch.cuda.synchronize()
    e_act = err(from_planes_t(act, geo, C), yt.detach())
    assert e_act < tol, e_act
    torch.testing.assert_close(m_avg.double(), 0.1 * m.detach(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(v_avg.double(), 0.9 + 0.1 * v.detach(), rtol=1e-5, atol=0)
    if pool:
        pt = Fn.max_pool2d(xt.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        assert torch.equal(from_planes_t(pooled, gp, C).double(), pt.detach())
        e_feat = 0.0
    else:
        f = from_feat_t(feat, B)
        e_feat = err(f, yt.detach().reshape(B, -1))
        assert e_feat < tol, e_feat
        assert not feat[:, B:].float().any()                          # rows past B untouched
    # backward
    dy = rnd(g, (B, H, H, C), dt)
    DY = to_planes_t(dy, geo).to(TD[dt])
    dp = rnd(g, (B, H // 2, H // 2, C), dt) if pool else None
    DP = to_planes_t(dp, gp).to(TD[dt]) if pool else None
    df = None if pool else rnd(g, (B, H * H * C), dt)
    DF = to_feat_t(df, Balloc).to(TD[dt]) if df is not None else None
    parts_b = torch.zeros(592 * 2 * C, device='cuda'); cnt = ctypes.c_int(0)
    L().bn_bwd_reduce(vp(LIN), vp(DY), vp(DF), Balloc, vp(ss), vp(mr), C, B, H, H, geo.G, geo.P,
                      vp(parts_b), 592, ctypes.byref(cnt), dt, None)
    sums = torch.zeros((2, C), device='cuda'); dg = torch.zeros(C, device='cuda'); dbt = torch.zeros(C, device='cuda')
    L().bn_bwd_finalize(vp(parts_b), cnt.value, C, vp(mr), vp(sums), vp(dg), vp(dbt), None)
    from lib.engine import _BN_BWD_FUSE, _host_struct
    acc = torch.zeros(2 * C + 1, dtype=torch.float64, device='cuda')
    sums_f = torch.zeros((2, C), device='cuda'); dg_f = torch.zeros(C, device='cuda'); db_f = torch.zeros(C, device='cuda')
    fb = _host_struct(_BN_BWD_FUSE, acc=vp(acc), sums=vp(sums_f), dgamma=vp(dg_f), dbeta=vp(db_f))
    L().bn_bwd_reduce_fused(vp(LIN), vp(DY), vp(DF), Balloc, vp(ss), vp(mr), C, B, H, H, geo.G, geo.P,
                            ctypes.c_void_p(fb.ctypes.data), dt, None)
    dlin = torch.zeros_like(LIN)
    dbias = torch.zeros(C, device='cuda')
    L().bn_relu_pool_bwd(vp(LIN), vp(DY), vp(DF), Balloc, vp(DP), gp.P if pool else 0, vp(ss), vp(mr), vp(sums),
                         count, C, B, H, H, geo.G, geo.P, vp(dlin), vp(dbias), dt, None)
    gtot = dy.double() + (df.double().view(B, H, H, C) if df is not None else 0)
    loss = (yt * gtot).sum()
    if pool:
        loss = loss + (pt * dp.double()).sum()
    loss.backward()
    torch.cuda.synchronize()
    scale = float(sums.abs().max())
    for a, b in ((sums, sums_f), (dg, dg_f), (dbt, db_f)):
        torch.testing.assert_close(b, a, rtol=2e-5, atol=2e-6 * scale)
    ref_dlin = xt.grad
    with torch.no_grad():
        kink = (gamma.double() * (xt - m) / torch.sqrt(v + EPS) + beta.double()).abs() < 1e-5
    got_dlin = from_planes_t(dlin, geo, C).double()
    e_dlin = err(got_dlin.masked_fill(kink, 0), ref_dlin.masked_fill(kink, 0))
    db_ref = ref_dlin.sum((0, 1, 2))
    db_tol = (1e-5 if dt == F32 else 2.0 ** -9) * ref_dlin.abs().sum((0, 1, 2))
    e_db = ((dbias.double() - db_ref).abs() / db_tol.clamp_min(1e-30)).max().item()
    print('bn B=%d H=%d C=%d %s %s: act %.2e, feat %.2e, dlin %.2e (tol %.0e each; %d elements at the kink), dbias %.2f of its bound'
          % (B, H, C, 'pool' if pool else 'feat', 'fp32' if dt == F32 else 'bf16', e_act, e_feat, e_dlin, tol,
             int(kink.sum()), e_db))
    assert e_dlin < tol, e_dlin
    assert bool(((dbias.double() - db_ref).abs() <= db_tol).all())
    assert float(acc.abs().max()) == 0.0


# --------------------------------------------------------------------------- #
# max-pool and global max-pool: exact, gradients to the first maximum
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('H,C', [(32, 16), (8, 64)])
def test_maxpool_and_global_maxpool_at_scale(B, dt, H, C):
    """mpnn_maxpool2_fwd/bwd and mpnn_global_maxpool_fwd/bwd on integer-valued inputs in [-3, 3] (exact in both
    types, ties in most windows): values, the flattened copy, argmax and both gradients must match exactly,
    the gradient going to the first maximum in window / row-major order."""
    g = gen(3000 + B + H + dt)
    geo, gp = Geo(B, H, H), Geo(B, H // 2, H // 2)
    Balloc = ru(B, 128)
    F = (H // 2) ** 2 * C
    x = ints(g, (B, H, H, C), -3, 4)
    X = to_planes_t(x, geo).to(TD[dt])
    out = torch.zeros((C // 8, gp.P, 8), dtype=TD[dt], device='cuda')
    feat = torch.zeros((F // 8, Balloc, 8), dtype=TD[dt], device='cuda')
    L().maxpool2_fwd(vp(X), C, B, H, H, geo.G, geo.P, vp(out), gp.P, vp(feat), Balloc, dt, None)
    blocks = x.view(B, H // 2, 2, H // 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(B, H // 2, H // 2, 4, C)
    ref, am = blocks.max(3).values, blocks.argmax(3)
    dout = ints(g, ref.shape, -4, 5)
    dfe = ints(g, (B, F), -4, 5)
    DOUT = to_planes_t(dout, gp).to(TD[dt]); DF = to_feat_t(dfe, Balloc).to(TD[dt])
    dx = torch.full_like(X, 7.0)                       # every valid row is written
    L().maxpool2_bwd(vp(X), vp(DOUT), vp(DF), Balloc, C, B, H, H, geo.G, geo.P, gp.P, vp(dx), dt, None)
    gf = torch.zeros((C // 8, Balloc, 8), dtype=TD[dt], device='cuda')
    arg = torch.zeros((C // 8, Balloc, 8), dtype=torch.int32, device='cuda')
    L().global_maxpool_fwd(vp(X), C, B, H, H, geo.G, geo.P, vp(gf), vp(arg), Balloc, dt, None)
    dgl = ints(g, (B, C), -4, 5)
    DG = to_feat_t(dgl, Balloc).to(TD[dt])
    dx2 = torch.full_like(X, 7.0)
    torch.cuda.synchronize()
    L().global_maxpool_bwd(vp(DG), vp(arg), Balloc, C, B, H, H, geo.G, geo.P, vp(dx2), dt, None)
    torch.cuda.synchronize()
    assert torch.equal(from_planes_t(out, gp, C).float(), ref)
    assert torch.equal(from_feat_t(feat, B).float(), ref.reshape(B, -1))
    d = dout + dfe.view(ref.shape)
    refdx = torch.zeros_like(blocks).scatter_(3, am.unsqueeze(3), d.unsqueeze(3))
    refdx = refdx.view(B, H // 2, H // 2, 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(B, H, H, C)
    assert torch.equal(from_planes_t(dx, geo, C).float(), refdx)
    xf = x.reshape(B, -1, C)
    assert torch.equal(from_feat_t(gf, B).float(), xf.max(1).values)
    garg = xf.argmax(1)
    assert torch.equal(from_feat_t(arg, B).long(), garg)
    ref2 = torch.zeros_like(xf).scatter_(1, garg.unsqueeze(1), dgl.unsqueeze(1))
    assert torch.equal(from_planes_t(dx2, geo, C).float(), ref2.view(B, H, H, C))
    print('maxpool B=%d H=%d %s: pooled, flattened copy, global max, argmax and both gradients exact (tol 0)'
          % (B, H, 'fp32' if dt == F32 else 'bf16'))


# --------------------------------------------------------------------------- #
# inference forward at the predictor's largest batch
# --------------------------------------------------------------------------- #
BIG = 16384          # the largest batch of tools/mb_predict.py


@pytest.mark.parametrize('dt,impl', [(F32, 0), (BF16, 1)])
@pytest.mark.parametrize('H,Cin,Cp,Cout', [(16, 32, 32, 32), (8, 64, 64, 64), (4, 128, 0, 128)])
def test_inference_forward_at_16384(dt, impl, H, Cin, Cp, Cout):
    """The forward kernels of routed inference at B = 16384 (4x the grid-stride passes of B = 4096; 4.7 M planes
    rows at 16x16), uncounted and counted (live batch B - 1 in device memory, as the predictor launches them):
      * mpnn_stencil_gemm without statistics (pooled second input) against the float64 conv: fp32 1e-5, bf16 4e-3
        (the tolerances of test_conv_forward_and_statistics_at_scale);
      * eval-mode BatchNorm -- mpnn_bn_finalize(train = 0) from running moments, then mpnn_bn_relu_pool_fwd with the
        pooled output (16x16, 8x8) or the flattened features of the head (4x4, F = 2048) -- against float64
        relu(a lin + c) of the stored lin: fp32 1e-5 (one fma of fp32 constants per element), bf16 4e-3 (stored);
        pooled values are the max of lin and must be exact;
      * mpnn_maxpool2_fwd (planes and flattened copy) and mpnn_global_maxpool_fwd (value and argmax) of the
        activations: exact, ties (zeros behind the ReLU) to the first maximum;
      * mpnn_fc_fwd of the flattened features (F = 2048, 10 classes): fp32 dot products of 2048 terms, 1e-5.
    A counted launch must equal the uncounted one bit for bit on the first B - 1 images and write nothing past."""
    B = BIG
    g = gen(9700 + H + impl)
    x = rnd(g, (B, H, H, Cin), dt)
    xp = rnd(g, (B, H, H, Cp), dt) if Cp else None
    w = rnd(g, (3, 3, Cin, Cout), dt, 1 / math.sqrt(9 * Cin))
    wv = rnd(g, (3, 3, Cp, Cout), dt, 1 / math.sqrt(9 * Cp)) if Cp else None
    bias = torch.randn(Cout, generator=g, device='cuda')
    geo, K0, Cp, A0, A1, Wp = conv_operands(x, xp, w, wv, dt)
    gp = Geo(B, H // 2, H // 2)
    Balloc = B
    cnt = torch.tensor([B - 1], dtype=torch.int32, device='cuda')
    past = geo.G + (B - 1) * geo.S                     # first planes row of the last image
    lin = torch.zeros((Cout // 8, geo.P, 8), dtype=TD[dt], device='cuda')
    lin_c = torch.zeros_like(lin)
    L().stencil_gemm(vp(A0), K0, vp(A1), Cp, vp(Wp), 9, vp(bias), vp(lin), Cout, 0, None, 0, 0,
                     B, H, H, geo.G, geo.P, None, 0, None, dt, dt, impl, None)
    L().stencil_gemm_counted(vp(A0), K0, vp(A1), Cp, vp(Wp), 9, vp(bias), vp(lin_c), Cout, 0, None, 0, 0,
                             B, H, H, geo.G, geo.P, None, 0, None, dt, dt, impl, vp(cnt), None)
    torch.cuda.synchronize()
    ref = conv3_ref(x, w) + bias.double()
    if Cp:
        ref += conv3_ref(xp, wv)
    lin_nhwc = from_planes_t(lin, geo, Cout)
    e_conv = err(lin_nhwc, ref)
    del ref
    assert torch.equal(lin_c[:, :past], lin[:, :past]) and not lin_c[:, past:].float().any()
    # eval-mode BatchNorm from running moments near the batch's own
    m, v = moments_ref(lin_nhwc)
    m_avg = (m * (1 + 0.1 * torch.rand(Cout, generator=g, device='cuda', dtype=torch.float64))).float()
    v_avg = (v * (1 + 0.1 * torch.rand(Cout, generator=g, device='cuda', dtype=torch.float64))).float()
    gamma = torch.randn(Cout, generator=g, device='cuda'); beta = 0.1 * torch.randn(Cout, generator=g, device='cuda')
    ss = torch.zeros((2, Cout), device='cuda'); mr = torch.zeros((2, Cout), device='cuda')
    L().bn_finalize(None, 0, Cout, float(B * H * H), vp(gamma), vp(beta), vp(m_avg), vp(v_avg), 0.9, EPS, 0,
                    vp(ss), vp(mr), None)
    pool = H > 4
    F = H * H * Cout
    act = torch.zeros_like(lin); act_c = torch.zeros_like(lin)
    pooled = torch.zeros((Cout // 8, gp.P, 8), dtype=TD[dt], device='cuda') if pool else None
    pooled_c = torch.zeros_like(pooled) if pool else None
    feat = None if pool else torch.zeros((F // 8, Balloc, 8), dtype=TD[dt], device='cuda')
    feat_c = None if pool else torch.zeros_like(feat)
    L().bn_relu_pool_fwd(vp(lin), Cout, B, H, H, geo.G, geo.P, vp(ss), None if not pool else vp(act), vp(pooled),
                         gp.P if pool else 0, vp(feat), Balloc, dt, None)
    L().bn_relu_pool_fwd_counted(vp(lin), Cout, B, H, H, geo.G, geo.P, vp(ss), None if not pool else vp(act_c),
                                 vp(pooled_c), gp.P if pool else 0, vp(feat_c), Balloc, dt, vp(cnt), None)
    torch.cuda.synchronize()
    a = gamma.double() / torch.sqrt(v_avg.double() + EPS)
    c = beta.double() - m_avg.double() * a
    ref_act = torch.relu(a * lin_nhwc.double() + c)
    tol = 1e-5 if dt == F32 else 4e-3
    if pool:
        e_bn = err(from_planes_t(act, geo, Cout), ref_act)
        assert torch.equal(act_c[:, :past], act[:, :past]) and not act_c[:, past:].float().any()
        pt = Fn.max_pool2d(lin_nhwc.permute(0, 3, 1, 2).float(), 2).permute(0, 2, 3, 1)
        assert torch.equal(from_planes_t(pooled, gp, Cout).float(), pt)
        pp = gp.G + (B - 1) * gp.S
        assert torch.equal(pooled_c[:, :pp], pooled[:, :pp]) and not pooled_c[:, pp:].float().any()
        del pt
        # max-pool of the activations (planes + flattened copy) and the global max-pool
        act_nhwc = from_planes_t(act, geo, Cout).float()
        mp = torch.zeros((Cout // 8, gp.P, 8), dtype=TD[dt], device='cuda')
        Fp = (H // 2) ** 2 * Cout
        mpf = torch.zeros((Fp // 8, Balloc, 8), dtype=TD[dt], device='cuda')
        L().maxpool2_fwd(vp(act), Cout, B, H, H, geo.G, geo.P, vp(mp), gp.P, vp(mpf), Balloc, dt, None)
        gf = torch.zeros((Cout // 8, Balloc, 8), dtype=TD[dt], device='cuda')
        arg = torch.zeros((Cout // 8, Balloc, 8), dtype=torch.int32, device='cuda')
        L().global_maxpool_fwd(vp(act), Cout, B, H, H, geo.G, geo.P, vp(gf), vp(arg), Balloc, dt, None)
        torch.cuda.synchronize()
        ref_mp = Fn.max_pool2d(act_nhwc.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        assert torch.equal(from_planes_t(mp, gp, Cout).float(), ref_mp)
        assert torch.equal(from_feat_t(mpf, B).float(), ref_mp.reshape(B, -1))
        af = act_nhwc.reshape(B, -1, Cout)
        assert torch.equal(from_feat_t(gf, B).float(), af.max(1).values)
        assert torch.equal(from_feat_t(arg, B).long(), af.argmax(1))
        e_fc = 0.0
    else:
        fnhwc = from_feat_t(feat, B)
        e_bn = err(fnhwc, ref_act.reshape(B, -1))
        last = slice(B - 1, None)
        assert torch.equal(feat_c[:, :B - 1], feat[:, :B - 1]) and not feat_c[:, last].float().any()
        # the classifier head on the flattened features, uncounted and counted
        n = 10
        W = torch.randn((F, n), generator=g, device='cuda') / 10
        bl = torch.randn(n, generator=g, device='cuda')
        Z = torch.zeros((B, n), device='cuda'); Z_c = torch.zeros_like(Z)
        L().fc_fwd(vp(feat), F, Balloc, B, vp(W), vp(bl), None, n, vp(Z), dt, None)
        L().fc_fwd_counted(vp(feat), F, Balloc, B, vp(W), vp(bl), None, n, vp(Z_c), dt, vp(cnt), None)
        torch.cuda.synchronize()
        e_fc = err(Z, fnhwc.double() @ W.double() + bl.double())
        assert torch.equal(Z_c[:B - 1], Z[:B - 1]) and not Z_c[B - 1:].any()
        assert e_fc < 1e-5, e_fc
    print('inference B=%d H=%d %s: conv %.2e, bn %.2e (tol %.0e each), fc %.2e (tol 1e-5); pooled, max-pools and '
          'counted launches exact' % (B, H, 'fp32' if dt == F32 else 'bf16', e_conv, e_bn, tol, e_fc))
    assert e_conv < tol and e_bn < tol


# --------------------------------------------------------------------------- #
# weight gradient
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('dt,impl,shape', [(BF16, 1, (32, 16, 16, 16)), (BF16, 1, (16, 32, 32, 32)),
                                           (F32, 0, (16, 32, 32, 32))])
def test_stencil_wgrad_at_scale(dt, impl, shape):
    """mpnn_stencil_wgrad at B = 4096: every weight is a sum over n = B*H*W = 4.2 M (32x32) or 1.0 M (16x16)
    pixels.  The products of bf16 operands are exact in fp32, so all error is fp32 summation.  The deterministic
    bound of a recursive fp32 sum, n u sum|terms| (0.25 relative at 4.2 M terms), says nothing here, so the
    tolerance is a probabilistic estimate instead: for independent zero-mean summands the rounding errors of one
    sequential chain of n terms have an rms of ~ u sqrt(n/2) |sum| (Higham & Mary), and the tolerance is u sqrt(n):
    1.2e-4 at 32x32, 6.1e-5 at 16x16 (relative Frobenius error of dW and dbias).  The kernel accumulates per CTA in
    TMEM and then across CTAs, i.e. in far shorter chains; the measured error is ~1e-5 in bf16 and ~2e-7 in fp32,
    an order of magnitude or more inside the estimate."""
    H, Cin, Cp, Cout = shape
    B = 4096
    g = gen(4000 + H + impl)
    x = rnd(g, (B, H, H, Cin), dt)
    xp = rnd(g, (B, H, H, Cp), dt)
    gr = rnd(g, (B, H, H, Cout), dt)
    geo = Geo(B, H, H)
    K0 = ru(Cin, 16 if dt == BF16 else 8)
    A0 = to_planes_t(x, geo, K0).to(TD[dt]); A1 = to_planes_t(xp, geo).to(TD[dt]); G = to_planes_t(gr, geo).to(TD[dt])
    dW0 = torch.zeros((9, Cin, Cout), device='cuda'); dW1 = torch.zeros((9, Cp, Cout), device='cuda')
    db = torch.zeros(Cout, device='cuda')
    L().stencil_wgrad(vp(A0), K0, Cin, vp(dW0), vp(A1), Cp, Cp, vp(dW1), vp(G), Cout, Cout, vp(db), 9,
                      B, H, H, geo.G, geo.P, dt, impl, None)
    torch.cuda.synchronize()
    tol = U * math.sqrt(B * H * H)
    g2 = gr.double().reshape(-1, Cout)
    errs = []
    for xin, dW, C in ((x, dW0, Cin), (xp, dW1, Cp)):
        xpd = Fn.pad(xin.double(), (0, 0, 1, 1, 1, 1))
        ref = torch.stack([xpd[:, t // 3:t // 3 + H, t % 3:t % 3 + H].reshape(-1, C).T @ g2 for t in range(9)])
        errs.append(err(dW, ref))
    errs.append(err(db, g2.sum(0)))
    print('wgrad H=%d %s: dW0 %.2e, dW1 %.2e, dbias %.2e (tol %.2e, probabilistic)'
          % (H, 'fp32' if dt == F32 else 'bf16', *errs, tol))
    assert max(errs) < tol


# --------------------------------------------------------------------------- #
# heads
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('n,extra', [(10, False), (16, True)])
def test_fc_fwd_bwd_at_scale(B, dt, n, extra):
    """mpnn_fc_fwd / fc_bwd_data / fc_bwd_weight with F = 2048 (the 4x4x128 stage flattened) and, for the
    router layer, the `extra` feature.  fc_fwd: fp32 dot products of F+1 terms, probabilistic error
    ~ sqrt(2049) u = 3e-6 -> 1e-5.  fc_bwd_weight: sums over the batch, ~ sqrt(4097) u = 4e-6 -> 1e-5 (dW, db).
    fc_bwd_data: n + 16 terms per output, 1e-5 in fp32, 4e-3 in bf16 (stored in bf16)."""
    F = 2048
    g = gen(5000 + B + n + dt)
    Balloc = ru(B, 128)
    x = rnd(g, (B, F), dt)
    W = torch.randn((F + (1 if extra else 0), n), generator=g, device='cuda') / 10
    bias = torch.randn(n, generator=g, device='cuda')
    ex = torch.randn(B, generator=g, device='cuda') if extra else None
    X = to_feat_t(x, Balloc).to(TD[dt])
    Z = torch.zeros((B, n), device='cuda')
    L().fc_fwd(vp(X), F, Balloc, B, vp(W), vp(bias), vp(ex), n, vp(Z), dt, None)
    dZ = torch.randn((B, n), generator=g, device='cuda')
    dZ2 = torch.randn((B, 16), generator=g, device='cuda')
    W2 = torch.randn((F, 16), generator=g, device='cuda') / 10
    dX = torch.zeros_like(X)
    L().fc_bwd_data(vp(dZ), vp(W), n, vp(dZ2), vp(W2), 16, F, Balloc, B, vp(dX), dt, None)
    dW = torch.zeros_like(W); db = torch.zeros(n, device='cuda')
    L().fc_bwd_weight(vp(X), F, Balloc, B, vp(ex), vp(dZ), n, vp(dW), vp(db), dt, None)
    torch.cuda.synchronize()
    xf = torch.cat([x, ex[:, None]], 1).double() if extra else x.double()
    e = [err(Z, xf @ W.double() + bias.double()),
         err(from_feat_t(dX, B), dZ.double() @ W[:F].double().T + dZ2.double() @ W2.double().T),
         err(dW, xf.T @ dZ.double()), err(db, dZ.double().sum(0))]
    tol_d = 1e-5 if dt == F32 else 4e-3
    print('fc B=%d n=%d %s: fwd %.2e (tol 1e-5), bwd_data %.2e (tol %.0e), dW %.2e (tol 1e-5), db %.2e (tol 1e-5)'
          % (B, n, 'fp32' if dt == F32 else 'bf16', e[0], e[1], tol_d, e[2], e[3]))
    assert e[0] < 1e-5 and e[1] < tol_d and e[2] < 1e-5 and e[3] < 1e-5
    assert not dX[:, B:].float().any()


@pytest.mark.parametrize('B', [4096, 4097, 16384])
def test_fc_heads_umma_at_scale(B):
    """The tensor-core head GEMM of test_fc_heads_umma (leaf and router layer packed side by side, router feature
    in the extra K slice; fc_wgrad; data gradient through the stencil GEMM with ntaps = 1) with Balloc = ru(B, 128):
    at 4097 the last 128-row feature tile holds one image, 16384 is the predictor's largest batch.  bf16 operands,
    fp32 accumulation over K = 2064 (logits) or B (weight gradients): ~ sqrt(16384) u = 8e-6 -> 1e-4 as at small
    B; data gradient stored in bf16, 4e-3."""
    import numpy as np
    F, n_cls = 2048, 10
    g = gen(6000 + B)
    Balloc = ru(B, 128)
    Fext = F + 16
    x = rnd(g, (B, F), BF16)
    kx = torch.rand(B, generator=g, device='cuda').to(torch.bfloat16).float()
    Wl = torch.randn((F, n_cls), generator=g, device='cuda') / 10
    Wr = torch.randn((F + 1, 16), generator=g, device='cuda') / 10
    bl = torch.randn(n_cls, generator=g, device='cuda'); br = torch.randn(16, generator=g, device='cuda')
    X = torch.zeros((Fext // 8, Balloc, 8), dtype=torch.bfloat16, device='cuda')
    X[:F // 8] = to_feat_t(x, Balloc).to(torch.bfloat16)
    X[F // 8, :B, 0] = kx.to(torch.bfloat16)
    Wfc = torch.zeros((1, Fext // 8, 32, 8), dtype=torch.bfloat16, device='cuda')
    bias = torch.zeros(32, device='cuda')
    desc = np.zeros(4, dtype=np.dtype([('w', '<u8'), ('packed', '<u8')] + [(k, '<i4') for k in (
        'ntaps', 'I', 'O', 'mode', 'k_off', 'Ktot', 'n_off', 'Ntot')], align=True))
    desc[0] = (Wl.data_ptr(), Wfc.data_ptr(), 1, F, n_cls, 0, 0, Fext, 0, 32)
    desc[1] = (Wr.data_ptr(), Wfc.data_ptr(), 1, F + 1, 16, 0, 0, Fext, 16, 32)
    desc[2] = (bl.data_ptr(), bias.data_ptr(), 1, 1, n_cls, 2, 0, 8, 0, 32)
    desc[3] = (br.data_ptr(), bias.data_ptr(), 1, 1, 16, 2, 0, 8, 16, 32)
    D = torch.from_numpy(desc.view(np.uint8).copy()).cuda()
    L().pack_weights_batched(vp(D), 4, 8, BF16, None)
    Z16 = torch.zeros((B, 16), device='cuda'); Z1 = torch.zeros((B, 16), device='cuda')
    L().stencil_gemm(vp(X), Fext, None, 0, vp(Wfc), 1, vp(bias), vp(Z16), 16, 0, vp(Z1), 16, 0,
                     B, 0, 0, 0, Balloc, None, 0, None, BF16, 2, 1, None)
    dz = rnd(g, (B, 32), BF16)
    dz[:, n_cls:16] = 0
    P = to_feat_t(dz, Balloc).to(torch.bfloat16)
    gWl = torch.zeros_like(Wl); gWr = torch.zeros_like(Wr)
    L().fc_wgrad(vp(X), Fext, Balloc, B, vp(P), 32, 16, vp(gWl), F, n_cls, vp(gWr), F + 1, 16, None)
    Wfd = torch.zeros((1, 4, F, 8), dtype=torch.bfloat16, device='cuda')
    desc2 = desc[:2].copy()
    desc2[0] = (Wl.data_ptr(), Wfd.data_ptr(), 1, F, n_cls, 1, 0, 32, 0, F)
    desc2[1] = (Wr.data_ptr(), Wfd.data_ptr(), 1, F, 16, 1, 16, 32, 0, F)
    D2 = torch.from_numpy(desc2.view(np.uint8).copy()).cuda()
    L().pack_weights_batched(vp(D2), 2, 8, BF16, None)
    dX = torch.zeros((F // 8, Balloc, 8), dtype=torch.bfloat16, device='cuda')
    L().stencil_gemm(vp(P), 32, None, 0, vp(Wfd), 1, None, vp(dX), F, 0, None, 0, 0,
                     B, 0, 0, 0, Balloc, None, 0, None, BF16, BF16, 1, None)
    torch.cuda.synchronize()
    bfr = lambda t: t.to(torch.bfloat16).double()
    xd = x.double()
    xf = torch.cat([xd, kx.double()[:, None]], 1)
    e = [err(Z16[:, :n_cls], xd @ bfr(Wl) + bl.double()), err(Z1, xf @ bfr(Wr) + br.double()),
         err(gWl, xd.T @ dz[:, :n_cls].double()), err(gWr, xf.T @ dz[:, 16:].double()),
         err(from_feat_t(dX, B), dz[:, :n_cls].double() @ bfr(Wl).T + dz[:, 16:].double() @ bfr(Wr[:F]).T)]
    print('fc_heads_umma B=%d: leaf %.2e, router %.2e, dWl %.2e, dWr %.2e (tol 1e-4 each), dX %.2e (tol 4e-3)' % (B, *e))
    assert max(e[:4]) < 1e-4 and e[4] < 4e-3
    assert not dX[:, B:].float().any()


# --------------------------------------------------------------------------- #
# activity cost and dropout
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('H,C', [(32, 16), (8, 64)])
def test_activity_cost_at_scale(B, dt, H, C):
    """mpnn_activity_fwd: cost[b] = alpha sum x^2, an fp32 sum of C*H*W positive terms in chains of C*H*W/256
    fmas plus the warp / CTA trees: gamma_n with n = C*H*W/256 + 13 (<= 77) -> rtol 1e-5.  mpnn_activity_bwd
    with coefficients, writing (acc = 0) and accumulating (acc = 1) into dx: one fma per element, 1e-6 in fp32,
    4e-3 in bf16 (stored in bf16)."""
    g = gen(7000 + B + H + dt)
    geo = Geo(B, H, H)
    x = rnd(g, (B, H, H, C), dt)
    X = to_planes_t(x, geo).to(TD[dt])
    alpha = 1e-3
    cost = torch.zeros(B, device='cuda')
    L().activity_fwd(vp(X), C, B, H, H, geo.G, geo.P, alpha, vp(cost), dt, None)
    coef = torch.rand(B, generator=g, device='cuda')
    scale = 2 * alpha / B
    d0 = rnd(g, (B, H, H, C), dt, 1e-6)
    dx_w = to_planes_t(d0, geo).to(TD[dt])
    dx_a = dx_w.clone()
    L().activity_bwd(vp(X), C, B, H, H, geo.G, geo.P, vp(coef), scale, vp(dx_w), 0, dt, None)
    L().activity_bwd(vp(X), C, B, H, H, geo.G, geo.P, vp(coef), scale, vp(dx_a), 1, dt, None)
    dx_n = torch.zeros_like(X)
    L().activity_bwd(vp(X), C, B, H, H, geo.G, geo.P, None, scale, vp(dx_n), 0, dt, None)
    torch.cuda.synchronize()
    xd = x.double()
    ref_c = alpha * (xd ** 2).sum((1, 2, 3))
    e_c = ((cost.double() - ref_c).abs() / ref_c).max().item()
    k = scale * coef.double()[:, None, None, None]
    tol = 1e-6 if dt == F32 else 4e-3
    e = [err(from_planes_t(dx_w, geo, C), k * xd), err(from_planes_t(dx_a, geo, C), d0.double() + k * xd),
         err(from_planes_t(dx_n, geo, C), scale * xd)]
    print('activity B=%d H=%d %s: cost %.2e (tol 1e-5), write %.2e, acc %.2e, no coef %.2e (tol %.0e each)'
          % (B, H, 'fp32' if dt == F32 else 'bf16', e_c, *e, tol))
    assert e_c < 1e-5 and max(e) < tol


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('feat', [0, 1])
def test_dropout_at_scale(B, dt, feat):
    """mpnn_dropout in the planes layout and in the flattened-feature layout against dropout_mask_t (the torch
    restatement of util.dropout_mask): x * (1/keep) where kept, 0 elsewhere, exactly (the same fp32 product,
    rounded once to the storage type).  33.6 M elements, so the element index passes 2^24 and the grid-stride
    loop runs many passes."""
    H, C, keep, seed, draw = 16, 32, 0.75, 0x1234567, 5
    g = gen(8000 + B + dt + 10 * feat)
    geo = Geo(B, H, H)
    Balloc = ru(B, 128)
    x = rnd(g, (B, H, H, C), dt)
    T = (to_feat_t(x.reshape(B, -1), Balloc) if feat else to_planes_t(x, geo)).to(TD[dt])
    hyp = torch.zeros(8, device='cuda')
    hyp.view(torch.int32)[6] = draw                  # MPNN_HYP_DRAW: bits of a uint32
    L().dropout(vp(T), C, B, H, H, geo.G, geo.P, feat, Balloc, keep, seed, vp(hyp), dt, None)
    mask = dropout_mask_t(seed, draw, (B, H, H, C), keep, 'cuda')
    ref = torch.where(mask, x * torch.tensor(1.0 / keep, dtype=torch.float32).cuda(), torch.zeros_like(x)).to(TD[dt])
    torch.cuda.synchronize()
    got = from_feat_t(T, B).view(B, H, H, C) if feat else from_planes_t(T, geo, C)
    assert torch.equal(got, ref)
    if feat:
        assert not T[:, B:].float().any()
    assert abs(mask.float().mean().item() - keep) < 1e-3
    print('dropout B=%d %s %s: exact (tol 0), kept fraction %.5f' % (B, 'feat' if feat else 'planes',
                                                                     'fp32' if dt == F32 else 'bf16', mask.float().mean().item()))


# --------------------------------------------------------------------------- #
# BatchNorm statistics of channels with large means
# --------------------------------------------------------------------------- #
RATIOS = (0, 1, 10, 100, 1000)          # |mean| / std; 1000 is measured and printed, not asserted


def _channel_plan(C):
    """per channel: (ratio, std, offset); every sixth channel has zero spread and outputs only its bias, 1"""
    plan = []
    for c in range(C):
        if c % 6 == 5:
            plan.append((None, 0.0, 1.0))
        else:
            std = 2.0 ** ((c // 6) % 3 - 1)
            r = RATIOS[c % 6]
            plan.append((r, std, (-1) ** c * r * std))
    return plan


def _check_stats(tag, mean, rstd, y, plan):
    """mean / rstd as the consumer sees them against two-pass float64 moments of y: mean error <= 1e-3 std,
    rstd relative error <= 1e-3 for ratios <= 100; a zero-spread channel must give mean = 1 and
    rstd = 1/sqrt(eps) to fp32 rounding.  Returns the worst errors per ratio."""
    m, v = moments_ref(y)
    s = torch.sqrt(v)
    rstd_ref = 1 / torch.sqrt(v + EPS)
    em = ((mean.double() - m).abs() / s).tolist()
    er = ((rstd.double() - rstd_ref).abs() / rstd_ref).tolist()
    worst = {}
    for c, (r, _, off) in enumerate(plan):
        if r is None:
            assert float(v[c]) == 0.0
            assert mean[c].item() == off, (tag, c, mean[c].item())
            z = 1.0 / math.sqrt(float(torch.tensor(EPS, dtype=torch.float32)))
            assert abs(rstd[c].item() - z) <= 4 * U * z, (tag, c, rstd[c].item())
            worst['zero'] = max(worst.get('zero', 0.0), abs(rstd[c].item() - z) / z)
            continue
        worst[r] = max(worst.get(r, (0, 0))[0], em[c]), max(worst.get(r, (0, 0))[1], er[c])
    print('%s: ' % tag + ', '.join('ratio %s: mean %.1e std, rstd %.1e' % (r, *worst[r]) for r in RATIOS if r in worst)
          + ', zero spread: rstd %.1e (tol 1e-3 for ratios <= 100, 4u for zero spread; 1000 not asserted)'
          % worst.get('zero', 0.0))
    for r in RATIOS:
        if r in worst and r <= 100:
            assert worst[r][0] <= 1e-3 and worst[r][1] <= 1e-3, (tag, r, worst[r])
    return worst


@pytest.mark.parametrize('n_parts', [1, 512])
def test_bn_finalize_variance_from_exact_sums(n_parts):
    """mpnn_bn_finalize with partial sums that carry no rounding: count = 4096*32*32 = 2^22 and every channel's
    sums s = count m, s2 = count q (m, q fp32) split into n_parts equal rows (powers of two: all exact), so the
    finalisation is the only arithmetic.  In float64, var = q - m^2 is then exact up to 2^-53 relative to m^2,
    so mean and rstd must be correct to fp32 rounding (rstd relative error <= 1e-6) at every ratio |mean|/std up
    to 1000 -- an fp32 evaluation of m^2 would be off by ~2^-24 ratio^2 (6e-4 at 100)."""
    count = 2.0 ** 22
    g = gen(9900)
    C = 32
    plan = _channel_plan(C)
    std = torch.tensor([p[1] for p in plan], dtype=torch.float64, device='cuda')
    off = torch.tensor([p[2] for p in plan], dtype=torch.float64, device='cuda')
    m = (off * (1 + 1e-3 * torch.rand(C, generator=g, device='cuda', dtype=torch.float64))).float()
    q = (m.double() ** 2 + std ** 2).float()
    var = (q.double() - m.double() ** 2).clamp_min(0)
    row = torch.stack([m.double(), q.double()]) * (count / n_parts)
    parts = row.float().repeat(n_parts, 1).contiguous()
    assert torch.equal(parts.double().view(n_parts, 2, C).sum(0), torch.stack([m.double(), q.double()]) * count)
    ss = torch.zeros((2, C), device='cuda'); mr = torch.zeros((2, C), device='cuda')
    one, zero = torch.ones(C, device='cuda'), torch.zeros(C, device='cuda')
    L().bn_finalize(vp(parts), n_parts, C, count, vp(one), vp(zero), None, None, 0.9, EPS, 1, vp(ss), vp(mr), None)
    torch.cuda.synchronize()
    rstd_ref = 1 / torch.sqrt(var.float().double() + EPS)
    er = ((mr[1].double() - rstd_ref).abs() / rstd_ref).max().item()
    print('bn_finalize exact sums, %d rows: mean exact %s, rstd rel err %.1e (tol 1e-6)' % (n_parts, torch.equal(mr[0], m), er))
    assert torch.equal(mr[0], m)
    assert er <= 1e-6


@pytest.mark.parametrize('producer', ['stencil_gemm+bn_finalize', 'conv_bn_stats', 'conv_bn_stats defer'])
@pytest.mark.parametrize('dt,impl', [(F32, 0), (BF16, 1)])
@pytest.mark.parametrize('H,Cin,Cout', [(32, 16, 16), (16, 32, 32)])
def test_bn_statistics_with_large_channel_means_conv(producer, dt, impl, H, Cin, Cout):
    """BatchNorm batch statistics of conv outputs lin = offset_c + conv_c with |offset| / std in {0, 1, 10, 100,
    1000} and zero-spread channels, at B = 4096, through each producer: the conv epilogue's per-CTA sums finalised
    by mpnn_bn_finalize, mpnn_conv_bn_stats (last CTA finalises), and mpnn_conv_bn_stats with defer = 1 finalised
    by mpnn_bn_relu_pool_fwd_acc.  Bar: see _check_stats."""
    B = 4096
    g = gen(9000 + H + impl)
    plan = _channel_plan(Cout)
    x = rnd(g, (B, H, H, Cin), dt)
    w = rnd(g, (3, 3, Cin, Cout), dt, 1 / math.sqrt(9 * Cin))
    w *= torch.tensor([p[1] for p in plan], device='cuda')           # powers of two: exact in bf16
    bias = torch.tensor([p[2] for p in plan], device='cuda')
    geo, K0, _, A0, _, Wp = conv_operands(x, None, w, None, dt)
    count = B * H * H
    out = torch.zeros((Cout // 8, geo.P, 8), dtype=TD[dt], device='cuda')
    if producer == 'stencil_gemm+bn_finalize':
        stats = torch.zeros(592 * 2 * Cout, device='cuda'); cnt = ctypes.c_int(0)
        L().stencil_gemm(vp(A0), K0, None, 0, vp(Wp), 9, vp(bias), vp(out), Cout, 0, None, 0, 0,
                         B, H, H, geo.G, geo.P, vp(stats), 592, ctypes.byref(cnt), dt, dt, impl, None)
        ss = torch.zeros((2, Cout), device='cuda'); mr = torch.zeros((2, Cout), device='cuda')
        one, zero = torch.ones(Cout, device='cuda'), torch.zeros(Cout, device='cuda')
        L().bn_finalize(vp(stats), cnt.value, Cout, float(count), vp(one), vp(zero), None, None, 0.9, EPS, 1,
                        vp(ss), vp(mr), None)
    else:
        defer = int(producer.endswith('defer'))
        b, fp = bn_fuse(Cout, count, defer)
        L().conv_bn_stats(vp(A0), K0, None, 0, vp(Wp), vp(bias), vp(out), Cout, B, H, H, geo.G, geo.P, fp, dt, impl, None)
        if defer:
            act = torch.zeros_like(out)
            L().bn_relu_pool_fwd_acc(vp(out), Cout, B, H, H, geo.G, geo.P, fp, vp(act), None, 0, None, 0, dt, None)
        mr = b['mr']
    torch.cuda.synchronize()
    y = conv3_ref(x, w) + bias.double()
    _check_stats('%s %s H=%d' % (producer, 'fp32' if dt == F32 else 'bf16', H), mr[0], mr[1], y, plan)


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('B,H,C', [(128, 8, 64), (512, 4, 128)])
def test_bn_statistics_with_large_channel_means_bn_fwd_small(dt, B, H, C):
    """The same channels through mpnn_bn_fwd_small at its largest eligible size (B*H*W = 8192 pixels): the
    coarse scales of the real net at the reference's training batch.  lin is rounded to the storage type first;
    the reference moments are those of the stored values."""
    g = gen(9500 + B + dt)
    plan = _channel_plan(C)
    geo = Geo(B, H, H)
    std = torch.tensor([p[1] for p in plan], device='cuda'); off = torch.tensor([p[2] for p in plan], device='cuda')
    lin = (torch.randn((B, H, H, C), generator=g, device='cuda') * std + off).to(TD[dt])
    LIN = to_planes_t(lin, geo)
    ss = torch.zeros((2, C), device='cuda'); mr = torch.zeros((2, C), device='cuda')
    one, zero = torch.ones(C, device='cuda'), torch.zeros(C, device='cuda')
    act = torch.zeros_like(LIN)
    L().bn_fwd_small(vp(LIN), C, B, H, H, geo.G, geo.P, vp(one), vp(zero), None, None, 0.9, EPS, vp(ss), vp(mr),
                     vp(act), None, 0, dt, None)
    torch.cuda.synchronize()
    _check_stats('bn_fwd_small %s B=%d H=%d' % ('fp32' if dt == F32 else 'bf16', B, H), mr[0], mr[1], lin.double(), plan)


# --------------------------------------------------------------------------- #
# the routing walks: mpnn_route_fwd / mpnn_route_bwd
# --------------------------------------------------------------------------- #
RT_STAGED_MAX = 32      # csrc/route.cu: trees up to this size run the staged walk, larger ones the global one


@functools.lru_cache(None)
def _plan_of(name):
    """(routing tables, n_theta, segment tables) of a dry-run plan of a full-size net (lib/engine.py)"""
    import arch_and_hypers as ah
    from lib import engine as E
    eng = E.Engine(getattr(ah, name)(k_cpt=4e-9)((32, 32, 3), (10,)), precision='fp32', impl=0, dry_run=True)
    plan = eng._plan(128, True, True)
    seg = {k: getattr(eng, k).clone() for k in ('seg_start', 'seg_node', 'seg_mult', 'seg_l2')}
    return tree_tables(plan), eng.n_theta, len(eng.nodes), seg


def tree_of(spec):
    if isinstance(spec, str):
        return _plan_of(spec)[0]
    n, ns = spec
    return random_tree(np.random.default_rng(31 * n + ns), n, ns)


def _ptrs(ts):
    return torch.tensor([x.data_ptr() for x in ts] or [0], dtype=torch.int64, device='cuda')


def route_launch(t, R, tau, eps, B, c_err=None, d_cor=None, k_cpt=None, critic=0, k_dec=0.0, k_cre=0.0,
                 optimistic=0, use_cls_err=0, kc=4e-9, bwd=True):
    """mpnn_route_fwd (+ mpnn_route_bwd) on tables t (NumPy) and device logits R[slot]; outputs start as NaN / -1
    so that an unwritten element cannot pass"""
    T = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in t.items()}
    n = len(t['parent'])
    hyp = torch.zeros(8, device='cuda')
    hyp[2], hyp[3], hyp[4] = tau, eps, kc
    Rt = _ptrs(R)
    o = dict(p_tr=torch.full((n, B), math.nan, device='cuda'), p_ev=torch.full((n, B), math.nan, device='cuda'),
             dec=torch.full((max(len(R), 1), B), -1, dtype=torch.int32, device='cuda'))
    L().route_fwd(vp(T['parent']), vp(T['sink_idx']), vp(T['n_sinks']), vp(T['floor']), vp(T['sw']), n, vp(Rt),
                  vp(hyp), B, vp(o['p_tr']), vp(o['p_ev']), vp(o['dec']), None)
    if bwd:
        o['dR'] = [torch.full_like(r, math.nan) for r in R]
        o['c_data'] = torch.full((B,), math.nan, device='cuda')
        scratch = torch.zeros(3 * n * B, device='cuda')
        ce_t, dc_t, dR_t = _ptrs(c_err), _ptrs(d_cor), _ptrs(o['dR'])
        L().route_bwd(vp(T['parent']), vp(T['sink_idx']), vp(T['n_sinks']), vp(T['child']), vp(T['floor']),
                      vp(T['sw']), vp(T['ops']), vp(T['err']), n, vp(Rt), vp(hyp), B, vp(o['p_tr']), vp(o['p_ev']),
                      vp(ce_t), vp(dc_t), vp(k_cpt), critic, k_dec, k_cre, optimistic, use_cls_err, vp(dR_t),
                      vp(scratch), vp(o['c_data']), None)
    torch.cuda.synchronize()
    return o


LOGITS = {'normal': 0.6, 'integer': 1.0, 'sharp': 0.1}       # logits kind -> tau


def route_inputs(t, B, kind, seed):
    g = gen(seed)
    n_err = int((t['err'] >= 0).sum())
    R = []
    for i in range(len(t['parent'])):
        ns = int(t['n_sinks'][i])
        if ns < 2:
            continue
        if kind == 'normal':
            r = 2 * torch.randn((B, ns), generator=g, device='cuda')
        elif kind == 'integer':                  # ties: the first maximum decides dec and p_ev
            r = torch.randint(-2, 3, (B, ns), generator=g, device='cuda').float()
        else:                                    # about +-50 at tau = 0.1 (the tau_cr schedule): exponents to 1000
            r = (25 * torch.randn((B, ns), generator=g, device='cuda')).clamp(-50, 50)
        R.append(r)
    ce = [3 * torch.rand(B, generator=g, device='cuda') for _ in range(n_err)]
    dc = [(torch.rand(B, generator=g, device='cuda') < 0.6).float() for _ in range(n_err)]
    kv = 1e-8 * torch.rand(B, generator=g, device='cuda')
    return R, ce, dc, kv


MODES = {'actor k_dec': dict(critic=0, k_dec=0.01), 'actor k_cpt vector': dict(critic=0, k_dec=0.01, vec=True),
         'critic': dict(critic=1, k_cre=1e-3), 'critic optimistic': dict(critic=1, k_cre=1e-3, optimistic=1),
         'critic use_cls_err': dict(critic=1, k_cre=1e-3, use_cls_err=1, vec=True)}


def p_tr_bound(t, ref, tau, eps, X):
    """First-order bound on |p_tr(fp32) - p_tr| per node and example, propagated down the tree.  A softmax
    probability in fp32 carries a relative error kappa <= (8X + 14) u: the exponent x_j - max x, with x = R / tau
    rounded and |x| <= X, is off by <= 4X u in absolute terms, expf adds 2 ulp, the sum of <= 8 terms 8u, the
    reciprocal and product 2u.  Then p_tr[i] = q p + eps fl[i] with q = p_tr[par] - eps fl[par] gives
      E[i] = p (E[par] + u eps fl[par] + u q) + q p (kappa + u) + u eps fl[i] + u p_tr[i]."""
    kappa = (8 * X + 14) * U
    eps32, n = float(np.float32(eps)), len(t['parent'])
    E = [torch.zeros_like(ref['p_tr'][0])] * n
    for i in range(1, n):
        par = int(t['parent'][i])
        if t['n_sinks'][par] < 2:
            E[i] = E[par]
            continue
        p = ref['sm'][int(t['sw'][par])][:, int(t['sink_idx'][i])]
        fp, fi = eps32 * float(t['floor'][par]), eps32 * float(t['floor'][i])
        q = ref['p_tr'][par] - fp
        E[i] = p * (E[par] + U * fp + U * q) + q * p * (kappa + U) + U * fi + U * ref['p_tr'][i]
    return torch.stack(E), kappa


def _depth(t):
    d = [0] * len(t['parent'])
    for i in range(1, len(d)):
        par = int(t['parent'][i])
        d[i] = d[par] + (1 if t['n_sinks'][par] >= 2 else 0)
    return max(d)


def route_bounds(t, ref, mode, tau, eps, R, E, kappa):
    """Bounds on dR (per element) and c_data (per example), from the float64 intermediates of route_ref:
      * actor: gs_j = g[child_j] (p_tr - eps fl) and dR_j = sm_j (gs_j - sum_k sm_k gs_k) / tau + 2 k_dec p_tr R_j / B.
        g (sums of <= n products of <= D probabilities, all terms >= 0) is good to K_g u = (D kappa / u + n + 4) u
        relative, so |d dR_j| <= (K_g + kappa / u + 8) u sm_j (|gs_j| + sum_k sm_k |gs_k|) / tau
        + sm_j (|g_j| + sum_k sm_k |g_k|) (E + 2u p_tr) / tau + |k_dec term| (E / p_tr + 6u);
      * critic: the target (a sum of <= n terms >= 0) is good to (n + 2) u relative, so
        |d dR_j| <= 2 k_cre p_tr / B ((n + 3) u (|R_j| + target_j)) + |dR_j| (E / p_tr + 6u);
      * c_data = sum_i p_tr w_i: |d| <= sum_i (E w_i + p_tr dw_i) + (n + 4) u sum_i p_tr w_i, with dw the bound of
        each weight (local cost: 3u; k_dec |R|^2: 12u; critic regression: 2 (n + 4) u k_cre sum_j (|R_j| + t_j)^2)."""
    n, D = len(t['parent']), _depth(t)
    tau32, B = float(np.float32(tau)), R[0].shape[0] if R else 1
    Kg = D * kappa / U + n + 4
    k_dec, k_cre = float(np.float32(mode.get('k_dec', 0.0))), float(np.float32(mode.get('k_cre', 0.0)))
    eps32 = float(np.float32(eps))
    bdR, terms, dterms = [None] * len(R), [], []
    p = ref['p_tr']
    for i in range(n):
        ns = int(t['n_sinks'][i])
        if ns < 2:
            continue
        s, ks = int(t['sw'][i]), list(t['child'][i, :ns])
        r = R[s].double()
        pt, Ei = p[i][:, None], E[i][:, None]
        if not mode['critic']:
            sm = ref['sm'][s]
            gc = ref['g'][ks].T
            gs = gc * (pt - eps32 * float(t['floor'][i]))
            a1 = sm * (gs.abs() + (sm * gs.abs()).sum(1, keepdim=True)) / tau32
            a2 = sm * (gc.abs() + (sm * gc.abs()).sum(1, keepdim=True)) / tau32
            kd = (2 * k_dec * pt * r / B).abs()
            bdR[s] = (Kg + kappa / U + 8) * U * a1 + a2 * (Ei + 2 * U * pt) + kd * (Ei / pt + 6 * U)
            terms.append(k_dec * p[i] * (r ** 2).sum(1)); dterms.append(E[i] * k_dec * (r ** 2).sum(1) + 12 * U * terms[-1])
        else:
            tg = ref['tgt'][s]
            bdR[s] = 2 * k_cre * pt / B * (n + 3) * U * (r.abs() + tg) + ref['dR'][s].abs() * (Ei / pt + 6 * U)
            w = k_cre * ((r.abs() + tg) ** 2).sum(1)
            terms.append(p[i] * w); dterms.append(E[i] * w + p[i] * 2 * (n + 4) * U * w)
    return bdR, terms, dterms


def c_data_bound(t, ref, mode, ce, kc, E, terms, dterms):
    n = len(t['parent'])
    ops = torch.tensor(t['ops'], dtype=torch.float64, device='cuda')
    tot, dtot = list(terms), list(dterms)
    for i in range(n):
        e = ce[int(t['err'][i])].double() if t['err'][i] >= 0 else 0.0
        w = e + (0.0 if mode['critic'] else kc * ops[i])
        w = w if torch.is_tensor(w) else torch.full_like(ref['p_tr'][i], w)
        tot.append(ref['p_tr'][i] * w); dtot.append(E[i] * w + 3 * U * ref['p_tr'][i] * w)
    return sum(dtot) + (n + 4) * U * sum(tot)


def _ratio(got, ref, bound):
    return float(((got.double() - ref).abs() / bound.clamp_min(1e-300)).max())


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('logits', list(LOGITS))
@pytest.mark.parametrize('tree', [(11, 2), (11, 4), (11, 8), (32, 2), (32, 4), (32, 8), (33, 2), (33, 4), (33, 8),
                                  'ac_tree', 'cr_tree'])
def test_route_walks_at_scale(tree, logits, B):
    """mpnn_route_fwd / _bwd on random trees of 11, 32 (staged walk) and 33 nodes (global walk) whose widest switch
    has 2, 4 or 8 sinks (every NS instantiation of the staged walk), and on the 95-node tables of the full-size
    ac_tree and cr_tree (global walk), against route_ref: actor with k_dec, actor with a per-example k_cpt,
    critic plain, optimistic and use_cls_err; random logits (tau 0.6), integer logits (ties, tau 1) and logits of
    about +-50 at tau = 0.1; eps = 1e-6 and 0.1 (at 1e-6 the floor terms are below every tolerance, at 0.1 they are
    not).  p_ev and dec are exact; p_tr, dR and c_data are held to the bounds of p_tr_bound and route_bounds,
    which scale with X = max |R| / tau (2 ulp of a softmax exponent of 1000 is 1e-4 relative)."""
    t = tree_of(tree)
    n = len(t['parent'])
    assert (n > RT_STAGED_MAX) == (tree == 'ac_tree' or tree == 'cr_tree' or tree[0] > 32)
    tau = LOGITS[logits]
    R, ce, dc, kv = route_inputs(t, B, logits, 7100 + n + B + len(logits))
    X = max(float(r.abs().max()) for r in R) / float(np.float32(tau))
    worst = {}
    for eps in (1e-6, 0.1):
        for name, m in MODES.items():
            k_cpt = kv if m.get('vec') else None
            got = route_launch(t, R, tau, eps, B, ce, dc, k_cpt, m['critic'], m.get('k_dec', 0.0), m.get('k_cre', 0.0),
                               m.get('optimistic', 0), m.get('use_cls_err', 0))
            ref = route_ref(t, R, tau, eps, c_err=ce, d_cor=dc, k_cpt=kv if m.get('vec') else 4e-9,
                            critic=bool(m['critic']), k_dec=m.get('k_dec', 0.0), k_cre=m.get('k_cre', 0.0),
                            optimistic=bool(m.get('optimistic')), use_cls_err=bool(m.get('use_cls_err')))
            assert torch.equal(got['p_ev'].double(), ref['p_ev']), name
            assert torch.equal(got['dec'][:len(R)].long(), ref['dec']), name
            E, kappa = p_tr_bound(t, ref, tau, eps, X)
            bdR, terms, dterms = route_bounds(t, ref, m, tau, eps, R, E, kappa)
            kc = kv.double() if m.get('vec') else float(np.float32(4e-9))
            bc = c_data_bound(t, ref, m, ce, kc, E, terms, dterms)
            r = dict(p_tr=_ratio(got['p_tr'], ref['p_tr'], E + 1e-300),
                     dR=max(_ratio(a, b, c) for a, b, c in zip(got['dR'], ref['dR'], bdR)),
                     c_data=_ratio(got['c_data'], ref['c_data'], bc))
            for k, v in r.items():
                worst[k] = max(worst.get(k, 0.0), v)
            assert max(r.values()) <= 1.0, (name, eps, r)
    print('route %s n=%d B=%d %s (X = %.0f): worst |err| / bound over 2 eps x 5 modes: p_tr %.2f, dR %.2f, '
          'c_data %.2f (tol 1 each); p_ev, dec exact' % (tree, n, B, logits, X, worst['p_tr'], worst['dR'],
                                                        worst['c_data']))


@pytest.mark.parametrize('tree', [(11, 2), (11, 4), (11, 8), (32, 2), (32, 4), (32, 8), 'ac_chain'])
@pytest.mark.parametrize('logits', ['normal', 'sharp'])
def test_staged_walk_equals_global_walk_bit_for_bit(tree, logits):
    """A tree of <= 32 nodes runs the staged walk; the same tree padded past 32 nodes with a chain of 1-sink
    nodes below its last node (ops 0, err -1) runs the global walk.  The padding changes no original node's
    values and only adds exact zeros to c_data, and the two walks do the same arithmetic in the same order, so
    p_tr, p_ev, dec, dR and c_data must agree bit for bit, in every mode and at both eps."""
    B = 4097
    t = tree_of(tree)
    n = len(t['parent'])
    assert n <= RT_STAGED_MAX
    tp = pad_tree(t, 40)
    tau = LOGITS[logits]
    R, ce, dc, kv = route_inputs(t, B, logits, 7300 + n)
    for eps in (1e-6, 0.1):
        for name, m in MODES.items():
            a = [route_launch(x, R, tau, eps, B, ce, dc, kv if m.get('vec') else None, m['critic'],
                              m.get('k_dec', 0.0), m.get('k_cre', 0.0), m.get('optimistic', 0),
                              m.get('use_cls_err', 0)) for x in (t, tp)]
            st, gl = a
            for k in ('p_tr', 'p_ev'):
                assert torch.equal(st[k], gl[k][:n]), (name, eps, k)
                assert torch.equal(gl[k][n:], gl[k][n - 1:n].expand(40 - n, B)), (name, eps, k)
            assert torch.equal(st['dec'], gl['dec']), (name, eps)
            assert torch.equal(st['c_data'], gl['c_data']), (name, eps)
            for x, y in zip(st['dR'], gl['dR']):
                assert torch.equal(x, y), (name, eps)
    print('staged vs global walk %s %s: p_tr, p_ev, dec, dR, c_data bit-identical (2 eps x 5 modes)' % (tree, logits))


def test_first_argmax_on_the_device():
    from oracle.torch_ref import first_argmax
    x = torch.tensor([[0., 0., 0.], [1., 3., 3.], [2., 1., 2.]], device='cuda')
    assert first_argmax(x, 1).tolist() == [0, 1, 0]


# --------------------------------------------------------------------------- #
# node moments and path compaction on the 95-node walk
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('B', [1, 127] + list(BATCHES) + [BIG])
def test_node_moments_and_compact_paths_on_the_tree_walk(B):
    """p_tr and p_ev of the global walk on the ac_tree tables (random logits, eps 0.1) into mpnn_node_moments and
    mpnn_compact_paths.  Moments: each thread sums ceil(B / 256) terms, then 5 shuffle levels and 8 warp partials,
    all terms >= 0, so |d sum| <= (ceil(B / 256) + 13) u sum (+ u for p^2, + u for the division by B), against
    float64 sums of the same fp32 p_tr.  Index lists and counts: exact, ascending."""
    t = tree_of('ac_tree')
    n = len(t['parent'])
    R, _, _, _ = route_inputs(t, B, 'normal', 7500 + B)
    o = route_launch(t, R, 0.6, 0.1, B, bwd=False)
    stats = torch.full((n, 2), math.nan, device='cuda')
    L().node_moments(vp(o['p_tr']), n, B, vp(stats), None)
    idx = torch.full((n, B), -1, dtype=torch.int32, device='cuda')
    cnt = torch.full((n,), -1, dtype=torch.int32, device='cuda')
    L().compact_paths(vp(o['p_ev']), n, B, vp(idx), vp(cnt), None)
    torch.cuda.synchronize()
    p = o['p_tr'].double()
    ref = torch.stack([(p ** 2).mean(1), p.mean(1)], 1)
    k = -(-B // 256) + 13
    tol = torch.tensor([k + 3, k + 2], dtype=torch.float64, device='cuda') * U
    e = ((stats.double() - ref).abs() / ref).max(0).values
    print('node_moments B=%d: mean p^2 %.2e (tol %.1e), mean p %.2e (tol %.1e); compaction exact'
          % (B, e[0], tol[0], e[1], tol[1]))
    assert bool((e <= tol).all())
    assert int(o['p_ev'][0].sum()) == B
    for i in range(n):
        want = torch.nonzero(o['p_ev'][i] > 0.5).flatten()
        assert int(cnt[i]) == want.numel()
        assert torch.equal(idx[i, :want.numel()].long(), want)



# --------------------------------------------------------------------------- #
# error layers: softmax + cross-entropy, squared error, superclass targets
# --------------------------------------------------------------------------- #
def logits_rows(g, B, n, ldz):
    """[B][ldz] logits (columns >= n hold garbage the kernels must not read): normal * 3, every 16th row all equal
    (ties to the first class), every 16th row (offset 5) of +-80 values; one-hot labels [B][n]"""
    Z = 3 * torch.randn((B, ldz), generator=g, device='cuda')
    Z[:, n:] = 1e30
    Z[::16, :n] = 0.25
    s = torch.randint(0, 2, (B, n), generator=g, device='cuda').float() * 160 - 80
    Z[5::16, :n] = s[5::16]
    y = Fn.one_hot(torch.randint(0, n, (B,), generator=g, device='cuda'), n).float()
    return Z.contiguous(), y


def planes_with_sentinel(B, Balloc):
    """two bf16 planes [2][Balloc][8]: rows < B hold 7 (every one must be written), rows B .. Balloc zero, as the
    engine allocates them (the kernels leave those rows alone, and the head GEMMs read them as zero rows)"""
    t = torch.zeros((2, Balloc, 8), dtype=torch.bfloat16, device='cuda')
    t[:, :B] = 7.0
    return t


def softmax_ce_ref(z, y, eps, n):
    """float64 softmax and c_err of fp32 operands (eps and eps / n as the kernel rounds them)"""
    p = torch.softmax(z, 1)
    a = float(np.float32(np.float32(eps) / np.float32(n))) + float(np.float32(1 - np.float32(eps))) * p
    return p, -(y.double() * torch.log(a)).sum(1)


@pytest.mark.parametrize('B', list(BATCHES) + [BIG])
@pytest.mark.parametrize('n', [2, 10, 16, 17, 32])
@pytest.mark.parametrize('ldz', ['n', 32])
def test_softmax_ce_at_scale(B, n, ldz):
    """mpnn_softmax_ce_fwd / _bwd with 16 (n <= 16) and 32 lanes per example, row stride n or 32 (the head GEMM's
    row), eps 1e-6 and 0.1, a per-example coef.  With m = max_j |z_j - max z| of a row, every fp32 probability of
    the row is good to kappa = (m + n + 5) u relative (exponent rounding m u, expf 2 ulp, sum n u, reciprocal and
    product 2u), so
      prob:  |d p_j| <= kappa p_j (+ 2^-126 for results in the subnormal range);
      c_err: -log(eps/n + (1-eps) p_y): |d| <= kappa + 4u + u |c_err|;
      d_cor: exact, the reference argmax taken from the kernel's own prob (checked above);
      dZ:    k p_j (g_j - sum_k p_k g_k), g = dc/dp: |d| <= (3 kappa + (n + 12) u) k p_j (|g_j| + |sum_k p_k g_k|),
             against float64 autograd of sum_b k_b c_err_b from the logits;
      dZp:   the bf16 rounding of the kernel's own dZ, exactly, columns n .. 16 zero, rows B .. Balloc still zero;
      dbias: float atomics of ~B / 8 CTA partial sums (each of 8 rows): |d| <= sum_b |d dZ| + (B / 8 + 8) u
             sum_b |dZ|."""
    ldz = n if ldz == 'n' else ldz
    g = gen(8100 + B + n + ldz)
    Balloc = ru(B, 128)
    Z, y = logits_rows(g, B, n, ldz)
    coef = torch.rand(B, generator=g, device='cuda')
    worst = {}
    for eps in (1e-6, 0.1):
        prob = torch.full((B, n), math.nan, device='cuda')
        ce = torch.full((B,), math.nan, device='cuda'); dc = torch.full((B,), math.nan, device='cuda')
        L().softmax_ce_fwd(vp(Z), ldz, vp(y), B, n, eps, vp(prob), vp(ce), vp(dc), None)
        dZ = torch.full((B, n), math.nan, device='cuda')
        dZp = planes_with_sentinel(B, Balloc) if n <= 16 else None
        dbias = torch.zeros(n, device='cuda') if n <= 16 else None
        L().softmax_ce_bwd(vp(prob), vp(y), B, n, eps, vp(coef), 1.0 / B, vp(dZ), vp(dZp), Balloc, vp(dbias), None)
        torch.cuda.synchronize()
        z = Z[:, :n].double().requires_grad_(True)
        p, c = softmax_ce_ref(z, y, eps, n)
        k = coef.double() * float(np.float32(1.0 / B))
        (c * k).sum().backward()
        zd = z.detach()
        kappa = ((zd - zd.max(1, keepdim=True).values).abs().max(1, keepdim=True).values + n + 5) * U
        e_p = _ratio(prob, p.detach(), kappa * p.detach() + 2.0 ** -126)
        e_c = _ratio(ce, c.detach(), kappa[:, 0] + 4 * U + U * c.detach().abs())
        from oracle.torch_ref import first_argmax
        assert torch.equal(dc, (first_argmax(prob, 1) == first_argmax(y, 1)).float())
        pd = p.detach()
        a = float(np.float32(np.float32(eps) / np.float32(n))) + float(np.float32(1 - np.float32(eps))) * pd
        gr = -y.double() * float(np.float32(1 - np.float32(eps))) / a
        dot = (pd * gr).sum(1, keepdim=True)
        bz = (3 * kappa + (n + 12) * U) * k[:, None] * pd * (gr.abs() + dot.abs()) + 2.0 ** -126
        e_z = _ratio(dZ, z.grad, bz)
        r = dict(prob=e_p, c_err=e_c, dZ=e_z)
        if n <= 16:
            assert torch.equal(from_feat_t(dZp, B)[:, :n], dZ.to(torch.bfloat16))
            assert not from_feat_t(dZp, B)[:, n:].float().any() and not dZp[:, B:].float().any()
            bb = bz.sum(0) + (B / 8 + 8) * U * z.grad.abs().sum(0)
            r['dbias'] = _ratio(dbias, z.grad.sum(0), bb)
        for kk, v in r.items():
            worst[kk] = max(worst.get(kk, 0.0), v)
        assert max(r.values()) <= 1.0, (eps, r)
    print('softmax_ce B=%d n=%d ldz=%d: worst |err| / bound over eps 1e-6, 0.1: %s (tol 1 each); d_cor%s exact'
          % (B, n, ldz, ', '.join('%s %.2f' % kv for kv in worst.items()), ', dZp' if n <= 16 else ''))


@pytest.mark.parametrize('B', list(BATCHES) + [BIG])
@pytest.mark.parametrize('n', [2, 10, 16, 17, 32])
@pytest.mark.parametrize('ldz', ['n', 32])
def test_squared_err_at_scale(B, n, ldz):
    """mpnn_squared_err_fwd / _bwd on integer-valued x (ties everywhere) and targets with ties (every 4th row of
    y all zero, every 4th (offset 1) with two ones, the rest one-hot): out an exact copy of x, d_cor exact (first
    maximum of x against first maximum of y), c_err = sum (x - y)^2 (an fma chain of n terms: (n + 2) u relative,
    all terms >= 0), dZ = 2 k (x - y) (2u), dZp exact (bf16 of the kernel's dZ), dbias as in test_softmax_ce_at_scale."""
    ldz = n if ldz == 'n' else ldz
    g = gen(8300 + B + n + ldz)
    Balloc = ru(B, 128)
    Z = ints(g, (B, ldz), -2, 3)
    Z[:, n:] = 1e30
    y = Fn.one_hot(torch.randint(0, n, (B,), generator=g, device='cuda'), n).float()
    y[::4] = 0
    y[1::4, 0] = 1
    y[1::4, n - 1] = 1
    coef = torch.rand(B, generator=g, device='cuda')
    out = torch.full((B, n), math.nan, device='cuda')
    ce = torch.full((B,), math.nan, device='cuda'); dc = torch.full((B,), math.nan, device='cuda')
    L().squared_err_fwd(vp(Z), ldz, vp(y), B, n, vp(out), vp(ce), vp(dc), None)
    dZ = torch.full((B, n), math.nan, device='cuda')
    dZp = planes_with_sentinel(B, Balloc) if n <= 16 else None
    dbias = torch.zeros(n, device='cuda') if n <= 16 else None
    L().squared_err_bwd(vp(out), vp(y), B, n, vp(coef), 1.0 / B, vp(dZ), vp(dZp), Balloc, vp(dbias), None)
    torch.cuda.synchronize()
    from oracle.torch_ref import first_argmax
    x = Z[:, :n]
    assert torch.equal(out, x)
    assert torch.equal(dc, (first_argmax(x, 1) == first_argmax(y, 1)).float())
    xd = x.double().requires_grad_(True)
    c = ((xd - y.double()) ** 2).sum(1)
    k = coef.double() * float(np.float32(1.0 / B))
    (c * k).sum().backward()
    e_c = _ratio(ce, c.detach(), (n + 2) * U * c.detach())
    bz = 4 * U * xd.grad.abs()
    e_z = _ratio(dZ, xd.grad, bz + 1e-300)
    r = dict(c_err=e_c, dZ=e_z)
    if n <= 16:
        assert torch.equal(from_feat_t(dZp, B)[:, :n], dZ.to(torch.bfloat16))
        assert not from_feat_t(dZp, B)[:, n:].float().any() and not dZp[:, B:].float().any()
        r['dbias'] = _ratio(dbias, xd.grad.sum(0), bz.sum(0) + (B / 8 + 8) * U * xd.grad.abs().sum(0))
    print('squared_err B=%d n=%d ldz=%d: %s (|err| / bound, tol 1 each); out, d_cor%s exact'
          % (B, n, ldz, ', '.join('%s %.2f' % kv for kv in r.items()), ', dZp' if n <= 16 else ''))
    assert max(r.values()) <= 1.0, r


@pytest.mark.parametrize('B', [4097, BIG])
@pytest.mark.parametrize('n_cls', [10, 100])
@pytest.mark.parametrize('n_sup', [2, 5, 20])
def test_superclass_targets_at_scale(B, n_cls, n_sup):
    """mpnn_superclass_targets: y_sup = y @ w_cls.  With the 0/1 weights of a class -> superclass map (class j in
    superclass j mod n_sup) every product is exact and the result must be too; with random weights it is an fma
    chain of n_cls terms, |d| <= n_cls u sum_j |y_j w_jk|.  Every 7th row of y is a soft target of multiples of 1/8
(exact sums).  Then chained into mpnn_softmax_ce_fwd with n = n_sup,
    as the engine runs a SuperclassCrossEntropyError leaf: c_err and d_cor against the float64 restatement on
    the exact targets (bounds of test_softmax_ce_at_scale)."""
    g = gen(8500 + B + n_cls + n_sup)
    y = Fn.one_hot(torch.randint(0, n_cls, (B,), generator=g, device='cuda'), n_cls).float()
    y[::7] = torch.randint(0, 9, (len(range(0, B, 7)), n_cls), generator=g, device='cuda') / 8.0   # soft rows (dyadic)
    w01 = torch.eye(n_sup, device='cuda')[torch.arange(n_cls, device='cuda') % n_sup].contiguous()
    wr = torch.rand((n_cls, n_sup), generator=g, device='cuda')
    outs = []
    for w in (w01, wr):
        ys = torch.full((B, n_sup), math.nan, device='cuda')
        L().superclass_targets(vp(y), vp(w), B, n_cls, n_sup, vp(ys), None)
        outs.append(ys)
    Z, _ = logits_rows(g, B, n_sup, 32)
    prob = torch.zeros((B, n_sup), device='cuda'); ce = torch.zeros(B, device='cuda'); dc = torch.zeros(B, device='cuda')
    L().softmax_ce_fwd(vp(Z), 32, vp(outs[0]), B, n_sup, 1e-6, vp(prob), vp(ce), vp(dc), None)
    torch.cuda.synchronize()
    ref01 = y.double() @ w01.double()
    assert torch.equal(outs[0].double(), ref01)
    refr = y.double() @ wr.double()
    e = _ratio(outs[1], refr, n_cls * U * (y.double().abs() @ wr.double().abs()))
    from oracle.torch_ref import first_argmax
    z = Z[:, :n_sup].double()
    p, c = softmax_ce_ref(z, ref01, 1e-6, n_sup)
    kappa = ((z - z.max(1, keepdim=True).values).abs().max(1).values + n_sup + 5) * U
    # c_err = -sum_k y_k log(a_k) with soft targets: |d| <= sum_k y_k (kappa + 4u + u |log a_k|)
    a = float(np.float32(np.float32(1e-6) / np.float32(n_sup))) + float(np.float32(1 - np.float32(1e-6))) * p
    bc = (ref01 * (kappa[:, None] + 4 * U + U * torch.log(a).abs())).sum(1) + n_sup * U * c.abs()
    e_c = _ratio(ce, c, bc + 1e-300)
    assert torch.equal(dc, (first_argmax(prob, 1) == first_argmax(outs[0], 1)).float())
    print('superclass_targets B=%d n_cls=%d n_sup=%d: 0/1 weights exact, random weights %.2f of the bound, '
          'chained c_err %.2f of the bound, d_cor exact' % (B, n_cls, n_sup, e, e_c))
    assert e <= 1.0 and e_c <= 1.0



# --------------------------------------------------------------------------- #
# compaction copies and the optimiser step
# --------------------------------------------------------------------------- #
CAP = 4096


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('H,C', [(32, 16), (16, 32), (8, 64), (4, 128)])
def test_gather_scatter_images_at_scale(H, C, dt):
    """mpnn_gather_images / mpnn_scatter_add_images between planes tensors of capacity 4096 at every stage
    geometry, with counts 0, 1, 4095 and 4096 (at 32x32x16 the capped grid of 148*16 CTAs makes 15 grid-stride
    passes).  Gather: destination image j is the whole S-row block of source image idx[j], the rest of the
    destination untouched.  Scatter-add into a destination that is not zero: block idx[j] += block j, one fp32
    addition rounded once to the storage type, the rest untouched.  All exact."""
    g = gen(8700 + H + dt)
    geo = Geo(CAP, H, H)
    KG, S = C // 8, geo.S
    src = to_planes_t(rnd(g, (CAP, H, H, C), dt), geo).to(TD[dt])
    base = to_planes_t(rnd(g, (CAP, H, H, C), dt), geo).to(TD[dt])
    blk = lambda t: t[:, geo.G:geo.G + CAP * S].view(KG, CAP, S, 8)
    for count in (0, 1, CAP - 1, CAP):
        idx = torch.randperm(CAP, generator=g, device='cuda')[:count].sort().values.int()
        idx_full = torch.zeros(CAP, dtype=torch.int32, device='cuda')
        idx_full[:count] = idx
        cnt = torch.tensor([count], dtype=torch.int32, device='cuda')
        dst = torch.full_like(src, 3.0)
        L().gather_images(vp(src), CAP, geo.P, vp(idx_full), vp(cnt), vp(dst), CAP, geo.P, C, H, H, geo.G, dt, None)
        acc = base.clone()
        L().scatter_add_images(vp(src), CAP, geo.P, vp(idx_full), vp(cnt), vp(acc), CAP, geo.P, C, H, H, geo.G, dt, None)
        torch.cuda.synchronize()
        il = idx.long()
        want = torch.full_like(src, 3.0)
        blk(want)[:, :count] = blk(src)[:, il]
        assert torch.equal(dst, want), count
        want = base.clone()
        blk(want)[:, il] = (blk(base)[:, il].float() + blk(src)[:, :count].float()).to(TD[dt])
        assert torch.equal(acc, want), count
    print('gather / scatter-add %dx%dx%d %s, counts 0, 1, 4095, 4096: exact (tol 0)' % (H, H, C, 'fp32' if dt == F32 else 'bf16'))


@pytest.mark.parametrize('net', ['ac_chain', 'ac_tree'])
@pytest.mark.parametrize('talr,stats', [(0, False), (1, False), (0, True), (1, True)])
@pytest.mark.parametrize('gscale', [1.0, 0.125])
def test_talr_momentum_step_at_scale(net, talr, stats, gscale):
    """mpnn_talr_momentum_step over the parameter buffer of the full-size net (n_theta 680,826 in 178 segments for
    ac_chain, 5,010,238 in 917 for ac_tree: the grid of 148*8 CTAs of 256 threads makes up to 17 grid-stride
    passes, and every segment boundary is crossed) against a float64 restatement of csrc/optim.cu element by
    element:  coef = m1 gs, scale = mult / sqrt(m2 gs) (talr, node stats present), g = (grad gs + 2 l2 coef theta)
    scale, a = mu a + g, theta -= lr a.  Each fp32 operation rounds once, so |d a| <= 10 u (mu |a| + |g terms|)
    and |d theta| <= lr (|d a| + 2u |a|) + 2u |theta|: the last rounding alone reaches u |theta| at the bottom of
    a binade (measured: 0.99 u |theta|), the second u leaves room for everything of second order."""
    _, n_theta, n_nodes, seg = _plan_of(net)
    g = gen(8900 + n_theta % 1000 + 10 * talr + int(stats) + int(8 * gscale))
    seg = {k: v.cuda() for k, v in seg.items()}
    n_seg = seg['seg_node'].numel()
    th = torch.randn(n_theta, generator=g, device='cuda')
    gr = torch.randn(n_theta, generator=g, device='cuda')
    acc = torch.randn(n_theta, generator=g, device='cuda')
    m2 = 0.01 + 0.5 * torch.rand(n_nodes, generator=g, device='cuda')
    m1 = m2.sqrt() + (1 - m2.sqrt()) * torch.rand(n_nodes, generator=g, device='cuda')
    st = (torch.stack([m2, m1], 1) / gscale).contiguous() if stats else None     # moments ride in the scaled tail
    hyp = torch.zeros(8, device='cuda')
    hyp[0], hyp[1], hyp[5] = 0.05, 0.9, gscale
    TH, A = th.clone(), acc.clone()
    L().talr_momentum_step(vp(TH), vp(gr), vp(A), n_theta, vp(seg['seg_start']), vp(seg['seg_node']),
                           vp(seg['seg_mult']), vp(seg['seg_l2']), n_seg, vp(st), talr, vp(hyp), None)
    torch.cuda.synchronize()
    sid = torch.repeat_interleave(torch.arange(n_seg, device='cuda'), (seg['seg_start'][1:] - seg['seg_start'][:-1]).long())
    node = seg['seg_node'].long()[sid]
    mult, l2 = seg['seg_mult'].double()[sid], seg['seg_l2'].double()[sid]
    gs, lr, mu = float(np.float32(gscale)), float(np.float32(0.05)), float(np.float32(0.9))
    if stats:
        coef = st[:, 1].double()[node] * gs
        scale = mult / torch.sqrt(st[:, 0].double()[node] * gs) if talr else mult
    else:
        coef, scale = torch.ones_like(mult), mult
    t0, t1 = gr.double() * gs, 2 * l2 * coef * th.double()
    a = mu * acc.double() + (t0 + t1) * scale
    thn = th.double() - lr * a
    ba = 10 * U * (mu * acc.double().abs() + (t0.abs() + t1.abs()) * scale.abs())
    bt = lr * (ba + 2 * U * a.abs()) + 2 * U * thn.abs()
    e = (_ratio(A, a, ba + 1e-300), _ratio(TH, thn, bt + 1e-300))
    print('talr_momentum_step %s n=%d talr=%d stats=%s gscale=%g: accum %.2f, theta %.2f of the bound (tol 1)'
          % (net, n_theta, talr, stats, gscale, *e))
    assert max(e) <= 1.0
