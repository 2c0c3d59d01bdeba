"""Kernel parity at the benchmark's batch (B200): libmpnn_sm100 entry points, called through the C ABI at
B = 4096 and the ragged 4095 / 4097 on the real architecture's stages (32x32x16 .. 4x4x128), against float64
references computed on the device with plain torch.

At these sizes the grid-stride loops run their second and later passes, the BN statistics are the two-pass
(not the one-launch) kernels, the head GEMMs see a partly-filled 128-row tile, and every reduction is thousands
of times longer than in test_kernels_gpu.py.  Tolerances are derived in each docstring; u = 2^-24 is the fp32
unit roundoff.  Run with -s to see the measured errors."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as Fn

from util import Geo, dropout_mask_t, from_feat_t, from_planes_t, to_feat_t, to_planes_t

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
