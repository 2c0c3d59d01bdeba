"""Graph-replayed routed inference (`Net.predictor`, lib/compact_eval.py RoutedPredictor): the counted entry points
(live batch read from device memory, grid sized for a capacity) against the uncounted ones called with the live
batch, bit for bit, with the rows past the count untouched; the predictor against `Net.predict`, bit for bit; no host
synchronisation per call; and `classify-net --graph` against the run without it."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'multipath-nn_b200')
for p in (ROOT, PKG, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

from util import Geo, batch, randomize_routers, to_planes, tiny_net  # noqa: E402

pytestmark = pytest.mark.gpu
F32, BF16 = 0, 1
K_MIX = np.array([0.0, 4e-9, 1.6e-8, 6.4e-8], np.float32)
CASES = [('ac', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('sr', {}),
         ('ac', dict(dyn_k_cpt=True))]
_KEEP = []


def L():
    from lib import _cabi
    return _cabi.lib()


def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    t = t if dtype is None else t.to(dtype)
    _KEEP.append(t)                   # the kernels are asynchronous: keep inputs alive until the test syncs
    return t


def counts(B):
    return sorted({0, 1, 37, B - 1, B})


def cnt_of(m):
    return dev(np.array([m], np.int32))


def bits(t):
    t = t.detach().cpu()
    return t.view(torch.int16 if t.element_size() == 2 else (torch.int64 if t.element_size() == 8 else torch.int32))


def same(a, b):
    assert a.shape == b.shape and torch.equal(bits(a), bits(b))


def untouched(t, sentinel):
    assert torch.equal(bits(t), bits(torch.full_like(t, sentinel)))


# ---------------------------------------------------------------- counted kernels
@pytest.mark.parametrize('dt,impl', [(BF16, 1), (F32, 0)])
def test_stencil_gemm_counted_conv(dt, impl):
    """3x3 conv with a pooled second operand (A1), tcgen05 and SIMT"""
    B, H, K0, K1, N = 70, 8, 16, 16, 32
    rng = np.random.default_rng(1)
    geo = Geo(B, H, H)
    td = torch.bfloat16 if dt == BF16 else torch.float32
    A0 = dev(to_planes(rng.standard_normal((B, H, H, K0)).astype(np.float32), geo), td)
    A1 = dev(to_planes(rng.standard_normal((B, H, H, K1)).astype(np.float32), geo), td)
    Wp = dev(rng.standard_normal((9, (K0 + K1) // 8, N, 8)).astype(np.float32) * 0.1, td)
    bias = dev(rng.standard_normal(N).astype(np.float32))
    for m in counts(B):
        ref = torch.full((N // 8, geo.P, 8), 7.0, dtype=td, device='cuda')
        got = torch.full_like(ref, 7.0)
        if m:
            L().stencil_gemm(vp(A0), K0, vp(A1), K1, vp(Wp), 9, vp(bias), vp(ref), N, 0, None, 0, 0,
                             m, H, H, geo.G, geo.P, None, 0, None, dt, dt, impl, None)
        L().stencil_gemm_counted(vp(A0), K0, vp(A1), K1, vp(Wp), 9, vp(bias), vp(got), N, 0, None, 0, 0,
                                 B, H, H, geo.G, geo.P, None, 0, None, dt, dt, impl, vp(cnt_of(m)), None)
        torch.cuda.synchronize()
        end = geo.G + m * geo.S
        same(got[:, geo.G:end], ref[:, geo.G:end])
        untouched(got[:, end:], 7.0)
        untouched(got[:, :geo.G], 7.0)


def test_stencil_gemm_counted_head_gemm():
    """the H = W = 0 head GEMM [W_leaf | W_r1] with fp32 row-major outputs"""
    B, Fext = 300, 64
    Balloc = (B + 127) // 128 * 128
    rng = np.random.default_rng(2)
    X = dev(rng.standard_normal((Fext // 8, Balloc, 8)).astype(np.float32), torch.bfloat16)
    Wfc = dev(rng.standard_normal((1, Fext // 8, 32, 8)).astype(np.float32) * 0.1, torch.bfloat16)
    bias = dev(rng.standard_normal(32).astype(np.float32))
    for m in counts(B):
        outs = [torch.full((B, 16), -5.0, device='cuda') for _ in range(4)]
        if m:
            L().stencil_gemm(vp(X), Fext, None, 0, vp(Wfc), 1, vp(bias), vp(outs[0]), 16, 0, vp(outs[1]), 16, 0,
                             m, 0, 0, 0, Balloc, None, 0, None, BF16, 2, 1, None)
        L().stencil_gemm_counted(vp(X), Fext, None, 0, vp(Wfc), 1, vp(bias), vp(outs[2]), 16, 0, vp(outs[3]), 16, 0,
                                 B, 0, 0, 0, Balloc, None, 0, None, BF16, 2, 1, vp(cnt_of(m)), None)
        torch.cuda.synchronize()
        for r, g in ((outs[0], outs[2]), (outs[1], outs[3])):
            same(g[:m], r[:m])
            untouched(g[m:], -5.0)


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('mode', ['pooled', 'feat'])
def test_bn_relu_pool_fwd_counted(dt, mode):
    B, H, C = 90, 8, 16
    rng = np.random.default_rng(3)
    geo, gp = Geo(B, H, H), Geo(B, H // 2, H // 2)
    assert gp.G == geo.G
    td = torch.bfloat16 if dt == BF16 else torch.float32
    lin = dev(to_planes(rng.standard_normal((B, H, H, C)).astype(np.float32), geo), td)
    ss = dev(np.concatenate([rng.random(C) + 0.5, rng.standard_normal(C)]).astype(np.float32))
    Balloc = (B + 127) // 128 * 128
    for m in counts(B):
        def outs():
            act = torch.full((C // 8, geo.P, 8), 3.0, dtype=td, device='cuda')
            if mode == 'pooled':
                return act, torch.full((C // 8, gp.P, 8), 3.0, dtype=td, device='cuda'), None
            return act, None, torch.full((H * H * C // 8, Balloc, 8), 3.0, dtype=td, device='cuda')
        ra, rp, rf = outs()
        ga, gpool, gf = outs()
        Pp = gp.P if mode == 'pooled' else 0
        if m:
            L().bn_relu_pool_fwd(vp(lin), C, m, H, H, geo.G, geo.P, vp(ss), vp(ra), vp(rp), Pp, vp(rf), Balloc, dt, None)
        L().bn_relu_pool_fwd_counted(vp(lin), C, B, H, H, geo.G, geo.P, vp(ss), vp(ga), vp(gpool), Pp, vp(gf), Balloc,
                                     dt, vp(cnt_of(m)), None)
        torch.cuda.synchronize()
        end = geo.G + m * geo.S
        same(ga[:, :end], ra[:, :end])
        untouched(ga[:, end:], 3.0)
        if mode == 'pooled':
            endp = gp.G + m * gp.S
            same(gpool[:, :endp], rp[:, :endp])
            untouched(gpool[:, endp:], 3.0)
        else:
            same(gf[:, :m], rf[:, :m])
            untouched(gf[:, m:], 3.0)


@pytest.mark.parametrize('dt', [F32, BF16])
def test_fc_fwd_counted_with_extra(dt):
    B, F, n = 200, 64, 16
    Balloc = 256
    rng = np.random.default_rng(4)
    td = torch.bfloat16 if dt == BF16 else torch.float32
    X = dev(rng.standard_normal((F // 8, Balloc, 8)).astype(np.float32), td)
    W = dev(rng.standard_normal((F + 1, n)).astype(np.float32) * 0.1)
    bias = dev(rng.standard_normal(n).astype(np.float32))
    extra = dev(rng.random(Balloc).astype(np.float32))
    for m in counts(B):
        ref = torch.full((B, n), 9.0, device='cuda')
        got = torch.full_like(ref, 9.0)
        if m:
            L().fc_fwd(vp(X), F, Balloc, m, vp(W), vp(bias), vp(extra), n, vp(ref), dt, None)
        L().fc_fwd_counted(vp(X), F, Balloc, B, vp(W), vp(bias), vp(extra), n, vp(got), dt, vp(cnt_of(m)), None)
        torch.cuda.synchronize()
        same(got[:m], ref[:m])
        untouched(got[m:], 9.0)


@pytest.mark.parametrize('B', [1000, 3000, 6000, 9000])      # RPT 1 / 2 / 4 and the re-reading cluster kernel
def test_router_tail_fwd_batched_counted(B):
    from lib.engine import _RT_FWD
    rng = np.random.default_rng(B)
    C, ns = 16, 3
    Z1 = dev(rng.standard_normal((B, C)).astype(np.float32) * 2 + 0.3)
    P = {k: dev(rng.standard_normal(sh).astype(np.float32) * sc) for k, sh, sc in [
        ('g1', C, 1), ('b1', C, .3), ('W2', (C, C), .3), ('c2', C, .1), ('g2', C, 1), ('b2', C, .3),
        ('W3', (C, ns), .3), ('c3', ns, .1)]}
    mom = [dev(np.full(C, v, np.float32)) for v in (0.1, 1.5, -0.2, 0.7)]

    def run(n, count):
        Z2 = torch.full((B, C), -1.0, device='cuda')
        R = torch.full((B, ns), -1.0, device='cuda')
        save = torch.full((64,), -1.0, device='cuda')
        ptr = lambda t: t.data_ptr()
        row = (ptr(Z1), ptr(P['g1']), ptr(P['b1']), ptr(mom[0]), ptr(mom[1]), ptr(P['W2']), ptr(P['c2']),
               ptr(P['g2']), ptr(P['b2']), ptr(mom[2]), ptr(mom[3]), ptr(P['W3']), ptr(P['c3']),
               ptr(Z2), ptr(R), ptr(save), ns, 0)
        table = dev(np.frombuffer(np.array([row], dtype=_RT_FWD).tobytes(), np.uint8).copy(), torch.uint8)
        if count is None:
            if n:
                L().router_tail_fwd_batched(vp(table), 1, n, C, 0.9, 1e-6, 0, None)
        else:
            L().router_tail_fwd_batched_counted(vp(table), 1, B, C, 0.9, 1e-6, 0, vp(count), None)
        torch.cuda.synchronize()
        return Z2, R, save

    for m in counts(B):
        rz, rr, rs = run(m, None)
        gz, gr, gs = run(B, cnt_of(m))
        same(gz[:m], rz[:m]); untouched(gz[m:], -1.0)
        same(gr[:m], rr[:m]); untouched(gr[m:], -1.0)
        if m:
            same(gs, rs)


@pytest.mark.parametrize('ns', [2, 8])
def test_route_compact_counted_with_parent_orig(ns):
    B = 3000
    rng = np.random.default_rng(ns)
    R = dev(rng.standard_normal((B, ns)).astype(np.float32))
    porig = dev(rng.permutation(5000)[:B].astype(np.int32))
    for m in counts(B):
        def outs():
            return (torch.full((ns, B), -4, dtype=torch.int32, device='cuda'),
                    torch.full((ns, B), -4, dtype=torch.int32, device='cuda'),
                    torch.full((ns,), -4, dtype=torch.int32, device='cuda'))
        rp, ro, rc = outs()
        gp, go, gc = outs()
        L().route_compact(vp(R), ns, ns, m, vp(porig), B, None, vp(rp), vp(ro), vp(rc), None)
        L().route_compact_counted(vp(R), ns, ns, B, vp(porig), B, None, vp(gp), vp(go), vp(gc), vp(cnt_of(m)), None)
        torch.cuda.synchronize()
        same(gc, rc)
        same(gp, rp)
        same(go, ro)
        assert int(gc.sum()) == m


@pytest.mark.parametrize('dt,step', [(F32, 1), (BF16, 2)])
def test_pack_input_counted(dt, step):
    B, H0, C0, Cpad = 80, 16, 3, 8
    rng = np.random.default_rng(5)
    x0 = dev(rng.random((B, H0, H0, C0)).astype(np.float32))
    geo = Geo(B, H0 // step, H0 // step)
    td = torch.bfloat16 if dt == BF16 else torch.float32
    for m in counts(B):
        ref = torch.full((Cpad // 8, geo.P, 8), 2.0, dtype=td, device='cuda')
        got = torch.full_like(ref, 2.0)
        L().pack_input(vp(x0), m, H0, H0, C0, step, vp(ref), Cpad, geo.G, geo.P, dt, None)
        L().pack_input_counted(vp(x0), B, H0, H0, C0, step, vp(got), Cpad, geo.G, geo.P, dt, vp(cnt_of(m)), None)
        torch.cuda.synchronize()
        same(got, ref)


# ---------------------------------------------------------------- the predictor against net.predict
def _trained(kind, hy, prec, seed=2):
    net = tiny_net(kind, seed=seed, **hy)
    if net.dynamic:
        randomize_routers(net)
    net.configure(precision=prec)
    x0, y = batch(64, seed=3)
    for t in range(2):                                   # non-trivial running BN moments
        net.train.run(_train_feed(net, hy, x0, y))
    return net


def _train_feed(net, hy, x0, y):
    f = {net.x0: x0, net.y: y, net.mode: 'tr', net.λ_lrn: 0.01}
    if net.dynamic:
        f[net.τ] = 0.5
    if hy.get('dyn_k_cpt'):
        f[net.k_cpt] = np.full(len(x0), 4e-9, np.float32)
    return f


def _mixed_k(n, seed=5):
    return np.random.default_rng(seed).choice(K_MIX, n)


def _equal(got, want):
    for f in ('cls', 'prob', 'exit', 'ops'):
        g = getattr(got, f)
        assert g.is_cuda, f
        g = g.cpu().numpy()
        w = getattr(want, f)
        assert g.dtype == w.dtype and g.shape == w.shape and g.tobytes() == w.tobytes(), f


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('kind,hy', CASES)
def test_predictor_equals_predict(kind, hy, prec):
    net = _trained(kind, hy, prec)
    n = 200
    x0, _ = batch(n, seed=9)
    kc = _mixed_k(n) if hy.get('dyn_k_cpt') else None
    want = net.predict(x0, k_cpt=kc, batch=256)
    p = net.predictor(256)
    assert net.predictor(256) is p
    _equal(p(x0, k_cpt=kc), want)
    if net.dynamic:
        assert len(set(want.exit.tolist())) > 1


def test_one_graph_serves_every_n():
    net = _trained('actree', dict(k_cpt=2e-9), 'bf16')
    B = 128
    p = net.predictor(B)
    x0, _ = batch(3 * B, seed=12)
    xd = torch.from_numpy(x0).cuda()
    graph = None
    for n in (B, 1, 77, B - 1, 5, B):
        lo = n % 50
        _equal(p(xd[lo:lo + n]), net.predict(x0[lo:lo + n], batch=B))
        graph = graph or p.graph
        assert p.graph is graph                          # captured once, replayed
    e = p(xd[:0])
    assert e.prob.shape == (0, 10) and e.cls.shape == e.exit.shape == e.ops.shape == (0,)
    with pytest.raises(ValueError, match='capacity'):
        p(xd[:B + 1])


def test_mixed_k_cpt_and_device_k_cpt():
    net = _trained('ac', dict(dyn_k_cpt=True), 'bf16')
    n = 150
    x0, _ = batch(n, seed=14)
    kc = _mixed_k(n, seed=8)
    p = net.predictor(160)
    want = net.predict(x0, k_cpt=kc, batch=160)
    _equal(p(x0, k_cpt=kc), want)
    _equal(p(torch.from_numpy(x0).cuda(), k_cpt=torch.from_numpy(kc).cuda()), want)
    _equal(p(x0, k_cpt=1.6e-8), net.predict(x0, k_cpt=1.6e-8, batch=160))
    assert len(set(want.ops.tolist())) > 1


@pytest.mark.parametrize('kind,hy', [('ac', dict(k_cpt=4e-9)), ('ac', dict(dyn_k_cpt=True))])
def test_a_call_after_a_training_step_sees_the_new_parameters(kind, hy):
    net = _trained(kind, hy, 'bf16')
    x0, y = batch(100, seed=15)
    kc = 4e-9 if hy.get('dyn_k_cpt') else None
    p = net.predictor(128)
    before = p(x0, k_cpt=kc)
    before = {f: getattr(before, f).cpu().numpy() for f in ('cls', 'prob', 'exit', 'ops')}
    xt, yt = batch(64, seed=16)
    net.train.run(_train_feed(net, hy, xt, yt))
    want = net.predict(x0, k_cpt=kc, batch=128)
    assert want.prob.tobytes() != before['prob'].tobytes()            # the step changed the answers
    _equal(p(x0, k_cpt=kc), want)


def test_no_host_synchronisation_with_device_inputs():
    net = _trained('ac', dict(dyn_k_cpt=True), 'bf16')
    x0, _ = batch(100, seed=17)
    xd = torch.from_numpy(x0).cuda()
    kd = torch.from_numpy(_mixed_k(100, seed=9)).cuda()
    p = net.predictor(128)
    p(xd, k_cpt=kd)                                      # first call: capture (synchronises once)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        out = p(xd, k_cpt=kd)
        out2 = p(xd[:50], k_cpt=kd[:50])
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert out2.cls.shape == (50,)
    want = net.predict(x0[:50], k_cpt=kd[:50].cpu().numpy(), batch=128)
    _equal(out2, want)
    del out


@pytest.mark.parametrize('arch', ['ac_chain', 'ac_tree'])
def test_full_architecture_with_randomized_routers(arch):
    import arch_and_hypers as ah
    from lib import layer_types
    layer_types.seed(0)
    net = getattr(ah, arch)(k_cpt=4e-9)((32, 32, 3), (10,))
    randomize_routers(net)
    net.configure(precision='bf16')
    x0 = np.random.default_rng(1).random((512, 32, 32, 3)).astype(np.float32)
    want = net.predict(x0, batch=512)
    _equal(net.predictor(512)(x0), want)
    assert len(set(want.exit.tolist())) > 1


# ---------------------------------------------------------------- driver
def _run(script, args, cwd):
    r = subprocess.run([sys.executable, os.path.join(PKG, script)] + args, cwd=cwd, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout


def test_classify_net_graph_equals_the_host_walk(tmp_path):
    _run('train-nets', ['cifar10-ac', '--synthetic', '--n-iter', '20', '--t-log', '20', '--nets', '0'], str(tmp_path))
    _run('train-adaptive-nets', ['hybrid-ac-dynkcpt', '--synthetic', '--n-iter', '20'], str(tmp_path))
    for net, extra in (('nets/cifar10-ac/0000.npy', []), ('nets/hybrid-ac-dynkcpt/net.npy', ['--k-cpt', '0', '1.6e-8'])):
        args = [str(tmp_path / net), '--synthetic', '--batch', '200'] + extra
        a = _run('classify-net', args + ['--out', 'a.npz'], str(tmp_path))
        b = _run('classify-net', args + ['--graph', '--out', 'b.npz'], str(tmp_path))
        assert a == b
        da, db = np.load(tmp_path / 'a.npz'), np.load(tmp_path / 'b.npz')
        assert sorted(da.files) == sorted(db.files)
        for f in da.files:
            assert da[f].dtype == db[f].dtype and da[f].shape == db[f].shape and da[f].tobytes() == db[f].tobytes(), f
