"""Routed inference (`Net.predict`, lib/compact_eval.py, `classify-net`): the leaf-emit and feature-gather kernels
against NumPy, predictions against the dense 'ev' pass (an example's arithmetic does not depend on its batch-mates,
so prob is expected bit-equal and ops exactly the dense moc), chunking, per-example k_cpt, the full architecture
against the oracle, and the driver."""
import ctypes
import os
import re
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

from oracle.torch_ref import OracleNet  # noqa: E402
from util import batch, node_paths, randomize_routers, record_of, tiny_net  # noqa: E402

pytestmark = pytest.mark.gpu
K_MIX = np.array([0.0, 4e-9, 1.6e-8, 6.4e-8], np.float32)


def L():
    from lib import _cabi
    return _cabi.lib()


def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---------------------------------------------------------------- kernels
@pytest.mark.parametrize('n_cls', [2, 10, 16, 17, 32])
def test_leaf_emit_matches_numpy(n_cls):
    rng = np.random.default_rng(n_cls)
    n_par, n_out, n, live = 300, 500, 200, 150          # parent rows, original ids, host bound, device count
    ldz = n_cls + 3
    Z = rng.standard_normal((n_par, ldz)).astype(np.float32)
    tie = rng.choice(n_par, 40, replace=False)
    Z[tie, n_cls - 1] = Z[tie, 0] = Z[tie, :n_cls].max(1) + 1.0           # tied maxima: the first index wins
    pos = rng.permutation(n_par)[:n].astype(np.int32)
    orig = rng.permutation(n_out)[:n].astype(np.int32)
    prob = torch.full((n_out, n_cls), -7.0, device='cuda')
    cls = torch.full((n_out,), -7, dtype=torch.int32, device='cuda')
    ext = torch.full_like(cls, -7)
    ops = torch.full((n_out,), -7.0, dtype=torch.float64, device='cuda')
    cnt = torch.tensor([live], dtype=torch.int32, device='cuda')
    Zd, pd, od = dev(Z), dev(pos), dev(orig)
    L().leaf_emit(vp(Zd), ldz, n_cls, vp(pd), vp(od), vp(cnt), n, 3, 1.25e6, vp(prob), vp(cls), vp(ext), vp(ops), None)
    L().leaf_emit(vp(Zd), ldz, n_cls, None, None, None, 0, 5, 9.0, None, None, None, None, None)     # n = 0: no-op
    # the dense path's softmax on the same rows
    rows = Zd[dev(pos[:live]).long()].contiguous()
    y = torch.zeros((live, n_cls), device='cuda')
    y[:, 0] = 1
    ref = torch.empty((live, n_cls), device='cuda')
    ce, dc = torch.empty(live, device='cuda'), torch.empty(live, device='cuda')
    L().softmax_ce_fwd(vp(rows), ldz, vp(y), live, n_cls, 0.0, vp(ref), vp(ce), vp(dc), None)
    torch.cuda.synchronize()
    P, C, E, O = prob.cpu().numpy(), cls.cpu().numpy(), ext.cpu().numpy(), ops.cpu().numpy()
    o = orig[:live]
    np.testing.assert_array_equal(P[o].view(np.int32), ref.cpu().numpy().view(np.int32))         # same bits
    z = Z[pos[:live], :n_cls].astype(np.float64)
    want = np.exp(z - z.max(1, keepdims=True))
    want /= want.sum(1, keepdims=True)
    np.testing.assert_allclose(P[o], want, rtol=0, atol=1e-6)
    np.testing.assert_array_equal(C[o], P[o].argmax(1))                                          # first argmax
    tied = np.isin(pos[:live], tie)
    assert tied.any() and (C[o][tied] == 0).all()
    assert (E[o] == 3).all() and (O[o] == 1.25e6).all()
    rest = np.setdiff1d(np.arange(n_out), o)                                  # rows not addressed keep the sentinel
    assert (P[rest] == -7).all() and (C[rest] == -7).all() and (E[rest] == -7).all() and (O[rest] == -7).all()


def test_gather_feature_matches_numpy():
    rng = np.random.default_rng(4)
    n_src, n, live = 1000, 600, 450
    src = (rng.random(n_src) * 10.0 ** rng.integers(-3, 3, n_src)).astype(np.float32)
    # exact bf16 halfway points: round to even both ways
    src[:8] = np.array([1 + 2 ** -8, 1 + 3 * 2 ** -8, 2 + 2 ** -7, 0.16, 0.04, 0.64, 1e7 * 4e-9, 1e7 * 6.4e-8], np.float32)
    orig = rng.permutation(n_src)[:n].astype(np.int32)
    orig[:8] = np.arange(8)
    sd, od = dev(src), dev(orig)
    cnt = torch.tensor([live], dtype=torch.int32, device='cuda')
    dst = torch.full((n,), -1.0, device='cuda')
    col = torch.full((n, 8), -3.0, device='cuda').to(torch.bfloat16)
    L().gather_feature(vp(sd), vp(od), vp(cnt), n, vp(dst), vp(col), 8, 1, None)
    col32 = torch.full((n, 4), -3.0, device='cuda')
    L().gather_feature(vp(sd), None, None, n, None, vp(col32), 4, 0, None)           # orig NULL, count NULL
    L().gather_feature(vp(sd), vp(od), vp(cnt), 0, vp(dst), None, 0, 0, None)       # n = 0: no-op
    torch.cuda.synchronize()
    g = src[orig[:live]]
    D = dst.cpu().numpy()
    np.testing.assert_array_equal(D[:live], g)
    assert (D[live:] == -1).all()
    want = torch.from_numpy(g).cuda().to(torch.bfloat16)        # torch's fp32 -> bf16 copy_
    got = col.cpu()
    assert torch.equal(got[:live, 0].view(torch.int16), want.cpu().view(torch.int16))
    assert (got[live:, 0] == -3).all() and (got[:, 1:] == -3).all()
    c32 = col32.cpu().numpy()
    np.testing.assert_array_equal(c32[:, 0], src[:n])
    assert (c32[:, 1:] == -3).all()


# ---------------------------------------------------------------- net.predict against the dense pass
def _trained(kind, hy, prec, seed=2):
    net = tiny_net(kind, seed=seed, **hy)
    if net.dynamic:
        randomize_routers(net)
    net.configure(precision=prec)
    x0, y = batch(64, seed=3)
    for t in range(2):                                   # non-trivial running BN moments
        f = {net.x0: x0, net.y: y, net.mode: 'tr', net.λ_lrn: 0.01}
        if net.dynamic:
            f[net.τ] = 0.5
        if hy.get('dyn_k_cpt'):
            f[net.k_cpt] = np.full(64, 4e-9, np.float32)
        net.train.run(f)
    return net


def _mixed_k(n, seed=5):
    return np.random.default_rng(seed).choice(K_MIX, n)


CASES = [('ac', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('sr', {}),
         ('ac', dict(dyn_k_cpt=True))]


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('kind,hy', CASES)
def test_predict_equals_the_dense_path(kind, hy, prec):
    net = _trained(kind, hy, prec)
    eng = net._get_engine()
    n = 200
    x0, y = batch(n, seed=9)
    kc = _mixed_k(n) if hy.get('dyn_k_cpt') else None
    feed = {net.x0: x0, net.y: y}
    if net.dynamic:
        feed[net.τ] = 0.5
    if kc is not None:
        feed[net.k_cpt] = kc
    moc = net.eval_stats(feed)[(net, 'moc')]
    plan = eng._plan(n, False, False)                    # the buffers of that dense forward
    p_ev = plan.p_ev.cpu().numpy() if net.dynamic else np.ones((len(eng.nodes), n), np.float32)
    got = net.predict(x0, k_cpt=kc, batch=128)           # two chunks: 128 + 72
    assert got.cls.dtype == np.int32 and got.exit.dtype == np.int32 and got.ops.dtype == np.float64
    assert got.prob.dtype == np.float32 and got.prob.shape == (n, 10)
    seen = np.zeros(n, bool)
    worst = 0.0
    for i, leaf in enumerate(eng.leaves):
        here = p_ev[leaf.idx] == 1
        assert not (seen & here).any()
        seen |= here
        np.testing.assert_array_equal(got.exit == i, here)
        dense = plan.reg[leaf.idx].prob.cpu().numpy()[:n]
        worst = max(worst, float(np.abs(got.prob[here] - dense[here]).max(initial=0.0)))
        np.testing.assert_array_equal(got.cls[here], dense[here].argmax(1))
    assert seen.all()
    print('predict vs dense %s %s %s: max |prob difference| %g' % (kind, hy, prec, worst))
    assert worst <= 1e-6
    np.testing.assert_array_equal(got.ops, moc)
    if net.dynamic:
        assert len(set(got.exit.tolist())) > 1                  # the routers spread the examples


def test_predict_in_chunks_equals_one_call():
    net = _trained('ac', dict(dyn_k_cpt=True), 'bf16')
    n = 160                                                # 2.5 x batch
    x0, _ = batch(n, seed=11)
    kc = _mixed_k(n, seed=6)
    one = net.predict(x0, k_cpt=kc, batch=256)
    chunked = net.predict(torch.from_numpy(x0).cuda(), k_cpt=torch.from_numpy(kc), batch=64)      # device input
    for f in ('cls', 'prob', 'exit', 'ops'):
        a, b = getattr(one, f), getattr(chunked, f)
        assert a.shape == b.shape and a.tobytes() == b.tobytes(), f
    empty = net.predict(x0[:0], k_cpt=kc[:0], batch=64)
    assert empty.prob.shape == (0, 10) and empty.cls.shape == empty.exit.shape == empty.ops.shape == (0,)


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
def test_per_example_k_cpt_equals_the_scalar_call_on_each_subset(prec):
    net = _trained('ac', dict(dyn_k_cpt=True), prec)
    n = 240
    x0, y = batch(n, seed=13)
    kc = _mixed_k(n, seed=7)
    vec = net.predict(x0, k_cpt=kc, batch=128)
    for k in K_MIX:
        sub = kc == k
        one = net.predict(x0[sub], k_cpt=float(k), batch=128)
        for f in ('cls', 'prob', 'exit', 'ops'):
            assert getattr(vec, f)[sub].tobytes() == getattr(one, f).tobytes(), (k, f)
    assert len(set(vec.ops.tolist())) > 1
    # the statistics entry point takes the same vector: equal to the dense means on the exact keys
    feed = {net.x0: x0, net.y: y, net.τ: 0.5, net.k_cpt: kc}
    dense = {k: np.asarray(v, np.float64).mean(0) for k, v in net.eval_stats(feed).items()}
    ev = net.compact_evaluator(128)
    ev.reset()
    for i in range(0, n, 128):
        ev.run_batch(x0[i:i + 128], y[i:i + 128], k_cpt=kc[i:i + 128])
    got = ev.result()
    assert got[(net, 'acc')] == pytest.approx(dense[(net, 'acc')], abs=1e-12)
    assert got[(net, 'moc')] == pytest.approx(dense[(net, 'moc')], rel=1e-12)
    for leaf in net.leaves:
        for name in ('p_cor', 'p_inc', 'p_cor_by_cls', 'p_inc_by_cls'):
            np.testing.assert_allclose(got[(leaf, name)], dense[(leaf, name)], rtol=0, atol=1e-12)


# ---------------------------------------------------------------- full architecture against the oracle
def test_predict_matches_the_oracle_on_the_full_net():
    import arch_and_hypers as ah
    from lib import layer_types
    layer_types.seed(0)
    net = ah.ac_chain(k_cpt=4e-9)((32, 32, 3), (10,)).configure(precision='fp32')
    rng = np.random.default_rng(1)
    for l in net.layers:
        if l.router is not None:
            w = l.router.comps[-1].params.w
            w.assign((0.5 * rng.standard_normal(w.shape)).astype(np.float32))
    x0 = rng.random((512, 32, 32, 3)).astype(np.float32)
    y = np.eye(10, dtype=np.float32)[rng.integers(0, 10, 512)]
    for t in range(12):                                  # move the running BN moments away from (0, 1)
        net.train.run({net.x0: x0[:128], net.y: y[:128], net.τ: 1.0, net.mode: 'tr', net.λ_lrn: 0.0})
    got = net.predict(x0, batch=256)
    with torch.no_grad():
        out = OracleNet(record_of(net), torch.float64).forward(x0, y, mode='ev', tau=0.5)
    paths = [p for p, l in node_paths(net) if not l.sinks]
    exit_ref = np.full(512, -1)
    for i, p in enumerate(paths):
        exit_ref[out.nodes[p].p_ev.numpy() == 1] = i
    assert (exit_ref >= 0).all()
    margin = np.full(512, np.inf)                        # smallest top-2 router margin along each example's path
    for p in out.order:
        nd = out.nodes[p]
        if nd.router is not None and len(nd.rec['sinks']) > 1:
            r = np.sort(nd.router.x.detach().numpy(), 1)
            m = r[:, -1] - r[:, -2]
            on = nd.p_ev.numpy() == 1
            margin[on] = np.minimum(margin[on], m[on])
    agree = got.exit == exit_ref
    print('predict vs oracle: exit agreement %.4f, smallest margin among disagreements %s'
          % (agree.mean(), margin[~agree].min(initial=np.inf)))
    assert agree.mean() >= 0.99
    assert agree[margin > 1e-4].all()
    for i, p in enumerate(paths):
        sel = agree & (exit_ref == i)
        if sel.any():
            ref = out.nodes[p].x.detach().numpy()[sel]
            np.testing.assert_allclose(got.prob[sel], ref, rtol=0, atol=1e-4)
    assert (got.cls[agree] == got.prob[agree].argmax(1)).all()


# ---------------------------------------------------------------- driver
def _run(script, args, cwd):
    r = subprocess.run([sys.executable, os.path.join(PKG, script)] + args, cwd=cwd, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout


def test_classify_net_driver(tmp_path):
    from lib.data import Dataset, synthetic_archive
    from lib.serdes import read_net
    _run('train-nets', ['cifar10-ac', '--synthetic', '--n-iter', '20', '--t-log', '20', '--compact-stats', '--nets', '0'],
         str(tmp_path))
    path = str(tmp_path / 'nets' / 'cifar10-ac' / '0000.npy')
    out = _run('classify-net', [path, '--synthetic', '--split', 'test', '--out', 'preds.npz'], str(tmp_path))
    d = np.load(tmp_path / 'preds.npz')
    assert d['cls'].dtype == np.int32 and d['cls'].shape == (512,)
    assert d['exit'].dtype == np.int32 and d['exit'].shape == (512,) and 0 <= d['exit'].min() and d['exit'].max() < 8
    assert d['ops'].dtype == np.float64 and d['ops'].shape == (512,) and (d['ops'] > 0).all()
    assert d['prob'].dtype == np.float32 and d['prob'].shape == (512, 10)
    assert 'k_cpt' not in d
    acc = float(re.search(r'^  accuracy\s+([0-9.]+)', out, re.M).group(1))
    net = read_net(path).configure(precision='bf16')
    ds = Dataset(archive=synthetic_archive(2048, 512, (32, 32, 3), 10))
    ev = net.compact_evaluator()
    ev.reset()
    ev.run_batch(ds.x0_ts, ds.y_ts)
    assert acc == pytest.approx(ev.result()[(net, 'acc')], abs=1e-12)
    with pytest.raises(AssertionError, match='k-cpt'):                   # refused for a fixed-k_cpt net
        _run('classify-net', [path, '--synthetic', '--k-cpt', '1e-8'], str(tmp_path))

    _run('train-adaptive-nets', ['hybrid-ac-dynkcpt', '--synthetic', '--n-iter', '20'], str(tmp_path))
    path = str(tmp_path / 'nets' / 'hybrid-ac-dynkcpt' / 'net.npy')
    out = _run('classify-net', [path, '--synthetic', '--k-cpt', '0', '1.6e-8', '--out', 'dyn.npz'], str(tmp_path))
    assert len(re.findall(r'^k_cpt ', out, re.M)) == len(re.findall(r'^  accuracy ', out, re.M)) == 2
    assert 'k_cpt 1.6e-08' in out
    d = np.load(tmp_path / 'dyn.npz')
    assert d['cls'].shape == (2, 512) and d['prob'].shape == (2, 512, 10)
    np.testing.assert_array_equal(d['k_cpt'], np.float32([0, 1.6e-8]))
