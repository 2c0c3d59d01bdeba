"""Routed inference and compacted statistics for Conv-block trees, MultiscaleLLN pyramids, GlobalMaxPool and
superclass classifiers, on the B200: the counted LLN and GlobalMaxPool kernels against the uncounted ones (sentinel
rows, count 0, graph replay), the target-aware leaf statistics and the strided leaf emit against NumPy and the dense
kernels, `net.predict` / `net.predictor` / the compacted statistics against the dense 'ev' pass bit for bit, the
Conv-block net against the fp64 oracle, and the drivers."""
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

from oracle.torch_ref import OracleNet  # noqa: E402
from test_predict_blocks_cpu import make  # noqa: E402
from test_predictor_gpu import _equal, _mixed_k  # noqa: E402
from util import Geo, batch, node_paths, randomize_routers, record_of, superclasses, to_planes  # noqa: E402

pytestmark = pytest.mark.gpu
F32, BF16 = 0, 1
X6 = ['cnv', 'cnvpyr', 'srlln', 'srsce', 'aclln', 'acsce', 'crsce']          # served in bf16x6 too
CASES = [(k, {}) for k in X6 + ['cnvactor']] + [('acsce', dict(dyn_k_cpt=True)), ('cnvactor', dict(dyn_k_cpt=True))]
ROUTED = [('aclln', {}), ('acsce', {}), ('crsce', {}), ('cnvactor', {}), ('acsce', dict(dyn_k_cpt=True))]


def L():
    from lib import _cabi
    return _cabi.lib()


def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def bits(t):
    t = t.detach().cpu()
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def cnt(m):
    return torch.tensor([m], dtype=torch.int32, device='cuda')


# ---------------------------------------------------------------- counted kernels against uncounted ones
def test_lln_counted_matches_lln():
    B, H0, step = 37, 16, 2
    rng = np.random.default_rng(1)
    x0 = dev(rng.random((B, H0, H0, 3)).astype(np.float32))
    H = H0 // step
    ref = torch.full((B, H, H, 3), -5.0, device='cuda')
    L().lln(vp(x0), B, H0, H0, 3, step, 2.0, 1e-3, vp(ref), None)
    for m in (0, 1, 20, B):
        got = torch.full_like(ref, -5.0)
        L().lln_counted(vp(x0), B, H0, H0, 3, step, 2.0, 1e-3, vp(got), vp(cnt(m)), None)
        torch.cuda.synchronize()
        assert torch.equal(bits(got[:m]), bits(ref[:m])) and (got[m:] == -5.0).all(), m
    got = torch.full_like(ref, -5.0)
    L().lln_counted(vp(x0), B, H0, H0, 3, step, 2.0, 1e-3, vp(got), None, None)             # count NULL: all B
    torch.cuda.synchronize()
    assert torch.equal(bits(got), bits(ref))
    # one captured launch reads the count on every replay
    c = cnt(B)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        L().lln_counted(vp(x0), B, H0, H0, 3, step, 2.0, 1e-3, vp(got), vp(c),
                        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    for m in (9, 30, 0):
        got.fill_(-5.0)
        c.fill_(m)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(bits(got[:m]), bits(ref[:m])) and (got[m:] == -5.0).all(), m


@pytest.mark.parametrize('dt', [F32, BF16])
def test_global_maxpool_fwd_counted_matches_the_uncounted_forward(dt):
    B, H, C = 45, 8, 32
    Balloc = 48
    geo = Geo(B, H, H)
    rng = np.random.default_rng(2)
    x = rng.integers(-3, 4, (B, H, H, C)).astype(np.float32)            # ties: the first maximum in both
    td = torch.float32 if dt == F32 else torch.bfloat16
    X = dev(to_planes(x, geo)).to(td)
    ref = torch.full((C // 8, Balloc, 8), -9.0, device='cuda').to(td)
    arg = torch.zeros((C // 8, Balloc, 8), dtype=torch.int32, device='cuda')
    L().global_maxpool_fwd(vp(X), C, B, H, H, geo.G, geo.P, vp(ref), vp(arg), Balloc, dt, None)
    for m in (0, 1, 30, B):
        got = torch.full_like(ref, -9.0)
        a2 = torch.full_like(arg, -1)
        L().global_maxpool_fwd_counted(vp(X), C, B, H, H, geo.G, geo.P, vp(got), vp(a2), Balloc, dt, vp(cnt(m)), None)
        got2 = torch.full_like(ref, -9.0)                # arg NULL: the same features, no argmax
        L().global_maxpool_fwd_counted(vp(X), C, B, H, H, geo.G, geo.P, vp(got2), None, Balloc, dt, vp(cnt(m)), None)
        torch.cuda.synchronize()
        assert torch.equal(bits(got[:, :m]), bits(ref[:, :m])) and (got[:, m:] == -9.0).all(), m
        assert torch.equal(bits(got2), bits(got)), m
        assert torch.equal(a2[:, :m], arg[:, :m]) and (a2[:, m:] == -1).all(), m
    got = torch.full_like(ref, -9.0)                     # count and arg NULL: all B images
    L().global_maxpool_fwd_counted(vp(X), C, B, H, H, geo.G, geo.P, vp(got), None, Balloc, dt, None, None)
    torch.cuda.synchronize()
    assert torch.equal(bits(got[:, :B]), bits(ref[:, :B])) and (got[:, B:] == -9.0).all()
    c = cnt(B)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        L().global_maxpool_fwd_counted(vp(X), C, B, H, H, geo.G, geo.P, vp(got), None, Balloc, dt, vp(c),
                                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    for m in (11, 44, 0):
        got.fill_(-9.0)
        c.fill_(m)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(bits(got[:, :m]), bits(ref[:, :m])) and (got[:, m:] == -9.0).all(), m


@pytest.mark.parametrize('n_out', [4, 10, 20])
def test_leaf_stats_targets_match_the_dense_loss_kernel(n_out):
    """cor is the dense d_cor of mpnn_softmax_ce_fwd on the targets; the bins follow the labels"""
    rng = np.random.default_rng(n_out)
    n_par, n_cls, B, n = 700, 10, 2000, 300
    ldz = 32
    Z = rng.standard_normal((n_par, ldz)).astype(np.float32)
    tie = rng.choice(n_par, 60, replace=False)
    Z[tie, 1] = Z[tie, 0] = Z[tie, :n_out].max(1) + 1.0               # tied maxima: the first index wins
    y = np.eye(n_cls, dtype=np.float32)[rng.integers(0, n_cls, B)]
    w = superclasses(n_cls, n_out) if n_out < n_cls else rng.standard_normal((n_cls, n_out)).astype(np.float32)
    t = (y @ w).astype(np.float32)
    pos = np.sort(rng.choice(n_par, n, replace=False)).astype(np.int32)
    orig = rng.choice(B, n, replace=False).astype(np.int32)
    out = torch.zeros(2 + 2 * n_cls, dtype=torch.float64, device='cuda')
    Zd, td, yd, pd, od = dev(Z), dev(t), dev(y), dev(pos), dev(orig)
    for rep in range(2):                                             # accumulates
        L().leaf_stats_targets(vp(Zd), ldz, n_out, vp(td), vp(yd), n_cls, vp(pd), vp(od), vp(cnt(n)), n, vp(out), None)
    # the dense loss kernel on the same rows and targets
    rows = Zd[pd.long()].contiguous()
    prob, ce, dc = (torch.empty((n, n_out), device='cuda'), torch.empty(n, device='cuda'),
                    torch.empty(n, device='cuda'))
    L().softmax_ce_fwd(vp(rows), ldz, vp(td[od.long()].contiguous()), n, n_out, 0.1, vp(prob), vp(ce), vp(dc), None)
    torch.cuda.synchronize()
    cor = dc.cpu().numpy() == 1.0
    assert cor.any() and (~cor).any()
    yo = y[orig]
    want = np.concatenate([[cor.sum(), (~cor).sum()], (cor[:, None] * yo).sum(0), ((~cor)[:, None] * yo).sum(0)])
    np.testing.assert_array_equal(out.cpu().numpy(), 2 * want)
    if n_out == n_cls:                   # mpnn_leaf_stats is the t = y case: the dense d_cor against the labels
        got = [torch.zeros_like(out) for _ in range(2)]
        L().leaf_stats(vp(Zd), ldz, n_cls, vp(yd), vp(pd), vp(od), vp(cnt(n)), n, vp(got[0]), None)
        L().leaf_stats_targets(vp(Zd), ldz, n_cls, vp(yd), vp(yd), n_cls, vp(pd), vp(od), vp(cnt(n)), n, vp(got[1]),
                               None)
        L().softmax_ce_fwd(vp(rows), ldz, vp(yd[od.long()].contiguous()), n, n_cls, 0.1, vp(prob), vp(ce), vp(dc), None)
        torch.cuda.synchronize()
        cor = dc.cpu().numpy() == 1.0
        want = np.concatenate([[cor.sum(), (~cor).sum()], (cor[:, None] * yo).sum(0), ((~cor)[:, None] * yo).sum(0)])
        for g in got:
            np.testing.assert_array_equal(g.cpu().numpy(), want)


@pytest.mark.parametrize('n_out', [4, 10, 20])
def test_leaf_emit_strided_zero_fills_the_row(n_out):
    rng = np.random.default_rng(n_out + 1)
    n_par, n_rows, n, live, ldp = 300, 500, 200, 150, 24
    ldz = 32
    Z = dev(rng.standard_normal((n_par, ldz)).astype(np.float32))
    pos, orig = dev(rng.permutation(n_par)[:n].astype(np.int32)), dev(rng.permutation(n_rows)[:n].astype(np.int32))
    outs = lambda w: [torch.full((n_rows, w), -7.0, device='cuda'), torch.full((n_rows,), -7, dtype=torch.int32,
                      device='cuda'), torch.full((n_rows,), -7, dtype=torch.int32, device='cuda'),
                      torch.full((n_rows,), -7.0, dtype=torch.float64, device='cuda')]
    a, b = outs(ldp), outs(n_out)
    L().leaf_emit_strided(vp(Z), ldz, n_out, vp(pos), vp(orig), vp(cnt(live)), n, 2, 3.5e5, vp(a[0]), ldp,
                          *(vp(t) for t in a[1:]), None)
    L().leaf_emit(vp(Z), ldz, n_out, vp(pos), vp(orig), vp(cnt(live)), n, 2, 3.5e5, *(vp(t) for t in b), None)
    torch.cuda.synchronize()
    o = orig[:live].long().cpu()
    rest = np.setdiff1d(np.arange(n_rows), o.numpy())
    assert torch.equal(bits(a[0][o, :n_out]), bits(b[0][o])) and (a[0][o, n_out:] == 0).all()
    assert (a[0][rest] == -7).all()
    for x, y in zip(a[1:], b[1:]):
        assert torch.equal(x, y)


# ---------------------------------------------------------------- the walk against the dense 'ev' pass
# router weights per net that send the examples down several paths: MultiscaleLLN rescales the images, and at the
# default scale every randomized router of 'aclln' picks sink 0 (checked against the fp64 oracle after the same two
# training steps: 60 / 98 / 42 of the 200 test examples at its three leaves)
ROUTERS = {'aclln': dict(seed=5, scale=8.0)}


def _trained(kind, hy, prec, seed=2):
    net = make(kind, seed=seed, **hy)
    if net.dynamic:
        randomize_routers(net, **ROUTERS.get(kind, {}))
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


def _feed(net, hy, x0, y, kc):
    feed = {net.x0: x0, net.y: y}
    if net.dynamic:
        feed[net.τ] = 0.5
    if kc is not None:
        feed[net.k_cpt] = kc
    return feed


def _precisions(kind):
    return ['fp32', 'bf16'] + (['bf16x6'] if kind in X6 else [])


@pytest.mark.parametrize('kind,hy,prec', [(k, h, p) for k, h in CASES for p in _precisions(k)])
def test_predict_equals_the_dense_path(kind, hy, prec):
    net = _trained(kind, hy, prec)
    eng = net._get_engine()
    n = 200
    x0, y = batch(n, seed=9)
    kc = _mixed_k(n) if hy.get('dyn_k_cpt') else None
    moc = net.eval_stats(_feed(net, hy, x0, y, kc))[(net, 'moc')]
    plan = eng._plan(n, False, False)                    # the buffers of that dense forward
    p_ev = plan.p_ev.cpu().numpy() if net.dynamic else np.ones((len(eng.nodes), n), np.float32)
    got = net.predict(x0, k_cpt=kc, batch=128)           # two chunks: 128 + 72
    assert got.prob.dtype == np.float32 and got.prob.shape == (n, 10)
    seen = np.zeros(n, bool)
    for i, leaf in enumerate(eng.leaves):
        here = p_ev[leaf.idx] == 1
        assert not (seen & here).any()
        seen |= here
        np.testing.assert_array_equal(got.exit == i, here)
        dense = plan.reg[leaf.idx].prob.cpu().numpy()[:n]
        w = dense.shape[1]                               # the leaf's outputs: its classes or its superclasses
        assert w == (4 if kind.endswith('sce') else 10)
        assert got.prob[here][:, :w].tobytes() == dense[here].tobytes()          # max |Δ| = 0
        assert (got.prob[here][:, w:] == 0).all()
        np.testing.assert_array_equal(got.cls[here], dense[here].argmax(1))
    assert seen.all()
    np.testing.assert_array_equal(got.ops, moc)
    if len(eng.leaves) > 1:
        assert len(set(got.exit.tolist())) > 1                  # the routers spread the examples


@pytest.mark.parametrize('kind,hy,prec', [(k, h, p) for k, h in CASES for p in _precisions(k)])
def test_predictor_equals_predict(kind, hy, prec):
    net = _trained(kind, hy, prec)
    n = 200
    x0, _ = batch(n, seed=10)
    kc = _mixed_k(n) if hy.get('dyn_k_cpt') else None
    want = net.predict(x0, k_cpt=kc, batch=256)
    p = net.predictor(256)
    _equal(p(x0, k_cpt=kc), want)
    _equal(p(x0[:77], k_cpt=kc[:77] if kc is not None else None), net.predict(x0[:77], k_cpt=kc[:77] if kc is not None
                                                                              else None, batch=256))


@pytest.mark.parametrize('kind,hy', [('acsce', dict(dyn_k_cpt=True)), ('cnvactor', dict(dyn_k_cpt=True)),
                                     ('aclln', {})])
def test_no_host_synchronisation_with_device_inputs(kind, hy):
    net = _trained(kind, hy, 'bf16')
    x0, _ = batch(100, seed=17)
    xd = torch.from_numpy(x0).cuda()
    kd = torch.from_numpy(_mixed_k(100, seed=9)).cuda() if hy.get('dyn_k_cpt') else None
    p = net.predictor(128)
    p(xd, k_cpt=kd)                                      # first call: capture (synchronises once)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        out = p(xd[:50], k_cpt=kd[:50] if kd is not None else None)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    _equal(out, net.predict(x0[:50], k_cpt=kd[:50].cpu().numpy() if kd is not None else None, batch=128))


EXACT = ('p_cor', 'p_inc', 'p_cor_by_cls', 'p_inc_by_cls')


@pytest.mark.parametrize('kind,hy,prec', [(k, h, p) for k, h in ROUTED for p in _precisions(k)])
def test_compact_statistics_equal_the_dense_path(kind, hy, prec):
    net = _trained(kind, hy, prec)
    n = 200
    x0, y = batch(n, seed=9)
    kc = np.full(n, 1.6e-8, np.float32) if hy.get('dyn_k_cpt') else None
    dense = {k: np.asarray(v, np.float64).mean(0) for k, v in net.eval_stats(_feed(net, hy, x0, y, kc)).items()}
    ev = net.compact_evaluator(128)                      # two batches: 128 + 72
    ev.reset()
    for i in range(0, n, 128):
        ev.run_batch(x0[i:i + 128], y[i:i + 128], k_cpt=kc[i:i + 128] if kc is not None else None)
    got = ev.result()
    assert got[(net, 'acc')] == pytest.approx(dense[(net, 'acc')], abs=1e-12)
    assert got[(net, 'moc')] == pytest.approx(dense[(net, 'moc')], rel=1e-12)
    for leaf in net.leaves:
        for name in EXACT:
            np.testing.assert_array_equal(np.asarray(got[(leaf, name)]), dense[(leaf, name)], err_msg=name)
        assert len(got[(leaf, 'p_cor_by_cls')]) == 10            # bins over the classes, also at superclass leaves
    assert sum(got[(leaf, 'p_cor')] + got[(leaf, 'p_inc')] for leaf in net.leaves) == pytest.approx(1.0, abs=1e-12)


# ---------------------------------------------------------------- the Conv-block net against the oracle
@pytest.mark.parametrize('kind', ['cnvactor', 'aclln', 'acsce'])
def test_fp32_predict_matches_the_oracle(kind):
    net = _trained(kind, {}, 'fp32')
    n = 256
    x0, y = batch(n, seed=21)
    got = net.predict(x0, batch=128)
    with torch.no_grad():
        out = OracleNet(record_of(net), torch.float64).forward(x0, y, mode='ev', tau=0.5)
    paths = [p for p, l in node_paths(net) if not l.sinks]
    exit_ref = np.full(n, -1)
    for i, p in enumerate(paths):
        exit_ref[out.nodes[p].p_ev.numpy() == 1] = i
    assert (exit_ref >= 0).all()
    agree = got.exit == exit_ref
    assert agree.mean() >= 0.99 if len(paths) > 1 else agree.all()
    worst = 0.0
    for i, p in enumerate(paths):
        sel = agree & (exit_ref == i)
        if sel.any():
            ref = out.nodes[p].x.detach().numpy()[sel]
            worst = max(worst, float(np.abs(got.prob[sel][:, :ref.shape[1]] - ref).max()))
    print('%s fp32 predict vs oracle: exit agreement %.4f, max |prob error| %g' % (kind, agree.mean(), worst))
    assert worst <= 1e-3


# ---------------------------------------------------------------- drivers
def _run(script, args, cwd):
    r = subprocess.run([sys.executable, os.path.join(PKG, script)] + args, cwd=cwd, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout


@pytest.mark.parametrize('kind,hy', [('cnvactor', {}), ('aclln', {}), ('acsce', {}), ('srsce', {}), ('cnvpyr', {})])
def test_classify_net(kind, hy, tmp_path):
    import re
    from lib.data import Dataset, synthetic_archive
    from lib.serdes import write_net
    net = _trained(kind, hy, 'bf16')
    path = str(tmp_path / 'net.npy')
    write_net(path, net)
    args = [path, '--synthetic', '--batch', '200']
    a = _run('classify-net', args + ['--out', 'a.npz'], str(tmp_path))
    b = _run('classify-net', args + ['--graph', '--out', 'b.npz'], str(tmp_path))
    assert a == b and '  accuracy ' in a
    da, db = np.load(tmp_path / 'a.npz'), np.load(tmp_path / 'b.npz')
    for f in da.files:
        assert da[f].dtype == db[f].dtype and da[f].tobytes() == db[f].tobytes(), f
    assert da['prob'].shape == (512, 10)
    # the printed accuracy scores a superclass exit against argmax(y @ w_cls): the compacted statistics' acc
    acc = float(re.search(r'^  accuracy\s+([0-9.]+)', a, re.M).group(1))
    ds = Dataset(archive=synthetic_archive(2048, 512, (16, 16, 3), 10))
    eng = net._get_engine()
    label = ds.y_ts.argmax(1)
    cor = np.zeros(512, bool)
    for i, nd in enumerate(eng.leaves):
        t = (ds.y_ts @ nd.w_cls).argmax(1) if nd.loss == 'sce' else label
        here = da['exit'] == i
        cor[here] = da['cls'][here] == t[here]
    assert acc == pytest.approx(cor.mean(), abs=1e-12)
    if net.dynamic:
        ev = net.compact_evaluator()
        ev.reset()
        ev.run_batch(ds.x0_ts, ds.y_ts)
        assert acc == pytest.approx(ev.result()[(net, 'acc')], abs=1e-12)


def test_compact_stats_net_desc_on_a_routed_superclass_net():
    """the `--compact-stats` statistics pass of train-nets (net_desc(compact=True)) on a routed superclass net"""
    from lib.data import Dataset, synthetic_archive
    from lib.desc import net_desc, render_net_desc, state_tensors
    net = _trained('acsce', {}, 'bf16')
    ds = Dataset(archive=synthetic_archive(512, 256, (16, 16, 3), 10))
    hy = {net.τ: 0.5}
    compact = net_desc(net, ds, hy, state_tensors(net), compact=True)
    dense = net_desc(net, ds, hy, state_tensors(net))
    for split in ('stats_tr', 'stats_ts'):
        assert compact[split]['acc'] == pytest.approx(dense[split]['acc'], abs=1e-12)
        assert compact[split]['moc'] == pytest.approx(dense[split]['moc'], rel=1e-12)
    assert 'acc' in render_net_desc(compact)
