"""Routed inference and compacted statistics in bf16x6 precision (lib/compact_eval.py's split branch): the counted
three-way split against the whole-tensor one, bit for bit, with the rows past the live images untouched and one
captured graph serving every count; `net.predict`, `net.predictor` and the compacted statistics against the dense
bf16x6 'ev' pass (the same kernels on the same rows, so the same bits); the full architecture against the fp64
oracle with the fp32 bounds; and the drivers."""
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
from test_compact_eval_gpu import test_compact_evaluator_equals_the_dense_path as _stats_equal_dense  # noqa: E402
from test_predict_gpu import test_predict_equals_the_dense_path as _predict_equals_dense  # noqa: E402
from test_predictor_gpu import test_predictor_equals_predict as _predictor_equals_predict  # noqa: E402
from test_predictor_gpu import _equal, _mixed_k, _trained  # noqa: E402
from util import Geo, batch, node_paths, record_of, to_planes  # noqa: E402

pytestmark = pytest.mark.gpu
CASES = [('ac', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('sr', {}),
         ('ac', dict(dyn_k_cpt=True))]


def L():
    from lib import _cabi
    return _cabi.lib()


def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def bits(t):
    return t.detach().cpu().view(torch.int16)


# ---------------------------------------------------------------- the counted split
def test_split_planes3_counted_matches_the_whole_tensor_split():
    B, H, C = 70, 8, 32
    geo = Geo(B, H, H)
    rng = np.random.default_rng(1)
    x = rng.standard_normal((B, H, H, C)).astype(np.float32) * 10.0 ** rng.integers(-6, 4, (B, H, H, C))
    src = torch.from_numpy(to_planes(x, geo)).cuda()
    ref = torch.full((3 * C // 8, geo.P, 8), -9.0, dtype=torch.bfloat16, device='cuda')
    L().split_planes3(vp(src), C, geo.P, vp(ref), None)
    cnt = torch.zeros(1, dtype=torch.int32, device='cuda')
    for m in (0, 1, B // 2, B):
        got = torch.full_like(ref, -9.0)
        cnt.fill_(m)
        L().split_planes3_counted(vp(src), C, B, H, H, geo.G, geo.P, vp(got), vp(cnt), None)
        torch.cuda.synchronize()
        end = geo.G + m * geo.S if m else 0
        assert torch.equal(bits(got[:, :end]), bits(ref[:, :end])), m
        assert (got[:, end:] == -9.0).all(), m
    got = torch.full_like(ref, -9.0)                     # count NULL: all B images
    L().split_planes3_counted(vp(src), C, B, H, H, geo.G, geo.P, vp(got), None, None)
    torch.cuda.synchronize()
    end = geo.G + B * geo.S
    assert torch.equal(bits(got[:, :end]), bits(ref[:, :end])) and (got[:, end:] == -9.0).all()


def test_split_planes3_counted_in_a_graph_reads_the_count_per_replay():
    B, H, C = 40, 16, 16
    geo = Geo(B, H, H)
    rng = np.random.default_rng(2)
    src = torch.from_numpy(to_planes(rng.standard_normal((B, H, H, C)).astype(np.float32), geo)).cuda()
    ref = torch.zeros((3 * C // 8, geo.P, 8), dtype=torch.bfloat16, device='cuda')
    L().split_planes3(vp(src), C, geo.P, vp(ref), None)
    dst = torch.full_like(ref, -9.0)
    cnt = torch.full((1,), B, dtype=torch.int32, device='cuda')
    L().split_planes3_counted(vp(src), C, B, H, H, geo.G, geo.P, vp(dst), vp(cnt), None)     # module load outside capture
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        L().split_planes3_counted(vp(src), C, B, H, H, geo.G, geo.P, vp(dst), vp(cnt),
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    for m in (7, 23, 0):
        dst.fill_(-9.0)
        cnt.fill_(m)
        g.replay()
        torch.cuda.synchronize()
        end = geo.G + m * geo.S if m else 0
        assert torch.equal(bits(dst[:, :end]), bits(ref[:, :end])), m
        assert (dst[:, end:] == -9.0).all(), m


# ---------------------------------------------------------------- the walk against the dense bf16x6 pass
@pytest.mark.parametrize('kind,hy', CASES)
def test_predict_equals_the_dense_path_in_bf16x6(kind, hy):
    _predict_equals_dense(kind, hy, 'bf16x6')


@pytest.mark.parametrize('kind,hy', CASES)
def test_predictor_equals_predict_in_bf16x6(kind, hy):
    _predictor_equals_predict(kind, hy, 'bf16x6')


def test_one_bf16x6_graph_serves_every_n_and_mixed_k_cpt():
    net = _trained('ac', dict(dyn_k_cpt=True), 'bf16x6')
    B = 160
    p = net.predictor(B)
    x0, _ = batch(B, seed=14)
    graph = None
    for n, seed in ((150, 8), (61, 9)):
        kc = _mixed_k(n, seed=seed)
        want = net.predict(x0[:n], k_cpt=kc, batch=B)
        _equal(p(x0[:n], k_cpt=kc), want)
        assert len(set(want.ops.tolist())) > 1
        graph = graph or p.graph
        assert p.graph is graph                          # captured once, replayed


@pytest.mark.parametrize('kind,hy', [c for c in CASES if c[0] != 'sr'])
def test_compact_statistics_equal_the_dense_path_in_bf16x6(kind, hy):
    _stats_equal_dense(kind, hy, 'bf16x6')


# ---------------------------------------------------------------- full architecture against the oracle
def test_bf16x6_predict_matches_the_oracle_on_the_full_net():
    """test_predict_gpu.py's fp32 check in bf16x6: the tensor-core mode is held to the same bounds"""
    import arch_and_hypers as ah
    from lib import layer_types
    layer_types.seed(0)
    net = ah.ac_chain(k_cpt=4e-9)((32, 32, 3), (10,)).configure(precision='bf16x6')
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
    worst = 0.0
    for i, p in enumerate(paths):
        sel = agree & (exit_ref == i)
        if sel.any():
            ref = out.nodes[p].x.detach().numpy()[sel]
            worst = max(worst, float(np.abs(got.prob[sel] - ref).max()))
    print('bf16x6 predict vs oracle: exit agreement %.4f, smallest margin among disagreements %s, max |prob error| %g'
          % (agree.mean(), margin[~agree].min(initial=np.inf), worst))
    assert agree.mean() >= 0.99
    assert agree[margin > 1e-4].all()
    assert worst <= 1e-4
    assert (got.cls[agree] == got.prob[agree].argmax(1)).all()
    assert len(set(got.exit.tolist())) > 1


# ---------------------------------------------------------------- drivers
def _run(script, args, cwd):
    r = subprocess.run([sys.executable, os.path.join(PKG, script)] + args, cwd=cwd, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout


def test_drivers_in_bf16x6(tmp_path):
    _run('train-nets', ['cifar10-ac', '--synthetic', '--n-iter', '4', '--t-log', '4', '--nets', '0',
                        '--precision', 'bf16x6', '--compact-stats'], str(tmp_path))
    d = tmp_path / 'nets' / 'cifar10-ac'
    stats = np.load(d / '0000-stats.npy', allow_pickle=True)[()]
    assert stats['type'] == 'ActorNet'
    for split in ('stats_tr', 'stats_ts'):
        assert 0.0 <= stats[split]['acc'] <= 1.0 and stats[split]['moc'] > 0
    path = str(d / '0000.npy')
    args = [path, '--synthetic', '--precision', 'bf16x6', '--batch', '200']
    a = _run('classify-net', args + ['--out', 'a.npz'], str(tmp_path))
    b = _run('classify-net', args + ['--graph', '--out', 'b.npz'], str(tmp_path))
    assert a == b and '  accuracy ' in a
    da, db = np.load(tmp_path / 'a.npz'), np.load(tmp_path / 'b.npz')
    assert da['cls'].shape == (512,) and da['prob'].shape == (512, 10) and (da['ops'] > 0).all()
    for f in da.files:
        assert da[f].dtype == db[f].dtype and da[f].tobytes() == db[f].tobytes(), f
