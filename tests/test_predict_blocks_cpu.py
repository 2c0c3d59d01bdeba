"""Routed inference and compacted statistics for Conv-block trees, MultiscaleLLN pyramids, GlobalMaxPool and
superclass classifiers, on the host: the C ABI of the new counted / strided / target-aware entry points and their
argument checks, the compositions the walk now serves and the ones it still refuses, and the walk's launches against
the dense eval plan's, operand for operand -- on dry-run engines, which plan without a device."""
import ctypes
import os
import sys
from types import SimpleNamespace as Ns

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

from lib import _cabi  # noqa: E402
from lib.compact_eval import _LeafEmit, _LeafStats  # noqa: E402
from lib.layer_types import (ActivityError, BatchNorm, Chain, Conv, CrossEntropyError, Dropout,  # noqa: E402
                             GlobalMaxPool, LinTrans, Rect, Softmax)
from lib.net_types import ActorNet  # noqa: E402
from test_predict_cpu import _dropout_net, _Recorder  # noqa: E402
from util import K_L2, tiny_net  # noqa: E402

F32, BF16 = 0, 1


def _dry(net, precision='fp32'):
    return net.configure(precision=precision, dry_run=True, impl=0 if precision == 'fp32' else 1)


def conv_actor(n_cls=10, seed=0, **hypers):
    """An ActorNet of Conv blocks: a Conv-BN-ReLU root on the image behind an identity Dropout, a block with an
    ActivityError cost, and a GlobalMaxPool classifier.  It has one path: a router's leading Select picks a scale of a
    multiscale tensor, so in this layer library only MultiscaleConvMax nodes can be switches, and a Conv block cannot
    sit below one (it takes a single tensor)."""
    from lib import layer_types as lt
    lt.seed(seed)
    blk = lambda n, tail, *sinks: Chain(name='ConvBlock', sinks=sinks, comps=[
        Conv(n_chan=n, supp=3, k_l2=K_L2, σ_w=1), BatchNorm(), Rect()] + list(tail))
    gmp = Chain(name='LogReg', comps=[GlobalMaxPool(), LinTrans(n_chan=n_cls, k_l2=K_L2, σ_w=1), Softmax(),
                                      CrossEntropyError()])
    root = blk(16, [Dropout()], blk(32, [ActivityError(α=1e-3)], gmp))
    if not hypers.get('dyn_k_cpt'):
        hypers.setdefault('k_cpt', 4e-9)
    return ActorNet(x0_shape=(16, 16, 3), y_shape=(n_cls,), root=root, **hypers)


def make(kind, **hy):
    if kind == 'cnvactor':
        return conv_actor(**hy)
    if kind[:2] in ('ac', 'cr') and not hy.get('dyn_k_cpt'):
        hy.setdefault('k_cpt', 4e-9)
    return tiny_net(kind, **hy)


SERVED = ['cnv', 'cnvpyr', 'srlln', 'srsce', 'aclln', 'acsce', 'crsce', 'cnvactor']


# ---------------------------------------------------------------- the C ABI
def test_new_entry_points_are_declared_and_exported():
    protos = _cabi.parse_header()
    want = {
        'mpnn_lln_counted': ['x0', 'B', 'H0', 'W0', 'C0', 'step', 'sigma', 'eps', 'out', 'count', 'stream'],
        'mpnn_global_maxpool_fwd_counted': ['x', 'C', 'B', 'H', 'W', 'G', 'P', 'feat', 'arg', 'Balloc', 'dtype',
                                            'count', 'stream'],
        'mpnn_leaf_stats_targets': ['Z', 'ldz', 'n_out', 't', 'y', 'n_cls', 'pos', 'orig', 'count', 'n', 'out',
                                    'stream'],
        'mpnn_leaf_emit_strided': ['Z', 'ldz', 'n_out', 'pos', 'orig', 'count', 'n', 'leaf', 'path_ops', 'prob', 'ldp',
                                   'cls', 'exit_id', 'ops', 'stream'],
    }
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for name, names in want.items():
        assert protos[name][2] == names, name
        assert hasattr(lib, name), name
    assert protos['mpnn_lln_counted'][1][6] is ctypes.c_float and protos['mpnn_leaf_emit_strided'][1][8] is ctypes.c_double
    # the entry points they generalise keep their prototypes
    assert len(protos['mpnn_leaf_emit'][1]) == 14 and len(protos['mpnn_leaf_stats'][1]) == 10
    assert len(protos['mpnn_lln'][1]) == 10 and len(protos['mpnn_global_maxpool_fwd'][1]) == 12


def test_argument_checks_raise_before_any_launch():
    L = _cabi.lib()
    p = ctypes.c_void_p(16)                       # never dereferenced: every call below fails its checks first
    before = L.launches
    with pytest.raises(_cabi.MpnnError, match='3 channels'):
        L.lln_counted(p, 4, 8, 8, 4, 1, 2.0, 1e-3, p, p, None)
    with pytest.raises(_cabi.MpnnError, match='step'):
        L.lln_counted(p, 4, 8, 8, 3, 3, 2.0, 1e-3, p, p, None)
    with pytest.raises(_cabi.MpnnError, match='B=-1'):
        L.lln_counted(p, -1, 8, 8, 3, 1, 2.0, 1e-3, p, p, None)
    with pytest.raises(_cabi.MpnnError, match='global_maxpool_fwd_counted'):
        L.global_maxpool_fwd_counted(p, 12, 4, 8, 8, 64, 4096, p, None, 8, F32, p, None)       # C % 8
    with pytest.raises(_cabi.MpnnError, match='global_maxpool_fwd_counted'):
        L.global_maxpool_fwd_counted(p, 16, 9, 8, 8, 64, 4096, p, None, 8, F32, p, None)       # Balloc < B
    with pytest.raises(_cabi.MpnnError, match='global_maxpool_fwd_counted'):
        L.global_maxpool_fwd_counted(None, 16, 4, 8, 8, 64, 4096, p, None, 8, F32, p, None)
    with pytest.raises(_cabi.MpnnError, match='leaf_stats: n_out=33'):
        L.leaf_stats_targets(p, 40, 33, p, p, 10, None, None, p, 4, p, None)
    with pytest.raises(_cabi.MpnnError, match='leaf_stats: n_out=4 ldz=3'):
        L.leaf_stats_targets(p, 3, 4, p, p, 10, None, None, p, 4, p, None)
    with pytest.raises(_cabi.MpnnError, match='leaf_stats'):
        L.leaf_stats_targets(p, 16, 4, None, p, 10, None, None, p, 4, p, None)                 # no targets
    with pytest.raises(_cabi.MpnnError, match='leaf_emit: n=4 n_out=4 ldz=16 ldp=3'):
        L.leaf_emit_strided(p, 16, 4, None, None, p, 4, 0, 1.0, p, 3, p, p, p, None)
    with pytest.raises(_cabi.MpnnError, match='leaf_emit: NULL operand'):
        L.leaf_emit_strided(p, 16, 4, None, None, p, 4, 0, 1.0, None, 10, p, p, p, None)
    L.leaf_emit_strided(p, 16, 4, None, None, p, 0, 0, 1.0, None, 10, None, None, None, None)   # n = 0: no-op
    L.lln_counted(p, 0, 8, 8, 3, 1, 2.0, 1e-3, p, p, None)                                        # capacity 0: no-op
    L.global_maxpool_fwd_counted(p, 16, 0, 8, 8, 64, 4096, p, None, 8, F32, p, None)
    assert L.launches == before + 3                  # the three no-ops return success without a kernel


# ---------------------------------------------------------------- what the walk serves and refuses
@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'bf16x6'])
@pytest.mark.parametrize('kind', SERVED)
def test_served_compositions_plan_a_walk(kind, precision):
    if precision == 'bf16x6' and kind == 'cnvactor':
        pytest.skip('the engine trains ActivityError / GlobalMaxPool blocks in fp32 and bf16 only')
    net = _dry(make(kind), precision)
    ev = net.compact_evaluator(16)
    assert net.compact_evaluator(16) is ev
    p = net.predictor(16)
    n_sup = 4 if kind.endswith('sce') else None
    assert ev.n_prob == 10 and tuple(p.prob.shape) == (16, 10)            # max(n_cls, widest leaf)
    assert len(ev.sce) == (len(list(net.leaves)) if n_sup else 0)
    out = net.predict(np.zeros((0, 16, 16, 3), np.float32), batch=16)     # n = 0: the shapes, nothing launched
    assert out.prob.shape == (0, 10) and out.cls.shape == out.exit.shape == out.ops.shape == (0,)
    e = p(np.zeros((0, 16, 16, 3), np.float32))
    assert tuple(e.prob.shape) == (0, 10) and p.graph is None


def test_bf16x6_refuses_the_conv_actor_in_the_engine():
    with pytest.raises(NotImplementedError, match='ActivityError'):
        _dry(conv_actor(), 'bf16x6')._get_engine()


@pytest.mark.parametrize('make_net,precision,reason', [
    (lambda: tiny_net('cnvmp'), 'fp32', 'MaxPool'),
    (lambda: tiny_net('cnvact'), 'fp32', 'MaxPool'),
    (lambda: tiny_net('cnvgmp'), 'bf16', 'MaxPool'),
    (lambda: tiny_net('cnvdrop'), 'fp32', 'MaxPool'),
    (_dropout_net, 'bf16', 'Dropout'),
    (lambda: tiny_net('acsq', k_cpt=4e-9), 'fp32', 'CrossEntropyError'),
    (lambda: tiny_net('srsq'), 'bf16', 'CrossEntropyError'),
    (lambda: tiny_net('acsce', k_cpt=4e-9), 'bf16x3', 'bf16x3'),
    (lambda: tiny_net('cnv'), 'bf16x3', 'bf16x3'),
])
def test_still_refused(make_net, precision, reason):
    net = _dry(make_net(), precision)
    with pytest.raises(NotImplementedError, match=reason):
        net.predict(np.zeros((2, 16, 16, 3), np.float32), batch=16)
    with pytest.raises(NotImplementedError, match=reason):
        net.predictor(16)
    with pytest.raises(NotImplementedError, match=reason):
        net.compact_evaluator(16)


# ---------------------------------------------------------------- the walk against the dense eval plan
def _dense_calls(plan, rec):
    """the dense eval plan's forward launches (pack ops excluded), recorded"""
    for op in plan.fwd_ops:
        op()
    return rec.calls


def _walk_calls(ev, rec, leaf, n, monkeypatch):
    monkeypatch.setattr(torch.cuda, 'current_stream', lambda *a: Ns(cuda_stream=0))

    def every_sink(nd, sw, stream):                      # each switch sends its whole batch down every sink
        for s in range(len(nd.kids)):
            yield s, (n, None), stream
    rec.calls = []
    ev._walk((n, None), leaf, every_sink)
    return rec.calls


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'bf16x6'])
@pytest.mark.parametrize('kind,hy', [(k, {}) for k in SERVED] + [('cnvactor', dict(dyn_k_cpt=True)),
                                                                  ('acsce', dict(dyn_k_cpt=True))])
def test_walk_launches_the_dense_eval_plans_kernels(kind, hy, precision, monkeypatch):
    if precision == 'bf16x6' and kind == 'cnvactor':
        pytest.skip('the engine trains ActivityError / GlobalMaxPool blocks in fp32 and bf16 only')
    net = _dry(make(kind, **hy), precision)
    eng = net._get_engine()
    x6 = precision == 'bf16x6'
    dt = BF16 if precision == 'bf16' else F32
    rec = _Recorder()
    eng.L = rec
    n = 24
    ev = net.compact_evaluator(32)
    plan = ev.plan
    dense = _dense_calls(plan, rec)
    by = lambda calls, name: [a for c, a in calls if c == name]
    walk = _walk_calls(ev, rec, _LeafStats(ev), n, monkeypatch)
    # gathers below a switch move the parent's tensors into the compact inputs: the convs read those copies
    to_src = {}
    for i, bufs in ev.cin.items():
        for slot, t in zip(plan.node[i].pin, bufs):
            to_src[t.data_ptr()] = (slot.split if x6 else slot.t).data_ptr()
    assert len(by(walk, 'gather_images')) == sum(len(b) for b in ev.cin.values())
    src = lambda p: to_src.get(p, p)

    # input: LLN / pack / split, every operand but the batch (the walk's n and its count)
    assert [a[:1] + a[2:9] for a in by(walk, 'lln_counted')] == [a[:1] + a[2:9] for a in by(dense, 'lln')]
    assert bool(by(walk, 'lln_counted')) == kind.endswith('lln')
    assert all(a[1] == n and a[9] is None for a in by(walk, 'lln_counted'))
    pk_w, pk_d = by(walk, 'pack_input_counted'), by(dense, 'pack_input')
    assert pk_w and [a[:1] + a[2:11] for a in pk_w] == [a[:1] + a[2:11] for a in pk_d]
    assert all(a[1] == n and a[11] is None for a in pk_w)
    sp_w = by(walk, 'split_planes3_counted')
    assert sorted((a[0], a[1], a[7]) for a in sp_w) == sorted((a[0], a[1], a[3]) for a in by(dense, 'split_planes3'))
    assert bool(sp_w) == x6 and all(a[2] == n and a[8] is None for a in sp_w)

    # convs: the dense plan's passes on the (gathered) inputs
    if x6:
        # conv_acc_bn_stats(A0, K0, A1, K1, Wp, bias, out, N, acc, B, H, W, G, P, bn, dtype, out_dtype, impl, stream)
        cd = [a[:9] + a[10:14] + a[15:18] for a in by(dense, 'conv_acc_bn_stats')]
    else:
        # stencil_gemm(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1, N1, acc1, B, H, W, G, P, stats,
        #              stats_cap, n_parts, dtype, out_dtype, impl, stream)
        cd = [a[:5] + a[6:10] + a[14:18] + a[21:24] for a in by(dense, 'stencil_gemm') if a[5] == 9]
    cw = [(src(a[0]),) + a[1:2] + (src(a[2]),) + a[3:5] + a[6:10] + a[14:18] + a[21:24]
          for a in by(walk, 'stencil_gemm_counted') if a[5] == 9]
    assert all(a[13] == n for a in by(walk, 'stencil_gemm_counted'))
    assert cd and sorted(cw, key=repr) == sorted(cd, key=repr)

    # BN / ReLU / pool: bn_relu_pool_fwd(lin, C, B, H, W, G, P, ss, act, pooled, Pp, feat, Balloc, dtype, stream)
    bw, bd = by(walk, 'bn_relu_pool_fwd_counted'), by(dense, 'bn_relu_pool_fwd')
    assert bd and sorted(a[:2] + a[3:14] for a in bw) == sorted(a[:2] + a[3:14] for a in bd)
    assert all(a[2] == n and a[13] == dt and a[14] is None for a in bw)
    # GlobalMaxPool: every operand of the dense launch but the argmax the 'ev' pass does not need
    gw, gd = by(walk, 'global_maxpool_fwd_counted'), by(dense, 'global_maxpool_fwd')
    assert [a[:2] + a[3:8] + a[9:11] for a in gw] == [a[:2] + a[3:8] + a[9:11] for a in gd]
    assert bool(gw) == (kind == 'cnvactor') and all(a[2] == n and a[8] is None for a in gw)
    # nothing the 'ev' pass does not need: no ActivityError cost, no Dropout, no BN statistics
    for name in ('activity_fwd', 'dropout', 'conv_bn_stats', 'bn_fwd_small', 'maxpool2_fwd'):
        assert not by(walk, name), name
    assert bool(by(dense, 'activity_fwd')) == (kind == 'cnvactor')


@pytest.mark.parametrize('kind', ['acsce', 'srsce', 'crsce'])
def test_superclass_leaves_score_their_targets_and_bin_the_labels(kind, monkeypatch):
    net = _dry(make(kind), 'bf16')
    eng = net._get_engine()
    rec = _Recorder()
    eng.L = rec
    ev = net.compact_evaluator(32)
    plan = ev.plan
    n = 20
    walk = _walk_calls(ev, rec, _LeafStats(ev), n, monkeypatch)
    st = [a for c, a in walk if c == 'leaf_stats_targets']
    assert len(st) == len(eng.regs)
    for a, nd in zip(st, eng.regs):
        r = plan.reg[nd.idx]
        # (Z, ldz, n_out, t, y, n_cls, pos, orig, count, n, out, stream)
        assert a[2] == 4 and a[3] == r.y.data_ptr() != plan.y.data_ptr() and a[4] == plan.y.data_ptr() and a[5] == 10
        assert tuple(r.y.shape) == (32, 4) and tuple(r.w_cls.shape) == (10, 4)
    buf = torch.zeros(64)
    walk = _walk_calls(ev, rec, _LeafEmit(ev, *(buf.data_ptr() + 4 * i for i in range(4))), n, monkeypatch)
    em = [a for c, a in walk if c == 'leaf_emit_strided']
    # (Z, ldz, n_out, pos, orig, count, n, leaf, path_ops, prob, ldp, cls, exit, ops, stream): 4 columns, rows of 10
    assert len(em) == len(eng.leaves) and all(a[2] == 4 and a[10] == 10 for a in em)

