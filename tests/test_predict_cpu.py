"""Routed inference (`Net.predict`, lib/compact_eval.py) on the host: argument checks, the compositions the
compacted walk refuses, the per-leaf path cost table, and the walk's launches against the dense eval plan's -- all on
dry-run engines, which plan without a device (their library calls are recorded instead of run)."""
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
from lib.compact_eval import _LeafStats  # noqa: E402
from lib.layer_types import BatchNorm, Chain, Conv, CrossEntropyError, Dropout, LinTrans, Rect, Softmax  # noqa: E402
from lib.net_types import SRNet  # noqa: E402
from util import tiny_net  # noqa: E402


def _dry(net, precision='fp32'):
    return net.configure(precision=precision, dry_run=True, impl=0 if precision == 'fp32' else 1)


def test_new_entry_points_are_declared_and_exported():
    protos = _cabi.parse_header()
    for name in ('mpnn_leaf_emit', 'mpnn_gather_feature'):
        assert name in protos, name
    assert len(protos['mpnn_leaf_emit'][1]) == 14 and protos['mpnn_leaf_emit'][1][8] is ctypes.c_double
    assert len(protos['mpnn_gather_feature'][1]) == 9
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    assert hasattr(lib, 'mpnn_leaf_emit') and hasattr(lib, 'mpnn_gather_feature')


def test_k_cpt_is_checked_before_any_launch():
    x0 = np.zeros((5, 16, 16, 3), np.float32)
    y = np.zeros((5, 10), np.float32)
    dyn = _dry(tiny_net('ac', dyn_k_cpt=True))
    with pytest.raises(ValueError, match='per-example k_cpt'):
        dyn.predict(x0, batch=64)
    with pytest.raises(ValueError, match='3 values for 5 examples'):
        dyn.predict(x0, k_cpt=[1e-8, 2e-8, 3e-8], batch=64)
    with pytest.raises(ValueError, match='3 values for 5 examples'):
        dyn.compact_evaluator(64).run_batch(x0, y, k_cpt=np.ones(3))
    fixed = _dry(tiny_net('ac', k_cpt=4e-9))
    with pytest.raises(ValueError, match='dyn_k_cpt'):
        fixed.predict(x0, k_cpt=4e-9, batch=64)
    sr = _dry(tiny_net('sr'))
    with pytest.raises(ValueError, match='dyn_k_cpt'):
        sr.predict(x0, k_cpt=[1e-8], batch=64)
    with pytest.raises(ValueError, match='shape'):
        sr.predict(np.zeros((5, 8, 8, 3), np.float32), batch=64)
    with pytest.raises(ValueError, match='dynamically-routed'):         # statistics stay for routed nets
        sr.compact_evaluator(64).run_batch(x0, y)


def _dropout_net():
    blk = Chain(name='ConvBlock', comps=[Conv(n_chan=16, supp=3, k_l2=1e-4, σ_w=1), BatchNorm(), Rect(), Dropout(λ=0.5)],
                sinks=[Chain(name='LogReg', comps=[LinTrans(n_chan=10, k_l2=1e-4, σ_w=1), Softmax(), CrossEntropyError()])])
    return SRNet(x0_shape=(16, 16, 3), y_shape=(10,), root=blk)


@pytest.mark.parametrize('make,precision,reason', [
    (lambda: tiny_net('ac', k_cpt=4e-9), 'bf16x3', 'bf16x3'),
    (lambda: tiny_net('acsq', k_cpt=4e-9), 'fp32', 'CrossEntropyError'),
    (lambda: tiny_net('cnvmp'), 'fp32', 'MaxPool'),
    (_dropout_net, 'fp32', 'Dropout'),
])
def test_refused_compositions_name_their_reason(make, precision, reason):
    net = _dry(make(), precision)
    with pytest.raises(NotImplementedError, match=reason):
        net.predict(np.zeros((2, 16, 16, 3), np.float32), batch=16)


@pytest.mark.parametrize('kind,hy', [('ac', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('sr', {})])
def test_path_cost_table_is_the_dense_moc_of_every_one_hot_route(kind, hy):
    net = _dry(tiny_net(kind, **hy), 'bf16')
    ev = net.compact_evaluator(32)
    eng = ev.eng
    leaves = list(net.leaves)
    assert len(ev.path_ops) == len(leaves) == len(eng.leaves)
    for i, leaf in enumerate(eng.leaves):
        assert leaf.layer is leaves[i]
        p_ev = np.zeros((len(eng.nodes), 1))
        j = leaf.idx
        while j is not None:
            p_ev[j] = 1.0
            j = eng.nodes[j].parent
        moc = np.zeros(1)                                    # Engine.eval_stats
        for nd in eng.nodes:
            ops = nd.layer.n_ops + (nd.router.n_ops if nd.router is not None else 0)
            moc += p_ev[nd.idx] * ops
        assert ev.path_ops[i] == moc[0] > 0
    assert len(ev.path_ops) == 1 if kind == 'sr' else len(set(ev.path_ops)) > 1


class _Recorder:
    """stands in for the C library: every call is recorded as (name, args), pointers as ints"""
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        name = name[5:] if name.startswith('mpnn_') else name

        def call(*args):
            self.calls.append((name, tuple(a.value if isinstance(a, ctypes.c_void_p) else a for a in args)))
            return 0
        return call

    def take(self, name):
        out = [a for n, a in self.calls if n == name]
        self.calls = []
        return out


F32, BF16 = 0, 1


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'bf16x6'])
@pytest.mark.parametrize('kind,hy', [('ac', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)),
                                     ('sr', {}), ('ac', dict(dyn_k_cpt=True))])
def test_walk_launches_the_dense_eval_plans_convs_and_splits(kind, hy, precision, monkeypatch):
    net = _dry(tiny_net(kind, **hy), precision)
    eng = net._get_engine()
    x6 = precision == 'bf16x6'
    dt = BF16 if precision == 'bf16' else F32
    rec = _Recorder()
    eng.L = rec
    n = 24
    ev = net.compact_evaluator(32)                       # its plan is the dense eval plan, built on the recorder
    plan = ev.plan
    for op in plan.fwd_ops:
        if getattr(op, 'kind', '') == 'conv_fwd':
            op()
    if x6:
        # conv_acc_bn_stats(A0, K0, A1, K1, Wp, bias, out, N, acc, B, H, W, G, P, bn, dtype, out_dtype, impl, stream)
        dense = [a[:9] + a[15:18] for a in rec.take('conv_acc_bn_stats')]
    else:
        # stencil_gemm(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1, N1, acc1, B, H, W, G, P, stats,
        #              stats_cap, n_parts, dtype, out_dtype, impl, stream)
        dense = [a[:5] + a[6:10] + a[21:24] for a in rec.take('stencil_gemm')]
    for op in plan.fwd_ops:
        if getattr(op, 'kind', '') == 'split':
            op()
    dense_splits = sorted((a[0], a[1], a[3]) for a in rec.take('split_planes3'))        # (src, C, dst)
    assert bool(dense_splits) == x6

    monkeypatch.setattr(torch.cuda, 'current_stream', lambda *a: Ns(cuda_stream=0))

    def every_sink(nd, sw, stream):                      # each switch sends its whole batch down every sink
        for s in range(len(nd.kids)):
            yield s, (n, None), stream
    ev._walk((n, None), _LeafStats(ev), every_sink)
    calls = rec.calls
    # the gathers below a switch move the parent's tensors -- in bf16x6 its split planes (3C bf16 channels) -- into
    # the compact inputs
    to_src = {}
    for i, bufs in ev.cin.items():
        for slot, t in zip(plan.node[i].pin, bufs):
            to_src[t.data_ptr()] = (slot.split if x6 else slot.t).data_ptr()
    gathers = [a for name, a in calls if name == 'gather_images']
    assert len(gathers) == sum(len(b) for b in ev.cin.values())
    for a in gathers:
        assert to_src[a[5]] == a[0] and a[12] == (BF16 if x6 else dt)
    # stencil_gemm_counted(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1, N1, acc1, B, H, W, G, P, stats,
    #                      stats_cap, n_parts, dtype, out_dtype, impl, count, stream)
    walk = []
    for name, a in calls:
        if name == 'stencil_gemm_counted' and (x6 or a[5] == 9):         # (ntaps 1: the tcgen05 heads' GEMM)
            assert a[5] == 9
            assert a[10] is None and a[13] == n
            walk.append((to_src.get(a[0], a[0]), a[1], to_src.get(a[2], a[2]), a[3], a[4], a[6], a[7], a[8], a[9],
                         a[21], a[22], a[23]))
    n_scales = 0
    for st in plan.node.values():
        for sc in getattr(st, 'sc', []):
            lin = sc.lin.data_ptr()
            d = [c for c in dense if c[6] == lin]
            w = [c for c in walk if c[6] == lin]
            assert len(d) == len(sc.passes) == len(w) and d == w
            assert len(w) >= 2 if x6 else len(w) == 1
            assert [c[4] for c in w] == [ps.W.data_ptr() for ps in sc.passes]
            assert w[0][5] is not None and w[0][8] == 0 and all(c[5] is None and c[8] == 1 for c in w[1:])
            assert all(c[9:] == ((BF16, F32, 1) if x6 else (dt, dt, eng.impl)) for c in w)
            n_scales += 1
    assert n_scales and len(walk) == len(dense)
    # the walk splits every tensor the dense plan splits, on the live images
    splits = [a for name, a in calls if name == 'split_planes3_counted']
    assert all(a[2] == n and a[8] is None for a in splits)
    assert sorted((a[0], a[1], a[7]) for a in splits) == dense_splits
