"""Routed inference (`Net.predict`, lib/compact_eval.py) on the host: argument checks, the compositions the
compacted walk refuses, and the per-leaf path cost table -- all on dry-run engines, which plan without a device."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

from lib import _cabi  # noqa: E402
from lib.layer_types import BatchNorm, Chain, Conv, CrossEntropyError, Dropout, LinTrans, Rect, Softmax  # noqa: E402
from lib.net_types import SRNet  # noqa: E402
from util import tiny_net  # noqa: E402


def _dry(net, precision='fp32'):
    return net.configure(precision=precision, dry_run=True, impl=0 if precision == 'fp32' else 1)


def test_new_entry_points_are_declared_and_exported():
    protos = _cabi.parse_header()
    for name in ('mpnn_leaf_emit', 'mpnn_gather_feature'):
        assert name in protos, name
    import ctypes
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
