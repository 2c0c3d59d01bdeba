"""Routed inference and compacted statistics in bf16x6 precision on the host: the counted three-way split is declared
and exported, the walk accepts bf16x6 and still refuses bf16x3, and the walk launches the dense eval plan's convs and
splits -- on dry-run engines, whose library calls are recorded instead of run."""
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
from util import tiny_net  # noqa: E402

CASES = [('ac', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('sr', {}),
         ('ac', dict(dyn_k_cpt=True))]
F32, BF16 = 0, 1


def _dry(net, precision='bf16x6'):
    return net.configure(precision=precision, dry_run=True, impl=1)


def test_counted_split_is_declared_and_exported():
    protos = _cabi.parse_header()
    _, args, names = protos['mpnn_split_planes3_counted']
    assert names == ['src', 'C', 'B', 'H', 'W', 'G', 'P', 'dst', 'count', 'stream']
    assert args[1:7] == [ctypes.c_int] * 6 and args[8] is ctypes.c_void_p
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    assert hasattr(lib, 'mpnn_split_planes3_counted') and hasattr(lib, 'mpnn_split_planes3')


@pytest.mark.parametrize('kind,hy', CASES)
def test_bf16x6_builds_the_evaluator_and_the_predictor(kind, hy):
    net = _dry(tiny_net(kind, **hy))
    ev = net.compact_evaluator(64)
    assert ev.eng.split == 3 and not ev.plan.umma_heads
    assert net.predictor(64).ev is ev
    for i, bufs in ev.cin.items():                       # compact inputs below a switch: the split planes
        for slot, t in zip(ev.plan.node[i].pin, bufs):
            assert t.dtype == torch.bfloat16 and tuple(t.shape) == tuple(slot.split.shape)


def test_bf16x3_is_still_refused():
    net = _dry(tiny_net('ac', k_cpt=4e-9), 'bf16x3')
    for call in (lambda: net.compact_evaluator(16), lambda: net.predictor(16),
                 lambda: net.predict(np.zeros((2, 16, 16, 3), np.float32), batch=16)):
        with pytest.raises(NotImplementedError, match='bf16x3'):
            call()


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


@pytest.mark.parametrize('kind,hy', CASES)
def test_walk_launches_the_dense_eval_plans_convs_and_splits(kind, hy, monkeypatch):
    net = _dry(tiny_net(kind, **hy))
    eng = net._get_engine()
    rec = _Recorder()
    eng.L = rec
    n = 24
    ev = net.compact_evaluator(32)                       # its plan is the dense eval plan, built on the recorder
    plan = ev.plan
    for op in plan.fwd_ops:
        if getattr(op, 'kind', '') == 'conv_fwd':
            op()
    # conv_acc_bn_stats(A0, K0, A1, K1, Wp, bias, out, N, acc, B, H, W, G, P, bn, dtype, out_dtype, impl, stream)
    dense = [a[:9] + a[15:18] for a in rec.take('conv_acc_bn_stats')]
    for op in plan.fwd_ops:
        if getattr(op, 'kind', '') == 'split':
            op()
    dense_splits = sorted((a[0], a[1], a[3]) for a in rec.take('split_planes3'))        # (src, C, dst)

    monkeypatch.setattr(torch.cuda, 'current_stream', lambda *a: Ns(cuda_stream=0))

    def every_sink(nd, sw, stream):                      # each switch sends its whole batch down every sink
        for s in range(len(nd.kids)):
            yield s, (n, None), stream
    ev._walk((n, None), _LeafStats(ev), every_sink)
    calls = rec.calls
    # the gathers below a switch move the parent's split planes (3C bf16 channels) into the compact inputs
    to_split = {}
    for i, bufs in ev.cin.items():
        for slot, t in zip(plan.node[i].pin, bufs):
            to_split[t.data_ptr()] = slot.split.data_ptr()
    gathers = [a for name, a in calls if name == 'gather_images']
    assert len(gathers) == sum(len(b) for b in ev.cin.values())
    for a in gathers:
        assert to_split[a[5]] == a[0] and a[12] == BF16
    # stencil_gemm_counted(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1, N1, acc1, B, H, W, G, P, stats,
    #                      stats_cap, n_parts, dtype, out_dtype, impl, count, stream)
    walk = []
    for name, a in calls:
        if name == 'stencil_gemm_counted':
            assert a[5] == 9 and a[10] is None and a[13] == n
            walk.append((to_split.get(a[0], a[0]), a[1], to_split.get(a[2], a[2]), a[3], a[4], a[6], a[7], a[8], a[9],
                         a[21], a[22], a[23]))
    n_scales = 0
    for st in plan.node.values():
        for sc in getattr(st, 'sc', []):
            lin = sc.lin.data_ptr()
            d = [c for c in dense if c[6] == lin]
            w = [c for c in walk if c[6] == lin]
            assert len(d) == len(sc.passes) == len(w) >= 2 and d == w
            assert [c[4] for c in w] == [ps.W.data_ptr() for ps in sc.passes]
            assert w[0][5] is not None and w[0][8] == 0 and all(c[5] is None and c[8] == 1 for c in w[1:])
            assert all(c[9:] == (BF16, F32, 1) for c in w)
            n_scales += 1
    assert n_scales and len(walk) == len(dense)
    # the walk splits every tensor the dense plan splits, on the live images
    splits = [a for name, a in calls if name == 'split_planes3_counted']
    assert all(a[2] == n and a[8] is None for a in splits)
    assert sorted((a[0], a[1], a[7]) for a in splits) == dense_splits
