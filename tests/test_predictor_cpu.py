"""Graph-replayed routed inference (`Net.predictor`) on the host: the counted entry points of the C ABI, and the
argument checks and refused compositions the predictor shares with `Net.predict` -- on dry-run engines, which plan
without a device."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

from lib import _cabi  # noqa: E402
from test_predict_cpu import _dropout_net  # noqa: E402
from util import tiny_net  # noqa: E402

COUNTED = ['mpnn_pack_input', 'mpnn_stencil_gemm', 'mpnn_bn_relu_pool_fwd', 'mpnn_fc_fwd',
           'mpnn_router_tail_fwd_batched', 'mpnn_route_compact']


def _dry(net, precision='fp32'):
    return net.configure(precision=precision, dry_run=True, impl=0 if precision == 'fp32' else 1)


def test_counted_entry_points_are_the_uncounted_ones_plus_a_count():
    protos = _cabi.parse_header()
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for name in COUNTED:
        _, args, names = protos[name]
        _, cargs, cnames = protos[name + '_counted']
        assert len(cargs) == len(args) + 1, name
        assert cnames[:-2] == names[:-1] and cnames[-1] == 'stream', name         # the count goes before the stream
        assert cargs[-2] is ctypes.c_void_p and cnames[-2] in ('count', 'n_count'), name
        assert hasattr(lib, name + '_counted'), name


def test_predictor_checks_its_arguments_like_predict():
    x0 = np.zeros((5, 16, 16, 3), np.float32)
    dyn = _dry(tiny_net('ac', dyn_k_cpt=True))
    p = dyn.predictor(64)
    assert dyn.predictor(64) is p and dyn.predictor(32) is not p
    with pytest.raises(ValueError, match='per-example k_cpt'):
        p(x0)
    with pytest.raises(ValueError, match='3 values for 5 examples'):
        p(x0, k_cpt=[1e-8, 2e-8, 3e-8])
    fixed = _dry(tiny_net('ac', k_cpt=4e-9))
    with pytest.raises(ValueError, match='dyn_k_cpt'):
        fixed.predictor(64)(x0, k_cpt=4e-9)
    sr = _dry(tiny_net('sr'))
    with pytest.raises(ValueError, match='dyn_k_cpt'):
        sr.predictor(64)(x0, k_cpt=[1e-8])
    with pytest.raises(ValueError, match='shape'):
        sr.predictor(64)(np.zeros((5, 8, 8, 3), np.float32))


def test_n_above_the_capacity_is_refused_before_any_launch():
    net = _dry(tiny_net('ac', k_cpt=4e-9))
    p = net.predictor(16)
    L = _cabi.lib()
    before = L.launches
    with pytest.raises(ValueError, match='17 > predictor capacity 16'):
        p(np.zeros((17, 16, 16, 3), np.float32))
    assert L.launches == before and p.graph is None
    e = p(np.zeros((0, 16, 16, 3), np.float32))              # n = 0: empty outputs, nothing launched
    assert tuple(e.prob.shape) == (0, 10) and tuple(e.cls.shape) == (0,) and p.graph is None


@pytest.mark.parametrize('make,precision,reason', [
    (lambda: tiny_net('ac', k_cpt=4e-9), 'bf16x3', 'bf16x3'),
    (lambda: tiny_net('acsq', k_cpt=4e-9), 'fp32', 'CrossEntropyError'),
    (lambda: tiny_net('cnvmp'), 'fp32', 'MaxPool'),
    (_dropout_net, 'fp32', 'Dropout'),
])
def test_predictor_refuses_what_predict_refuses(make, precision, reason):
    net = _dry(make(), precision)
    with pytest.raises(NotImplementedError, match=reason):
        net.predictor(16)
