"""Routed inference and compacted statistics in bf16x6 precision on the host: the counted three-way split is declared
and exported, and the walk accepts bf16x6 and still refuses bf16x3 -- on dry-run engines, which plan without a device.
(That the walk launches the dense eval plan's convs and splits is checked for every precision in test_predict_cpu.py.)"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

from lib import _cabi  # noqa: E402
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
