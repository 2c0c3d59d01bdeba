"""Device statistics (`Net.stats_evaluator`, lib/dense_stats.py) on the host: the C ABI of the accumulate launch, the
refusals and argument checks, the descriptor table and the launch list of one chunk -- on dry-run engines, which plan
without a device."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

from lib import _cabi  # noqa: E402
from lib.desc import state_tensors  # noqa: E402
from test_predict_cpu import _dropout_net  # noqa: E402
from util import tiny_net  # noqa: E402

PKG = os.path.join(ROOT, 'multipath-nn_b200')


def _dry(net, precision='fp32'):
    return net.configure(precision=precision, dry_run=True, impl=0 if precision == 'fp32' else 1)


def test_accumulate_prototype_is_declared_and_exported():
    protos = _cabi.parse_header()
    _, args, names = protos['mpnn_stats_accumulate']
    assert names == ['descs', 'n_leaf', 'n_sw', 'y', 'n_cls', 'node_p_ev', 'ops', 'n_nodes', 'B', 'work', 'total',
                     'count', 'stream']
    assert [a is ctypes.c_int for a in args] == [False, True, True, False, True, False, False, True, True, False,
                                                 False, False, False]
    assert hasattr(ctypes.CDLL(_cabi.LIB_PATH), 'mpnn_stats_accumulate')


def test_dropout_is_refused_with_its_reason():
    net = _dry(_dropout_net())
    with pytest.raises(NotImplementedError, match=r'Dropout\(λ < 1\).*batch layout'):
        net.stats_evaluator(16)


def test_capacity_and_shape_errors_come_before_any_launch():
    net = _dry(tiny_net('ac', k_cpt=4e-9))
    ev = net.stats_evaluator(16)
    assert net.stats_evaluator(16) is ev and net.stats_evaluator(32) is not ev
    L = _cabi.lib()
    before = L.launches
    x0, y = np.zeros((17, 16, 16, 3), np.float32), np.zeros((17, 10), np.float32)
    with pytest.raises(ValueError, match='17 > evaluator capacity 16'):
        ev.run_batch(x0, y)
    with pytest.raises(ValueError, match='x0: shape'):
        ev.run_batch(np.zeros((5, 8, 8, 3), np.float32), y[:5])
    with pytest.raises(ValueError, match='y: shape'):
        ev.run_batch(x0[:5], y[:4])
    ev.run_batch(x0[:0], y[:0])                               # n = 0: nothing to run
    with pytest.raises(RuntimeError, match='dry-run'):
        ev.run_batch(x0[:5], y[:5])
    assert L.launches == before and ev.graph is None and ev.n_seen == 0


def _decode(ev):
    from lib.dense_stats import _STATS
    return np.frombuffer(ev.tab.numpy().tobytes(), dtype=_STATS)


@pytest.mark.parametrize('kind,hy', [('ac', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('sr', {}),
                                     ('crsce', dict(k_cpt=4e-9))])
def test_descriptor_table_decodes_to_the_plans_buffers(kind, hy):
    net = _dry(tiny_net(kind, **hy), 'bf16')
    ev = net.stats_evaluator(32)
    eng, plan = ev.eng, ev.plan
    assert plan is eng._plan(32, False, False)               # the engine's dense eval plan at the capacity
    tab = _decode(ev)
    assert len(tab) == len(eng.regs) + len(eng.switches)
    ptr = lambda t: 0 if t is None else t.data_ptr()
    for row, nd in zip(tab, eng.regs):
        r = plan.reg[nd.idx]
        assert row['d_cor'] == ptr(r.d_cor) and row['c_err'] == ptr(r.c_err) and row['R'] == 0 and row['ns'] == 0
        if eng.dynamic:
            assert row['p_ev'] == ptr(plan.p_ev[nd.idx]) and row['p_tr'] == ptr(plan.p_tr[nd.idx])
        else:
            assert row['p_ev'] == 0 and row['p_tr'] == 0
    for row, nd in zip(tab[len(eng.regs):], eng.switches):
        assert row['R'] == ptr(plan.rtr[nd.idx].R) and row['ns'] == len(nd.kids)
        assert row['p_ev'] == row['p_tr'] == row['d_cor'] == row['c_err'] == 0
    # one total per statistic of state_tensors, in the layout of include/mpnn.h
    n_keys = sum(1 if name not in ('p_cor_by_cls', 'p_inc_by_cls') else ev.n_cls for _, name in state_tensors(net))
    assert ev.M == n_keys + (0 if eng.dynamic else len(eng.regs))          # SR nets keep an unused p_tr column
    assert ev.work.numel() == -(-32 // 32) * ev.M


class _Recorder:
    """stands in for the C library: records the names of the entry points a launch list calls"""
    def __init__(self):
        self.calls = []
        self.launches = 0

    def __getattr__(self, name):
        if name.startswith('__'):
            raise AttributeError(name)

        def call(*args):
            self.calls.append(name)
            return 0
        return call


@pytest.mark.parametrize('kind,hy,prec', [('ac', dict(k_cpt=4e-9), 'bf16'), ('sr', {}, 'fp32'),
                                          ('acsce', dict(k_cpt=4e-9), 'fp32'), ('ac', dict(k_cpt=4e-9), 'bf16x6')])
def test_a_chunk_launches_the_dense_eval_plan_and_one_accumulate(kind, hy, prec):
    net = _dry(tiny_net(kind, **hy), prec)
    eng = net._get_engine()
    eng.L = rec = _Recorder()                                # before the plan is built: its ops call the recorder
    ev = net.stats_evaluator(64)
    plan = ev.plan
    assert ev.op_lists[0] is plan.pack_ops and ev.op_lists[1] is plan.fwd_ops and len(ev.op_lists[2]) == 1

    def run(ops):
        rec.calls = []
        for op in ops:
            op()
        return rec.calls
    want = run(plan.pack_ops) + run(plan.fwd_ops)
    got = run([op for ops in ev.op_lists for op in ops])
    assert got == want + ['stats_accumulate']
    if kind.endswith('sce'):                                 # the superclass targets read each chunk's labels
        assert 'superclass_targets' in run(plan.pack_ops)


def test_device_and_compact_statistics_exclude_each_other():
    r = subprocess.run([sys.executable, os.path.join(PKG, 'train-nets'), 'cifar10-ac', '--synthetic', '--device-stats',
                        '--compact-stats'], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and 'choose one' in r.stderr
    r = subprocess.run([sys.executable, os.path.join(PKG, 'train-adaptive-nets'), 'hybrid-ac-dynkcpt', '--synthetic',
                        '--device-stats', '--compact-stats'], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and 'choose one' in r.stderr


def test_net_desc_refuses_compact_and_device_together():
    from lib.data import Dataset, synthetic_archive
    from lib.desc import net_desc
    net = _dry(tiny_net('ac', k_cpt=4e-9))
    ds = Dataset(archive=synthetic_archive(8, 8, (16, 16, 3), 10))
    with pytest.raises(ValueError, match='choose one'):
        net_desc(net, ds, {}, state_tensors(net), compact=True, device=True)
