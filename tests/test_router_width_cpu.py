"""Routers of hidden width W = 16, 32 or 64 (arch_and_hypers.router_n_chan) on the host: dry-run plans size every
router buffer and head by W and pass W to every router-tail launch; the recording stand-in of test_schedule_cpu.py
finds every conflicting pair of launches ordered; unserved widths are refused by name."""
import contextlib
import os
import re
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import arch_and_hypers as ah  # noqa: E402
import util  # noqa: E402
from lib import _cabi, layer_types, engine as E  # noqa: E402
from lib.layer_types import BatchNorm, Chain, Rect, Select  # noqa: E402
from test_schedule_cpu import Recorder, _check, _tensor_index  # noqa: E402

KINDS = [('ac', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('ac', dict(dyn_k_cpt=True))]


def _router(widths):
    """util.router with hidden widths (w1, w2) in place of (16, 16)"""
    def make(n_sinks):
        if n_sinks < 2:
            return None
        return Chain(name='Router', comps=[Select(i=-1), util._fc(widths[0]), BatchNorm(), Rect(), util._fc(widths[1]),
                                           BatchNorm(), Rect(), util._fc(n_sinks, 0)])
    return make


@contextlib.contextmanager
def router_widths(*per_router):
    """tiny nets built inside get routers of these hidden widths: an int W, a pair (w1, w2), or one entry per
    router in build order (the last one repeats)"""
    made = [0]
    orig = util.router

    def make(n_sinks):
        if n_sinks < 2:
            return None
        w = per_router[min(made[0], len(per_router) - 1)]
        made[0] += 1
        return _router(w if isinstance(w, tuple) else (w, w))(n_sinks)
    util.router = make
    try:
        yield
    finally:
        util.router = orig


def tiny_wide(W, kind, **hy):
    with router_widths(W):
        return util.tiny_net(kind, **hy)


@contextlib.contextmanager
def router_n_chan(W):
    old = ah.router_n_chan
    ah.router_n_chan = W
    try:
        yield
    finally:
        ah.router_n_chan = old


class ArgLog:
    """C ABI stand-in that keeps the name and arguments of every call"""
    def __init__(self, real):
        self.protos, self.launches, self.calls = real.protos, 0, []

    def __getattr__(self, name):
        def call(*args):
            self.calls.append((name, args))
            self.launches += 1
            return 0
        return call


def _engine(net, prec):
    return E.Engine(net, precision=prec, impl=0 if prec == 'fp32' else 1, dry_run=True)


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('W', [32, 64])
@pytest.mark.parametrize('kind,hy', KINDS)
def test_plan_sizes_router_buffers_and_launches_by_width(kind, hy, W, prec):
    B = 12
    eng = _engine(tiny_wide(W, kind, **hy), prec)
    assert eng.router_width == W
    eng.L = log = ArgLog(eng.L)
    plan = eng._plan(B, True, True)
    assert plan.rtr and plan.umma_heads == (prec == 'bf16')
    for idx, rt in plan.rtr.items():
        assert tuple(rt.Z1.shape) == (B, W) and tuple(rt.Z2.shape) == (B, W) and tuple(rt.dZ1.shape) == (B, W)
        assert rt.save.numel() >= 4 * W and rt.scratch.numel() >= 2 * B * W
        if plan.umma_heads:
            hd = plan.heads[idx]
            assert hd.N == (16 if hd.leaf_off is not None else 0) + W
            assert tuple(hd.dZ.shape) == (hd.N // 8, plan.Balloc, 8) and hd.r_off + W == hd.N
    log.calls = []
    for op in plan.pack_ops + plan.fwd_ops + plan.bwd_ops:
        op()
    by = {}
    for name, args in log.calls:
        by.setdefault(name, []).append(args)
    assert [a[3] for a in by['router_tail_fwd_batched']] == [W]
    assert [a[3] for a in by['router_tail_bwd_batched']] == [W]
    if plan.umma_heads:
        for a in by['fc_wgrad']:                     # (X, F, Balloc, B, dZ, N, Nsplit, dWa, Fa, na, dWb, Fb, nb)
            assert a[5] in (W, 16 + W, 16) and (a[9] == W or a[12] == W or a[5] == 16)
            assert a[6] == (16 if a[5] != W else W)
    else:
        assert sorted({a[7] for a in by['fc_fwd']}) == sorted({10, W})                         # leaves and fc1
        assert {a[6] for a in by['fc_bwd_weight']} == {10, W}
        assert all(a[5] in (0, W) for a in by['fc_bwd_data'])


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('W', [32, 64])
@pytest.mark.parametrize('kind,hy', KINDS)
def test_every_conflicting_pair_of_launches_is_ordered_at_width(kind, hy, W, prec):
    eng = _engine(tiny_wide(W, kind, **hy), prec)
    holder = {}
    eng.L = Recorder(eng.L, lambda ptr: holder['lookup'](ptr)[2])
    plan = eng._plan(12, True, True)
    holder['lookup'] = _tensor_index(eng, plan)
    problems = _check(eng, plan)
    assert not problems, problems[:8]


@pytest.mark.parametrize('W', [16, 32, 64])
def test_fullsize_ac_chain_keeps_the_tensor_core_heads(W):
    """router_n_chan set the reference's way: router() reads it when the net is built"""
    layer_types.seed(0)
    with router_n_chan(W):
        net = ah.ac_chain(k_cpt=4e-9)((32, 32, 3), (10,))
    assert all(nd.router is None or nd.router.comps[1].hypers.n_chan == W for nd in _nodes(net))
    eng = E.Engine(net, precision='bf16', impl=1, dry_run=True)
    plan = eng._plan(128, True, True)
    assert eng.router_width == W and plan.umma_heads
    assert sorted({hd.N for hd in plan.heads.values()}) == [16, 16 + W]


def _nodes(net):
    out, todo = [], [net.root]
    while todo:
        ℓ = todo.pop()
        out.append(ℓ)
        todo += list(getattr(ℓ, 'sinks', []))
    return out


def test_router_n_chan_default_is_16():
    assert ah.router_n_chan == 16


@pytest.mark.parametrize('widths,what', [
    ((24,), 'hidden widths 24 and 24'),
    (((32, 16),), 'hidden widths 32 and 16'),
    ((32, 64), 'different widths'),
])
def test_unserved_widths_are_refused_naming_the_served_set(widths, what):
    with router_widths(*widths):
        net = util.tiny_net('ac', k_cpt=4e-9)
    with pytest.raises(NotImplementedError) as e:
        _engine(net, 'fp32')
    assert what in str(e.value) and '(16, 32, 64)' in str(e.value)


# the router-tail and FC-head prototypes as the parent commit declares them: wider routers reuse the C argument
PROTOTYPES = {
    'mpnn_router_tail_fwd_batched': 'int mpnn_router_tail_fwd_batched(const mpnn_router_fwd_desc* descs, int n, int B, '
                                    'int C, float d, float eps, int train, void* stream);',
    'mpnn_router_tail_fwd_batched_counted': 'int mpnn_router_tail_fwd_batched_counted(const mpnn_router_fwd_desc* descs, '
                                            'int n, int B, int C, float d, float eps, int train, const int* count, '
                                            'void* stream);',
    'mpnn_router_tail_bwd_batched': 'int mpnn_router_tail_bwd_batched(const mpnn_router_bwd_desc* descs, int n, int B, '
                                    'int C, void* stream);',
}


def test_router_tail_prototypes_are_unchanged():
    src = re.sub(r'/\*.*?\*/', ' ', open(_cabi.HEADER).read(), flags=re.S)
    src = re.sub(r'//[^\n]*', ' ', src)
    for name, proto in PROTOTYPES.items():
        m = re.search(r'\bint\s+' + name + r'\s*\([^;]*\)\s*;', src)
        assert m is not None, name
        assert ' '.join(m.group(0).split()) == proto, name

