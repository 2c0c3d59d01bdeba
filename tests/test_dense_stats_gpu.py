"""Device statistics on the B200: mpnn_stats_accumulate against a NumPy restatement, and `net_desc(device=True)`
(lib/dense_stats.py) against the host path `net_desc(...)` (Engine.eval_stats per 128-example slice, NumPy sums) on
the same trained net in the same process.  Count-valued statistics (p_cor, p_inc, the per-class entries, acc, moc)
are sums of integers in fp64 and must have the same bits; c_err, p_tr and x_rte differ by summation order only."""
import ctypes
import os
import sys
import warnings

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

from lib.data import Dataset, synthetic_archive  # noqa: E402
from lib.desc import net_desc, state_tensors  # noqa: E402
from util import randomize_routers, tiny_net  # noqa: E402

pytestmark = pytest.mark.gpu

COUNT_KEYS = ('p_cor', 'p_inc', 'p_cor_by_cls', 'p_inc_by_cls', 'acc', 'moc')


def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


# --------------------------------------------------------------------------- #
# the kernel
# --------------------------------------------------------------------------- #
def _kernel_case(B, n_cls, seed):
    rng = np.random.default_rng(seed)
    n_leaf, n_sw, n_nodes = 3, 2, 6
    leaf_nodes = [1, 3, 5]
    p_ev = (rng.random((n_nodes, B)) < 0.5).astype(np.float32)
    p_ev[leaf_nodes] = np.eye(n_leaf, dtype=np.float32)[rng.integers(0, n_leaf, B)].T       # one-hot over the leaves
    c = dict(
        p_ev=p_ev, p_tr=rng.random((n_leaf, B)).astype(np.float32),
        d_cor=(rng.random((n_leaf, B)) < 0.6).astype(np.float32),
        c_err=(3 * rng.random((n_leaf, B))).astype(np.float32),
        R=[rng.standard_normal((B, ns)).astype(np.float32) for ns in (2, 3)],
        y=np.eye(n_cls, dtype=np.float32)[rng.integers(0, n_cls, B)],
        ops=rng.integers(1, 10 ** 7, n_nodes).astype(np.float64), leaf_nodes=leaf_nodes, n_sw=n_sw)
    return c


def _numpy_totals(c, n, dynamic):
    """the host reduction (Engine.eval_stats + _RunningMean) of the first n examples, in the kernel's layout"""
    y = c['y'][:n].astype(np.float64)
    out = []
    acc = np.zeros(n)
    for l, node in enumerate(c['leaf_nodes']):
        pe = c['p_ev'][node, :n].astype(np.float64) if dynamic else np.ones(n)
        dc = c['d_cor'][l, :n].astype(np.float64)
        acc += pe * dc
        out += [(pe * dc).sum(), (pe * (1 - dc)).sum(), c['c_err'][l, :n].astype(np.float64).sum(),
                c['p_tr'][l, :n].astype(np.float64).sum() if dynamic else 0.0]
        out += list(((pe * dc)[:, None] * y).sum(0)) + list(((pe * (1 - dc))[:, None] * y).sum(0))
    for r in c['R']:
        out.append(np.abs(r[:n].astype(np.float64)).mean(1).sum())
    moc = np.zeros(n)
    for i in range(len(c['ops'])):
        moc += (c['p_ev'][i, :n].astype(np.float64) if dynamic else 1.0) * c['ops'][i]
    out += [acc.sum(), moc.sum()]
    return np.array(out)


def _launch(c, B, count, dynamic, total, work):
    from lib import _cabi
    from lib.dense_stats import _STATS
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    keep = {k: dev(c[k]) for k in ('p_ev', 'p_tr', 'd_cor', 'c_err', 'y', 'ops')}
    keep['R'] = [dev(r) for r in c['R']]
    rows = np.zeros(len(c['leaf_nodes']) + c['n_sw'], _STATS)
    for l, node in enumerate(c['leaf_nodes']):
        if dynamic:
            rows[l]['p_ev'] = keep['p_ev'][node].data_ptr()
            rows[l]['p_tr'] = keep['p_tr'][l].data_ptr()
        rows[l]['d_cor'] = keep['d_cor'][l].data_ptr()
        rows[l]['c_err'] = keep['c_err'][l].data_ptr()
    for s, r in enumerate(keep['R']):
        rows[len(c['leaf_nodes']) + s]['R'] = r.data_ptr()
        rows[len(c['leaf_nodes']) + s]['ns'] = r.shape[1]
    tab = torch.from_numpy(rows.view(np.uint8).copy()).cuda()
    cnt = None if count is None else torch.tensor([count], dtype=torch.int32, device='cuda')
    _cabi.lib().stats_accumulate(vp(tab), len(c['leaf_nodes']), c['n_sw'], vp(keep['y']), c['y'].shape[1],
                                 vp(keep['p_ev']) if dynamic else None, vp(keep['ops']), len(c['ops']), B, vp(work),
                                 vp(total), vp(cnt), None)
    torch.cuda.synchronize()


def _n_cols(c):
    return len(c['leaf_nodes']) * (4 + 2 * c['y'].shape[1]) + c['n_sw'] + 2


def _check_totals(got, want, c):
    per_leaf = 4 + 2 * c['y'].shape[1]
    n_leaf = len(c['leaf_nodes'])
    exact = np.ones(len(want), bool)
    for l in range(n_leaf):
        exact[l * per_leaf + 2:l * per_leaf + 4] = False             # c_err, p_tr
    exact[n_leaf * per_leaf:n_leaf * per_leaf + c['n_sw']] = False   # x_rte
    np.testing.assert_array_equal(got[exact], want[exact])
    np.testing.assert_allclose(got[~exact], want[~exact], rtol=1e-12, atol=0)


@pytest.mark.parametrize('n_cls', [10, 100])
@pytest.mark.parametrize('B', [128, 4096, 4097])
def test_accumulate_matches_numpy(B, n_cls):
    c = _kernel_case(B, n_cls, seed=B + n_cls)
    M = _n_cols(c)
    work = torch.full((-(-B // 32) * M,), float('nan'), dtype=torch.float64, device='cuda')
    for dynamic in (True, False):
        for count in (0, 1, 4095, B, None):
            if count is not None and count > B:
                continue
            n = B if count is None else count
            total = torch.zeros(M, dtype=torch.float64, device='cuda')
            _launch(c, B, count, dynamic, total, work)
            got = total.cpu().numpy()
            want = _numpy_totals(c, n, dynamic)
            if n == 0:
                np.testing.assert_array_equal(got, np.zeros(M))         # n = 0 adds nothing
                continue
            _check_totals(got, want, c)
            _launch(c, B, count, dynamic, total, work)                  # accumulates; same bits twice
            np.testing.assert_array_equal(total.cpu().numpy(), got + got)


def test_accumulate_clamps_the_count_to_the_capacity():
    c = _kernel_case(128, 10, seed=5)
    M = _n_cols(c)
    work = torch.zeros(4 * M, dtype=torch.float64, device='cuda')
    total = torch.zeros(M, dtype=torch.float64, device='cuda')
    _launch(c, 128, 4095, True, total, work)
    _check_totals(total.cpu().numpy(), _numpy_totals(c, 128, True), c)


# --------------------------------------------------------------------------- #
# the evaluator against the host path
# --------------------------------------------------------------------------- #
def _walk(a, b, path=()):
    assert type(a) is type(b), path
    if isinstance(a, dict):
        assert a.keys() == b.keys(), (path, set(a) ^ set(b))
        for k in a:
            yield from _walk(a[k], b[k], path + (k,))
    elif isinstance(a, list) and a and isinstance(a[0], dict):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            yield from _walk(x, y, path + (i,))
    else:
        yield path, a, b


def assert_desc_equal(got, want):
    n = 0
    for path, a, b in _walk(got, want):
        if path[-1] in COUNT_KEYS:
            assert a == b, (path, a, b)
            n += 1
        elif path[-1] in ('c_err', 'p_tr', 'x_rte'):
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=0, err_msg=str(path))
            n += 1
        else:
            assert a == b, path
    assert n > 0


NETS = {'sr': {}, 'ac': dict(k_cpt=4e-9), 'cr': dict(k_cpt=4e-9), 'actree': dict(k_cpt=2e-9),
        'acdyn': dict(dyn_k_cpt=True), 'srsq': {}, 'acsq': dict(k_cpt=4e-9), 'srsce': {}, 'crsce': dict(k_cpt=4e-9),
        'cnv': {}, 'cnvpyr': {}, 'cnvmp': {}, 'cnvgmp': {}, 'cnvact': {}, 'srlln': {}, 'aclln': dict(k_cpt=4e-9)}
CASES = [(k, p) for k in NETS for p in ('fp32', 'bf16')] + [(k, p) for k in ('ac', 'sr') for p in ('bf16x6', 'bf16x3')]


def _trained(kind, prec, steps=2):
    hy = NETS[kind]
    net = tiny_net('ac' if kind == 'acdyn' else kind, seed=2, **hy)
    net = randomize_routers(net).configure(precision=prec) if net.dynamic else net.configure(precision=prec)
    ds = Dataset(archive=synthetic_archive(1000, 300, (16, 16, 3), 10, seed=4), seed=0)
    for t in range(steps):                               # non-trivial running BatchNorm moments
        net.train.run(_train_feed(net, ds, hy))
    return net, ds, hy


def _train_feed(net, ds, hy):
    x0, y = ds.training_batch(64)
    f = {net.x0: x0, net.y: y, net.mode: 'tr', net.λ_lrn: 0.01}
    if net.dynamic:
        f[net.τ] = 0.5
    if hy.get('dyn_k_cpt'):
        f[net.k_cpt] = np.full(64, 4e-9, np.float32)
    return f


def _hypers(net, hy):
    h = {net.τ: 0.5} if net.dynamic else {}
    if hy.get('dyn_k_cpt'):
        h[net.k_cpt] = [1.6e-8]                           # the length-1 feed of train-adaptive-nets:102-105
    return h


@pytest.mark.parametrize('kind,prec', CASES)
def test_device_statistics_equal_the_host_path(kind, prec):
    net, ds, hy = _trained(kind, prec)
    h, state = _hypers(net, hy), state_tensors(net)
    want = net_desc(net, ds, h, state)
    got = net_desc(net, ds, h, state, device=True, batch=256)    # 1000 = 3 x 256 + 232, 300 = 256 + 44
    assert_desc_equal(got, want)


def test_current_parameters_and_reproducible_passes():
    net, ds, hy = _trained('ac', 'bf16')
    h, state = _hypers(net, hy), state_tensors(net)
    first = net_desc(net, ds, h, state, device=True, batch=256)
    again = net_desc(net, ds, h, state, device=True, batch=256)
    for path, a, b in _walk(again, first):                # same data, same chunking: the same bits for every key
        assert a == b, path
    net.train.run({**_train_feed(net, ds, hy), net.λ_lrn: 0.1})   # new weights and running moments
    after = net_desc(net, ds, h, state, device=True, batch=256)
    assert after != first
    assert_desc_equal(after, net_desc(net, ds, h, state))


def test_no_host_synchronisation_per_chunk_and_one_read():
    net, ds, hy = _trained('ac', 'bf16', steps=1)
    ev = net.stats_evaluator(128)
    x0, y = ds.training_set(1000, device=True).__next__()
    h = _hypers(net, hy)
    ev.reset()
    ev.run_batch(x0[:128], y[:128], h)                   # captures the graph (that synchronises once)
    torch.cuda.synchronize()
    ev.reset()
    torch.cuda.set_sync_debug_mode('error')
    try:
        for i in range(0, 1000, 128):
            ev.run_batch(x0[i:i + 128], y[i:i + 128], h)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.set_sync_debug_mode('warn')
    try:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter('always')
            res = ev.result()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len([m for m in w if 'synchroniz' in str(m.message)]) == 1, [str(m.message) for m in w]
    assert ev.n_seen == 1000 and set(res) == set(state_tensors(net))


# --------------------------------------------------------------------------- #
# the real architecture
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize('kind', ['cifar10-ac', 'cifar10-sr'])
def test_full_architecture_at_capacity_4096(kind):
    import arch_and_hypers as ah
    from lib import layer_types
    layer_types.seed(0)
    ctor = ah.ac_chain(k_cpt=4e-9) if kind == 'cifar10-ac' else ah.sr_chain(len(ah.arch))
    net = ctor((32, 32, 3), (10,)).configure(precision='bf16', graphs=True)
    if net.dynamic:
        randomize_routers(net)
    ds = Dataset(archive=synthetic_archive(10000, 1000, (32, 32, 3), 10, seed=1), seed=0)
    for t in range(3):
        x0, y = ds.augmented_training_batch_gpu(128)
        net.train.run({net.x0: x0, net.y: y, net.mode: 'tr', net.λ_lrn: 0.01, **({net.τ: 1.0} if net.dynamic else {})})
    h, state = ({net.τ: 0.5} if net.dynamic else {}), state_tensors(net)
    assert_desc_equal(net_desc(net, ds, h, state, device=True, batch=4096), net_desc(net, ds, h, state))


# --------------------------------------------------------------------------- #
# the drivers
# --------------------------------------------------------------------------- #
def test_drivers_write_the_reference_layout_with_device_statistics(tmp_path):
    from test_drivers_gpu import _check_stats, _run
    _run('train-nets', ['cifar10-ac', '--synthetic', '--n-iter', '4', '--t-log', '2', '--nets', '0',
                        '--device-stats'], str(tmp_path))
    d = tmp_path / 'nets' / 'cifar10-ac'
    for f in ('0000.npy', '0000-stats.npy', '0000-log.txt', '0000-stats/00000002.npy', '0000-stats/00000004.npy'):
        assert (d / f).exists(), f
    stats = np.load(d / '0000-stats.npy', allow_pickle=True)[()]
    assert _check_stats(stats, dynamic=True) == 8
    _run('train-adaptive-nets', ['hybrid-ac-dynkcpt', '--synthetic', '--n-iter', '2', '--device-stats'], str(tmp_path))
    d = tmp_path / 'nets' / 'hybrid-ac-dynkcpt'
    for i in range(8):
        stats = np.load(d / ('%.4i-stats.npy' % i), allow_pickle=True)[()]
        assert _check_stats(stats, dynamic=True) == 8
