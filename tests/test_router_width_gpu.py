"""Routers of hidden width 32 and 64 on the device: the batched router-tail kernels against a float64 torch
restatement, the counted forward against the uncounted one, reproducible statistics, and the end-to-end paths
(oracle parity of a training step, training, routed inference, compacted statistics, the full architecture) with
the nets of the existing tests rebuilt with wider routers."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import test_compact_eval_gpu as CE  # noqa: E402
import test_fullsize_parity_gpu as FP  # noqa: E402
import test_parity_gpu as PG  # noqa: E402
import test_predict_gpu as PD  # noqa: E402
import test_predictor_gpu as PR  # noqa: E402
from test_predictor_gpu import L, cnt_of, counts, same, untouched, vp  # noqa: E402
from test_router_width_cpu import router_n_chan, router_widths  # noqa: E402
from util import batch, randomize_routers, tiny_net  # noqa: E402

pytestmark = pytest.mark.gpu

D, EPS = 0.9, 1e-6
NS = (2, 5, 8)                         # routers of different fan-out in one launch
BATCHES = [128, 4096, 4097, 8192, 16384]


def _tails(W, B, seed):
    """one descriptor row per router in NS, with its parameters, running moments and output buffers"""
    rng = np.random.default_rng(seed)
    f = lambda *sh, s=1.0, m=0.0: torch.tensor((rng.standard_normal(sh) * s + m).astype(np.float32), device='cuda')
    out = []
    for ns in NS:
        t = dict(ns=ns, Z1=f(B, W, s=2.0, m=0.3), g1=f(W), b1=f(W, s=0.3), W2=f(W, W, s=1.0 / np.sqrt(W)), c2=f(W, s=0.1),
                 g2=f(W), b2=f(W, s=0.3), W3=f(W, ns, s=0.5), c3=f(ns, s=0.1), dR=f(B, ns))
        t['mom'] = [f(W, s=0.1), (f(W, s=0.2) ** 2 + 1.0), f(W, s=0.1), (f(W, s=0.2) ** 2 + 1.0)]
        out.append(t)
    return out


def _fwd(tails, W, B, train, count=None):
    """runs the batched forward on copies of the running moments; returns per router (Z2, R, save, moments)"""
    from lib.engine import _RT_FWD
    rows, res = [], []
    for t in tails:
        mom = [m.clone() for m in t['mom']]
        r = dict(Z2=torch.full((B, W), -1.0, device='cuda'), R=torch.full((B, t['ns']), -1.0, device='cuda'),
                 save=torch.full((4 * W,), -1.0, device='cuda'), mom=mom)
        p = lambda x: x.data_ptr()
        rows.append((p(t['Z1']), p(t['g1']), p(t['b1']), p(mom[0]), p(mom[1]), p(t['W2']), p(t['c2']), p(t['g2']),
                     p(t['b2']), p(mom[2]), p(mom[3]), p(t['W3']), p(t['c3']), p(r['Z2']), p(r['R']), p(r['save']),
                     t['ns'], 0))
        res.append(r)
    table = torch.tensor(np.frombuffer(np.array(rows, dtype=_RT_FWD).tobytes(), np.uint8).copy(), device='cuda')
    if count is None:
        L().router_tail_fwd_batched(vp(table), len(rows), B, W, D, EPS, train, None)
    else:
        L().router_tail_fwd_batched_counted(vp(table), len(rows), B, W, D, EPS, train, vp(count), None)
    torch.cuda.synchronize()
    return res


def _bwd(tails, fwd, W, B):
    from lib.engine import _RT_BWD
    Balloc = -(-B // 128) * 128
    rows, res = [], []
    for t, f in zip(tails, fwd):
        g = {k: torch.zeros_like(t[k]) for k in ('g1', 'b1', 'W2', 'c2', 'g2', 'b2', 'W3', 'c3')}
        g['c1'] = torch.zeros(W, device='cuda')
        g['dZ1'] = torch.full((B, W), -1.0, device='cuda')
        g['dZ1p'] = torch.zeros((W // 8, Balloc, 8), dtype=torch.bfloat16, device='cuda')
        p = lambda x: x.data_ptr()
        rows.append((p(t['Z1']), p(f['Z2']), p(t['dR']), p(t['g1']), p(t['b1']), p(t['W2']), p(t['g2']), p(t['b2']),
                     p(t['W3']), p(f['save']), p(g['g1']), p(g['b1']), p(g['W2']), p(g['c2']), p(g['g2']), p(g['b2']),
                     p(g['W3']), p(g['c3']), p(g['dZ1']), 0, p(g['dZ1p']), p(g['c1']), t['ns'], Balloc))
        res.append(g)
    table = torch.tensor(np.frombuffer(np.array(rows, dtype=_RT_BWD).tobytes(), np.uint8).copy(), device='cuda')
    L().router_tail_bwd_batched(vp(table), len(rows), B, W, None)
    torch.cuda.synchronize()
    return res


def _kernel_gates(t, f, W):
    """the ReLU gates the kernels applied: sign(fmaf(a, z, c)) with a = g * rs and c = b - mean * a in fp32, from the
    kernel's own statistics (save) and Z2.  The sign of a * z + c survives fp32 rounding, so it is taken exactly in
    fp64; c is formed both with and without a fused multiply-add, and elements where the two disagree are reported."""
    save = f['save']
    out = []
    for z, g, b, m, rs in ((t['Z1'], t['g1'], t['b1'], save[:W], save[W:2 * W]),
                           (f['Z2'], t['g2'], t['b2'], save[2 * W:3 * W], save[3 * W:])):
        a = g * rs
        c_fused = (b.double() - m.double() * a.double()).float()
        c_plain = b - m * a
        u = [a.double() * z.double() + c.double() for c in (c_fused, c_plain)]
        out.append(((u[0] > 0).double(), int(((u[0] > 0) != (u[1] > 0)).sum())))
    return out


def _reference(t, train, gates=None):
    """float64 restatement of the tail (tf.nn.moments-style batch statistics in training, running moments otherwise)
    and, by autograd, of its gradients for the loss sum(R * dR); gates: the kernel's ReLU decisions, which the
    backward then follows (a pre-activation within rounding of zero may fall either way)"""
    d = lambda x: x.detach().double().requires_grad_(True)
    P = {k: d(t[k]) for k in ('g1', 'b1', 'W2', 'c2', 'g2', 'b2', 'W3', 'c3')}
    Z1 = d(t['Z1'])
    save, pre = [], []

    def bn(z, g, b, m_run, v_run):
        if train:
            m = z.mean(0)
            v = ((z - m) ** 2).mean(0)
        else:
            m, v = m_run.double(), v_run.double()
        rs = 1.0 / torch.sqrt(v + EPS)
        save.extend([m.detach(), rs.detach()])
        u = (z - m) * rs * g + b
        h = torch.relu(u) if gates is None else u * gates[len(pre)][0]
        pre.append(u.detach())
        return h, m.detach(), v.detach()
    h1, m1, v1 = bn(Z1, P['g1'], P['b1'], t['mom'][0], t['mom'][1])
    Z2 = h1 @ P['W2'] + P['c2']
    h2, m2, v2 = bn(Z2, P['g2'], P['b2'], t['mom'][2], t['mom'][3])
    R = h2 @ P['W3'] + P['c3']
    (R * t['dR'].double()).sum().backward()
    grads = {k: P[k].grad for k in P}
    grads['dZ1'] = Z1.grad
    return dict(Z2=Z2.detach(), R=R.detach(), save=torch.cat(save), grads=grads, stats=(m1, v1, m2, v2), pre=pre)


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('W', [32, 64])
def test_tail_forward_and_backward_against_float64(W, B):
    """Training-mode forward, then backward on its outputs, against float64.

    Tolerances.  Every output is a chain of fp32 dot products of length <= W = 64 and of batch sums of <= 16384
    terms, the sums formed in blocks (per thread, per warp by shuffles, per CTA, then 8 CTAs in fp64 or rank
    order), so the rounding of a sum grows like u * (log2 B + rows per thread) with u = 2^-24 = 6e-8, about 1e-6
    relative to the largest term; the BN backward subtracts batch means of such sums from per-row terms, which
    amplifies it by the ratio of max |dz| to the typical |dz|, a few units here.  Relative to the largest entry of
    each tensor: 2e-5 for the forward values and statistics, 2e-4 for the gradients (an order above the estimate
    each).  The bf16 planes copy of dZ1 is its round-to-nearest.  A pre-activation within rounding of zero may be
    gated differently in fp32 and fp64, which would move the backward by O(1) in its row: the reference backward
    follows the kernel's gates (_kernel_gates), so the bounds hold without masking."""
    tails = _tails(W, B, seed=W + B)
    fwd = _fwd(tails, W, B, train=1)
    bwd = _bwd(tails, fwd, W, B)
    for t, f, g in zip(tails, fwd, bwd):
        gates = _kernel_gates(t, f, W)
        assert [n for _, n in gates] == [0, 0]
        ref = _reference(t, train=True, gates=gates)
        assert _rel(f['Z2'], ref['Z2']) < 2e-5 and _rel(f['R'], ref['R']) < 2e-5
        assert _rel(f['save'], ref['save']) < 2e-5
        m1, v1, m2, v2 = ref['stats']
        for got, old, new in zip(f['mom'], t['mom'], (m1, v1, m2, v2)):
            assert _rel(got, D * old.double() + (1 - D) * new) < 2e-5
        G = ref['grads']
        for k in ('g1', 'b1', 'W2', 'g2', 'b2', 'W3', 'c3', 'dZ1'):
            assert _rel(g[k], G[k]) < 2e-4, (k, _rel(g[k], G[k]))
        # biases in front of train-mode BatchNorm: zero gradient, rounding noise only
        scale = float(G['c3'].abs().max())
        assert float(g['c2'].abs().max()) < 1e-4 * scale and float(g['c1'].abs().max()) < 1e-4 * scale
        planes = g['dZ1p'][:, :B].permute(1, 0, 2).reshape(B, W)
        assert torch.equal(planes, g['dZ1'].to(torch.bfloat16))


@pytest.mark.parametrize('B', [128, 4097, 16384])
@pytest.mark.parametrize('W', [32, 64])
def test_tail_eval_forward_against_float64(W, B):
    """Eval mode (running moments): dot products only, tolerance 2e-5 as above; the moments are left unchanged."""
    tails = _tails(W, B, seed=7 * W + B)
    fwd = _fwd(tails, W, B, train=0)
    for t, f in zip(tails, fwd):
        ref = _reference(t, train=False)
        assert _rel(f['Z2'], ref['Z2']) < 2e-5 and _rel(f['R'], ref['R']) < 2e-5
        for got, old in zip(f['mom'], t['mom']):
            assert torch.equal(got, old)


@pytest.mark.parametrize('B', [128, 4097, 9000])
@pytest.mark.parametrize('W', [32, 64])
def test_counted_forward_equals_the_uncounted_call(W, B):
    tails = _tails(W, B, seed=3)
    for m in counts(B):
        ref = _fwd(tails, W, m, train=0) if m else None
        got = _fwd(tails, W, B, train=0, count=cnt_of(m))
        for i, g in enumerate(got):
            untouched(g['Z2'][m:], -1.0)
            untouched(g['R'][m:], -1.0)
            if m:
                same(g['Z2'][:m], ref[i]['Z2'][:m])
                same(g['R'][:m], ref[i]['R'][:m])
                same(g['save'], ref[i]['save'])


@pytest.mark.parametrize('B', [128, 4097, 16384])
@pytest.mark.parametrize('W', [32, 64])
def test_statistics_are_reproducible(W, B):
    """the batch statistics are combined in a fixed order (warp, CTA, cluster rank): two runs agree bit for bit"""
    tails = _tails(W, B, seed=11)
    runs = []
    for _ in range(2):
        fwd = _fwd(tails, W, B, train=1)
        runs.append((fwd, _bwd(tails, fwd, W, B)))
    (f0, b0), (f1, b1) = runs
    for a, b in zip(f0, f1):
        for k in ('Z2', 'R', 'save'):
            same(a[k], b[k])
        for x, y in zip(a['mom'], b['mom']):
            same(x, y)
    for a, b in zip(b0, b1):
        for k in ('g1', 'b1', 'g2', 'b2', 'dZ1'):
            same(a[k], b[k])


def test_unserved_width_is_refused_by_the_kernels():
    from lib._cabi import MpnnError
    tails = _tails(16, 128, seed=1)
    with pytest.raises(MpnnError, match='16, 32 or 64'):
        _fwd(tails, 24, 128, train=1)


# ---------------------------------------------------------------- end to end, with the nets of the existing tests
TINY = [('ac', dict(k_cpt=4e-9)), ('cr', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9))]
# test_parity_gpu's per-case bf16 gradient bound ('_bf16_grad'), raised for one (net, width) only.  In the actree net
# built with 32-wide routers, seven tensors exceed 0.15 in bf16, all of one subtree: the router of node 0/2 (w 0.289,
# beta 0.263) and the conv stage it feeds (0.19-0.21).  The same net in fp32 is within 1e-3, and the nets built from
# the same seed with 16- and 64-wide routers peak at 0.051 on the same kernels.  So this is test_parity_gpu's documented
# amplification: that router's gradient is a difference of its children's costs that nearly cancel for this draw of
# parameters.  It is not an error of the wide heads or dZ1 planes, which the 64-wide net runs too.
BF16_GRAD = {('actree', 32): 0.35}


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('W', [32, 64])
@pytest.mark.parametrize('kind,hy', TINY)
def test_training_step_matches_the_oracle(kind, hy, W, prec):
    """test_parity_gpu's forward / routing-decision / gradient check, at its bounds, with W-wide routers"""
    if (kind, W) in BF16_GRAD:
        hy = dict(hy, _bf16_grad=BF16_GRAD[kind, W])
    with router_widths(W):
        PG.test_forward_and_gradients(kind, hy, prec)


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('W', [32, 64])
def test_twenty_steps_stay_finite_and_reduce_the_loss(W, prec):
    with router_widths(W):
        net = tiny_net('ac', seed=4, k_cpt=4e-9)
    randomize_routers(net)
    net.configure(precision=prec)
    x0, y = batch(64, seed=5)
    eng = net._get_engine()
    losses = []
    for _ in range(20):
        net.train.run(PR._train_feed(net, dict(k_cpt=4e-9), x0, y))
        torch.cuda.synchronize()
        losses.append(eng.c_tot(eng._plan(64, True, True)))
    assert np.all(np.isfinite(losses)) and np.all(np.isfinite(eng.theta.cpu().numpy()))
    assert np.mean(losses[-3:]) < np.mean(losses[:3]), losses


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('kind,hy', [('ac', dict(k_cpt=4e-9)), ('actree', dict(k_cpt=2e-9)), ('ac', dict(dyn_k_cpt=True))])
def test_routed_inference_equals_the_dense_pass(kind, hy, prec):
    """net.predict against the dense 'ev' pass, and net.predictor against net.predict, bit for bit, at W = 32"""
    with router_widths(32):
        PD.test_predict_equals_the_dense_path(kind, hy, prec)
        PR.test_predictor_equals_predict(kind, hy, prec)


@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
@pytest.mark.parametrize('kind,hy', [('ac', dict(k_cpt=4e-9)), ('ac', dict(dyn_k_cpt=True))])
def test_compacted_statistics_equal_the_dense_ones(kind, hy, prec):
    with router_widths(32):
        CE.test_compact_evaluator_equals_the_dense_path(kind, hy, prec)


@pytest.mark.parametrize('W,prec', [(32, 'fp32'), (32, 'bf16'), (64, 'bf16')])
def test_full_architecture_with_wide_routers_matches_the_oracle(W, prec):
    """cifar10-ac with router_n_chan = W, B = 128, at the bounds of test_fullsize_parity_gpu.  In bf16 the head GEMM
    [W_leaf | W_r1] of the F = 2048 stages has N = 48 / 80 and runs as 3 / 5 slices of 16 columns over blockIdx.y."""
    with router_n_chan(W):
        FP.test_full_architecture_matches_the_oracle('cifar10-ac', prec)
