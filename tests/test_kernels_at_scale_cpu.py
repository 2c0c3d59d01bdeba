"""The torch helpers of tests/util.py (used on the device by test_kernels_at_scale_gpu.py) against independent
restatements: the NumPy planes emulation and the flattened-feature layout on small ragged shapes, the random
routing trees and the float64 routing reference against a per-example recursion; and the routing tables of the
full-size trees.  Runs without a GPU."""
import math

import numpy as np
import pytest
import torch

from util import (RT_MAXS, Geo, dropout_mask, dropout_mask_t, from_feat_t, from_planes, from_planes_t, pad_tree,
                  random_tree, route_ref, to_feat_t, to_planes, to_planes_t, tree_tables)


@pytest.mark.parametrize('seed,draw,keep', [(0, 0, 0.5), (12345, 7, 0.75), (0xFFFFFFFF, 0xDEADBEEF, 0.1)])
def test_torch_dropout_mask_equals_the_numpy_restatement(seed, draw, keep):
    shape = (3, 5, 7, 16)
    ref = dropout_mask(seed, draw, shape, keep)
    got = dropout_mask_t(seed, draw, shape, keep, 'cpu')
    np.testing.assert_array_equal(got.numpy().astype(np.float32), ref)
    assert 0 < ref.mean() < 1


@pytest.mark.parametrize('B,H,W,C,Cpad', [(1, 4, 4, 8, None), (3, 8, 8, 3, 16), (5, 4, 6, 24, None), (2, 32, 32, 16, 32),
                                          (7, 2, 2, 13, 16)])
def test_planes_helpers_equal_the_numpy_layout(B, H, W, C, Cpad):
    rng = np.random.default_rng(B * 100 + H)
    x = rng.standard_normal((B, H, W, C)).astype(np.float32)
    geo = Geo(B, H, W)
    ref = to_planes(x, geo, Cpad)
    got = to_planes_t(torch.from_numpy(x), geo, Cpad)
    assert got.dtype == torch.float32 and tuple(got.shape) == ref.shape
    np.testing.assert_array_equal(got.numpy(), ref)
    np.testing.assert_array_equal(from_planes_t(got, geo, C).numpy(), from_planes(ref, geo, C))
    np.testing.assert_array_equal(from_planes_t(got, geo, C).numpy(), x)
    # dtype follows the input, and a bf16 round trip is the identity on bf16 values
    xb = torch.from_numpy(x).to(torch.bfloat16)
    tb = to_planes_t(xb, geo, Cpad)
    assert tb.dtype == torch.bfloat16
    assert torch.equal(from_planes_t(tb, geo, C), xb)


@pytest.mark.parametrize('B,F,Balloc', [(1, 8, 8), (5, 256, 8), (37, 64, 128), (129, 40, 256)])
def test_feature_helpers_equal_the_loop_layout(B, F, Balloc):
    rng = np.random.default_rng(F + B)
    x = rng.standard_normal((B, F)).astype(np.float32)
    ref = np.zeros((F // 8, Balloc, 8), np.float32)
    for i in range(F // 8):                       # the layout as test_kernels_gpu.py builds it
        ref[i, :B] = x[:, i * 8:(i + 1) * 8]
    got = to_feat_t(torch.from_numpy(x), Balloc)
    np.testing.assert_array_equal(got.numpy(), ref)
    np.testing.assert_array_equal(from_feat_t(got, B).numpy(), np.concatenate([ref[i, :B] for i in range(F // 8)], 1))


# --------------------------------------------------------------------------- #
# routing trees and the float64 routing reference
# --------------------------------------------------------------------------- #
def check_tables(t, leaf_slots=True):
    """the invariants of include/mpnn.h "Tree tables": preorder (every subtree a contiguous range starting at its
    root, children in sink order), parent before child, sinks numbered 0 .. n_sinks-1, child consistent with
    parent, switch slots (and with leaf_slots, classifier slots of the leaves) numbered in preorder,
    floor = n_leaves(i) / n_leaves(root).  Returns n_leaves per node."""
    n = len(t['parent'])
    assert t['parent'][0] == -1 and all(0 <= t['parent'][i] < i for i in range(1, n))
    leaves, size = np.zeros(n, np.int64), np.ones(n, np.int64)
    for i in reversed(range(n)):
        ns = int(t['n_sinks'][i])
        kids = [c for c in range(n) if t['parent'][c] == i]
        assert 0 <= ns <= RT_MAXS and len(kids) == ns
        assert list(t['child'][i, :ns]) == kids and all(t['child'][i, ns:] == -1)
        assert [t['sink_idx'][c] for c in kids] == list(range(ns))
        at = i + 1
        for c in kids:                           # preorder
            assert c == at
            at += size[c]
        size[i] = at - i
        leaves[i] = 1 if ns == 0 else leaves[kids].sum()
    assert size[0] == n
    sw = [i for i in range(n) if t['n_sinks'][i] >= 2]
    assert list(t['sw'][sw]) == list(range(len(sw))) and all(t['sw'][i] == -1 for i in range(n) if i not in sw)
    if leaf_slots:
        lv = [i for i in range(n) if t['n_sinks'][i] == 0]
        assert list(t['err'][lv]) == list(range(len(lv)))
        assert all(t['err'][i] == -1 for i in range(n) if i not in lv)
    np.testing.assert_array_equal(t['floor'], (leaves / leaves[0]).astype(np.float32))
    return leaves


@pytest.mark.parametrize('n_nodes', [11, 32, 33, 60])
@pytest.mark.parametrize('max_sinks', [2, 4, 8])
def test_random_tree_invariants(n_nodes, max_sinks):
    rng = np.random.default_rng(100 * n_nodes + max_sinks)
    kinds = set()
    for _ in range(4):
        t = random_tree(rng, n_nodes, max_sinks)
        check_tables(t)
        assert len(t['parent']) == n_nodes and int(t['n_sinks'].max()) == max_sinks
        assert all(t['ops'] > 0) and all(t['err'][t['n_sinks'] == 0] >= 0)
        kinds |= {min(int(k), 2) for k in t['n_sinks']}
        p = pad_tree(t, 40 if n_nodes < 40 else n_nodes + 3)
        leaves = check_tables(p, leaf_slots=False)
        n = n_nodes
        for k in t:                             # the original nodes keep their tables, except the former last leaf
            np.testing.assert_array_equal(p[k][:n - 1], t[k][:n - 1])
        assert p['err'][n - 1] == t['err'][n - 1] and p['n_sinks'][n - 1] == 1
        assert all(p['ops'][n:] == 0) and all(p['err'][n:] == -1) and leaves[0] == (t['n_sinks'] == 0).sum()
    assert kinds == {0, 1, 2} or n_nodes < 32    # leaves, chain nodes and switches


def _walk_naive(t, R, tau, eps, ce, dc, kc, b, critic, k_dec, k_cre, optimistic, use_cls_err, R_frozen=None):
    """one example, by recursion over the tree in Python floats: (p_tr, p_ev, dec, c_data, dR, c_ev)"""
    n = len(t['parent'])
    f = lambda v: float(np.float32(v))
    tau, eps, k_dec, k_cre = f(tau), f(eps), f(k_dec), f(k_cre)
    fl = [eps * f(x) for x in t['floor']]
    kids = lambda i: [int(c) for c in t['child'][i, :t['n_sinks'][i]]]
    p_tr, p_ev, dec, dR = [0.0] * n, [0.0] * n, {}, {}

    def soft(i, Rsrc):
        r = [float(v) for v in Rsrc[int(t['sw'][i])][b]]
        m = max(x / tau for x in r)
        e = [math.exp(x / tau - m) for x in r]
        return r, [v / sum(e) for v in e], next(j for j, x in enumerate(r) if x == max(r))

    def down(i, pt, pe):
        p_tr[i], p_ev[i] = pt, pe
        ks = kids(i)
        if len(ks) >= 2:
            r, sm, d = soft(i, R)
            dec[int(t['sw'][i])] = d
            for j, c in enumerate(ks):
                down(c, (pt - fl[i]) * sm[j] + fl[c], pe * (1.0 if d == j else 0.0))
        else:
            for c in ks:
                down(c, pt, pe)
    down(0, 1.0, 1.0)
    cerr = lambda i: float(ce[int(t['err'][i])][b]) if t['err'][i] >= 0 else 0.0
    if not critic:
        pf = p_tr if R_frozen is None else _walk_naive(t, R_frozen, tau, eps, ce, dc, kc, b, 0, 0, 0, 0, 0)[0]
        tot = sum(p_tr[i] * (cerr(i) + kc * f(t['ops'][i])) for i in range(n))
        for i in range(n):
            if t['n_sinks'][i] >= 2:
                tot += pf[i] * k_dec * sum(float(v) ** 2 for v in R[int(t['sw'][i])][b])
        return p_tr, p_ev, dec, tot, None, None
    tot = 0.0

    def up(i):
        nonlocal tot
        loss = (1.0 - float(dc[int(t['err'][i])][b]) if t['err'][i] >= 0 else 0.0) if use_cls_err else cerr(i)
        base = loss + kc * f(t['ops'][i])
        ks = kids(i)
        res = [up(c) for c in ks]
        cre = 0.0
        if len(ks) < 2:
            ev, op = base + sum(e for e, _ in res), base + sum(o for _, o in res)
        else:
            r, _, d = soft(i, R)
            tg = [o if optimistic else e for e, o in res]
            dR[int(t['sw'][i])] = [p_tr[i] / len(R[0]) * k_cre * 2 * (r[j] + tg[j]) for j in range(len(ks))]
            cre = k_cre * sum((r[j] + tg[j]) ** 2 for j in range(len(ks)))
            ev, op = base + res[d][0], base + min(o for _, o in res)
        tot += p_tr[i] * (cerr(i) + cre)
        return ev, op
    c_ev = up(0)[0]
    return p_tr, p_ev, dec, tot, dR, c_ev


@pytest.mark.parametrize('mode', ['actor', 'actor k_cpt vector', 'critic', 'critic optimistic', 'critic use_cls_err'])
@pytest.mark.parametrize('n_nodes,max_sinks,eps', [(7, 2, 1e-6), (12, 3, 0.1), (16, 8, 0.1)])
def test_route_ref_matches_a_recursion(mode, n_nodes, max_sinks, eps):
    """route_ref (vectorised over the batch, actor gradient by autograd) against a per-example recursion over the
    tree in Python floats, with the actor's dR by central differences of the mean cost (h = 1e-5 on the logits:
    truncation ~ h^2, so 1e-6 relative)"""
    rng = np.random.default_rng(n_nodes)
    t = random_tree(rng, n_nodes, max_sinks)
    B, tau = 5, 0.7
    n_sw, n_err = int((t['n_sinks'] >= 2).sum()), int((t['n_sinks'] == 0).sum())
    R = [torch.from_numpy(rng.standard_normal((B, int(t['n_sinks'][i]))).astype(np.float32))
         for i in range(n_nodes) if t['n_sinks'][i] >= 2]
    R[0][0] = 1.0                                    # a tie: the first maximum decides
    ce = [torch.from_numpy((rng.random(B) * 3).astype(np.float32)) for _ in range(n_err)]
    dc = [torch.from_numpy((rng.random(B) < 0.5).astype(np.float32)) for _ in range(n_err)]
    critic = mode.startswith('critic')
    kv = 'vector' in mode
    kc = torch.from_numpy((rng.random(B) * 1e-8).astype(np.float32)) if kv else 4e-9
    hy = dict(critic=critic, k_dec=0.0 if critic else 0.01, k_cre=1e-3 if critic else 0.0,
              optimistic='optimistic' in mode, use_cls_err='cls' in mode)
    ref = route_ref(t, R, tau, eps, c_err=ce, d_cor=dc, k_cpt=kc, **hy)
    assert len(ref['dR']) == n_sw and ref['dec'].shape == (n_sw, B)
    args = lambda b: (t, [r.numpy() for r in R], tau, eps, [c.numpy() for c in ce], [d.numpy() for d in dc],
                      float(kc[b]) if kv else float(np.float32(kc)), b, critic, hy['k_dec'], hy['k_cre'],
                      hy['optimistic'], hy['use_cls_err'])
    for b in range(B):
        p_tr, p_ev, dec, tot, dR, c_ev = _walk_naive(*args(b))
        np.testing.assert_allclose(ref['p_tr'][:, b].numpy(), p_tr, rtol=1e-12)
        np.testing.assert_array_equal(ref['p_ev'][:, b].numpy(), p_ev)
        assert [int(ref['dec'][s, b]) for s in range(n_sw)] == [dec[s] for s in range(n_sw)]
        assert math.isclose(float(ref['c_data'][b]), tot, rel_tol=1e-12)
        if critic:
            assert math.isclose(float(ref['c_ev'][0, b]), c_ev, rel_tol=1e-12)
            for s in range(n_sw):
                np.testing.assert_allclose(ref['dR'][s][b].numpy(), dR[s], rtol=1e-12)
    if not critic:                                   # d mean_b c_data / dR with sg(p_tr) in the k_dec term
        h = 1e-5
        Rn = [r.numpy().astype(np.float64) for r in R]
        for s in range(n_sw):
            fd = np.zeros(Rn[s].shape)
            for b in range(B):
                for j in range(Rn[s].shape[1]):
                    val = []
                    for sgn in (1, -1):
                        Rp = [r.copy() for r in Rn]
                        Rp[s][b, j] += sgn * h
                        a = list(args(b)); a[1] = Rp
                        val.append(_walk_naive(*a, R_frozen=Rn)[3])
                    fd[b, j] = (val[0] - val[1]) / (2 * h) / B
            np.testing.assert_allclose(ref['dR'][s].numpy(), fd, rtol=1e-6, atol=1e-9 * np.abs(fd).max())
        # the explicit dL/dp_tr of the reference gives the same gradient as autograd
        g = ref['g']
        for i in range(n_nodes):
            if t['n_sinks'][i] >= 2:
                s, sm = int(t['sw'][i]), ref['sm'][int(t['sw'][i])]
                ks = t['child'][i, :t['n_sinks'][i]]
                gs = g[ks].T * (ref['p_tr'][i] - float(np.float32(eps)) * float(t['floor'][i]))[:, None]
                dot = (sm * gs).sum(1, keepdim=True)
                r = R[s].double()
                exp = sm * (gs - dot) / float(np.float32(tau)) + ref['p_tr'][i][:, None] * float(np.float32(0.01)) * 2 * r / B
                np.testing.assert_allclose(ref['dR'][s].numpy(), exp.numpy(), rtol=1e-10, atol=1e-15)


@pytest.mark.parametrize('name', ['ac_tree', 'cr_tree', 'ac_chain'])
def test_full_size_routing_tables(name):
    """The tables a dry-run plan of the full-size nets hands to mpnn_route_fwd / _bwd (lib/engine.py
    _build_routing): valid, and for both trees more than RT_STAGED_MAX = 32 nodes, so the at-scale GPU cases on
    these tables run the global-memory walk of csrc/route.cu (ac_chain, 17 nodes, runs the staged walk)."""
    import arch_and_hypers as ah
    from lib import engine as E
    net = getattr(ah, name)(k_cpt=4e-9)((32, 32, 3), (10,))
    plan = E.Engine(net, precision='fp32', impl=0, dry_run=True)._plan(128, True, True)
    t = tree_tables(plan)
    check_tables(t)
    n = len(t['parent'])
    if name == 'ac_chain':
        assert n == 17 and n <= 32
    else:
        assert n == 95 > 32 and int((t['n_sinks'] >= 2).sum()) == 39 and int(t['n_sinks'].max()) == 3
