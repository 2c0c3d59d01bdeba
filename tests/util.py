"""Shared helpers for the test-suite: small nets, planes-layout emulation in
NumPy (the layout of csrc/common.cuh), comparison helpers."""
import copy

import numpy as np

from lib import layer_types as lt
from lib import serdes
from lib.layer_types import (ActivityError, BatchNorm, Chain, Conv, CrossEntropyError, Dropout, GlobalMaxPool, LinTrans,
                             MaxPool, MultiscaleBatchNorm, MultiscaleConvMax, MultiscaleLLN, MultiscaleRect, Rect, Select, Softmax,
                             SquaredError, SuperclassCrossEntropyError, ToPyramid)
from lib.net_types import ActorNet, CriticNet, SRNet

K_L2 = 1e-4


def _fc(n, s=1):
    return LinTrans(n_chan=n, k_l2=K_L2, σ_w=s)


def router(n_sinks):
    if n_sinks < 2:
        return None
    return Chain(name='Router', comps=[Select(i=-1), _fc(16), BatchNorm(), Rect(), _fc(16), BatchNorm(),
                                       Rect(), _fc(n_sinks, 0)])


_LLN = [False]          # local luminance normalisation behind ToPyramid (set by tiny_net for the '...lln' kinds)


def pyr(n_scales, *sinks):
    comps = [ToPyramid(n_scales=n_scales)] + ([MultiscaleLLN(σ=2)] if _LLN[0] else [])
    return Chain(name='ToPyramid', sinks=sinks, comps=comps)


def rcm(n_chan, *sinks):
    return Chain(name='ReConvMax', sinks=sinks, router=router(len(sinks)), comps=[
        MultiscaleConvMax(n_chan=list(n_chan), supp=3, k_l2=K_L2, σ_w=1), MultiscaleBatchNorm(), MultiscaleRect()])


N_SUP = 4


def superclasses(n_cls, n_sup=N_SUP):
    """class j belongs to superclass j mod n_sup"""
    return np.eye(n_sup, dtype=np.float32)[np.arange(n_cls) % n_sup]


_LEAF = ['ce']          # error layer of the classifiers built by reg(): 'ce' | 'sq' | 'sce' (set by tiny_net)


def reg(n_cls):
    if _LEAF[0] == 'sq':      # SquaredError on the LinTrans output (layer_types.py:255-260)
        return Chain(name='LinReg', comps=[Select(i=-1), _fc(n_cls), SquaredError()])
    if _LEAF[0] == 'sce':     # SuperclassCrossEntropyError (layer_types.py:274-285)
        return Chain(name='LogReg', comps=[Select(i=-1), _fc(N_SUP), Softmax(),
                                           SuperclassCrossEntropyError(w_cls=superclasses(n_cls))])
    return Chain(name='LogReg', comps=[Select(i=-1), _fc(n_cls), Softmax(), CrossEntropyError()])


def tiny_net(kind='ac', n_cls=10, x0_shape=(16, 16, 3), seed=0, **hypers):
    """16x16 input, 3-scale pyramid, stages [16,16,16] -> [16,16] -> [32];
    'sr' is a chain, 'ac'/'cr' route at both inner stages, 'tree' has a 3-way switch."""
    lt.seed(seed)
    _LEAF[0] = 'ce'
    for suffix in ('sq', 'sce'):          # 'srsq', 'acsce', ...: the same nets with another error layer on the leaves
        if kind.endswith(suffix) and kind not in ('sq', 'sce'):
            kind, _LEAF[0] = kind[:-len(suffix)], suffix
    if kind.endswith('lln'):              # 'srlln', 'aclln': MultiscaleLLN (layer_types.py:126-147) on every pyramid scale
        kind, _LLN[0] = kind[:-3], True
    try:
        return _tiny_net(kind, n_cls, x0_shape, **hypers)
    finally:
        _LEAF[0], _LLN[0] = 'ce', False


def _tiny_net(kind, n_cls, x0_shape, **hypers):
    if kind in ('cnvmp', 'cnvgmp', 'cnvact', 'cnvdrop'):
        # the plain-CNN layers of layer_types.py:86-100, 212-217, 287-293: Conv-BN-ReLU-MaxPool blocks (with the
        # identity-configured Dropout / ActivityError in the chain) and a GlobalMaxPool classifier
        blk = lambda n, *sinks, tail=(): Chain(name='ConvBlock', sinks=sinks, comps=[
            Conv(n_chan=n, supp=3, k_l2=K_L2, σ_w=1), BatchNorm(), Rect()] + list(tail))
        if kind == 'cnvmp':
            flat = Chain(name='LogReg', comps=[Dropout(), _fc(n_cls), Softmax(), CrossEntropyError()])
            root = blk(16, blk(32, flat, tail=[MaxPool(stride=2, supp=2)]), tail=[ActivityError(), MaxPool(stride=2, supp=2)])
        elif kind == 'cnvdrop':     # Dropout(keep < 1) behind the ReLU, in front of a MaxPool and in front of the classifier
            flat = Chain(name='LogReg', comps=[_fc(n_cls), Softmax(), CrossEntropyError()])
            root = blk(16, blk(32, flat, tail=[Dropout(λ=0.75)]), tail=[Dropout(λ=0.5), MaxPool(stride=2, supp=2)])
        elif kind == 'cnvact':      # an activity cost on both blocks, with and without a MaxPool behind it
            flat = Chain(name='LogReg', comps=[_fc(n_cls), Softmax(), CrossEntropyError()])
            root = blk(16, blk(32, flat, tail=[ActivityError(α=2e-3)]), tail=[ActivityError(α=1e-3), MaxPool(stride=2, supp=2)])
        else:
            gap = Chain(name='LogReg', comps=[GlobalMaxPool(), _fc(n_cls), Softmax(), CrossEntropyError()])
            root = blk(16, blk(32, gap), tail=[MaxPool(stride=2, supp=2)])
        return SRNet(x0_shape=x0_shape, y_shape=(n_cls,), root=root)
    if kind in ('cnv', 'cnvpyr'):
        # standalone Conv (layer_types.py:55-74) chains: on the image itself, or on one pyramid scale via Select
        cnv = lambda n, *sinks, pre=(): Chain(name='ConvBlock', sinks=sinks, comps=list(pre) + [
            Conv(n_chan=n, supp=3, k_l2=K_L2, σ_w=1), BatchNorm(), Rect()])
        flat = Chain(name='LogReg', comps=[_fc(n_cls), Softmax(), CrossEntropyError()])
        if kind == 'cnv':
            root = cnv(16, cnv(32, flat))
        else:
            root = pyr(2, cnv(16, cnv(16, flat), pre=[Select(i=1)]))
        return SRNet(x0_shape=x0_shape, y_shape=(n_cls,), root=root)
    if kind == 'sr':
        root = pyr(3, rcm([16, 16, 16], rcm([16, 16], rcm([32], reg(n_cls)))))
        return SRNet(x0_shape=x0_shape, y_shape=(n_cls,), root=root)
    cls = CriticNet if kind.startswith('cr') else ActorNet
    if kind.endswith('tree'):
        root = pyr(3, rcm([16, 16, 16], reg(n_cls),
                          rcm([16, 16], reg(n_cls), rcm([32], reg(n_cls))),
                          rcm([16, 16], reg(n_cls), rcm([32], reg(n_cls)))))
    else:
        root = pyr(3, rcm([16, 16, 16], reg(n_cls), rcm([16, 16], reg(n_cls), rcm([32], reg(n_cls)))))
    return cls(x0_shape=x0_shape, y_shape=(n_cls,), root=root, **hypers)


def dropout_mask(seed, draw, shape, keep):
    """numpy restatement of the device's Dropout mask (csrc/activity.cu): keep <=> mix(mix(i * 0x9E3779B9 + seed)
    ^ (draw * 0x85EBCA6B)) < keep * 2^32 over the NHWC element index i"""
    def mix(x):
        x = x.copy()
        x ^= x >> np.uint32(16); x *= np.uint32(0x7feb352d); x ^= x >> np.uint32(15)
        x *= np.uint32(0x846ca68b); x ^= x >> np.uint32(16)
        return x
    with np.errstate(over='ignore'):
        i = np.arange(int(np.prod(shape)), dtype=np.uint32)
        u = mix(mix(i * np.uint32(0x9E3779B9) + np.uint32(seed)) ^ np.uint32((draw * 0x85EBCA6B) & 0xFFFFFFFF))
    return (u.astype(np.uint64) < np.uint64(int(keep * 4294967296.0))).reshape(shape).astype(np.float32)


def _mul32(x, c):
    """x * c mod 2^32 for int64 tensors holding uint32 values, without int64 overflow"""
    return (x * (c & 0xFFFF) + (((x * (c >> 16)) & 0xFFFF) << 16)) & 0xFFFFFFFF


def _mix32(x):
    x = x ^ (x >> 16); x = _mul32(x, 0x7feb352d); x = x ^ (x >> 15); x = _mul32(x, 0x846ca68b)
    return x ^ (x >> 16)


def dropout_mask_t(seed, draw, shape, keep, device):
    """torch restatement of dropout_mask on any device (bool tensor of `shape`, NHWC element order)"""
    import torch
    n = 1
    for s in shape:
        n *= int(s)
    i = torch.arange(n, dtype=torch.int64, device=device)
    u = _mix32(_mix32((_mul32(i, 0x9E3779B9) + seed) & 0xFFFFFFFF) ^ ((draw * 0x85EBCA6B) & 0xFFFFFFFF))
    return (u < int(keep * 4294967296.0)).view(*shape)


def randomize_routers(net, seed=1, scale=0.5):
    """The reference zero-initialises the last router layer (all decisions tie
    to sink 0); give it weights so parity tests see non-trivial routing."""
    rng = np.random.default_rng(seed)
    for l in net.layers:
        if l.router is not None:
            last = l.router.comps[-1]
            last.params.w.assign((scale * rng.standard_normal(last.params.w.shape)).astype(np.float32))
            last.params.b.assign((0.1 * rng.standard_normal(last.params.b.shape)).astype(np.float32))
    return net


def batch(B, x0_shape=(16, 16, 3), n_cls=10, seed=0):
    rng = np.random.default_rng(seed)
    x0 = rng.random((B,) + tuple(x0_shape)).astype(np.float32)
    y = np.eye(n_cls, dtype=np.float32)[rng.integers(0, n_cls, B)]
    return x0, y


def record_of(net):
    return copy.deepcopy(serdes.encode_net(net))


def node_paths(net):
    """preorder list of (path, layer) matching oracle path naming."""
    out = []

    def walk(l, path):
        out.append((path, l))
        for i, s in enumerate(l.sinks):
            walk(s, (path + '/' if path else '') + str(i))
    walk(net.root, '')
    return out


def rel_err(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    d = np.linalg.norm(a - b)
    n = np.linalg.norm(b)
    return d / n if n > 0 else d


# ---- planes layout emulation ------------------------------------------------ #
class Geo:
    def __init__(self, B, H, W):
        self.B, self.H, self.W = B, H, W
        self.Wp = W + 1
        self.S = (H + 1) * (W + 1)
        self.rows = B * self.S
        self.G = max(64, (W + 2 + 7) // 8 * 8)
        self.P = (self.G + self.rows + 128 + self.G + 7) // 8 * 8


def to_planes(x, geo, Cpad=None, dtype=np.float32):
    """NHWC -> [Cpad/8][P][8] with zero pads/guards."""
    B, H, W, C = x.shape
    Cpad = C if Cpad is None else Cpad
    t = np.zeros((Cpad // 8, geo.P, 8), dtype)
    xp = np.zeros((B, H, W, Cpad), dtype)
    xp[..., :C] = x
    rows = (geo.G + np.arange(B)[:, None, None] * geo.S + (np.arange(H)[None, :, None] + 1) * geo.Wp
            + (np.arange(W)[None, None, :] + 1))
    for kg in range(Cpad // 8):
        t[kg, rows.reshape(-1)] = xp[..., kg * 8:(kg + 1) * 8].reshape(-1, 8)
    return t


def from_planes(t, geo, C):
    B, H, W = geo.B, geo.H, geo.W
    rows = (geo.G + np.arange(B)[:, None, None] * geo.S + (np.arange(H)[None, :, None] + 1) * geo.Wp
            + (np.arange(W)[None, None, :] + 1)).reshape(-1)
    out = np.concatenate([t[kg, rows] for kg in range(t.shape[0])], 1)
    return out.reshape(B, H, W, -1)[..., :C]


def _planes_view(t, geo):
    """[KG][P][8] -> view [KG][B][H+1][W+1][8] of the image blocks (row G + n*S + r*Wp + c is [n][r][c]);
    the valid pixel (h, w) is [h+1][w+1], row 0 and column 0 of a block are its zero pads."""
    return t[:, geo.G:geo.G + geo.rows].view(t.shape[0], geo.B, geo.H + 1, geo.W + 1, 8)


def to_planes_t(x, geo, Cpad=None):
    """torch version of to_planes on x's device and dtype: NHWC -> [Cpad/8][P][8] with zero pads / guards"""
    B, H, W, C = x.shape
    Cpad = C if Cpad is None else Cpad
    t = x.new_zeros((Cpad // 8, geo.P, 8))
    v = _planes_view(t, geo)[:, :, 1:, 1:, :]
    for kg in range(Cpad // 8):          # one plane at a time: no NHWC-sized temporary
        c = min(8, max(C - kg * 8, 0))
        if c:
            v[kg, ..., :c] = x[..., kg * 8:kg * 8 + c]
    return t


def from_planes_t(t, geo, C):
    """torch version of from_planes: [KG][P][8] -> NHWC (first C channels), a new tensor"""
    v = _planes_view(t, geo)[:, :, 1:, 1:, :]
    return v.permute(1, 2, 3, 0, 4).reshape(geo.B, geo.H, geo.W, -1)[..., :C].contiguous()


def to_feat_t(x, Balloc):
    """(B, F) -> the flattened-feature layout [F/8][Balloc][8] of the heads, rows >= B zero"""
    B, F = x.shape
    t = x.new_zeros((F // 8, Balloc, 8))
    t[:, :B] = x.view(B, F // 8, 8).permute(1, 0, 2)
    return t


def from_feat_t(t, B):
    """[F/8][Balloc][8] -> (B, F)"""
    return t[:, :B].permute(1, 0, 2).reshape(B, -1)


def stencil_offsets(Wp):
    return [(t // 3 - 1) * Wp + (t % 3 - 1) for t in range(9)]


# ---- routing tree tables (include/mpnn.h, "Tree tables") and a float64 restatement of both walks ---------- #
RT_MAXS = 8             # sinks per switch (csrc/route.cu)


def random_tree(rng, n_nodes, max_sinks):
    """Random tables for mpnn_route_fwd / _bwd: n_nodes nodes in preorder, a mix of leaves, 1-sink chain nodes and
    switches of 2 .. max_sinks sinks, at least one switch of exactly max_sinks sinks (the root).  Every leaf is a
    classifier (err = its leaf slot), switches get slots in preorder, ops are positive, and
    floor = n_leaves(i) / n_leaves(root) as the engine writes it.  NumPy arrays, keyed by the C argument names."""
    assert 2 <= max_sinks <= RT_MAXS and n_nodes > max_sinks
    kids = [[]]
    open_, left = [0], n_nodes - 1
    while left:
        v = open_.pop(len(open_) - 1 - int(rng.integers(min(3, len(open_)))))     # mostly the newest: deep trees
        if v == 0:
            ns = max_sinks
        else:
            r = rng.random()
            ns = 0 if r < 0.3 else 1 if r < 0.55 else int(rng.integers(2, max_sinks + 1))
            ns = min(ns, left)
            if ns == 0 and not open_:           # the last open node must not close the tree early
                ns = 1
        for _ in range(ns):
            kids.append([])
            kids[v].append(len(kids) - 1)
            open_.append(len(kids) - 1)
        left -= ns
    order = []                                   # preorder relabelling

    def walk(v):
        order.append(v)
        for c in kids[v]:
            walk(c)
    walk(0)
    new = {v: i for i, v in enumerate(order)}
    n = n_nodes
    t = dict(parent=np.full(n, -1, np.int32), sink_idx=np.zeros(n, np.int32), n_sinks=np.zeros(n, np.int32),
             child=np.full((n, RT_MAXS), -1, np.int32), floor=np.zeros(n, np.float32), sw=np.full(n, -1, np.int32),
             ops=np.zeros(n, np.float32), err=np.full(n, -1, np.int32))
    for v in order:
        i = new[v]
        t['n_sinks'][i] = len(kids[v])
        for j, c in enumerate(kids[v]):
            t['parent'][new[c]], t['sink_idx'][new[c]], t['child'][i, j] = i, j, new[c]
    n_sw = n_err = 0
    for i in range(n):
        if t['n_sinks'][i] >= 2:
            t['sw'][i], n_sw = n_sw, n_sw + 1
        if t['n_sinks'][i] == 0:
            t['err'][i], n_err = n_err, n_err + 1
    leaves = np.zeros(n, np.int64)
    for i in reversed(range(n)):
        leaves[i] = 1 if t['n_sinks'][i] == 0 else sum(leaves[c] for c in t['child'][i, :t['n_sinks'][i]])
    t['floor'][:] = leaves / leaves[0]
    t['ops'][:] = rng.uniform(1e6, 3e8, n).astype(np.float32)
    return t


def tree_tables(plan):
    """the routing tables of an engine plan (lib/engine.py _build_routing) as NumPy arrays, keyed as random_tree's"""
    return {k: getattr(plan, 't_' + a).cpu().numpy() for k, a in (
        ('parent', 'parent'), ('sink_idx', 'sink'), ('n_sinks', 'nsinks'), ('child', 'child'), ('floor', 'floor'),
        ('sw', 'sw'), ('ops', 'ops'), ('err', 'err'))}


def pad_tree(t, n_total):
    """t with a chain of 1-sink nodes hung below its last node in preorder (a leaf) up to n_total nodes: ops 0,
    err -1, so the padding changes no original node's p_tr, p_ev, c_ev or c_opt, and adds exact zeros to c_data.
    The former last node keeps its err slot."""
    n = len(t['parent'])
    assert t['n_sinks'][n - 1] == 0 and n_total > n
    p = {k: v.copy() for k, v in t.items()}
    extra = n_total - n
    for k in ('parent', 'sink_idx', 'n_sinks', 'floor', 'sw', 'ops', 'err'):
        fill = {'parent': 0, 'sink_idx': 0, 'n_sinks': 1, 'floor': t['floor'][n - 1], 'sw': -1, 'ops': 0, 'err': -1}[k]
        p[k] = np.concatenate([p[k], np.full(extra, fill, p[k].dtype)])
    p['child'] = np.concatenate([p['child'], np.full((extra, RT_MAXS), -1, np.int32)])
    for i in range(n - 1, n_total):
        if i > n - 1:
            p['parent'][i] = i - 1
        if i < n_total - 1:
            p['n_sinks'][i], p['child'][i, 0] = 1, i + 1
    p['n_sinks'][n_total - 1] = 0
    return p


def _f32(v):
    return float(np.float32(v))


def route_ref(t, R, tau, eps, c_err=None, d_cor=None, k_cpt=0.0, critic=False, k_dec=0.0, k_cre=0.0,
              optimistic=False, use_cls_err=False):
    """Both routing walks of csrc/route.cu (lib/net_types.py:108-131 actor, :193-243 critic) in float64 torch, from
    the tables alone, on the device of R.  R[slot]: [B][n_sinks] logits of each switch slot; c_err[leaf], d_cor[leaf]:
    [B]; k_cpt: a number or a [B] vector.  The scalars are rounded to fp32 first, as the kernels receive them.
      p_tr[i] = (p_tr[par] - eps floor[par]) softmax(R / tau)[sink_idx[i]] + eps floor[i]   below a switch,
      p_ev[i] = p_ev[par] [first argmax R == sink_idx[i]],   dec[slot] = first argmax R.
    Actor: c_data = sum_i p_tr (c_err + k_cpt ops) + sum_switches sg(p_tr) k_dec |R|^2, dR = d mean_b(c_data) / dR by
    autograd; 'g' is the explicit dL/dp_tr of every node (the `gp` of the kernels), for error bounds.
    Critic: c_ev / c_opt bottom-up (ce = 1 - d_cor with use_cls_err), dR = p_tr / B k_cre 2 (R + target) with
    target = c_opt (optimistic) or c_ev of each sink, c_data = sum_i p_tr (c_err + k_cre sum_j (R_j + target_j)^2).
    Returns a dict of p_tr, p_ev [n][B], dec [n_sw][B] (int64), c_data [B], dR [slot] and the intermediates."""
    from oracle.torch_ref import first_argmax
    import torch
    L = {k: (v.tolist() if hasattr(v, 'tolist') else list(v)) for k, v in t.items()}
    n = len(L['parent'])
    dev = R[0].device if len(R) else (c_err[0].device if c_err else 'cpu')
    B = R[0].shape[0] if len(R) else c_err[0].shape[0]
    dt = torch.float64
    tau, eps, k_dec, k_cre = _f32(tau), _f32(eps), _f32(k_dec), _f32(k_cre)
    fl = [eps * _f32(f) for f in L['floor']]
    ops = [_f32(o) for o in L['ops']]
    kc = k_cpt.double() if hasattr(k_cpt, 'double') else _f32(k_cpt)
    Rt = [r.detach().double().requires_grad_(not critic) for r in R]
    sm = [torch.softmax(r / tau, 1) for r in Rt]
    dec = [first_argmax(r.detach(), 1) for r in Rt]
    one = torch.ones(B, dtype=dt, device=dev)
    zero = torch.zeros(B, dtype=dt, device=dev)
    p_tr, p_ev = [one] + [None] * (n - 1), [one] + [None] * (n - 1)
    for i in range(1, n):
        par = L['parent'][i]
        if L['n_sinks'][par] >= 2:
            s, si = L['sw'][par], L['sink_idx'][i]
            p_tr[i] = (p_tr[par] - fl[par]) * sm[s][:, si] + fl[i]
            p_ev[i] = p_ev[par] * (dec[s] == si).to(dt)
        else:
            p_tr[i], p_ev[i] = p_tr[par], p_ev[par]
    ce = [c_err[L['err'][i]].double() if L['err'][i] >= 0 else zero for i in range(n)]
    out = dict(sm=[s.detach() for s in sm], dec=torch.stack(dec) if dec else None)
    if not critic:
        local = [ce[i] + kc * ops[i] for i in range(n)]
        tot = sum(p_tr[i] * local[i] for i in range(n))
        for i in range(n):
            if L['n_sinks'][i] >= 2:
                tot = tot + p_tr[i].detach() * k_dec * (Rt[L['sw'][i]] ** 2).sum(1)
        if Rt:
            (tot.sum() / B).backward()
        with torch.no_grad():
            g = [(local[i] / B).detach().clone() for i in range(n)]
            for i in range(n - 1, 0, -1):
                par = L['parent'][i]
                w = sm[L['sw'][par]][:, L['sink_idx'][i]].detach() if L['n_sinks'][par] >= 2 else 1.0
                g[par] = g[par] + g[i] * w
        out.update(dR=[r.grad for r in Rt], g=torch.stack(g), c_data=tot.detach())
    else:
        ce_loss = [(1.0 - d_cor[L['err'][i]].double()) if L['err'][i] >= 0 else zero for i in range(n)] \
            if use_cls_err else ce
        cev, cop, dR, tgt = [None] * n, [None] * n, [None] * len(R), [None] * len(R)
        tot = zero
        for i in range(n - 1, -1, -1):
            base = ce_loss[i] + kc * ops[i]
            ks = L['child'][i][:L['n_sinks'][i]]
            cre = zero
            if len(ks) < 2:
                cev[i] = base + sum((cev[c] for c in ks), zero)
                cop[i] = base + sum((cop[c] for c in ks), zero)
            else:
                s = L['sw'][i]
                tg = torch.stack([(cop if optimistic else cev)[c] for c in ks], 1)
                r = Rt[s]
                dR[s] = p_tr[i][:, None] / B * k_cre * 2 * (r + tg)
                tgt[s] = tg
                cre = k_cre * ((r + tg) ** 2).sum(1)
                cev[i] = base + torch.stack([cev[c] for c in ks], 1).gather(1, dec[s][:, None])[:, 0]
                cop[i] = base + torch.stack([cop[c] for c in ks], 1).min(1).values
            tot = tot + p_tr[i] * (ce[i] + cre)
        out.update(dR=dR, tgt=tgt, c_ev=torch.stack(cev), c_opt=torch.stack(cop), c_data=tot)
    out.update(p_tr=torch.stack([p.detach() for p in p_tr]), p_ev=torch.stack(p_ev))
    return out
