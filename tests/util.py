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
