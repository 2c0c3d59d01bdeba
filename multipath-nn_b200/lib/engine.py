"""Execution engine: compiles a linked net (lib.net_types) into a static plan
of libmpnn_sm100 kernel launches over preallocated "padded planes" buffers and
runs forward / backward / TALR+momentum on one B200.  PyTorch supplies device
memory, streams, CUDA graphs and torch.distributed -- no arithmetic.

What the reference expresses as a TF graph + autodiff
(/root/reference/scripts/lib/net_types.py:137-181, 245-284) is laid out here
explicitly:  forward in preorder over the sink tree, routing walk, backward in
reverse preorder, one fused optimiser kernel over the flat parameter buffer.
Every node is evaluated densely on the whole batch, exactly like the
reference (SURVEY F2).
"""
import contextlib
import ctypes
import gc
import os
from types import SimpleNamespace as Ns

import numpy as np
import torch

from lib import _cabi
from lib.layer_types import (ActivityError, BatchNorm, Chain, Conv, CrossEntropyError, Dropout, GlobalMaxPool,
                             LinTrans, MaxPool, MultiscaleBatchNorm, MultiscaleConvMax, MultiscaleLLN,
                             MultiscaleRect, Param, Rect, Select, Softmax, SquaredError,
                             SuperclassCrossEntropyError, ToPyramid)
from lib.net_types import n_leaves

F32, BF16 = 0, 1
HYP_LR, HYP_MU, HYP_TAU, HYP_EPS, HYP_KCPT, HYP_GSCALE, HYP_DRAW, HYP_COUNT = 0, 1, 2, 3, 4, 5, 6, 8
MAXS = 8


def _struct(ptrs, ints):
    """numpy dtype mirroring a C struct of pointers followed by ints (include/mpnn.h)"""
    return np.dtype([(k, '<u8') for k in ptrs] + [(k, '<i4') for k in ints], align=True)


_PACK = _struct(['w', 'packed'], ['ntaps', 'I', 'O', 'mode', 'k_off', 'Ktot', 'n_off', 'Ntot'])
_RT_FWD = _struct(['Z1', 'g1', 'b1', 'm1', 'v1', 'W2', 'bias2', 'g2', 'b2', 'm2', 'v2', 'W3', 'bias3',
                   'Z2', 'R', 'save'], ['ns', 'reserved'])
_RT_BWD = _struct(['Z1', 'Z2', 'dR', 'g1', 'b1', 'W2', 'g2', 'b2', 'W3', 'save', 'dg1', 'dbt1', 'dW2',
                   'dbias2', 'dg2', 'dbt2', 'dW3', 'dbias3', 'dZ1', 'scratch', 'dZ1p', 'dbias1'],
                  ['ns', 'Balloc'])
_BN_FUSE = np.dtype([(k, '<u8') for k in ('acc', 'gamma', 'beta', 'm_avg', 'v_avg', 'ss', 'mr')]
                    + [('count', '<f8'), ('d', '<f4'), ('eps', '<f4'), ('defer', '<i4'), ('reserved', '<i4')], align=True)
_BN_BWD_FUSE = _struct(['acc', 'sums', 'dgamma', 'dbeta'], [])
_BN_BWD_EPI = _struct(['lin', 'ss', 'mr', 'acc', 'sums', 'dgamma', 'dbeta'], [])
assert _PACK.itemsize == 48 and _RT_FWD.itemsize == 136 and _RT_BWD.itemsize == 184
# mpnn_p2p_desc (include/mpnn.h): the exchange buffers of all ranks as mapped into this process
_P2P_MAX, _P2P_FLAG_BYTES, _P2P_HANDLE_BYTES = 16, 4096, 64
_BN_SMALL_MAX_PIXELS = 8192            # MPNN_BN_SMALL_MAX_PIXELS (include/mpnn.h)
_P2P = np.dtype([('base', '<u8', (_P2P_MAX,)), ('world', '<i4'), ('rank', '<i4'), ('off_grad', '<i8'),
                 ('off_theta', '<i8'), ('off_accum', '<i8'), ('g0', '<i4'), ('n', '<i4')], align=True)
assert _P2P.itemsize == 168


ROUTER_WIDTHS = (16, 32, 64)


def _router_width(nodes):
    """Hidden width W of the net's routers, Chain([Select(-1), LinTrans(W), BatchNorm, Rect, LinTrans(W), BatchNorm,
    Rect, LinTrans(n_sinks)]) (arch_and_hypers.router_n_chan).  Both hidden layers and every router of a net have the
    same W, because the tails of all routers run as one launch of one width; 16 when the net has no router."""
    widths = {}
    for nd in nodes:
        if nd.router is None:
            continue
        c = nd.router.comps
        w = (c[1].hypers.n_chan, c[4].hypers.n_chan)
        if w[0] != w[1] or w[0] not in ROUTER_WIDTHS:
            raise NotImplementedError('engine: router %r has hidden widths %d and %d; both must be one of %s'
                                      % (nd.layer.name, w[0], w[1], ROUTER_WIDTHS))
        widths[w[0]] = nd.layer.name
    if len(widths) > 1:
        raise NotImplementedError('engine: routers of different widths in one net (%s); all must share one of %s'
                                  % (', '.join('%s: %d' % (n, w) for w, n in sorted(widths.items())), ROUTER_WIDTHS))
    return next(iter(widths), 16)


class _DevMem:
    """device memory that is not torch's (the cudaMalloc'ed exchange buffer of the fused data-parallel tail) as
    a zero-copy torch tensor, through __cuda_array_interface__"""
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = dict(shape=(int(n),), typestr='<f4', data=(int(ptr), False), version=2)
assert _BN_FUSE.itemsize == 80 and _BN_BWD_FUSE.itemsize == 32 and _BN_BWD_EPI.itemsize == 56


def _host_struct(dtype, **fields):
    """one C struct in host memory (numpy record); pointers given as c_void_p / int / None"""
    rec = np.zeros(1, dtype)
    for k, v in fields.items():
        rec[k] = (v.value or 0) if isinstance(v, ctypes.c_void_p) else (0 if v is None else v)
    return rec


def _ru(a, b):
    return (a + b - 1) // b * b


def _vp(t):
    """device pointer of a tensor (or None) as c_void_p"""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


@contextlib.contextmanager
def _gc_off():
    """Around a CUDA graph capture.  The cyclic garbage collector must not run inside capture: freeing a tensor of an
    engine that was dropped earlier (plans and their launch closures are reference cycles) makes the allocator record
    an event on a capturing stream, which invalidates the capture.  Collect now, keep the collector off until capture
    ends."""
    gc.collect()
    was_on = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if was_on:
            gc.enable()


def _comps(layer):
    """comps of a chain without the ones that are the identity as configured: Dropout(λ=1) (tf.nn.dropout with
    keep_prob 1, the default of lib/layer_types.py:212-217) and ActivityError (:287-293; α = 0 is no cost at all, α != 0
    behind the Rect of a Conv block is picked up by _activity)"""
    out = []
    for c in layer.comps:
        if type(c) is Dropout:
            prev = out[-1] if out else None
            if float(c.hypers.λ) != 1.0 and not (isinstance(prev, Rect) and len(out) >= 3 and isinstance(out[-3], Conv)):
                raise NotImplementedError('engine: Dropout(λ=%r) is served directly behind the Rect of a '
                                          'Conv-BatchNorm-Rect block (elsewhere only keep_prob 1)' % c.hypers.λ)
            continue
        if type(c) is ActivityError:
            prev = out[-1] if out else None
            if float(c.hypers.α) != 0.0 and not (isinstance(prev, Rect) and len(out) >= 3 and isinstance(out[-3], Conv)):
                raise NotImplementedError('engine: ActivityError(α=%r) is served directly behind the Rect of a '
                                          'Conv-BatchNorm-Rect block (elsewhere only α = 0)' % c.hypers.α)
            continue
        out.append(c)
    return out


def _dropout(layer):
    """keep probability of the Dropout behind the Rect of a Conv block (1: none)"""
    keep = [float(c.hypers.λ) for c in layer.comps if type(c) is Dropout and float(c.hypers.λ) != 1.0]
    if len(keep) > 1:
        raise NotImplementedError('engine: more than one Dropout in a block')
    return keep[0] if keep else 1.0


def _activity(layer):
    """α of the ActivityError behind the Rect of a Conv block (0: none)"""
    return sum(float(c.hypers.α) for c in layer.comps if type(c) is ActivityError)


def _is_chain(layer, types):
    if not isinstance(layer, Chain):
        return False
    comps = _comps(layer)
    return len(comps) == len(types) and all(isinstance(c, t) for c, t in zip(comps, types))


_PYR = [ToPyramid]
_RCM = [MultiscaleConvMax, MultiscaleBatchNorm, MultiscaleRect]
# split-precision modes: the launches of one source tensor as (parts of A0, parts of A1, weight pack modes along K).
# x3 (two parts): [hi | lo | hi] x [hi; hi; lo]; x6 (three parts): [hi | mid | lo] x [hi; hi; hi], then
# [hi | mid | hi] x [mid; mid; lo].  Pack modes: 0 = bf16(w), 4 = first residual, 8 = second residual.
_SPLIT_PASSES = {2: [(2, 1, (0, 0, 4))], 3: [(3, 0, (0, 0, 0)), (2, 1, (4, 4, 8))]}

# standalone Conv (lib/layer_types.py:55-74) as a tree node: 3x3 SAME conv + bias -> BatchNorm -> ReLU on ONE
# tensor -- the input image, a pyramid scale picked by a leading Select, or the tensor of the node above --
# and a classifier that flattens a tensor without a Select.  Arithmetically a one-scale MultiscaleConvMax
# stage: the same kernels serve it (mpnn_conv_bn_stats / mpnn_stencil_gemm with A1 = NULL).
_CNV = [Conv, BatchNorm, Rect]
_CNVS = [Select, Conv, BatchNorm, Rect]
_RTR = [Select, LinTrans, BatchNorm, Rect, LinTrans, BatchNorm, Rect, LinTrans]


def _leaf_spec(layer):
    """[Select | GlobalMaxPool,] LinTrans + one of the error layers of lib/layer_types.py:255-285 -> (select, fc, error layer, kind):
    'ce' Softmax + CrossEntropyError, 'sce' Softmax + SuperclassCrossEntropyError, 'sq' SquaredError (on the
    LinTrans output itself); None for anything else"""
    if not isinstance(layer, Chain):
        return None
    comps = _comps(layer)
    sel = comps.pop(0) if comps and isinstance(comps[0], (Select, GlobalMaxPool)) else None
    if not comps or not isinstance(comps[0], LinTrans):
        return None
    fc, tail = comps[0], comps[1:]
    if len(tail) == 2 and isinstance(tail[0], Softmax) and type(tail[1]) is CrossEntropyError:
        return sel, fc, tail[1], 'ce'
    if len(tail) == 2 and isinstance(tail[0], Softmax) and type(tail[1]) is SuperclassCrossEntropyError:
        return sel, fc, tail[1], 'sce'
    if len(tail) == 1 and type(tail[0]) is SquaredError:
        return sel, fc, tail[0], 'sq'
    return None


class Geo:
    """Padded-planes geometry of one scale (see csrc/common.cuh)."""

    def __init__(self, B, H, W):
        self.B, self.H, self.W = B, H, W
        self.Wp = W + 1
        self.S = (H + 1) * (W + 1)
        self.rows = B * self.S
        self.G = max(64, _ru(W + 2, 8))
        self.P = _ru(self.G + self.rows + 128 + self.G, 8)

    def args(self):
        return (self.B, self.H, self.W, self.G, self.P)


class Engine:
    def __init__(self, net, precision='fp32', device=None, graphs=False, dist=False, impl=None,
                 dry_run=False):
        # dry_run: build plans on host memory without launching anything (used by
        # the CPU test-suite to exercise the planner); it cannot execute.
        self.dry = bool(dry_run)
        if not self.dry and not torch.cuda.is_available():
            raise RuntimeError('multipath-nn_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        self.L = _cabi.lib()
        self.net = net
        if self.dry:
            self.dev = torch.device('cpu')
        else:
            self.dev = torch.device('cuda', torch.cuda.current_device() if device is None else device)
        assert precision in ('fp32', 'bf16', 'bf16x3', 'bf16x6')
        # 'bf16x3': fp32 storage and elementwise arithmetic like 'fp32', but the convolutions run on the tensor
        # cores: every fp32 operand is split into two bf16 planes sets (x = hi + lo, mpnn_split_planes) and a
        # product is evaluated as a_hi*b_hi + a_lo*b_hi + a_hi*b_lo with fp32 accumulation (2^-16 relative) --
        # the reference's fp32 arithmetic (layer_types.py:106-107) on tcgen05 within the 1e-3 tolerance
        # 'bf16x6': the same with three-way splits (x = hi + mid + lo, 24 significant bits, mpnn_split_planes3) and
        # the six products of relative size >= 2^-16 -- the tensor-core mode that meets 1e-3 on gradients too.
        # self.split = number of bf16 parts per fp32 operand (0: no splitting)
        self.split = {'bf16x3': 2, 'bf16x6': 3}.get(precision, 0)
        self.dtype = BF16 if precision == 'bf16' else F32
        self.tdtype = torch.bfloat16 if precision == 'bf16' else torch.float32
        # stencil implementation: 0 = SIMT fp32-accumulate, 1 = tcgen05
        self.impl = (1 if (precision != 'fp32' and self.L.mpnn_has_umma()) else 0) if impl is None else impl
        if self.split and self.impl != 1:
            raise RuntimeError('precision %s needs the tcgen05 kernels' % precision)
        # weight gradient follows the conv implementation (per launch it drops back to the
        # SIMT kernel when the shape exceeds what the tcgen05 wgrad tiles: K0+K1 > 128)
        self.impl_w = self.impl
        self.use_graphs = graphs
        self.dist = dist
        self.world = torch.distributed.get_world_size() if dist else 1
        self.dynamic = bool(net.dynamic)
        self.critic = type(net).__name__ == 'CriticNet'
        self.stream = None
        self.comm = None
        self.graph_collective = os.environ.get('MPNN_DIST_GRAPH', '1') != '0'
        self.overlap_allreduce = os.environ.get('MPNN_DIST_OVERLAP', '1') != '0'
        # data-parallel step tail as ONE kernel over NVLink peer memory (csrc/p2p.cu: reduce-scatter by peer loads,
        # TALR + momentum on the owned slice, all-gather by peer stores) instead of ncclAllReduce + optimiser
        self.fused_dp = bool(dist) and self.world > 1 and not self.dry and os.environ.get('MPNN_DIST_FUSED', '0') != '0'
        self._p2p_desc = None
        self.lane_priority = os.environ.get('MPNN_LANE_PRIORITY', '0') != '0'
        # classifier / router-input heads rotate over this many lanes (1: all on the one heads lane, in stage order)
        self.head_lanes = max(1, int(os.environ.get('MPNN_HEAD_LANES', '4')))
        self.pack_blocks = max(1, int(os.environ.get('MPNN_PACK_BLOCKS', '32')))      # CTAs per weight tensor in the packing launch
        # train-mode BN statistics: the conv only accumulates the totals, the BN / ReLU / pool kernel behind it derives
        # the constants (MPNN_DEFER_BN=0: the conv's last CTA finalises them, as in round 1)
        self.defer_bn = os.environ.get('MPNN_DEFER_BN', '0') != '0'
        # BatchNorm backward of small tensors without a pooling branch as one launch (MPNN_BN_SMALL=0: the two-pass pair)
        self.bn_small = os.environ.get('MPNN_BN_SMALL', '1') != '0'
        self._snapshot = False
        self._analyse()
        self._alloc_params()
        if self.fused_dp:
            self._init_p2p()
        self._plans = {}
        self._graphs = {}
        self._lanes = None
        self._copy_stream, self._stage, self._stage_i = None, {}, 0
        self.multistream = os.environ.get('MPNN_MULTISTREAM', '1') != '0'
        self.fuse_bn_red = os.environ.get('MPNN_FUSE_BNRED', '1') != '0'
        self.fuse_bn_red_min_rows = int(os.environ.get('MPNN_FUSE_BNRED_MIN_ROWS', 65536))
        # per-step scalars travel host->device asynchronously from pinned memory; a ring of slots
        # (each guarded by an event) keeps step t+1's values from overwriting step t's before its
        # copy has executed
        self._hyp_ring = [torch.zeros(HYP_COUNT, dtype=torch.float32) for _ in range(1 if self.dry else 16)]
        if not self.dry:
            self._hyp_ring = [t.pin_memory() for t in self._hyp_ring]
        self._hyp_ev = [None] * len(self._hyp_ring)
        self._hyp_i = 0
        self.draw = 0
        self.hyp_host = self._hyp_ring[0]
        self.hyp = torch.zeros(HYP_COUNT, dtype=torch.float32, device=self.dev)

    # ------------------------------------------------------------------ #
    # static analysis of the layer tree
    # ------------------------------------------------------------------ #
    def _analyse(self):
        net = self.net
        self.nodes = []

        def visit(layer, parent, sink_idx):
            nd = Ns(layer=layer, idx=len(self.nodes), parent=parent, sink_idx=sink_idx, kids=[],
                    router=layer.router)
            if _is_chain(layer, _PYR) or _is_chain(layer, _PYR + [MultiscaleLLN]):
                nd.kind = 'pyr'
                nd.lln = _comps(layer)[1] if len(_comps(layer)) > 1 else None     # local luminance normalisation of every scale
                if nd.lln is not None and net.hypers.x0_shape[2] != 3:
                    raise ValueError('MultiscaleLLN weighs R, G, B: the input has %d channels' % net.hypers.x0_shape[2])
            elif _is_chain(layer, _RCM):
                nd.kind = 'rcm'
                nd.cm, nd.mbn, nd.sel = _comps(layer)[0], _comps(layer)[1], None
                if nd.cm.hypers.supp != 3:
                    raise NotImplementedError('engine: MultiscaleConvMax supp=%r' % nd.cm.hypers.supp)
            elif any(_is_chain(layer, pat) for pat in (_CNV, _CNVS, _CNV + [MaxPool], _CNVS + [MaxPool])):
                nd.kind = 'rcm'
                comps = _comps(layer)
                off = 1 if isinstance(comps[0], Select) else 0
                conv, bn = comps[off], comps[off + 1]
                nd.maxpool = isinstance(comps[-1], MaxPool)
                nd.act_alpha = _activity(layer)
                nd.keep = _dropout(layer)
                if (nd.act_alpha or nd.keep != 1.0) and self.split:
                    raise NotImplementedError('engine: ActivityError / Dropout in bf16x3 precision')
                if nd.act_alpha and nd.keep != 1.0:
                    raise NotImplementedError('engine: ActivityError and Dropout in one block')
                if nd.maxpool and (comps[-1].hypers.stride, comps[-1].hypers.supp) != (2, 2):
                    # tf.nn.max_pool(x, strides, k_shape): window = stride, step = supp (SURVEY F8)
                    raise NotImplementedError('engine: MaxPool(stride=%r, supp=%r): the 2 / 2 window is served'
                                              % (comps[-1].hypers.stride, comps[-1].hypers.supp))
                if nd.maxpool and self.split:
                    raise NotImplementedError('engine: MaxPool in bf16x3 precision')
                if conv.hypers.supp != 3 or conv.hypers.res:
                    raise NotImplementedError('engine: standalone Conv with supp=%r res=%r (3x3 without the residual '
                                              'initialisation is what the stencil kernels serve)' % (conv.hypers.supp, conv.hypers.res))
                if conv.hypers.n_chan % 16:
                    raise NotImplementedError('engine: Conv n_chan=%d (multiples of 16)' % conv.hypers.n_chan)
                # the stage code reads a MultiscaleConvMax / MultiscaleBatchNorm pair: present the Conv as one scale
                nd.cm = Ns(hypers=Ns(n_chan=[conv.hypers.n_chan], supp=3, k_l2=conv.hypers.k_l2),
                           params=Ns(w_horz_0=conv.params.w, b_0=conv.params.b))
                nd.mbn = Ns(comps=[bn])
                nd.sel = comps[0].hypers.i if off else None
                nd.tensor_in = not off
            elif _leaf_spec(layer) is not None:
                nd.kind = 'reg'
                sel, nd.fc, nd.ce, nd.loss = _leaf_spec(layer)
                nd.gmp = isinstance(sel, GlobalMaxPool)
                if sel is not None and not nd.gmp and sel.hypers.i != -1:
                    raise NotImplementedError('engine: LogReg must select the coarsest scale')
                n_cls, n_out = net.hypers.y_shape[0], nd.fc.hypers.n_chan
                if nd.loss == 'sce':
                    w_cls = None if nd.ce.hypers.w_cls is None else np.asarray(nd.ce.hypers.w_cls, np.float32)
                    if w_cls is None or w_cls.shape != (n_cls, n_out):
                        raise ValueError('SuperclassCrossEntropyError of %r: w_cls must be (%d, %d)' % (layer.name, n_cls, n_out))
                    nd.w_cls = w_cls
                elif n_out != n_cls:
                    raise ValueError('classifier %r has %d outputs for %d classes' % (layer.name, n_out, n_cls))
            else:
                raise NotImplementedError(
                    'engine: tree node %r (%s) is not one of the hot-path compositions '
                    '(ToPyramid | ConvMax+BN+Rect | Select+LinTrans+Softmax+CrossEntropy)'
                    % (layer.name, [type(c).__name__ for c in layer.comps]))
            if layer.router is not None:
                if not _is_chain(layer.router, _RTR):
                    raise NotImplementedError('engine: router of %r is not the FC-BN-ReLU x2 + FC chain' % layer.name)
                if len(layer.sinks) < 2 or len(layer.sinks) > MAXS:
                    raise NotImplementedError('engine: router with %d sinks' % len(layer.sinks))
            elif len(layer.sinks) > 1:
                raise ValueError('switch %r has no router' % layer.name)
            self.nodes.append(nd)
            if parent is not None:
                self.nodes[parent].kids.append(nd.idx)
            for i, s in enumerate(layer.sinks):
                visit(s, nd.idx, i)
        visit(net.root, None, 0)
        if self.nodes[0].kind != 'pyr' and not getattr(self.nodes[0], 'tensor_in', False):
            raise NotImplementedError('engine: the root must be the ToPyramid chain or a Conv-BatchNorm-Rect chain')
        for nd in self.nodes:
            par = self.nodes[nd.parent] if nd.parent is not None else None
            if getattr(nd, 'tensor_in', False) and par is not None and par.kind == 'pyr':
                raise NotImplementedError('engine: %r takes a tensor but sits under the pyramid (lead with Select)' % nd.layer.name)
            if nd.kind == 'rcm' and nd.sel is not None and (par is None or par.kind != 'pyr'):
                raise NotImplementedError('engine: Select + Conv must sit directly under the ToPyramid node')
        for nd in self.nodes:
            if nd.kind == 'reg' and getattr(nd, 'gmp', False):
                par = self.nodes[nd.parent]
                if len(par.kids) != 1 or par.router is not None or not hasattr(par, 'tensor_in') \
                        or getattr(par, 'maxpool', False) or self.split:
                    raise NotImplementedError('engine: a GlobalMaxPool classifier must be the only sink of a '
                                              'Conv-BatchNorm-Rect block (no router, no MaxPool, not bf16x3)')
                par.gmp = True
            if nd.kind == 'reg' and nd.kids:
                raise NotImplementedError('engine: LogReg with sinks')
            if nd.kind in ('rcm', 'reg') and nd.parent is not None and self.nodes[nd.parent].kind == 'reg':
                raise NotImplementedError('engine: node under a LogReg')
            if nd.kind == 'pyr' and nd.idx != 0:
                raise NotImplementedError('engine: nested ToPyramid')
            if nd.kind == 'pyr' and (nd.router is not None):
                raise NotImplementedError('engine: router on the ToPyramid node')
        self.leaves = [nd for nd in self.nodes if not nd.kids]
        self.switches = [nd for nd in self.nodes if len(nd.kids) > 1]
        for s, nd in enumerate(self.switches):
            nd.sw = s
        for e, nd in enumerate(nd for nd in self.nodes if nd.kind == 'reg'):
            nd.err = e
        self.regs = [nd for nd in self.nodes if nd.kind == 'reg']
        if not self.dynamic and self.switches:
            raise NotImplementedError('engine: SRNet with switches')
        self.router_width = _router_width(self.nodes)

    # ------------------------------------------------------------------ #
    # parameters: flat trainable buffer + flat state buffer (BN EMAs)
    # ------------------------------------------------------------------ #
    def _alloc_params(self):
        net = self.net
        hy = net.hypers
        a_rtr = float(getattr(hy, 'α_rtr', 1.0)) if self.dynamic else 1.0
        self.tparams, self.sparams = [], []
        seg_start, seg_node, seg_mult, seg_l2 = [], [], [], []
        off_t = off_s = 0

        def walk(layer, node_idx, mult):
            nonlocal off_t, off_s
            if layer is None:
                return
            for key, p in vars(layer.params).items():
                assert isinstance(p, Param)
                if p.trainable:
                    l2 = 0.0
                    if isinstance(layer, LinTrans) and key == 'w':
                        if getattr(layer.hypers, 'res', False):
                            raise NotImplementedError('engine: LinTrans(res=True)')
                        l2 = float(layer.hypers.k_l2)
                    elif isinstance(layer, MultiscaleConvMax) and key.startswith('w_'):
                        l2 = float(layer.hypers.k_l2)
                    elif isinstance(layer, Conv) and key == 'w':
                        l2 = float(layer.hypers.k_l2)
                    off_t = _ru(off_t, 4)          # 16-byte aligned: vector reductions into the gradient
                    p._bind = (self, 'theta', off_t)
                    self.tparams.append(p)
                    seg_start.append(off_t); seg_node.append(node_idx)
                    seg_mult.append(mult); seg_l2.append(l2)
                    off_t += p.value.size
                else:
                    p._bind = (self, 'state', off_s)
                    self.sparams.append(p)
                    off_s += p.value.size
            for c in layer.comps:
                walk(c, node_idx, mult)
        for nd in self.nodes:
            walk(nd.layer, nd.idx, 1.0)
            walk(nd.router, nd.idx, a_rtr)
        self.n_theta, self.n_state = off_t, off_s
        seg_start.append(off_t)
        n_nodes = len(self.nodes)
        dev = self.dev
        self.theta = None if self.fused_dp else torch.zeros(off_t, dtype=torch.float32, device=dev)
        # gradient buffer = [per-node p_tr moments (2 per node, padded to 16 bytes) | gradients]: the moments
        # travel with the gradients through the all-reduce (data-parallel TALR stays replica-consistent) and
        # sit in FRONT so that the two buckets of the overlapped all-reduce are contiguous: [moments | shallow
        # stages] and [deep stages] (their gradients are complete first, see _Plan._build)
        self.g0 = _ru(2 * n_nodes, 4)
        if self.fused_dp:
            # [flags | grad | theta | accum] in one cudaMalloc'ed, zero-filled buffer that the other ranks map (CUDA IPC).
            # It is deliberately never freed: a peer may still hold the mapping when this engine goes away, and the
            # flag epochs must stay monotonic for the life of the process (a few MB per engine).
            ng, nt = _ru(self.g0 + off_t, 4), _ru(off_t, 4)
            o_g = _P2P_FLAG_BYTES
            o_t = _ru(o_g + 4 * ng, 256)
            o_a = _ru(o_t + 4 * nt, 256)
            base = ctypes.c_void_p()
            with torch.cuda.device(dev):
                self.L.p2p_alloc(ctypes.byref(base), _ru(o_a + 4 * nt, 256))
                self.grad = torch.as_tensor(_DevMem(base.value + o_g, self.g0 + off_t), device=dev)
                self.theta = torch.as_tensor(_DevMem(base.value + o_t, off_t), device=dev)
                self.accum = torch.as_tensor(_DevMem(base.value + o_a, off_t), device=dev)
            self._p2p_base, self._p2p_offs = base.value, (o_g, o_t, o_a)
        else:
            self.grad = torch.zeros(self.g0 + off_t, dtype=torch.float32, device=dev)
            self.accum = torch.zeros(off_t, dtype=torch.float32, device=dev)
        self.state = torch.zeros(max(off_s, 1), dtype=torch.float32, device=dev)
        self.seg_start = torch.tensor(seg_start, dtype=torch.int32, device=dev)
        self.seg_node = torch.tensor(seg_node, dtype=torch.int32, device=dev)
        self.seg_mult = torch.tensor(seg_mult, dtype=torch.float32, device=dev)
        self.seg_l2 = torch.tensor(seg_l2, dtype=torch.float32, device=dev)
        self.n_seg = len(seg_node)
        self.seg_node_list = list(seg_node)
        for p in self.tparams + self.sparams:
            self.push_param(p)

    def _buf(self, p):
        kind, off = p._bind[1], p._bind[2]
        return (self.theta if kind == 'theta' else self.state)[off:off + p.value.size]

    def push_param(self, p):
        self._buf(p).copy_(torch.from_numpy(p.value.reshape(-1)))

    def fetch_param(self, p):
        if self._snapshot:
            return                                    # p.value is current (host_snapshot)
        p.value = self._buf(p).cpu().numpy().reshape(p.value.shape).copy()

    def host_snapshot(self):
        """Context manager: fetch ALL parameters with one device-to-host copy per flat buffer (trainable |
        state) and serve `Param.eval()` from the host copies while it is open (serdes / checkpoints read
        ~150 tensors; one blocking copy each is most of their cost)."""
        import contextlib

        @contextlib.contextmanager
        def cm():
            th, st = self.theta.cpu().numpy(), self.state.cpu().numpy()
            for p in self.tparams + self.sparams:
                src = th if p._bind[1] == 'theta' else st
                p.value = src[p._bind[2]:p._bind[2] + p.value.size].reshape(p.value.shape).copy()
            self._snapshot = True
            try:
                yield self
            finally:
                self._snapshot = False
        return cm()

    def momentum_numpy(self):
        """optimiser accumulators, one array per trainable tensor in `self.tparams` order (one D2H copy)"""
        a = self.accum.cpu().numpy()
        return [a[p._bind[2]:p._bind[2] + p.value.size].reshape(p.value.shape).copy() for p in self.tparams]

    def load_momentum(self, arrays):
        if len(arrays) != len(self.tparams):
            raise ValueError('load_momentum: %d arrays for %d trainable tensors' % (len(arrays), len(self.tparams)))
        for p, a in zip(self.tparams, arrays):
            a = np.asarray(a, dtype=np.float32)
            if a.shape != p.value.shape:
                raise ValueError('load_momentum: shape %s != %s' % (a.shape, p.value.shape))
            self.accum[p._bind[2]:p._bind[2] + a.size].copy_(torch.from_numpy(np.ascontiguousarray(a).reshape(-1)))

    def tptr(self, p):
        return ctypes.c_void_p(self.theta.data_ptr() + 4 * p._bind[2]) if p._bind[1] == 'theta' \
            else ctypes.c_void_p(self.state.data_ptr() + 4 * p._bind[2])

    def gptr(self, p):
        assert p._bind[1] == 'theta'
        return ctypes.c_void_p(self.grad.data_ptr() + 4 * (self.g0 + p._bind[2]))

    def grads_numpy(self, with_l2=False):
        """{Param: gradient ndarray} of the last backward (before TALR).  The L2
        (c_mod) term is applied inside the optimiser kernel; with_l2 adds it here
        the same way (2 k_l2 mean(p_tr) theta) so the result is d c_tot / d theta."""
        gall = self.grad.cpu().numpy().astype(np.float64)
        g = gall[self.g0:]
        out = {}
        if with_l2:
            th = self.theta.cpu().numpy().astype(np.float64)
            l2 = self.seg_l2.cpu().numpy(); node = self.seg_node.cpu().numpy()
            stats = gall[:2 * len(self.nodes)].reshape(-1, 2)
        for s, p in enumerate(self.tparams):
            sl = slice(p._bind[2], p._bind[2] + p.value.size)
            v = g[sl].copy()
            if with_l2 and l2[s] > 0:
                coef = stats[node[s], 1] if self.dynamic else 1.0
                v += 2.0 * l2[s] * coef * th[sl]
            out[p] = v.reshape(p.value.shape)
        return out

    # ------------------------------------------------------------------ #
    # plan construction
    # ------------------------------------------------------------------ #
    def _plan(self, B, bn_train, need_bwd):
        key = (B, bool(bn_train), bool(need_bwd))
        if key not in self._plans:
            self._plans[key] = _Plan(self, B, bn_train, need_bwd)
        return self._plans[key]

    # ------------------------------------------------------------------ #
    # feeding
    # ------------------------------------------------------------------ #
    def _to_dev(self, v, shape, name):
        if isinstance(v, torch.Tensor):
            t = v
            if t.dtype != torch.float32:
                t = t.float()
        else:
            t = torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32))
        if tuple(t.shape) != tuple(shape):
            raise ValueError('feed %s: shape %s, expected %s' % (name, tuple(t.shape), tuple(shape)))
        return t

    def _feed(self, plan, feed, train):
        net = self.net
        hy = net.hypers
        x0 = feed[net.x0]
        y = feed[net.y]
        B = plan.B
        self._upload(plan, self._to_dev(x0, (B,) + tuple(hy.x0_shape), 'x0'),
                     self._to_dev(y, (B,) + tuple(hy.y_shape), 'y'))
        i = self._hyp_i = (self._hyp_i + 1) % len(self._hyp_ring)
        if self._hyp_ev[i] is not None:
            self._hyp_ev[i].synchronize()
        h = self.hyp_host = self._hyp_ring[i]
        h[HYP_LR] = float(feed.get(net.λ_lrn, hy.λ_lrn))
        h[HYP_MU] = float(feed.get(net.μ_lrn, hy.μ_lrn))
        h[HYP_GSCALE] = 1.0 / self.world
        self.draw = (self.draw + 1) & 0xFFFFFFFF       # Dropout masks: one draw per evaluation (bits of a uint32)
        h.view(torch.int32)[HYP_DRAW] = self.draw - (1 << 32) if self.draw >= (1 << 31) else self.draw
        if self.dynamic:
            h[HYP_TAU] = float(feed.get(net.τ, hy.τ))
            h[HYP_EPS] = float(feed.get(net.ϵ, hy.ε))
            if hy.dyn_k_cpt:
                kc = np.asarray(feed[net.k_cpt], dtype=np.float32).reshape(-1)
                if kc.size == 1:
                    kc = np.full(B, kc[0], np.float32)      # train-adaptive-nets:102-105
                if kc.size != B:
                    raise ValueError('feed k_cpt: %d values for batch %d' % (kc.size, B))
                plan.kcpt.copy_(torch.from_numpy(kc), non_blocking=True)
                plan.kextra.copy_(torch.from_numpy(kc * np.float32(hy.α_cpt)), non_blocking=True)
                for col in plan.kplanes:          # tcgen05 heads: the feature is one more input column
                    col[:B].copy_(plan.kextra)
            else:
                h[HYP_KCPT] = float(hy.k_cpt)
        self.hyp.copy_(h, non_blocking=True)
        if self._hyp_ev[i] is None:
            self._hyp_ev[i] = torch.cuda.Event()
        self._hyp_ev[i].record()

    def _upload(self, plan, x0, y):
        """Host batch -> plan.x0 / plan.y.  Host tensors go through a double-buffered device
        staging slot on a copy stream, so the PCIe transfer of step t+1 overlaps the kernels of
        step t; the step itself starts with a device-to-device copy out of the slot."""
        if x0.is_cuda and y.is_cuda:
            plan.x0.copy_(x0, non_blocking=True)
            plan.y.copy_(y, non_blocking=True)
            return
        main = torch.cuda.current_stream(self.dev)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(self.dev)
        slots = self._stage.get(plan.B)
        if slots is None:
            slots = self._stage[plan.B] = [Ns(x=torch.empty_like(plan.x0), y=torch.empty_like(plan.y),
                                              ready=torch.cuda.Event(), consumed=None, src=None)
                                           for _ in range(2)]
        self._stage_i ^= 1
        sl = slots[self._stage_i]
        cs = self._copy_stream
        if sl.consumed is not None:
            cs.wait_event(sl.consumed)             # the step that read this slot two uploads ago
        with torch.cuda.stream(cs):
            sl.src = (x0, y)                       # keep pinned sources alive until the slot is reused
            sl.x.copy_(x0, non_blocking=True)
            sl.y.copy_(y, non_blocking=True)
            sl.ready.record(cs)
        main.wait_event(sl.ready)
        plan.x0.copy_(sl.x, non_blocking=True)
        plan.y.copy_(sl.y, non_blocking=True)
        if sl.consumed is None:
            sl.consumed = torch.cuda.Event()
        sl.consumed.record(main)

    def _batch_of(self, feed):
        x0 = feed[self.net.x0]
        return int(x0.shape[0])

    # ------------------------------------------------------------------ #
    # public steps
    # ------------------------------------------------------------------ #
    def _run(self, ops):
        if self.dry:
            raise RuntimeError('dry-run engine cannot execute: the hot path is CUDA-only')
        main = torch.cuda.current_stream(self.dev)
        main_p = self.stream = ctypes.c_void_p(main.cuda_stream)
        if not self.multistream:
            for op in ops:
                self.stream = main_p
                op()
            return
        # Lanes (one CUDA stream each).  0: input packing, routing, optimiser.  1: classifier and
        # router heads, which only feed the losses (forward) or start from them (backward).
        # 9 / 10+k: weight gradients of the heads / of the convs at scale k, which only feed the
        # optimiser and are mutually independent.  3+k: the conv / BN / data-gradient
        # ops of pyramid scale k -- layer L at scale k depends on layer L-1 at scale k (same lane)
        # and on layer L at scale k-1 (pooled input; the neighbouring lane), so the scales advance
        # as a wavefront and the small, latency-bound coarse-scale launches hide behind the large
        # fine-scale ones.  Every lane forks from the main stream at the head of an op list and joins
        # it at the end (valid under capture); all other cross-lane edges are explicit
        # (op.deps -> events), including those from lane-0 ops issued earlier in the same list.
        if self._lanes is None:
            self._lanes = {}
        used = sorted({getattr(op, 'lane', 0) for op in ops} - {0})
        for lane in used:                         # fork: every lane starts after what main holds now
            if lane not in self._lanes:
                # the conv / BN chain of the pyramid scales (3..7) and the heads (1) are the critical path of the
                # step; weight gradients (9, 10+k), TALR moments (8) and the gradient all-reduce (20) only feed the
                # optimiser: they run at lower stream priority, so their CTAs fill SMs the chain leaves idle
                # instead of delaying it.  Measured: +2 % at B = 128, -3 % at B = 4096 -> off unless MPNN_LANE_PRIORITY=1
                hi = self.lane_priority and (lane in (1, 3, 4, 5, 6, 7) or 21 <= lane < 40)
                self._lanes[lane] = torch.cuda.Stream(self.dev, priority=-1 if hi else 0)
            self._lanes[lane].wait_stream(main)
        for op in ops:
            lane = getattr(op, 'lane', 0)
            st = main if lane == 0 else self._lanes[lane]
            for d in getattr(op, 'deps', ()):
                if getattr(d, 'lane', 0) != lane and getattr(d, '_ev', None) is not None:
                    st.wait_event(d._ev)
            if getattr(op, 'wait_all', False):      # ordered after everything issued so far, on every lane
                for other in [0] + used:
                    if other != lane:
                        ev = torch.cuda.Event()
                        ev.record(main if other == 0 else self._lanes[other])
                        st.wait_event(ev)
            self.stream = main_p if lane == 0 else ctypes.c_void_p(st.cuda_stream)
            op()
            if getattr(op, 'signal', False):
                op._ev = torch.cuda.Event()
                op._ev.record(st)
        self.stream = main_p
        for lane in used:
            main.wait_stream(self._lanes[lane])

    def train_step(self, feed, update=True):
        """One `net.train.run(...)`: forward ('tr'), backward, TALR + momentum."""
        B = self._batch_of(feed)
        plan = self._plan(B, True, True)
        with torch.cuda.device(self.dev):
            self._feed(plan, feed, True)
            self.run_resident(plan, update)

    def run_resident(self, plan, update=True):
        """Step on inputs already resident in plan.x0 / plan.y / self.hyp."""
        if self.use_graphs and update:
            g = self._graphs.get(id(plan))
            if g is None:
                g = self._capture(plan)
            g[0].replay()                        # pack + forward + backward (+ all-reduce + optimiser when captured)
            if g[1] is not None:
                if self.dist and not self.fused_dp:
                    self._allreduce(0, plan.ar_split)   # MPNN_DIST_GRAPH=0: issued eagerly between two graphs
                g[1].replay()                    # TALR + momentum
            return
        self._compute_ops(plan)
        if update:
            if self.dist and not self.fused_dp:
                self._allreduce(0, plan.ar_split)
            self._run(plan.opt_ops)

    def _init_comm(self):
        """Our own NCCL communicator (C ABI: mpnn_comm_*): rank 0 makes the unique id, the existing process
        group ships its 128 bytes, every rank joins.  Owning the communicator keeps the all-reduce on the
        step's stream and lets it be captured into the step's CUDA graph."""
        import torch.distributed as dist
        rank = dist.get_rank()
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            self.L.comm_unique_id(ctypes.c_void_p(uid.data_ptr()))
        t = uid.to(self.dev) if dist.get_backend() == 'nccl' else uid
        dist.broadcast(t, 0)
        uid = t.cpu().contiguous()
        comm = ctypes.c_void_p()
        with torch.cuda.device(self.dev):
            self.L.comm_init_rank(ctypes.byref(comm), self.world, rank, ctypes.c_void_p(uid.data_ptr()))
        self.comm = comm

    def _init_p2p(self):
        """exchange the CUDA-IPC handles of the exchange buffers over the process group and map the peers' buffers
        (collective: every rank builds its engine at the same point); one node only"""
        import torch.distributed as dist
        rank, world = dist.get_rank(), self.world
        if world > _P2P_MAX or int(os.environ.get('LOCAL_WORLD_SIZE', world)) != world:
            raise RuntimeError('MPNN_DIST_FUSED: the fused data-parallel tail maps peer memory of ONE node, up to %d ranks'
                               % _P2P_MAX)
        h = torch.zeros(_P2P_HANDLE_BYTES, dtype=torch.uint8)
        self.L.p2p_export(ctypes.c_void_p(self._p2p_base), ctypes.c_void_p(h.data_ptr()))
        on_dev = dist.get_backend() == 'nccl'
        mine = h.to(self.dev) if on_dev else h
        hs = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(hs, mine)
        rec = np.zeros(1, _P2P)
        with torch.cuda.device(self.dev):
            for r in range(world):
                if r == rank:
                    rec['base'][0, r] = self._p2p_base
                else:
                    hr = hs[r].cpu().contiguous()
                    p = ctypes.c_void_p()
                    self.L.p2p_import(ctypes.c_void_p(hr.data_ptr()), ctypes.byref(p))
                    rec['base'][0, r] = p.value
        rec['world'], rec['rank'] = world, rank
        rec['off_grad'], rec['off_theta'], rec['off_accum'] = self._p2p_offs
        rec['g0'], rec['n'] = self.g0, self.n_theta
        self._p2p_desc = rec
        dist.barrier()

    def p2p_status(self):
        """0, or 1 if a wait inside the fused tail timed out (a rank never arrived)"""
        st = ctypes.c_int(0)
        self.L.p2p_status(ctypes.c_void_p(self._p2p_base), ctypes.byref(st))
        return st.value

    def _allreduce(self, lo=0, hi=None, stream=None):
        """the collective of a step: sum of [TALR moments | gradients] over the replicas, in place.  With the
        overlapped schedule it is issued as two buckets: grad[split:] (the deep stages, complete first) under
        the rest of the backward pass, grad[:split] at its end."""
        if self.comm is None:
            self._init_comm()
        hi = self.grad.numel() if hi is None else hi
        if hi <= lo:
            return
        st = stream if stream is not None else ctypes.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)
        self.L.allreduce_flat(self.comm, ctypes.c_void_p(self.grad.data_ptr() + 4 * lo), hi - lo, st)

    def average_state(self):
        """BatchNorm running moments are per-replica (each replica normalises with its own shard's moments,
        SURVEY F3): average them over the replicas before they are serialised or used for statistics"""
        if self.dist and self.world > 1:
            if self.comm is None:
                self._init_comm()
            st = ctypes.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)
            self.L.allreduce_flat(self.comm, _vp(self.state), self.state.numel(), st)
            self.state.mul_(1.0 / self.world)

    def _compute_ops(self, plan):
        self._run(plan.pack_ops)
        self._run(plan.fwd_ops)
        self.grad.zero_()
        self._run(plan.bwd_ops)

    def _capture(self, plan):
        """One CUDA graph per plan holds the whole step: pack + forward + backward, the gradient all-reduce
        (data parallel; captured through our own NCCL communicator) and the optimiser.  MPNN_DIST_GRAPH=0
        keeps the collective out of capture: two graphs (compute | optimiser) with the all-reduce issued
        eagerly in between."""
        s = torch.cuda.Stream(self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        keep = (self.theta.clone(), self.accum.clone(), self.state.clone())
        with torch.cuda.stream(s):               # warm-up: allocations, lazy module loads
            self._compute_ops(plan)
            self._run(plan.opt_ops)
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        self.theta.copy_(keep[0]); self.accum.copy_(keep[1]); self.state.copy_(keep[2])
        g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        before = self.L.launches
        one_graph = (not self.dist) or self.graph_collective or self.fused_dp
        if self.dist and self.comm is None and not self.fused_dp:
            self._init_comm()
        if self.dist and not self.fused_dp:
            with torch.cuda.stream(s):           # the communicator's first collective (channel setup) stays out of capture
                self._allreduce()
            torch.cuda.synchronize(self.dev)
        with _gc_off():
            if one_graph:
                # the whole step is ONE graph: with our own communicator the NCCL launch is captured like any kernel
                with torch.cuda.graph(g1):
                    self._compute_ops(plan)
                    if self.dist and not self.fused_dp:
                        self._allreduce(0, plan.ar_split)
                    self._run(plan.opt_ops)
                g2 = None
            else:
                with torch.cuda.graph(g1):
                    self._compute_ops(plan)
                with torch.cuda.graph(g2):
                    self._run(plan.opt_ops)
        plan.graph_launches = self.L.launches - before
        self._graphs[id(plan)] = (g1, g2)
        return self._graphs[id(plan)]

    def forward(self, feed, mode=None):
        """Forward only; returns the plan (buffers hold the results)."""
        net = self.net
        mode = feed.get(net.mode, 'ev') if mode is None else mode
        B = self._batch_of(feed)
        plan = self._plan(B, mode == 'tr', False)
        with torch.cuda.device(self.dev):
            self._feed(plan, feed, False)
            self._run(plan.pack_ops)
            self._run(plan.fwd_ops)
        return plan

    def eval_stats(self, feed):
        """state_tensors of train-nets:111-130 for one batch (numpy)."""
        net = self.net
        plan = self.forward(feed)
        B = plan.B
        torch.cuda.synchronize(self.dev)
        y = plan.y.cpu().numpy().astype(np.float64)
        if self.dynamic:
            p_ev = plan.p_ev.cpu().numpy().astype(np.float64)
            p_tr = plan.p_tr.cpu().numpy().astype(np.float64)
        else:
            p_ev = np.ones((len(self.nodes), B))
            p_tr = None
        out = {}
        acc = np.zeros(B)
        moc = np.zeros(B)
        for nd in self.nodes:
            ops = nd.layer.n_ops + (nd.router.n_ops if nd.router is not None else 0)
            moc += p_ev[nd.idx] * ops
        for nd in self.regs:
            l = nd.layer
            d_cor = plan.reg[nd.idx].d_cor.cpu().numpy().astype(np.float64)
            c_err = plan.reg[nd.idx].c_err.cpu().numpy().astype(np.float64)
            pe = p_ev[nd.idx]
            acc += pe * d_cor
            out[(l, 'p_cor')] = pe * d_cor
            out[(l, 'p_inc')] = pe * (1 - d_cor)
            out[(l, 'p_cor_by_cls')] = (pe * d_cor)[:, None] * y
            out[(l, 'p_inc_by_cls')] = (pe * (1 - d_cor))[:, None] * y
            if p_tr is not None:
                out[(l, 'p_tr')] = p_tr[nd.idx]
            out[(l, 'c_err')] = c_err
        for nd in self.switches:
            r = plan.rtr[nd.idx].R.cpu().numpy().astype(np.float64)
            out[(nd.layer, 'x_rte')] = np.abs(r).mean(1)
        out[(net, 'acc')] = acc
        out[(net, 'moc')] = moc
        return out

    def debug_forward(self, feed, mode='tr'):
        """Internal tensors of one forward for the parity tests (numpy, by node index)."""
        plan = self.forward(feed, mode)
        torch.cuda.synchronize(self.dev)
        res = Ns(logits={}, c_err={}, d_cor={}, R={}, p_tr=None, p_ev=None, dec=None, plan=plan)
        for nd in self.regs:
            res.logits[nd.idx] = plan.reg[nd.idx].Z.cpu().numpy()
            res.c_err[nd.idx] = plan.reg[nd.idx].c_err.cpu().numpy()
            res.d_cor[nd.idx] = plan.reg[nd.idx].d_cor.cpu().numpy()
        for nd in self.switches:
            res.R[nd.idx] = plan.rtr[nd.idx].R.cpu().numpy()
        if self.dynamic:
            res.p_tr = plan.p_tr.cpu().numpy()
            res.p_ev = plan.p_ev.cpu().numpy()
            res.dec = plan.dec.cpu().numpy()
        return res

    def c_tot(self, plan):
        """Value of the training objective for the plan's last forward+backward
        (data term from the route kernel + L2 terms; logging / tests only)."""
        B = plan.B
        if self.dynamic:
            data = float(plan.c_data.double().mean())
            w = plan.p_tr.double().mean(1)
        else:
            data = float(sum(plan.reg[nd.idx].c_err.double().mean() for nd in self.regs))
            w = torch.ones(len(self.nodes), dtype=torch.float64, device=self.dev)
        for idx, sc in plan.activity:               # per-example ActivityError costs, weighted like the node's c_mod
            data += float((sc.c_act.double() * (plan.p_tr[idx].double() if self.dynamic else 1.0)).mean())
        mod = 0.0
        seg_l2 = self.seg_l2.cpu().numpy(); seg_node = self.seg_node.cpu().numpy()
        for s, p in enumerate(self.tparams):
            if seg_l2[s] > 0:
                mod += float(w[seg_node[s]]) * seg_l2[s] * float((self._buf(p).double() ** 2).sum())
        return data + mod


class _Plan:
    """Buffers + launch list for one (batch size, BN mode, needs-backward)."""

    def __init__(self, eng, B, bn_train, need_bwd):
        self.eng, self.B, self.bn_train, self.need_bwd = eng, B, bn_train, need_bwd
        self.pack_ops, self.fwd_ops, self.bwd_ops, self.opt_ops = [], [], [], []
        self.graph_launches = 0
        self._build()

    @staticmethod
    def _tag(fn, kind, flops=0.0, nbytes=0.0, desc=''):
        """algorithmic work of one launch (bench.py roofline); untagged ops are 'misc'"""
        fn.kind, fn.flops, fn.nbytes, fn.desc = kind, float(flops), float(nbytes), desc
        if kind == 'conv_wgrad':
            fn.lane = 2

    @staticmethod
    def _after(op, *deps):
        """op must run after deps (ops possibly on other lanes)"""
        deps = [d for d in deps if d is not None]
        op.deps = list(getattr(op, 'deps', ())) + deps
        for d in deps:
            d.signal = True
        return op

    # -- allocation helpers ------------------------------------------------ #
    # Every buffer of a plan is a view into a few large zero-filled arenas (bump allocation, 256-byte
    # aligned): a plan has ~450 buffers, and one torch.zeros each was ~450 fill launches in front of
    # the first step (they also hid the step's own kernels from a launch-count-limited profiler).
    _ESZ = {torch.float32: 4, torch.bfloat16: 2, torch.float64: 8, torch.int32: 4, torch.int64: 8, torch.uint8: 1}

    def zeros(self, shape, dtype):
        shape = tuple(int(v) for v in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        n = 1
        for v in shape:
            n *= v
        nbytes = _ru(max(n, 1) * self._ESZ[dtype], 256)
        if getattr(self, '_arena', None) is None or self._arena_off + nbytes > self._arena.numel():
            chunk = max(nbytes, (256 << 20) if self.B > 512 else (32 << 20))
            self._arena = torch.zeros(chunk, dtype=torch.uint8, device=self.eng.dev)
            self._arena_off = 0
            self.arenas = getattr(self, 'arenas', []) + [self._arena]
        raw = self._arena[self._arena_off:self._arena_off + n * self._ESZ[dtype]]
        self._arena_off += nbytes
        return raw.view(dtype).view(shape)

    def planes(self, C, geo):
        return self.zeros((C // 8, geo.P, 8), self.eng.tdtype)

    def _acc_f(self, n):
        """fp64 accumulator of deferred forward BN statistics: a slice of one pool that a single memset at the head
        of the step clears (the deferred protocol does not clean up after itself)"""
        if getattr(self, '_accpool', None) is None:
            self._accpool = self.zeros(1 << 14, torch.float64)
            self._accpool_off = 0
            pool = self._accpool
            self.pack_ops.append(lambda: pool.zero_())
        off = self._accpool_off
        n = _ru(n, 2)
        if off + n > self._accpool.numel():
            raise RuntimeError('engine: BN accumulator pool exhausted')
        self._accpool_off = off + n
        return self._accpool[off:off + n]

    def _image_slot(self):
        """pseudo parent of a Conv chain at the root: the input image as one padded-planes tensor"""
        if getattr(self, '_img', None) is None:
            eng, L, B = self.eng, self.eng.L, self.B
            H0, W0, C0 = eng.net.hypers.x0_shape
            cpad = _ru(C0, 16 if (eng.dtype == BF16 or eng.split) else 8)
            geo = Geo(B, H0, W0)
            t = self.planes(cpad, geo)
            slot = Ns(t=t, C=cpad, Creal=C0, geo=geo, dact=None, writers=0, sc=None, consumers=0, fused_red=False,
                      split=None, split_op=None)
            # (planes beyond the image's channels stay at their one-time zero fill: only the live ones are written)
            pk = lambda: L.pack_input(_vp(self.x0), B, H0, W0, C0, 1, _vp(t), min(cpad, _ru(C0, 8)), geo.G, geo.P, eng.dtype, eng.stream)
            pk.lane = 3
            self.fwd_ops.append(pk)
            if eng.split:
                slot.split, slot.split_op = self._split(t, cpad, geo, 3)
            self._img = Ns(out=[slot], needs_grad=False)
        return self._img

    def _split(self, t, C, geo, lane, ops=None):
        """bf16x3 / bf16x6 modes: (hi | lo) or (hi | mid | lo) bf16 copy of an fp32 planes tensor and the launch
        that fills it"""
        eng, L = self.eng, self.eng.L
        dst = self.zeros((eng.split * C // 8, geo.P, 8), torch.bfloat16)
        fn = L.split_planes3 if eng.split == 3 else L.split_planes

        def sp():
            fn(_vp(t), C, geo.P, _vp(dst), eng.stream)
        self._tag(sp, 'split', nbytes=C * geo.P * (4 + 2 * eng.split))
        sp.lane = lane
        (self.fwd_ops if ops is None else ops).append(sp)
        return dst, sp

    def f32(self, *shape):
        return self.zeros(shape, torch.float32)

    def _build(self):
        eng, L, B = self.eng, self.eng.L, self.B
        net = eng.net
        dt, impl = eng.dtype, eng.impl
        dev = eng.dev
        train, bwd = self.bn_train, self.need_bwd
        H0, W0, C0 = net.hypers.x0_shape
        n_cls = net.hypers.y_shape[0]
        self.x0 = self.f32(B, H0, W0, C0)
        self.y = self.f32(B, n_cls)
        self.kcpt = self.f32(B)
        self.kextra = self.f32(B)
        S = lambda: eng.stream
        # fully-connected heads on the tensor cores (bf16/tcgen05 mode): one GEMM per conv stage
        # computes the LogReg logits and the first router layer from the shared feature matrix
        def head_features(nd):              # inputs of the heads of a stage: its coarsest (or only) output, flattened
            x = nd.layer.x
            x = x[-1] if isinstance(x, (list, tuple)) else x
            return int(np.prod(x.shape))
        with_heads = [nd for nd in eng.nodes if nd.kind == 'rcm' and (
            nd.router is not None or any(eng.nodes[k].kind == 'reg' for k in nd.kids))]
        # the head GEMM keeps [W_leaf | W_r1] resident in shared memory: F/8 x 32 x 16 bytes must fit (F = 2048 at the
        # reference architecture; a Conv chain at full resolution has F = H*W*C and takes the CUDA-core heads)
        # a wider head (N = 16 + W = 48 or 80) is split over blockIdx.y into slices of 16 columns (stencil_umma.cu), so
        # the same bound holds for every router width
        fits = all((head_features(nd) + 16) // 8 * 32 * 16 <= 150 * 1024 for nd in with_heads)
        self.umma_heads = eng.impl == 1 and all(nd.fc.hypers.n_chan <= 16 for nd in eng.regs) and not eng.split and fits
        Balloc = _ru(B, 128) if self.umma_heads else _ru(B, 8)
        self.Balloc = Balloc
        self.node = {}
        self.reg, self.rtr, self.heads = {}, {}, {}
        self.pack_list, self.rt_fwd, self.keep, self.kplanes = [], [], [], []
        self.last_head_op = None
        self.head_ops = []
        self.activity = []                       # (node, scale) pairs that carry an ActivityError cost
        cpad_q = 16 if (dt == BF16 or eng.split) else 8
        dyn_k = eng.dynamic and bool(net.hypers.dyn_k_cpt)

        # ---------------- forward ---------------- #
        for nd in eng.nodes:
            lay = nd.layer
            st = Ns()
            self.node[nd.idx] = st
            if nd.kind == 'pyr':
                n_sc = _comps(lay)[0].hypers.n_scales
                cpad = _ru(C0, cpad_q)
                st.out = []
                for i in range(n_sc):
                    geo = Geo(B, H0 // 2 ** i, W0 // 2 ** i)
                    t = self.planes(cpad, geo)
                    st.out.append(Ns(t=t, C=cpad, Creal=C0, geo=geo, dact=None, writers=0, sc=None, consumers=0, fused_red=False,
                                     split=None, split_op=None))
                    if getattr(nd, 'lln', None) is not None:
                        # MultiscaleLLN behind ToPyramid: normalise the scale in fp32 NHWC, then pack that
                        tmp = self.f32(B, geo.H, geo.W, C0)

                        def lln(i=i, tmp=tmp, hy=nd.lln.hypers):
                            L.lln(_vp(self.x0), B, H0, W0, C0, 2 ** i, float(hy.σ), float(hy.ϵ), _vp(tmp), S())
                        lln.lane = 3 + i
                        self.fwd_ops.append(lln)
                    # channel planes beyond the image's own (padding to the MMA's K = 16) are never written after the
                    # arena's zero fill: pack only the live planes (half of the bytes for a 3-channel image)
                    clive = min(cpad, _ru(C0, 8))
                    if getattr(nd, 'lln', None) is not None:
                        pk = lambda t=t, geo=geo, tmp=tmp: L.pack_input(
                            _vp(tmp), B, geo.H, geo.W, C0, 1, _vp(t), clive, geo.G, geo.P, dt, S())
                    else:
                        pk = lambda t=t, i=i, geo=geo: L.pack_input(
                            _vp(self.x0), B, H0, W0, C0, 2 ** i, _vp(t), clive, geo.G, geo.P, dt, S())
                    pk.lane = 3 + i
                    self.fwd_ops.append(pk)
                    if eng.split:
                        st.out[-1].split, st.out[-1].split_op = self._split(t, cpad, geo, 3 + i)
                st.needs_grad = False
            elif nd.kind == 'rcm':
                self._build_rcm_fwd(nd, st, Balloc)
            elif nd.kind == 'reg':
                par = self.node[nd.parent]
                fc = nd.fc
                n_out = fc.hypers.n_chan           # = n_cls, or the number of superclasses
                eps = float(nd.ce.hypers.ε) if nd.loss != 'sq' else 0.0
                if self.umma_heads:
                    hd = self.heads[nd.parent]          # logits come from the parent's head GEMM
                    r = Ns(Zbuf=hd.Z16, Z=hd.Z16[:, :n_out], ldz=16, prob=self.f32(B, n_out),
                           c_err=self.f32(B), d_cor=self.f32(B), dZ=None, fc=fc, eps=eps)
                else:
                    zb = self.f32(B, n_out)
                    r = Ns(Zbuf=zb, Z=zb, ldz=n_out, prob=self.f32(B, n_out), c_err=self.f32(B),
                           d_cor=self.f32(B), dZ=self.f32(B, n_out) if bwd else None, fc=fc, eps=eps)
                    F = par.F
                    fcf = lambda par=par, r=r, fc=fc, F=F, n_out=n_out: L.fc_fwd(
                        _vp(par.feat), F, Balloc, B, eng.tptr(fc.params.w), eng.tptr(fc.params.b), None,
                        n_out, _vp(r.Zbuf), dt, S())
                    self.fwd_ops.append(self._after(fcf, getattr(par, 'feat_op', None)))
                r.n, r.loss, r.y = n_out, nd.loss, self.y
                if nd.loss == 'sce':
                    # SuperclassCrossEntropyError (lib/layer_types.py:274-285): the targets are y @ w_cls, refreshed
                    # with the labels at the head of every step
                    w_cls = torch.tensor(nd.w_cls, dtype=torch.float32, device=eng.dev)
                    r.y = self.f32(B, n_out)
                    self.keep.append(w_cls)
                    self.pack_ops.append(lambda r=r, w_cls=w_cls, n_out=n_out: L.superclass_targets(
                        _vp(self.y), _vp(w_cls), B, n_cls, n_out, _vp(r.y), S()))
                self.reg[nd.idx] = r
                if nd.loss == 'sq':                    # SquaredError on the LinTrans output; r.prob keeps that output
                    ce = lambda r=r: L.squared_err_fwd(
                        _vp(r.Zbuf), r.ldz, _vp(r.y), B, r.n, _vp(r.prob), _vp(r.c_err), _vp(r.d_cor), S())
                else:
                    ce = lambda r=r: L.softmax_ce_fwd(
                        _vp(r.Zbuf), r.ldz, _vp(r.y), B, r.n, r.eps, _vp(r.prob), _vp(r.c_err), _vp(r.d_cor), S())
                if self.umma_heads:
                    ce.lane = hd.lane                 # follows its head GEMM on that head's lane
                    self.last_head_op = ce
                    self.head_ops.append(ce)
                self.fwd_ops.append(ce)
            if nd.router is not None:
                self._build_router_fwd(nd, Balloc, dyn_k, emit_fc=not self.umma_heads)
            if nd.kind == 'rcm' and self.umma_heads and getattr(st, 'feat', None) is not None:
                self._build_heads_fwd(nd, st, dyn_k)

        # ---------------- routers (all tails in one launch), routing ---------------- #
        if self.rt_fwd:
            bn0 = self.rtr[eng.switches[0].idx].bn1
            for sw in eng.switches:       # the batched tail launch takes ONE (d, eps) for every router BatchNorm
                for bn in (self.rtr[sw.idx].bn1, self.rtr[sw.idx].bn2):
                    if (float(bn.hypers.d), float(bn.hypers.ε)) != (float(bn0.hypers.d), float(bn0.hypers.ε)):
                        raise NotImplementedError(
                            'engine: router BatchNorm hypers differ between routers (%r: d=%r, eps=%r vs d=%r, eps=%r)'
                            % (sw.layer.name, bn.hypers.d, bn.hypers.ε, bn0.hypers.d, bn0.hypers.ε))
            tab = self._desc_table(_RT_FWD, self.rt_fwd)
            self.keep.append(tab)
            tails = lambda: L.router_tail_fwd_batched(
                _vp(tab), len(self.rt_fwd), B, eng.router_width, float(bn0.hypers.d), float(bn0.hypers.ε),
                1 if self.bn_train else 0, S())
            # the tails need the head GEMMs that write a router's first layer -- not the classifiers' losses, and not the
            # head of a stage without a router (the last stage: its GEMM and loss then run beside the tails and the
            # routing walk instead of in front of them; the backward list starts when every lane has drained)
            feeders = [op for op in self.head_ops if getattr(op, 'feeds_router', False)]
            if os.environ.get('MPNN_TAILS_WAIT_ALL', '0') != '0':      # A/B switch: the round-2 dependency (every head op)
                feeders = []
            self.fwd_ops.append(self._after(tails, *(feeders or self.head_ops or [self.last_head_op])))
        if eng.dynamic:
            self._build_routing()

        if not bwd:
            self._finish_pack()
            return
        # ---------------- backward ---------------- #
        if eng.dynamic:
            hy = net.hypers
            self.bwd_ops.append(lambda: L.route_bwd(
                _vp(self.t_parent), _vp(self.t_sink), _vp(self.t_nsinks), _vp(self.t_child), _vp(self.t_floor),
                _vp(self.t_sw), _vp(self.t_ops), _vp(self.t_err), len(eng.nodes), _vp(self.R_tab), _vp(eng.hyp), B,
                _vp(self.p_tr), _vp(self.p_ev), _vp(self.cerr_tab), _vp(self.dcor_tab),
                _vp(self.kcpt) if dyn_k else None,
                1 if eng.critic else 0, float(getattr(hy, 'k_dec', 0.0)), float(getattr(hy, 'k_cre', 0.0)),
                1 if getattr(hy, 'optimistic', False) else 0, 1 if getattr(hy, 'use_cls_err', False) else 0,
                _vp(self.dR_tab), _vp(self.route_scratch), _vp(self.c_data), S()))
            moments = lambda: L.node_moments(
                _vp(self.p_tr), len(eng.nodes), B, _vp(eng.grad), S())
            moments.lane = 8                     # only the optimiser reads the TALR moments: off the chain
            self.bwd_ops.append(moments)
            if eng.switches:
                # every dR is known right after route_bwd: all router tails backward in one launch
                rows = [self._router_bwd_desc(nd) for nd in eng.switches]
                tabb = self._desc_table(_RT_BWD, rows)
                self.keep.append(tabb)
                self.bwd_ops.append(lambda: L.router_tail_bwd_batched(_vp(tabb), len(rows), B, eng.router_width, S()))
        main_ops = [op for op in self.bwd_ops if getattr(op, 'lane', 0) == 0]
        self.bwd_head_dep = main_ops[-1] if main_ops else None             # routing gradients are complete
        # data parallel: the gradients of the DEEP stages are complete long before the backward pass ends (it
        # runs deepest-first) and they are most of the parameters (stages 4-7: 80 % of the conv weights).  Their
        # all-reduce goes out on its own lane as soon as every launch that writes them has been issued, and
        # overlaps the backward pass of the shallow stages; the rest [moments | shallow stages] follows the
        # backward list.  Split = first parameter of the conv stage nearest to half of the parameters.
        self.ar_split = None                     # None: one all-reduce over the whole buffer
        split_node = None
        if eng.dist and eng.overlap_allreduce:
            offs = {}
            for sidx, p in enumerate(eng.tparams):
                offs.setdefault(eng.seg_node_list[sidx], p._bind[2])          # first parameter of each node
            best = None
            for cand in eng.nodes:
                if cand.kind != 'rcm' or cand.idx not in offs:
                    continue
                # a classifier's gradients are written by its PARENT's head launches: every node of the deep
                # bucket must have its parent in the bucket too (except the split node itself)
                if any(o.idx > cand.idx and o.parent is not None and o.parent < cand.idx for o in eng.nodes):
                    continue
                frac = offs[cand.idx] / max(eng.n_theta, 1)                   # share of the parameters in FRONT of it
                if 0.1 <= frac <= 0.6 and (best is None or abs(frac - 0.3) < abs(best[0] - 0.3)):
                    best = (frac, cand)
            if best is not None:
                split_node = best[1]
                self.ar_split = eng.g0 + offs[split_node.idx]
        for nd in reversed(eng.nodes):
            if nd.kind == 'reg':
                r = self.reg[nd.idx]
                par = self.node[nd.parent]
                coef = (lambda nd=nd: ctypes.c_void_p(self.p_tr.data_ptr() + 4 * nd.idx * B)) if eng.dynamic \
                    else (lambda: None)
                if self.umma_heads:
                    hd = self.heads[nd.parent]
                    dzp = ctypes.c_void_p(hd.dZ.data_ptr() + (hd.leaf_off // 8) * Balloc * 16)
                    ceb = lambda r=r, coef=coef, dzp=dzp: self._loss_bwd(r, coef(), None, dzp, eng.gptr(r.fc.params.b))
                    ceb.lane = hd.lane
                    # a stage without a router only needs p_tr (forward): its head gradients are issued
                    # ahead of the routing backward so the deepest conv chain starts under it
                    ceb.early = eng.nodes[nd.parent].router is None
                    hd.ceb_op = ceb
                    self.bwd_ops.append(ceb if ceb.early else self._after(ceb, self.bwd_head_dep))
                else:
                    self.bwd_ops.append(lambda r=r, coef=coef: self._loss_bwd(r, coef(), _vp(r.dZ), None, None))
                    self.bwd_ops.append(lambda r=r, par=par: L.fc_bwd_weight(
                        _vp(par.feat), par.F, Balloc, B, None, _vp(r.dZ), r.n,
                        eng.gptr(r.fc.params.w), eng.gptr(r.fc.params.b), dt, S()))
            if nd.router is not None and not self.umma_heads:
                self._build_router_bwd(nd, Balloc, dyn_k)
            if nd.kind == 'rcm':
                self._build_rcm_bwd(nd, Balloc)
            if split_node is not None and nd.idx == split_node.idx:
                if eng.fused_dp:
                    # the deep stages' slice of the fused tail (reduce + TALR / momentum + all-gather) on its own
                    # flag channel, under the rest of the backward pass: nothing issued later in the step reads
                    # those parameters (convs read the copies packed at the head of the step, and every launch
                    # that reads a deep-stage parameter directly also writes one of its gradients)
                    def ar_deep():
                        self._p2p_tail(self.ar_split - eng.g0, 0, 1)
                else:
                    def ar_deep():
                        eng._allreduce(self.ar_split, None, stream=S())
                ar_deep.kind, ar_deep.lane, ar_deep.wait_all = 'allreduce', 20, True
                self.bwd_ops.append(ar_deep)
        early = [op for op in self.bwd_ops if getattr(op, 'early', False)]
        self.bwd_ops = early + [op for op in self.bwd_ops if not getattr(op, 'early', False)]
        # ---------------- optimiser ---------------- #
        talr = 1 if (eng.dynamic and bool(net.hypers.talr)) else 0
        stats_ptr = (lambda: _vp(eng.grad)) if eng.dynamic else (lambda: None)
        if eng.fused_dp:
            # reduce-scatter + TALR / momentum + all-gather over peer memory in ONE launch (csrc/p2p.cu); with the
            # overlapped schedule the deep stages went out earlier (ar_deep) and this is [moments | shallow stages]
            talr_, dyn_ = talr, 1 if eng.dynamic else 0

            def p2p_tail(lo, hi, channel):
                L.allreduce_talr_p2p(ctypes.c_void_p(eng._p2p_desc.ctypes.data), _vp(eng.seg_start), _vp(eng.seg_node),
                                     _vp(eng.seg_mult), _vp(eng.seg_l2), eng.n_seg, dyn_, talr_, _vp(eng.hyp), 1,
                                     lo, hi, channel, S())
            self._p2p_tail = p2p_tail
            fused = lambda: p2p_tail(0, (self.ar_split - eng.g0) if self.ar_split is not None else 0, 0)
            self._tag(fused, 'allreduce_talr_p2p')
            self.opt_ops.append(fused)
        else:
            self.opt_ops.append(lambda: L.talr_momentum_step(
                _vp(eng.theta), ctypes.c_void_p(eng.grad.data_ptr() + 4 * eng.g0), _vp(eng.accum), eng.n_theta,
                _vp(eng.seg_start), _vp(eng.seg_node),
                _vp(eng.seg_mult), _vp(eng.seg_l2), eng.n_seg, stats_ptr(), talr, _vp(eng.hyp), S()))
        self._finish_pack()

    # -- descriptor tables (device arrays of C structs, see include/mpnn.h) -- #
    def _desc_table(self, dtype, rows):
        arr = np.zeros(len(rows), dtype=dtype)
        for i, row in enumerate(rows):
            for k, v in row.items():
                if isinstance(v, ctypes.c_void_p):
                    v = v.value or 0
                elif isinstance(v, torch.Tensor):
                    v = v.data_ptr()
                arr[i][k] = 0 if v is None else v
        return torch.from_numpy(arr.view(np.uint8).copy()).to(self.eng.dev)

    def _finish_pack(self):
        """one launch packs every conv weight tensor of the step (fwd + dgrad operands)"""
        if not self.pack_list:
            return
        eng, L = self.eng, self.eng.L
        tab = self._desc_table(_PACK, self.pack_list)
        self.keep.append(tab)
        n = len(self.pack_list)
        self.pack_ops.append(lambda: L.pack_weights_batched(_vp(tab), n, eng.pack_blocks, BF16 if eng.split else eng.dtype, eng.stream))

    def _pack(self, param, packed, I, O, mode, k_off, Ktot, n_off, Ntot, ntaps=9):
        """mode 0: forward operand, 1: dgrad operand (transposed, taps flipped), 2: fp32 vector copy"""
        self.pack_list.append(dict(w=self.eng.tptr(param), packed=packed, ntaps=ntaps, I=I, O=O, mode=mode,
                                   k_off=k_off, Ktot=Ktot, n_off=n_off, Ntot=Ntot))

    # -- fully-connected heads on the tensor cores ---------------------------- #
    def _build_heads_fwd(self, nd, st, dyn_k):
        """One tcgen05 GEMM per conv stage: [LogReg logits | first router layer] = X @ [W_leaf | W_r1] + b
        (lib/layer_types.py:39-53 twice, sharing the flattened coarsest scale X)."""
        eng, L, B, Balloc = self.eng, self.eng.L, self.B, self.Balloc
        S = lambda: eng.stream
        n_cls = eng.net.hypers.y_shape[0]
        leaves = [k for k in nd.kids if eng.nodes[k].kind == 'reg']
        if len(leaves) > 1:
            raise NotImplementedError('engine: more than one LogReg under one node')
        rt = self.rtr.get(nd.idx)
        W = eng.router_width
        hd = Ns(leaf_off=0 if leaves else None, r_off=(16 if leaves else 0) if rt is not None else None)
        hd.N = 16 * bool(leaves) + (W if rt is not None else 0)
        # heads only feed the losses / the routers: off the conv lanes, and spread over a few lanes of their own so
        # that a head never queues behind the head of another stage
        hd.lane = 1 if eng.head_lanes == 1 else 21 + len(self.heads) % eng.head_lanes
        F, Fext = st.F, st.Fext
        hd.Z16 = self.f32(B, 16) if leaves else None
        hd.Wfc = self.zeros((1, Fext // 8, hd.N, 8), eng.tdtype)
        hd.bias = self.f32(hd.N)
        hd.dZ = self.zeros((hd.N // 8, Balloc, 8), eng.tdtype) if self.need_bwd else None
        if leaves:
            fc = eng.nodes[leaves[0]].fc
            hd.fc_leaf = fc
            self._pack(fc.params.w, hd.Wfc, F, fc.hypers.n_chan, 0, 0, Fext, hd.leaf_off, hd.N, ntaps=1)
            self._pack(fc.params.b, hd.bias, 1, fc.hypers.n_chan, 2, 0, 8, hd.leaf_off, hd.N, ntaps=1)
        if rt is not None:
            rows = F + (1 if dyn_k else 0)
            self._pack(rt.fc1.params.w, hd.Wfc, rows, W, 0, 0, Fext, hd.r_off, hd.N, ntaps=1)
            self._pack(rt.fc1.params.b, hd.bias, 1, W, 2, 0, 8, hd.r_off, hd.N, ntaps=1)
        outs = [(hd.Z16, 16)] if leaves else []
        if rt is not None:
            outs.append((rt.Z1, W))
        outs.append((None, 0))
        (o0, n0), (o1, n1) = outs[0], outs[1]
        self.heads[nd.idx] = hd

        def gemm():
            L.stencil_gemm(_vp(st.feat), Fext, None, 0, _vp(hd.Wfc), 1, _vp(hd.bias), _vp(o0), n0, 0, _vp(o1), n1, 0,
                           B, 0, 0, 0, Balloc, None, 0, None, BF16, 2, 1, S())
        self._tag(gemm, 'fc_fwd', desc='F%d N%d' % (Fext, hd.N), flops=2.0 * B * F * hd.N, nbytes=B * F * 2)
        gemm.lane = hd.lane
        gemm.feeds_router = rt is not None
        self._after(gemm, getattr(st, 'feat_op', None))
        self.last_head_op = gemm
        self.head_ops.append(gemm)
        self.fwd_ops.append(gemm)

    def _loss_bwd(self, r, coef, dZ, dZp, dbias):
        """gradient of a leaf's error layer wrt the LinTrans output (fp32 rows and / or the bf16 planes operand)"""
        L, B = self.eng.L, self.B
        if r.loss == 'sq':
            L.squared_err_bwd(_vp(r.prob), _vp(r.y), B, r.n, coef, 1.0 / B, dZ, dZp, self.Balloc if dZp else 0,
                              dbias, self.eng.stream)
        else:
            L.softmax_ce_bwd(_vp(r.prob), _vp(r.y), B, r.n, r.eps, coef, 1.0 / B, dZ, dZp,
                             self.Balloc if dZp else 0, dbias, self.eng.stream)

    def _build_heads_bwd(self, nd, st, dyn_k):
        eng, L, B, Balloc = self.eng, self.eng.L, self.B, self.Balloc
        S = lambda: eng.stream
        n_cls = eng.net.hypers.y_shape[0]
        hd = self.heads[nd.idx]
        rt = self.rtr.get(nd.idx)
        F, Fext = st.F, st.Fext
        leaf = getattr(hd, 'fc_leaf', None)
        # weight gradients of both heads in one launch
        a = (eng.gptr(leaf.params.w), F, leaf.hypers.n_chan) if leaf is not None else (None, 0, 0)
        b = (eng.gptr(rt.fc1.params.w), F + (1 if dyn_k else 0), eng.router_width) if rt is not None else (None, 0, 0)
        if leaf is None:
            a, b = b, (None, 0, 0)
        nsplit = 16 if leaf is not None else hd.N           # columns of dZ that belong to the first head

        def wgrad():
            L.fc_wgrad(_vp(st.feat), Fext, Balloc, B, _vp(hd.dZ), hd.N, nsplit, a[0], a[1], a[2], b[0], b[1], b[2], S())
        self._tag(wgrad, 'fc_wgrad', desc='F%d N%d' % (Fext, hd.N), flops=2.0 * B * F * hd.N, nbytes=B * F * 2)
        wgrad.lane = 9                               # off the heads lane: the data gradient below is what the chain waits for
        wgrad.early = rt is None
        self._after(wgrad, getattr(hd, 'ceb_op', None))
        self.bwd_ops.append(wgrad if wgrad.early else self._after(wgrad, self.bwd_head_dep))
        # data gradient towards the flattened coarsest scale
        hd.Wfd = self.zeros((1, hd.N // 8, F, 8), eng.tdtype)
        if leaf is not None:
            self._pack(leaf.params.w, hd.Wfd, F, leaf.hypers.n_chan, 1, hd.leaf_off, hd.N, 0, F, ntaps=1)
        if rt is not None:
            self._pack(rt.fc1.params.w, hd.Wfd, F, eng.router_width, 1, hd.r_off, hd.N, 0, F, ntaps=1)
        st.dfeat = self.zeros((F // 8, Balloc, 8), eng.tdtype)

        def dgrad():
            L.stencil_gemm(_vp(hd.dZ), hd.N, None, 0, _vp(hd.Wfd), 1, None, _vp(st.dfeat), F, 0, None, 0, 0,
                           B, 0, 0, 0, Balloc, None, 0, None, BF16, BF16, 1, S())
        self._tag(dgrad, 'fc_dgrad', desc='N%d F%d' % (hd.N, F), flops=2.0 * B * F * hd.N, nbytes=B * F * 2)
        dgrad.lane = hd.lane
        dgrad.early = rt is None
        st.dfeat_op = dgrad                          # the conv chain of this node waits for it
        # the router half of dZ comes from the routing backward on lane 0 (normally already ordered through
        # the leaf's softmax gradient on this lane; explicit for stages that have a router but no leaf)
        self.bwd_ops.append(dgrad if dgrad.early else self._after(dgrad, self.bwd_head_dep))

    def _router_bwd_desc(self, nd):
        eng = self.eng
        rt = self.rtr[nd.idx]
        P = lambda lay, k: eng.tptr(getattr(lay.params, k))
        Gp = lambda lay, k: eng.gptr(getattr(lay.params, k))
        return dict(Z1=rt.Z1, Z2=rt.Z2, dR=rt.dR, g1=P(rt.bn1, 'γ'), b1=P(rt.bn1, 'β'), W2=P(rt.fc2, 'w'),
                    g2=P(rt.bn2, 'γ'), b2=P(rt.bn2, 'β'), W3=P(rt.fc3, 'w'), save=rt.save,
                    dg1=Gp(rt.bn1, 'γ'), dbt1=Gp(rt.bn1, 'β'), dW2=Gp(rt.fc2, 'w'), dbias2=Gp(rt.fc2, 'b'),
                    dg2=Gp(rt.bn2, 'γ'), dbt2=Gp(rt.bn2, 'β'), dW3=Gp(rt.fc3, 'w'), dbias3=Gp(rt.fc3, 'b'),
                    dZ1=rt.dZ1, scratch=rt.scratch, ns=rt.ns, Balloc=self.Balloc,
                    dZ1p=self._router_planes(nd), dbias1=Gp(rt.fc1, 'b') if self.umma_heads else None)

    def _router_planes(self, nd):
        """bf16 planes slot of dZ1 inside the node's head-gradient operand (tcgen05 heads only)"""
        if not self.umma_heads:
            return None
        hd = self.heads[nd.idx]
        return ctypes.c_void_p(hd.dZ.data_ptr() + (hd.r_off // 8) * self.Balloc * 16)

    # -- conv stage -------------------------------------------------------- #
    def _build_rcm_fwd(self, nd, st, Balloc):
        eng, L, B = self.eng, self.eng.L, self.B
        dt, impl = eng.dtype, eng.impl
        S = lambda: eng.stream
        lay = nd.layer
        cm, mbn = nd.cm, nd.mbn
        if nd.parent is None:                     # a Conv chain at the root: its input tensor is the image itself
            par = self._image_slot()
        else:
            par = self.node[nd.parent]
        n_chan = list(cm.hypers.n_chan)
        n = len(n_chan)
        if nd.sel is not None:                    # Select(i) + Conv: one scale of the pyramid
            pin = [par.out[nd.sel]]
        else:
            pin = par.out[len(par.out) - n:]
        st.pin = pin
        st.needs_grad = True
        st.out, st.sc = [], []
        kid_rcm = [k for k in nd.kids if eng.nodes[k].kind == 'rcm']
        has_heads = any(eng.nodes[k].kind == 'reg' for k in nd.kids) or nd.router is not None

        def live(k):
            for c in kid_rcm:
                m = len(eng.nodes[c].cm.hypers.n_chan)
                if k >= n - m:
                    return True
            return k == n - 1 and has_heads
        train, bwd = self.bn_train, self.need_bwd
        for k in range(n):
            src = pin[k]
            src.consumers += 1
            geo = src.geo
            N = n_chan[k]
            K0 = src.C
            K1 = n_chan[k - 1] if k > 0 else 0
            sc = Ns(k=k, geo=geo, N=N, K0=K0, K0real=src.Creal, K1=K1, src=src, live=live(k),
                    dpooled=None, geo_p=None)
            sc.lin = self.planes(N, geo)
            pooled_out = getattr(nd, 'maxpool', False)          # [Conv, BN, Rect, MaxPool]: the sinks see the pooled tensor
            gmp = getattr(nd, 'gmp', False)                     # the classifier below takes GlobalMaxPool features
            act_alpha = getattr(nd, 'act_alpha', 0.0)           # ActivityError behind the ReLU: a per-example cost
            sc.act = self.planes(N, geo) if pooled_out or gmp or act_alpha or any(
                k >= n - len(eng.nodes[c].cm.hypers.n_chan) for c in kid_rcm) else None
            sc.pooled = None
            if k < n - 1:
                sc.geo_p = pin[k + 1].geo
                sc.pooled = self.planes(N, sc.geo_p)
            sc.feat = None
            if k == n - 1 and has_heads:
                st.F = N if gmp else (geo.H // 2) * (geo.W // 2) * N if pooled_out else geo.H * geo.W * N
                # tcgen05 heads with a per-example k_cpt feature (net_types.py:149-160): the feature
                # alpha_cpt*k_cpt lives in channel 0 of one extra (16-aligned) pair of planes
                ext = 16 if (self.umma_heads and nd.router is not None and eng.dynamic
                             and bool(eng.net.hypers.dyn_k_cpt)) else 0
                st.Fext = st.F + ext
                sc.feat = self.zeros((st.Fext // 8, Balloc, 8), eng.tdtype)
                st.feat = sc.feat
                if ext:
                    self.kplanes.append(sc.feat[st.F // 8, :, 0])
                if pooled_out or gmp:
                    sc.feat = None                  # written by the pooling kernel (st.feat), not by BN / ReLU
            sc.Wf = None if eng.split else self.zeros((9, (K0 + K1) // 8, N, 8), eng.tdtype)
            sc.ss = self.f32(2, N)
            sc.mr = self.f32(2, N)
            sc.bn = mbn.comps[k]
            wh = getattr(cm.params, 'w_horz_%i' % k)
            wv = getattr(cm.params, 'w_vert_%i' % (k - 1)) if k > 0 else None
            bk = getattr(cm.params, 'b_%i' % k)
            sc.wh, sc.wv, sc.bk = wh, wv, bk
            if tuple(wh.shape[:2]) != (3, 3):
                raise NotImplementedError('engine: conv window %s' % (wh.shape[:2],))
            if not eng.split:
                self._pack(wh, sc.Wf, sc.K0real, sc.N, 0, 0, sc.K0 + sc.K1, 0, sc.N)
                if wv is not None:
                    self._pack(wv, sc.Wf, sc.K1, sc.N, 0, sc.K0, sc.K0 + sc.K1, 0, sc.N)
            prev = st.sc[k - 1] if k > 0 else None
            use_stats = sc.live and train
            if eng.split:
                self._build_conv_fwd_split(sc, prev, use_stats, B, Balloc, st)
                st.sc.append(sc)
                st.out.append(Ns(t=sc.act, C=N, Creal=N, geo=geo, dact=None, writers=0, sc=sc, consumers=0, fused_red=False,
                                 split=getattr(sc, 'act_split', None), split_op=getattr(sc, 'post_op', None)))
                continue

            # small tensors without a pooled output (the coarsest scale of a stage at the reference's batch): the conv
            # stores `lin` only, and ONE cluster launch takes the statistics and applies BN / ReLU (mpnn_bn_fwd_small)
            small_f = (use_stats and not eng.defer_bn and eng.bn_small and sc.pooled is None
                       and B * geo.H * geo.W <= _BN_SMALL_MAX_PIXELS and (sc.act is not None or sc.feat is not None))
            if use_stats and not small_f:
                # train-mode BN statistics ride on the conv launch (last CTA finalises): no bn_finalize
                bn = sc.bn
                sc.acc_f = self._acc_f(2 * N + 1) if eng.defer_bn else self.zeros(2 * N + 1, torch.float64)
                sc.bnf = _host_struct(_BN_FUSE, acc=_vp(sc.acc_f), gamma=eng.tptr(bn.params.γ), beta=eng.tptr(bn.params.β),
                                      m_avg=eng.tptr(bn.params.m_avg), v_avg=eng.tptr(bn.params.v_avg),
                                      ss=_vp(sc.ss), mr=_vp(sc.mr), count=float(B * geo.H * geo.W),
                                      d=float(bn.hypers.d), eps=float(bn.hypers.ε), defer=1 if eng.defer_bn else 0)

                def conv(sc=sc, prev=prev):
                    L.conv_bn_stats(_vp(sc.src.t), sc.K0, _vp(prev.pooled) if prev is not None else None, sc.K1,
                                    _vp(sc.Wf), eng.tptr(sc.bk), _vp(sc.lin), sc.N, *sc.geo.args(),
                                    ctypes.c_void_p(sc.bnf.ctypes.data), dt, impl, S())
            else:
                def conv(sc=sc, prev=prev):
                    L.stencil_gemm(_vp(sc.src.t), sc.K0, _vp(prev.pooled) if prev is not None else None, sc.K1,
                                   _vp(sc.Wf), 9, eng.tptr(sc.bk), _vp(sc.lin), sc.N, 0, None, 0, 0,
                                   *sc.geo.args(), None, 0, None, dt, dt, impl, S())
            self._tag(conv, 'conv_fwd', desc='H%d K%d+%d N%d' % (sc.geo.H, sc.K0, sc.K1, sc.N), flops=2.0 * B * sc.geo.H * sc.geo.W * 9 * (sc.K0real + sc.K1) * sc.N,
                      nbytes=B * sc.geo.H * sc.geo.W * (sc.K0 + sc.K1 + sc.N) * (2 if dt == BF16 else 4))
            sc.lane = 3 + int(round(np.log2(eng.net.hypers.x0_shape[0] / geo.H)))
            conv.lane = sc.lane
            self._after(conv, getattr(prev, 'post_op', None) if prev is not None else None)   # pooled input
            self._after(conv, getattr(src, 'op', None))        # a MaxPool-ed parent tensor comes from another lane
            self.fwd_ops.append(conv)
            if sc.live and not use_stats:
                bn = sc.bn

                def fin(sc=sc, bn=bn):             # inference: scale/shift from the running moments
                    L.bn_finalize(None, 0, sc.N,
                                  float(B * sc.geo.H * sc.geo.W), eng.tptr(bn.params.γ), eng.tptr(bn.params.β),
                                  eng.tptr(bn.params.m_avg), eng.tptr(bn.params.v_avg),
                                  float(bn.hypers.d), float(bn.hypers.ε), 0,
                                  _vp(sc.ss), _vp(sc.mr), S())
                self._tag(fin, 'bn_finalize')
                fin.lane = sc.lane
                self.fwd_ops.append(fin)
            if sc.live or sc.pooled is not None:
                if small_f:
                    def post(sc=sc, bn=sc.bn):
                        L.bn_fwd_small(_vp(sc.lin), sc.N, *sc.geo.args(), eng.tptr(bn.params.γ), eng.tptr(bn.params.β),
                                       eng.tptr(bn.params.m_avg), eng.tptr(bn.params.v_avg), float(bn.hypers.d),
                                       float(bn.hypers.ε), _vp(sc.ss), _vp(sc.mr), _vp(sc.act), _vp(sc.feat), Balloc, dt, S())
                elif use_stats and eng.defer_bn:
                    def post(sc=sc):
                        L.bn_relu_pool_fwd_acc(_vp(sc.lin), sc.N, *sc.geo.args(), ctypes.c_void_p(sc.bnf.ctypes.data),
                                               _vp(sc.act), _vp(sc.pooled), sc.geo_p.P if sc.pooled is not None else 0,
                                               _vp(sc.feat), Balloc, dt, S())
                else:
                    def post(sc=sc):
                        L.bn_relu_pool_fwd(_vp(sc.lin), sc.N, *sc.geo.args(), _vp(sc.ss) if sc.live else None,
                                           _vp(sc.act), _vp(sc.pooled), sc.geo_p.P if sc.pooled is not None else 0,
                                           _vp(sc.feat), Balloc, dt, S())
                self._tag(post, 'bn_fwd', desc='H%d C%d' % (sc.geo.H, sc.N), nbytes=B * sc.geo.H * sc.geo.W * sc.N * (2 if dt == BF16 else 4) * (1 + (sc.act is not None) + 0.25 * (sc.pooled is not None) + (sc.feat is not None)))
                post.lane = sc.lane
                sc.post_op = post
                self.fwd_ops.append(post)
                if sc.feat is not None:
                    st.feat_op = post
            st.sc.append(sc)
            sc.keep = getattr(nd, 'keep', 1.0)
            if sc.keep != 1.0:
                # Dropout behind the ReLU: the activations (and the flattened copy the heads read) are scaled in
                # place by m / keep; every sink sees the dropped tensor
                sc.drop_seed = (0x9E3779B9 * (nd.idx + 1)) & 0xFFFFFFFF

                def drop(sc=sc):
                    if sc.act is not None:
                        L.dropout(_vp(sc.act), sc.N, *sc.geo.args(), 0, 0, sc.keep, sc.drop_seed, _vp(eng.hyp), dt, S())
                    if sc.feat is not None:
                        L.dropout(_vp(sc.feat), sc.N, *sc.geo.args(), 1, Balloc, sc.keep, sc.drop_seed, _vp(eng.hyp), dt, S())
                drop.lane = sc.lane
                self.fwd_ops.append(drop)
                sc.post_op = drop
                if sc.feat is not None:
                    st.feat_op = drop
            sc.act_alpha = act_alpha
            if act_alpha:
                sc.c_act = self.f32(B)

                def acost(sc=sc):
                    L.activity_fwd(_vp(sc.act), sc.N, *sc.geo.args(), sc.act_alpha, _vp(sc.c_act), dt, S())
                acost.lane = sc.lane
                self.fwd_ops.append(acost)
                self.activity.append((nd.idx, sc))
            if pooled_out or gmp:
                # the features of the heads come from the pooling kernel, not from the BN / ReLU kernel
                # (sc.feat was cleared before `post` was built, see below)
                geo_q = Geo(B, geo.H // 2, geo.W // 2) if pooled_out else None
                sc.mp = Ns(feat=st.feat if has_heads else None, geo=geo_q,
                           out=self.planes(N, geo_q) if pooled_out and kid_rcm else None,
                           arg=self.zeros((N // 8, Balloc, 8), torch.int32) if gmp else None)
                if pooled_out:
                    def pool(sc=sc):
                        L.maxpool2_fwd(_vp(sc.act), sc.N, *sc.geo.args(), _vp(sc.mp.out), sc.mp.geo.P,
                                       _vp(sc.mp.feat), Balloc, dt, S())
                else:
                    def pool(sc=sc):
                        L.global_maxpool_fwd(_vp(sc.act), sc.N, *sc.geo.args(), _vp(sc.mp.feat), _vp(sc.mp.arg), Balloc, dt, S())
                self._tag(pool, 'pool_fwd', nbytes=B * geo.H * geo.W * N * (2 if dt == BF16 else 4) * 1.25)
                pool.lane = sc.lane
                self.fwd_ops.append(pool)
                if sc.mp.feat is not None:
                    st.feat_op = pool
                if pooled_out:
                    st.out.append(Ns(t=sc.mp.out, C=N, Creal=N, geo=geo_q, dact=None, writers=0, sc=None, consumers=0,
                                     fused_red=False, split=None, split_op=None, op=pool, dact_ops=[]))
                    continue
            st.out.append(Ns(t=sc.act, C=N, Creal=N, geo=geo, dact=None, writers=0, sc=sc, consumers=0, fused_red=False,
                             split=getattr(sc, 'act_split', None), split_op=getattr(sc, 'post_op', None)))

    def _build_conv_fwd_split(self, sc, prev, use_stats, B, Balloc, st):
        """bf16x3 mode: the conv of one scale as up to two tcgen05 launches over (hi | lo) operands --
        horizontal input, then the pooled predecessor accumulated on top -- with fp32 planes out; the BN moments
        ride on the last launch.  Followed by the fp32 BN / ReLU / pool kernel and the splits of what it wrote."""
        eng, L = self.eng, self.eng.L
        S = lambda: eng.stream
        geo, N, K0, K1 = sc.geo, sc.N, sc.K0, sc.K1
        sc.lane = 3 + int(round(np.log2(eng.net.hypers.x0_shape[0] / geo.H)))

        # launches of one source tensor as (parts of A0, parts of A1, weight parts along K): x3 = one launch
        # [hi | lo | hi] x [hi; hi; lo]; x6 = two launches [hi | mid | lo] x [hi; hi; hi] and
        # [hi | mid | hi] x [mid; mid; lo] (pack modes: 0 = hi, 4 = first residual, 8 = second residual)
        passes = _SPLIT_PASSES[eng.split]

        def packs(w, K, Kreal):
            out = []
            for _, _, wparts in passes:
                W3 = self.zeros((9, 3 * K // 8, N, 8), torch.bfloat16)
                for j, mode in enumerate(wparts):
                    self._pack(w, W3, Kreal, N, mode, j * K, 3 * K, 0, N)
                out.append(W3)
            return out
        sc.W3h = packs(sc.wh, K0, sc.K0real)
        sc.W3v = packs(sc.wv, K1, K1) if sc.wv is not None else None
        bnp = None
        if use_stats:
            bn = sc.bn
            sc.acc_f = self._acc_f(2 * N + 1) if eng.defer_bn else self.zeros(2 * N + 1, torch.float64)
            sc.bnf = _host_struct(_BN_FUSE, acc=_vp(sc.acc_f), gamma=eng.tptr(bn.params.γ), beta=eng.tptr(bn.params.β),
                                  m_avg=eng.tptr(bn.params.m_avg), v_avg=eng.tptr(bn.params.v_avg),
                                  ss=_vp(sc.ss), mr=_vp(sc.mr), count=float(B * geo.H * geo.W),
                                  d=float(bn.hypers.d), eps=float(bn.hypers.ε), defer=1 if eng.defer_bn else 0)
            bnp = ctypes.c_void_p(sc.bnf.ctypes.data)
        # the scale's launches in order -- source ('h': the split input, 'v': the split pooled predecessor), its K,
        # parts of it in A0 / A1, packed weights, first (bias, no accumulation) / last (BN moments) -- read by the ops
        # below and by the compacted walk (lib/compact_eval.py), which launches the same list on its own batch
        sc.passes = [Ns(src='h', K=K0, Kreal=sc.K0real, na0=na0, na1=na1, W=W) for (na0, na1, _), W in zip(passes, sc.W3h)]
        if prev is not None:
            sc.passes += [Ns(src='v', K=K1, Kreal=K1, na0=na0, na1=na1, W=W) for (na0, na1, _), W in zip(passes, sc.W3v)]
        for i, ps in enumerate(sc.passes):
            ps.first, ps.last = i == 0, i == len(sc.passes) - 1
            src, dep = (sc.src.split, sc.src.split_op) if ps.src == 'h' else (prev.pooled_split, prev.post_op)

            def conv(src=src, ps=ps):
                L.conv_acc_bn_stats(_vp(src), ps.na0 * ps.K, _vp(src) if ps.na1 else None, ps.na1 * ps.K, _vp(ps.W),
                                    eng.tptr(sc.bk) if ps.first else None, _vp(sc.lin), N, 0 if ps.first else 1,
                                    *geo.args(), bnp if ps.last else None, BF16, F32, 1, S())
            self._tag(conv, 'conv_fwd', desc='H%d K3x%d N%d%s' % (geo.H, ps.K, N, '' if ps.first else ' +acc'),
                      flops=3 * 2.0 * B * geo.H * geo.W * 9 * ps.Kreal * N,
                      nbytes=B * geo.H * geo.W * (3 * ps.K * 2 + (1 if ps.first else 2) * N * 4))
            conv.lane = sc.lane
            self._after(conv, dep)
            self.fwd_ops.append(conv)
        if sc.live and not use_stats:
            bn = sc.bn

            def fin(sc=sc, bn=bn):             # inference: scale/shift from the running moments
                L.bn_finalize(None, 0, N, float(B * geo.H * geo.W), eng.tptr(bn.params.γ), eng.tptr(bn.params.β),
                              eng.tptr(bn.params.m_avg), eng.tptr(bn.params.v_avg),
                              float(bn.hypers.d), float(bn.hypers.ε), 0, _vp(sc.ss), _vp(sc.mr), S())
            self._tag(fin, 'bn_finalize')
            fin.lane = sc.lane
            self.fwd_ops.append(fin)
        sc.act_split = sc.pooled_split = None
        if sc.live or sc.pooled is not None:
            if use_stats and eng.defer_bn:
                def post(sc=sc):
                    L.bn_relu_pool_fwd_acc(_vp(sc.lin), N, *geo.args(), bnp, _vp(sc.act), _vp(sc.pooled),
                                           sc.geo_p.P if sc.pooled is not None else 0, _vp(sc.feat), Balloc, F32, S())
            else:
                def post(sc=sc):
                    L.bn_relu_pool_fwd(_vp(sc.lin), N, *geo.args(), _vp(sc.ss) if sc.live else None,
                                       _vp(sc.act), _vp(sc.pooled), sc.geo_p.P if sc.pooled is not None else 0,
                                       _vp(sc.feat), Balloc, F32, S())
            self._tag(post, 'bn_fwd', desc='H%d C%d' % (geo.H, N), nbytes=B * geo.H * geo.W * N * 4 * (1 + (sc.act is not None) + 0.25 * (sc.pooled is not None) + (sc.feat is not None)))
            post.lane = sc.lane
            self.fwd_ops.append(post)
            sc.post_op = post
            if sc.feat is not None:
                st.feat_op = post
            if sc.act is not None:
                sc.act_split, sc.post_op = self._split(sc.act, N, geo, sc.lane)
            if sc.pooled is not None:
                sc.pooled_split, sc.post_op = self._split(sc.pooled, N, sc.geo_p, sc.lane)

    def _bn_bwd_bufs(self, sc):
        """sums / fp64 accumulator / finalisation struct of a scale's BatchNorm backward (shared by the
        stand-alone reduction and the one fused into the consumer's data gradient)"""
        eng = self.eng
        if getattr(sc, 'sums', None) is None:
            sc.sums = self.f32(2, sc.N)
            if getattr(sc, 'acc', None) is None:
                sc.acc = self.zeros(2 * sc.N + 1, torch.float64)
            bn = sc.bn
            sc.bnb = _host_struct(_BN_BWD_FUSE, acc=_vp(sc.acc), sums=_vp(sc.sums),
                                  dgamma=eng.gptr(bn.params.γ), dbeta=eng.gptr(bn.params.β))

    def _build_rcm_bwd(self, nd, Balloc):
        eng, L, B = self.eng, self.eng.L, self.B
        dt, impl = eng.dtype, eng.impl
        S = lambda: eng.stream
        st = self.node[nd.idx]
        lay = nd.layer
        n = len(st.sc)
        par = self.node[nd.parent] if nd.parent is not None else self._image_slot()
        par_grad = par.needs_grad
        # gradient of the heads wrt the flattened coarsest scale
        heads = [k for k in nd.kids if eng.nodes[k].kind == 'reg']
        st.dfeat = None
        if (heads or nd.router is not None) and self.umma_heads:
            self._build_heads_bwd(nd, st, eng.dynamic and bool(eng.net.hypers.dyn_k_cpt))
        elif heads or nd.router is not None:
            if len(heads) > 1:
                raise NotImplementedError('engine: more than one LogReg under one node')
            st.dfeat = self.zeros(tuple(st.feat.shape), st.feat.dtype)
            pairs = []
            if heads:
                r = self.reg[heads[0]]
                pairs.append((r.dZ, r.fc.params.w, r.dZ.shape[1]))
            if nd.router is not None:
                rt = self.rtr[nd.idx]
                pairs.append((rt.dZ1, rt.fc1.params.w, eng.router_width))
            p0 = pairs[0]
            p1 = pairs[1] if len(pairs) > 1 else (None, None, 0)
            fbd = lambda p0=p0, p1=p1: L.fc_bwd_data(
                _vp(p0[0]), eng.tptr(p0[1]), p0[2], _vp(p1[0]), eng.tptr(p1[1]) if p1[1] is not None else None,
                p1[2], st.F, Balloc, B, _vp(st.dfeat), dt, S())
            st.dfeat_op = fbd
            self.bwd_ops.append(fbd)
        for k in range(n - 1, -1, -1):
            sc = st.sc[k]
            geo = sc.geo
            sc.dlin = self.planes(sc.N, geo)
            dact = st.out[k].dact                    # written by child conv stages (already built)
            dfeat = st.dfeat if (k == n - 1) else None
            dpooled = sc.dpooled      # gradient wrt pooled(lin_k), set by scale k+1's dgrad below
            mp = getattr(sc, 'mp', None)
            if mp is not None and (dact is not None or dfeat is not None):
                # MaxPool / GlobalMaxPool behind the ReLU: route the sinks' gradients back to the maxima first
                full = self.planes(sc.N, geo)
                if mp.arg is None:
                    def unpool(sc=sc, dact=dact, dfeat=dfeat, full=full):
                        L.maxpool2_bwd(_vp(sc.act), _vp(dact), _vp(dfeat), Balloc, sc.N, *sc.geo.args(),
                                       sc.mp.geo.P, _vp(full), dt, S())
                else:
                    def unpool(sc=sc, dfeat=dfeat, full=full):
                        L.global_maxpool_bwd(_vp(dfeat), _vp(sc.mp.arg), Balloc, sc.N, *sc.geo.args(), _vp(full), dt, S())
                self._tag(unpool, 'pool_bwd', nbytes=B * geo.H * geo.W * sc.N * (2 if dt == BF16 else 4) * 2.25)
                unpool.lane = sc.lane
                self._after(unpool, getattr(st, 'dfeat_op', None) if dfeat is not None else None,
                            *getattr(st.out[k], 'dact_ops', []))
                self.bwd_ops.append(unpool)
                dact, dfeat = full, None
            if getattr(sc, 'keep', 1.0) != 1.0 and (dact is not None or dfeat is not None):
                def dropb(sc=sc, dact=dact, dfeat=dfeat):
                    if dact is not None:
                        L.dropout(_vp(dact), sc.N, *sc.geo.args(), 0, 0, sc.keep, sc.drop_seed, _vp(eng.hyp), dt, S())
                    if dfeat is not None:
                        L.dropout(_vp(dfeat), sc.N, *sc.geo.args(), 1, Balloc, sc.keep, sc.drop_seed, _vp(eng.hyp), dt, S())
                dropb.lane = sc.lane
                self._after(dropb, getattr(st, 'dfeat_op', None) if dfeat is not None else None,
                            *getattr(st.out[k], 'dact_ops', []))
                self.bwd_ops.append(dropb)
            if getattr(sc, 'act_alpha', 0.0):
                # gradient of alpha * sum x^2, weighted like the node's other costs: 1/B, times p_tr when routed
                acc = 1 if dact is not None else 0
                if dact is None:
                    dact = self.planes(sc.N, geo)
                coef = (lambda nd=nd: ctypes.c_void_p(self.p_tr.data_ptr() + 4 * nd.idx * B)) if eng.dynamic \
                    else (lambda: None)

                def agrad(sc=sc, dact=dact, acc=acc, coef=coef):
                    L.activity_bwd(_vp(sc.act), sc.N, *sc.geo.args(), coef(), 2.0 * sc.act_alpha / B, _vp(dact), acc, dt, S())
                agrad.lane = sc.lane
                if getattr(sc, 'mp', None) is None:
                    self._after(agrad, *getattr(st.out[k], 'dact_ops', []))
                self.bwd_ops.append(agrad)
            live = sc.live and (dact is not None or dfeat is not None)
            self._bn_bwd_bufs(sc)
            # small tensors without a pooling branch (the coarsest scale of a stage at the reference's batch): the
            # reduction and the gradient in ONE launch (mpnn_bn_bwd_small: cluster per plane, rows in registers)
            small = (live and not st.out[k].fused_red and dpooled is None and eng.bn_small
                     and B * sc.geo.H * sc.geo.W <= _BN_SMALL_MAX_PIXELS)
            if live and not st.out[k].fused_red and not small:   # (fused: the sums arrive with the consumer's data gradient)

                def red(sc=sc, dact=dact, dfeat=dfeat):
                    L.bn_bwd_reduce_fused(_vp(sc.lin), _vp(dact), _vp(dfeat), Balloc, _vp(sc.ss), _vp(sc.mr), sc.N,
                                          *sc.geo.args(), ctypes.c_void_p(sc.bnb.ctypes.data), dt, S())
                self._tag(red, 'bn_bwd_reduce', desc='H%d C%d' % (sc.geo.H, sc.N), nbytes=B * sc.geo.H * sc.geo.W * sc.N * (2 if dt == BF16 else 4) * 2)
                red.lane = sc.lane
                if dfeat is not None:
                    self._after(red, getattr(st, 'dfeat_op', None))
                self.bwd_ops.append(red)
            if not live and dpooled is None:
                raise RuntimeError('engine: scale %d of %r has no gradient path' % (k, lay.name))

            if small:
                def elt(sc=sc, dact=dact, dfeat=dfeat):
                    bn = sc.bn
                    L.bn_bwd_small(_vp(sc.lin), _vp(dact), _vp(dfeat), Balloc, _vp(sc.ss), _vp(sc.mr), sc.N,
                                   *sc.geo.args(), _vp(sc.sums), eng.gptr(bn.params.γ), eng.gptr(bn.params.β),
                                   float(B * sc.geo.H * sc.geo.W), _vp(sc.dlin), eng.gptr(sc.bk), dt, S())
            else:
                def elt(sc=sc, dact=dact, dfeat=dfeat, dpooled=dpooled, live=live):
                    L.bn_relu_pool_bwd(_vp(sc.lin), _vp(dact), _vp(dfeat), Balloc, _vp(dpooled),
                                       sc.geo_p.P if dpooled is not None else 0,
                                       _vp(sc.ss) if live else None, _vp(sc.mr), _vp(sc.sums),
                                       float(B * sc.geo.H * sc.geo.W), sc.N, *sc.geo.args(), _vp(sc.dlin),
                                       eng.gptr(sc.bk), dt, S())
            self._tag(elt, 'bn_bwd', desc='H%d C%d%s' % (sc.geo.H, sc.N, ' 1-launch' if small else ''),
                      nbytes=B * sc.geo.H * sc.geo.W * sc.N * (2 if dt == BF16 else 4) * (3 + 0.25 * (dpooled is not None)))
            elt.lane = sc.lane
            if dfeat is not None:
                self._after(elt, getattr(st, 'dfeat_op', None))
            self._after(elt, getattr(sc, 'dpooled_op', None))      # written by scale k+1's data gradient
            self.bwd_ops.append(elt)
            prev = st.sc[k - 1] if k > 0 else None
            if eng.split:
                self._build_conv_bwd_split(sc, prev, elt, par_grad, B)
                continue

            def wgrad(sc=sc, prev=prev):
                L.stencil_wgrad(_vp(sc.src.t), sc.K0, sc.K0real, eng.gptr(sc.wh),
                                _vp(prev.pooled) if prev is not None else None, sc.K1, sc.K1,
                                eng.gptr(sc.wv) if sc.wv is not None else None,
                                _vp(sc.dlin), sc.N, sc.N, None, 9, *sc.geo.args(), dt,   # db: see bn_relu_pool_bwd
                                eng.impl_w if (sc.K0 + sc.K1 <= 128 and sc.N <= 256) else 0, S())
            self._tag(wgrad, 'conv_wgrad', desc='H%d K%d+%d N%d' % (sc.geo.H, sc.K0, sc.K1, sc.N), flops=2.0 * B * sc.geo.H * sc.geo.W * 9 * (sc.K0real + sc.K1) * sc.N,
                      nbytes=B * sc.geo.H * sc.geo.W * (sc.K0 + sc.K1 + sc.N) * (2 if dt == BF16 else 4))
            wgrad.lane = 10 + (sc.lane - 3)          # weight gradients are mutually independent: one lane per scale
            self.bwd_ops.append(self._after(wgrad, elt))
            # data gradient: towards the parent's activation (N0) and the pooled predecessor (N1)
            N0 = sc.K0 if par_grad else 0
            N1 = sc.K1
            if N0 + N1 == 0:
                continue
            sc.Wd = self.zeros((9, sc.N // 8, N0 + N1, 8), eng.tdtype)
            if N0:
                self._pack(sc.wh, sc.Wd, sc.K0real, sc.N, 1, 0, sc.N, 0, N0 + N1)
            if N1:
                self._pack(sc.wv, sc.Wd, sc.K1, sc.N, 1, 0, sc.N, N0, N0 + N1)
            acc0 = 0
            out0 = None
            if N0:
                slot = sc.src
                if slot.dact is None:
                    slot.dact = self.planes(slot.C, geo)
                acc0 = 1 if slot.writers > 0 else 0
                slot.writers += 1
                out0 = slot.dact
            if N1:
                prev.dpooled = self.planes(sc.K1, geo)
            # BatchNorm-backward sums of the layer below ride on this data gradient when it is the only
            # producer of that layer's dAct (one consumer, no head gradient at that scale): removes the
            # bn_bwd_reduce pass over (lin, dAct)
            psc = sc.src.sc if N0 else None
            # (measured: a win where the 16- / 32-wide fast epilogue applies and the tensor is large; on
            #  small tensors and in the generic epilogue the stand-alone reduction is as fast or faster)
            fuse = (psc is not None and eng.fuse_bn_red and impl == 1 and self.bn_train and sc.src.consumers == 1
                    and psc.live and psc.feat is None and psc.N == N0 and (N0 + N1) in (16, 32)
                    and not getattr(psc, 'act_alpha', 0.0) and getattr(psc, 'keep', 1.0) == 1.0
                    and B * sc.geo.H * sc.geo.W >= eng.fuse_bn_red_min_rows)
            if fuse:
                sc.src.fused_red = True
                self._bn_bwd_bufs(psc)
                sc.epi = _host_struct(_BN_BWD_EPI, lin=_vp(psc.lin), ss=_vp(psc.ss), mr=_vp(psc.mr), acc=_vp(psc.acc),
                                      sums=_vp(psc.sums), dgamma=eng.gptr(psc.bn.params.γ),
                                      dbeta=eng.gptr(psc.bn.params.β))

                def dgrad(sc=sc, out0=out0, N0=N0, N1=N1, prev=prev):
                    L.conv_dgrad_bn_reduce(_vp(sc.dlin), sc.N, _vp(sc.Wd), _vp(out0), N0,
                                           _vp(prev.dpooled) if N1 else None, N1, *sc.geo.args(),
                                           ctypes.c_void_p(sc.epi.ctypes.data), dt, impl, S())
            else:
                def dgrad(sc=sc, out0=out0, N0=N0, N1=N1, acc0=acc0, prev=prev):
                    L.stencil_gemm(_vp(sc.dlin), sc.N, None, 0, _vp(sc.Wd), 9, None,
                                   _vp(out0), N0, acc0, _vp(prev.dpooled) if N1 else None, N1, 0,
                                   *sc.geo.args(), None, 0, None, dt, dt, impl, S())
            self._tag(dgrad, 'conv_dgrad', desc='H%d K%d N%d+%d%s' % (sc.geo.H, sc.N, N0, N1, ' +bnred' if fuse else ''),
                      flops=2.0 * B * sc.geo.H * sc.geo.W * 9 * sc.N * (N0 + N1),
                      nbytes=B * sc.geo.H * sc.geo.W * (sc.N + N0 + N1 + (N0 if fuse else 0)) * (2 if dt == BF16 else 4))
            dgrad.lane = sc.lane
            if N1:
                prev.dpooled_op = dgrad
            if N0 and hasattr(sc.src, 'dact_ops'):
                sc.src.dact_ops.append(dgrad)
            self.bwd_ops.append(dgrad)

    def _build_conv_bwd_split(self, sc, prev, elt, par_grad, B):
        """bf16x3 mode: dLin (fp32) is split into (hi | lo); the weight gradient is three tcgen05 launches
        (A_hi x G_hi, A_lo x G_hi, A_hi x G_lo, all reduced into the same fp32 gradient tensors), the data
        gradient one launch over [G_hi | G_lo | G_hi] x [W_hi; W_hi; W_lo] with fp32 planes out."""
        eng, L = self.eng, self.eng.L
        S = lambda: eng.stream
        geo, N, K0, K1 = sc.geo, sc.N, sc.K0, sc.K1
        sc.dlin_split, sp = self._split(sc.dlin, N, geo, sc.lane, ops=self.bwd_ops)
        self._after(sp, elt)
        part = lambda t, C, j: ctypes.c_void_p(t.data_ptr() + j * (C // 8) * geo.P * 16) if t is not None else None
        psp = prev.pooled_split if prev is not None else None
        dWv = eng.gptr(sc.wv) if sc.wv is not None else None
        # (activation part, gradient part) of every product kept: all pairs with i + j < number of parts
        pairs = [(i, j) for j in range(eng.split) for i in range(eng.split - j)]
        for n_, (i, j) in enumerate(pairs):
            a0, a1, g = part(sc.src.split, K0, i), part(psp, K1, i), part(sc.dlin_split, N, j)

            def wgrad(a0=a0, a1=a1, g=g):
                L.stencil_wgrad(a0, K0, sc.K0real, eng.gptr(sc.wh), a1, K1, K1, dWv, g, N, N, None, 9,
                                *geo.args(), BF16, 1 if (K0 + K1 <= 128 and N <= 256) else 0, S())
            self._tag(wgrad, 'conv_wgrad', desc='H%d K%d+%d N%d x%d[%d]' % (geo.H, K0, K1, N, len(pairs), n_),
                      flops=2.0 * B * geo.H * geo.W * 9 * (sc.K0real + K1) * N, nbytes=B * geo.H * geo.W * (K0 + K1 + N) * 2)
            wgrad.lane = 10 + (sc.lane - 3)
            self.bwd_ops.append(self._after(wgrad, sp))
        N0 = K0 if par_grad else 0
        N1 = K1
        if N0 + N1 == 0:
            return
        passes = _SPLIT_PASSES[eng.split]
        sc.Wd3 = []
        for _, _, wparts in passes:
            Wd = self.zeros((9, 3 * N // 8, N0 + N1, 8), torch.bfloat16)
            for j, mode in enumerate(wparts):                                  # parts along K (= output channels)
                if N0:
                    self._pack(sc.wh, Wd, sc.K0real, N, mode | 1, j * N, 3 * N, 0, N0 + N1)
                if N1:
                    self._pack(sc.wv, Wd, K1, N, mode | 1, j * N, 3 * N, N0, N0 + N1)
            sc.Wd3.append(Wd)
        acc0, out0 = 0, None
        if N0:
            slot = sc.src
            if slot.dact is None:
                slot.dact = self.planes(slot.C, geo)
            acc0 = 1 if slot.writers > 0 else 0
            slot.writers += 1
            out0 = slot.dact
        if N1:
            prev.dpooled = self.planes(K1, geo)
        for i, ((na0, na1, _), Wd) in enumerate(zip(passes, sc.Wd3)):
            def dgrad(out0=out0, acc0=acc0 if i == 0 else 1, acc1=0 if i == 0 else 1, na0=na0, na1=na1, Wd=Wd):
                L.stencil_gemm(_vp(sc.dlin_split), na0 * N, _vp(sc.dlin_split) if na1 else None, na1 * N, _vp(Wd), 9, None,
                               _vp(out0), N0, acc0, _vp(prev.dpooled) if N1 else None, N1, acc1,
                               *geo.args(), None, 0, None, BF16, F32, 1, S())
            self._tag(dgrad, 'conv_dgrad', desc='H%d K3x%d N%d+%d%s' % (geo.H, N, N0, N1, ' +acc' if i else ''),
                      flops=3 * 2.0 * B * geo.H * geo.W * 9 * N * (N0 + N1),
                      nbytes=B * geo.H * geo.W * (3 * N * 2 + (N0 + N1) * 4 * (2 if i else 1)))
            dgrad.lane = sc.lane
            if N1:
                prev.dpooled_op = dgrad
            self.bwd_ops.append(dgrad)

    # -- router ------------------------------------------------------------ #
    def _build_router_fwd(self, nd, Balloc, dyn_k, emit_fc=True):
        eng, L, B = self.eng, self.eng.L, self.B
        dt = eng.dtype
        S = lambda: eng.stream
        st = self.node[nd.idx]
        c = nd.router.comps
        fc1, bn1, fc2, bn2, fc3 = c[1], c[2], c[4], c[5], c[7]
        if c[0].hypers.i != -1:
            raise NotImplementedError('engine: router must select the coarsest scale')
        ns = len(nd.kids)
        if fc3.hypers.n_chan != ns:
            raise NotImplementedError('engine: router output width %d for %d sinks' % (fc3.hypers.n_chan, ns))
        W = eng.router_width                    # hidden width, checked for the whole net by _router_width
        bwd = self.need_bwd
        rt = Ns(fc1=fc1, bn1=bn1, fc2=fc2, bn2=bn2, fc3=fc3, ns=ns,
                Z1=self.f32(B, W), Z2=self.f32(B, W), R=self.f32(B, ns), save=self.f32(4 * W),
                dR=self.f32(B, ns) if bwd else None, dZ1=self.f32(B, W) if bwd else None,
                scratch=self.f32(2 * B * W) if bwd else None)
        self.rtr[nd.idx] = rt
        if emit_fc:
            fcr = lambda: L.fc_fwd(
                _vp(st.feat), st.F, Balloc, B, eng.tptr(fc1.params.w), eng.tptr(fc1.params.b),
                _vp(self.kextra) if dyn_k else None, W, _vp(rt.Z1), dt, S())
            self.fwd_ops.append(self._after(fcr, getattr(st, 'feat_op', None)))
        P = lambda lay, k: eng.tptr(getattr(lay.params, k))
        # the tails of all routers run as ONE launch after the conv pipeline (see _build)
        self.rt_fwd.append(dict(
            Z1=rt.Z1, g1=P(bn1, 'γ'), b1=P(bn1, 'β'), m1=P(bn1, 'm_avg'), v1=P(bn1, 'v_avg'),
            W2=P(fc2, 'w'), bias2=P(fc2, 'b'), g2=P(bn2, 'γ'), b2=P(bn2, 'β'), m2=P(bn2, 'm_avg'),
            v2=P(bn2, 'v_avg'), W3=P(fc3, 'w'), bias3=P(fc3, 'b'), Z2=rt.Z2, R=rt.R, save=rt.save, ns=ns))

    def _build_router_bwd(self, nd, Balloc, dyn_k):
        eng, L, B = self.eng, self.eng.L, self.B
        dt = eng.dtype
        S = lambda: eng.stream
        st = self.node[nd.idx]
        rt = self.rtr[nd.idx]
        Gp = lambda lay, k: eng.gptr(getattr(lay.params, k))
        # (the tail itself ran in the batched launch right after route_bwd)
        self.bwd_ops.append(lambda: L.fc_bwd_weight(
            _vp(st.feat), st.F, Balloc, B, _vp(self.kextra) if dyn_k else None, _vp(rt.dZ1), eng.router_width,
            Gp(rt.fc1, 'w'), Gp(rt.fc1, 'b'), dt, S()))

    # -- routing ----------------------------------------------------------- #
    def _build_routing(self):
        eng, L, B = self.eng, self.eng.L, self.B
        S = lambda: eng.stream
        dev = eng.dev
        nodes = eng.nodes
        nn = len(nodes)
        root_leaves = n_leaves(eng.net.root)
        ti = lambda v: torch.tensor(v, dtype=torch.int32, device=dev)
        tf = lambda v: torch.tensor(v, dtype=torch.float32, device=dev)
        self.t_parent = ti([nd.parent if nd.parent is not None else -1 for nd in nodes])
        self.t_sink = ti([nd.sink_idx for nd in nodes])
        self.t_nsinks = ti([len(nd.kids) for nd in nodes])
        child = np.full((nn, MAXS), -1, np.int32)
        for nd in nodes:
            child[nd.idx, :len(nd.kids)] = nd.kids
        self.t_child = ti(child)
        self.t_floor = tf([n_leaves(nd.layer) / root_leaves for nd in nodes])
        self.t_sw = ti([getattr(nd, 'sw', -1) if len(nd.kids) > 1 else -1 for nd in nodes])
        self.t_ops = tf([float(nd.layer.n_ops + (nd.router.n_ops if nd.router is not None else 0)) for nd in nodes])
        self.t_err = ti([nd.err if nd.kind == 'reg' else -1 for nd in nodes])
        self.p_tr = self.f32(nn, B)
        self.p_ev = self.f32(nn, B)
        n_sw = max(len(eng.switches), 1)
        self.dec = self.zeros((n_sw, B), torch.int32)
        tp = lambda ts: torch.tensor([t.data_ptr() for t in ts] or [0], dtype=torch.int64, device=dev)
        self.R_tab = tp([self.rtr[nd.idx].R for nd in eng.switches])
        self.cerr_tab = tp([self.reg[nd.idx].c_err for nd in eng.regs])
        self.dcor_tab = tp([self.reg[nd.idx].d_cor for nd in eng.regs])
        self.fwd_ops.append(lambda: L.route_fwd(
            _vp(self.t_parent), _vp(self.t_sink), _vp(self.t_nsinks), _vp(self.t_floor), _vp(self.t_sw), nn,
            _vp(self.R_tab), _vp(eng.hyp), B, _vp(self.p_tr), _vp(self.p_ev), _vp(self.dec), S()))
        if self.need_bwd:
            self.dR_tab = tp([self.rtr[nd.idx].dR for nd in eng.switches])
            self.route_scratch = self.f32(3 * nn * B)
            self.c_data = self.f32(B)
