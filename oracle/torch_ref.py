"""CPU oracle (TEST INFRASTRUCTURE ONLY) -- a define-by-run restatement, on
PyTorch-CPU autograd, of the reference's TensorFlow graph for the hot path.

  PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures
  (SURVEY.md section 4 / 8c) and TensorFlow <= 0.12 cannot be installed in this
  image, so this restatement cannot be checked against outputs of the
  reference itself.  It is cross-checked against an independent NumPy fp64
  forward (oracle/np_ref.py) and finite differences (tests/test_oracle.py).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs may import this module.  The product (multipath-nn_b200/)
never does.

The oracle interprets the *serialised* net record (the dict tree written by
the reference's serdes, /root/reference/scripts/lib/serdes.py:13-19,40-44) so
that product and oracle consume byte-identical weights.  Every rule cites the
reference lines it follows (paths relative to /root/reference/scripts).

Nodes of the sink tree are named by their path from the root: '' is the
root, '0' its first sink, '0/1' the second sink of that, and so on.
"""
from __future__ import annotations

import math
from types import SimpleNamespace as Ns

import numpy as np
import torch
import torch.nn.functional as F

__all__ = ['OracleNet']


def _eps(hy, default=1e-6):
    """The reference spells the hyper `\u03f5` (U+03F5); Python NFKC-normalises
    identifiers, so the attribute / record key is `\u03b5` (U+03B5)."""
    for k in ('\u03b5', '\u03f5'):
        if k in hy:
            return hy[k]
    return default


# --------------------------------------------------------------------------- #
# TF op semantics (SURVEY App. A)
# --------------------------------------------------------------------------- #

def _same_pad(n, k, s=1):
    """TF 'SAME': total = max((ceil(n/s)-1)*s + k - n, 0); extra goes last."""
    out = -(-n // s)
    tot = max((out - 1) * s + k - n, 0)
    return tot // 2, tot - tot // 2


def tf_conv2d_same(x, w):
    """tf.nn.conv2d(x NHWC, w HWIO, stride 1, 'SAME') -- cross-correlation.
    lib/layer_types.py:106-107."""
    kh, kw = w.shape[0], w.shape[1]
    pt, pb = _same_pad(x.shape[1], kh)
    pl, pr = _same_pad(x.shape[2], kw)
    xc = F.pad(x.permute(0, 3, 1, 2), (pl, pr, pt, pb))
    return F.conv2d(xc, w.permute(3, 2, 0, 1)).permute(0, 2, 3, 1)


def tf_max_pool_same(x, k, s):
    """tf.nn.max_pool(x NHWC, ksize k, stride s, 'SAME'); padding never wins."""
    pt, pb = _same_pad(x.shape[1], k, s)
    pl, pr = _same_pad(x.shape[2], k, s)
    xc = F.pad(x.permute(0, 3, 1, 2), (pl, pr, pt, pb), value=-math.inf)
    return F.max_pool2d(xc, k, s).permute(0, 2, 3, 1)


def tf_resize_legacy(x, h, w):
    """tf.image.resize_images (TF<=0.12 bilinear, align_corners=False): source
    coordinate = dst * (in/out).  For the integer factors the pyramid uses the
    interpolation weight is zero, i.e. strided subsampling.  Non-integer
    factors fall back to the same formula with interpolation.
    lib/layer_types.py:123-125."""
    ih, iw = x.shape[1], x.shape[2]
    if ih % h == 0 and iw % w == 0:
        return x[:, ::ih // h, ::iw // w, :]
    ys = torch.arange(h, dtype=x.dtype) * (ih / h)
    xs = torch.arange(w, dtype=x.dtype) * (iw / w)
    y0 = ys.floor().long(); x0 = xs.floor().long()
    y1 = (y0 + 1).clamp(max=ih - 1); x1 = (x0 + 1).clamp(max=iw - 1)
    fy = (ys - y0)[None, :, None, None]; fx = (xs - x0)[None, None, :, None]
    top = x[:, y0][:, :, x0] * (1 - fx) + x[:, y0][:, :, x1] * fx
    bot = x[:, y1][:, :, x0] * (1 - fx) + x[:, y1][:, :, x1] * fx
    return top * (1 - fy) + bot * fy


def first_argmax(x, dim):
    """tf.argmax: index of the FIRST maximal element."""
    m = x.max(dim, keepdim=True).values
    idx = torch.arange(x.shape[dim], device=x.device).reshape(
        [-1 if d == dim % x.dim() else 1 for d in range(x.dim())])
    big = x.shape[dim]
    return torch.where(x == m, idx, big).min(dim).values


# --------------------------------------------------------------------------- #
# Optional emulation of bf16 STORAGE (quant='bf16'): the CUDA path keeps conv
# operands / activations / activation gradients in bf16 and accumulates in
# fp32.  Rounding only those tensors here gives an oracle "in the arithmetic
# the device stores in", so kernel bugs are not masked by (or mistaken for)
# the number format's own error.
# --------------------------------------------------------------------------- #

class _RoundBoth(torch.autograd.Function):
    """value and incoming gradient rounded to bf16 (activations, lin, pooled)"""
    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype)


class _RoundFwd(torch.autograd.Function):
    """value rounded to bf16, gradient untouched (packed weights, input pyramid)"""
    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


# --------------------------------------------------------------------------- #
# Layer interpreter
# --------------------------------------------------------------------------- #

class _Node(Ns):
    """Per-record link state: x, c_err, c_mod, n_ops, delta_cor, p (params)."""


def _n_leaves(rec):
    # lib/net_types.py:14-16
    return 1 if not rec['sinks'] else sum(_n_leaves(s) for s in rec['sinks'])


class OracleNet:
    """Restatement of SRNet / ActorNet / CriticNet (lib/net_types.py:85-284).

    record : dict as produced by serdes.encode_net
    dtype  : torch.float32 (reference precision) or torch.float64
    """

    def __init__(self, record, dtype=torch.float32, quant=None):
        assert quant in (None, 'bf16')
        self.quant = quant
        self.rec = record
        self.kind = record['type']
        self.dtype = dtype
        self.hy = dict(record['hypers'])
        self.params = {}     # id(param record dict) -> {key: tensor}
        self.trainable = []  # (owner_path, role, key, tensor); role 'layer'|'router'
        self._collect(record['root'], '')
        self.momentum = {id(t): torch.zeros_like(t) for _, _, _, t in self.trainable}
        # TF's dropout stream cannot be restated: a test that exercises Dropout(λ < 1) supplies the keep masks of
        # one evaluation here, in the order the Dropout layers are linked (preorder)
        self.dropout_masks = None
        self._drop_i = 0

    # -- parameters ------------------------------------------------------- #
    def _collect(self, rec, path):
        def grab(r, role):
            if r is None:
                return
            store = {}
            for k, v in r['params'].items():
                t = torch.tensor(np.asarray(v), dtype=self.dtype)
                if k not in ('m_avg', 'v_avg'):     # layer_types.py:229-230
                    t.requires_grad_(True)
                    self.trainable.append((path, role, k, t))
                store[k] = t
            self.params[id(r)] = store
            for c in r['comps']:
                grab(c, role)
        grab(rec, 'layer')
        grab(rec['router'], 'router')
        for i, s in enumerate(rec['sinks']):
            self._collect(s, (path + '/' if path else '') + str(i))

    def write_back(self):
        """Copy current parameter values back into the record (numpy fp32)."""
        def put(r):
            if r is None:
                return
            for k, t in self.params[id(r)].items():
                r['params'][k] = t.detach().to(torch.float32).numpy().copy()
            for c in r['comps']:
                put(c)
            put(r['router'])
            for s in r['sinks']:
                put(s)
        put(self.rec['root'])

    def _q(self, x):
        return _RoundBoth.apply(x) if self.quant else x

    def _qf(self, x):
        return _RoundFwd.apply(x) if self.quant else x

    # -- layer link rules -------------------------------------------------- #
    def _link(self, rec, x, y, mode):
        """Returns a _Node; mirrors Layer.link (layer_types.py:22-26)."""
        kind = rec['type']
        hy = rec['hypers']
        p = self.params[id(rec)]
        nd = _Node(x=x, c_err=0.0, c_mod=0.0, n_ops=0, delta_cor=None, comps=[])
        if kind == 'NoOp':
            pass
        elif kind == 'Chain':                       # layer_types.py:299-310
            for i, c in enumerate(rec['comps']):
                # (bf16 restatement: the device rounds the pyramid where it is packed, i.e. behind a MultiscaleLLN)
                nxt = rec['comps'][i + 1]['type'] if i + 1 < len(rec['comps']) else None
                self._raw_pyramid = c['type'] == 'ToPyramid' and nxt == 'MultiscaleLLN'
                cn = self._link(c, x, y, mode)
                nd.comps.append(cn)
                x = cn.x
            nd.x = x
            nd.c_err = sum(c.c_err for c in nd.comps) if nd.comps else 0.0
            nd.c_mod = sum(c.c_mod for c in nd.comps) if nd.comps else 0.0
            nd.n_ops = sum(c.n_ops for c in nd.comps) if nd.comps else 0
            if nd.comps and nd.comps[-1].delta_cor is not None:
                nd.delta_cor = nd.comps[-1].delta_cor
        elif kind == 'LinTrans':                    # layer_types.py:39-53
            n_in = int(np.prod(x.shape[1:]))
            w_eq = (torch.eye(n_in, hy['n_chan'], dtype=self.dtype)
                    if hy.get('res', False) else 0)
            nd.x = x.reshape(-1, n_in) @ p['w'] + p['b']
            nd.c_mod = hy.get('k_l2', 0) * ((p['w'] - w_eq) ** 2).sum()
            nd.n_ops = n_in * hy['n_chan']
        elif kind == 'Conv':                        # layer_types.py:55-74
            n_in = x.shape[3]
            supp = hy.get('supp', 1)
            if hy.get('res', False):
                sel = (np.arange(supp) == supp // 2)
                w_eq = torch.tensor(
                    sel[:, None, None, None] * sel[:, None, None]
                    * np.eye(n_in, hy['n_chan']), dtype=self.dtype)
            else:
                w_eq = 0
            nd.x = tf_conv2d_same(x, p['w']) + p['b']
            nd.c_mod = hy.get('k_l2', 0) * ((p['w'] - w_eq) ** 2).sum()
            nd.n_ops = int(np.prod(x.shape[1:3])) * supp ** 2 * n_in * hy['n_chan']
        elif kind == 'Rect':                        # layer_types.py:76-79
            nd.x = torch.relu(x)
        elif kind == 'Softmax':                     # layer_types.py:81-84
            nd.x = torch.softmax(x, 1)
        elif kind == 'MaxPool':                     # layer_types.py:86-94
            # the reference passes (strides, k_shape) into (ksize, strides):
            # the window is `stride` wide and the step is `supp` (SURVEY F8)
            nd.x = tf_max_pool_same(x, hy.get('stride', 1), hy.get('supp', 1))
        elif kind == 'GlobalMaxPool':               # layer_types.py:96-100
            nd.x = x.amax(tuple(range(1, x.dim() - 1)))
        elif kind == 'ToPyramid':                   # layer_types.py:118-125
            h, w = x.shape[1:3]
            qf = (lambda t: t) if getattr(self, '_raw_pyramid', False) else self._qf
            nd.x = [qf(tf_resize_legacy(x, h // 2 ** i, w // 2 ** i))
                    for i in range(hy.get('n_scales', 1))]
        elif kind == 'MultiscaleLLN':               # layer_types.py:126-147
            sig, e = hy.get('σ', 3), hy.get('ϵ', 1e-3)
            s = int(np.ceil(2 * sig))
            u = np.linspace(-s, s, 2 * s + 1)[:, None, None, None]
            v = np.linspace(-s, s, 2 * s + 1)[:, None, None]
            k = (np.exp(-(u ** 2 + v ** 2) / (2 * sig ** 2)) / (2 * np.pi * sig ** 2)
                 * np.array([[0.2126], [0.7152], [0.0722]]))                      # HWIO, (2s+1, 2s+1, 3, 1)
            kt = torch.tensor(k, dtype=self.dtype)
            out = []
            for x_i in x:
                # pad by s, SAME conv, crop the middle = the zero-padded correlation at every pixel
                lum = tf_conv2d_same(x_i, kt)
                den = tf_conv2d_same(torch.ones_like(x_i), kt)
                out.append(self._qf(x_i / (lum / den + e)))
            nd.x = out
        elif kind == 'MultiscaleConvMax':           # layer_types.py:149-194
            n = len(hy['n_chan'])
            xin = x[len(x) - n:]
            out = []
            n_ops = 0
            sq = 0.0
            for k in range(n):
                wh = p['w_horz_%i' % k]
                o = p['b_%i' % k] + tf_conv2d_same(xin[k], self._qf(wh))
                sq = sq + (wh ** 2).sum()
                ops = wh.numel()
                if k > 0:
                    wv = p['w_vert_%i' % (k - 1)]
                    o = o + tf_conv2d_same(self._q(tf_max_pool_same(out[k - 1], 2, 2)), self._qf(wv))
                    sq = sq + (wv ** 2).sum()
                    ops += wv.numel()
                n_ops += int(o.shape[1] * o.shape[2]) * ops
                out.append(self._q(o))
            nd.x = out
            nd.c_mod = hy.get('k_l2', 0) * sq
            nd.n_ops = n_ops
        elif kind == 'MultiscaleRect':              # layer_types.py:196-199
            nd.x = [self._q(torch.relu(v)) for v in x]
        elif kind == 'Select':                      # layer_types.py:201-206
            nd.x = x[hy.get('i', 0)]
        elif kind == 'BatchNorm':                   # layer_types.py:219-239
            nd.x = self._batch_norm(p, hy, x, mode)
        elif kind == 'MultiscaleBatchNorm':         # layer_types.py:241-249
            nd.x = [self._batch_norm(self.params[id(c)], c['hypers'] or hy, v, mode)
                    for c, v in zip(rec['comps'], x)]
        elif kind == 'CrossEntropyError':           # layer_types.py:262-272
            eps = _eps(hy)
            n_cls = y.shape[1]
            p_cls = eps / n_cls + (1 - eps) * x
            nd.c_err = -(y * torch.log(p_cls)).sum(1)
            # self.x is the layer INPUT (layer_types.py:23, SURVEY F8)
            nd.delta_cor = (first_argmax(x, 1) == first_argmax(y, 1)).to(self.dtype)
        elif kind == 'SquaredError':                # layer_types.py:255-260
            nd.c_err = ((x - y) ** 2).sum(1)
            nd.delta_cor = (first_argmax(x, 1) == first_argmax(y, 1)).to(self.dtype)
        elif kind == 'SuperclassCrossEntropyError':  # layer_types.py:274-285
            eps = _eps(hy)
            y_sup = y @ torch.as_tensor(np.asarray(hy['w_cls']), dtype=self.dtype)
            n_sup = y_sup.shape[1]
            p_cls = eps / n_sup + (1 - eps) * x
            nd.c_err = -(y_sup * torch.log(p_cls)).sum(1)
            nd.delta_cor = (first_argmax(x, 1) == first_argmax(y_sup, 1)).to(self.dtype)
        elif kind == 'ActivityError':               # layer_types.py:287-293 (c_mod is PER EXAMPLE here)
            nd.c_mod = hy.get('α', 0.0) * (x ** 2).sum(tuple(range(1, x.dim())))
        elif kind == 'Dropout':                     # layer_types.py:212-217: tf.nn.dropout(x, keep_prob=λ), every mode
            lam = hy.get('λ', 1)
            if lam != 1:
                if self.dropout_masks is None:
                    raise NotImplementedError('oracle: Dropout(λ=%r) draws from TF\'s random stream '
                                              '(set dropout_masks)' % lam)
                m = torch.as_tensor(np.asarray(self.dropout_masks[self._drop_i]), dtype=self.dtype)
                self._drop_i += 1
                nd.x = self._q(x * m / lam)
        else:
            raise NotImplementedError('oracle: layer type %r' % kind)
        return nd

    def _batch_norm(self, p, hy, x, mode):
        d = hy.get('d', 0.9)
        eps = _eps(hy)
        if mode == 'tr':
            dims = tuple(range(x.dim() - 1))
            m = x.mean(dims)
            v = ((x - m) ** 2).mean(dims)           # tf.nn.moments: biased
            with torch.no_grad():
                p['m_avg'].copy_(d * p['m_avg'] + (1 - d) * m)
                p['v_avg'].copy_(d * p['v_avg'] + (1 - d) * v)
            return p['γ'] * (x - m) / torch.sqrt(v + eps) + p['β']
        return p['γ'] * (x - p['m_avg']) / torch.sqrt(p['v_avg'] + eps) + p['β']

    # -- net link + routing -------------------------------------------------- #
    def forward(self, x0, y, mode='ev', tau=None, k_cpt=None, eps=None):
        """One link of the whole net.  Returns Ns(c_tot, nodes{path: Ns}).

        Per node: x (output), c_err, c_mod, n_ops, delta_cor, p_tr, p_ev,
        router (Ns(x, c_mod, n_ops)) or None, and for critics c_ev/c_opt/c_cre.
        """
        dt = self.dtype
        self._drop_i = 0
        x0 = torch.as_tensor(np.asarray(x0), dtype=dt)
        y = torch.as_tensor(np.asarray(y), dtype=dt)
        B = x0.shape[0]
        hy = self.hy
        dyn = self.kind != 'SRNet'
        if dyn:
            tau = hy.get('τ') if tau is None else tau
            eps = _eps(hy) if eps is None else eps
            if hy.get('dyn_k_cpt', False):
                k_cpt = torch.as_tensor(np.asarray(k_cpt), dtype=dt).reshape(-1)
            else:
                k_cpt = hy.get('k_cpt', 0.0) if k_cpt is None else k_cpt
        nodes = {}
        order = []

        def link_layer(rec, x, path):               # net_types.py:56-63,146-164
            nd = self._link(rec, x, y, mode)
            nd.rec = rec
            nd.router = None
            if rec['router'] is not None:
                xr = nd.x
                if dyn and hy.get('dyn_k_cpt', False):
                    def cat(v):
                        return torch.cat([
                            v.reshape(B, -1),
                            hy.get('α_cpt', 1e7) * k_cpt[:, None] * torch.ones(B, 1, dtype=dt)], 1)
                    xr = [cat(v) for v in xr] if isinstance(xr, list) else cat(xr)
                nd.router = self._link(rec['router'], xr, y, mode)
            nodes[path] = nd
            order.append(path)
            for i, s in enumerate(rec['sinks']):
                link_layer(s, nd.x, (path + '/' if path else '') + str(i))

        link_layer(self.rec['root'], x0, '')
        ones = torch.ones(B, dtype=dt)

        if not dyn:                                  # net_types.py:88-97
            for nd in nodes.values():
                nd.p_ev = ones
                nd.p_tr = None
            c_tot = sum(nd.c_err + nd.c_mod for nd in nodes.values())
            c_tot = (c_tot * ones).mean()
            return Ns(c_tot=c_tot, nodes=nodes, order=order)

        n_root = _n_leaves(self.rec['root'])

        def floor(rec):                              # net_types.py:121-122
            return eps * _n_leaves(rec) / n_root

        def rops(nd):
            return nd.router.n_ops if nd.router is not None else 0

        critic = self.kind == 'CriticNet'
        use_cls = bool(hy.get('use_cls_err', False))

        def route(path, p_tr, p_ev):                 # net_types.py:108-131,193-243
            nd = nodes[path]
            rec = nd.rec
            nd.p_tr, nd.p_ev = p_tr, p_ev
            kids = [(path + '/' if path else '') + str(i) for i in range(len(rec['sinks']))]
            if critic:
                if use_cls:
                    c_err = 1 - (nd.delta_cor if nd.delta_cor is not None else 1)
                else:
                    c_err = nd.c_err
            if len(kids) < 2:
                for k in kids:
                    route(k, p_tr, p_ev)
                if critic:
                    base = c_err + k_cpt * nd.n_ops
                    nd.c_ev = base + sum(nodes[k].c_ev for k in kids)
                    nd.c_opt = base + sum(nodes[k].c_opt for k in kids)
                    nd.c_cre = 0.0
                return
            r = nd.router.x
            pi_tr = ((1 - floor(rec) / p_tr[:, None]) * torch.softmax(r / tau, 1)
                     + torch.tensor([floor(s) for s in rec['sinks']], dtype=dt) / p_tr[:, None])
            pi_ev = F.one_hot(first_argmax(r, 1), len(kids)).to(dt)
            nd.pi_ev = pi_ev
            for i, k in enumerate(kids):
                route(k, p_tr * pi_tr[:, i], p_ev * pi_ev[:, i])
            if critic:
                base = c_err + k_cpt * (nd.n_ops + nd.router.n_ops)
                nd.c_ev = base + sum(pi_ev[:, i] * nodes[k].c_ev for i, k in enumerate(kids))
                c_min = nodes[kids[0]].c_opt * ones
                for k in kids[1:]:
                    c_min = torch.minimum(c_min, nodes[k].c_opt * ones)
                nd.c_opt = base + c_min
                opt = bool(hy.get('optimistic', False))
                nd.c_cre = hy.get('k_cre', 1e-3) * sum(
                    (r[:, i] + ((nodes[k].c_opt if opt else nodes[k].c_ev) * ones).detach()) ** 2
                    for i, k in enumerate(kids))

        route('', ones, ones)
        L = [nodes[p] for p in order]

        def rmod(nd):
            return nd.router.c_mod if nd.router is not None else 0.0

        if not critic:                               # net_types.py:167-177
            c_err = sum(nd.p_tr * nd.c_err for nd in L)
            c_cpt = sum(nd.p_tr * k_cpt * (nd.n_ops + rops(nd)) for nd in L)
            c_mod = sum(nd.p_tr.detach() * (nd.c_mod + rmod(nd)) for nd in L)
            c_dec = sum(nd.p_tr.detach() * hy.get('k_dec', 0.01) * (nd.router.x ** 2).sum(1)
                        for nd in L if len(nd.rec['sinks']) > 1)
            c_tot = (c_err + c_cpt + c_mod + c_dec).mean()
        else:                                        # net_types.py:275-280
            c_err = sum(nd.p_tr.detach() * nd.c_err for nd in L)
            c_cre = sum(nd.p_tr.detach() * nd.c_cre for nd in L)
            c_mod = sum(nd.p_tr.detach() * (nd.c_mod + rmod(nd)) for nd in L)
            c_tot = (c_err + c_cre + c_mod).mean()
        return Ns(c_tot=c_tot, nodes=nodes, order=order)

    # -- training step -------------------------------------------------------- #
    def grads(self, x0, y, tau=None, k_cpt=None):
        """c_tot and raw d c_tot / d theta (before TALR), mode 'tr'."""
        for _, _, _, t in self.trainable:
            t.grad = None
        out = self.forward(x0, y, 'tr', tau=tau, k_cpt=k_cpt)
        out.c_tot.backward()
        g = {}
        for path, role, key, t in self.trainable:
            g[(path, role, key, id(t))] = (
                t.grad.detach().clone() if t.grad is not None else torch.zeros_like(t))
        return out, g

    def train_step(self, x0, y, lr=None, mu=None, tau=None, k_cpt=None):
        """minimize_expectation (net_types.py:24-37) + MomentumOptimizer
        (non-Nesterov: a <- mu a + g ; theta <- theta - lr a)."""
        hy = self.hy
        lr = hy.get('λ_lrn', 1e-3) if lr is None else lr
        mu = hy.get('μ_lrn', 0.9) if mu is None else mu
        out, g = self.grads(x0, y, tau=tau, k_cpt=k_cpt)
        talr = self.kind != 'SRNet' and bool(hy.get('talr', True))
        a_rtr = hy.get('α_rtr', 1.0) if self.kind != 'SRNet' else 1.0
        scale = {}
        for path, nd in out.nodes.items():
            s = 1.0
            if talr:
                s = 1.0 / torch.sqrt((nd.p_tr.detach() ** 2).mean())
            scale[(path, 'layer')] = s
            scale[(path, 'router')] = a_rtr * s
        with torch.no_grad():
            for (path, role, key, tid), gr in g.items():
                t = next(tt for pp, rr, kk, tt in self.trainable if id(tt) == tid)
                # TF only returns gradients for variables c_tot depends on;
                # a parameter with no path to c_tot (dead BN scales) keeps
                # grad None and is skipped (net_types.py:36).
                if t.grad is None:
                    continue
                acc = self.momentum[tid]
                acc.mul_(mu).add_(scale[(path, role)] * gr)
                t.sub_(lr * acc)
        return out

    # -- statistics (scripts/train-nets:111-130) ------------------------------ #
    def state(self, x0, y, tau=None, k_cpt=None):
        """Per-example statistic tensors of `state_tensors`, mode 'ev'."""
        with torch.no_grad():
            out = self.forward(x0, y, 'ev', tau=tau, k_cpt=k_cpt)
        yt = torch.as_tensor(np.asarray(y), dtype=self.dtype)
        st = {}
        L = [(p, out.nodes[p]) for p in out.order]
        leaves = [(p, nd) for p, nd in L if not nd.rec['sinks']]

        def tot_ops(nd):
            return nd.n_ops + (nd.router.n_ops if nd.router is not None else 0)

        st[('net', 'acc')] = sum(nd.p_ev * nd.delta_cor for _, nd in leaves)
        st[('net', 'moc')] = sum(nd.p_ev * tot_ops(nd) for _, nd in L)
        for p, nd in leaves:
            st[(p, 'p_cor')] = nd.p_ev * nd.delta_cor
            st[(p, 'p_inc')] = nd.p_ev * (1 - nd.delta_cor)
            st[(p, 'p_cor_by_cls')] = (nd.p_ev * nd.delta_cor)[:, None] * yt
            st[(p, 'p_inc_by_cls')] = (nd.p_ev * (1 - nd.delta_cor))[:, None] * yt
            if nd.p_tr is not None:
                st[(p, 'p_tr')] = nd.p_tr
            st[(p, 'c_err')] = nd.c_err
        for p, nd in L:
            if nd.router is not None:
                st[(p, 'x_rte')] = nd.router.x.abs().mean(1)
        return {k: v.numpy() for k, v in st.items()}, out
