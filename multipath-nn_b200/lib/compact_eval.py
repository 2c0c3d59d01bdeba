"""Compacted 'ev'-mode evaluation: the second hot loop of the reference
(/root/reference/scripts/lib/desc.py:10-22 called from scripts/train-nets:144-155 -- full passes over the
training and test sets every t_log steps).

The reference evaluates every node of the tree on the whole batch and multiplies the statistics with the
one-hot p_ev (scripts/lib/net_types.py:127-131, scripts/train-nets:117-130).  In 'ev' mode BatchNorm uses
its running moments, so examples are independent and an example only needs the nodes ON ITS OWN PATH:
after every switch the batch is compacted (mpnn_route_compact: first-max argmax, ballot + prefix scan into
per-sink index lists), the activation pyramids of the examples that continue are gathered into the child's
input buffers (mpnn_gather_images) and the child runs on the smaller batch; classifiers are scored only on
the examples that exit at them (mpnn_leaf_stats_targets: correct against the labels, or against y @ w_cls at a
SuperclassCrossEntropyError classifier, binned by the labels).  All sums stay on the device and are read back once
per data set.

The root is a ToPyramid (each scale packed from the image, or from mpnn_lln_counted's output behind a
MultiscaleLLN) or a Conv chain on the image (packed into the dense plan's image slot; the root then runs as an
ordinary node).  Conv blocks run like one-scale stages; ActivityError costs and
Dropout(λ = 1) need no launch in 'ev' mode, and a GlobalMaxPool classifier reads the features of
mpnn_global_maxpool_fwd_counted.  Refused: bf16x3, MaxPool blocks, SquaredError classifiers, Dropout(λ < 1).

Exact for every p_ev-weighted statistic -- acc, moc, and per leaf p_cor, p_inc, p_cor_by_cls, p_inc_by_cls
(what make-acc-eff-plots / make-nlds / make-routing-hists read).  The three entries of `state_tensors` that
are NOT p_ev-weighted (per-leaf c_err and p_tr, per-switch x_rte; train-nets:125-128) are defined on examples
a compacted pass never evaluates: they are absent from its result (use the dense `Engine.eval_stats` for them).

The same walk serves routed inference (`predict`, behind `Net.predict`): at a classifier it writes each
example's softmax, predicted class, exit leaf and path cost (mpnn_leaf_emit_strided: rows of max(n_cls, widest
leaf) columns, a superclass classifier's superclasses zero-filled to that width) instead of adding statistics.
Nets with a per-example k_cpt carry the router feature alpha_cpt * k_cpt through the compaction by original
example id (mpnn_gather_feature), so one batch may mix cost budgets.

Every scale launches the dense eval plan's list of conv passes (`sc.passes`, _Plan._conv_passes) on the node's
inputs: one launch in fp32 and bf16.  In bf16x6 precision the convs read only the (hi | mid | lo) bf16 splits of their
fp32 inputs: the root splits every pyramid scale after packing it, the gathers below a switch move the parent's split
planes, and the passes write fp32 planes, followed by BN / ReLU / pool in fp32 and the counted splits
(mpnn_split_planes3_counted) of what the next convs read.  The heads are the CUDA-core fp32 ones, as in the dense
plan.

One walker serves both ways of running the tree.  Every kernel takes its live batch as a pair (launch batch,
device count) through the counted entry points, and only the step at a switch differs:
  * host-synced (`run_batch`, `predict`): a node runs at its batch n with no count (the uncounted launch).  A switch
    reads its sinks' counts back to the host, because they are the launch batches below it, and walks the non-empty
    sinks on the same stream.
  * graph (`RoutedPredictor`, behind `Net.predictor`): every node is launched in a static order at the capacity
    `batch` and reads its live batch from the parent switch's device-side count (zero for the subtrees no example
    takes).  Sinks 1.. of a switch fork side streams.  The walk has no host round trip, so it is captured once as a
    CUDA graph and replayed per call.
"""
import ctypes
from types import SimpleNamespace as Ns

import numpy as np
import torch

from lib.engine import BF16, _RT_FWD, _gc_off, _vp, node_ops

__all__ = ['CompactEvaluator', 'RoutedPredictor']


class _LeafStats:
    """leaf action of `run_batch`: count every node's examples in `visits` and add each classifier's statistics"""
    def __init__(self, ev):
        self.ev = ev

    def visit(self, nd, n):
        self.ev.visits[nd.idx] += n

    def __call__(self, nd, n, orig, pos, sink_cnt, S):
        ev = self.ev
        r = ev.plan.reg[nd.idx]
        # correct against r.y (the labels, or a superclass leaf's targets y @ w_cls), binned by the labels
        ev.L.leaf_stats_targets(_vp(r.Zbuf), r.ldz, r.n, _vp(r.y), _vp(ev.plan.y), ev.n_cls, _vp(pos), _vp(orig),
                                _vp(sink_cnt), n, _vp(ev.acc[nd.err]), S)


class _LeafEmit:
    """leaf action of prediction: write the results of the examples that exit at each classifier to four device
    arrays, given by the addresses of their first rows"""
    def __init__(self, ev, prob, cls, exit, ops):
        self.ev = ev
        self.out = [ctypes.c_void_p(p) for p in (prob, cls, exit, ops)]

    def visit(self, nd, n):
        pass

    def __call__(self, nd, n, orig, pos, sink_cnt, S):
        ev = self.ev
        r = ev.plan.reg[nd.idx]
        no = ev.leaf_no[nd.idx]
        prob, cls, exit, ops = self.out
        ev.L.leaf_emit_strided(_vp(r.Zbuf), r.ldz, r.n, _vp(pos), _vp(orig), _vp(sink_cnt), n, no, ev.path_ops[no],
                               prob, ev.n_prob, cls, exit, ops, S)


class CompactEvaluator:
    def __init__(self, eng, batch=4096):
        if eng.split == 2:
            raise NotImplementedError('compacted evaluation runs in fp32, bf16 or bf16x6 precision (not bf16x3)')
        if any(getattr(nd, 'maxpool', False) for nd in eng.nodes):
            raise NotImplementedError('compacted evaluation does not cover MaxPool blocks')
        if any(nd.loss not in ('ce', 'sce') for nd in eng.regs):
            # a SquaredError leaf has no softmax: its prob would mean something else
            raise NotImplementedError('compacted evaluation scores Softmax + CrossEntropyError / '
                                      'SuperclassCrossEntropyError classifiers only')
        if any(getattr(nd, 'keep', 1.0) != 1.0 for nd in eng.nodes):
            # the reference applies Dropout in every mode: an 'ev' pass through it is random, and this walk has no mask
            raise NotImplementedError('compacted evaluation does not cover Dropout(λ < 1) blocks')
        self.eng, self.L, self.B = eng, eng.L, int(batch)
        self.plan = plan = eng._plan(self.B, False, False)      # buffers, packed operands, BN constants
        self.n_cls = eng.net.hypers.y_shape[0]
        # columns of predict's prob: a superclass leaf writes its n_out softmax outputs, zero-filled to this width
        self.n_prob = max([self.n_cls] + [plan.reg[nd.idx].n for nd in eng.regs])
        self.sce = [plan.reg[nd.idx] for nd in eng.regs if nd.loss == 'sce']
        B = self.B
        dev = eng.dev
        self.dyn_k = eng.dynamic and bool(eng.net.hypers.dyn_k_cpt)
        # alpha_cpt * k_cpt of the chunk's examples by original id (the dense path's router feature)
        self.kfeat = torch.zeros(B, dtype=torch.float32, device=dev) if self.dyn_k else None
        # per classifier: its index in `net.leaves` and the ops of the nodes on its root-to-leaf path, summed in node
        # order like the dense `moc` (Engine.eval_stats) with a one-hot p_ev
        self.leaf_no = {nd.idx: i for i, nd in enumerate(eng.leaves)}
        self.path_ops = []
        for nd in eng.leaves:
            on_path, i = set(), nd.idx
            while i is not None:
                on_path.add(i)
                i = eng.nodes[i].parent
            tot = 0.0
            for i in sorted(on_path):
                tot += float(node_ops(eng.nodes[i]))
            self.path_ops.append(tot)
        zi = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=dev)
        self.sw = {}
        for nd in eng.nodes:
            if len(nd.kids) > 1:
                ns = len(nd.kids)
                tab = plan._desc_table(_RT_FWD, [plan.rtr[nd.idx].fwd_desc])
                host = torch.zeros(ns, dtype=torch.int32)
                self.sw[nd.idx] = dict(tab=tab, pos=zi(ns, B), orig=zi(ns, B), count=zi(ns),
                                       host=host if eng.dry else host.pin_memory())
        # compacted inputs of every conv stage below a switch: one planes tensor per scale it consumes (bf16x6: the
        # (hi | mid | lo) split planes, the only form of the input its convs read)
        self.cin = {}
        for nd in eng.nodes:
            if nd.kind == 'rcm' and nd.parent is not None and len(eng.nodes[nd.parent].kids) > 1:
                st = plan.node[nd.idx]
                self.cin[nd.idx] = [plan.zeros((3 * s.C // 8, s.geo.P, 8), torch.bfloat16) if eng.split
                                    else plan.planes(s.C, s.geo) for s in st.pin]
        # each router of the CUDA-core heads gets its own k_cpt feature vector: in the graph, sibling subtrees run
        # concurrently
        self._kext = {i: torch.zeros(B, dtype=torch.float32, device=dev) for i in plan.rtr} \
            if self.dyn_k and not plan.umma_heads else {}
        n_leaf = len(eng.regs)
        self.acc = torch.zeros((n_leaf, 2 + 2 * self.n_cls), dtype=torch.float64, device=dev)
        self.visits = np.zeros(len(eng.nodes), np.int64)
        self.n_seen = 0
        self._prepared = False

    # ------------------------------------------------------------------ #
    def reset(self):
        self.acc.zero_()
        self.visits[:] = 0
        self.n_seen = 0
        self._prepared = False            # parameters may have changed since the last data set

    def _S(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.eng.dev).cuda_stream)

    def _prepare(self):
        """once per data set: pack the conv / head operands and turn the running BN moments into scale / shift"""
        eng, plan = self.eng, self.plan
        eng.stream = self._S()
        for op in plan.pack_ops:
            op()
        for op in plan.fwd_ops:
            if getattr(op, 'kind', '') == 'bn_finalize':
                op()
        self._prepared = True

    # ------------------------------------------------------------------ #
    def _k_feature(self, k_cpt, n):
        """alpha_cpt * k_cpt per example as fp32 (the dense feed's arithmetic, Engine._feed), or None for nets with
        a fixed k_cpt; k_cpt is a scalar, one value or n values"""
        hy = self.eng.net.hypers
        if not self.dyn_k:
            if k_cpt is not None:
                raise ValueError('k_cpt is fed to nets with a per-example k_cpt (dyn_k_cpt) only')
            return None
        if k_cpt is None:
            raise ValueError('this net routes on a per-example k_cpt: pass k_cpt (a scalar, one value or n values)')
        if isinstance(k_cpt, torch.Tensor) and k_cpt.is_cuda:      # stays on the device (no host round trip)
            kc = k_cpt.to(torch.float32).reshape(-1)
            if kc.numel() == 1:
                kc = kc.expand(n)
            if kc.numel() != n:
                raise ValueError('k_cpt: %d values for %d examples' % (kc.numel(), n))
            return kc * float(np.float32(hy.α_cpt))                 # fp32 product, as below
        kc = np.asarray(k_cpt, dtype=np.float32).reshape(-1)
        if kc.size == 1:
            kc = np.full(n, kc[0], np.float32)
        if kc.size != n:
            raise ValueError('k_cpt: %d values for %d examples' % (kc.size, n))
        return kc * np.float32(hy.α_cpt)

    def _load(self, x0, n, kf):
        """copy the chunk x0 (n <= batch examples, host or device) and its router features kf (or None) into the
        walk's input buffers"""
        eng = self.eng
        self.plan.x0[:n].copy_(eng._to_dev(x0, (n,) + tuple(eng.net.hypers.x0_shape), 'x0'), non_blocking=True)
        if kf is not None:
            self.kfeat[:n].copy_(torch.as_tensor(kf), non_blocking=True)

    def _walk(self, live, leaf, split):
        """run the loaded chunk down the tree on the current stream.  live: its (launch batch, device count), (n, None)
        or (B, count of the chunk); leaf: the leaf action; split: the switch step"""
        eng, plan, L = self.eng, self.plan, self.L
        H0, W0, C0 = eng.net.hypers.x0_shape
        stream = torch.cuda.current_stream(eng.dev)
        S = ctypes.c_void_p(stream.cuda_stream)
        root = eng.nodes[0]
        pyr = root.kind == 'pyr'
        # the pyramid's scales, or the image a Conv chain at the root reads (the dense plan's _image_slot)
        lln = getattr(root, 'lln', None)
        for i, slot in enumerate(plan.node[0].out if pyr else plan._image_slot().out):
            g = slot.geo
            src, H, W, step = plan.x0, H0, W0, 2 ** i
            if lln is not None:                     # MultiscaleLLN: normalise the scale, then pack the fp32 result
                L.lln_counted(_vp(plan.x0), live[0], H0, W0, C0, step, float(lln.hypers.σ), float(lln.hypers.ϵ),
                              _vp(slot.lln), _vp(live[1]), S)
                src, H, W, step = slot.lln, g.H, g.W, 1
            L.pack_input_counted(_vp(src), live[0], H, W, C0, step, _vp(slot.t), min(slot.C, (C0 + 7) // 8 * 8),
                                 g.G, g.P, eng.dtype, _vp(live[1]), S)
            if eng.split:
                L.split_planes3_counted(_vp(slot.t), slot.C, live[0], g.H, g.W, g.G, g.P, _vp(slot.split),
                                        _vp(live[1]), S)
        if live[0] == 0:                            # run_batch of no examples
            leaf.visit(root, 0)
            return
        if not pyr:                                 # a Conv chain at the root: an ordinary node
            self._node(root, live, live, None, None, live[1], stream, leaf, split)
            return
        leaf.visit(root, live[0])
        for k in root.kids:
            self._node(eng.nodes[k], live, live, None, None, live[1], stream, leaf, split)

    def run_batch(self, x0, y, k_cpt=None):
        """accumulate the statistics of one batch (n <= batch examples; host or device arrays).  k_cpt (nets with a
        per-example k_cpt only): a scalar, one value or one per example."""
        eng, plan = self.eng, self.plan
        if not eng.dynamic:
            raise ValueError('compacted evaluation is for dynamically-routed nets (an SRNet has one path)')
        n = int(x0.shape[0])
        if n > self.B:
            raise ValueError('batch %d > evaluator capacity %d' % (n, self.B))
        kf = self._k_feature(k_cpt, n)
        with torch.cuda.device(eng.dev):
            if not self._prepared:
                self._prepare()
            y = eng._to_dev(y, (n,) + tuple(eng.net.hypers.y_shape), 'y')
            plan.y[:n].copy_(y, non_blocking=True)
            for r in self.sce if n else ():         # a superclass leaf is scored against y @ w_cls of these labels
                self.L.superclass_targets(_vp(plan.y), _vp(r.w_cls), n, self.n_cls, r.n, _vp(r.y), self._S())
            self.n_seen += n
            self._load(x0, n, kf)
            self._walk((n, None), _LeafStats(self), self._host_split)

    def _check_x0(self, x0):
        hy = self.eng.net.hypers
        if tuple(x0.shape[1:]) != tuple(hy.x0_shape):
            raise ValueError('x0: shape %s, expected (n,) + %s' % (tuple(x0.shape), tuple(hy.x0_shape)))
        return int(x0.shape[0])

    def predict(self, x0, k_cpt=None):
        """Routed inference (see `Net.predict`): Ns(cls, prob, exit, ops) of numpy arrays, one row per example of x0
        (any n, host or device), run in chunks of `batch` examples."""
        eng = self.eng
        n = self._check_x0(x0)
        kf = self._k_feature(k_cpt, n)
        nc = self.n_prob
        # one byte buffer holds the four outputs, so that one device-to-host copy returns them
        o_prob = 8 * n
        o_cls = o_prob + 4 * n * nc
        o_exit = o_cls + 4 * n
        nbytes = o_exit + 4 * n
        if n == 0:
            host = np.zeros(nbytes, np.uint8)
        else:
            with torch.cuda.device(eng.dev):
                self._prepare()                      # every call: the current parameters and running moments
                buf = torch.empty(nbytes, dtype=torch.uint8, device=eng.dev)
                kfd = torch.as_tensor(kf).to(eng.dev, non_blocking=True) if kf is not None else None
                p = buf.data_ptr()
                for b0 in range(0, n, self.B):
                    m = min(self.B, n - b0)
                    self._load(x0[b0:b0 + m], m, kfd[b0:b0 + m] if kfd is not None else None)
                    emit = _LeafEmit(self, p + o_prob + 4 * nc * b0, p + o_cls + 4 * b0, p + o_exit + 4 * b0, p + 8 * b0)
                    self._walk((m, None), emit, self._host_split)
                host = buf.cpu().numpy()
        return Ns(cls=host[o_cls:o_exit].view(np.int32), prob=host[o_prob:o_cls].view(np.float32).reshape(n, nc),
                  exit=host[o_exit:nbytes].view(np.int32), ops=host[:o_prob].view(np.float64))

    def _host_split(self, nd, sw, stream):
        """switch step of the host-synced walk: the sinks' counts are the launch batches below them, so they are read
        back; the non-empty sinks run one after another on the switch's stream"""
        sw['host'].copy_(sw['count'], non_blocking=True)
        stream.synchronize()
        for s, c in enumerate(sw['host'].tolist()):
            if c:
                yield s, (c, None), stream

    # ------------------------------------------------------------------ #
    def _node(self, nd, live, par, orig, pos, sink_cnt, stream, leaf, split):
        """Run node `nd` and its subtree on `stream`.  live / par: the (launch batch, device count or None) of this
        node's examples and of its parent's compact batch; orig / pos: the examples' original ids and rows in the
        parent's compact batch (None = identity, no switch above); sink_cnt: the device count of the switch sink (or
        of the chunk) the examples come from, which the gathers and the leaf action read; leaf: the leaf action;
        split(nd, sw, stream): the switch step, yields (sink, its live pair, its stream) for the sinks to run."""
        eng, plan, L = self.eng, self.plan, self.L
        dt = eng.dtype
        n, cnt = live
        S = ctypes.c_void_p(stream.cuda_stream)
        leaf.visit(nd, n)
        if nd.kind == 'reg':
            if not plan.umma_heads:
                pst = plan.node[nd.parent]
                r = plan.reg[nd.idx]
                # logits of the parent's compact batch (rows of the examples that exit here are read through pos)
                L.fc_fwd_counted(_vp(pst.feat), pst.F, plan.Balloc, par[0], eng.tptr(r.fc.params.w),
                                 eng.tptr(r.fc.params.b), None, r.n, _vp(r.Zbuf), dt, _vp(par[1]), S)
            leaf(nd, n, orig, pos, sink_cnt, S)
            return
        st = plan.node[nd.idx]
        x6 = bool(eng.split)                        # bf16x6: the convs read the split planes only
        ins = [s.split if x6 else s.t for s in st.pin]
        if pos is not None:                         # below a switch: gather the inputs of the examples that continue
            for slot, src, dst in zip(st.pin, ins, self.cin[nd.idx]):
                g = slot.geo
                L.gather_images(_vp(src), par[0], g.P, _vp(pos), _vp(sink_cnt), _vp(dst), n, g.P,
                                3 * slot.C if x6 else slot.C, g.H, g.W, g.G, BF16 if x6 else dt, S)
            ins = self.cin[nd.idx]
        rt = plan.rtr.get(nd.idx)
        if self.dyn_k and rt is not None:           # the router's k_cpt feature, in this node's compact order
            if plan.umma_heads:                      # channel 0 of the extra planes of the head GEMM's input
                L.gather_feature(_vp(self.kfeat), _vp(orig), _vp(sink_cnt), n, None, _vp(st.feat[st.F // 8, :, 0]), 8,
                                 dt, S)
            else:
                L.gather_feature(_vp(self.kfeat), _vp(orig), _vp(sink_cnt), n, _vp(self._kext[nd.idx]), None, 0, 0, S)
        for k, sc in enumerate(st.sc):
            g = sc.geo
            prev = st.sc[k - 1] if k > 0 else None
            for ps in sc.passes:                    # the dense plan's conv launches (Plan._conv_passes)
                A0, K0, A1, K1 = plan.pass_operands(sc, prev, ps, h=ins[k])
                L.stencil_gemm_counted(_vp(A0), K0, _vp(A1), K1, _vp(ps.W), 9, eng.tptr(sc.bk) if ps.first else None,
                                       _vp(sc.lin), sc.N, 0 if ps.first else 1, None, 0, 0, n, g.H, g.W, g.G, g.P,
                                       None, 0, None, *plan.conv_dtypes, _vp(cnt), S)
            if sc.live or sc.pooled is not None:
                L.bn_relu_pool_fwd_counted(_vp(sc.lin), sc.N, n, g.H, g.W, g.G, g.P, _vp(sc.ss) if sc.live else None,
                                           _vp(sc.act), _vp(sc.pooled), sc.geo_p.P if sc.pooled is not None else 0,
                                           _vp(sc.feat), plan.Balloc, dt, _vp(cnt), S)
                if x6:                              # the split operands of the convs that read act / pooled
                    if sc.act_split is not None:
                        L.split_planes3_counted(_vp(sc.act), sc.N, n, g.H, g.W, g.G, g.P, _vp(sc.act_split), _vp(cnt), S)
                    if sc.pooled_split is not None:
                        q = sc.geo_p
                        L.split_planes3_counted(_vp(sc.pooled), sc.N, n, q.H, q.W, q.G, q.P, _vp(sc.pooled_split),
                                                _vp(cnt), S)
            # (Dropout(λ = 1) is the identity, and an ActivityError cost enters the training objective only)
            if getattr(nd, 'gmp', False):           # the GlobalMaxPool classifier's features, without the argmax
                L.global_maxpool_fwd_counted(_vp(sc.act), sc.N, n, g.H, g.W, g.G, g.P, _vp(st.feat), None, plan.Balloc,
                                             dt, _vp(cnt), S)
        if not nd.kids:
            return
        if plan.umma_heads and nd.idx in plan.heads:
            hd = plan.heads[nd.idx]
            o0, n0, o1, n1 = hd.outs
            L.stencil_gemm_counted(_vp(st.feat), st.Fext, None, 0, _vp(hd.Wfc), 1, _vp(hd.bias), _vp(o0), n0, 0,
                                   _vp(o1), n1, 0, n, 0, 0, 0, plan.Balloc, None, 0, None, BF16, 2, 1, _vp(cnt), S)
        elif rt is not None:
            L.fc_fwd_counted(_vp(st.feat), st.F, plan.Balloc, n, eng.tptr(rt.fc1.params.w), eng.tptr(rt.fc1.params.b),
                             _vp(self._kext[nd.idx]) if self.dyn_k else None, eng.router_width, _vp(rt.Z1), dt,
                             _vp(cnt), S)
        if len(nd.kids) == 1:                       # no switch: the only sink sees every example of this node
            self._node(eng.nodes[nd.kids[0]], live, live, orig, None, cnt, stream, leaf, split)
            return
        sw = self.sw[nd.idx]
        ns = len(nd.kids)
        L.router_tail_fwd_batched_counted(_vp(sw['tab']), 1, n, eng.router_width, float(rt.bn1.hypers.d),
                                          float(rt.bn1.hypers.ε), 0, _vp(cnt), S)
        L.route_compact_counted(_vp(rt.R), ns, ns, n, _vp(orig), self.B, None, _vp(sw['pos']), _vp(sw['orig']),
                                _vp(sw['count']), _vp(cnt), S)
        for s, sink, sink_stream in split(nd, sw, stream):
            self._node(eng.nodes[nd.kids[s]], sink, live, sw['orig'][s], sw['pos'][s], sw['count'][s:s + 1],
                       sink_stream, leaf, split)

    # ------------------------------------------------------------------ #
    def result(self):
        """{(object, name): mean over the data set} in `mean_net_state`'s form (desc.py:10-22) for the exact keys"""
        eng = self.eng
        n = max(self.n_seen, 1)
        a = self.acc.cpu().numpy() / n                       # the one device-to-host read of the data set
        nc = self.n_cls
        out = {}
        acc = 0.0
        for nd in eng.regs:
            row = a[nd.err]
            l = nd.layer
            out[(l, 'p_cor')] = float(row[0])
            out[(l, 'p_inc')] = float(row[1])
            out[(l, 'p_cor_by_cls')] = row[2:2 + nc].tolist()
            out[(l, 'p_inc_by_cls')] = row[2 + nc:2 + 2 * nc].tolist()
            acc += float(row[0])
        moc = 0.0
        for nd in eng.nodes:
            moc += self.visits[nd.idx] * float(node_ops(nd))
        out[(eng.net, 'acc')] = acc
        out[(eng.net, 'moc')] = moc / n
        return out


class RoutedPredictor:
    """Routed inference as one CUDA graph (see `Net.predictor`).  `p(x0, k_cpt=None)` runs n <= batch examples and
    returns Ns(cls, prob, exit, ops) of device tensors with the dtypes and meaning of `Net.predict`.  They are views
    [:n] of the predictor's own output buffers: the next call overwrites them (clone what you keep).

    A call copies x0 into the walk's input buffer, writes n and the per-example router feature with device copies,
    and replays the graph on the current stream: with device inputs it does not synchronise the host.  The graph
    starts with the weight packing and the BatchNorm constants of the running moments (what `predict` runs before its
    walk), so every call sees the current parameters."""

    def __init__(self, ev):
        self.ev, eng = ev, ev.eng
        self.B = ev.B
        dev = eng.dev
        B, nc = ev.B, ev.n_prob
        self.n_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.cls = torch.zeros(B, dtype=torch.int32, device=dev)
        self.prob = torch.zeros((B, nc), dtype=torch.float32, device=dev)
        self.exit = torch.zeros(B, dtype=torch.int32, device=dev)
        self.ops = torch.zeros(B, dtype=torch.float64, device=dev)
        self._out = _LeafEmit(ev, self.prob.data_ptr(), self.cls.data_ptr(), self.exit.data_ptr(), self.ops.data_ptr())
        self._side = {}
        self._joins = []
        self.graph = None
        self.graph_launches = 0

    def _split(self, nd, sw, stream):
        """switch step of the graph: every sink runs at the capacity with its device count.  Sink 0 continues on the
        switch's stream and the others fork side streams, so the graph's critical path is one root-to-leaf chain."""
        ev = torch.cuda.Event()
        ev.record(stream)
        for s in range(len(nd.kids)):
            st = stream
            if s > 0:
                if (nd.idx, s) not in self._side:
                    self._side[(nd.idx, s)] = torch.cuda.Stream(self.ev.eng.dev)
                st = self._side[(nd.idx, s)]
                st.wait_event(ev)
                self._joins.append(st)
            yield s, (self.B, sw['count'][s:s + 1]), st

    def _ops(self):
        ev = self.ev
        main = torch.cuda.current_stream(ev.eng.dev)
        ev._prepare()
        self._joins = []
        ev._walk((self.B, self.n_dev), self._out, self._split)
        for st in self._joins:                   # every side stream rejoins the origin (required under capture)
            main.wait_stream(st)

    def _capture(self):
        eng = self.ev.eng
        s = torch.cuda.Stream(eng.dev)
        s.wait_stream(torch.cuda.current_stream(eng.dev))
        with torch.cuda.stream(s):               # warm-up: lazy module loads and per-kernel attributes stay out of capture
            self._ops()
        torch.cuda.current_stream(eng.dev).wait_stream(s)
        torch.cuda.synchronize(eng.dev)
        g = torch.cuda.CUDAGraph()
        before = eng.L.launches
        with _gc_off():
            with torch.cuda.graph(g):
                self._ops()
        self.graph_launches = eng.L.launches - before
        self.graph = g

    def __call__(self, x0, k_cpt=None):
        ev = self.ev
        n = ev._check_x0(x0)
        if n > self.B:
            raise ValueError('batch %d > predictor capacity %d' % (n, self.B))
        kf = ev._k_feature(k_cpt, n)
        if n > 0:
            with torch.cuda.device(ev.eng.dev):
                if self.graph is None:
                    self._capture()
                ev._load(x0, n, kf)
                self.n_dev.fill_(n)
                self.graph.replay()
        return Ns(cls=self.cls[:n], prob=self.prob[:n], exit=self.exit[:n], ops=self.ops[:n])
