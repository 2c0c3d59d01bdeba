"""Dense 'ev'-mode statistics on the device: `mean_net_state` (lib/desc.py) for EVERY key of `state_tensors`, from
graph-replayed forwards at a batch that fills the GPU.

The host path (`Engine.eval_stats`) runs an eager dense forward per 128-example slice and reads about two dozen small
tensors back per slice.  Here one chunk of up to `batch` examples is one replay of a CUDA graph that holds

    the plan's pack ops   weight packing and SuperclassCrossEntropyError targets (they read this chunk's labels),
    the plan's fwd ops    the dense 'ev' forward at the capacity, BatchNorm constants from the current running moments,
    one accumulate launch mpnn_stats_accumulate: the chunk's per-example statistics, summed in a fixed order into a
                          device fp64 total,

so every chunk sees the current parameters and its own labels, and the only device-to-host read of a data set is the
one in `result()`.  The live n is a device int: the forward runs at the capacity (in 'ev' mode the examples are
independent) and rows at or past n are never summed.

Against the host path the count-valued statistics (p_cor, p_inc, the per-class entries, acc, moc: sums of integers in
fp64) have the same bits; c_err, p_tr and x_rte differ only by summation order.
"""
import ctypes

import numpy as np
import torch

from lib.engine import _gc_off, _struct, _vp, node_ops

__all__ = ['DenseStatsEvaluator']

# mpnn_stats_desc (include/mpnn.h)
_STATS = _struct(['p_ev', 'p_tr', 'd_cor', 'c_err', 'R'], ['ns', 'reserved'])
_STATS_ROWS = 32                       # MPNN_STATS_ROWS (include/mpnn.h)
assert _STATS.itemsize == 48


class DenseStatsEvaluator:
    def __init__(self, eng, batch=4096):
        if any(getattr(nd, 'keep', 1.0) != 1.0 for nd in eng.nodes):
            # the reference applies Dropout in every mode; the masks hash the example's position in the batch and the
            # per-evaluation draw, so a pass at another chunking would be another random draw
            raise NotImplementedError('device statistics do not cover Dropout(λ < 1) blocks: their masks depend on the '
                                      'batch layout and the per-evaluation draw')
        self.eng, self.B = eng, int(batch)
        if self.B < 1:
            raise ValueError('capacity %d < 1' % self.B)
        self.plan = plan = eng._plan(self.B, False, False)
        self.n_cls = eng.net.hypers.y_shape[0]
        self.per_leaf = 4 + 2 * self.n_cls
        n_leaf, n_sw = len(eng.regs), len(eng.switches)
        self.M = n_leaf * self.per_leaf + n_sw + 2
        dev = eng.dev
        rows = []
        for nd in eng.regs:
            r = plan.reg[nd.idx]
            rows.append(dict(p_ev=plan.p_ev[nd.idx] if eng.dynamic else None,
                             p_tr=plan.p_tr[nd.idx] if eng.dynamic else None, d_cor=r.d_cor, c_err=r.c_err, ns=0))
        for nd in eng.switches:
            rows.append(dict(R=plan.rtr[nd.idx].R, ns=len(nd.kids)))
        self.tab = plan._desc_table(_STATS, rows)
        self.ops = torch.tensor([float(node_ops(nd)) for nd in eng.nodes], dtype=torch.float64, device=dev)
        self.work = torch.zeros(-(-self.B // _STATS_ROWS) * self.M, dtype=torch.float64, device=dev)
        self.total = torch.zeros(self.M, dtype=torch.float64, device=dev)
        self.n_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        node_p_ev = plan.p_ev if eng.dynamic else None
        L = eng.L

        def accumulate():
            L.stats_accumulate(_vp(self.tab), n_leaf, n_sw, _vp(plan.y), self.n_cls, _vp(node_p_ev), _vp(self.ops),
                               len(eng.nodes), self.B, _vp(self.work), _vp(self.total), _vp(self.n_dev), eng.stream)
        accumulate.kind = 'stats_accumulate'
        # one chunk: the dense eval plan's pack and forward ops, then the accumulate launch (each list is issued by
        # Engine._run, which joins its lanes at the end, so the accumulate launch follows the whole forward)
        self.op_lists = (plan.pack_ops, plan.fwd_ops, [accumulate])
        self.graph = None
        self.graph_launches = 0
        self.n_seen = 0

    # ------------------------------------------------------------------ #
    def reset(self):
        if not self.eng.dry:
            self.total.zero_()
        self.n_seen = 0

    def _ops(self):
        for ops in self.op_lists:
            self.eng._run(ops)

    def _capture(self):
        eng = self.eng
        self.n_dev.zero_()                       # the warm-up adds nothing
        s = torch.cuda.Stream(eng.dev)
        s.wait_stream(torch.cuda.current_stream(eng.dev))
        with torch.cuda.stream(s):               # warm-up: lazy module loads, the engine's lanes
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

    def run_batch(self, x0, y, hypers={}):
        """add the statistics of n <= batch examples (x0, y: numpy or torch, host or device).  hypers: the feed of
        `mean_net_state` (tau, eps, k_cpt: one value or n values).  With device inputs nothing synchronises the host."""
        eng = self.eng
        hy = eng.net.hypers
        n = int(x0.shape[0])
        if n > self.B:
            raise ValueError('batch %d > evaluator capacity %d' % (n, self.B))
        x0 = eng._to_dev(x0, (n,) + tuple(hy.x0_shape), 'x0')
        y = eng._to_dev(y, (n,) + tuple(hy.y_shape), 'y')
        if n == 0:
            return
        if eng.dry:
            raise RuntimeError('dry-run engine cannot execute: the hot path is CUDA-only')
        plan = self.plan
        with torch.cuda.device(eng.dev):
            if self.graph is None:
                self._capture()
            plan.x0[:n].copy_(x0, non_blocking=True)
            plan.y[:n].copy_(y, non_blocking=True)
            eng._feed_hyp(plan, hypers, n)
            self.n_dev.fill_(n)
            self.graph.replay()
        self.n_seen += n

    def result(self):
        """{key: mean over the examples run since `reset`} for every key of `state_tensors(net)`, in the form of
        `mean_net_state` (python floats, lists for the per-class entries)"""
        eng = self.eng
        tot = self.total.cpu().numpy()              # the one device-to-host read of the data set
        n = max(self.n_seen, 1)
        nc, pl = self.n_cls, self.per_leaf
        out = {}
        for e, nd in enumerate(eng.regs):
            row, l = tot[e * pl:(e + 1) * pl], nd.layer
            out[(l, 'p_cor')] = (row[0] / n).tolist()
            out[(l, 'p_inc')] = (row[1] / n).tolist()
            out[(l, 'p_cor_by_cls')] = (row[4:4 + nc] / n).tolist()
            out[(l, 'p_inc_by_cls')] = (row[4 + nc:4 + 2 * nc] / n).tolist()
            if eng.dynamic:
                out[(l, 'p_tr')] = (row[3] / n).tolist()
            out[(l, 'c_err')] = (row[2] / n).tolist()
        base = len(eng.regs) * pl
        for s, nd in enumerate(eng.switches):
            out[(nd.layer, 'x_rte')] = (tot[base + s] / n).tolist()
        out[(eng.net, 'acc')] = (tot[base + len(eng.switches)] / n).tolist()
        out[(eng.net, 'moc')] = (tot[base + len(eng.switches) + 1] / n).tolist()
        return out
