"""Routed inference (`net.predict`, and `net.predictor`, the same walk replayed as one CUDA graph) against the dense
'ev' forward (`Engine.forward` on an eval plan) on cifar10-ac at the real architecture in bf16 (or --precision fp32 /
bf16x6), for three router settings and B in {128, 4096, 16384}:

  (a) fresh net: the zero-initialised last router layer ties, every example exits at stage 0;
  (b) every switch biased to continue: every example runs the whole chain (worst case for the compaction);
  (c) randomized routers (tests/util.py::randomize_routers).

CUDA events around each call, warm-up first, the two paths alternated in one process, and a 256 MB buffer
rewritten before every timed call so that no path reads its inputs or weights from L2 (126 MB).  Reports
ms per call (median of the repeats), images/s, mean ops as a fraction of the whole tree, the exit histogram,
the host synchronisations of one predict call (one per switch visited per chunk, plus the final read-back) and
those of one predictor call with device inputs (counted by torch's sync debug mode)."""
import argparse
import os
import subprocess
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import arch_and_hypers as ah  # noqa: E402
from lib import layer_types  # noqa: E402
from util import randomize_routers  # noqa: E402

BATCHES = [int(b) for b in os.environ.get('BATCHES', '128,4096,16384').split(',')]
REPS = int(os.environ.get('REPS', 10))


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else 'nvidia-smi failed'


def make_net(setting, precision):
    layer_types.seed(0)
    net = ah.ac_chain(k_cpt=4e-9)((32, 32, 3), (10,))
    if setting == 'continue':
        for l in net.layers:
            if l.router is not None:
                last = l.router.comps[-1]
                last.params.w.assign(np.zeros(last.params.w.shape, np.float32))
                b = np.zeros(last.params.b.shape, np.float32)
                b[1:] = 1.0                                 # sink 0 is the stage's classifier, sink 1 the next stage
                last.params.b.assign(b)
    elif setting == 'random':
        randomize_routers(net)
    return net.configure(precision=precision)


def switches_visited(eng, exit_, B):
    """host synchronisations of one predict call: per chunk, every switch that some example of the chunk reaches"""
    below = {}
    for i, leaf in enumerate(eng.leaves):
        j = eng.nodes[leaf.idx].parent
        while j is not None:
            below.setdefault(j, set()).add(i)
            j = eng.nodes[j].parent
    n = 0
    for b0 in range(0, len(exit_), B):
        seen = set(exit_[b0:b0 + B].tolist())
        n += sum(1 for sw in eng.switches if below[sw.idx] & seen)
    return n + 1


def predictor_syncs(call):
    """host synchronisations torch sees during one call"""
    torch.cuda.synchronize()
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        torch.cuda.set_sync_debug_mode('warn')
        try:
            call()
        finally:
            torch.cuda.set_sync_debug_mode(0)
    return sum('called a synchronizing' in str(x.message) for x in w)        # not the mode's own prototype notice


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32', 'bf16x6'])
    args = ap.parse_args()
    torch.cuda.init()
    print('card (name, power limit, max SM clock): %s' % card())
    rng = np.random.default_rng(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    print('%-9s %6s %10s %10s %10s %11s %11s %11s %7s %7s %8s %6s %6s  %s' % (
        'routers', 'B', 'dense ms', 'predict', 'predictor', 'dense im/s', 'predict', 'predictor', 'x pred', 'x dense',
        'ops frac', 'syncs', 'graph', 'exits'))
    for setting in ('fresh', 'continue', 'random'):
        net = make_net(setting, args.precision)
        eng = net._get_engine()
        ops_tree = float(sum(l.n_ops + (l.router.n_ops if l.router is not None else 0) for l in net.layers))
        for B in BATCHES:
            x0 = torch.from_numpy(rng.random((B, 32, 32, 3), dtype=np.float32)).cuda()
            y = torch.from_numpy(np.eye(10, dtype=np.float32)[rng.integers(0, 10, B)]).cuda()
            feed = {net.x0: x0, net.y: y, net.τ: 0.5}
            dense = lambda: eng.forward(feed, 'ev')
            routed = lambda: net.predict(x0, batch=B)
            graph = lambda: net.predictor(B)(x0)

            def timed(fn):
                flush.fill_(1)
                ev0.record()
                r = fn()
                ev1.record()
                ev1.synchronize()
                return ev0.elapsed_time(ev1), r
            for _ in range(3):                                # warm-up: plans, packing, module loads, graph capture
                timed(dense), timed(routed), timed(graph)
            t_d, t_p, t_g = [], [], []
            for _ in range(REPS):                             # alternated
                t_d.append(timed(dense)[0])
                t, r = timed(routed)
                t_p.append(t)
                t, g = timed(graph)
                t_g.append(t)
            assert g.exit.cpu().numpy().tobytes() == r.exit.tobytes()
            md, mp, mg = float(np.median(t_d)), float(np.median(t_p)), float(np.median(t_g))
            hist = np.bincount(r.exit, minlength=len(eng.leaves))
            print('%-9s %6d %10.3f %10.3f %10.3f %11.0f %11.0f %11.0f %7.2f %7.2f %8.3f %6d %6d  %s' % (
                setting, B, md, mp, mg, B / md * 1e3, B / mp * 1e3, B / mg * 1e3, mp / mg, md / mg,
                r.ops.mean() / ops_tree, switches_visited(eng, r.exit, B), predictor_syncs(graph), hist.tolist()),
                flush=True)
        del net, eng
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
