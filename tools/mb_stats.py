"""One full statistics pass (`net_desc`: the training and the test split) on the host path against the device path,
for cifar10-ac and cifar10-sr at the real architecture in bf16 and fp32, on synthetic CIFAR-shaped sets of 50 k / 10 k
examples.

  host    `net_desc(...)`: Engine.eval_stats per 128-example slice (eager dense 'ev' forward, per-slice read-back,
          NumPy sums) -- what train-nets runs by default every t_log steps
  device  `net_desc(..., device=True)`: graph-replayed dense forward + mpnn_stats_accumulate per 4096-example chunk,
          both splits resident in HBM, one read-back per split (lib/dense_stats.py)

Wall clock around each whole pass (both paths end in a device-to-host read, so the clock covers the device work), one
warm-up pass of each path first (graph capture, upload of the resident splits), then the two paths alternated REPS
times in this process; the median is reported.  The card's name and power limit are read in the same run.  The data
set (615 MB of fp32 training images) exceeds the 126 MB L2, so neither path reads its inputs from L2 across passes.
Also checks that the two passes agree (count keys bit-identical, the rest within 1e-12 relative)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import arch_and_hypers as ah  # noqa: E402
from lib import layer_types  # noqa: E402
from lib.data import Dataset, synthetic_archive  # noqa: E402
from lib.desc import net_desc, state_tensors  # noqa: E402
from util import randomize_routers  # noqa: E402

COUNT_KEYS = ('p_cor', 'p_inc', 'p_cor_by_cls', 'p_inc_by_cls', 'acc', 'moc')


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else 'nvidia-smi failed'


def worst_difference(a, b):
    """(count keys identical, largest relative difference of c_err / p_tr / x_rte)"""
    same, worst = True, 0.0

    def walk(x, y, key=None):
        nonlocal same, worst
        if isinstance(x, dict):
            for k in x:
                walk(x[k], y[k], k)
        elif isinstance(x, list) and x and isinstance(x[0], dict):
            for u, v in zip(x, y):
                walk(u, v)
        elif key in COUNT_KEYS:
            same = same and x == y
        elif key in ('c_err', 'p_tr', 'x_rte'):
            worst = max(worst, abs(x - y) / max(abs(y), 1e-300))
    walk(a, b)
    return same, worst


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--n-train', type=int, default=50000)
    ap.add_argument('--n-test', type=int, default=10000)
    ap.add_argument('--out', help='also write the result lines to this JSON file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('mb_stats: needs a CUDA device')
    line = card()
    print('card: %s' % line, flush=True)
    ds = Dataset(archive=synthetic_archive(args.n_train, args.n_test, (32, 32, 3), 10, seed=0), seed=0)
    rows = []
    for kind in ('cifar10-ac', 'cifar10-sr'):
        for prec in ('bf16', 'fp32'):
            layer_types.seed(0)
            ctor = ah.ac_chain(k_cpt=4e-9) if kind == 'cifar10-ac' else ah.sr_chain(len(ah.arch))
            net = ctor((32, 32, 3), (10,)).configure(precision=prec, graphs=True)
            if net.dynamic:
                randomize_routers(net)
            h, state = ({net.τ: 0.5} if net.dynamic else {}), state_tensors(net)
            paths = {'host': lambda: net_desc(net, ds, h, state),
                     'device': lambda: net_desc(net, ds, h, state, device=True)}
            out = {p: f() for p, f in paths.items()}                 # warm-up
            same, worst = worst_difference(out['device'], out['host'])
            times = {p: [] for p in paths}
            for r in range(args.reps):
                for p, f in paths.items():
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    f()
                    torch.cuda.synchronize()
                    times[p].append(time.perf_counter() - t0)
            med = {p: statistics.median(v) for p, v in times.items()}
            n = args.n_train + args.n_test
            row = dict(net=kind, precision=prec, examples=n, host_s=med['host'], device_s=med['device'],
                       host_all=times['host'], device_all=times['device'], speedup=med['host'] / med['device'],
                       device_images_per_s=n / med['device'], count_keys_identical=same, worst_rel_diff=worst,
                       card=line)
            rows.append(row)
            print('%-10s %-5s  host %.3f s  device %.3f s  (x%.1f, %.2f M images/s)  count keys identical: %s, '
                  'c_err/p_tr/x_rte within %.1e' % (kind, prec, med['host'], med['device'], row['speedup'],
                                                     row['device_images_per_s'] / 1e6, same, worst), flush=True)
            del net
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
