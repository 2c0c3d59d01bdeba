"""Cost of wider routers (arch_and_hypers.router_n_chan = 16, 32, 64) on the B200:

  (1) router-tail kernels alone: one batched forward (train mode) and one batched backward launch for the 7 two-way
      routers of cifar10-ac, at B = 128 and 4096; CUDA events around REPS back-to-back launches, after a warm-up;
  (2) the cifar10-ac training step in bf16 at the same batches, timed like bench.py (bench.Run.device_timed: the
      batch resident in HBM, one event pair per CUDA-graph step, a 256 MB buffer rewritten between steps so that no
      step reads L2-resident data).

Prints the card's name, power limit and max SM clock first, then one line per measurement."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'multipath-nn_b200'), os.path.join(ROOT, 'tests')]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import arch_and_hypers as ah  # noqa: E402
import bench  # noqa: E402
from lib import _cabi  # noqa: E402
from lib.engine import _RT_BWD, _RT_FWD  # noqa: E402

WIDTHS = [int(w) for w in os.environ.get('WIDTHS', '16,32,64').split(',')]
BATCHES = [int(b) for b in os.environ.get('BATCHES', '128,4096').split(',')]
REPS = int(os.environ.get('REPS', 200))
STEPS = int(os.environ.get('STEPS', 50))
N_ROUTERS, NS = 7, 2


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else 'nvidia-smi failed'


def tail_tables(W, B, keep):
    """descriptor tables of N_ROUTERS tails of width W on random data (forward train mode, then backward)"""
    rng = np.random.default_rng(W + B)
    f = lambda *sh, s=1.0: keep.append(torch.tensor(rng.standard_normal(sh).astype(np.float32) * s,
                                                    device='cuda')) or keep[-1]
    z = lambda *sh: keep.append(torch.zeros(sh, device='cuda')) or keep[-1]
    fr, br = [], []
    Balloc = -(-B // 128) * 128
    for _ in range(N_ROUTERS):
        P = dict(Z1=f(B, W), g1=f(W), b1=f(W), m1=z(W), v1=f(W) ** 2 + 1, W2=f(W, W, s=W ** -0.5), c2=f(W), g2=f(W),
                 b2=f(W), m2=z(W), v2=f(W) ** 2 + 1, W3=f(W, NS), c3=f(NS), Z2=z(B, W), R=z(B, NS), save=z(4 * W),
                 dR=f(B, NS), dZ1=z(B, W), dZ1p=keep.append(torch.zeros((W // 8, Balloc, 8), dtype=torch.bfloat16,
                                                                       device='cuda')) or keep[-1])
        keep.append(P)
        g = {k: z(*P[k].shape) for k in ('g1', 'b1', 'W2', 'c2', 'g2', 'b2', 'W3', 'c3')}
        p = lambda k: P[k].data_ptr()
        fr.append((p('Z1'), p('g1'), p('b1'), p('m1'), p('v1'), p('W2'), p('c2'), p('g2'), p('b2'), p('m2'), p('v2'),
                   p('W3'), p('c3'), p('Z2'), p('R'), p('save'), NS, 0))
        br.append((p('Z1'), p('Z2'), p('dR'), p('g1'), p('b1'), p('W2'), p('g2'), p('b2'), p('W3'), p('save'),
                   g['g1'].data_ptr(), g['b1'].data_ptr(), g['W2'].data_ptr(), g['c2'].data_ptr(), g['g2'].data_ptr(),
                   g['b2'].data_ptr(), g['W3'].data_ptr(), g['c3'].data_ptr(), p('dZ1'), 0, p('dZ1p'),
                   0, NS, Balloc))
    tab = lambda rows, dt: torch.tensor(np.frombuffer(np.array(rows, dtype=dt).tobytes(), np.uint8).copy(), device='cuda')
    return tab(fr, _RT_FWD), tab(br, _RT_BWD)


def time_launches(launch):
    for _ in range(20):
        launch()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(REPS):
        launch()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1000.0 / REPS


def main():
    L = _cabi.lib()
    vp = lambda t: __import__('ctypes').c_void_p(t.data_ptr())
    print('# card (name, power limit, max SM clock):', card(), flush=True)
    for B in BATCHES:
        for W in WIDTHS:
            keep = []
            tf, tb = tail_tables(W, B, keep)
            fwd = time_launches(lambda: L.router_tail_fwd_batched(vp(tf), N_ROUTERS, B, W, 0.9, 1e-6, 1, None))
            bwd = time_launches(lambda: L.router_tail_bwd_batched(vp(tb), N_ROUTERS, B, W, None))
            print('tails   B=%5d W=%2d  fwd %7.2f us  bwd %7.2f us  (%d routers, one launch each)'
                  % (B, W, fwd, bwd, N_ROUTERS), flush=True)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device='cuda')
    old = ah.router_n_chan
    for B in BATCHES:
        for W in WIDTHS:
            ah.router_n_chan = W
            try:
                run = bench.Run('cifar10-ac', B, 'bf16', torch.device('cuda'), 0, 1)
            finally:
                ah.router_n_chan = old
            assert run.eng.router_width == W and run.plan.umma_heads
            run.warm(5)
            ms, _ = run.device_timed(STEPS, 5, flush)
            print('step    B=%5d W=%2d  %8.3f ms per training step (cifar10-ac bf16, mean of %d)'
                  % (B, W, ms / STEPS, STEPS), flush=True)
            del run
            torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
