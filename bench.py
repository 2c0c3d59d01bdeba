#!/usr/bin/env python3
"""Benchmark of the hot path: one training step (forward 'tr' + backward + TALR / momentum) of the
reference's nets on synthetic data of the datasets' shapes.

  python bench.py --gpus N --steps K --warmup W [--config C] [--batch B] [--precision bf16|fp32]
  python bench.py --impl reference ...      # CPU arm: the oracle port of the reference on the host cores
  python bench.py ... --dump-outputs DIR    # also write what the last timed step computed, DIR/<name>.npy

Headline workload = `cifar10-ac` (ac_chain, /root/reference/scripts/arch_and_hypers.py:76-139, experiment
table scripts/train-nets:84-87) at --batch per GPU (default 4096; the reference trains at 128, reported in
the `configs` array next to it).  Other configs of BASELINE.json (SURVEY F4):
  cifar10-sr / mnist-sr = sr_chain(8) on 32x32x3 / 32x32x1, cifar10-cr = cr_chain(k_cpt) with the tau_cr
  schedule, hybrid-ac-dyn = ac_chain(dyn_k_cpt=True) with k_cpt ~ choice(k_cpts, B) per example
  (scripts/train-adaptive-nets:24-45).

One JSON line on rank 0 (driver contract).  `value` = images/s with the batch already resident in HBM
(device-timed, per-step CUDA events, L2 flushed between steps); `e2e` = images/s through
net.train.run(feed) with pinned HOST batches (H2D inside the timed region, loss vector read back);
`configs` = the same two numbers for every config at B = 128 and B = 4096 (fp32 mode included).
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'multipath-nn_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

K_CPT = 4e-9            # k_cpts[3] of arch_and_hypers.py:15


def lam(t):
    return 0.1 / 2 ** (t / 10000)


def tau_ds(t):
    return 1 / 2 ** (t / 20000)


def tau_cr(t):
    return 0.1 / 2 ** (t / 20000)


def _configs():
    import arch_and_hypers as ah
    return {
        'cifar10-ac': dict(make=lambda: ah.ac_chain(k_cpt=K_CPT), C=3, tau=tau_ds,
                           what='ac_chain(k_cpt=4e-9), 32x32x3, 10 classes'),
        'cifar10-cr': dict(make=lambda: ah.cr_chain(k_cpt=K_CPT), C=3, tau=tau_cr,
                           what='cr_chain(k_cpt=4e-9), tau_cr schedule, 32x32x3, 10 classes'),
        'cifar10-sr': dict(make=lambda: ah.sr_chain(8), C=3, tau=None, what='sr_chain(8), 32x32x3, 10 classes'),
        'mnist-sr': dict(make=lambda: ah.sr_chain(8), C=1, tau=None, what='sr_chain(8), 32x32x1 (MNIST-shaped), 10 classes'),
        'hybrid-ac-dyn': dict(make=lambda: ah.ac_chain(dyn_k_cpt=True), C=3, tau=tau_ds, dyn=True,
                              what='ac_chain(dyn_k_cpt=True), k_cpt ~ choice(k_cpts, B) per example, 32x32x3, 10 classes'),
    }


CONFIG_NAMES = ['cifar10-ac', 'cifar10-cr', 'cifar10-sr', 'mnist-sr', 'hybrid-ac-dyn']


def make_net(config='cifar10-ac', seed=0):
    from lib import layer_types
    cfg = _configs()[config]
    layer_types.seed(seed)
    return cfg['make']()((32, 32, cfg['C']), (10,))


def train_flop_per_img(net):
    """Algorithmic work of one dense training step per image from the reference's own n_ops formulas
    (layer_types.py:53,189-194): 1 MAC = 2 flop, training = forward + data gradient + weight gradient
    = 3 x forward MACs minus the stage-0 data gradient towards the input image, which nobody needs
    (SURVEY section 8(d): 123.02 MFLOP for ac_chain, 122.13 for sr_chain(8))."""
    fwd = 0
    for l in net.layers:
        fwd += l.n_ops + (l.router.n_ops if l.router is not None else 0)
    first = net.root.sinks[0].comps[0]                     # MultiscaleConvMax of stage 0
    c0 = net.hypers.x0_shape[2]
    n = len(first.hypers.n_chan)
    h0 = net.hypers.x0_shape[0]
    scales = [h0 // 2 ** i for i in range(4)][-n:]
    skip = sum(h * h * 9 * c0 * c for h, c in zip(scales, first.hypers.n_chan))
    return 2.0 * (3 * fwd - skip)


def synth(B, n, seed, C=3):
    rng = np.random.default_rng(seed)
    xs = [torch.from_numpy(rng.random((B, 32, 32, C), dtype=np.float32)) for _ in range(n)]
    ys = [torch.from_numpy(np.eye(10, dtype=np.float32)[rng.integers(0, 10, B)]) for _ in range(n)]
    return xs, ys


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


class Clocks:
    """nvidia-smi sampler (recipe's clocks line) running during the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu):
        self.rows, self.proc, self.gpu, self.mark = [], None, gpu, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '25'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        # samples of the timed regions; a very short run (few steps) may have none, then the samples taken
        # under the warm-up load stand in and the line says so
        rows = self.rows[self.mark:]
        window = 'timed region'
        if not rows:
            rows, window = list(self.rows), 'warm-up (timed region shorter than the sampling interval)'
        sm = [float(r[1]) for r in rows if len(r) > 2 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm), 'window': window}


# --------------------------------------------------------------------------- #
# CPU arm: the oracle port of the reference (TF <= 0.12 is not installable offline)
# --------------------------------------------------------------------------- #
def _oracle(config):
    import copy
    from lib import serdes
    from oracle.torch_ref import OracleNet
    return OracleNet(copy.deepcopy(serdes.encode_net(make_net(config))), torch.float32)


def _oracle_step(o, cfg, x, y, t, rng):
    import arch_and_hypers as ah
    kc = rng.choice(ah.k_cpts, len(x)).astype(np.float32) if cfg.get('dyn') else None
    o.train_step(x.numpy(), y.numpy(), lr=lam(t), tau=cfg['tau'](t) if cfg['tau'] else None, k_cpt=kc)


def cpu_oracle_rate(config, B, budget_s=15.0, max_steps=400):
    """Reference semantics restated on PyTorch-CPU (oracle/torch_ref.py): full train steps (forward 'tr',
    autograd backward, TALR + momentum) on a bounded sample of the workload."""
    cfg = _configs()[config]
    o = _oracle(config)
    xs, ys = synth(B, 2, 1, cfg['C'])
    rng = np.random.default_rng(0)
    _oracle_step(o, cfg, xs[0], ys[0], 0, rng)        # warm-up
    t0 = time.perf_counter()
    n = 0
    while n < max_steps and (n == 0 or time.perf_counter() - t0 < budget_s):
        _oracle_step(o, cfg, xs[n % 2], ys[n % 2], n, rng)
        n += 1
    dt = time.perf_counter() - t0
    return n * B / dt, n, dt


def run_reference(args, rank, world, emit):
    """--impl reference: the reference's CPU implementation of the path (its oracle port; the TF graph itself
    cannot be installed here) on the box's host cores, same config / batch / steps / warm-up as our arm.  Only if
    the whole run would exceed a few minutes the per-step sample is cut to a smaller batch (stated in `sample`)."""
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = _configs()[args.config]
    B, steps, warm = args.batch, args.steps, max(0, args.warmup)
    o = _oracle(args.config)
    rng = np.random.default_rng(0)
    probe_B = min(B, 256)
    xs, ys = synth(probe_B, 1, 2, cfg['C'])
    _oracle_step(o, cfg, xs[0], ys[0], 0, rng)                      # first call: thread pool, allocator
    t0 = time.perf_counter()
    _oracle_step(o, cfg, xs[0], ys[0], 0, rng)
    rate = probe_B / (time.perf_counter() - t0)                     # images/s estimate
    budget = float(os.environ.get('MPNN_REF_BUDGET_S', 240.0))
    sample_B = B
    if (steps + warm) * B / rate > budget:
        sample_B = max(128, int(budget * rate / (steps + warm)) // 128 * 128)
        sample_B = min(sample_B, B)
    o = _oracle(args.config)                                        # fresh parameters for the timed run
    xs, ys = synth(sample_B, 2, 1, cfg['C'])
    for w in range(warm):
        _oracle_step(o, cfg, xs[w % 2], ys[w % 2], w, rng)
    t0 = time.perf_counter()
    for t in range(steps):
        _oracle_step(o, cfg, xs[t % 2], ys[t % 2], warm + t, rng)
    dt = time.perf_counter() - t0
    v = steps * sample_B / dt
    sample = '%d train steps at batch %d%s (reference semantics restated on PyTorch-CPU; TF<=0.12 not installable offline)' % (
        steps, sample_B, '' if sample_B == B else ' -- a bounded sample of the batch-%d workload' % B)
    line = {
        'impl': 'reference', 'metric': 'train images/sec', 'value': v, 'unit': 'images/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': warm, 'ms_per_step': 1e3 * dt / steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': '%s: %s train step (fwd tr + bwd + TALR/momentum), dense as in the reference'
                               % (args.config, cfg['what']),
                   'batch_per_gpu': B, 'sample_batch': sample_B},
        'cpu_baseline': {'value': v, 'unit': 'images/s', 'cores': torch.get_num_threads(), 'kind': 'port', 'sample': sample},
        'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    emit(line)


# --------------------------------------------------------------------------- #
# our arm
# --------------------------------------------------------------------------- #
class Run:
    """one (config, batch, precision) on this rank's GPU"""

    def __init__(self, config, B, precision, dev, rank, world, graphs=True):
        import arch_and_hypers as ah
        self.cfg, self.config, self.B, self.dev, self.world = _configs()[config], config, B, dev, world
        self.net = make_net(config).configure(precision=precision, graphs=graphs, dist=world > 1)
        self.eng = self.net._get_engine()
        xs, ys = synth(B, 4, 100 + rank, self.cfg['C'])
        self.xs = [x.pin_memory() for x in xs]
        self.ys = [y.pin_memory() for y in ys]
        rng = np.random.default_rng(200 + rank)
        self.kcs = [rng.choice(ah.k_cpts, B).astype(np.float32) for _ in range(4)] if self.cfg.get('dyn') else None
        self.plan = self.eng._plan(B, True, True)
        self.flop = train_flop_per_img(self.net)
        # parameters, momentum and layer state as initialised (seeded): the last device-timed step starts from them
        self.init = [t.clone() for t in (self.eng.theta, self.eng.accum, self.eng.state)]

    def feed(self, t):
        net = self.net
        f = {net.x0: self.xs[t % 4], net.y: self.ys[t % 4], net.mode: 'tr', net.λ_lrn: lam(t)}
        if self.cfg['tau'] is not None:
            f[net.τ] = self.cfg['tau'](t)
        if self.kcs is not None:
            f[net.k_cpt] = self.kcs[t % 4]
        return f

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(self.dev)

    def warm(self, n):
        for t in range(n):
            self.net.train.run(self.feed(t))
        self.barrier()

    def _max_over_ranks(self, v):
        tt = torch.tensor([v], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        return float(tt.item())

    def device_timed(self, steps, warmup, flush):
        """K steps with the batch resident in HBM, one CUDA event pair per step, L2 flushed in between.  The last
        step starts again from the initial parameters: the step's fp32 weight-gradient sums are unordered, so two
        runs differ in the last bits, and consecutive steps on one batch amplify that to percents within 25 steps.
        Restarting the last step from the seeded state keeps what it computes (--dump-outputs) reproducible to those
        last bits; it runs the same kernels on the same shapes as the others.  The K end-to-end steps that follow
        (e2e_timed, whose mean objective is the line's `loss`) therefore continue from the initial parameters plus
        one step, not plus the warm-up and K steps."""
        eng, plan = self.eng, self.plan
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        eng._feed(plan, self.feed(warmup), True)
        self.barrier()
        l0 = eng.L.launches
        for t in range(steps):
            if t == steps - 1:
                for buf, init in zip((eng.theta, eng.accum, eng.state), self.init):
                    buf.copy_(init)
            flush.zero_()                                  # evict L2 between timed iterations
            ev[t][0].record()
            eng.run_resident(plan, True)
            ev[t][1].record()
        self.barrier()
        launches = (plan.graph_launches * steps) if eng.use_graphs else (eng.L.launches - l0)
        return self._max_over_ranks(sum(a.elapsed_time(b) for a, b in ev)), int(launches)

    def e2e_timed(self, steps, warmup):
        """the public API with pinned host batches: H2D copies inside, per-example objective read back"""
        host_loss = torch.empty(self.B, dtype=torch.float32).pin_memory()
        obj = self.plan.c_data if self.net.dynamic else self.plan.reg[self.eng.regs[-1].idx].c_err
        self.barrier()
        t0 = time.perf_counter()
        for t in range(steps):
            self.net.train.run(self.feed(warmup + t))
            host_loss.copy_(obj, non_blocking=True)
        torch.cuda.synchronize(self.dev)
        s = time.perf_counter() - t0
        return self._max_over_ranks(s), float(host_loss.mean())

    def hbm_bytes_per_step(self):
        p = self.plan
        return sum(getattr(op, 'nbytes', 0.0) for op in p.pack_ops + p.fwd_ops + p.bwd_ops + p.opt_ops)

    def summary(self, steps, warmup, flush, pk):
        self.warm(max(warmup, 3))
        ms, launches = self.device_timed(steps, warmup, flush)
        e2e_s, loss = self.e2e_timed(steps, warmup)
        value = self.world * self.B * steps / (ms * 1e-3)
        return {
            'config': self.config, 'workload': self.cfg['what'], 'batch_per_gpu': self.B,
            'dtype': 'bf16' if self.eng.dtype == 1 else ('f32 (%s on tcgen05)' % {2: 'bf16x3', 3: 'bf16x6'}[self.eng.split] if self.eng.split else 'f32'),
            'conv_impl': 'tcgen05' if self.eng.impl == 1 else 'simt', 'value': value, 'unit': 'images/s',
            'ms_per_step': ms / steps, 'e2e': self.world * self.B * steps / e2e_s, 'steps': steps,
            'launches_per_step': launches // max(steps, 1), 'train_mflop_per_img': self.flop / 1e6,
            'tensor_frac_of_step': value / self.world * self.flop / (pk['bf16_tflops_sustained'] * 1e12),
            'hbm_frac_of_step': (self.hbm_bytes_per_step() / (pk['hbm_gbs'] * 1e9)) / (ms / steps * 1e-3),
            'loss': loss}


DUMP_BYTES = 60 << 20          # leaves room for the .npy headers under 64 MB


def dump_outputs(run, out_dir):
    """What the last device-timed step (one training step from the initial parameters on the resident batch) left
    for a caller, one float32 DIR/<name>.npy each: the updated parameters (`theta`), momentum and layer state, the
    step's gradient buffer ([per-node TALR moments | gradients]), every leaf's logits / per-example error /
    correctness and, for routed nets, the routing weights `p_tr`, decisions `p_ev` (nodes x batch) and per-example
    objective `c_data`.  The inputs are seeded, so two builds run with the same arguments can be compared array for
    array.  A batch whose arrays would pass 64 MB in all is cut to a fixed, seeded sample of examples (their indices
    in `examples.npy`)."""
    eng, plan = run.eng, run.plan
    whole = {'theta': eng.theta, 'momentum': eng.accum, 'grad': eng.grad, 'state': eng.state[:eng.n_state]}
    per_ex = {}                                   # name -> (tensor, batch axis)
    for k, nd in enumerate(eng.regs):
        r = plan.reg[nd.idx]
        per_ex.update({'leaf%d_logits' % k: (r.Z, 0), 'leaf%d_c_err' % k: (r.c_err, 0), 'leaf%d_d_cor' % k: (r.d_cor, 0)})
    if eng.dynamic:
        per_ex.update(p_tr=(plan.p_tr, 1), p_ev=(plan.p_ev, 1), c_data=(plan.c_data, 0))
    out = {k: t.detach().float().cpu().numpy() for k, t in whole.items()}
    per_ex = {k: (t.detach().float().cpu().numpy(), ax) for k, (t, ax) in per_ex.items()}
    B = plan.B
    fixed = sum(a.nbytes for a in out.values())
    per_example = sum(a.nbytes for a, _ in per_ex.values()) / B
    keep = int((DUMP_BYTES - fixed - 8 * B) // per_example) if per_example else B
    if keep < B:
        idx = np.sort(np.random.default_rng(0).choice(B, max(keep, 1), replace=False))
        per_ex = {k: (np.take(a, idx, axis=ax), ax) for k, (a, ax) in per_ex.items()}
        out['examples'] = idx.astype(np.float64)
    out.update({k: a for k, (a, _) in per_ex.items()})
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def per_launch_profile(run):
    """eager replay of the step's launch list on ONE stream, a CUDA event pair around every launch (3 passes, the
    last one kept).  Returns [(op, ms)] with op.kind / op.desc / op.flops / op.nbytes (lib/engine.py::_tag)."""
    eng, plan, L = run.eng, run.plan, run.eng.L
    # (collectives are left out: this replay runs on rank 0 alone)
    ops = [op for op in plan.pack_ops + plan.fwd_ops + plan.bwd_ops + plan.opt_ops if getattr(op, 'kind', '') != 'allreduce']
    called, saved = [], {}
    for name in L.protos:                                   # untagged launches are labelled by their C-ABI entry
        short = name[5:]
        try:
            fn = getattr(L, short)
        except AttributeError:
            continue
        saved[short] = fn
        L.__dict__[short] = (lambda fn, short: (lambda *a: (called.append(short), fn(*a))[1]))(fn, short)
    out = []
    for rep in range(3):
        evs = []
        eng.grad.zero_()
        eng.stream = __import__('ctypes').c_void_p(torch.cuda.current_stream(run.dev).cuda_stream)
        for op in ops:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            del called[:]
            a.record(); op(); b.record()
            if not hasattr(op, 'kind'):
                op.kind = called[0] if called else 'misc'
            evs.append((op, a, b))
        torch.cuda.synchronize(run.dev)
        if rep == 2:
            out = [(op, a.elapsed_time(b)) for op, a, b in evs]
    L.__dict__.update(saved)
    return out


def roofline_of(prof, pk, pk_src, B):
    """`roofline` = the single dominant LAUNCH of the step against the ceiling that binds it (the larger of its
    HBM time at the measured copy bandwidth and its tensor time at the measured cuBLAS bf16 rate); `families`
    = per kernel family: launches, time, share of the serialised step, achieved rate and fraction."""
    tot = sum(ms for _, ms in prof)

    def rates(flops, nbytes, ms):
        tf, gb = flops / (ms * 1e-3) / 1e12, nbytes / (ms * 1e-3) / 1e9
        t_hbm, t_tc = nbytes / (pk['hbm_gbs'] * 1e9), flops / (pk['bf16_tflops'] * 1e12)
        if t_tc > t_hbm:
            return dict(bound='tensor', achieved=tf, peak=pk['bf16_tflops'], unit='TFLOP/s', frac=tf / pk['bf16_tflops'],
                        other_ceiling=dict(bound='hbm', achieved=gb, frac=gb / pk['hbm_gbs']))
        return dict(bound='hbm', achieved=gb, peak=pk['hbm_gbs'], unit='GB/s', frac=gb / pk['hbm_gbs'],
                    other_ceiling=dict(bound='tensor', achieved=tf, frac=tf / pk['bf16_tflops']))
    tagged = [(op, ms) for op, ms in prof if getattr(op, 'nbytes', 0.0) > 0]
    op, ms = max(tagged, key=lambda t: t[1])
    roof = rates(op.flops, op.nbytes, ms)
    name = ('%s %s' % (op.kind, getattr(op, 'desc', ''))).strip()
    roof.update(kernel=name, launch_ms=ms, share_of_step=ms / tot, algorithmic_bytes=op.nbytes,
                algorithmic_flops=op.flops, traffic=None,
                peak_source=pk_src + ' (burst; the launch is timed alone with CUDA events on its stream)')
    try:                                                    # measured DRAM bytes of exactly this launch at exactly this batch
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json'))).get('B%d' % B, {}).get(name)
        if tr:
            roof['traffic'] = tr['dram_bytes']
            roof['traffic_source'] = tr['source']
    except Exception:
        pass
    fam = {}
    for o, t in prof:
        d = fam.setdefault(getattr(o, 'kind', 'misc'), dict(n=0, ms=0.0, flops=0.0, bytes=0.0))
        d['n'] += 1; d['ms'] += t; d['flops'] += getattr(o, 'flops', 0.0); d['bytes'] += getattr(o, 'nbytes', 0.0)
    families = {}
    for k, d in sorted(fam.items(), key=lambda kv: -kv[1]['ms']):
        row = dict(launches=d['n'], ms=round(d['ms'], 4), share=round(d['ms'] / tot, 4))
        if d['bytes'] > 0:
            r = rates(d['flops'], d['bytes'], d['ms'])
            row.update(bound=r['bound'], achieved=round(r['achieved'], 1), unit=r['unit'], frac=round(r['frac'], 4))
        families[k] = row
    return roof, families, tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--config', default='cifar10-ac', choices=CONFIG_NAMES)
    ap.add_argument('--batch', type=int, default=int(os.environ.get('MPNN_BENCH_BATCH', 4096)),
                    help='examples per GPU per step (reference trains at 128; see DESIGN.md)')
    ap.add_argument('--precision', default=os.environ.get('MPNN_PRECISION', 'bf16'))
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--no-graphs', action='store_true')
    ap.add_argument('--no-sweep', action='store_true', help='skip the `configs` array (other configs / batches)')
    ap.add_argument('--profile', action='store_true', help='print per-kernel-kind time shares')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    # stdout carries exactly ONE JSON line: anything a library prints to fd 1 meanwhile (NCCL's version banner on
    # the first communicator) is sent to stderr, and the real stdout comes back for the final print
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        return run_reference(args, rank, world, emit)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    if os.environ.get('NCCL_DEBUG', '').upper() in ('VERSION', 'WARN'):
        del os.environ['NCCL_DEBUG']               # NCCL's version banner goes to stdout, which carries the ONE JSON line
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=180))
    pk, pk_src = peaks()
    B = args.batch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    run = Run(args.config, B, args.precision, dev, rank, world, graphs=not args.no_graphs)

    # ---------------- warm-up (also captures the CUDA graphs) --------------- #
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()                                 # nvidia-smi needs ~0.2 s before its first sample
    run.warm(args.warmup)
    if rank == 0:
        # wait for the sampler WITHOUT issuing work: a training step contains the all-reduce, so every
        # rank must run exactly the same number of them
        t_wait = time.perf_counter()
        while not clocks.rows and time.perf_counter() - t_wait < 3.0:
            time.sleep(0.01)
        clocks.mark = len(clocks.rows)                 # samples from here on fall inside the timed regions
    run.barrier()
    dev_ms, launches = run.device_timed(args.steps, args.warmup, flush)
    if args.dump_outputs and rank == 0:
        dump_outputs(run, args.dump_outputs)
    e2e_s, loss = run.e2e_timed(args.steps, args.warmup)
    clk = clocks.stop() if rank == 0 else None

    # ---------------- other configs / batches (every rank runs the same sequence) ---------------- #
    sweep = []
    if not args.no_sweep:
        todo = [(args.config, 128, args.precision)] if B != 128 else []
        if world == 1:
            for c in CONFIG_NAMES:
                for b in (128, 4096):
                    if (c, b) != (args.config, B) and (c, b, args.precision) not in todo:
                        todo.append((c, b, args.precision))
            todo += [(args.config, b, p) for p in ('bf16x3', 'bf16x6', 'fp32') for b in (128, 4096)]
        for c, b, prec in todo:
            r = Run(c, b, prec, dev, rank, world)
            sweep.append(r.summary(30 if b > 128 else 100, 3, flush, pk))
            del r
            gc.collect()                              # plans are reference cycles: free the run's buffers now
            torch.cuda.empty_cache()

    # ---------------- per-launch profile (rank 0) ---------------- #
    prof = per_launch_profile(run) if rank == 0 else []
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    roof, families, tot_ms = roofline_of(prof, pk, pk_src, B)
    if args.profile:
        for k, v in families.items():
            print('# %-22s n=%3d %8.3f ms  %5.1f%%  %s' % (k, v['launches'], v['ms'], 100 * v['share'],
                                                          ('%.1f %s (%.0f%% of %s peak)' % (v['achieved'], v['unit'], 100 * v['frac'], v['bound']))
                                                          if 'unit' in v else ''), file=sys.stderr)
        for op, ms in prof:
            if getattr(op, 'desc', ''):
                print('#   %-11s %-24s %7.3f ms %7.1f TFLOP/s %7.0f GB/s' % (
                    op.kind, op.desc, ms, op.flops / ms / 1e9, op.nbytes / ms / 1e6), file=sys.stderr)

    cfg = run.cfg
    torch.set_num_threads(os.cpu_count() or 1)
    cpu_B = min(B, 256)
    cpu = None
    if world == 1 and not os.environ.get('MPNN_BENCH_NO_CPU'):
        cpu_v, cpu_n, cpu_dt = cpu_oracle_rate(args.config, cpu_B, budget_s=15.0)
        cpu = {'value': cpu_v, 'unit': 'images/s', 'cores': torch.get_num_threads(), 'kind': 'port',
               'sample': '%d train steps at batch %d in %.1f s (reference semantics restated on PyTorch-CPU; '
                         'TF<=0.12 not installable offline)' % (cpu_n, cpu_B, cpu_dt)}
    value = world * B * args.steps / (dev_ms * 1e-3)
    e2e = world * B * args.steps / e2e_s
    eng = run.eng
    h2d = B * (32 * 32 * cfg['C'] + 10) * 4 + 8 * 4 + (B * 4 if cfg.get('dyn') else 0)
    line = {
        'metric': 'train images/sec', 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dev_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'bf16' if args.precision == 'bf16' else 'f32', 'data': 'synthetic',
        'config': {'workload': '%s: %s train step (fwd tr + bwd + TALR/momentum), dense as in the reference'
                               % (args.config, cfg['what']),
                   'batch_per_gpu': B, 'global_batch': B * world, 'parallelism': 'dp%d' % world,
                   'l2': 'flushed between timed steps (256 MiB memset outside the event pairs)',
                   'cuda_graph': bool(eng.use_graphs), 'conv_impl': 'tcgen05' if eng.impl == 1 else 'simt',
                   'wgrad_impl': 'tcgen05' if eng.impl_w == 1 else 'simt',
                   'dp_tail': None if world == 1 else ('one kernel over NVLink peer memory (MPNN_DIST_FUSED=1)' if eng.fused_dp
                                                       else 'ncclAllReduce in two buckets (deep stages under the backward pass) + optimiser')},
        'e2e': {'value': e2e, 'unit': 'images/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': B * 4,
                'timing': 'wall clock around net.train.run(feed) with pinned host batches', 'loss': loss},
        'gpu_launches': int(launches), 'train_mflop_per_img': run.flop / 1e6,
        'tensor_frac_of_step': value / world * run.flop / (pk['bf16_tflops_sustained'] * 1e12),
        # whole step against the HBM ceiling: algorithmic bytes of every launch (op tags) / measured copy bandwidth
        'hbm_frac_of_step': (run.hbm_bytes_per_step() / (pk['hbm_gbs'] * 1e9)) / (dev_ms / args.steps * 1e-3),
        'roofline': roof, 'families': families, 'serialised_kernel_ms': tot_ms,
        'configs': sweep, 'cpu_baseline': cpu, 'clocks': clk}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
