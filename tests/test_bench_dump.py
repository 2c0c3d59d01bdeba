"""bench.py --dump-outputs on the host: which arrays it writes, their dtype, and the seeded example sample that keeps
a large batch under the size budget (engine and plan stand-ins with the buffers dump_outputs reads; every
per-example value encodes its example index, so a sample taken along the wrong axis shows)."""
import os
from types import SimpleNamespace as Ns

import numpy as np
import torch

import bench


def _run(B, n_nodes=5, n_leaves=2, n_theta=1000):
    ex = torch.arange(B, dtype=torch.float32)
    zbuf = ex[:, None] * 16 + torch.arange(16, dtype=torch.float32)       # a 16-wide buffer, 10 live columns
    nodes = torch.arange(n_nodes, dtype=torch.float32)[:, None] * 1e6
    eng = Ns(theta=torch.linspace(-1, 1, n_theta), accum=torch.full((n_theta,), 0.5), grad=torch.ones(n_theta + 8),
             state=torch.arange(40, dtype=torch.float32), n_state=30, dynamic=True,
             regs=[Ns(idx=i) for i in range(n_leaves)])
    plan = Ns(B=B, reg={i: Ns(Z=zbuf[:, :10], c_err=ex + 0.25, d_cor=ex + 0.5) for i in range(n_leaves)},
              p_tr=nodes + ex, p_ev=nodes - ex, c_data=ex * 2)
    return Ns(eng=eng, plan=plan)


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_writes_every_output_whole(tmp_path):
    run = _run(64)
    bench.dump_outputs(run, str(tmp_path))
    got = _load(tmp_path)
    assert set(got) == {'theta', 'momentum', 'grad', 'state', 'p_tr', 'p_ev', 'c_data'} | {
        'leaf%d_%s' % (i, k) for i in range(2) for k in ('logits', 'c_err', 'd_cor')}
    assert all(a.dtype == np.float32 for a in got.values())
    np.testing.assert_array_equal(got['theta'], run.eng.theta.numpy())
    np.testing.assert_array_equal(got['state'], np.arange(30, dtype=np.float32))      # the live state only
    np.testing.assert_array_equal(got['leaf1_logits'], run.plan.reg[1].Z.numpy())
    np.testing.assert_array_equal(got['p_ev'], run.plan.p_ev.numpy())


def test_dump_samples_a_large_batch_under_the_budget(tmp_path, monkeypatch):
    budget = 256 << 10
    monkeypatch.setattr(bench, 'DUMP_BYTES', budget)
    B = 4096                                          # 35 floats per example: 590 KB in all without the sample
    bench.dump_outputs(_run(B), str(tmp_path / 'a'))
    got = _load(tmp_path / 'a')
    assert sum(os.path.getsize(os.path.join(tmp_path, 'a', f)) for f in os.listdir(tmp_path / 'a')) <= budget
    idx = got.pop('examples')
    assert idx.dtype == np.float64 and 0 < len(idx) < B and np.all(np.diff(idx) > 0)
    n = len(idx)
    assert got['theta'].shape == (1000,) and got['grad'].shape == (1008,)            # whole, never sampled
    for i in range(2):
        np.testing.assert_array_equal(got['leaf%d_logits' % i], idx[:, None] * 16 + np.arange(10))
        np.testing.assert_array_equal(got['leaf%d_c_err' % i], idx + 0.25)
    np.testing.assert_array_equal(got['p_tr'], np.arange(5)[:, None] * 1e6 + idx)     # batch axis 1
    np.testing.assert_array_equal(got['p_ev'], np.arange(5)[:, None] * 1e6 - idx)
    np.testing.assert_array_equal(got['c_data'], idx * 2)
    assert got['p_tr'].shape == (5, n)
    bench.dump_outputs(_run(B), str(tmp_path / 'b'))                                  # the sample is fixed
    np.testing.assert_array_equal(np.load(tmp_path / 'b' / 'examples.npy'), idx)
