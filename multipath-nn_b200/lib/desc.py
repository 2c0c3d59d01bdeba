"""Network statistics (`net_desc`) and their log rendering.

Schema and text layout are those of /root/reference/scripts/lib/desc.py:10-79
(SURVEY App. C), because the plotting scripts and the `NNNN-stats.npy` /
`NNNN-log.txt` files of `train-nets` consume them:

    net_desc   = {'type', 'stats_tr', 'stats_ts', 'root': layer_desc}
    layer_desc = {'name', 'stats_tr', 'stats_ts', 'sinks': [layer_desc]}

with every statistic the mean over a whole dataset split of a per-example
quantity.  Here the per-example quantities come from `net.eval_stats` (one GPU
forward in 'ev' mode per batch) instead of a TF session; the reduction -- sum over
examples in float64 on the host, divided by the example count -- is unchanged.
"""
import numpy as np

__all__ = ['state_tensors', 'mean_net_state', 'mean_net_state_compact', 'mean_net_state_device', 'net_desc',
           'render_net_desc']

_SPLITS = ('stats_tr', 'stats_ts')
_RULE = '─' * 59


# --------------------------------------------------------------------------- #
# which statistics exist (scripts/train-nets:111-130)
# --------------------------------------------------------------------------- #
def state_tensors(net):
    """{key: key} for every statistic `net.eval_stats` returns; key = (owner, name) where the owner is
    the net (accuracy, mean op count), a leaf (outcome probabilities, losses) or a switch (|logit|)"""
    per_leaf = ['p_cor', 'p_inc', 'p_cor_by_cls', 'p_inc_by_cls'] + (['p_tr'] if net.dynamic else []) + ['c_err']
    keys = [(net, 'acc'), (net, 'moc')]
    keys += [(leaf, name) for leaf in net.leaves for name in per_leaf]
    keys += [(layer, 'x_rte') for layer in net.layers if layer.router is not None]
    return dict(zip(keys, keys))


# --------------------------------------------------------------------------- #
# dataset means
# --------------------------------------------------------------------------- #
class _RunningMean:
    """float64 sums over the example axis of a stream of batches"""

    def __init__(self, keys):
        self.total = dict.fromkeys(keys, 0)
        self.n = 0

    def add(self, batch_stats, n_examples):
        for key in self.total:
            self.total[key] = self.total[key] + np.asarray(batch_stats[key], dtype=np.float64).sum(0)
        self.n += n_examples

    def result(self):
        return {key: (value / self.n).tolist() for key, value in self.total.items()}


def mean_net_state(net, tensors, data, hypers):
    """mean of every requested statistic over the batches `data` yields, as python floats / lists"""
    if not tensors:
        return {}
    mean = _RunningMean(tensors.keys())
    for x0, y in data:
        feed = {net.x0: x0, net.y: y}
        feed.update(hypers)
        mean.add(net.eval_stats(feed), len(x0))
    return mean.result()


def _owned_by(owner, stats):
    """the statistics of one owner, keyed by name (identity comparison, like the reference's `t == l`)"""
    return {name: value for (who, name), value in stats.items() if who is owner}


def layer_desc(layer, stats_tr, stats_ts):
    node = {'name': layer.name}
    for split, stats in zip(_SPLITS, (stats_tr, stats_ts)):
        node[split] = _owned_by(layer, stats)
    node['sinks'] = [layer_desc(child, stats_tr, stats_ts) for child in layer.sinks]
    return node


def mean_net_state_compact(net, data, hypers, batch=4096):
    """`mean_net_state` for the p_ev-weighted statistics through the compacted evaluator (lib/compact_eval.py):
    every example only runs the nodes on its own path, the sums stay on the device and are read once.  In 'ev'
    mode examples are independent (BatchNorm uses its running moments), so the batch size of the pass is free:
    the 128-example slices the data set yields are regrouped into batches of `batch`."""
    ev = net.compact_evaluator(batch)
    ev.reset()
    k_cpt = hypers.get(getattr(net, 'k_cpt', None)) if net.hypers.__dict__.get('dyn_k_cpt') else None
    xs, ys, n = [], [], 0

    def flush():
        nonlocal xs, ys, n
        if n:
            ev.run_batch(np.concatenate(xs), np.concatenate(ys), k_cpt=k_cpt)
        xs, ys, n = [], [], 0
    for x0, y in data:
        if n + len(x0) > batch:
            flush()
        xs.append(np.asarray(x0, dtype=np.float32)); ys.append(np.asarray(y, dtype=np.float32)); n += len(x0)
    flush()
    return ev.result()


def mean_net_state_device(net, data, hypers, batch=4096):
    """`mean_net_state` for every key of `state_tensors(net)` through the device evaluator (lib/dense_stats.py): one
    graph-replayed dense forward and accumulate launch per chunk, one device-to-host read per data set.  The slices
    `data` yields (numpy or torch, host or device) are regrouped into chunks of `batch`.  Count-valued statistics have
    the host path's bits; c_err, p_tr and x_rte differ from it in the last bits (another summation order)."""
    import torch
    ev = net.stats_evaluator(batch)
    ev.reset()
    xs, ys, n = [], [], 0

    def cat(parts):
        if len(parts) == 1:
            return parts[0]
        if all(isinstance(p, torch.Tensor) for p in parts):
            return torch.cat(parts)
        return np.concatenate([p.cpu().numpy() if isinstance(p, torch.Tensor) else np.asarray(p, np.float32)
                               for p in parts])

    def flush():
        nonlocal xs, ys, n
        if n:
            ev.run_batch(cat(xs), cat(ys), hypers)
        xs, ys, n = [], [], 0
    for x0, y in data:
        if n + len(x0) > batch:
            flush()
        xs.append(x0); ys.append(y); n += len(x0)
    flush()
    return ev.result()


def net_desc(net, dataset, hypers={}, state={}, compact=False, device=False, batch=4096):
    """compact=True (dynamically-routed nets): statistics from the compacted evaluator -- exact for acc, moc,
    p_cor, p_inc and the per-class entries; c_err / p_tr / x_rte, which the reference defines on examples
    that never reach the node, are omitted (no plotting script reads them).
    device=True: the statistics of `state` from the device evaluator, over both splits kept resident in HBM
    (`Dataset.training_set(device=True)` / `test_set(device=True)`), in chunks of `batch` examples."""
    if compact and device:
        raise ValueError('net_desc: compact and device statistics are two different passes; choose one')
    if device:
        per_split = [{k: v for k, v in mean_net_state_device(net, batches, hypers, batch).items() if k in state}
                     for batches in (dataset.training_set(batch, device=True), dataset.test_set(batch, device=True))]
    elif compact and net.dynamic:
        per_split = [mean_net_state_compact(net, batches, hypers)
                     for batches in (dataset.training_set(), dataset.test_set())]
    else:
        per_split = [mean_net_state(net, state, batches, hypers)
                     for batches in (dataset.training_set(), dataset.test_set())]
    out = {'type': type(net).__name__}
    for split, stats in zip(_SPLITS, per_split):
        out[split] = _owned_by(net, stats)
    out['root'] = layer_desc(net.root, *per_split)
    return out


# --------------------------------------------------------------------------- #
# rendering (the NNNN-log.txt format)
# --------------------------------------------------------------------------- #
def _scalars(stats):
    """'(a=1; b=2)' over the scalar statistics in key order; vectors (per-class entries) are skipped"""
    shown = ['%s=%.3g' % (name, stats[name]) for name in sorted(stats) if np.ndim(stats[name]) == 0]
    return '(%s)' % '; '.join(shown) if stats else ''


def _tree(node, split):
    """one line per layer; sinks hang below their parent on '↳', siblings are joined by '| ' rails"""
    text = '%s %s' % (node['name'], _scalars(node[split]))
    last = len(node['sinks']) - 1
    for i, child in enumerate(node['sinks']):
        rail = '\n  ' if i == last else '\n| '
        text += '\n↳ ' + _tree(child, split).replace('\n', rail)
    return text


def render_net_desc(desc, name='Network'):
    rows = ['┌' + _RULE, '│ ' + name, '├' + _RULE]
    for title, split in (('Training Set:', 'stats_tr'), ('Test Set:', 'stats_ts')):
        rows += ['│ ' + title, '│',
                 '│   [%s] %s' % (desc['type'], _scalars(desc[split])),
                 '│     ' + _tree(desc['root'], split).replace('\n', '\n│     '),
                 '│']
    return '\n'.join(rows)
