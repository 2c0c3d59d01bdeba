"""Datasets in the reference's `.npz` schema (x0_tr, x0_ts, y_tr, y_ts, m_sym;
/root/reference/scripts/lib/data.py:54-85, scripts/prep-data) plus a synthetic
generator of the same schema (datasets cannot be downloaded offline).

CPU data preparation is outside the GPU hot path (SURVEY section 2.1); the
augmentation here is a vectorised NumPy restatement of data.py:10-34 (random
flip for symmetric classes, +-r_shift pixel shift with per-image-mean fill,
sampling with replacement, float64 output).
"""
import numpy as np

__all__ = ['Dataset', 'synthetic_archive']


def synthetic_archive(n_tr=512, n_ts=256, shape=(32, 32, 3), n_cls=10, seed=0):
    """Random data with prep-data's output schema: images uniform in [0,1)
    (CIFAR is gamma-decoded into [0,1], prep-data:94-96), one-hot labels."""
    rng = np.random.default_rng(seed)

    def labels(n):
        y = np.zeros((n, n_cls))
        y[np.arange(n), rng.integers(0, n_cls, n)] = 1
        return y
    return dict(x0_tr=rng.random((n_tr, *shape)), x0_ts=rng.random((n_ts, *shape)),
                y_tr=labels(n_tr), y_ts=labels(n_ts), m_sym=np.ones(n_cls, bool))


class Dataset:
    def __init__(self, path=None, archive=None, seed=None):
        if archive is None:
            archive = np.load(path, allow_pickle=True)['arr_0'][()]
        self.x0_tr = archive['x0_tr']
        self.x0_ts = archive['x0_ts']
        self.y_tr = archive['y_tr']
        self.y_ts = archive['y_ts']
        # prep-data writes m_sym as float64 ones/zeros (mnist, cifar-*) or a Python int list (hybrid):
        # normalise once to a boolean mask (a float & bool raises, an int array would index, not mask)
        self.m_sym = np.asarray(archive['m_sym']).astype(bool)
        self.x0_vl = self.x0_tr[:0]
        self.y_vl = self.y_tr[:0]
        self.rng = np.random.default_rng(seed)

    @property
    def x0_shape(self):
        return self.x0_tr.shape[1:]

    @property
    def y_shape(self):
        return self.y_tr.shape[1:]

    def augmented_training_batch(self, n=128, r_shift=4):
        rng = self.rng
        j = rng.integers(0, len(self.x0_tr), n)
        x = np.asarray(self.x0_tr[j], dtype=np.float64)
        y = np.asarray(self.y_tr[j], dtype=np.float64)
        flip = self.m_sym[np.argmax(y, 1)] & (rng.random(n) >= 0.5)
        x[flip] = x[flip][:, :, ::-1]
        h, w = x.shape[1:3]
        out = np.empty_like(x)
        out[:] = x.mean((1, 2), keepdims=True)
        du = rng.integers(-r_shift, r_shift + 1, n)
        dv = rng.integers(-r_shift, r_shift + 1, n)
        for i in range(n):
            a, b = du[i], dv[i]
            out[i, max(-a, 0):min(h - a, h), max(-b, 0):min(w - b, w)] = \
                x[i, max(a, 0):min(h + a, h), max(b, 0):min(w + b, w)]
        return out, y

    def to_device(self, device='cuda'):
        """keep the training set resident in HBM for `augmented_training_batch_gpu`"""
        import torch
        self._dev = (torch.from_numpy(np.ascontiguousarray(self.x0_tr, dtype=np.float32)).to(device),
                     torch.from_numpy(np.ascontiguousarray(self.y_tr, dtype=np.float32)).to(device))
        return self

    def test_to_device(self, device='cuda'):
        """keep the test set resident in HBM for `test_set(device=True)`, so a statistics pass over it does not upload
        the data set again"""
        import torch
        self._dev_ts = (torch.from_numpy(np.ascontiguousarray(self.x0_ts, dtype=np.float32)).to(device),
                        torch.from_numpy(np.ascontiguousarray(self.y_ts, dtype=np.float32)).to(device))
        return self

    def augmented_training_batch_gpu(self, n=128, r_shift=4, shard=None):
        """`augmented_training_batch` with the per-example work on the GPU (csrc/augment.cu).  The
        random numbers are drawn on the host in the same order, so a seeded sampler produces the same
        batches either way; returns device tensors (x0 fp32 NHWC, y one-hot) that `net.train.run`
        accepts as feed values.  shard=(rank, world): this rank's part of the global batch."""
        import ctypes
        import torch
        from lib import _cabi
        if getattr(self, '_dev', None) is None:
            self.to_device()
        xd, yd = self._dev
        rng = self.rng
        j = rng.integers(0, len(self.x0_tr), n)
        flip = self.m_sym[np.argmax(self.y_tr[j], 1)] & (rng.random(n) >= 0.5)
        du = rng.integers(-r_shift, r_shift + 1, n)
        dv = rng.integers(-r_shift, r_shift + 1, n)
        if shard is not None:
            # data parallel: every rank draws the SAME global batch (same seed) and keeps its contiguous shard,
            # so the union over the ranks is the batch a single process would have drawn
            rank, world = shard
            if n % world:
                raise ValueError('batch %d does not divide over %d ranks' % (n, world))
            sl = slice(rank * (n // world), (rank + 1) * (n // world))
            j, flip, du, dv = j[sl], flip[sl], du[sl], dv[sl]
            n = n // world
        draws = torch.from_numpy(np.stack([j, flip, du, dv]).astype(np.int32)).to(xd.device)
        h, w, c = self.x0_tr.shape[1:]
        n_cls = self.y_tr.shape[1]
        x0 = torch.empty((n, h, w, c), dtype=torch.float32, device=xd.device)
        y = torch.empty((n, n_cls), dtype=torch.float32, device=xd.device)
        vp = lambda t: ctypes.c_void_p(t.data_ptr())
        _cabi.lib().augment_batch(vp(xd), vp(yd), len(self.x0_tr), h, w, c, n_cls, vp(draws[0]), vp(draws[1]),
                                  vp(draws[2]), vp(draws[3]), n, vp(x0), vp(y),
                                  ctypes.c_void_p(torch.cuda.current_stream(xd.device).cuda_stream))
        self._keep = draws          # the launch is asynchronous: keep its operands alive until the next batch
        return x0, y

    def _batch(self, x0, y, n):
        i = self.rng.integers(0, len(x0), n)
        return np.take(x0, i, axis=0), np.take(y, i, axis=0)

    def training_batch(self, n=128):
        return self._batch(self.x0_tr, self.y_tr, n)

    def test_batch(self, n=128):
        return self._batch(self.x0_ts, self.y_ts, n)

    @staticmethod
    def _full_set(x0, y, n):
        for i in range(0, len(x0), n):
            yield x0[i:i + n], y[i:i + n]

    def training_set(self, n=128, device=False):
        """the training set in slices of n; device=True: slices (views) of the fp32 copy resident in HBM"""
        if device:
            if getattr(self, '_dev', None) is None:
                self.to_device()
            yield from self._full_set(*self._dev, n)
        else:
            yield from self._full_set(self.x0_tr, self.y_tr, n)

    def test_set(self, n=128, device=False):
        """the test set in slices of n; device=True: slices (views) of the fp32 copy resident in HBM"""
        if device:
            if getattr(self, '_dev_ts', None) is None:
                self.test_to_device()
            yield from self._full_set(*self._dev_ts, n)
        else:
            yield from self._full_set(self.x0_ts, self.y_ts, n)
