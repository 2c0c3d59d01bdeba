"""Net types of the B200 build -- SRNet / ActorNet / CriticNet with the
reference's constructor, hypers, feed keys and tree iterators
(/root/reference/scripts/lib/net_types.py:43-284).  `link` only wires shapes
and parameters; routing, costs, gradients and the TALR + momentum update run
in `lib.engine` (libmpnn_sm100, CUDA sm_100a).

TF-session idioms map as follows:
    net.train.run({net.x0: x0, net.y: y, net.mode: 'tr', net.λ_lrn: ..})
        -> one fused forward / backward / update step on the GPU
    session.run(state_tensors, {net.x0: x0, net.y: y, **hypers})
        -> net.eval_stats({...}) (see lib.desc.mean_net_state)
"""
from types import SimpleNamespace as Ns

from lib.layer_types import Layer, NoOp, Sym

__all__ = ['n_leaves', 'params_list_rec', 'Placeholder', 'Net', 'SRNet', 'ActorNet', 'CriticNet']

# ---- support functions (net_types.py:14-22) --------------------------------


def n_leaves(ℓ):
    return 1 if len(ℓ.sinks) == 0 else sum(map(n_leaves, ℓ.sinks))


def params_list_rec(ℓ):
    if ℓ is not None:
        yield from vars(ℓ.params).values()
        for c in getattr(ℓ, 'comps', []):
            yield from params_list_rec(c)


class Placeholder:
    """Hashable feed key (stands in for tf.placeholder[_with_default])."""

    def __init__(self, name, default=None):
        self.name = name
        self.default = default

    def __repr__(self):
        return '<feed %s>' % self.name


class _TrainOp:
    def __init__(self, net):
        self.net = net

    def run(self, feed_dict=None):
        return self.net._get_engine().train_step(feed_dict or {})

# ---- root network class (net_types.py:43-79) -------------------------------


class Net:
    default_hypers = Ns(x0_shape=(), y_shape=())
    dynamic = False

    def __init__(self, **options):
        self.root = options.pop('root', None) or NoOp()
        self.hypers = Ns(**{**vars(type(self).default_hypers), **options})
        self.hypers.x0_shape = tuple(self.hypers.x0_shape)
        self.hypers.y_shape = tuple(self.hypers.y_shape)
        self.params = Ns()
        self.x0 = Placeholder('x0')
        self.y = Placeholder('y')
        self.mode = Placeholder('mode', 'ev')
        self.train = _TrainOp(self)
        self._engine = None
        self._engine_opts = {}
        self.link()

    def link(self):
        x0 = Sym(self.hypers.x0_shape, self, 'x0')
        y = Sym(self.hypers.y_shape, self, 'y')

        def link_layer(ℓ, x):
            ℓ.link(x, y, self.mode)
            if ℓ.router is not None:
                ℓ.router.link(self._router_input(ℓ.x), y, self.mode)
            for s in ℓ.sinks:
                link_layer(s, ℓ.x)
        link_layer(self.root, x0)

    def _router_input(self, x):
        return x

    @property
    def layers(self):
        def all_in_tree(layer):
            yield layer
            for sink in layer.sinks:
                yield from all_in_tree(sink)
        yield from all_in_tree(self.root)

    @property
    def leaves(self):
        return (ℓ for ℓ in self.layers if len(ℓ.sinks) == 0)

    @property
    def switches(self):
        return (ℓ for ℓ in self.layers if len(ℓ.sinks) > 1)

    # ---- execution -------------------------------------------------------- #
    def configure(self, **opts):
        """Engine options: precision='fp32'|'bf16'|'bf16x3'|'bf16x6', device, graphs=bool,
        dist=bool.  Must be called before the first run."""
        if self._engine is not None:
            raise RuntimeError('configure() after the engine was built')
        self._engine_opts.update(opts)
        return self

    def _get_engine(self):
        if self._engine is None:
            from lib.engine import Engine
            self._engine = Engine(self, **self._engine_opts)
            pending = getattr(self, '_pending_momentum', None)
            if pending is not None:                  # restored checkpoint (lib/checkpoint.py)
                self._engine.load_momentum(pending)
                self._pending_momentum = None
        return self._engine

    def compact_evaluator(self, batch=4096):
        """compacted 'ev'-mode evaluator of this net (lib/compact_eval.py), cached per batch capacity"""
        cache = self.__dict__.setdefault('_compact_eval', {})
        if batch not in cache:
            from lib.compact_eval import CompactEvaluator
            cache[batch] = CompactEvaluator(self._get_engine(), batch)
        return cache[batch]

    def stats_evaluator(self, batch=4096):
        """dense 'ev'-mode statistics on the device (lib/dense_stats.py), cached per batch capacity: `reset()`,
        `run_batch(x0, y, hypers)` for n <= batch examples, `result()` = `mean_net_state` for every key of
        `state_tensors(net)`.  Each chunk replays one CUDA graph (weight packing, the dense forward with the current
        BatchNorm moments, one accumulate launch); nets with Dropout(λ < 1) raise NotImplementedError."""
        cache = self.__dict__.setdefault('_stats_eval', {})
        if batch not in cache:
            from lib.dense_stats import DenseStatsEvaluator
            cache[batch] = DenseStatsEvaluator(self._get_engine(), batch)
        return cache[batch]

    def predict(self, x0, k_cpt=None, batch=4096):
        """Routed inference: run every example of x0 (numpy or torch, host or device, any n) only along its own
        path in 'ev' mode, in chunks of `batch` on the cached `compact_evaluator(batch)`.  No labels.  Returns
        Ns of numpy arrays:
            cls  int32 (n,)            predicted class (first argmax of prob)
            prob float32 (n, n_prob)   softmax of the classifier the example exits at
            exit int32 (n,)            that classifier's index in list(net.leaves)
            ops  float64 (n,)          ops of the nodes and routers on the example's path (the dense `moc`)
        n_prob = max(n_cls, widest classifier), which is n_cls unless a SuperclassCrossEntropyError classifier has
        more superclasses than the net has classes.  For an example that exits at a superclass classifier, prob is
        the softmax over that classifier's superclasses (zero-filled to n_prob columns) and cls is the superclass.
        k_cpt: required for nets with a per-example k_cpt (dyn_k_cpt) -- a scalar, one value or n values --
        and None for the others.  The weights are packed and the BatchNorm moments finalised on every call, so a
        call between training steps sees the current parameters."""
        return self.compact_evaluator(batch).predict(x0, k_cpt)

    def predictor(self, batch=4096):
        """Routed inference replayed as one CUDA graph (lib/compact_eval.py, RoutedPredictor), cached per capacity.
        `p = net.predictor(batch)`; `p(x0, k_cpt=None)` takes n <= batch examples (host or device) and returns the
        Ns(cls, prob, exit, ops) of `predict` (the same widths and superclass meaning) as DEVICE torch tensors -- views [:n] of the predictor's output buffers,
        overwritten by the next call.  With device inputs a call does not synchronise the host.  The checks, the
        refused compositions and the use of the current parameters are those of `predict`; n > batch raises
        ValueError.  The graph is captured on the first call with n > 0."""
        cache = self.__dict__.setdefault('_predictors', {})
        if batch not in cache:
            from lib.compact_eval import RoutedPredictor
            cache[batch] = RoutedPredictor(self.compact_evaluator(batch))
        return cache[batch]

    def eval_stats(self, feed_dict):
        """Per-example `state_tensors` (train-nets:111-130) for one batch, as a
        dict {(net|layer, name): ndarray}; `mode` defaults to 'ev'."""
        return self._get_engine().eval_stats(feed_dict)

# ---- statically-routed networks (net_types.py:85-97) -----------------------


class SRNet(Net):
    default_hypers = Ns(λ_lrn=1e-3, μ_lrn=0.9)

    def link(self):
        super().link()
        ϕ = self.hypers
        self.λ_lrn = Placeholder('λ_lrn', ϕ.λ_lrn)
        self.μ_lrn = Placeholder('μ_lrn', ϕ.μ_lrn)

# ---- dynamically-routed networks (net_types.py:103-284) --------------------


class _DynNet(Net):
    dynamic = True

    def link(self):
        ϕ = self.hypers
        self.λ_lrn = Placeholder('λ_lrn', ϕ.λ_lrn)
        self.μ_lrn = Placeholder('μ_lrn', ϕ.μ_lrn)
        self.ϵ = Placeholder('ϵ', ϕ.ϵ)
        self.τ = Placeholder('τ', ϕ.τ)
        # a feed key when k_cpt varies per example, else the scalar hyper
        self.k_cpt = Placeholder('k_cpt') if ϕ.dyn_k_cpt else ϕ.k_cpt
        super().link()

    def _router_input(self, x):
        # dyn_k_cpt appends the feature α_cpt·k_cpt to the flattened router
        # input of every scale (net_types.py:149-160)
        if not self.hypers.dyn_k_cpt:
            return x

        def cat(s):
            n = 1
            for d in s.shape:
                n *= d
            return Sym((n + 1,), s.owner, s.name + '+k_cpt')
        return [cat(s) for s in x] if isinstance(x, list) else cat(x)


class ActorNet(_DynNet):
    default_hypers = Ns(
        k_cpt=0.0, k_dec=0.01, ϵ=1e-6, τ=1.0, λ_lrn=1e-3, μ_lrn=0.9,
        dyn_k_cpt=False, α_cpt=1e7, talr=True, α_rtr=1.0)


class CriticNet(_DynNet):
    default_hypers = Ns(
        k_cpt=0.0, k_cre=1e-3, ϵ=1e-6, τ=0.01, optimistic=False,
        dyn_k_cpt=False, α_cpt=1e7, use_cls_err=False, λ_lrn=1e-3, μ_lrn=0.9,
        talr=True, α_rtr=1.0)
