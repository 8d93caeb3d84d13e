"""Driver: mirror of Henbun/model.py (Model :13-123, Indexer :126-153, AutoOptimize :155-188,
Optimizer :190-269).

The reference compiles the user's objective into one TF graph and loops ``session.run(optimize_op)``.
``Optimizer.compile`` traces the objective once (trace.py) and binds a recognised graph -- the notebook's
variational GP regression, the linear-operator model, the amortised encoder/decoder model -- to its
whole-step C entry point (fused.py): one C call per step writes the gradient into the flat buffer.  Any
other objective is evaluated eagerly on device tensors every step (each heavy op is one of this package's
CUDA kernels) with torch's autograd tape driving the hand-written backward kernels.  Either way the TF-1
Adam rule is applied by one fused kernel on the flat parameter buffer -- after a single NCCL all-reduce
of the flat gradient when torch.distributed is initialised (one process per GPU; the GP binding
additionally shares ONE block-cyclic factorisation between the ranks).

New, non-reference knobs (SURVEY.md 8b): ``compile(n_samples=S, seed=...)`` and
``run/optimize(eps={variational: tensor})``.
"""
from __future__ import annotations

from functools import wraps

import numpy as np
import torch

from . import ops
from .param import Parameterized, Variable, Data, MinibatchData, graph_key, _device
from .train import AdamOptimizer
from .variationals import RunContext
from ._settings import settings


class _Session(object):
    """Stand-in for the reference's tf.Session handle (Model._session): a CUDA stream owner."""

    def __init__(self):
        self.closed = False

    def run(self, fetch, feed_dict=None):
        if callable(fetch):
            fetch = fetch()
        if isinstance(fetch, (list, tuple)):
            return [self.run(f) for f in fetch]
        if isinstance(fetch, torch.Tensor):
            return fetch.detach().cpu().numpy()
        return fetch


class Model(Parameterized):
    """Base class of every model; parameters are defined in ``setUp`` (Henbun/model.py:13-123)."""

    def __init__(self, name='model', **kw):
        Parameterized.__init__(self)
        self._name = name
        self._session = _Session()
        self._index = Indexer()
        self._run_ctx = RunContext()
        self.setUp(**kw)

    @property
    def name(self):
        return self._name

    def setUp(self):
        pass

    def initialize(self):
        """Apply pending assignments (Henbun/model.py:76-82)."""
        for op in self.initialize_ops:
            op()
        self.finalize()

    def _feed(self, feed_dict):
        for var, value in feed_dict.items():
            if isinstance(var, MinibatchData):
                var._gather(value)
            elif isinstance(var, Data):
                var._upload(value)

    def run(self, tensor, feed_dict=None, n_samples=1, eps=None, seed=None):
        """Evaluate ``tensor`` with the current parameters (Henbun/model.py:84-96).  Because evaluation is
        eager, pass a zero-argument callable to get a fresh sample per call (it is executed inside
        tf_mode); an already evaluated tensor is simply copied to the host."""
        self.initialize()
        if feed_dict is None:
            feed_dict = self.get_feed_dict()
        self._feed(feed_dict)
        if callable(tensor):
            self._begin_run(n_samples, eps, seed)
            was = object.__getattribute__(self, '_tf_mode')
            if was:
                out = tensor()
            else:
                with self.tf_mode():
                    out = tensor()
            return self._session.run(out)
        out = self._session.run(tensor)
        # the value was computed eagerly before this call; start a new run so that the next access to
        # a variational draws a fresh sample (the reference re-samples on every session.run)
        self._new_run(self._run_ctx)
        return out

    def _begin_run(self, n_samples=1, eps=None, seed=None, shard=None):
        ctx = self._run_ctx
        ctx.n_samples = int(n_samples)
        ctx.eps = eps or {}
        if seed is not None:
            ctx.seed = int(seed)
        # (first sample of this rank, samples over all ranks): ranks read disjoint windows of one Philox stream
        ctx.first_sample, ctx.total_samples = shard if shard is not None else (0, int(n_samples))
        self._new_run(ctx)

    def validate(self):
        """Henbun/model.py:98-117."""
        minibatch_data = [d for d in self.get_variables(graph_key.DATA) if isinstance(d, MinibatchData)]
        if len(minibatch_data) > 1:
            for d in minibatch_data:
                if d.data_size != minibatch_data[0].data_size:
                    raise ValueError('Minibatch data' + d.long_name + ' is not the same size.')
        if len(minibatch_data) > 0:
            data_size = minibatch_data[0].data_size
            if self._index.data_size is None or self._index.data_size != data_size:
                self._index.setUp(data_size)

    def test_feed_dict(self, minibatch_size=None):
        return self.get_feed_dict(self._index.test_index(minibatch_size))


class Indexer(object):
    """Train/test split and random-with-replacement minibatch indices (Henbun/model.py:126-153)."""

    def __init__(self):
        self.data_size = None
        self.test_frac = 0.1

    def setUp(self, data_size):
        self.data_size = data_size
        self.test_size = int(np.floor(self.data_size * self.test_frac))
        self.train_size = data_size - self.test_size
        index = np.array(range(self.data_size))
        np.random.shuffle(index)
        self._train_index = index[:self.train_size]
        self._test_index = index[self.train_size:]

    def train_index(self, minibatch_size):
        return self._train_index[np.random.randint(0, self.train_size, minibatch_size)]

    def test_index(self, minibatch_size):
        return self._test_index[np.random.randint(0, self.test_size, minibatch_size)]

    # ---- the same draws on the device: no host RNG, no host gather, no H2D copy per step (SURVEY.md 8f rank 3) ----
    def _device_pool(self, which):
        key = '_dev_' + which
        if getattr(self, key, None) is None or getattr(self, key + '_src', None) is not getattr(self, '_' + which + '_index'):
            host = getattr(self, '_' + which + '_index')
            setattr(self, key, torch.as_tensor(np.asarray(host, dtype=np.int64)).to(_device()))
            setattr(self, key + '_src', host)
        return getattr(self, key)

    def device_index(self, minibatch_size, seed, offset, training=True):
        """int64 device tensor of `minibatch_size` indices drawn with replacement from the train (test) split by the
        Philox stream (seed, offset) -- hb_random_index."""
        pool = self._device_pool('train' if training else 'test')
        out = torch.empty(int(minibatch_size), dtype=torch.int64, device=pool.device)
        ops._lib.check(ops._L().hb_random_index(ops.ptr(out), int(minibatch_size), ops.ptr(pool), pool.numel(), int(seed),
                                                int(offset), ops.stream()), "hb_random_index")
        return out


class AutoOptimize(object):
    """Decorator turning a model method into an Optimizer factory (Henbun/model.py:155-188)."""

    def __init__(self):
        pass

    def __call__(self, method):
        @wraps(method)
        def runnable(instance):
            optimizer_name = '_' + method.__name__ + '_AF_optimizer'
            if hasattr(instance, optimizer_name):
                optimizer = getattr(instance, optimizer_name)
            else:
                optimizer = Optimizer(instance, method)
                object.__setattr__(instance, optimizer_name, optimizer)
            return optimizer

        return runnable


_default_adam = AdamOptimizer()


class Optimizer(object):
    """Henbun/model.py:190-269."""

    def __init__(self, model_instance, likelihood_method):
        self.model = model_instance
        self.likelihood_method = likelihood_method
        self.method_op = None
        self.optimize_op = None
        self.n_samples = 1
        self._flat = None
        self._compiled_settings = None

    # ---- compile: bind parameters to flat buffers, create Adam slots ----
    def compile(self, optimizer=None, collection=graph_key.VARIABLES, global_step=None, n_samples=1, seed=0,
                verbose=True, shard=None, fused=True, device_index=True, shared_factorisation=True):
        """``shard`` (multi-GPU, one process per GPU): 'samples' splits the n_samples draws over the ranks
        (contiguous windows of ONE Philox stream, so the union over ranks is the single-GPU draw), 'batch' keeps
        n_samples per rank and splits the minibatch (each rank draws its own indices and its own Philox window).
        Default: 'batch' when the model holds MinibatchData, else 'samples'.  ``fused=True`` lets compile bind a
        recognised objective to one of the fused C entry points (henbun_b200/fused.py)."""
        if verbose:
            print('compiling...')
        m = self.model
        self.optimizer = optimizer if optimizer is not None else _default_adam
        self.n_samples = int(n_samples)
        self.global_step = global_step
        self._seed = int(seed)
        self._shard_mode = shard
        self._shared_factorisation = bool(shared_factorisation)   # multi-GPU GP objective: one block-cyclic Cholesky for all ranks
        self._want_fused = bool(fused)
        self._fused = None
        self._device_index = bool(device_index)    # minibatch indices drawn on the device (False: numpy's global RNG, as upstream)
        self._index_draws = 0
        m.initialize()
        variables = [v for v in m.get_variables(collection) if isinstance(v, Variable) and v.is_parameter]
        # de-duplicate while keeping the reference's name-sorted order (param.py:467-475)
        seen, var_list = set(), []
        for v in variables:
            if id(v) not in seen:
                seen.add(id(v)); var_list.append(v)
        # graph building: trace the objective once; a recognised graph is bound to its whole-step C entry point and
        # the flat buffer takes that entry point's parameter packing (SURVEY.md section 7, step 2)
        binding = self._trace_and_bind() if fused else None
        if binding is not None and {id(v) for v in binding.var_order} == {id(v) for v in var_list}:
            var_list = list(binding.var_order)
            self._fused = binding
        self.var_list = var_list
        dev = _device()
        sizes = [int(np.prod(v._host.shape)) for v in var_list]
        pad = (lambda s: s) if self._fused is not None else (lambda s: (s + 3) // 4 * 4)
        offs = np.concatenate([[0], np.cumsum([pad(s) for s in sizes])]).astype(np.int64)
        total = int(offs[-1])
        self._flat = torch.zeros(max(total, 4), device=dev)
        self._flat_grad = torch.zeros(max(total, 4), device=dev)
        self._slices = [(int(o), int(s)) for o, s in zip(offs[:-1], sizes)]
        self._bind_all()
        # Adam slots are (re)created at every compile, parameter values are kept (test_model.py:61-74)
        self._m = torch.zeros_like(self._flat)
        self._v = torch.zeros_like(self._flat)
        self._step = torch.zeros(1, dtype=torch.int32, device=dev)
        m._run_ctx.seed = int(seed)
        self._compiled_settings = settings.get_settings()     # jitter / clip are read at compile time
        self.method_op = self._evaluate
        self.optimize_op = self._step_once
        m.validate()
        # one evaluation now: shape errors and unfed LOCAL variables surface here, like graph building
        # (a traced-and-bound graph has been validated already: no need to allocate the eager path's buffers)
        if self._fused is None:
            self._evaluate(self.feed_dict(None) if self._no_minibatch() else None, dry=True)
        m._run_ctx.offset = 0                     # the training stream starts at position 0 whichever executor was bound
        if verbose:
            print('finished.')

    def _trace_and_bind(self):
        from . import trace, fused
        m = self.model
        if bool(settings.numerics.clip_by_value):
            return None                       # the whole-step entry points implement the default (clip off) graph
        tree = None
        try:
            with trace.tracing():
                with m.tf_mode():
                    tree = self.likelihood_method(m)
        except Exception:
            tree = None
        finally:
            for v in fused._variationals_of(m):
                if '_sym_feed' in v.__dict__:
                    del v.__dict__['_sym_feed']
        if not isinstance(tree, trace.Sym):
            return None
        return fused.bind(tree, m)

    @property
    def fused_entry(self):
        """Name of the whole-step C entry point this objective was bound to at compile time (None: eager tape)."""
        return type(self._fused).__name__ if self._fused is not None else None

    def _bind_all(self):
        for v, (o, s) in zip(self.var_list, self._slices):
            v._rebind(self._flat[o:o + s], self._flat_grad[o:o + s])

    def _ensure_bound(self):
        """Another Optimizer compiled over some of the same variables re-binds them to ITS flat buffers (TF minimize
        ops share tf.Variables: testing/test_gp.py compiles likelihood_ana then likelihood_var).  Take the
        variables back -- current values are copied into this optimizer's buffer, Adam slots are kept."""
        for v, (o, s) in zip(self.var_list, self._slices):
            t = v._tensor
            if t is None or t.data_ptr() != self._flat.data_ptr() + 4 * o or t.grad is None or \
                    t.grad.data_ptr() != self._flat_grad.data_ptr() + 4 * o:
                v._rebind(self._flat[o:o + s], self._flat_grad[o:o + s])

    def _shard(self):
        """(first_sample, local_count, total_count, world) of this rank for the compiled n_samples."""
        from . import parallel
        world, rank = parallel.world()
        S = self.n_samples
        if world == 1:
            return 0, S, S, 1
        mode = self._shard_mode or ('samples' if self._no_minibatch() else 'batch')
        if mode == 'samples' and S % world == 0:
            first, count = parallel.shard_samples(S, world, rank)
            return first, count, S, world
        return rank * S, S, S * world, world        # every rank draws S samples of its own window

    def _no_minibatch(self):
        return not any(isinstance(d, MinibatchData) for d in self.model.get_variables(graph_key.DATA))

    def feed_dict(self, minibatch_size=None, training=True):
        if minibatch_size is None:
            return self.model.get_feed_dict(None)
        if getattr(self, '_device_index', False) and self.model._index.data_size is not None:
            # a Philox stream of its own (key = seed + 1): index draws never collide with the eps windows
            from . import parallel
            _, rank = parallel.world()
            per = (int(minibatch_size) + 1) // 2 * 4
            off = self._index_draws * per
            self._index_draws += 1
            idx = self.model._index.device_index(minibatch_size, self._seed + 1 + 7919 * rank, off, training)
            return self.model.get_feed_dict(idx)
        elif training:
            return self.model.get_feed_dict(self.model._index.train_index(minibatch_size))
        return self.model.get_feed_dict(self.model._index.test_index(minibatch_size))

    # ---- one objective evaluation (the reference's session.run(method_op)) ----
    def _evaluate(self, feed_dict, eps=None, dry=False, grad=False):
        m = self.model
        if feed_dict is None and dry:
            return None
        m.initialize()                           # pending assignments apply at the next run (Henbun/model.py:84-96)
        m._feed(feed_dict or {})
        self._ensure_bound()
        first, count, total, _ = self._shard()
        with settings.temp_settings(self._compiled_settings):
            m._begin_run(count, eps, shard=(first, total))
            with torch.set_grad_enabled(grad):
                with m.tf_mode():
                    obj = self.likelihood_method(m)
        if not isinstance(obj, torch.Tensor):
            obj = torch.as_tensor(obj, dtype=torch.float32, device=_device())
        return obj.reshape(()) / float(count)

    def run(self, minibatch_size=None, training=True, eps=None):
        """Objective value with the current parameters (mean over the compiled n_samples)."""
        self._require_compiled()
        try:
            val = self._evaluate(self.feed_dict(minibatch_size, training), eps=eps)
            ops.check_numerics()
            return val.detach().cpu().numpy()
        except KeyboardInterrupt:
            raise KeyboardInterrupt

    def _require_compiled(self):
        if self._flat is None:
            raise RuntimeError('call .compile() first')

    def _fused_step(self, feed_dict, eps):
        """One step through the bound whole-step entry point: same Philox windows, same Adam rule as the tape path."""
        m, b = self.model, self._fused
        m.initialize()
        m._feed(feed_dict or {})
        self._ensure_bound()
        first, count, total, world = self._shard()
        with settings.temp_settings(self._compiled_settings):
            m._begin_run(count, eps, shard=(first, total))
        ctx = m._run_ctx
        qs = getattr(b, 'qs', None)
        if qs is not None:
            # several variationals: one eps (or Philox window, taken in the order the tape takes them) per variational
            es = [None if not eps else eps.get(q, None) for q in qs]
            offsets = [ctx.take_sharded(b.per_sample()) if e is None else 0 for e in es]
            return b.step(self, count, es, ctx.seed, offsets, world)
        q = b.q
        e = None if not eps else eps.get(q, None)
        offset = ctx.take_sharded(b.per_sample()) if e is None else 0
        o = self.optimizer
        if getattr(b, 'fused_adam', False):
            return b.step(self, count, e, ctx.seed, offset, world)
        obj = b.step(self, count, e, ctx.seed, offset)
        if world > 1:
            torch.distributed.all_reduce(self._flat_grad)
        ops._lib.check(ops._L().hb_increment_i32(ops.ptr(self._step), ops.stream()), "hb_increment_i32")
        ops.adam_tf1_(self._flat, self._flat_grad, self._m, self._v, self._step, o.learning_rate, o.beta1, o.beta2,
                      o.epsilon, grad_scale=-1.0 / world)
        return obj

    def _step_once(self, feed_dict, eps=None):
        if self._fused is not None:
            world = self._shard()[3]
            if world == 1 or not getattr(self._fused, 'fused_adam', False):
                return self._fused_step(feed_dict, eps)
        self._flat_grad.zero_()
        obj = self._evaluate(feed_dict, eps=eps, grad=True)
        obj.backward()
        world = 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            world = torch.distributed.get_world_size()
            if world > 1:
                torch.distributed.all_reduce(self._flat_grad)      # the single collective of a step
        o = self.optimizer
        ops._lib.check(ops._L().hb_increment_i32(ops.ptr(self._step), ops.stream()), "hb_increment_i32")
        ops.adam_tf1_(self._flat, self._flat_grad, self._m, self._v, self._step, o.learning_rate, o.beta1, o.beta2,
                      o.epsilon, grad_scale=-1.0 / world)            # minimise(-objective)
        return obj

    def optimize(self, maxiter=1, minibatch_size=None, eps=None, check_every=100):
        """Henbun/model.py:255-269: maxiter Adam steps on -objective."""
        self._require_compiled()
        iteration = 0
        last = None
        if minibatch_size is not None:
            # batch-sharded multi-GPU run: each rank draws minibatch_size / world rows of its own
            world = self._shard()[3]
            if world > 1 and (self._shard_mode or 'batch') == 'batch':
                minibatch_size = max(1, int(minibatch_size) // world)
        while iteration < maxiter:
            try:
                last = self._step_once(self.feed_dict(minibatch_size), eps=eps)
                iteration += 1
                if check_every and iteration % check_every == 0:
                    ops.check_numerics()
            except KeyboardInterrupt:
                raise KeyboardInterrupt
        # a failed factorisation must not go unnoticed whatever maxiter is (tf.cholesky raises immediately upstream):
        # one flag read per optimize() call
        ops.check_numerics()
        self.last_objective = last
        return last
