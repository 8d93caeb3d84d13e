"""A minimal TensorFlow-1.x graph-mode shim (lazy graph over torch-CPU float64) -- TEST TOOLING ONLY.

Purpose: TensorFlow cannot be installed in this image, but the reference (fujii-team/Henbun) is pure
Python on top of ~60 TF-1 symbols.  This shim provides exactly those symbols so that
``tests/golden/make_golden.py`` can import and execute the UNMODIFIED reference modules from
a checkout of it and record what the reference's own code computes (sampler, KL, kernels, Cholesky,
NeuralNet, LOCAL feed, ELBO of the notebook models, tf.gradients of all of it, AdamOptimizer steps).
The recorded vectors are committed under tests/golden/*.npz and pin the oracle.

What is restated here (from TF-1 documentation) is only the semantics of the individual TF ops;
every composition -- which op is applied to what, in which order, with which shapes -- is the
reference's own code.  All arithmetic is float64 so the vectors are exact to ~1e-15.
Nothing in the product or in the GPU tests imports this file.
"""
from __future__ import annotations

import math
import sys
import types

import numpy as np
import torch

DT = torch.float64


class DType(object):
    def __init__(self, name, tdt):
        self.name = name
        self.torch = tdt
        self.as_numpy_dtype = {"float32": np.float32, "float64": np.float64, "int32": np.int32, "int64": np.int64,
                               "float16": np.float16, "int16": np.int16}[name]

    def __repr__(self):
        return "tf." + self.name


float16 = DType("float16", DT)
float32 = DType("float32", DT)          # every float computes in float64 (see module docstring)
float64 = DType("float64", DT)
int16 = DType("int16", torch.int64)
int32 = DType("int32", torch.int64)
int64 = DType("int64", torch.int64)


class Dim(object):
    def __init__(self, v):
        self.value = v


class TShape(object):
    def __init__(self, dims):
        self.dims = None if dims is None else [d for d in dims]
        self.ndims = None if dims is None else len(dims)

    def __getitem__(self, i):
        return self.dims[i]

    def __len__(self):
        return len(self.dims)

    def as_list(self):
        return list(self.dims)


class _Graph(object):
    def __init__(self):
        self.variables = []
        self.seed = None
        self.rng = np.random.RandomState(0)


_graph = _Graph()


def reset_default_graph():
    global _graph
    _graph = _Graph()


def set_random_seed(seed):
    _graph.seed = seed
    _graph.rng = np.random.RandomState(seed)


def _as_t(v):
    if isinstance(v, torch.Tensor):
        return v
    a = np.asarray(v)
    if a.dtype.kind in "iub":
        return torch.as_tensor(a.astype(np.int64))
    return torch.as_tensor(a.astype(np.float64))


class Tensor(object):
    """A node of the lazy graph."""
    _count = 0
    __array_ufunc__ = None      # numpy operands defer to the reflected operators below

    def __init__(self, fn, inputs=(), static_shape=None, name=None):
        self.fn = fn
        self.inputs = list(inputs)
        self._static = static_shape
        Tensor._count += 1
        self.name = (name or "node") + "_%d:0" % Tensor._count
        self.op = types.SimpleNamespace(name=self.name[:-2])

    # --- evaluation ---
    is_source = False        # random draws: realised once per session.run, reused by gradient re-evaluation

    def _eval(self, env):
        src = env["_src"]
        if id(self) in src:
            return src[id(self)]
        if id(self) in env:
            return env[id(self)]
        args = [(_ev(i, env)) for i in self.inputs]
        out = self.fn(*args)
        (src if self.is_source else env)[id(self)] = out
        return out

    def get_shape(self):
        return TShape(self._static)

    @property
    def shape(self):
        return TShape(self._static)

    # --- operators ---
    def __add__(self, o): return _bin(torch.add, self, o)
    def __radd__(self, o): return _bin(torch.add, o, self)
    def __sub__(self, o): return _bin(torch.sub, self, o)
    def __rsub__(self, o): return _bin(torch.sub, o, self)
    def __mul__(self, o): return _bin(torch.mul, self, o)
    def __rmul__(self, o): return _bin(torch.mul, o, self)
    def __truediv__(self, o): return _bin(torch.div, self, o)
    def __rtruediv__(self, o): return _bin(torch.div, o, self)
    __div__ = __truediv__
    __rdiv__ = __rtruediv__
    def __neg__(self): return _un(torch.neg, self)
    def __pow__(self, o): return _bin(torch.pow, self, o)
    def __getitem__(self, idx): return Tensor(lambda x: x[idx], [self])
    __hash__ = object.__hash__


def _ev(x, env):
    if isinstance(x, Tensor):
        return x._eval(env)
    if isinstance(x, (list, tuple)):
        return [_ev(i, env) for i in x]
    return x


def _v(x):
    """torch value of an already evaluated argument or a python/numpy constant."""
    return x if isinstance(x, torch.Tensor) else _as_t(x)


def _shape_of(x):
    if isinstance(x, Tensor):
        return x._static
    try:
        return list(np.shape(x))
    except Exception:
        return None


def _bshape(a, b):
    sa, sb = _shape_of(a), _shape_of(b)
    if sa is None or sb is None:
        return None
    try:
        return list(np.broadcast_shapes(tuple(1 if d is None else d for d in sa), tuple(1 if d is None else d for d in sb)))
    except Exception:
        return None


def _bin(f, a, b):
    def go(x, y):
        x, y = _v(x), _v(y)
        if x.is_floating_point() or y.is_floating_point():
            x, y = x.to(DT), y.to(DT)
        return f(x, y)
    return Tensor(go, [a, b], _bshape(a, b))


def _un(f, a, shape_same=True):
    return Tensor(lambda x: f(_v(x)), [a], _shape_of(a) if shape_same else None)


class Variable(Tensor):
    def __init__(self, initial_value=None, dtype=None, collections=None, name=None, trainable=True):
        Tensor.__init__(self, None, [], _shape_of(initial_value), name or "Variable")
        self._init = initial_value
        self.value_t = None
        self.collections = collections
        self.initialized = False
        _graph.variables.append(self)
        self.initializer = Op(lambda: self._do_init())

    def _do_init(self):
        env = {"_src": {}}
        v = _ev(self._init, env)
        self.value_t = _v(v).detach().clone().to(DT)
        self.initialized = True

    def _eval(self, env):
        if id(self) in env["_src"]:
            return env["_src"][id(self)]
        if id(self) in env:
            return env[id(self)]
        if not self.initialized:
            raise RuntimeError("Attempting to use uninitialized value " + self.name)
        env[id(self)] = self.value_t
        return self.value_t

    def assign(self, value):
        def do():
            val = _v(_ev(value, {"_src": {}})).detach().clone().to(DT)
            self.value_t = val.reshape(self.value_t.shape) if self.value_t is not None else val
            self.initialized = True
        return Op(do)


class Op(object):
    """A stateful graph operation (initialiser, assign, optimiser step)."""

    def __init__(self, fn):
        self.fn = fn


def variables_initializer(var_list, name=None):
    return Op(lambda: [v._do_init() for v in var_list])


def global_variables():
    return list(_graph.variables)


def is_variable_initialized(v):
    return Tensor(lambda: torch.tensor(bool(v.initialized)), [])


class GraphKeys(object):
    GLOBAL_VARIABLES = "variables"
    VARIABLES = "variables"


class Session(object):
    def __init__(self, *a, **k):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def run(self, fetches, feed_dict=None):
        env = {"_src": {}}
        for k, v in (feed_dict or {}).items():
            env["_src"][id(k)] = _as_t(v).to(DT) if _as_t(v).is_floating_point() else _as_t(v)
        return self._run(fetches, env)

    def _run(self, f, env):
        if isinstance(f, (list, tuple)):
            return [self._run(x, env) for x in f]
        if isinstance(f, Op):
            f.fn()
            return None
        if isinstance(f, Tensor):
            out = f._eval(env)
            if isinstance(out, torch.Tensor):
                a = out.detach().numpy()
                return a if a.ndim else a[()]
            return out
        return f


# --------------------------------------------------------------------------- sources
def placeholder(dtype=None, shape=None, name=None):
    def missing():
        raise RuntimeError("placeholder was not fed")
    return Tensor(missing, [], None if shape is None else list(shape), name or "Placeholder")


def constant(value, dtype=None, shape=None, name=None):
    t = _as_t(value)
    return Tensor(lambda: t, [], list(t.shape))


def convert_to_tensor(value, dtype=None, name=None):
    if isinstance(value, Tensor):
        return value
    return constant(value, dtype)


def _static_or_none(shape):
    try:
        return [int(s) for s in shape]
    except Exception:
        return None


def _resolve_shape(shape):
    return [int(_v(s)) if not isinstance(s, int) else s for s in shape]


def random_normal(shape, mean=0.0, stddev=1.0, dtype=None, seed=None, name=None):
    def draw(*dyn):
        shp = _resolve_shape(dyn[0]) if dyn else list(shape)
        return torch.as_tensor(mean + stddev * _graph.rng.standard_normal(size=tuple(shp)))
    if isinstance(shape, Tensor) or any(isinstance(s, Tensor) for s in (shape if isinstance(shape, (list, tuple)) else [])):
        t = Tensor(lambda s: draw(s), [list(shape) if isinstance(shape, (list, tuple)) else shape], None)
    else:
        t = Tensor(lambda: draw(), [], _static_or_none(shape))
    t.is_source = True
    return t


def truncated_normal(shape, mean=0.0, stddev=1.0, dtype=None, seed=None, name=None):
    def draw():
        out = _graph.rng.standard_normal(size=tuple(shape))
        bad = np.abs(out) > 2.0
        while bad.any():
            out[bad] = _graph.rng.standard_normal(size=int(bad.sum()))
            bad = np.abs(out) > 2.0
        return torch.as_tensor(mean + stddev * out)
    return Tensor(draw, [], _static_or_none(shape))


def ones(shape, dtype=None, name=None):
    if isinstance(shape, Tensor) or any(isinstance(s, Tensor) for s in shape):
        return Tensor(lambda s: torch.ones(_resolve_shape(s), dtype=DT), [list(shape) if isinstance(shape, (list, tuple)) else shape])
    return Tensor(lambda: torch.ones(list(shape), dtype=DT), [], list(shape))


def zeros(shape, dtype=None, name=None):
    shp = list(shape) if isinstance(shape, (list, tuple)) else [shape]
    return Tensor(lambda: torch.zeros(shp, dtype=DT), [], shp)


def ones_like(x, dtype=None): return _un(torch.ones_like, x)
def zeros_like(x, dtype=None): return _un(torch.zeros_like, x)


# --------------------------------------------------------------------------- elementwise / reductions
def exp(x, name=None): return _un(torch.exp, x)
def log(x, name=None): return _un(torch.log, x)
def sqrt(x, name=None): return _un(torch.sqrt, x)
def square(x, name=None): return _un(torch.square, x)
def abs(x, name=None): return _un(torch.abs, x)  # noqa: A001
def negative(x, name=None): return _un(torch.neg, x)
def identity(x, name=None): return _un(lambda t: t, x)
def lgamma(x, name=None): return _un(torch.lgamma, x)
def sigmoid(x, name=None): return _un(torch.sigmoid, x)
def tanh(x, name=None): return _un(torch.tanh, x)
def add(a, b, name=None): return _bin(torch.add, a, b)
def multiply(a, b, name=None): return _bin(torch.mul, a, b)
def cast(x, dtype, name=None): return _un(lambda t: t.to(dtype.torch), x)
def clip_by_value(x, lo, hi, name=None): return _un(lambda t: torch.clamp(t, lo, hi), x)
def equal(a, b): return _bin(torch.eq, a, b)
def select(cond, a, b):                                        # TF <= 0.12 name of tf.where (densities.py:36)
    return Tensor(lambda c, x, y: torch.where(_v(c), _as_t(_v(x)), _as_t(_v(y))), [cond, a, b], None)


def _red(f):
    def r(x, axis=None, keep_dims=False, name=None, reduction_indices=None):
        ax = axis if axis is not None else reduction_indices
        def go(t):
            t = _v(t)
            if ax is None:
                return f(t)
            return f(t, dim=ax, keepdim=keep_dims)
        return Tensor(go, [x], None)
    return r


reduce_sum = _red(torch.sum)
reduce_mean = _red(torch.mean)
reduce_max = _red(lambda t, **k: torch.amax(t, **k) if k else torch.max(t))


def rank(x):
    s = _shape_of(x)
    return len(s) if s is not None else Tensor(lambda t: torch.tensor(_v(t).dim()), [x])


def size(x): return Tensor(lambda t: torch.tensor(_v(t).numel()), [x])


def shape(x, name=None):
    return Tensor(lambda t: torch.tensor(list(_v(t).shape), dtype=torch.int64), [x], None)


def reshape(x, shp, name=None):
    def go(t, s):
        s = [int(_v(i)) for i in s] if isinstance(s, (list, tuple)) else [int(i) for i in _v(s)]
        return _v(t).reshape(s)
    static = None
    if isinstance(shp, (list, tuple)) and all(isinstance(i, int) for i in shp):
        static = [None if i == -1 else i for i in shp]
    return Tensor(go, [x, list(shp) if isinstance(shp, (list, tuple)) else shp], static)


def expand_dims(x, axis, name=None):
    s = _shape_of(x)
    static = None
    if s is not None:
        static = list(s); static.insert(axis if axis >= 0 else len(s) + 1 + axis, 1)
    return Tensor(lambda t: _v(t).unsqueeze(axis), [x], static)


def squeeze(x, axis=None, name=None, squeeze_dims=None):
    ax = axis if axis is not None else squeeze_dims
    def go(t):
        t = _v(t)
        if ax is None:
            return t.squeeze()
        for a in sorted([a % t.dim() for a in (ax if isinstance(ax, (list, tuple)) else [ax])], reverse=True):
            t = t.squeeze(a)
        return t
    return Tensor(go, [x], None)


def slice(x, begin, size, name=None):  # noqa: A001
    def go(t, b, s):
        t = _v(t); b = [int(i) for i in _v(b)]; s = [int(i) for i in _v(s)]
        idx = tuple(builtins_slice(bi, None if si == -1 else bi + si) for bi, si in zip(b, s))
        return t[idx]
    return Tensor(go, [x, begin, size], None)


builtins_slice = __builtins__["slice"] if isinstance(__builtins__, dict) else __builtins__.slice


def tile(x, multiples, name=None):
    def go(t, m):
        return _v(t).repeat(*[int(_v(i)) for i in m])
    return Tensor(go, [x, list(multiples)], None)


def stack(values, axis=0, name=None):
    return Tensor(lambda vs: torch.stack([_v(v) for v in vs], dim=axis), [list(values)], None)


def transpose(x, perm=None, name=None):
    return Tensor(lambda t: _v(t).permute(*perm) if perm is not None else _v(t).t(), [x], None)


# --------------------------------------------------------------------------- linear algebra
def matmul(a, b, transpose_a=False, transpose_b=False, name=None):
    def go(x, y):
        x = _v(x).to(DT); y = _v(y).to(DT)
        if transpose_a:
            x = x.transpose(-1, -2)
        if transpose_b:
            y = y.transpose(-1, -2)
        return torch.matmul(x, y)
    sa, sb = _shape_of(a), _shape_of(b)
    static = None
    if sa is not None and sb is not None and len(sa) >= 2 and len(sb) >= 2:
        m = sa[-1] if transpose_a else sa[-2]
        n = sb[-2] if transpose_b else sb[-1]
        static = list(sa[:-2]) + [m, n]
    return Tensor(go, [a, b], static)


def matrix_band_part(x, num_lower, num_upper, name=None):
    def go(t):
        t = _v(t)
        if num_lower == -1 and num_upper == 0:
            return torch.tril(t)
        if num_lower == 0 and num_upper == -1:
            return torch.triu(t)
        raise NotImplementedError
    return Tensor(go, [x], _shape_of(x))


def matrix_diag_part(x, name=None):
    return Tensor(lambda t: torch.diagonal(_v(t), dim1=-2, dim2=-1), [x], None)


diag_part = matrix_diag_part


def diag(x, name=None):
    return Tensor(lambda t: torch.diag(_v(t)), [x], None)


def cholesky(x, name=None):
    return Tensor(lambda t: torch.linalg.cholesky(_v(t)), [x], _shape_of(x))


def matrix_triangular_solve(matrix, rhs, lower=True, adjoint=False, name=None):
    def go(m, r):
        m = _v(m); r = _v(r)
        if adjoint:
            m = m.transpose(-1, -2)
        return torch.linalg.solve_triangular(m, r, upper=(not lower) != adjoint)
    return Tensor(go, [matrix, rhs], _shape_of(rhs))


# --------------------------------------------------------------------------- autodiff + Adam
def _leaf_eval(ys, xs, parent_env):
    """Evaluate ys with fresh leaf copies of the variables xs (feeds and random draws of the
    current session.run are shared); returns (values, leaves)."""
    env = {"_src": parent_env["_src"]}
    leaves = []
    for x in xs:
        base = x._eval({"_src": parent_env["_src"]}) if not isinstance(x, Variable) else x.value_t
        leaf = _v(base).detach().clone().to(DT).requires_grad_(True)
        env[id(x)] = leaf
        leaves.append(leaf)
    vals = [y._eval(env) for y in ys]
    return vals, leaves


class _GradTensor(Tensor):
    def __init__(self, y, xs, i):
        Tensor.__init__(self, None, [], None, "grad")
        self.y, self.xs, self.i = y, xs, i

    def _eval(self, env):
        key = ("grads", id(self.y), tuple(id(x) for x in self.xs))
        if key not in env:
            vals, leaves = _leaf_eval([self.y], self.xs, env)
            gs = torch.autograd.grad(vals[0].sum(), leaves, allow_unused=True)
            env[key] = gs
        g = env[key][self.i]
        return g


def gradients(ys, xs, name=None):
    y = ys[0] if isinstance(ys, (list, tuple)) else ys
    xs = list(xs)
    out = []
    for i, x in enumerate(xs):
        out.append(_GradTensor(y, xs, i))
    return out


class _Nn(object):
    @staticmethod
    def softplus(x, name=None):
        return _un(lambda t: torch.clamp(t, min=0) + torch.log1p(torch.exp(-torch.abs(t))), x)

    sigmoid = staticmethod(sigmoid)
    tanh = staticmethod(tanh)

    @staticmethod
    def relu(x, name=None):
        return _un(torch.relu, x)


nn = _Nn()


class _AdamOptimizer(object):
    """tf.train.AdamOptimizer (TF 1.x): lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m,v EMAs;
    var -= lr_t * m / (sqrt(v) + eps)."""

    def __init__(self, learning_rate=0.001, beta1=0.9, beta2=0.999, epsilon=1e-08, use_locking=False, name="Adam"):
        self.lr, self.b1, self.b2, self.eps = learning_rate, beta1, beta2, epsilon

    def minimize(self, loss, var_list=None, global_step=None, name=None):
        var_list = list(var_list)
        state = {"t": 0, "m": [None] * len(var_list), "v": [None] * len(var_list)}
        slot = Variable(initial_value=np.zeros(1), name="adam_slots")     # so "initialise the uninitialised" sees it
        opt = self

        class StepOp(Op):
            pass

        step = StepOp(None)

        def run_with_env(env):
            vals, leaves = _leaf_eval([loss], var_list, env)
            gs = torch.autograd.grad(vals[0].sum(), leaves, allow_unused=True)
            state["t"] += 1
            t = state["t"]
            lr_t = opt.lr * math.sqrt(1 - opt.b2 ** t) / (1 - opt.b1 ** t)
            for i, (v, g) in enumerate(zip(var_list, gs)):
                if g is None:
                    continue
                if state["m"][i] is None:
                    state["m"][i] = torch.zeros_like(g); state["v"][i] = torch.zeros_like(g)
                state["m"][i] = opt.b1 * state["m"][i] + (1 - opt.b1) * g
                state["v"][i] = opt.b2 * state["v"][i] + (1 - opt.b2) * g * g
                v.value_t = (v.value_t - lr_t * state["m"][i] / (torch.sqrt(state["v"][i]) + opt.eps)).detach()
        step.run_with_env = run_with_env
        step.fn = lambda: run_with_env({"_src": {}})
        return step


class _Saver(object):
    def __init__(self, var_dict=None):
        self.var_dict = var_dict or {}

    def save(self, sess, path, **kw):
        np.savez(path, **{k: v.value_t.numpy() for k, v in self.var_dict.items()})
        return path

    def restore(self, sess, path):
        d = np.load(path if path.endswith(".npz") else path + ".npz")
        for k, v in self.var_dict.items():
            v.value_t = torch.as_tensor(d[k]); v.initialized = True


train = types.SimpleNamespace(AdamOptimizer=_AdamOptimizer, Saver=_Saver)


class name_scope(object):
    def __init__(self, *a, **k):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


# Session.run must hand the feed environment to optimiser steps
_orig_run = Session._run


def _run(self, f, env):
    if isinstance(f, Op) and hasattr(f, "run_with_env"):
        f.run_with_env(env)
        return None
    return _orig_run(self, f, env)


Session._run = _run


def install():
    """Register this module as ``tensorflow`` and patch py3.10+ incompatibilities of the reference."""
    import collections
    import collections.abc
    if not hasattr(collections, "Mapping"):
        collections.Mapping = collections.abc.Mapping          # Henbun/_settings.py:114
    sys.modules["tensorflow"] = sys.modules[__name__]
    return sys.modules[__name__]
