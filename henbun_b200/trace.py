"""Symbolic pass over a user objective, the stand-in for the reference's graph building
(Henbun/model.py:217-221: ``method_op = likelihood_method(model)`` inside tf_mode builds ONE TensorFlow graph that
every ``session.run`` replays).  ``Optimizer.compile`` runs the objective once with every parameter / data / sample
replaced by a ``Sym`` leaf; the ops of the hot path (tf.matmul, kern.Cholesky, densities.gaussian, tf.reduce_sum,
tf.sqrt, tf.sigmoid, NeuralNet calls, LOCAL feeds, KL()) build an expression tree instead of launching kernels.
``fused.py`` matches that tree against the graphs that have a whole-step C entry point (variational GP regression, the
mixture of GP experts in float64, the linear operator model, the amortised encoder/decoder model).  Anything the tracer
does not understand raises, and the Optimizer keeps the eager tape path -- tracing never changes results, it only selects
the faster executor."""
from __future__ import annotations

import contextlib

_ACTIVE = [False]
_DRAWS = []          # variationals of the current (or last) trace, in the order their first 'sample' node was created


def active() -> bool:
    return _ACTIVE[0]


def draws():
    """Variationals sampled by the last traced objective, in the order it first sampled them.  The eager tape takes each
    variational's Philox window at its first sample, so this is the order of those windows."""
    return list(_DRAWS)


@contextlib.contextmanager
def tracing():
    _ACTIVE[0] = True
    del _DRAWS[:]
    try:
        yield
    finally:
        _ACTIVE[0] = False


class TraceError(TypeError):
    pass


class Sym(object):
    """Node of the traced objective: op name, positional children (Sym, python scalars or model objects), attributes."""
    __slots__ = ("op", "args", "kw")
    __array_priority__ = 1000      # numpy scalars defer to Sym's reflected operators

    def __init__(self, op, *args, **kw):
        self.op, self.args, self.kw = op, args, kw
        if op == 'sample' and _ACTIVE[0] and not any(q is args[0] for q in _DRAWS):
            _DRAWS.append(args[0])

    def _bin(self, op, other, swap=False):
        if not isinstance(other, (Sym, int, float)):
            raise TraceError(f"cannot trace {op} with {type(other).__name__}")
        return Sym(op, other, self) if swap else Sym(op, self, other)

    def __add__(self, o): return self._bin("add", o)
    def __radd__(self, o): return self._bin("add", o, True)
    def __sub__(self, o): return self._bin("sub", o)
    def __rsub__(self, o): return self._bin("sub", o, True)
    def __mul__(self, o): return self._bin("mul", o)
    def __rmul__(self, o): return self._bin("mul", o, True)
    def __truediv__(self, o): return self._bin("div", o)
    def __rtruediv__(self, o): return self._bin("div", o, True)
    def __neg__(self): return Sym("neg", self)

    # anything else a tensor could do is outside the traced vocabulary
    def __getattr__(self, name):
        raise TraceError(f"'{name}' is not traced")

    def __getitem__(self, key):
        raise TraceError("indexing is not traced")

    def __array__(self, *a, **k):
        raise TraceError("conversion to an array is not traced")

    def __bool__(self):
        raise TraceError("truth value of a traced tensor")

    def __repr__(self):
        def r(a):
            return repr(a) if isinstance(a, Sym) else (type(a).__name__ if not isinstance(a, (int, float, str, type(None))) else repr(a))
        return f"{self.op}({', '.join(r(a) for a in self.args)})"


def is_sym(*xs) -> bool:
    return any(isinstance(x, Sym) for x in xs)
