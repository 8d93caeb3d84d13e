"""Feed-forward networks, mirror of Henbun/nn.py (MatBias :10-32, NeuralNet :34-87).

``MatBias.__call__`` = activation(clip(x w + b)) is ONE CUDA kernel here (GEMM with bias/clip/
activation epilogue); the reference emits matmul, add, clip and the activation as separate TF ops
(nn.py:32,83).  Activations are named by the tf-compat callables in henbun_b200.tf (tf.sigmoid,
tf.nn.relu, tf.tanh) or by string."""
from __future__ import annotations

import numpy as np

from . import ops
from .param import Variable, Parameterized, graph_key
from ._settings import settings


def sigmoid(x, name=None):
    import torch
    from . import trace as _trace
    if isinstance(x, _trace.Sym):
        return _trace.Sym('sigmoid', x)
    return torch.sigmoid(x)


def relu(x, name=None):
    import torch
    return torch.relu(x)


def tanh(x, name=None):
    import torch
    return torch.tanh(x)


sigmoid._hb_act = 'sigmoid'
relu._hb_act = 'relu'
tanh._hb_act = 'tanh'


def _act_name(fn):
    if fn is None:
        return 'none'
    if isinstance(fn, str):
        return fn
    return getattr(fn, '_hb_act', None)


def _per_layer(spec, count):
    """A single value (repeated) or an explicit per-layer list."""
    return list(spec) if isinstance(spec, list) else [spec] * count


class MatBias(Parameterized):
    """One dense layer: parameters w [*n_layers, fan_in, fan_out] and b [*n_layers, 1, fan_out] (nn.py:23-29); calling
    it evaluates activation(clip(x w + b)) as ONE kernel (GEMM with the bias / clip / activation epilogue)."""

    def __init__(self, nodes, n_layers=[], mean=0.0, stddev=1.0, variable=Variable,
                 collections=[graph_key.VARIABLES]):
        assert len(nodes) == 2                                    # [fan_in, fan_out] (nn.py:23)
        fan_in, fan_out = nodes
        Parameterized.__init__(self)
        common = dict(n_layers=n_layers, mean=mean, stddev=stddev, collections=collections)
        self.w = variable(shape=[fan_in, fan_out], **common)
        self.b = variable(shape=[1, fan_out], **common)

    def __call__(self, x, activation=None):
        from . import trace as _trace
        if isinstance(x, _trace.Sym):
            raise _trace.TraceError("a bare MatBias call is not traced")
        numerics = settings.numerics
        return ops.matbias(x, self.w, self.b, act=activation if activation else 'none',
                           clip=bool(numerics.clip_by_value), lo=numerics.clip_value_min, hi=numerics.clip_value_max)


class NeuralNet(Parameterized):
    """Chain of MatBias layers over the widths in ``nodes``; hidden layers use ``neuron_types`` (one callable or a list),
    the output layer is linear (nn.py:34-87).  Layers are reachable as ``net[i]`` and as attributes ``matbias<i>``
    (the names the reference's parameter tree / checkpoints use)."""

    def __init__(self, nodes, n_layers=[], mean=0.0, stddev=1.0, variable_types=Variable,
                 neuron_types=sigmoid, collections=[graph_key.VARIABLES]):
        Parameterized.__init__(self)
        self.nodes = nodes
        n_dense = len(nodes) - 1
        self.neuron_types = _per_layer(neuron_types, n_dense - 1)
        self._matbias_list = []
        for i, (width_in, width_out, vtype) in enumerate(zip(nodes[:-1], nodes[1:], _per_layer(variable_types, n_dense))):
            layer = MatBias([width_in, width_out], n_layers=n_layers, mean=mean, stddev=stddev, variable=vtype,
                            collections=collections)
            self._matbias_list.append(layer)
            setattr(self, 'matbias%d' % i, layer)

    def __call__(self, x):
        """Must run in tf_mode.  A named activation (tf.sigmoid / tf.nn.relu / tf.tanh or its string) goes into the
        GEMM epilogue; any other callable is applied to the layer's linear output."""
        from . import trace as _trace
        if isinstance(x, _trace.Sym):
            return _trace.Sym('nn', self, x)
        *hidden, last = self._matbias_list
        y = x
        for layer, act in zip(hidden, self.neuron_types):
            fused = _act_name(act)
            y = layer(y, activation=fused) if fused is not None else act(layer(y))
        return last(y)

    def __getitem__(self, i):
        return self._matbias_list[i]
