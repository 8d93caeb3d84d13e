"""Parameter tree and ``tf_mode``: mirror of Henbun/param.py (graph_key :29-47, Parentable :49-95,
Variable :97-314, Parameterized :316-603, ParamList :605-674, Data :676-714, MinibatchData :716-739).

Storage differs from the reference (which keeps ``tf.Variable``s in a ``tf.Session``): every global
parameter is a fp32 leaf tensor in HBM holding the *free-space* value; in ``tf_mode`` attributes
resolve to device tensors exactly as the reference's resolve to TF tensors.  Host copies exist only
for initialisation, assignment (``m.p = ndarray``) and ``.value``.
"""
from __future__ import annotations

from contextlib import contextmanager
from functools import reduce

import numpy as np
import torch

from . import transforms
from . import trace as _trace
from ._lib import HenbunB200Error

np_float_type = np.float32


class _GraphKey(object):
    """VARIABLES / LOCAL / DATA flags (Henbun/param.py:29-47)."""

    def __init__(self):
        self.VARIABLES = 'variables'      # the value of tf.GraphKeys.GLOBAL_VARIABLES
        self.LOCAL = 'LOCAL'
        self.DATA = 'DATA'

    @property
    def not_parameters(self):
        return [self.LOCAL, self.DATA]


graph_key = _GraphKey()


def _is(collections, key):
    return isinstance(collections, str) and collections == key


def _in_collection(collection, collections):
    """`collection in self.collections` of the reference (list membership, or substring for str)."""
    if collection is None:
        return True
    return collection in collections


def _device():
    if not torch.cuda.is_available():
        raise HenbunB200Error("henbun_b200 evaluates on a CUDA device only (no CPU fallback); no GPU is visible")
    return torch.device('cuda', torch.cuda.current_device())


def _truncated_normal(shape, mean, stddev, rng=None):
    """tf.truncated_normal: N(mean, stddev) re-drawn until within 2 stddev (param.py:206-208)."""
    rng = rng or np.random
    out = rng.standard_normal(size=shape)
    bad = np.abs(out) > 2.0
    while np.any(bad):
        out[bad] = rng.standard_normal(size=int(bad.sum()))
        bad = np.abs(out) > 2.0
    return (mean + stddev * out).astype(np_float_type)


class Parentable(object):
    """Tree node that knows its parent and can derive its own name (Henbun/param.py:49-95)."""

    def __init__(self):
        self._parent = None

    @property
    def highest_parent(self):
        if self._parent is None:
            return self
        return self._parent.highest_parent

    @property
    def name(self):
        if self._parent is None:
            return 'unnamed'
        if isinstance(self._parent, ParamList):
            return 'item%i' % self._parent._list.index(self)
        matches = [key for key, value in self._parent.__dict__.items() if value is self]
        if len(matches) == 0:
            raise ValueError("mis-specified parent. This Param's _parent does not contain a reference to it.")
        if len(matches) > 1:
            raise ValueError("This Param appears to be doubly referenced by a parent")
        return matches[0]

    @property
    def long_name(self):
        if self._parent is None:
            return self.name
        return self._parent.long_name + '.' + self.name


class Variable(Parentable):
    """Global parameter, LOCAL parameter or DATA holder (Henbun/param.py:97-314).
    Storage shape is n_layers + [n_batch]? + shape; values live in free space and ``tensor()``
    applies the transform (param.py:211-218)."""

    def __init__(self, shape, n_layers=[], n_batch=None, mean=0.0, stddev=1.0,
                 transform=transforms.Identity(), collections=[graph_key.VARIABLES]):
        Parentable.__init__(self)
        if isinstance(shape, (int, np.integer)):
            shape = [int(shape)]
        self.transform = transform
        self.collections = collections
        self.n_batch = n_batch
        self.shape = list(shape)
        self.n_layers = list(n_layers)
        self._assigned = True
        self._tensor = None
        self._host = None        # host master copy of the free-space value (parameters only)
        self._pending = None
        if not self.is_parameter:
            return
        if self.n_batch is None:
            _shape = list(n_layers) + list(shape)
        else:
            _shape = list(n_layers) + [self.n_batch] + list(shape)
        self._host = _truncated_normal(tuple(int(s) for s in _shape), mean, stddev)
        self._pending = self._host

    # --- collection helpers ---
    @property
    def is_parameter(self):
        return not (_is(self.collections, graph_key.LOCAL) or _is(self.collections, graph_key.DATA))

    @property
    def is_local(self):
        return _is(self.collections, graph_key.LOCAL)

    # --- device storage ---
    def _ensure_device(self):
        if self.is_parameter and self._tensor is None:
            self._tensor = torch.from_numpy(np.ascontiguousarray(self._host)).to(_device()).requires_grad_(True)
        return self._tensor

    def _rebind(self, storage_view, grad_view):
        """Make this parameter alias a slice of the optimizer's flat buffers (one Adam launch, one
        all-reduce per step).  Current values are preserved."""
        cur = self._ensure_device().detach()
        with torch.no_grad():
            storage_view.copy_(cur.reshape(storage_view.shape))
        t = storage_view.view(cur.shape).detach().requires_grad_(True)
        t.grad = grad_view.view(cur.shape)
        self._tensor = t

    def tensor(self):
        """In tf_mode this object is seen as transform(free value) (param.py:211-218)."""
        if _trace.active():
            return _trace.Sym('param' if self.is_parameter else 'local', self)
        if not self.is_parameter:
            return self._tensor
        return self.transform.tf_forward(self._ensure_device())

    def get_tf_variables(self, collection=None):
        if _in_collection(collection, self.collections):
            if self.is_parameter:
                self._ensure_device()
            return [self._tensor]
        return []

    def get_variables(self, collection=None):
        if _in_collection(collection, self.collections):
            return [self]
        return []

    def assign(self, value):
        """Store transform.backward(value); applied at the next initialize() (param.py:241-248)."""
        if self.is_parameter:
            v = np.asarray(self.transform.backward(np.asarray(value, dtype=np.float64)), dtype=np_float_type)
            self._pending = np.broadcast_to(v, self._host.shape).copy() if v.shape != self._host.shape else v
            self._assigned = True

    def _apply_pending(self):
        if self.is_parameter and self._assigned and self._pending is not None:
            self._host = np.ascontiguousarray(self._pending, dtype=np_float_type)
            if self._tensor is not None:
                with torch.no_grad():
                    self._tensor.copy_(torch.from_numpy(self._host).reshape(self._tensor.shape))
            self._pending = None

    @property
    def initialize_ops(self):
        if self.is_parameter and self._assigned:
            return [self._apply_pending]
        return []

    def finalize(self):
        self._assigned = False

    def _free_numpy(self):
        if self._tensor is not None and self.is_parameter:
            return self._tensor.detach().cpu().numpy()
        return self._host

    @property
    def value(self):
        """Current (constrained-space) value (param.py:268-279)."""
        assert hasattr(self.highest_parent, '_session')
        if self.is_parameter:
            if self._assigned:
                self._apply_pending()
                self.finalize()
            return self.transform.forward(self._free_numpy())
        t = self.tensor()
        return None if t is None else t.detach().cpu().numpy()

    @property
    def feed_size(self):
        if self.is_local:
            return int(reduce(np.multiply, self.shape, 1))
        return 0

    def feed(self, x):
        """LOCAL: take x [*n_layers, N, prod(shape)] and view it as n_layers+[N]+shape (param.py:291-304).
        The view is strided -- no slice copy is made."""
        if self.is_local:
            if self.n_batch is not None and x.shape[-2] is not None:
                assert x.shape[-2] == self.n_batch
            if len(self.shape) == 1:
                self._tensor = x
            else:
                self._tensor = x.reshape(list(self.n_layers) + [x.shape[-2]] + self.shape)

    def get_feed_dict(self, minibatch_index):
        if _is(self.collections, graph_key.DATA):
            raise NotImplementedError
        return {}


class Parameterized(Parentable):
    """Holds Variables / Parameterized children; implements tf_mode (Henbun/param.py:316-603)."""

    def __init__(self):
        Parentable.__init__(self)
        self._tf_mode = False
        self.scoped_keys = []
        self._saver = None

    def __getattribute__(self, key):
        o = object.__getattribute__(self, key)
        try:
            if not object.__getattribute__(self, '_tf_mode'):
                return o
        except AttributeError:
            return o
        if key == '_parent':
            return o
        if isinstance(o, (Parameterized, Variable)) and hasattr(o, 'tensor'):
            return o.tensor()
        return o

    def __setattr__(self, key, value):
        if key in self.__dict__.keys():
            p = object.__getattribute__(self, key)
            try:
                if object.__getattribute__(self, '_tf_mode'):
                    if isinstance(p, (Variable, Parameterized)):
                        p.feed(value)
                        return
            except (KeyError, AttributeError):
                pass
            if isinstance(p, Variable):
                if isinstance(value, (float, int)):
                    value = np.array([value], dtype=np_float_type)
                if isinstance(value, np.ndarray):
                    p.assign(value)
                    return
            if isinstance(p, (Variable, Parameterized)) and isinstance(value, (Variable, Parameterized)):
                p._parent = None
                if hasattr(self, '_needs_recompile'):
                    self.highest_parent._needs_recompile = True
        object.__setattr__(self, key, value)
        if isinstance(value, Parentable) and key != '_parent':
            value._parent = self

    @contextmanager
    def tf_mode(self):
        self._begin_tf_mode()
        try:
            yield
        finally:
            self._end_tf_mode()

    def _begin_tf_mode(self):
        [child._begin_tf_mode() for child in self.sorted_variables if isinstance(child, Parameterized)]
        self._tf_mode = True

    def _end_tf_mode(self):
        [child._end_tf_mode() for child in self.sorted_variables if isinstance(child, Parameterized)]
        self._tf_mode = False

    def _new_run(self, ctx):
        """Start of one objective evaluation (one ``session.run`` of the reference): variationals draw
        fresh samples.  ctx carries n_samples / seed / injected eps."""
        for child in self.sorted_variables:
            if isinstance(child, Parameterized):
                child._new_run(ctx)

    @property
    def sorted_variables(self):
        variables = [child for key, child in object.__getattribute__(self, '__dict__').items()
                     if isinstance(child, (Variable, Parameterized)) and key != '_parent']
        return sorted(variables, key=lambda x: x.name)

    def get_tf_variables(self, collection=None):
        params = []
        for p in self.sorted_variables:
            params += p.get_tf_variables(collection)
        return params

    def get_variables(self, collection=None):
        params = []
        for p in self.sorted_variables:
            params += p.get_variables(collection)
        return params

    @property
    def initialize_ops(self):
        params = []
        for p in self.sorted_variables:
            params += p.initialize_ops
        return params

    def finalize(self):
        for p in self.sorted_variables:
            p.finalize()

    @property
    def feed_size(self):
        return int(np.sum([p.feed_size for p in self.get_variables(graph_key.LOCAL)], dtype=int))

    def feed(self, x):
        """Split the last axis of x over the LOCAL children in name-sorted order (param.py:516-537)."""
        if _trace.active():
            object.__setattr__(self, '_sym_feed', x)
            return
        local = self.get_variables(graph_key.LOCAL)
        if len(local) == 0:
            return
        n_layers = local[0].n_layers
        for p in local:
            assert len(p.n_layers) == len(n_layers)
            assert all([n == n0 for n, n0 in zip(p.n_layers, n_layers)]), \
                'n_layers of all the LOCAL variables should be same for using this method.'
        begin = 0
        for p in self.sorted_variables:
            size = p.feed_size
            p.feed(x[..., begin:begin + size])
            begin += size

    def get_feed_dict(self, minibatch_index=None):
        feed_dict = {}
        for p in self.sorted_variables:
            feed_dict.update(p.get_feed_dict(minibatch_index))
        return feed_dict

    def KL(self, collection=None):
        """Sum of the children's KL (param.py:549-560)."""
        if _trace.active():
            return _trace.Sym('KL', self, collection)
        KL_list = [p.KL(collection) for p in self.sorted_variables if hasattr(p, 'KL')]
        KL_list = [k for k in KL_list if isinstance(k, torch.Tensor)]      # drop the numpy zeros of KL-less children
        if len(KL_list) == 0:
            return np.zeros([], dtype=np_float_type)
        return reduce(lambda a, b: a + b, KL_list)

    # --- checkpointing: {long_name: free-space array} (param.py:562-603; Adam slots are not saved there either) ---
    def _var_dict(self):
        d = {v.long_name: v for v in self.get_variables() if v.is_parameter}
        if len(d) == 0:
            raise ValueError('This class does not contain any global variables.')
        return d

    def save(self, save_path=None, **_ignored):
        if save_path is None:
            save_path = self.name + '.ckpt'
        self.highest_parent.initialize()
        arrays = {k: v._free_numpy() for k, v in self._var_dict().items()}
        with open(save_path, 'wb') as f:
            np.savez(f, **arrays)
        return save_path

    def restore(self, save_path=None):
        if save_path is None:
            save_path = self.name + '.ckpt'
        with np.load(save_path) as data:
            for k, v in self._var_dict().items():
                v._pending = data[k].astype(np_float_type)
                v._assigned = True
                v._apply_pending()
        [v.finalize() for v in self.get_variables()]


class ParamList(Parameterized):
    """A list of parameters visible to the tree (Henbun/param.py:605-674)."""

    def __init__(self, list_of_params=[]):
        Parameterized.__init__(self)
        for item in list_of_params:
            assert isinstance(item, (Variable, Parameterized))
            item._parent = self
        self._list = list_of_params

    @property
    def sorted_variables(self):
        return object.__getattribute__(self, '_list')

    def __getitem__(self, key):
        o = self.sorted_variables[key]
        if isinstance(o, Variable) and object.__getattribute__(self, '_tf_mode'):
            return o.tensor()
        return o

    def append(self, item):
        assert isinstance(item, (Variable, Parameterized)), "this object is for containing parameters"
        item._parent = self
        self.sorted_variables.append(item)

    def __len__(self):
        return len(self.sorted_variables)

    def __setitem__(self, key, value):
        p = self.sorted_variables[key]
        if isinstance(value, np.ndarray):
            p._pending = value.astype(np_float_type); p._assigned = True
            return
        elif isinstance(value, (float, int)):
            p._pending = np.array([value], dtype=np_float_type); p._assigned = True
            return
        raise TypeError


class Data(Variable):
    """Data fed into the objective on every run (Henbun/param.py:676-714).  The reference pushes the whole array through
    feed_dict on every session.run (param.py:701-705); here the array stays RESIDENT in HBM and is copied again (from
    pinned host memory) only when a different array object is fed or assigned -- config 5 would otherwise move its
    4.3 GB operator over PCIe every step (92 of 115 ms).  In-place edits of the same numpy array are therefore not
    picked up: assign the array again (``model.A = arr``) or call ``invalidate()``."""

    def __init__(self, data):
        Variable.__init__(self, data.shape, n_layers=[], n_batch=None, collections=graph_key.DATA)
        self._dtype = self._get_type(data)
        self.data = data
        self._pinned = None
        self._fed_version = -1

    def _get_type(self, array):
        if any([array.dtype == np.dtype(t) for t in [np.float32, np.float64]]):
            return torch.float32
        elif any([array.dtype == np.dtype(t) for t in [np.int16, np.int32, np.int64]]):
            return torch.int32
        raise NotImplementedError("unknown dtype")

    def invalidate(self):
        """Force the next feed to copy the host array again."""
        self._resident_src = None

    def _upload(self, array):
        if self._tensor is not None and getattr(self, '_resident_src', None) is array:
            return                                   # already resident
        self._resident_src = array
        t = torch.as_tensor(np.ascontiguousarray(array)).to(self._dtype)
        if self._pinned is None or self._pinned.shape != t.shape:
            self._pinned = torch.empty(t.shape, dtype=self._dtype).pin_memory()
            self._h2d_done = None
        if self._tensor is None or self._tensor.shape != t.shape:
            self._tensor = torch.empty(t.shape, dtype=self._dtype, device=_device())
        if getattr(self, '_h2d_done', None) is not None:
            self._h2d_done.synchronize()      # the previous async copy out of the staging buffer must have drained
        self._pinned.copy_(t)
        self._tensor.copy_(self._pinned, non_blocking=True)
        self._h2d_done = torch.cuda.Event()
        self._h2d_done.record()

    def get_feed_dict(self, minibatch_index=None):
        return {self: self.data}

    def tensor(self):
        if _trace.active():
            return _trace.Sym('data', self)
        if self._tensor is None or getattr(self, '_resident_src', None) is None:
            self._upload(self.data)
        return self._tensor

    def assign(self, value):
        if not np.all(value.shape == self.data.shape):
            raise ValueError('The shape of data must be the same.')
        self.data = value
        self._resident_src = None          # next feed copies the new array (device buffer and staging are kept)

    @property
    def value(self):
        return self.data


class MinibatchData(Data):
    """Minibatched data (Henbun/param.py:716-739).  The whole array stays resident in HBM; a feed
    gathers the indexed rows on the device (K15) instead of a host fancy-index + H2D copy."""

    def __init__(self, data):
        Variable.__init__(self, data.shape[1:], n_layers=[], n_batch=None, collections=graph_key.DATA)
        self._dtype = self._get_type(data)
        self.data = data
        self._resident = None
        self._pinned = None

    @property
    def data_size(self):
        return self.data.shape[0]

    def get_feed_dict(self, minibatch_index):
        if minibatch_index is None:
            return {}
        return {self: minibatch_index}

    def _gather(self, index):
        from . import ops
        if self._resident is None:
            self._resident = torch.as_tensor(np.ascontiguousarray(self.data)).to(self._dtype).to(_device())
        idx = index if isinstance(index, torch.Tensor) else torch.as_tensor(np.asarray(index, dtype=np.int64))
        self.last_index = idx               # the rows of this feed, for a binding that gathers its own copy of the data
        if self._dtype == torch.float32:
            self._tensor = ops.gather_rows(self._resident, idx.to(self._resident.device))
        else:
            self._tensor = self._resident[idx.to(self._resident.device)]

    def tensor(self):
        if _trace.active():
            return _trace.Sym('mbdata', self)
        return self._tensor

    def assign(self, value):
        self.data = value
        self._resident = None
        self._tensor = None
