"""Whole-step entry points of the C ABI, for drivers that do not need the autograd tape in between.

``LinearOperatorStep`` = BASELINE config 5 (full-covariance ``variationals.Normal([n])`` through a dense forward
operator with ``densities.gaussian``): forward, backward and the TF-1 Adam update are two C calls
(``hb_linop_elbo_local`` / ``hb_linop_elbo_update``, csrc/linop.cu) with ONE all-reduce in between when the operator
is row-sharded over ranks (SURVEY.md 8e).  Same numbers as the model written against the Python API
(tests/test_gpu_linop.py compares the two), without the n x n gradient ever being materialised.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib, parallel
from ._lib import ptr, stream, check


class LinearOperatorStep(object):
    """params packing: [ q_sqrt (n*n) | q_mu (n) | var (1) ], all in free space (var = softplus(free) + 1e-6).

    A_rows / y_rows: this rank's rows of the operator and of the data (device tensors, resident).
    m_total: rows of the whole operator (defaults to this rank's count = single GPU)."""

    def __init__(self, A_rows: torch.Tensor, y_rows: torch.Tensor, n_samples: int, m_total: int = None, seed: int = 0,
                 lr: float = 1e-3, beta1: float = 0.9, beta2: float = 0.999, epsilon: float = 1e-8, presplit: bool = None):
        self.lib = _lib.load()
        self.A = _lib.f32(A_rows).contiguous()
        self.y = _lib.f32(y_rows).contiguous().reshape(-1)
        M, n = self.A.shape
        if self.y.numel() != M:
            raise ValueError("y must have one entry per row of A")
        self.n, self.S = int(n), int(n_samples)
        if presplit is None:
            presplit = self.presplit_ok(M, n, self.S)
        self.cfg = _lib.LinopConfig(int(M), int(m_total if m_total is not None else M), self.n, self.S, int(seed), 0,
                                    1 if presplit else 0)
        dev = self.A.device
        self.count = int(self.lib.hb_linop_param_count(C.byref(self.cfg)))
        self.params = torch.zeros(self.count, device=dev)
        self.m = torch.zeros(self.count, device=dev)
        self.v = torch.zeros(self.count, device=dev)
        self.zbar_stats = torch.empty(self.S * self.n + 4, device=dev)
        self.out4 = torch.zeros(4, device=dev)
        self.ws_bytes = int(self.lib.hb_linop_workspace_bytes(C.byref(self.cfg)))
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.step_dev = torch.ones(1, dtype=torch.int32, device=dev)      # Adam's t (starts at 1)
        self.hyper = (float(lr), float(beta1), float(beta2), float(epsilon))
        self._stride = (self.S * self.n + 3) // 4 * 4
        self.prepare()

    @staticmethod
    def presplit_ok(M, n, S):
        """The pre-split engine (fp16 hi/lo shadow of the operator, + 4 bytes per element of A of workspace) streams A at
        HBM speed from 64 MB on; TMA needs 16-byte rows."""
        return M % 8 == 0 and n % 8 == 0 and S % 8 == 0 and S <= 256 and M * n >= (1 << 24)

    def prepare(self):
        """(Re)build the operator's shadow -- call again after changing A in place."""
        if self.cfg.presplit:
            check(self.lib.hb_linop_prepare(C.byref(self.cfg), ptr(self.A), ptr(self.ws), self.ws_bytes, stream()), "hb_linop_prepare")

    # ---- parameter access (free space) ----
    @property
    def q_sqrt(self):
        return self.params[:self.n * self.n].view(self.n, self.n)

    @property
    def q_mu(self):
        return self.params[self.n * self.n:self.n * self.n + self.n]

    @property
    def var_free(self):
        return self.params[self.n * self.n + self.n:]

    def set_params(self, q_mu, q_sqrt, var_free):
        dev = self.params.device
        self.q_sqrt.copy_(torch.as_tensor(np.asarray(q_sqrt, np.float32), device=dev))
        self.q_mu.copy_(torch.as_tensor(np.asarray(q_mu, np.float32), device=dev).reshape(-1))
        self.var_free.copy_(torch.as_tensor(np.asarray(var_free, np.float32), device=dev).reshape(-1))

    # ---- the step ----
    def local(self, eps=None, step_index=0):
        """Sampler, F = Z A^T, log-lik, partial Zbar = R A on this rank's rows -> self.zbar_stats."""
        self.cfg.offset = int(step_index) * self._stride
        check(self.lib.hb_linop_elbo_local(C.byref(self.cfg), ptr(self.A), ptr(self.y), ptr(self.params),
                                           ptr(eps) if eps is not None else None, ptr(self.zbar_stats), ptr(self.ws),
                                           self.ws_bytes, stream()), "hb_linop_elbo_local")
        return self.zbar_stats

    def update(self, grads: torch.Tensor = None, apply_adam: bool = True):
        """mu-bar, var-bar and the fused (gradient of q_sqrt + Adam) pass; returns out4 = {ELBO, loglik, kl, 0}."""
        lr, b1, b2, e = self.hyper
        check(self.lib.hb_linop_elbo_update(C.byref(self.cfg), ptr(self.params), ptr(self.zbar_stats), ptr(grads),
                                            ptr(self.m) if apply_adam else None, ptr(self.v) if apply_adam else None,
                                            lr, b1, b2, e, ptr(self.step_dev), 0, ptr(self.out4), ptr(self.ws),
                                            self.ws_bytes, stream()), "hb_linop_elbo_update")
        if apply_adam:
            check(self.lib.hb_increment_i32(ptr(self.step_dev), stream()), "hb_increment_i32")
        return self.out4

    def step(self, eps=None, step_index=0):
        """One ELBO + gradient + Adam step; the only collective is the all-reduce of [S*n + 4] floats."""
        self.local(eps, step_index)
        parallel.allreduce_sum_(self.zbar_stats)
        return self.update()

    def value_and_grads(self, eps=None):
        """ELBO and d ELBO / d params without touching the parameters (parity tests)."""
        g = torch.zeros(self.count, device=self.params.device)
        self.local(eps)
        parallel.allreduce_sum_(self.zbar_stats)
        out = self.update(grads=g, apply_adam=False)
        return out, g


# ------------------------------------------------------------------------------------------------------------------
# Binding of traced objectives (trace.py) to the whole-step entry points: what Optimizer.compile does with the tree
# ------------------------------------------------------------------------------------------------------------------
def _is_positive_scalar(v):
    from . import transforms
    from .param import Variable
    return isinstance(v, Variable) and v.is_parameter and isinstance(v.transform, transforms.Log1pe) and \
        int(np.prod(v._host.shape)) == 1 and abs(float(getattr(v.transform, '_lower', 1e-6)) - 1e-6) < 1e-12


def _leaf(node, op):
    from .trace import Sym
    return node.args[0] if isinstance(node, Sym) and node.op == op else None


def _variationals_of(model):
    from .variationals import Variational
    from .param import Parameterized
    out = []

    def walk(p):
        for c in p.sorted_variables:
            if isinstance(c, Variational):
                out.append(c)
            if isinstance(c, Parameterized):
                walk(c)
    walk(model)
    return out


def _split_elbo(tree, model):
    """tree = reduce_sum(gaussian(data, f, var)) - KL(model)  ->  (data variable, f, var variable) or None."""
    from .trace import Sym
    from .param import graph_key
    if not (isinstance(tree, Sym) and tree.op == 'sub' and len(tree.args) == 2):
        return None
    ll, kl = tree.args
    if not (isinstance(kl, Sym) and kl.op == 'KL' and kl.args[0] is model):
        return None
    if not (isinstance(ll, Sym) and ll.op == 'reduce_sum' and ll.kw.get('axis') is None):
        return None
    g = ll.args[0]
    if not (isinstance(g, Sym) and g.op == 'gaussian'):
        return None
    y, f, var = g.args
    yv, vv = _leaf(y, 'data'), _leaf(var, 'param')
    if yv is None or vv is None or not _is_positive_scalar(vv):
        return None
    return yv, f, vv, kl.args[1]


class _Float64Masters(object):
    """float_type = float64 (henbunrc:7) for a whole-step entry point whose parameters are packed at the start of the
    Optimizer's flat buffers: fp64 master copies of the parameters, their gradient and the Adam moments live in the binding,
    and the fp32 flat buffer mirrors them after every step (so .value, save() and the eager evaluation keep working).
    A binding whose entry point never writes a flat gradient sets _grad64 = False: no fp64 gradient is allocated or pushed."""
    _p64 = None
    _src64 = None
    _grad64 = True

    def _data64(self, dev):
        """fp64 device copies of X and Y, refreshed when new data is fed."""
        if self._src64 is None or self._src64[0] is not self.X.data or self._src64[1] is not self.Y.data:
            self._X64 = torch.as_tensor(np.ascontiguousarray(self.X.data, dtype=np.float64)).to(dev)
            self._Y64 = torch.as_tensor(np.ascontiguousarray(self.Y.data, dtype=np.float64)).to(dev).reshape(-1)
            self._src64 = (self.X.data, self.Y.data)
        return self._X64, self._Y64

    def _pull64(self, opt, npar, dev):
        """Masters before a step: created from the fp32 buffers at the first step, afterwards taking every entry of the
        fp32 mirror that was edited from outside since the last step."""
        if self._p64 is None:
            self._p64 = opt._flat[:npar].double()
            self._g64 = torch.zeros(npar, dtype=torch.float64, device=dev) if self._grad64 else None
            self._m64 = opt._m[:npar].double(); self._v64 = opt._v[:npar].double()
        else:
            # entries of the fp32 mirror that no longer equal the rounded master were edited from outside since the last
            # step (an assignment, restore(), another Optimizer over the same variables): the master takes them
            cur = opt._flat[:npar]
            self._p64 = torch.where(cur != self._p64.float(), cur.double(), self._p64)

    def _push64(self, opt, npar):
        opt._flat[:npar].copy_(self._p64)
        if self._grad64:
            opt._flat_grad[:npar].copy_(self._g64)


class GpElboBinding(_Float64Masters):
    """notebooks/GaussianProcess.ipynb:109-148 recognised in a traced objective:
        y_fit = matmul(kern.Cholesky(X), q) * sqrt(k_var);  ELBO = reduce_sum(gaussian(Y, y_fit, var)) - KL()
    with q = variationals.Gaussian([n, 1]) (diagonal or fullrank), kern = UnitRBF.  One call of hb_gp_elbo_step writes the
    ELBO and d ELBO / d (free parameters) straight into the Optimizer's flat gradient buffer, which is laid out in the
    entry point's packing [q_mu | q_sqrt | scale | lengthscales | k_var | var]."""

    def __init__(self, model, q, kern, k_var, var, X, Y):
        self.model, self.q, self.kern, self.k_var, self.var, self.X, self.Y = model, q, kern, k_var, var, X, Y
        g = object.__getattribute__
        self.var_order = [g(q, 'q_mu'), g(q, 'q_sqrt'), g(q, 'scale'), g(kern, 'lengthscales'), k_var, var]
        self.lib = _lib.load()
        self._ws = None
        self._key = None
        self._p64 = None
        self._src64 = None

    @staticmethod
    def match(tree, model):
        from .trace import Sym
        from .variationals import Gaussian, OffsetGaussian
        from .gp.kernels import UnitRBF
        from .param import Data, MinibatchData, graph_key, _is
        from . import transforms
        parts = _split_elbo(tree, model)
        if parts is None:
            return None
        Y, f, var, kl_coll = parts
        if kl_coll not in (None, graph_key.VARIABLES):
            return None
        if not (isinstance(f, Sym) and f.op == 'mul'):
            return None
        a, b = f.args
        if isinstance(a, Sym) and a.op == 'sqrt':
            a, b = b, a
        if not (isinstance(b, Sym) and b.op == 'sqrt'):
            return None
        k_var = _leaf(b.args[0], 'param')
        if k_var is None or not _is_positive_scalar(k_var):
            return None
        mm = a
        if not (isinstance(mm, Sym) and mm.op == 'matmul' and not mm.kw['ta'] and not mm.kw['tb']):
            return None
        ch, smp = mm.args
        if not (isinstance(ch, Sym) and ch.op == 'cholesky' and isinstance(smp, Sym) and smp.op == 'sample'):
            return None
        kern, Xs = ch.args
        X = _leaf(Xs, 'data')
        q = smp.args[0]
        if X is None or isinstance(X, MinibatchData) or isinstance(Y, MinibatchData):
            return None
        if type(kern) is not UnitRBF or type(q) is not Gaussian or smp.args[1] is not None:
            return None
        ell = object.__getattribute__(kern, 'lengthscales')
        from .param import Variable
        if not (isinstance(ell, Variable) and ell.is_parameter and isinstance(ell.transform, transforms.Log1pe)
                and abs(float(ell.transform._lower) - 1e-6) < 1e-12):
            return None
        if X.data.ndim != 2 or Y.data.shape != (X.data.shape[0], 1):
            return None
        n, D = X.data.shape
        if list(q._shape) != [n, 1] or q.n_layers or q.n_batch is not None or q.is_local or D > 32:
            return None
        if int(np.prod(ell._host.shape)) not in (1, D):
            return None
        scale = object.__getattribute__(q, 'scale')
        if not _is_positive_scalar(scale) or not isinstance(q.transform, transforms.Identity):
            return None
        if _variationals_of(model) != [q]:           # KL() must be exactly this variational's
            return None
        return GpElboBinding(model, q, kern, k_var, var, X, Y)

    def per_sample(self):
        return int(self.X.data.shape[0])

    SHARED_MIN_N = 4096      # below this a factorisation is a handful of leaves: every rank keeps its own

    # float_type = float64 (henbunrc:7): the whole step, Adam included, is hb_gp_elbo_step_f64 -- one persistent CTA for
    # notebook-sized models (csrc/gp_small.cu), the fp64 kernel chain at any larger n (csrc/f64.cu)
    @property
    def fused_adam(self):
        # in fp32 hb_gp_elbo_step already takes the one-CTA kernel for n <= 128 and the separate Adam launch is faster than Adam
        # inside it (168 vs 180 us)
        return self._f64() and parallel.world()[0] == 1

    @staticmethod
    def _f64():
        from ._settings import settings
        return str(settings.dtypes.float_type) == 'float64'

    def _cfg(self, opt, count, seed, offset):
        n, D = self.X.data.shape
        n_ell = int(np.prod(object.__getattribute__(self.kern, 'lengthscales')._host.shape))
        full = 1 if self.q.q_shape == 'fullrank' else 0
        return _lib.GpConfig(int(n), int(D), int(count), n_ell, full, float(opt._compiled_settings.numerics.jitter_level),
                             int(seed), int(offset)), (n, D, count, n_ell, full)

    def _eps(self, eps, count, n, device, dtype):
        if eps is None:
            return None
        e = torch.as_tensor(np.asarray(eps), dtype=dtype) if not isinstance(eps, torch.Tensor) else eps
        return e.to(device, dtype).reshape(count, n).contiguous()

    def step(self, opt, count, eps, seed, offset, world=None):
        """Forward + backward into opt._flat_grad; returns the ELBO (mean over the `count` samples) as a 0-d tensor.
        Called with `world` (fused_adam): the Adam update happens inside the same kernel."""
        from . import ops
        X, Y = self.X.tensor(), self.Y.tensor()
        n, D = X.shape
        cfg, key = self._cfg(opt, count, seed, offset)
        with_adam = world is not None
        f64 = with_adam and self._f64()
        # More than one rank: the ranks share ONE column-block-cyclic factorisation and reverse mode (csrc/linalg.cu:
        # potrf_flat / chol_rev_flat) instead of each factoring K itself; samples stay sharded (each rank its own Philox window).
        nranks = parallel.world()[0]
        shared = (not with_adam) and nranks > 1 and n >= self.SHARED_MIN_N and getattr(opt, '_shared_factorisation', True)
        key = key + (with_adam, f64, shared, _lib.OPTIONS.small_gp_kernel)     # the option picks the fp64 route and its workspace
        if self._key != key:
            self._env = parallel.block_cyclic_env(shard_samples=True) if shared else None
            if f64:
                self._wsb = int(self.lib.hb_gp_elbo_f64_workspace_bytes(C.byref(cfg)))
            elif with_adam:
                self._wsb = int(self.lib.hb_gp_small_workspace_bytes(C.byref(cfg), 0))
            elif shared:
                self._wsb = int(self.lib.hb_gp_elbo_dist_workspace_bytes(C.byref(cfg), C.byref(self._env)))
            else:
                self._wsb = int(self.lib.hb_gp_elbo_workspace_bytes(C.byref(cfg)))
            self._ws = torch.empty(self._wsb, dtype=torch.uint8, device=X.device)
            self._out4 = torch.zeros(4, device=X.device, dtype=torch.float64 if f64 else torch.float32)
            self._p64 = None
            self._key = key
        err = ops.err_flag(X.device)
        if not with_adam:
            e = self._eps(eps, count, n, X.device, torch.float32)
            if shared:
                check(self.lib.hb_gp_elbo_step_dist(C.byref(cfg), C.byref(self._env), ptr(X), ptr(Y), ptr(opt._flat), ptr(e),
                                                    ptr(opt._flat_grad), ptr(self._out4), ptr(self._ws), self._wsb, ptr(err), stream()),
                      "hb_gp_elbo_step_dist")
                torch.distributed.all_reduce(err, op=torch.distributed.ReduceOp.MAX)    # a failing block flags its owner only
                return self._out4[0]
            check(self.lib.hb_gp_elbo_step(C.byref(cfg), ptr(X), ptr(Y), ptr(opt._flat), ptr(e), ptr(opt._flat_grad), ptr(self._out4),
                                           ptr(self._ws), self._wsb, ptr(err), stream()), "hb_gp_elbo_step")
            return self._out4[0]
        o = opt.optimizer
        check(self.lib.hb_increment_i32(ptr(opt._step), stream()), "hb_increment_i32")
        adam = _lib.AdamConfig(float(o.learning_rate), float(o.beta1), float(o.beta2), float(o.epsilon), -1.0,
                               C.c_void_p(opt._step.data_ptr()), 0)
        npar = int(self.lib.hb_gp_param_count(C.byref(cfg)))
        if not f64:
            e = self._eps(eps, count, n, X.device, torch.float32)
            check(self.lib.hb_gp_small_step(C.byref(cfg), ptr(X), ptr(Y), ptr(opt._flat), ptr(e), ptr(opt._flat_grad), ptr(self._out4),
                                            ptr(opt._m), ptr(opt._v), C.byref(adam), ptr(self._ws), self._wsb, ptr(err), stream()),
                  "hb_gp_small_step")
            return self._out4[0]
        # float_type = float64 (henbunrc:7): fp64 master copies of parameters / moments (_Float64Masters)
        dev = X.device
        X64, Y64 = self._data64(dev)
        self._pull64(opt, npar, dev)
        e = self._eps(eps, count, n, X.device, torch.float64)
        check(self.lib.hb_gp_elbo_step_f64(C.byref(cfg), ptr(X64), ptr(Y64), ptr(self._p64), ptr(e), ptr(self._g64),
                                           ptr(self._out4), ptr(self._m64), ptr(self._v64), C.byref(adam), ptr(self._ws), self._wsb,
                                           ptr(err), stream()), "hb_gp_elbo_step_f64")
        self._push64(opt, npar)
        return self._out4[0]


def _operands(node, op):
    """(a, b) of a binary `op` node, or None."""
    from .trace import Sym
    if isinstance(node, Sym) and node.op == op and len(node.args) == 2:
        return node.args
    return None


def _commuted(node, op, first):
    """Operands of a commutative `op` node as (x, y) with first(x) true, trying both orders; None if neither fits."""
    ab = _operands(node, op)
    if ab is None:
        return None
    for x, y in (ab, ab[::-1]):
        if first(x):
            return x, y
    return None


def _gp_projection(node):
    """matmul(kern.Cholesky(X), q) with a UnitRBF kernel (Log1pe lengthscales) and a variationals.Gaussian q of shape [n, 1]
    -> (kern, X data variable, q), else None."""
    from .trace import Sym
    from .variationals import Gaussian
    from .gp.kernels import UnitRBF
    from .param import Variable
    from . import transforms
    if not (isinstance(node, Sym) and node.op == 'matmul' and not node.kw['ta'] and not node.kw['tb']):
        return None
    ch, smp = node.args
    if not (isinstance(ch, Sym) and ch.op == 'cholesky' and isinstance(smp, Sym) and smp.op == 'sample'):
        return None
    kern, Xs = ch.args
    X, q = _leaf(Xs, 'data'), smp.args[0]
    if X is None or type(kern) is not UnitRBF or type(q) is not Gaussian or smp.args[1] is not None:
        return None
    ell = object.__getattribute__(kern, 'lengthscales')
    if not (isinstance(ell, Variable) and ell.is_parameter and isinstance(ell.transform, transforms.Log1pe)
            and abs(float(ell.transform._lower) - 1e-6) < 1e-12):
        return None
    if q.n_layers or q.n_batch is not None or q.is_local or not isinstance(q.transform, transforms.Identity):
        return None
    if not _is_positive_scalar(object.__getattribute__(q, 'scale')):
        return None
    return kern, X, q


class MixtureGpElboBinding(_Float64Masters):
    """notebooks/Expert_GPR.ipynb:101-149 (BASELINE config 2) recognised in a traced objective under float_type = float64:
        f_s = matmul(kern_s.Cholesky(X), q_s);  f_l = matmul(kern_l.Cholesky(X), q_l)
        f_r = matmul(kern_r.Cholesky(X), q_r) * sqrt(k_var_r);  fraction = sigmoid(f_r)
        ELBO = reduce_sum(gaussian(Y, (fraction * f_s + (1 - fraction) * f_l) * k_var, var)) - KL()
    (either operand order of every mul and add) with three distinct UnitRBF kernels and three distinct
    variationals.Gaussian([n, 1]).  One call of hb_moe_gp_elbo_step_f64 (csrc/moe64.cu) runs the step, TF-1 Adam included,
    on fp64 master copies (_Float64Masters) packed as [q_s.q_mu | q_s.q_sqrt | q_s.scale | kern_s.lengthscales | the same for
    l and r | k_var | k_var_r | var].  `qs` lists the variationals in the order the objective samples them, the order of
    their Philox windows on the eager tape."""

    fused_adam = True

    def __init__(self, model, experts, k_var, k_var_r, var, X, Y, qs):
        self.model, self.experts, self.X, self.Y, self.qs = model, experts, X, Y, qs
        self.k_var, self.k_var_r, self.var = k_var, k_var_r, var
        g = object.__getattribute__
        order = []
        for kern, q in experts:
            order += [g(q, 'q_mu'), g(q, 'q_sqrt'), g(q, 'scale'), g(kern, 'lengthscales')]
        self.var_order = order + [k_var, k_var_r, var]
        self.lib = _lib.load()
        self._key = None

    @staticmethod
    def match(tree, model):
        from .trace import Sym, draws
        from .param import MinibatchData, graph_key
        from ._settings import settings
        if str(settings.dtypes.float_type) != 'float64' or parallel.world()[0] != 1:
            return None
        parts = _split_elbo(tree, model)
        if parts is None:
            return None
        Y, f, var, kl_coll = parts
        if kl_coll not in (None, graph_key.VARIABLES):
            return None
        param = lambda x: _leaf(x, 'param') is not None and _is_positive_scalar(_leaf(x, 'param'))
        sig = lambda x: isinstance(x, Sym) and x.op == 'sigmoid'
        one_minus = lambda x: (isinstance(x, Sym) and x.op == 'sub' and isinstance(x.args[0], (int, float))
                               and x.args[0] == 1 and sig(x.args[1]))
        # (mixture) * k_var
        mk = _commuted(f, 'mul', lambda x: not param(x))
        if mk is None or not param(mk[1]):
            return None
        mix, k_var = mk[0], _leaf(mk[1], 'param')
        # sigmoid(f_r) * f_s + (1 - sigmoid(f_r)) * f_l
        sl = _commuted(mix, 'add', lambda x: _commuted(x, 'mul', sig) is not None)
        if sl is None:
            return None
        gate_s, f_s = _commuted(sl[0], 'mul', sig)
        gl = _commuted(sl[1], 'mul', one_minus)
        if gl is None:
            return None
        gate_l, f_l = gl[0].args[1], gl[1]
        # f_r = matmul(kern_r.Cholesky(X), q_r) * sqrt(k_var_r), the same gate on both experts
        gates = []
        for gate in (gate_s, gate_l):
            fr = _commuted(gate.args[0], 'mul', lambda x: isinstance(x, Sym) and x.op == 'sqrt' and param(x.args[0]))
            if fr is None:
                return None
            gates.append((_leaf(fr[0].args[0], 'param'), _gp_projection(fr[1])))
        if gates[0][1] is None or gates[1][1] is None or gates[0][0] is not gates[1][0] or \
                any(a is not b for a, b in zip(gates[0][1], gates[1][1])):
            return None
        k_var_r, proj_r = gates[0]
        projs = [_gp_projection(f_s), _gp_projection(f_l), proj_r]
        if any(pr is None for pr in projs):
            return None
        kerns, Xs, qs = zip(*projs)
        X = Xs[0]
        if any(x is not X for x in Xs) or isinstance(X, MinibatchData) or isinstance(Y, MinibatchData):
            return None
        if len({id(k) for k in kerns}) != 3 or len({id(q) for q in qs}) != 3:
            return None
        if len({id(v) for v in (k_var, k_var_r, var)}) != 3:
            return None
        if X.data.ndim != 2 or Y.data.shape != (X.data.shape[0], 1):
            return None
        n, D = X.data.shape
        if D > 32 or any(list(q._shape) != [n, 1] for q in qs):
            return None
        if any(int(np.prod(object.__getattribute__(k, 'lengthscales')._host.shape)) not in (1, D) for k in kerns):
            return None
        found = _variationals_of(model)          # KL() must be exactly these three variationals'
        if len(found) != 3 or {id(q) for q in found} != {id(q) for q in qs}:
            return None
        order = [q for q in draws() if any(q is r for r in qs)]
        if len(order) != 3:
            return None
        return MixtureGpElboBinding(model, list(zip(kerns, qs)), k_var, k_var_r, var, X, Y, order)

    def per_sample(self):
        return int(self.X.data.shape[0])

    def step(self, opt, count, eps, seed, offsets, world=None):
        """One ELBO + gradient + Adam step.  eps / offsets: one per variational of `qs` (an injected [count, n] draw or None;
        the Philox stream position of a variational without one)."""
        from . import ops
        X = self.X.tensor()
        n, D = X.shape
        dev = X.device
        role = {id(q): i for i, (_, q) in enumerate(self.experts)}       # s, l, r
        e64, off = [None] * 3, [0] * 3
        for q, e, o in zip(self.qs, eps, offsets):
            i = role[id(q)]
            e64[i] = None if e is None else (torch.as_tensor(np.asarray(e), dtype=torch.float64) if not isinstance(e, torch.Tensor)
                                             else e).to(dev, torch.float64).reshape(count, n).contiguous()
            off[i] = int(o)
        n_ell = [int(np.prod(object.__getattribute__(k, 'lengthscales')._host.shape)) for k, _ in self.experts]
        full = [1 if q.q_shape == 'fullrank' else 0 for _, q in self.experts]
        cfg = _lib.MoeGpConfig(int(n), int(D), int(count), (C.c_int * 3)(*n_ell), (C.c_int * 3)(*full),
                               float(opt._compiled_settings.numerics.jitter_level), int(seed), (C.c_ulonglong * 3)(*off))
        key = (int(n), int(D), int(count), tuple(n_ell), tuple(full))
        if self._key != key:
            self._wsb = int(self.lib.hb_moe_gp_f64_workspace_bytes(C.byref(cfg)))
            self._ws = torch.empty(self._wsb, dtype=torch.uint8, device=dev)
            self._out4 = torch.zeros(4, dtype=torch.float64, device=dev)
            self._p64 = None
            self._key = key
        npar = int(self.lib.hb_moe_gp_param_count(C.byref(cfg)))
        X64, Y64 = self._data64(dev)
        self._pull64(opt, npar, dev)
        err = ops.err_flag(dev)
        check(self.lib.hb_increment_i32(ptr(opt._step), stream()), "hb_increment_i32")
        o = opt.optimizer
        adam = _lib.AdamConfig(float(o.learning_rate), float(o.beta1), float(o.beta2), float(o.epsilon), -1.0,
                               C.c_void_p(opt._step.data_ptr()), 0)
        check(self.lib.hb_moe_gp_elbo_step_f64(C.byref(cfg), ptr(X64), ptr(Y64), ptr(self._p64), ptr(e64[0]), ptr(e64[1]),
                                               ptr(e64[2]), ptr(self._g64), ptr(self._out4), ptr(self._m64), ptr(self._v64),
                                               C.byref(adam), ptr(self._ws), self._wsb, ptr(err), stream()),
              "hb_moe_gp_elbo_step_f64")
        self._push64(opt, npar)
        return self._out4[0]


class LinopElboBinding(_Float64Masters):
    """BASELINE config 5 recognised in a traced objective:
        f = matmul(q, A, transpose_b=True);  ELBO = reduce_sum(gaussian(y, f, var)) - KL()
    with q = variationals.Normal([n], 'fullrank').  The step runs hb_linop_elbo_local / _update on the Optimizer's flat
    buffers (packing [q_sqrt | q_mu | var]); the q_sqrt gradient is formed and consumed by Adam in one pass.
    Under float_type = float64 (henbunrc:7) with one process (`f64`, fixed when compile() binds), the step is the fp64 pair
    hb_linop_elbo_local_f64 / _update_f64 (csrc/linop64.cu) on fp64 master copies (_Float64Masters) and fp64 device copies
    of A and y."""

    _grad64 = False                     # neither route writes the flat gradient: no n x n fp64 gradient either

    def __init__(self, model, q, var, A, y, f64=False):
        self.model, self.q, self.var, self.A, self.y = model, q, var, A, y
        g = object.__getattribute__
        self.var_order = [g(q, 'q_sqrt'), g(q, 'q_mu'), var]
        self.fused_adam = True
        self.f64 = bool(f64)
        self._st = None
        self._key64 = None

    @staticmethod
    def match(tree, model):
        from .trace import Sym
        from .variationals import Normal
        from .param import MinibatchData, graph_key
        from . import transforms
        parts = _split_elbo(tree, model)
        if parts is None:
            return None
        y, f, var, kl_coll = parts
        if kl_coll not in (None, graph_key.VARIABLES):
            return None
        if not (isinstance(f, Sym) and f.op == 'matmul' and not f.kw['ta'] and f.kw['tb']):
            return None
        smp, As = f.args
        A = _leaf(As, 'data')
        if not (isinstance(smp, Sym) and smp.op == 'sample') or A is None:
            return None
        q = smp.args[0]
        if type(q) is not Normal or q.q_shape != 'fullrank' or q.n_layers or q.n_batch is not None or q.is_local:
            return None
        if isinstance(A, MinibatchData) or isinstance(y, MinibatchData) or A.data.ndim != 2:
            return None
        M, n = A.data.shape
        if list(q._shape) != [n] or int(np.prod(y.data.shape)) != M:
            return None
        if _variationals_of(model) != [q]:
            return None
        from ._settings import settings
        f64 = str(settings.dtypes.float_type) == 'float64' and parallel.world()[0] == 1
        return LinopElboBinding(model, q, var, A, y, f64=f64)

    def per_sample(self):
        return int(self.A.data.shape[1])

    def _operator64(self, dev):
        """fp64 device copies of A and y, built from the host arrays that are resident for the fp32 route and rebuilt
        when new data is fed."""
        src = (getattr(self.A, '_resident_src', None), getattr(self.y, '_resident_src', None))
        if self._src64 is None or self._src64[0] is not src[0] or self._src64[1] is not src[1]:
            self._A64 = self._y64 = None                 # release the old copy before the new one is made
            self._A64 = torch.as_tensor(np.ascontiguousarray(src[0])).to(dev).to(torch.float64)
            self._y64 = torch.as_tensor(np.ascontiguousarray(src[1])).to(dev).to(torch.float64).reshape(-1)
            self._src64 = src
        return self._A64, self._y64

    def _step64(self, opt, count, eps, seed, offset):
        A, _ = self.A.tensor(), self.y.tensor()          # keep the fp32 residents (and their _resident_src) current
        dev = A.device
        M, n = (int(s) for s in A.shape)
        A64, y64 = self._operator64(dev)
        lib = _lib.load()
        cfg = _lib.LinopConfig(M, M, n, int(count), int(seed), int(offset), 0)
        if self._key64 != (M, n, int(count)):
            self._wsb = int(lib.hb_linop_f64_workspace_bytes(C.byref(cfg)))
            self._ws = torch.empty(self._wsb, dtype=torch.uint8, device=dev)
            self._zbar64 = torch.empty(int(count) * n + 4, dtype=torch.float64, device=dev)
            self._out4 = torch.zeros(4, dtype=torch.float64, device=dev)
            self._key64 = (M, n, int(count))
        npar = int(lib.hb_linop_param_count(C.byref(cfg)))
        self._pull64(opt, npar, dev)
        e = None
        if eps is not None:
            e = torch.as_tensor(np.asarray(eps), dtype=torch.float64) if not isinstance(eps, torch.Tensor) else eps
            e = e.to(dev, torch.float64).reshape(count, n).contiguous()
        check(lib.hb_linop_elbo_local_f64(C.byref(cfg), ptr(A64), ptr(y64), ptr(self._p64), ptr(e), ptr(self._zbar64),
                                          ptr(self._ws), self._wsb, stream()), "hb_linop_elbo_local_f64")
        check(lib.hb_increment_i32(ptr(opt._step), stream()), "hb_increment_i32")
        o = opt.optimizer
        adam = _lib.AdamConfig(float(o.learning_rate), float(o.beta1), float(o.beta2), float(o.epsilon), -1.0,
                               C.c_void_p(opt._step.data_ptr()), 0)
        check(lib.hb_linop_elbo_update_f64(C.byref(cfg), ptr(self._p64), ptr(self._zbar64), None, ptr(self._m64), ptr(self._v64),
                                           C.byref(adam), ptr(self._out4), ptr(self._ws), self._wsb, stream()),
              "hb_linop_elbo_update_f64")
        self._push64(opt, npar)
        return self._out4[0]

    def step(self, opt, count, eps, seed, offset, world):
        if self.f64 and world == 1:
            return self._step64(opt, count, eps, seed, offset)
        A, y = self.A.tensor(), self.y.tensor()
        if self._st is None or self._st.S != count:
            st = LinearOperatorStep.__new__(LinearOperatorStep)
            st.lib = _lib.load()
            st.A, st.y = A, y.reshape(-1)
            M, n = A.shape
            st.n, st.S = int(n), int(count)
            st.cfg = _lib.LinopConfig(int(M), int(M), st.n, st.S, int(seed), 0,
                                      1 if LinearOperatorStep.presplit_ok(int(M), int(n), int(count)) else 0)
            st.count = int(st.lib.hb_linop_param_count(C.byref(st.cfg)))
            st.params, st.m, st.v = opt._flat[:st.count], opt._m[:st.count], opt._v[:st.count]
            st.zbar_stats = torch.empty(st.S * st.n + 4, device=A.device)
            st.out4 = torch.zeros(4, device=A.device)
            st.ws_bytes = int(st.lib.hb_linop_workspace_bytes(C.byref(st.cfg)))
            st.ws = torch.empty(st.ws_bytes, dtype=torch.uint8, device=A.device)
            st.step_dev = opt._step
            self._st = st
            self._prepared_src = None
        if self._prepared_src is not getattr(self.A, '_resident_src', None):     # a new operator was fed: its shadow is stale
            self._st.A = A
            self._st.prepare()
            self._prepared_src = getattr(self.A, '_resident_src', None)
        st = self._st
        st.A, st.y = A, y.reshape(-1)
        o = opt.optimizer
        st.hyper = (float(o.learning_rate), float(o.beta1), float(o.beta2), float(o.epsilon))
        st.cfg.seed = int(seed)
        st.cfg.offset = int(offset)
        e = None
        if eps is not None:
            e = torch.as_tensor(np.asarray(eps), dtype=torch.float32) if not isinstance(eps, torch.Tensor) else eps
            e = e.to(A.device, torch.float32).reshape(count, st.n).contiguous()
        check(st.lib.hb_linop_elbo_local(C.byref(st.cfg), ptr(st.A), ptr(st.y), ptr(st.params), ptr(e), ptr(st.zbar_stats),
                                         ptr(st.ws), st.ws_bytes, stream()), "hb_linop_elbo_local")
        # Adam's t: the Optimizer's counter holds the number of finished steps; the kernel wants the 1-based step
        check(st.lib.hb_increment_i32(ptr(opt._step), stream()), "hb_increment_i32")
        lr, b1, b2, ep = st.hyper
        check(st.lib.hb_linop_elbo_update(C.byref(st.cfg), ptr(st.params), ptr(st.zbar_stats), None, ptr(st.m), ptr(st.v),
                                          lr, b1, b2, ep, ptr(opt._step), 0, ptr(st.out4), ptr(st.ws), st.ws_bytes, stream()),
              "hb_linop_elbo_update")
        return st.out4[0]


class AmortisedElboBinding(_Float64Masters):
    """BASELINE config 4 recognised in a traced objective:
        self.q_local = self.enc(self.X);  x_rec = self.dec(self.q_local)
        ELBO = reduce_sum(gaussian(self.X, x_rec, self.var)) - self.KL(graph_key.LOCAL)
    with enc / dec = nn.NeuralNet, q_local = LOCAL variationals.Normal([latent]) (diagonal), X = MinibatchData.
    One call of hb_amortised_elbo_step (csrc/amortised.cu) on the gathered minibatch writes every gradient into the
    Optimizer's flat buffer, laid out as [enc w0 | enc b0 | ... | dec w0 | dec b0 | ... | var].
    Under float_type = float64 (henbunrc:7) with one process (`f64`, fixed when compile() binds), the step, TF-1 Adam
    included, is hb_amortised_elbo_step_f64 (csrc/amortised64.cu) on fp64 master copies (_Float64Masters) and on this
    step's rows gathered from a resident fp64 copy of the data."""

    _grad64 = False                     # the fp64 step keeps its gradient in its workspace

    def __init__(self, model, X, enc, dec, q, var, f64=False):
        self.model, self.X, self.enc, self.dec, self.q, self.var = model, X, enc, dec, q, var
        g = object.__getattribute__
        order = []
        for net in (enc, dec):
            for layer in net._matbias_list:
                order += [g(layer, 'w'), g(layer, 'b')]
        self.var_order = order + [var]
        self.f64 = bool(f64)
        self.fused_adam = self.f64
        self.lib = _lib.load()
        self._key = None

    @staticmethod
    def _net_ok(net):
        from .nn import NeuralNet, _act_name
        from .param import Variable
        from . import transforms
        if type(net) is not NeuralNet or len(net._matbias_list) > _lib.HB_MAX_LAYERS:
            return False
        g = object.__getattribute__
        for layer in net._matbias_list:
            for v in (g(layer, 'w'), g(layer, 'b')):
                if type(v) is not Variable or not v.is_parameter or v.n_layers or not isinstance(v.transform, transforms.Identity):
                    return False
        return all(_act_name(a) in ('none', 'sigmoid', 'relu', 'tanh') for a in net.neuron_types)

    @staticmethod
    def match(tree, model):
        from .trace import Sym
        from .variationals import Normal
        from .param import MinibatchData, graph_key
        parts = _split_elbo_mb(tree, model)
        if parts is None:
            return None
        X, f, var, kl_coll = parts
        if kl_coll != graph_key.LOCAL or not isinstance(X, MinibatchData) or X.data.ndim != 2:
            return None
        if not (isinstance(f, Sym) and f.op == 'nn'):
            return None
        dec, smp = f.args
        if not (isinstance(smp, Sym) and smp.op == 'sample'):
            return None
        q, fed = smp.args
        if not (isinstance(fed, Sym) and fed.op == 'nn'):
            return None
        enc, xin = fed.args
        if _leaf(xin, 'mbdata') is not X:
            return None
        if type(q) is not Normal or q.q_shape != 'diagonal' or not q.is_local or q.n_layers or len(q._shape) != 1:
            return None
        if not (AmortisedElboBinding._net_ok(enc) and AmortisedElboBinding._net_ok(dec)):
            return None
        lat, Dx = q._shape[0], X.data.shape[1]
        if enc.nodes[0] != Dx or enc.nodes[-1] != 2 * lat or dec.nodes[0] != lat or dec.nodes[-1] != Dx:
            return None
        if _variationals_of(model) != [q]:
            return None
        from ._settings import settings
        f64 = str(settings.dtypes.float_type) == 'float64' and parallel.world()[0] == 1
        return AmortisedElboBinding(model, X, enc, dec, q, var, f64=f64)

    def per_sample(self):
        return int(self.X.tensor().shape[0]) * int(self.q._shape[0])

    def _config(self, B, count, f64):
        from .nn import _act_name
        key = (B, count, f64)
        if self._key != key:
            cfg = _lib.AmortisedConfig()
            cfg.B, cfg.S, cfg.latent = B, int(count), int(self.q._shape[0])
            for name, net in (('enc', self.enc), ('dec', self.dec)):
                setattr(cfg, 'n_' + name, len(net._matbias_list))
                nodes = getattr(cfg, name + '_nodes'); acts = getattr(cfg, name + '_act')
                for i, w in enumerate(net.nodes):
                    nodes[i] = int(w)
                for i, a in enumerate(net.neuron_types):
                    acts[i] = _lib.ACT[_act_name(a)]
            self._cfg = cfg
            size = self.lib.hb_amortised_f64_workspace_bytes if f64 else self.lib.hb_amortised_workspace_bytes
            self._wsb = int(size(C.byref(cfg)))
            if self._wsb == 0:
                raise _lib.HenbunB200Error("hb_amortised_elbo_step rejected the network shapes")
            dev = self.X.tensor().device
            self._ws = None                              # release the old workspace before the new one is made
            self._ws = torch.empty(self._wsb, dtype=torch.uint8, device=dev)
            self._out4 = torch.zeros(4, device=dev, dtype=torch.float64 if f64 else torch.float32)
            self._key = key
        return self._cfg

    def _eps(self, eps, count, B, dev, dtype):
        if eps is None:
            return None
        e = torch.as_tensor(np.asarray(eps), dtype=dtype) if not isinstance(eps, torch.Tensor) else eps
        return e.to(dev, dtype).reshape(count, B, int(self.q._shape[0])).contiguous()

    def _minibatch64(self, dev):
        """This step's rows (the index the fp32 route gathered) from an fp64 device copy of X.data, rebuilt when the data
        is replaced."""
        src = self.X.data
        if self._src64 is not src:
            self._X64 = None                             # release the old copy before the new one is made
            self._X64 = torch.as_tensor(np.ascontiguousarray(src, dtype=np.float64)).to(dev)
            self._src64 = src
        idx = self.X.last_index.to(device=dev, dtype=torch.int64).contiguous()
        row = int(self._X64.shape[1])
        out = torch.empty((idx.numel(), row), dtype=torch.float64, device=dev)
        check(self.lib.hb_gather_rows_f64(ptr(out), ptr(self._X64), ptr(idx), idx.numel(), row, stream()), "hb_gather_rows_f64")
        return out

    def _step64(self, opt, count, eps, seed, offset):
        dev = self.X.tensor().device
        X64 = self._minibatch64(dev)
        B = int(X64.shape[0])
        cfg = self._config(B, int(count), True)
        cfg.seed, cfg.offset = int(seed), int(offset)
        npar = int(self.lib.hb_amortised_param_count(C.byref(cfg)))
        self._pull64(opt, npar, dev)
        check(self.lib.hb_increment_i32(ptr(opt._step), stream()), "hb_increment_i32")
        o = opt.optimizer
        adam = _lib.AdamConfig(float(o.learning_rate), float(o.beta1), float(o.beta2), float(o.epsilon), -1.0,
                               C.c_void_p(opt._step.data_ptr()), 0)
        e = self._eps(eps, count, B, dev, torch.float64)
        check(self.lib.hb_amortised_elbo_step_f64(C.byref(cfg), ptr(X64), ptr(self._p64), ptr(e), None, ptr(self._out4),
                                                  ptr(self._m64), ptr(self._v64), C.byref(adam), ptr(self._ws), self._wsb,
                                                  stream()), "hb_amortised_elbo_step_f64")
        self._push64(opt, npar)
        return self._out4[0]

    def step(self, opt, count, eps, seed, offset, world=None):
        """Called with `world` (fused_adam: the float64 route) the step applies Adam itself; without it the fp32 step
        writes the gradient into opt._flat_grad and the caller applies Adam."""
        if world is not None:
            return self._step64(opt, count, eps, seed, offset)
        X = self.X.tensor()
        B = int(X.shape[0])
        cfg = self._config(B, int(count), False)
        cfg.seed, cfg.offset = int(seed), int(offset)
        e = self._eps(eps, count, B, X.device, torch.float32)
        check(self.lib.hb_amortised_elbo_step(C.byref(cfg), ptr(X), ptr(opt._flat), ptr(e), ptr(opt._flat_grad), ptr(self._out4),
                                              ptr(self._ws), self._wsb, stream()), "hb_amortised_elbo_step")
        return self._out4[0]


def _split_elbo_mb(tree, model):
    """As _split_elbo with a MinibatchData observation."""
    from .trace import Sym
    if not (isinstance(tree, Sym) and tree.op == 'sub' and len(tree.args) == 2):
        return None
    ll, kl = tree.args
    if not (isinstance(kl, Sym) and kl.op == 'KL' and kl.args[0] is model):
        return None
    if not (isinstance(ll, Sym) and ll.op == 'reduce_sum' and ll.kw.get('axis') is None):
        return None
    g = ll.args[0]
    if not (isinstance(g, Sym) and g.op == 'gaussian'):
        return None
    y, f, var = g.args
    yv, vv = _leaf(y, 'mbdata'), _leaf(var, 'param')
    if yv is None or vv is None or not _is_positive_scalar(vv):
        return None
    return yv, f, vv, kl.args[1]


BINDINGS = (GpElboBinding, MixtureGpElboBinding, LinopElboBinding, AmortisedElboBinding)


def bind(tree, model):
    """First whole-step entry point whose graph equals the traced objective, or None."""
    for cls in BINDINGS:
        try:
            b = cls.match(tree, model)
        except Exception:       # a shape the matcher did not foresee: keep the eager path
            b = None
        if b is not None:
            return b
    return None
