"""Host-side contract of the float64 mixture-of-experts GP entry point (csrc/moe64.cu) and of its binding to traced
objectives (fused.MixtureGpElboBinding): parameter counts, workspace sizes, the argument checks that return before anything
reaches a device, and which graphs the binder accepts.  No kernel is launched, so these run without a GPU."""
import ctypes as C

import numpy as np
import pytest

HB_OK, HB_ERR_ARG, HB_ERR_WORKSPACE = 0, 1, 3
FAKE = C.c_void_p(4096)          # a non-NULL device address; every call below is rejected before it is dereferenced


@pytest.fixture(scope="module")
def lib():
    from henbun_b200 import _lib
    return _lib.load()


def cfg(n, D=1, S=4, n_ell=(1, 1, 1), full=(1, 1, 0), offset=(0, 0, 0)):
    from henbun_b200 import _lib
    return _lib.MoeGpConfig(n, D, S, (C.c_int * 3)(*n_ell), (C.c_int * 3)(*full), 3e-4, 0, (C.c_ulonglong * 3)(*offset))


SHAPES = [(q, a) for q in ((0, 0, 0), (1, 1, 0), (1, 1, 1), (0, 1, 0)) for a in ((1, 1, 1), (3, 3, 3), (1, 3, 1))]


@pytest.mark.parametrize("full,n_ell", SHAPES)
def test_param_count_and_workspace(lib, full, n_ell):
    n, D, S = 50, 3, 4
    c = cfg(n, D, S, n_ell, full)
    want = sum(n + (n * n if f else n) + 1 + k for f, k in zip(full, n_ell)) + 3
    assert lib.hb_moe_gp_param_count(C.byref(c)) == want
    # three GPs, each with its Gram / factor and K-bar matrices, five [S, n] buffers and its own split-K partial tiles
    assert lib.hb_moe_gp_f64_workspace_bytes(C.byref(c)) >= 3 * (2 * n * n * 8 + 5 * S * n * 8 + 32 * 128 * 128 * 8)


def test_sizes_of_invalid_configs_are_zero(lib):
    for c in (cfg(0), cfg(10, D=33, n_ell=(1, 1, 1)), cfg(10, D=3, n_ell=(2, 1, 1)), cfg(10, full=(2, 0, 0))):
        assert lib.hb_moe_gp_param_count(C.byref(c)) == 0
        assert lib.hb_moe_gp_f64_workspace_bytes(C.byref(c)) == 0


def step(lib, c, X=FAKE, Y=FAKE, params=FAKE, eps=(FAKE, FAKE, FAKE), grads=FAKE, out4=FAKE, m=None, v=None, adam=None,
         ws=FAKE, wsb=None):
    if wsb is None:
        wsb = lib.hb_moe_gp_f64_workspace_bytes(C.byref(c)) or 1 << 40
    return lib.hb_moe_gp_elbo_step_f64(C.byref(c), X, Y, params, eps[0], eps[1], eps[2], grads, out4, m, v, adam, ws, wsb,
                                       None, None)


def test_step_rejects_bad_arguments(lib):
    from henbun_b200 import _lib
    c = cfg(20)
    assert lib.hb_moe_gp_elbo_step_f64(None, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None, None, None, FAKE, 1,
                                       None, None) == HB_ERR_ARG
    for k in ("X", "Y", "params", "grads", "out4"):
        assert step(lib, c, **{k: None}) == HB_ERR_ARG, k
    assert step(lib, cfg(0), wsb=1 << 40) == HB_ERR_ARG
    assert step(lib, cfg(-3), wsb=1 << 40) == HB_ERR_ARG
    assert step(lib, cfg(20, S=0), wsb=1 << 40) == HB_ERR_ARG
    assert step(lib, cfg(20, D=33, n_ell=(1, 1, 1)), wsb=1 << 40) == HB_ERR_ARG
    assert step(lib, cfg(20, D=3, n_ell=(3, 2, 3)), wsb=1 << 40) == HB_ERR_ARG
    assert step(lib, cfg(20, D=3, n_ell=(3, 3, 0)), wsb=1 << 40) == HB_ERR_ARG
    # a Philox window must start on a multiple of 4 -- only when that variational draws from it
    for e in range(3):
        off = [0, 0, 0]; off[e] = 6
        eps = [FAKE, FAKE, FAKE]; eps[e] = None
        assert step(lib, cfg(20, offset=off), eps=eps) == HB_ERR_ARG, e
    # Adam needs both moments and its configuration
    a = _lib.AdamConfig(1e-3, 0.9, 0.999, 1e-8, -1.0, None, 1)
    assert step(lib, c, m=FAKE) == HB_ERR_ARG
    assert step(lib, c, m=FAKE, v=FAKE) == HB_ERR_ARG
    assert step(lib, c, m=FAKE, adam=C.byref(a)) == HB_ERR_ARG


def test_step_rejects_a_short_workspace(lib):
    c = cfg(100)
    wsb = lib.hb_moe_gp_f64_workspace_bytes(C.byref(c))
    assert step(lib, c, wsb=wsb - 1) == HB_ERR_WORKSPACE
    assert step(lib, c, ws=None) == HB_ERR_WORKSPACE


# ---------------------------------------------------------------------------------------------------------------------
# the binder
# ---------------------------------------------------------------------------------------------------------------------
def _trace(model, method):
    from henbun_b200 import trace
    with trace.tracing():
        with model.tf_mode():
            return method.__wrapped__(model)


def _models():
    import henbun_b200 as hb
    import henbun_b200.tf as tf
    rng = np.random.RandomState(0)
    X = rng.randn(20, 2); Y = rng.randn(20, 1)

    class Experts(hb.model.Model):                         # notebooks/Expert_GPR.ipynb:101-149
        def setUp(self, minibatch=False, fourth=False, q_shapes=('fullrank', 'fullrank', 'diagonal')):
            self.X = hb.param.MinibatchData(X) if minibatch else hb.param.Data(X)
            self.Y = hb.param.MinibatchData(Y) if minibatch else hb.param.Data(Y)
            self.q_s = hb.variationals.Gaussian(shape=[20, 1], q_shape=q_shapes[0])
            self.q_l = hb.variationals.Gaussian(shape=[20, 1], q_shape=q_shapes[1])
            self.q_r = hb.variationals.Gaussian(shape=[20, 1], q_shape=q_shapes[2])
            if fourth:
                self.q_x = hb.variationals.Normal([3])
            self.kern_s = hb.gp.kernels.UnitRBF(np.ones(1) * 0.2)
            self.kern_l = hb.gp.kernels.UnitRBF(np.ones(1))
            self.kern_r = hb.gp.kernels.UnitRBF(np.ones(2))
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.k_var_r = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        def _f(self):
            self.f_s = tf.matmul(self.kern_s.Cholesky(self.X), self.q_s)
            self.f_l = tf.matmul(self.kern_l.Cholesky(self.X), self.q_l)
            self.f_r = tf.matmul(self.kern_r.Cholesky(self.X), self.q_r) * tf.sqrt(self.k_var_r)

        @hb.model.AutoOptimize()
        def ELBO(self):
            self._f()
            fraction = tf.sigmoid(self.f_r)
            self.f = (fraction * self.f_s + (1 - fraction) * self.f_l) * self.k_var
            return tf.reduce_sum(hb.densities.gaussian(self.Y, self.f, self.var)) - self.KL()

        @hb.model.AutoOptimize()
        def ELBO_commuted(self):                           # the gate first, every product and sum written the other way
            f_r = tf.sqrt(self.k_var_r) * tf.matmul(self.kern_r.Cholesky(self.X), self.q_r)
            f_l = tf.matmul(self.kern_l.Cholesky(self.X), self.q_l)
            f_s = tf.matmul(self.kern_s.Cholesky(self.X), self.q_s)
            fraction = tf.nn.sigmoid(f_r)
            f = self.k_var * (f_l * (1 - fraction) + f_s * fraction)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, f, self.var)) - self.KL()

        @hb.model.AutoOptimize()
        def ELBO_sqrt_kvar(self):                          # sqrt(k_var) on the mixture: not the notebook's graph
            self._f()
            fraction = tf.sigmoid(self.f_r)
            f = (fraction * self.f_s + (1 - fraction) * self.f_l) * tf.sqrt(self.k_var)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, f, self.var)) - self.KL()

        @hb.model.AutoOptimize()
        def ELBO_shared_kernel(self):                      # both experts on kern_s
            f_s = tf.matmul(self.kern_s.Cholesky(self.X), self.q_s)
            f_l = tf.matmul(self.kern_s.Cholesky(self.X), self.q_l)
            fraction = tf.sigmoid(tf.matmul(self.kern_r.Cholesky(self.X), self.q_r) * tf.sqrt(self.k_var_r))
            f = (fraction * f_s + (1 - fraction) * f_l) * self.k_var
            return tf.reduce_sum(hb.densities.gaussian(self.Y, f, self.var)) - self.KL()

        @hb.model.AutoOptimize()
        def ELBO_gate_on_l_only(self):
            self._f()
            fraction = tf.sigmoid(self.f_r)
            f = (self.f_s + (1 - fraction) * self.f_l) * self.k_var
            return tf.reduce_sum(hb.densities.gaussian(self.Y, f, self.var)) - self.KL()

    return Experts


def _bind(m, method):
    from henbun_b200 import fused
    return fused.bind(_trace(m, method), m)


def _float64():
    import henbun_b200 as hb
    cfg = hb.settings.get_settings(); cfg.dtypes.float_type = 'float64'
    return hb.settings.temp_settings(cfg)


def test_binder_accepts_the_notebook_model_in_float64():
    Experts = _models()
    with _float64():
        for method in (Experts.ELBO, Experts.ELBO_commuted):
            m = Experts()
            b = _bind(m, method)
            assert type(b).__name__ == 'MixtureGpElboBinding', method.__name__
            assert [v.long_name for v in b.var_order] == [
                'model.q_s.q_mu', 'model.q_s.q_sqrt', 'model.q_s.scale', 'model.kern_s.lengthscales',
                'model.q_l.q_mu', 'model.q_l.q_sqrt', 'model.q_l.scale', 'model.kern_l.lengthscales',
                'model.q_r.q_mu', 'model.q_r.q_sqrt', 'model.q_r.scale', 'model.kern_r.lengthscales',
                'model.k_var', 'model.k_var_r', 'model.var']
            assert b.per_sample() == 20
        m = Experts(q_shapes=('diagonal', 'diagonal', 'diagonal'))
        assert type(_bind(m, Experts.ELBO)).__name__ == 'MixtureGpElboBinding'


def test_binder_refuses_everything_else():
    Experts = _models()
    m = Experts()
    assert _bind(m, Experts.ELBO) is None                  # float32: the eager tape stays the fp32 route
    with _float64():
        for kw in (dict(fourth=True), dict(minibatch=True)):
            m = Experts(**kw)
            assert _bind(m, Experts.ELBO) is None, kw
        for method in (Experts.ELBO_shared_kernel, Experts.ELBO_sqrt_kvar, Experts.ELBO_gate_on_l_only):
            m = Experts()
            assert _bind(m, method) is None, method.__name__


def test_draw_order_follows_the_objective():
    from henbun_b200 import trace
    Experts = _models()
    g = object.__getattribute__
    m = Experts()
    _trace(m, Experts.ELBO)
    assert trace.draws() == [g(m, 'q_s'), g(m, 'q_l'), g(m, 'q_r')]
    _trace(m, Experts.ELBO_commuted)
    assert trace.draws() == [g(m, 'q_r'), g(m, 'q_l'), g(m, 'q_s')]
    with _float64():
        b = _bind(m, Experts.ELBO_commuted)
    assert b.qs == [g(m, 'q_r'), g(m, 'q_l'), g(m, 'q_s')]
    assert [q for _, q in b.experts] == [g(m, 'q_s'), g(m, 'q_l'), g(m, 'q_r')]


def test_sigmoid_outside_a_trace_is_unchanged():
    import torch
    import henbun_b200.tf as tf
    x = torch.linspace(-3, 3, 7)
    assert torch.equal(tf.sigmoid(x), torch.sigmoid(x))
    assert torch.equal(tf.nn.sigmoid(x), torch.sigmoid(x))
