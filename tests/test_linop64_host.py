"""Host-side contract of the float64 linear-operator pair (csrc/linop64.cu, BASELINE config 5) and of the route its binding
(fused.LinopElboBinding) takes: workspace sizes, the argument checks that return before anything reaches a device, and
which route the binder picks under each float_type.  No kernel is launched, so these run without a GPU."""
import ctypes as C

import numpy as np
import pytest
import torch

HB_OK, HB_ERR_ARG, HB_ERR_WORKSPACE = 0, 1, 3
FAKE = C.c_void_p(4096)          # a non-NULL device address; every call below is rejected before it is dereferenced


@pytest.fixture(scope="module")
def lib():
    from henbun_b200 import _lib
    return _lib.load()


def cfg(M=300, n=70, S=5, M_total=None, offset=0, presplit=0):
    from henbun_b200 import _lib
    return _lib.LinopConfig(M, M if M_total is None else M_total, n, S, 0, offset, presplit)


def wsb(lib, c):
    return lib.hb_linop_f64_workspace_bytes(C.byref(c))


def test_workspace_grows_with_every_dimension(lib):
    base = wsb(lib, cfg())
    assert base > 0
    # U, Z, Zt [S, n] and F [S, M] in double, plus the split-K partial tiles of the fp64 GEMM
    assert base >= (3 * 5 * 70 + 5 * 300) * 8 + (8 << 20)
    assert wsb(lib, cfg(M=3000)) > base
    assert wsb(lib, cfg(n=700)) > base
    assert wsb(lib, cfg(S=50)) > base
    # the named size: F alone is S * M doubles
    assert wsb(lib, cfg(M=65536, n=16384, S=64)) >= 64 * 65536 * 8
    # the parameter count is the fp32 route's
    assert lib.hb_linop_param_count(C.byref(cfg())) == 70 * 70 + 70 + 1


def test_sizes_of_invalid_configs_are_zero(lib):
    for c in (cfg(n=0), cfg(n=-2), cfg(S=0), cfg(M=0), cfg(M=-1), cfg(M=300, M_total=299), cfg(presplit=1)):
        assert wsb(lib, c) == 0
    assert lib.hb_linop_f64_workspace_bytes(None) == 0


def local(lib, c, A=FAKE, y=FAKE, params=FAKE, eps=FAKE, zbar=FAKE, ws=FAKE, nbytes=None):
    if nbytes is None:
        nbytes = wsb(lib, c) or 1 << 40
    return lib.hb_linop_elbo_local_f64(C.byref(c), A, y, params, eps, zbar, ws, nbytes, None)


def update(lib, c, params=FAKE, zbar=FAKE, grads=None, m=None, v=None, adam=None, out4=FAKE, ws=FAKE, nbytes=None):
    if nbytes is None:
        nbytes = wsb(lib, c) or 1 << 40
    return lib.hb_linop_elbo_update_f64(C.byref(c), params, zbar, grads, m, v, adam, out4, ws, nbytes, None)


def test_local_rejects_bad_arguments(lib):
    assert lib.hb_linop_elbo_local_f64(None, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 1 << 40, None) == HB_ERR_ARG
    c = cfg()
    for k in ("A", "y", "params", "zbar"):
        assert local(lib, c, **{k: None}) == HB_ERR_ARG, k
    for bad in (cfg(n=0), cfg(n=-5), cfg(S=0), cfg(M=0), cfg(M=-3), cfg(M=300, M_total=200), cfg(presplit=1)):
        assert local(lib, bad, nbytes=1 << 40) == HB_ERR_ARG
    # a Philox window must start on a multiple of 4 -- only when the samples are drawn from it
    assert local(lib, cfg(offset=6), eps=None) == HB_ERR_ARG


def test_update_rejects_bad_arguments(lib):
    from henbun_b200 import _lib
    assert lib.hb_linop_elbo_update_f64(None, FAKE, FAKE, None, None, None, None, FAKE, FAKE, 1 << 40, None) == HB_ERR_ARG
    c = cfg()
    for k in ("params", "zbar", "out4"):
        assert update(lib, c, **{k: None}) == HB_ERR_ARG, k
    for bad in (cfg(n=0), cfg(S=0), cfg(M=0), cfg(M=300, M_total=200), cfg(presplit=1)):
        assert update(lib, bad, nbytes=1 << 40) == HB_ERR_ARG
    # Adam needs both moments and its configuration
    a = _lib.AdamConfig(1e-3, 0.9, 0.999, 1e-8, -1.0, None, 1)
    assert update(lib, c, m=FAKE) == HB_ERR_ARG
    assert update(lib, c, v=FAKE, adam=C.byref(a)) == HB_ERR_ARG
    assert update(lib, c, m=FAKE, v=FAKE) == HB_ERR_ARG


def test_short_workspace_is_rejected(lib):
    c = cfg()
    n = wsb(lib, c)
    assert local(lib, c, nbytes=n - 1) == HB_ERR_WORKSPACE
    assert local(lib, c, ws=None) == HB_ERR_WORKSPACE
    assert update(lib, c, nbytes=n - 1) == HB_ERR_WORKSPACE
    assert update(lib, c, ws=None) == HB_ERR_WORKSPACE


# ---------------------------------------------------------------------------------------------------------------------
# the binder
# ---------------------------------------------------------------------------------------------------------------------
def _model(M=40, n=12):
    import henbun_b200 as hb
    import henbun_b200.tf as tf
    rng = np.random.RandomState(0)
    A = rng.randn(M, n); y = rng.randn(M)

    class LinearOperator(hb.model.Model):
        def setUp(self):
            self.A = hb.param.Data(A); self.y = hb.param.Data(y)
            self.q = hb.variationals.Normal([n], q_shape='fullrank', stddev=0.1)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            f = tf.matmul(self.q, self.A, transpose_b=True)
            return tf.reduce_sum(hb.densities.gaussian(self.y, f, self.var)) - self.KL()

    return LinearOperator


def _bind(m, method):
    from henbun_b200 import fused, trace
    with trace.tracing():
        with m.tf_mode():
            tree = method.__wrapped__(m)
    return fused.bind(tree, m)


def _float64():
    import henbun_b200 as hb
    s = hb.settings.get_settings(); s.dtypes.float_type = 'float64'
    return hb.settings.temp_settings(s)


def test_binder_picks_the_route_of_the_float_type():
    Model = _model()
    m = Model()
    b32 = _bind(m, Model.ELBO)
    assert type(b32).__name__ == 'LinopElboBinding' and b32.f64 is False
    with _float64():
        m = Model()
        b64 = _bind(m, Model.ELBO)
    assert type(b64).__name__ == 'LinopElboBinding' and b64.f64 is True
    for b in (b32, b64):
        assert [v.long_name for v in b.var_order] == ['model.q.q_sqrt', 'model.q.q_mu', 'model.var']
        assert b.fused_adam and b.per_sample() == 12


def test_float64_masters_keep_no_gradient():
    """The fp64 route never writes a flat gradient (nor does the fp32 one): its masters hold parameters and moments only, and
    pushing them leaves the flat gradient buffer alone."""
    from henbun_b200 import fused
    Model = _model()
    with _float64():
        b = _bind(Model(), Model.ELBO)

    class Opt(object):
        _flat = torch.arange(8, dtype=torch.float32) / 3
        _flat_grad = torch.full((8,), 7.0)
        _m = torch.zeros(8); _v = torch.ones(8)

    opt = Opt()
    b._pull64(opt, 6, 'cpu')
    assert b._g64 is None and b._p64.dtype == torch.float64 and b._m64.shape == (6,)
    b._p64 += 1.0
    b._push64(opt, 6)
    assert torch.equal(opt._flat[:6], b._p64.float())
    assert torch.equal(opt._flat_grad, torch.full((8,), 7.0))
    assert fused.GpElboBinding._grad64 and fused.MixtureGpElboBinding._grad64
