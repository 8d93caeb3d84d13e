"""Host-side contract of the float64 amortised model (csrc/amortised64.cu, BASELINE config 4) and of the route its binding
(fused.AmortisedElboBinding) takes: workspace sizes, the argument checks that return before anything reaches a device, which
route the binder picks, and why the route exists: on data with a large common level the oracle in fp32 misses 1e-5 on the
gradients by more than 10x.  No kernel is launched, so these run without a GPU."""
import ctypes as C

import numpy as np
import pytest

HB_OK, HB_ERR_ARG, HB_ERR_WORKSPACE = 0, 1, 3
FAKE = C.c_void_p(4096)          # a non-NULL device address; every call below is rejected before it is dereferenced
ACT = {"sigmoid": 1, "relu": 2, "tanh": 3}


@pytest.fixture(scope="module")
def lib():
    from henbun_b200 import _lib
    return _lib.load()


def cfg(enc=(12, 16, 8), dec=(4, 16, 12), acts=("sigmoid",), B=32, S=5, offset=0):
    from henbun_b200 import _lib
    c = _lib.AmortisedConfig()
    c.B, c.S, c.latent = B, S, dec[0]
    c.n_enc, c.n_dec = len(enc) - 1, len(dec) - 1
    for i, w in enumerate(enc): c.enc_nodes[i] = w
    for i, w in enumerate(dec): c.dec_nodes[i] = w
    for i, a in enumerate(acts[:len(enc) - 2]): c.enc_act[i] = ACT[a]
    for i, a in enumerate(acts[:len(dec) - 2]): c.dec_act[i] = ACT[a]
    c.offset = offset
    return c


def wsb(lib, c):
    return lib.hb_amortised_f64_workspace_bytes(C.byref(c))


def test_workspace_grows_with_every_dimension(lib):
    base = wsb(lib, cfg())
    assert base > 0
    # the decoder's activations alone are S B (4 + 16 + 12) doubles
    assert base >= 5 * 32 * (4 + 16 + 12) * 8
    assert wsb(lib, cfg(B=320)) > base
    assert wsb(lib, cfg(S=50)) > base
    assert wsb(lib, cfg(enc=(12, 160, 8), dec=(4, 160, 12))) > base
    # the named size: two [S B, 784] gradient buffers and the decoder's activations in double
    named = cfg(enc=(784, 512, 512, 128), dec=(64, 512, 512, 784), acts=("sigmoid", "sigmoid"), B=4096, S=32)
    assert wsb(lib, named) >= 32 * 4096 * (2 * 784 + 64 + 512 + 512 + 784) * 8
    # the parameter count is the fp32 route's
    assert lib.hb_amortised_param_count(C.byref(cfg())) == 12 * 16 + 16 + 16 * 8 + 8 + 4 * 16 + 16 + 16 * 12 + 12 + 1


def test_sizes_of_invalid_configs_are_zero(lib):
    bad = [cfg(B=0), cfg(S=0), cfg(enc=(12, 16, 9)), cfg(dec=(4, 16, 11)), cfg(dec=(3, 16, 12))]
    c = cfg(); c.n_enc = 0; bad.append(c)
    c = cfg(); c.n_dec = 9; bad.append(c)
    c = cfg(); c.enc_act[0] = 4; bad.append(c)
    for c in bad:
        assert wsb(lib, c) == 0
        assert lib.hb_amortised_workspace_bytes(C.byref(c)) == 0       # the fp32 route agrees on what is valid
    assert lib.hb_amortised_f64_workspace_bytes(None) == 0


def step(lib, c, X=FAKE, params=FAKE, eps=FAKE, grads=FAKE, out4=FAKE, m=None, v=None, adam=None, ws=FAKE, nbytes=None):
    if nbytes is None:
        nbytes = wsb(lib, c) or 1 << 40
    return lib.hb_amortised_elbo_step_f64(C.byref(c), X, params, eps, grads, out4, m, v, adam, ws, nbytes, None)


def test_step_rejects_bad_arguments(lib):
    from henbun_b200 import _lib
    assert lib.hb_amortised_elbo_step_f64(None, FAKE, FAKE, FAKE, FAKE, FAKE, None, None, None, FAKE, 1 << 40, None) == HB_ERR_ARG
    c = cfg()
    for k in ("X", "params", "out4"):
        assert step(lib, c, **{k: None}) == HB_ERR_ARG, k
    for bad in (cfg(B=0), cfg(S=-1), cfg(enc=(12, 16, 9))):
        assert step(lib, bad, nbytes=1 << 40) == HB_ERR_ARG
    # a Philox window must start on a multiple of 4 -- only when the samples are drawn from it
    assert step(lib, cfg(offset=6), eps=None) == HB_ERR_ARG
    # Adam needs both moments and its configuration; without Adam the gradient needs somewhere to go
    a = _lib.AdamConfig(1e-3, 0.9, 0.999, 1e-8, -1.0, None, 1)
    assert step(lib, c, m=FAKE) == HB_ERR_ARG
    assert step(lib, c, v=FAKE, adam=C.byref(a)) == HB_ERR_ARG
    assert step(lib, c, m=FAKE, v=FAKE) == HB_ERR_ARG
    assert step(lib, c, grads=None) == HB_ERR_ARG
    # S B rows must fit the products' int row count
    assert step(lib, cfg(B=1 << 16, S=1 << 15), nbytes=1 << 62) == HB_ERR_ARG


def test_short_workspace_is_rejected(lib):
    from henbun_b200 import _lib
    c = cfg()
    n = wsb(lib, c)
    assert step(lib, c, nbytes=n - 1) == HB_ERR_WORKSPACE
    assert step(lib, c, ws=None) == HB_ERR_WORKSPACE
    a = _lib.AdamConfig(1e-3, 0.9, 0.999, 1e-8, -1.0, None, 1)
    assert step(lib, c, grads=None, m=FAKE, v=FAKE, adam=C.byref(a), nbytes=n - 1) == HB_ERR_WORKSPACE


# ---------------------------------------------------------------------------------------------------------------------
# the binder
# ---------------------------------------------------------------------------------------------------------------------
def _model():
    import henbun_b200 as hb
    import henbun_b200.tf as tf

    class Amortised(hb.model.Model):
        def setUp(self, X=None, latent=4, hidden=16):
            self.X = hb.param.MinibatchData(X)
            self.enc = hb.nn.NeuralNet([X.shape[1], hidden, 2 * latent], stddev=0.3, neuron_types=tf.tanh)
            self.dec = hb.nn.NeuralNet([latent, hidden, X.shape[1]], stddev=0.3)
            self.q_local = hb.variationals.Normal([latent], collections=hb.param.graph_key.LOCAL)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            self.q_local = self.enc(self.X)
            x_rec = self.dec(self.q_local)
            return tf.reduce_sum(hb.densities.gaussian(self.X, x_rec, self.var)) - self.KL(hb.param.graph_key.LOCAL)

    return Amortised


def _bind(m, method):
    from henbun_b200 import fused, trace
    try:
        with trace.tracing():
            with m.tf_mode():
                tree = method.__wrapped__(m)
    finally:
        for v in fused._variationals_of(m):
            v.__dict__.pop('_sym_feed', None)
    return fused.bind(tree, m)


def _float64():
    import henbun_b200 as hb
    s = hb.settings.get_settings(); s.dtypes.float_type = 'float64'
    return hb.settings.temp_settings(s)


def test_binder_picks_the_float64_route_only_with_float64_and_one_process(monkeypatch):
    from henbun_b200 import parallel
    Model = _model()
    X = np.random.RandomState(0).randn(50, 12)
    b32 = _bind(Model(X=X), Model.ELBO)
    assert type(b32).__name__ == 'AmortisedElboBinding' and b32.f64 is False and b32.fused_adam is False
    with _float64():
        b64 = _bind(Model(X=X), Model.ELBO)
        assert type(b64).__name__ == 'AmortisedElboBinding' and b64.f64 is True and b64.fused_adam is True
        monkeypatch.setattr(parallel, 'world', lambda: (2, 0))
        bw = _bind(Model(X=X), Model.ELBO)
        assert type(bw).__name__ == 'AmortisedElboBinding' and bw.f64 is False and bw.fused_adam is False
    names = [v.long_name for v in b64.var_order]
    assert names == ['model.enc.matbias0.w', 'model.enc.matbias0.b', 'model.enc.matbias1.w', 'model.enc.matbias1.b',
                     'model.dec.matbias0.w', 'model.dec.matbias0.b', 'model.dec.matbias1.w', 'model.dec.matbias1.b', 'model.var']
    assert b64._grad64 is False


def test_minibatch_records_the_index_it_was_fed():
    import henbun_b200 as hb
    d = hb.param.MinibatchData(np.zeros((10, 3)))
    d._resident = 'resident'                       # the gather itself is not reached on a CPU-only box
    try:
        d._gather([3, 1, 4])
    except Exception:
        pass
    assert list(np.asarray(d.last_index)) == [3, 1, 4]


# ---------------------------------------------------------------------------------------------------------------------
# why: the oracle in fp32 on the offset input of tests/test_gpu_amortised64.py
# ---------------------------------------------------------------------------------------------------------------------
def offset_case(c=1e4, seed=0):
    """enc 32-64-16, dec 8-64-32, sigmoid, B = 256, S = 4, data c + 0.5 randn; the decoder's last bias starts at the level c
    and var at about 0.25."""
    rng = np.random.RandomState(seed)
    enc, dec, B, S = [32, 64, 16], [8, 64, 32], 256, 4
    X = c + 0.5 * rng.randn(B, enc[0])
    U = rng.randn(S, B, dec[0])
    p = {}
    for name, nodes in (("enc", enc), ("dec", dec)):
        for i in range(len(nodes) - 1):
            p[f"{name}.w{i}"] = rng.randn(nodes[i], nodes[i + 1]) / np.sqrt(nodes[i]) * (0.3 / c if name == "enc" and i == 0 else 1.0)
            p[f"{name}.b{i}"] = 0.1 * rng.randn(1, nodes[i + 1])
    p["dec.b1"] = p["dec.b1"] + c
    p["var"] = np.array([np.log(np.expm1(0.25))])
    return enc, dec, ["sigmoid"], ["sigmoid"], B, S, X, U, p


def oracle_block_errors(case, dtype):
    import torch
    from oracle import henbun_oracle as O
    enc, dec, ea, da, B, S, X, U, p = case
    _, g64 = O.value_and_grads(lambda pp, X_, U_: O.amortised_elbo(pp, X_, U_, ea, da), p, X, U)
    _, g = O.value_and_grads(lambda pp, X_, U_: O.amortised_elbo(pp, X_, U_, ea, da), p, X, U, dtype=dtype)
    return {k: np.linalg.norm(g[k] - g64[k]) / max(np.linalg.norm(g64[k]), 1e-300) for k in g64}


def test_fp32_arithmetic_misses_the_offset_input_by_more_than_10x():
    import torch
    errs = oracle_block_errors(offset_case(), torch.float32)
    assert max(errs.values()) > 10 * 1e-5, errs
