"""float64 amortised model (csrc/amortised64.cu, BASELINE config 4): hb_amortised_elbo_step_f64 against the fp64 oracle
(oracle.amortised_elbo + autograd, and + the TF-1 Adam rule) at small ragged sizes and at the named size, on data with a
large common level where fp32 loses the gradients, its Philox route, its repeatability, and the float64 route through the
model API (fused.AmortisedElboBinding)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import henbun_oracle as O
from test_amortised64_host import offset_case

pytestmark = pytest.mark.gpu
ACT = {"sigmoid": 1, "relu": 2, "tanh": 3}
NAMED = ([784, 512, 512, 128], [64, 512, 512, 784], ["sigmoid", "sigmoid"], ["sigmoid", "sigmoid"], 4096, 32)


@pytest.fixture(scope="module")
def lib():
    from henbun_b200 import _lib
    return _lib.load()


def rel_err(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def make_case(enc, dec, ea, da, B, S, seed, scale=0.3):
    rng = np.random.RandomState(seed)
    X = rng.randn(B, enc[0])
    U = rng.randn(S, B, dec[0])
    p = {}
    for name, nodes in (("enc", enc), ("dec", dec)):
        for i in range(len(nodes) - 1):
            p[f"{name}.w{i}"] = scale * rng.randn(nodes[i], nodes[i + 1]) / np.sqrt(nodes[i]) * 3
            p[f"{name}.b{i}"] = 0.1 * rng.randn(1, nodes[i + 1])
    p["var"] = np.array([0.3])
    return enc, dec, ea, da, B, S, X, U, p


def keys(enc, dec):
    return [f"{n}.{k}{i}" for n, nodes in (("enc", enc), ("dec", dec)) for i in range(len(nodes) - 1) for k in "wb"] + ["var"]


def pack(case):
    enc, dec, _, _, _, _, _, _, p = case
    return np.concatenate([np.asarray(p[k], np.float64).ravel() for k in keys(enc, dec)])


def unpack(case, flat):
    enc, dec, _, _, _, _, _, _, p = case
    out, o = {}, 0
    for k in keys(enc, dec):
        n = int(np.prod(np.shape(p[k])))
        out[k] = flat[o:o + n].reshape(np.shape(p[k])); o += n
    return out


class Step(object):
    """hb_amortised_elbo_step_f64 (or the fp32 hb_amortised_elbo_step) on one case."""

    def __init__(self, lib, case, dtype=torch.float64):
        from henbun_b200 import _lib
        enc, dec, ea, da, B, S, X, U, p = case
        self.lib, self.case, self.dtype = lib, case, dtype
        c = _lib.AmortisedConfig()
        c.B, c.S, c.latent = B, S, dec[0]
        c.n_enc, c.n_dec = len(enc) - 1, len(dec) - 1
        for i, w in enumerate(enc): c.enc_nodes[i] = w
        for i, w in enumerate(dec): c.dec_nodes[i] = w
        for i, a in enumerate(ea): c.enc_act[i] = ACT[a]
        for i, a in enumerate(da): c.dec_act[i] = ACT[a]
        self.cfg = c
        self.npar = int(lib.hb_amortised_param_count(C.byref(c)))
        size = lib.hb_amortised_f64_workspace_bytes if dtype == torch.float64 else lib.hb_amortised_workspace_bytes
        self.wsb = int(size(C.byref(c)))
        self.ws = torch.empty(self.wsb, dtype=torch.uint8, device="cuda")
        self.X = torch.as_tensor(X, dtype=dtype).cuda().contiguous()
        self.params = torch.as_tensor(pack(case), dtype=dtype).cuda()
        assert self.params.numel() == self.npar
        self.grads = torch.zeros(self.npar, dtype=dtype, device="cuda")
        self.out4 = torch.zeros(4, dtype=dtype, device="cuda")

    def __call__(self, U=None, seed=0, offset=0, m=None, v=None, adam=None, grads=True):
        from henbun_b200._lib import ptr, stream, check
        self.cfg.seed, self.cfg.offset = int(seed), int(offset)
        e = None if U is None else torch.as_tensor(np.asarray(U) if not isinstance(U, torch.Tensor) else U).to("cuda", self.dtype).contiguous()
        g = self.grads if grads else None
        if self.dtype == torch.float64:
            rc = self.lib.hb_amortised_elbo_step_f64(C.byref(self.cfg), ptr(self.X), ptr(self.params), ptr(e), ptr(g), ptr(self.out4),
                                                     ptr(m), ptr(v), adam, ptr(self.ws), self.wsb, stream())
        else:
            rc = self.lib.hb_amortised_elbo_step(C.byref(self.cfg), ptr(self.X), ptr(self.params), ptr(e), ptr(g), ptr(self.out4),
                                                 ptr(self.ws), self.wsb, stream())
        check(rc, "amortised step")
        torch.cuda.synchronize()
        return self.out4.double().cpu().numpy(), self.grads.double().cpu().numpy()


def oracle(case, device="cpu", p=None):
    enc, dec, ea, da, B, S, X, U, p0 = case
    return O.value_and_grads(lambda pp, X_, U_: O.amortised_elbo(pp, X_, U_, list(ea), list(da)), p0 if p is None else p, X, U,
                             device=device)


def block_errors(case, got, gref):
    g = unpack(case, got)
    return {k: rel_err(g[k], gref[k]) for k in g}


@pytest.mark.parametrize("enc,dec,ea,da,B,S", [
    ([12, 16, 8], [4, 16, 12], ["sigmoid"], ["sigmoid"], 32, 5),
    ([7, 6], [3, 7], [], [], 9, 1),                                        # single linear layers
    ([20, 33, 17, 10], [5, 9, 31, 20], ["tanh", "relu"], ["relu", "tanh"], 50, 3),
    ([64, 128, 128, 32], [16, 128, 128, 64], ["sigmoid", "sigmoid"], ["sigmoid", "sigmoid"], 512, 8),
])
def test_step_matches_the_fp64_oracle(lib, enc, dec, ea, da, B, S):
    case = make_case(enc, dec, ea, da, B, S, seed=B + S)
    out4, got = Step(lib, case)(case[7])
    ref, gref = oracle(case)
    assert abs(out4[0] - ref) <= 1e-10 * abs(ref)
    for k, e in block_errors(case, got, gref).items():
        assert e < 1e-8, (k, e)


def test_named_size_matches_the_fp64_oracle_on_the_device(lib):
    """784-512-512-2x64 encoder + mirrored decoder, minibatch 4096, S = 32: the dW reductions over 131072 rows run split-K."""
    case = make_case(*NAMED, seed=0, scale=0.05 / 3 * np.sqrt(512))
    out4, got = Step(lib, case)(case[7])
    ref, gref = oracle(case, device="cuda")
    assert abs(out4[0] - ref) <= 1e-10 * abs(ref)
    for k, e in block_errors(case, got, gref).items():
        assert e < 1e-8, (k, e)


def test_offset_input_meets_1e5_where_fp32_does_not(lib):
    case = offset_case()
    ref, gref = oracle(case)
    out4, got = Step(lib, case)(case[7])
    errs = block_errors(case, got, gref)
    _, got32 = Step(lib, case, torch.float32)(case[7])
    errs32 = block_errors(case, got32, gref)
    print("fp32 entry on the offset input:", {k: "%.1e" % e for k, e in errs32.items()})
    print("fp64 entry on the offset input:", {k: "%.1e" % e for k, e in errs.items()})
    assert abs(out4[0] - ref) <= 1e-10 * abs(ref)
    for k, e in errs.items():
        assert e < 1e-5, (k, e)


def test_philox_route_equals_injected_draws_and_repeats_bitwise(lib):
    from henbun_b200 import ops
    case = make_case([20, 33, 17, 10], [5, 9, 31, 20], ["tanh", "relu"], ["relu", "tanh"], 50, 3, seed=3)
    st = Step(lib, case)
    seed, offset = 17, 4 * 1001
    o_a, g_a = st(None, seed, offset)
    o_b, g_b = st(None, seed, offset)
    assert np.array_equal(o_a, o_b) and np.array_equal(g_a, g_b)
    U = ops.randn_philox((3, 50, 5), seed, offset, "cuda").double()
    o_c, g_c = st(U)
    assert np.array_equal(o_a, o_c) and np.array_equal(g_a, g_c)


def test_fp64_and_fp32_routes_agree_on_a_well_conditioned_input(lib):
    case = make_case([12, 16, 8], [4, 16, 12], ["sigmoid"], ["sigmoid"], 32, 5, seed=7)
    o64, g64 = Step(lib, case)(None, 5, 8)
    o32, g32 = Step(lib, case, torch.float32)(None, 5, 8)
    assert abs(o64[0] - o32[0]) <= 1e-5 * abs(o64[0])
    for k, e in block_errors(case, g32, unpack(case, g64)).items():
        assert e < 1e-5, (k, e)


def test_ten_fused_adam_steps_match_the_oracle(lib):
    from henbun_b200 import _lib
    case = make_case([20, 33, 17, 10], [5, 9, 31, 20], ["tanh", "sigmoid"], ["sigmoid", "tanh"], 50, 3, seed=5)
    st = Step(lib, case)
    m = torch.zeros(st.npar, dtype=torch.float64, device="cuda"); v = torch.zeros_like(m)
    theta = pack(case); mh = np.zeros_like(theta); vh = np.zeros_like(theta)
    rng = np.random.RandomState(9)
    lr = 0.01
    for t in range(1, 11):
        U = rng.randn(3, 50, 5)
        adam = _lib.AdamConfig(lr, 0.9, 0.999, 1e-8, -1.0, None, t)
        st(U, m=m, v=v, adam=C.byref(adam), grads=(t % 2 == 0))          # the gradient buffer is optional under Adam
        c = case[:7] + (U,) + case[8:]
        _, g = oracle(c, p=unpack(case, theta))
        gflat = np.concatenate([np.asarray(g[k]).ravel() for k in keys(case[0], case[1])])
        theta, mh, vh = O.adam_tf1_step(theta, -gflat, mh, vh, t, lr=lr)
    assert rel_err(st.params.cpu().numpy(), theta) < 1e-7


# ---------------------------------------------------------------------------------------------------------------------
# through the model API
# ---------------------------------------------------------------------------------------------------------------------
def _amortised():
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


def _float64():
    import henbun_b200 as hb
    s = hb.settings.get_settings(); s.dtypes.float_type = 'float64'
    return hb.settings.temp_settings(s)


def test_binding_in_float64_matches_the_eager_tape():
    import henbun_b200.tf as tf
    Amortised = _amortised()
    Xall = np.random.RandomState(0).randn(500, 12)
    res = []
    with _float64():
        for fused in (True, False):
            np.random.seed(11)
            m = Amortised(X=Xall)
            m.ELBO().compile(optimizer=tf.train.AdamOptimizer(0.01), n_samples=5, seed=2, verbose=False, fused=fused)
            if fused:
                b = m.ELBO()._fused
                assert m.ELBO().fused_entry == 'AmortisedElboBinding' and b.f64 and b.fused_adam
            else:
                assert m.ELBO().fused_entry is None
            objs = [float(m.ELBO().optimize(maxiter=1, minibatch_size=64)) for _ in range(4)]
            res.append((objs, [v._free_numpy().astype(np.float64).ravel() for v in m.get_variables() if v.is_parameter]))
    assert np.allclose(res[0][0], res[1][0], rtol=1e-4)
    for a, b in zip(res[0][1], res[1][1]):
        assert np.allclose(a, b, rtol=1e-4, atol=2e-5)


def test_float64_route_follows_new_data_and_assignments():
    import henbun_b200.tf as tf
    Amortised = _amortised()
    rng = np.random.RandomState(1)
    X1 = rng.randn(300, 12)
    with _float64():
        m = Amortised(X=X1)
        opt = m.ELBO()
        opt.compile(optimizer=tf.train.AdamOptimizer(0.01), n_samples=3, seed=4, verbose=False)
        b = opt._fused
        assert b.f64
        objs = [float(opt.optimize(maxiter=1, minibatch_size=32)) for _ in range(3)]      # device-drawn minibatches
        assert np.all(np.isfinite(objs))
        assert torch.equal(b._X64.cpu(), torch.from_numpy(X1))
        # the fp32 mirror tracks the masters
        npar = b._p64.numel()
        assert torch.equal(opt._flat[:npar], b._p64.float())
        # new data reaches the fp64 copy, and the rows the step sees are this feed's
        X2 = 100.0 + rng.randn(300, 12)
        m.X = X2
        opt.optimize(maxiter=1, minibatch_size=32)
        assert torch.equal(b._X64.cpu(), torch.from_numpy(X2))
        # an assignment to a weight reaches the master: one Adam step moves it by at most about lr
        g = object.__getattribute__
        bvar = g(g(m.dec, 'matbias1'), 'b')
        m.dec.matbias1.b = np.full(bvar._host.shape, 5.0)
        opt.optimize(maxiter=1, minibatch_size=32)
        o, s = opt._slices[[id(v) for v in opt.var_list].index(id(bvar))]
        assert torch.all(torch.abs(b._p64[o:o + s] - 5.0) <= 0.0101)
        assert torch.equal(opt._flat[:npar], b._p64.float())
