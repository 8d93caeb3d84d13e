"""CPU-side logic of the Henbun-shaped API mirror (no GPU, no kernels): parameter tree, naming,
assignment, LOCAL feed sizes, settings, transforms, Indexer, and the "no silent fallback" rule.
Ports of testing/test_param.py, test_data.py, test_transforms.py, test_model.py host-side checks."""
import numpy as np
import pytest
import torch

import henbun_b200 as hb


def test_tree_names_and_parents():                   # test_param.py naming / parent links
    m = hb.model.Model()
    m.p = hb.param.Variable([2, 3])
    m.k = hb.gp.kernels.UnitRBF(np.ones(2))
    m.q = hb.variationals.Gaussian([4, 1], q_shape='fullrank')
    assert m.p.long_name == 'model.p' and m.k.lengthscales.long_name == 'model.k.lengthscales'
    assert m.q.q_mu._parent is m.q and m.q._parent is m and m.p.highest_parent is m
    names = [v.long_name for v in m.get_variables()]
    assert names == ['model.k.lengthscales', 'model.p', 'model.q.q_mu', 'model.q.q_sqrt', 'model.q.scale']   # name-sorted
    assert m.q.q_sqrt.shape == [4, 4] and m.q.size == 4


def test_truncated_normal_init_range():              # test_param.py:286-296
    v = hb.param.Variable([2000], mean=1.0, stddev=0.5)
    assert v._host.dtype == np.float32
    assert np.all(np.abs(v._host - 1.0) <= 2 * 0.5 + 1e-6)
    assert abs(v._host.mean() - 1.0) < 0.05


def test_assignment_is_deferred_until_initialize():  # test_model.py:53-59, param.py docstring
    m = hb.model.Model()
    m.p = hb.param.Variable([2, 1])
    m.initialize()
    m.p = np.zeros((2, 1))
    assert m.p._assigned
    m.initialize()
    assert not m.p._assigned and np.allclose(m.p.value, 0)
    m.s = hb.param.Variable([1], transform=hb.transforms.positive)
    m.s = 2.5
    assert np.allclose(m.s.value, 2.5, atol=1e-5)            # stored in free space, read back transformed
    assert np.allclose(m.s._free_numpy(), np.log(np.expm1(2.5 - 1e-6)), atol=1e-5)


def test_variational_initialisation_rules():        # variationals.py:84-96, 266-273
    g = hb.variationals.Gaussian([3], mean=0.1, stddev=2.0)
    assert abs(g.q_mu._host.mean() - 0.05) < 0.3 and abs(g.q_sqrt._host.mean() - 0.0) < 0.3      # log(1)=0
    g2 = hb.variationals.Gaussian([3], mean=5.0, stddev=1.0)                                     # |mean| >= stddev
    assert abs(g2.q_mu._host.mean() - 1.0) < 0.1 and abs(g2.q_sqrt._host.mean() - np.log(0.2)) < 0.3
    f = hb.variationals.Normal([5], q_shape='fullrank', stddev=0.5)
    assert f.q_sqrt._host.shape == (5, 5) and np.all(f.q_sqrt._host > 0)                        # every entry ~ stddev
    with pytest.raises(AssertionError):
        hb.variationals.Normal([5], q_shape='lowrank')


def test_local_feed_sizes_and_einsum_strings():      # test_variationals.py:15-24, param.py:281-289
    LOCAL = hb.param.graph_key.LOCAL
    v = hb.variationals.Normal((2, 3), n_layers=[2, 3], q_shape='fullrank')
    vl = hb.variationals.Normal((2, 3), n_layers=[2, 3], q_shape='fullrank', collections=LOCAL)
    assert v._einsum_matmul() == 'abcd,abd->abc' and vl._einsum_matmul() == 'abcde,abce->abcd'
    assert vl.feed_size == 6 + 36 and v.feed_size == 0
    d = hb.variationals.Gaussian([4], collections=LOCAL)
    assert d.feed_size == 4 + 4 + 1                                     # q_mu | q_sqrt | scale, name-sorted
    assert d.get_variables(LOCAL) and not d.get_variables(hb.param.graph_key.VARIABLES)
    assert d.KL(hb.param.graph_key.VARIABLES).shape == ()               # zero for another collection


def test_data_and_minibatch_data():                  # test_data.py, test_model.py:116-135
    m = hb.model.Model()
    m.d = hb.param.Data(np.arange(6.0).reshape(3, 2))
    assert np.array_equal(m.d.value, np.arange(6.0).reshape(3, 2))
    m.d = np.ones((3, 2))
    assert np.array_equal(m.d.value, np.ones((3, 2)))
    with pytest.raises(ValueError):
        m.d = np.ones((4, 2))                                           # param.py:712-713
    with pytest.raises(NotImplementedError):
        hb.param.Data(np.array(['a']))
    m.mb = hb.param.MinibatchData(np.zeros((100, 3)))
    m.validate()
    assert m._index.data_size == 100 and m._index.train_size == 90 and m._index.test_size == 10
    idx = m._index.train_index(7)
    assert idx.shape == (7,) and set(idx) <= set(m._index._train_index)
    assert set(m._index.test_index(5)) <= set(m._index._test_index)
    m.mb2 = hb.param.MinibatchData(np.zeros((50, 3)))
    with pytest.raises(ValueError):
        m.validate()                                                    # model.py:113


def test_settings_temp_context():                    # _settings.py:26-63, Expert_GPR.ipynb:203,224
    assert hb.settings.numerics.jitter_level == 1e-5 and hb.settings.numerics.clip_by_value is False
    assert hb.settings.dtypes.float_type == 'float32'
    cfg = hb.settings.get_settings()
    cfg.numerics.jitter_level = 3e-4
    with hb.settings.temp_settings(cfg):
        assert hb.settings.numerics.jitter_level == 3e-4
    assert hb.settings.numerics.jitter_level == 1e-5


def test_transforms_numpy_roundtrip():               # test_transforms.py:49-53
    x = np.random.RandomState(0).randn(10)
    for t in (hb.transforms.Identity(), hb.transforms.Exp(), hb.transforms.Log1pe(), hb.transforms.Logistic(7.3, 19.4)):
        assert np.allclose(t.backward(t.forward(x)), x, atol=1e-4)
    assert hb.transforms.positive.__class__ is hb.transforms.Log1pe
    # the device side (tf_forward / tf_log_jacobian, test_transforms.py:39-47) is a CUDA kernel: tests/test_gpu_transforms.py.
    # On a CPU tensor it must raise, not fall back.
    with pytest.raises(Exception):
        hb.transforms.Log1pe().tf_forward(torch.tensor(x, dtype=torch.float32))
    assert hb.transforms.Identity().tf_forward(torch.tensor(x)) is not None


def test_paramlist_and_aliases():
    pl = hb.param.ParamList([hb.param.Variable([1]), hb.param.Variable([2])])
    assert len(pl) == 2 and pl[0].name == 'item0'
    pl.append(hb.param.Variable([3]))
    assert pl[2].name == 'item2'
    assert hb.param.Param is hb.param.Variable and hb.gp.kern.RBF is hb.gp.kernels.UnitRBF
    assert hb.gp.kern.Stationary is hb.gp.kernels.UnitStationary


def test_no_silent_cpu_fallback():
    """Evaluating anything needs the CUDA library and a device; without a GPU it must raise, not fall back."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    m = hb.model.Model()
    m.q = hb.variationals.Normal([3])
    with pytest.raises(Exception) as e:
        with m.tf_mode():
            m.q
    assert 'CUDA' in str(e.value) or 'cuda' in str(e.value)
    from henbun_b200 import _lib
    with pytest.raises(_lib.HenbunB200Error):
        _lib.ptr(torch.zeros(3))


def test_priors_host_side():                         # priors.py:44-116 (strings, hyper-parameter storage)
    g = hb.priors.Gaussian(0.5, [1.0, 2.0])
    assert g.mu.dtype == np.float32 and g.mu.shape == (1,) and g.var.shape == (2,)
    assert str(g) == "N(" + str(g.mu) + "," + str(g.var) + ")"
    assert str(hb.priors.LogNormal(0.0, 1.0)).startswith("logN(") and str(hb.priors.Gamma(2.0, 1.5)).startswith("Ga(")
    assert str(hb.priors.Laplace(0.0, 1.0)).startswith("Lap.(") and str(hb.priors.Normal()) == "N(0,1)"
    u = hb.priors.Uniform(1.0, 3.0)
    assert str(u) == "U(1.0,3.0)" and np.isclose(u.log_height, -np.log(2.0))
    assert np.isclose(u.logp(torch.zeros(5, 2)), 10 * -np.log(2.0))                  # constant: no kernel involved
    with pytest.raises(NotImplementedError):
        hb.priors.Prior().logp(torch.zeros(1))
    with pytest.raises(TypeError):
        hb.priors.Gaussian.__mro__[1].__init__(hb.priors.Gaussian.__new__(hb.priors.Gaussian), 1.0)   # wrong hyper count


def test_neural_net_structure():                     # nn.py:34-87, test_nn.py shapes
    net = hb.nn.NeuralNet([6, 5, 4, 3], n_layers=[2], stddev=0.3)
    assert [net[i].w.shape for i in range(3)] == [[6, 5], [5, 4], [4, 3]]
    assert [net[i].b.shape for i in range(3)] == [[1, 5], [1, 4], [1, 3]]
    assert net.matbias1 is net[1] and len(net.neuron_types) == 2
    assert net[0].w._host.shape == (2, 6, 5)                                         # [*n_layers, in, out]
    names = [v.long_name for v in net.get_variables()]
    assert names == sorted(names) and len(names) == 6
    with pytest.raises(AssertionError):
        hb.nn.MatBias([3, 4, 5])
    mixed = hb.nn.NeuralNet([3, 3, 3, 2], neuron_types=[hb.nn.tanh, hb.nn.relu])
    assert mixed.neuron_types == [hb.nn.tanh, hb.nn.relu]


def test_bench_cpu_extrapolation_rule():
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("bench", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    assert bench.extrapolation_factor(4096, 4096, 64) == 1.0
    f = bench.extrapolation_factor(65536, 16384, 64)
    assert 16.0 < f < 64.0 and abs(f - 62.9) < 0.1                                   # cubic term dominates at S = 64
    assert bench.extrapolation_factor(65536, 16384, 512) < f                          # more samples -> larger quadratic share
    assert bench.host_threads() >= 1


def test_bench_dump_outputs_cap_and_fixed_sample(tmp_path, monkeypatch):
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("bench", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    assert bench.DUMP_BYTES + 4096 < 64e6
    monkeypatch.setattr(bench, "DUMP_BYTES", 8192)                                   # shares of 4 KB: "big" is sampled
    big = torch.arange(100000, dtype=torch.float32).reshape(250, 400)
    small = torch.tensor([[1.0, 2.0]], dtype=torch.float64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"big": big, "small": small})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and 0 < a.nbytes <= 4096 and np.array_equal(a, b)    # same positions in every run
    assert np.all(np.diff(a) > 0) and a[-1] < 100000                                  # distinct elements of the array
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float64 and s.shape == (1, 2) and np.array_equal(s, [[1.0, 2.0]])


def test_philox4x32_10_published_algorithm_reproduces_the_kat_vectors():
    """Independent restatement of Philox-4x32-10 (Salmon et al. 2011: multipliers 0xD2511F53 / 0xCD9E8D57, Weyl key
    increments 0x9E3779B9 / 0xBB67AE85) against the three Random123 known-answer vectors that the GPU test
    (tests/test_gpu_parity_named.py) pins the device generator to."""
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85

    def philox(c, k):
        c = list(c); k = list(k)
        for _ in range(10):
            p0 = M0 * c[0]; p1 = M1 * c[2]
            c = [(p1 >> 32) ^ c[1] ^ k[0], p1 & 0xffffffff, (p0 >> 32) ^ c[3] ^ k[1], p0 & 0xffffffff]
            k = [(k[0] + W0) & 0xffffffff, (k[1] + W1) & 0xffffffff]
        return tuple(c)
    kat = [((0,) * 4, (0,) * 2, (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for c, k, want in kat:
        assert philox(c, k) == want


# ------------------------------------------------------------------ graph tracing / binding (no kernels are launched)
def _trace(model, method):
    from henbun_b200 import trace
    with trace.tracing():
        with model.tf_mode():
            return method.__wrapped__(model)


def test_tracer_recognises_the_gp_and_linear_operator_objectives():
    import henbun_b200 as hb
    import henbun_b200.tf as tf
    from henbun_b200 import fused
    rng = np.random.RandomState(0)
    X = rng.randn(20, 3); Y = rng.randn(20, 1)

    class GPR(hb.model.Model):
        def setUp(self, q_shape='diagonal'):
            self.X = hb.param.Data(X); self.Y = hb.param.Data(Y)
            self.q = hb.variationals.Gaussian(shape=[20, 1], q_shape=q_shape)
            self.kern = hb.gp.kernels.UnitRBF()
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            y_fit = tf.matmul(self.kern.Cholesky(self.X), self.q) * tf.sqrt(self.k_var)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, y_fit, self.var)) - self.KL()

        @hb.model.AutoOptimize()
        def ELBO_student(self):          # a graph with no whole-step entry point
            y_fit = tf.matmul(self.kern.Cholesky(self.X), self.q) * tf.sqrt(self.k_var)
            return tf.reduce_sum(hb.densities.student_t(self.Y, y_fit, self.var, 3.0)) - self.KL()

    for q_shape in ('diagonal', 'fullrank'):
        m = GPR(q_shape=q_shape)
        b = fused.bind(_trace(m, GPR.ELBO), m)
        assert type(b).__name__ == 'GpElboBinding'
        assert [v.long_name for v in b.var_order] == ['model.q.q_mu', 'model.q.q_sqrt', 'model.q.scale', 'model.kern.lengthscales',
                                                      'model.k_var', 'model.var']
    m = GPR()
    with pytest.raises(Exception):
        _trace(m, GPR.ELBO_student)                      # untraced op: compile() falls back to the eager tape
    assert m._tf_mode is False                           # tf_mode was left cleanly

    A = rng.randn(30, 8).astype(np.float32); y = rng.randn(30).astype(np.float32)

    class LO(hb.model.Model):
        def setUp(self):
            self.A = hb.param.Data(A); self.y = hb.param.Data(y)
            self.q = hb.variationals.Normal([8], q_shape='fullrank', stddev=0.1)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            f = tf.matmul(self.q, self.A, transpose_b=True)
            return tf.reduce_sum(hb.densities.gaussian(self.y, f, self.var)) - self.KL()

    m2 = LO()
    b2 = fused.bind(_trace(m2, LO.ELBO), m2)
    assert type(b2).__name__ == 'LinopElboBinding'
    assert [v.long_name for v in b2.var_order] == ['model.q.q_sqrt', 'model.q.q_mu', 'model.var']


def test_tracer_rejects_graphs_that_only_look_similar():
    import henbun_b200 as hb
    import henbun_b200.tf as tf
    from henbun_b200 import fused
    rng = np.random.RandomState(0)
    X = rng.randn(20, 3); Y = rng.randn(20, 1)

    class TwoQ(hb.model.Model):                          # a second variational contributes to KL(): not the fused graph
        def setUp(self):
            self.X = hb.param.Data(X); self.Y = hb.param.Data(Y)
            self.q = hb.variationals.Gaussian(shape=[20, 1])
            self.q2 = hb.variationals.Normal([3])
            self.kern = hb.gp.kernels.UnitRBF()
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            y_fit = tf.matmul(self.kern.Cholesky(self.X), self.q) * tf.sqrt(self.k_var)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, y_fit, self.var)) - self.KL()

    m = TwoQ()
    assert fused.bind(_trace(m, TwoQ.ELBO), m) is None

    class NoSqrt(hb.model.Model):                        # k_var instead of sqrt(k_var)
        def setUp(self):
            self.X = hb.param.Data(X); self.Y = hb.param.Data(Y)
            self.q = hb.variationals.Gaussian(shape=[20, 1])
            self.kern = hb.gp.kernels.UnitRBF()
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            y_fit = tf.matmul(self.kern.Cholesky(self.X), self.q) * self.k_var
            return tf.reduce_sum(hb.densities.gaussian(self.Y, y_fit, self.var)) - self.KL()

    m = NoSqrt()
    assert fused.bind(_trace(m, NoSqrt.ELBO), m) is None


def test_run_context_windows_of_one_philox_stream():
    """Ranks of a sample-sharded run read disjoint, contiguous windows whose union is the single-GPU draw."""
    from henbun_b200.variationals import RunContext
    per_sample, S, world = 1000, 8, 4
    single = RunContext(n_samples=S); single.total_samples = S
    o0 = single.take_sharded(per_sample)
    offs = []
    for r in range(world):
        c = RunContext(n_samples=S // world); c.first_sample, c.total_samples = r * (S // world), S
        offs.append(c.take_sharded(per_sample))
        assert c.offset == single.offset                  # every rank reserves the block of ALL samples
    assert offs == [o0 + r * (S // world) * per_sample for r in range(world)]
