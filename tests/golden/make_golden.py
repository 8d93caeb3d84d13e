#!/usr/bin/env python
"""Generate tests/golden/*.npz by executing the UNMODIFIED reference (a checkout of fujii-team/Henbun) on the
TF-1 shim of tests/golden/tf1_shim.py (TensorFlow itself is not installable here).

    HENBUN_REFERENCE=<checkout of fujii-team/Henbun> python tests/golden/make_golden.py

Every vector below is produced by the reference's own Python: its Variational sampler / KL, kernels,
Cholesky wrapper, NeuralNet, LOCAL feed routing, densities, transforms, the notebook models' ELBO,
tf.gradients of those graphs and tf.train.AdamOptimizer steps.  Inputs use the same seeds as the
reference's tests (np.random.RandomState(0)); eps is injected with feed_dict={variational.u: eps}.
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import tf1_shim  # noqa: E402

tf = tf1_shim.install()
sys.path.insert(0, os.environ["HENBUN_REFERENCE"])
warnings.simplefilter("ignore")
import Henbun as hb  # noqa: E402  (the reference)

LOCAL = hb.param.graph_key.LOCAL


def free_values(model):
    """{long_name: free-space value} of every global variable, in the reference's order."""
    out = {}
    for v in model.get_variables():
        if v.collections not in hb.param.graph_key.not_parameters:
            out[v.long_name] = np.array(model._session.run(v._tensor))
    return out


def grads_of(model, op, feed):
    vs = [v for v in model.get_variables() if v.collections not in hb.param.graph_key.not_parameters]
    g = tf.gradients(op, [v._tensor for v in vs])
    vals = model._session.run(g, feed_dict=feed)
    return {v.long_name: (np.zeros_like(model._session.run(v._tensor)) if gv is None else np.array(gv))
            for v, gv in zip(vs, vals)}


def save(name, **arrays):
    flat = {}
    for k, v in arrays.items():
        if isinstance(v, dict):
            for kk, vv in v.items():
                flat[k + "/" + kk] = np.asarray(vv)
        else:
            flat[k] = np.asarray(v)
    path = os.path.join(os.environ.get("HB_GOLDEN_OUT", HERE), name + ".npz")
    np.savez_compressed(path, **flat)
    print("wrote", path, {k: np.shape(v) for k, v in flat.items()})


# ------------------------------------------------------------------------------------------------
def golden_variationals():
    """testing/test_variationals.py:31-122 setup: Normal(10, n_layers=[3]) fullrank / diagonal."""
    rng = np.random.RandomState(0)
    sqrts = {'fullrank': rng.randn(3, 10, 10) * 0.5, 'diagonal': rng.randn(3, 10) * 0.5 - 0.5}
    for i in range(3):
        for j in range(10):
            sqrts['fullrank'][i, j, j] = np.exp(sqrts['fullrank'][i, j, j])
            for k in range(j + 1, 10):
                sqrts['fullrank'][i, j, k] = 0.
    x = rng.randn(3, 10) * 0.3
    u = rng.randn(3, 10)
    out = dict(x=x, u=u, sqrt_fullrank=sqrts['fullrank'], sqrt_diagonal=sqrts['diagonal'])
    for shape in ('fullrank', 'diagonal'):
        m = hb.model.Model()
        m.m = hb.variationals.Normal(x.shape[-1], n_layers=[3], q_shape=shape)
        m.m.q_mu = x
        m.m.q_sqrt = sqrts[shape]
        m.initialize()
        v = object.__getattribute__(m, 'm')
        with m.tf_mode():
            out['sample_' + shape] = m._session.run(v._sample(tf.convert_to_tensor(u)))
            out['logdet_' + shape] = m._session.run(v.logdet)
            out['kl_' + shape] = m._session.run(v.KL(), feed_dict={v.u: u})
            out['tensor_' + shape] = m._session.run(v.tensor(), feed_dict={v.u: u})
    save("variationals", **out)


def golden_local_feed():
    """LOCAL feed order / shapes (testing/test_variationals.py:166-203, test_param.py:117-124)."""
    rng = np.random.RandomState(0)
    m = hb.model.Model()
    m.v = hb.variationals.Normal([2, 3], n_layers=[4], collections=LOCAL)
    x = rng.randn(4, 7, 12)
    u = rng.randn(4, 7, 6)
    with m.tf_mode():
        m.v = tf.constant(x)
        v = object.__getattribute__(m, 'v')
        feed = {v.u: u}
        out = dict(x=x, u=u,
                   q_mu=m._session.run(v.q_mu), q_sqrt=m._session.run(v.q_sqrt),
                   sample=m._session.run(v.tensor(), feed_dict=feed),
                   logdet=m._session.run(v.logdet),
                   kl=m._session.run(v.KL(LOCAL), feed_dict=feed))
    save("local_feed", **out)


def golden_kernels():
    """testing/test_kernels.py:66-226 setup."""
    rng = np.random.RandomState(0)
    m = hb.model.Model()
    l1 = np.exp(rng.randn(1)); l2 = np.exp(rng.randn(2))
    m.k1 = hb.gp.kernels.UnitRBF(lengthscales=l1)
    m.k2 = hb.gp.kernels.UnitRBF(lengthscales=l2)
    m.k3 = hb.gp.kernels.UnitCsymRBF(lengthscales=l1)
    X = rng.randn(5, 2); X2 = rng.randn(6, 2); Xb = rng.randn(10, 5, 2); X2b = rng.randn(10, 6, 2)
    m.initialize()
    out = dict(l1=l1, l2=l2, X=X, X2=X2, Xb=Xb, X2b=X2b, jitter=hb.settings.numerics.jitter_level)
    run = m._session.run
    with m.tf_mode():
        for name, k in (('k1', m.k1), ('k2', m.k2), ('k3', m.k3)):
            out[name + '_K'] = run(k.K(X)); out[name + '_K2'] = run(k.K(X, X2))
            out[name + '_Kb'] = run(k.K(Xb)); out[name + '_K2b'] = run(k.K(Xb, X2b))
            out[name + '_Kdiag'] = run(k.Kdiag(X))
            out[name + '_chol'] = run(k.Cholesky(X)); out[name + '_cholb'] = run(k.Cholesky(Xb))
        out['sqdist_k2'] = run(m.k2.square_dist(X, X2))
        loss = tf.reduce_sum(m.k2.K(X, X2))
        out['grad_sumK2'] = grads_of(m, loss, {})
        loss = tf.reduce_sum(m.k1.Cholesky(X))
        out['grad_sumChol1'] = grads_of(m, loss, {})
    out['free'] = free_values(m)
    save("kernels", **out)


def golden_nn():
    """testing/test_nn.py:11-52."""
    rng = np.random.RandomState(0)
    tf.set_random_seed(0)
    m = hb.model.Model()
    m.nn = hb.nn.NeuralNet([3, 2, 4], n_layers=[5], neuron_types=tf.sigmoid)
    m.nn2 = hb.nn.NeuralNet([3, 2, 4, 5], n_layers=[6, 5], neuron_types=[tf.nn.sigmoid, tf.nn.relu])
    m.initialize()
    x1 = rng.randn(5, 6, 3); x2 = rng.randn(6, 5, 6, 3)
    with m.tf_mode():
        y1 = m._session.run(m.nn(tf.constant(x1)))
        y2 = m._session.run(m.nn2(tf.constant(x2)))
        loss = tf.reduce_sum(tf.square(m.nn(tf.constant(x1))))
        g = grads_of(m, loss, {})
    save("nn", x1=x1, x2=x2, y1=y1, y2=y2, free=free_values(m), grad_sumsq_y1=g)


def golden_densities_transforms():
    rng = np.random.RandomState(0)
    a = rng.randn(2, 3, 4); mu = rng.randn(2, 3, 4); var = np.exp(rng.randn(2, 3, 4))
    xs = rng.randn(10)
    with tf.Session() as sess:
        g1 = sess.run(hb.densities.gaussian(tf.constant(a), 0.0, 2.0))
        g2 = sess.run(hb.densities.gaussian(tf.constant(a), tf.constant(mu), tf.constant(var)))
        st = sess.run(hb.densities.student_t(tf.constant(a), tf.constant(mu), tf.constant(np.sqrt(var)), 3.0))
        t = hb.transforms.Log1pe()
        fw = sess.run(t.tf_forward(tf.constant(xs))); lj = sess.run(t.tf_log_jacobian(tf.constant(xs)))
        lg = hb.transforms.Logistic(7.3, 19.4)
        fwl = sess.run(lg.tf_forward(tf.constant(xs))); ljl = sess.run(lg.tf_log_jacobian(tf.constant(xs)))
        ex = hb.transforms.Exp()
        fwe = sess.run(ex.tf_forward(tf.constant(xs)))
    save("densities_transforms", a=a, mu=mu, var=var, gauss_scalar=g1, gauss_tensor=g2, student_t3=st, xs=xs,
         log1pe_fwd=fw, log1pe_logjac=lj, log1pe_np_fwd=t.forward(xs), log1pe_np_bwd=t.backward(t.forward(xs)),
         logistic_fwd=fwl, logistic_logjac=ljl, exp_fwd=fwe)


def golden_densities_all():
    """Every non-Gaussian density of Henbun/densities.py:30-103 and its tf.gradients w.r.t. each tensor
    argument (d sum(w * logp) with a fixed random weighting w, so that every element's derivative is pinned)."""
    rng = np.random.RandomState(0)
    shp = (3, 5, 4)
    pos = lambda *s: np.exp(0.5 * rng.randn(*s))
    cases = {
        # name: (function, [argument arrays in the reference's order])
        "lognormal": (hb.densities.lognormal, [pos(*shp), rng.randn(5, 4), pos(4)]),
        "bernoulli": (hb.densities.bernoulli, [rng.uniform(0.05, 0.95, shp), (rng.rand(*shp) < 0.5).astype(np.float64)]),
        "poisson": (hb.densities.poisson, [pos(*shp), rng.poisson(3.0, shp).astype(np.float64)]),
        "exponential": (hb.densities.exponential, [pos(5, 4), pos(*shp)]),
        "gamma": (hb.densities.gamma, [pos(4) + 0.5, pos(5, 4), pos(*shp)]),
        "student_t": (hb.densities.student_t, [rng.randn(*shp), rng.randn(5, 4), pos(4), pos(*shp) * 3.0]),
        "beta": (hb.densities.beta, [pos(5, 4) + 0.5, pos(4) + 0.5,
                                     np.concatenate([rng.uniform(0.02, 0.98, (3, 5, 3)), np.array([0.0, 1.0, 0.5] * 5).reshape(3, 5, 1)], -1)]),
        "laplace": (hb.densities.laplace, [rng.randn(5, 4), pos(4), rng.randn(*shp)]),
        "bimixture": (hb.densities.bimixture, [rng.uniform(0.05, 0.95, (5, 4)), rng.randn(*shp) * 3, rng.randn(*shp) * 3]),
    }
    out = {}
    with tf.Session() as sess:
        for name, (fn, args) in cases.items():
            w = rng.randn(*shp)
            ts = [tf.constant(a) for a in args]
            val = fn(*ts)
            out[name + "/out"] = sess.run(val)
            out[name + "/w"] = w
            gs = sess.run(tf.gradients(tf.reduce_sum(val * tf.constant(w)), ts))
            for i, (a, g) in enumerate(zip(args, gs)):
                out[f"{name}/arg{i}"] = a
                out[f"{name}/grad{i}"] = np.zeros_like(a) if g is None else np.asarray(g)
    save("densities_all", **out)


def _gpr_class(X, Y, q_shape):
    class GPR(hb.model.Model):                 # notebooks/GaussianProcess.ipynb:109-148, verbatim structure
        def setUp(self):
            self.X = hb.param.Data(X)
            self.Y = hb.param.Data(Y)
            self.q = hb.variationals.Gaussian(shape=X.shape[:1] + (1,), q_shape=q_shape)
            self.kern = hb.gp.kernels.UnitRBF()
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO_gaussian(self):
            y_fit = tf.matmul(self.kern.Cholesky(self.X), self.q) * tf.sqrt(self.k_var)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, y_fit, self.var)) - self.KL()
    return GPR


def golden_gpr():
    """ELBO, all gradients and a 5-step Adam trajectory of the GaussianProcess.ipynb model, S one-sample
    evaluations with injected eps (mean over S = the S-sample ELBO of BASELINE.json)."""
    for tag, n, D, q_shape, jitter, S in (("c1_fullrank", 40, 1, 'fullrank', 1e-3, 4), ("c3_diag", 64, 8, 'diagonal', 1e-5, 4)):
        rng = np.random.RandomState(0)
        tf.set_random_seed(0)
        if D == 1:
            X = np.linspace(0, 6, n).reshape(-1, 1); Y = np.sin(X) + rng.randn(n, 1) * 0.3
        else:
            X = rng.randn(n, D); Y = np.sin(X.sum(1, keepdims=True) / np.sqrt(D)) + 0.1 * rng.randn(n, 1)
        cfg = hb.settings.get_settings(); cfg.numerics.jitter_level = jitter
        m = _gpr_class(X, Y, q_shape)()
        if q_shape == 'fullrank':      # a sane full-rank start (the default init has every entry ~ stddev)
            m.q.q_sqrt = 0.3 * np.eye(n) + 0.02 * np.tril(rng.randn(n, n))
        with hb.settings.temp_settings(cfg):
            m.ELBO_gaussian().compile(tf.train.AdamOptimizer(0.01))
        opt = m.ELBO_gaussian()
        free0 = free_values(m)
        U = rng.randn(S, n, 1)
        q = object.__getattribute__(m, 'q')
        elbos, grads = [], None
        for s in range(S):
            feed = dict(m.get_feed_dict()); feed[q.u] = U[s].reshape(-1)
            elbos.append(m._session.run(opt.method_op, feed_dict=feed))
            g = grads_of(m, opt.method_op, feed)
            grads = g if grads is None else {k: grads[k] + g[k] for k in g}
        grads = {k: v / S for k, v in grads.items()}
        # Adam trajectory: 5 reference steps, one sample per step (exactly what Optimizer.optimize does)
        Ua = rng.randn(5, n, 1)
        for t in range(5):
            feed = dict(m.get_feed_dict()); feed[q.u] = Ua[t].reshape(-1)
            m._session.run(opt.optimize_op, feed_dict=feed)
        save("gpr_" + tag, X=X, Y=Y, U=U, jitter=jitter, elbo_per_sample=np.array(elbos), elbo_mean=np.mean(elbos),
             free=free0, grad_mean=grads, U_adam=Ua, free_after_5_adam=free_values(m), adam_lr=0.01)


def golden_amortised():
    """Encoder -> LOCAL Normal -> decoder model (BASELINE config 4 at toy size) on the reference."""
    rng = np.random.RandomState(0)
    tf.set_random_seed(0)
    Xall = rng.randn(50, 6)

    class Amortised(hb.model.Model):
        def setUp(self):
            self.X = hb.param.MinibatchData(Xall)
            self.enc = hb.nn.NeuralNet([6, 5, 2 * 3], stddev=0.3)
            self.dec = hb.nn.NeuralNet([3, 5, 6], stddev=0.3)
            self.q_local = hb.variationals.Normal([3], collections=LOCAL)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            self.q_local = self.enc(self.X)
            x_rec = self.dec(self.q_local)
            return tf.reduce_sum(hb.densities.gaussian(self.X, x_rec, self.var)) - self.KL(LOCAL)

    m = Amortised()
    m.ELBO().compile()
    opt = m.ELBO()
    idx = np.arange(8) * 5
    S = 3
    U = rng.randn(S, 8, 3)
    ql = object.__getattribute__(m, 'q_local')
    free0 = free_values(m)
    elbos, grads = [], None
    for s in range(S):
        feed = dict(m.get_feed_dict(idx)); feed[ql.u] = U[s]
        elbos.append(m._session.run(opt.method_op, feed_dict=feed))
        g = grads_of(m, opt.method_op, feed)
        grads = g if grads is None else {k: grads[k] + g[k] for k in g}
    grads = {k: v / S for k, v in grads.items()}
    save("amortised", Xall=Xall, idx=idx, U=U, elbo_per_sample=np.array(elbos), elbo_mean=np.mean(elbos), free=free0,
         grad_mean=grads)


def golden_expert_gpr():
    """notebooks/Expert_GPR.ipynb:101-149 (ELBO) at N=30, one sample."""
    rng = np.random.RandomState(0)
    tf.set_random_seed(0)
    n = 30
    X = np.linspace(0, 6, n).reshape(-1, 1)
    Y = np.sin(0.1 * X * X * X) + rng.randn(*X.shape) * 0.1

    class ExpertGPR(hb.model.Model):
        def setUp(self):
            self.X = hb.param.Data(X)
            self.Y = hb.param.Data(Y)
            self.q_s = hb.variationals.Gaussian(shape=X.shape, q_shape='fullrank')
            self.q_l = hb.variationals.Gaussian(shape=X.shape, q_shape='fullrank')
            self.q_r = hb.variationals.Gaussian(shape=X.shape, q_shape='fullrank')
            self.kern_s = hb.gp.kernels.UnitRBF(np.ones(1) * 0.2)
            self.kern_l = hb.gp.kernels.UnitRBF(np.ones(1) * 1)
            self.kern_r = hb.gp.kernels.UnitRBF(np.ones(1) * 1)
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.k_var_r = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            self.f_s = tf.matmul(self.kern_s.Cholesky(self.X), self.q_s)
            self.f_l = tf.matmul(self.kern_l.Cholesky(self.X), self.q_l)
            self.f_r = tf.matmul(self.kern_r.Cholesky(self.X), self.q_r) * tf.sqrt(self.k_var_r)
            fraction = tf.sigmoid(self.f_r)
            self.f = (fraction * self.f_s + (1 - fraction) * self.f_l) * self.k_var
            return tf.reduce_sum(hb.densities.gaussian(self.Y, self.f, self.var)) - self.KL()

    m = ExpertGPR()
    for nm in ('q_s', 'q_l', 'q_r'):
        getattr(m, nm).q_sqrt = 0.3 * np.eye(n) + 0.02 * np.tril(rng.randn(n, n))
    cfg = hb.settings.get_settings(); cfg.numerics.jitter_level = 3.0e-4          # Expert_GPR.ipynb:203
    with hb.settings.temp_settings(cfg):
        m.ELBO().compile()
    opt = m.ELBO()
    U = {nm: rng.randn(n) for nm in ('q_s', 'q_l', 'q_r')}
    feed = dict(m.get_feed_dict())
    for nm in U:
        feed[object.__getattribute__(m, nm).u] = U[nm]
    save("expert_gpr", X=X, Y=Y, U=U, jitter=3.0e-4, elbo=m._session.run(opt.method_op, feed_dict=feed),
         free=free_values(m), grad=grads_of(m, opt.method_op, feed))


if __name__ == "__main__":
    golden_variationals()
    golden_local_feed()
    golden_kernels()
    golden_nn()
    golden_densities_transforms()
    golden_densities_all()
    golden_gpr()
    golden_amortised()
    golden_expert_gpr()
