"""Pin the oracle: every function of oracle/henbun_oracle.py is checked against the vectors in
tests/golden/*.npz, which were produced by executing the UNMODIFIED reference on the TF-1 shim
(tests/golden/make_golden.py).  CPU only."""
import os

import numpy as np
import torch

from oracle import henbun_oracle as O

G = os.path.join(os.path.dirname(__file__), "golden")
T = lambda a: torch.tensor(np.asarray(a, dtype=np.float64))


def load(name):
    d = np.load(os.path.join(G, name + ".npz"))
    out, nested = {}, {}
    for k in d.files:
        if "/" in k:
            a, b = k.split("/", 1)
            nested.setdefault(a, {})[b] = d[k]
        else:
            out[k] = d[k]
    out.update(nested)
    return out


def test_sampler_logdet_kl():
    g = load("variationals")
    x, u = T(g["x"]), T(g["u"])
    z = O.sample_fullrank(x, T(g["sqrt_fullrank"]), u)
    assert np.allclose(z.numpy(), g["sample_fullrank"], rtol=1e-12, atol=1e-12)
    assert np.allclose(O.logdet_fullrank(T(g["sqrt_fullrank"])).numpy(), g["logdet_fullrank"], atol=1e-12)
    assert np.allclose(O.kl_normal(O.logdet_fullrank(T(g["sqrt_fullrank"])), u, z).item(), g["kl_fullrank"], rtol=1e-12)
    z = O.sample_diag(x, T(g["sqrt_diagonal"]), u)
    assert np.allclose(z.numpy(), g["sample_diagonal"], rtol=1e-12, atol=1e-12)
    assert np.allclose(O.logdet_diag(T(g["sqrt_diagonal"])).numpy(), g["logdet_diagonal"], atol=1e-12)
    assert np.allclose(O.kl_normal(O.logdet_diag(T(g["sqrt_diagonal"])), u, z).item(), g["kl_diagonal"], rtol=1e-12)
    assert np.allclose(g["tensor_diagonal"], g["sample_diagonal"])


def test_local_feed_split_order():
    g = load("local_feed")
    mu, om = O.local_feed_split(T(g["x"]), [6, 6])
    assert np.array_equal(mu.numpy(), g["q_mu"]) and np.array_equal(om.numpy(), g["q_sqrt"])
    z = O.sample_diag(mu, om, T(g["u"]))
    assert np.allclose(z.numpy().reshape(4, 7, 2, 3), g["sample"], rtol=1e-12)
    assert np.allclose(O.kl_normal(O.logdet_diag(om), T(g["u"]), z).item(), g["kl"], rtol=1e-12)


def test_kernels_and_cholesky():
    g = load("kernels")
    j = float(g["jitter"])
    for name, ell, fn in (("k1", g["l1"], O.rbf_K), ("k2", g["l2"], O.rbf_K), ("k3", g["l1"], O.csym_rbf_K)):
        ell = T(ell)
        assert np.allclose(fn(T(g["X"]), ell).numpy(), g[name + "_K"], atol=1e-12)
        assert np.allclose(fn(T(g["X"]), ell, T(g["X2"])).numpy(), g[name + "_K2"], atol=1e-12)
        assert np.allclose(fn(T(g["Xb"]), ell).numpy(), g[name + "_Kb"], atol=1e-12)
        assert np.allclose(fn(T(g["Xb"]), ell, T(g["X2b"])).numpy(), g[name + "_K2b"], atol=1e-12)
        assert np.allclose(O.kern_cholesky(T(g["X"]), ell, j, fn).numpy(), g[name + "_chol"], atol=1e-10)
        assert np.allclose(O.kern_cholesky(T(g["Xb"]), ell, j, fn).numpy(), g[name + "_cholb"], atol=1e-10)
    assert np.allclose(O.Kdiag(T(g["X"])).numpy(), g["k1_Kdiag"])
    assert np.allclose(O.square_dist(T(g["X"]), T(g["l2"]), T(g["X2"])).numpy(), g["sqdist_k2"], atol=1e-12)
    # gradients through the positive transform (lengthscale free variable)
    f2 = torch.tensor(g["free"]["model.k2.lengthscales"], requires_grad=True)
    O.rbf_K(T(g["X"]), O.log1pe_forward(f2), T(g["X2"])).sum().backward()
    assert np.allclose(f2.grad.numpy(), g["grad_sumK2"]["model.k2.lengthscales"], rtol=1e-10)
    f1 = torch.tensor(g["free"]["model.k1.lengthscales"], requires_grad=True)
    O.kern_cholesky(T(g["X"]), O.log1pe_forward(f1), j).sum().backward()
    assert np.allclose(f1.grad.numpy(), g["grad_sumChol1"]["model.k1.lengthscales"], rtol=1e-8)


def test_cholesky_reverse_mode_matches_reference_gradient():
    """The recursive reverse-mode Cholesky the CUDA host code follows reproduces the reference's
    d sum(chol(K+jI)) / d lengthscale."""
    g = load("kernels")
    j = float(g["jitter"]); X = g["X"]
    free = g["free"]["model.k1.lengthscales"]
    ell = np.logaddexp(0, free) + 1e-6
    K = O.rbf_K(T(X), T(ell)).numpy()
    L = np.linalg.cholesky(K + j * np.eye(5))
    Gm = O.chol_rev_recursive(L, np.tril(np.ones((5, 5))), nb=2)
    D2 = ((X[:, None, :] - X[None, :, :]) ** 2).sum(-1)
    g_ell = np.sum(Gm * K * D2) / ell[0] ** 3
    g_free = g_ell / (1 + np.exp(-free[0]))
    assert np.allclose(g_free, g["grad_sumChol1"]["model.k1.lengthscales"][0], rtol=1e-8)


def test_neural_net():
    g = load("nn")
    f = {k: T(v) for k, v in g["free"].items()}
    y1 = O.neural_net(T(g["x1"]), [f["model.nn.matbias0.w"], f["model.nn.matbias1.w"]],
                      [f["model.nn.matbias0.b"], f["model.nn.matbias1.b"]], ["sigmoid"])
    assert np.allclose(y1.numpy(), g["y1"], atol=1e-12)
    y2 = O.neural_net(T(g["x2"]), [f[f"model.nn2.matbias{i}.w"] for i in range(3)],
                      [f[f"model.nn2.matbias{i}.b"] for i in range(3)], ["sigmoid", "relu"])
    assert np.allclose(y2.numpy(), g["y2"], atol=1e-12)
    leaves = {k: T(v).requires_grad_(True) for k, v in g["free"].items() if k.startswith("model.nn.")}
    y = O.neural_net(T(g["x1"]), [leaves["model.nn.matbias0.w"], leaves["model.nn.matbias1.w"]],
                     [leaves["model.nn.matbias0.b"], leaves["model.nn.matbias1.b"]], ["sigmoid"])
    (y ** 2).sum().backward()
    for k, v in leaves.items():
        assert np.allclose(v.grad.numpy(), g["grad_sumsq_y1"][k], rtol=1e-10, atol=1e-12)


def test_all_densities_and_their_gradients():
    """Every density of densities.py:30-103 and tf.gradients of it, as the unmodified reference computed them."""
    d = np.load(os.path.join(G, "densities_all.npz"))
    for name, fn in O.DENSITIES.items():
        if name == "gaussian":
            continue
        n_args = len([k for k in d.files if k.startswith(name + "/arg")])
        args = [torch.tensor(d[f"{name}/arg{i}"], dtype=torch.float64, requires_grad=True) for i in range(n_args)]
        out = fn(*args)
        assert np.allclose(out.detach().numpy(), d[name + "/out"], rtol=1e-12, atol=1e-12), name
        (out * torch.tensor(d[name + "/w"])).sum().backward()
        for i, a in enumerate(args):
            got = np.zeros_like(d[f"{name}/grad{i}"]) if a.grad is None else a.grad.numpy()
            assert np.allclose(got, d[f"{name}/grad{i}"], rtol=1e-10, atol=1e-12), (name, i)


def test_densities_and_transforms():
    g = load("densities_transforms")
    assert np.allclose(O.gaussian(T(g["a"]), T(0.0), T(2.0)).numpy(), g["gauss_scalar"], atol=1e-12)
    assert np.allclose(O.gaussian(T(g["a"]), T(g["mu"]), T(g["var"])).numpy(), g["gauss_tensor"], atol=1e-12)
    assert np.allclose(O.student_t(T(g["a"]), T(g["mu"]), np.sqrt(g["var"]), 3.0).numpy(), g["student_t3"], atol=1e-12)
    xs = T(g["xs"])
    assert np.allclose(O.log1pe_forward(xs).numpy(), g["log1pe_fwd"], atol=1e-12)
    assert np.allclose(O.log1pe_log_jacobian(xs).item(), g["log1pe_logjac"], rtol=1e-12)
    assert np.allclose(O.log1pe_backward(g["log1pe_np_fwd"]), g["xs"], atol=1e-8)
    assert np.allclose(O.logistic_forward(xs, 7.3, 19.4).numpy(), g["logistic_fwd"], atol=1e-12)
    assert np.allclose(O.logistic_log_jacobian(xs, 7.3, 19.4).item(), g["logistic_logjac"], rtol=1e-12)
    assert np.allclose(O.exp_forward(xs).numpy(), g["exp_fwd"], atol=1e-12)


def gpr_params(free, n, full):
    return dict(q_mu=free["model.q.q_mu"].reshape(n), q_sqrt=free["model.q.q_sqrt"].reshape((n, n) if full else (n,)),
                scale=free["model.q.scale"].reshape(1), lengthscales=free["model.kern.lengthscales"].reshape(-1),
                k_var=free["model.k_var"].reshape(1), var=free["model.var"].reshape(1))


GPR_KEYS = {"q_mu": "model.q.q_mu", "q_sqrt": "model.q.q_sqrt", "scale": "model.q.scale",
            "lengthscales": "model.kern.lengthscales", "k_var": "model.k_var", "var": "model.var"}


def test_gpr_elbo_gradients_and_adam_trajectory():
    for tag, full in (("c1_fullrank", True), ("c3_diag", False)):
        g = load("gpr_" + tag)
        n = g["X"].shape[0]
        p = gpr_params(g["free"], n, full)
        qs = "fullrank" if full else "diagonal"
        fn = lambda pp, *a: O.gpr_elbo(pp, *a, q_shape=qs, jitter=float(g["jitter"]))
        U = g["U"][:, :, 0]
        for s in range(U.shape[0]):         # the reference's one-sample ELBO, sample by sample
            v, _ = O.value_and_grads(fn, p, g["X"], g["Y"][:, 0], U[s:s + 1])
            assert np.allclose(v, g["elbo_per_sample"][s], rtol=1e-10)
        v, gr = O.value_and_grads(fn, p, g["X"], g["Y"][:, 0], U)
        assert np.allclose(v, g["elbo_mean"], rtol=1e-10)
        for k, name in GPR_KEYS.items():
            assert np.allclose(gr[k].ravel(), g["grad_mean"][name].ravel(), rtol=1e-7, atol=1e-9), (tag, k)
        if not full:                      # closed-form backward (the CUDA blueprint) on the reference's numbers
            v2, g2 = O.gpr_elbo_closed_form_grads(p, g["X"], g["Y"][:, 0], U, jitter=float(g["jitter"]))
            assert np.allclose(v2, g["elbo_mean"], rtol=1e-10)
            for k, name in GPR_KEYS.items():
                assert np.allclose(g2[k].ravel(), g["grad_mean"][name].ravel(), rtol=1e-7, atol=1e-9), (tag, k)
        # 5 reference Adam steps (tf.train.AdamOptimizer(0.01).minimize(-ELBO)), one sample per step
        mom = {k: np.zeros_like(v) for k, v in p.items()}; vel = {k: np.zeros_like(v) for k, v in p.items()}
        for t in range(5):
            _, gr = O.value_and_grads(fn, p, g["X"], g["Y"][:, 0], g["U_adam"][t, :, 0][None, :])
            for k in p:
                p[k], mom[k], vel[k] = O.adam_tf1_step(p[k], -gr[k], mom[k], vel[k], t + 1, lr=float(g["adam_lr"]))
        for k, name in GPR_KEYS.items():
            assert np.allclose(p[k].ravel(), g["free_after_5_adam"][name].ravel(), rtol=1e-8, atol=1e-10), (tag, k)


def test_amortised_model():
    g = load("amortised")
    f = g["free"]
    p = {"var": f["model.var"]}
    for i in range(2):
        p[f"enc.w{i}"] = f[f"model.enc.matbias{i}.w"]; p[f"enc.b{i}"] = f[f"model.enc.matbias{i}.b"]
        p[f"dec.w{i}"] = f[f"model.dec.matbias{i}.w"]; p[f"dec.b{i}"] = f[f"model.dec.matbias{i}.b"]
    Xmb = g["Xall"][g["idx"]]
    fn = lambda pp, X_, U_: O.amortised_elbo(pp, X_, U_, ["sigmoid"], ["sigmoid"])
    v, gr = O.value_and_grads(fn, p, Xmb, g["U"])
    assert np.allclose(v, g["elbo_mean"], rtol=1e-10)
    assert np.allclose(gr["var"], g["grad_mean"]["model.var"], rtol=1e-8)
    for i in range(2):
        assert np.allclose(gr[f"enc.w{i}"], g["grad_mean"][f"model.enc.matbias{i}.w"], rtol=1e-7, atol=1e-10)
        assert np.allclose(gr[f"dec.b{i}"], g["grad_mean"][f"model.dec.matbias{i}.b"], rtol=1e-7, atol=1e-10)


def test_expert_gpr_model():
    g = load("expert_gpr")
    f = g["free"]; n = g["X"].shape[0]
    p = {"k_var": f["model.k_var"], "k_var_r": f["model.k_var_r"], "var": f["model.var"]}
    for nm in ("s", "l", "r"):
        p[f"q_{nm}.q_mu"] = f[f"model.q_{nm}.q_mu"].reshape(n)
        p[f"q_{nm}.q_sqrt"] = f[f"model.q_{nm}.q_sqrt"].reshape(n, n)
        p[f"q_{nm}.scale"] = f[f"model.q_{nm}.scale"].reshape(1)
        p[f"kern_{nm}.lengthscales"] = f[f"model.kern_{nm}.lengthscales"]
    U3 = {nm: g["U"]["q_" + nm][None, :] for nm in ("s", "l", "r")}
    v, gr = O.value_and_grads(lambda pp, X_, Y_, U_: O.expert_gpr_elbo(pp, X_, Y_, U_, jitter=float(g["jitter"])), p,
                              g["X"], g["Y"][:, 0], U3)
    assert np.allclose(v, g["elbo"], rtol=1e-10)
    for k in p:
        assert np.allclose(gr[k].ravel(), g["grad"]["model." + k].ravel(), rtol=1e-6, atol=1e-9), k


def test_golden_vectors_regenerate_from_the_reference(tmp_path):
    """The committed vectors are exactly what the UNMODIFIED reference (the checkout of fujii-team/Henbun that
    HENBUN_REFERENCE names, on the TF-1 shim) produces: re-run the generator into a scratch directory and compare array by
    array.  Skipped when no reference checkout is named."""
    import subprocess
    import sys
    import pytest
    ref = os.environ.get("HENBUN_REFERENCE")
    if not ref or not os.path.isdir(os.path.join(ref, "Henbun")):
        pytest.skip("no reference checkout: set HENBUN_REFERENCE to a checkout of fujii-team/Henbun")
    env = dict(os.environ, HB_GOLDEN_OUT=str(tmp_path))
    subprocess.run([sys.executable, os.path.join(G, "make_golden.py")], check=True, env=env, stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL, timeout=600)
    names = sorted(f for f in os.listdir(G) if f.endswith(".npz"))
    assert names and sorted(f for f in os.listdir(tmp_path) if f.endswith(".npz")) == names
    for f in names:
        a, b = np.load(os.path.join(G, f)), np.load(os.path.join(tmp_path, f))
        assert set(a.files) == set(b.files), f
        for k in a.files:
            assert np.array_equal(a[k], b[k]), (f, k)
