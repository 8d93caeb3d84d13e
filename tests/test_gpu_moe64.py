"""float64 mixture-of-experts GP regression (csrc/moe64.cu, BASELINE config 2 = notebooks/Expert_GPR.ipynb:101-149):
hb_moe_gp_elbo_step_f64 against the unmodified reference's vectors and the fp64 oracle at the named size, its Philox route,
its repeatability, its non-positive-pivot flag, and the float64 route through the model API (fused.MixtureGpElboBinding)
against the eager fp32 tape and against the oracle's Adam trajectory."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import henbun_oracle as O

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
ROLES = ("s", "l", "r")


@pytest.fixture(scope="module")
def lib():
    from henbun_b200 import _lib
    return _lib.load()


def P(t):
    from henbun_b200._lib import ptr
    return ptr(t)


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64).cuda()


def rel_err(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def blocks(p):
    """(oracle key, size) in the entry point's packing"""
    keys = []
    for nm in ROLES:
        keys += [f"q_{nm}.q_mu", f"q_{nm}.q_sqrt", f"q_{nm}.scale", f"kern_{nm}.lengthscales"]
    return [(k, np.asarray(p[k]).size) for k in keys + ["k_var", "k_var_r", "var"]]


def pack(p):
    return np.concatenate([np.asarray(p[k], np.float64).ravel() for k, _ in blocks(p)])


def run_moe(lib, X, Y, p, U3, q_shapes, jitter, S, seed=0, offsets=(0, 0, 0), adam_t=None, check_err=True):
    from henbun_b200 import _lib
    n, D = X.shape
    full = [1 if q == "fullrank" else 0 for q in q_shapes]
    n_ell = [np.asarray(p[f"kern_{nm}.lengthscales"]).size for nm in ROLES]
    cfg = _lib.MoeGpConfig(n, D, S, (C.c_int * 3)(*n_ell), (C.c_int * 3)(*full), jitter, seed, (C.c_ulonglong * 3)(*offsets))
    npar = lib.hb_moe_gp_param_count(C.byref(cfg))
    params = dev(pack(p))
    assert params.numel() == npar
    grads, out4 = torch.zeros(npar, dtype=torch.float64, device="cuda"), torch.zeros(4, dtype=torch.float64, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    wsb = lib.hb_moe_gp_f64_workspace_bytes(C.byref(cfg))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    Xd, Yd = dev(X), dev(np.asarray(Y).reshape(-1))
    eps = [None if U3 is None else dev(U3[nm]) for nm in ROLES]
    m = v = acfg = None
    if adam_t is not None:
        m, v = torch.zeros_like(params), torch.zeros_like(params)
        acfg = C.byref(_lib.AdamConfig(0.01, 0.9, 0.999, 1e-8, -1.0, None, adam_t))
    rc = lib.hb_moe_gp_elbo_step_f64(C.byref(cfg), P(Xd), P(Yd), P(params), P(eps[0]), P(eps[1]), P(eps[2]), P(grads), P(out4),
                                     P(m), P(v), acfg, P(ws), wsb, P(err), _lib.stream())
    torch.cuda.synchronize()
    assert rc == 0
    if check_err:
        assert err.item() == 0
    return out4.cpu().numpy(), grads.cpu().numpy(), params.cpu().numpy(), err.item()


def oracle(p, X, Y, U3, q_shapes, jitter, device="cuda"):
    fn = lambda pp, X_, Y_, U_: O.expert_gpr_elbo(pp, X_, Y_, U_, q_shapes=q_shapes, jitter=jitter)
    return O.value_and_grads(fn, p, X, np.asarray(Y).reshape(-1), U3, device=device)


def block_errors(grads, gref, p):
    out, off = {}, 0
    for k, sz in blocks(p):
        out[k] = rel_err(grads[off:off + sz], np.asarray(gref[k]).ravel())
        off += sz
    return out


def test_against_the_reference_vectors(lib):
    """tests/golden/expert_gpr.npz: the unmodified reference in fp64 at N = 30, one sample, full-rank q everywhere (its r^2
    expansion changes the fp64 oracle by 5e-15 on the ELBO and 1.1e-12 on the gradients, well inside the bars)."""
    d = np.load(os.path.join(G, "expert_gpr.npz"))
    X, Y, n = d["X"], d["Y"], d["X"].shape[0]
    p = {}
    for nm in ROLES:
        p[f"q_{nm}.q_mu"] = d[f"free/model.q_{nm}.q_mu"].reshape(n)
        p[f"q_{nm}.q_sqrt"] = d[f"free/model.q_{nm}.q_sqrt"].reshape(n, n)
        p[f"q_{nm}.scale"] = d[f"free/model.q_{nm}.scale"].reshape(1)
        p[f"kern_{nm}.lengthscales"] = d[f"free/model.kern_{nm}.lengthscales"].reshape(-1)
    for k in ("k_var", "k_var_r", "var"):
        p[k] = d["free/model." + k].reshape(1)
    U3 = {nm: d[f"U/q_{nm}"].reshape(1, n) for nm in ROLES}
    out4, grads, _, _ = run_moe(lib, X, Y, p, U3, ("fullrank",) * 3, float(d["jitter"]), 1)
    ref = float(d["elbo"])
    e_val = abs(out4[0] - ref) / abs(ref)
    gref = {k: d["grad/model." + k] for k, _ in blocks(p)}
    errs = block_errors(grads, gref, p)
    print(f"N=30 vs the reference: ELBO {e_val:.1e}, gradient blocks", {k: f"{e:.1e}" for k, e in errs.items()})
    assert e_val <= 1e-10
    for k, e in errs.items():
        assert e <= 1e-8, (k, e)


def notebook_problem(n, S, q_shapes, seed=0):
    """Expert_GPR.ipynb:56-57 input (X = linspace(0, 6, n), Y = sin(0.1 X^3) + 0.1 eps), lengthscales (0.2, 1, 1)."""
    rng = np.random.RandomState(seed)
    X = np.linspace(0, 6, n).reshape(-1, 1)
    Y = np.sin(0.1 * X ** 3) + 0.1 * rng.randn(n, 1)
    p = {}
    for nm, qs, ell in zip(ROLES, q_shapes, (0.2, 1.0, 1.0)):
        p[f"q_{nm}.q_mu"] = 0.1 * rng.randn(n)
        p[f"q_{nm}.q_sqrt"] = (np.log(0.3) + 0.1 * rng.randn(n) if qs == "diagonal"
                               else 0.3 * np.eye(n) + (0.2 / np.sqrt(n)) * np.tril(rng.randn(n, n)))
        p[f"q_{nm}.scale"] = np.array([float(O.log1pe_backward(1.0)) + 0.1 * rng.randn()])
        p[f"kern_{nm}.lengthscales"] = np.array([float(O.log1pe_backward(ell))])
    p["k_var"] = np.array([0.5]); p["k_var_r"] = np.array([0.3]); p["var"] = np.array([-2.0])
    U3 = {nm: rng.randn(S, n) for nm in ROLES}
    return X, Y, p, U3


@pytest.mark.parametrize("q_shapes", [("fullrank", "fullrank", "diagonal"), ("fullrank", "fullrank", "fullrank")])
def test_named_size_meets_the_parity_bar(lib, q_shapes):
    """N = 2000, S = 4, jitter 3e-4 (cond(K + 3e-4 I) ~ 2.5e6 for the l = 1 kernels): the ELBO and every gradient block
    within 1e-5 of the fp64 oracle, where the fp32 tape is held to 0.023."""
    n, S, jitter = 2000, 4, 3e-4
    X, Y, p, U3 = notebook_problem(n, S, q_shapes)
    val, gref = oracle(p, X, Y, U3, q_shapes, jitter)
    out4, grads, _, _ = run_moe(lib, X, Y, p, U3, q_shapes, jitter, S)
    e_val = abs(out4[0] - val) / abs(val)
    errs = block_errors(grads, gref, p)
    print(f"config 2 in fp64 {q_shapes}: ELBO {e_val:.1e}, gradient blocks", {k: f"{e:.1e}" for k, e in errs.items()})
    assert e_val <= 1e-5
    for k, e in errs.items():
        assert e <= 1e-5, (k, e)


def test_ard_lengthscales_per_expert(lib):
    """D = 3 with one lengthscale for expert s and one per dimension for l and the gate r (n_ell = 1, 3, 3): each expert's
    lengthscale slots, Gram backward partial sums and gradient blocks against the fp64 oracle."""
    rng = np.random.RandomState(7)
    n, D, S, jitter = 400, 3, 4, 1e-2
    q_shapes = ("diagonal", "fullrank", "diagonal")
    X = rng.randn(n, D); Y = np.sin(X.sum(1, keepdims=True)) + 0.1 * rng.randn(n, 1)
    p = {}
    for nm, qs, ell in zip(ROLES, q_shapes, ([0.7], [0.5, 1.0, 2.0], [1.5, 0.8, 1.2])):
        p[f"q_{nm}.q_mu"] = 0.1 * rng.randn(n)
        p[f"q_{nm}.q_sqrt"] = (np.log(0.3) + 0.1 * rng.randn(n) if qs == "diagonal"
                               else 0.3 * np.eye(n) + (0.2 / np.sqrt(n)) * np.tril(rng.randn(n, n)))
        p[f"q_{nm}.scale"] = np.array([float(O.log1pe_backward(1.0)) + 0.1 * rng.randn()])
        p[f"kern_{nm}.lengthscales"] = np.array([float(O.log1pe_backward(v)) for v in ell])
    p["k_var"] = np.array([0.5]); p["k_var_r"] = np.array([0.3]); p["var"] = np.array([-2.0])
    U3 = {nm: rng.randn(S, n) for nm in ROLES}
    val, gref = oracle(p, X, Y, U3, q_shapes, jitter)
    out4, grads, _, _ = run_moe(lib, X, Y, p, U3, q_shapes, jitter, S)
    e_val = abs(out4[0] - val) / abs(val)
    errs = block_errors(grads, gref, p)
    print(f"ARD (1, 3, 3): ELBO {e_val:.1e}, gradient blocks", {k: f"{e:.1e}" for k, e in errs.items()})
    assert e_val <= 1e-10
    for k, e in errs.items():
        assert e <= 1e-8, (k, e)


def test_philox_route_and_repeatability(lib):
    """eps = NULL draws the library's Philox stream at each variational's offset: the same numbers, bit for bit, as
    injecting those draws widened to double.  Two calls are bitwise identical."""
    from henbun_b200 import ops
    n, S, seed = 700, 4, 11
    q_shapes = ("fullrank", "diagonal", "fullrank")
    X, Y, p, _ = notebook_problem(n, S, q_shapes, seed=3)
    offsets = (0, 4 * S * n, 12 * S * n)
    drawn = {nm: ops.randn_philox((S, n), seed, off, "cuda").double().cpu().numpy() for nm, off in zip(ROLES, offsets)}
    a = run_moe(lib, X, Y, p, None, q_shapes, 3e-4, S, seed=seed, offsets=offsets)
    b = run_moe(lib, X, Y, p, drawn, q_shapes, 3e-4, S, seed=seed, offsets=offsets)
    c = run_moe(lib, X, Y, p, None, q_shapes, 3e-4, S, seed=seed, offsets=offsets)
    for x, y in ((a, b), (a, c)):
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1])
    # a different window is a different draw
    d = run_moe(lib, X, Y, p, None, q_shapes, 3e-4, S, seed=seed, offsets=(0, 4 * S * n, 16 * S * n))
    assert not np.array_equal(a[1], d[1])


def test_fused_adam_step(lib):
    n, S, t = 300, 4, 3
    q_shapes = ("fullrank", "fullrank", "diagonal")
    X, Y, p, U3 = notebook_problem(n, S, q_shapes, seed=5)
    _, grads, _, _ = run_moe(lib, X, Y, p, U3, q_shapes, 1e-2, S)
    _, _, params, _ = run_moe(lib, X, Y, p, U3, q_shapes, 1e-2, S, adam_t=t)
    z = np.zeros_like(grads)
    want, _, _ = O.adam_tf1_step(pack(p), -grads, z, z, t, lr=0.01)
    off = 0
    for k, sz in blocks(p):                                 # the strict upper triangle of a full-rank q_sqrt never moves
        if k.endswith("q_sqrt") and sz == n * n:
            q = np.triu(np.ones((n, n), bool), 1).ravel()
            want[off:off + sz][q] = pack(p)[off:off + sz][q]
        off += sz
    assert rel_err(params, want) <= 1e-12


def test_non_positive_pivot_sets_the_flag(lib):
    n, S = 200, 2
    X, Y, p, U3 = notebook_problem(n, S, ("diagonal",) * 3)
    _, _, _, err = run_moe(lib, X, Y, p, U3, ("diagonal",) * 3, -2.0, S, check_err=False)
    assert err == 1                                         # 1 + row 0: the first pivot is 1 - 2 < 0


# ---------------------------------------------------------------------------------------------------------------------
# through the model API
# ---------------------------------------------------------------------------------------------------------------------
def _model_class():
    import henbun_b200 as hb
    import henbun_b200.tf as tf

    class ExpertGPR(hb.model.Model):                        # notebooks/Expert_GPR.ipynb:101-149
        def setUp(self, X=None, Y=None, q_shapes=("fullrank", "fullrank", "diagonal"), ell=(0.2, 1.0, 1.0)):
            self.X = hb.param.Data(X)
            self.Y = hb.param.Data(Y)
            self.q_s = hb.variationals.Gaussian(shape=[X.shape[0], 1], q_shape=q_shapes[0])
            self.q_l = hb.variationals.Gaussian(shape=[X.shape[0], 1], q_shape=q_shapes[1])
            self.q_r = hb.variationals.Gaussian(shape=[X.shape[0], 1], q_shape=q_shapes[2])
            self.kern_s = hb.gp.kernels.UnitRBF(np.ones(1) * ell[0])
            self.kern_l = hb.gp.kernels.UnitRBF(np.ones(1) * ell[1])
            self.kern_r = hb.gp.kernels.UnitRBF(np.ones(1) * ell[2])
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

        @hb.model.AutoOptimize()
        def ELBO_gate_first(self):                          # q_r sampled first, then q_l, then q_s
            f_r = tf.matmul(self.kern_r.Cholesky(self.X), self.q_r) * tf.sqrt(self.k_var_r)
            f_l = tf.matmul(self.kern_l.Cholesky(self.X), self.q_l)
            f_s = tf.matmul(self.kern_s.Cholesky(self.X), self.q_s)
            fraction = tf.sigmoid(f_r)
            f = self.k_var * (f_l * (1 - fraction) + fraction * f_s)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, f, self.var)) - self.KL()

    return ExpertGPR


def _settings(float_type, jitter):
    import henbun_b200 as hb
    cfg = hb.settings.get_settings(); cfg.dtypes.float_type = float_type; cfg.numerics.jitter_level = jitter
    return hb.settings.temp_settings(cfg)


def _per_variable(opt, flat):
    return {v.long_name: flat[o:o + s].detach().double().cpu().numpy() for v, (o, s) in zip(opt.var_list, opt._slices)}


@pytest.mark.parametrize("method", ["ELBO", "ELBO_gate_first"])
def test_binding_matches_the_eager_tape(method):
    """Un-injected Philox draws on a well-conditioned input (X = randn(300, 3), l = 0.3, jitter 1e-2, cond(K) ~ 570): the
    float64 step and the eager fp32 tape agree to 1e-4 on the ELBO and every gradient block, so each variational reads the
    Philox window the tape gives it (a wrong window is off by O(1))."""
    import henbun_b200 as hb
    ExpertGPR = _model_class()
    rng = np.random.RandomState(1)
    n, S = 300, 4
    X = rng.randn(n, 3); Y = np.sin(X.sum(1, keepdims=True)) + 0.1 * rng.randn(n, 1)
    m = ExpertGPR(X=X, Y=Y, ell=(0.3, 0.3, 0.3))
    for nm in ("q_s", "q_l"):
        getattr(m, nm).q_sqrt = 0.3 * np.eye(n) + (0.2 / np.sqrt(n)) * np.tril(rng.randn(n, n))
    opt = getattr(m, method)()
    with _settings('float32', 1e-2):
        opt.compile(n_samples=S, verbose=False)
        assert opt.fused_entry is None
        opt._flat_grad.zero_()
        val = opt._evaluate(opt.feed_dict(None), grad=True)
        val.backward()
        tape = {v.long_name: v._tensor.grad.detach().double().cpu().numpy().ravel() for v in opt.var_list}
        tape_val = float(val)
    with _settings('float64', 1e-2):
        opt.compile(n_samples=S, verbose=False)
        assert opt.fused_entry == 'MixtureGpElboBinding'
        got_val = float(opt.optimize(maxiter=1))
        got = _per_variable(opt, opt._fused._g64)
    e_val = abs(got_val - tape_val) / abs(tape_val)
    errs = {k: rel_err(got[k], tape[k]) for k in tape}
    print(f"{method}: ELBO {e_val:.1e}, gradient blocks", {k: f"{e:.1e}" for k, e in errs.items()})
    assert e_val <= 1e-4
    for k, e in errs.items():
        assert e <= 1e-4, (k, e)


def test_adam_through_the_api():
    """Ten Adam steps of optimize() in float64 follow the oracle's gradient + TF-1 Adam to 1e-7; a value assigned between
    steps reaches the fp64 master copy."""
    import henbun_b200 as hb
    import henbun_b200.tf as tf
    ExpertGPR = _model_class()
    rng = np.random.RandomState(2)
    n, S, jitter = 300, 4, 1e-2
    q_shapes = ("fullrank", "fullrank", "diagonal")
    X = rng.randn(n, 2); Y = np.sin(X.sum(1, keepdims=True)) + 0.1 * rng.randn(n, 1)
    m = ExpertGPR(X=X, Y=Y, q_shapes=q_shapes, ell=(0.5, 1.0, 1.0))
    for nm in ("q_s", "q_l"):
        getattr(m, nm).q_sqrt = 0.3 * np.eye(n) + (0.2 / np.sqrt(n)) * np.tril(rng.randn(n, n))
    with _settings('float64', jitter):
        m.ELBO().compile(optimizer=tf.train.AdamOptimizer(0.01), n_samples=S, verbose=False)
        assert m.ELBO().fused_entry == 'MixtureGpElboBinding'
        # the fp64 master copy starts from the Optimizer's fp32 flat buffer: so does the reference trajectory
        g = lambda v: v._free_numpy().astype(np.float32).astype(np.float64)
        p = {}
        for nm, qs in zip(ROLES, q_shapes):
            q = getattr(m, "q_" + nm)
            p[f"q_{nm}.q_mu"] = g(q.q_mu).reshape(n)
            p[f"q_{nm}.q_sqrt"] = g(q.q_sqrt).reshape((n, n) if qs == "fullrank" else (n,))
            p[f"q_{nm}.scale"] = g(q.scale).reshape(1)
            p[f"kern_{nm}.lengthscales"] = g(getattr(m, "kern_" + nm).lengthscales).reshape(-1)
        for k in ("k_var", "k_var_r", "var"):
            p[k] = g(getattr(m, k)).reshape(1)
        mom = {k: np.zeros_like(v) for k, v in p.items()}; vel = {k: np.zeros_like(v) for k, v in p.items()}
        qv = {nm: object.__getattribute__(m, "q_" + nm) for nm in ROLES}
        for t in range(1, 11):
            U3 = {nm: rng.randn(S, n) for nm in ROLES}
            m.ELBO().optimize(maxiter=1, eps={qv[nm]: U3[nm].reshape(S, n, 1) for nm in ROLES})
            _, gr = oracle(p, X, Y, U3, q_shapes, jitter)
            for k in p:
                p[k], mom[k], vel[k] = O.adam_tf1_step(p[k], -gr[k], mom[k], vel[k], t, lr=0.01)
        got = m.ELBO()._fused._p64.cpu().numpy()
        mirror = m.q_r.q_mu._free_numpy().ravel().copy()
        m.k_var = 7.5
        m.ELBO().optimize(maxiter=1, eps={qv[nm]: rng.randn(S, n, 1) for nm in ROLES})
        k_var_after = float(np.ravel(m.k_var.value)[0])
    print("Adam through the API: max |param - oracle trajectory|", np.max(np.abs(got - pack(p))))
    assert np.allclose(got, pack(p), rtol=1e-7, atol=1e-9)
    assert np.allclose(mirror, p["q_r.q_mu"], rtol=1e-5, atol=1e-6)      # the fp32 mirror follows
    assert abs(k_var_after - 7.5) < 0.2, k_var_after                      # an assignment reaches the master copy


def test_non_positive_pivot_raises_through_the_api():
    import henbun_b200 as hb
    ExpertGPR = _model_class()
    rng = np.random.RandomState(3)
    X = rng.randn(150, 2); Y = rng.randn(150, 1)
    m = ExpertGPR(X=X, Y=Y)
    with _settings('float64', -2.0):                        # every expert's first pivot is 1 - 2 < 0
        m.ELBO().compile(n_samples=2, verbose=False)
        assert m.ELBO().fused_entry == 'MixtureGpElboBinding'
        with pytest.raises(FloatingPointError):
            m.ELBO().optimize(maxiter=1)
