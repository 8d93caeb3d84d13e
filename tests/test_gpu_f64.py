"""float64 at any size (csrc/f64.cu): the fp64 GEMM, the blocked Cholesky and its reverse mode, and hb_gp_elbo_step_f64
against CPU / torch fp64 references and the fp64 oracle, the two fp64 routes against each other, and the float64 route
through the model API beyond the one-CTA kernel's n <= 112."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import henbun_oracle as O
from test_gpu_small import ORDER, pack, problem

pytestmark = pytest.mark.gpu
U53 = 2.0 ** -53


@pytest.fixture(scope="module")
def lib():
    from henbun_b200 import _lib
    return _lib.load()


def P(t):
    from henbun_b200._lib import ptr
    return ptr(t)


def ST():
    from henbun_b200._lib import stream
    return stream()


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64).cuda()


def rel_err(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


# ---------------------------------------------------------------------------------------------------------------------
# hb_gemm_f64
# ---------------------------------------------------------------------------------------------------------------------
def op_mask(tri, rows, cols, a_side):
    r = np.arange(rows)[:, None]; c = np.arange(cols)[None, :]
    if a_side:                         # (m, k)
        m, k = r, c
        return {0: np.ones((rows, cols), bool), 1: k <= m, 2: k >= m, 3: k > m, 4: k < m}[tri]
    k, n = r, c                        # (k, n)
    return {0: np.ones((rows, cols), bool), 1: n <= k, 2: n >= k, 3: n > k, 4: n < k}[tri]


def run_gemm(lib, M, N, K, tA, tB, at, bt, ct, alpha, beta, rng, ws=None, C0=None):
    A = rng.randn(K, M) if tA else rng.randn(M, K)
    B = rng.randn(N, K) if tB else rng.randn(K, N)
    C0 = rng.randn(M, N) if C0 is None else C0
    opA = (A.T if tA else A) * op_mask(at, M, K, True)
    opB = (B.T if tB else B) * op_mask(bt, K, N, False)
    ref = alpha * opA @ opB + (beta * C0 if beta != 0 else 0.0)
    bound = 4 * max(K, 1) * U53 * (abs(alpha) * np.abs(opA) @ np.abs(opB) + (abs(beta) * np.abs(C0) if beta != 0 else 0.0)) + 1e-300
    Ad, Bd, Cd = dev(A), dev(B), dev(C0)
    wsb = 0 if ws is None else ws.numel()
    rc = lib.hb_gemm_f64(P(Ad), A.shape[1], tA, at, P(Bd), B.shape[1], tB, bt, P(Cd), N, ct, M, N, K, alpha, beta,
                         P(ws), wsb, ST())
    torch.cuda.synchronize()
    assert rc == 0
    got = Cd.cpu().numpy()
    low = np.tril(np.ones((M, N), bool)) if ct else np.ones((M, N), bool)
    assert np.all(np.abs(got - ref)[low] <= bound[low]), (M, N, K, tA, tB, at, bt, ct, np.max((np.abs(got - ref) / bound)[low]))
    if ct:                                                    # the strict upper part of C is untouched
        assert np.array_equal(got[~low], C0[~low])
    return got


def test_gemm_every_layout_and_mask(lib):
    rng = np.random.RandomState(0)
    for tA in (0, 1):
        for tB in (0, 1):
            for at in range(5):
                for bt in range(5):
                    for ct in (0, 1):
                        run_gemm(lib, 97, 75, 83, tA, tB, at, bt, ct, -2.0, 0.5, rng)


def test_gemm_ragged_shapes(lib):
    rng = np.random.RandomState(1)
    sizes = (1, 63, 65, 1000)
    for M in sizes:
        for N in sizes:
            for K in sizes:
                run_gemm(lib, M, N, K, rng.randint(2), rng.randint(2), 0, 0, 0, 1.0, 0.0, rng)


@pytest.mark.parametrize("S", [1, 10, 64])
def test_gemm_sample_rows(lib, S):
    """the S-row products of the GP step: F = Z L^T and W = R L with a triangular L, and Z += U tril(Lq)^T"""
    rng = np.random.RandomState(S)
    n = 1500
    run_gemm(lib, S, n, n, 0, 1, 0, 2, 0, 1.0, 0.0, rng)
    run_gemm(lib, S, n, n, 0, 0, 0, 1, 0, 1.0, 0.0, rng)
    run_gemm(lib, S, n, n, 0, 1, 0, 2, 0, 1.0, 1.0, rng)
    run_gemm(lib, n, n, S, 1, 0, 0, 0, 1, 1.0, 0.0, rng)     # tril(R^T Z)


def test_gemm_split_k_is_deterministic(lib):
    rng = np.random.RandomState(2)
    ws = torch.empty(8 << 20, dtype=torch.uint8, device="cuda")
    a = run_gemm(lib, 64, 64, 20000, 1, 0, 0, 0, 1, -2.0, 1.0, np.random.RandomState(5), ws=ws)
    b = run_gemm(lib, 64, 64, 20000, 1, 0, 0, 0, 1, -2.0, 1.0, np.random.RandomState(5), ws=ws)
    assert np.array_equal(a, b)
    run_gemm(lib, 130, 70, 5000, 0, 1, 0, 0, 0, 1.0, 0.0, rng, ws=ws)


def test_gemm_beta_zero_does_not_read_c(lib):
    run_gemm(lib, 70, 70, 50, 0, 0, 0, 0, 0, 1.0, 0.0, np.random.RandomState(3), C0=np.full((70, 70), np.nan))


# ---------------------------------------------------------------------------------------------------------------------
# hb_potrf_lower_f64 / hb_potrf_lower_bwd_f64
# ---------------------------------------------------------------------------------------------------------------------
def spd(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    B = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
    return B @ B.T / n + 0.5 * torch.eye(n, dtype=torch.float64, device="cuda")


@pytest.mark.parametrize("n", [1, 63, 64, 65, 500, 2000, 4224, 8200])
def test_potrf_f64(lib, n):
    A = spd(n, n)
    wsb = lib.hb_potrf_f64_workspace_bytes(n)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    Lk = A.clone() + torch.triu(torch.full_like(A, float("nan")), 1)     # the strict upper triangle is never read
    assert lib.hb_potrf_lower_f64(P(Lk), n, n, P(ws), wsb, P(err), ST()) == 0
    torch.cuda.synchronize()
    assert err.item() == 0
    L = torch.tril(Lk)
    assert torch.isnan(Lk[torch.triu(torch.ones(n, n, dtype=torch.bool, device="cuda"), 1)]).all()   # ... nor written
    rt = (torch.linalg.norm(L @ L.T - A) / torch.linalg.norm(A)).item()
    ev = torch.linalg.eigvalsh(A)
    cond = (ev[-1] / ev[0]).item()
    Lref = torch.linalg.cholesky(A)
    fe = (torch.linalg.norm(L - Lref) / torch.linalg.norm(Lref)).item()
    print(f"n={n}: round trip {rt:.2e}, factor vs torch {fe:.2e} (cond {cond:.1f})")
    assert rt <= 1e-14
    assert fe <= 64 * cond * U53

    # reverse mode against torch autograd (symmetric-input convention: compare the lower triangles of sym(grad))
    g = torch.Generator(device="cuda").manual_seed(n + 1)
    Lb = torch.tril(torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g))
    tA = A.clone().requires_grad_(True)
    torch.sum(torch.linalg.cholesky(tA) * Lb).backward()
    Gref = torch.tril(0.5 * (tA.grad + tA.grad.T))
    runs = []
    for _ in range(2):
        G = Lb + torch.triu(torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g), 1)   # ignored above the diagonal
        assert lib.hb_potrf_lower_bwd_f64(P(L), n, P(G), n, n, P(ws), wsb, ST()) == 0
        torch.cuda.synchronize()
        runs.append(torch.tril(G))
    be = (torch.linalg.norm(runs[0] - Gref) / torch.linalg.norm(Gref)).item()
    print(f"n={n}: reverse mode vs torch autograd {be:.2e}")
    assert be <= 1e-10
    assert torch.equal(runs[0], runs[1])                                   # bitwise reproducible
    # the factorisation is deterministic too
    L2 = A.clone()
    assert lib.hb_potrf_lower_f64(P(L2), n, n, P(ws), wsb, P(err), ST()) == 0
    torch.cuda.synchronize()
    assert torch.equal(torch.tril(L2), L)


@pytest.mark.parametrize("n,bad", [(6, 3), (300, 200)])
def test_potrf_f64_flags_a_non_positive_pivot(lib, n, bad):
    A = torch.eye(n, dtype=torch.float64, device="cuda")
    A[bad, bad] = -1.0
    wsb = lib.hb_potrf_f64_workspace_bytes(n)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    assert lib.hb_potrf_lower_f64(P(A), n, n, P(ws), wsb, P(err), ST()) == 0
    torch.cuda.synchronize()
    assert err.item() == bad + 1                                            # 1 + the failing row, as the fp32 path


# ---------------------------------------------------------------------------------------------------------------------
# hb_gp_elbo_step_f64
# ---------------------------------------------------------------------------------------------------------------------
def run_step(lib, X, Y, p, U, jitter, full, small_gp_kernel=1, adam_t=None, seed=0):
    from henbun_b200 import _lib
    n, D = X.shape; S = U.shape[0] if U is not None else 4
    o = _lib.Options(0, 2048, 2, 1, small_gp_kernel, 0, 1, 0)
    cfg = _lib.GpConfig(n, D, S, p["lengthscales"].size, 1 if full else 0, jitter, seed, 0)
    cfg.opt = C.pointer(o)
    npar = lib.hb_gp_param_count(C.byref(cfg))
    params, grads, out4 = dev(pack(p)), torch.zeros(npar, dtype=torch.float64, device="cuda"), \
        torch.zeros(4, dtype=torch.float64, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    wsb = lib.hb_gp_elbo_f64_workspace_bytes(C.byref(cfg))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    Xd, Yd = dev(X), dev(Y)
    Ud = dev(U) if U is not None else None
    m = v = acfg = None
    if adam_t is not None:
        m, v = torch.zeros_like(params), torch.zeros_like(params)
        acfg = C.byref(_lib.AdamConfig(0.01, 0.9, 0.999, 1e-8, -1.0, None, adam_t))
    rc = lib.hb_gp_elbo_step_f64(C.byref(cfg), P(Xd), P(Yd), P(params), P(Ud), P(grads), P(out4), P(m), P(v), acfg, P(ws), wsb,
                                 P(err), ST())
    torch.cuda.synchronize()
    assert rc == 0 and err.item() == 0
    return out4.cpu().numpy(), grads.cpu().numpy(), params.cpu().numpy()


def oracle(p, X, Y, U, jitter, full):
    j32 = float(np.float32(jitter))                        # hb_gp_config carries the jitter as a float
    return O.value_and_grads(lambda pp, *a: O.gpr_elbo(pp, *a, q_shape='fullrank' if full else 'diagonal', jitter=j32),
                             p, X, Y, U, device="cuda")


@pytest.mark.parametrize("n", [113, 500, 2000, 8200])
@pytest.mark.parametrize("full", [False, True])
@pytest.mark.parametrize("ard", [False, True])
@pytest.mark.parametrize("S", [1, 10])
def test_step_matches_oracle_fp64(lib, n, full, ard, S):
    D = 3
    X, Y, p, U, jitter = problem(n, D, S, full, ard, seed=n + S + 2 * full + ard)
    val, g = oracle(p, X, Y, U, jitter, full)
    out4, grads, _ = run_step(lib, X, Y, p, U, jitter, full)
    e_val, e_grad = abs(out4[0] - val) / abs(val), rel_err(grads, pack(g))
    print(f"n={n} full={full} ard={ard} S={S}: ELBO {e_val:.1e}, gradient {e_grad:.1e}")
    assert e_val <= 1e-10
    assert e_grad <= 1e-8
    if full:
        assert np.count_nonzero(np.triu(grads[n:n + n * n].reshape(n, n), 1)) == 0


def test_step_matches_oracle_fp64_n16384(lib):
    n, S = 16384, 4
    X, Y, p, U, jitter = problem(n, 3, S, False, False, seed=7)
    val, g = oracle(p, X, Y, U, jitter, False)
    out4, grads, _ = run_step(lib, X, Y, p, U, jitter, False)
    e_val, e_grad = abs(out4[0] - val) / abs(val), rel_err(grads, pack(g))
    print(f"n={n}: ELBO {e_val:.1e}, gradient {e_grad:.1e}")
    assert e_val <= 1e-10 and e_grad <= 1e-8


@pytest.mark.parametrize("n", [37, 100, 112])
@pytest.mark.parametrize("full", [False, True])
@pytest.mark.parametrize("philox", [False, True])
def test_chain_equals_the_one_cta_kernel(lib, n, full, philox):
    S = 10
    X, Y, p, U, jitter = problem(n, 2, S, full, True, seed=n)
    U = None if philox else U
    a = run_step(lib, X, Y, p, U, jitter, full, small_gp_kernel=1, seed=11)
    b = run_step(lib, X, Y, p, U, jitter, full, small_gp_kernel=0, seed=11)
    assert abs(a[0][0] - b[0][0]) <= 1e-12 * abs(a[0][0])
    assert rel_err(b[1], a[1]) <= 1e-12
    a2 = run_step(lib, X, Y, p, U, jitter, full, small_gp_kernel=1, adam_t=3, seed=11)
    b2 = run_step(lib, X, Y, p, U, jitter, full, small_gp_kernel=0, adam_t=3, seed=11)
    assert rel_err(b2[2], a2[2]) <= 1e-12


def test_expert_gpr_input_meets_the_parity_bar(lib):
    """The Expert_GPR notebook's 1-D grid (X = linspace(0, 6, 2000), jitter 3e-4, lengthscale 1: cond ~ 2.5e6), where the
    fp32 path has to be held to a condition-scaled bar: in float64 the ELBO and every gradient block meet 1e-5."""
    n, S = 2000, 10
    for full in (False, True):
        X, Y, p, U, _ = problem(n, 1, S, full, False, seed=0, grid=True)
        jitter = 3e-4
        p["lengthscales"] = np.array([float(O.log1pe_backward(1.0))])
        val, g = oracle(p, X, Y, U, jitter, full)
        out4, grads, _ = run_step(lib, X, Y, p, U, jitter, full)
        gref = pack(g)
        assert abs(out4[0] - val) <= 1e-5 * abs(val)
        off = 0
        for k in ORDER:
            sz = np.asarray(p[k]).size
            e = rel_err(grads[off:off + sz], gref[off:off + sz])
            print(f"full={full} {k}: {e:.1e}")
            assert e <= 1e-5, k
            off += sz


def test_fused_adam_step(lib):
    n, S, t = 700, 10, 4
    X, Y, p, U, jitter = problem(n, 2, S, True, False, seed=5)
    _, grads, _ = run_step(lib, X, Y, p, U, jitter, True)
    _, _, params = run_step(lib, X, Y, p, U, jitter, True, adam_t=t)
    z = np.zeros_like(grads)
    want, _, _ = O.adam_tf1_step(pack(p), -grads, z, z, t, lr=0.01)
    q = np.triu(np.ones((n, n), bool), 1).ravel()           # the strict upper triangle of q_sqrt never moves
    want[n:n + n * n][q] = pack(p)[n:n + n * n][q]
    assert rel_err(params, want) <= 1e-12


def test_float64_through_the_api_beyond_the_one_cta_kernel():
    """float_type = 'float64' at n = 1000: the bound GP graph takes hb_gp_elbo_step_f64 (the kernel chain, Adam included).
    jitter 1e-3: with the default 1e-5 this 1-D grid has cond(K) ~ 4e7, and the first Adam steps' g / (|g| + eps) turn the
    cond * 2^-53 error of the smallest gradient entries into parameter differences of 1e-8 between ANY two fp64
    implementations (measured against the oracle: gradient 2e-10, four of 1e6 parameters outside rtol 1e-7)."""
    import henbun_b200 as hb
    import henbun_b200.tf as tf
    rng = np.random.RandomState(0)
    n, S = 1000, 10
    X = np.linspace(0, 6, n).reshape(-1, 1); Y = np.sin(X) + 0.3 * rng.randn(n, 1)

    class GPR(hb.model.Model):
        def setUp(self):
            self.X = hb.param.Data(X); self.Y = hb.param.Data(Y)
            self.q = hb.variationals.Gaussian(shape=[n, 1], q_shape='fullrank')
            self.kern = hb.gp.kernels.UnitRBF()
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            y_fit = tf.matmul(self.kern.Cholesky(self.X), self.q) * tf.sqrt(self.k_var)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, y_fit, self.var)) - self.KL()

    m = GPR()
    m.q.q_sqrt = 0.3 * np.eye(n) + 0.02 * np.tril(rng.randn(n, n))
    cfg = hb.settings.get_settings(); cfg.dtypes.float_type = 'float64'; cfg.numerics.jitter_level = 1e-3
    with hb.settings.temp_settings(cfg):
        m.ELBO().compile(optimizer=tf.train.AdamOptimizer(0.01), n_samples=S, verbose=False)
        assert m.ELBO().fused_entry == 'GpElboBinding'
        jitter = float(np.float32(m.ELBO()._compiled_settings.numerics.jitter_level))
        # the fp64 master copy starts from the Optimizer's fp32 flat buffer: so does the reference trajectory
        g = lambda v: v._free_numpy().astype(np.float32).astype(np.float64)
        p = dict(q_mu=g(m.q.q_mu).reshape(n), q_sqrt=g(m.q.q_sqrt).reshape(n, n), scale=g(m.q.scale).reshape(1),
                 lengthscales=g(m.kern.lengthscales).reshape(-1), k_var=g(m.k_var).reshape(1), var=g(m.var).reshape(1))
        mom = {k: np.zeros_like(v) for k, v in p.items()}; vel = {k: np.zeros_like(v) for k, v in p.items()}
        q = object.__getattribute__(m, 'q')
        for t in range(1, 11):
            U = rng.randn(S, n, 1)
            m.ELBO().optimize(maxiter=1, eps={q: U})
            _, gr = O.value_and_grads(lambda pp, *a: O.gpr_elbo(pp, *a, q_shape='fullrank', jitter=jitter), p, X, Y[:, 0],
                                      U[:, :, 0], device="cuda")
            for k in p:
                p[k], mom[k], vel[k] = O.adam_tf1_step(p[k], -gr[k], mom[k], vel[k], t, lr=0.01)
        got = m.ELBO()._fused._p64.cpu().numpy()
        mirror = m.q.q_mu._free_numpy().ravel().copy()
        m.k_var = 7.5
        m.ELBO().optimize(maxiter=1, eps={q: rng.randn(S, n, 1)})
        k_var_after = float(np.ravel(m.k_var.value)[0])
    assert np.allclose(got, pack(p), rtol=1e-7, atol=1e-9)
    assert np.allclose(mirror, p["q_mu"], rtol=1e-5, atol=1e-6)      # the fp32 mirror follows
    assert abs(k_var_after - 7.5) < 0.2, k_var_after                  # an assignment between steps reaches the master copy
