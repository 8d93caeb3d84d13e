"""Host-side contract of the float64 entry points (csrc/f64.cu): workspace sizes and the argument / workspace checks that
return before anything reaches a device, so these run without a GPU."""
import ctypes as C

import pytest

HB_OK, HB_ERR_ARG, HB_ERR_WORKSPACE = 0, 1, 3
FAKE = C.c_void_p(4096)          # a non-NULL device address; every call below is rejected before it is dereferenced


@pytest.fixture(scope="module")
def lib():
    from henbun_b200 import _lib
    return _lib.load()


def cfg(n, D=1, S=10, n_ell=1, full=0, small_gp_kernel=1, offset=0):
    from henbun_b200 import _lib
    o = _lib.Options(0, 2048, 2, 1, small_gp_kernel, 0, 1, 0)
    c = _lib.GpConfig(n, D, S, n_ell, full, 3e-4, 0, offset)
    c.opt = C.pointer(o)
    c._keep = o
    return c


@pytest.mark.parametrize("n", [113, 500, 2000, 16384])
def test_chain_workspace_holds_two_gram_matrices(lib, n):
    c = cfg(n)
    assert lib.hb_gp_elbo_f64_workspace_bytes(C.byref(c)) >= 2 * n * n * 8 + 5 * 10 * n * 8


@pytest.mark.parametrize("n", [1, 37, 100, 112])
def test_notebook_sizes_take_the_one_cta_figure(lib, n):
    c = cfg(n)
    assert lib.hb_gp_elbo_f64_workspace_bytes(C.byref(c)) == lib.hb_gp_small_workspace_bytes(C.byref(c), 1)
    # with the one-CTA kernel switched off the same sizes run the chain and need its workspace
    c0 = cfg(n, small_gp_kernel=0)
    assert lib.hb_gp_elbo_f64_workspace_bytes(C.byref(c0)) >= 2 * n * n * 8


def test_potrf_workspace(lib):
    assert lib.hb_potrf_f64_workspace_bytes(0) == 0
    assert lib.hb_potrf_f64_workspace_bytes(64) == 0                    # one leaf: no product
    for n in (65, 2000, 16384):
        assert lib.hb_potrf_f64_workspace_bytes(n) >= 32 * 128 * 128 * 8   # split-K partial tiles of the reductions


def gemm(lib, A=FAKE, lda=8, tA=0, at=0, B=FAKE, ldb=8, tB=0, bt=0, Cp=FAKE, ldc=8, ct=0, M=8, N=8, K=8, ws=None, wsb=0):
    return lib.hb_gemm_f64(A, lda, tA, at, B, ldb, tB, bt, Cp, ldc, ct, M, N, K, 1.0, 0.0, ws, wsb, None)


def test_gemm_rejects_bad_arguments(lib):
    assert gemm(lib, M=-1) == HB_ERR_ARG
    assert gemm(lib, K=-1) == HB_ERR_ARG
    assert gemm(lib, at=5) == HB_ERR_ARG
    assert gemm(lib, bt=-1) == HB_ERR_ARG
    assert gemm(lib, ct=2) == HB_ERR_ARG
    assert gemm(lib, tA=2) == HB_ERR_ARG
    assert gemm(lib, lda=7) == HB_ERR_ARG                      # A stored [M, K]
    assert gemm(lib, tA=1, M=9, lda=8) == HB_ERR_ARG           # A stored [K, M]
    assert gemm(lib, ldb=7) == HB_ERR_ARG
    assert gemm(lib, ldc=7) == HB_ERR_ARG
    assert gemm(lib, A=None) == HB_ERR_ARG
    assert gemm(lib, Cp=None) == HB_ERR_ARG
    assert gemm(lib, wsb=1 << 20) == HB_ERR_WORKSPACE          # a size without a buffer
    assert gemm(lib, M=0) == HB_OK                              # empty output: nothing to launch


def test_potrf_rejects_bad_arguments(lib):
    err = FAKE
    assert lib.hb_potrf_lower_f64(FAKE, 100, -1, None, 0, err, None) == HB_ERR_ARG
    assert lib.hb_potrf_lower_f64(FAKE, 99, 100, None, 0, err, None) == HB_ERR_ARG
    assert lib.hb_potrf_lower_f64(None, 100, 100, None, 0, err, None) == HB_ERR_ARG
    assert lib.hb_potrf_lower_f64(FAKE, 100, 100, None, 0, err, None) == HB_ERR_WORKSPACE
    assert lib.hb_potrf_lower_f64(FAKE, 100, 0, None, 0, err, None) == HB_OK
    assert lib.hb_potrf_lower_bwd_f64(FAKE, 100, FAKE, 99, 100, None, 0, None) == HB_ERR_ARG
    assert lib.hb_potrf_lower_bwd_f64(FAKE, 100, None, 100, 100, None, 0, None) == HB_ERR_ARG
    ws_small = lib.hb_potrf_f64_workspace_bytes(100) - 1
    assert lib.hb_potrf_lower_bwd_f64(FAKE, 100, FAKE, 100, 100, FAKE, ws_small, None) == HB_ERR_WORKSPACE


def step(lib, c, eps=FAKE, m=None, v=None, adam=None, ws=FAKE, wsb=None):
    if wsb is None:
        wsb = lib.hb_gp_elbo_f64_workspace_bytes(C.byref(c)) if c is not None else 0
    ref = C.byref(c) if c is not None else None
    return lib.hb_gp_elbo_step_f64(ref, FAKE, FAKE, FAKE, eps, FAKE, FAKE, m, v, adam, ws, wsb, FAKE, None)


def test_step_rejects_bad_arguments(lib):
    from henbun_b200 import _lib
    assert step(lib, None) == HB_ERR_ARG
    assert step(lib, cfg(500, D=33, n_ell=1)) == HB_ERR_ARG
    assert step(lib, cfg(500, D=3, n_ell=2)) == HB_ERR_ARG
    assert step(lib, cfg(500, S=0)) == HB_ERR_ARG
    assert step(lib, cfg(500, offset=2), eps=None) == HB_ERR_ARG            # Philox offsets are multiples of 4
    assert step(lib, cfg(500), m=FAKE) == HB_ERR_ARG                        # moments without an Adam config
    adam = _lib.AdamConfig(0.01, 0.9, 0.999, 1e-8, -1.0, None, 1)
    assert step(lib, cfg(500), m=FAKE, adam=C.byref(adam)) == HB_ERR_ARG    # m without v
    for n, small in ((500, 1), (100, 0), (100, 1)):
        c = cfg(n, small_gp_kernel=small)
        assert step(lib, c, wsb=lib.hb_gp_elbo_f64_workspace_bytes(C.byref(c)) - 1) == HB_ERR_WORKSPACE
        assert step(lib, c, ws=None) == HB_ERR_WORKSPACE
