"""ctypes binding of libhenbun_b200.so (the C ABI declared in include/henbun_b200.h).

There is no CPU fallback: if the shared library is missing, ``load()`` raises, and every wrapper
refuses tensors that are not fp32 CUDA tensors.  torch is used only to own device memory and the
current stream.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhenbun_b200.so")

HB_OK, HB_ERR_ARG, HB_ERR_CUDA, HB_ERR_WORKSPACE = 0, 1, 2, 3
ACT = {"none": 0, None: 0, "identity": 0, "sigmoid": 1, "relu": 2, "tanh": 3}

_c_f = C.c_void_p        # device pointers travel as void*
_ll = C.c_longlong
_ull = C.c_ulonglong
_i = C.c_int
_fl = C.c_float
_sz = C.c_size_t


class Options(C.Structure):
    """hb_options (include/henbun_b200.h): behavioural switches that travel with every call."""
    _fields_ = [("gemm_engine", _i), ("exact_below", _i), ("panel_refinement", _i), ("presplit_engine", _i),
                ("small_gp_kernel", _i), ("tc_option", _i), ("lookahead", _i), ("schedule", _i)]


# The process-wide DEFAULT the Python layer passes when a caller gives no options of its own.  The C library itself keeps
# no configuration; `lib.hb_set_*` below are Python-side conveniences that edit this object (tests, A/B runs).
OPTIONS = Options(0, 2048, 2, 1, 1, 0, 1, 0)


class GpConfig(C.Structure):
    _fields_ = [("n", _i), ("D", _i), ("S", _i), ("n_ell", _i), ("q_fullrank", _i), ("jitter", _fl),
                ("seed", _ull), ("offset", _ull), ("opt", C.POINTER(Options))]


class MoeGpConfig(C.Structure):
    """hb_moe_gp_config: per-expert arrays in the order s, l, r."""
    _fields_ = [("n", _i), ("D", _i), ("S", _i), ("n_ell", _i * 3), ("q_fullrank", _i * 3), ("jitter", C.c_double),
                ("seed", _ull), ("offset", _ull * 3), ("opt", C.POINTER(Options))]


class Dist(C.Structure):
    """hb_dist: this rank's place in a column-block-cyclic factorisation (comm from hb_comm_create; NULL when world == 1)."""
    _fields_ = [("comm", C.c_void_p), ("rank", _i), ("world", _i), ("block", _i), ("shard_samples", _i), ("batch", _i), ("block_bwd", _i), ("turn", _i)]


class AdamConfig(C.Structure):
    _fields_ = [("lr", C.c_double), ("b1", C.c_double), ("b2", C.c_double), ("eps", C.c_double), ("grad_scale", C.c_double),
                ("step_dev", C.c_void_p),
                ("step_host", _i)]


HB_MAX_LAYERS = 8


class AmortisedConfig(C.Structure):
    _fields_ = [("B", _i), ("S", _i), ("latent", _i),
                ("n_enc", _i), ("enc_nodes", _i * (HB_MAX_LAYERS + 1)), ("enc_act", _i * HB_MAX_LAYERS),
                ("n_dec", _i), ("dec_nodes", _i * (HB_MAX_LAYERS + 1)), ("dec_act", _i * HB_MAX_LAYERS),
                ("seed", _ull), ("offset", _ull), ("opt", C.POINTER(Options))]


class LinopConfig(C.Structure):
    _fields_ = [("M", _i), ("M_total", _ll), ("n", _i), ("S", _i), ("seed", _ull), ("offset", _ull), ("presplit", _i),
                ("opt", C.POINTER(Options))]


# name -> (restype, argtypes); kept in one table so tests can check that every symbol the header
# declares is exported.
SIGNATURES = {
    "hb_version": (_i, []),
    "hb_launch_count": (_ull, []),
    "hb_reduce_workspace_bytes": (_sz, []),
    "hb_options_init": (None, [C.POINTER(Options)]),
    "hb_profile_begin": (_i, [_i]),
    "hb_profile_end": (_i, [C.POINTER(C.c_double)]),
    "hb_profile_dump_csv": (_i, [C.c_char_p]),
    "hb_profile_end_ex": (_i, [C.POINTER(C.c_double)]),
    "hb_phase_begin": (_i, []),
    "hb_phase_end": (_i, [C.POINTER(C.c_double), _i]),
    "hb_randn_philox": (_i, [_c_f, _ll, _ull, _ull, _c_f]),
    "hb_philox4x32_10": (_i, [_c_f, _ll, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), _c_f]),
    "hb_sample_diag_fwd": (_i, [_c_f, _ll, _c_f, _ll, _i, _i, _c_f, _ull, _ull, _i, _c_f, _c_f, _c_f, _sz, _c_f]),
    "hb_sample_diag_bwd": (_i, [_c_f, _ll, _c_f, _ll, _i, _i, _c_f, _ull, _ull, _i, _c_f, _c_f, _fl, _c_f, _c_f, _ll,
                                _c_f, _ll, _fl, _c_f]),
    "hb_sample_tril_fwd": (_i, [_c_f, _c_f, _i, _i, _c_f, _i, _c_f, _c_f, _c_f, _sz, _c_f]),
    "hb_sample_tril_bwd": (_i, [_c_f, _i, _i, _c_f, _c_f, _i, _c_f, _fl, _c_f, _c_f, _c_f, _c_f]),
    "hb_gaussian_logpdf": (_i, [_c_f, _ll, _c_f, _ll, _c_f, _ll, _ll, _c_f, _c_f]),
    "hb_gaussian_logpdf_bwd": (_i, [_c_f, _ll, _c_f, _ll, _c_f, _ll, _ll, _c_f, _c_f, _c_f, _c_f]),
    "hb_transform_fwd": (_i, [_i, _c_f, _ll, _fl, _fl, _c_f, _c_f]),
    "hb_transform_bwd": (_i, [_i, _c_f, _ll, _fl, _fl, _c_f, _c_f, _c_f]),
    "hb_transform_logjac": (_i, [_i, _c_f, _ll, _fl, _fl, _c_f, _c_f, _sz, _c_f]),
    "hb_transform_logjac_bwd": (_i, [_i, _c_f, _ll, _fl, _fl, _c_f, _c_f, _c_f]),
    "hb_density_nargs": (_i, [_i]),
    "hb_density_logpdf": (_i, [_i, _c_f, _c_f, _ll, _c_f, _c_f]),
    "hb_density_logpdf_bwd": (_i, [_i, _c_f, _c_f, _ll, _c_f, _ll, _c_f, _c_f, _sz, _c_f]),
    "hb_gather_rows": (_i, [_c_f, _c_f, _c_f, _ll, _ll, _c_f]),
    "hb_random_index": (_i, [_c_f, _ll, _c_f, _ll, _ull, _ull, _c_f]),
    "hb_gauss_loglik_fwd": (_i, [_c_f, _c_f, _c_f, _ll, _ll, _c_f, _fl, _c_f, _c_f, _c_f, _sz, _c_f]),
    "hb_rbf_gram_fwd": (_i, [_c_f, _c_f, _i, _i, _i, _i, _c_f, _i, _c_f, _ll, _ll, _fl, _i, _i, _c_f]),
    "hb_rbf_gram_bwd": (_i, [_c_f, _ll, _ll, _c_f, _c_f, _i, _i, _i, _i, _c_f, _i, _i, _i, _c_f, _c_f, _c_f, _sz,
                             _c_f]),
    "hb_rbf_gram_bwd_x2": (_i, [_c_f, _ll, _ll, _c_f, _c_f, _i, _i, _i, _i, _c_f, _i, _i, _fl, _c_f, _c_f]),
    "hb_potrf_workspace_bytes": (_sz, [_i]),
    "hb_potrf_lower": (_i, [_c_f, _ll, _ll, _i, _i, _i, _c_f, _sz, _c_f, _c_f, C.POINTER(Options)]),
    "hb_potrf_lower_bwd": (_i, [_c_f, _ll, _ll, _c_f, _ll, _ll, _i, _i, _c_f, _sz, _c_f, C.POINTER(Options)]),
    "hb_trsm_workspace_bytes": (_sz, [_i, _i]),
    "hb_trsm_right_lower": (_i, [_c_f, _ll, _c_f, _ll, _i, _i, _i, _c_f, _sz, _c_f, C.POINTER(Options)]),
    "hb_gemm": (_i, [_c_f, _ll, _ll, _i, _i, _c_f, _ll, _ll, _i, _i, _c_f, _ll, _ll, _i, _i, _i, _i, _i, _fl, _fl,
                     _c_f, _ll, _i, _i, _fl, _fl, _c_f]),
    "hb_gemm_ws": (_i, [_c_f, _ll, _ll, _i, _i, _c_f, _ll, _ll, _i, _i, _c_f, _ll, _ll, _i, _i, _i, _i, _i, _fl, _fl,
                        _c_f, _ll, _i, _i, _fl, _fl, _c_f, _sz, _c_f, C.POINTER(Options)]),
    "hb_gemm_tc_workspace_bytes": (_sz, [_i, _i, _i]),
    "hb_gemm_tn_tc": (_i, [_c_f, _ll, _c_f, _ll, _c_f, _ll, _i, _i, _i, _i, _fl, _fl, _c_f, _sz, _c_f]),
    "hb_gemm_presplit_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "hb_gemm_presplit": (_i, [_c_f, _ll, _i, _c_f, _ll, _i, _c_f, _ll, _i, _i, _i, _i, _fl, _fl, _i, _i, _i, _c_f, _sz, _c_f,
                              C.POINTER(Options)]),
    "hb_act_bwd_colsum_workspace_bytes": (_sz, [_i, _i]),
    "hb_act_bwd_colsum_ws": (_i, [_c_f, _c_f, _c_f, _i, _i, _ll, _i, _i, _fl, _fl, _c_f, _c_f, _sz, _c_f]),
    "hb_act_bwd_colsum": (_i, [_c_f, _c_f, _c_f, _i, _i, _ll, _i, _i, _fl, _fl, _c_f, _c_f]),
    "hb_colsum": (_i, [_c_f, _ll, _i, _i, _fl, _fl, _c_f, _c_f]),
    "hb_adam_tf1": (_i, [_c_f, _c_f, _c_f, _c_f, _ll, _fl, _fl, _fl, _fl, _fl, _c_f, _i, _c_f]),
    "hb_increment_i32": (_i, [_c_f, _c_f]),
    "hb_transpose2d": (_i, [_c_f, _ll, _c_f, _ll, _i, _i, _fl, _c_f]),
    "hb_zero_strict_upper": (_i, [_c_f, _ll, _i, _c_f]),
    "hb_linop_param_count": (_sz, [C.POINTER(LinopConfig)]),
    "hb_linop_workspace_bytes": (_sz, [C.POINTER(LinopConfig)]),
    "hb_linop_prepare": (_i, [C.POINTER(LinopConfig), _c_f, _c_f, _sz, _c_f]),
    "hb_linop_elbo_local": (_i, [C.POINTER(LinopConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _sz, _c_f]),
    "hb_linop_elbo_update": (_i, [C.POINTER(LinopConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _fl, _fl, _fl, _fl, _c_f, _i,
                                  _c_f, _c_f, _sz, _c_f]),
    "hb_amortised_param_count": (_sz, [C.POINTER(AmortisedConfig)]),
    "hb_amortised_workspace_bytes": (_sz, [C.POINTER(AmortisedConfig)]),
    "hb_amortised_elbo_step": (_i, [C.POINTER(AmortisedConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _sz, _c_f]),
    "hb_gp_small_max_n": (_i, [_i]),
    "hb_gp_small_workspace_bytes": (_sz, [C.POINTER(GpConfig), _i]),
    "hb_gp_small_step": (_i, [C.POINTER(GpConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, C.POINTER(AdamConfig), _c_f, _sz,
                              _c_f, _c_f]),
    "hb_gp_small_step_f64": (_i, [C.POINTER(GpConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, C.POINTER(AdamConfig), _c_f,
                                  _sz, _c_f, _c_f]),
    "hb_gp_param_count": (_sz, [C.POINTER(GpConfig)]),
    "hb_gp_elbo_workspace_bytes": (_sz, [C.POINTER(GpConfig)]),
    "hb_gp_elbo_step": (_i, [C.POINTER(GpConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _sz, _c_f, _c_f]),
    "hb_gemm_f64": (_i, [_c_f, _ll, _i, _i, _c_f, _ll, _i, _i, _c_f, _ll, _i, _i, _i, _i, C.c_double, C.c_double, _c_f, _sz, _c_f]),
    "hb_potrf_f64_workspace_bytes": (_sz, [_i]),
    "hb_potrf_lower_f64": (_i, [_c_f, _ll, _i, _c_f, _sz, _c_f, _c_f]),
    "hb_potrf_lower_bwd_f64": (_i, [_c_f, _ll, _c_f, _ll, _i, _c_f, _sz, _c_f]),
    "hb_gp_elbo_f64_workspace_bytes": (_sz, [C.POINTER(GpConfig)]),
    "hb_gp_elbo_step_f64": (_i, [C.POINTER(GpConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, C.POINTER(AdamConfig), _c_f,
                                 _sz, _c_f, _c_f]),
    "hb_moe_gp_param_count": (_sz, [C.POINTER(MoeGpConfig)]),
    "hb_moe_gp_f64_workspace_bytes": (_sz, [C.POINTER(MoeGpConfig)]),
    "hb_moe_gp_elbo_step_f64": (_i, [C.POINTER(MoeGpConfig), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f,
                                     C.POINTER(AdamConfig), _c_f, _sz, _c_f, _c_f]),
    "hb_comm_unique_id": (_i, [C.c_void_p]),
    "hb_comm_create": (_i, [C.c_void_p, _i, _i, C.POINTER(C.c_void_p)]),
    "hb_comm_destroy": (_i, [C.c_void_p]),
    "hb_flat_trace_begin": (_i, []),
    "hb_flat_trace_end": (_i, [C.POINTER(C.c_double), _i]),
    "hb_potrf_dist_workspace_bytes": (_sz, [_i, C.POINTER(Dist)]),
    "hb_potrf_lower_dist": (_i, [_c_f, _ll, _i, C.POINTER(Dist), _c_f, _sz, _c_f, _c_f, C.POINTER(Options)]),
    "hb_potrf_lower_bwd_dist": (_i, [_c_f, _ll, _c_f, _ll, _i, C.POINTER(Dist), _c_f, _sz, _c_f, C.POINTER(Options)]),
    "hb_gp_elbo_dist_workspace_bytes": (_sz, [C.POINTER(GpConfig), C.POINTER(Dist)]),
    "hb_gp_elbo_step_dist": (_i, [C.POINTER(GpConfig), C.POINTER(Dist), _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _sz, _c_f, _c_f]),
}

_lib: Optional[C.CDLL] = None


class HenbunB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the CUDA library; fail loudly if it has not been built (no fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HenbunB200Error(
            f"{LIB_PATH} not found: build it with `make` (or __graft_entry__.build()). "
            "henbun_b200 has no CPU or PyTorch fallback path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _install_option_plumbing(lib)
    # A/B switches from the environment (accuracy vs speed of the factorisations) edit the Python-side default
    if os.environ.get("HB_EXACT_BELOW") is not None:
        lib.hb_set_exact_below(int(os.environ["HB_EXACT_BELOW"]))
    if os.environ.get("HB_PANEL_REFINEMENT") is not None:
        lib.hb_set_panel_refinement(int(os.environ["HB_PANEL_REFINEMENT"]))
    _lib = lib
    return lib


# entry points whose LAST argument is `const hb_options*`, and whole-step entry points whose config struct carries it
_TRAILING_OPT = ("hb_gemm_ws", "hb_potrf_lower", "hb_potrf_lower_bwd", "hb_trsm_right_lower", "hb_gemm_presplit",
                 "hb_potrf_lower_dist", "hb_potrf_lower_bwd_dist")
_CFG_OPT = ("hb_gp_elbo_step", "hb_gp_elbo_step_dist", "hb_gp_elbo_step_f64", "hb_gp_elbo_f64_workspace_bytes",
            "hb_moe_gp_elbo_step_f64", "hb_moe_gp_f64_workspace_bytes",
            "hb_linop_prepare", "hb_linop_elbo_local", "hb_linop_elbo_update",
            "hb_amortised_elbo_step")


def _install_option_plumbing(lib):
    """Callers that do not pass options get the Python-side default OPTIONS; `lib.hb_set_*` edit that default.  (The C
    functions of those names were removed in round 2: configuration travels with the call.)"""
    def trailing(fn, nargs):
        def call(*args):
            if len(args) == nargs - 1:
                args = args + (C.byref(OPTIONS),)
            return fn(*args)
        call.__name__ = fn.__name__
        return call

    def cfg_first(fn):
        def call(cfg_ref, *args):
            cfg = getattr(cfg_ref, "_obj", None)
            if cfg is not None and not cfg.opt:
                cfg.opt = C.pointer(OPTIONS)
            return fn(cfg_ref, *args)
        call.__name__ = fn.__name__
        return call
    for name in _TRAILING_OPT:
        setattr(lib, name, trailing(getattr(lib, name), len(SIGNATURES[name][1])))
    for name in _CFG_OPT:
        setattr(lib, name, cfg_first(getattr(lib, name)))

    def set_engine(mode):
        if mode < 0 or mode > 3:
            return HB_ERR_ARG
        OPTIONS.gemm_engine = int(mode)
        return HB_OK

    def set_refinement(mode):
        OPTIONS.panel_refinement = int(mode) if 0 <= mode <= 3 else 2
        return OPTIONS.panel_refinement

    def set_field(field, conv=int):
        def f(v):
            setattr(OPTIONS, field, conv(v))
            return getattr(OPTIONS, field)
        return f
    lib.hb_set_gemm_engine = set_engine
    lib.hb_get_gemm_engine = lambda: OPTIONS.gemm_engine
    lib.hb_set_panel_refinement = set_refinement
    lib.hb_set_exact_below = set_field("exact_below", lambda v: max(0, int(v)))
    lib.hb_set_presplit_engine = set_field("presplit_engine", lambda v: 1 if v else 0)
    lib.hb_set_small_gp_kernel = set_field("small_gp_kernel", lambda v: 1 if v else 0)
    lib.hb_set_schedule = set_field("schedule", int)
    lib.hb_set_tc_option = lambda v: (setattr(OPTIONS, "tc_option", int(v)), HB_OK)[1]


_ERR = {HB_ERR_ARG: "invalid argument", HB_ERR_CUDA: "CUDA launch/runtime failure",
        HB_ERR_WORKSPACE: "workspace missing or too small"}


def check(rc: int, what: str) -> None:
    if rc == HB_ERR_ARG:
        raise ValueError(f"{what}: {_ERR[rc]}")
    if rc != HB_OK:
        raise HenbunB200Error(f"{what}: {_ERR.get(rc, rc)}")


def ptr(t: Optional[torch.Tensor]):
    """Device pointer of a contiguous-enough fp32/int32 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise HenbunB200Error("henbun_b200 kernels need CUDA tensors (no CPU fallback)")
    return C.c_void_p(t.data_ptr())


def stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def f32(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32 or not t.is_cuda:
        raise HenbunB200Error(f"expected a float32 CUDA tensor, got {t.dtype} on {t.device}")
    return t


_reduce_ws = {}


def reduce_ws(device=None) -> torch.Tensor:
    """Per-device scratch for reducing kernels (caller-owned, reused across calls on one stream)."""
    dev = torch.device(device if device is not None else torch.cuda.current_device())
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    w = _reduce_ws.get(key)
    if w is None:
        w = torch.empty(load().hb_reduce_workspace_bytes(), dtype=torch.uint8, device=dev)
        _reduce_ws[key] = w
    return w
