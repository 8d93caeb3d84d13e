"""Rates of the float64 path (csrc/f64.cu) on the GPU, with CUDA events after warm-up, next to the fp32 step:

  hb_gemm_f64                          at 4096^3 and 8192^3 (useful FLOP 2 M N K)
  hb_potrf_lower_f64 / _bwd_f64        at n in {2000, 8192, 16384} (useful FLOP n^3/3 forward, 2 n^3/3 reverse)
  hb_gp_elbo_step_f64, S = 10          at the same n
  hb_gp_elbo_step (fp32), S = 10       at the same n

Prints the card's name, power limit and maximum SM clock (nvidia-smi, read only) first.  Operands of the 8192^3 product and
of the factorisations at n >= 8192 are larger than the 126 MB L2.

    python tools/f64_probe.py [--out FILE]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from henbun_b200 import _lib  # noqa: E402
from henbun_b200._lib import ptr, stream  # noqa: E402


def timed(fn, reps, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    assert torch.cuda.is_available(), "f64_probe measures on the GPU"
    lib = _lib.load()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    say("# " + smi.replace("\n", " | "))
    say("# FP64 tensor-core rate of NVIDIA's HGX B200 data sheet: 296 TFLOP/s for eight GPUs, 37 TFLOP/s per GPU (data-sheet figure)")
    st = stream()
    g = torch.Generator(device="cuda").manual_seed(0)

    for n in (4096, 8192):
        A = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
        B = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
        Cm = torch.empty(n, n, dtype=torch.float64, device="cuda")

        def run():
            _lib.check(lib.hb_gemm_f64(ptr(A), n, 0, 0, ptr(B), n, 0, 0, ptr(Cm), n, 0, n, n, n, 1.0, 0.0, None, 0, st),
                       "hb_gemm_f64")
        ms = timed(run, 10 if n == 4096 else 4)
        fl = 2.0 * n ** 3
        err = (torch.linalg.norm(Cm - A @ B) / torch.linalg.norm(A @ B)).item()
        say(f"hb_gemm_f64 {n}^3: {ms:.2f} ms, {fl / ms / 1e9:.1f} TFLOP/s (vs torch fp64 rel {err:.1e})")
        del A, B, Cm

    for n in (2000, 8192, 16384):
        Bm = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
        K = Bm @ Bm.T / n + 0.5 * torch.eye(n, dtype=torch.float64, device="cuda")
        del Bm
        wsb = lib.hb_potrf_f64_workspace_bytes(n)
        ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device="cuda")
        err = torch.zeros(1, dtype=torch.int32, device="cuda")
        L = K.clone()
        Lb = torch.tril(torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g))
        G = Lb.clone()

        def fwd():
            L.copy_(K)
            _lib.check(lib.hb_potrf_lower_f64(ptr(L), n, n, ptr(ws), wsb, ptr(err), st), "hb_potrf_lower_f64")

        def bwd():
            G.copy_(Lb)
            _lib.check(lib.hb_potrf_lower_bwd_f64(ptr(L), n, ptr(G), n, n, ptr(ws), wsb, st), "hb_potrf_lower_bwd_f64")
        reps = 5 if n < 16384 else 3
        copy_ms = timed(lambda: L.copy_(K), reps)
        ms_f = timed(fwd, reps) - copy_ms
        ms_b = timed(bwd, reps) - copy_ms
        assert err.item() == 0
        say(f"hb_potrf_lower_f64 n={n}: {ms_f:.2f} ms, {n ** 3 / 3 / ms_f / 1e9:.2f} TFLOP/s; "
            f"hb_potrf_lower_bwd_f64: {ms_b:.2f} ms, {2 * n ** 3 / 3 / ms_b / 1e9:.2f} TFLOP/s")
        del K, L, Lb, G, ws

        S, D = 10, 8
        rng = np.random.RandomState(n)
        X = rng.randn(n, D); Y = np.sin(X.sum(1) / np.sqrt(D)) + 0.1 * rng.randn(n)
        p = np.concatenate([0.1 * rng.randn(n), -1.0 + 0.1 * rng.randn(n), [0.54, 0.54, 0.3, -0.5]])
        U = rng.randn(S, n)
        for f64 in (True, False):
            dt = torch.float64 if f64 else torch.float32
            d = lambda a: torch.as_tensor(a, dtype=dt).cuda()
            cfg = _lib.GpConfig(n, D, S, 1, 0, 1e-3, 0, 0)
            Xd, Yd, Ud, params = d(X), d(Y), d(U), d(p)
            grads, out4 = torch.zeros_like(params), torch.zeros(4, dtype=dt, device="cuda")
            if f64:
                wsb = lib.hb_gp_elbo_f64_workspace_bytes(C.byref(cfg))
                ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

                def step():
                    _lib.check(lib.hb_gp_elbo_step_f64(C.byref(cfg), ptr(Xd), ptr(Yd), ptr(params), ptr(Ud), ptr(grads), ptr(out4),
                                                       None, None, None, ptr(ws), wsb, ptr(err), st), "hb_gp_elbo_step_f64")
            else:
                wsb = lib.hb_gp_elbo_workspace_bytes(C.byref(cfg))
                ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

                def step():
                    _lib.check(lib.hb_gp_elbo_step(C.byref(cfg), ptr(Xd), ptr(Yd), ptr(params), ptr(Ud), ptr(grads), ptr(out4),
                                                   ptr(ws), wsb, ptr(err), st), "hb_gp_elbo_step")
            ms = timed(step, reps)
            fl = n ** 3 / 3 + 2 * n ** 3 / 3
            say(f"{'hb_gp_elbo_step_f64' if f64 else 'hb_gp_elbo_step (fp32)'} n={n} S={S}: {ms:.2f} ms per step "
                f"({fl / ms / 1e9:.2f} TFLOP/s of factorisation FLOP n^3)")
            del ws, Xd, Yd, Ud, params, grads
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
