"""Time of the float64 linear-operator pair (csrc/linop64.cu, BASELINE config 5) on the GPU, with CUDA events after warm-up:

  the whole fp64 step (hb_linop_elbo_local_f64 + hb_linop_elbo_update_f64 with TF-1 Adam),
  its two operator products F = Z A^T and Zbar = R A alone, on hb_gemm_f64 (TFLOP/s of 2 S M n each),
  its update call alone (GB/s of the Adam pass over the lower triangle: L_q, m, v read and written, 6 * 8 n^2 / 2 bytes), and
  the fp32 step (fused.LinearOperatorStep, the route float_type = float32 takes) in the same run,

at (M, n, S) = (65536, 16384, 64), the named size, and (16384, 4096, 64), eps injected.  Prints the card's name, power limit
and maximum SM clock (nvidia-smi, read only) first.

    python tools/linop64_probe.py [--out FILE]        (default: profiles/r5_linop64_probe.txt)
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from henbun_b200 import _lib  # noqa: E402
from henbun_b200._lib import ptr, stream, check  # noqa: E402


def timed(fn, reps, warm=2):
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
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r5_linop64_probe.txt"))
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    assert torch.cuda.is_available(), "linop64_probe measures on the GPU"
    lib = _lib.load()
    from henbun_b200.fused import LinearOperatorStep
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    say("# " + smi.replace("\n", " | "))
    say("# CUDA-event time per call after warm-up, eps injected")
    st = stream()
    for M, n, S in ((65536, 16384, 64), (16384, 4096, 64)):
        reps = 5
        gen = torch.Generator(device="cuda").manual_seed(0)
        A = torch.randn(M, n, device="cuda", dtype=torch.float64, generator=gen) / n ** 0.5
        y = A[:, :256] @ torch.randn(256, device="cuda", dtype=torch.float64, generator=gen)
        U = torch.randn(S, n, device="cuda", dtype=torch.float64, generator=gen)
        cfg = _lib.LinopConfig(M, M, n, S, 0, 0, 0)
        count = int(lib.hb_linop_param_count(C.byref(cfg)))
        params = torch.zeros(count, dtype=torch.float64, device="cuda")
        params[:n * n].view(n, n).copy_(0.1 * torch.eye(n, dtype=torch.float64, device="cuda"))
        params[n * n:n * n + n].normal_(0.0, 0.1, generator=gen)
        params[-1] = 0.3
        m, v = torch.zeros_like(params), torch.zeros_like(params)
        zbar = torch.empty(S * n + 4, dtype=torch.float64, device="cuda")
        out4 = torch.zeros(4, dtype=torch.float64, device="cuda")
        wsb = int(lib.hb_linop_f64_workspace_bytes(C.byref(cfg)))
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
        step = torch.ones(1, dtype=torch.int32, device="cuda")
        adam = _lib.AdamConfig(1e-6, 0.9, 0.999, 1e-8, -1.0, C.c_void_p(step.data_ptr()), 0)

        def local():
            check(lib.hb_linop_elbo_local_f64(C.byref(cfg), ptr(A), ptr(y), ptr(params), ptr(U), ptr(zbar), ptr(ws), wsb, st),
                  "hb_linop_elbo_local_f64")

        def update():
            check(lib.hb_linop_elbo_update_f64(C.byref(cfg), ptr(params), ptr(zbar), None, ptr(m), ptr(v), C.byref(adam),
                                               ptr(out4), ptr(ws), wsb, st), "hb_linop_elbo_update_f64")

        def whole():
            local()
            update()
        ms_step = timed(whole, reps)
        ms_upd = timed(update, reps)

        # the two operator products alone, on the same GEMM
        Z = U.clone()
        F = torch.empty(S, M, dtype=torch.float64, device="cuda")
        Zb = torch.empty(S, n, dtype=torch.float64, device="cuda")
        gws = torch.empty(8 << 20, dtype=torch.uint8, device="cuda")

        def fwd():
            check(lib.hb_gemm_f64(ptr(Z), n, 0, 0, ptr(A), n, 1, 0, ptr(F), M, 0, S, M, n, 1.0, 0.0, ptr(gws), 8 << 20, st),
                  "hb_gemm_f64")

        def back():
            check(lib.hb_gemm_f64(ptr(F), M, 0, 0, ptr(A), n, 0, 0, ptr(Zb), n, 0, S, n, M, 1.0, 0.0, ptr(gws), 8 << 20, st),
                  "hb_gemm_f64")
        ms_f, ms_b = timed(fwd, reps), timed(back, reps)
        flop = 2.0 * S * M * n
        gb = 6 * 8 * n * n / 2 / 1e9
        A32 = A.float()
        del A, F, Zb, gws, ws, m, v, params
        torch.cuda.empty_cache()

        st32 = LinearOperatorStep(A32, y.float(), S, lr=1e-6)
        st32.q_sqrt.copy_(0.1 * torch.eye(n, device="cuda"))
        st32.var_free.fill_(0.3)
        U32 = U.float()
        ms_32 = timed(lambda: st32.step(U32), reps)
        say(f"M={M} n={n} S={S}: fp64 step (local + update with Adam) {ms_step:.2f} ms | F = Z A^T {ms_f:.2f} ms "
            f"{flop / ms_f / 1e9:.1f} TFLOP/s, Zbar = R A {ms_b:.2f} ms {flop / ms_b / 1e9:.1f} TFLOP/s | update {ms_upd:.2f} ms "
            f"({gb / (ms_upd / 1e3):.0f} GB/s of the Adam pass) | fp32 step (presplit={st32.cfg.presplit}) {ms_32:.2f} ms, "
            f"fp64 / fp32 = {ms_step / ms_32:.1f}")
        del st32, A32, U32, y, U, Z
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
