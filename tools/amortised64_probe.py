"""Time of the float64 amortised step (csrc/amortised64.cu, BASELINE config 4) on the GPU, with CUDA events after warm-up,
at the named size (784-512-512-2x64 encoder + mirrored decoder, sigmoid, minibatch B = 4096, S = 32, eps injected):

  the whole fp64 step (hb_amortised_elbo_step_f64 with TF-1 Adam), its achieved FLOP/s over the 3 x 2 x rows x in x out of
  every MatBias product (forward, dW, gx),
  the same step split into GEMM (the DMMA kernel and its split-K reductions) and non-GEMM kernel time, from a separate
  torch.profiler run, and
  the fp32 step (hb_amortised_elbo_step, the route float_type = float32 takes) in the same run.

Prints the card's name, power limit and maximum SM clock (nvidia-smi, read only) first.

    python tools/amortised64_probe.py [--out FILE]        (default: profiles/r6_amortised64_probe.txt)
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

ENC, DEC, B, S = [784, 512, 512, 128], [64, 512, 512, 784], 4096, 32


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


def config():
    c = _lib.AmortisedConfig()
    c.B, c.S, c.latent = B, S, DEC[0]
    c.n_enc, c.n_dec = len(ENC) - 1, len(DEC) - 1
    for i, w in enumerate(ENC): c.enc_nodes[i] = w
    for i, w in enumerate(DEC): c.dec_nodes[i] = w
    for i in range(len(ENC) - 2): c.enc_act[i] = 1
    for i in range(len(DEC) - 2): c.dec_act[i] = 1
    return c


def flops():
    f = sum(2.0 * B * ENC[i] * ENC[i + 1] for i in range(len(ENC) - 1))
    f += sum(2.0 * S * B * DEC[i] * DEC[i + 1] for i in range(len(DEC) - 1))
    return 3 * f


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r6_amortised64_probe.txt"))
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    assert torch.cuda.is_available(), "amortised64_probe measures on the GPU"
    lib = _lib.load()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    say("# " + smi.replace("\n", " | "))
    say("# CUDA-event time per call after warm-up, eps injected; GEMM / non-GEMM split from a separate torch.profiler run")
    st = stream()
    cfg = config()
    npar = int(lib.hb_amortised_param_count(C.byref(cfg)))
    gen = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn(B, ENC[0], device="cuda", dtype=torch.float64, generator=gen)
    U = torch.randn(S, B, DEC[0], device="cuda", dtype=torch.float64, generator=gen)
    params = 0.03 * torch.randn(npar, device="cuda", dtype=torch.float64, generator=gen)
    m, v = torch.zeros_like(params), torch.zeros_like(params)
    out4 = torch.zeros(4, dtype=torch.float64, device="cuda")
    wsb = int(lib.hb_amortised_f64_workspace_bytes(C.byref(cfg)))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    step = torch.ones(1, dtype=torch.int32, device="cuda")
    adam = _lib.AdamConfig(1e-6, 0.9, 0.999, 1e-8, -1.0, C.c_void_p(step.data_ptr()), 0)

    def step64():
        check(lib.hb_amortised_elbo_step_f64(C.byref(cfg), ptr(X), ptr(params), ptr(U), None, ptr(out4), ptr(m), ptr(v),
                                             C.byref(adam), ptr(ws), wsb, st), "hb_amortised_elbo_step_f64")
    reps = 10
    ms64 = timed(step64, reps)

    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            step64()
        torch.cuda.synchronize()
    gemm_us = other_us = 0.0
    for ev in prof.key_averages():
        t = ev.self_device_time_total if hasattr(ev, "self_device_time_total") else ev.self_cuda_time_total
        if "f64_kernel" in ev.key and ("gemm" in ev.key or "splitk" in ev.key):
            gemm_us += t
        elif t > 0:
            other_us += t
    gemm_ms, other_ms = gemm_us / 3e3, other_us / 3e3

    X32, U32, p32 = X.float(), U.float(), params.float()
    g32 = torch.zeros(npar, device="cuda")
    out32 = torch.zeros(4, device="cuda")
    wsb32 = int(lib.hb_amortised_workspace_bytes(C.byref(cfg)))
    del ws
    torch.cuda.empty_cache()
    ws32 = torch.empty(wsb32, dtype=torch.uint8, device="cuda")

    def step32():
        check(lib.hb_amortised_elbo_step(C.byref(cfg), ptr(X32), ptr(p32), ptr(U32), ptr(g32), ptr(out32), ptr(ws32), wsb32, st),
              "hb_amortised_elbo_step")
    ms32 = timed(step32, reps)
    f = flops()
    say(f"B={B} S={S} enc {'-'.join(map(str, ENC))} dec {'-'.join(map(str, DEC))}: fp64 step (with Adam) {ms64:.2f} ms, "
        f"{f / ms64 / 1e9:.1f} TFLOP/s over {f:.3g} FLOP of MatBias products | kernel time per step: GEMM {gemm_ms:.2f} ms "
        f"({f / gemm_ms / 1e9:.1f} TFLOP/s), non-GEMM {other_ms:.2f} ms | fp32 step (gradient only) {ms32:.2f} ms, "
        f"fp64 / fp32 = {ms64 / ms32:.1f}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
