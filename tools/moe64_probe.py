"""Time of the float64 mixture-of-experts step (csrc/moe64.cu, BASELINE config 2) on the GPU, with CUDA events after
warm-up, next to

  hb_gp_elbo_step_f64 (one fp64 GP) at the same n and S, with a full-rank and with a diagonal q,
  hb_potrf_lower_f64 and hb_potrf_lower_bwd_f64 at the same n (the two longest phases of every GP chain), and
  the fp32 config-2 step through the model API (the eager tape: Optimizer.optimize with float_type float32),

at n in {2000, 8192} and S in {4, 10}, on the notebook's input (X = linspace(0, 6, n), jitter 3e-4, lengthscales 0.2, 1, 1,
q shapes full, full, diagonal).  The three GP chains of the mixture step run concurrently, so the step is expected well
below three single-GP steps: its ratio to the full-rank single step (two of its three chains are full rank) and to the
diagonal one are printed.  Prints the card's name, power limit and maximum SM clock (nvidia-smi, read only) first.

    python tools/moe64_probe.py [--out FILE]        (default: profiles/r4_moe64_probe.txt)
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


def problem(n, S, seed=0):
    rng = np.random.RandomState(seed)
    X = np.linspace(0, 6, n).reshape(-1, 1)
    Y = np.sin(0.1 * X[:, 0] ** 3) + 0.1 * rng.randn(n)
    sp_inv = lambda y: float(np.log(np.expm1(y - 1e-6)))
    segs = []
    for full, ell in ((1, 0.2), (1, 1.0), (0, 1.0)):
        sq = (0.3 * np.eye(n) + (0.2 / np.sqrt(n)) * np.tril(rng.randn(n, n))).ravel() if full else np.log(0.3) + 0.1 * rng.randn(n)
        segs += [0.1 * rng.randn(n), sq, [sp_inv(1.0)], [sp_inv(ell)]]
    segs.append([0.5, 0.3, -2.0])
    return X, Y, np.concatenate([np.asarray(s, np.float64).ravel() for s in segs]), {k: rng.randn(S, n) for k in "slr"}


def api_fp32_step(n, S, X, Y):
    """Optimizer.optimize step of the notebook model in float32 (no fused entry point: the eager tape)."""
    import henbun_b200 as hb
    import henbun_b200.tf as tf

    class ExpertGPR(hb.model.Model):
        def setUp(self):
            self.X = hb.param.Data(X); self.Y = hb.param.Data(Y.reshape(-1, 1))
            self.q_s = hb.variationals.Gaussian(shape=[n, 1], q_shape='fullrank')
            self.q_l = hb.variationals.Gaussian(shape=[n, 1], q_shape='fullrank')
            self.q_r = hb.variationals.Gaussian(shape=[n, 1], q_shape='diagonal')
            self.kern_s = hb.gp.kernels.UnitRBF(np.ones(1) * 0.2)
            self.kern_l = hb.gp.kernels.UnitRBF(np.ones(1))
            self.kern_r = hb.gp.kernels.UnitRBF(np.ones(1))
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.k_var_r = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            f_s = tf.matmul(self.kern_s.Cholesky(self.X), self.q_s)
            f_l = tf.matmul(self.kern_l.Cholesky(self.X), self.q_l)
            f_r = tf.matmul(self.kern_r.Cholesky(self.X), self.q_r) * tf.sqrt(self.k_var_r)
            fraction = tf.sigmoid(f_r)
            f = (fraction * f_s + (1 - fraction) * f_l) * self.k_var
            return tf.reduce_sum(hb.densities.gaussian(self.Y, f, self.var)) - self.KL()

    m = ExpertGPR()
    for nm in ("q_s", "q_l"):
        getattr(m, nm).q_sqrt = 0.3 * np.eye(n) + (0.2 / np.sqrt(n)) * np.tril(np.random.RandomState(1).randn(n, n))
    cfg = hb.settings.get_settings(); cfg.numerics.jitter_level = 3e-4
    with hb.settings.temp_settings(cfg):
        opt = m.ELBO()
        opt.compile(n_samples=S, verbose=False)
        assert opt.fused_entry is None
    fd = opt.feed_dict(None)
    return lambda: opt._step_once(fd)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r4_moe64_probe.txt"))
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    assert torch.cuda.is_available(), "moe64_probe measures on the GPU"
    lib = _lib.load()
    from henbun_b200 import ops
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    say("# " + smi.replace("\n", " | "))
    say("# CUDA-event time per step after warm-up, eps injected; the mixture step has q (full, full, diagonal), the single "
        "fp64 GP step is timed with a full-rank and with a diagonal q")
    st = stream()
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    for n in (2000, 8192):
        for S in (4, 10):
            reps = 10 if n == 2000 else 4
            X, Y, p, U = problem(n, S)
            d = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64).cuda()
            Xd, Yd, params = d(X), d(Y), d(p)
            Ud = {k: d(v) for k, v in U.items()}
            cfg = _lib.MoeGpConfig(n, 1, S, (C.c_int * 3)(1, 1, 1), (C.c_int * 3)(1, 1, 0), 3e-4, 0, (C.c_ulonglong * 3)(0, 0, 0))
            assert lib.hb_moe_gp_param_count(C.byref(cfg)) == params.numel()
            grads, out4 = torch.zeros_like(params), torch.zeros(4, dtype=torch.float64, device="cuda")
            wsb = lib.hb_moe_gp_f64_workspace_bytes(C.byref(cfg))
            ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

            def moe():
                _lib.check(lib.hb_moe_gp_elbo_step_f64(C.byref(cfg), ptr(Xd), ptr(Yd), ptr(params), ptr(Ud["s"]), ptr(Ud["l"]),
                                                       ptr(Ud["r"]), ptr(grads), ptr(out4), None, None, None, ptr(ws), wsb,
                                                       ptr(err), st), "hb_moe_gp_elbo_step_f64")
            ms_moe = timed(moe, reps)
            assert err.item() == 0
            del ws

            ms_gp = {}
            for full in (1, 0):
                gcfg = _lib.GpConfig(n, 1, S, 1, full, 3e-4, 0, 0)
                gp = d(np.concatenate([p[:n + n * n] if full else np.concatenate([p[:n], np.log(0.3) * np.ones(n)]),
                                       [0.54, 0.54, 0.5, -2.0]]))
                ggrads, gout4 = torch.zeros_like(gp), torch.zeros(4, dtype=torch.float64, device="cuda")
                gwsb = lib.hb_gp_elbo_f64_workspace_bytes(C.byref(gcfg))
                gws = torch.empty(gwsb, dtype=torch.uint8, device="cuda")

                def single():
                    _lib.check(lib.hb_gp_elbo_step_f64(C.byref(gcfg), ptr(Xd), ptr(Yd), ptr(gp), ptr(Ud["s"]), ptr(ggrads),
                                                       ptr(gout4), None, None, None, ptr(gws), gwsb, ptr(err), st),
                               "hb_gp_elbo_step_f64")
                ms_gp[full] = timed(single, reps)
                assert err.item() == 0
                del gws, gp, ggrads
            del Xd, Yd, params, grads, Ud

            ms_f = ms_b = None
            if S == 4:                                   # the factorisation does not depend on S
                Bm = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n))
                K = Bm @ Bm.T / n + 0.5 * torch.eye(n, dtype=torch.float64, device="cuda")
                del Bm
                pwsb = lib.hb_potrf_f64_workspace_bytes(n)
                pws = torch.empty(max(pwsb, 1), dtype=torch.uint8, device="cuda")
                Lf = K.clone()
                Lb = torch.tril(torch.ones_like(K))
                G = Lb.clone()

                def fwd():
                    Lf.copy_(K)
                    _lib.check(lib.hb_potrf_lower_f64(ptr(Lf), n, n, ptr(pws), pwsb, ptr(err), st), "hb_potrf_lower_f64")

                def bwd():
                    G.copy_(Lb)
                    _lib.check(lib.hb_potrf_lower_bwd_f64(ptr(Lf), n, ptr(G), n, n, ptr(pws), pwsb, st), "hb_potrf_lower_bwd_f64")
                copy_ms = timed(lambda: Lf.copy_(K), reps)
                ms_f = timed(fwd, reps) - copy_ms
                ms_b = timed(bwd, reps) - copy_ms
                del K, Lf, Lb, G, pws

            fp32 = api_fp32_step(n, S, X, Y)
            ms_api = timed(fp32, reps)
            flagged = ""
            try:
                ops.check_numerics()
            except FloatingPointError as e:
                flagged = f" (fp32 factorisation flagged: {e})"
            say(f"n={n} S={S}: hb_moe_gp_elbo_step_f64 (q full, full, diag) {ms_moe:.2f} ms | hb_gp_elbo_step_f64 q full "
                f"{ms_gp[1]:.2f} ms, q diag {ms_gp[0]:.2f} ms (mixture / full single = {ms_moe / ms_gp[1]:.2f}, "
                f"mixture / (2 full + 1 diag singles) = {ms_moe / (2 * ms_gp[1] + ms_gp[0]):.2f}) | "
                f"fp32 config-2 step through the API {ms_api:.2f} ms{flagged}")
            if ms_f is not None:
                say(f"n={n}: phases of one chain: hb_potrf_lower_f64 {ms_f:.2f} ms, hb_potrf_lower_bwd_f64 {ms_b:.2f} ms")
            del fp32
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
