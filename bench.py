#!/usr/bin/env python
"""Headline benchmark: ELBO + gradient (+ TF-1 Adam update) evaluations per second of the variational GP of
BASELINE.json config 3 (N=65536, D=8, S=64 MC samples, RBF kernel, blocked Cholesky), on N B200s of one node.

  python bench.py --gpus N --steps K --warmup W            # our arm
  python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference path (rank 0 only)
  python bench.py --workload c4|c5 ...                     # the other BASELINE configs as the main line

A step = one pass of the hot path on one batch of synthetic inputs: K(X,X)+jI -> Cholesky -> reparameterised sampler +
one-sample KL -> F = sqrt(k_var) L (s z) -> Gaussian log-likelihood -> full backward (incl. reverse-mode Cholesky and the
lengthscale gradient) -> Adam.  evals = S * N per step.
  value : inputs resident in HBM, hb_gp_elbo_step + hb_adam_tf1 through the C ABI, CUDA events around K steps.
  e2e   : the SAME step through the Henbun API a user calls -- ``m.ELBO_gaussian().optimize(maxiter=1)`` on a model whose
          objective is the notebook's Python (Optimizer.compile traces it and binds it to the fused entry point) -- with
          X, Y re-fed from host memory every step and the ELBO read back.
Multi-GPU: `value` is weak scaling in S (S samples per rank, each rank its own window of one Philox stream) on top of ONE
column-block-cyclic factorisation + reverse mode shared by the ranks (hb_gp_elbo_step_dist: panel broadcasts over NCCL, one
all-gather of Z / R, one all-reduce of the packed gradient per step); ``multi_gpu`` adds the strong-scaling figure (S in
total) and the round-1 path (every rank factors K itself).  The default line also carries short measurements of BASELINE
configs 1, 4 and 5 (``other_workloads``; C4 minibatch-sharded and C5 row-sharded when N > 1).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "elbo_grad_evals_per_sec"
UNIT = "evals/s (MC samples x data points / s)"
LENGTHSCALE = 0.5


def workload_string(n, D, S):
    return (f"variational GP regression N={n} D={D} S={S}/GPU, UnitRBF lengthscale={LENGTHSCALE} jitter=1e-5, mean-field q, "
            f"ELBO+grad+Adam (BASELINE config 3; lengthscale 0.5 instead of SURVEY's 1.0: K + 1e-5 I is not positive definite in "
            f"fp32 at lengthscale 1)")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c4", "c5"])
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--dim", type=int, default=8)
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--cpu-n", type=int, default=16384, help="size of the bounded CPU-baseline sample of our arm")
    ap.add_argument("--ref-n", type=int, default=12288, help="size of the bounded sample each step of the reference arm runs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short config 1 / 4 / 5 measurements")
    ap.add_argument("--no-api-leg", action="store_true", help="e2e through the C ABI only (skips the Henbun-API leg)")
    ap.add_argument("--engine", type=int, default=0, help="GEMM engine: 0 auto, 1 SIMT fp32, 2 tcgen05 3xTF32")
    ap.add_argument("--profile-csv", default=None, help="dump the per-launch GEMM events of the profiled step to this file")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs --impl ours (the reference arm draws other samples at another N)")
    return a


DUMP_BYTES = 60 << 20          # all files of --dump-outputs together, .npy headers included, stay under 64 MB


def dump_outputs(path, arrays):
    """Write each tensor of `arrays` ({name: fp32 or fp64 tensor}) as path/<name>.npy.  A tensor larger than its equal share of
    DUMP_BYTES is written as a sample of its flattened elements at seeded positions, the same in every run, so that the
    files of two builds compare element for element."""
    import torch
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = torch.as_tensor(t).detach()
        if t.numel() * t.element_size() > share:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), share // t.element_size()))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def extrapolation_factor(n_full, n_sample, S):
    """CPU time at n_full / CPU time at n_sample from the step's flop counts: n^3 (Cholesky n^3/3 + its reverse mode
    2n^3/3) scales cubically, the 6 n^2 S of the three sample projections quadratically."""
    r = n_full / n_sample
    q = 6.0 * S / (6.0 * S + n_sample)          # quadratic share at the sample size
    return (1.0 - q) * r ** 3 + q * r ** 2


def host_threads():
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1 to every rank: override it)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:  # pragma: no cover
        return max(1, os.cpu_count() or 1)


def cpu_baseline(n_full, D, S, n_sample, steps=3, warmup=1):
    """Oracle (torch-CPU fp32) ELBO+grad+Adam step on a bounded sample (median of `steps`), extrapolated by flop count."""
    from oracle import cpu_baseline as cb
    n_sample = min(n_sample, n_full)
    t, _, threads = cb.time_gpr_steps(n_sample, D, S, steps=steps, warmup=warmup, threads=host_threads())
    scale = extrapolation_factor(n_full, n_sample, S)
    t_full = t * scale
    return {
        "value": S * n_full / t_full, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": (f"torch-CPU fp32 oracle, full ELBO+grad+Adam step at N={n_sample}, D={D}, S={S}: "
                   f"{t:.3f} s/step (median of {steps}); extrapolated x{scale:.1f} to N={n_full} by flop count "
                   f"(n^3 Cholesky + reverse mode cubically, 6 n^2 S sample projections quadratically)"),
        "sample_n": n_sample, "sample_evals_per_sec": S * n_sample / t, "sample_s_per_step": t, "extrapolated": n_sample != n_full,
    }


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.TemporaryFile("w+")
        self.idx = gpu_index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        hi = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
        return {"sm_mhz": float(np.median(hi)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(pw)), "samples": len(sm)}


# ======================================================================================================================
# reference arm: the oracle port of the reference graph on the box's host cores (TensorFlow is not installable here)
# ======================================================================================================================
def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_baseline as cb
    n_s = min(a.ref_n, a.n)
    # same job as our arm at --gpus N: weak scaling in S, i.e. S * N samples per step on the one host.  Each of the K
    # timed steps is one full ELBO+grad+Adam step of the bounded sample (N = n_s); `value` extrapolates to the named N.
    S_tot = a.samples * max(1, a.gpus)
    t, _, threads = cb.time_gpr_steps(n_s, a.dim, S_tot, steps=max(1, a.steps), warmup=max(0, a.warmup), threads=host_threads(),
                                      reduce="mean")
    scale = extrapolation_factor(a.n, n_s, S_tot)
    val = S_tot * a.n / (t * scale)
    sample = (f"torch-CPU fp32 restatement of the reference graph (TensorFlow is not installable here), {a.steps} timed "
              f"ELBO+grad+Adam steps at N={n_s}, S={S_tot}: {t:.3f} s/step (mean); value extrapolated x{scale:.1f} to N={a.n} by flop "
              f"count (n^3 cubically, 6 n^2 S quadratically); ms_per_step is the MEASURED step of the bounded sample")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * t, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(a.n, a.dim, a.samples), "timing": "host wall clock, CPU only",
                   "sample_n": n_s, "extrapolation_factor": scale, "extrapolated_ms_per_full_step": 1e3 * t * scale},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ======================================================================================================================
# our arm
# ======================================================================================================================
class Dist:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ms(self, ms):
        if self.world > 1:
            t = self.torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return t.item()
        return ms

    def timed(self, fn, nsteps):
        """CUDA events on the current stream around nsteps calls, barrier + synchronize on both sides, max over ranks."""
        torch = self.torch
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record()
        for i in range(nsteps):
            fn(i)
        ev1.record()
        self.barrier()
        return self.max_ms(ev0.elapsed_time(ev1))


def peaks():
    """The ceilings the rooflines divide by: bf16 dense sustained TFLOP/s and HBM copy GB/s (BASELINE.md section 2)."""
    return 1415.5, 6550.0, "measured on one B200 at its 1,000 W power limit: bf16 dense sustained / HBM copy (BASELINE.md section 2)"


def ncu_traffic():
    """DRAM bytes of one captured launch of the dominant kernel (ncu --set full, summary committed in profiles/)."""
    try:
        tr = {}
        path = os.path.join(ROOT, "profiles", "r2_ncu_prof_h2_pair_r2.csv")
        for ln in open(path):
            c = ln.strip().split(",")
            if len(c) >= 3 and c[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                tr[c[0]] = float(c[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(c[2], 1.0)
        if len(tr) == 2:
            return {"bytes_per_launch": sum(tr.values()), "launch": "gemm_h2_pair_kernel, M=N=K=8192 (tools/h2_one.py)",
                    "algorithmic_bytes": 3 * 8192 * 8192 * 4, "source": "profiles/r2_ncu_prof_h2_pair_r2.csv (committed capture, not this run)"}
    except Exception:
        pass
    return None


class GpCabi:
    """Config 3 through the C ABI: hb_gp_elbo_step (+ all-reduce) + hb_adam_tf1 on caller-owned buffers."""

    def __init__(self, d, n, D, S, seed_rank_offset=True, shared=None, block=None, batch=None):
        """shared (default: whenever there is more than one rank): the ranks share ONE column-block-cyclic factorisation
        and reverse mode (hb_gp_elbo_step_dist, shard_samples = 1); False: every rank factors K itself (round 1)."""
        import torch
        from henbun_b200 import _lib, parallel
        from henbun_b200.synthetic import make_gp_problem, pack_gp_params
        self.d, self.n, self.D, self.S = d, n, D, S
        self.lib = lib = _lib.load()
        self.shared = (d.world > 1 and n >= 4096) if shared is None else bool(shared and d.world > 1)
        self.env = parallel.block_cyclic_env(block, batch, shard_samples=True) if self.shared else None
        X, Y, p = make_gp_problem(n, D, S, seed=0, lengthscale=LENGTHSCALE)
        self.X, self.Y, self.p = X, Y, p
        params_h = pack_gp_params(p)
        self.cfg = _lib.GpConfig(n, D, S, 1, 0, 1e-5, 1000, 0)
        self.npar = npar = lib.hb_gp_param_count(C.byref(self.cfg))
        assert npar == params_h.size
        dev = d.dev
        self.params = torch.from_numpy(params_h).to(dev)
        self.grads = torch.zeros(npar, device=dev)
        self.adam_m = torch.zeros(npar, device=dev); self.adam_v = torch.zeros(npar, device=dev)
        self.step_ctr = torch.zeros(1, dtype=torch.int32, device=dev)
        self.out4 = torch.zeros(4, device=dev)
        self.err = torch.zeros(1, dtype=torch.int32, device=dev)
        self.wsb = (lib.hb_gp_elbo_dist_workspace_bytes(C.byref(self.cfg), C.byref(self.env)) if self.shared
                    else lib.hb_gp_elbo_workspace_bytes(C.byref(self.cfg)))
        self.ws = torch.empty(self.wsb, dtype=torch.uint8, device=dev)
        self.Xd = torch.from_numpy(X).to(dev); self.Yd = torch.from_numpy(Y).to(dev)
        self.Xh = torch.from_numpy(X).pin_memory(); self.Yh = torch.from_numpy(Y).pin_memory()
        self.out_h = torch.zeros(4).pin_memory()
        self.it = 0
        self._lib = _lib

    def step(self, host_io=False):
        _lib, lib, d = self._lib, self.lib, self.d
        st = _lib.stream
        if host_io:      # the reference feeds Data through feed_dict on every session.run (param.py:701-705)
            self.Xd.copy_(self.Xh, non_blocking=True); self.Yd.copy_(self.Yh, non_blocking=True)
        # ranks read disjoint windows of one Philox stream: the union over ranks is the single-GPU draw of S * world samples
        per_step = (self.S * d.world * self.n + 3) // 4 * 4
        self.cfg.offset = C.c_ulonglong(self.it * per_step + (d.rank * self.S * self.n) // 4 * 4)
        if self.shared:
            _lib.check(lib.hb_gp_elbo_step_dist(C.byref(self.cfg), C.byref(self.env), _lib.ptr(self.Xd), _lib.ptr(self.Yd),
                                                _lib.ptr(self.params), None, _lib.ptr(self.grads), _lib.ptr(self.out4), _lib.ptr(self.ws),
                                                self.wsb, _lib.ptr(self.err), st()), "hb_gp_elbo_step_dist")
        else:
            _lib.check(lib.hb_gp_elbo_step(C.byref(self.cfg), _lib.ptr(self.Xd), _lib.ptr(self.Yd), _lib.ptr(self.params), None,
                                           _lib.ptr(self.grads), _lib.ptr(self.out4), _lib.ptr(self.ws), self.wsb, _lib.ptr(self.err), st()),
                       "hb_gp_elbo_step")
        if d.world > 1:
            d.dist.all_reduce(self.grads)          # one NCCL all-reduce of the packed gradient (sum); mean below
        _lib.check(lib.hb_increment_i32(_lib.ptr(self.step_ctr), st()), "hb_increment_i32")
        _lib.check(lib.hb_adam_tf1(_lib.ptr(self.params), _lib.ptr(self.grads), _lib.ptr(self.adam_m), _lib.ptr(self.adam_v), self.npar,
                                   -1.0 / d.world, 1e-3, 0.9, 0.999, 1e-8, _lib.ptr(self.step_ctr), 0, st()), "hb_adam_tf1")
        if host_io:
            self.out_h.copy_(self.out4, non_blocking=True)
        self.it += 1

    def check(self):
        self.d.barrier()
        elbo = self.out4[0].item()
        if self.d.world > 1:                       # a failing block sets the flag on its owner only
            self.d.dist.all_reduce(self.err, op=self.d.dist.ReduceOp.MAX)
        if self.err.item() != 0:
            raise RuntimeError(f"Cholesky failed: non-positive pivot at row {self.err.item() - 1}")
        if not math.isfinite(elbo):
            raise RuntimeError(f"non-finite ELBO {elbo}")
        return elbo

    def free(self):
        import torch
        for k in ("ws", "params", "grads", "adam_m", "adam_v", "Xd", "Yd"):
            setattr(self, k, None)
        torch.cuda.empty_cache()


def build_gpr_model(X, Y, p, lengthscale):
    """notebooks/GaussianProcess.ipynb:109-148 written against the mirrored API."""
    import henbun_b200 as hb
    import henbun_b200.tf as tf

    class GPR(hb.model.Model):
        def setUp(self):
            self.X = hb.param.Data(X)
            self.Y = hb.param.Data(Y.reshape(-1, 1))
            self.q = hb.variationals.Gaussian(shape=[X.shape[0], 1], q_shape='diagonal')
            self.kern = hb.gp.kernels.UnitRBF(np.ones(1) * lengthscale)
            self.k_var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO_gaussian(self):
            y_fit = tf.matmul(self.kern.Cholesky(self.X), self.q) * tf.sqrt(self.k_var)
            return tf.reduce_sum(hb.densities.gaussian(self.Y, y_fit, self.var)) - self.KL()

    m = GPR()
    m.q.q_mu = np.asarray(p["q_mu"]).reshape(-1)
    m.q.q_sqrt = np.asarray(p["q_sqrt"]).reshape(-1)
    m.q.scale = np.ones((1, 1)); m.k_var = np.ones(1); m.var = np.ones(1)
    return m


def api_leg(d, a, X, Y, p):
    """The e2e measurement: the step a Henbun user runs, host-fed every step."""
    import torch
    n, D, S = a.n, a.dim, a.samples
    m = build_gpr_model(X, Y, p, LENGTHSCALE)
    opt = m.ELBO_gaussian()
    opt.compile(n_samples=S * d.world, seed=1000, shard='samples', verbose=False)
    Xh, Yh = X, Y.reshape(-1, 1)
    last = [0.0]

    def step(_i):
        m.X = Xh; m.Y = Yh                      # re-fed from host memory every step (pinned staging + H2D inside optimize)
        obj = opt.optimize(maxiter=1)           # ends with the numerics check: one device->host read
        last[0] = float(obj)                    # the ELBO comes back to the host
    for i in range(min(a.warmup, 3)):
        step(i)
    ms = d.timed(step, a.steps)
    out = {"ms_per_step": ms / a.steps, "fused_entry": opt.fused_entry, "elbo_last": last[0]}
    del m, opt
    torch.cuda.empty_cache()
    return out


def run_c3(d, a):
    import torch
    from henbun_b200 import _lib
    lib = _lib.load()
    lib.hb_set_gemm_engine(a.engine)
    n, D, S = a.n, a.dim, a.samples
    g = GpCabi(d, n, D, S)
    for _ in range(a.warmup):
        g.step()
    g.check()

    clocks = ClockSampler(d.local)
    if d.rank == 0:
        clocks.start()
    l0 = lib.hb_launch_count()
    try:
        ms = d.timed(lambda i: g.step(), a.steps)
    finally:                                   # the nvidia-smi sampler must not outlive a failing step
        clk = clocks.stop() if d.rank == 0 else None
    launches = lib.hb_launch_count() - l0
    if a.dump_outputs and d.rank == 0:         # out4 = {ELBO, loglik_sum, kl_sum, 0}; params after the step's Adam update
        dump_outputs(a.dump_outputs, {"out4": g.out4, "grads": g.grads, "params": g.params})
    ms_cabi_e2e = d.timed(lambda i: g.step(host_io=True), min(a.steps, 3)) / min(a.steps, 3)
    # separate, untimed passes for the evidence: per-launch GEMM events (roofline) and per-phase events
    d.barrier()
    # the timed step overlaps the narrow steps of a block (chain stream) with the trailing updates (caller's stream);
    # for per-launch durations the same products are issued on one stream (hb_options.lookahead = 0)
    _lib.OPTIONS.lookahead = 0
    g.step()
    lib.hb_profile_begin(200000)
    ms_prof = d.timed(lambda i: g.step(), 1)
    buf = (C.c_double * 8)()
    lib.hb_profile_end_ex(buf)
    _lib.OPTIONS.lookahead = 1
    prof = list(buf)
    if a.profile_csv and d.rank == 0:
        lib.hb_profile_dump_csv(a.profile_csv.encode())
    lib.hb_phase_begin()
    g.step()                                   # every rank steps (the step holds a collective); rank 0 reports
    pbuf = (C.c_double * 16)()
    npz = lib.hb_phase_end(pbuf, 16)
    names = ["scalars+gram_fwd", "potrf", "sampler+F+loglik+W", "sampler_bwd+Lbar", "potrf_bwd", "gram_bwd+scalar_grads"]
    phases = {names[i] if i < len(names) else f"phase{i}": round(pbuf[i], 3) for i in range(max(npz, 0))}
    elbo = g.check()
    X, Y, p = g.X, g.Y, g.p
    shared = g.shared
    g.free()

    # strong scaling (same S in total, split over the ranks) and the round-1 path (every rank factors K itself)
    multi = None
    if d.world > 1 and shared:
        multi = {}
        if S % d.world == 0:
            gs = GpCabi(d, n, D, S // d.world)
            for _ in range(2):
                gs.step()
            gs.check()
            k = min(a.steps, 3)
            multi["strong"] = {"samples_total": S, "samples_per_rank": S // d.world, "ms_per_step": d.timed(lambda i: gs.step(), k) / k,
                               "what": "the single-GPU job (S samples in total) on N ranks: shared factorisation, S / N samples per rank"}
            gs.free()
        gr = GpCabi(d, n, D, S, shared=False)
        for _ in range(2):
            gr.step()
        gr.check()
        k = min(a.steps, 3)
        multi["replicated"] = {"samples_per_rank": S, "ms_per_step": d.timed(lambda i: gr.step(), k) / k,
                               "what": "round-1 path: every rank factors K itself, samples sharded, one all-reduce"}
        gr.free()

    # like-for-like pair at the CPU sample size (GPU side; the CPU side is cpu_baseline.sample_s_per_step)
    same_n = None
    if d.world == 1 and not a.no_cpu_baseline and a.cpu_n < n:
        gs = GpCabi(d, a.cpu_n, D, S)
        for _ in range(3):
            gs.step()
        gs.check()
        same_n = {"n": a.cpu_n, "gpu_ms_per_step": d.timed(lambda i: gs.step(), 5) / 5}
        gs.free()

    api, api_error = None, None
    if not a.no_api_leg:
        try:
            api = api_leg(d, a, X, Y, p)
        except Exception as e:       # the main line must survive; e2e then falls back to the host-fed C-ABI step and says why
            api_error = f"{type(e).__name__}: {e}"[:300]
            torch.cuda.empty_cache()

    if d.rank != 0:
        return None
    evals = float(S) * n * d.world
    peak, _hbm, peak_src = peaks()
    n_gemm, gemm_ms, gemm_flop, n_pair, pair_ms, pair_flop, h2_ms, h2_flop = prof[:8]
    achieved = gemm_flop / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    h2_achieved = h2_flop / (h2_ms * 1e-3) / 1e12 if h2_ms > 0 else 0.0
    eng = lib.hb_get_gemm_engine()
    e2e_ms = api["ms_per_step"] if api else ms_cabi_e2e
    line = {
        "metric": METRIC, "value": evals * a.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": d.world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": workload_string(n, D, S),
            "parallelism": (f"ONE column-block-cyclic factorisation + reverse mode shared by {d.world} ranks (panel broadcasts over "
                            f"NCCL), samples sharded: S={S} per rank (weak scaling in S), one all-gather of Z/R + one all-reduce "
                            f"of the packed gradient per step") if shared else
                           f"sample-sharded (weak scaling in S), {d.world} rank(s), factorisation on every rank",
            "schedule": "right-looking two-stream schedule over column blocks (hb_options.schedule = 0: auto)",
            "l2": "inputs larger than L2 (K/L and Lbar/Kbar are N^2 fp32 = %.1f GB each)" % (4.0 * n * n / 1e9),
            "eps": "device Philox-4x32-10, regenerated in the backward; ranks read disjoint windows of one stream",
            "gemm_engine": {0: "auto", 1: "simt-fp32", 2: "tcgen05", 3: "simt-kloop"}.get(eng, str(eng)),
            "presplit_engine": bool(_lib.OPTIONS.presplit_engine),
            "elbo_last": elbo,
        },
        "e2e": {"value": evals / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": int(X.size * 4 + Y.size * 4), "d2h_bytes_per_step": 8,
                "ms_per_step": e2e_ms,
                "api": ("model.ELBO_gaussian().optimize(maxiter=1) on the notebook's objective written against the mirrored Henbun API "
                        "(compile() traced it and bound it to " + str(api and api["fused_entry"]) + "), X/Y re-assigned from host "
                        "arrays every step, ELBO read back") if api else
                       "hb_gp_elbo_step + hb_adam_tf1 through the C ABI, X/Y fed from pinned host memory every step",
                "c_abi_ms_per_step": ms_cabi_e2e, "api_ms_per_step": api["ms_per_step"] if api else None,
                **({"api_error": api_error} if api_error else {})},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": {
            "bound": "tensor",
            "kernel": "gemm_h2_pair_kernel (tcgen05 cta_group::2, kind::f16 on fp16 hi/lo shadow operands, 3 MMAs per k-step): the big "
                      "products of potrf / potrf_bwd",
            "achieved": h2_achieved, "peak": peak, "unit": "TFLOP/s", "frac": h2_achieved / peak if peak else None,
            "traffic": ncu_traffic(), "peak_source": peak_src,
            "kernel_ms_per_step": h2_ms, "kernel_share_of_step": h2_ms / ms_prof if ms_prof > 0 else None,
            "useful_flop_per_step": h2_flop,
            "all_level3": {"what": "every GEMM launch of the step (pre-split pair kernel, in-kernel-split tcgen05 kernels, short-K SIMT)",
                           "launches": int(n_gemm), "ms_per_step": gemm_ms, "useful_flop_per_step": gemm_flop,
                           "achieved": achieved, "frac": achieved / peak if peak else None,
                           "share_of_step": gemm_ms / ms_prof if ms_prof > 0 else None},
            "note": ("fp32 parity (1e-5) needs a split product: operands are split once into fp16 hi/lo pairs (22 mantissa bits) and "
                     "multiplied as hi*hi + lo*hi + hi*lo = 3 tensor-pipe slots where a plain bf16 GEMM needs 1, i.e. frac <= 0.333 "
                     "against the bf16 peak for this formulation (round 1: tf32 + 2 bf16 terms = 4 slots, 0.25)"),
            "how": "CUDA-event pair around every GEMM launch of one extra (untimed) step on the launching stream; achieved = useful "
                   "FLOP (trapezoid / block-mask shares counted, padding not) / summed launch time.  The timed steps run the block "
                   "chain and the trailing updates on two concurrent streams; this pass issues the same products on ONE "
                   "stream (hb_options.lookahead = 0) so that a launch's duration is its own",
            "serialised_step_ms": ms_prof,
            "step_level": {"what": "useful level-3 FLOP of the step / ms_per_step of the TIMED (two-stream) steps",
                           "achieved": gemm_flop / (ms / a.steps * 1e-3) / 1e12 if ms > 0 else None,
                           "frac": gemm_flop / (ms / a.steps * 1e-3) / 1e12 / peak if ms > 0 and peak else None},
        },
        "phases_ms": phases,
    }
    if multi:
        line["multi_gpu"] = multi
    if d.world == 1 and not a.no_cpu_baseline:
        cb = cpu_baseline(n, D, S, a.cpu_n)
        line["cpu_baseline"] = cb
        if same_n:
            same_n["cpu_s_per_step"] = cb["sample_s_per_step"]
            same_n["measured_ratio"] = cb["sample_s_per_step"] * 1e3 / same_n["gpu_ms_per_step"]
            same_n["note"] = "both sides measured at this N in this run (no extrapolation)"
            line["same_n_pair"] = same_n
    return line


# ---------------------------------------------------------------------------------------------------------------------
# the other BASELINE configs (short measurements; main line with --workload c4|c5)
# ---------------------------------------------------------------------------------------------------------------------
def run_c1(d, steps=200):
    """Config 1 (GP regression N=100, 1-D, full-covariance q, S=10) through the fused C entry: eager launches and a CUDA
    graph replay of the same step."""
    import torch
    from henbun_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(0)
    n, D, S, jitter = 100, 1, 10, 1e-3
    X = np.linspace(0, 6, n).reshape(-1, 1).astype(np.float32); Y = (np.sin(X[:, 0]) + 0.3 * rng.randn(n)).astype(np.float32)
    cfg = _lib.GpConfig(n, D, S, 1, 1, jitter, 0, 0)
    npar = lib.hb_gp_param_count(C.byref(cfg))
    q_sqrt = (0.3 * np.eye(n) + 0.02 * np.tril(rng.randn(n, n))).astype(np.float32)
    dev = d.dev
    params = torch.tensor(np.concatenate([0.1 * rng.randn(n), q_sqrt.ravel(), [0.54], [0.54], [0.54], [-0.5]]).astype(np.float32), device=dev)
    grads = torch.zeros(npar, device=dev); am = torch.zeros(npar, device=dev); av = torch.zeros(npar, device=dev)
    ctr = torch.zeros(1, dtype=torch.int32, device=dev); out4 = torch.zeros(4, device=dev); err = torch.zeros(1, dtype=torch.int32, device=dev)
    wsb = lib.hb_gp_elbo_workspace_bytes(C.byref(cfg)); ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    Xd, Yd = torch.tensor(X, device=dev), torch.tensor(Y, device=dev)

    def step(it):
        cfg.offset = C.c_ulonglong(it * ((S * n + 3) // 4 * 4))
        _lib.check(lib.hb_gp_elbo_step(C.byref(cfg), _lib.ptr(Xd), _lib.ptr(Yd), _lib.ptr(params), None, _lib.ptr(grads), _lib.ptr(out4),
                                       _lib.ptr(ws), wsb, _lib.ptr(err), _lib.stream()), "hb_gp_elbo_step")
        _lib.check(lib.hb_increment_i32(_lib.ptr(ctr), _lib.stream()), "inc")
        _lib.check(lib.hb_adam_tf1(_lib.ptr(params), _lib.ptr(grads), _lib.ptr(am), _lib.ptr(av), npar, -1.0, 1e-3, 0.9, 0.999, 1e-8,
                                   _lib.ptr(ctr), 0, _lib.stream()), "adam")
    def measure():
        for i in range(20):
            step(i)
        l0_ = lib.hb_launch_count(); step(20); per_ = lib.hb_launch_count() - l0_
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for i in range(steps):
            step(21 + i)
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps * 1e3, per_
    lib.hb_set_small_gp_kernel(0)
    try:
        multi_us, multi_launches = measure()               # the 23-kernel path (round 1)
    finally:
        lib.hb_set_small_gp_kernel(1)
    for i in range(20):
        step(i)
    l0 = lib.hb_launch_count(); step(20); per_step = lib.hb_launch_count() - l0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); ev0.record()
    for i in range(steps):
        step(21 + i)
    ev1.record(); torch.cuda.synchronize()
    eager = ev0.elapsed_time(ev1) / steps * 1e3
    # the same step as ONE persistent CTA with Adam inside (csrc/gp_small.cu; also the float64 route)
    adam = _lib.AdamConfig(1e-3, 0.9, 0.999, 1e-8, -1.0, C.c_void_p(ctr.data_ptr()), 0)

    def one(it):
        cfg.offset = C.c_ulonglong(it * ((S * n + 3) // 4 * 4))
        lib.hb_increment_i32(_lib.ptr(ctr), _lib.stream())
        _lib.check(lib.hb_gp_small_step(C.byref(cfg), _lib.ptr(Xd), _lib.ptr(Yd), _lib.ptr(params), None, _lib.ptr(grads), _lib.ptr(out4),
                                        _lib.ptr(am), _lib.ptr(av), C.byref(adam), _lib.ptr(ws), wsb, _lib.ptr(err), _lib.stream()),
                   "hb_gp_small_step")
    for i in range(10):
        one(1000 + i)
    torch.cuda.synchronize(); ev0.record()
    for i in range(steps):
        one(1100 + i)
    ev1.record(); torch.cuda.synchronize()
    single = ev0.elapsed_time(ev1) / steps * 1e3
    return {"workload": "BASELINE config 1: GP regression N=100 1-D, full-covariance q, S=10, fused C entry + Adam",
            "us_per_step": eager, "evals_per_sec": S * n / eager * 1e6, "kernels_per_step": int(per_step),
            "with_adam_inside_the_kernel_us_per_step": single,
            "multi_kernel_path_us_per_step": multi_us, "multi_kernel_path_launches": int(multi_launches),
            "note": "default = ONE persistent CTA for the whole ELBO + gradient (blocked shared-memory factorisation, closed-form reverse mode) "
                    "+ the Adam launch; hb_options.small_gp_kernel = 0 is the multi-kernel path",
            "elbo_last": float(out4[0]), "err_flag": int(err.item())}


def run_c5(d, steps, warmup, dump=None, S=64, M=65536, n=16384):
    """Config 5: full-covariance q over n = 16384 latents seen through a dense 65536 x 16384 operator; the operator is
    row-sharded over the ranks (strong scaling in M), one all-reduce of [S n + 4] floats per step."""
    import torch
    from henbun_b200.fused import LinearOperatorStep
    from henbun_b200 import parallel
    first, rows = parallel.shard_rows(M, d.world, d.rank)
    gen = torch.Generator(device=d.dev).manual_seed(0)
    w_true = torch.randn(256, device=d.dev, generator=gen)
    gen_r = torch.Generator(device=d.dev).manual_seed(100 + d.rank)
    A = torch.randn(rows, n, device=d.dev, generator=gen_r) / np.sqrt(n)
    y = A[:, :256] @ w_true + 0.1 * torch.randn(rows, device=d.dev, generator=gen_r)
    st = LinearOperatorStep(A, y, S, m_total=M, lr=1e-3)
    st.q_sqrt.copy_(0.1 * torch.eye(n, device=d.dev) + 1e-3 * torch.tril(torch.randn(n, n, device=d.dev, generator=gen)))
    yh = y.cpu().pin_memory(); out_h = torch.zeros(4).pin_memory()
    it = [0]

    def step(host_io):
        if host_io:
            st.y.copy_(yh, non_blocking=True)
        st.step(None, it[0]); it[0] += 1
        if host_io:
            out_h.copy_(st.out4, non_blocking=True)
    for _ in range(warmup):
        step(False)
    ms = d.timed(lambda i: step(False), steps) / steps
    if dump and d.rank == 0:
        dump_outputs(dump, {"out4": st.out4, "q_mu": st.q_mu, "q_sqrt": st.q_sqrt, "var_free": st.var_free})
    ms_e2e = d.timed(lambda i: step(True), steps) / steps
    tri = n * (n + 1) / 2
    bytes_step = 2 * 4.0 * rows * n + 4 * tri + 4.0 * S * (3 * rows + 4 * n) + 6 * 4 * tri + 4.0 * S * n * 4
    _tf, hbm, src = peaks()
    evals = float(S) * M
    out = {"workload": f"BASELINE config 5: n={n} full-covariance q, A {M}x{n} row-sharded over {d.world} rank(s), S={S}, fused "
                       f"hb_linop_elbo_local/_update (ELBO+grad+Adam)",
           "metric": METRIC, "value": evals / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "scaling": "strong", "n_gpus": d.world,
           "e2e": {"value": evals / (ms_e2e * 1e-3), "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(rows * 4), "d2h_bytes_per_step": 16,
                   "api": "LinearOperatorStep.step through the C ABI, y re-fed from pinned host memory, ELBO read back"},
           "roofline": {"bound": "hbm", "achieved": bytes_step / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                        "frac": bytes_step / (ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes_per_rank_step": bytes_step, "peak_source": src},
           "elbo_last": float(st.out4[0])}
    del st, A
    torch.cuda.empty_cache()
    return out


def run_c4(d, steps, warmup, dump=None, n_data=1000000, B=4096, S=32, latent=64):
    """Config 4: amortised encoder 784-512-512-2x64 + mirrored decoder, 1 M synthetic points resident in HBM, minibatch
    4096 (split over the ranks), S = 32, through the Henbun API."""
    import torch
    import henbun_b200 as hb
    import henbun_b200.tf as tf

    class Amortised(hb.model.Model):
        def setUp(self, X=None):
            self.X = hb.param.MinibatchData(X)
            self.enc = hb.nn.NeuralNet([784, 512, 512, 2 * latent], stddev=0.05)
            self.dec = hb.nn.NeuralNet([latent, 512, 512, 784], stddev=0.05)
            self.q_local = hb.variationals.Normal([latent], collections=hb.param.graph_key.LOCAL)
            self.var = hb.param.Variable(shape=[1], transform=hb.transforms.positive)

        @hb.model.AutoOptimize()
        def ELBO(self):
            self.q_local = self.enc(self.X)
            x_rec = self.dec(self.q_local)
            return tf.reduce_sum(hb.densities.gaussian(self.X, x_rec, self.var)) - self.KL(hb.param.graph_key.LOCAL)

    rows = n_data // d.world                       # each rank holds its shard of the data set
    X = np.random.default_rng(d.rank).standard_normal((rows, 784), dtype=np.float32)
    np.random.seed(1234)                           # Variable init draws from numpy's global RNG: same weights on every rank
    m = Amortised(X=X)
    np.random.seed(99 + d.rank)                    # ... the Indexer too: ranks draw different minibatches
    opt = m.ELBO()
    opt.compile(n_samples=S, seed=7, shard='batch', verbose=False)
    last = [0.0]

    def step(read):
        obj = opt.optimize(maxiter=1, minibatch_size=B)
        if read:
            last[0] = float(obj)
    for _ in range(warmup):
        step(False)
    ms = d.timed(lambda i: step(False), steps) / steps
    if dump and d.rank == 0:                   # the objective optimize() returned and the flat parameter vector it updated
        dump_outputs(dump, {"elbo": opt.last_objective, "params": opt._flat})
    ms_e2e = d.timed(lambda i: step(True), steps) / steps
    flop = 3 * 2.0 * B * (784 * 512 + 512 * 512 + 512 * 2 * latent) + 3 * 2.0 * B * S * (latent * 512 + 512 * 512 + 512 * 784)
    tf_peak, _h, src = peaks()
    evals = float(S) * B
    out = {"workload": f"BASELINE config 4: encoder 784-512-512-2x{latent} + mirrored decoder, {n_data} points resident, minibatch {B} "
                       f"over {d.world} rank(s), S={S}, Henbun API (" + str(opt.fused_entry or "eager tape over the CUDA operators") + ")",
           "metric": METRIC, "value": evals / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "scaling": "strong", "n_gpus": d.world,
           "e2e": {"value": evals / (ms_e2e * 1e-3), "ms_per_step": ms_e2e, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 8,
                   "api": "model.ELBO().optimize(maxiter=1, minibatch_size=4096): data resident, minibatch indices drawn and rows gathered on the device, ELBO read back"},
           "roofline": {"bound": "tensor", "achieved": flop / d.world / (ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                        "frac": flop / d.world / (ms * 1e-3) / 1e12 / tf_peak, "algorithmic_flop_per_step": flop, "peak_source": src},
           "elbo_last": last[0]}
    del m, opt, X
    torch.cuda.empty_cache()
    return out


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    # stdout carries exactly ONE line, the JSON: anything a library prints there meanwhile (NCCL's version banner when a
    # communicator is created) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        d, line = measure(a)
    finally:
        sys.stdout.flush()
        try:
            C.CDLL(None).fflush(None)          # C stdio buffers too, before fd 1 is the real stdout again
        except Exception:
            pass
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if d.rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
    if d.world > 1:
        d.dist.destroy_process_group()


def measure(a):
    d = Dist()
    line = None
    if a.workload == "c3":
        line = run_c3(d, a)
        if not a.no_extras:
            extras = {}
            for name, fn in (("c1", lambda: run_c1(d) if d.world == 1 else None),
                             ("c5", lambda: run_c5(d, 10, 3)),
                             ("c4", lambda: run_c4(d, 10, 3))):
                try:
                    r = fn()
                except Exception as e:  # the main line must survive a failing side measurement
                    r = {"error": f"{type(e).__name__}: {e}"[:300]}
                    try:
                        d.torch.cuda.empty_cache()
                    except Exception:
                        pass
                if r is not None:
                    extras[name] = r
            if line is not None:
                line["other_workloads"] = extras
    else:
        r = (run_c5 if a.workload == "c5" else run_c4)(d, a.steps, a.warmup, a.dump_outputs)
        if d.rank == 0:
            line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": d.world, "steps": a.steps, "warmup": a.warmup,
                    "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                    "data": "synthetic", "config": {"workload": r["workload"]}, "e2e": dict(r["e2e"], unit=UNIT),
                    "roofline": r["roofline"], "gpu_launches": None}
    return d, line


if __name__ == "__main__":
    main()
