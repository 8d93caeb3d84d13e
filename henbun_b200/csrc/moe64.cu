// float64 mixture-of-experts GP regression (notebooks/Expert_GPR.ipynb:101-149, BASELINE config 2): the ELBO + gradient
// (+ TF-1 Adam) of two GP experts s, l and a GP gate r in double, the reference's float_type = float64 (henbunrc:7).
//
//   G_e  = a_e Z_e L_e^T   (a_e = softplus(scale_e) + 1e-6, Z_e the sampler of q_e, L_e = chol(rbf_{ell_e}(X) + jitter I))
//   frac = sigmoid(sqrt(k_var_r) G_r),  f = k_var (frac G_s + (1 - frac) G_l),  ELBO = [sum gaussian(Y, f, var) - sum_e KL_e] / S
//
// Each GP runs the per-GP kernels of f64.cu's step on its own slice of the workspace.  The three chains are independent
// except at the mixture log-likelihood (which needs every F_e and hands back every residual R_e = d ll / d G_e / S) and at
// the scalar chain rules, so expert s runs on the caller's stream and l, r on two side streams forked from it by events
// and joined back before those two kernels: at n = 2000 one factorisation plus its reverse mode is a chain of latency-bound
// leaves and panel solves, and three of them overlap.  Every kernel reduces in a fixed order and nothing is summed across
// experts outside the joins, so results are bitwise repeatable.  When the call returns the caller's stream has waited on all
// of the work.
#include "../../include/henbun_b200.h"
#include "f64.cuh"
#include "gemm.cuh"
#include "tmath.cuh"
#include <algorithm>

namespace hb {
namespace {

constexpr int NE = 3;                                    // experts s, l and the gate r, in packing order

// mix: [0] k_var, [1] k_var_r, [2] var, [3] loglik, [4] sum E^2, [5] d ll / d k_var, [6] sum (d ll / d g) G_r,
//      [7..10) d ELBO / d a_e
constexpr int MIX_N = 16;
constexpr int MIX_THREADS = 512;                         // one CTA; 128 registers a thread keep the 7 sums out of local memory

struct MoeLayout {
  size_t seg_params[NE];                                 // offset of each expert's segment in params / grads (elements)
  size_t off_K[NE], off_G[NE], off_Z[NE], off_F[NE], off_R[NE], off_W[NE], off_U[NE], off_sc[NE], off_red[NE], off_split[NE];
  size_t off_mix, total;
  size_t nparams;
};

size_t seg_count(const hb_moe_gp_config& c, int e) {
  return (size_t)c.n + (c.q_fullrank[e] ? (size_t)c.n * c.n : (size_t)c.n) + 1 + c.n_ell[e];
}

MoeLayout moe_layout(const hb_moe_gp_config& c) {
  MoeLayout L{};
  const size_t nn = (size_t)c.n * c.n * sizeof(double), sn = (size_t)c.S * c.n * sizeof(double);
  size_t o = 0, p = 0;
  for (int e = 0; e < NE; ++e) {
    L.seg_params[e] = p; p += seg_count(c, e);
    L.off_K[e] = o; o += align256(nn);
    L.off_G[e] = o; o += align256(nn);
    L.off_Z[e] = o; o += align256(sn);
    L.off_F[e] = o; o += align256(sn);
    L.off_R[e] = o; o += align256(sn);
    L.off_W[e] = o; o += align256(sn);
    L.off_U[e] = o; o += align256(sn);
    L.off_sc[e] = o; o += align256((size_t)(SC_ELL + c.n_ell[e]) * sizeof(double));
    L.off_red[e] = o; o += align256((size_t)kGramBwdBlocks * c.n_ell[e] * sizeof(double));
    L.off_split[e] = o; o += align256(kSplitWsBytes);
  }
  L.off_mix = o; o += align256(MIX_N * sizeof(double));
  L.total = o;
  L.nparams = p + 3;                                     // + k_var, k_var_r, var
  return L;
}

bool config_ok(const hb_moe_gp_config& c) {
  if (c.n <= 0 || c.D <= 0 || c.D > 32 || c.S <= 0) return false;
  for (int e = 0; e < NE; ++e) {
    if (c.n_ell[e] != 1 && c.n_ell[e] != c.D) return false;
    if (c.q_fullrank[e] != 0 && c.q_fullrank[e] != 1) return false;
  }
  return true;
}

// the per-expert pointers the kernels below take by value
struct MoePtrs {
  const double* p_scale[NE];
  const double* p_ell[NE];
  double* g_scale[NE];
  double* g_ell[NE];
  int n_ell[NE];
  double* sc[NE];
  const double* red[NE];
  const double* F[NE];
  double* R[NE];
  const double* p_glob;                                  // [k_var, k_var_r, var]
  double* g_glob;
  double* mix;
};

// every transformed parameter: a_e (sc[0] and, as the amp the per-GP kernels read, sc[3]), the lengthscales, and the three
// shared scalars
__global__ void moe64_prep_kernel(MoePtrs p) {
  for (int e = 0; e < NE; ++e) {
    if (threadIdx.x == 0) {
      const double a = t_softplus<double>(*p.p_scale[e]) + 1e-6;
      p.sc[e][0] = a; p.sc[e][3] = a;
    }
    for (int d = threadIdx.x; d < p.n_ell[e]; d += blockDim.x) p.sc[e][SC_ELL + d] = t_softplus<double>(p.p_ell[e][d]) + 1e-6;
  }
  if (threadIdx.x < 3) p.mix[threadIdx.x] = t_softplus<double>(p.p_glob[threadIdx.x]) + 1e-6;
}

// The mixture log-likelihood, one CTA in a fixed order: with G_e = a_e F_e, g = sqrt(k_var_r) G_r, frac = sigmoid(g),
// m = frac G_s + (1 - frac) G_l, E = Y - k_var m, it writes R_s = k_var frac E / var / S, R_l = k_var (1 - frac) E / var / S,
// R_r = sqrt(k_var_r) k_var (G_s - G_l) frac (1 - frac) E / var / S (d ll / d G_e / S) and reduces ll, sum E^2, sum m E / var,
// sum (d ll / d g) G_r and sum_e R_e F_e (= d ELBO / d a_e).
__global__ void __launch_bounds__(MIX_THREADS) moe64_loglik_kernel(MoePtrs p, const double* Y, int n, int S) {
  __shared__ double red[7 * 32];
  const double kv = p.mix[0], skr = sqrt(p.mix[1]), var = p.mix[2], lv = log(var), invS = 1.0 / (double)S;
  const double as = p.sc[0][0], al = p.sc[1][0], ar = p.sc[2][0];
  double v[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (long long e = threadIdx.x; e < (long long)S * n; e += MIX_THREADS) {
    const double fs = p.F[0][e], fl = p.F[1][e], fr = p.F[2][e];
    const double Gs = as * fs, Gl = al * fl, Gr = ar * fr;
    const double frac = 1.0 / (1.0 + exp(-skr * Gr));
    const double m = frac * Gs + (1.0 - frac) * Gl;
    const double E = Y[e % n] - kv * m, dldf = E / var;
    const double dg = dldf * kv * (Gs - Gl) * frac * (1.0 - frac);
    const double Rs = kv * frac * dldf * invS, Rl = kv * (1.0 - frac) * dldf * invS, Rr = skr * dg * invS;
    p.R[0][e] = Rs; p.R[1][e] = Rl; p.R[2][e] = Rr;
    v[0] += -0.9189385332046727 - 0.5 * lv - 0.5 * E * E / var;
    v[1] += E * E;
    v[2] += m * dldf;
    v[3] += dg * Gr;
    v[4] += Rs * fs;
    v[5] += Rl * fl;
    v[6] += Rr * fr;
  }
  block_sum<7>(v, red);
  if (threadIdx.x == 0)
    for (int i = 0; i < 7; ++i) p.mix[3 + i] = v[i];
}

// lengthscale gradients (K-bar came without the factor a_e: the reverse-mode Cholesky is linear in L-bar), the scale
// gradients, the three shared scalars' gradients and out4
__global__ void moe64_scalar_kernel(MoePtrs p, int n, int S, double* out4) {
  const double invS = 1.0 / (double)S;
  for (int e = 0; e < NE; ++e) {
    const double a = p.sc[e][0];
    for (int d = threadIdx.x; d < p.n_ell[e]; d += blockDim.x) {
      double t = 0.0;
      for (int b = 0; b < kGramBwdBlocks; ++b) t += p.red[e][(long long)b * p.n_ell[e] + d];
      p.g_ell[e][d] = a * t / p.sc[e][SC_ELL + d] * t_sigmoid<double>(p.p_ell[e][d]);
    }
  }
  if (threadIdx.x == 0) {
    const double* mx = p.mix;
    const double kvr = mx[1], v = mx[2], ll = mx[3], sumE2 = mx[4];
    double kl = 0.0;
    for (int e = 0; e < NE; ++e) {
      *p.g_scale[e] = mx[7 + e] * t_sigmoid<double>(*p.p_scale[e]);
      kl += p.sc[e][7];
    }
    p.g_glob[0] = invS * mx[5] * t_sigmoid<double>(p.p_glob[0]);
    p.g_glob[1] = invS * mx[6] / (2.0 * sqrt(kvr)) * t_sigmoid<double>(p.p_glob[1]);
    p.g_glob[2] = invS * (-0.5 * (double)S * n / v + 0.5 * sumE2 / (v * v)) * t_sigmoid<double>(p.p_glob[2]);
    out4[0] = (ll - kl) * invS; out4[1] = ll; out4[2] = kl; out4[3] = 0.0;
  }
}

// The two side streams and the events that fork them from, and join them back to, the caller's stream: created once per
// device, a resource cache like linalg.cu's side stream.
struct MoeStreams {
  cudaStream_t side[NE - 1] = {nullptr, nullptr};
  cudaEvent_t fork = nullptr, done[NE - 1] = {nullptr, nullptr};
  bool tried = false, ok = false;
};
MoeStreams g_moe[64];

MoeStreams* moe_streams() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  MoeStreams& s = g_moe[dev];
  if (!s.tried) {
    s.tried = true;
    bool ok = cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < NE - 1; ++i)
      ok = ok && cudaStreamCreateWithFlags(&s.side[i], cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&s.done[i], cudaEventDisableTiming) == cudaSuccess;
    s.ok = ok;
  }
  return s.ok ? &s : nullptr;
}

int fork_sides(const MoeStreams& s, cudaStream_t st) {
  if (cudaEventRecord(s.fork, st) != cudaSuccess) return HB_ERR_CUDA;
  for (int i = 0; i < NE - 1; ++i)
    if (cudaStreamWaitEvent(s.side[i], s.fork, 0) != cudaSuccess) return HB_ERR_CUDA;
  return HB_OK;
}

int join_sides(const MoeStreams& s, cudaStream_t st) {
  int rc = HB_OK;
  for (int i = 0; i < NE - 1; ++i)                       // every side stream, even after one fails
    if (cudaEventRecord(s.done[i], s.side[i]) != cudaSuccess || cudaStreamWaitEvent(st, s.done[i], 0) != cudaSuccess)
      rc = HB_ERR_CUDA;
  return rc;
}

// fn(e) for every expert between a fork and a join.  The join happens even when a launch fails, so the caller's stream
// has waited on whatever the side streams had queued; the first error is returned.
template <class Fn>
int on_chains(const MoeStreams& s, cudaStream_t st, Fn fn) {
  HB_TRY(fork_sides(s, st));
  int rc = HB_OK;
  for (int e = 0; e < NE && rc == HB_OK; ++e) rc = fn(e);
  const int rj = join_sides(s, st);
  return rc != HB_OK ? rc : rj;
}

// one expert's chain up to its raw projection F_e = Z_e L_e^T: Gram, factorisation, sampler + KL, projection
int expert_forward(const Ctx64& cx, const hb_moe_gp_config& c, int e, const double* X, const double* p_mu, const double* p_sq,
                   const double* eps, double* sc, double* K, double* Z, double* F, double* U) {
  const int n = c.n, S = c.S, full = c.q_fullrank[e];
  const long long Sn = (long long)S * n;
  const int ew_blocks = (int)std::min<long long>((Sn + 255) / 256, 148 * 8);
  gp64_gram_kernel<<<dim3(cdiv(n, 32), cdiv(n, 32)), dim3(32, 8), 0, cx.st>>>(X, n, c.D, sc, c.n_ell[e], c.jitter, K);
  HB_CHECK_LAUNCH();
  HB_TRY(potrf_cols64(cx, K, n, 0, n, n));
  gp64_sample_kernel<<<ew_blocks, 256, 0, cx.st>>>(p_mu, p_sq, full, n, S, eps, c.seed, c.offset[e], U, Z);
  HB_CHECK_LAUNCH();
  if (full) HB_TRY(gemm64(cx, U, n, 0, 0, p_sq, n, 1, 2, Z, n, 0, S, n, n, 1.0, 1.0));          // Z += U tril(Lq)^T
  gp64_kl_kernel<<<1, RED_THREADS, 0, cx.st>>>(p_sq, full, n, S, U, Z, sc);
  HB_CHECK_LAUNCH();
  return gemm64(cx, Z, n, 0, 0, K, n, 1, 2, F, n, 0, S, n, n, 1.0, 0.0);
}

// the rest of the chain from the residual R_e: W = R L, z-bar, sampler backward, L-bar / a_e = tril(R^T Z), reverse-mode
// Cholesky, Gram backward partial sums
int expert_backward(const Ctx64& cx, const hb_moe_gp_config& c, int e, const double* X, const double* p_sq, const double* sc,
                    double* K, double* G, double* Z, double* F, double* R, double* W, double* U, double* red, double* g_mu,
                    double* g_sq) {
  const int n = c.n, S = c.S, full = c.q_fullrank[e];
  const long long Sn = (long long)S * n;
  const int ew_blocks = (int)std::min<long long>((Sn + 255) / 256, 148 * 8);
  HB_TRY(gemm64(cx, R, n, 0, 0, K, n, 0, 1, W, n, 0, S, n, n, 1.0, 0.0));
  gp64_zbar_kernel<<<ew_blocks, 256, 0, cx.st>>>(W, Z, sc, Sn, S, F);                          // F is free: z-bar
  HB_CHECK_LAUNCH();
  if (full) {
    if (cudaMemsetAsync(g_sq, 0, (size_t)n * n * sizeof(double), cx.st) != cudaSuccess) return HB_ERR_CUDA;
    HB_TRY(gemm64(cx, F, n, 1, 0, U, n, 0, 0, g_sq, n, 1, n, n, S, 1.0, 0.0));              // tril(z-bar^T U)
  }
  gp64_sampler_bwd_kernel<<<cdiv(n, 256), 256, 0, cx.st>>>(F, U, p_sq, full, n, S, g_mu, g_sq);
  HB_CHECK_LAUNCH();
  HB_TRY(gemm64(cx, R, n, 1, 0, Z, n, 0, 0, G, n, 1, n, n, S, 1.0, 0.0));
  HB_TRY(chol_rev_cols64(cx, K, n, G, n, 0, n, n));
  gp64_gram_bwd_kernel<<<kGramBwdBlocks, 256, 0, cx.st>>>(G, X, n, c.D, sc, c.n_ell[e], red);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

int moe_step_f64(const hb_moe_gp_config& c, const double* X, const double* Y, double* params, const double* const eps[NE],
                 double* grads, double* out4, double* adam_m, double* adam_v, const hb_adam_config* adam, void* ws,
                 int* err_flag, cudaStream_t st) {
  const MoeLayout L = moe_layout(c);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  auto at = [&](size_t off) { return reinterpret_cast<double*>(base + off); };
  const int n = c.n;
  HB_TRY(ensure_attrs64());
  const MoeStreams* ms = moe_streams();
  if (!ms) return HB_ERR_CUDA;

  MoePtrs p{};
  const double* p_mu[NE];
  const double* p_sq[NE];
  double* g_mu[NE];
  double* g_sq[NE];
  Ctx64 cx[NE];
  for (int e = 0; e < NE; ++e) {
    const size_t nq = c.q_fullrank[e] ? (size_t)n * n : (size_t)n;
    p_mu[e] = params + L.seg_params[e];
    p_sq[e] = p_mu[e] + n;
    p.p_scale[e] = p_sq[e] + nq;
    p.p_ell[e] = p.p_scale[e] + 1;
    g_mu[e] = grads + L.seg_params[e];
    g_sq[e] = g_mu[e] + n;
    p.g_scale[e] = g_sq[e] + nq;
    p.g_ell[e] = p.g_scale[e] + 1;
    p.n_ell[e] = c.n_ell[e];
    p.sc[e] = at(L.off_sc[e]);
    p.red[e] = at(L.off_red[e]);
    p.F[e] = at(L.off_F[e]);
    p.R[e] = at(L.off_R[e]);
    cx[e] = Ctx64{e == 0 ? st : ms->side[e - 1], err_flag, base + L.off_split[e], kSplitWsBytes};
  }
  p.p_glob = params + L.nparams - 3;
  p.g_glob = grads + L.nparams - 3;
  p.mix = at(L.off_mix);

  moe64_prep_kernel<<<1, 32, 0, st>>>(p);
  HB_CHECK_LAUNCH();
  HB_TRY(on_chains(*ms, st, [&](int e) {
    return expert_forward(cx[e], c, e, X, p_mu[e], p_sq[e], eps[e], p.sc[e], at(L.off_K[e]), at(L.off_Z[e]), at(L.off_F[e]),
                          at(L.off_U[e]));
  }));
  moe64_loglik_kernel<<<1, MIX_THREADS, 0, st>>>(p, Y, n, c.S);
  HB_CHECK_LAUNCH();
  HB_TRY(on_chains(*ms, st, [&](int e) {
    return expert_backward(cx[e], c, e, X, p_sq[e], p.sc[e], at(L.off_K[e]), at(L.off_G[e]), at(L.off_Z[e]), at(L.off_F[e]),
                           at(L.off_R[e]), at(L.off_W[e]), at(L.off_U[e]), at(L.off_red[e]), g_mu[e], g_sq[e]);
  }));
  moe64_scalar_kernel<<<1, 32, 0, st>>>(p, n, c.S, out4);
  HB_CHECK_LAUNCH();

  if (adam_m) {
    // each expert's segment has the GP entry's layout (q_sqrt at offset n), then the three trailing scalars
    auto run = [&](size_t off, long long npar, int full) {
      gp64_adam_kernel<<<(int)std::min<long long>((npar + 255) / 256, 148 * 8), 256, 0, st>>>(
          params + off, grads + off, adam_m + off, adam_v + off, npar, n, full, adam->step_dev, adam->step_host, adam->lr,
          adam->b1, adam->b2, adam->eps, adam->grad_scale);
    };
    for (int e = 0; e < NE; ++e) {
      run(L.seg_params[e], (long long)seg_count(c, e), c.q_fullrank[e]);
      HB_CHECK_LAUNCH();
    }
    run(L.nparams - 3, 3, 0);
    HB_CHECK_LAUNCH();
  }
  return HB_OK;
}

}  // namespace
}  // namespace hb

using namespace hb;

extern "C" {

size_t hb_moe_gp_param_count(const hb_moe_gp_config* cfg) {
  if (!cfg || !config_ok(*cfg)) return 0;
  return moe_layout(*cfg).nparams;
}

size_t hb_moe_gp_f64_workspace_bytes(const hb_moe_gp_config* cfg) {
  if (!cfg || !config_ok(*cfg)) return 0;
  return moe_layout(*cfg).total + 256;
}

int hb_moe_gp_elbo_step_f64(const hb_moe_gp_config* cfg, const double* X, const double* Y, double* params, const double* eps_s,
                            const double* eps_l, const double* eps_r, double* grads, double* out4, double* adam_m,
                            double* adam_v, const hb_adam_config* adam, void* ws, size_t ws_bytes, int* err_flag, void* stream) {
  if (!cfg || !X || !Y || !params || !grads || !out4) return HB_ERR_ARG;
  OptScope scope(cfg->opt);
  const hb_moe_gp_config c = *cfg;
  if (!config_ok(c)) return HB_ERR_ARG;
  const double* eps[NE] = {eps_s, eps_l, eps_r};
  for (int e = 0; e < NE; ++e)
    if (!eps[e] && (c.offset[e] & 3ull)) return HB_ERR_ARG;
  if ((adam_m || adam_v) && (!adam || !adam_m || !adam_v)) return HB_ERR_ARG;
  if (!ws || ws_bytes < moe_layout(c).total + 256) return HB_ERR_WORKSPACE;
  return moe_step_f64(c, X, Y, params, eps, grads, out4, adam_m, adam_v, adam, ws, err_flag, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
