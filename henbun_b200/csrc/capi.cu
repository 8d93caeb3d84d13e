// extern "C" boundary of libhenbun_b200.so -- see include/henbun_b200.h for the contract.
#include "../../include/henbun_b200.h"
#include "gemm.cuh"
#include "kernels.cuh"
#include "comm.cuh"
#include "gemm_h2.cuh"
#include <vector>
#include <cstdio>
#include <cstdlib>

namespace hb {

// ---- options of the call in flight (include/henbun_b200.h: hb_options) ------------------------------------------------
// The library keeps no mutable configuration.  Every extern "C" entry point that reaches the level-3 engine installs the
// caller's hb_options for its own duration on the calling thread (OptScope) and the kernels' host code reads them through
// the opt_*() accessors; outside any call, and for NULL, the defaults of hb_options_init apply.
static const hb_options kDefaultOptions = {0, 2048, 2, 1, 1, 0, 1, 0};
static thread_local const hb_options* tl_options = nullptr;
static inline const hb_options& cur_opt() { return tl_options ? *tl_options : kDefaultOptions; }
int opt_gemm_engine() { const int e = cur_opt().gemm_engine; return (e < 0 || e > 3) ? 0 : e; }
int opt_exact_below() { const int n = cur_opt().exact_below; return n < 0 ? 0 : n; }
int opt_panel_refinement() { const int m = cur_opt().panel_refinement; return (m < 0 || m > 3) ? 2 : m; }
int opt_presplit_engine() { return cur_opt().presplit_engine != 0; }
int opt_small_gp_kernel() { return cur_opt().small_gp_kernel != 0; }
int opt_tc_option() { return cur_opt().tc_option; }
int opt_lookahead() { return cur_opt().lookahead != 0; }
int opt_schedule() { return cur_opt().schedule; }
OptScope::OptScope(const ::hb_options* o) : prev(tl_options) { if (o) tl_options = o; }
OptScope::~OptScope() { tl_options = prev; }
#define g_engine (opt_gemm_engine())

int gemm_tc2(const GemmParams& p, cudaStream_t stream);  // gemm_tc2.cu (in-kernel hi/lo split, no workspace)
bool gemm_tc2_eligible(const GemmParams& p);
bool gemm_tc2_uses_pair(const GemmParams& p);
int get_tc_option();

// shapes worth a tensor-core launch
static bool tc_worth(const GemmParams& p) {
  if (p.N < 64 || p.K < 32) return false;
  if ((double)p.M * p.N * p.K >= 256.0 * 256.0 * 256.0) return true;
  return p.K >= 512 && p.M >= 64 && p.ws != nullptr;     // long-K reductions into a small tile: split-K on tensor cores
}
// short-K products: the whole-K SIMT kernel wins until there are enough 128-row tiles to fill the tensor-core grid
static bool prefer_small(const GemmParams& p) {
  if (!gemm_small_eligible(p)) return false;
  const long long tiles = (long long)((p.M + 127) / 128) * ((p.N + 255) / 256);
  return !(tiles >= 24 && gemm_tc2_eligible(p) && tc_worth(p));
}
static int tc_run(const GemmParams& p, cudaStream_t st, bool force) {
  if (gemm_tc2_eligible(p) && (force || tc_worth(p))) return gemm_tc2(p, st);
  return -1;
}

// engine: 0 auto | 1 fp32 SIMT only (short-K kernel + k-looped kernel) | 2 force tcgen05 | 3 k-looped SIMT kernel only
static int gemm_dispatch(const GemmParams& p, cudaStream_t st) {
  if (p.C == p.A && p.N > 128) return HB_ERR_ARG;      // in-place needs one column tile per row block
  if (g_engine == 3) return gemm_simt(p, st);
  if (p.force_simt) return gemm_small_eligible(p) ? gemm_small(p, st) : gemm_simt(p, st);
  if (g_engine == 2) { const int rc = tc_run(p, st, true); return rc < 0 ? HB_ERR_ARG : rc; }
  if (g_engine == 1 ? gemm_small_eligible(p) : prefer_small(p)) return gemm_small(p, st);
  if (g_engine == 0) { const int rc = tc_run(p, st, false); if (rc >= 0) return rc; }
  if (gemm_small_eligible(p)) return gemm_small(p, st);
  return gemm_simt(p, st);
}

// Optional per-launch GEMM timing (CUDA events on the launching stream) for bench.py's roofline.
struct GemmProfiler {
  bool on = false;
  size_t used = 0;
  std::vector<cudaEvent_t> ev0, ev1;
  std::vector<double> flops;
  std::vector<long long> shape;   // M, N, K, engine(1 = tensor core) per launch
} g_prof;

// Optional phase timing of the fused GP step (events on the launching stream; enabled by hb_phase_begin).
struct PhaseProfiler {
  bool on = false;
  int used = 0;
  cudaEvent_t ev[16];
  bool made = false;
} g_phase;
static void phase_mark(cudaStream_t st) {
  if (g_phase.on && g_phase.used < 16) cudaEventRecord(g_phase.ev[g_phase.used++], st);
}

static double gemm_useful_flops(const GemmParams& p) {
  double f = 2.0 * (double)p.M * (double)p.N * (double)p.K * (double)p.batch;
  if (p.c_tri) {   // lower trapezoid: M*N - N(N-1)/2 outputs when M >= N
    const double M = p.M, N = p.N;
    const double outs = (M >= N) ? M * N - 0.5 * N * (N - 1.0) : 0.5 * M * (M + 1.0);
    f *= outs / (M * N);
  }
  if (p.a_tri || p.b_tri) f *= 0.5;
  return f;
}

int gemm_prof_begin(double useful_flops, int M, int N, int K, int kind, cudaStream_t st) {
  if (!g_prof.on || g_prof.used >= g_prof.ev0.size()) return -1;
  const size_t i = g_prof.used++;
  g_prof.flops[i] = useful_flops;
  g_prof.shape[4 * i] = M; g_prof.shape[4 * i + 1] = N; g_prof.shape[4 * i + 2] = K; g_prof.shape[4 * i + 3] = kind;
  cudaEventRecord(g_prof.ev0[i], st);
  return (int)i;
}
void gemm_prof_end(int slot, cudaStream_t st) {
  if (slot >= 0) cudaEventRecord(g_prof.ev1[slot], st);
}

int gemm(const GemmParams& p, cudaStream_t st) {
  if (!g_prof.on || g_prof.used >= g_prof.ev0.size() || p.M <= 0 || p.N <= 0 || p.batch <= 0)
    return gemm_dispatch(p, st);
  const size_t i = g_prof.used++;
  g_prof.flops[i] = gemm_useful_flops(p);
  g_prof.shape[4 * i] = p.M; g_prof.shape[4 * i + 1] = p.N; g_prof.shape[4 * i + 2] = p.K;
  g_prof.shape[4 * i + 3] = p.force_simt ? 0 : (g_engine == 2 || (g_engine == 0 && !prefer_small(p) && (gemm_tc2_eligible(p) && tc_worth(p)))) ? 1 : 0;
  if (g_prof.shape[4 * i + 3] && gemm_tc2_eligible(p) && gemm_tc2_uses_pair(p)) g_prof.shape[4 * i + 3] = 2;
  cudaEventRecord(g_prof.ev0[i], st);
  const int rc = gemm_dispatch(p, st);
  cudaEventRecord(g_prof.ev1[i], st);
  return rc;
}

namespace {

inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// ---- scalar glue of the fused GP step (all on device, no host round trip) ----
// sc layout: [0]=scale s, [1]=k_var, [2]=var, [3]=a=sqrt(k_var)*s, [4..4+n_ell)=ell
__global__ void gp_prep_scalars_kernel(const float* __restrict__ p_scale, const float* __restrict__ p_ell, int n_ell,
                                       const float* __restrict__ p_kvar, const float* __restrict__ p_var, float* sc) {
  if (threadIdx.x == 0) {
    const float s = softplus_f(*p_scale) + 1e-6f;
    const float kv = softplus_f(*p_kvar) + 1e-6f;
    const float v = softplus_f(*p_var) + 1e-6f;
    sc[0] = s; sc[1] = kv; sc[2] = v; sc[3] = sqrtf(kv) * s;
  }
  for (int d = threadIdx.x; d < n_ell; d += blockDim.x) sc[4 + d] = softplus_f(p_ell[d]) + 1e-6f;
}

// ll3 = {loglik, sum E^2, sum E*F}; writes ELBO pieces and the scalar free-space gradients.
__global__ void gp_scalar_bwd_kernel(const float* __restrict__ sc, const float* __restrict__ ll3,
                                     const float* __restrict__ kl, long long total, int S, const float* p_scale,
                                     const float* p_ell, int n_ell, const float* p_kvar, const float* p_var,
                                     float* g_scale, float* g_ell, float* g_kvar, float* g_var, float* out4) {
  if (threadIdx.x == 0) {
    const double s = sc[0], kv = sc[1], v = sc[2], a = sc[3];
    const double invS = 1.0 / (double)S;
    const double sumE2 = ll3[1], sumEF = ll3[2];
    // d ELBO / d a  = sum R .* Fraw,  R = -(1/S) E / v,  Fraw = F / a
    const double ga = -invS * sumEF / (v * a);
    const double gs = ga * sqrt(kv);
    const double gkv = ga * s / (2.0 * sqrt(kv));
    const double gv = invS * (-0.5 * (double)total / v + 0.5 * sumE2 / (v * v));
    *g_scale = (float)(gs * (double)sigmoid_f(*p_scale));
    *g_kvar = (float)(gkv * (double)sigmoid_f(*p_kvar));
    *g_var = (float)(gv * (double)sigmoid_f(*p_var));
    out4[0] = (float)(((double)ll3[0] - (double)*kl) * invS);
    out4[1] = ll3[0];
    out4[2] = *kl;
    out4[3] = 0.f;
  }
  // lengthscale chain rule (g_ell currently holds d ELBO / d ell)
  for (int d = threadIdx.x; d < n_ell; d += blockDim.x) g_ell[d] *= sigmoid_f(p_ell[d]);
}

// zt = a*wb - c*z (full-rank path)
__global__ void gp_zbar_total_kernel(const float* __restrict__ wb, const float* __restrict__ z, const float* __restrict__ a,
                                     float c, long long n, float* zt) {
  const float aa = *a;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    zt[e] = aa * wb[e] - c * z[e];
}

struct GpLayout {
  size_t off_K, off_G, off_Z, off_F, off_R, off_W, off_U, off_sc, off_red, off_potrf, off_ZA, off_RA, total;
  size_t potrf_bytes;
};

GpLayout gp_layout(const hb_gp_config& c, const DistEnv* d = nullptr) {
  GpLayout L{};
  const size_t nn = (size_t)c.n * c.n * sizeof(float), sn = (size_t)c.S * c.n * sizeof(float);
  size_t o = 0;
  L.off_K = o; o += align_up(nn);
  L.off_G = o; o += align_up(nn);
  L.off_Z = o; o += align_up(sn);
  L.off_F = o; o += align_up(sn);
  L.off_R = o; o += align_up(sn);
  L.off_W = o; o += align_up(sn);
  L.off_U = o; o += align_up(c.q_fullrank ? sn : 0);
  L.off_sc = o; o += align_up((size_t)(16 + c.n_ell) * sizeof(float));
  L.off_red = o; o += align_up(kReduceWsBytes);
  L.potrf_bytes = potrf_workspace_bytes(c.n);
  if (d) {
    DistEnv wide = *d;
    wide.block = max(d->block, d->block_bwd);
    L.potrf_bytes = potrf_dist_workspace_bytes(c.n, wide);
  }
  L.off_potrf = o; o += align_up(L.potrf_bytes);
  const size_t gathered = (d && d->world > 1 && d->shard_samples) ? sn * d->world : 0;     // Z and R of every rank
  L.off_ZA = o; o += align_up(gathered);
  L.off_RA = o; o += align_up(gathered);
  L.total = o;
  return L;
}

}  // namespace
}  // namespace hb

using namespace hb;

extern "C" {

int hb_version(void) { return 100; }
unsigned long long hb_launch_count(void) { return g_launches; }
size_t hb_reduce_workspace_bytes(void) { return kReduceWsBytes; }
void hb_options_init(hb_options* opt) { if (opt) *opt = kDefaultOptions; }

int hb_profile_begin(int max_gemm_launches) {
  if (max_gemm_launches < 0) return HB_ERR_ARG;
  while ((int)g_prof.ev0.size() < max_gemm_launches) {
    cudaEvent_t a, b;
    if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return HB_ERR_CUDA;
    g_prof.ev0.push_back(a); g_prof.ev1.push_back(b);
  }
  g_prof.flops.assign(g_prof.ev0.size(), 0.0);
  g_prof.shape.assign(4 * g_prof.ev0.size(), 0);
  g_prof.used = 0;
  g_prof.on = true;
  return HB_OK;
}
// Synchronises the device. out4 = {gemm launches timed, total gemm ms, total useful gemm FLOP, 0}.
int hb_profile_end(double* out4_host) {
  g_prof.on = false;
  if (!out4_host) return HB_ERR_ARG;
  if (cudaDeviceSynchronize() != cudaSuccess) return HB_ERR_CUDA;
  double ms = 0.0, fl = 0.0;
  for (size_t i = 0; i < g_prof.used; ++i) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, g_prof.ev0[i], g_prof.ev1[i]) != cudaSuccess) return HB_ERR_CUDA;
    ms += t; fl += g_prof.flops[i];
  }
  out4_host[0] = (double)g_prof.used; out4_host[1] = ms; out4_host[2] = fl; out4_host[3] = 0.0;
  return HB_OK;
}
// Per-launch dump of the last profiled region (call after hb_profile_end[_ex], before the next hb_profile_begin).
int hb_profile_dump_csv(const char* path) {
  if (!path) return HB_ERR_ARG;
  FILE* f = fopen(path, "w");
  if (!f) return HB_ERR_ARG;
  fprintf(f, "M,N,K,tc,useful_flop,ms\n");
  for (size_t i = 0; i < g_prof.used; ++i) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, g_prof.ev0[i], g_prof.ev1[i]) != cudaSuccess) { fclose(f); return HB_ERR_CUDA; }
    fprintf(f, "%lld,%lld,%lld,%lld,%.0f,%.6f\n", g_prof.shape[4 * i], g_prof.shape[4 * i + 1], g_prof.shape[4 * i + 2],
            g_prof.shape[4 * i + 3], g_prof.flops[i], t);
  }
  fclose(f);
  return HB_OK;
}
// Same, but also splits out the launches that ran the CTA-pair tcgen05 kernel (the dominant kernel):
// out8 = {launches, ms, useful FLOP, pair launches, pair ms, pair useful FLOP, 0, 0}.  Call INSTEAD of hb_profile_end.
int hb_profile_end_ex(double* out8_host) {
  if (!out8_host) return HB_ERR_ARG;
  const size_t used = g_prof.used;
  const int rc = hb_profile_end(out8_host);
  if (rc != HB_OK) return rc;
  double pn = 0.0, pms = 0.0, pfl = 0.0, hms = 0.0, hfl = 0.0;
  for (size_t i = 0; i < used; ++i) {
    const long long kind = g_prof.shape[4 * i + 3];
    if (kind != 2 && kind != 3) continue;
    float t = 0.f;
    if (cudaEventElapsedTime(&t, g_prof.ev0[i], g_prof.ev1[i]) != cudaSuccess) return HB_ERR_CUDA;
    if (kind == 2) { pn += 1.0; pms += t; pfl += g_prof.flops[i]; }
    else { hms += t; hfl += g_prof.flops[i]; }
  }
  out8_host[3] = pn; out8_host[4] = pms; out8_host[5] = pfl; out8_host[6] = hms; out8_host[7] = hfl;
  return HB_OK;
}

// Phase timing of ONE hb_gp_elbo_step call: hb_phase_begin(); step; hb_phase_end(out) -> ms of
// {prep+Gram fwd, potrf, sampler+F+loglik+W, sampler bwd + Lbar, potrf_bwd, Gram bwd + scalars}; returns #phases.
int hb_phase_begin(void) {
  if (!g_phase.made) {
    for (int i = 0; i < 16; ++i) if (cudaEventCreate(&g_phase.ev[i]) != cudaSuccess) return HB_ERR_CUDA;
    g_phase.made = true;
  }
  g_phase.used = 0; g_phase.on = true;
  return HB_OK;
}
int hb_phase_end(double* out_ms, int capacity) {
  g_phase.on = false;
  if (!out_ms) return -1;
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  int n = 0;
  for (int i = 0; i + 1 < g_phase.used && n < capacity; ++i, ++n) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, g_phase.ev[i], g_phase.ev[i + 1]) != cudaSuccess) return -1;
    out_ms[n] = t;
  }
  return n;
}

int hb_randn_philox(float* out, long long count, unsigned long long seed, unsigned long long offset, void* stream) {
  return randn_philox(out, count, seed, offset, S(stream));
}

int hb_philox4x32_10(unsigned int* out, long long n_blocks, const unsigned int* ctr4_host, const unsigned int* key2_host,
                     void* stream) {
  return philox_raw(out, n_blocks, ctr4_host, key2_host, S(stream));
}

int hb_sample_diag_fwd(const float* mu, long long ld_mu, const float* omega, long long ld_omega, int rows, int cols,
                       const float* eps, unsigned long long seed, unsigned long long offset, int Sn, float* z,
                       float* kl_out, void* ws, size_t ws_bytes, void* stream) {
  return sample_diag_fwd(mu, ld_mu, omega, ld_omega, rows, cols, eps, seed, offset, Sn, z, kl_out, ws, ws_bytes, S(stream));
}

int hb_sample_diag_bwd(const float* mu, long long ld_mu, const float* omega, long long ld_omega, int rows, int cols,
                       const float* eps, unsigned long long seed, unsigned long long offset, int Sn,
                       const float* zbar, const float* zbar_scale, float kl_coef, const float* kl_coef_dev, float* gmu,
                       long long ld_gmu,
                       float* gomega, long long ld_gomega, float beta, void* stream) {
  return sample_diag_bwd(mu, ld_mu, omega, ld_omega, rows, cols, eps, seed, offset, Sn, zbar, zbar_scale, kl_coef, kl_coef_dev, gmu,
                         ld_gmu, gomega, ld_gomega, beta, S(stream));
}

int hb_sample_tril_fwd(const float* mu, const float* Lq, int n, int batch, const float* eps, int Sn, float* z,
                       float* kl_out, void* ws, size_t ws_bytes, void* stream) {
  if (n < 0 || batch < 0 || Sn < 0) return HB_ERR_ARG;
  if ((long long)n * batch * Sn == 0) return kl_out ? fill_f32(kl_out, 1, 0.f, S(stream)) : HB_OK;
  if (!mu || !Lq || !eps || !z) return HB_ERR_ARG;
  // z[b] (S x n) = eps[b] (S x n) * tril(Lq[b])^T : op(B)[k][j] = Lq[j][k], keep k <= j (upper in (k,n))
  GemmParams g;
  g.A = eps; g.lda = n; g.sA = (long long)Sn * n;
  g.B = Lq; g.ldb = n; g.sB = (long long)n * n; g.transB = 1; g.b_tri = 2;
  g.C = z; g.ldc = n; g.sC = (long long)Sn * n;
  g.M = Sn; g.N = n; g.K = n; g.batch = batch;
  g.bias = mu; g.sBias = n;
  HB_TRY(gemm(g, S(stream)));
  if (kl_out)
    HB_TRY(tril_logdet_kl(Lq, n, (long long)n * n, n, batch, eps, z, (long long)batch * Sn * n, Sn, kl_out, ws, ws_bytes, S(stream)));
  return HB_OK;
}

int hb_sample_tril_bwd(const float* Lq, int n, int batch, const float* eps, const float* z, int Sn,
                       const float* zbar, float kl_coef, float* gmu, float* gLq, float* scratch, void* stream) {
  if (n < 0 || batch < 0 || Sn < 0) return HB_ERR_ARG;
  const long long cnt = (long long)batch * Sn * n;
  if (cnt == 0) return HB_OK;
  if (!Lq || !eps || !z || !gmu || !gLq || !scratch) return HB_ERR_ARG;
  cudaStream_t st = S(stream);
  // zt = zbar - c*z
  if (zbar) {
    HB_TRY(copy2d(scratch, cnt, zbar, cnt, 1, (int)cnt, 1.f, st));
    HB_TRY(axpby(scratch, z, cnt, -kl_coef, 1.f, st));
  } else {
    HB_TRY(axpby(scratch, z, cnt, -kl_coef, 0.f, st));
  }
  for (int b = 0; b < batch; ++b)
    HB_TRY(colsum(scratch + (long long)b * Sn * n, n, Sn, n, 1.f, 0.f, gmu + (long long)b * n, st));
  HB_TRY(fill_f32(gLq, (long long)batch * n * n, 0.f, st));
  GemmParams g;   // gLq[b] = tril(zt[b]^T eps[b])
  g.A = scratch; g.lda = n; g.sA = (long long)Sn * n; g.transA = 1;
  g.B = eps; g.ldb = n; g.sB = (long long)Sn * n; g.transB = 0;
  g.C = gLq; g.ldc = n; g.sC = (long long)n * n; g.c_tri = 1;
  g.M = n; g.N = n; g.K = Sn; g.batch = batch;
  HB_TRY(gemm(g, st));
  return tril_diag_grad(gLq, n, (long long)n * n, Lq, n, (long long)n * n, n, batch, kl_coef * (float)Sn, st);
}

int hb_gaussian_logpdf(const float* x, long long x_period, const float* mu, long long mu_period, const float* var,
                       long long var_period, long long total, float* out, void* stream) {
  return gaussian_logpdf(x, x_period, mu, mu_period, var, var_period, total, out, S(stream));
}

int hb_gaussian_logpdf_bwd(const float* x, long long x_period, const float* mu, long long mu_period, const float* var,
                           long long var_period, long long total, const float* g, float* dmu, float* dvar,
                           void* stream) {
  return gaussian_logpdf_bwd(x, x_period, mu, mu_period, var, var_period, total, g, dmu, dvar, S(stream));
}
int hb_transform_fwd(int kind, const float* x, long long total, float p0, float p1, float* y, void* stream) {
  return transform_fwd(kind, x, total, p0, p1, y, S(stream));
}
int hb_transform_bwd(int kind, const float* x, long long total, float p0, float p1, const float* gy, float* gx, void* stream) {
  return transform_bwd(kind, x, total, p0, p1, gy, gx, S(stream));
}
int hb_transform_logjac(int kind, const float* x, long long total, float p0, float p1, float* out1, void* ws, size_t ws_bytes,
                        void* stream) {
  return transform_logjac(kind, x, total, p0, p1, out1, ws, ws_bytes, S(stream));
}
int hb_transform_logjac_bwd(int kind, const float* x, long long total, float p0, float p1, const float* g1, float* gx,
                            void* stream) {
  return transform_logjac_bwd(kind, x, total, p0, p1, g1, gx, S(stream));
}

int hb_density_nargs(int kind) { return density_nargs_host(kind); }

int hb_density_logpdf(int kind, const float* const* args, const long long* periods, long long total, float* out,
                      void* stream) {
  return density_logpdf(kind, args, periods, total, out, S(stream));
}

int hb_density_logpdf_bwd(int kind, const float* const* args, const long long* periods, long long total, const float* g,
                          long long g_period, float* const* dargs, void* ws, size_t ws_bytes, void* stream) {
  return density_logpdf_bwd(kind, args, periods, total, g, g_period, dargs, ws, ws_bytes, S(stream));
}

int hb_gather_rows(float* dst, const float* src, const long long* index, long long n_index, long long row_elems,
                   void* stream) {
  return gather_rows(dst, src, index, n_index, row_elems, S(stream));
}

int hb_gather_rows_f64(double* dst, const double* src, const long long* index, long long n_index, long long row_elems,
                       void* stream) {
  return gather_rows_f64(dst, src, index, n_index, row_elems, S(stream));
}

int hb_random_index(long long* out, long long n_index, const long long* pool, long long pool_size, unsigned long long seed,
                    unsigned long long offset, void* stream) {
  return random_index(out, n_index, pool, pool_size, seed, offset, S(stream));
}

int hb_gauss_loglik_fwd(const float* f, const float* f_scale, const float* y, long long total, long long y_period,
                        const float* var, float rcoef, float* resid, float* out3, void* ws, size_t ws_bytes,
                        void* stream) {
  return gauss_loglik_fwd(f, f_scale, y, total, y_period, var, rcoef, resid, out3, ws, ws_bytes, S(stream));
}

int hb_rbf_gram_fwd(const float* X, const float* X2, int n, int n2, int D, int batch, const float* ell, int n_ell,
                    float* K, long long ldk, long long strideK, float jitter, int lower_only, int csym, void* stream) {
  return rbf_gram_fwd(X, X2, n, n2, D, (long long)n * D, (long long)n2 * D, ell, n_ell, K, ldk, strideK, batch, jitter,
                      lower_only, csym, S(stream));
}

int hb_rbf_gram_bwd(const float* G, long long ldg, long long strideG, const float* X, const float* X2, int n, int n2,
                    int D, int batch, const float* ell, int n_ell, int sym_lower, int csym, const float* out_scale,
                    float* g_ell, void* ws, size_t ws_bytes, void* stream) {
  return rbf_gram_bwd(G, ldg, strideG, X, X2, n, n2, D, (long long)n * D, (long long)n2 * D, ell, n_ell, batch, sym_lower,
                      csym, out_scale, g_ell, ws, ws_bytes, S(stream));
}

int hb_rbf_gram_bwd_x2(const float* G, long long ldg, long long strideG, const float* X, const float* X2, int n, int n2,
                       int D, int batch, const float* ell, int n_ell, int sym_lower, float scale, float* dX2, void* stream) {
  return rbf_gram_bwd_x2(G, ldg, strideG, X, X2 ? X2 : X, n, n2, D, (long long)n * D, (long long)n2 * D, ell, n_ell, batch,
                         sym_lower, scale, dX2, S(stream));
}

size_t hb_potrf_workspace_bytes(int n) { return potrf_workspace_bytes(n); }
int hb_potrf_lower(float* A, long long lda, long long strideA, int n, int batch, int zero_upper, void* ws,
                   size_t ws_bytes, int* err_flag, void* stream, const hb_options* opt) {
  OptScope scope(opt);
  return potrf_lower(A, lda, strideA, n, batch, zero_upper, ws, ws_bytes, err_flag, S(stream));
}
int hb_potrf_lower_bwd(const float* L, long long ldl, long long strideL, float* G, long long ldg, long long strideG,
                       int n, int batch, void* ws, size_t ws_bytes, void* stream, const hb_options* opt) {
  OptScope scope(opt);
  return potrf_lower_bwd(L, ldl, strideL, G, ldg, strideG, n, batch, ws, ws_bytes, S(stream));
}
size_t hb_trsm_workspace_bytes(int m, int n) { return trsm_workspace_bytes(m, n); }
int hb_trsm_right_lower(const float* L, long long ldl, float* X, long long ldx, int m, int n, int trans, void* ws,
                        size_t ws_bytes, void* stream, const hb_options* opt) {
  OptScope scope(opt);
  return trsm_right_lower(L, ldl, X, ldx, m, n, trans, ws, ws_bytes, S(stream));
}

int hb_gemm(const float* A, long long lda, long long strideA, int transA, int a_tri, const float* B, long long ldb,
            long long strideB, int transB, int b_tri, float* C, long long ldc, long long strideC, int c_tri, int M,
            int N, int K, int batch, float alpha, float beta, const float* bias, long long strideBias, int act,
            int clip, float clip_lo, float clip_hi, void* stream) {
  return hb_gemm_ws(A, lda, strideA, transA, a_tri, B, ldb, strideB, transB, b_tri, C, ldc, strideC, c_tri, M, N, K,
                    batch, alpha, beta, bias, strideBias, act, clip, clip_lo, clip_hi, nullptr, 0, stream, nullptr);
}

int hb_gemm_ws(const float* A, long long lda, long long strideA, int transA, int a_tri, const float* B, long long ldb,
               long long strideB, int transB, int b_tri, float* C, long long ldc, long long strideC, int c_tri, int M,
               int N, int K, int batch, float alpha, float beta, const float* bias, long long strideBias, int act,
               int clip, float clip_lo, float clip_hi, void* ws, size_t ws_bytes, void* stream, const hb_options* opt) {
  OptScope scope(opt);
  GemmParams g;
  g.ws = ws; g.ws_bytes = ws_bytes;
  g.A = A; g.lda = lda; g.sA = strideA; g.transA = transA; g.a_tri = a_tri;
  g.B = B; g.ldb = ldb; g.sB = strideB; g.transB = transB; g.b_tri = b_tri;
  g.C = C; g.ldc = ldc; g.sC = strideC; g.c_tri = c_tri;
  g.M = M; g.N = N; g.K = K; g.batch = batch; g.alpha = alpha; g.beta = beta;
  g.bias = bias; g.sBias = strideBias; g.act = act; g.clip = clip; g.clip_lo = clip_lo; g.clip_hi = clip_hi;
  if (M > 0 && N > 0 && batch > 0) {
    const long long minA = transA ? M : K, minB = transB ? K : N;
    if ((K > 0 && (lda < minA || ldb < minB)) || ldc < N) return HB_ERR_ARG;
  }
  return gemm(g, S(stream));
}

size_t hb_gemm_tc_workspace_bytes(int, int, int) { return 0; }   // the engine consumes operands in place
int hb_gemm_tn_tc(const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc, int c_tri, int M,
                  int N, int K, float alpha, float beta, void* ws, size_t ws_bytes, void* stream) {
  GemmParams g;
  g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.transB = 1; g.C = C; g.ldc = ldc; g.c_tri = c_tri;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.beta = beta; g.ws = ws; g.ws_bytes = ws_bytes;
  const int rc = tc_run(g, S(stream), true);   // bypasses the size heuristic: always a tensor-core engine
  return rc < 0 ? HB_ERR_ARG : rc;
}

// ---- pre-split fp16 hi/lo engine (gemm_h2.cu), standalone: split both operands, then multiply --------------------
static size_t h2_probe_layout(int M, int N, int K, int transA, int transB, size_t off[6]) {
  const long long ra = transA ? K : M, ca = transA ? M : K, rb = transB ? N : K, cb = transB ? K : N;
  const long long lda = (ca + 63) / 64 * 64, ldb = (cb + 63) / 64 * 64;
  size_t o = 0;
  off[0] = o; o += align_up((size_t)ra * lda * 2);
  off[1] = o; o += align_up((size_t)ra * lda * 2);
  off[2] = o; o += align_up((size_t)rb * ldb * 2);
  off[3] = o; o += align_up((size_t)rb * ldb * 2);
  off[4] = o; o += align_up((size_t)(4 * ((ca + 127) / 128) + 32) * sizeof(float));   // max bits | inverse scales of A's column blocks (+ diagonal blocks)
  off[5] = o; o += align_up(16 * sizeof(float));                                       // B: max bits, {s, 1/s}
  return o + 256;
}
size_t hb_gemm_presplit_workspace_bytes(int M, int N, int K, int transA, int transB) {
  size_t off[6];
  return h2_probe_layout(M, N, K, transA, transB, off);
}
int hb_gemm_presplit(const float* A, long long lda, int transA, const float* B, long long ldb, int transB, float* C,
                     long long ldc, int c_tri, int M, int N, int K, float alpha, float beta, int a_bmode, int a_blockscale,
                     int skip_split, void* ws, size_t ws_bytes, void* stream, const hb_options* opt) {
  OptScope scope(opt);
  if (M <= 0 || N <= 0 || K <= 0) return HB_OK;
  if (!A || !B || !C) return HB_ERR_ARG;
  size_t off[6];
  if (!ws || ws_bytes < h2_probe_layout(M, N, K, transA, transB, off)) return HB_ERR_WORKSPACE;
  cudaStream_t st = S(stream);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  const long long ra = transA ? K : M, ca = transA ? M : K, rb = transB ? N : K, cb = transB ? K : N;
  const long long ldah = (ca + 63) / 64 * 64, ldbh = (cb + 63) / 64 * 64;
  __half* ah = reinterpret_cast<__half*>(base + off[0]); __half* al = reinterpret_cast<__half*>(base + off[1]);
  __half* bh = reinterpret_cast<__half*>(base + off[2]); __half* bl = reinterpret_cast<__half*>(base + off[3]);
  const int nblk = (int)((ca + 127) / 128);
  unsigned* amax = reinterpret_cast<unsigned*>(base + off[4]);
  float* ainv = reinterpret_cast<float*>(base + off[4]) + 2 * nblk + 8;
  unsigned* dmax = amax + nblk + 4;
  float* dinv = ainv + nblk + 4;
  unsigned* bmax = reinterpret_cast<unsigned*>(base + off[5]);
  float* bsc = reinterpret_cast<float*>(base + off[5]) + 4;
  if (!skip_split) {
    if (cudaMemsetAsync(base + off[4], 0, (size_t)(2 * nblk + 8) * 4, st) != cudaSuccess) return HB_ERR_CUDA;
    if (cudaMemsetAsync(base + off[5], 0, 16, st) != cudaSuccess) return HB_ERR_CUDA;
    if (a_blockscale) {       // one scale per 128-column block of the stored A
      if (ca % 128) return HB_ERR_ARG;
      for (int b = 0; b < nblk; ++b) {
        HB_TRY(h2_absmax(A + 128 * b, lda, ra, 128, 0, 0, amax + b, st));
        HB_TRY(h2_split(A + 128 * b, lda, ra, 128, nullptr, amax + b, ainv + b, 0, 0, ah + 128 * b, al + 128 * b, ldah, st));
        if (a_bmode == 1 && !transA) {   // the diagonal block of a K-major square A gets its own scale (as the reverse-mode leaves do)
          const float* D = A + (long long)128 * b * lda + 128 * b;
          HB_TRY(h2_absmax(D, lda, 128, 128, 0, 0, dmax + b, st));
          HB_TRY(h2_split(D, lda, 128, 128, nullptr, dmax + b, dinv + b, 0, 0, ah + (long long)128 * b * ldah + 128 * b,
                          al + (long long)128 * b * ldah + 128 * b, ldah, st));
        }
      }
    } else {
      if (ca % 8) return HB_ERR_ARG;
      HB_TRY(h2_absmax(A, lda, ra, (int)ca, 0, 0, amax, st));
      HB_TRY(h2_split(A, lda, ra, (int)ca, nullptr, amax, ainv, 0, 0, ah, al, ldah, st));
    }
    if (cb % 8) return HB_ERR_ARG;
    HB_TRY(h2_absmax(B, ldb, rb, (int)cb, 0, 0, bmax, st));
    HB_TRY(h2_scale_from_max(bmax, 0, bsc, st));
    HB_TRY(h2_split(B, ldb, rb, (int)cb, bsc, nullptr, nullptr, 0, 0, bh, bl, ldbh, st));
  }
  H2Gemm g;
  g.a_hi = ah; g.a_lo = al; g.lda = ldah; g.a_kmajor = transA ? 0 : 1;
  g.b_hi = bh; g.b_lo = bl; g.ldb = ldbh; g.b_kmajor = transB ? 1 : 0;
  g.C = C; g.ldc = ldc; g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.beta = beta; g.c_tri = c_tri; g.a_bmode = a_bmode;
  if (a_blockscale) { if (transA) g.a_minv = ainv; else { g.a_kinv = ainv; if (a_bmode == 1) g.a_dinv = dinv; } }
  else g.a_inv = ainv;
  g.b_inv = bsc + 1;
  return gemm_h2(g, st);
}

size_t hb_act_bwd_colsum_workspace_bytes(int rows, int cols) { return act_bwd_colsum_workspace_bytes(rows, cols); }
int hb_act_bwd_colsum_ws(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act, int clip,
                         float clip_lo, float clip_hi, float* dbias, void* ws, size_t ws_bytes, void* stream) {
  return act_bwd_colsum_ws(dy, y, dz, rows, cols, ld, act, clip, clip_lo, clip_hi, dbias, ws, ws_bytes, S(stream));
}
int hb_act_bwd_colsum(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act, int clip,
                      float clip_lo, float clip_hi, float* dbias, void* stream) {
  return act_bwd_colsum(dy, y, dz, rows, cols, ld, act, clip, clip_lo, clip_hi, dbias, S(stream));
}
int hb_colsum(const float* a, long long lda, int rows, int cols, float alpha, float beta, float* out, void* stream) {
  return colsum(a, lda, rows, cols, alpha, beta, out, S(stream));
}

int hb_adam_tf1(float* theta, const float* grad, float* m, float* v, long long n, float grad_scale, float lr, float b1,
                float b2, float eps, const int* step_dev, int step_host, void* stream) {
  return adam_tf1(theta, grad, m, v, n, grad_scale, lr, b1, b2, eps, step_dev, step_host, S(stream));
}
int hb_increment_i32(int* counter, void* stream) { return increment_i32(counter, S(stream)); }

int hb_transpose2d(float* dst, long long ldd, const float* src, long long lds, int rows, int cols, float scale, void* stream) {
  return transpose2d(dst, ldd, src, lds, rows, cols, scale, S(stream));
}
int hb_zero_strict_upper(float* a, long long lda, int n, void* stream) { return zero_strict_upper(a, lda, n, S(stream)); }

// ---------------------------------------------------------------------------------------------
// fused variational-GP ELBO + gradient
// ---------------------------------------------------------------------------------------------
int hb_gp_small_max_n(int f64) { return gp_small_max_n(f64); }
size_t hb_gp_small_workspace_bytes(const hb_gp_config* c, int f64) {
  if (!c) return 0;
  return gp_small_workspace_elems(c->n, c->S) * (f64 ? 8 : 4) + 256;
}
int hb_gp_small_step(const hb_gp_config* cfg, const float* X, const float* Y, float* params, const float* eps, float* grads,
                     float* out4, float* adam_m, float* adam_v, const hb_adam_config* adam, void* ws, size_t ws_bytes,
                     int* err_flag, void* stream) {
  if (!cfg) return HB_ERR_ARG;
  if (!ws || ws_bytes < hb_gp_small_workspace_bytes(cfg, 0)) return HB_ERR_WORKSPACE;
  if ((adam_m || adam_v) && (!adam || !adam_m || !adam_v)) return HB_ERR_ARG;
  float* w = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  return gp_small_step_f32(cfg->n, cfg->D, cfg->S, cfg->n_ell, cfg->q_fullrank, cfg->jitter, cfg->seed, cfg->offset, X, Y, params, eps,
                           grads, out4, w, err_flag, adam_m, adam_v, adam ? adam->step_dev : nullptr, adam ? adam->step_host : 0,
                           adam ? adam->lr : 0.0, adam ? adam->b1 : 0.0, adam ? adam->b2 : 0.0, adam ? adam->eps : 0.0,
                           adam ? adam->grad_scale : 0.0, S(stream));
}
int hb_gp_small_step_f64(const hb_gp_config* cfg, const double* X, const double* Y, double* params, const double* eps, double* grads,
                         double* out4, double* adam_m, double* adam_v, const hb_adam_config* adam, void* ws, size_t ws_bytes,
                         int* err_flag, void* stream) {
  if (!cfg) return HB_ERR_ARG;
  if (!ws || ws_bytes < hb_gp_small_workspace_bytes(cfg, 1)) return HB_ERR_WORKSPACE;
  if ((adam_m || adam_v) && (!adam || !adam_m || !adam_v)) return HB_ERR_ARG;
  double* w = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  return gp_small_step_f64(cfg->n, cfg->D, cfg->S, cfg->n_ell, cfg->q_fullrank, (double)cfg->jitter, cfg->seed, cfg->offset, X, Y, params,
                           eps, grads, out4, w, err_flag, adam_m, adam_v, adam ? adam->step_dev : nullptr, adam ? adam->step_host : 0,
                           adam ? adam->lr : 0.0, adam ? adam->b1 : 0.0, adam ? adam->b2 : 0.0, adam ? adam->eps : 0.0,
                           adam ? adam->grad_scale : 0.0, S(stream));
}

size_t hb_gp_param_count(const hb_gp_config* c) {
  if (!c) return 0;
  return (size_t)c->n + (c->q_fullrank ? (size_t)c->n * c->n : (size_t)c->n) + 1 + c->n_ell + 2;
}
size_t hb_gp_elbo_workspace_bytes(const hb_gp_config* c) {
  if (!c) return 0;
  return gp_layout(*c).total + 256;
}

static DistEnv to_env(const hb_dist* d) {
  DistEnv e;
  e.comm = d->comm; e.rank = d->rank; e.world = d->world; e.block = d->block > 0 ? d->block : 2048;
  e.batch = d->batch > 0 ? d->batch : 1;
  e.shard_samples = d->shard_samples ? 1 : 0;
  e.turn = d->turn > 0 ? d->turn : 1;
  e.block_bwd = d->block_bwd > 0 ? d->block_bwd : 0;
  return e;
}

int hb_comm_unique_id(void* out128_host) { return comm_unique_id(out128_host); }
int hb_comm_create(const void* id128_host, int rank, int world, void** comm_out) { return comm_create(id128_host, rank, world, comm_out); }
int hb_comm_destroy(void* comm) { return comm_destroy(comm); }

int hb_flat_trace_begin(void) { return flat_trace_begin(); }
int hb_flat_trace_end(double* out3_host, int capacity) { return flat_trace_end(out3_host, capacity); }
size_t hb_potrf_dist_workspace_bytes(int n, const hb_dist* d) { return d ? potrf_dist_workspace_bytes(n, to_env(d)) : 0; }
int hb_potrf_lower_dist(float* A, long long lda, int n, const hb_dist* d, void* ws, size_t ws_bytes, int* err_flag, void* stream,
                        const hb_options* opt) {
  if (!d) return HB_ERR_ARG;
  OptScope scope(opt);
  return potrf_lower_dist(A, lda, n, to_env(d), ws, ws_bytes, err_flag, S(stream));
}
int hb_potrf_lower_bwd_dist(const float* L, long long ldl, float* G, long long ldg, int n, const hb_dist* d, void* ws,
                            size_t ws_bytes, void* stream, const hb_options* opt) {
  if (!d) return HB_ERR_ARG;
  OptScope scope(opt);
  return potrf_lower_bwd_dist(L, ldl, G, ldg, n, to_env(d), ws, ws_bytes, S(stream), 0);
}

static int gp_elbo_step_impl(const hb_gp_config* cfg, const DistEnv* dist, const float* X, const float* Y, const float* params,
                             const float* eps, float* grads, float* out4, void* ws, size_t ws_bytes, int* err_flag, void* stream);

size_t hb_gp_elbo_dist_workspace_bytes(const hb_gp_config* c, const hb_dist* d) {
  if (!c || !d) return 0;
  const DistEnv e = to_env(d);
  return gp_layout(*c, &e).total + 256;
}
int hb_gp_elbo_step_dist(const hb_gp_config* cfg, const hb_dist* d, const float* X, const float* Y, const float* params,
                         const float* eps, float* grads, float* out4, void* ws, size_t ws_bytes, int* err_flag, void* stream) {
  if (!d) return HB_ERR_ARG;
  const DistEnv e = to_env(d);
  return gp_elbo_step_impl(cfg, &e, X, Y, params, eps, grads, out4, ws, ws_bytes, err_flag, stream);
}
int hb_gp_elbo_step(const hb_gp_config* cfg, const float* X, const float* Y, const float* params, const float* eps,
                    float* grads, float* out4, void* ws, size_t ws_bytes, int* err_flag, void* stream) {
  return gp_elbo_step_impl(cfg, nullptr, X, Y, params, eps, grads, out4, ws, ws_bytes, err_flag, stream);
}

static int gp_elbo_step_impl(const hb_gp_config* cfg, const DistEnv* dist, const float* X, const float* Y, const float* params,
                             const float* eps, float* grads, float* out4, void* ws, size_t ws_bytes, int* err_flag, void* stream) {
  if (!cfg || !X || !Y || !params || !grads || !out4) return HB_ERR_ARG;
  OptScope scope(cfg->opt);
  const hb_gp_config c = *cfg;
  if (c.n <= 0 || c.D <= 0 || c.D > 32 || c.S <= 0 || (c.n_ell != 1 && c.n_ell != c.D)) return HB_ERR_ARG;
  if (!eps && (c.offset & 3ull)) return HB_ERR_ARG;
  if (dist && c.n <= 128) dist = nullptr;        // one leaf: nothing to schedule
  const GpLayout L = gp_layout(c, dist);
  if (!ws || ws_bytes < L.total + 256) return HB_ERR_WORKSPACE;
  cudaStream_t st = S(stream);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  float* K = reinterpret_cast<float*>(base + L.off_K);
  float* G = reinterpret_cast<float*>(base + L.off_G);
  float* Z = reinterpret_cast<float*>(base + L.off_Z);
  float* F = reinterpret_cast<float*>(base + L.off_F);
  float* R = reinterpret_cast<float*>(base + L.off_R);
  float* W = reinterpret_cast<float*>(base + L.off_W);
  float* U = reinterpret_cast<float*>(base + L.off_U);
  float* sc = reinterpret_cast<float*>(base + L.off_sc);
  void* red = base + L.off_red;
  void* pws = base + L.off_potrf;
  float* ll3 = sc + 8 + c.n_ell;       // 3 floats
  float* kl = ll3 + 3;                 // 1 float

  const int n = c.n, Sn = c.S;
  if (n <= gp_small_max_n(0) && opt_small_gp_kernel()) {
    // notebook-sized model: the whole step is ONE persistent CTA (gp_small.cu); Z | F | R | W are adjacent -> 4 S n floats
    return gp_small_step_f32(n, c.D, Sn, c.n_ell, c.q_fullrank, c.jitter, c.seed, c.offset, X, Y, const_cast<float*>(params), eps,
                             grads, out4, Z, err_flag, nullptr, nullptr, nullptr, 0, 0.0, 0.0, 0.0, 0.0, 0.0, st);
  }
  const size_t nq = c.q_fullrank ? (size_t)n * n : (size_t)n;
  const float* p_mu = params;
  const float* p_sq = params + n;
  const float* p_scale = p_sq + nq;
  const float* p_ell = p_scale + 1;
  const float* p_kvar = p_ell + c.n_ell;
  const float* p_var = p_kvar + 1;
  float* g_mu = grads;
  float* g_sq = grads + n;
  float* g_scale = g_sq + nq;
  float* g_ell = g_scale + 1;
  float* g_kvar = g_ell + c.n_ell;
  float* g_var = g_kvar + 1;
  const float invS = 1.f / (float)Sn;

  phase_mark(st);
  gp_prep_scalars_kernel<<<1, 32, 0, st>>>(p_scale, p_ell, c.n_ell, p_kvar, p_var, sc);
  HB_CHECK_LAUNCH();
  const float* d_var = sc + 2;
  const float* d_a = sc + 3;
  const float* d_ell = sc + 4;

  // K = rbf(X) + jitter I (lower tiles), L = chol(K) in place
  HB_TRY(rbf_gram_fwd(X, nullptr, n, n, c.D, 0, 0, d_ell, c.n_ell, K, n, 0, 1, c.jitter, 1, 0, st));
  phase_mark(st);
  if (dist) HB_TRY(potrf_lower_dist(K, n, n, *dist, pws, L.potrf_bytes, err_flag, st));
  else HB_TRY(potrf_lower(K, n, 0, n, 1, 0, pws, L.potrf_bytes, err_flag, st));
  phase_mark(st);

  // sampler + KL
  const float* eps_used = eps;
  if (!c.q_fullrank) {
    HB_TRY(sample_diag_fwd(p_mu, n, p_sq, n, 1, n, eps, c.seed, c.offset, Sn, Z, kl, red, kReduceWsBytes, st));
  } else {
    if (!eps) {
      HB_TRY(randn_philox(U, (long long)Sn * n, c.seed, c.offset, st));
      eps_used = U;
    }
    HB_TRY(hb_sample_tril_fwd(p_mu, p_sq, n, 1, eps_used, Sn, Z, kl, red, kReduceWsBytes, stream));
  }

  // Fraw [S,n] = Z L^T : op(B)[k][j] = L[j][k], keep k <= j
  {
    GemmParams g;
    g.A = Z; g.lda = n; g.B = K; g.ldb = n; g.transB = 1; g.b_tri = 2;
    g.C = F; g.ldc = n; g.M = Sn; g.N = n; g.K = n;
    HB_TRY(gemm(g, st));
  }
  HB_TRY(gauss_loglik_fwd(F, d_a, Y, (long long)Sn * n, n, d_var, invS, R, ll3, red, kReduceWsBytes, st));
  // Wb_raw [S,n] = R L : op(B)[k][j] = L[k][j], keep k >= j (lower)
  {
    GemmParams g;
    g.A = R; g.lda = n; g.B = K; g.ldb = n; g.transB = 0; g.b_tri = 1;
    g.C = W; g.ldc = n; g.M = Sn; g.N = n; g.K = n;
    HB_TRY(gemm(g, st));
  }
  phase_mark(st);
  if (!c.q_fullrank) {
    HB_TRY(sample_diag_bwd(p_mu, n, p_sq, n, 1, n, eps, c.seed, c.offset, Sn, W, d_a, invS, nullptr, g_mu, n, g_sq, n, 0.f, st));
  } else {
    // zt = a*W - Z/S (into F, which is free now); gmu = colsum(zt); gLq = tril(zt^T eps) + diag(1/Lq_ii)
    gp_zbar_total_kernel<<<148 * 4, 256, 0, st>>>(W, Z, d_a, invS, (long long)Sn * n, F);
    HB_CHECK_LAUNCH();
    HB_TRY(colsum(F, n, Sn, n, 1.f, 0.f, g_mu, st));
    HB_TRY(fill_f32(g_sq, (long long)n * n, 0.f, st));
    GemmParams g;
    g.A = F; g.lda = n; g.transA = 1; g.B = eps_used; g.ldb = n; g.transB = 0;
    g.C = g_sq; g.ldc = n; g.c_tri = 1; g.M = n; g.N = n; g.K = Sn;
    HB_TRY(gemm(g, st));
    HB_TRY(tril_diag_grad(g_sq, n, 0, p_sq, n, 0, n, 1, 1.f, st));
  }
  // Lbar_raw = tril(R^T Z)  (the factor a = sqrt(k_var)*scale is applied at the very end: the
  // reverse-mode Cholesky is linear in Lbar)
  {
    GemmParams g;
    g.A = R; g.lda = n; g.transA = 1; g.B = Z; g.ldb = n; g.transB = 0;
    g.C = G; g.ldc = n; g.c_tri = 1; g.M = n; g.N = n; g.K = Sn;
    if (dist && dist->world > 1 && dist->shard_samples) {
      // Sample-sharded ranks share ONE factorisation: its gradient is linear in L-bar, so the ranks' residuals and samples
      // are gathered (2 x world x S x n floats) and every rank forms the L-bar of the rank-averaged objective itself.
      float* ZA = reinterpret_cast<float*>(base + L.off_ZA);
      float* RA = reinterpret_cast<float*>(base + L.off_RA);
      HB_TRY(comm_allgather_f32(dist->comm, Z, ZA, (size_t)Sn * n, st));
      HB_TRY(comm_allgather_f32(dist->comm, R, RA, (size_t)Sn * n, st));
      g.A = RA; g.B = ZA; g.K = Sn * dist->world; g.alpha = 1.f / (float)dist->world;
      // ... and only for the column blocks it owns: the others arrive as finished K-bar panels before anything reads them
      const int W = dist->block_bwd > 0 ? dist->block_bwd : dist->block, nblocks = (n + W - 1) / W;   // the reverse mode's blocks
      for (int b = 0; b < nblocks; ++b) {
        if ((b / dist->turn) % dist->world != dist->rank) continue;
        const int c0 = b * W, w = min(W, n - c0);
        GemmParams q = g;
        q.A = RA + c0; q.B = ZA + c0; q.C = G + (long long)c0 * n + c0; q.M = n - c0; q.N = w;
        HB_TRY(gemm(q, st));
      }
    } else {
      HB_TRY(gemm(g, st));
    }
  }
  phase_mark(st);
  if (dist) {
    DistEnv rev = *dist;
    if (dist->block_bwd > 0) rev.block = dist->block_bwd;
    HB_TRY(potrf_lower_bwd_dist(K, n, G, n, n, rev, pws, L.potrf_bytes, st, /*l_shadow_valid=*/1));
  }
  else HB_TRY(potrf_lower_bwd(K, n, 0, G, n, 0, n, 1, pws, L.potrf_bytes, st, /*l_shadow_valid=*/1));
  phase_mark(st);
  HB_TRY(rbf_gram_bwd(G, n, 0, X, nullptr, n, n, c.D, 0, 0, d_ell, c.n_ell, 1, 1, 0, d_a, g_ell, red, kReduceWsBytes, st));
  gp_scalar_bwd_kernel<<<1, 32, 0, st>>>(sc, ll3, kl, (long long)Sn * n, Sn, p_scale, p_ell, c.n_ell, p_kvar, p_var,
                                         g_scale, g_ell, g_kvar, g_var, out4);
  HB_CHECK_LAUNCH();
  phase_mark(st);
  return HB_OK;
}

}  // extern "C"
