// float64 linear-operator model (BASELINE config 5): the ELBO + gradient (+ TF-1 Adam) of csrc/linop.cu in double, the
// reference's float_type = float64 (henbunrc:7).
//     z = mu + tril(L_q) u,  KL = -1/2 sum(log diag(L_q)^2 + u^2 - z^2),  ELBO = [sum gaussian(y, A z, var) - KL] / S
// The problem is an inverse one: when the fit is good the residual E = y - A z is a small difference of large numbers, and
// Zbar = R A sums M of them, so in fp32 every gradient inherits the relative error |y| / |E| 2^-24 of E.
//
// Same two-call split as the fp32 pair, so a row-sharded operator needs exactly one collective in between:
//   hb_linop_elbo_local_f64  : sampler + KL (f64.cu's kernels), F = Z A^T, log-likelihood + residual, partial Zbar = R A
//   (all-reduce zbar_stats [S*n + 4] over the ranks)
//   hb_linop_elbo_update_f64 : Zt = Zbar - Z/S, mu-bar, var-bar, fused L_q gradient + Adam over the lower triangle
// Both operator products run on the fp64 GEMM of f64.cu (DMMA).  Every reduction has a fixed order and nothing is summed
// with atomics, so results are bitwise repeatable.  The workspace carries U, Z and the scalars between the two calls.
#include "../../include/henbun_b200.h"
#include "f64.cuh"
#include "tmath.cuh"
#include <algorithm>

namespace hb {
namespace {

constexpr int LL_BLOCKS = 296;                           // partial sums of sum E^2, finished in block order
constexpr int LL_THREADS = 256;
// sc: [0] var, [1] d var / d free, [7] kl (gp64_kl_kernel's slot)
constexpr int SC_N = 16;

struct Linop64Layout {
  size_t off_U, off_Z, off_Zt, off_F, off_sc, off_part, off_gt, off_split, total;
};

Linop64Layout linop64_layout(const hb_linop_config& c) {
  Linop64Layout L{};
  const size_t sn = (size_t)c.S * c.n * sizeof(double);
  size_t o = 0;
  L.off_U = o; o += align256(sn);
  L.off_Z = o; o += align256(sn);
  L.off_Zt = o; o += align256(sn);
  L.off_F = o; o += align256((size_t)c.S * c.M * sizeof(double));
  L.off_sc = o; o += align256(SC_N * sizeof(double));
  L.off_part = o; o += align256(LL_BLOCKS * sizeof(double));
  L.off_gt = o; o += align256(((size_t)c.n + 1) * sizeof(double));
  L.off_split = o; o += align256(kSplitWsBytes);
  L.total = o;
  return L;
}

bool cfg64_ok(const hb_linop_config& c) {
  return c.n > 0 && c.S > 0 && c.M > 0 && (long long)c.M <= c.M_total && c.presplit == 0;
}

__global__ void linop64_prep_kernel(const double* __restrict__ p_var, double* sc) {
  if (threadIdx.x == 0) {
    const double x = *p_var;
    sc[0] = t_softplus<double>(x) + 1e-6;
    sc[1] = t_sigmoid<double>(x);
  }
}

// R = E / var / S with E = y - F, in place over F [S, M]; block b writes its partial sum E^2 to part[b].  The element
// assignment depends on the fixed grid only, so the sums are the same on every call.
__global__ void __launch_bounds__(LL_THREADS) linop64_resid_kernel(double* __restrict__ F, const double* __restrict__ y, int M,
                                                                   long long total, const double* __restrict__ sc, double invS,
                                                                   double* __restrict__ part) {
  __shared__ double red[32];
  const double scale = invS / sc[0];
  double v[1] = {0.0};
  for (long long e = blockIdx.x * (long long)LL_THREADS + threadIdx.x; e < total; e += (long long)LL_BLOCKS * LL_THREADS) {
    const double E = y[e % M] - F[e];
    v[0] += E * E;
    F[e] = E * scale;
  }
  block_sum<1>(v, red);
  if (threadIdx.x == 0) part[blockIdx.x] = v[0];
}

// stats4 = {loglik, sum E^2, 0, 0} appended to the partial Zbar (one all-reduce carries both).  The log-likelihood of
// S * M terms is -S M (log(2 pi) + log var) / 2 - sum E^2 / (2 var): linear in the row count, so the ranks' values add up.
__global__ void linop64_stats_kernel(const double* __restrict__ part, const double* __restrict__ sc, double elems, double* stats4) {
  if (threadIdx.x == 0) {
    double e2 = 0.0;
    for (int b = 0; b < LL_BLOCKS; ++b) e2 += part[b];
    const double var = sc[0];
    stats4[0] = -elems * (0.9189385332046727 + 0.5 * log(var)) - 0.5 * e2 / var;
    stats4[1] = e2;
    stats4[2] = 0.0;
    stats4[3] = 0.0;
  }
}

// Zt = Zbar - Z / S (d ELBO_mean / d z: likelihood part minus the KL's z / S)
__global__ void linop64_zt_kernel(const double* __restrict__ zbar, const double* __restrict__ z, double invS, long long cnt,
                                  double* __restrict__ zt) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < cnt; e += (long long)gridDim.x * blockDim.x)
    zt[e] = zbar[e] - invS * z[e];
}

// mu-bar = column sums of Zt over the samples, in sample order
__global__ void linop64_colsum_kernel(const double* __restrict__ zt, int n, int S, double* __restrict__ g_mu) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int r = 0; r < S; ++r) s += zt[(long long)r * n + k];
    g_mu[k] = s;
  }
}

// d ELBO_mean / d var_free from the all-reduced {loglik, sum E^2}; out4 = {ELBO, loglik, kl, 0}
__global__ void linop64_scalars_kernel(const double* __restrict__ stats4, const double* __restrict__ sc, double total_elems,
                                       double invS, double* g_var, double* out4) {
  if (threadIdx.x == 0) {
    const double v = sc[0], kl = sc[7];
    *g_var = (-0.5 * total_elems / v + 0.5 * stats4[1] / (v * v)) * invS * sc[1];
    out4[0] = (stats4[0] - kl) * invS;
    out4[1] = stats4[0];
    out4[2] = kl;
    out4[3] = 0.0;
  }
}

// Fused gradient of L_q + TF-1 Adam over the lower triangle, the fp64 twin of linop.cu's tril_rank_adam_kernel.  One CTA
// per 64 x 64 lower-triangle tile of (i, j), 4 x 4 entries per thread:
//   g_ij = sum_s Zt[s,i] U[s,j] + (i == j) / L_ii              (d ELBO_mean / d L_ij, j <= i)
//   gl = grad_scale g;  m = b1 m + (1-b1) gl;  v = b2 v + (1-b2) gl^2;  L -= lr_t m / (sqrt(v) + eps)
// The n x n gradient is never materialised and nothing above the diagonal is read or written.  m == NULL: no update;
// gout != NULL: g is stored as well (lower triangle only).
constexpr int TA_TILE = 64, TA_SCHUNK = 32;

__global__ void __launch_bounds__(256) tril_rank_adam_f64_kernel(double* __restrict__ Lq, double* __restrict__ m,
                                                                 double* __restrict__ v, double* __restrict__ gout,
                                                                 const double* __restrict__ Zt, const double* __restrict__ U,
                                                                 int n, int S, double lr, double b1, double b2, double eps,
                                                                 double grad_scale, const int* step_dev, int step_host) {
  const long long kblk = blockIdx.x;
  int ti = (int)((sqrt(8.0 * (double)kblk + 1.0) - 1.0) * 0.5);
  while ((long long)ti * (ti + 1) / 2 > kblk) --ti;
  while ((long long)(ti + 1) * (ti + 2) / 2 <= kblk) ++ti;
  const int tj = (int)(kblk - (long long)ti * (ti + 1) / 2);
  __shared__ __align__(16) double Zs[TA_SCHUNK][TA_TILE];
  __shared__ __align__(16) double Us[TA_SCHUNK][TA_TILE];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int i0 = ti * TA_TILE, j0 = tj * TA_TILE;
  double acc[4][4];
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 4; ++y) acc[x][y] = 0.0;
  for (int s0 = 0; s0 < S; s0 += TA_SCHUNK) {
    for (int idx = tid; idx < TA_SCHUNK * TA_TILE; idx += 256) {
      const int sr = idx / TA_TILE, c = idx % TA_TILE;
      const bool sv = (s0 + sr) < S;
      Zs[sr][c] = (sv && (i0 + c) < n) ? __ldg(Zt + (long long)(s0 + sr) * n + i0 + c) : 0.0;
      Us[sr][c] = (sv && (j0 + c) < n) ? __ldg(U + (long long)(s0 + sr) * n + j0 + c) : 0.0;
    }
    __syncthreads();
    const int sl = min(TA_SCHUNK, S - s0);
    for (int sr = 0; sr < sl; ++sr) {
      const double2 a01 = *reinterpret_cast<const double2*>(&Zs[sr][ty * 4]);
      const double2 a23 = *reinterpret_cast<const double2*>(&Zs[sr][ty * 4 + 2]);
      const double2 b01 = *reinterpret_cast<const double2*>(&Us[sr][tx * 4]);
      const double2 b23 = *reinterpret_cast<const double2*>(&Us[sr][tx * 4 + 2]);
      const double a[4] = {a01.x, a01.y, a23.x, a23.y}, b[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = fma(a[x], b[y], acc[x][y]);
    }
    __syncthreads();
  }
  double lr_t = 0.0;
  if (m) {
    const int t = step_dev ? *step_dev : step_host;
    lr_t = lr * sqrt(1.0 - pow(b2, (double)t)) / (1.0 - pow(b1, (double)t));
  }
  const int jb = j0 + tx * 4;
#pragma unroll
  for (int x = 0; x < 4; ++x) {
    const int i = i0 + ty * 4 + x;
    if (i >= n) continue;
#pragma unroll
    for (int y = 0; y < 4; ++y) {
      const int j = jb + y;
      if (j > i || j >= n) continue;
      const long long off = (long long)i * n + j;
      double l = __ldcs(Lq + off);
      const double g = acc[x][y] + ((j == i) ? 1.0 / l : 0.0);
      if (gout) gout[off] = g;
      if (m) {
        const double gl = grad_scale * g;
        const double mm = b1 * __ldcs(m + off) + (1.0 - b1) * gl;
        const double vv = b2 * __ldcs(v + off) + (1.0 - b2) * gl * gl;
        l -= lr_t * mm / (sqrt(vv) + eps);
        __stcs(m + off, mm);
        __stcs(v + off, vv);
        __stcs(Lq + off, l);
      }
    }
  }
}

struct Linop64Ptrs {
  double *U, *Z, *Zt, *F, *sc, *part, *gt;
  Ctx64 cx;
};

Linop64Ptrs linop64_ptrs(const hb_linop_config& c, void* ws, cudaStream_t st) {
  const Linop64Layout L = linop64_layout(c);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  auto at = [&](size_t off) { return reinterpret_cast<double*>(base + off); };
  return Linop64Ptrs{at(L.off_U), at(L.off_Z), at(L.off_Zt), at(L.off_F), at(L.off_sc), at(L.off_part), at(L.off_gt),
                     Ctx64{st, nullptr, base + L.off_split, kSplitWsBytes}};
}

}  // namespace
}  // namespace hb

using namespace hb;

extern "C" {

size_t hb_linop_f64_workspace_bytes(const hb_linop_config* cfg) {
  if (!cfg || !cfg64_ok(*cfg)) return 0;
  return linop64_layout(*cfg).total + 256;
}

int hb_linop_elbo_local_f64(const hb_linop_config* cfg, const double* A, const double* y, const double* params,
                            const double* eps, double* zbar_stats, void* ws, size_t ws_bytes, void* stream) {
  if (!cfg || !A || !y || !params || !zbar_stats) return HB_ERR_ARG;
  const hb_linop_config c = *cfg;
  if (!cfg64_ok(c)) return HB_ERR_ARG;
  if (!eps && (c.offset & 3ull)) return HB_ERR_ARG;
  if (!ws || ws_bytes < linop64_layout(c).total + 256) return HB_ERR_WORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const Linop64Ptrs P = linop64_ptrs(c, ws, st);
  const int n = c.n, S = c.S, M = c.M;
  const double* p_sq = params;
  const double* p_mu = params + (size_t)n * n;
  const double* p_var = p_mu + n;
  const long long Sn = (long long)S * n;

  linop64_prep_kernel<<<1, 32, 0, st>>>(p_var, P.sc);
  HB_CHECK_LAUNCH();
  // U = eps (or the Philox stream widened to double) and Z = mu, then Z += U tril(L_q)^T; U stays for the update call
  gp64_sample_kernel<<<(int)std::min<long long>((Sn + 255) / 256, 148 * 8), 256, 0, st>>>(p_mu, p_sq, 1, n, S, eps, c.seed,
                                                                                          c.offset, P.U, P.Z);
  HB_CHECK_LAUNCH();
  HB_TRY(gemm64(P.cx, P.U, n, 0, 0, p_sq, n, 1, 2, P.Z, n, 0, S, n, n, 1.0, 1.0));
  gp64_kl_kernel<<<1, RED_THREADS, 0, st>>>(p_sq, 1, n, S, P.U, P.Z, P.sc);
  HB_CHECK_LAUNCH();
  // F [S, M] = Z A^T, then R = (y - F) / var / S in place
  HB_TRY(gemm64(P.cx, P.Z, n, 0, 0, A, n, 1, 0, P.F, M, 0, S, M, n, 1.0, 0.0));
  linop64_resid_kernel<<<LL_BLOCKS, LL_THREADS, 0, st>>>(P.F, y, M, (long long)S * M, P.sc, 1.0 / (double)S, P.part);
  HB_CHECK_LAUNCH();
  // partial Zbar [S, n] = R A (this rank's rows), then the stats
  HB_TRY(gemm64(P.cx, P.F, M, 0, 0, A, n, 0, 0, zbar_stats, n, 0, S, n, M, 1.0, 0.0));
  linop64_stats_kernel<<<1, 32, 0, st>>>(P.part, P.sc, (double)S * (double)M, zbar_stats + Sn);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

int hb_linop_elbo_update_f64(const hb_linop_config* cfg, double* params, const double* zbar_stats, double* grads, double* m,
                             double* v, const hb_adam_config* adam, double* out4, void* ws, size_t ws_bytes, void* stream) {
  if (!cfg || !params || !zbar_stats || !out4) return HB_ERR_ARG;
  const hb_linop_config c = *cfg;
  if (!cfg64_ok(c)) return HB_ERR_ARG;
  if ((m == nullptr) != (v == nullptr) || (m && !adam)) return HB_ERR_ARG;
  if (!ws || ws_bytes < linop64_layout(c).total + 256) return HB_ERR_WORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const Linop64Ptrs P = linop64_ptrs(c, ws, st);
  const int n = c.n, S = c.S;
  const size_t nn = (size_t)n * n;
  const double invS = 1.0 / (double)S;
  const long long Sn = (long long)S * n;

  linop64_zt_kernel<<<(int)std::min<long long>((Sn + 255) / 256, 148 * 8), 256, 0, st>>>(zbar_stats, P.Z, invS, Sn, P.Zt);
  HB_CHECK_LAUNCH();
  linop64_colsum_kernel<<<cdiv(n, 256), 256, 0, st>>>(P.Zt, n, S, P.gt);
  HB_CHECK_LAUNCH();
  linop64_scalars_kernel<<<1, 32, 0, st>>>(zbar_stats + Sn, P.sc, (double)S * (double)c.M_total, invS, P.gt + n, out4);
  HB_CHECK_LAUNCH();
  if (grads && cudaMemcpyAsync(grads + nn, P.gt, ((size_t)n + 1) * sizeof(double), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    return HB_ERR_CUDA;
  const double lr = m ? adam->lr : 0.0, b1 = m ? adam->b1 : 0.0, b2 = m ? adam->b2 : 0.0, ea = m ? adam->eps : 0.0;
  const double gs = m ? adam->grad_scale : 0.0;
  const int* step_dev = m ? adam->step_dev : nullptr;
  const int step_host = m ? adam->step_host : 0;
  const long long t = cdiv(n, TA_TILE);
  tril_rank_adam_f64_kernel<<<(unsigned)(t * (t + 1) / 2), 256, 0, st>>>(params, m, v, grads, P.Zt, P.U, n, S, lr, b1, b2, ea, gs,
                                                                       step_dev, step_host);
  HB_CHECK_LAUNCH();
  if (m) {
    gp64_adam_kernel<<<cdiv(n + 1, 256), 256, 0, st>>>(params + nn, P.gt, m + nn, v + nn, (long long)n + 1, n, 0, step_dev,
                                                       step_host, lr, b1, b2, ea, gs);
    HB_CHECK_LAUNCH();
  }
  return HB_OK;
}

}  // extern "C"
