// float64 amortised local-variable model (BASELINE config 4): the step of csrc/amortised.cu in double, the reference's
// float_type = float64 (henbunrc:7).
//     h = enc(X) = [mu | log sigma],  z = mu + exp(log sigma) u,  x_rec = dec(z)
//     ELBO = [sum gaussian(X, x_rec, var) - KL(LOCAL)] / S,  KL = -1/2 sum(2 log sigma + u^2 - z^2)
// Data that is not centred is where fp32 loses: the decoder's last bias carries the common level c and every gradient
// flows from the small difference X - x_rec, so fp32 errors grow in proportion to c.
//
// The chain mirrors amortised.cu launch for launch.  MatBias products run on f64.cu's DMMA GEMM with the bias and
// activation in its epilogue; the weight gradients dW = x^T dz reduce over S B rows by split-K in a fixed split order.  The
// sampler reads mu | log sigma as strided halves of the encoder's output row and writes its gradient back the same way; the
// log-likelihood is reduced in the pass that writes d ELBO / d x_rec (the [S B, Dx] log-density tensor is never stored);
// activation backward is fused with the bias-gradient column sums.  Every reduction sums fixed partials in a fixed order
// and nothing uses atomics, so results are bitwise repeatable.
#include "../../include/henbun_b200.h"
#include "amortised.cuh"
#include "f64.cuh"
#include "gemm.cuh"
#include "tmath.cuh"
#include <algorithm>

namespace hb {
namespace {

constexpr int RB_THREADS = 256;
constexpr int RB_BLOCKS = 148 * 8;                       // fixed partial sums of sum E^2 and of the KL terms
constexpr int CS_MAX_ROWBLOCKS = 128;                    // row blocks of the column sums (partials per column)
// sc: [0] var, [1] d var / d free
constexpr int SC_N = 16;

struct Am64Layout {
  size_t a_enc[HB_MAX_LAYERS + 1], a_dec[HB_MAX_LAYERS + 1];   // activations (a_enc[0] is the caller's X)
  size_t U, g0, g1, sc, part_ll, part_kl, part_cs, grad, split, total;
  size_t split_bytes;
};

int max_width(const hb_amortised_config& c) {
  int m = 0;
  for (int i = 0; i <= c.n_enc; ++i) m = std::max(m, c.enc_nodes[i]);
  for (int i = 0; i <= c.n_dec; ++i) m = std::max(m, c.dec_nodes[i]);
  return m;
}

size_t npar_of(const hb_amortised_config& c) {
  size_t w[HB_MAX_LAYERS], b[HB_MAX_LAYERS];
  return amortised_net_params(c.dec_nodes, c.n_dec, amortised_net_params(c.enc_nodes, c.n_enc, 0, w, b), w, b) + 1;
}

Am64Layout am64_layout(const hb_amortised_config& c) {
  Am64Layout L{};
  const size_t rows_d = (size_t)c.S * c.B, d = sizeof(double);
  size_t o = 0;
  for (int i = 1; i <= c.n_enc; ++i) { L.a_enc[i] = o; o += align256((size_t)c.B * c.enc_nodes[i] * d); }
  for (int i = 0; i <= c.n_dec; ++i) { L.a_dec[i] = o; o += align256(rows_d * c.dec_nodes[i] * d); }
  L.U = o; o += align256(rows_d * c.latent * d);
  const size_t gbytes = align256(rows_d * max_width(c) * d);
  L.g0 = o; o += gbytes;
  L.g1 = o; o += gbytes;
  L.sc = o; o += align256(SC_N * d);
  L.part_ll = o; o += align256(RB_BLOCKS * d);
  L.part_kl = o; o += align256(RB_BLOCKS * d);
  L.part_cs = o; o += align256((size_t)CS_MAX_ROWBLOCKS * max_width(c) * d);
  L.grad = o; o += align256(npar_of(c) * d);
  // partial tiles: the tall dW reductions' splits, at least what the GEMM's own small-output rule may take
  size_t sb = kSplitWsBytes;
  for (int net = 0; net < 2; ++net) {
    const int n = net ? c.n_dec : c.n_enc;
    const int* nodes = net ? c.dec_nodes : c.enc_nodes;
    const int rows = net ? (int)std::min<size_t>(rows_d, 0x7fffffff) : c.B;
    for (int l = 0; l < n; ++l) sb = std::max(sb, gemm64_split_bytes(nodes[l], nodes[l + 1], rows, 1));
  }
  L.split_bytes = align256(sb);
  L.split = o; o += L.split_bytes;
  L.total = o;
  return L;
}

__global__ void am64_prep_kernel(const double* __restrict__ p_var, double* sc) {
  if (threadIdx.x == 0) {
    const double x = *p_var;
    sc[0] = t_softplus<double>(x) + 1e-6;
    sc[1] = t_sigmoid<double>(x);
  }
}

// U = eps (or the library's Philox stream widened to double: element e of [S, B, latent] is stream position offset + e, as in
// sampler.cu's sample_diag_fwd), Z = mu + exp(log sigma) U with mu | log sigma the halves of h's row b.  Block b writes its
// partial sum of the KL terms 2 log sigma + u^2 - z^2 to part[b]; the element assignment depends on the fixed grid only.
__global__ void __launch_bounds__(RB_THREADS) am64_sample_kernel(const double* __restrict__ h, int L, long long P, long long total,
                                                               const double* __restrict__ eps, unsigned long long seed,
                                                               unsigned long long offset, double* __restrict__ U,
                                                               double* __restrict__ Z, double* __restrict__ part) {
  __shared__ double red[32];
  double v[1] = {0.0};
  const long long ngroups = (total + 3) / 4;
  for (long long g = blockIdx.x * (long long)RB_THREADS + threadIdx.x; g < ngroups; g += (long long)RB_BLOCKS * RB_THREADS) {
    float u4[4] = {0.f, 0.f, 0.f, 0.f};
    if (!eps) philox_normal4(seed, (offset >> 2) + (unsigned long long)g, u4);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const long long e = 4 * g + q;
      if (e >= total) break;
      const double u = eps ? eps[e] : (double)u4[q];
      const long long p = e % P, b = p / L;
      const int j = (int)(p % L);
      const double om = h[b * 2 * L + L + j];
      const double z = h[b * 2 * L + j] + exp(om) * u;
      U[e] = u;
      Z[e] = z;
      v[0] += 2.0 * om + u * u - z * z;
    }
  }
  block_sum<1>(v, red);
  if (threadIdx.x == 0) part[blockIdx.x] = v[0];
}

// R = (X - x_rec) / var / S = d ELBO / d x_rec with X [B, Dx] broadcast over the S samples; block b writes its partial sum
// of E^2 to part[b]
__global__ void __launch_bounds__(RB_THREADS) am64_loglik_kernel(const double* __restrict__ xr, const double* __restrict__ X,
                                                               long long period, long long total, const double* __restrict__ sc,
                                                               double invS, double* __restrict__ R, double* __restrict__ part) {
  __shared__ double red[32];
  const double scale = invS / sc[0];
  double v[1] = {0.0};
  for (long long e = blockIdx.x * (long long)RB_THREADS + threadIdx.x; e < total; e += (long long)RB_BLOCKS * RB_THREADS) {
    const double E = X[e % period] - xr[e];
    v[0] += E * E;
    R[e] = E * scale;
  }
  block_sum<1>(v, red);
  if (threadIdx.x == 0) part[blockIdx.x] = v[0];
}

// dz = gy act'(y) (written only for a hidden layer; a linear layer's dz is gy) fused with the column sums of dz: block
// (x, y) takes 32 columns and the rows of chunk y, and writes one partial per column to part[y * cols + c]
__global__ void __launch_bounds__(256) am64_act_bwd_colsum_kernel(const double* __restrict__ gy, const double* __restrict__ y,
                                                                double* __restrict__ dz, int rows, int cols, int act, int chunk,
                                                                double* __restrict__ part) {
  __shared__ double red[8][33];
  const int tx = threadIdx.x, ty = threadIdx.y, c = blockIdx.x * 32 + tx;
  const int r0 = blockIdx.y * chunk, r1 = min(rows, r0 + chunk);
  double s = 0.0;
  if (c < cols) {
    for (int r = r0 + ty; r < r1; r += 8) {
      const long long i = (long long)r * cols + c;
      double g = gy[i];
      if (act != ACT_NONE) {
        const double yv = y[i];
        g *= act == ACT_SIGMOID ? yv * (1.0 - yv) : act == ACT_RELU ? (yv > 0.0 ? 1.0 : 0.0) : 1.0 - yv * yv;
        dz[i] = g;
      }
      s += g;
    }
  }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && c < cols) {
    double t = 0.0;
    for (int k = 0; k < 8; ++k) t += red[k][tx];
    part[(long long)blockIdx.y * cols + c] = t;
  }
}

__global__ void am64_colsum_finish_kernel(const double* __restrict__ part, int nrb, int cols, double* __restrict__ out) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int b = 0; b < nrb; ++b) s += part[(long long)b * cols + c];
    out[c] = s;
  }
}

// sampler backward into dh [B, 2 latent] (strided halves), the KL included: with zt = zbar - z / S,
//   d mu = sum_s zt,  d log sigma = exp(log sigma) sum_s zt u + 1
__global__ void am64_sampler_bwd_kernel(const double* __restrict__ zbar, const double* __restrict__ U, const double* __restrict__ Z,
                                        const double* __restrict__ h, int L, long long P, int S, double invS,
                                        double* __restrict__ dh) {
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < P; p += (long long)gridDim.x * blockDim.x) {
    const long long b = p / L;
    const int j = (int)(p % L);
    double gm = 0.0, go = 0.0;
    for (int s = 0; s < S; ++s) {
      const long long i = (long long)s * P + p;
      const double zt = zbar[i] - invS * Z[i];
      gm += zt;
      go += zt * U[i];
    }
    dh[b * 2 * L + j] = gm;
    dh[b * 2 * L + L + j] = go * exp(h[b * 2 * L + L + j]) + 1.0;
  }
}

// the ELBO pieces from the partials (block order) and the free-space gradient of var; out4 = {ELBO, loglik, kl, 0}
__global__ void am64_finish_kernel(const double* __restrict__ sc, const double* __restrict__ part_ll,
                                   const double* __restrict__ part_kl, double elems, double invS, double* g_var, double* out4) {
  if (threadIdx.x == 0) {
    double e2 = 0.0, k = 0.0;
    for (int b = 0; b < RB_BLOCKS; ++b) e2 += part_ll[b];
    for (int b = 0; b < RB_BLOCKS; ++b) k += part_kl[b];
    const double v = sc[0], kl = -0.5 * k;
    const double ll = -elems * (0.9189385332046727 + 0.5 * log(v)) - 0.5 * e2 / v;
    *g_var = invS * (-0.5 * elems / v + 0.5 * e2 / (v * v)) * sc[1];
    out4[0] = (ll - kl) * invS;
    out4[1] = ll;
    out4[2] = kl;
    out4[3] = 0.0;
  }
}

// backward of y = act(x W + b) over `rows` rows: db, dW = x^T dz (tall reduction: split-K) and, when gx is not null,
// gx = dz W^T.  dz = gy act'(y) goes to dz_buf for a hidden layer and is gy itself for a linear one; gx must not alias it.
int layer_bwd64(const Ctx64& cx, const double* gy, const double* y, const double* x, const double* W, double* dz_buf, double* dW,
                double* db, double* gx, int rows, int in, int out, int act, double* part) {
  const int nrb = std::min(CS_MAX_ROWBLOCKS, cdiv(rows, 64));
  const int chunk = cdiv(rows, nrb);
  am64_act_bwd_colsum_kernel<<<dim3(cdiv(out, 32), nrb), dim3(32, 8), 0, cx.st>>>(gy, y, dz_buf, rows, out, act, chunk, part);
  HB_CHECK_LAUNCH();
  am64_colsum_finish_kernel<<<cdiv(out, 256), 256, 0, cx.st>>>(part, nrb, out, db);
  HB_CHECK_LAUNCH();
  const double* dz = act != ACT_NONE ? dz_buf : gy;
  HB_TRY(gemm64_ex(cx, x, in, 1, dz, out, 0, dW, out, in, out, rows, 0.0, nullptr, ACT_NONE, 1));
  if (gx) HB_TRY(gemm64_ex(cx, dz, out, 0, W, out, 1, gx, in, rows, in, out, 0.0, nullptr, ACT_NONE, 0));
  return HB_OK;
}

// backward through the layers of one net from gy (the gradient of its output, in *gy) down to its input: on return *gy
// holds the gradient of the net's input (when want_gx) and *spare is free
int net_bwd64(const Ctx64& cx, const double* params, double* G, const int* nodes, const int* acts, int n, const size_t* w_off,
              const size_t* b_off, const double* const* a, int rows, bool want_gx, double** gy, double** spare, double* part) {
  for (int l = n - 1; l >= 0; --l) {
    const int act = (l + 1 < n) ? acts[l] : ACT_NONE;
    const bool gx_wanted = want_gx || l > 0;
    // a hidden layer's dz goes to *spare and *gy is dead after it: gx overwrites *gy; a linear layer's dz is *gy: gx goes to *spare
    double* gx = !gx_wanted ? nullptr : (act != ACT_NONE ? *gy : *spare);
    HB_TRY(layer_bwd64(cx, *gy, a[l + 1], a[l], params + w_off[l], *spare, G + w_off[l], G + b_off[l], gx, rows, nodes[l],
                       nodes[l + 1], act, part));
    if (gx && act == ACT_NONE) std::swap(*gy, *spare);
  }
  return HB_OK;
}

}  // namespace
}  // namespace hb

using namespace hb;

extern "C" {

size_t hb_amortised_f64_workspace_bytes(const hb_amortised_config* cfg) {
  if (!cfg || !amortised_valid(*cfg)) return 0;
  return am64_layout(*cfg).total + 256;
}

int hb_amortised_elbo_step_f64(const hb_amortised_config* cfg, const double* X, double* params, const double* eps, double* grads,
                               double* out4, double* adam_m, double* adam_v, const hb_adam_config* adam, void* ws,
                               size_t ws_bytes, void* stream) {
  if (!cfg || !X || !params || !out4) return HB_ERR_ARG;
  const hb_amortised_config c = *cfg;
  if (!amortised_valid(c)) return HB_ERR_ARG;
  if ((adam_m == nullptr) != (adam_v == nullptr) || (adam_m && !adam) || (!adam_m && !grads)) return HB_ERR_ARG;
  if (!eps && (c.offset & 3ull)) return HB_ERR_ARG;
  const long long rows_d = (long long)c.S * c.B;
  if (rows_d > 0x7fffffffLL) return HB_ERR_ARG;
  const Am64Layout Lw = am64_layout(c);
  if (!ws || ws_bytes < Lw.total + 256) return HB_ERR_WORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  auto D = [&](size_t off) { return reinterpret_cast<double*>(base + off); };
  const Ctx64 cx{st, nullptr, base + Lw.split, Lw.split_bytes};
  size_t ew[HB_MAX_LAYERS], eb[HB_MAX_LAYERS], dw[HB_MAX_LAYERS], db[HB_MAX_LAYERS];
  const size_t var_off = amortised_net_params(c.dec_nodes, c.n_dec, amortised_net_params(c.enc_nodes, c.n_enc, 0, ew, eb), dw, db);
  const size_t npar = var_off + 1;
  double* G = grads ? grads : D(Lw.grad);
  double* sc = D(Lw.sc);
  double* U = D(Lw.U);
  double* part_cs = D(Lw.part_cs);
  const int B = c.B, S = c.S, lat = c.latent, Dx = c.enc_nodes[0];
  const double invS = 1.0 / (double)S;
  const double* a_enc[HB_MAX_LAYERS + 1];
  const double* a_dec[HB_MAX_LAYERS + 1];
  a_enc[0] = X;
  for (int i = 1; i <= c.n_enc; ++i) a_enc[i] = D(Lw.a_enc[i]);
  for (int i = 0; i <= c.n_dec; ++i) a_dec[i] = D(Lw.a_dec[i]);

  am64_prep_kernel<<<1, 32, 0, st>>>(params + var_off, sc);
  HB_CHECK_LAUNCH();
  // ---- encoder forward: h [B, 2 latent] = mu | log sigma ----
  for (int l = 0; l < c.n_enc; ++l) {
    const int act = (l + 1 < c.n_enc) ? c.enc_act[l] : ACT_NONE;
    HB_TRY(gemm64_ex(cx, a_enc[l], c.enc_nodes[l], 0, params + ew[l], c.enc_nodes[l + 1], 0, D(Lw.a_enc[l + 1]), c.enc_nodes[l + 1],
                     B, c.enc_nodes[l + 1], c.enc_nodes[l], 0.0, params + eb[l], act, 0));
  }
  const double* h = a_enc[c.n_enc];
  // ---- LOCAL sampler + KL partials: z [S, B, latent] ----
  const long long P = (long long)B * lat;
  am64_sample_kernel<<<RB_BLOCKS, RB_THREADS, 0, st>>>(h, lat, P, rows_d * lat, eps, c.seed, c.offset, U, D(Lw.a_dec[0]),
                                                      D(Lw.part_kl));
  HB_CHECK_LAUNCH();
  // ---- decoder forward ----
  for (int l = 0; l < c.n_dec; ++l) {
    const int act = (l + 1 < c.n_dec) ? c.dec_act[l] : ACT_NONE;
    HB_TRY(gemm64_ex(cx, a_dec[l], c.dec_nodes[l], 0, params + dw[l], c.dec_nodes[l + 1], 0, D(Lw.a_dec[l + 1]), c.dec_nodes[l + 1],
                     (int)rows_d, c.dec_nodes[l + 1], c.dec_nodes[l], 0.0, params + db[l], act, 0));
  }
  // ---- log-likelihood partials + d ELBO / d x_rec in one pass ----
  double* gy = D(Lw.g0);
  double* spare = D(Lw.g1);
  am64_loglik_kernel<<<RB_BLOCKS, RB_THREADS, 0, st>>>(a_dec[c.n_dec], X, (long long)B * Dx, rows_d * Dx, sc, invS, gy,
                                                      D(Lw.part_ll));
  HB_CHECK_LAUNCH();
  // ---- decoder backward: *gy ends as d ELBO / d z [S, B, latent] (likelihood path) ----
  HB_TRY(net_bwd64(cx, params, G, c.dec_nodes, c.dec_act, c.n_dec, dw, db, a_dec, (int)rows_d, true, &gy, &spare, part_cs));
  // ---- sampler backward into dh [B, 2 latent], KL included ----
  am64_sampler_bwd_kernel<<<cdiv(P, 256), 256, 0, st>>>(gy, U, a_dec[0], h, lat, P, S, invS, spare);
  HB_CHECK_LAUNCH();
  std::swap(gy, spare);
  // ---- encoder backward ----
  HB_TRY(net_bwd64(cx, params, G, c.enc_nodes, c.enc_act, c.n_enc, ew, eb, a_enc, B, false, &gy, &spare, part_cs));
  am64_finish_kernel<<<1, 32, 0, st>>>(sc, D(Lw.part_ll), D(Lw.part_kl), (double)rows_d * (double)Dx, invS, G + var_off, out4);
  HB_CHECK_LAUNCH();
  if (adam_m) {
    gp64_adam_kernel<<<(int)std::min<long long>(((long long)npar + 255) / 256, 148 * 8), 256, 0, st>>>(
        params, G, adam_m, adam_v, (long long)npar, 0, 0, adam->step_dev, adam->step_host, adam->lr, adam->b1, adam->b2, adam->eps,
        adam->grad_scale);
    HB_CHECK_LAUNCH();
  }
  return HB_OK;
}

}  // extern "C"
