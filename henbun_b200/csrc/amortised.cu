// Whole-step entry point of the amortised local-variable model (BASELINE config 4):
//     q_local = enc(X)                       nn.NeuralNet, Henbun/nn.py:34-87 (MatBias :10-32)
//     x_rec   = dec(q_local)                 LOCAL Normal fed by the encoder: param.py:386-392, 516-537; sampler variationals.py:138-142
//     ELBO    = reduce_sum(gaussian(X, x_rec, var)) - KL(LOCAL)        densities.py:25-27, variationals.py:225-230
// The reference emits ~40 TensorFlow ops per direction for this graph and the round-1 port replayed it through the autograd
// tape.  Here the step is one host-sequenced chain of this library's kernels with no Python, no tape and no temporaries
// between them: MatBias products with the bias / activation epilogue, the sampler reading mu | log sigma as strided
// halves of the encoder's output row and writing its gradient back the same way, the log-likelihood reduced in the same
// pass that writes dELBO/dx_rec (the [S B, 784] log-density tensor is never materialised), activation-backward fused with
// the bias-gradient column sums, tall dW reductions by deterministic split-K.
#include "../../include/henbun_b200.h"
#include "amortised.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

namespace hb {
namespace {

inline size_t au(size_t x) { return (x + 255) / 256 * 256; }

__global__ void am_prep_kernel(const float* p_var, float* sc) {
  if (threadIdx.x == 0) sc[0] = softplus_f(*p_var) + 1e-6f;
}
// out3 = {loglik, sum E^2, .}: ELBO pieces and the free-space gradient of var
__global__ void am_finish_kernel(const float* sc, const float* out3, const float* kl, double total, int S, const float* p_var,
                                 float* g_var, float* out4) {
  if (threadIdx.x == 0) {
    const double v = sc[0], invS = 1.0 / (double)S;
    const double gv = invS * (-0.5 * total / v + 0.5 * (double)out3[1] / (v * v));
    *g_var = (float)(gv * (double)sigmoid_f(*p_var));
    out4[0] = (float)(((double)out3[0] - (double)*kl) * invS);
    out4[1] = out3[0]; out4[2] = *kl; out4[3] = 0.f;
  }
}

struct Net {
  int n;                     // layers
  const int* nodes;          // n + 1 widths
  const int* act;            // n - 1 hidden activations
  size_t w_off[HB_MAX_LAYERS], b_off[HB_MAX_LAYERS];   // offsets into params / grads
};

struct Layout {
  size_t a_enc[HB_MAX_LAYERS + 1], a_dec[HB_MAX_LAYERS + 1];   // activations (a_enc[0] is the caller's X)
  size_t g0, g1, sc, red, tc, total;
  size_t tc_bytes;
};

size_t max_width(const hb_amortised_config& c) {
  int m = 0;
  for (int i = 0; i <= c.n_enc; ++i) m = c.enc_nodes[i] > m ? c.enc_nodes[i] : m;
  for (int i = 0; i <= c.n_dec; ++i) m = c.dec_nodes[i] > m ? c.dec_nodes[i] : m;
  return (size_t)m;
}

Layout layout(const hb_amortised_config& c) {
  Layout L{};
  size_t o = 0;
  const size_t rows_d = (size_t)c.S * c.B;
  for (int i = 1; i <= c.n_enc; ++i) { L.a_enc[i] = o; o += au((size_t)c.B * c.enc_nodes[i] * 4); }
  for (int i = 0; i <= c.n_dec; ++i) { L.a_dec[i] = o; o += au(rows_d * c.dec_nodes[i] * 4); }
  const size_t gbytes = au(rows_d * max_width(c) * 4);
  L.g0 = o; o += gbytes;
  L.g1 = o; o += gbytes;
  L.sc = o; o += au(64 * 4);
  L.red = o; o += au(kReduceWsBytes);
  L.tc_bytes = (size_t)64 << 20;
  L.tc = o; o += au(L.tc_bytes);
  L.total = o;
  return L;
}

// y[rows, out] = act(x[rows, in] W + b)
int layer_fwd(const float* x, const float* W, const float* b, float* y, int rows, int in, int out, int act, void* ws, size_t wsb,
              cudaStream_t st) {
  GemmParams g;
  g.A = x; g.lda = in; g.B = W; g.ldb = out; g.C = y; g.ldc = out; g.M = rows; g.N = out; g.K = in;
  g.bias = b; g.act = act; g.ws = ws; g.ws_bytes = wsb;
  return gemm(g, st);
}

// backward of one layer: gy -> (dz in place of scratch), dW, db, gx (may be null)
int layer_bwd(const float* gy, const float* y, const float* x, const float* W, float* dz, float* dW, float* db, float* gx,
              long long ld_gx, int rows, int in, int out, int act, void* red, void* ws, size_t wsb, cudaStream_t st) {
  HB_TRY(act_bwd_colsum_ws(gy, y, dz, rows, out, out, act, 0, 0.f, 0.f, db, ws, wsb, st));
  (void)red;
  {
    GemmParams g;     // dW[in, out] = x^T dz  (tall reduction over the rows)
    g.A = x; g.lda = in; g.transA = 1; g.B = dz; g.ldb = out; g.C = dW; g.ldc = out; g.M = in; g.N = out; g.K = rows;
    g.ws = ws; g.ws_bytes = wsb; g.hint_split_waves = 1;
    HB_TRY(gemm(g, st));
  }
  if (gx) {
    GemmParams g;     // gx[rows, in] = dz W^T
    g.A = dz; g.lda = out; g.B = W; g.ldb = out; g.transB = 1; g.C = gx; g.ldc = ld_gx; g.M = rows; g.N = in; g.K = out;
    g.ws = ws; g.ws_bytes = wsb;
    HB_TRY(gemm(g, st));
  }
  return HB_OK;
}

}  // namespace

bool amortised_valid(const hb_amortised_config& c) {
  if (c.B <= 0 || c.S <= 0 || c.latent <= 0) return false;
  if (c.n_enc < 1 || c.n_enc > HB_MAX_LAYERS || c.n_dec < 1 || c.n_dec > HB_MAX_LAYERS) return false;
  if (c.enc_nodes[c.n_enc] != 2 * c.latent || c.dec_nodes[0] != c.latent) return false;
  if (c.dec_nodes[c.n_dec] != c.enc_nodes[0]) return false;          // gaussian(X, dec(z), var): same width as the data
  for (int i = 0; i <= c.n_enc; ++i) if (c.enc_nodes[i] <= 0) return false;
  for (int i = 0; i <= c.n_dec; ++i) if (c.dec_nodes[i] <= 0) return false;
  for (int i = 0; i + 1 < c.n_enc; ++i) if (c.enc_act[i] < 0 || c.enc_act[i] > 3) return false;
  for (int i = 0; i + 1 < c.n_dec; ++i) if (c.dec_act[i] < 0 || c.dec_act[i] > 3) return false;
  return true;
}

size_t amortised_net_params(const int* nodes, int n, size_t start, size_t* w_off, size_t* b_off) {
  size_t o = start;
  for (int l = 0; l < n; ++l) {
    w_off[l] = o; o += (size_t)nodes[l] * nodes[l + 1];
    b_off[l] = o; o += (size_t)nodes[l + 1];
  }
  return o;
}

}  // namespace hb

using namespace hb;

extern "C" {

size_t hb_amortised_param_count(const hb_amortised_config* c) {
  if (!c || !amortised_valid(*c)) return 0;
  size_t w[HB_MAX_LAYERS], b[HB_MAX_LAYERS];
  size_t o = amortised_net_params(c->enc_nodes, c->n_enc, 0, w, b);
  o = amortised_net_params(c->dec_nodes, c->n_dec, o, w, b);
  return o + 1;
}

size_t hb_amortised_workspace_bytes(const hb_amortised_config* c) {
  if (!c || !amortised_valid(*c)) return 0;
  return layout(*c).total + 256;
}

int hb_amortised_elbo_step(const hb_amortised_config* cfg, const float* X, const float* params, const float* eps, float* grads,
                           float* out4, void* ws, size_t ws_bytes, void* stream) {
  if (!cfg || !X || !params || !grads || !out4) return HB_ERR_ARG;
  OptScope scope(cfg->opt);
  const hb_amortised_config c = *cfg;
  if (!amortised_valid(c)) return HB_ERR_ARG;
  if (!eps && (c.offset & 3ull)) return HB_ERR_ARG;
  const Layout L = layout(c);
  if (!ws || ws_bytes < L.total + 256) return HB_ERR_WORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  auto F = [&](size_t off) { return reinterpret_cast<float*>(base + off); };
  size_t ew[HB_MAX_LAYERS], eb[HB_MAX_LAYERS], dw[HB_MAX_LAYERS], db[HB_MAX_LAYERS];
  size_t o = amortised_net_params(c.enc_nodes, c.n_enc, 0, ew, eb);
  o = amortised_net_params(c.dec_nodes, c.n_dec, o, dw, db);
  const size_t var_off = o;
  float* sc = F(L.sc);
  float* out3 = sc + 8;
  float* kl = sc + 16;
  void* red = base + L.red;
  void* tcw = base + L.tc;
  const int B = c.B, S = c.S, lat = c.latent;
  const long long rows_d = (long long)S * B;
  if (rows_d > 0x7fffffffLL) return HB_ERR_ARG;

  am_prep_kernel<<<1, 32, 0, st>>>(params + var_off, sc);
  HB_CHECK_LAUNCH();

  // ---- encoder forward ----
  const float* a = X;
  for (int l = 0; l < c.n_enc; ++l) {
    const int act = (l + 1 < c.n_enc) ? c.enc_act[l] : ACT_NONE;
    HB_TRY(layer_fwd(a, params + ew[l], params + eb[l], F(L.a_enc[l + 1]), B, c.enc_nodes[l], c.enc_nodes[l + 1], act, tcw, L.tc_bytes, st));
    a = F(L.a_enc[l + 1]);
  }
  const float* h = a;                                           // [B, 2 latent]: mu | log sigma
  // ---- LOCAL sampler + KL: z [S, B, latent] ----
  HB_TRY(sample_diag_fwd(h, 2 * lat, h + lat, 2 * lat, B, lat, eps, c.seed, c.offset, S, F(L.a_dec[0]), kl, red, kReduceWsBytes, st));
  // ---- decoder forward ----
  a = F(L.a_dec[0]);
  for (int l = 0; l < c.n_dec; ++l) {
    const int act = (l + 1 < c.n_dec) ? c.dec_act[l] : ACT_NONE;
    HB_TRY(layer_fwd(a, params + dw[l], params + db[l], F(L.a_dec[l + 1]), (int)rows_d, c.dec_nodes[l], c.dec_nodes[l + 1], act, tcw,
                     L.tc_bytes, st));
    a = F(L.a_dec[l + 1]);
  }
  // ---- log-likelihood + dELBO/dx_rec in one pass (x broadcast over the S samples) ----
  const int Dx = c.enc_nodes[0];
  const long long total = rows_d * Dx;
  float* g_cur = F(L.g0);
  float* g_alt = F(L.g1);
  HB_TRY(gauss_loglik_fwd(a, nullptr, X, total, (long long)B * Dx, sc, 1.f / (float)S, g_cur, out3, red, kReduceWsBytes, st));

  // ---- decoder backward ----
  for (int l = c.n_dec - 1; l >= 0; --l) {
    const int act = (l + 1 < c.n_dec) ? c.dec_act[l] : ACT_NONE;
    float* dz = g_alt;
    // gradient w.r.t. this layer's input goes to where the incoming gradient lived (it is dead after act_bwd)
    HB_TRY(layer_bwd(g_cur, F(L.a_dec[l + 1]), F(L.a_dec[l]), params + dw[l], dz, grads + dw[l], grads + db[l], g_cur,
                     c.dec_nodes[l], (int)rows_d, c.dec_nodes[l], c.dec_nodes[l + 1], act, red, tcw, L.tc_bytes, st));
  }
  // g_cur = dELBO/dz [S, B, latent] (likelihood path)
  // ---- sampler backward into dh [B, 2 latent] (strided halves), KL included ----
  float* dh = g_alt;
  HB_TRY(sample_diag_bwd(h, 2 * lat, h + lat, 2 * lat, B, lat, eps, c.seed, c.offset, S, g_cur, nullptr, 1.f / (float)S, nullptr,
                         dh, 2 * lat, dh + lat, 2 * lat, 0.f, st));
  // ---- encoder backward ----
  float* gy = dh;
  float* other = g_cur;
  for (int l = c.n_enc - 1; l >= 0; --l) {
    const int act = (l + 1 < c.n_enc) ? c.enc_act[l] : ACT_NONE;
    const float* xin = (l == 0) ? X : F(L.a_enc[l]);
    // dz may not alias gy here (gy is read by act_bwd while dz is written elementwise: same index -> safe), use `other`
    HB_TRY(layer_bwd(gy, F(L.a_enc[l + 1]), xin, params + ew[l], other, grads + ew[l], grads + eb[l], (l > 0) ? gy : nullptr,
                     c.enc_nodes[l], B, c.enc_nodes[l], c.enc_nodes[l + 1], act, red, tcw, L.tc_bytes, st));
  }
  am_finish_kernel<<<1, 32, 0, st>>>(sc, out3, kl, (double)total, S, params + var_off, grads + var_off, out4);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

}  // extern "C"
