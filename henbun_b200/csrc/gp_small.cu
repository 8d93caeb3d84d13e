// One persistent CTA for the whole ELBO + gradient (+ TF-1 Adam) step of the variational GP regression graph when the
// model is notebook sized (n <= 128 in fp32, n <= 112 in fp64):
//     notebooks/GaussianProcess.ipynb:109-148   y_fit = matmul(kern.Cholesky(X), q) * sqrt(k_var)
//                                                ELBO  = reduce_sum(gaussian(Y, y_fit, var)) - KL()
// The reference launches ~60 TensorFlow ops per session.run for this graph; round 1 of this library needed 23 kernels
// (0.24 ms per step, 60 % of it in two one-CTA leaf kernels that also computed block inverses nobody needs at this
// size).  Here the Gram matrix, its Cholesky factor and the adjoint live in shared memory from the first to the last
// instruction: Gram -> potrf (right-looking, one column per step) -> sampler + KL -> F = a L Z^T -> log-likelihood ->
// z-bar, L-bar -> sampler backward -> reverse-mode Cholesky (level-2 form of Murray 2016, in place, no inverse) ->
// Gram backward -> scalar chain rules -> optional Adam.  The arithmetic type is a template parameter: the fp64
// instantiation is the float_type = float64 path of the reference (henbunrc:7) for the 1-D notebook inputs, whose Gram
// matrices (cond 1e6) put an fp32 factorisation 3 orders of magnitude away from the 1e-5 parity bar.
#include "kernels.cuh"
#include "leaf_smem.cuh"
#include "tmath.cuh"

namespace hb {

namespace {

constexpr int GS_THREADS = 512;

template <typename T> struct SmallLimits;
template <> struct SmallLimits<float> { static constexpr int max_n = 128; };
template <> struct SmallLimits<double> { static constexpr int max_n = 112; };

template <typename T>
struct SmallArgs {
  int n, D, S, n_ell, q_fullrank;
  T jitter;
  unsigned long long seed, offset;
  const T* X; const T* Y; T* params; const T* eps; T* grads; T* out4;
  T* ws;                 // 4 * S * n elements: Z | U | R | Zbar
  int* err_flag;
  // optional fused Adam (m == nullptr: gradients only)
  T* m; T* v; const int* step_dev; int step_host; double lr, b1, b2, eps_adam, grad_scale;
  int vec_smem = 0;      // gp_leaf_step_kernel: Z | U | R | Zbar in shared memory (set by the launcher)
};

// block-wide sum of one double per thread; result broadcast to every thread
__device__ __forceinline__ double block_sum_all(double v, double* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < GS_THREADS / 32; ++i) t += red[i];
  return t;
}

template <typename T>
__global__ void __launch_bounds__(GS_THREADS, 1) gp_small_step_kernel(const SmallArgs<T> a) {
  extern __shared__ __align__(16) unsigned char gs_smem[];
  const int n = a.n, S = a.S, D = a.D, tid = threadIdx.x;
  const int LD = n | 1;                                  // odd leading dimension: conflict-free column walks
  T* L = reinterpret_cast<T*>(gs_smem);                  // K, then its Cholesky factor (lower)
  T* G = L + (size_t)n * LD;                             // L-bar, then K-bar (lower)
  T* ell = G + (size_t)n * LD;                           // [n_ell]
  T* colv = ell + 32;                                    // [n] scratch column
  __shared__ double red[GS_THREADS / 32];
  __shared__ int sh_bad;

  const size_t nq = a.q_fullrank ? (size_t)n * n : (size_t)n;
  T* p_mu = a.params; T* p_sq = a.params + n; T* p_scale = p_sq + nq; T* p_ell = p_scale + 1;
  T* p_kvar = p_ell + a.n_ell; T* p_var = p_kvar + 1;
  T* g_mu = a.grads; T* g_sq = a.grads + n; T* g_scale = g_sq + nq; T* g_ell = g_scale + 1;
  T* g_kvar = g_ell + a.n_ell; T* g_var = g_kvar + 1;
  T* Z = a.ws; T* U = Z + (size_t)S * n; T* R = U + (size_t)S * n; T* Zb = R + (size_t)S * n;

  // ---- positive hyper-parameters (transforms.positive: softplus + 1e-6, transforms.py:133-134) ----
  const T s_q = t_softplus<T>(*p_scale) + T(1e-6);
  const T kv = t_softplus<T>(*p_kvar) + T(1e-6);
  const T var = t_softplus<T>(*p_var) + T(1e-6);
  const T amp = t_sqrt<T>(kv) * s_q;
  for (int d = tid; d < a.n_ell; d += GS_THREADS) ell[d] = t_softplus<T>(p_ell[d]) + T(1e-6);
  __syncthreads();

  // ---- K = rbf(X) + jitter I, lower triangle (gp/kernels.py:54-84, 100-101, 110-111) ----
  for (int e = tid; e < n * n; e += GS_THREADS) {
    const int i = e / n, j = e % n;
    T val = T(0);
    if (j <= i) {
      T r2 = T(0);
      for (int d = 0; d < D; ++d) {
        const T df = (a.X[i * D + d] - a.X[j * D + d]) / ell[a.n_ell == 1 ? 0 : d];
        r2 += df * df;
      }
      val = t_exp<T>(T(-0.5) * r2) + (i == j ? a.jitter : T(0));
    }
    L[i * LD + j] = val;
  }
  __syncthreads();

  // ---- potrf, right-looking, one column per step (tf.cholesky) ----
  const int bad = potrf_cols_smem<T, GS_THREADS>(L, LD, n, colv, &sh_bad);
  if (tid == 0 && bad != 0 && a.err_flag) atomicCAS(a.err_flag, 0, bad);

  // ---- sampler + one-sample KL (variationals.py:138-146, 183-186, 225-230) ----
  double kl_part = 0.0;
  for (int e = tid; e < S * n; e += GS_THREADS) {
    const T u = a.eps ? a.eps[e] : (T)philox_normal_at(a.seed, a.offset, (unsigned long long)e);
    U[e] = u;
  }
  __syncthreads();
  if (a.q_fullrank) {       // stage q_sqrt in the adjoint's buffer (free until L-bar is formed): coalesced, read once
    for (int e = tid; e < n * n; e += GS_THREADS) G[(e / n) * LD + (e % n)] = p_sq[e];
    __syncthreads();
  }
  for (int e = tid; e < S * n; e += GS_THREADS) {
    const int s = e / n, i = e % n;
    T z, logdet;
    if (!a.q_fullrank) {
      z = p_mu[i] + t_exp<T>(p_sq[i]) * U[e];
      logdet = T(2) * p_sq[i];
    } else {
      T acc = p_mu[i];
      const T* lq = G + (size_t)i * LD;
      const T* ur = U + (size_t)s * n;
      for (int k = 0; k <= i; ++k) acc += lq[k] * ur[k];
      z = acc;
      logdet = t_log<T>(lq[i] * lq[i]);
    }
    Z[e] = z;
    const T u = U[e];
    kl_part += (double)(logdet + u * u - z * z);
  }
  const double kl = -0.5 * block_sum_all(kl_part, red);
  __syncthreads();

  // ---- F = amp * Z L^T, log-likelihood, residual R = dELBO/dF (densities.py:25-27) ----
  double ll_part = 0.0, e2_part = 0.0, ef_part = 0.0;
  const T inv_S = T(1) / (T)S;
  for (int e = tid; e < S * n; e += GS_THREADS) {
    const int s = e / n, i = e % n;
    T acc = T(0);
    const T* zr = Z + (size_t)s * n;
    for (int k = 0; k <= i; ++k) acc += L[i * LD + k] * zr[k];
    const T F = amp * acc;
    const T E = a.Y[i] - F;
    ll_part += (double)(T(-0.9189385332046727) - T(0.5) * t_log<T>(var) - T(0.5) * E * E / var);
    e2_part += (double)(E * E);
    ef_part += (double)(E * acc);                        // sum E * Fraw
    R[e] = E / var * inv_S;
  }
  const double ll = block_sum_all(ll_part, red);
  const double sumE2 = block_sum_all(e2_part, red);
  const double sumEFraw = block_sum_all(ef_part, red);
  __syncthreads();

  // ---- z-bar = amp * R L  (+ the KL's -z/S), L-bar = amp * tril(R^T Z) ----
  for (int e = tid; e < S * n; e += GS_THREADS) {
    const int s = e / n, k = e % n;
    T acc = T(0);
    const T* rr = R + (size_t)s * n;
    for (int i = k; i < n; ++i) acc += rr[i] * L[i * LD + k];
    Zb[e] = amp * acc - Z[e] * inv_S;
  }
  for (int e = tid; e < n * n; e += GS_THREADS) {
    const int i = e / n, k = e % n;
    T acc = T(0);
    if (k <= i) {
      for (int s = 0; s < S; ++s) acc += R[s * n + i] * Z[s * n + k];
      acc *= amp;
    }
    G[i * LD + k] = acc;
  }
  __syncthreads();

  // ---- sampler backward ----
  for (int k = tid; k < n; k += GS_THREADS) {
    T gm = T(0), go = T(0);
    for (int s = 0; s < S; ++s) {
      const T zt = Zb[s * n + k];
      gm += zt;
      if (!a.q_fullrank) go += zt * U[s * n + k];
    }
    g_mu[k] = gm;
    if (!a.q_fullrank) g_sq[k] = go * t_exp<T>(p_sq[k]) + T(1);
  }
  if (a.q_fullrank) {
    for (int e = tid; e < n * n; e += GS_THREADS) {
      const int i = e / n, k = e % n;
      T acc = T(0);
      if (k <= i) {
        for (int s = 0; s < S; ++s) acc += Zb[s * n + i] * U[s * n + k];
        if (k == i) acc += T(1) / p_sq[(size_t)i * n + i];
      }
      g_sq[(size_t)i * n + k] = acc;
    }
  }

  // ---- reverse-mode Cholesky, level-2, in place: G (L-bar) -> dELBO / dK over the stored lower triangle ----
  potrf_rev_cols_smem<T, GS_THREADS>(L, G, LD, n, colv);

  // ---- Gram backward: dELBO / d ell (K recomputed from X; the diagonal does not depend on ell) ----
  {
    double acc_e[4] = {0.0, 0.0, 0.0, 0.0};
    for (int d0 = 0; d0 < a.n_ell; d0 += 4) {
      for (int q = 0; q < 4; ++q) acc_e[q] = 0.0;
      for (int e = tid; e < n * n; e += GS_THREADS) {
        const int i = e / n, j = e % n;
        if (j >= i) continue;
        T r2 = T(0);
        for (int d = 0; d < D; ++d) {
          const T df = (a.X[i * D + d] - a.X[j * D + d]) / ell[a.n_ell == 1 ? 0 : d];
          r2 += df * df;
        }
        const T gk = G[i * LD + j] * t_exp<T>(T(-0.5) * r2);
        if (a.n_ell == 1) {
          acc_e[0] += (double)(gk * r2 / ell[0]);          // dK/d ell = K r2 / ell
        } else {
          for (int q = 0; q < 4 && d0 + q < a.n_ell; ++q) {
            const T df = (a.X[i * D + d0 + q] - a.X[j * D + d0 + q]) / ell[d0 + q];
            acc_e[q] += (double)(gk * df * df / ell[d0 + q]);
          }
        }
      }
      for (int q = 0; q < 4 && d0 + q < a.n_ell; ++q) {
        const double t = block_sum_all(acc_e[q], red);
        if (tid == 0) g_ell[d0 + q] = (T)t * t_sigmoid<T>(p_ell[d0 + q]);
      }
    }
  }

  // ---- scalar gradients and the ELBO ----
  if (tid == 0) {
    const double v = (double)var, am = (double)amp, sq = (double)s_q, kvd = (double)kv;
    const double invS = 1.0 / (double)S;
    const double ga = invS * sumEFraw / v;                         // dELBO / d amp = sum R * Fraw
    const double gv = invS * (-0.5 * (double)S * n / v + 0.5 * sumE2 / (v * v));
    *g_scale = (T)(ga * sqrt(kvd) * (double)t_sigmoid<T>(*p_scale));
    *g_kvar = (T)(ga * sq / (2.0 * sqrt(kvd)) * (double)t_sigmoid<T>(*p_kvar));
    *g_var = (T)(gv * (double)t_sigmoid<T>(*p_var));
    (void)am;
    a.out4[0] = (T)((ll - kl) * invS); a.out4[1] = (T)ll; a.out4[2] = (T)kl; a.out4[3] = T(0);
  }

  // ---- optional TF-1 Adam on -ELBO (model.py:206,220) ----
  if (a.m) {
    __threadfence_block();
    __syncthreads();
    const int t = a.step_dev ? *a.step_dev : a.step_host;
    const double lr_t = a.lr * sqrt(1.0 - pow(a.b2, (double)t)) / (1.0 - pow(a.b1, (double)t));
    const size_t npar = (size_t)n + nq + 3 + a.n_ell;
    for (size_t i = tid; i < npar; i += GS_THREADS) {
      if (a.q_fullrank && i >= (size_t)n && i < (size_t)n + nq) {
        const size_t q = i - n;
        if (q % n > q / n) continue;                     // strict upper triangle of q_sqrt: zero gradient upstream, never moves
      }
      const T g = (T)a.grad_scale * a.grads[i];
      const T mm = (T)a.b1 * a.m[i] + (T)(1.0 - a.b1) * g;
      const T vv = (T)a.b2 * a.v[i] + (T)(1.0 - a.b2) * g * g;
      a.m[i] = mm; a.v[i] = vv;
      a.params[i] -= (T)lr_t * mm / (t_sqrt<T>(vv) + (T)a.eps_adam);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// fp32: the same step on the BLOCKED shared-memory building blocks of the 128 x 128 leaf kernels (leaf_smem.cuh) instead of
// one-column-at-a-time loops -- 16-wide panels for the factorisation (3 barriers per panel instead of 2 per column) and the
// closed form  K-bar = sym(L^-T Phi(L^T L-bar) L^-1)  for its reverse mode (a blocked triangular inverse + three masked 128^3
// products, all level 3) in place of the level-2 reverse sweep.  Three 128 x 129 buffers (198 KB): B0 = K, then L;
// B1 = staged q_sqrt, then L^-1; B2 = scratch, L-bar, K-bar.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GS_THREADS, 1) gp_leaf_step_kernel(const SmallArgs<float> a) {
  using namespace leaf;
  extern __shared__ __align__(16) unsigned char gs_smem[];
  const int n = a.n, S = a.S, D = a.D, tid = threadIdx.x;
  float* B0 = reinterpret_cast<float*>(gs_smem);
  float* B1 = B0 + NB * LDS;
  float* B2 = B1 + NB * LDS;
  float* ell = B2 + NB * LDS;                            // [n_ell <= 32]
  __shared__ double red[GS_THREADS / 32];

  const size_t nq = a.q_fullrank ? (size_t)n * n : (size_t)n;
  float* p_mu = a.params; float* p_sq = a.params + n; float* p_scale = p_sq + nq; float* p_ell = p_scale + 1;
  float* p_kvar = p_ell + a.n_ell; float* p_var = p_kvar + 1;
  float* g_mu = a.grads; float* g_sq = a.grads + n; float* g_scale = g_sq + nq; float* g_ell = g_scale + 1;
  float* g_kvar = g_ell + a.n_ell; float* g_var = g_kvar + 1;
  // the S x n sample vectors live in shared memory when they fit (the notebook sizes do), else in the caller's workspace
  float* vec = (a.vec_smem) ? (ell + 32) : a.ws;
  float* Z = vec; float* U = Z + (size_t)S * n; float* R = U + (size_t)S * n; float* Zb = R + (size_t)S * n;
  float* Xs = B1;                                        // X / ell, [n][D]: B1 is free until q_sqrt is staged
  // instrumentation: cycles at the phase boundaries go to the 16 spare floats behind the caller's 4 S n workspace elements
  float* stamps = a.ws + (size_t)4 * S * n;
  const long long t_begin = clock64();
  int stamp_i = 0;
  auto stamp = [&]() { if (tid == 0 && stamp_i < 16) stamps[stamp_i] = (float)(clock64() - t_begin); ++stamp_i; };

  const float s_q = t_softplus<float>(*p_scale) + 1e-6f;
  const float kv = t_softplus<float>(*p_kvar) + 1e-6f;
  const float var = t_softplus<float>(*p_var) + 1e-6f;
  const float amp = sqrtf(kv) * s_q;
  for (int d = tid; d < a.n_ell; d += GS_THREADS) ell[d] = t_softplus<float>(p_ell[d]) + 1e-6f;
  __syncthreads();
  for (int e = tid; e < n * D; e += GS_THREADS) Xs[e] = a.X[e] / ell[a.n_ell == 1 ? 0 : e % D];
  __syncthreads();

  // ---- K = rbf(X) + jitter I, lower triangle, identity padded to 128 x 128 ----
  for (int e = tid; e < NB * NB; e += GS_THREADS) {
    const int i = e >> 7, j = e & (NB - 1);
    float val = (i == j) ? 1.f : 0.f;
    if (i < n && j <= i) {
      float r2 = 0.f;
      for (int d = 0; d < D; ++d) {
        const float df = Xs[i * D + d] - Xs[j * D + d];
        r2 = fmaf(df, df, r2);
      }
      val = expf(-0.5f * r2) + (i == j ? a.jitter : 0.f);
    } else if (i < n) {
      val = 0.f;
    }
    B0[i * LDS + j] = val;
  }
  stamp();   // 0: hyper-parameters + Gram
  potrf_smem(B0, n, a.err_flag, 0);                      // blocked, in place; flags 1 + row of a non-positive pivot
  stamp();   // 1: potrf

  // ---- sampler + one-sample KL ----
  double kl_part = 0.0;
  for (int e = tid; e < S * n; e += GS_THREADS)
    U[e] = a.eps ? a.eps[e] : philox_normal_at(a.seed, a.offset, (unsigned long long)e);
  if (a.q_fullrank)
    for (int e = tid; e < n * n; e += GS_THREADS) B1[(e / n) * LDS + (e % n)] = p_sq[e];
  __syncthreads();
  for (int e = tid; e < S * n; e += GS_THREADS) {
    const int s = e / n, i = e % n;
    float z, logdet;
    if (!a.q_fullrank) {
      z = p_mu[i] + expf(p_sq[i]) * U[e];
      logdet = 2.f * p_sq[i];
    } else {
      float acc = p_mu[i];
      const float* lq = B1 + i * LDS;
      const float* ur = U + (size_t)s * n;
      for (int k = 0; k <= i; ++k) acc = fmaf(lq[k], ur[k], acc);
      z = acc;
      logdet = logf(lq[i] * lq[i]);
    }
    Z[e] = z;
    const float u = U[e];
    kl_part += (double)(logdet + u * u - z * z);
  }
  const double kl = -0.5 * block_sum_all(kl_part, red);
  __syncthreads();

  // ---- F = amp * Z L^T, log-likelihood, residual ----
  double ll_part = 0.0, e2_part = 0.0, ef_part = 0.0;
  const float inv_S = 1.f / (float)S;
  for (int e = tid; e < S * n; e += GS_THREADS) {
    const int s = e / n, i = e % n;
    float acc = 0.f;
    const float* zr = Z + (size_t)s * n;
    for (int k = 0; k <= i; ++k) acc = fmaf(B0[i * LDS + k], zr[k], acc);
    const float F = amp * acc;
    const float E = a.Y[i] - F;
    ll_part += (double)(-0.9189385332046727f - 0.5f * logf(var) - 0.5f * E * E / var);
    e2_part += (double)(E * E);
    ef_part += (double)(E * acc);
    R[e] = E / var * inv_S;
  }
  const double ll = block_sum_all(ll_part, red);
  const double sumE2 = block_sum_all(e2_part, red);
  const double sumEFraw = block_sum_all(ef_part, red);
  __syncthreads();

  // ---- z-bar = amp * R L - Z / S ----
  for (int e = tid; e < S * n; e += GS_THREADS) {
    const int s = e / n, k = e % n;
    float acc = 0.f;
    const float* rr = R + (size_t)s * n;
    for (int i = k; i < n; ++i) acc = fmaf(rr[i], B0[i * LDS + k], acc);
    Zb[e] = amp * acc - Z[e] * inv_S;
  }
  __syncthreads();

  // ---- sampler backward ----
  for (int k = tid; k < n; k += GS_THREADS) {
    float gm = 0.f, go = 0.f;
    for (int s = 0; s < S; ++s) {
      const float zt = Zb[s * n + k];
      gm += zt;
      if (!a.q_fullrank) go = fmaf(zt, U[s * n + k], go);
    }
    g_mu[k] = gm;
    if (!a.q_fullrank) g_sq[k] = go * expf(p_sq[k]) + 1.f;
  }
  if (a.q_fullrank) {
    for (int e = tid; e < n * n; e += GS_THREADS) {
      const int i = e / n, k = e % n;
      float acc = 0.f;
      if (k <= i) {
        for (int s = 0; s < S; ++s) acc = fmaf(Zb[s * n + i], U[s * n + k], acc);
        if (k == i) acc += 1.f / B1[i * LDS + i];
      }
      g_sq[(size_t)i * n + k] = acc;
    }
  }
  __syncthreads();

  stamp();   // 2: sampler, projection, log-likelihood, z-bar, sampler backward
  // ---- reverse-mode Cholesky, closed form on the blocked building blocks ----
  trinv_smem(B0, B1, B2);                                // B1 = L^-1 (identity padded), B2 scratch
  stamp();   // 3: triangular inverse
  for (int e = tid; e < NB * NB; e += GS_THREADS) {      // B2 = L-bar = amp * tril(R^T Z), zero padded
    const int i = e >> 7, k = e & (NB - 1);
    float acc = 0.f;
    if (i < n && k <= i) {
      for (int s = 0; s < S; ++s) acc = fmaf(R[s * n + i], Z[s * n + k], acc);
      acc *= amp;
    }
    B2[i * LDS + k] = acc;
  }
  __syncthreads();
  stamp();   // 4: L-bar
  mm_smem<true, false, 1>(B2, B0, B2);                   // P = L^T L-bar
  __syncthreads();
  for (int e = tid; e < NB * NB; e += GS_THREADS) {      // Phi: lower triangle, halved diagonal
    const int i = e >> 7, j = e & (NB - 1);
    float v = B2[i * LDS + j];
    if (j > i) v = 0.f;
    else if (j == i) v *= 0.5f;
    B2[i * LDS + j] = v;
  }
  __syncthreads();
  mm_smem<false, false, 2>(B0, B2, B1);                  // M1 = P L^-1        (L is dead: B0 receives M1)
  __syncthreads();
  mm_smem<true, false, 1>(B2, B1, B0);                   // S = L^-T M1;  dELBO/dK (symmetric) = (S + S^T) / 2
  __syncthreads();

  stamp();   // 5: three masked 128^3 products
  // ---- Gram backward: the stored lower entry (i, j) stands for both (i, j) and (j, i): weight S_ij + S_ji ----
  {
    float* Xr = B0;                                      // X / ell again (M1 is dead)
    for (int e = tid; e < n * D; e += GS_THREADS) Xr[e] = a.X[e] / ell[a.n_ell == 1 ? 0 : e % D];
    __syncthreads();
    double acc_e[4] = {0.0, 0.0, 0.0, 0.0};
    for (int d0 = 0; d0 < a.n_ell; d0 += 4) {
      for (int q = 0; q < 4; ++q) acc_e[q] = 0.0;
      float part[4] = {0.f, 0.f, 0.f, 0.f};              // a thread sums ~20 entries in fp32, the block reduction runs in fp64
      for (int e = tid; e < n * n; e += GS_THREADS) {
        const int i = e / n, j = e % n;
        if (j >= i) continue;
        float r2 = 0.f;
        for (int d = 0; d < D; ++d) {
          const float df = Xr[i * D + d] - Xr[j * D + d];
          r2 = fmaf(df, df, r2);
        }
        const float gk = (B2[i * LDS + j] + B2[j * LDS + i]) * expf(-0.5f * r2);
        if (a.n_ell == 1) {
          part[0] = fmaf(gk, r2, part[0]);
        } else {
          for (int q = 0; q < 4 && d0 + q < a.n_ell; ++q) {
            const float df = Xr[i * D + d0 + q] - Xr[j * D + d0 + q];
            part[q] = fmaf(gk * df, df, part[q]);
          }
        }
      }
      for (int q = 0; q < 4; ++q) acc_e[q] = (double)part[q] / (double)ell[a.n_ell == 1 ? 0 : min(d0 + q, a.n_ell - 1)];
      for (int q = 0; q < 4 && d0 + q < a.n_ell; ++q) {
        const double t = block_sum_all(acc_e[q], red);
        if (tid == 0) g_ell[d0 + q] = (float)t * t_sigmoid<float>(p_ell[d0 + q]);
      }
    }
  }

  if (tid == 0) {
    const double v = (double)var, sq = (double)s_q, kvd = (double)kv;
    const double invS = 1.0 / (double)S;
    const double ga = invS * sumEFraw / v;
    const double gv = invS * (-0.5 * (double)S * n / v + 0.5 * sumE2 / (v * v));
    *g_scale = (float)(ga * sqrt(kvd) * (double)t_sigmoid<float>(*p_scale));
    *g_kvar = (float)(ga * sq / (2.0 * sqrt(kvd)) * (double)t_sigmoid<float>(*p_kvar));
    *g_var = (float)(gv * (double)t_sigmoid<float>(*p_var));
    a.out4[0] = (float)((ll - kl) * invS); a.out4[1] = (float)ll; a.out4[2] = (float)kl; a.out4[3] = 0.f;
  }

  stamp();   // 6: Gram backward + scalar gradients
  if (a.m) {                                             // optional TF-1 Adam on -ELBO (model.py:206,220)
    __threadfence_block();
    __syncthreads();
    const int t = a.step_dev ? *a.step_dev : a.step_host;
    const double lr_t = a.lr * sqrt(1.0 - pow(a.b2, (double)t)) / (1.0 - pow(a.b1, (double)t));
    const size_t npar = (size_t)n + nq + 3 + a.n_ell;
    for (size_t i = tid; i < npar; i += GS_THREADS) {
      if (a.q_fullrank && i >= (size_t)n && i < (size_t)n + nq) {
        const size_t q = i - n;
        if (q % n > q / n) continue;
      }
      const float g = (float)a.grad_scale * a.grads[i];
      const float mm = (float)a.b1 * a.m[i] + (float)(1.0 - a.b1) * g;
      const float vv = (float)a.b2 * a.v[i] + (float)(1.0 - a.b2) * g * g;
      a.m[i] = mm; a.v[i] = vv;
      a.params[i] -= (float)lr_t * mm / (sqrtf(vv) + (float)a.eps_adam);
    }
  }
}

static int launch_leaf_step(SmallArgs<float> a, cudaStream_t st) {
  if (a.n <= 0 || a.n > leaf::NB || a.D <= 0 || a.D > 32 || a.S <= 0 || (a.n_ell != 1 && a.n_ell != a.D)) return HB_ERR_ARG;
  if (!a.X || !a.Y || !a.params || !a.grads || !a.out4 || !a.ws) return HB_ERR_ARG;
  if (!a.eps && (a.offset & 3ull)) return HB_ERR_ARG;
  const size_t base = (size_t)(3 * leaf::NB * leaf::LDS + 32) * sizeof(float) + 64;
  const size_t vecs = (size_t)4 * a.S * a.n * sizeof(float);
  constexpr size_t kBudget = 216 * 1024;                 // + 8.3 KB of static shared memory (panel staging, reductions) <= 227 KB
  a.vec_smem = (base + vecs <= kBudget) ? 1 : 0;
  const size_t smem = base + (a.vec_smem ? vecs : 0);
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(gp_leaf_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBudget) != cudaSuccess) return HB_ERR_CUDA;
    attr_set = true;
  }
  gp_leaf_step_kernel<<<1, GS_THREADS, smem, st>>>(a);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

template <typename T>
size_t small_smem_bytes(int n) {
  const size_t LD = (size_t)(n | 1);
  return (2 * (size_t)n * LD + 32 + (size_t)n + 8) * sizeof(T) + 64;
}

template <typename T>
int launch_small(const SmallArgs<T>& a, cudaStream_t st) {
  if (a.n <= 0 || a.n > SmallLimits<T>::max_n || a.D <= 0 || a.D > 32 || a.S <= 0 || (a.n_ell != 1 && a.n_ell != a.D))
    return HB_ERR_ARG;
  if (!a.X || !a.Y || !a.params || !a.grads || !a.out4 || !a.ws) return HB_ERR_ARG;
  if (!a.eps && (a.offset & 3ull)) return HB_ERR_ARG;
  const size_t smem = small_smem_bytes<T>(a.n);
  static size_t attr_set = 0;
  if (smem > attr_set) {
    // 227 KB per CTA minus this kernel's static shared memory (reduction scratch)
    if (cudaFuncSetAttribute(gp_small_step_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(226 * 1024)) != cudaSuccess)
      return HB_ERR_CUDA;
    attr_set = 226 * 1024;
  }
  gp_small_step_kernel<T><<<1, GS_THREADS, smem, st>>>(a);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

}  // namespace

int gp_small_max_n(int f64) { return f64 ? SmallLimits<double>::max_n : SmallLimits<float>::max_n; }
size_t gp_small_workspace_elems(int n, int S) { return 4 * (size_t)S * n + 16; }

int gp_small_step_f32(int n, int D, int S, int n_ell, int q_fullrank, float jitter, unsigned long long seed, unsigned long long offset,
                      const float* X, const float* Y, float* params, const float* eps, float* grads, float* out4, float* ws,
                      int* err_flag, float* m, float* v, const int* step_dev, int step_host, double lr, double b1, double b2,
                      double eps_adam, double grad_scale, cudaStream_t st) {
  SmallArgs<float> a{n, D, S, n_ell, q_fullrank, jitter, seed, offset, X, Y, params, eps, grads, out4, ws, err_flag,
                     m, v, step_dev, step_host, lr, b1, b2, eps_adam, grad_scale};
  return launch_leaf_step(a, st);      // blocked building blocks; the column-at-a-time template stays the fp64 route
}

int gp_small_step_f64(int n, int D, int S, int n_ell, int q_fullrank, double jitter, unsigned long long seed, unsigned long long offset,
                      const double* X, const double* Y, double* params, const double* eps, double* grads, double* out4, double* ws,
                      int* err_flag, double* m, double* v, const int* step_dev, int step_host, double lr, double b1, double b2,
                      double eps_adam, double grad_scale, cudaStream_t st) {
  SmallArgs<double> a{n, D, S, n_ell, q_fullrank, jitter, seed, offset, X, Y, params, eps, grads, out4, ws, err_flag,
                      m, v, step_dev, step_host, lr, b1, b2, eps_adam, grad_scale};
  return launch_small<double>(a, st);
}

}  // namespace hb
