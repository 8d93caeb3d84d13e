// Internal declarations of the fp64 building blocks of f64.cu that other whole-step entry points chain (moe64.cu): the
// GEMM and column-recursion context, the blocked Cholesky and its reverse mode, and the per-GP kernels of the ELBO step.
#pragma once
#include "common.cuh"

namespace hb {

constexpr size_t kSplitWsBytes = (size_t)8 << 20;       // 32 partial 128 x 128 tiles, 64 partial 64 x 64 ones
// sc (per GP): [0] scale s, [1] k_var, [2] var, [3] amp, [4] loglik, [5] sum E^2, [6] sum E Fraw, [7] kl, [8..) ell
constexpr int SC_ELL = 8;
constexpr int kGramBwdBlocks = 296;
constexpr int RED_THREADS = 1024;

inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }

// one stream of the column recursion: its error flag and its own split-K partial tiles
struct Ctx64 {
  cudaStream_t st;
  int* err;
  void* ws;                // split-K partial tiles
  size_t ws_bytes;
};

int ensure_attrs64();
int gemm64(const Ctx64& c, const double* A, long long lda, int transA, int a_tri, const double* B, long long ldb, int transB,
           int b_tri, double* C, long long ldc, int c_tri, int M, int N, int K, double alpha, double beta);
// C = act(op(A) op(B) + beta C + bias) without triangular masks (bias [N] or nullptr, act ACT_* of gemm.cuh).  split_tall:
// split a long K over CTAs even when the output has many tiles (tall reductions), in a fixed split order.  The bytes of
// partial tiles it may use: gemm64_split_bytes.
int gemm64_ex(const Ctx64& c, const double* A, long long lda, int transA, const double* B, long long ldb, int transB, double* C,
              long long ldc, int M, int N, int K, double beta, const double* bias, int act, int split_tall);
size_t gemm64_split_bytes(int M, int N, int K, int split_tall);
int potrf_cols64(const Ctx64& c, double* A, long long lda, int c0, int w, int n);
int chol_rev_cols64(const Ctx64& c, const double* L, long long ldl, double* G, long long ldg, int c0, int w, int n);

__global__ void gp64_gram_kernel(const double* X, int n, int D, const double* sc, int n_ell, double jitter, double* K);
__global__ void gp64_sample_kernel(const double* p_mu, const double* p_sq, int full, int n, int S, const double* eps,
                                   unsigned long long seed, unsigned long long offset, double* U, double* Z);
__global__ void __launch_bounds__(RED_THREADS) gp64_kl_kernel(const double* p_sq, int full, int n, int S, const double* U,
                                                            const double* Z, double* sc);
__global__ void gp64_zbar_kernel(const double* W, const double* Z, const double* sc, long long total, int S, double* Zb);
__global__ void gp64_sampler_bwd_kernel(const double* Zb, const double* U, const double* p_sq, int full, int n, int S, double* g_mu,
                                        double* g_sq);
__global__ void __launch_bounds__(256) gp64_gram_bwd_kernel(const double* G, const double* X, int n, int D, const double* sc, int n_ell,
                                                          double* red);
__global__ void gp64_adam_kernel(double* params, const double* grads, double* m, double* v, long long npar, int n, int full,
                                 const int* step_dev, int step_host, double lr, double b1, double b2, double eps, double grad_scale);

}  // namespace hb
