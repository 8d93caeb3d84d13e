// Internal C++ declarations of every kernel launcher in the library (the C ABI in capi.cu wraps these).
#pragma once
#include "common.cuh"

namespace hb {

constexpr int kReduceBlocks = 1024;                       // max partial-sum blocks of a reducing kernel
constexpr size_t kReduceWsBytes = kReduceBlocks * 40 * sizeof(double);  // up to 40 values per block

// ---- utilities (elementwise.cu) ----
int copy2d(float* dst, long long ldd, const float* src, long long lds, int rows, int cols, float scale, cudaStream_t st);
int scale2d(float* a, long long lda, int rows, int cols, float s, cudaStream_t st);
int transpose2d(float* dst, long long ldd, const float* src, long long lds, int rows, int cols, float scale, cudaStream_t st);
int zero_strict_upper(float* a, long long lda, int n, cudaStream_t st);
int fill_f32(float* a, long long n, float v, cudaStream_t st);
int randn_philox(float* out, long long count, unsigned long long seed, unsigned long long offset, cudaStream_t st);
int random_index(long long* out, long long n_index, const long long* pool, long long pool_size, unsigned long long seed,
                 unsigned long long offset, cudaStream_t st);
int philox_raw(uint32_t* out, long long n_blocks, const uint32_t* ctr4_host, const uint32_t* key2_host, cudaStream_t st);

// ---- persistent single-CTA variational-GP step for notebook-sized models (gp_small.cu) ----
int gp_small_max_n(int f64);
size_t gp_small_workspace_elems(int n, int S);
int gp_small_step_f32(int n, int D, int S, int n_ell, int q_fullrank, float jitter, unsigned long long seed, unsigned long long offset,
                      const float* X, const float* Y, float* params, const float* eps, float* grads, float* out4, float* ws,
                      int* err_flag, float* m, float* v, const int* step_dev, int step_host, double lr, double b1, double b2,
                      double eps_adam, double grad_scale, cudaStream_t st);
int gp_small_step_f64(int n, int D, int S, int n_ell, int q_fullrank, double jitter, unsigned long long seed, unsigned long long offset,
                      const double* X, const double* Y, double* params, const double* eps, double* grads, double* out4, double* ws,
                      int* err_flag, double* m, double* v, const int* step_dev, int step_host, double lr, double b1, double b2,
                      double eps_adam, double grad_scale, cudaStream_t st);

// ---- Variational sampler + one-sample KL (sampler.cu) ----
int sample_diag_fwd(const float* mu, long long ld_mu, const float* omega, long long ld_om, int rows, int cols,
                    const float* eps, unsigned long long seed, unsigned long long offset, int S, float* z,
                    float* kl_out, void* ws, size_t ws_bytes, cudaStream_t st);
int sample_diag_bwd(const float* mu, long long ld_mu, const float* omega, long long ld_om, int rows, int cols,
                    const float* eps, unsigned long long seed, unsigned long long offset, int S, const float* zbar,
                    const float* zbar_scale, float kl_coef, const float* kl_coef_dev, float* gmu, long long ld_gmu, float* gom,
                    long long ld_gom, float beta,
                    cudaStream_t st);
int tril_logdet_kl(const float* Lq, long long ld, long long stride, int n, int batch, const float* eps,
                   const float* z, long long count, int S, float* kl_out, void* ws, size_t ws_bytes, cudaStream_t st);
int tril_diag_grad(float* gL, long long ld, long long stride, const float* Lq, long long ldl, long long strideL,
                   int n, int batch, float coef, cudaStream_t st);
int add_rowvec(float* z, long long ldz, const float* mu, int rows, int cols, cudaStream_t st);
int colsum(const float* a, long long lda, int rows, int cols, float alpha, float beta, float* out, cudaStream_t st);
int axpby(float* y, const float* x, long long n, float a, float b, cudaStream_t st);

// ---- densities.gaussian (density.cu) ----
int gauss_loglik_fwd(const float* f, const float* f_scale, const float* y, long long total, long long y_period,
                     const float* var, float rcoef, float* resid, float* out3, void* ws, size_t ws_bytes, cudaStream_t st);
int gauss_loglik_fwd_ex(const float* f, const float* f_scale, const float* y, long long total, long long y_period,
                        long long y_div, const float* var, float rcoef, float* resid, float* out3, void* ws, size_t ws_bytes,
                        cudaStream_t st);
int gaussian_logpdf(const float* x, long long x_period, const float* mu, long long mu_period, const float* var,
                    long long var_period, long long total, float* out, cudaStream_t st);

int gaussian_logpdf_bwd(const float* x, long long x_period, const float* mu, long long mu_period, const float* var,
                        long long var_period, long long total, const float* g, float* dmu, float* dvar,
                        cudaStream_t st);
// ---- the whole densities.py family (density_family.cu) ----
int density_nargs_host(int kind);
int density_logpdf(int kind, const float* const* args, const long long* periods, long long total, float* out,
                   cudaStream_t st);
int density_logpdf_bwd(int kind, const float* const* args, const long long* periods, long long total, const float* g,
                       long long g_period, float* const* dargs, void* ws, size_t ws_bytes, cudaStream_t st);
// ---- transforms.py as kernels (transforms.cu) ----
int transform_fwd(int kind, const float* x, long long total, float p0, float p1, float* y, cudaStream_t st);
int transform_bwd(int kind, const float* x, long long total, float p0, float p1, const float* gy, float* gx, cudaStream_t st);
int transform_logjac(int kind, const float* x, long long total, float p0, float p1, float* out1, void* ws, size_t ws_bytes,
                     cudaStream_t st);
int transform_logjac_bwd(int kind, const float* x, long long total, float p0, float p1, const float* g1, float* gx,
                         cudaStream_t st);
int gather_rows(float* dst, const float* src, const long long* index, long long n_index, long long row_elems,
                cudaStream_t st);
int gather_rows_f64(double* dst, const double* src, const long long* index, long long n_index, long long row_elems,
                    cudaStream_t st);

// ---- UnitRBF Gram (gram.cu) ----
int rbf_gram_fwd(const float* X, const float* X2, int n, int n2, int D, long long sX, long long sX2,
                 const float* ell, int n_ell, float* K, long long ldk, long long sK, int batch, float jitter,
                 int lower_only, int csym, cudaStream_t st);
int rbf_gram_bwd(const float* G, long long ldg, long long sG, const float* X, const float* X2, int n, int n2,
                 int D, long long sX, long long sX2, const float* ell, int n_ell, int batch, int sym_lower,
                 int csym, const float* out_scale, float* g_ell, void* ws, size_t ws_bytes, cudaStream_t st);

int rbf_gram_bwd_x2(const float* G, long long ldg, long long sG, const float* X, const float* X2, int n, int n2, int D,
                    long long sX, long long sX2, const float* ell, int n_ell, int batch, int sym_lower, float scale,
                    float* dX2, cudaStream_t st);

// ---- NN helpers (nn.cu) ----
size_t act_bwd_colsum_workspace_bytes(int rows, int cols);
int act_bwd_colsum_ws(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act, int clip,
                      float clip_lo, float clip_hi, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st);
int act_bwd_colsum(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act, int clip,
                   float clip_lo, float clip_hi, float* dbias, cudaStream_t st);

// ---- Adam, TF-1 flavour (adam.cu) ----
int adam_tf1(float* theta, const float* grad, float* m, float* v, long long n, float grad_scale, float lr, float b1,
             float b2, float eps, const int* step_dev, int step_host, cudaStream_t st);
int increment_i32(int* p, cudaStream_t st);

// ---- linalg.cu ----
size_t potrf_workspace_bytes(int n);
size_t trsm_workspace_bytes(int m, int n);
int potrf_lower(float* A, long long lda, long long strideA, int n, int batch, int zero_upper, void* ws,
                size_t ws_bytes, int* err_flag, cudaStream_t st);
int potrf_lower_bwd(const float* L, long long ldl, long long strideL, float* G, long long ldg, long long strideG,
                    int n, int batch, void* ws, size_t ws_bytes, cudaStream_t st, int l_shadow_valid = 0);
int trsm_right_lower(const float* L, long long ldl, float* X, long long ldx, int m, int n, int trans, void* ws,
                     size_t ws_bytes, cudaStream_t st);
int flat_trace_begin();
int flat_trace_end(double* out3, int capacity);
// right-looking schedule over column blocks, one GPU or a column-block-cyclic group (comm.cuh: DistEnv)
struct DistEnv;
size_t potrf_dist_workspace_bytes(int n, const DistEnv& d);
int potrf_lower_dist(float* A, long long lda, int n, const DistEnv& d, void* ws, size_t ws_bytes, int* err_flag,
                     cudaStream_t st);
int potrf_lower_bwd_dist(const float* L, long long ldl, float* G, long long ldg, int n, const DistEnv& d, void* ws,
                         size_t ws_bytes, cudaStream_t st, int l_shadow_valid = 0);

}  // namespace hb
