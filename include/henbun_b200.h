/* henbun_b200 -- C ABI of the B200-native Monte-Carlo ELBO hot path of Henbun.
 *
 * The reference (fujii-team/Henbun) has NO native/FFI boundary: ext_modules=[] (setup.py:28) and the
 * only vestige is a commented-out tf.load_op_library block (Henbun/tf_wraps.py:50-71).  Every entry
 * point below therefore replaces a group of TensorFlow ops that the reference's Python emits on the
 * hot path; the reference call site each one stands for is cited per function.
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless the name ends in _host.  Tensors are contiguous
 *    row-major fp32 unless a leading dimension / stride argument says otherwise.
 *  - The caller owns every buffer including workspaces; the library keeps no device state.
 *  - `stream` is a cudaStream_t passed as void*.  Calls are asynchronous and stream-ordered; no call
 *    synchronises the host.  All calls are CUDA-graph capturable.
 *  - Return value: 0 = launched, HB_ERR_ARG = bad argument (reference: ValueError/AssertionError,
 *    e.g. Henbun/param.py:712-713, variationals.py:82), HB_ERR_CUDA = launch failure,
 *    HB_ERR_WORKSPACE = workspace missing/too small.
 *  - Numerical failure is reported asynchronously: a non-positive Cholesky pivot writes
 *    (1 + global row index) into *err_flag (reference: InvalidArgumentError from tf.cholesky).
 *  - Triangular matrices use full-square storage; only the lower triangle is read or written.
 */
#ifndef HENBUN_B200_H
#define HENBUN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HB_OK 0
#define HB_ERR_ARG 1
#define HB_ERR_CUDA 2
#define HB_ERR_WORKSPACE 3

#define HB_ACT_NONE 0
#define HB_ACT_SIGMOID 1
#define HB_ACT_RELU 2
#define HB_ACT_TANH 3

/* Behavioural switches travel WITH THE CALL (the library keeps no mutable configuration: two models with different accuracy
 * settings can run side by side in one process).  Every entry point that reaches the level-3 engine takes a
 * `const hb_options*` -- a trailing argument of the building blocks, the last field of the whole-step config structs --
 * and NULL means hb_options_init()'s defaults.
 *   gemm_engine      0 auto | 1 fp32 SIMT kernels only | 2 force tcgen05 (HB_ERR_ARG if the shape does not qualify) | 3 k-looped SIMT only
 *   exact_below      factorisations (potrf / potrf_bwd / trsm) of order <= this run their products on the exact-fp32 SIMT
 *                    kernels (default 2048: latency-bound sizes, where the notebook models live and where the split product's
 *                    error shows on ill-conditioned inputs); 0 disables
 *   panel_refinement panel solves multiply by explicit inverses of the 128 x 128 diagonal blocks; 0 inverse only, 1 one step of
 *                    iterative refinement against the triangular block (LAPACK-grade on ill-conditioned matrices, two more
 *                    short-K products per panel), 2 (default) refined for n <= 8192, 3 substitution kernel (no inverse)
 *   presplit_engine  1 (default): factorisations of order >= 4096 (n % 8 == 0) keep fp16 hi/lo shadows of every finished panel
 *                    of L and K-bar in their workspace and run their big products on csrc/gemm_h2.cu; 0: round-1 behaviour
 *   small_gp_kernel  1 (default): hb_gp_elbo_step runs n <= 128 as ONE persistent CTA (csrc/gp_small.cu: 168 us per step at
 *                    N = 100 against 239 us for the 23-kernel path); 0: the multi-kernel path
 *   tc_option        bit 2: no CTA pairs in the in-kernel-split engine, bit 3: three TF32 passes instead of TF32 + bf16 terms
 *   lookahead        1 (default): leaf kernels of potrf / potrf_bwd run on a high-priority side stream
 *   schedule         order of the blocked factorisation and of its reverse mode.  0 (default): from n = 32768 on the
 *                    right-looking two-stream schedule over n/16-column blocks (the narrow steps of a block on a high-priority
 *                    stream next to the trailing updates of the previous one; see hb_potrf_lower_dist), below that the plain
 *                    column recursion; 1: column recursion always; >= 128: right-looking with blocks of that many columns
 *                    (orders below 8192 always take the column recursion: their workspace carries no scratch for the second
 *                    stream; hb_potrf_lower_dist / hb_gp_elbo_step_dist with world = 1 run the schedule at any order) */
typedef struct hb_options {
  int gemm_engine, exact_below, panel_refinement, presplit_engine, small_gp_kernel, tc_option, lookahead, schedule;
} hb_options;
void hb_options_init(hb_options* opt);

/* library / bookkeeping */
int hb_version(void);
unsigned long long hb_launch_count(void);           /* kernels launched by this library so far */
size_t hb_reduce_workspace_bytes(void);             /* workspace every reducing call needs */
/* Optional instrumentation for bench.py: CUDA-event pairs around every GEMM launch on its stream.
 * hb_profile_end synchronises and fills a HOST array {launches, total ms, useful FLOP, 0}. */
int hb_profile_begin(int max_gemm_launches);
int hb_profile_end(double* out4_host);
/* per-launch dump of the last profiled region (M,N,K,engine,useful FLOP,ms); call before the next hb_profile_begin */
int hb_profile_dump_csv(const char* path_host);
/* As hb_profile_end, plus the shares of the two CTA-pair tcgen05 kernels: out8 = {launches, ms, useful FLOP,
 * in-kernel-split pair kernel launches, ms, useful FLOP, pre-split (fp16 hi/lo) pair kernel ms, useful FLOP}. */
int hb_profile_end_ex(double* out8_host);
/* Phase timing of one hb_gp_elbo_step: hb_phase_begin(); step; n = hb_phase_end(ms, cap) fills ms[0..n) with
 * {scalars + Gram fwd, potrf, sampler + F + log-lik + W, sampler bwd + Lbar, potrf_bwd, Gram bwd + scalar grads}. */
int hb_phase_begin(void);
int hb_phase_end(double* out_ms_host, int capacity);

/* tf.random_normal (variationals.py:107,127): Philox-4x32-10 + Box-Muller, counter based.
 * Element i of the stream (seed, offset) is identical whether it is materialised here or
 * regenerated inside hb_sample_diag_{fwd,bwd}.  offset must be a multiple of 4. */
int hb_randn_philox(float* out, long long count, unsigned long long seed, unsigned long long offset, void* stream);
/* The raw generator underneath (known-answer tests against the Random123 vectors): out[4b .. 4b+3] =
 * Philox-4x32-10(counter = ctr4 + b on its low 64 bits, key = key2).  ctr4_host / key2_host are HOST arrays of 4 / 2
 * words.  The library's own streams use counter = (offset/4 + block, 0, 0), key = seed. */
int hb_philox4x32_10(unsigned int* out, long long n_blocks, const unsigned int* ctr4_host, const unsigned int* key2_host,
                     void* stream);

/* Variational._sample 'diagonal' (variationals.py:138-142) fused with Normal._KL (:225-230) and
 * logdet (:183-184).  mu/omega: [rows, cols] with row strides (LOCAL variationals read the two halves
 * of an encoder row, param.py:529-537).  eps: [S, rows, cols] or NULL (Philox).  z: [S, rows, cols].
 * kl_out (1 float, may be NULL) = -0.5*sum(2*omega + eps^2 - z^2) over all S samples. */
int hb_sample_diag_fwd(const float* mu, long long ld_mu, const float* omega, long long ld_omega, int rows, int cols,
                       const float* eps, unsigned long long seed, unsigned long long offset, int S, float* z,
                       float* kl_out, void* ws, size_t ws_bytes, void* stream);
/* Backward of the above for an objective  obj = g(z) - c*KL, c = kl_coef * (*kl_coef_dev if non-NULL):
 * zbar = dg/dz [S,rows,cols] (NULL = 0), optionally multiplied by the device scalar *zbar_scale.
 * g* = beta*g* + grad. */
int hb_sample_diag_bwd(const float* mu, long long ld_mu, const float* omega, long long ld_omega, int rows, int cols,
                       const float* eps, unsigned long long seed, unsigned long long offset, int S,
                       const float* zbar, const float* zbar_scale, float kl_coef, const float* kl_coef_dev, float* gmu,
                       long long ld_gmu,
                       float* gomega, long long ld_gomega, float beta, void* stream);

/* Variational._sample 'fullrank' (variationals.py:144-146): z[b,s,:] = mu[b,:] + tril(Lq[b]) eps[b,s,:].
 * Lq: [batch, n, n]; mu: [batch, n]; eps, z: [batch, S, n].  kl_out as above with
 * logdet = log(diag(Lq)^2) (:185-186). */
int hb_sample_tril_fwd(const float* mu, const float* Lq, int n, int batch, const float* eps, int S, float* z,
                       float* kl_out, void* ws, size_t ws_bytes, void* stream);
/* gmu [batch,n], gLq [batch,n,n] (lower triangle written, strict upper zeroed). zbar may be NULL. */
int hb_sample_tril_bwd(const float* Lq, int n, int batch, const float* eps, const float* z, int S,
                       const float* zbar, float kl_coef, float* gmu, float* gLq, float* scratch_Sn, void* stream);

/* densities.gaussian (densities.py:25-27) elementwise with modular broadcasting:
 * out[i] = logN(x[i % x_period]; mu[i % mu_period], var[i % var_period]). */
int hb_gaussian_logpdf(const float* x, long long x_period, const float* mu, long long mu_period, const float* var,
                       long long var_period, long long total, float* out, void* stream);
/* Backward of hb_gaussian_logpdf: dmu[i] = g[i]*dlogN/dmu, dvar[i] = g[i]*dlogN/dvar (full size; the
 * caller reduces over broadcast axes; dlogN/dx = -dlogN/dmu).  dmu / dvar may be NULL. */
int hb_gaussian_logpdf_bwd(const float* x, long long x_period, const float* mu, long long mu_period, const float* var,
                           long long var_period, long long total, const float* g, float* dmu, float* dvar,
                           void* stream);
/* Constrained-parameter transforms (Henbun/transforms.py) on device tensors: y = T(x), the log-Jacobian sum that the
 * generic Variational._KL subtracts (variationals.py:204-208), and their backward passes.
 *   HB_TRANSFORM_EXP 1      (transforms.py:90-107)   y = exp(x) + p0
 *   HB_TRANSFORM_LOG1PE 2   (transforms.py:110-143)  y = log(1 + exp(x)) + p0        (transforms.positive, p0 = 1e-6)
 *   HB_TRANSFORM_LOGISTIC 3 (transforms.py:146-180)  y = p0 + (p1 - p0) / (1 + exp(-x))
 * bwd: gx = gy * T'(x).  logjac: *out1 = sum_e log|T'(x_e)| (deterministic; ws of hb_reduce_workspace_bytes()).
 * logjac_bwd: gx = *g1 * d logjac / dx (g1 a device scalar). */
#define HB_TRANSFORM_EXP 1
#define HB_TRANSFORM_LOG1PE 2
#define HB_TRANSFORM_LOGISTIC 3
int hb_transform_fwd(int kind, const float* x, long long total, float p0, float p1, float* y, void* stream);
int hb_transform_bwd(int kind, const float* x, long long total, float p0, float p1, const float* gy, float* gx, void* stream);
int hb_transform_logjac(int kind, const float* x, long long total, float p0, float p1, float* out1, void* ws, size_t ws_bytes,
                        void* stream);
int hb_transform_logjac_bwd(int kind, const float* x, long long total, float p0, float p1, const float* g1, float* gx,
                            void* stream);
/* The log-densities of Henbun/densities.py as one elementwise family (csrc/density_family.cu).
 * kind (operands in the reference function's argument order, file:line in densities.py):
 *   HB_DENSITY_GAUSSIAN 0 (x, mu, var) :25-27      HB_DENSITY_GAMMA 5 (shape, scale, x) :49-51
 *   HB_DENSITY_LOGNORMAL 1 (x, mu, var) :30-32     HB_DENSITY_STUDENT_T 6 (x, mean, scale, deg_free) :54-61
 *   HB_DENSITY_BERNOULLI 2 (p, y) :35-36           HB_DENSITY_BETA 7 (alpha, beta, y) :64-70
 *   HB_DENSITY_POISSON 3 (lamb, y) :39-40          HB_DENSITY_LAPLACE 8 (mu, sigma, y) :73-74
 *   HB_DENSITY_EXPONENTIAL 4 (lamb, y) :43-44      HB_DENSITY_BIMIXTURE 9 (fraction, logp0, logp1) :95-103
 * args / periods: HOST arrays of hb_density_nargs(kind) device pointers and their modular periods
 * (operand i is read at flat index e % periods[i]; 1 = scalar, total = full tensor).  out[e], e < total. */
#define HB_DENSITY_GAUSSIAN 0
#define HB_DENSITY_LOGNORMAL 1
#define HB_DENSITY_BERNOULLI 2
#define HB_DENSITY_POISSON 3
#define HB_DENSITY_EXPONENTIAL 4
#define HB_DENSITY_GAMMA 5
#define HB_DENSITY_STUDENT_T 6
#define HB_DENSITY_BETA 7
#define HB_DENSITY_LAPLACE 8
#define HB_DENSITY_BIMIXTURE 9
int hb_density_nargs(int kind);   /* -1 for an unknown kind */
int hb_density_logpdf(int kind, const float* const* args, const long long* periods, long long total, float* out,
                      void* stream);
/* Backward of hb_density_logpdf (what tf.gradients emits for the same graph).  g: incoming gradient read at
 * e % g_period (1 = the scalar a reduce_sum sends back).  dargs: HOST array of device pointers, NULL = not wanted.
 * For an operand with period 1 (and total > 1) dargs[i][0] = sum_e g[e] * dlogp/d operand_i, reduced in-kernel
 * (deterministic; needs ws of hb_reduce_workspace_bytes()); otherwise dargs[i][e] = g[e] * dlogp/d operand_i at
 * full size and the caller sums over the broadcast axes. */
int hb_density_logpdf_bwd(int kind, const float* const* args, const long long* periods, long long total, const float* g,
                          long long g_period, float* const* dargs, void* ws, size_t ws_bytes, void* stream);
/* MinibatchData.get_feed_dict (param.py:733-739) on device: dst[i,:] = src[index[i],:], index int64. */
int hb_gather_rows(float* dst, const float* src, const long long* index, long long n_index, long long row_elems,
                   void* stream);
/* Indexer.train_index (model.py:147-149) on device: out[i] = pool[j_i], j_i uniform in [0, pool_size) with replacement,
 * drawn from Philox(seed, offset) (two 32-bit words per index; 2 * ceil(n_index / 2) stream positions).  pool == NULL:
 * out[i] = j_i.  Feeds hb_gather_rows without any host work or host->device copy per step. */
int hb_random_index(long long* out, long long n_index, const long long* pool, long long pool_size, unsigned long long seed,
                    unsigned long long offset, void* stream);
/* reduce_sum(densities.gaussian(y, f_scale*f, var)) fused with the residual for the backward.
 * f: [total]; y: [y_period] broadcast; var, f_scale: device scalars (f_scale may be NULL = 1).
 * resid (may be NULL) = -rcoef*(f_scale*f - y)/var.  out3 = {loglik, sum E^2, sum E*(f_scale*f)}. */
int hb_gauss_loglik_fwd(const float* f, const float* f_scale, const float* y, long long total, long long y_period,
                        const float* var, float rcoef, float* resid, float* out3, void* ws, size_t ws_bytes,
                        void* stream);

/* UnitRBF.K / UnitCsymRBF.K (gp/kernels.py:54-84,110-111,122-126), + jitter*I when X2 == NULL
 * (UnitStationary.Cholesky :100-101).  X [batch,n,D], X2 [batch,n2,D] or NULL, ell [n_ell] with
 * n_ell in {1, D} (already transformed to the positive space).  lower_only skips tiles above the
 * diagonal (requires X2 == NULL). */
int hb_rbf_gram_fwd(const float* X, const float* X2, int n, int n2, int D, int batch, const float* ell, int n_ell,
                    float* K, long long ldk, long long strideK, float jitter, int lower_only, int csym,
                    void* stream);
/* Gradient w.r.t. the SECOND kernel argument (SparseGP inducing points, Henbun/gp/gp.py:95-98, 146-174):
 * dX2[b][j][d] = scale * sum_i Geff_ij K(x_i, x2_j) (x_id - x2_jd) / ell_d^2, Geff = G or (sym_lower, n == n2) the
 * symmetric matrix whose lower triangle G holds.  X2 == NULL means X.  The gradient w.r.t. the first argument is the
 * same call on G^T with the arguments swapped.  UnitRBF only (no Csym term); D <= 32. */
int hb_rbf_gram_bwd_x2(const float* G, long long ldg, long long strideG, const float* X, const float* X2, int n, int n2,
                       int D, int batch, const float* ell, int n_ell, int sym_lower, float scale, float* dX2, void* stream);
/* g_ell[n_ell] = *out_scale * sum_ij G_ij dK_ij/d ell.  sym_lower: G's lower triangle holds a symmetric
 * gradient (full-symmetric convention), off-diagonal entries count twice. */
int hb_rbf_gram_bwd(const float* G, long long ldg, long long strideG, const float* X, const float* X2, int n, int n2,
                    int D, int batch, const float* ell, int n_ell, int sym_lower, int csym, const float* out_scale,
                    float* g_ell, void* ws, size_t ws_bytes, void* stream);

/* tf.cholesky (gp/kernels.py:101; gp/gp.py:135), batched, in place, lower. */
size_t hb_potrf_workspace_bytes(int n);
int hb_potrf_lower(float* A, long long lda, long long strideA, int n, int batch, int zero_upper, void* ws,
                   size_t ws_bytes, int* err_flag, void* stream, const hb_options* opt);
/* Reverse mode of tf.cholesky (TF's _CholeskyGrad, reached through Optimizer.compile, model.py:220).
 * In: G lower = dObj/dL.  Out: G lower = dObj/dK for the symmetric input (off-diagonals of a
 * symmetric perturbation count twice). */
int hb_potrf_lower_bwd(const float* L, long long ldl, long long strideL, float* G, long long ldg, long long strideG,
                       int n, int batch, void* ws, size_t ws_bytes, void* stream, const hb_options* opt);
/* tf.matrix_triangular_solve from the right: X <- X L^{-T} (trans=1) or X L^{-1} (trans=0)
 * (gp/gp.py:162,169 and densities.py:84 use the transposed-left forms of the same solves). */
size_t hb_trsm_workspace_bytes(int m, int n);
int hb_trsm_right_lower(const float* L, long long ldl, float* X, long long ldx, int m, int n, int trans, void* ws,
                        size_t ws_bytes, void* stream, const hb_options* opt);

/* tf.matmul (GaussianProcess.ipynb:144, gp/gp.py:50, nn.py:32, variationals.py:146) with the fused
 * MatBias epilogue clip(x w + b) -> activation (nn.py:32,83).
 * C[M,N] = act(clip(alpha*op(A) op(B) + beta*C + bias)).  transA=0: A stored [M,K]; 1: [K,M].
 * transB=0: B stored [K,N]; 1: [N,K].  Triangular masks: see csrc/gemm.cuh.  Batched by strides. */
int hb_gemm(const float* A, long long lda, long long strideA, int transA, int a_tri, const float* B, long long ldb,
            long long strideB, int transB, int b_tri, float* C, long long ldc, long long strideC, int c_tri, int M,
            int N, int K, int batch, float alpha, float beta, const float* bias, long long strideBias, int act,
            int clip, float clip_lo, float clip_hi, void* stream);
/* hb_gemm with an optional scratch buffer and options.  Engine choice (opt->gemm_engine == 0, the default):
 *   - K <= 256 and few output tiles          -> short-K fp32 SIMT kernel (whole K staged in one round trip)
 *   - batch 1, 16-byte aligned A/B, ld % 4 == 0, N >= 64, K >= 32 and M*N*K >= 256^3 (or K >= 512 with ws given)
 *                                            -> tcgen05 engine (gemm_tc2.cu): any transposition, triangular masks,
 *                                               alpha/beta/bias/activation epilogue, C may alias A when N <= 256;
 *                                               CTA-pair kernel from 64 tiles of 256x256, split-K (needs ws: partial
 *                                               tiles, <= 40 MiB) for long-K products with a small output
 *   - everything else (batched, unaligned)   -> k-looped fp32 SIMT kernel.
 * Results are fp32-grade on every path (product error vs fp64 <= 3e-6 relative, tests/test_gpu_tc.py). */
int hb_gemm_ws(const float* A, long long lda, long long strideA, int transA, int a_tri, const float* B, long long ldb,
               long long strideB, int transB, int b_tri, float* C, long long ldc, long long strideC, int c_tri, int M,
               int N, int K, int batch, float alpha, float beta, const float* bias, long long strideBias, int act,
               int clip, float clip_lo, float clip_hi, void* ws, size_t ws_bytes, void* stream, const hb_options* opt);
/* Force the tensor-core engine on C[M,N] = alpha*A[M,K]*B[N,K]^T + beta*C (both operands K-major); HB_ERR_ARG if the
 * operands do not qualify. */
size_t hb_gemm_tc_workspace_bytes(int M, int N, int K);
int hb_gemm_tn_tc(const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc, int c_tri, int M,
                  int N, int K, float alpha, float beta, void* ws, size_t ws_bytes, void* stream);
/* The engine behind the big products of hb_potrf_lower / hb_potrf_lower_bwd at n >= 4096 (csrc/gemm_h2.cu), standalone:
 * both fp32 operands are split once into fp16 hi/lo pairs scaled by a power of two taken from their absolute maximum
 * (22 mantissa bits; a_blockscale = 1: one scale per 128-column block of the stored A), then multiplied by three
 * kind::f16 tcgen05 MMAs per k-step with two-level fp32 accumulation.  C = alpha op(A) op(B) + beta C, layouts as
 * hb_gemm (transA = 0: A stored [M, K]; transB = 0: B stored [K, N]).  a_bmode (square op(A), 128-blocks): 1 keeps
 * k-block <= row-block, 2 keeps k-block > row-block.  skip_split = 1 reuses the shadows a previous call left in ws
 * (timing the product alone).  M, N > 128; K, lda, ldb multiples of 8. */
size_t hb_gemm_presplit_workspace_bytes(int M, int N, int K, int transA, int transB);
int hb_gemm_presplit(const float* A, long long lda, int transA, const float* B, long long ldb, int transB, float* C,
                     long long ldc, int c_tri, int M, int N, int K, float alpha, float beta, int a_bmode, int a_blockscale,
                     int skip_split, void* ws, size_t ws_bytes, void* stream, const hb_options* opt);
/* Backward helper of MatBias: dz = dy * act'(y) (through the output y), dbias[c] = sum_r dz[r,c]. */
/* Same with a scratch buffer of hb_act_bwd_colsum_workspace_bytes(rows, cols): full-grid kernel + deterministic partial
 * reduction (the scratch-free entry point uses one block per 32 columns).  Falls back to it when ws is NULL / too small. */
size_t hb_act_bwd_colsum_workspace_bytes(int rows, int cols);
int hb_act_bwd_colsum_ws(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act,
                         int clip, float clip_lo, float clip_hi, float* dbias, void* ws, size_t ws_bytes, void* stream);
int hb_act_bwd_colsum(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act,
                      int clip, float clip_lo, float clip_hi, float* dbias, void* stream);
int hb_colsum(const float* a, long long lda, int rows, int cols, float alpha, float beta, float* out, void* stream);

/* tf.train.AdamOptimizer.minimize(-objective) (model.py:206,220), TF-1 update rule:
 * g = grad_scale*grad; lr_t = lr*sqrt(1-b2^t)/(1-b1^t); theta -= lr_t*m/(sqrt(v)+eps).
 * t is read from *step_dev when non-NULL (graph-capturable), else step_host. */
int hb_adam_tf1(float* theta, const float* grad, float* m, float* v, long long n, float grad_scale, float lr,
                float b1, float b2, float eps, const int* step_dev, int step_host, void* stream);
int hb_increment_i32(int* counter, void* stream);

/* small utilities used by the host layer */
int hb_transpose2d(float* dst, long long ldd, const float* src, long long lds, int rows, int cols, float scale, void* stream);
int hb_zero_strict_upper(float* a, long long lda, int n, void* stream);

/* ---- fused ELBO + gradient of the variational GP regression graph -------------------------------
 * notebooks/GaussianProcess.ipynb:109-148 (ELBO_gaussian), S-sample mean:
 *   y_fit = matmul(kern.Cholesky(X), q) * sqrt(k_var);  ELBO = sum gaussian(Y, y_fit, var) - KL()
 * with q = variationals.Gaussian(shape=[n,1], q_shape) = scale * Normal.
 * params / grads packing (free space, floats):
 *   [ q_mu (n) | q_sqrt (n if mean-field else n*n) | scale (1) | lengthscales (n_ell) | k_var (1) | var (1) ]
 * out4 = { ELBO, loglik_sum, kl_sum, 0 }.  eps: [S,n] or NULL (Philox(seed, offset)). */
typedef struct {
  int n, D, S, n_ell;
  int q_fullrank;
  float jitter;
  unsigned long long seed, offset;
  const hb_options* opt;   /* NULL = defaults */
} hb_gp_config;
size_t hb_gp_param_count(const hb_gp_config* cfg);
/* Notebook-sized models (n <= hb_gp_small_max_n(0) = 128 in fp32, hb_gp_small_max_n(1) = 112 in fp64): the whole step --
 * Gram, Cholesky, sampler + KL, projection, log-likelihood, the complete backward and, when adam_m / adam_v are given,
 * the TF-1 Adam update -- is ONE persistent CTA with K / L / K-bar resident in shared memory (csrc/gp_small.cu).
 * hb_gp_elbo_step takes this path for n <= 128 (opt->small_gp_kernel, default on).  fp32 runs on the blocked shared-memory
 * building blocks of the 128 x 128 leaf kernels -- 16-wide panels for the factorisation, the closed form
 * K-bar = sym(L^-T Phi(L^T L-bar) L^-1) as a blocked triangular inverse + three masked 128^3 products for its reverse mode:
 * 168 us per step at N = 100, S = 10 against 239 us for the 23-kernel path (a first version with one column per step: 280 us);
 * fp64 keeps the column-at-a-time form.
 * The _f64 variant is the reference's float_type = float64 (henbunrc:7) for this graph: every pointer is double,
 * same packing.  adam: grad_scale = -1 minimises -ELBO; step counter read from *step_dev when non-NULL. */
typedef struct {
  double lr, b1, b2, eps, grad_scale;
  const int* step_dev;
  int step_host;
} hb_adam_config;
int hb_gp_small_max_n(int f64);
size_t hb_gp_small_workspace_bytes(const hb_gp_config* cfg, int f64);
int hb_gp_small_step(const hb_gp_config* cfg, const float* X, const float* Y, float* params, const float* eps, float* grads,
                     float* out4, float* adam_m, float* adam_v, const hb_adam_config* adam, void* ws, size_t ws_bytes,
                     int* err_flag, void* stream);
int hb_gp_small_step_f64(const hb_gp_config* cfg, const double* X, const double* Y, double* params, const double* eps,
                         double* grads, double* out4, double* adam_m, double* adam_v, const hb_adam_config* adam, void* ws,
                         size_t ws_bytes, int* err_flag, void* stream);
size_t hb_gp_elbo_workspace_bytes(const hb_gp_config* cfg);
int hb_gp_elbo_step(const hb_gp_config* cfg, const float* X, const float* Y, const float* params, const float* eps,
                    float* grads, float* out4, void* ws, size_t ws_bytes, int* err_flag, void* stream);

/* ---- float64 at any size (csrc/f64.cu) --------------------------------------------------------------------------------
 * The reference's float_type = float64 (henbunrc:7) beyond the one-CTA kernel's n <= 112.  Every pointer is double.
 *
 * hb_gemm_f64: C[M,N] = alpha op(A) op(B) + beta C on the fp64 tensor cores (mma.sync f64 -> DMMA).  Layouts and the
 * triangular masks a_tri / b_tri (0..4) / c_tri (0, 1) as hb_gemm; with c_tri = 1 nothing above the diagonal of C is
 * written.  beta = 0 does not read C.  ws (optional): outputs of fewer than 74 tiles with K >= 1024 split K over CTAs
 * into partial tiles of ws (splits * M * N doubles, at most 32 splits) and sum them in a fixed order, so results are
 * deterministic either way.  No bias, activation or batch.
 *
 * hb_potrf_lower_f64 / hb_potrf_lower_bwd_f64: the conventions of hb_potrf_lower / hb_potrf_lower_bwd (lower triangle
 * only; a non-positive pivot writes 1 + its row into *err_flag; the reverse mode takes G lower = dObj/dL and leaves
 * dObj/dK in the symmetric-input convention) for one matrix.  The column recursion over 64-column leaves, every
 * product on hb_gemm_f64, panels solved by substitution (no explicit inverse).  ws of hb_potrf_f64_workspace_bytes(n).
 *
 * hb_gp_elbo_step_f64: hb_gp_small_step_f64 at any n, same arguments (adam_m / adam_v NULL: gradient only).  For
 * n <= hb_gp_small_max_n(1) with opt->small_gp_kernel on (the default) it IS hb_gp_small_step_f64; otherwise, and always
 * with small_gp_kernel = 0, it runs a chain of kernels: Gram, hb_potrf_lower_f64, sampler + KL, the two S-row
 * products, log-likelihood, sampler backward, hb_potrf_lower_bwd_f64, Gram backward, scalar chain rules, Adam.  eps NULL
 * draws the library's Philox stream (the fp32 draw widened to double), the same samples on both routes.
 * ws of hb_gp_elbo_f64_workspace_bytes(cfg) (which follows cfg->opt to the route). */
int hb_gemm_f64(const double* A, long long lda, int transA, int a_tri, const double* B, long long ldb, int transB, int b_tri,
                double* C, long long ldc, int c_tri, int M, int N, int K, double alpha, double beta, void* ws, size_t ws_bytes,
                void* stream);
size_t hb_potrf_f64_workspace_bytes(int n);
int hb_potrf_lower_f64(double* A, long long lda, int n, void* ws, size_t ws_bytes, int* err_flag, void* stream);
int hb_potrf_lower_bwd_f64(const double* L, long long ldl, double* G, long long ldg, int n, void* ws, size_t ws_bytes,
                           void* stream);
size_t hb_gp_elbo_f64_workspace_bytes(const hb_gp_config* cfg);
int hb_gp_elbo_step_f64(const hb_gp_config* cfg, const double* X, const double* Y, double* params, const double* eps,
                        double* grads, double* out4, double* adam_m, double* adam_v, const hb_adam_config* adam, void* ws,
                        size_t ws_bytes, int* err_flag, void* stream);

/* ---- float64 mixture-of-experts GP regression (csrc/moe64.cu) ----------------------------------------------------------
 * notebooks/Expert_GPR.ipynb:101-149 (BASELINE config 2), S-sample mean, every pointer double: experts s, l and gate r,
 *   f_e = matmul(kern_e.Cholesky(X), q_e),  frac = sigmoid(f_r * sqrt(k_var_r)),
 *   ELBO = sum gaussian(Y, (frac f_s + (1 - frac) f_l) * k_var, var) - KL()
 * with q_e = variationals.Gaussian(shape=[n,1], q_fullrank[e]) and kern_e = UnitRBF (n_ell[e] = 1 or D lengthscales).
 * params / grads packing (free space): [ q_mu | q_sqrt | scale | lengthscales ] for s, then l, then r (each segment laid
 * out as hb_gp_config's packing up to its lengthscales), then [ k_var | k_var_r | var ].  out4 = { ELBO, loglik_sum, kl_sum over the three, 0 }.
 * eps_e: [S,n] or NULL (the library's Philox stream at (seed, offset[e]), the fp32 draw widened to double; offset[e] a
 * multiple of 4).  adam_m / adam_v NULL: gradient only; otherwise the TF-1 Adam update of hb_gp_elbo_step_f64 follows.
 * A non-positive pivot in any expert's factorisation writes 1 + its row into *err_flag; the three factorisations run
 * concurrently, so when several fail the row is that of whichever got there first, and the expert is not identified.  The three GP chains run
 * concurrently on two side streams forked from `stream` and joined back into it; results are bitwise repeatable and
 * `stream` has waited on all of the work when the call returns.  D <= 32.  ws of hb_moe_gp_f64_workspace_bytes(cfg). */
typedef struct {
  int n, D, S;
  int n_ell[3];                        /* 1 or D; experts s, l, gate r */
  int q_fullrank[3];
  double jitter;
  unsigned long long seed, offset[3];  /* Philox window per variational; each a multiple of 4 when its eps is NULL */
  const hb_options* opt;               /* NULL = defaults */
} hb_moe_gp_config;
size_t hb_moe_gp_param_count(const hb_moe_gp_config* cfg);
size_t hb_moe_gp_f64_workspace_bytes(const hb_moe_gp_config* cfg);
int hb_moe_gp_elbo_step_f64(const hb_moe_gp_config* cfg, const double* X, const double* Y, double* params, const double* eps_s,
                            const double* eps_l, const double* eps_r, double* grads, double* out4, double* adam_m,
                            double* adam_v, const hb_adam_config* adam, void* ws, size_t ws_bytes, int* err_flag, void* stream);

/* ---- the same step with the factorisation and its reverse mode on a right-looking schedule over column blocks, on one GPU
 * or SHARED BY A GROUP OF GPUs (strong scaling of BASELINE config 3; the reference has no multi-device path, SURVEY.md 8e:
 * tf.cholesky, gp/kernels.py:100-101, and its gradient run on one device).
 * Column blocks of `block` columns (a multiple of 128; 0 = 2048) are dealt round-robin (`turn` at a time): block b belongs to rank (b / turn) % world.
 * Its owner factors it (all rows below; the column recursion restricted to the block) on a high-priority "chain" stream while
 * every rank applies the previous panels to the blocks it owns on the caller's stream; a finished panel travels to the other
 * ranks by ncclBroadcast on a third stream and is unpacked into each rank's own copy of the matrix, fp16 hi/lo shadows and
 * scales rebuilt bit-identically -- so after hb_potrf_lower_dist every rank holds the complete factor, after
 * hb_potrf_lower_bwd_dist the complete gradient, and the rest of the step needs no further exchange.  world == 1
 * (comm == NULL) is the same two-stream schedule on one GPU.
 * hb_comm_*: a communicator of this library's own over the NCCL the process already carries (bound at run time; rank 0 calls
 * hb_comm_unique_id, the 128 bytes travel to the other ranks by any means -- torch.distributed in the Python layer --, every
 * rank calls hb_comm_create with its device current).  All ranks must make the same sequence of *_dist calls.
 * err_flag is set on the rank that owns the failing block only: reduce it (max) across ranks before trusting a step. */
typedef struct hb_dist {
  void* comm;            /* from hb_comm_create; NULL when world == 1 */
  int rank, world;
  int block;             /* columns per block, multiple of 128; 0 = 2048 */
  int shard_samples;     /* hb_gp_elbo_step_dist: 1 = every rank draws its OWN S samples (its own eps / Philox window) and the
                            ranks share one factorisation: Z and the residuals are all-gathered (2 world S n floats) before
                            L-bar is formed, K-bar and the lengthscale gradient come out as the rank-averaged ones on every
                            rank, the remaining gradients are per-rank means to be averaged by the caller's all-reduce.
                            0 = every rank evaluates the same samples (nothing to reduce afterwards) */
  int batch;             /* blocks further than two from the current one take the finished panels `batch` at a time, as ONE
                            product over all their columns (long-K products from narrow blocks); 0 = 1 */
  int block_bwd;         /* hb_gp_elbo_step_dist: block width of the reverse mode when it should differ from the forward pass
                            (every rank holds the complete factor in between, so the two distributions are independent; measured:
                            the forward chain prefers 1024-column blocks, the reverse 2048); 0 = block */
  int turn;              /* consecutive blocks a rank owns before the next rank's turn: block b belongs to rank (b / turn) % world.
                            Panels travel block by block, so with turn > 1 the broadcast of a block overlaps the factorisation
                            of the owner's next one; 0 = 1 */
} hb_dist;
int hb_comm_unique_id(void* out128_host);
int hb_comm_create(const void* id128_host, int rank, int world, void** comm_out);
int hb_comm_destroy(void* comm);
/* Optional timeline of the schedule (instrumentation, like hb_profile_*): timing events at the stations of every block --
 * tag 0 chain: factorisation of block p starts | 1 done | 2 panel p available on this rank (sent, or received + unpacked) |
 * 3 chain: the update the next block still lacked is done | 4 main: updates with panel p may start | 5 main: done.
 * hb_flat_trace_end synchronises the device, fills rows {tag, block, ms since the first station}, returns the row count. */
int hb_flat_trace_begin(void);
int hb_flat_trace_end(double* out3_host, int capacity);
size_t hb_potrf_dist_workspace_bytes(int n, const hb_dist* d);
int hb_potrf_lower_dist(float* A, long long lda, int n, const hb_dist* d, void* ws, size_t ws_bytes, int* err_flag, void* stream,
                        const hb_options* opt);
int hb_potrf_lower_bwd_dist(const float* L, long long ldl, float* G, long long ldg, int n, const hb_dist* d, void* ws,
                            size_t ws_bytes, void* stream, const hb_options* opt);
size_t hb_gp_elbo_dist_workspace_bytes(const hb_gp_config* cfg, const hb_dist* d);
int hb_gp_elbo_step_dist(const hb_gp_config* cfg, const hb_dist* d, const float* X, const float* Y, const float* params,
                         const float* eps, float* grads, float* out4, void* ws, size_t ws_bytes, int* err_flag, void* stream);

/* ---- fused ELBO + gradient of the amortised local-variable model (BASELINE config 4) ----------------------------
 *   q_local = enc(X);  x_rec = dec(q_local);  ELBO = sum gaussian(X, x_rec, var) - KL(LOCAL),  S-sample mean
 * enc / dec = nn.NeuralNet (nn.py:34-87: hidden layers act(x w + b), last layer linear), q_local = LOCAL
 * variationals.Normal([latent]) fed with the encoder's output row [mu | log sigma] (param.py:516-537).
 * X: this step's minibatch [B, enc_nodes[0]] (e.g. from hb_gather_rows).  eps: [S, B, latent] or NULL (Philox).
 * params / grads packing (free space): enc w0 [in, out] | enc b0 [out] | enc w1 | ... | dec w0 | dec b0 | ... | var (1).
 * out4 = {ELBO, loglik_sum, kl_sum, 0}.  *_act: HB_ACT_* of the hidden layers (n - 1 entries). */
#define HB_MAX_LAYERS 8
typedef struct {
  int B, S, latent;
  int n_enc, enc_nodes[HB_MAX_LAYERS + 1], enc_act[HB_MAX_LAYERS];
  int n_dec, dec_nodes[HB_MAX_LAYERS + 1], dec_act[HB_MAX_LAYERS];
  unsigned long long seed, offset;
  const hb_options* opt;   /* NULL = defaults */
} hb_amortised_config;
size_t hb_amortised_param_count(const hb_amortised_config* cfg);
size_t hb_amortised_workspace_bytes(const hb_amortised_config* cfg);
int hb_amortised_elbo_step(const hb_amortised_config* cfg, const float* X, const float* params, const float* eps, float* grads,
                           float* out4, void* ws, size_t ws_bytes, void* stream);

/* ---- fused ELBO + gradient + Adam of the linear-operator model (BASELINE config 5) ---------------------
 * q = variationals.Normal([n], q_shape='fullrank') (variationals.py:94-96,144-146,185-186,225-230) observed through a
 * dense operator A [M, n]:  ELBO = sum gaussian(y, A z, var) - KL  (densities.py:25-27), S-sample mean.
 * params / grads / m / v packing (free space, floats):  [ q_sqrt (n*n, row-major, lower triangle used) | q_mu (n) | var (1) ]
 * Row-sharded across ranks: each rank holds M rows of the M_total-row operator and calls hb_linop_elbo_local, the
 * ranks all-reduce (sum) zbar_stats [S*n + 4], every rank calls hb_linop_elbo_update.  On one GPU M == M_total
 * and the two calls run back to back.  Both calls take the SAME workspace (it carries eps and z between them).
 *   local : eps [S,n] or NULL (Philox(seed, offset), identical on every rank).
 *   update: grads may be NULL; when given it receives d ELBO_mean / d params (strict upper triangle of q_sqrt
 *           untouched).  m, v NULL -> gradient only; otherwise the TF-1 Adam rule of hb_adam_tf1 on -ELBO is applied
 *           in the same pass that forms the q_sqrt gradient (never materialised).  out4 = {ELBO, loglik, kl, 0}. */
typedef struct {
  int M;                 /* rows of A held by this rank */
  long long M_total;     /* rows of the whole operator (== M on one GPU) */
  int n, S;
  unsigned long long seed, offset;
  int presplit;          /* 1: both passes over A run on the pre-split tcgen05 engine from an fp16 hi/lo shadow of A that
                            hb_linop_prepare writes into the workspace once per operator (+ 4 bytes per element of A of
                            workspace; n % 8 == 0, M % 8 == 0).  0: A is consumed as fp32 (in-kernel split). */
  const hb_options* opt; /* NULL = defaults */
} hb_linop_config;
size_t hb_linop_param_count(const hb_linop_config* cfg);
size_t hb_linop_workspace_bytes(const hb_linop_config* cfg);
/* presplit = 1 only: split the operator into the workspace's shadow.  Call once, and again whenever A changes. */
int hb_linop_prepare(const hb_linop_config* cfg, const float* A, void* ws, size_t ws_bytes, void* stream);
int hb_linop_elbo_local(const hb_linop_config* cfg, const float* A, const float* y, const float* params, const float* eps,
                        float* zbar_stats, void* ws, size_t ws_bytes, void* stream);
int hb_linop_elbo_update(const hb_linop_config* cfg, float* params, const float* zbar_stats, float* grads, float* m, float* v,
                         float lr, float b1, float b2, float eps_adam, const int* step_dev, int step_host, float* out4,
                         void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HENBUN_B200_H */
