// Utility kernels: strided copies/transposes, Philox fill, column sums, activation backward,
// TF-1 Adam.  All HBM-bound; vectorised where alignment allows, grid sized from the SM count.
#include "kernels.cuh"
#include "gemm.cuh"

namespace hb {

unsigned long long g_launches = 0;

namespace {

constexpr int kSMs = 148;

inline int grid_for(long long work_items, int threads, int max_blocks = kSMs * 16) {
  long long b = (work_items + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return (int)b;
}

__global__ void copy2d_kernel(float* __restrict__ dst, long long ldd, const float* __restrict__ src, long long lds,
                              int rows, int cols, float scale) {
  const long long total = (long long)rows * cols;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / cols; const int c = (int)(e % cols);
    dst[r * ldd + c] = scale * src[r * lds + c];
  }
}

__global__ void scale2d_kernel(float* a, long long lda, int rows, int cols, float s) {
  const long long total = (long long)rows * cols;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / cols; const int c = (int)(e % cols);
    a[r * lda + c] *= s;
  }
}

__global__ void transpose2d_kernel(float* __restrict__ dst, long long ldd, const float* __restrict__ src,
                                   long long lds, int rows, int cols, float scale) {
  __shared__ float t[32][33];
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = by + i, c = bx + threadIdx.x;
    t[i][threadIdx.x] = (r < rows && c < cols) ? src[(long long)r * lds + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = bx + i, r = by + threadIdx.x;   // dst[c][r]
    if (r < rows && c < cols) dst[(long long)c * ldd + r] = scale * t[threadIdx.x][i];
  }
}

__global__ void zero_strict_upper_kernel(float* a, long long lda, int n) {
  const long long total = (long long)n * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / n; const int c = (int)(e % n);
    if (c > r) a[r * lda + c] = 0.f;
  }
}

__global__ void fill_kernel(float* a, long long n, float v) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) a[e] = v;
}

__global__ void randn_kernel(float* out, long long count, unsigned long long seed, unsigned long long offset) {
  // offset is a multiple of 4: group g covers flat stream positions [offset+4g, offset+4g+4)
  const long long ngroups = (count + 3) / 4;
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < ngroups; g += (long long)gridDim.x * blockDim.x) {
    float z[4];
    philox_normal4(seed, (offset >> 2) + (unsigned long long)g, z);
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (4 * g + c < count) out[4 * g + c] = z[c];
  }
}

__global__ void add_rowvec_kernel(float* z, long long ldz, const float* __restrict__ mu, int rows, int cols) {
  const long long total = (long long)rows * cols;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / cols; const int c = (int)(e % cols);
    z[r * ldz + c] += mu[c];
  }
}

// out[c] = alpha * sum_r a[r][c] + beta * out[c]; one thread per column, coalesced across columns,
// rows split over blockDim.y with a shared-memory combine (deterministic).
__global__ void colsum_kernel(const float* __restrict__ a, long long lda, int rows, int cols, float alpha, float beta,
                              float* out) {
  __shared__ double part[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  double s = 0.0;
  if (c < cols)
    for (int r = threadIdx.y; r < rows; r += blockDim.y) s += (double)a[(long long)r * lda + c];
  part[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    double t = 0.0;
    for (int y = 0; y < blockDim.y; ++y) t += part[y][threadIdx.x];
    const float prev = (beta != 0.f) ? out[c] : 0.f;
    out[c] = alpha * (float)t + beta * prev;
  }
}

__global__ void axpby_kernel(float* y, const float* __restrict__ x, long long n, float a, float b) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    y[e] = a * x[e] + (b != 0.f ? b * y[e] : 0.f);
}

__device__ __forceinline__ float act_grad_from_output(float y, int act) {
  switch (act) {
    case ACT_SIGMOID: return y * (1.f - y);
    case ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case ACT_TANH: return 1.f - y * y;
    default: return 1.f;
  }
}

// dz = dy * act'(y) (expressed through the output y); dbias[c] = sum_r dz[r][c].
// Clip, when enabled, precedes the activation in the reference (nn.py:32 then :83): its gradient
// mask cannot be recovered from y for saturating activations, so for clip=1 the caller passes the
// pre-activation in `y` with act=ACT_NONE and applies the mask |y|<hi here.
__global__ void act_bwd_colsum_kernel(const float* __restrict__ dy, const float* __restrict__ y, float* dz, int rows,
                                      int cols, long long ld, int act, int clip, float lo, float hi, float* dbias) {
  __shared__ double part[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  double s = 0.0;
  if (c < cols)
    for (int r = threadIdx.y; r < rows; r += blockDim.y) {
      const long long idx = (long long)r * ld + c;
      const float yy = y[idx];
      float g = dy[idx] * act_grad_from_output(yy, act);
      if (clip && (yy <= lo || yy >= hi)) g = 0.f;
      dz[idx] = g;
      s += (double)g;
    }
  part[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (dbias && threadIdx.y == 0 && c < cols) {
    double t = 0.0;
    for (int yb = 0; yb < blockDim.y; ++yb) t += part[yb][threadIdx.x];
    dbias[c] = (float)t;
  }
}

// Full-grid version: the one-block-per-32-columns kernel above runs on cols/32 SMs (25 of 148 for a 784-wide layer:
// 27 ms of a 34 ms config-4 step).  Here a block owns a [rows_per_block x 128] slab (float4 per lane along the
// columns), writes dz and a per-block column partial (double) into `partials[blockIdx.y][col]`; a second small kernel
// sums the partials in a fixed order (deterministic, no atomics).
__global__ void __launch_bounds__(256) act_bwd_tile_kernel(const float* __restrict__ dy, const float* __restrict__ y, float* dz,
                                                           int rows, int cols, long long ld, int act, int clip, float lo, float hi,
                                                           int rows_per_block, double* partials) {
  __shared__ double red[8][128];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  const int r_begin = blockIdx.y * rows_per_block, r_end = min(rows, r_begin + rows_per_block);
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  double dacc[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < cols) {
    int n = 0;
    for (int r = r_begin + w; r < r_end; r += 8) {
      const long long idx = (long long)r * ld + c;
      const float4 yy = *reinterpret_cast<const float4*>(y + idx);
      const float4 dd = *reinterpret_cast<const float4*>(dy + idx);
      float g[4] = {dd.x * act_grad_from_output(yy.x, act), dd.y * act_grad_from_output(yy.y, act),
                    dd.z * act_grad_from_output(yy.z, act), dd.w * act_grad_from_output(yy.w, act)};
      if (clip) {
        const float yv[4] = {yy.x, yy.y, yy.z, yy.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) if (yv[e] <= lo || yv[e] >= hi) g[e] = 0.f;
      }
      *reinterpret_cast<float4*>(dz + idx) = make_float4(g[0], g[1], g[2], g[3]);
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[e] += g[e];
      if (++n == 64) {      // bound the fp32 running sums
#pragma unroll
        for (int e = 0; e < 4; ++e) { dacc[e] += (double)acc[e]; acc[e] = 0.f; }
        n = 0;
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) red[w][lane * 4 + e] = dacc[e] + (double)acc[e];
  __syncthreads();
  if (partials && threadIdx.x < 128) {
    const int cc = blockIdx.x * 128 + threadIdx.x;
    if (cc < cols) {
      double t = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
      partials[(long long)blockIdx.y * cols + cc] = t;
    }
  }
}
__global__ void colsum_partials_kernel(const double* __restrict__ partials, int nb, int cols, float* out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  double t = 0.0;
  for (int b = 0; b < nb; ++b) t += partials[(long long)b * cols + c];
  out[c] = (float)t;
}

// tf.train.AdamOptimizer on loss = -objective: g = grad_scale * grad (grad_scale = -1 for maximise).
__global__ void adam_tf1_kernel(float* theta, const float* __restrict__ grad, float* m, float* v, long long n,
                                float gs, float lr, float b1, float b2, float eps, const int* step_dev, int step_host) {
  const int t = step_dev ? *step_dev : step_host;
  const float lr_t = lr * sqrtf(1.f - powf(b2, (float)t)) / (1.f - powf(b1, (float)t));
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const float g = gs * grad[e];
    const float mm = b1 * m[e] + (1.f - b1) * g;
    const float vv = b2 * v[e] + (1.f - b2) * g * g;
    m[e] = mm; v[e] = vv;
    theta[e] -= lr_t * mm / (sqrtf(vv) + eps);
  }
}

__global__ void increment_kernel(int* p) { *p += 1; }

// dst[i, :] = src[index[i], :]  (MinibatchData.get_feed_dict, Henbun/param.py:733-739, on device)
template <typename T>
__global__ void gather_rows_kernel(T* __restrict__ dst, const T* __restrict__ src,
                                   const long long* __restrict__ index, long long n_index, long long row) {
  const long long total = n_index * row;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / row, c = e % row;
    dst[e] = src[index[i] * row + c];
  }
}

}  // namespace

int copy2d(float* dst, long long ldd, const float* src, long long lds, int rows, int cols, float scale, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return HB_OK;
  copy2d_kernel<<<grid_for((long long)rows * cols, 256), 256, 0, st>>>(dst, ldd, src, lds, rows, cols, scale);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int scale2d(float* a, long long lda, int rows, int cols, float s, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return HB_OK;
  scale2d_kernel<<<grid_for((long long)rows * cols, 256), 256, 0, st>>>(a, lda, rows, cols, s);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int transpose2d(float* dst, long long ldd, const float* src, long long lds, int rows, int cols, float scale, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return HB_OK;
  dim3 grid(cdiv(cols, 32), cdiv(rows, 32));
  if (grid.y > 65535) return HB_ERR_ARG;
  transpose2d_kernel<<<grid, dim3(32, 8), 0, st>>>(dst, ldd, src, lds, rows, cols, scale);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int zero_strict_upper(float* a, long long lda, int n, cudaStream_t st) {
  if (n <= 0) return HB_OK;
  zero_strict_upper_kernel<<<grid_for((long long)n * n, 256), 256, 0, st>>>(a, lda, n);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int fill_f32(float* a, long long n, float v, cudaStream_t st) {
  if (n <= 0) return HB_OK;
  fill_kernel<<<grid_for(n, 256), 256, 0, st>>>(a, n, v);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
// Indexer.train_index on the device (Henbun/model.py:147-149: pool[np.random.randint(0, len(pool), B)], with replacement):
// out[i] = pool[floor(u_i * pool_size)], u_i from two Philox words (64-bit multiply-shift), pool == nullptr -> identity.
__global__ void random_index_kernel(long long* out, long long n_index, const long long* __restrict__ pool, unsigned long long pool_size,
                                    unsigned long long seed, unsigned long long offset) {
  const long long ngroups = (n_index + 1) / 2;
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < ngroups; g += (long long)gridDim.x * blockDim.x) {
    uint32_t r[4];
    philox4x32_10(seed, (offset >> 2) + (unsigned long long)g, r);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const long long i = 2 * g + c;
      if (i >= n_index) break;
      const unsigned long long w = ((unsigned long long)r[2 * c + 1] << 32) | r[2 * c];
      const unsigned long long j = __umul64hi(w, pool_size);
      out[i] = pool ? pool[j] : (long long)j;
    }
  }
}
int random_index(long long* out, long long n_index, const long long* pool, long long pool_size, unsigned long long seed,
                 unsigned long long offset, cudaStream_t st) {
  if (n_index <= 0) return HB_OK;
  if (!out || pool_size <= 0 || (offset & 3ull)) return HB_ERR_ARG;
  random_index_kernel<<<grid_for((n_index + 1) / 2, 256), 256, 0, st>>>(out, n_index, pool, (unsigned long long)pool_size, seed, offset);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

// Raw Philox-4x32-10 blocks (known-answer tests): block b = core(counter = ctr4 + b on the low 64 bits, key).
__global__ void philox_raw_kernel(uint32_t* out, long long n_blocks, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                  uint32_t k0, uint32_t k1) {
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < n_blocks; b += (long long)gridDim.x * blockDim.x) {
    const unsigned long long lo = (((unsigned long long)c1 << 32) | c0) + (unsigned long long)b;
    uint32_t c[4] = {(uint32_t)lo, (uint32_t)(lo >> 32), c2, c3};
    philox4x32_10_core(c, k0, k1);
    out[4 * b] = c[0]; out[4 * b + 1] = c[1]; out[4 * b + 2] = c[2]; out[4 * b + 3] = c[3];
  }
}
int philox_raw(uint32_t* out, long long n_blocks, const uint32_t* ctr4, const uint32_t* key2, cudaStream_t st) {
  if (n_blocks <= 0) return HB_OK;
  if (!out || !ctr4 || !key2) return HB_ERR_ARG;
  philox_raw_kernel<<<grid_for(n_blocks, 256), 256, 0, st>>>(out, n_blocks, ctr4[0], ctr4[1], ctr4[2], ctr4[3], key2[0], key2[1]);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int randn_philox(float* out, long long count, unsigned long long seed, unsigned long long offset, cudaStream_t st) {
  if (count <= 0) return HB_OK;
  if (!out || (offset & 3ull)) return HB_ERR_ARG;
  randn_kernel<<<grid_for((count + 3) / 4, 256), 256, 0, st>>>(out, count, seed, offset);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int add_rowvec(float* z, long long ldz, const float* mu, int rows, int cols, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return HB_OK;
  add_rowvec_kernel<<<grid_for((long long)rows * cols, 256), 256, 0, st>>>(z, ldz, mu, rows, cols);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int colsum(const float* a, long long lda, int rows, int cols, float alpha, float beta, float* out, cudaStream_t st) {
  if (cols <= 0) return HB_OK;
  colsum_kernel<<<cdiv(cols, 32), dim3(32, 8), 0, st>>>(a, lda, rows, cols, alpha, beta, out);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int axpby(float* y, const float* x, long long n, float a, float b, cudaStream_t st) {
  if (n <= 0) return HB_OK;
  axpby_kernel<<<grid_for(n, 256), 256, 0, st>>>(y, x, n, a, b);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
size_t act_bwd_colsum_workspace_bytes(int rows, int cols) {
  (void)rows;
  return (size_t)148 * 8 * (size_t)(cols > 0 ? cols : 0) * sizeof(double) + 256;
}
int act_bwd_colsum_ws(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act, int clip,
                      float clip_lo, float clip_hi, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return HB_OK;
  const bool vec = (cols % 4 == 0) && (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(dy) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(y) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dz) & 15) == 0);
  if (!vec || !ws || ws_bytes < act_bwd_colsum_workspace_bytes(rows, cols) || rows < 512)
    return act_bwd_colsum(dy, y, dz, rows, cols, ld, act, clip, clip_lo, clip_hi, dbias, st);
  const int col_tiles = cdiv(cols, 128);
  int row_blocks = (148 * 8) / col_tiles;                       // ~8 blocks per SM in total
  if (row_blocks < 1) row_blocks = 1;
  int rpb = cdiv(rows, row_blocks);
  if (rpb < 64) rpb = 64;
  rpb = (rpb + 7) / 8 * 8;
  row_blocks = cdiv(rows, rpb);
  double* part = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  act_bwd_tile_kernel<<<dim3((unsigned)col_tiles, (unsigned)row_blocks), 256, 0, st>>>(dy, y, dz, rows, cols, ld, act, clip, clip_lo,
                                                                                      clip_hi, rpb, dbias ? part : nullptr);
  HB_CHECK_LAUNCH();
  if (dbias) {
    colsum_partials_kernel<<<cdiv(cols, 128), 128, 0, st>>>(part, row_blocks, cols, dbias);
    HB_CHECK_LAUNCH();
  }
  return HB_OK;
}
int act_bwd_colsum(const float* dy, const float* y, float* dz, int rows, int cols, long long ld, int act, int clip,
                   float clip_lo, float clip_hi, float* dbias, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return HB_OK;
  act_bwd_colsum_kernel<<<cdiv(cols, 32), dim3(32, 8), 0, st>>>(dy, y, dz, rows, cols, ld, act, clip, clip_lo, clip_hi, dbias);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int adam_tf1(float* theta, const float* grad, float* m, float* v, long long n, float grad_scale, float lr, float b1,
             float b2, float eps, const int* step_dev, int step_host, cudaStream_t st) {
  if (n <= 0) return HB_OK;
  if (!theta || !grad || !m || !v) return HB_ERR_ARG;
  adam_tf1_kernel<<<grid_for(n, 256), 256, 0, st>>>(theta, grad, m, v, n, grad_scale, lr, b1, b2, eps, step_dev, step_host);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
template <typename T>
int gather_rows_t(T* dst, const T* src, const long long* index, long long n_index, long long row_elems, cudaStream_t st) {
  if (n_index < 0 || row_elems < 0) return HB_ERR_ARG;
  if (n_index * row_elems == 0) return HB_OK;
  if (!dst || !src || !index) return HB_ERR_ARG;
  gather_rows_kernel<T><<<grid_for(n_index * row_elems, 256), 256, 0, st>>>(dst, src, index, n_index, row_elems);
  HB_CHECK_LAUNCH();
  return HB_OK;
}
int gather_rows(float* dst, const float* src, const long long* index, long long n_index, long long row_elems,
                cudaStream_t st) {
  return gather_rows_t(dst, src, index, n_index, row_elems, st);
}
int gather_rows_f64(double* dst, const double* src, const long long* index, long long n_index, long long row_elems,
                    cudaStream_t st) {
  return gather_rows_t(dst, src, index, n_index, row_elems, st);
}
int increment_i32(int* p, cudaStream_t st) {
  increment_kernel<<<1, 1, 0, st>>>(p);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

}  // namespace hb
