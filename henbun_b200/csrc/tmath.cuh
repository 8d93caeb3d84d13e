// Type-generic device math and the column-at-a-time shared-memory Cholesky pair shared by the fp64 kernels
// (gp_small.cu's one-CTA step, f64.cu's leaves of the blocked recursion).
#pragma once
#include "common.cuh"

namespace hb {

template <typename T> __device__ __forceinline__ T t_exp(T x);
template <> __device__ __forceinline__ float t_exp<float>(float x) { return expf(x); }
template <> __device__ __forceinline__ double t_exp<double>(double x) { return exp(x); }
template <typename T> __device__ __forceinline__ T t_log(T x);
template <> __device__ __forceinline__ float t_log<float>(float x) { return logf(x); }
template <> __device__ __forceinline__ double t_log<double>(double x) { return log(x); }
template <typename T> __device__ __forceinline__ T t_sqrt(T x);
template <> __device__ __forceinline__ float t_sqrt<float>(float x) { return sqrtf(x); }
template <> __device__ __forceinline__ double t_sqrt<double>(double x) { return sqrt(x); }
template <typename T> __device__ __forceinline__ T t_softplus(T x) {
  const T ax = x < T(0) ? -x : x;
  return (x > T(0) ? x : T(0)) + (T)log1p((double)t_exp<T>(-ax));
}
template <typename T> __device__ __forceinline__ T t_sigmoid(T x) { return T(1) / (T(1) + t_exp<T>(-x)); }

// Right-looking Cholesky of the n x n lower triangle of L (leading dimension LD, shared memory), one column per step,
// by a CTA of NT threads (NT a multiple of 512: a 16 x 32 grid per trailing update).  colv: [n] shared scratch.
// Returns, in every thread, 0 or 1 + the first column with a non-positive pivot (the factorisation goes on with pivot 1).
template <typename T, int NT>
__device__ __forceinline__ int potrf_cols_smem(T* L, int LD, int n, T* colv, int* sh_bad) {
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  constexpr int NY = NT / 32;
  if (tid == 0) *sh_bad = 0;
  __syncthreads();
  for (int j = 0; j < n; ++j) {
    const T d = L[j * LD + j];                           // every thread takes the pivot itself: two barriers per column
    if (tid == 0 && !(d > T(0)) && *sh_bad == 0) *sh_bad = j + 1;
    const T piv = t_sqrt<T>(d > T(0) ? d : T(1)), rp = T(1) / piv;
    for (int i = j + 1 + tid; i < n; i += NT) {
      const T x = L[i * LD + j] * rp;
      L[i * LD + j] = x;
      colv[i] = x;
    }
    __syncthreads();
    if (tid == 0) L[j * LD + j] = piv;
    for (int r = j + 1 + ty; r < n; r += NY) {
      const T lr = colv[r];
      for (int c = j + 1 + tx; c <= r; c += 32) L[r * LD + c] -= lr * colv[c];
    }
    __syncthreads();
  }
  return *sh_bad;
}

// Reverse mode of potrf_cols_smem, level 2 (Murray 2016), in place: on entry the lower triangle of G holds dObj/dL, on exit
// dObj/dA for every stored lower entry A[r][c] (an off-diagonal entry stands for both A[r][c] and A[c][r]).  colv: [n] scratch.
template <typename T, int NT>
__device__ __forceinline__ void potrf_rev_cols_smem(const T* L, T* G, int LD, int n, T* colv) {
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  constexpr int NY = NT / 32;
  for (int j = n - 1; j >= 0; --j) {
    // reverse of the trailing update of column j: Lbar[r, j] -= sum_c (Abar[r, c] + Abar[c, r]) L[c, j]  (r, c > j):
    // warp ty owns rows ty + NY i, its lanes split the columns, one shuffle reduction per row
    for (int r = j + 1 + ty; r < n; r += NY) {
      T acc = T(0);
      for (int c = j + 1 + tx; c < n; c += 32) {
        const T ab = (c <= r) ? G[r * LD + c] : G[c * LD + r];
        acc += ab * L[c * LD + j] * ((c == r) ? T(2) : T(1));
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (tx == 0) colv[r] = acc;
    }
    __syncthreads();
    if (ty == 0) {           // column phase in one warp: scale the column, dot product for the diagonal, no block-wide reduction
      const T ljj = L[j * LD + j];
      T dot = T(0);
      for (int r = j + 1 + tx; r < n; r += 32) {
        const T lb = G[r * LD + j] - colv[r];            // adjoint of L[r, j]
        G[r * LD + j] = lb / ljj;                        // reverse of the column scaling: adjoint of A[r, j]
        dot += lb * L[r * LD + j];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      if (tx == 0) {
        const T lbjj = G[j * LD + j] - dot / ljj;        // adjoint of L[j, j]
        G[j * LD + j] = lbjj / (T(2) * ljj);             // reverse of the square root
      }
    }
    __syncthreads();
  }
}

}  // namespace hb
