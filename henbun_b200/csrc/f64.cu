// float64 at any size: the fp64 GEMM (DMMA tensor cores), the blocked Cholesky and its reverse mode on it, and the whole
// ELBO + gradient (+ TF-1 Adam) step of the variational GP regression graph as a chain of kernels -- the reference's
// float_type = float64 (henbunrc:7) beyond the n <= 112 of the one-CTA kernel (gp_small.cu).
//
//   GEMM        mma.sync.m16n8k16 f64 (DMMA.8x8x4 in SASS on sm_100a; tcgen05 has no f64 kind).  64 x 64 CTA tiles, or
//               16 x 64 when M <= 16 (the S-row products F = Z L^T, W = R L).  Triangular operand masks narrow the k range
//               a tile visits; a lower-trapezoid output skips the tiles above the diagonal.  Small outputs with long K
//               split K over CTAs into a workspace and sum the partial tiles in a fixed order (deterministic).
//   Cholesky    the column recursion of linalg.cu (potrf_cols / chol_rev_cols) on one stream, 64-column leaves: a
//               64 x 64 double block (32 KB) is factored / reversed column by column in shared memory (tmath.cuh), the
//               panel below it is solved by substitution -- no explicit inverse, so no digits are lost on the
//               ill-conditioned Gram matrices fp64 is chosen for.
#include "../../include/henbun_b200.h"
#include "gemm.cuh"
#include "f64.cuh"
#include "kernels.cuh"
#include "tmath.cuh"
#include <algorithm>

namespace hb {

namespace {

inline cudaStream_t S_(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ------------------------------------------------------------------------------------------------------------------
// fp64 GEMM:  C[M,N] = alpha op(A) op(B) + beta C,  masks as GemmParams (gemm.cuh)
// ------------------------------------------------------------------------------------------------------------------
struct G64 {
  const double* A; long long lda; int transA, a_tri;
  const double* B; long long ldb; int transB, b_tri;
  double* C; long long ldc; int c_tri;
  int M, N, K;
  double alpha, beta;
  double* part;        // split-K partial tiles [splits][M][N] (nullptr: one split)
  int kchunk;          // k range per split (multiple of BK)
};

constexpr int BK = 16;

__device__ __forceinline__ bool keep_a(int tri, int m, int k) {
  switch (tri) {
    case 1: return k <= m;
    case 2: return k >= m;
    case 3: return k > m;
    case 4: return k < m;
    default: return true;
  }
}
__device__ __forceinline__ bool keep_b(int tri, int k, int n) {
  switch (tri) {
    case 1: return n <= k;
    case 2: return n >= k;
    case 3: return n > k;
    case 4: return n < k;
    default: return true;
  }
}

// the k range [kb, ke) a tile of rows [m0, m0 + bm) and columns [n0, n0 + bn) can see through the operand masks
__host__ __device__ inline void tile_k_range(const G64& p, int m0, int bm, int n0, int bn, int& kb, int& ke) {
  kb = 0; ke = p.K;
  switch (p.a_tri) {
    case 1: ke = min(ke, m0 + bm); break;
    case 2: kb = max(kb, m0); break;
    case 3: kb = max(kb, m0 + 1); break;
    case 4: ke = min(ke, m0 + bm - 1); break;
    default: break;
  }
  switch (p.b_tri) {
    case 1: kb = max(kb, n0); break;
    case 2: ke = min(ke, n0 + bn); break;
    case 3: ke = min(ke, n0 + bn - 1); break;
    case 4: kb = max(kb, n0 + 1); break;
    default: break;
  }
}

__device__ __forceinline__ void dmma16816(double (&c)[4], const double (&a)[8], const double (&b)[4]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, {%12,%13,%14,%15}, "
      "{%0,%1,%2,%3};"
      : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
      : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(a[4]), "d"(a[5]), "d"(a[6]), "d"(a[7]), "d"(b[0]), "d"(b[1]),
        "d"(b[2]), "d"(b[3]));
}

// CTA tile BM x BN, warp tile WM x WN (WM multiple of 16, WN of 8).  Shared tiles are k-major with a leading dimension
// of 4 mod 16 doubles: the fragment reads (k = tig + 4 i, row = g) of a half-warp hit 16 different bank pairs.
template <int BM, int BN, int WM, int WN>
struct Tile {
  static constexpr int NT = (BM / WM) * (BN / WN) * 32;
  static constexpr int LDA = BM + 4, LDB = BN + 4;
  static constexpr int LA = BM * BK / NT, LB = BN * BK / NT;   // elements each thread stages per k-tile
  static constexpr int MI = WM / 16, NJ = WN / 8;
};

template <int BM, int BN, int WM, int WN>
__global__ void __launch_bounds__(Tile<BM, BN, WM, WN>::NT) gemm_f64_kernel(const G64 p) {
  using T = Tile<BM, BN, WM, WN>;
  __shared__ __align__(16) double As[2][BK * T::LDA];
  __shared__ __align__(16) double Bs[2][BK * T::LDB];
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  if (p.c_tri && n0 > m0 + BM - 1) return;               // entirely above the diagonal
  int kb, ke;
  tile_k_range(p, m0, BM, n0, BN, kb, ke);
  if (p.part) {                                          // this CTA's share of the k range
    const int s0 = kb + blockIdx.z * p.kchunk;
    ke = min(ke, s0 + p.kchunk);
    kb = s0;
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tig = lane & 3;
  const int wm0 = (warp / (BN / WN)) * WM, wn0 = (warp % (BN / WN)) * WN;

  double ra[T::LA], rb[T::LB];
  auto load = [&](int k0) {
#pragma unroll
    for (int l = 0; l < T::LA; ++l) {
      const int idx = tid + l * T::NT;
      const int m = p.transA ? idx % BM : idx / BK, k = p.transA ? idx / BM : idx % BK;
      const int gm = m0 + m, gk = k0 + k;
      double v = 0.0;
      if (gm < p.M && gk < ke && keep_a(p.a_tri, gm, gk))
        v = p.transA ? p.A[(long long)gk * p.lda + gm] : p.A[(long long)gm * p.lda + gk];
      ra[l] = v;
    }
#pragma unroll
    for (int l = 0; l < T::LB; ++l) {
      const int idx = tid + l * T::NT;
      const int n = p.transB ? idx / BK : idx % BN, k = p.transB ? idx % BK : idx / BN;
      const int gn = n0 + n, gk = k0 + k;
      double v = 0.0;
      if (gn < p.N && gk < ke && keep_b(p.b_tri, gk, gn))
        v = p.transB ? p.B[(long long)gn * p.ldb + gk] : p.B[(long long)gk * p.ldb + gn];
      rb[l] = v;
    }
  };
  auto store = [&](int buf) {
#pragma unroll
    for (int l = 0; l < T::LA; ++l) {
      const int idx = tid + l * T::NT;
      const int m = p.transA ? idx % BM : idx / BK, k = p.transA ? idx / BM : idx % BK;
      As[buf][k * T::LDA + m] = ra[l];
    }
#pragma unroll
    for (int l = 0; l < T::LB; ++l) {
      const int idx = tid + l * T::NT;
      const int n = p.transB ? idx / BK : idx % BN, k = p.transB ? idx % BK : idx / BN;
      Bs[buf][k * T::LDB + n] = rb[l];
    }
  };

  double acc[T::MI][T::NJ][4];
#pragma unroll
  for (int i = 0; i < T::MI; ++i)
#pragma unroll
    for (int j = 0; j < T::NJ; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.0;

  if (kb < ke) {
    load(kb);
    store(0);
    __syncthreads();
    int buf = 0;
    for (int k0 = kb; k0 < ke; k0 += BK) {
      const bool more = k0 + BK < ke;
      if (more) load(k0 + BK);                           // global loads in flight behind the MMAs of this k-tile
      const double* as = As[buf];
      const double* bs = Bs[buf];
      double af[T::MI][8], bf[T::NJ][4];
#pragma unroll
      for (int i = 0; i < T::MI; ++i)
#pragma unroll
        for (int q = 0; q < 8; ++q) af[i][q] = as[((q >> 1) * 4 + tig) * T::LDA + wm0 + i * 16 + g + (q & 1) * 8];
#pragma unroll
      for (int j = 0; j < T::NJ; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) bf[j][q] = bs[(q * 4 + tig) * T::LDB + wn0 + j * 8 + g];
#pragma unroll
      for (int i = 0; i < T::MI; ++i)
#pragma unroll
        for (int j = 0; j < T::NJ; ++j) dmma16816(acc[i][j], af[i], bf[j]);
      if (more) {
        store(buf ^ 1);
        __syncthreads();
        buf ^= 1;
      }
    }
  }

#pragma unroll
  for (int i = 0; i < T::MI; ++i)
#pragma unroll
    for (int j = 0; j < T::NJ; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int r = m0 + wm0 + i * 16 + g + (q >> 1) * 8, c = n0 + wn0 + j * 8 + 2 * tig + (q & 1);
        if (r >= p.M || c >= p.N) continue;
        if (p.part) {
          p.part[((long long)blockIdx.z * p.M + r) * p.N + c] = acc[i][j][q];
        } else if (!(p.c_tri && c > r)) {
          double* cp = p.C + (long long)r * p.ldc + c;
          *cp = p.alpha * acc[i][j][q] + (p.beta != 0.0 ? p.beta * *cp : 0.0);
        }
      }
}

// C = alpha * (sum of the partial tiles, in split order) + beta C
__global__ void splitk_reduce_f64_kernel(const G64 p, int splits) {
  const long long total = (long long)p.M * p.N;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(e / p.N), c = (int)(e % p.N);
    if (p.c_tri && c > r) continue;
    double s = 0.0;
    for (int z = 0; z < splits; ++z) s += p.part[(long long)z * total + e];
    double* cp = p.C + (long long)r * p.ldc + c;
    *cp = p.alpha * s + (p.beta != 0.0 ? p.beta * *cp : 0.0);
  }
}

template <int BM, int BN, int WM, int WN>
int launch_gemm_f64(G64 p, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int gx = cdiv(p.N, BN), gy = cdiv(p.M, BM);
  // the widest k range any tile sees (masks only narrow it)
  int kb, ke;
  G64 q = p; q.a_tri = 0; q.b_tri = 0;
  tile_k_range(q, 0, BM, 0, BN, kb, ke);
  const int klen = ke - kb;
  int splits = 1;
  const long long tiles = (long long)gx * gy;
  if (ws && tiles < 74 && klen >= 1024) {                // small output, long K: spread K over about two waves of CTAs
    splits = (int)std::min<long long>(std::min(32, klen / 256), (296 + tiles - 1) / tiles);
    while (splits > 1 && (size_t)splits * p.M * p.N * sizeof(double) > ws_bytes) --splits;
  }
  if (splits > 1) {
    p.part = reinterpret_cast<double*>(ws);
    p.kchunk = (cdiv(klen, splits) + BK - 1) / BK * BK;
    splits = cdiv(klen, p.kchunk);
  }
  gemm_f64_kernel<BM, BN, WM, WN><<<dim3(gx, gy, splits), Tile<BM, BN, WM, WN>::NT, 0, st>>>(p);
  HB_CHECK_LAUNCH();
  if (splits > 1) {
    const long long total = (long long)p.M * p.N;
    splitk_reduce_f64_kernel<<<(int)std::min<long long>((total + 255) / 256, 148 * 8), 256, 0, st>>>(p, splits);
    HB_CHECK_LAUNCH();
  }
  return HB_OK;
}

int gemm_f64(const G64& p0, void* ws, size_t ws_bytes, cudaStream_t st) {
  G64 p = p0;
  p.part = nullptr; p.kchunk = 0;
  if (p.M <= 0 || p.N <= 0) return HB_OK;
  if (p.M <= 16) return launch_gemm_f64<16, 64, 16, 16>(p, ws, ws_bytes, st);
  return launch_gemm_f64<64, 64, 32, 32>(p, ws, ws_bytes, st);
}

int check_g64(const G64& p) {
  if (p.M < 0 || p.N < 0 || p.K < 0) return HB_ERR_ARG;
  if (p.transA < 0 || p.transA > 1 || p.transB < 0 || p.transB > 1 || p.a_tri < 0 || p.a_tri > 4 || p.b_tri < 0 ||
      p.b_tri > 4 || p.c_tri < 0 || p.c_tri > 1)
    return HB_ERR_ARG;
  if (p.M == 0 || p.N == 0) return HB_OK;
  if (!p.C || p.ldc < p.N) return HB_ERR_ARG;
  if (p.K > 0) {
    if (!p.A || !p.B) return HB_ERR_ARG;
    if (p.lda < (p.transA ? p.M : p.K) || p.ldb < (p.transB ? p.K : p.N)) return HB_ERR_ARG;
  }
  return HB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// leaves: one 64 x 64 diagonal block in shared memory
// ------------------------------------------------------------------------------------------------------------------
constexpr int NB64 = 64;
constexpr int LD64 = NB64 + 1;                           // odd leading dimension: conflict-free column walks
constexpr int LEAF64_THREADS = 512;
constexpr size_t kLeaf64Smem = (size_t)(2 * NB64 * LD64 + NB64) * sizeof(double);

__global__ void __launch_bounds__(LEAF64_THREADS) potrf_leaf_f64_kernel(double* A, long long lda, int w, int* err, int err_base) {
  extern __shared__ __align__(16) unsigned char sm64[];
  double* L = reinterpret_cast<double*>(sm64);
  double* colv = L + NB64 * LD64;
  __shared__ int sh_bad;
  for (int e = threadIdx.x; e < w * w; e += LEAF64_THREADS) {
    const int i = e / w, j = e % w;
    if (j <= i) L[i * LD64 + j] = A[(long long)i * lda + j];
  }
  __syncthreads();
  const int bad = potrf_cols_smem<double, LEAF64_THREADS>(L, LD64, w, colv, &sh_bad);
  if (threadIdx.x == 0 && bad != 0 && err) atomicCAS(err, 0, err_base + bad);
  for (int e = threadIdx.x; e < w * w; e += LEAF64_THREADS) {
    const int i = e / w, j = e % w;
    if (j <= i) A[(long long)i * lda + j] = L[i * LD64 + j];
  }
}

// G (lower, dObj/dL of the block) -> dObj/dK of the block in the symmetric-input convention (off-diagonals halved)
__global__ void __launch_bounds__(LEAF64_THREADS) chol_rev_leaf_f64_kernel(const double* Lg, long long ldl, double* Gg, long long ldg,
                                                                         int w) {
  extern __shared__ __align__(16) unsigned char sm64[];
  double* L = reinterpret_cast<double*>(sm64);
  double* G = L + NB64 * LD64;
  double* colv = G + NB64 * LD64;
  for (int e = threadIdx.x; e < w * w; e += LEAF64_THREADS) {
    const int i = e / w, j = e % w;
    if (j <= i) {
      L[i * LD64 + j] = Lg[(long long)i * ldl + j];
      G[i * LD64 + j] = Gg[(long long)i * ldg + j];
    }
  }
  __syncthreads();
  potrf_rev_cols_smem<double, LEAF64_THREADS>(L, G, LD64, w, colv);
  for (int e = threadIdx.x; e < w * w; e += LEAF64_THREADS) {
    const int i = e / w, j = e % w;
    if (j <= i) Gg[(long long)i * ldg + j] = (i == j) ? G[i * LD64 + j] : 0.5 * G[i * LD64 + j];
  }
}

// Panel solve by substitution, one thread per row: TRANS: Bp <- alpha Bp D^-T (x_j = (b_j - sum_{k<j} x_k D_jk) / D_jj),
// else Bp <- alpha Bp D^-1 (x_j = (b_j - sum_{k>j} x_k D_kj) / D_jj, j descending).  D: w x w lower, w <= 64.
constexpr int PS64_ROWS = 128;
constexpr size_t kPanel64Smem = (size_t)(NB64 * PS64_ROWS + NB64 * LD64) * sizeof(double);

template <bool TRANS>
__global__ void __launch_bounds__(PS64_ROWS) panel_solve_f64_kernel(const double* D, long long ldd, double* Bp, long long ldb, int m,
                                                                   int w, double alpha) {
  extern __shared__ __align__(16) unsigned char sm64[];
  double* Xs = reinterpret_cast<double*>(sm64);          // Xs[k * ROWS + r]: row r of the panel as a column
  double* Ds = Xs + NB64 * PS64_ROWS;
  const int r0 = blockIdx.x * PS64_ROWS, rows = min(PS64_ROWS, m - r0), tid = threadIdx.x;
  for (int e = tid; e < w * w; e += PS64_ROWS) {
    const int i = e / w, j = e % w;
    if (j <= i) Ds[i * LD64 + j] = D[(long long)i * ldd + j];
  }
  for (int e = tid; e < rows * w; e += PS64_ROWS) {
    const int r = e / w, k = e % w;
    Xs[k * PS64_ROWS + r] = alpha * Bp[(long long)(r0 + r) * ldb + k];
  }
  __syncthreads();
  if (tid < rows) {
    double* x = Xs + tid;
    if (TRANS) {
      for (int j = 0; j < w; ++j) {
        const double* dj = Ds + j * LD64;
        double a0 = x[j * PS64_ROWS], a1 = 0.0;
        int k = 0;
        for (; k + 1 < j; k += 2) {
          a0 -= x[k * PS64_ROWS] * dj[k];
          a1 -= x[(k + 1) * PS64_ROWS] * dj[k + 1];
        }
        if (k < j) a0 -= x[k * PS64_ROWS] * dj[k];
        x[j * PS64_ROWS] = (a0 + a1) / dj[j];
      }
    } else {
      for (int j = w - 1; j >= 0; --j) {
        double a0 = x[j * PS64_ROWS], a1 = 0.0;
        int k = j + 1;
        for (; k + 1 < w; k += 2) {
          a0 -= x[k * PS64_ROWS] * Ds[k * LD64 + j];
          a1 -= x[(k + 1) * PS64_ROWS] * Ds[(k + 1) * LD64 + j];
        }
        if (k < w) a0 -= x[k * PS64_ROWS] * Ds[k * LD64 + j];
        x[j * PS64_ROWS] = (a0 + a1) / Ds[j * LD64 + j];
      }
    }
  }
  __syncthreads();
  for (int e = tid; e < rows * w; e += PS64_ROWS) {
    const int r = e / w, k = e % w;
    Bp[(long long)(r0 + r) * ldb + k] = Xs[k * PS64_ROWS + r];
  }
}

}  // namespace

int ensure_attrs64() {
  static bool done = false;
  if (done) return HB_OK;
  if (cudaFuncSetAttribute(chol_rev_leaf_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLeaf64Smem) != cudaSuccess ||
      cudaFuncSetAttribute(potrf_leaf_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLeaf64Smem) != cudaSuccess ||
      cudaFuncSetAttribute(panel_solve_f64_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPanel64Smem) != cudaSuccess ||
      cudaFuncSetAttribute(panel_solve_f64_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPanel64Smem) != cudaSuccess)
    return HB_ERR_CUDA;
  done = true;
  return HB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// the column recursion (linalg.cu: potrf_cols / chol_rev_cols) with every product on the fp64 GEMM
// ------------------------------------------------------------------------------------------------------------------
namespace {

inline int split64(int w) { return ((cdiv(w, NB64) + 1) / 2) * NB64; }

}  // namespace

int gemm64(const Ctx64& c, const double* A, long long lda, int transA, int a_tri, const double* B, long long ldb, int transB,
           int b_tri, double* C, long long ldc, int c_tri, int M, int N, int K, double alpha, double beta) {
  G64 p{A, lda, transA, a_tri, B, ldb, transB, b_tri, C, ldc, c_tri, M, N, K, alpha, beta, nullptr, 0};
  return gemm_f64(p, c.ws, c.ws_bytes, c.st);
}

namespace {

int panel_solve64(const Ctx64& c, const double* D, long long ldd, double* Bp, long long ldb, int m, int w, bool trans, double alpha) {
  if (trans) panel_solve_f64_kernel<true><<<cdiv(m, PS64_ROWS), PS64_ROWS, kPanel64Smem, c.st>>>(D, ldd, Bp, ldb, m, w, alpha);
  else panel_solve_f64_kernel<false><<<cdiv(m, PS64_ROWS), PS64_ROWS, kPanel64Smem, c.st>>>(D, ldd, Bp, ldb, m, w, alpha);
  HB_CHECK_LAUNCH();
  return HB_OK;
}

}  // namespace

int potrf_cols64(const Ctx64& c, double* A, long long lda, int c0, int w, int n) {
  double* D = A + (long long)c0 * lda + c0;
  if (w <= NB64) {
    potrf_leaf_f64_kernel<<<1, LEAF64_THREADS, kLeaf64Smem, c.st>>>(D, lda, w, c.err, c0);
    HB_CHECK_LAUNCH();
    const int below = n - (c0 + w);
    return below > 0 ? panel_solve64(c, D, lda, D + (long long)w * lda, lda, below, w, true, 1.0) : HB_OK;
  }
  const int w1 = split64(w), w2 = w - w1;
  HB_TRY(potrf_cols64(c, A, lda, c0, w1, n));
  // A[c0+w1 .. n, c0+w1 .. c0+w) -= L[c0+w1 .. n, c0 .. c0+w1) L[c0+w1 .. c0+w, c0 .. c0+w1)^T  (lower trapezoid)
  double* P = A + (long long)(c0 + w1) * lda + c0;
  HB_TRY(gemm64(c, P, lda, 0, 0, P, lda, 1, 0, P + w1, lda, 1, n - (c0 + w1), w2, w1, -1.0, 1.0));
  return potrf_cols64(c, A, lda, c0 + w1, w2, n);
}

// rev_cols(c0, w) owns G[c0 .. n, c0 .. c0+w): on entry dObj/dL with every contribution of the columns to the right
// applied, on exit dObj/dK in the symmetric-input convention.  The steps are those of linalg.cu's chol_rev_cols.
int chol_rev_cols64(const Ctx64& c, const double* L, long long ldl, double* G, long long ldg, int c0, int w, int n) {
  double* GD = G + (long long)c0 * ldg + c0;
  const double* LD = L + (long long)c0 * ldl + c0;
  if (w <= NB64) {
    const int below = n - (c0 + w);
    if (below > 0) {
      double* Gp = GD + (long long)w * ldg;
      const double* Lp = LD + (long long)w * ldl;
      HB_TRY(panel_solve64(c, LD, ldl, Gp, ldg, below, w, false, 0.5));               // S = G_below L_DD^-1 / 2
      HB_TRY(gemm64(c, Gp, ldg, 1, 0, Lp, ldl, 0, 0, GD, ldg, 1, w, w, below, -2.0, 1.0));   // G_DD -= 2 tril(S^T L_below)
    }
    chol_rev_leaf_f64_kernel<<<1, LEAF64_THREADS, kLeaf64Smem, c.st>>>(LD, ldl, GD, ldg, w);
    HB_CHECK_LAUNCH();
    return HB_OK;
  }
  const int w1 = split64(w), w2 = w - w1;
  const int r1 = c0 + w1, rb = c0 + w, nb = n - rb;
  HB_TRY(chol_rev_cols64(c, L, ldl, G, ldg, r1, w2, n));
  double* G_T_left = G + (long long)r1 * ldg + c0;
  const double* L_T_left = L + (long long)r1 * ldl + c0;
  if (nb > 0) {
    const double* G_R_right = G + (long long)rb * ldg + r1;
    double* G_R_left = G + (long long)rb * ldg + c0;
    const double* L_R_left = L + (long long)rb * ldl + c0;
    HB_TRY(gemm64(c, G_R_right, ldg, 0, 0, L_T_left, ldl, 0, 0, G_R_left, ldg, 0, nb, w1, w2, -2.0, 1.0));
    HB_TRY(gemm64(c, G_R_right, ldg, 1, 0, L_R_left, ldl, 0, 0, G_T_left, ldg, 0, w2, w1, nb, -2.0, 1.0));
  }
  // G[T, left] -= 2 sym(G[T, right]) L[T, left], sym from the lower triangle: its lower part, then its strict upper part
  const double* G_TT = G + (long long)r1 * ldg + r1;
  HB_TRY(gemm64(c, G_TT, ldg, 0, 1, L_T_left, ldl, 0, 0, G_T_left, ldg, 0, w2, w1, w2, -2.0, 1.0));
  HB_TRY(gemm64(c, G_TT, ldg, 1, 3, L_T_left, ldl, 0, 0, G_T_left, ldg, 0, w2, w1, w2, -2.0, 1.0));
  return chol_rev_cols64(c, L, ldl, G, ldg, c0, w1, n);
}

namespace {

size_t potrf64_ws_bytes(int n) { return n > NB64 ? kSplitWsBytes + 256 : 0; }

int make_ctx64(Ctx64& c, int n, void* ws, size_t ws_bytes, int* err, cudaStream_t st) {
  if (ws_bytes < potrf64_ws_bytes(n) || (potrf64_ws_bytes(n) && !ws)) return HB_ERR_WORKSPACE;
  c.st = st; c.err = err;
  c.ws = ws ? reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255)) : nullptr;
  c.ws_bytes = ws ? ws_bytes - ((char*)c.ws - (char*)ws) : 0;
  return ensure_attrs64();
}

int potrf_lower_f64(double* A, long long lda, int n, void* ws, size_t ws_bytes, int* err, cudaStream_t st) {
  if (n < 0 || (n > 0 && (!A || lda < n))) return HB_ERR_ARG;
  if (n == 0) return HB_OK;
  Ctx64 c;
  HB_TRY(make_ctx64(c, n, ws, ws_bytes, err, st));
  return potrf_cols64(c, A, lda, 0, n, n);
}

int potrf_lower_bwd_f64(const double* L, long long ldl, double* G, long long ldg, int n, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (n < 0 || (n > 0 && (!L || !G || ldl < n || ldg < n))) return HB_ERR_ARG;
  if (n == 0) return HB_OK;
  Ctx64 c;
  HB_TRY(make_ctx64(c, n, ws, ws_bytes, nullptr, st));
  return chol_rev_cols64(c, L, ldl, G, ldg, 0, n, n);
}

// ------------------------------------------------------------------------------------------------------------------
// the rest of the GP step in double (the formulas of gp_small.cu's step, as separate kernels)
// sc: [0] scale s, [1] k_var, [2] var, [3] amp = sqrt(k_var) s, [4] loglik, [5] sum E^2, [6] sum E Fraw, [7] kl, [8..) ell
// ------------------------------------------------------------------------------------------------------------------
__global__ void gp64_prep_kernel(const double* p_scale, const double* p_ell, int n_ell, const double* p_kvar, const double* p_var,
                                 double* sc) {
  if (threadIdx.x == 0) {
    const double s = t_softplus<double>(*p_scale) + 1e-6, kv = t_softplus<double>(*p_kvar) + 1e-6;
    sc[0] = s; sc[1] = kv; sc[2] = t_softplus<double>(*p_var) + 1e-6; sc[3] = sqrt(kv) * s;
  }
  for (int d = threadIdx.x; d < n_ell; d += blockDim.x) sc[SC_ELL + d] = t_softplus<double>(p_ell[d]) + 1e-6;
}

}  // namespace

// K = rbf(X) + jitter I, 32 x 32 tiles on and below the diagonal
__global__ void gp64_gram_kernel(const double* X, int n, int D, const double* sc, int n_ell, double jitter, double* K) {
  if (blockIdx.x > blockIdx.y) return;
  const double* ell = sc + SC_ELL;
  const int j = blockIdx.x * 32 + threadIdx.x;
  for (int i = blockIdx.y * 32 + threadIdx.y; i < min(n, (int)blockIdx.y * 32 + 32); i += blockDim.y) {
    if (j > i || j >= n) continue;
    double r2 = 0.0;
    for (int d = 0; d < D; ++d) {
      const double df = (X[(long long)i * D + d] - X[(long long)j * D + d]) / ell[n_ell == 1 ? 0 : d];
      r2 += df * df;
    }
    K[(long long)i * n + j] = exp(-0.5 * r2) + (i == j ? jitter : 0.0);
  }
}

// U = eps (or the library's Philox stream widened to double, as gp_small.cu draws it); Z = mu + exp(omega) U, or mu for the
// full-rank q (its U Lq^T follows as a product)
__global__ void gp64_sample_kernel(const double* p_mu, const double* p_sq, int full, int n, int S, const double* eps,
                                   unsigned long long seed, unsigned long long offset, double* U, double* Z) {
  const long long total = (long long)S * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e % n);
    const double u = eps ? eps[e] : (double)philox_normal_at(seed, offset, (unsigned long long)e);
    U[e] = u;
    Z[e] = full ? p_mu[i] : p_mu[i] + exp(p_sq[i]) * u;
  }
}

// kl = -0.5 sum_{s,i} (logdet_i + u^2 - z^2): one CTA, fixed order
__global__ void __launch_bounds__(RED_THREADS) gp64_kl_kernel(const double* p_sq, int full, int n, int S, const double* U,
                                                            const double* Z, double* sc) {
  __shared__ double red[32];
  double v[1] = {0.0};
  for (long long e = threadIdx.x; e < (long long)S * n; e += RED_THREADS) {
    const int i = (int)(e % n);
    double logdet;
    if (full) { const double l = p_sq[(long long)i * n + i]; logdet = log(l * l); }
    else logdet = 2.0 * p_sq[i];
    v[0] += logdet + U[e] * U[e] - Z[e] * Z[e];
  }
  block_sum<1>(v, red);
  if (threadIdx.x == 0) sc[7] = -0.5 * v[0];
}

namespace {

// log-likelihood of Y under F = amp Fraw, sum E^2, sum E Fraw, residual R = E / var / S: one CTA, fixed order
__global__ void __launch_bounds__(RED_THREADS) gp64_loglik_kernel(const double* Fraw, const double* Y, int n, int S, double* R,
                                                                double* sc) {
  __shared__ double red[3 * 32];
  const double amp = sc[3], var = sc[2], lv = log(var), invS = 1.0 / (double)S;
  double v[3] = {0.0, 0.0, 0.0};
  for (long long e = threadIdx.x; e < (long long)S * n; e += RED_THREADS) {
    const double fr = Fraw[e], E = Y[e % n] - amp * fr;
    v[0] += -0.9189385332046727 - 0.5 * lv - 0.5 * E * E / var;
    v[1] += E * E;
    v[2] += E * fr;
    R[e] = E / var * invS;
  }
  block_sum<3>(v, red);
  if (threadIdx.x == 0) { sc[4] = v[0]; sc[5] = v[1]; sc[6] = v[2]; }
}

}  // namespace

// z-bar = amp W - Z / S  (W = R L)
__global__ void gp64_zbar_kernel(const double* W, const double* Z, const double* sc, long long total, int S, double* Zb) {
  const double amp = sc[3], invS = 1.0 / (double)S;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x)
    Zb[e] = amp * W[e] - Z[e] * invS;
}

// sampler backward: g_mu = sum_s z-bar; mean-field g_omega = exp(omega) sum_s z-bar u + 1; full rank: the diagonal's
// 1 / Lq_ii is added to the tril(z-bar^T U) a product already wrote
__global__ void gp64_sampler_bwd_kernel(const double* Zb, const double* U, const double* p_sq, int full, int n, int S, double* g_mu,
                                        double* g_sq) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    double gm = 0.0, go = 0.0;
    for (int s = 0; s < S; ++s) {
      const double zt = Zb[(long long)s * n + k];
      gm += zt;
      if (!full) go += zt * U[(long long)s * n + k];
    }
    g_mu[k] = gm;
    if (!full) g_sq[k] = go * exp(p_sq[k]) + 1.0;
    else g_sq[(long long)k * n + k] += 1.0 / p_sq[(long long)k * n + k];
  }
}

// partial sums of d ELBO / d ell over the strict lower triangle of the symmetric-convention K-bar (each entry counts twice):
// block b takes rows b, b + gridDim.x, ...; red[b * n_ell + d]
__global__ void __launch_bounds__(256) gp64_gram_bwd_kernel(const double* G, const double* X, int n, int D, const double* sc, int n_ell,
                                                          double* red) {
  __shared__ double sred[8 * 32];
  const double* ell = sc + SC_ELL;
  for (int d0 = 0; d0 < n_ell; d0 += 8) {
    double v[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
      for (int j = threadIdx.x; j < i; j += blockDim.x) {
        double r2 = 0.0;
        for (int d = 0; d < D; ++d) {
          const double df = (X[(long long)i * D + d] - X[(long long)j * D + d]) / ell[n_ell == 1 ? 0 : d];
          r2 += df * df;
        }
        const double gk = 2.0 * G[(long long)i * n + j] * exp(-0.5 * r2);
        if (n_ell == 1) {
          v[0] += gk * r2;
        } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            if (d0 + q < n_ell) {
              const double df = (X[(long long)i * D + d0 + q] - X[(long long)j * D + d0 + q]) / ell[d0 + q];
              v[q] += gk * df * df;
            }
          }
        }
      }
    }
    block_sum<8>(v, sred);
    if (threadIdx.x == 0)
      for (int q = 0; q < 8 && d0 + q < n_ell; ++q) red[(long long)blockIdx.x * n_ell + d0 + q] = v[q];
  }
}

namespace {

// lengthscale gradient (K-bar came without the factor amp: the reverse-mode Cholesky is linear in L-bar), scalar chain rules,
// the ELBO
__global__ void gp64_scalar_bwd_kernel(const double* sc, const double* red, int nblk, int n_ell, int n, int S, const double* p_scale,
                                       const double* p_ell, const double* p_kvar, const double* p_var, double* g_scale, double* g_ell,
                                       double* g_kvar, double* g_var, double* out4) {
  const double amp = sc[3];
  for (int d = threadIdx.x; d < n_ell; d += blockDim.x) {
    double t = 0.0;
    for (int b = 0; b < nblk; ++b) t += red[(long long)b * n_ell + d];
    g_ell[d] = amp * t / sc[SC_ELL + d] * t_sigmoid<double>(p_ell[d]);
  }
  if (threadIdx.x == 0) {
    const double sq = sc[0], kv = sc[1], v = sc[2], ll = sc[4], sumE2 = sc[5], sumEF = sc[6], kl = sc[7];
    const double invS = 1.0 / (double)S;
    const double ga = invS * sumEF / v;
    const double gv = invS * (-0.5 * (double)S * n / v + 0.5 * sumE2 / (v * v));
    *g_scale = ga * sqrt(kv) * t_sigmoid<double>(*p_scale);
    *g_kvar = ga * sq / (2.0 * sqrt(kv)) * t_sigmoid<double>(*p_kvar);
    *g_var = gv * t_sigmoid<double>(*p_var);
    out4[0] = (ll - kl) * invS; out4[1] = ll; out4[2] = kl; out4[3] = 0.0;
  }
}

}  // namespace

// TF-1 Adam on -ELBO (model.py:206,220); the strict upper triangle of a full-rank q_sqrt never moves
__global__ void gp64_adam_kernel(double* params, const double* grads, double* m, double* v, long long npar, int n, int full,
                                 const int* step_dev, int step_host, double lr, double b1, double b2, double eps, double grad_scale) {
  const int t = step_dev ? *step_dev : step_host;
  const double lr_t = lr * sqrt(1.0 - pow(b2, (double)t)) / (1.0 - pow(b1, (double)t));
  const long long nq = full ? (long long)n * n : n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < npar; i += (long long)gridDim.x * blockDim.x) {
    if (full && i >= n && i < n + nq) {
      const long long q = i - n;
      if (q % n > q / n) continue;
    }
    const double g = grad_scale * grads[i];
    const double mm = b1 * m[i] + (1.0 - b1) * g;
    const double vv = b2 * v[i] + (1.0 - b2) * g * g;
    m[i] = mm; v[i] = vv;
    params[i] -= lr_t * mm / (sqrt(vv) + eps);
  }
}

namespace {

struct Gp64Layout {
  size_t off_K, off_G, off_Z, off_F, off_R, off_W, off_U, off_sc, off_red, off_potrf, total;
};

Gp64Layout gp64_layout(const hb_gp_config& c) {
  Gp64Layout L{};
  const size_t nn = (size_t)c.n * c.n * sizeof(double), sn = (size_t)c.S * c.n * sizeof(double);
  size_t o = 0;
  L.off_K = o; o += align256(nn);
  L.off_G = o; o += align256(nn);
  L.off_Z = o; o += align256(sn);
  L.off_F = o; o += align256(sn);
  L.off_R = o; o += align256(sn);
  L.off_W = o; o += align256(sn);
  L.off_U = o; o += align256(sn);
  L.off_sc = o; o += align256((size_t)(SC_ELL + c.n_ell) * sizeof(double));
  L.off_red = o; o += align256((size_t)kGramBwdBlocks * c.n_ell * sizeof(double));
  L.off_potrf = o; o += align256(kSplitWsBytes);
  L.total = o;
  return L;
}

bool gp64_forwards_to_small(const hb_gp_config& c) { return c.n <= gp_small_max_n(1) && opt_small_gp_kernel(); }

int gp_elbo_step_f64_chain(const hb_gp_config& c, const double* X, const double* Y, double* params, const double* eps,
                           double* grads, double* out4, double* adam_m, double* adam_v, const hb_adam_config* adam, void* ws,
                           size_t ws_bytes, int* err_flag, cudaStream_t st) {
  const Gp64Layout L = gp64_layout(c);
  if (!ws || ws_bytes < L.total + 256) return HB_ERR_WORKSPACE;
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  double* K = reinterpret_cast<double*>(base + L.off_K);
  double* G = reinterpret_cast<double*>(base + L.off_G);
  double* Z = reinterpret_cast<double*>(base + L.off_Z);
  double* F = reinterpret_cast<double*>(base + L.off_F);
  double* R = reinterpret_cast<double*>(base + L.off_R);
  double* W = reinterpret_cast<double*>(base + L.off_W);
  double* U = reinterpret_cast<double*>(base + L.off_U);
  double* sc = reinterpret_cast<double*>(base + L.off_sc);
  double* red = reinterpret_cast<double*>(base + L.off_red);
  Ctx64 cx{st, err_flag, base + L.off_potrf, kSplitWsBytes};
  HB_TRY(ensure_attrs64());

  const int n = c.n, S = c.S, full = c.q_fullrank;
  const size_t nq = full ? (size_t)n * n : (size_t)n;
  const double* p_mu = params;
  const double* p_sq = params + n;
  const double* p_scale = p_sq + nq;
  const double* p_ell = p_scale + 1;
  const double* p_kvar = p_ell + c.n_ell;
  const double* p_var = p_kvar + 1;
  double* g_mu = grads;
  double* g_sq = grads + n;
  double* g_scale = g_sq + nq;
  double* g_ell = g_scale + 1;
  double* g_kvar = g_ell + c.n_ell;
  double* g_var = g_kvar + 1;
  const long long Sn = (long long)S * n;
  const int ew_blocks = (int)std::min<long long>((Sn + 255) / 256, 148 * 8);

  gp64_prep_kernel<<<1, 32, 0, st>>>(p_scale, p_ell, c.n_ell, p_kvar, p_var, sc);
  HB_CHECK_LAUNCH();
  gp64_gram_kernel<<<dim3(cdiv(n, 32), cdiv(n, 32)), dim3(32, 8), 0, st>>>(X, n, c.D, sc, c.n_ell, (double)c.jitter, K);
  HB_CHECK_LAUNCH();
  HB_TRY(potrf_cols64(cx, K, n, 0, n, n));

  // sampler + KL
  gp64_sample_kernel<<<ew_blocks, 256, 0, st>>>(p_mu, p_sq, full, n, S, eps, c.seed, c.offset, U, Z);
  HB_CHECK_LAUNCH();
  if (full) HB_TRY(gemm64(cx, U, n, 0, 0, p_sq, n, 1, 2, Z, n, 0, S, n, n, 1.0, 1.0));          // Z += U tril(Lq)^T
  gp64_kl_kernel<<<1, RED_THREADS, 0, st>>>(p_sq, full, n, S, U, Z, sc);
  HB_CHECK_LAUNCH();

  // Fraw = Z L^T, log-likelihood and residual, W = R L, z-bar
  HB_TRY(gemm64(cx, Z, n, 0, 0, K, n, 1, 2, F, n, 0, S, n, n, 1.0, 0.0));
  gp64_loglik_kernel<<<1, RED_THREADS, 0, st>>>(F, Y, n, S, R, sc);
  HB_CHECK_LAUNCH();
  HB_TRY(gemm64(cx, R, n, 0, 0, K, n, 0, 1, W, n, 0, S, n, n, 1.0, 0.0));
  gp64_zbar_kernel<<<ew_blocks, 256, 0, st>>>(W, Z, sc, Sn, S, F);                              // F is free: z-bar
  HB_CHECK_LAUNCH();

  // sampler backward
  if (full) {
    if (cudaMemsetAsync(g_sq, 0, nq * sizeof(double), st) != cudaSuccess) return HB_ERR_CUDA;
    HB_TRY(gemm64(cx, F, n, 1, 0, U, n, 0, 0, g_sq, n, 1, n, n, S, 1.0, 0.0));                  // tril(z-bar^T U)
  }
  gp64_sampler_bwd_kernel<<<cdiv(n, 256), 256, 0, st>>>(F, U, p_sq, full, n, S, g_mu, g_sq);
  HB_CHECK_LAUNCH();

  // L-bar / amp = tril(R^T Z), reverse-mode Cholesky, Gram backward, scalars
  HB_TRY(gemm64(cx, R, n, 1, 0, Z, n, 0, 0, G, n, 1, n, n, S, 1.0, 0.0));
  HB_TRY(chol_rev_cols64(cx, K, n, G, n, 0, n, n));
  gp64_gram_bwd_kernel<<<kGramBwdBlocks, 256, 0, st>>>(G, X, n, c.D, sc, c.n_ell, red);
  HB_CHECK_LAUNCH();
  gp64_scalar_bwd_kernel<<<1, 32, 0, st>>>(sc, red, kGramBwdBlocks, c.n_ell, n, S, p_scale, p_ell, p_kvar, p_var, g_scale, g_ell,
                                           g_kvar, g_var, out4);
  HB_CHECK_LAUNCH();

  if (adam_m) {
    const long long npar = (long long)(n + nq + 3 + c.n_ell);
    gp64_adam_kernel<<<(int)std::min<long long>((npar + 255) / 256, 148 * 8), 256, 0, st>>>(
        params, grads, adam_m, adam_v, npar, n, full, adam->step_dev, adam->step_host, adam->lr, adam->b1, adam->b2, adam->eps,
        adam->grad_scale);
    HB_CHECK_LAUNCH();
  }
  return HB_OK;
}

}  // namespace
}  // namespace hb

using namespace hb;

extern "C" {

int hb_gemm_f64(const double* A, long long lda, int transA, int a_tri, const double* B, long long ldb, int transB, int b_tri,
                double* C, long long ldc, int c_tri, int M, int N, int K, double alpha, double beta, void* ws, size_t ws_bytes,
                void* stream) {
  G64 p{A, lda, transA, a_tri, B, ldb, transB, b_tri, C, ldc, c_tri, M, N, K, alpha, beta, nullptr, 0};
  HB_TRY(check_g64(p));
  if (ws_bytes && !ws) return HB_ERR_WORKSPACE;
  void* w = ws ? reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255)) : nullptr;
  const size_t wb = ws ? (ws_bytes > (size_t)((char*)w - (char*)ws) ? ws_bytes - ((char*)w - (char*)ws) : 0) : 0;
  return gemm_f64(p, wb ? w : nullptr, wb, S_(stream));
}

size_t hb_potrf_f64_workspace_bytes(int n) { return potrf64_ws_bytes(n); }

int hb_potrf_lower_f64(double* A, long long lda, int n, void* ws, size_t ws_bytes, int* err_flag, void* stream) {
  return potrf_lower_f64(A, lda, n, ws, ws_bytes, err_flag, S_(stream));
}

int hb_potrf_lower_bwd_f64(const double* L, long long ldl, double* G, long long ldg, int n, void* ws, size_t ws_bytes, void* stream) {
  return potrf_lower_bwd_f64(L, ldl, G, ldg, n, ws, ws_bytes, S_(stream));
}

size_t hb_gp_elbo_f64_workspace_bytes(const hb_gp_config* cfg) {
  if (!cfg || cfg->n <= 0 || cfg->S <= 0 || cfg->n_ell <= 0) return 0;
  OptScope scope(cfg->opt);
  if (gp64_forwards_to_small(*cfg)) return hb_gp_small_workspace_bytes(cfg, 1);
  return gp64_layout(*cfg).total + 256;
}

int hb_gp_elbo_step_f64(const hb_gp_config* cfg, const double* X, const double* Y, double* params, const double* eps, double* grads,
                        double* out4, double* adam_m, double* adam_v, const hb_adam_config* adam, void* ws, size_t ws_bytes,
                        int* err_flag, void* stream) {
  if (!cfg || !X || !Y || !params || !grads || !out4) return HB_ERR_ARG;
  OptScope scope(cfg->opt);
  const hb_gp_config c = *cfg;
  if (c.n <= 0 || c.D <= 0 || c.D > 32 || c.S <= 0 || (c.n_ell != 1 && c.n_ell != c.D)) return HB_ERR_ARG;
  if (!eps && (c.offset & 3ull)) return HB_ERR_ARG;
  if ((adam_m || adam_v) && (!adam || !adam_m || !adam_v)) return HB_ERR_ARG;
  if (gp64_forwards_to_small(c))
    return hb_gp_small_step_f64(cfg, X, Y, params, eps, grads, out4, adam_m, adam_v, adam, ws, ws_bytes, err_flag, stream);
  return gp_elbo_step_f64_chain(c, X, Y, params, eps, grads, out4, adam_m, adam_v, adam, ws, ws_bytes, err_flag, S_(stream));
}

}  // extern "C"
