// gemm.cu — general row-major GEMM  C = alpha*op(A)*op(B) + beta*C  for the Cholesky trailing
// update (SYRK), the inverse-based TRSM steps, A A^T, A^T f and tril(q_sqrt)^T A.
//   fp64: legacy tensor path  mma.sync.m8n8k4.f64 (DMMA) — tcgen05 has no f64 kind (SURVEY 7.3 #1);
//         the tcgen05 paths live in gemm_tc.cu (int8-sliced fp64 SYRK) and gemm_tf32.cu (3xTF32 fp32 GEMM).
//   fp32: CUDA-core register-tiled kernel with the same tile-shape menu as the DMMA kernel (small / ragged shapes).
// Replaces tf.linalg.matmul call sites: gpflow/models/sgpr.py:205,263, conditionals/util.py:144,157,
// posteriors.py:497,535,539,728,734, and the GEMM inside tf.linalg.cholesky / triangular_solve.
//
// In-place contract used by potrf/trsm: a CTA reads every A/B element it needs before its first
// store to C, so C may alias A when one tile spans n and may alias B when one tile spans m (the shape
// selection keeps BN >= n resp. BM >= m in those cases).
#include "common.cuh"

namespace gpk {

constexpr int GB = 128;  // CTA tile edge (both kernels)

// ------------------------------------------------------------------------------------------------
// shared epilogue
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void atomic_add_t(T* p, T v) { atomicAdd(p, v); }

// ------------------------------------------------------------------------------------------------
// fp64: DMMA m8n8k4, 512 threads, 4x4 warps of 32x32, BK = 16
// ------------------------------------------------------------------------------------------------
constexpr int DK = 16;          // k chunk
constexpr int DS_K = DK + 4;    // row stride of a k-minor tile  [128][20]
constexpr int DS_M = GB + 4;    // row stride of a m-minor tile  [16][132]
constexpr int DTILE = GB * DS_K;  // 2560 doubles >= 16*132 = 2112

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// Loads this thread's share of one operand chunk (ROWS x 16) into registers.
// STORED_KMINOR: global operand is [rows][k] (k contiguous); else [k][rows] (rows contiguous).
// tri: 0 none; 1 = stored matrix is lower triangular (zero where stored_col > stored_row).
template <bool STORED_KMINOR, int ROWS, int NT>
__device__ __forceinline__ void dload(double (&reg)[ROWS * DK / NT], const double* P, int64_t ld, int64_t r0,
                                      int64_t nrows, int64_t k0, int64_t kend, int tid, int tri) {
#pragma unroll
  for (int i = 0; i < ROWS * DK / NT; ++i) {
    const int e = tid + i * NT;
    int rr, kk;
    if (STORED_KMINOR) { kk = e % DK; rr = e / DK; } else { rr = e % ROWS; kk = e / ROWS; }
    const int64_t gr = r0 + rr, gk = k0 + kk;
    double v = 0.0;
    if (gr < nrows && gk < kend) {
      const int64_t srow = STORED_KMINOR ? gr : gk, scol = STORED_KMINOR ? gk : gr;
      if (!(tri && scol > srow)) v = P[srow * ld + scol];
    }
    reg[i] = v;
  }
}

template <bool STORED_KMINOR, int ROWS, int NT>
__device__ __forceinline__ void dstore(const double (&reg)[ROWS * DK / NT], double* __restrict__ S, int tid) {
#pragma unroll
  for (int i = 0; i < ROWS * DK / NT; ++i) {
    const int e = tid + i * NT;
    if (STORED_KMINOR) { const int kk = e % DK, rr = e / DK; S[rr * DS_K + kk] = reg[i]; }
    else { const int rr = e % ROWS, kk = e / ROWS; S[kk * (ROWS + 4) + rr] = reg[i]; }
  }
}

// CTA tile BM x BN (multiples of 32), one warp per 32x32 sub-tile.  128x128 is the throughput shape;
// 64x128 / 32x128 / 128x64 / 128x32 spread the narrow GEMMs of the recursion (a single 128-wide block
// column or row: panel solves, K=128 updates) over more SMs — one SM needs >= 17 us for a 128^3 tile.
template <bool TA, bool TB, int BM, int BN>
__global__ void __launch_bounds__((BM / 32) * (BN / 32) * 32)
gemm_dmma_kernel(int64_t m, int64_t n, int64_t k, double alpha, const double* A, int64_t lda,
                 const double* B, int64_t ldb, double beta, double* C, int64_t ldc,
                 int flags, int* head_flag) {
  constexpr int NT = (BM / 32) * (BN / 32) * 32;
  constexpr int WN = BN / 32;
  constexpr int ATILE = BM * DS_K > DK * (BM + 4) ? BM * DS_K : DK * (BM + 4);
  constexpr int BTILE = BN * DS_K > DK * (BN + 4) ? BN * DS_K : DK * (BN + 4);
  // head_flag != nullptr: grid is (row tiles, column tiles) so column block 0 is dispatched first
  const int64_t m0 = (int64_t)(head_flag ? blockIdx.x : blockIdx.y) * BM;
  const int64_t n0 = (int64_t)(head_flag ? blockIdx.y : blockIdx.x) * BN;
  if ((flags & GPK_GEMM_LOWER_ONLY) && n0 > m0 + BM - 1) return;
  extern __shared__ __align__(16) double dsm[];
  double* sA = dsm;                // [2][ATILE]
  double* sB = dsm + 2 * ATILE;    // [2][BTILE]
  __shared__ double s_col[BN];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = (warp / WN) * 32, wn = (warp % WN) * 32;
  const int g = lane >> 2, t = lane & 3;

  // k range; a lower-triangular stored A restricts it (rows of op(A) in this tile: m0..m0+BM-1)
  int64_t kb = 0, ke = k;
  const int triA = (flags & GPK_GEMM_A_LOWER) ? 1 : 0;
  if (triA) {
    if (TA) kb = (m0 / DK) * DK;                // op(A)[i][kk] = S[kk][i], nonzero iff kk >= i
    else ke = min(k, m0 + BM);                  // op(A)[i][kk] = S[i][kk], nonzero iff kk <= i
  }

  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  double ra[BM * DK / NT], rb[BN * DK / NT];
  const int nchunks = (int)((ke - kb + DK - 1) / DK);
  if (nchunks > 0) {
    dload<!TA, BM, NT>(ra, A, lda, m0, m, kb, ke, tid, triA);
    dload<TB, BN, NT>(rb, B, ldb, n0, n, kb, ke, tid, 0);
    dstore<!TA, BM, NT>(ra, sA, tid);
    dstore<TB, BN, NT>(rb, sB, tid);
  }
  __syncthreads();
  for (int c = 0; c < nchunks; ++c) {
    const int cur = c & 1;
    if (c + 1 < nchunks) {
      dload<!TA, BM, NT>(ra, A, lda, m0, m, kb + (int64_t)(c + 1) * DK, ke, tid, triA);
      dload<TB, BN, NT>(rb, B, ldb, n0, n, kb + (int64_t)(c + 1) * DK, ke, tid, 0);
    }
    const double* cA = sA + cur * ATILE;
    const double* cB = sB + cur * BTILE;
#pragma unroll
    for (int k4 = 0; k4 < DK; k4 += 4) {
      double af[4], bf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        af[i] = !TA ? cA[(wm + i * 8 + g) * DS_K + k4 + t] : cA[(k4 + t) * (BM + 4) + wm + i * 8 + g];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        bf[j] = TB ? cB[(wn + j * 8 + g) * DS_K + k4 + t] : cB[(k4 + t) * (BN + 4) + wn + j * 8 + g];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
    if (c + 1 < nchunks) {
      dstore<!TA, BM, NT>(ra, sA + (cur ^ 1) * ATILE, tid);
      dstore<TB, BN, NT>(rb, sB + (cur ^ 1) * BTILE, tid);
    }
    __syncthreads();
  }

  if (flags & GPK_GEMM_COLSUMSQ) {
    if (tid < BN) s_col[tid] = 0.0;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int64_t gi = m0 + wm + i * 8 + g;
          const double v = alpha * acc[i][j][h];
          if (gi < m) s += v * v;
        }
        // reduce over the 8 row-groups g (lanes with equal t)
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        s += __shfl_xor_sync(0xffffffffu, s, 8);
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        if (g == 0) atomicAdd(&s_col[wn + j * 8 + 2 * t + h], s);
      }
    __syncthreads();
    if (tid < BN && n0 + tid < n) atomicAdd(&C[n0 + tid], s_col[tid]);
    return;
  }

  const bool vec_ok = ((uintptr_t)C % 16 == 0) && (ldc % 2 == 0);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t gi = m0 + wm + i * 8 + g;
    if (gi >= m) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t gj = n0 + wn + j * 8 + 2 * t;
      double* dst = C + gi * ldc + gj;
      double v0 = alpha * acc[i][j][0], v1 = alpha * acc[i][j][1];
      if (gj + 1 < n && vec_ok) {
        if (beta != 0.0) {
          const double2 old = *reinterpret_cast<const double2*>(dst);
          v0 += beta * old.x; v1 += beta * old.y;
        }
        *reinterpret_cast<double2*>(dst) = make_double2(v0, v1);
      } else {
        if (gj < n) dst[0] = beta != 0.0 ? v0 + beta * dst[0] : v0;
        if (gj + 1 < n) dst[1] = beta != 0.0 ? v1 + beta * dst[1] : v1;
      }
    }
  }
  if (head_flag && n0 < 128) {  // publish progress on the leading block column / the leading 128x128 block
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      atomicAdd(head_flag, 1);
      const int u = diag_units_tile(m0, n0, BM, BN, m, n);
      if (u) atomicAdd(head_flag + 1, u);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// generic CUDA-core kernel (fp32; fp64 runs on the DMMA kernel above): 128x128x8, 256 threads, 8x8
// ------------------------------------------------------------------------------------------------
constexpr int SK = 8;

// BM x BN tile, 16 x 16 threads, (BM/16) x (BN/16) accumulators per thread in groups of up to 4 consecutive
// rows / columns.  Narrow shapes (32/64 x 128, 128 x 32/64) exist for the same reason as in the DMMA kernel: the
// small-K GEMMs of the factorisation and of trsm have few 128 x 128 tiles (measured before: 54 launches = 2.0 ms of
// the 5.7 ms SVGP evaluation at 2.6 TFLOP/s), and the in-place contract needs one tile across the aliased operand.
template <typename T, bool TA, bool TB, int BM, int BN>
__global__ void __launch_bounds__(256)
gemm_simt_kernel(int64_t m, int64_t n, int64_t k, T alpha, const T* A, int64_t lda,
                 const T* B, int64_t ldb, T beta, T* C, int64_t ldc, int flags, int* head_flag) {
  constexpr int TM = BM / 16, TN = BN / 16, GM = TM < 4 ? TM : 4, GN = TN < 4 ? TN : 4;
  const int64_t m0 = (int64_t)(head_flag ? blockIdx.x : blockIdx.y) * BM;
  const int64_t n0 = (int64_t)(head_flag ? blockIdx.y : blockIdx.x) * BN;
  if ((flags & GPK_GEMM_LOWER_ONLY) && n0 > m0 + BM - 1) return;
  __shared__ __align__(16) T sA[2][SK][BM + 4];
  __shared__ __align__(16) T sB[2][SK][BN + 4];
  __shared__ T s_col[BN];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  auto rowi = [&](int i) { return (i / GM) * (16 * GM) + ty * GM + (i % GM); };  // tile row of accumulator row i
  auto coli = [&](int j) { return (j / GN) * (16 * GN) + tx * GN + (j % GN); };

  int64_t kb = 0, ke = k;
  const int triA = (flags & GPK_GEMM_A_LOWER) ? 1 : 0;
  if (triA) {
    if (TA) kb = (m0 / SK) * SK; else ke = min(k, m0 + BM);
  }
  T acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = T(0);

  constexpr int LA = BM * SK / 256, LB = BN * SK / 256;  // elements of each operand chunk per thread
  T ra[LA], rb[LB];
  auto gload = [&](int64_t k0) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = tid + i * 256;
      int rr, kk;
      if (!TA) { kk = e % SK; rr = e / SK; } else { rr = e % BM; kk = e / BM; }
      const int64_t gr = m0 + rr, gk = k0 + kk;
      T v = T(0);
      if (gr < m && gk < ke) {
        const int64_t srow = !TA ? gr : gk, scol = !TA ? gk : gr;
        if (!(triA && scol > srow)) v = A[srow * lda + scol];
      }
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      const int e = tid + i * 256;
      int rr, kk;
      if (TB) { kk = e % SK; rr = e / SK; } else { rr = e % BN; kk = e / BN; }
      const int64_t gr = n0 + rr, gk = k0 + kk;
      T v = T(0);
      if (gr < n && gk < ke) v = TB ? B[gr * ldb + gk] : B[gk * ldb + gr];
      rb[i] = v;
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = tid + i * 256;
      int rr, kk;
      if (!TA) { kk = e % SK; rr = e / SK; } else { rr = e % BM; kk = e / BM; }
      sA[buf][kk][rr] = ra[i];
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      const int e = tid + i * 256;
      int rr, kk;
      if (TB) { kk = e % SK; rr = e / SK; } else { rr = e % BN; kk = e / BN; }
      sB[buf][kk][rr] = rb[i];
    }
  };

  const int nchunks = (int)((ke - kb + SK - 1) / SK);
  if (nchunks > 0) { gload(kb); sstore(0); }
  __syncthreads();
  for (int c = 0; c < nchunks; ++c) {
    const int cur = c & 1;
    if (c + 1 < nchunks) gload(kb + (int64_t)(c + 1) * SK);
#pragma unroll
    for (int kk = 0; kk < SK; ++kk) {
      T a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = sA[cur][kk][rowi(i)];
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = sB[cur][kk][coli(j)];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
    if (c + 1 < nchunks) sstore(cur ^ 1);
    __syncthreads();
  }

  if (flags & GPK_GEMM_COLSUMSQ) {
    if (tid < BN) s_col[tid] = T(0);
    __syncthreads();
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      T s = T(0);
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        const int64_t gi = m0 + rowi(i);
        const T v = alpha * acc[i][j];
        if (gi < m) s += v * v;
      }
      s += __shfl_xor_sync(0xffffffffu, s, 16);  // the two ty rows held by one warp
      if ((tid & 16) == 0) atomic_add_t(&s_col[coli(j)], s);
    }
    __syncthreads();
    if (tid < BN && n0 + tid < n) atomic_add_t(&C[n0 + tid], s_col[tid]);
    return;
  }

#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int64_t gi = m0 + rowi(i);
    if (gi >= m) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int64_t gj = n0 + coli(j);
      if (gj >= n) continue;
      T* dst = C + gi * ldc + gj;
      const T v = alpha * acc[i][j];
      *dst = beta != T(0) ? v + beta * *dst : v;
    }
  }
  if (head_flag && n0 < 128) {
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      atomicAdd(head_flag, 1);
      const int u = diag_units_tile(m0, n0, BM, BN, m, n);
      if (u) atomicAdd(head_flag + 1, u);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// skinny right-hand sides (n <= 16, B stored [k][n]):  A^T q_mu, A err, the TRSM updates of alpha / c
// (conditionals/util.py:144, models/sgpr.py:263-264, logdensities.py:150).  Memory-bound on A.
// ------------------------------------------------------------------------------------------------
constexpr int SKN = 16;

template <typename T, bool TA>
__global__ void __launch_bounds__(256)
gemm_skinny_kernel(int64_t m, int n, int64_t k, T alpha, const T* A, int64_t lda, const T* B, int64_t ldb, T beta,
                   T* C, int64_t ldc) {
  T acc[SKN];
#pragma unroll
  for (int j = 0; j < SKN; ++j) acc[j] = T(0);
  if (!TA) {
    // one CTA (8 warps) per output row: the warps split k, lanes stride over it (row of A contiguous),
    // 4 independent loads in flight per lane; partial sums meet in shared memory
    __shared__ T red[8][SKN];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int64_t i = blockIdx.x;
    const T* arow = A + i * lda;
    const int64_t kchunk = (k + 7) / 8, k0 = wp * kchunk, k1 = min(k, k0 + kchunk);
    int64_t kk = k0 + lane;
    for (; kk + 96 < k1; kk += 128) {
      const T a0 = arow[kk], a1 = arow[kk + 32], a2 = arow[kk + 64], a3 = arow[kk + 96];
#pragma unroll
      for (int j = 0; j < SKN; ++j)
        if (j < n) {
          acc[j] = fma(a0, B[kk * ldb + j], acc[j]);
          acc[j] = fma(a1, B[(kk + 32) * ldb + j], acc[j]);
          acc[j] = fma(a2, B[(kk + 64) * ldb + j], acc[j]);
          acc[j] = fma(a3, B[(kk + 96) * ldb + j], acc[j]);
        }
    }
    for (; kk < k1; kk += 32) {
      const T a = arow[kk];
#pragma unroll
      for (int j = 0; j < SKN; ++j)
        if (j < n) acc[j] = fma(a, B[kk * ldb + j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < SKN; ++j)
      if (j < n) {
        const T s = warp_sum(acc[j]);
        if (lane == 0) red[wp][j] = s;
      }
    __syncthreads();
    if (threadIdx.x < n) {
      T s = T(0);
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) s += red[w8][threadIdx.x];
      T* dst = C + i * ldc + threadIdx.x;
      *dst = beta != T(0) ? alpha * s + beta * *dst : alpha * s;
    }
  } else {
    // A stored [k][m]: a CTA covers 32 output rows (lanes -> consecutive rows: coalesced), its 8 warps split k with
    // 4 loads in flight per lane; partial sums meet in shared memory.  (One thread per row over the whole k was
    // latency-bound: 1.0 ms for the SVGP mean A^T q_mu at M = 2048, B = 4096.)
    __shared__ T red[8][32][SKN + 1];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 32 + lane;
    const int64_t kchunk = (k + 7) / 8, k0 = wp * kchunk, k1 = min(k, k0 + kchunk);
    if (i < m) {
      int64_t kk = k0;
      for (; kk + 3 < k1; kk += 4) {
        const T a0 = A[kk * lda + i], a1 = A[(kk + 1) * lda + i], a2 = A[(kk + 2) * lda + i], a3 = A[(kk + 3) * lda + i];
#pragma unroll
        for (int j = 0; j < SKN; ++j)
          if (j < n) {
            acc[j] = fma(a0, B[kk * ldb + j], acc[j]);
            acc[j] = fma(a1, B[(kk + 1) * ldb + j], acc[j]);
            acc[j] = fma(a2, B[(kk + 2) * ldb + j], acc[j]);
            acc[j] = fma(a3, B[(kk + 3) * ldb + j], acc[j]);
          }
      }
      for (; kk < k1; ++kk) {
        const T a = A[kk * lda + i];
#pragma unroll
        for (int j = 0; j < SKN; ++j)
          if (j < n) acc[j] = fma(a, B[kk * ldb + j], acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < SKN; ++j) red[wp][lane][j] = acc[j];
    __syncthreads();
    if (i < m)
      for (int j = wp; j < n; j += 8) {
        T sum = T(0);
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) sum += red[w8][lane][j];
        T* dst = C + i * ldc + j;
        *dst = beta != T(0) ? alpha * sum + beta * *dst : alpha * sum;
      }
  }
}

template <typename T>
static int launch_skinny(int ta, int64_t m, int n, int64_t k, T alpha, const T* A, int64_t lda, const T* B, int64_t ldb,
                         T beta, T* C, int64_t ldc, cudaStream_t st) {
  if (!ta)
    gemm_skinny_kernel<T, false><<<(unsigned)m, 256, 0, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc);
  else
    gemm_skinny_kernel<T, true><<<(unsigned)((m + 31) / 32), 256, 0, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc);
  GPK_LAUNCH_OK();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// dispatch
// ------------------------------------------------------------------------------------------------
template <typename T, int BM, int BN>
static int launch_simt_shape(int ta, int tb, int64_t m, int64_t n, int64_t k, T alpha, const T* A, int64_t lda,
                             const T* B, int64_t ldb, T beta, T* C, int64_t ldc, int flags, cudaStream_t st, int* hf) {
  dim3 grid((unsigned)((n + BN - 1) / BN), (unsigned)((m + BM - 1) / BM));
  if (hf) grid = dim3(grid.y, grid.x);  // row tiles fastest: column block 0 first
  GPK_CHECK_ARG(grid.y <= 65535, "gemm: too many tiles for the grid");
#define GO(TA_, TB_) gemm_simt_kernel<T, TA_, TB_, BM, BN><<<grid, 256, 0, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags, hf)
  if (!ta && !tb) GO(false, false); else if (!ta && tb) GO(false, true);
  else if (ta && !tb) GO(true, false); else GO(true, true);
#undef GO
  GPK_LAUNCH_OK();
  return 0;
}

// shape selection, same rules as launch_dmma: 128x128 when there are enough tiles to fill the machine, otherwise
// narrower tiles; C aliasing A needs one tile across n (BN >= n), C aliasing B one tile across m
template <typename T>
static int launch_simt(int ta, int tb, int64_t m, int64_t n, int64_t k, T alpha, const T* A, int64_t lda,
                       const T* B, int64_t ldb, T beta, T* C, int64_t ldc, int flags, cudaStream_t st, int* hf) {
  const bool alias_a = (const void*)C == (const void*)A, alias_b = (const void*)C == (const void*)B;
  const int64_t t128 = ((m + 127) / 128) * ((n + 127) / 128);
#define SHAPE(BM_, BN_) return launch_simt_shape<T, BM_, BN_>(ta, tb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags, st, hf)
  if (t128 >= 120 || (flags & GPK_GEMM_COLSUMSQ)) SHAPE(128, 128);
  if (alias_b || (m <= 128 && !alias_a)) {          // short and wide: split the columns finer
    if ((n + 63) / 64 >= 100) SHAPE(128, 64);
    SHAPE(128, 32);
  }
  if (alias_a || n <= 128) {                        // tall and narrow: split the rows finer
    if ((m + 63) / 64 >= 100) SHAPE(64, 128);
    SHAPE(32, 128);
  }
  if (((m + 63) / 64) * ((n + 127) / 128) >= 100) SHAPE(64, 128);
  SHAPE(32, 128);
#undef SHAPE
}

template <int BM, int BN>
static int launch_dmma_shape(int ta, int tb, int64_t m, int64_t n, int64_t k, double alpha, const double* A, int64_t lda,
                             const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags,
                             cudaStream_t st, int* hf) {
  constexpr int NT = (BM / 32) * (BN / 32) * 32;
  constexpr int ATILE = BM * DS_K > DK * (BM + 4) ? BM * DS_K : DK * (BM + 4);
  constexpr int BTILE = BN * DS_K > DK * (BN + 4) ? BN * DS_K : DK * (BN + 4);
  const size_t smem = (size_t)(2 * ATILE + 2 * BTILE) * sizeof(double);
  static PerDeviceOnce attr_once;  // function attributes are per device
  GPK_TRY(attr_once.run([&]() -> int {
    GPK_CUDA_OK(cudaFuncSetAttribute(gemm_dmma_kernel<false, false, BM, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GPK_CUDA_OK(cudaFuncSetAttribute(gemm_dmma_kernel<false, true, BM, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GPK_CUDA_OK(cudaFuncSetAttribute(gemm_dmma_kernel<true, false, BM, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GPK_CUDA_OK(cudaFuncSetAttribute(gemm_dmma_kernel<true, true, BM, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
  }));
  dim3 grid((unsigned)((n + BN - 1) / BN), (unsigned)((m + BM - 1) / BM));
  if (hf) grid = dim3(grid.y, grid.x);  // row tiles fastest: column block 0 first
  GPK_CHECK_ARG(grid.y <= 65535, "gemm: too many tiles for the grid");
#define GO(TA_, TB_) gemm_dmma_kernel<TA_, TB_, BM, BN><<<grid, NT, smem, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags, hf)
  if (!ta && !tb) GO(false, false); else if (!ta && tb) GO(false, true);
  else if (ta && !tb) GO(true, false); else GO(true, true);
#undef GO
  GPK_LAUNCH_OK();
  return 0;
}

static int launch_dmma(int ta, int tb, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                       int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags,
                       cudaStream_t st, int* hf) {
  // shape selection: 128x128 when there are enough tiles to fill the machine, otherwise narrower tiles.
  // In-place contract: C aliasing A needs one tile across n (BN >= n), C aliasing B one tile across m.
  const bool alias_a = (const void*)C == (const void*)A, alias_b = (const void*)C == (const void*)B;
  const int64_t t128 = ((m + 127) / 128) * ((n + 127) / 128);
#define SHAPE(BM_, BN_) return launch_dmma_shape<BM_, BN_>(ta, tb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags, st, hf)
  if (t128 >= 120 || (flags & GPK_GEMM_COLSUMSQ)) SHAPE(128, 128);
  if (alias_b || (m <= 128 && !alias_a)) {          // short and wide: split the columns finer
    if ((n + 63) / 64 >= 100) SHAPE(128, 64);
    SHAPE(128, 32);
  }
  if (alias_a || n <= 128) {                        // tall and narrow: split the rows finer
    if ((m + 63) / 64 >= 100) SHAPE(64, 128);
    SHAPE(32, 128);
  }
  if (((m + 63) / 64) * ((n + 127) / 128) >= 100) SHAPE(64, 128);
  SHAPE(32, 128);
#undef SHAPE
}

template <typename T>
int gemm_t(int transa, int transb, int64_t m, int64_t n, int64_t k, T alpha, const T* A, int64_t lda, const T* B,
           int64_t ldb, T beta, T* C, int64_t ldc, int flags, cudaStream_t st, const GemmOpts* opts) {
  if (m <= 0 || n <= 0) return 0;
  int* hf = opts ? opts->head_flag : nullptr;
  // skinny right-hand side: never when C aliases an operand row-block larger than one thread's reach
  if (!hf && n <= SKN && !transb && flags == 0 && (const void*)C != (const void*)B && (const void*)C != (const void*)A) {
    ProfScope ps(PROF_SKINNY, st);
    return launch_skinny<T>(transa, m, (int)n, k, alpha, A, lda, B, ldb, beta, C, ldc, st);
  }
  if (sizeof(T) == 4 && !hf && gemm_tf32_eligible(m, n, k, A, B, C, flags))
    return gemm_tf32(transa, transb, m, n, k, (float)alpha, (const float*)A, lda, (const float*)B, ldb, (float)beta,
                     (float*)C, ldc, flags, st);
  // work = MACs the launch computes (tiles strictly above the diagonal are skipped for LOWER_ONLY: about half)
  ProfScope ps(PROF_GEMM, st, (double)m * (double)n * (double)k * ((flags & GPK_GEMM_LOWER_ONLY) && m == n ? 0.5 : 1.0));
  if constexpr (sizeof(T) == 8)
    return launch_dmma(transa, transb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags, st, hf);
  else
    return launch_simt<T>(transa, transb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags, st, hf);
}

template int gemm_t<float>(int, int, int64_t, int64_t, int64_t, float, const float*, int64_t, const float*, int64_t,
                           float, float*, int64_t, int, cudaStream_t, const GemmOpts*);
template int gemm_t<double>(int, int, int64_t, int64_t, int64_t, double, const double*, int64_t, const double*,
                            int64_t, double, double*, int64_t, int, cudaStream_t, const GemmOpts*);

}  // namespace gpk
