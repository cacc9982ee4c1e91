// potrf.cu — blocked Cholesky and triangular solves for sm_100a.
//
// Replaces tf.linalg.cholesky (gpflow/models/gpr.py:102, posteriors.py:422,533,538,703,
// models/sgpr.py:201,207, conditionals/util.py:67, kullback_leiblers.py:107) and
// tf.linalg.triangular_solve (logdensities.py:150, conditionals/util.py:125,139, sgpr.py:204,264,
// posteriors.py:495-496,534,540,707,710, kullback_leiblers.py:114,152).
//
// Structure (row-major, lower): recursive blocked factorisation whose leaves are 128x128 diagonal
// blocks handled by ONE CTA entirely in shared memory (warp-cooperative 32x32 register Cholesky,
// per-row substitution panels, 4x4 register-tiled updates with in-leaf look-ahead).
//   fp64, n > 128 ("slim"): the leaf also emits the inverses of its two 64x64 diagonal sub-blocks and
//   potrf_panel_kernel solves the rows below on DMMA; the full 128x128 block inverses that trsm consumes
//   are produced afterwards, all blocks in parallel (trtri_diag_kernel).
//   fp32 / single block: the leaf emits the INVERSE of the whole diagonal block and the panel solve
//   X = B L_jj^-T is one dense GEMM with it.
// Trailing updates C -= A A^T (gemm.cu / gemm_tc.cu / gemm_tf32.cu, K >= 128) publish progress on the next
// diagonal block so that the next leaf overlaps them on a side stream (look-ahead).
// Rows below the square part (`rows > n`) ride along, so appending (Y-m)^T as extra rows yields
// alpha^T = (L^-1 (Y-m))^T without a separate TRSV (logdensities.py:150).
#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"
#include <type_traits>
#include "planes.cuh"

namespace gpk {

constexpr int LS = NB + 1;  // shared row stride of the leaf matrix

template <typename T> __device__ __forceinline__ T sqrt_t(T x);
template <> __device__ __forceinline__ double sqrt_t<double>(double x) { return sqrt(x); }
template <> __device__ __forceinline__ float sqrt_t<float>(float x) { return sqrtf(x); }

// Leaf design notes (measured with gpk_debug_leaf on B200, cycles @1.9 GHz):
//  * shared-memory read-modify-write loops serialise on load/store aliasing (~55 cycles per fma);
//    all O(n^3) phases therefore accumulate 4x4 micro-tiles in registers from read-only operands;
//  * micro-tiles are INTERLEAVED (thread (tr,tc) owns rows tr+TR*i, cols tc+TC*j) so the lanes of a
//    warp touch consecutive rows of the stride-129 array: bank-conflict free;
//  * the serial part (32x32 diagonal Cholesky, one warp) keeps its row in registers and exchanges
//    columns by shuffles.

// asynchronous global -> shared copies (all of a thread's copies in flight at once; cp_async_wait_all + a barrier publish them)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {  // !valid: 16 zero bytes
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int nbytes = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(nbytes) : "memory");
}
template <typename T>
__device__ __forceinline__ void cp_async_elem(T* smem_dst, const T* gsrc) {  // one element (4 or 8 bytes)
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  if (sizeof(T) == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void dmma884p(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c[0]), "+d"(c[1])
               : "d"(a), "d"(b));
}

// ---- one 32x32 block pair of the in-leaf trailing update: C[R0.., C0..] -= S[R0.., jb:jb+32] S[C0.., jb:jb+32]^T (c <= r) -------
// 64 threads (sub = 0..63) per pair.  fp64: two warps x (2 m-blocks x 4 n-blocks) of mma.sync.m8n8k4.f64 -- 48 shared loads +
// 64 DMMAs per warp instead of 256 loads + 512 DFMAs of the 4x4 micro-tile form (4.3k -> cycles measured on the pair that
// gates the next diagonal block, scripts/leaf_timing.py).  fp32: 8 x 8 threads, interleaved 4x4 micro-tiles.
// one 16-row half (wv = 0, 1) of a pair by ONE warp
__device__ __forceinline__ void leaf_pair_half(double* S, int R0, int C0, int jb, int wv, int lane) {
  const int g = lane >> 2, q = lane & 3;
  double acc[2][4][2];
#pragma unroll
  for (int mb = 0; mb < 2; ++mb)
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
  // k-step ks covers k = ks, ks + 8, ks + 16, ks + 24 (lane q supplies k = ks + 8 q): with the odd row stride the 32 lanes of a
  // fragment load then touch every 8-byte bank exactly twice (2 wavefronts, the minimum for 256 bytes) instead of up to 4
  // times with k = 4 ks + q -- the shared-memory pipe also carries the shuffles of the concurrent 32x32 factorisation
  const double* Ra = S + (R0 + 16 * wv + g) * LS + jb + 8 * q;
  const double* Rb = S + (C0 + g) * LS + jb + 8 * q;
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    double a[2], b[4];
#pragma unroll
    for (int mb = 0; mb < 2; ++mb) a[mb] = Ra[mb * 8 * LS + ks];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) b[nb] = Rb[nb * 8 * LS + ks];
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) dmma884p(acc[mb][nb], a[mb], b[nb]);
  }
#pragma unroll
  for (int mb = 0; mb < 2; ++mb)
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      const int r = R0 + 16 * wv + 8 * mb + g, c = C0 + 8 * nb + 2 * q;
      if (c <= r) S[r * LS + c] -= acc[mb][nb][0];
      if (c + 1 <= r) S[r * LS + c + 1] -= acc[mb][nb][1];
    }
}
__device__ __forceinline__ void leaf_pair_update(double* S, int R0, int C0, int jb, int sub) {
  leaf_pair_half(S, R0, C0, jb, sub >> 5, sub & 31);
}
// the pair that IS the next diagonal block (R0 = C0 = t0), spread over all 8 warps: warp w takes the 8-row block w >> 1 and the
// two 8-column blocks 2 (w & 1), +1 (those not above the diagonal): 16 DMMAs per warp, then everybody meets at a barrier and
// warp 0 factors the block while the others apply the rest of the update
__device__ __forceinline__ void leaf_pair0_all(double* S, int t0, int jb, int w, int lane) {
  const int g = lane >> 2, q = lane & 3, mb = w >> 1, nb0 = 2 * (w & 1);
  if (nb0 > mb) return;  // both column blocks above the diagonal
  double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
  const double* Ra = S + (t0 + 8 * mb + g) * LS + jb + 8 * q;  // (k = ks + 8 q, see leaf_pair_half)
  const double* Rb = S + (t0 + 8 * nb0 + g) * LS + jb + 8 * q;
  const bool second = nb0 + 1 <= mb;
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    const double a = Ra[ks];
    dmma884p(acc[0], a, Rb[ks]);
    if (second) dmma884p(acc[1], a, Rb[8 * LS + ks]);
  }
  const int r = t0 + 8 * mb + g;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int c = t0 + 8 * (nb0 + j) + 2 * q;
    if (j == 1 && !second) break;
    if (c <= r) S[r * LS + c] -= acc[j][0];
    if (c + 1 <= r) S[r * LS + c + 1] -= acc[j][1];
  }
}

template <typename T> __device__ __forceinline__ T rsqrt_t(T x);
// MUFU.RSQ64H seed (rsqrt.approx.f64: ~2^-22 relative, no fp64 <-> fp32 conversions) + ONE third-order step
// y1 = y0 (1 + e/2 + 3 e^2/8), e = 1 - x y0^2: error ~ e^3 = 2^-66 before rounding.  Four dependent fp64 operations
// instead of the six of two Newton steps -- this sits on the serial pivot chain of the diagonal-block factorisation.
template <> __device__ __forceinline__ double rsqrt_t<double>(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double t = x * y;
  const double e = fma(-t, y, 1.0);
  const double p = fma(0.375, e, 0.5);
  const double q = y * e;
  return fma(q, p, y);
}
template <> __device__ __forceinline__ float rsqrt_t<float>(float x) { return rsqrtf(x); }

// ---- 32x32 diagonal block Cholesky by one warp: lane i owns row i in registers ---------------------
// On return S holds L (strict lower part), ldiag the diagonal of L, and S's diagonal 1/L_kk.
// Cross-lane traffic is shuffles only (a shared-memory column broadcast variant took 18.4k cycles, a pure
// shared-memory loop 27k, the right-looking register version 10-11.5k).
template <typename T>
__device__ __forceinline__ int warp_chol32(T* S, int jb, T* ldiag) {
  const int lane = threadIdx.x & 31;
  T a[32];
#pragma unroll
  for (int c = 0; c < 32; ++c) a[c] = c <= lane ? S[(jb + lane) * LS + jb + c] : T(0);
  int bad = 0;
  T my_inv = T(1), my_diag = T(1);
  // left-looking: corrections from columns < j-1 go into four independent partial sums, only the last one sits on
  // the pivot chain; entries above the diagonal accumulate harmless garbage (never read or stored).  Measured on B200,
  // cycles per block: 8.1k (right-looking: 9.4k, blocked by 8 columns: 9.8k, pivots formed by every lane: 8.4k)
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    if (j >= 2) {
      T p0 = T(0), p1 = T(0), p2 = T(0), p3 = T(0);
#pragma unroll
      for (int k = 0; k < 32; ++k)
        if (k < j - 1) {
          const T ljk = __shfl_sync(0xffffffffu, a[k], j);
          if ((k & 3) == 0) p0 = fma(a[k], ljk, p0);
          else if ((k & 3) == 1) p1 = fma(a[k], ljk, p1);
          else if ((k & 3) == 2) p2 = fma(a[k], ljk, p2);
          else p3 = fma(a[k], ljk, p3);
        }
      a[j] -= (p0 + p1) + (p2 + p3);
    }
    if (j >= 1) a[j] = fma(-a[j - 1], __shfl_sync(0xffffffffu, a[j - 1], j), a[j]);
    T d = __shfl_sync(0xffffffffu, a[j], j);
    if (!(d > T(0))) {
      if (bad == 0) bad = j + 1;
      d = T(1);
    }
    const T inv = rsqrt_t<T>(d);
    if (lane == j) { my_inv = inv; my_diag = d * inv; }
    a[j] *= inv;
  }
#pragma unroll
  for (int c = 0; c < 32; ++c)
    if (c < lane) S[(jb + lane) * LS + jb + c] = a[c];
  S[(jb + lane) * LS + jb + lane] = my_inv;  // diagonal slot now holds inv(L)_kk
  ldiag[jb + lane] = my_diag;
  __syncwarp();
  return bad;
}

// ---- inverse of one 32x32 lower-triangular diagonal block by one warp ----------------------------
// lane j solves L x = e_j with x in registers (L broadcast from shared memory); x_i (i > j) goes to
// the TRANSPOSED slot S[jb+j][jb+i]; the diagonal slot already holds 1/L_jj.
template <typename T>
__device__ __forceinline__ void warp_inv32(T* S, int jb) {
  const int lane = threadIdx.x & 31;
  T x[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) x[i] = i == lane ? T(1) : T(0);
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    x[k] *= S[(jb + k) * LS + jb + k];
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (i > k) x[i] -= S[(jb + i) * LS + jb + k] * x[k];
  }
  __syncwarp();  // every lane has finished reading the lower triangle before the upper slots are written
#pragma unroll
  for (int i = 0; i < 32; ++i)
    if (i > lane) S[(jb + lane) * LS + jb + i] = x[i];
  __syncwarp();
}

// 4x4 register micro-tile accumulation: acc[i][j] += sum_k fa(i,k) * fb(j,k), k in [k0,k1)
template <typename T, class FA, class FB>
__device__ __forceinline__ void mt_acc(T (&acc)[4][4], int k0, int k1, FA fa, FB fb) {
#pragma unroll 4
  for (int k = k0; k < k1; ++k) {
    T av[4], bv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) av[i] = fa(i, k);
#pragma unroll
    for (int j = 0; j < 4; ++j) bv[j] = fb(j, k);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
  }
}

template <typename T>
__device__ __forceinline__ void mt_zero(T (&acc)[4][4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = T(0);
}

__device__ __forceinline__ void leaf_pair_update(float* S, int R0, int C0, int jb, int sub) {
  const int ptr_ = sub >> 3, ptc = sub & 7;
  float acc[4][4];
  mt_zero(acc);
  const float* Ra = S + (R0 + ptr_) * LS + jb;
  const float* Rb = S + (C0 + ptc) * LS + jb;
  mt_acc<float>(acc, 0, 32,
                [&](int i, int k) { return Ra[i * 8 * LS + k]; },
                [&](int j, int k) { return Rb[j * 8 * LS + k]; });
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = R0 + ptr_ + 8 * i, c = C0 + ptc + 8 * j;
      if (c <= r) S[r * LS + c] -= acc[i][j];
    }
}

// level 32 of the inverse on DMMA (fp64): X = -Linv_II (L_IJ Linv_JJ) for the pairs (I,J) = (1,0), (3,2); warps 0-1 / 2-3 take
// one pair each (16 rows x 32 columns per warp), the rest of the CTA only joins the barriers.  Storage conventions as in
// invert_offdiag_128 below (Linv transposed in the upper triangle of S, diagonal included).
__device__ __forceinline__ void invert_level32_dmma(double* S, double* tmp) {
  const int tid = threadIdx.x, pair = tid >> 6, wv = (tid >> 5) & 1, lane = tid & 31, g = lane >> 2, q = lane & 3;
  const int J = 2 * pair, I = J + 1;
  double acc[2][4][2];
  if (pair < 2) {  // T = L_IJ Linv_JJ;  Linv_JJ[k][c] = S[J*32+c][J*32+k] for k >= c
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
    const double* La = S + (I * 32 + 16 * wv + g) * LS + J * 32 + q;
    const double* Lb = S + (J * 32 + g) * LS + J * 32 + q;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      double a[2], b[4];
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) a[mb] = La[mb * 8 * LS + 4 * ks];
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) {
        const double v = Lb[nb * 8 * LS + 4 * ks];
        b[nb] = (4 * ks + q >= 8 * nb + g) ? v : 0.0;
      }
#pragma unroll
      for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int nb = 0; nb < 4; ++nb)
          if (4 * ks + 3 >= 8 * nb) dmma884p(acc[mb][nb], a[mb], b[nb]);  // (k-steps entirely above the diagonal are zero)
    }
    double* tp = tmp + pair * 1024;
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int nb = 0; nb < 4; ++nb)
        *reinterpret_cast<double2*>(tp + (16 * wv + 8 * mb + g) * 32 + 8 * nb + 2 * q) = make_double2(acc[mb][nb][0], acc[mb][nb][1]);
  }
  __syncthreads();
  if (pair < 2) {  // X = -Linv_II T;  Linv_II[r][k] = S[I*32+k][I*32+r] for r >= k;  stored transposed: S[J*32+c][I*32+r]
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
    const double* tp = tmp + pair * 1024;
    const double* Li = S + (I * 32 + q) * LS + I * 32 + 16 * wv + g;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      double a[2], b[4];
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) {
        const double v = Li[4 * ks * LS + 8 * mb];
        a[mb] = (16 * wv + 8 * mb + g >= 4 * ks + q) ? v : 0.0;
      }
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) b[nb] = tp[(4 * ks + q) * 32 + 8 * nb + g];
#pragma unroll
      for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) dmma884p(acc[mb][nb], a[mb], b[nb]);
    }
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) {
        const int r = 16 * wv + 8 * mb + g, c = 8 * nb + 2 * q;
        S[(J * 32 + c) * LS + I * 32 + r] = -acc[mb][nb][0];
        S[(J * 32 + c + 1) * LS + I * 32 + r] = -acc[mb][nb][1];
      }
  }
  __syncthreads();
}

// ---- off-diagonal blocks of the inverse (diagonal 32x32 blocks already inverted) ---------------------
// Linv is stored TRANSPOSED in the upper triangle of S INCLUDING the diagonal: Linv[r][c] = S[c][r],
// r >= c.  The strict lower triangle of S still holds L.  tmp: 4096-element scratch.
// Block recursion  [A 0; C D]^-1 = [A^-1 0; -D^-1 C A^-1, D^-1]:
//   level 32: inside each 64x64 diagonal block (2 independent pairs, 64 threads each, 2 products)
//   level 64: the 64x64 block (rows 64.., cols 0..63) with all 256 threads (2 products of depth 64)
template <typename T>
__device__ void invert_offdiag_128(T* S, T* tmp, bool level64 = true) {
  const int tid = threadIdx.x;
  T acc[4][4];
  if (sizeof(T) == 8) {  // ---- level 32 on DMMA: pairs (I,J) = (1,0) and (3,2), two warps per pair
    invert_level32_dmma(reinterpret_cast<double*>(S), reinterpret_cast<double*>(tmp));
  } else {  // ---- level 32: pairs (I,J) = (1,0) and (3,2)
    const int pair = tid >> 6, sub = tid & 63, tr = sub >> 3, tc = sub & 7;
    const int J = 2 * pair, I = J + 1;
    if (pair < 2) {
      mt_zero(acc);
      const T* La = S + (I * 32 + tr) * LS + J * 32;   // L_IJ rows tr + 8 i
      const T* Lb = S + (J * 32 + tc) * LS + J * 32;   // Linv_JJ[k][c] = S[J*32+c][J*32+k], k >= c
      mt_acc<T>(acc, 0, 32,
                [&](int i, int k) { return La[i * 8 * LS + k]; },
                [&](int j, int k) { const T v = Lb[j * 8 * LS + k]; return k >= tc + 8 * j ? v : T(0); });
      T* tp = tmp + pair * 1024;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) tp[(tr + 8 * i) * 32 + tc + 8 * j] = acc[i][j];
    }
    __syncthreads();
    if (pair < 2) {
      const T* tp = tmp + pair * 1024;
      const T* Li = S + (I * 32) * LS + I * 32 + tr;   // Linv_II[r][k] = S[I*32+k][I*32+r], r >= k
      mt_zero(acc);
      mt_acc<T>(acc, 0, 32,
                [&](int i, int k) { const T v = Li[k * LS + 8 * i]; return (tr + 8 * i >= k) ? v : T(0); },
                [&](int j, int k) { return tp[k * 32 + tc + 8 * j]; });
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) S[(J * 32 + tc + 8 * j) * LS + I * 32 + tr + 8 * i] = -acc[i][j];
    }
    __syncthreads();
  }
  if (level64) {  // ---- level 64: X = -D^-1 (C A^-1), C = L[64:128, 0:64], A^-1 = Linv[0:64,0:64], D^-1 = Linv[64:,64:]
    const int tr = tid >> 4, tc = tid & 15;            // 16 x 16 threads, rows tr + 16 i, cols tc + 16 j
    mt_zero(acc);
    const T* Ca = S + (64 + tr) * LS;                  // C[r][k] = S[64+r][k]
    const T* Ab = S + tc * LS;                         // A^-1[k][c] = S[c][k], k >= c
    mt_acc<T>(acc, 0, 64,
              [&](int i, int k) { return Ca[i * 16 * LS + k]; },
              [&](int j, int k) { const T v = Ab[j * 16 * LS + k]; return k >= tc + 16 * j ? v : T(0); });
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) tmp[(tr + 16 * i) * 64 + tc + 16 * j] = acc[i][j];
    __syncthreads();
    mt_zero(acc);
    const T* Di = S + 64 * LS + 64 + tr;               // D^-1[r][k] = S[64+k][64+r], r >= k
    mt_acc<T>(acc, 0, 64,
              [&](int i, int k) { const T v = Di[k * LS + 16 * i]; return (tr + 16 * i >= k) ? v : T(0); },
              [&](int j, int k) { return tmp[k * 64 + tc + 16 * j]; });
    // Linv[64+r][c] = -acc  ->  S[c][64+r]
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) S[(tc + 16 * j) * LS + 64 + tr + 16 * i] = -acc[i][j];
    __syncthreads();
  }
}

// lower triangle of an n x n block (identity-padded to 128) as asynchronous element copies: every thread has its up to 64
// loads in flight at once (the row stride 129 rules out 16-byte copies); the caller's barrier follows cp_async_wait_all
template <typename T>
__device__ __forceinline__ void load_lower_block(T* S, const T* __restrict__ A, int64_t lda, int n) {
  const int c = threadIdx.x & 127, rh = threadIdx.x >> 7;  // 2 rows per pass
#pragma unroll 8
  for (int u = 0; u < 64; ++u) {
    const int r = 2 * u + rh;
    if (r < n && c <= r) cp_async_elem<T>(S + r * LS + c, A + (int64_t)r * lda + c);
    else S[r * LS + c] = (r >= n && c == r) ? T(1) : T(0);
  }
  cp_async_wait_all();
}

template <typename T>
__device__ __forceinline__ void write_dinv(const T* S, T* __restrict__ dinv) {
  const int c = threadIdx.x & 127, rh = threadIdx.x >> 7;
#pragma unroll 8
  for (int r0 = 0; r0 < NB; r0 += 2) {
    const int r = r0 + rh;
    dinv[r * NB + c] = c <= r ? S[c * LS + r] : T(0);
  }
}

// inverses of the two 64x64 diagonal sub-blocks only: dinv64[b][r][c], b = 0, 1 (slim leaf, see potrf_panel_kernel)
template <typename T>
__device__ __forceinline__ void write_dinv64(const T* S, T* __restrict__ dinv) {
  const int c = threadIdx.x & 63, rq = threadIdx.x >> 6;  // 4 rows per pass
#pragma unroll 4
  for (int e = 0; e < 32; ++e) {
    const int b = e >> 4, r = (e & 15) * 4 + rq;
    dinv[b * 4096 + r * 64 + c] = c <= r ? S[(64 * b + c) * LS + 64 * b + r] : T(0);
  }
}

// ---- leaf: factor + invert one diagonal block (n <= 128) ------------------------------------------
// SLIM = false: leaves the full 128x128 inverse of the block in dinv (inverse-based panel solve by one GEMM).
// SLIM = true : leaves only the inverses of the two 64x64 diagonal sub-blocks ([2][64][64]); the rows below are
//               solved by potrf_panel_kernel, which needs no more, and the 64x64 off-diagonal block of the
//               inverse (two 64^3 products on ONE SM, ~13 us) leaves the critical path of the factorisation.
template <typename T, bool SLIM>
__global__ void __launch_bounds__(256, 1)
potrf_leaf_kernel(T* __restrict__ A, int64_t lda, int n, T* __restrict__ dinv, int32_t* info, int info_base,
                  long long* dbg, int* wait_flag, int wait_target, int64_t batch_stride, int* done_flag) {
  // grid > 1: a BATCH of independent blocks (gpk_potrf_batched, n <= 128), block b at A + b * batch_stride with its own
  // inverse slot and info word
  A += (int64_t)blockIdx.x * batch_stride;
  dinv += (size_t)blockIdx.x * NB * NB;
  if (info) info += blockIdx.x;
  extern __shared__ __align__(16) unsigned char leaf_smem[];
  T* S = reinterpret_cast<T*>(leaf_smem);  // [128][129]
  T* ldiag = S + NB * LS;                  // [128] diagonal of L
  T* tmp = ldiag + NB;                     // 4096-element scratch (panel staging / inverse products)
  const int tid = threadIdx.x;
  const int tr = tid >> 3, tc = tid & 7;   // 32 x 8 thread grid, interleaved 4x4 micro-tiles

#define GPK_DBG(i) do { if (dbg && tid == 0) dbg[i] = clock64(); } while (0)
  if (tid == 0 && blockIdx.x == 0) trace_mark(1, 0);
  if (wait_flag) {  // look-ahead: the trailing update still running on the main stream publishes its
    if (tid == 0) { // head tiles (this block's inputs) through a counter; bounded spin, never a hang
      unsigned spins = 0;
      while (atomicAdd(wait_flag, 0) < wait_target) {
        __nanosleep(256);
        if (++spins > (1u << 24)) __trap();
      }
      __threadfence();
    }
    __syncthreads();
  }
  GPK_DBG(0);
  if (tid == 0 && blockIdx.x == 0) trace_mark(1, 1);  // inputs ready
  load_lower_block<T>(S, A, lda, n);
  __syncthreads();
  GPK_DBG(1);

  // Per 32-column step J: rows below by substitution, trailing update with IN-LEAF LOOK-AHEAD -- the first block
  // pair of the update is the next diagonal block, and as soon as the two warps that own it are done (named
  // barrier) warp 0 factors it while the other warps finish the update.  Step -1 only factors block 0.  (One call
  // site per phase: the fully unrolled phases are large and the kernel must stay inside the instruction cache.)
#pragma unroll 1
  for (int J = -1; J < 3; ++J) {
    const int jb = J * 32;
    const int t0 = jb + 32, nr = NB - t0;
    const int grp = tid >> 6;
    if (J >= 0) {
      // panel rows t0..127:  X = B L_JJ^-T by forward substitution, ONE THREAD PER ROW with the row's 32 entries
      // in registers; L_JJ (strict lower part) and 1/diag are warp-wide broadcasts from shared memory
      if (tid < nr) {
        T* rowp = S + (t0 + tid) * LS + jb;
        const T* Lj = S + jb * LS + jb;
        T b[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) b[k] = rowp[k];
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const T xk = b[k] * Lj[k * LS + k];  // diagonal slot holds 1/L_kk
          b[k] = xk;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j > k) b[j] = fma(-xk, Lj[j * LS + k], b[j]);
        }
#pragma unroll
        for (int k = 0; k < 32; ++k) rowp[k] = b[k];
      }
      __syncthreads();
      if (J == 0) GPK_DBG(4);
      // trailing update by 32x32 block pairs (rb >= cb):  C[r][c] -= sum_k S[r][jb+k] S[c][jb+k]
      const int nblk = nr / 32, npairs = nblk * (nblk + 1) / 2;
      if (sizeof(T) == 8) {
        // fp64 (DMMA): pair 0 = the next diagonal block by ALL warps (0.6k cycles instead of 3.6k on two warps that share
        // their DP pipes with the rest), barrier, then warp 0 factors it while warps 1-3 and 5-7 apply the other pairs in
        // 16-row halves; warp 4 shares warp 0's scheduler and stays idle (the concurrent update slowed the 32x32
        // factorisation from 8.6k to 10.6k cycles: scripts/leaf_timing.py)
        const int w8 = tid >> 5;
        leaf_pair0_all(reinterpret_cast<double*>(S), t0, jb, w8, tid & 31);
        __syncthreads();
        if (J == 0) GPK_DBG(10);
        if (w8 != 0 && w8 != 4) {
          const int wi = w8 < 4 ? w8 - 1 : w8 - 2;  // 0..5
          for (int u = wi; u < 2 * (npairs - 1); u += 6) {
            const int pr = 1 + (u >> 1);
            int rbk = 0, rem = pr;
            while (rem > rbk) { rem -= rbk + 1; ++rbk; }  // pr -> (rbk, cbk = rem), cbk <= rbk
            leaf_pair_half(reinterpret_cast<double*>(S), t0 + rbk * 32, t0 + rem * 32, jb, u & 1, tid & 31);
          }
        }
      } else {
        // fp32: 64 threads (8x8 interleaved 4x4 micro-tiles) per pair; pair 0 = the next diagonal block, done by warps 0-1 only
        const int sub = tid & 63;
        int pr = grp;
        while (pr < npairs) {
          int rbk = 0, rem = pr;
          while (rem > rbk) { rem -= rbk + 1; ++rbk; }  // pr -> (rbk, cbk = rem), cbk <= rbk
          const int cbk = rem;
          const int R0 = t0 + rbk * 32, C0 = t0 + cbk * 32;
          leaf_pair_update(S, R0, C0, jb, sub);
          if (grp == 0) break;              // warps 0-1 go on to the next diagonal block
          pr = pr < 4 ? 3 + grp : pr + 3;   // the other three groups share the remaining pairs
        }
        if (grp == 0) asm volatile("bar.sync 1, 64;" ::: "memory");  // the next diagonal block is up to date
        if (J == 0) GPK_DBG(10);
      }
    }
    if (__all_sync(0xffffffffu, tid < 32)) {  // warp-uniform by construction: the vote tells the compiler so
      const int bad = warp_chol32<T>(S, t0, ldiag);
      if (bad && tid == 0 && info) atomicCAS(info, 0, info_base + t0 + bad);
      if (J == 0) GPK_DBG(11);
    }
    __syncthreads();
    if (J == -1) { GPK_DBG(2); GPK_DBG(3); }
    if (J == 0) GPK_DBG(5);
  }
  GPK_DBG(6);

  // L back to global (lower part of the first n rows), coalesced along columns
  {
    const int c = tid & 127, rh = tid >> 7;
#pragma unroll 1
    for (int r0 = 0; r0 < NB; r0 += 64) {
      T v[32];
#pragma unroll
      for (int u = 0; u < 32; ++u) {
        const int r = r0 + 2 * u + rh;
        v[u] = c == r ? ldiag[r] : S[r * LS + c];
      }
#pragma unroll
      for (int u = 0; u < 32; ++u) {
        const int r = r0 + 2 * u + rh;
        if (r < n && c <= r) A[(int64_t)r * lda + c] = v[u];
      }
    }
  }
  GPK_DBG(7);
  if (__all_sync(0xffffffffu, tid < 128)) warp_inv32<T>(S, (tid >> 5) * 32);  // the four 32x32 diagonal inverses, one warp each
  __syncthreads();
  invert_offdiag_128<T>(S, tmp, !SLIM);
  GPK_DBG(8);
  if (SLIM) write_dinv64<T>(S, dinv); else write_dinv<T>(S, dinv);
  __syncthreads();
  GPK_DBG(9);
  if (done_flag && tid == 0) {  // (after the barrier above: L and the inverses of every thread are stored) the panel kernel
    __threadfence();            // below this block is already resident and polls this counter instead of waiting for a launch
    atomicAdd(done_flag, 1);
  }
  if (tid == 0 && blockIdx.x == 0) trace_mark(1, 2);
#undef GPK_DBG
}

// ---- panel solve below a diagonal block (fp64): X = B L^-T for 64 rows per CTA -------------------------
// With L = [A 0; C D] (64x64 blocks):  X1 = B1 A^-T,  T = B2 - X1 C^T,  X2 = T D^-T  -- three 64-deep products on
// DMMA (mma.sync.m8n8k4.f64), the triangular ones skipping their zero k-blocks.  Each WARP owns 8 rows through
// all three phases (operands A^-1, C, D^-1 are CTA-shared and read-only), so the phases need only __syncwarp.
constexpr int PR = 64;    // panel rows per CTA
constexpr int PLB = 132;  // row stride of the staged panel rows (= 4 mod 16: minimal-wavefront fragment loads)
constexpr int PLW = 68;   // row stride of the 64-wide operands


// Optional extras of the panel kernel (both off = the plain solve):
//  * PanelEmit: the finished rows are also written as int8 digit planes into the plane store (planes.cuh), with the
//    static row scales -- this replaces the slicing pass over L in front of every tcgen05 update;
//  * PanelFuse: the K = 128 trailing update of the NEXT block column, C[rows, 0:uc] -= X X_top^T with X_top = the first
//    `uc` solved rows (they belong to the first two CTAs, which publish them through a counter), is applied by the same
//    CTA while X is still in shared memory; CTAs holding rows of the next diagonal block report them to the look-ahead
//    counter, so the next leaf starts while the rest of the grid is still updating.
struct PanelEmit {
  TcPlanes pl;        // pl.planes == nullptr: off
  int64_t row_g0;     // global row index of B's first row
  int64_t col_g0;     // global column index of the block
  int64_t dyn_k0;     // dyn_K > 0: the tcgen05 update of the k-range [dyn_k0, dyn_k0 + dyn_K) follows this panel (it ends at
  int64_t dyn_K;      // this block); the CTAs that own rows below the square part slice them for it (dynamic scales)
  int* leaf_flag;     // not nullptr: the leaf of this block runs CONCURRENTLY (other stream); its outputs (Lblk, dinv64) are
  int leaf_target;    // valid once *leaf_flag >= leaf_target.  The CTA's own rows are fetched before the wait.
};
constexpr int PCR = 16;  // rows per CRITICAL CTA of the fused panel (see the row mapping in the kernel)
struct PanelFuse {
  double* C;          // nullptr: off.  C[rows, uc] (same rows as B), leading dimension ldb
  int uc;             // columns of the update (<= 128)
  int ncrit;          // CTAs (PCR rows each) that cover the first uc rows = X_top = the next diagonal block
  int* flag;          // [1]: 32x32 units of the next diagonal block done, [2]: X_top CTAs finished (never reset during a
  int xtop_target;    // factorisation: waits compare against running totals) -- flag[2] value once all of X_top is stored
  int64_t mu, nu;     // shape of the whole update (rows, uc) for diag_units_tile
};

__global__ void __launch_bounds__(256, 1)
potrf_panel_kernel(double* __restrict__ B, int64_t ldb, int64_t rows, const double* __restrict__ Lblk, int64_t ldl,
                   int nb, const double* __restrict__ dinv64, PanelEmit em, PanelFuse fu) {
  extern __shared__ __align__(16) unsigned char leaf_smem[];
  double* Bs = reinterpret_cast<double*>(leaf_smem);  // [64][PLB]
  double* Ai = Bs + PR * PLB;                          // [64][PLW]  A^-1
  double* Di = Ai + 64 * PLW;                          // [64][PLW]  D^-1
  double* Cs = Di + 64 * PLW;                          // [64][PLW]  C = L[64:128, 0:64]
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, q = lane & 3;
  // Row mapping.  Plain: 64 rows per CTA.  Fused: the first fu.ncrit CTAs take PCR = 16 rows each of the CRITICAL rows (the
  // rows of the next diagonal block: X_top, and the block the next leaf is waiting for) -- two active warps per SM instead of
  // eight sharing the DMMA pipe, so their solve + update finish in a fraction of the time; the rest 64 rows each below them.
  const int ncrit = fu.C ? fu.ncrit : 0;
  const bool critical = (int)blockIdx.x < ncrit;
  const int nrows_cta = critical ? PCR : PR;
  const int64_t r0 = critical ? (int64_t)blockIdx.x * PCR : (int64_t)ncrit * PCR + (int64_t)(blockIdx.x - ncrit) * PR;
  const bool wact = w * 8 < nrows_cta;  // warps beyond the CTA's rows only help with the cooperative loads / emission
  const int trace_id = fu.C ? 2 : 3;
  if (tid == 0 && blockIdx.x == 0) trace_mark(trace_id, 0);
  double* Bw = Bs + (w * 8) * PLB;  // this warp's 8 rows
  // Operands (A^-1, D^-1, C: 3 x 32 KB) and the CTA's rows (up to 64 KB) come in as 16-byte asynchronous copies, all in
  // flight at once: one L2 round trip + the transfer (~1.7 us with every SM loading) instead of 16 dependent rounds of
  // 8-byte loads (4.1 us of the 12.9 us panel, device timeline profiles/r2/trace_c2_phases.csv).
  const bool async_ok = nb == NB && (ldb & 1) == 0 && (ldl & 1) == 0 && ((reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(Lblk) |
                                                                           reinterpret_cast<uintptr_t>(dinv64)) & 15) == 0;
  auto wait_leaf = [&]() {  // flag hop instead of a launch boundary between the leaf and this kernel (~3.5 us of the chain)
    if (!em.leaf_flag) return;
    if (tid == 0) {
      unsigned spins = 0;
      while (atomicAdd(em.leaf_flag, 0) < em.leaf_target) {
        __nanosleep(32);
        if (++spins > (1u << 25)) __trap();
      }
      __threadfence();
    }
    __syncthreads();
  };
  if (async_ok) {
    for (int e = tid; e < nrows_cta * 64; e += 256) {  // rows x 64 chunks (independent of the leaf: issued first)
      const int rl = e >> 6, c2 = (e & 63) * 2;
      const int64_t row = r0 + rl;
      cp_async16(Bs + rl * PLB + c2, B + (row < rows ? row : 0) * ldb + c2, row < rows);
    }
    wait_leaf();
    for (int e = tid; e < 2048; e += 256) {  // 64 rows x 32 chunks of 2 doubles
      const int i = e >> 5, j2 = (e & 31) * 2;
      cp_async16(Ai + i * PLW + j2, dinv64 + i * 64 + j2, true);
      cp_async16(Di + i * PLW + j2, dinv64 + 4096 + i * 64 + j2, true);
      cp_async16(Cs + i * PLW + j2, Lblk + (int64_t)(64 + i) * ldl + j2, true);
    }
    cp_async_wait_all();
  } else {
    wait_leaf();
    for (int e = tid; e < 4096; e += 256) {
      const int i = e >> 6, j = e & 63;
      Ai[i * PLW + j] = __ldcg(dinv64 + e);
      Di[i * PLW + j] = __ldcg(dinv64 + 4096 + e);
      Cs[i * PLW + j] = (64 + i < nb) ? __ldcg(Lblk + (int64_t)(64 + i) * ldl + j) : 0.0;
    }
    if (wact) {
#pragma unroll
      for (int rr = 0; rr < 8; ++rr) {
        const int64_t row = r0 + w * 8 + rr;
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const int c = lane + 32 * cc;
          Bw[rr * PLB + c] = (row < rows && c < nb) ? B[row * ldb + c] : 0.0;
        }
      }
    }
  }
  __syncthreads();
  if (tid == 0 && blockIdx.x == 0) trace_mark(trace_id, 10);  // operands + own rows staged

  double acc[8][2], af[16];
  if (wact) {
  // ---- phase 1: X1 = B1 A^-T;  (A^-T)[k][n] = Ai[n][k], zero for k > n
#pragma unroll
  for (int ks = 0; ks < 16; ++ks) af[ks] = Bw[g * PLB + ks * 4 + q];
#pragma unroll
  for (int cb = 0; cb < 8; ++cb) acc[cb][0] = acc[cb][1] = 0.0;
#pragma unroll
  for (int ks = 0; ks < 16; ++ks)  // k outer: consecutive DMMAs hit different accumulators (no dependent issue)
#pragma unroll
    for (int cb = ks >> 1; cb < 8; ++cb) dmma884p(acc[cb], af[ks], Ai[(cb * 8 + g) * PLW + ks * 4 + q]);
  __syncwarp();
#pragma unroll
  for (int cb = 0; cb < 8; ++cb)
    *reinterpret_cast<double2*>(Bw + g * PLB + cb * 8 + 2 * q) = make_double2(acc[cb][0], acc[cb][1]);
  __syncwarp();
  // ---- phase 2: T = B2 - X1 C^T
#pragma unroll
  for (int ks = 0; ks < 16; ++ks) af[ks] = -Bw[g * PLB + ks * 4 + q];
#pragma unroll
  for (int cb = 0; cb < 8; ++cb) {
    const double2 b2 = *reinterpret_cast<const double2*>(Bw + g * PLB + 64 + cb * 8 + 2 * q);
    acc[cb][0] = b2.x;
    acc[cb][1] = b2.y;
  }
#pragma unroll
  for (int ks = 0; ks < 16; ++ks)
#pragma unroll
    for (int cb = 0; cb < 8; ++cb) dmma884p(acc[cb], af[ks], Cs[(cb * 8 + g) * PLW + ks * 4 + q]);
  __syncwarp();
#pragma unroll
  for (int cb = 0; cb < 8; ++cb)
    *reinterpret_cast<double2*>(Bw + g * PLB + 64 + cb * 8 + 2 * q) = make_double2(acc[cb][0], acc[cb][1]);
  __syncwarp();
  // ---- phase 3: X2 = T D^-T
#pragma unroll
  for (int ks = 0; ks < 16; ++ks) af[ks] = Bw[g * PLB + 64 + ks * 4 + q];
#pragma unroll
  for (int cb = 0; cb < 8; ++cb) acc[cb][0] = acc[cb][1] = 0.0;
#pragma unroll
  for (int ks = 0; ks < 16; ++ks)
#pragma unroll
    for (int cb = ks >> 1; cb < 8; ++cb) dmma884p(acc[cb], af[ks], Di[(cb * 8 + g) * PLW + ks * 4 + q]);
  __syncwarp();
#pragma unroll
  for (int cb = 0; cb < 8; ++cb)
    *reinterpret_cast<double2*>(Bw + g * PLB + 64 + cb * 8 + 2 * q) = make_double2(acc[cb][0], acc[cb][1]);
  __syncwarp();
  // ---- own rows back to global
#pragma unroll
  for (int rr = 0; rr < 8; ++rr) {
    const int64_t row = r0 + w * 8 + rr;
    if (row < rows) {
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int c = lane + 32 * cc;
        if (c < nb) B[row * ldb + c] = Bw[rr * PLB + c];
      }
    }
  }
  }  // wact
  if (tid == 0 && blockIdx.x == 0) trace_mark(trace_id, 11);  // solved rows stored
  // ---- fused K = nb update of the next block column: X_top published first (everybody needs it)
  if (fu.C) {
    const int ntop = ncrit;                  // CTAs that own rows of X_top
    __syncthreads();                         // all warps' rows are in global memory
    if ((int)blockIdx.x < ntop && tid == 0) {
      __threadfence();
      atomicAdd(fu.flag + 2, 1);
    }
  }
  // ---- digit planes of the finished rows (static scales; the extra rows below the square part are sliced elsewhere).
  // One item = 16 consecutive k of one row = 16 contiguous bytes of every plane in the tile image; consecutive lanes
  // take consecutive rows, so a warp's 16-byte stores fill whole 128-byte lines (4-byte stores per lane cost 8 us per
  // launch: as much as the slicing pass this replaces).
  auto emit_planes = [&]() {
    if (!(em.pl.planes && nb == NB)) return;
    if (!fu.C) __syncthreads();  // (the fused path has passed a barrier already) all warps' rows are in Bs
    const int S = em.pl.S;
    const TcDigitizer dz(S);
#pragma unroll 1
    for (int e = tid; e < nrows_cta * 8; e += 256) {
      const int rl = e % nrows_cta, ch = e / nrows_cta;  // local row, 16-column chunk
      const int64_t row = r0 + rl, grow = em.row_g0 + row;
      if (row >= rows || grow >= em.pl.n_sq) continue;
      const double inv = 1.0 / em.pl.rowscale[grow];  // exact: a power of two
      double v[16];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const double2 t2 = *reinterpret_cast<const double2*>(Bs + rl * PLB + ch * 16 + 2 * u);
        v[2 * u] = t2.x * inv;
        v[2 * u + 1] = t2.y * inv;
      }
      const int64_t kcol = em.col_g0 + ch * 16;
      int8_t* tb = em.pl.tile(grow >> 7, kcol / TC_KB) + tc_tile_off((int)(grow & 127), (int)(kcol % TC_KB));
      // digit bytes of every value (planes.cuh), 4 x 4 byte transposes, then one 16-byte store per plane
      uint32_t wd[4][8];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const double v4[4] = {v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]};
        tc_digit_words(dz, v4, wd[g]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < S) *reinterpret_cast<uint4*>(tb + (size_t)(S - 1 - j) * TC_ATILE) = make_uint4(wd[0][j], wd[1][j], wd[2][j], wd[3][j]);
    }
  };
  // CTAs that hold rows of the next diagonal block update and publish them first (the next leaf is waiting for them) and
  // emit their planes afterwards; everybody else emits while waiting for X_top
  if (!critical) emit_planes();
  if (!fu.C) {
    // rows below the square part (the (Y - m)^T rows that ride along): sliced here for the update that follows, with the
    // scale of their maximum over its k-range -- everything left of this block is in global memory since earlier launches,
    // this block's columns since the stores above.  (A slicing launch between this panel and the update costs ~6 us of
    // the dependent chain, 31 times per evaluation at N = 8192.)
    if (em.dyn_K > 0 && em.pl.planes && em.row_g0 + r0 + nrows_cta > em.pl.n_sq) {
      __shared__ double wmax[8];
      __syncthreads();
      for (int rl = 0; rl < nrows_cta; ++rl) {
        const int64_t row = r0 + rl, grow = em.row_g0 + row;
        if (row >= rows || grow < em.pl.n_sq) continue;
        tc_slice_row_cta(B + row * ldb + (em.dyn_k0 - em.col_g0), grow, em.dyn_k0, em.dyn_K, em.pl, wmax);
      }
    }
    if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) trace_mark(trace_id, blockIdx.x == 0 ? 2 : 3);
    return;
  }
  // ---- C[own rows, 0:uc] -= X[own rows, 0:nb] X_top[0:uc, 0:nb]^T
  {
    double* Xt = Ai;  // [128][PLB] staged X_top: reuses the operand area (everybody passed the barrier above)
    if (tid == 0) {
      unsigned spins = 0;
      while (atomicAdd(fu.flag + 2, 0) < fu.xtop_target) {
        __nanosleep(64);
        if (++spins > (1u << 24)) __trap();
      }
      __threadfence();
    }
    __syncthreads();
    if (tid == 0 && blockIdx.x == 0) trace_mark(trace_id, 12);  // X_top complete (all critical CTAs stored)
    // (L2 copies: the rows were written by other CTAs of this grid; cp.async.cg does not look in L1)
    if ((ldb & 1) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0) {
      for (int e = tid; e < NB * 64; e += 256) {  // 128 rows x 64 chunks of 2 doubles
        const int i = e >> 6, c2 = (e & 63) * 2;
        cp_async16(Xt + i * PLB + c2, B + (int64_t)(i < fu.uc ? i : 0) * ldb + c2, i < fu.uc);
      }
      cp_async_wait_all();
    } else {
      for (int e = tid; e < NB * NB; e += 256) {
        const int i = e >> 7, c = e & 127;
        Xt[i * PLB + c] = i < fu.uc ? __ldcg(B + (int64_t)i * ldb + c) : 0.0;
      }
    }
    // accumulators = 8 rows of C (DMMA C-fragment layout: row g, columns 8 cb + 2q, +1).  Non-critical CTAs: warp w owns
    // rows 8w.. and all 16 column blocks.  Critical CTAs (16 rows) spread the update over all 8 warps -- warp w takes rows
    // 8 (w & 1).. and the 4 column blocks from 4 (w >> 1): 128 DMMAs per warp instead of 512 on two warps (the update was
    // 6.9 us of the 19 us between the start of the kernel and the publish; profiles/r2/trace_c2_phases.csv).
    auto update = [&](auto ncb_c, const int urow, const int cb0, const bool uact) {
      constexpr int NCB = decltype(ncb_c)::value;
      const double* Bu = Bs + urow * PLB;
      const int64_t crow = r0 + urow + g;
      const bool rok = uact && crow < rows;
      double cacc[NCB][2];
#pragma unroll
      for (int cbi = 0; cbi < NCB; ++cbi) {
        const int c = (cb0 + cbi) * 8 + 2 * q;
        cacc[cbi][0] = (rok && c < fu.uc) ? fu.C[crow * ldb + c] : 0.0;
        cacc[cbi][1] = (rok && c + 1 < fu.uc) ? fu.C[crow * ldb + c + 1] : 0.0;
      }
      __syncthreads();
      if (tid == 0 && blockIdx.x == 0) trace_mark(trace_id, 13);  // X_top staged, C fragments loaded
      if (uact) {
#pragma unroll 1
        for (int kh = 0; kh < 2; ++kh) {  // two halves of k keep the A fragments at 16 registers
#pragma unroll
          for (int ks = 0; ks < 16; ++ks) af[ks] = -Bu[g * PLB + kh * 64 + ks * 4 + q];
#pragma unroll
          for (int ks = 0; ks < 16; ++ks)
#pragma unroll
            for (int cbi = 0; cbi < NCB; ++cbi)
              dmma884p(cacc[cbi], af[ks], Xt[((cb0 + cbi) * 8 + g) * PLB + kh * 64 + ks * 4 + q]);
        }
      }
      if (rok) {
#pragma unroll
        for (int cbi = 0; cbi < NCB; ++cbi) {
          const int c = (cb0 + cbi) * 8 + 2 * q;
          if (c < fu.uc) fu.C[crow * ldb + c] = cacc[cbi][0];
          if (c + 1 < fu.uc) fu.C[crow * ldb + c + 1] = cacc[cbi][1];
        }
      }
    };
    if (critical) update(std::integral_constant<int, 4>{}, (w & 1) * 8, (w >> 1) * 4, true);
    else update(std::integral_constant<int, 16>{}, w * 8, 0, wact);
    // look-ahead: the critical CTAs hold the rows of the next diagonal block; the next leaf waits for all of them
    if (critical) {
      __syncthreads();
      if (tid == 0) {
        __threadfence();
        atomicAdd(fu.flag + 1, 1);
        if (blockIdx.x == 0) trace_mark(trace_id, 1);  // first critical CTA published
      }
    }
  }
  if (critical) emit_planes();
  if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) trace_mark(trace_id, blockIdx.x == 0 ? 2 : 3);
}

static size_t panel_smem_bytes(bool fused = false) {
  return (size_t)(PR * PLB + (fused ? NB * PLB : 3 * 64 * PLW)) * sizeof(double);
}

// ---- standalone inverse of the diagonal blocks of a given factor (for trsm without cached dinv) -----
template <typename T>
__global__ void __launch_bounds__(256, 1)
trtri_diag_kernel(const T* __restrict__ L, int64_t ldl, int64_t n, T* __restrict__ dinv) {
  extern __shared__ __align__(16) unsigned char leaf_smem[];
  T* S = reinterpret_cast<T*>(leaf_smem);
  T* tmp = S + NB * LS + NB;
  const int tid = threadIdx.x;
  const int64_t b0 = (int64_t)blockIdx.x * NB;
  const int nb = (int)min((int64_t)NB, n - b0);
  load_lower_block<T>(S, L + b0 * ldl + b0, ldl, nb);
  __syncthreads();
  if (tid < NB) S[tid * LS + tid] = T(1) / S[tid * LS + tid];  // diagonal slot holds inv(L)_kk
  __syncthreads();
  if (__all_sync(0xffffffffu, tid < 128)) warp_inv32<T>(S, (tid >> 5) * 32);
  __syncthreads();
  invert_offdiag_128<T>(S, tmp);
  write_dinv<T>(S, dinv + (size_t)blockIdx.x * NB * NB);
}

template <typename T>
static size_t leaf_smem_bytes() { return (size_t)(NB * LS + NB + 4096) * sizeof(T); }

template <typename T>
static int leaf_attr() {
  static PerDeviceOnce once;  // function attributes are per device
  return once.run([&]() -> int {
    GPK_CUDA_OK(cudaFuncSetAttribute(potrf_leaf_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)leaf_smem_bytes<T>()));
    GPK_CUDA_OK(cudaFuncSetAttribute(potrf_leaf_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)leaf_smem_bytes<T>()));
    GPK_CUDA_OK(cudaFuncSetAttribute(potrf_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)panel_smem_bytes(true)));
    GPK_CUDA_OK(cudaFuncSetAttribute(trtri_diag_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)leaf_smem_bytes<T>()));
    return 0;
  });
}

static inline int64_t split_point(int64_t n) { return ((n / NB + 1) / 2) * NB; }

// Updates with K below this use the DMMA kernel (slicing + epilogue overhead of the int8 path).
constexpr int64_t TC_MIN_K = 256;

// ---- look-ahead context ------------------------------------------------------------------------------
// The trailing update U (main stream) and the next diagonal-block factorisation (side stream) overlap:
// U processes the tiles of its first 128-column block first and counts them in `flag`; the leaf kernel
// spins on that counter, so it runs while U is still working on the remaining tiles.
struct LookAhead {
  cudaStream_t side = nullptr;
  cudaEvent_t ev_inputs = nullptr, ev_side = nullptr, ev_u = nullptr;
  int* flag = nullptr;     // device counters (in the workspace): [0] head tiles done, [1] diagonal units done, [2] X_top CTAs
  int target = 0;          // value of flag[1] the next leaf waits for
  int base1 = 0, base2 = 0;  // running totals of flag[1] / flag[2]: the counters are zeroed once per factorisation
  int64_t follow_k0 = -1, follow_K = 0;  // the tcgen05 update that directly follows the block being factored (0: none)
  int64_t dyn_k0 = -1, dyn_K = 0;        // k-range whose extra-row planes the last panel kernel has already written
  bool pending = false;
  bool flaghop = false;    // slim + look-ahead: leaves alone on the side stream, panels / updates on the main stream; a panel
  bool side_started = false;  // kernel waits for its leaf through flag[3] (leaves_done) instead of a cross-stream event
  int leaves_done = 0;
  bool enabled = false;
  bool slim = false;       // fp64, n > 128: slim leaves + potrf_panel_kernel (full block inverses filled in afterwards)
  bool fuse = false;       // slim + look-ahead: the K = 128 updates are applied by the panel kernel itself
  TcPlanes pl;             // digit-plane store of this factorisation (pl.planes == nullptr: tcgen05 updates off)
};

static int num_sms() {  // of the CURRENT device (a process may drive several)
  int dev = 0, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n > 0 ? n : 148;
}

// Polling panel kernels are only safe while no OTHER factorisation competes for the SMs with polling kernels of its own
// (four models on four streams: 4 x 64 polling CTAs fill the GPU and lock every leaf out).  One factorisation per device
// may poll at a time: a factorisation enqueued while the previous one on a different stream is still in flight keeps
// the event-ordered launches, whose only spinning kernels are single-CTA leaves.
struct FlightReg { cudaEvent_t ev = nullptr; cudaStream_t stream = nullptr; bool valid = false; };
static std::mutex g_flight_mu;
static std::map<int, FlightReg> g_flight;

// (both under g_flight_mu, which potrf_t holds from the check to the mark: the enqueue of one factorisation, ~1 ms of host time)
static bool flight_alone(cudaStream_t st) {
  int dev = 0;
  cudaGetDevice(&dev);
  auto it = g_flight.find(dev);
  if (it == g_flight.end() || !it->second.valid || it->second.stream == st) return true;
  const cudaError_t q = cudaEventQuery(it->second.ev);
  if (q == cudaSuccess) return true;
  cudaGetLastError();  // (cudaErrorNotReady is not an error here)
  return false;
}

static int flight_mark(cudaStream_t st) {
  int dev = 0;
  GPK_CUDA_OK(cudaGetDevice(&dev));
  FlightReg& r = g_flight[dev];
  if (!r.ev) GPK_CUDA_OK(cudaEventCreateWithFlags(&r.ev, cudaEventDisableTiming));
  GPK_CUDA_OK(cudaEventRecord(r.ev, st));
  r.stream = st;
  r.valid = true;
  return 0;
}

static int lookahead_init(LookAhead& la, int* flag, cudaStream_t st) {
  // one side stream + event set per (device, caller stream): independent factorisations issued on
  // different streams (e.g. one model per output) never share look-ahead state
  struct Res { cudaStream_t side; cudaEvent_t ev[3]; };
  static std::map<std::pair<int, cudaStream_t>, Res> pool;
  static std::mutex mu;
  if (!flag) return 0;
  int dev = 0;
  GPK_CUDA_OK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  auto it = pool.find({dev, st});
  if (it == pool.end()) {
    Res r;
    GPK_CUDA_OK(cudaStreamCreateWithFlags(&r.side, cudaStreamNonBlocking));
    for (int i = 0; i < 3; ++i) GPK_CUDA_OK(cudaEventCreateWithFlags(&r.ev[i], cudaEventDisableTiming));
    it = pool.emplace(std::make_pair(dev, st), r).first;
  }
  la.side = it->second.side;
  la.ev_inputs = it->second.ev[0];
  la.ev_side = it->second.ev[1];
  la.ev_u = it->second.ev[2];
  la.flag = flag;
  la.enabled = true;
  return 0;
}

// C = A[col0 + n1 :, col0 + n1 : col0 + n] -= P P[0 : n - n1]^T with P = the finished columns [col0, col0 + K) below
// eager creation of the (device, stream) look-ahead resources (gpk_warm): the first factorisation on a stream otherwise
// creates one side stream and three events lazily
int lookahead_warm(cudaStream_t st) {
  LookAhead la;
  int dummy = 0;
  return lookahead_init(la, &dummy, st);
}

// int32 accumulators: 128 * 128 * K * S < 2^31 (radix-256 digits; tests/test_digit_slicing_model.py); deeper updates use DMMA
template <typename T>
static bool tc_update_eligible(const LookAhead& la, int64_t m, int64_t n, int64_t K) {
  return sizeof(T) == 8 && la.pl.planes && K >= TC_MIN_K && K % 32 == 0 && n <= m && K * la.pl.S * 16384 < (1ll << 31);
}

template <typename T>
static int trailing_update(T* C, int64_t ldc, int64_t m, int64_t n, const T* P, int64_t ldp, int64_t K, int64_t col0,
                           LookAhead& la, cudaStream_t st) {
  GemmOpts opts;
  const bool use_tc = tc_update_eligible<T>(la, m, n, K);
  if (use_tc) {
    // operand rows without a static scale: the extra rows below the square part
    const int64_t r0 = col0 + K;
    const int64_t dyn0 = la.pl.n_sq > r0 ? la.pl.n_sq : r0;
    if (dyn0 < r0 + m && !(la.dyn_k0 == col0 && la.dyn_K == K))  // (else: the last panel kernel did it)
      GPK_TRY(tc_slice_rows((const double*)P + (dyn0 - r0) * ldp, ldp, dyn0, r0 + m - dyn0, col0, K, la.pl, st));
  }
  if (la.enabled) {
    opts.head_flag = la.flag;
    la.base1 += diag_units_total(m, n);  // 32x32 units of the next 128x128 diagonal block
    la.target = la.base1;
    if (!la.flaghop) GPK_CUDA_OK(cudaEventRecord(la.ev_inputs, st));  // everything the next leaf needs except U itself
    la.pending = true;
  }
  int rc;
  if (use_tc)
    rc = syrk_tc_planes((double*)C, ldc, m, n, la.pl, col0 + K, col0, K, 1, st, &opts);
  else
    rc = gemm_t<T>(0, 1, m, n, K, T(-1), P, ldp, P, ldp, T(1), C, ldc, GPK_GEMM_LOWER_ONLY, st, &opts);
  if (rc == 0 && la.enabled && !la.flaghop) GPK_CUDA_OK(cudaEventRecord(la.ev_u, st));  // U complete
  return rc;
}

// (fp32 factorisations by way of the fp64 path: potrf_f32_via_f64 below)
static bool f32_detour_applies(int64_t n, int64_t rows) { return rows <= n && n >= 512 && n <= 65535; }
struct F32Detour { int64_t ld64; size_t a_bytes, d_bytes, p_bytes; };
static F32Detour f32_detour_layout(int64_t n) {
  F32Detour d;
  d.ld64 = (n + 3) / 4 * 4;
  d.a_bytes = align_up((size_t)n * d.ld64 * sizeof(double), 256);
  d.d_bytes = align_up((size_t)((n + NB - 1) / NB) * NB * NB * sizeof(double) + 256, 256);
  d.p_bytes = align_up(tc_planes_bytes(n, n), 256);
  return d;
}

size_t potrf_tc_ws_bytes(int64_t n, int64_t rows, int dtype) {
  if (dtype == GPK_F32) {  // scratch of the fp64 detour of square fp32 factorisations (potrf_f32_via_f64)
    if (!f32_detour_applies(n, rows)) return 0;
    const F32Detour L = f32_detour_layout(n);
    return L.a_bytes + L.d_bytes + L.p_bytes;
  }
  if (n < 2 * 128) return 0;  // reserved from n >= 256; the updates use the planes once split_point(n) >= TC_MIN_K (n >= 384)
  return tc_planes_bytes(n, rows);
}

// One diagonal block (n <= 128) at global column col0: leaf, then the rows below.  fuse_cols > 0: the panel kernel
// also applies the K = n update of the next fuse_cols columns (the caller skips that trailing update).
template <typename T>
static int potrf_block(T* A, int64_t n, int64_t rows, int64_t lda, int32_t* info, T* dinv, int64_t col0, int fuse_cols,
                       LookAhead& la, cudaStream_t st) {
  T* dblk = dinv + (size_t)(col0 / NB) * NB * NB;
  // look-ahead: run the leaf (and its panel solve) on the side stream, gated by U's head-tile counter
  cudaStream_t ls = st;
  int* wf = nullptr;
  int wt = 0;
  int* done = nullptr;
  if (la.flaghop) {
    // Flag hops: every leaf runs on the side stream (one after the other), every panel / update on the main stream.  The leaf
    // waits for its diagonal block through flag[1] (published by the update or the fused panel before it), the panel below
    // it waits for the leaf through flag[3]; neither needs a launch boundary or a cross-stream event in between.
    if (!la.side_started) {  // the first leaf: its inputs are whatever precedes the factorisation on the caller's stream
      GPK_CUDA_OK(cudaEventRecord(la.ev_inputs, st));
      GPK_CUDA_OK(cudaStreamWaitEvent(la.side, la.ev_inputs, 0));
      la.side_started = true;
    }
    ls = la.side;
    if (la.pending) { wf = la.flag + 1; wt = la.target; }
    done = la.flag + 3;
    la.leaves_done += 1;
    la.pending = false;
  } else if (la.pending) {
    GPK_CUDA_OK(cudaStreamWaitEvent(la.side, la.ev_inputs, 0));
    ls = la.side;
    wf = la.flag + 1;  // the leaf needs only the diagonal block of U's output
    wt = la.target;
  }
  {
    ProfScope ps(PROF_LEAF, ls);
    if (la.slim)
      potrf_leaf_kernel<T, true><<<1, 256, leaf_smem_bytes<T>(), ls>>>(A, lda, (int)n, dblk, info, (int)col0, nullptr, wf, wt, 0, done);
    else
      potrf_leaf_kernel<T, false><<<1, 256, leaf_smem_bytes<T>(), ls>>>(A, lda, (int)n, dblk, info, (int)col0, nullptr, wf, wt, 0, done);
    GPK_LAUNCH_OK();
  }
  if (rows <= n) {
    if (la.pending) {
      GPK_CUDA_OK(cudaEventRecord(la.ev_side, la.side));
      GPK_CUDA_OK(cudaStreamWaitEvent(st, la.ev_side, 0));
      la.pending = false;
    }
    return 0;
  }
  PanelEmit em{};
  PanelFuse fu{};
  if (la.slim) {
    em.pl = la.pl;
    em.row_g0 = col0 + n;
    em.col_g0 = col0;
  }
  if (la.flaghop) {
    // The panel CTAs (one per SM: shared memory) spin until the leaf has finished, so the leaf must be able to get an SM
    // whatever the block scheduler does first: only grids that leave eight SMs free may poll (this leaf + the spinning
    // leaves of factorisations enqueued later on other streams, which never poll themselves: potrf_t); a larger grid
    // (N > ~9000) is ordered behind the leaf by an event, as a launch boundary would.
    const int64_t prow = rows - n;
    const int64_t ctas = fuse_cols > 0 ? (fuse_cols + PCR - 1) / PCR + (prow + PR - 1) / PR : (prow + PR - 1) / PR;
    if (ctas <= num_sms() - 8) {
      em.leaf_flag = la.flag + 3;
      em.leaf_target = la.leaves_done;
    } else {
      GPK_CUDA_OK(cudaEventRecord(la.ev_side, la.side));
      GPK_CUDA_OK(cudaStreamWaitEvent(st, la.ev_side, 0));
    }
  }
  if (la.slim && fuse_cols > 0) {
    // The fused panel + update plays the role of U: it runs on the MAIN stream (behind the previous U, which it needs
    // completely), publishes the next diagonal block through the counter and the next leaf overlaps it on the side stream.
    if (la.pending) {
      GPK_CUDA_OK(cudaEventRecord(la.ev_side, la.side));
      GPK_CUDA_OK(cudaStreamWaitEvent(st, la.ev_side, 0));
      la.pending = false;
    }
    fu.C = (double*)(A + n * lda + n);
    fu.uc = fuse_cols;
    fu.flag = la.flag;
    fu.mu = rows - n;
    fu.nu = fuse_cols;
    {
      const int64_t crit_rows = fuse_cols < rows - n ? fuse_cols : rows - n;   // rows of the next diagonal block
      fu.ncrit = (int)((crit_rows + PCR - 1) / PCR);
    }
    la.base1 += fu.ncrit;  // every critical CTA reports once
    la.base2 += fu.ncrit;  // ... and counts itself into flag[2] when its rows of X_top are stored
    la.target = la.base1;
    fu.xtop_target = la.base2;
    if (!la.flaghop) GPK_CUDA_OK(cudaEventRecord(la.ev_inputs, st));
    la.pending = true;
    {
      // work: MACs of the solve (half of rows x 128 x 128: triangular) + the fused K = 128 update
      ProfScope ps(PROF_PANEL, st, (double)(rows - n) * n * (0.5 * n + fuse_cols));
      const int64_t below = rows - n - (int64_t)fu.ncrit * PCR;
      const unsigned nblk = (unsigned)(fu.ncrit + (below > 0 ? (below + PR - 1) / PR : 0));
      potrf_panel_kernel<<<nblk, 256, panel_smem_bytes(true), st>>>((double*)(A + n * lda), lda, rows - n, (const double*)A, lda,
                                                                     (int)n, (const double*)dblk, em, fu);
      GPK_LAUNCH_OK();
    }
    if (!la.flaghop) GPK_CUDA_OK(cudaEventRecord(la.ev_u, st));
    return 0;
  }
  if (la.flaghop) ls = st;  // the panel runs on the main stream (behind the fused panel / update it needs completely)
  else if (la.pending) GPK_CUDA_OK(cudaStreamWaitEvent(la.side, la.ev_u, 0));  // the panel below needs all of U
  la.dyn_K = 0;
  if (la.slim && em.pl.planes && n == NB && la.follow_K > 0 && la.follow_k0 + la.follow_K == col0 + n && rows > la.pl.n_sq - col0) {
    // the tcgen05 update of [follow_k0, follow_k0 + follow_K) is the next launch: this panel also slices the extra rows for it
    em.dyn_k0 = la.dyn_k0 = la.follow_k0;
    em.dyn_K = la.dyn_K = la.follow_K;
  }
  if (la.slim) {
    ProfScope ps(PROF_PANEL, ls, (double)(rows - n) * n * 0.5 * n);
    const unsigned nblk = (unsigned)((rows - n + PR - 1) / PR);
    potrf_panel_kernel<<<nblk, 256, panel_smem_bytes(), ls>>>((double*)(A + n * lda), lda, rows - n, (const double*)A, lda,
                                                               (int)n, (const double*)dblk, em, fu);
    GPK_LAUNCH_OK();
  } else {  // one GEMM with the block inverse (single column tile)
    GPK_TRY(gemm_t<T>(0, 1, rows - n, n, n, T(1), A + n * lda, lda, dblk, NB, T(0), A + n * lda, lda, 0, ls));
  }
  if (la.pending) {
    GPK_CUDA_OK(cudaEventRecord(la.ev_side, la.side));
    GPK_CUDA_OK(cudaStreamWaitEvent(st, la.ev_side, 0));  // main stream joins (it also still holds U)
    la.pending = false;
  }
  return 0;
}

// (fk0, fK): the k-range of the trailing update that directly follows this sub-factorisation when it runs on tcgen05
// (fK = 0: none) -- the last panel kernel before it prepares the extra rows' digit planes (potrf_block)
template <typename T>
static int potrf_rec(T* A, int64_t n, int64_t rows, int64_t lda, int32_t* info, T* dinv, int64_t col0, LookAhead& la,
                     cudaStream_t st, int64_t fk0 = -1, int64_t fK = 0) {
  if (n <= NB) {
    la.follow_k0 = fk0;
    la.follow_K = fK;
    return potrf_block<T>(A, n, rows, lda, info, dinv, col0, 0, la, st);
  }
  const int64_t n1 = split_point(n);
  if (n <= 2 * NB && la.fuse) {  // two diagonal blocks: the K = 128 update between them is fused into the first panel
    la.follow_K = 0;
    GPK_TRY(potrf_block<T>(A, n1, rows, lda, info, dinv, col0, (int)(n - n1), la, st));
    return potrf_rec<T>(A + n1 * lda + n1, n - n1, rows - n1, lda, info, dinv, col0 + n1, la, st, fk0, fK);
  }
  const bool tc = tc_update_eligible<T>(la, rows - n1, n - n1, n1);
  GPK_TRY(potrf_rec<T>(A, n1, rows, lda, info, dinv, col0, la, st, col0, tc ? n1 : 0));
  // trailing update: A[n1:rows, n1:n] -= A[n1:rows, :n1] A[n1:n, :n1]^T  (lower tiles only)
  GPK_TRY(trailing_update<T>(A + n1 * lda + n1, lda, rows - n1, n - n1, A + n1 * lda, lda, n1, col0, la, st));
  return potrf_rec<T>(A + n1 * lda + n1, n - n1, rows - n1, lda, info, dinv, col0 + n1, la, st, fk0, fK);
}

// Number of base-256 digit planes of the tcgen05 trailing updates from what the caller knows about the conditioning
// (cond = max_i A_ii / lambda_min, e.g. (kernel variance + noise) / noise for GPR).  Measured with the NumPy emulation
// of this factorisation (scripts/radix_study.py; numerically low-rank matrices, static scales): S = 6 (+ the (3,3) product)
// moves L by ~1e-12 cond relative and the LML by <= 2e-8 relative up to cond 1e4; S = 7 resolves 2^-54 of the row scale and
// stays within ~3x of plain fp64 arithmetic for every conditioning tried (1e1 .. 1e8), so it serves everything else,
// including an unknown conditioning (a bare gpk_potrf).
static int g_last_slices = 0;  // diagnostic: digit planes of the most recent fp64 factorisation (0 = DMMA / none)
int potrf_last_slices() { return g_last_slices; }

static int pick_slices(double cond_hint) {
  return (cond_hint > 0.0 && cond_hint <= 1e4) ? 6 : 7;
}

// ---- fp32 factorisations by way of the fp64 path --------------------------------------------------------------------------
// The fp32 factorisation keeps the round-1 structure (full-inverse leaf, 63-70 us, panel solves and updates as CUDA-core
// GEMMs): chol(Kuu) at M = 2048 costs ~1.8 ms of the 3.3 ms SVGP step.  The fp64 path (slim DMMA leaf, panel kernel, tcgen05
// updates) factors the same matrix in ~1.0 ms, so a square fp32 matrix of n >= 512 is widened to fp64, factored there and
// rounded back; the fp32 block inverses the triangular solves consume are recomputed from the rounded factor.  (The factor
// is the correctly rounded fp64 factor instead of an fp32-accumulated one.)  The fp64 copy, its block-inverse slots and its
// digit planes live in the CALLER's workspace: potrf_tc_ws_bytes(n, rows, GPK_F32) is part of gpk_potrf_ws / the fused
// objectives' workspace queries.
__global__ void widen_lower_kernel(const float* __restrict__ A, int64_t lda, double* __restrict__ B, int64_t ldb, int64_t n) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c <= r && c < n) B[r * ldb + c] = (double)A[r * lda + c];
}
__global__ void narrow_lower_kernel(const double* __restrict__ B, int64_t ldb, float* __restrict__ A, int64_t lda, int64_t n) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c <= r && c < n) A[r * lda + c] = (float)B[r * ldb + c];
}

static int potrf_f32_via_f64(float* A, int64_t n, int64_t lda, int32_t* info, float* dinv, void* scratch, cudaStream_t st,
                             bool need_dinv) {
  const F32Detour L = f32_detour_layout(n);
  char* ws = (char*)scratch;
  double* A64 = (double*)ws;
  double* dinv64 = (double*)(ws + L.a_bytes);
  void* planes = ws + L.a_bytes + L.d_bytes;
  const dim3 grid((unsigned)((n + 255) / 256), (unsigned)n);
  {
    ProfScope ps(PROF_MISC, st);
    widen_lower_kernel<<<grid, 256, 0, st>>>(A, lda, A64, L.ld64, n);
    GPK_LAUNCH_OK();
  }
  GPK_TRY(potrf_t<double>(A64, n, n, L.ld64, info, dinv64, planes, L.p_bytes, st, /*need_dinv=*/false, /*cond_hint=*/0.0));
  {
    ProfScope ps(PROF_MISC, st);
    narrow_lower_kernel<<<grid, 256, 0, st>>>(A64, L.ld64, A, lda, n);
    GPK_LAUNCH_OK();
  }
  if (need_dinv) GPK_TRY(trtri_diag_t<float>(A, n, lda, dinv, st));
  return 0;
}

template <typename T>
int potrf_t(T* A, int64_t n, int64_t rows, int64_t lda, int32_t* info, T* dinv, void* tcws, size_t tcws_bytes,
            cudaStream_t st, bool need_dinv, double cond_hint) {
  if (n <= 0) return 0;
  if (sizeof(T) == 4 && f32_detour_applies(n, rows) && tcws && tcws_bytes >= potrf_tc_ws_bytes(n, rows, GPK_F32))
    return potrf_f32_via_f64(reinterpret_cast<float*>(A), n, lda, info, reinterpret_cast<float*>(dinv), tcws, st, need_dinv);
  GPK_TRY(leaf_attr<T>());
  if (info) GPK_CUDA_OK(cudaMemsetAsync(info, 0, sizeof(int32_t), st));
  LookAhead la;
  // the look-ahead counter lives in the last 256 bytes of the dinv area's alignment slack (see potrf_ws_bytes)
  int* flag = reinterpret_cast<int*>(reinterpret_cast<char*>(dinv) + (size_t)((n + NB - 1) / NB) * NB * NB * sizeof(T));
  if (n > NB) GPK_TRY(lookahead_init(la, flag, st));
  if (la.enabled) GPK_CUDA_OK(cudaMemsetAsync(la.flag, 0, 4 * sizeof(int), st));  // counters run up from here (la.base1 / base2)
  la.slim = sizeof(T) == 8 && n > NB;
  la.fuse = la.slim && la.enabled;
  std::unique_lock<std::mutex> flight_lock(g_flight_mu, std::defer_lock);
  if (la.enabled) flight_lock.lock();
  la.flaghop = la.slim && la.enabled && flight_alone(st);
  // digit-plane store for the tcgen05 trailing updates: fp64, slim panels (they emit the planes), split_point(n) >= TC_MIN_K
  const int S = pick_slices(cond_hint);
  if (sizeof(T) == 8) g_last_slices = 0;
  if (la.slim && tcws && split_point(n) >= TC_MIN_K && tcws_bytes >= tc_planes_bytes(n, rows)) {
    la.pl = tc_planes_layout(tcws, n, rows, S);
    g_last_slices = S;
    GPK_TRY(tc_row_exponents((const double*)A, lda, la.pl, st));  // from the ORIGINAL diagonal
  }
  GPK_TRY(potrf_rec<T>(A, n, rows, lda, info, dinv, 0, la, st));
  if (la.flaghop && la.side_started) {  // the caller's stream continues behind the last leaf
    GPK_CUDA_OK(cudaEventRecord(la.ev_side, la.side));
    GPK_CUDA_OK(cudaStreamWaitEvent(st, la.ev_side, 0));
  }
  if (la.enabled) GPK_TRY(flight_mark(st));
  // slim leaves left only the 64x64 diagonal inverses: the full 128x128 block inverses that gpk_trsm consumes are
  // computed now, all blocks in parallel, off the factorisation's critical path (skipped when nobody will use them)
  if (la.slim && need_dinv) GPK_TRY(trtri_diag_t<T>(A, n, lda, dinv, st));
  return 0;
}

// Batch of small factorisations (n <= 128): ONE launch, one CTA per matrix (multi-output Kuu stacks [L, M, M]).
template <typename T>
int potrf_batched_small_t(T* A, int64_t n, int64_t lda, int64_t stride, int batch, int32_t* info, T* dinv, cudaStream_t st) {
  if (n <= 0 || batch <= 0) return 0;
  GPK_CHECK_ARG(n <= NB, "potrf_batched_small: n = %lld > %d", (long long)n, NB);
  GPK_TRY(leaf_attr<T>());
  if (info) GPK_CUDA_OK(cudaMemsetAsync(info, 0, (size_t)batch * sizeof(int32_t), st));
  ProfScope ps(PROF_LEAF, st);
  potrf_leaf_kernel<T, false><<<(unsigned)batch, 256, leaf_smem_bytes<T>(), st>>>(A, lda, (int)n, dinv, info, 0, nullptr, nullptr,
                                                                                  0, stride, nullptr);
  GPK_LAUNCH_OK();
  return 0;
}
template int potrf_batched_small_t<float>(float*, int64_t, int64_t, int64_t, int, int32_t*, float*, cudaStream_t);
template int potrf_batched_small_t<double>(double*, int64_t, int64_t, int64_t, int, int32_t*, double*, cudaStream_t);

template <typename T>
int trtri_diag_t(const T* L, int64_t n, int64_t ldl, T* dinv, cudaStream_t st) {
  if (n <= 0) return 0;
  GPK_TRY(leaf_attr<T>());
  const unsigned nblk = (unsigned)((n + NB - 1) / NB);
  trtri_diag_kernel<T><<<nblk, 256, leaf_smem_bytes<T>(), st>>>(L, ldl, n, dinv);
  GPK_LAUNCH_OK();
  return 0;
}

template <typename T>
static int trsm_rec(int trans, const T* L, int64_t n, int64_t ldl, T* B, int64_t nrhs, int64_t ldb, const T* dinv,
                    int64_t col0, cudaStream_t st) {
  if (n <= NB) {
    const T* dblk = dinv + (size_t)(col0 / NB) * NB * NB;
    // B <- Linv B  or  Linv^T B, in place (single row tile)
    return gemm_t<T>(trans ? 1 : 0, 0, n, nrhs, n, T(1), dblk, NB, B, ldb, T(0), B, ldb, 0, st);
  }
  const int64_t n1 = split_point(n);
  const T* L21 = L + n1 * ldl;
  const T* L22 = L + n1 * ldl + n1;
  T* B2 = B + n1 * ldb;
  if (!trans) {
    GPK_TRY(trsm_rec<T>(0, L, n1, ldl, B, nrhs, ldb, dinv, col0, st));
    GPK_TRY(gemm_t<T>(0, 0, n - n1, nrhs, n1, T(-1), L21, ldl, B, ldb, T(1), B2, ldb, 0, st));
    return trsm_rec<T>(0, L22, n - n1, ldl, B2, nrhs, ldb, dinv, col0 + n1, st);
  }
  GPK_TRY(trsm_rec<T>(1, L22, n - n1, ldl, B2, nrhs, ldb, dinv, col0 + n1, st));
  GPK_TRY(gemm_t<T>(1, 0, n1, nrhs, n - n1, T(-1), L21, ldl, B2, ldb, T(1), B, ldb, 0, st));
  return trsm_rec<T>(1, L, n1, ldl, B, nrhs, ldb, dinv, col0, st);
}

template <typename T>
int trsm_t(int trans, const T* L, int64_t n, int64_t ldl, T* B, int64_t nrhs, int64_t ldb, const T* dinv,
           cudaStream_t st) {
  if (n <= 0 || nrhs <= 0) return 0;
  return trsm_rec<T>(trans, L, n, ldl, B, nrhs, ldb, dinv, 0, st);
}

// phase timing of one leaf launch (clock64 at phase boundaries), for tuning
int trace_set_potrf(TraceBuf tb) {
  GPK_CUDA_OK(cudaMemcpyToSymbol(g_trace, &tb, sizeof(tb)));
  return 0;
}

int leaf_debug(double* A, int64_t lda, int n, double* dinv, long long* dbg, cudaStream_t st) {
  GPK_TRY(leaf_attr<double>());
  potrf_leaf_kernel<double, false><<<1, 256, leaf_smem_bytes<double>(), st>>>(A, lda, n, dinv, nullptr, 0, dbg, nullptr, 0, 0, nullptr);
  GPK_LAUNCH_OK();
  return 0;
}

template int potrf_t<float>(float*, int64_t, int64_t, int64_t, int32_t*, float*, void*, size_t, cudaStream_t, bool, double);
template int potrf_t<double>(double*, int64_t, int64_t, int64_t, int32_t*, double*, void*, size_t, cudaStream_t, bool,
                             double);
template int trtri_diag_t<float>(const float*, int64_t, int64_t, float*, cudaStream_t);
template int trtri_diag_t<double>(const double*, int64_t, int64_t, double*, cudaStream_t);
template int trsm_t<float>(int, const float*, int64_t, int64_t, float*, int64_t, int64_t, const float*, cudaStream_t);
template int trsm_t<double>(int, const double*, int64_t, int64_t, double*, int64_t, int64_t, const double*,
                            cudaStream_t);

}  // namespace gpk
