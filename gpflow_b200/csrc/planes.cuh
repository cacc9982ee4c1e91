// planes.cuh — the digit-plane store of one fp64 factorisation (shared by gemm_tc.cu and potrf.cu).
//
// The tcgen05 trailing update (gemm_tc.cu) consumes L as S signed digit planes per element, radix 256 (round 2; radix 128 in
// round 1: one more plane for the same precision),
//     l_ik = 2^(e_i - 6) * sum_s 2^(-8 s) d_s(i,k),   d_0 in [-65, 65], d_s in [-128, 127] (s >= 1)  (int8),
// i.e. the integer I = rint(l_ik 2^(6 - e_i) 2^(8 (S - 1))) in balanced base 256.  S = 6 resolves 2^-46 of the row scale 2^e_i,
// S = 7 2^-54 (entries within 2^-2 of 2^e_i keep every bit; as accurate as fp64 arithmetic itself on every matrix of scripts/radix_study.py, cond up to 1e8).  The update
// keeps the digit products of order s + t < S; for even S it adds the (S/2, S/2) product, the only dropped term of order S
// whose mean on the diagonal of C is not zero (d^2 > 0 -- it biased sum log diag L by 1e-7 .. 1e-5 at S = 6 without it).
// Planes are stored PRE-TILED in the canonical no-swizzle K-major UMMA image: tile (rb, kb) = rows [128 rb, 128 rb + 128) x
// columns [32 kb, 32 kb + 32) holds S consecutive planes of 4096 bytes.  Row block rb only ever needs the k-blocks left
// of its diagonal block (kb < 4 rb; extra rows below the square part need all of them), so the tiles are packed
// triangularly: tile (rb, kb) starts at (plane_prefix(rb) + kb) * S * 4096 bytes.
//
// Static scales: |L_ik| <= sqrt(A_ii) for a positive-definite A, so e_i = ilogb(sqrt(A_ii)) + 1 is valid for every
// entry of row i BEFORE the row exists.  The panel-solve kernel (potrf.cu) therefore emits the planes of the columns it
// has just finished directly from shared memory, and no slicing pass over L is needed (the price -- rows of L are often
// well below sqrt(A_ii), so a few leading digit bits are unused -- is measured in scripts/static_scale_study.py and
// scripts/radix_study.py: max |dL| / max |L| = 2e-11 at S = 6, 1e-13 at S = 7 on BASELINE configs[1]).  Rows below the square part (the (Y - m)^T rows that ride along)
// have no such bound and are sliced with their running row maximum before each update (slice_rows_kernel).
#pragma once
#include "common.cuh"

namespace gpk {

constexpr int TC_BM = 128, TC_BN = 64, TC_KB = 32;   // CTA tile of the update, bytes (= int8 elements) per k-step
constexpr int TC_ATILE = TC_BM * TC_KB;              // 4096 B per digit plane of a 128-row tile
constexpr int TC_BTILE = TC_BN * TC_KB;              // 2048 B (one half of a 128-row tile)
constexpr int TC_MAXS = 8;                           // planes the store is sized for (S <= 7 is used)

// byte offset of element (row r in [0,128), k in [0,32)) inside one digit-plane tile:
// canonical no-swizzle K-major UMMA layout ((8,n),2):((1,SBO),LBO) in 16-byte units, LBO = 8, SBO = 16
__device__ __host__ __forceinline__ int tc_tile_off(int r, int k) {
  return (r >> 3) * 256 + (k >> 4) * 128 + (r & 7) * 16 + (k & 15);
}

// number of k-block tiles stored before row block rb; nbk = number of 128-column blocks of the square part
__device__ __host__ __forceinline__ int64_t plane_prefix(int64_t rb, int64_t nbk) {
  const int64_t q = rb < nbk + 1 ? rb : nbk + 1;
  return 2 * q * (q - 1) + (rb - q) * 4 * nbk;
}

// Conversions without the XU pipe (F2I / I2F / FRND run at 16 per clock per SM, a quarter of the fp64 FMA rate):
//  * digit extraction: t = v + 1.5 * 2^52 rounds v (|v| < 2^31) to the nearest integer (ties to even, like rint) in the
//    fp64 adder; the integer sits in the low word of t, the rounded value is t - 1.5 * 2^52;
//  * int32 -> double: the bit pattern 0x43300000'(x ^ 0x80000000) is 2^52 + 2^31 + x exactly.
constexpr int TC_RADIX_BITS = 8;
// The S balanced base-256 digits of I = rint(v 2^(8 (S - 1))), |v| < 64: d_s in [-128, 127] for s >= 1, the top digit d_0
// is what remains (|d_0| <= 65).  Adding the bias J = I + 0x80...80 (S - 1 bytes) makes every lower digit an unsigned byte
// u_s = d_s + 128 of J, and u_s ^ 0x80 is d_s as an int8; J >> 8 (S - 1) is d_0.  So the digit bytes of one value are
//     X = (I + flip) ^ flip,  flip = 0x80 repeated S - 1 times,  byte j of X = digit of plane S - 1 - j,
// and I comes out of the fp64 adder without a conversion instruction: the bit pattern of x + 1.5 2^52 is
// 0x433 << 52 | (2^51 + rint(x)) for |x| < 2^51 (S <= 6: |I| <= 2^46).  S >= 7 (|I| <= 2^54, 2^62) rounds the top 22 bits
// and the rest separately: hi = rint(v 2^16) (exact remainder r = v 2^16 - hi, |r| <= 1/2), I = hi 2^low + rint(r 2^low).
// 5 instructions per value at S <= 6, 11 at S >= 7 (a digit-by-digit loop costs ~10 per DIGIT).
struct TcDigitizer {
  double up;                     // 2^(8 (S - 1)) (S <= 6) or 2^low (S >= 7), low = 8 (S - 1) - 16
  unsigned long long c, flip;    // c = flip - (0x433 << 52) - 2^51
  int S, hshift;                 // S >= 7: hi enters at bit low = 32 + hshift
  __device__ __forceinline__ explicit TcDigitizer(int S_) : S(S_) {
    const int low = S <= 6 ? TC_RADIX_BITS * (S - 1) : TC_RADIX_BITS * (S - 1) - 16;
    up = __hiloint2double((1023 + low) << 20, 0);
    hshift = S <= 6 ? 0 : low - 32;
    flip = 0x8080808080808080ull >> (8 * (9 - S));
    c = flip - 0x4330000000000000ull - 0x0008000000000000ull;
  }
  __device__ __forceinline__ unsigned long long bytes(double v) const {
    const double magic = 6755399441055744.0;  // 1.5 * 2^52
    if (S <= 6) {
      const double t = fma(v, up, magic);
      return ((unsigned long long)__double_as_longlong(t) + c) ^ flip;
    }
    const double xh = v * 65536.0;
    const double th = xh + magic;             // low word = rint(v 2^16) as an int32
    const double r = xh - (th - magic);
    const double t2 = fma(r, up, magic);
    unsigned long long J = (unsigned long long)__double_as_longlong(t2) + c;
    J += (unsigned long long)(long long)__double2loint(th) << (32 + hshift);
    return J ^ flip;
  }
};
// 4 x 4 byte transpose: o[j] = byte j of a0 | byte j of a1 << 8 | byte j of a2 << 16 | byte j of a3 << 24 (8 PRMT)
__device__ __forceinline__ void tc_transpose4(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t (&o)[4]) {
  const uint32_t l01 = __byte_perm(a0, a1, 0x5140), h01 = __byte_perm(a0, a1, 0x7362);
  const uint32_t l23 = __byte_perm(a2, a3, 0x5140), h23 = __byte_perm(a2, a3, 0x7362);
  o[0] = __byte_perm(l01, l23, 0x5410);
  o[1] = __byte_perm(l01, l23, 0x7632);
  o[2] = __byte_perm(h01, h23, 0x5410);
  o[3] = __byte_perm(h01, h23, 0x7632);
}
// digit words of 4 consecutive k of one row: w[j] = the 32-bit word of plane S - 1 - j (j < S)
__device__ __forceinline__ void tc_digit_words(const TcDigitizer& dz, const double (&v)[4], uint32_t (&w)[8]) {
  unsigned long long x[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) x[q] = dz.bytes(v[q]);
  uint32_t lo[4], hi[4];
  tc_transpose4((uint32_t)x[0], (uint32_t)x[1], (uint32_t)x[2], (uint32_t)x[3], lo);
  tc_transpose4((uint32_t)(x[0] >> 32), (uint32_t)(x[1] >> 32), (uint32_t)(x[2] >> 32), (uint32_t)(x[3] >> 32), hi);
#pragma unroll
  for (int j = 0; j < 4; ++j) { w[j] = lo[j]; w[4 + j] = hi[j]; }
}
__device__ __forceinline__ double tc_int_to_double(int x) {
  return __hiloint2double(0x43300000, x ^ 0x80000000) - 4503601774854144.0;  // 2^52 + 2^31
}

struct TcPlanes {
  int8_t* planes = nullptr;   // digit planes, triangular tile packing
  double* rowscale = nullptr; // [rows_pad]: 2^(e_i - 6)
  int* err = nullptr;         // device word: protocol error code of the tcgen05 kernel (bounded waits)
  int S = 7;                  // digit planes per element: 6 or 7
  int64_t nbk = 0;            // 128-column blocks of the square part
  int64_t n_sq = 0;           // rows >= n_sq are "extra" rows (dynamic scales)
  __device__ __host__ int8_t* tile(int64_t rb, int64_t kb) const {
    return planes + (size_t)(plane_prefix(rb, nbk) + kb) * S * TC_ATILE;
  }
};

// Dynamic slicing of ONE row by a whole CTA (256 threads): the k-range [k0, k0 + K) of row r (src = &row[k0]) gets the scale
// of its maximum over that range -- the rows below the square part have no static bound.  wmax: 8 doubles of shared memory.
__device__ __forceinline__ void tc_slice_row_cta(const double* src, int64_t r, int64_t k0, int64_t K, const TcPlanes& pl,
                                                 double* wmax) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = pl.S;
  double mx = 0.0;
  for (int64_t k = threadIdx.x; k < K; k += 256) mx = fmax(mx, fabs(src[k]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  __syncthreads();  // (wmax may still be read by the previous row's threads)
  if (lane == 0) wmax[warp] = mx;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < 8; ++w) mx = fmax(mx, wmax[w]);
  int e = 0;
  if (mx > 0.0 && mx < 1e300) e = ilogb(mx) + 1;  // mx * 2^-e in [0.5, 1)
  const double sc = scalbn(1.0, -e + 6);          // x * 2^-e * 2^6
  if (threadIdx.x == 0) pl.rowscale[r] = scalbn(1.0, e - 6);
  int8_t* rowbase = pl.tile(r >> 7, k0 / TC_KB);
  const int rr = (int)(r & 127);
  const TcDigitizer dz(S);
  // each thread converts 4 consecutive k per iteration -> one 32-bit store per digit plane
  for (int64_t kq = (int64_t)threadIdx.x * 4; kq < K; kq += 1024) {
    double v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = src[kq + q] * sc;
    const int kb = (int)(kq / TC_KB), kk = (int)(kq % TC_KB);
    int8_t* tb = rowbase + (size_t)kb * S * TC_ATILE + tc_tile_off(rr, kk);
    uint32_t w[8];
    tc_digit_words(dz, v, w);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < S) *reinterpret_cast<uint32_t*>(tb + (size_t)(S - 1 - j) * TC_ATILE) = w[j];
  }
}

size_t tc_planes_bytes(int64_t n, int64_t rows);
TcPlanes tc_planes_layout(void* ws, int64_t n, int64_t rows, int S);
// rowscale[i] = 2^(ilogb(sqrt(A_ii)) + 1 - 6) for the square rows (reads the ORIGINAL diagonal: call before factorising)
int tc_row_exponents(const double* A, int64_t lda, const TcPlanes& pl, cudaStream_t st);
// slices rows [row0, row0 + nrows) (global indices) of the k-range [k0, k0 + K) with their running row maxima
int tc_slice_rows(const double* P, int64_t ld, int64_t row0, int64_t nrows, int64_t k0, int64_t K, const TcPlanes& pl,
                  cudaStream_t st);
// C[m, n] -= L[r0 : r0 + m, k0 : k0 + K] L[r0 : r0 + n, k0 : k0 + K]^T from the plane store (lower tiles only if `lower`)
int syrk_tc_planes(double* C, int64_t ldc, int64_t m, int64_t n, const TcPlanes& pl, int64_t r0, int64_t k0, int64_t K,
                   int lower, cudaStream_t st, const GemmOpts* opts = nullptr);

}  // namespace gpk
