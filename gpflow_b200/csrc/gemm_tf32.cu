// gemm_tf32.cu — fp32 GEMM on the 5th-generation tensor cores (tcgen05 kind::tf32, TMEM accumulators)
// with 3xTF32 error compensation:   a = a_hi + a_lo (both exactly representable in TF32)
//        a*b ~= a_hi*b_hi + a_hi*b_lo + a_lo*b_hi     (dropped a_lo*b_lo ~ 2^-22 relative)
// accumulated in ONE fp32 TMEM accumulator, so the result is as accurate as an fp32 FFMA GEMM while the
// contraction runs on the tensor pipe.  Serves the fp32 configs (SGPR / SVGP): the GEMM blocks of the
// inverse-based TRSM (sgpr.py:204, conditionals/util.py:125), A A^T (sgpr.py:205), tril(q_sqrt)^T A with
// the fused column-sum-of-squares (conditionals/util.py:151-164) and the Cholesky trailing updates.
//
//     C[m,n] = alpha * op(A) op(B) + beta * C          (row-major fp32, any op combination)
//
// A pre-pass (split_tiles_kernel) reads each operand once in whatever orientation it is stored,
// splits hi/lo and writes PRE-TILED K-major planes in the canonical no-swizzle UMMA shared-memory
// image, so the main kernel fills a pipeline stage with 1-D bulk copies and never needs a
// transposed (MN-major) descriptor.  Persistent CTAs, 320 threads:
//   warp 0 producer (cp.async.bulk + mbarrier; in a 2-CTA cluster each CTA fetches half of every B plane
//   and multicasts it), warp 1 MMA issuer (one elected lane, 3 MMAs per 8-deep k-step, tile 128 x 256,
//   runs of 64 k-elements into alternating TMEM buffers), warps 2-9 promotion + epilogue (tcgen05.ld of a
//   finished run, round-to-nearest add into fp32 register accumulators, then shared transpose -> coalesced
//   128-byte row segments, alpha/beta, optional split-K atomics, optional fused column sums of squares).
// The all-zero K range of a triangular A operand is skipped (tf_krange).
#include <algorithm>
#include <map>
#include <utility>

#include "tc_common.cuh"

namespace gpk {

constexpr int TF_BM = 128, TF_BN = 256;
constexpr int TF_KS = 16;                       // fp32 elements of K per pipeline stage (64 bytes per row)
constexpr int TF_STAGES = 4;
constexpr int TF_APLANE = TF_BM * TF_KS * 4;    // 8 KB
constexpr int TF_BPLANE = TF_BN * TF_KS * 4;    // 16 KB
constexpr int TF_STAGE_BYTES = 2 * TF_APLANE + 2 * TF_BPLANE;  // 48 KB
constexpr int TF_EPI_BYTES = 4 * 32 * 33 * 4;   // per-warp 32x33 transpose tiles

// byte offset of (row r, k) inside one plane tile of RB rows x 16 k (no-swizzle K-major canonical layout:
// 8x16-byte core matrices, LBO = 128 B between k chunks, SBO = 512 B between 8-row groups)
__device__ __forceinline__ int tf_tile_off(int r, int k) { return (r >> 3) * 512 + (k >> 2) * 128 + (r & 7) * 16 + (k & 3) * 4; }

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

// ------------------------------------------------------------------------------------------------
// pre-pass: operand (logical [R, K]) -> tiles[(rb, kb)][plane][RB x 16] with hi / lo planes
//   trans = 0: src[r * ld + k]     trans = 1: src[k * ld + r]
//   tri   = 1: the STORED matrix is lower triangular (band_part(-1,0)); entries with stored col > row read as 0
// ------------------------------------------------------------------------------------------------
// Index arithmetic without 64-bit divisions (the 1-D form of round 1 spent most of its time in them: 2.0 of the 7.5 ms of
// BASELINE configs[2] went to this pre-pass) and whole-line stores in both orientations:
//   trans = 0 (k contiguous in the source): a warp takes 8 rows x one 16-k tile column -- 8 x 64 B segments in, and the 4 core
//     matrices of those 8 rows (512 contiguous bytes of the tile image) out; block = 8 consecutive k-blocks, grid.(y,z) = row groups
//   trans = 1 (r contiguous): consecutive lanes walk r (coalesced loads, 128-byte runs of the core matrices out);
//     block = 256 consecutive rows, grid.(y,z) = k-chunks
constexpr int TF_SPLIT_YMAX = 32768;
template <int RB>
__global__ void __launch_bounds__(256)
split_tiles_kernel(const float* __restrict__ src, int64_t R, int64_t K, int64_t ld, int trans, int tri,
                   float* __restrict__ tiles, int64_t KBn, int64_t rows_per_batch, int64_t batch_stride) {
  // rows_per_batch > 0: the logical [R, K] operand is a vertical stack of R / rows_per_batch matrices stored
  // batch_stride elements apart (the P lower-triangular q_sqrt_p of the SVGP conditional): row r = (batch, r % rows)
  // one thread = one 16-byte k-chunk (4 consecutive k) of one row
  const int64_t Rpad = (R + RB - 1) / RB * RB;
  const int64_t nchunk = KBn * 4;  // k-chunks per row
  const int64_t slow = (int64_t)blockIdx.z * TF_SPLIT_YMAX + blockIdx.y;
  int64_t r, kc;
  if (!trans) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    r = slow * 8 + (lane & 7);
    kc = ((int64_t)blockIdx.x * 8 + w) * 4 + (lane >> 3);
  } else {
    r = (int64_t)blockIdx.x * 256 + threadIdx.x;
    kc = slow;
  }
  if (r >= Rpad || kc >= nchunk) return;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (r < R) {
    int64_t rl = r;
    const float* sb = src;
    if (rows_per_batch > 0) {
      const int64_t bi = r / rows_per_batch;
      rl = r - bi * rows_per_batch;
      sb = src + bi * batch_stride;
    }
    const int64_t k0 = kc * 4;
    if (!trans && k0 + 3 < K && !tri && (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(sb) & 15) == 0) {
      const float4 t4 = *reinterpret_cast<const float4*>(sb + rl * ld + k0);
      v[0] = t4.x; v[1] = t4.y; v[2] = t4.z; v[3] = t4.w;
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int64_t k = k0 + q;
        if (k < K) {
          const int64_t srow = trans ? k : rl, scol = trans ? rl : k;
          if (!(tri && scol > srow)) v[q] = sb[srow * ld + scol];
        }
      }
    }
  }
  float hi[4], lo[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    hi[q] = to_tf32(v[q]);
    lo[q] = to_tf32(v[q] - hi[q]);
  }
  const int64_t rb = r / RB, kb = kc >> 2;   // (RB is a power of two: shifts)
  const int rr = (int)(r % RB), kk = (int)(kc & 3) * 4;
  char* base = reinterpret_cast<char*>(tiles) + ((size_t)(rb * KBn + kb) * 2) * (RB * TF_KS * 4) + tf_tile_off(rr, kk);
  *reinterpret_cast<float4*>(base) = make_float4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<float4*>(base + RB * TF_KS * 4) = make_float4(lo[0], lo[1], lo[2], lo[3]);
}

template <int RB>
static void split_tiles_launch(const float* src, int64_t R, int64_t K, int64_t ld, int trans, int tri, float* tiles, int64_t KBn,
                               int64_t rows_per_batch, int64_t batch_stride, cudaStream_t st) {
  const int64_t Rpad = (R + RB - 1) / RB * RB;
  const int64_t fast = trans ? (Rpad + 255) / 256 : (KBn + 7) / 8;
  const int64_t slow = trans ? KBn * 4 : Rpad / 8;
  const dim3 grid((unsigned)fast, (unsigned)(slow < TF_SPLIT_YMAX ? slow : TF_SPLIT_YMAX),
                  (unsigned)((slow + TF_SPLIT_YMAX - 1) / TF_SPLIT_YMAX));
  split_tiles_kernel<RB><<<grid, 256, 0, st>>>(src, R, K, ld, trans, tri, tiles, KBn, rows_per_batch, batch_stride);
}

// ------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D = F32, A = B = TF32, K-major both, N = 256, M = 128
constexpr uint32_t TF_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TF_BN >> 3) << 17) |
                              ((uint32_t)(TF_BM >> 4) << 24);

struct TfWork {  // work unit = (CL vertically adjacent row tiles, column tile, k split); same enumeration in every role
  int64_t ntm, ntn;
  int nsplit, lower, cl, rank;
  int64_t idx, tm0, tm, tn;  // tm0 = first row tile of the unit, tm = this CTA's row tile (tm0 + rank)
  int ks;
  __device__ TfWork(int64_t m, int64_t n, int nsplit_, int lower_, int cl_, int rank_)
      : nsplit(nsplit_), lower(lower_), cl(cl_), rank(rank_), idx(-1), tm0(0), tm(0), tn(0), ks(-1) {
    ntm = (m + TF_BM - 1) / TF_BM;
    ntn = (n + TF_BN - 1) / TF_BN;
  }
  __device__ bool tile_skip(int64_t t) const { return lower && tn * TF_BN > t * TF_BM + TF_BM - 1; }
  __device__ bool unit_skip() const { return tile_skip(tm0 + cl - 1); }  // the lowest tile of the unit decides
  // this CTA's tile takes part in the loads / MMAs of its unit but is not stored when it is padding
  __device__ bool valid() const { return tm < ntm && !tile_skip(tm); }
  __device__ int64_t tm_load() const { return tm < ntm ? tm : ntm - 1; }
  // Order: k-splits innermost, then ROW units, column tiles outermost: the (large) B tile of a column
  // block is reused by consecutive work items while it is still in L2 (measured before: 4.5x re-reads
  // of the B planes from HBM with column tiles innermost).
  __device__ bool next() {
    const int64_t nclusters = gridDim.x / cl, my = blockIdx.x / cl;
    for (;;) {
      ++ks;
      if (ks >= nsplit) { ks = 0; tm0 += cl; }
      while (tn < ntn && (tm0 >= ntm || unit_skip())) {
        if (tm0 >= ntm) { tm0 = 0; ++tn; } else { tm0 += cl; }
      }
      if (tn >= ntn) return false;
      ++idx;
      if (idx % nclusters == my) { tm = tm0 + rank; return true; }
    }
  }
};

// The fp32 accumulation inside the tensor core truncates (round-toward-zero): every MMA adds up to one
// ulp of systematic error relative to the running accumulator, so a long K loop into ONE TMEM accumulator
// loses ~n_mma * 2^-24 (measured: 1.6e-5 relative at K = 640, 2e-3 on the SGPR ELBO at K = 1e5).
// Fix: the MMAs accumulate only TF_KP = 64 k-elements (24 MMAs) into a TMEM buffer; eight "promotion"
// warps then read the buffer (tcgen05.ld) and add it round-to-nearest into fp32 REGISTER accumulators
// while the MMAs continue into the other buffer.
constexpr int TF_KP = 64;                       // k elements per TMEM accumulation run
constexpr int TF_SPP = TF_KP / TF_KS;           // pipeline stages per run (4)
constexpr int TF_THREADS = 320;                 // warp 0 producer, warp 1 MMA, warps 2..9 promotion/epilogue

// Stage range [kb0, kb1) of k-split `ks` of row tile `tm`.  tri = 1: op(A) is lower triangular (k <= row), tri = 2:
// upper triangular (k >= row, e.g. tril(q_sqrt)^T): the all-zero part of the K range is skipped (whole runs), which
// halves the P batched products  tril(q_sqrt_p)^T A  of the SVGP conditional (conditionals/util.py:151-157).
__device__ __forceinline__ void tf_krange(int tri, int64_t tm_first, int64_t tm_last, int KB, int nsplit, int ks, int& kb0,
                                          int& kb1, int tpb = 0) {  // common range of the row tiles tm_first..tm_last of one unit
  if (tpb > 0) { tm_first %= tpb; tm_last %= tpb; }  // stacked triangular operands: position inside the own matrix
  int lo = 0, hi = KB;
  if (tri == 2) lo = (int)((tm_first * TF_BM / TF_KS) / TF_SPP * TF_SPP);
  if (tri == 1) { const int64_t e = ((tm_last + 1) * TF_BM + TF_KS - 1) / TF_KS; if (e < hi) hi = (int)e; }
  if (lo > hi) lo = hi;
  const int per = ((hi - lo + nsplit - 1) / nsplit + TF_SPP - 1) / TF_SPP * TF_SPP;  // whole runs per split
  kb0 = lo + ks * per;
  kb1 = kb0 + per < hi ? kb0 + per : hi;
  if (kb0 > kb1) kb0 = kb1;
}

// CL = 2: the two CTAs of a cluster work on vertically adjacent row tiles of the same column tile and share the B
// planes (each fetches half of every plane and multicasts it): 48 -> 32 KB of L2->SM traffic per stage per CTA.
template <int CL>
__global__ void __launch_bounds__(TF_THREADS, 1)
gemm_tf32_kernel(const float* __restrict__ Atiles, const float* __restrict__ Btiles, float* C, int64_t ldc, int64_t m,
                 int64_t n, int KB, int nsplit, float alpha, float beta, int flags, int tri, int* err, int tpb,
                 int64_t c_batch_stride) {
  // tpb > 0: op(A) is a vertical stack of matrices of tpb row tiles each (batched tril(q_sqrt_p)^T A); the fused column
  // sums of squares of matrix b go to C + b * c_batch_stride
  extern __shared__ __align__(1024) uint8_t tf_smem[];
  uint8_t* epi = tf_smem + TF_STAGES * TF_STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi + 2 * TF_EPI_BYTES);  // full[4], empty[4], tfull[2], tempty[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TF_STAGES + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + TF_STAGES);
  const uint32_t tfull0 = smem_u32(bars + 2 * TF_STAGES), tempty0 = smem_u32(bars + 2 * TF_STAGES + 2);
  const int lower = (flags & GPK_GEMM_LOWER_ONLY) ? 1 : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < TF_STAGES; ++i) { mbar_init(full0 + 8 * i, 1); mbar_init(empty0 + 8 * i, CL); }
    for (int i = 0; i < 2; ++i) { mbar_init(tfull0 + 8 * i, 1); mbar_init(tempty0 + 8 * i, 256); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // peer barriers initialised before any multicast copy / commit targets them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int rank = CL > 1 ? (int)cluster_ctarank() : 0;
  constexpr uint16_t cl_mask = (uint16_t)((1u << CL) - 1);

  if (__all_sync(0xffffffffu, warp == 0)) {  // vote: the role branch is warp-uniform and the compiler knows it
    // ===== producer =====
    TfWork w(m, n, nsplit, lower, CL, rank);
    uint32_t st = 0, ph = 0;
    while (w.next()) {
      int kb0, kb1;
      tf_krange(tri, w.tm0, w.tm0 + CL - 1, KB, nsplit, w.ks, kb0, kb1, tpb);
      const char* a_src = reinterpret_cast<const char*>(Atiles) + (size_t)w.tm_load() * KB * 2 * TF_APLANE;
      const char* b_src = reinterpret_cast<const char*>(Btiles) + (size_t)w.tn * KB * 2 * TF_BPLANE;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty0 + 8 * st, ph ^ 1, err, 201);
        if (elect_one()) {
          const uint32_t fb = full0 + 8 * st;
          mbar_expect_tx(fb, TF_STAGE_BYTES);
          const uint32_t sa = smem_u32(tf_smem + (size_t)st * TF_STAGE_BYTES);
          bulk_g2s(sa, a_src + (size_t)kb * 2 * TF_APLANE, 2 * TF_APLANE, fb);
          if (CL == 1) {
            bulk_g2s(sa + 2 * TF_APLANE, b_src + (size_t)kb * 2 * TF_BPLANE, 2 * TF_BPLANE, fb);
          } else {
            constexpr uint32_t part = TF_BPLANE / CL;
#pragma unroll
            for (int pl = 0; pl < 2; ++pl)
              bulk_g2s_mc(sa + 2 * TF_APLANE + pl * TF_BPLANE + rank * part,
                          b_src + (size_t)kb * 2 * TF_BPLANE + pl * TF_BPLANE + rank * part, part, fb, cl_mask);
          }
        }
        __syncwarp();
        if (++st == TF_STAGES) { st = 0; ph ^= 1; }
      }
    }
  } else if (__all_sync(0xffffffffu, warp == 1)) {
    // ===== MMA issuer: runs of TF_SPP stages into alternating TMEM buffers =====
    TfWork w(m, n, nsplit, lower, CL, rank);
    uint32_t st = 0, ph = 0, buf = 0, tph0 = 0, tph1 = 0;
    const uint64_t desc_hi = ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46);
    while (w.next()) {
      int kb0, kb1;
      tf_krange(tri, w.tm0, w.tm0 + CL - 1, KB, nsplit, w.ks, kb0, kb1, tpb);
      for (int kr = kb0; kr < kb1; kr += TF_SPP) {
        mbar_wait(tempty0 + 8 * buf, (buf ? tph1 : tph0) ^ 1, err, 202);
        tc_fence_after();
        const uint32_t d = tmem_base + buf * TF_BN;
        const int kre = min(kb1, kr + TF_SPP);
        for (int kb = kr; kb < kre; ++kb) {
          mbar_wait(full0 + 8 * st, ph, err, 203);
          tc_fence_after();
          const uint32_t sa = smem_u32(tf_smem + (size_t)st * TF_STAGE_BYTES);
          const uint64_t a_hi = desc_hi | (uint64_t)((sa & 0x3FFFFu) >> 4);
          const uint64_t a_lo = a_hi + (TF_APLANE >> 4);
          const uint64_t b_hi = a_hi + ((2 * TF_APLANE) >> 4);
          const uint64_t b_lo = b_hi + (TF_BPLANE >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k8 = 0; k8 < TF_KS / 8; ++k8) {  // 32 bytes (8 tf32) per MMA: two 16-byte chunks, LBO = 128 B
              const uint64_t o = (uint64_t)(k8 * 2 * 128) >> 4;
              // small terms first, then the leading term
              tc_mma_tf32(d, a_lo + o, b_hi + o, TF_IDESC, (kb > kr || k8 > 0) ? 1u : 0u);
              tc_mma_tf32(d, a_hi + o, b_lo + o, TF_IDESC, 1u);
              tc_mma_tf32(d, a_hi + o, b_hi + o, TF_IDESC, 1u);
            }
            if (CL == 1) tc_commit(empty0 + 8 * st); else tc_commit_mc(empty0 + 8 * st, cl_mask);
          }
          __syncwarp();
          if (++st == TF_STAGES) { st = 0; ph ^= 1; }
        }
        if (elect_one()) tc_commit(tfull0 + 8 * buf);
        __syncwarp();
        if (buf) tph1 ^= 1; else tph0 ^= 1;
        buf ^= 1;
      }
    }
  } else {
    // ===== promotion + epilogue: 8 warps; warp (w-2): lane quarter q = w & 3, column half h = (w-2) >> 2 =====
    const int q = warp & 3, h = (warp - 2) >> 2;
    float* tile = reinterpret_cast<float*>(epi) + (warp - 2) * 32 * 33;
    TfWork w(m, n, nsplit, lower, CL, rank);
    uint32_t buf = 0, tph0 = 0, tph1 = 0;
    while (w.next()) {
      int kb0, kb1;
      tf_krange(tri, w.tm0, w.tm0 + CL - 1, KB, nsplit, w.ks, kb0, kb1, tpb);
      float acc[128];
#pragma unroll
      for (int c = 0; c < 128; ++c) acc[c] = 0.f;
      for (int kr = kb0; kr < kb1; kr += TF_SPP) {
        mbar_wait(tfull0 + 8 * buf, buf ? tph1 : tph0, err, 204);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * TF_BN + h * 128;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          uint32_t v[32];
          tc_ld32(taddr + ch * 32, v);
#pragma unroll
          for (int c = 0; c < 32; ++c) acc[ch * 32 + c] += __uint_as_float(v[c]);  // round-to-nearest promotion
        }
        tc_fence_before();
        mbar_arrive(tempty0 + 8 * buf);
        if (buf) tph1 ^= 1; else tph0 ^= 1;
        buf ^= 1;
      }
      // write out: 32x32 blocks transposed through shared memory -> coalesced 128-byte row segments
      const int64_t row0 = w.tm * TF_BM + q * 32;
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const int64_t col0 = w.tn * TF_BN + h * 128 + ch * 32;
        if (col0 < n && w.valid()) {
#pragma unroll
          for (int c = 0; c < 32; ++c) tile[lane * 33 + c] = alpha * acc[ch * 32 + c];
          __syncwarp();
          const int64_t col = col0 + lane;
          if (flags & GPK_GEMM_COLSUMSQ) {  // column sums of squares over this warp's 32 rows (util.py:164)
            float s = 0.f;
            for (int r = 0; r < 32; ++r) {
              const float x = row0 + r < m ? tile[r * 33 + lane] : 0.f;
              s = fmaf(x, x, s);
            }
            if (col < n) atomicAdd(C + (tpb > 0 ? (w.tm / tpb) * c_batch_stride : 0) + col, s);
          } else if (col < n) {
            float* cbase = C + row0 * ldc + col;
            if (nsplit > 1) {
#pragma unroll 8
              for (int r = 0; r < 32; ++r)
                if (row0 + r < m) atomicAdd(cbase + r * ldc, tile[r * 33 + lane]);   // C was pre-scaled by beta
            } else if (beta != 0.f) {
              // read-modify-write: issue all 32 row loads before the first dependent FMA / store
              float old[32];
#pragma unroll
              for (int r = 0; r < 32; ++r) old[r] = row0 + r < m ? cbase[r * ldc] : 0.f;
#pragma unroll
              for (int r = 0; r < 32; ++r)
                if (row0 + r < m) cbase[r * ldc] = fmaf(beta, old[r], tile[r * 33 + lane]);
            } else {
#pragma unroll 8
              for (int r = 0; r < 32; ++r)
                if (row0 + r < m) cbase[r * ldc] = tile[r * 33 + lane];
            }
          }
          __syncwarp();
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // no CTA leaves while a peer may still multicast into its shared memory
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// scale the m x n region (lower tiles only if requested) of C by beta before a split-K accumulation
__global__ void scale_c_kernel(float* C, int64_t ldc, int64_t m, int64_t n, float beta) {
  const int64_t tot = m * n;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (int64_t)gridDim.x * blockDim.x) {
    float* p = C + (e / n) * ldc + e % n;
    *p = beta == 0.f ? 0.f : beta * *p;
  }
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
// Grow-only device scratch for the pre-tiled planes, one buffer per (device, stream): allocated on first
// use (warm-up), never on the steady-state path; the two streams of the Cholesky look-ahead get
// separate buffers.
static void* tf_scratch(size_t bytes, cudaStream_t st, int* rc) {
  struct Buf { void* p; size_t n; };
  static std::map<std::pair<int, cudaStream_t>, Buf> bufs;
  int dev = 0;
  cudaGetDevice(&dev);
  Buf& b = bufs[{dev, st}];
  if (b.n < bytes) {
    if (b.p) { cudaStreamSynchronize(st); cudaFree(b.p); }
    b.p = nullptr;
    b.n = 0;
    size_t want = bytes + bytes / 4;
    if (cudaMalloc(&b.p, want) != cudaSuccess) {
      cudaGetLastError();
      if (cudaMalloc(&b.p, bytes) != cudaSuccess) { *rc = -2; set_error("gemm_tf32: scratch allocation of %zu bytes failed", bytes); return nullptr; }
      want = bytes;
    }
    b.n = want;
  }
  *rc = 0;
  return b.p;
}

// eager reservation of the plane scratch for this (device, stream) (gpk_warm)
int tf32_reserve(size_t bytes, cudaStream_t st) {
  int rc = 0;
  tf_scratch(bytes, st, &rc);
  return rc;
}

static int tf_num_sms() {
  static int n = 0;
  if (n == 0) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); if (n <= 0) n = 148; }
  return n;
}

// eligibility: big enough to amortise the pre-pass; no aliasing of C with an operand (the pre-pass makes
// copies, but in-place callers rely on tile-local ordering which the persistent kernel does not give)
bool gemm_tf32_eligible(int64_t m, int64_t n, int64_t k, const void* A, const void* B, const void* C, int flags) {
  if (k < 64 || m < 64 || n < 64) return false;
  if ((double)m * n * k < 2.0e8) return false;
  (void)A; (void)B; (void)C; (void)flags;
  return true;
}

int gemm_tf32(int transa, int transb, int64_t m, int64_t n, int64_t k, float alpha, const float* A, int64_t lda,
              const float* B, int64_t ldb, float beta, float* C, int64_t ldc, int flags, cudaStream_t st, int batch,
              int64_t a_batch_stride, int64_t c_batch_stride) {
  // batch > 1 (COLSUMSQ only): op(A) = [op(A_0); ...; op(A_{batch-1})], A_b = A + b * a_batch_stride, all against the same
  // B; column sums of squares of block b accumulate into C + b * c_batch_stride.  ONE launch (B split once, one persistent
  // grid over batch * tiles) instead of `batch` launches with a 2-wave tail each.
  const int64_t m_per = m;
  if (batch > 1) {
    GPK_CHECK_ARG((flags & GPK_GEMM_COLSUMSQ) && m % (2 * TF_BM) == 0, "gemm_tf32: batched form needs COLSUMSQ and m %% 256 == 0");
    m *= batch;
  }
  const int64_t KB = (k + TF_KS - 1) / TF_KS;
  const int64_t mpad = (m + TF_BM - 1) / TF_BM * TF_BM, npad = (n + TF_BN - 1) / TF_BN * TF_BN;
  const size_t a_bytes = (size_t)mpad * KB * TF_KS * 4 * 2, b_bytes = (size_t)npad * KB * TF_KS * 4 * 2;
  int rc = 0;
  char* ws = (char*)tf_scratch(align_up(a_bytes, 256) + align_up(b_bytes, 256) + 256, st, &rc);
  if (!ws) return rc;
  float* At = (float*)ws;
  float* Bt = (float*)(ws + align_up(a_bytes, 256));
  int* err = (int*)(ws + align_up(a_bytes, 256) + align_up(b_bytes, 256));
  {
    ProfScope ps(PROF_MISC, st);
    // op(A) is [m, k]: stored [m,k] (transa = 0, k contiguous) or [k,m] (transa = 1)
    split_tiles_launch<TF_BM>(A, m, k, lda, transa ? 1 : 0, (flags & GPK_GEMM_A_LOWER) ? 1 : 0, At, KB, batch > 1 ? m_per : 0,
                              a_batch_stride, st);
    GPK_LAUNCH_OK();
    // op(B)^T is [n, k]: stored [n,k] (transb = 1) or [k,n] (transb = 0 -> read transposed)
    split_tiles_launch<TF_BN>(B, n, k, ldb, transb ? 0 : 1, 0, Bt, KB, 0, 0, st);
    GPK_LAUNCH_OK();
  }
  const int lower = (flags & GPK_GEMM_LOWER_ONLY) ? 1 : 0;
  const int64_t ntm = mpad / TF_BM, ntn = npad / TF_BN;
  // clusters of 2 row tiles share the B planes by multicast; a single row tile has no pair
  const int cl = ntm >= 2 ? 2 : 1;
  int64_t nunits = 0;  // work units of cl vertically adjacent row tiles (the lowest tile decides whether a unit is needed)
  for (int64_t tn = 0; tn < ntn; ++tn)
    for (int64_t t0 = 0; t0 < ntm; t0 += cl)
      if (!(lower && tn * TF_BN > (t0 + cl - 1) * TF_BM + TF_BM - 1)) ++nunits;
  if (nunits == 0) return 0;
  const int sms = tf_num_sms();
  int nsplit = 1;
  // split K when the tiles alone cannot fill the machine and K is deep
  while (nunits * cl * nsplit < sms && KB / (nsplit * 2) >= 64 && nsplit < 64) nsplit *= 2;
  if (nsplit > 1 && !(flags & GPK_GEMM_COLSUMSQ)) {
    scale_c_kernel<<<(unsigned)std::min<int64_t>((m * n + 255) / 256, 148 * 8), 256, 0, st>>>(C, ldc, m, n, beta);
    GPK_LAUNCH_OK();
  }
  if ((flags & GPK_GEMM_COLSUMSQ) && nsplit > 1) nsplit = 1;  // sums of squares need the complete dot products
  const size_t smem = (size_t)TF_STAGES * TF_STAGE_BYTES + 2 * TF_EPI_BYTES + 256;
  static PerDeviceOnce attr_once;  // function attributes are per device
  GPK_TRY(attr_once.run([&]() -> int {
    GPK_CUDA_OK(cudaFuncSetAttribute(gemm_tf32_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GPK_CUDA_OK(cudaFuncSetAttribute(gemm_tf32_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
  }));
  int grid = (int)std::min<int64_t>(sms / cl * cl, nunits * cl * nsplit);
  const int tri = (flags & GPK_GEMM_A_LOWER) ? (transa ? 2 : 1) : 0;
  ProfScope ps(PROF_TC, st, 3.0 * (double)m * (double)n * (double)k * (tri ? 0.5 : 1.0));  // (m already includes the batch)  // tf32 MACs issued (3xTF32)
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(TF_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cl;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  const float* Atc = At;
  const float* Btc = Bt;
  const int KBi = (int)KB;
  const int tpb = batch > 1 ? (int)(m_per / TF_BM) : 0;
  if (cl == 2)
    GPK_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tf32_kernel<2>, Atc, Btc, C, ldc, m, n, KBi, nsplit, alpha, beta, flags, tri, err,
                                   tpb, c_batch_stride));
  else
    GPK_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tf32_kernel<1>, Atc, Btc, C, ldc, m, n, KBi, nsplit, alpha, beta, flags, tri, err,
                                   tpb, c_batch_stride));
  count_launch();
  return 0;
}

}  // namespace gpk
