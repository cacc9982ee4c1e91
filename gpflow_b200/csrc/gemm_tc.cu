// gemm_tc.cu — fp64 symmetric rank-k update on the 5th-generation tensor cores (tcgen05 + TMEM).
//
//     C[m, n]  -=  A[m, K] * A[0:n, K]^T          (row-major fp64; the Cholesky trailing update)
//
// tcgen05.mma has no f64 kind (f16/tf32/f8f6f4/i8/mx* only), so the fp64 operands are split into
// balanced base-256 digits with a per-row power-of-two scale (an Ozaki-style splitting, planes.cuh):
//
//     a_ik = 2^(e_i - 6) * sum_s 2^(-8 s) d_s(i,k),   d_0 in [-65, 65], d_s in [-128, 127]  (int8),  s = 0..S-1
//
// The digit products accumulate EXACTLY in int32 on the tensor cores (kind::i8); products with the
// same weight s+t = g < S share one TMEM accumulator.  S = 6 adds the (3,3) product in a seventh accumulator (the only
// dropped term whose mean on the diagonal of C is not zero), so a CTA tile (128 x 64) holds 7 accumulators of 64 columns
// (448 of the 512 TMEM columns) at S = 6 and S = 7 alike and issues 22 / 28 digit products per 32-deep k-step in 8 / 10
// concatenated MMAs.  The epilogue converts the integer planes to fp64, recombines them with exact power-of-two
// weights and the row/column scales, and ADDS the update into C with bulk reductions.  Error per dot product:
// ~K * (S + 1) * 2^(-8S + 2) relative to the row scales from the dropped products (tests/test_digit_slicing_model.py).
//
// Pipeline (per persistent CTA, 192 threads):
//   warp 0   producer : cp.async.bulk (1-D TMA) of PRE-TILED digit planes global -> shared, mbarrier
//   warp 1   issuer   : one elected lane issues tcgen05.mma (SS, no-swizzle K-major descriptors)
//   warps 2-5 epilogue: tcgen05.ld TMEM -> registers, recombine, bulk reduction (add) of the update into C
// The slicing pre-pass (slice_rows_kernel) writes the digit planes directly in the canonical UMMA
// shared-memory image (8x16-byte core matrices), so a stage is filled by plain bulk copies: no tensor
// map, no swizzle to keep consistent between three places.
//
// Replaces the SYRK inside tf.linalg.cholesky (gpflow/models/gpr.py:102 etc.) for the large-K levels
// of the recursion in potrf.cu; small-K levels and ragged shapes use the DMMA kernel of gemm.cu.
#include "tc_common.cuh"
#include "planes.cuh"

namespace gpk {

// Epilogue staging: every epilogue thread owns one row of 32 doubles (256 B, rows 272 B apart: 16-byte stores of a quarter
// warp then hit 32 different banks) from which a bulk reduction adds its half row of the update into C.
constexpr int TC_EPI_ROW = 272;
constexpr int TC_EPI_BYTES = 128 * TC_EPI_ROW;
constexpr int TC_SMEM_BUDGET = 226 * 1024 - TC_EPI_BYTES;  // pipeline stages: as many as fit (S planes of A and B per stage, tightly packed)
__host__ __device__ constexpr int tc_stages(int S) { return TC_SMEM_BUDGET / (S * (TC_ATILE + TC_BTILE)) > 6 ? 6 : TC_SMEM_BUDGET / (S * (TC_ATILE + TC_BTILE)); }
constexpr int TC_TMEM_COLS = 512;
// CTAs per cluster: the two CTAs of a cluster compute horizontally adjacent tiles and share their A tile by multicast
// (the kernel is L2 -> SM bandwidth bound)
constexpr int TC_CL = 2;

// ------------------------------------------------------------------------------------------------
// scales and slicing
// ------------------------------------------------------------------------------------------------
// static row scales from the ORIGINAL diagonal (planes.cuh): rowscale[i] = 2^(e_i - 6), sqrt(A_ii) < 2^e_i
__global__ void row_exp_kernel(const double* __restrict__ A, int64_t lda, int64_t n, int64_t npad,
                               double* __restrict__ rowscale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npad) return;
  double sc = 0.0;
  if (i < n) {
    const double d = A[i * lda + i];
    int e = 0;
    if (d > 0.0 && d < 1e300) e = ilogb(sqrt(d)) + 1;
    sc = scalbn(1.0, e - 6);
  }
  rowscale[i] = sc;
}

// dynamic slicing, one CTA per row: rows [row0, row0 + nrows) of the k-range [k0, k0 + K) get the scale of their
// running maximum over that range (the extra rows below the square part)
__global__ void __launch_bounds__(256)
slice_rows_kernel(const double* __restrict__ P, int64_t ld, int64_t row0, int64_t nrows, int64_t k0, int64_t K,
                  TcPlanes pl) {
  __shared__ double wmax[8];
  const int64_t i = blockIdx.x;
  tc_slice_row_cta(P + i * ld, row0 + i, k0, K, pl, wmax);
}

// shared-memory matrix descriptor: K-major, no swizzle, LBO = 128 B (next 16-byte k chunk),
// SBO = 256 B (next group of 8 rows), version 1 (Blackwell)
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) |
         (1ull << 46);
}
// instruction descriptor: D = S32, A = B = signed int8, both K-major, N = 64, M = 128
__host__ __device__ constexpr uint32_t tc_idesc_n(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
}
constexpr uint32_t TC_IDESC = tc_idesc_n(TC_BN);

struct TcTileIter {  // identical enumeration in every warp role
  // Work unit = TC_CL horizontally adjacent tiles (tm, tnb .. tnb+TC_CL-1), one per CTA of a cluster, so the
  // cluster shares the A tile (multicast).  Order: pass 0 = the "head" units (first 128 columns) of every
  // row tile, pass 1 = the rest: the next diagonal block's inputs are complete early (look-ahead).
  static constexpr int64_t head_w = 128 / TC_BN;  // column tiles of the head
  int64_t ntm, ntn;
  int lower, pass, rank;
  int64_t tm, tnb, tn, idx;
  __device__ TcTileIter(int64_t m, int64_t n, int lower_, int rank_)
      : lower(lower_), pass(0), rank(rank_), tm(0), tnb(-TC_CL), tn(0), idx(-1) {
    ntm = (m + TC_BM - 1) / TC_BM;
    ntn = (n + TC_BN - 1) / TC_BN;
  }
  __device__ int64_t ncols(int64_t t) const {
    const int64_t lim = 2 * t + 2;  // column tiles touching the lower triangle of row tile t
    return lower ? (lim < ntn ? lim : ntn) : ntn;
  }
  __device__ bool is_head() const { return pass == 0; }
  // tile index used for LOADING B (clamped: the odd CTA of a last, half-empty unit loads valid memory and
  // its epilogue writes nothing because its columns are >= n)
  __device__ int64_t tn_load() const { return tn < ntn ? tn : ntn - 1; }
  // false for the padding tiles of a unit that sticks out of the (lower-triangular) tile set: computed, not stored
  __device__ bool valid() const { return tn < ncols(tm); }
  // advances to this cluster's next unit; false when exhausted
  __device__ bool next() {
    const int64_t nunits_grid = gridDim.x / TC_CL, my = blockIdx.x / TC_CL;
    for (;;) {
      tnb += TC_CL;
      for (;;) {
        if (pass == 0) {
          const int64_t lim = ncols(tm) < head_w ? ncols(tm) : head_w;
          if (tm < ntm && tnb >= lim) { ++tm; tnb = 0; continue; }
          if (tm >= ntm) { pass = 1; tm = 0; tnb = head_w; continue; }
        } else {
          if (tm < ntm && tnb >= ncols(tm)) { ++tm; tnb = head_w; continue; }
          if (tm >= ntm) return false;
        }
        break;
      }
      ++idx;
      if (idx % nunits_grid == my) { tn = tnb + rank; return true; }
    }
  }
};

template <int S>
__global__ void __launch_bounds__(192, 1)
syrk_i8_kernel(TcPlanes pl, int64_t rb0, int64_t kb0, double* __restrict__ C, int64_t ldc, int64_t m, int64_t n, int KB,
               int lower, int* head_flag) {
  // rows of C = global rows 128 rb0 + ..., columns of C = the same rows (C is the block right of the k-range
  // [32 kb0, 32 (kb0 + KB)) on the diagonal); operands come from the digit-plane store (planes.cuh)
  const double* __restrict__ rowscale = pl.rowscale + rb0 * TC_BM;
  int* err = pl.err;
  // even S (6): one more accumulator for the (S/2, S/2) digit product (planes.cuh)
  constexpr bool SQ = (S == 6);
  constexpr int H = S / 2, NACC = S + (SQ ? 1 : 0);
  extern __shared__ __align__(1024) uint8_t tc_smem[];
  constexpr uint32_t stage_bytes = (uint32_t)S * (TC_ATILE + TC_BTILE);
  constexpr int TC_STAGES = tc_stages(S);   // S = 7: 5 stages of 42 KB, S = 6: 6 of 36 KB
  constexpr uint32_t stage_stride = (uint32_t)S * (TC_ATILE + TC_BTILE);
  uint8_t* epi_area = tc_smem + TC_STAGES * (size_t)stage_stride;  // [128][TC_EPI_ROW]
  uint8_t* bar_area = epi_area + TC_EPI_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(bar_area);  // full[4], empty[4], tmem_full, tmem_empty
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_STAGES + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + TC_STAGES);
  const uint32_t tfull = smem_u32(bars + 2 * TC_STAGES), tempty = smem_u32(bars + 2 * TC_STAGES + 1);

  if (threadIdx.x == 0) {
    if (blockIdx.x == 0) trace_mark(4, 0);
    for (int i = 0; i < TC_STAGES; ++i) {
      mbar_init(full0 + 8 * i, 1);
      mbar_init(empty0 + 8 * i, TC_CL);  // every CTA of the cluster releases a stage (A is multicast into all)
    }
    mbar_init(tfull, 1);
    mbar_init(tempty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)TC_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // peer barriers initialised before any multicast copy / commit targets them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0 && blockIdx.x == 0) trace_mark(4, 10);  // prologue done (barriers, TMEM, cluster sync)
  const int rank = (int)cluster_ctarank();
  constexpr uint16_t cl_mask = (uint16_t)((1u << TC_CL) - 1);

  if (__all_sync(0xffffffffu, warp == 0)) {  // vote: the role branch is warp-uniform and the compiler knows it
    // ===== producer (whole warp runs the loop; one elected lane issues the copies) =====
    TcTileIter it(m, n, lower, rank);
    uint32_t st = 0, ph = 0;
    while (it.next()) {
      const int8_t* a_src = pl.tile(rb0 + it.tm, kb0);
      const int64_t tl = it.tn_load();
      const int8_t* b_src = pl.tile(rb0 + (tl >> 1), kb0) + (tl & 1) * TC_BTILE;
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(empty0 + 8 * st, ph ^ 1, err, 101);
        if (elect_one()) {
          const uint32_t fb = full0 + 8 * st;
          mbar_expect_tx(fb, stage_bytes);
          const uint32_t sa = smem_u32(tc_smem + (size_t)st * stage_stride);
          const uint32_t sb = sa + S * TC_ATILE;
          // each CTA fetches 1/TC_CL of every A plane (64 of the 128 rows) and multicasts it to the cluster
          constexpr uint32_t part = TC_ATILE / TC_CL;
#pragma unroll
          for (int s2 = 0; s2 < S; ++s2)
            bulk_g2s_mc(sa + s2 * TC_ATILE + rank * part, a_src + ((size_t)kb * S + s2) * TC_ATILE + rank * part, part, fb,
                        cl_mask);
#pragma unroll
          for (int t = 0; t < S; ++t)
            bulk_g2s(sb + t * TC_BTILE, b_src + ((size_t)kb * S + t) * TC_ATILE, TC_BTILE, fb);
        }
        __syncwarp();
        if (++st == TC_STAGES) { st = 0; ph ^= 1; }
      }
    }
  } else if (__all_sync(0xffffffffu, warp == 1)) {
    // ===== MMA issuer (uniform control flow, one elected lane issues) =====
    TcTileIter it(m, n, lower, rank);
    uint32_t st = 0, ph = 0, tph = 0;
    const uint64_t desc_hi = ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46);
    while (it.next()) {
      mbar_wait(tempty, tph ^ 1, err, 102);  // epilogue has drained the accumulators
      tc_fence_after();
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(full0 + 8 * st, ph, err, 103);
        tc_fence_after();
        const uint32_t sa = smem_u32(tc_smem + (size_t)st * stage_stride);
        const uint64_t ad0 = desc_hi | (uint64_t)((sa & 0x3FFFFu) >> 4);
        const uint64_t bd0 = ad0 + ((S * TC_ATILE) >> 4);
        if (elect_one()) {
          // the S-s digit products of A plane s share the A operand and write ADJACENT accumulators, and the B planes are
          // contiguous in shared memory with the same 8-row-group stride: one MMA with N = 64 (S-s) (split at 256) replaces
          // S-s MMAs with N = 64 -- 10 instructions per k-step instead of 28 for S = 7
#pragma unroll
          for (int s = 0; s < S; ++s)
#pragma unroll
            for (int t = 0; t + s < S; t += 4) {
              int c = (S - s - t) < 4 ? (S - s - t) : 4;
              // the square term rides on the MMA of A plane H (B planes 0 .. H instead of 0 .. H-1) except in the first
              // k-step, where its accumulator starts from zero while the others of that MMA already hold products
              if (SQ && s == H && t == 0 && kb > 0) c = H + 1;
              tc_mma_i8(tmem_base + (uint32_t)(s + t) * TC_BN, ad0 + (uint64_t)(s * (TC_ATILE >> 4)),
                        bd0 + (uint64_t)(t * (TC_BTILE >> 4)), tc_idesc_n(TC_BN * c), (kb > 0 || s > 0) ? 1u : 0u);
            }
          if (SQ && kb == 0)
            tc_mma_i8(tmem_base + (uint32_t)S * TC_BN, ad0 + (uint64_t)(H * (TC_ATILE >> 4)),
                      bd0 + (uint64_t)(H * (TC_BTILE >> 4)), TC_IDESC, 0u);
          // frees the stage (in every CTA of the cluster) once these copies / MMAs have read it
          tc_commit_mc(empty0 + 8 * st, cl_mask);
        }
        __syncwarp();
        if (++st == TC_STAGES) { st = 0; ph ^= 1; }
      }
      if (elect_one()) tc_commit(tfull);  // accumulators complete
      __syncwarp();
      tph ^= 1;
    }
  } else {
    // ===== epilogue (4 warps = 128 TMEM lanes) =====
    // One thread = one row of the tile.  Per 32-column half: drain the accumulators (tcgen05.ld), recombine the digit orders
    // in fp64, scale, write the half row of the UPDATE (-rs cs acc) into the thread's own 256-byte row of the staging
    // buffer and let a bulk reduction (cp.reduce.async.bulk .add.f64) add it into C in L2.  C is never read by the SM, the
    // global traffic is whole 256-byte row segments issued by the copy engine, and everything is thread-local (a thread's
    // fence.proxy.async orders its own shared-memory stores before its own bulk operation).  Every element of C receives
    // exactly one reduction per launch, so the result does not depend on any ordering.
    // (The previous read-modify-write epilogue -- 16-byte loads / stores of a thread's own row, 32 lines per warp
    // instruction -- took 7.7 us per tile on the LSU: profiles/r2/trace_c2_phases.csv.)
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    TcTileIter it(m, n, lower, rank);
    uint32_t tph = 0;
    const bool vec_ok = ((ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
    double* srow = reinterpret_cast<double*>(epi_area + (size_t)(q * 32 + lane) * TC_EPI_ROW);
    const uint32_t srow_s = smem_u32(srow);
    while (it.next()) {
      const int64_t row = it.tm * TC_BM + q * 32 + lane;
      const int64_t colb = it.tn * TC_BN;
      const bool live = row < m && it.valid();
      const bool fullw = vec_ok && colb + TC_BN <= n;
      double* crow = C + (live ? row : 0) * ldc + colb;
      const double rs = live ? -__ldg(rowscale + row) : 0.0;
      const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
      mbar_wait(tfull, tph, err, 104);
      tc_fence_after();
      const bool tr0 = blockIdx.x == 0 && tph == 0 && threadIdx.x == 64 && it.is_head();  // (first tile of CTA 0: timeline marks)
      if (tr0) trace_mark(4, 13);  // accumulators complete
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        const double* sc = rowscale + colb + half * 32;
        // the bulk reduction issued from this row one half ago has finished READING the staging row
        if (fullw) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
#pragma unroll
        for (int qq = 0; qq < 2; ++qq) {  // 16 columns at a time: all NACC accumulator reads in flight, one wait
          uint32_t v[NACC][16];
#pragma unroll
          for (int g = 0; g < NACC; ++g) tc_ld16_nowait(lane_addr + (uint32_t)(g * TC_BN + half * 32 + qq * 16), v[g]);
          tc_ld_wait();
          if (half == 1 && qq == 1) {  // accumulators drained: the MMA warp may start the next tile
            tc_fence_before();
            mbar_arrive(tempty);
          }
          double acc[16];
#pragma unroll
          for (int c = 0; c < 16; ++c) acc[c] = 0.0;
          double w = 1.0;
#pragma unroll
          for (int g = 0; g < NACC; ++g) {
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[c] = fma(tc_int_to_double((int)v[g][c]), w, acc[c]);
            w *= 0.00390625;  // 2^-8 (radix 256)
          }
          if (fullw) {
#pragma unroll
            for (int c2 = 0; c2 < 8; ++c2) {
              const double2 s2 = __ldg(reinterpret_cast<const double2*>(sc + qq * 16 + 2 * c2));
              double2 o;
              o.x = (rs * s2.x) * acc[2 * c2];
              o.y = (rs * s2.y) * acc[2 * c2 + 1];
              *reinterpret_cast<double2*>(srow + qq * 16 + 2 * c2) = o;
            }
          } else if (live) {  // ragged right edge / unaligned C: element-wise read-modify-write (rare)
#pragma unroll
            for (int c = 0; c < 16; ++c) {  // (fully unrolled: a runtime index would move acc[] to local memory)
              const int cc = half * 32 + qq * 16 + c;
              if (colb + cc < n) crow[cc] = fma(rs * __ldg(sc + qq * 16 + c), acc[c], crow[cc]);
            }
          }
        }
        if (tr0) trace_mark(4, 14 + 2 * half);  // TMEM drained + converted + staged (14 / 16)
        if (fullw) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          if (live)
            asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], 256;" ::"l"(crow + half * 32),
                         "r"(srow_s)
                         : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (tr0) trace_mark(4, 15 + 2 * half);  // update issued (15 / 17)
      }
      tph ^= 1;
      if (head_flag && it.is_head()) {  // publish this head tile once all four epilogue warps' reductions are complete
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        asm volatile("fence.proxy.async.global;" ::: "memory");  // the reductions (async proxy) before the generic-proxy release below
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (threadIdx.x == 64) {
          __threadfence();
          trace_mark(4, 1);  // a head tile published
          atomicAdd(head_flag, 1);
          const int u = diag_units_tile(it.tm * TC_BM, it.tn * TC_BN, TC_BM, TC_BN, m, n);
          if (u) atomicAdd(head_flag + 1, u);  // progress on the next diagonal block
        }
      }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // the staging rows stay valid until every reduction has read them
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) trace_mark(4, blockIdx.x == 0 ? 2 : 3);
  cluster_sync_all();  // no CTA leaves while a peer may still multicast into its shared memory
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TC_TMEM_COLS)
                 : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
int trace_set_tc(TraceBuf tb) {
  GPK_CUDA_OK(cudaMemcpyToSymbol(g_trace, &tb, sizeof(tb)));
  return 0;
}

size_t tc_planes_bytes(int64_t n, int64_t rows) {
  const int64_t nbk = (n + TC_BM - 1) / TC_BM, rbt = (rows + TC_BM - 1) / TC_BM;
  return align_up((size_t)plane_prefix(rbt, nbk) * TC_MAXS * TC_ATILE, 256) + align_up((size_t)rbt * TC_BM * sizeof(double), 256) + 256;
}

TcPlanes tc_planes_layout(void* ws, int64_t n, int64_t rows, int S) {
  const int64_t nbk = (n + TC_BM - 1) / TC_BM, rbt = (rows + TC_BM - 1) / TC_BM;
  TcPlanes pl;
  pl.planes = (int8_t*)ws;
  pl.rowscale = (double*)((char*)ws + align_up((size_t)plane_prefix(rbt, nbk) * TC_MAXS * TC_ATILE, 256));
  pl.err = (int*)((char*)pl.rowscale + align_up((size_t)rbt * TC_BM * sizeof(double), 256));
  pl.S = S;
  pl.nbk = nbk;
  pl.n_sq = n;
  return pl;
}

int tc_row_exponents(const double* A, int64_t lda, const TcPlanes& pl, cudaStream_t st) {
  const int64_t npad = (pl.n_sq + TC_BM - 1) / TC_BM * TC_BM;
  ProfScope ps(PROF_MISC, st);
  row_exp_kernel<<<(unsigned)((npad + 255) / 256), 256, 0, st>>>(A, lda, pl.n_sq, npad, pl.rowscale);
  GPK_LAUNCH_OK();
  return 0;
}

int tc_slice_rows(const double* P, int64_t ld, int64_t row0, int64_t nrows, int64_t k0, int64_t K, const TcPlanes& pl,
                  cudaStream_t st) {
  if (nrows <= 0) return 0;
  GPK_CHECK_ARG(K % TC_KB == 0 && k0 % TC_KB == 0, "tc_slice_rows: k-range must be a multiple of 32");
  ProfScope ps(PROF_MISC, st);
  slice_rows_kernel<<<(unsigned)nrows, 256, 0, st>>>(P, ld, row0, nrows, k0, K, pl);
  GPK_LAUNCH_OK();
  return 0;
}

static int tc_num_sms() {  // of the CURRENT device (a process may drive several)
  int dev = 0, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n > 0 ? n : 148;
}

// C[m,n] -= L[r0:r0+m, k0:k0+K] L[r0:r0+n, k0:k0+K]^T (lower tiles only if `lower`); K, k0 % 32 == 0, r0 % 128 == 0, n <= m.
int syrk_tc_planes(double* C, int64_t ldc, int64_t m, int64_t n, const TcPlanes& pl, int64_t r0, int64_t k0, int64_t K,
                   int lower, cudaStream_t st, const GemmOpts* opts) {
  const int S = pl.S;
  int* hf = opts ? opts->head_flag : nullptr;
  GPK_CHECK_ARG(K % TC_KB == 0 && K > 0 && n <= m && r0 % TC_BM == 0 && k0 % TC_KB == 0,
                "syrk_tc: unsupported shape m=%lld n=%lld K=%lld r0=%lld k0=%lld", (long long)m, (long long)n, (long long)K,
                (long long)r0, (long long)k0);
  const int64_t rb0 = r0 / TC_BM, kb0 = k0 / TC_KB;
  const size_t smem = tc_stages(S) * (size_t)S * (TC_ATILE + TC_BTILE) + TC_EPI_BYTES + 256;
  // Both operands from shared memory with the digit products of one A plane CONCATENATED along N (one MMA of N up to 256
  // instead of up to four of N = 64): scripts/mb_mma.cu measures 52.9 cycles per N = 64 SS MMA against a floor of 32,
  // but 128.0 per N = 256 MMA (= the floor), and the tcgen05.cp of the TS form costs 137 cycles per k-step on top.
  // C2: 8.70 ms (TS, N = 64) -> 8.14 ms (SS, concatenated).
  // number of work units (TC_CL adjacent tiles)
  const int64_t ntm = (m + TC_BM - 1) / TC_BM, ntn = (n + TC_BN - 1) / TC_BN;
  int64_t nunits = 0;
  for (int64_t t = 0; t < ntm; ++t) {
    const int64_t nc = lower ? (2 * t + 2 < ntn ? 2 * t + 2 : ntn) : ntn;
    nunits += (nc + TC_CL - 1) / TC_CL;
  }
  int grid = tc_num_sms() - (hf ? 1 : 0);  // look-ahead: leave one SM for the concurrent leaf kernel
  grid = grid / TC_CL * TC_CL;
  if (nunits * TC_CL < grid) grid = (int)(nunits * TC_CL);
  if (grid < 1) return 0;
  const int KBn = (int)(K / TC_KB);
  // issued int8 MACs: every tile of every unit (padding tiles included) x k-steps x S(S+1)/2 digit products
  ProfScope ps(PROF_TC, st, (double)nunits * TC_CL * KBn * (S * (S + 1) / 2 + (S == 6 ? 1 : 0)) * (double)(TC_BM * TC_BN * TC_KB));
  auto launch = [&](auto kern) -> int {
    GPK_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(192);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)TC_CL;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    GPK_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, pl, rb0, kb0, C, ldc, m, n, KBn, lower, hf));
    count_launch();
    return 0;
  };
  return S == 6 ? launch(syrk_i8_kernel<6>) : launch(syrk_i8_kernel<7>);
}

}  // namespace gpk
