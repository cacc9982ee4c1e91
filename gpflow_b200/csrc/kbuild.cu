// kbuild.cu — fused pairwise covariance builder (K-build) for sm_100a.
//
// One pass over the output: each CTA owns a 64x64 tile of K, stages the (weighted) active columns
// of its X / X2 row blocks in shared memory, forms the Gram term with a 4x4 register micro-tile,
// turns it into the scaled squared distance with the norm expansion the reference uses
// (gpflow/utilities/ops.py:105-122, on inputs scaled as in kernels/stationaries.py:77-79), applies
// every leaf function (stationaries.py:209-313, statics.py:57-91, linears.py:60-68) and folds the
// Sum/Product tree (kernels/base.py:281-314) in registers, adds the diagonal shift
// (utilities/model_utils.py:33-38, covariances/kuus.py:33) and writes K once with 16-byte
// vector stores.  The reference materialises one [N,N2] temporary per elementwise op instead.
//
// A single stationary leaf takes the fast path further down (persistent CTAs, register-prefetched operand
// pipeline, folded scales, table-driven exp / MUFU-seeded sqrt, lower tiles only + mirrored stores).
//
// Algorithmic HBM bytes per launch: T*(N*N2 + (N+N2)*D)  (GPK_LOWER: T*(N(N+1)/2 + N*D)).
#include <math.h>
#include <stdarg.h>

#include <vector>

#include <type_traits>
#include "common.cuh"

namespace gpk {

constexpr int KB_MAXG = 4;      // gram groups (distinct (active_dims, weights) sets)
constexpr int KB_MAXL = 12;     // leaves
constexpr int KB_MAXDIMS = 256; // total active dims over groups
constexpr int KB_MAXOPS = 32;
constexpr int KB_OP_ADD = 0xFE, KB_OP_MUL = 0xFF;
constexpr int KB_TILE = 64;     // output tile edge
constexpr int KB_KC = 32;       // dims staged per chunk

struct KProg {
  int n_groups, n_leaves, n_ops, symmetric;
  int g_ndims[KB_MAXG], g_off[KB_MAXG], g_weighted[KB_MAXG];
  int l_type[KB_MAXL], l_group[KB_MAXL];
  double l_scale[KB_MAXL], l_var[KB_MAXL], l_alpha[KB_MAXL];
  unsigned char ops[KB_MAXOPS];
  short dims[KB_MAXDIMS];
  double w[KB_MAXDIMS];
};
static_assert(sizeof(KProg) < 4000, "KProg must fit the kernel parameter space");

// ---------------------------------------------------------------------------------------------
// host: flatten the reference-shaped node list into groups / leaves / postfix ops
// ---------------------------------------------------------------------------------------------
static bool is_leaf_op(int op) { return (op >= GPK_K_RBF && op <= GPK_K_CONSTANT) || op == GPK_K_POLYNOMIAL; }
static bool uses_gram(int op) { return op <= GPK_K_LINEAR || op == GPK_K_POLYNOMIAL; }
static bool linear_like(int op) { return op == GPK_K_LINEAR || op == GPK_K_POLYNOMIAL; }  // variance weights on the A side

static int emit_ops(const gpk_knode* nodes, int idx, const std::vector<int>& leaf_of, KProg& p, int& depth,
                    int& max_depth) {
  const gpk_knode& nd = nodes[idx];
  if (is_leaf_op(nd.op)) {
    if (p.n_ops >= KB_MAXOPS) return -1;
    p.ops[p.n_ops++] = (unsigned char)leaf_of[idx];
    depth++;
    if (depth > max_depth) max_depth = depth;
    return 0;
  }
  if (nd.n_children < 1 || nd.n_children > GPK_MAX_CHILDREN) return -1;
  for (int c = 0; c < nd.n_children; ++c) {
    if (nd.child[c] < 0 || nd.child[c] >= idx) return -1;  // children precede parents
    if (emit_ops(nodes, nd.child[c], leaf_of, p, depth, max_depth)) return -1;
    if (c > 0) {
      if (p.n_ops >= KB_MAXOPS) return -1;
      p.ops[p.n_ops++] = nd.op == GPK_K_SUM ? KB_OP_ADD : KB_OP_MUL;
      depth--;
    }
  }
  return 0;
}

int compile_kprog(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, int64_t D,
                  KProg& p) {
  memset(&p, 0, sizeof(p));
  GPK_CHECK_ARG(nodes && n_nodes > 0, "kbuild: empty kernel expression");
  GPK_CHECK_ARG(D > 0 && D < 32768, "kbuild: bad input dimension D=%lld", (long long)D);
  std::vector<int> leaf_of(n_nodes, -1);
  int tot_dims = 0;
  for (int i = 0; i < n_nodes; ++i) {
    const gpk_knode& nd = nodes[i];
    GPK_CHECK_ARG(nd.op >= GPK_K_RBF && nd.op <= GPK_K_POLYNOMIAL, "kbuild: unknown kernel op %d", nd.op);
    if (!is_leaf_op(nd.op)) continue;
    GPK_CHECK_ARG(p.n_leaves < KB_MAXL, "kbuild: more than %d leaf kernels", KB_MAXL);
    int l = p.n_leaves++;
    leaf_of[i] = l;
    p.l_type[l] = nd.op;
    p.l_var[l] = nd.variance;
    p.l_alpha[l] = nd.alpha;
    p.l_scale[l] = nd.op == GPK_K_POLYNOMIAL ? nd.lengthscale : 1.0;  // Polynomial: the offset rides in this slot
    p.l_group[l] = -1;
    if (!uses_gram(nd.op)) continue;
    int nd_dims = nd.n_dims > 0 ? nd.n_dims : (int)D;
    GPK_CHECK_ARG(nd.n_dims == 0 || dims != nullptr, "kbuild: active dims given without index array");
    GPK_CHECK_ARG(nd.n_ard == 0 || (nd.n_ard == nd_dims && ard != nullptr),
                  "kbuild: size of ARD parameter (%d) does not match active dims (%d)", nd.n_ard, nd_dims);
    // weights of this leaf's gram term
    std::vector<double> w;
    if (nd.n_ard > 0) {
      w.resize(nd_dims);
      for (int d = 0; d < nd_dims; ++d) {
        double a = ard[nd.ard_off + d];
        w[d] = linear_like(nd.op) ? a : 1.0 / a;  // stationary: X/l on BOTH sides (stationaries.py:77-79)
      }
      if (linear_like(nd.op)) p.l_var[l] = 1.0;
    } else if (!linear_like(nd.op)) {
      p.l_scale[l] = 1.0 / (nd.lengthscale * nd.lengthscale);
    }
    // find or create the group
    int g = -1;
    for (int c = 0; c < p.n_groups && g < 0; ++c) {
      const int wmode = w.empty() ? 0 : (linear_like(nd.op) ? 1 : 2);
      if (p.g_ndims[c] != nd_dims || p.g_weighted[c] != wmode) continue;
      bool same = true;
      for (int d = 0; d < nd_dims && same; ++d) {
        int col = nd.n_dims > 0 ? dims[nd.dims_off + d] : d;
        same = p.dims[p.g_off[c] + d] == col && (w.empty() || p.w[p.g_off[c] + d] == w[d]);
      }
      if (same) g = c;
    }
    if (g < 0) {
      GPK_CHECK_ARG(p.n_groups < KB_MAXG, "kbuild: more than %d distinct (active_dims, ARD) groups", KB_MAXG);
      GPK_CHECK_ARG(tot_dims + nd_dims <= KB_MAXDIMS, "kbuild: more than %d active dims in total", KB_MAXDIMS);
      g = p.n_groups++;
      p.g_ndims[g] = nd_dims;
      p.g_off[g] = tot_dims;
      p.g_weighted[g] = w.empty() ? 0 : (linear_like(nd.op) ? 1 : 2);  // 1: A side only, 2: both sides
      for (int d = 0; d < nd_dims; ++d) {
        int col = nd.n_dims > 0 ? dims[nd.dims_off + d] : d;
        GPK_CHECK_ARG(col >= 0 && col < D, "kbuild: active dim %d out of range [0,%lld)", col, (long long)D);
        p.dims[tot_dims + d] = (short)col;
        p.w[tot_dims + d] = w.empty() ? 1.0 : w[d];
      }
      tot_dims += nd_dims;
    }
    p.l_group[l] = g;
  }
  int depth = 0, max_depth = 0;
  GPK_CHECK_ARG(emit_ops(nodes, n_nodes - 1, leaf_of, p, depth, max_depth) == 0,
                "kbuild: malformed or too large kernel expression (max %d postfix ops)", KB_MAXOPS);
  GPK_CHECK_ARG(max_depth <= 4, "kbuild: kernel expression nests deeper than the 4-entry evaluation stack");
  return 0;
}

// ---------------------------------------------------------------------------------------------
// device
// ---------------------------------------------------------------------------------------------
template <typename T>
struct KMath;
template <>
struct KMath<double> {
  static __device__ __forceinline__ double exp_(double x) { return exp(x); }
  static __device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
  static __device__ __forceinline__ double pow_(double x, double y) { return pow(x, y); }
};
template <>
struct KMath<float> {
  static __device__ __forceinline__ float exp_(float x) { return expf(x); }
  static __device__ __forceinline__ float sqrt_(float x) { return sqrtf(x); }
  static __device__ __forceinline__ float pow_(float x, float y) { return powf(x, y); }
};

// value of one leaf given the (weighted) gram term `dot` and the row / column norms
template <typename T>
__device__ __forceinline__ T leaf_value(int type, T dot, T na, T nb, T scale, T var, T alpha, bool on_diag) {
  using M = KMath<T>;
  if (type == GPK_K_LINEAR) return var * dot;
  if (type == GPK_K_POLYNOMIAL) return M::pow_(var * dot + scale, alpha);  // linears.py:108 (offset rides in `scale`)
  if (type == GPK_K_CONSTANT) return var;
  if (type == GPK_K_WHITE) return on_diag ? var : T(0);
  T r2 = scale * (na + nb - T(2) * dot);  // ops.py:113-122 — may be slightly negative
  if (type == GPK_K_RBF) return var * M::exp_(T(-0.5) * r2);                 // stationaries.py:210
  if (type == GPK_K_RQ) return var * M::pow_(T(1) + T(0.5) * r2 / alpha, -alpha);  // :238
  T r = M::sqrt_(fmax(r2, T(1e-36)));                                         // :114
  if (type == GPK_K_MATERN52) {                                               // :311-313
    const T s5 = T(2.23606797749978969641);
    return var * (T(1) + s5 * r + T(5.0 / 3.0) * r * r) * M::exp_(-s5 * r);
  }
  if (type == GPK_K_MATERN32) {                                               // :290-292
    const T s3 = T(1.73205080756887729353);
    return var * (T(1) + s3 * r) * M::exp_(-s3 * r);
  }
  if (type == GPK_K_MATERN12) return var * M::exp_(-r);                       // :270-271
  return var * M::exp_(T(-0.5) * r);                                          // Exponential :250-251
}

// element e (= r*4+c) of a register-resident 4x4 tile without dynamic register indexing
template <typename T>
__device__ __forceinline__ T sel16(const T (&d)[4][4], int e) {
  T v = d[0][0];
#pragma unroll
  for (int q = 1; q < 16; ++q)
    if (e == q) v = d[q >> 2][q & 3];
  return v;
}

template <typename T, int NG>
__global__ void __launch_bounds__(256)
kbuild_kernel(const __grid_constant__ KProg prog, const T* __restrict__ X, int64_t N, int64_t ldx,
              const T* __restrict__ X2, int64_t N2, int64_t ldx2, T* __restrict__ K, int64_t ldk, int lower,
              T diag_scalar, const T* __restrict__ diag_vec, int vec_ok) {
  const int bx = blockIdx.x, by = blockIdx.y;
  if (lower && bx > by) return;
  __shared__ __align__(16) T sA[KB_KC][KB_TILE];
  __shared__ __align__(16) T sB[KB_KC][KB_TILE];
  __shared__ T sNa[NG][KB_TILE];
  __shared__ T sNb[NG][KB_TILE];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t row0 = (int64_t)by * KB_TILE, col0 = (int64_t)bx * KB_TILE;
  const bool sym = prog.symmetric != 0;
  const T* Xb = sym ? X : X2;
  const int64_t ldb = sym ? ldx : ldx2;

  T dots[NG][4][4];
#pragma unroll
  for (int g = 0; g < NG; ++g)
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) dots[g][r][c] = T(0);

  if (tid < KB_TILE) {
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      sNa[g][tid] = T(0);
      sNb[g][tid] = T(0);
    }
  }

#pragma unroll
  for (int g = 0; g < NG; ++g) {
    if (g >= prog.n_groups) break;
    const int nd = prog.g_ndims[g], off = prog.g_off[g];
    for (int d0 = 0; d0 < nd; d0 += KB_KC) {
      const int kc = min(KB_KC, nd - d0);
      __syncthreads();
      // stage: sA[d][r] = w_d * X[row0+r, dims[d]],  sB[d][c] = X2[col0+c, dims[d]]
      for (int e = tid; e < kc * KB_TILE; e += 256) {
        const int d = e % kc, r = e / kc;  // consecutive threads walk one row's dims (same cache lines)
        const int col = prog.dims[off + d0 + d];
        const int64_t gr = row0 + r, gc = col0 + r;
        T a = gr < N ? X[gr * ldx + col] : T(0);
        T b = gc < N2 ? Xb[gc * ldb + col] : T(0);
        const T wv = T(prog.w[off + d0 + d]);
        sA[d][r] = a * wv;
        sB[d][r] = prog.g_weighted[g] == 2 ? b * wv : b;
      }
      __syncthreads();
      // squared norms of the staged (scaled) rows / columns: same expression on both sides
      if (tid < 2 * KB_TILE) {
        const int r = tid & (KB_TILE - 1);
        T acc = T(0);
        if (tid < KB_TILE) {
          for (int d = 0; d < kc; ++d) { const T a = sA[d][r]; acc = fma(a, a, acc); }
          sNa[g][r] += acc;
        } else {
          for (int d = 0; d < kc; ++d) { const T b = sB[d][r]; acc = fma(b, b, acc); }
          sNb[g][r] += acc;
        }
      }
      // gram micro-tile
      for (int d = 0; d < kc; ++d) {
        T a[4], b[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) a[r] = sA[d][ty * 4 + r];
#pragma unroll
        for (int c = 0; c < 4; ++c) b[c] = sB[d][tx * 4 + c];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) dots[g][r][c] = fma(a[r], b[c], dots[g][r][c]);
      }
    }
  }
  __syncthreads();

  // epilogue: leaf functions + postfix Sum/Product fold.  The 16 elements of the micro-tile are
  // processed by ONE rolled loop (values staged in a small local array): unrolling it replicates
  // the exp/sqrt/pow code 16x (180 KB of SASS) and makes the kernel instruction-fetch bound.
  T vals[16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) vals[r * 4 + c] = NG == 1 ? dots[0][r][c] : T(0);
  const int n_ops = prog.n_ops;
#pragma unroll 1
  for (int e = 0; e < 16; ++e) {
    const int r = e >> 2, c = e & 3;
    const int64_t gi = row0 + ty * 4 + r, gj = col0 + tx * 4 + c;
    const bool on_diag = sym && gi == gj;
    T s0 = T(0), s1 = T(0), s2 = T(0), s3 = T(0);
    for (int o = 0; o < n_ops; ++o) {
      const int op = prog.ops[o];
      if (op < KB_MAXL) {
        const int g = prog.l_group[op];
        T dot = T(0), na = T(0), nb = T(0);
        if (NG == 1) {
          dot = vals[e];
          if (g == 0) { na = sNa[0][ty * 4 + r]; nb = sNb[0][tx * 4 + c]; }
        } else {
#pragma unroll
          for (int gg = 0; gg < NG; ++gg)
            if (g == gg) {
              dot = sel16(dots[gg], e);
              na = sNa[gg][ty * 4 + r];
              nb = sNb[gg][tx * 4 + c];
            }
        }
        T v = leaf_value<T>(prog.l_type[op], dot, na, nb, T(prog.l_scale[op]), T(prog.l_var[op]),
                            T(prog.l_alpha[op]), on_diag);
        s3 = s2; s2 = s1; s1 = s0; s0 = v;
      } else {
        s0 = op == KB_OP_ADD ? s1 + s0 : s1 * s0;
        s1 = s2; s2 = s3;
      }
    }
    if (on_diag) s0 += diag_scalar + (diag_vec ? diag_vec[gi] : T(0));
    vals[e] = s0;
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int64_t gi = row0 + ty * 4 + r;
    if (gi < N) {
      const int64_t gj0 = col0 + tx * 4;
      T* dst = K + gi * ldk + gj0;
      if (vec_ok && gj0 + 3 < N2) {
        if (sizeof(T) == 8) {
          reinterpret_cast<double2*>(dst)[0] = make_double2((double)vals[r * 4 + 0], (double)vals[r * 4 + 1]);
          reinterpret_cast<double2*>(dst)[1] = make_double2((double)vals[r * 4 + 2], (double)vals[r * 4 + 3]);
        } else {
          reinterpret_cast<float4*>(dst)[0] =
              make_float4((float)vals[r * 4 + 0], (float)vals[r * 4 + 1], (float)vals[r * 4 + 2], (float)vals[r * 4 + 3]);
        }
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (gj0 + c < N2) dst[c] = vals[r * 4 + c];
      }
    }
  }
}

template <typename T>
__global__ void kdiag_kernel(const __grid_constant__ KProg prog, const T* __restrict__ X, int64_t N, int64_t ldx,
                             T* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  T s0 = T(0), s1 = T(0), s2 = T(0), s3 = T(0);
  for (int o = 0; o < prog.n_ops; ++o) {
    const int op = prog.ops[o];
    if (op < KB_MAXL) {
      T v = T(prog.l_var[op]);  // stationaries.py:82-83, statics.py:41-42
      if (prog.l_type[op] == GPK_K_LINEAR || prog.l_type[op] == GPK_K_POLYNOMIAL) {  // linears.py:67-68, 111-112
        const int g = prog.l_group[op];
        T acc = T(0);
        for (int d = 0; d < prog.g_ndims[g]; ++d) {
          T x = X[i * ldx + prog.dims[prog.g_off[g] + d]];
          acc += T(prog.w[prog.g_off[g] + d]) * x * x;
        }
        v *= acc;
        if (prog.l_type[op] == GPK_K_POLYNOMIAL) v = KMath<T>::pow_(v + T(prog.l_scale[op]), T(prog.l_alpha[op]));
      }
      s3 = s2; s2 = s1; s1 = s0; s0 = v;
    } else {
      s0 = op == KB_OP_ADD ? s1 + s0 : s1 * s0;
      s1 = s2; s2 = s3;
    }
  }
  out[i] = s0;
}


// =============================================================================================
// Fast path: ONE stationary leaf (RBF / Matern12 / Matern32 / Matern52 / Exponential) — the common
// case and BASELINE config 2.  fp64 on B200 is compute-bound (exp(double) 835 Gop/s, sqrt 1164 Gop/s
// measured vs 18.3 T DFMA/s), so this path
//   * evaluates only lower-triangle tiles of a symmetric K and, for GPK_FULL, writes the mirrored
//     tile through a shared-memory transpose (compute once, store twice: HBM-bound);
//   * uses a table-driven exp (2^(j/64) table + degree-5 polynomial, ~12 DFMA instead of ~22) and a
//     MUFU-seeded Newton square root (~9 instead of ~16);
//   * launches a 1-D grid over the needed tiles only.
// =============================================================================================
__constant__ double c_exp2_tab[64];
static double h_exp2_tab[64];

// The fast path works on x = c * r2 (c folded into the per-dimension weights on the host together with the
// 1/lengthscale^2 scale): RBF c = 1/2 (k = v exp(-x)), Matern12 c = 1 (u = sqrt x, k = v exp(-u)),
// Exponential c = 1/4, Matern32 c = 3 (k = v (1 + u) exp(-u)), Matern52 c = 5 (k = v (1 + u + x/3) exp(-u)).
// The reference's clip of r2 at 1e-36 (stationaries.py:130-136) becomes a clip of x at c * 1e-36.
template <int TYPE> __host__ __device__ constexpr double kf_fold() {
  return TYPE == GPK_K_RBF ? 0.5 : TYPE == GPK_K_MATERN32 ? 3.0 : TYPE == GPK_K_MATERN52 ? 5.0
       : TYPE == GPK_K_EXPONENTIAL ? 0.25 : 1.0;
}
template <int TYPE> __host__ __device__ constexpr bool kf_const_pre() {  // prefactor is just the variance
  return TYPE == GPK_K_RBF || TYPE == GPK_K_MATERN12 || TYPE == GPK_K_EXPONENTIAL;
}

// fp32 value (generic float path): plain library math, the SFU exp is accurate enough for fp32
template <int TYPE>
__device__ __forceinline__ float stationary_value_f32(float x, float var) {
  if (TYPE == GPK_K_RBF) return var * __expf(-fmaxf(x, 0.0f));
  const float xc = fmaxf(x, (float)(kf_fold<TYPE>() * 1e-36));
  const float u = sqrtf(xc);
  if (TYPE == GPK_K_MATERN52) return fmaf(var * (1.0f / 3.0f), xc, fmaf(var, u, var)) * __expf(-u);
  if (TYPE == GPK_K_MATERN32) return fmaf(var, u, var) * __expf(-u);
  return var * __expf(-u);
}

__device__ __forceinline__ float rsqrt_approx(float x) {
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Four fp64 elements at a time, stage by stage: every arithmetic step is issued for the four independent
// elements back to back, so the dependent chains (sqrt: 6, exp: 11 fp64 ops) overlap instead of each
// waiting out the fp64 latency alone.  fp64-pipe budget per element (Matern52): 2 (x) + 6 (sqrt) + 2 (pre)
// + 11 (exp) = 21 besides the D-term dot product; clamps, range checks and the 2^n scaling are integer ops.
//   tab: 2^(j/64) in SHARED memory (lanes hit different entries), pre-multiplied by the variance when the
//   prefactor is constant.  var_ok: variance >= 2^-100, so adding n to the exponent field cannot underflow
//   while n >= -900 (the slow path handles the rest, including exp underflow to 0 below -708).
template <int TYPE>
__device__ __forceinline__ void stationary_value4(const double (&xin)[4], double var, double var3, bool var_ok,
                                                  const double* __restrict__ tab, double (&out)[4]) {
  double u[4], pre[4];
  if (TYPE == GPK_K_RBF) {
#pragma unroll
    for (int q = 0; q < 4; ++q) u[q] = __double2hiint(xin[q]) < 0 ? 0.0 : xin[q];  // max(x, 0) on the integer pipe
  } else {
    constexpr double clampv = kf_fold<TYPE>() * 1e-36;
    double x[4], g[4], h[4], r[4], d[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      // x < clamp (or negative) by a signed compare of the high words: equal high words differ by < 2^-20 relative
      const int hi_c = (int)((unsigned long long)__double_as_longlong(clampv) >> 32);
      x[q] = __double2hiint(xin[q]) < hi_c ? clampv : xin[q];
    }
    // y0 ~ x^-1/2 to 2^-22 (MUFU); g = x y0 ~ sqrt x, h = y0/2; one coupled Newton step on g (2^-43), then a
    // Heron correction with the unrefined h: relative error 1.5 e0^3 ~ 2^-64 before rounding
#pragma unroll
    for (int q = 0; q < 4; ++q) h[q] = (double)rsqrt_approx((float)x[q]);
#pragma unroll
    for (int q = 0; q < 4; ++q) g[q] = x[q] * h[q];
#pragma unroll
    for (int q = 0; q < 4; ++q) h[q] = 0.5 * h[q];
#pragma unroll
    for (int q = 0; q < 4; ++q) r[q] = fma(-g[q], h[q], 0.5);
#pragma unroll
    for (int q = 0; q < 4; ++q) g[q] = fma(g[q], r[q], g[q]);
#pragma unroll
    for (int q = 0; q < 4; ++q) d[q] = fma(-g[q], g[q], x[q]);
#pragma unroll
    for (int q = 0; q < 4; ++q) u[q] = fma(h[q], d[q], g[q]);
    if (TYPE == GPK_K_MATERN52) {
#pragma unroll
      for (int q = 0; q < 4; ++q) pre[q] = fma(var3, x[q], fma(var, u[q], var));
    } else if (TYPE == GPK_K_MATERN32) {
#pragma unroll
      for (int q = 0; q < 4; ++q) pre[q] = fma(var, u[q], var);
    }
  }
  // exp(-u), u >= 0
  double sh[4], kd[4], rr[4], p[4];
  int k[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) sh[q] = fma(u[q], -92.33248261689366, 6755399441055744.0);  // round(-u 64/ln2) in the low bits
#pragma unroll
  for (int q = 0; q < 4; ++q) { kd[q] = sh[q] - 6755399441055744.0; k[q] = __double2loint(sh[q]); }
#pragma unroll
  for (int q = 0; q < 4; ++q) rr[q] = fma(kd[q], -0.01083042468962958, -u[q]);   // ln2/64 hi (kd * hi exact)
#pragma unroll
  for (int q = 0; q < 4; ++q) rr[q] = fma(kd[q], -6.619564634077006e-12, rr[q]);  // ln2/64 lo
#pragma unroll
  for (int q = 0; q < 4; ++q) p[q] = fma(rr[q], 8.3333333333333332e-03, 4.1666666666666664e-02);
#pragma unroll
  for (int q = 0; q < 4; ++q) p[q] = fma(p[q], rr[q], 1.6666666666666666e-01);
#pragma unroll
  for (int q = 0; q < 4; ++q) p[q] = fma(p[q], rr[q], 0.5);
#pragma unroll
  for (int q = 0; q < 4; ++q) p[q] = fma(p[q], rr[q], 1.0);
#pragma unroll
  for (int q = 0; q < 4; ++q) p[q] = fma(p[q], rr[q], 1.0);
  double w[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const double t = tab[k[q] & 63];
    w[q] = (kf_const_pre<TYPE>() ? t : pre[q] * t) * p[q];
  }
  const int kmin = min(min(k[0], k[1]), min(k[2], k[3]));
  if (var_ok && kmin >= -57600) {  // 2^n by an integer add on the exponent field (n >= -900, w >= 2^-101)
#pragma unroll
    for (int q = 0; q < 4; ++q)
      out[q] = __hiloint2double(__double2hiint(w[q]) + ((k[q] >> 6) << 20), __double2loint(w[q]));
  } else {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int n = max(k[q] >> 6, -1022);
      const double two_n = __longlong_as_double((long long)(n + 1023) << 52);
      out[q] = u[q] > 708.0 ? 0.0 : w[q] * two_n;
    }
  }
}

#ifndef KF_VARIANT
#define KF_VARIANT 0  // experiment switches (scripts/kb_variants.sh): 1 no stores, 2 no dots, 4 no evaluation
#endif
constexpr int KF_KC = 8;             // dims staged per chunk (fast path)
constexpr int KF_LD = KB_TILE + 4;   // shared row stride of a staged dim: 16-byte aligned rows, 2-way store conflicts

// Persistent CTAs over the needed tiles (lower-triangle tiles of a symmetric K).  Per (tile, chunk of 8 dims)
// the operand rows are fetched into REGISTERS one step ahead (the global-load latency overlaps the previous
// step's arithmetic), scaled by the folded weights and staged transposed in shared memory.  Thread (tx,ty) of
// a 16x16 grid owns a 4x4 micro-tile made of 2x2 blocks 32 apart (rows {2ty, 2ty+1, 32+2ty, 33+2ty}, columns
// likewise with tx), warps are 8(tx) x 4(ty): every 16-byte store instruction of a warp then writes whole
// 32-byte sectors -- 128-byte row runs for the direct tile, 64-byte runs for the MIRRORED tile of GPK_FULL,
// which is written straight from registers (K[j][i] = K[i][j] is a copy, so K is bit-symmetric).
template <typename T, int TYPE, int MINB>
__global__ void __launch_bounds__(256, MINB)
kbuild_fast_kernel(const __grid_constant__ KProg prog, const T* __restrict__ X, int64_t N, int64_t ldx,
                   const T* __restrict__ X2, int64_t N2, int64_t ldx2, T* __restrict__ K, int64_t ldk, int mode,
                   T diag_scalar, const T* __restrict__ diag_vec, int vec_ok, int64_t ntiles) {
  // mode: 0 rectangular, 1 symmetric lower-only, 2 symmetric full (mirror)
  __shared__ __align__(16) T sA[2 * KF_KC * KF_LD];  // double-buffered staged operands [buf][dim][row]
  __shared__ __align__(16) T sB[2 * KF_KC * KF_LD];
  __shared__ T sNa[2 * KB_TILE], sNb[2 * KB_TILE];    // squared row norms of the staged rows
  __shared__ double s_tab[64];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = (lane & 7) + 8 * (warp & 1), ty = (lane >> 3) + 4 * (warp >> 1);
  auto rowi = [&](int r) { return ((r >> 1) << 5) + ty * 2 + (r & 1); };  // tile row of micro-tile row r
  auto coli = [&](int c) { return ((c >> 1) << 5) + tx * 2 + (c & 1); };  // tile column of micro-tile column c
  const T var = T(prog.l_var[0]);
  if (tid < 64) s_tab[tid] = kf_const_pre<TYPE>() ? c_exp2_tab[tid] * (double)var : c_exp2_tab[tid];
  // prog.w carries sqrt(c / lengthscale^2) (kf_fold), so the norm expansion yields x = c r2 directly
  const double var3 = (double)var * (1.0 / 3.0);
  const bool var_ok = (double)var >= 7.888609052210118e-31;  // 2^-100
  const bool sym = mode != 0;
  const T* Xb = sym ? X : X2;
  const int64_t ldb = sym ? ldx : ldx2;
  const int nd = prog.g_ndims[0];
  const int nchunks = (nd + KF_KC - 1) / KF_KC;
  const int64_t ntx = (N2 + KB_TILE - 1) / KB_TILE;

  auto decode = [&](int t, int& by, int& bx) {  // tile counts fit 31 bits (checked on the host)
    if (mode == 0) {
      by = t / (int)ntx;
      bx = t - by * (int)ntx;
    } else {  // lower-triangle tile enumeration: t = by (by + 1) / 2 + bx, bx <= by
      by = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);  // fp32 estimate, exact after the fix-up loops
      while ((long long)by * (by + 1) / 2 > t) --by;
      while ((long long)(by + 1) * (by + 2) / 2 <= t) ++by;
      bx = t - (int)((long long)by * (by + 1) / 2);
    }
  };
  // Staging: this thread fetches rows sr0 and sr0 + 32 of both operands, dim sd of a chunk, one step ahead into
  // registers, scales them and later writes them transposed into the step's shared buffer.  The squared row norms
  // are reduced across the 8 lanes that hold one row (xor butterfly: every lane gets the same bits, and a row
  // staged as the A side or as the B side sums in the same order, so K stays bit-symmetric).
  const int sd = tid & 7, sr0 = tid >> 3;
  T pa[2], pb[2];          // fetched (scaled) operands of the step after next
  T qa[2] = {T(0), T(0)}, qb[2] = {T(0), T(0)};  // running squared norms of the rows this thread stages
  auto fetch = [&](int by, int bx, int ch) {
    const int d = ch * KF_KC + sd;
    const bool dok = d < nd;
    const int col = dok ? prog.dims[d] : 0;
    const T wv = dok ? T(prog.w[d]) : T(0);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int64_t gr = (int64_t)by * KB_TILE + sr0 + 32 * i, gc = (int64_t)bx * KB_TILE + sr0 + 32 * i;
      pa[i] = (dok && gr < N) ? X[gr * ldx + col] * wv : T(0);
      pb[i] = (dok && gc < N2) ? Xb[gc * ldb + col] * wv : T(0);
    }
  };
  auto stage = [&](int buf, int ch) {  // registers -> shared buffer `buf` (+ norms up to and including chunk ch)
    T* dA = sA + buf * (KF_KC * KF_LD);
    T* dB = sB + buf * (KF_KC * KF_LD);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      dA[sd * KF_LD + sr0 + 32 * i] = pa[i];
      dB[sd * KF_LD + sr0 + 32 * i] = pb[i];
      T va = pa[i] * pa[i], vb = pb[i] * pb[i];
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        va += __shfl_xor_sync(0xffffffffu, va, o);
        vb += __shfl_xor_sync(0xffffffffu, vb, o);
      }
      qa[i] = ch == 0 ? va : qa[i] + va;
      qb[i] = ch == 0 ? vb : qb[i] + vb;
      if (sd == 0) {
        sNa[buf * KB_TILE + sr0 + 32 * i] = qa[i];
        sNb[buf * KB_TILE + sr0 + 32 * i] = qb[i];
      }
    }
  };

  // software pipeline over steps (tile, chunk): compute step s from buffer s&1 while step s+1 is written to the
  // other buffer and step s+2 is in flight from global memory; ONE barrier per step
  // (tile coordinates are decoded once per tile, when it enters the pipeline, and handed down)
  const int nt = (int)ntiles, G = (int)gridDim.x;
  int t = blockIdx.x, ch = 0, by = 0, bx = 0;  // step s
  int t1 = t, ch1 = 0, by1 = 0, bx1 = 0;       // step s+1
  auto advance = [&](int& tt, int& cc, int& yy, int& xx) {
    if (cc + 1 < nchunks) { ++cc; return; }
    cc = 0;
    tt += G;
    if (tt < nt) decode(tt, yy, xx);
  };
  if (t < nt) { decode(t, by, bx); fetch(by, bx, 0); stage(0, 0); }
  by1 = by; bx1 = bx;
  advance(t1, ch1, by1, bx1);
  if (t1 < nt) fetch(by1, bx1, ch1);
  __syncthreads();
  int buf = 0;
  T dots[4][4];
  while (t < nt) {
    if (t1 < nt) stage(buf ^ 1, ch1);
    int t2 = t1, ch2 = ch1, by2 = by1, bx2 = bx1;
    if (t1 < nt) {
      advance(t2, ch2, by2, bx2);
      if (t2 < nt) fetch(by2, bx2, ch2);
    }
    if (ch == 0) {
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) dots[r][c] = T(0);
    }
    {
      const T* cA = sA + buf * (KF_KC * KF_LD);
      const T* cB = sB + buf * (KF_KC * KF_LD);
#pragma unroll
      for (int d = 0; d < ((KF_VARIANT & 2) ? 1 : KF_KC); ++d) {
        T a[4], b[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) a[r] = cA[d * KF_LD + rowi(r)];
#pragma unroll
        for (int c = 0; c < 4; ++c) b[c] = cB[d * KF_LD + coli(c)];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) dots[r][c] = fma(a[r], b[c], dots[r][c]);
      }
    }
#define KF_NEXT_STEP() do { buf ^= 1; t = t1; ch = ch1; by = by1; bx = bx1; t1 = t2; ch1 = ch2; by1 = by2; bx1 = bx2; } while (0)
    if (ch + 1 < nchunks) {  // more dims of this tile to come
      __syncthreads();
      KF_NEXT_STEP();
      continue;
    }
    const int64_t row0 = (int64_t)by * KB_TILE, col0 = (int64_t)bx * KB_TILE;

    T vals[16];
    T na[4], nb[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) { na[r] = sNa[buf * KB_TILE + rowi(r)]; nb[r] = sNb[buf * KB_TILE + coli(r)]; }
    // the sum of norms is formed FIRST so that (i,j) and (j,i) round identically inside a diagonal tile
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if (sizeof(T) == 8) {
        double r2[4], o[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) r2[c] = fma(-2.0, (double)dots[r][c], (double)na[r] + (double)nb[c]);
        if (KF_VARIANT & 4) {
#pragma unroll
          for (int c = 0; c < 4; ++c) o[c] = r2[c];
        } else {
          stationary_value4<TYPE>(r2, (double)var, var3, var_ok, s_tab, o);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) vals[r * 4 + c] = (T)o[c];
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const T sn = na[r] + nb[c];
          vals[r * 4 + c] = (T)stationary_value_f32<TYPE>((float)fma(T(-2), dots[r][c], sn), (float)var);
        }
      }
    }
    if (sym && bx == by && tx == ty) {  // diagonal shift: only diagonal micro-tiles carry diagonal elements
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int64_t gi = row0 + rowi(r);
        vals[r * 4 + r] += diag_scalar + ((diag_vec && gi < N) ? diag_vec[gi] : T(0));
      }
    }
    if (KF_VARIANT & 1) {  // keep the values alive without the store traffic
      T acc = T(0);
#pragma unroll
      for (int e = 0; e < 16; ++e) acc += vals[e];
      if (acc == T(-12345.678)) K[tid] = acc;
      __syncthreads();
      KF_NEXT_STEP();
      continue;
    }
    const bool interior = vec_ok && row0 + KB_TILE <= N && col0 + KB_TILE <= N2;  // uniform: no per-element checks
    if (interior) {
      using V2 = typename std::conditional<sizeof(T) == 8, double2, float2>::type;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        T* dst = K + (row0 + rowi(r)) * ldk + col0 + tx * 2;
        V2 v0, v1;
        v0.x = vals[r * 4 + 0]; v0.y = vals[r * 4 + 1];
        v1.x = vals[r * 4 + 2]; v1.y = vals[r * 4 + 3];
        *reinterpret_cast<V2*>(dst) = v0;
        *reinterpret_cast<V2*>(dst + 32) = v1;
      }
      if (mode == 2 && bx < by) {  // mirrored tile K[col0 + j][row0 + i] = tile[i][j]
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          T* dt = K + (col0 + coli(c)) * ldk + row0 + ty * 2;
          V2 v0, v1;
          v0.x = vals[0 * 4 + c]; v0.y = vals[1 * 4 + c];
          v1.x = vals[2 * 4 + c]; v1.y = vals[3 * 4 + c];
          *reinterpret_cast<V2*>(dt) = v0;
          *reinterpret_cast<V2*>(dt + 32) = v1;
        }
      }
    } else {  // ragged edge tiles / unaligned K: element-wise guarded stores
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int64_t gi = row0 + rowi(r);
        if (gi < N) {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (col0 + coli(c) < N2) K[gi * ldk + col0 + coli(c)] = vals[r * 4 + c];
        }
      }
      if (mode == 2 && bx < by) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int64_t gi = col0 + coli(c);
          if (gi < N2) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
              if (row0 + rowi(r) < N) K[gi * ldk + row0 + rowi(r)] = vals[r * 4 + c];
          }
        }
      }
    }
    __syncthreads();  // every reader of buffer `buf` is done; the other buffer is completely written
    KF_NEXT_STEP();
  }
#undef KF_NEXT_STEP
}

static bool fast_path_ok(const KProg& p) {
  if (p.n_leaves != 1 || p.n_ops != 1 || p.n_groups != 1) return false;
  const int t = p.l_type[0];
  return t == GPK_K_RBF || t == GPK_K_MATERN12 || t == GPK_K_MATERN32 || t == GPK_K_MATERN52 || t == GPK_K_EXPONENTIAL;
}

template <typename T, int TYPE, int MINB>
static int kbuild_fast_go(const KProg& p, const void* X, int64_t N, int64_t ldx, const void* X2, int64_t N2, int64_t ldx2,
                          void* K, int64_t ldk, int mode, double diag_scalar, const void* diag_vec, int vec_ok,
                          cudaStream_t st) {
  const int64_t nty = (N + KB_TILE - 1) / KB_TILE, ntx = (N2 + KB_TILE - 1) / KB_TILE;
  const int64_t ntiles = mode == 0 ? nty * ntx : nty * (nty + 1) / 2;
  static int grid_max = 0;  // persistent grid: resident CTAs per SM x SM count (the same on every B200 of a box)
  static PerDeviceOnce once;
  GPK_TRY(once.run([&]() -> int {
    int dev = 0, sms = 0, per_sm = 0;
    GPK_CUDA_OK(cudaGetDevice(&dev));
    GPK_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GPK_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kbuild_fast_kernel<T, TYPE, MINB>, 256, 0));
    grid_max = sms * (per_sm > 0 ? per_sm : 1);
    return 0;
  }));
  const int64_t grid = ntiles < grid_max ? ntiles : grid_max;
  kbuild_fast_kernel<T, TYPE, MINB><<<(unsigned)grid, 256, 0, st>>>(p, (const T*)X, N, ldx, (const T*)X2, N2, ldx2, (T*)K, ldk,
                                                               mode, (T)diag_scalar, (const T*)diag_vec, vec_ok, ntiles);
  GPK_LAUNCH_OK();
  return 0;
}

template <typename T>
static int kbuild_fast_launch(const KProg& p, const void* X, int64_t N, int64_t ldx, const void* X2, int64_t N2,
                              int64_t ldx2, void* K, int64_t ldk, int lower, double diag_scalar, const void* diag_vec,
                              cudaStream_t st) {
  static PerDeviceOnce tab_once;  // __constant__ symbols live per device
  GPK_TRY(tab_once.run([&]() -> int {
    for (int j = 0; j < 64; ++j) h_exp2_tab[j] = exp2((double)j / 64.0);
    GPK_CUDA_OK(cudaMemcpyToSymbol(c_exp2_tab, h_exp2_tab, sizeof(h_exp2_tab)));
    return 0;
  }));
  ProfScope ps(PROF_KBUILD, st);
  const int vec_ok = ((uintptr_t)K % 16 == 0) && ((ldk * sizeof(T)) % 16 == 0);
  const int mode = p.symmetric ? (lower ? 1 : 2) : 0;
  // resident CTAs per SM the kernel is compiled for: 2 (<= 128 registers) for fp64, 3 (<= 80) for fp32
  constexpr int minb = sizeof(T) == 8 ? 2 : 3;
  // fold c / lengthscale^2 into the per-dimension weights (applied to both operands): x = c r2 comes out of
  // the norm expansion with no further scaling
#define GPK_KF(TY)                                                                                         \
  do {                                                                                                     \
    KProg q = p;                                                                                           \
    const double f = sqrt(q.l_scale[0] * kf_fold<TY>());                                                   \
    for (int d = 0; d < q.g_ndims[0]; ++d) q.w[d] *= f;                                                    \
    q.l_scale[0] = 1.0;                                                                                    \
    return kbuild_fast_go<T, TY, minb>(q, X, N, ldx, X2, N2, ldx2, K, ldk, mode, diag_scalar, diag_vec, vec_ok, st); \
  } while (0)
  switch (p.l_type[0]) {
    case GPK_K_RBF: GPK_KF(GPK_K_RBF);
    case GPK_K_MATERN12: GPK_KF(GPK_K_MATERN12);
    case GPK_K_MATERN32: GPK_KF(GPK_K_MATERN32);
    case GPK_K_MATERN52: GPK_KF(GPK_K_MATERN52);
    default: GPK_KF(GPK_K_EXPONENTIAL);
  }
#undef GPK_KF
}

template <typename T>
static int kbuild_launch(const KProg& p, const void* X, int64_t N, int64_t ldx, const void* X2, int64_t N2,
                         int64_t ldx2, void* K, int64_t ldk, int lower, double diag_scalar, const void* diag_vec,
                         cudaStream_t st) {
  ProfScope ps(PROF_KBUILD, st);
  dim3 grid((unsigned)((N2 + KB_TILE - 1) / KB_TILE), (unsigned)((N + KB_TILE - 1) / KB_TILE));
  const int vec_ok = ((uintptr_t)K % 16 == 0) && ((ldk * sizeof(T)) % 16 == 0);
#define GPK_KB_GO(NG)                                                                                            \
  kbuild_kernel<T, NG><<<grid, 256, 0, st>>>(p, (const T*)X, N, ldx, (const T*)X2, N2, ldx2, (T*)K, ldk, lower,   \
                                              (T)diag_scalar, (const T*)diag_vec, vec_ok)
  switch (p.n_groups) {
    case 0:
    case 1: GPK_KB_GO(1); break;
    case 2: GPK_KB_GO(2); break;
    case 3: GPK_KB_GO(3); break;
    default: GPK_KB_GO(4); break;
  }
#undef GPK_KB_GO
  GPK_LAUNCH_OK();
  return 0;
}

int kbuild_impl(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X,
                int64_t N, int64_t ldx, const void* X2, int64_t N2, int64_t ldx2, int64_t D, void* K, int64_t ldk,
                int dtype, int uplo, double diag_scalar, const void* diag_vec, cudaStream_t st) {
  GPK_CHECK_ARG(dtype == GPK_F32 || dtype == GPK_F64, "kbuild: bad dtype %d", dtype);
  GPK_CHECK_ARG(X && K, "kbuild: null X or K");
  const bool sym = X2 == nullptr;
  if (sym) { N2 = N; ldx2 = ldx; }
  GPK_CHECK_ARG(N >= 0 && N2 >= 0 && ldx >= D && ldx2 >= D && ldk >= N2, "kbuild: bad shape/stride");
  GPK_CHECK_ARG(sym || (uplo == GPK_FULL && diag_scalar == 0.0 && diag_vec == nullptr),
                "kbuild: uplo=LOWER / diagonal shift need the symmetric form (X2 == NULL)");
  if (N == 0 || N2 == 0) return 0;
  KProg p;
  GPK_TRY(compile_kprog(nodes, n_nodes, dims, ard, D, p));
  p.symmetric = sym ? 1 : 0;
  if (fast_path_ok(p)) {
    if (dtype == GPK_F64)
      return kbuild_fast_launch<double>(p, X, N, ldx, X2, N2, ldx2, K, ldk, uplo == GPK_LOWER, diag_scalar, diag_vec, st);
    return kbuild_fast_launch<float>(p, X, N, ldx, X2, N2, ldx2, K, ldk, uplo == GPK_LOWER, diag_scalar, diag_vec, st);
  }
  if (dtype == GPK_F64)
    return kbuild_launch<double>(p, X, N, ldx, X2, N2, ldx2, K, ldk, uplo == GPK_LOWER, diag_scalar, diag_vec, st);
  return kbuild_launch<float>(p, X, N, ldx, X2, N2, ldx2, K, ldk, uplo == GPK_LOWER, diag_scalar, diag_vec, st);
}

int kdiag_impl(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X,
               int64_t N, int64_t ldx, int64_t D, void* out, int dtype, cudaStream_t st) {
  GPK_CHECK_ARG(dtype == GPK_F32 || dtype == GPK_F64, "kdiag: bad dtype %d", dtype);
  GPK_CHECK_ARG(X && out && ldx >= D, "kdiag: bad arguments");
  if (N == 0) return 0;
  KProg p;
  GPK_TRY(compile_kprog(nodes, n_nodes, dims, ard, D, p));
  const unsigned blocks = (unsigned)((N + 255) / 256);
  if (dtype == GPK_F64)
    kdiag_kernel<double><<<blocks, 256, 0, st>>>(p, (const double*)X, N, ldx, (double*)out);
  else
    kdiag_kernel<float><<<blocks, 256, 0, st>>>(p, (const float*)X, N, ldx, (float*)out);
  GPK_LAUNCH_OK();
  return 0;
}

}  // namespace gpk
