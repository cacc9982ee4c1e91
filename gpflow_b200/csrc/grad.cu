// grad.cu — device backward passes of GPR.log_marginal_likelihood (SURVEY.md 8(f) rank 1) and, further down, of the
// SGPR ELBO (DESIGN.md section 4.9).
//
// The reference gets d(LML)/d(theta) from TensorFlow autodiff through gpflow/models/gpr.py:91-107 (driven by
// gpflow/optimizers/scipy.py:78-228 via training_loss_closure, models/training_mixins.py:43-78).  Here the adjoint is
// written out:
//     dLML/dK = G = 1/2 (alpha alpha^T - P K^-1),   alpha = K^-1 (Y - m),   K = kernel(X) + sigma_n^2 I
//     dLML/dtheta = sum_ij G_ij dK_ij/dtheta ,      dLML/dsigma_n^2 = tr G
// with K^-1 = L^-T L^-1 from the factor the forward pass leaves behind:
//   1. alpha  = L^-T beta            (beta^T = the extra rows of the factorisation; one trsm)
//   2. L^-1   in place (recursive block inversion [A 0; C D]^-1 = [A^-1 0; -D^-1 C A^-1, D^-1]; the 128x128 diagonal
//             blocks are the block inverses potrf already produced; two triangular x dense GEMMs per level)
//   3. K^-1   = L^-T L^-1, lower triangle (recursive: C11 = lauum(A11) + A21^T A21, C21 = A22^T A21, C22 = lauum(A22))
//   4. one K-build-shaped pass over the lower-triangle tiles that re-evaluates k and dk/ds per element (s = scaled
//      squared distance, by direct differences), forms G_ij on the fly from alpha and K^-1, and reduces
//      sum G (.) dK/dtheta per parameter: registers -> warp shuffles -> one atomicAdd per CTA and parameter.
// Steps 2-3 run on the DMMA GEMM with the triangular operand's zero k-range skipped (GPK_GEMM_A_LOWER): 2 N^3 / 3 flops.
// Covered kernels: a single stationary leaf (SquaredExponential, Matern12/32/52, Exponential) with a scalar or ARD
// lengthscale; the Python layer raises NotImplementedError for anything else.
#include "internal.cuh"

namespace gpk {

constexpr int GR_MAXD = 32;
struct GradKern {
  int type;            // GPK_K_RBF / MATERN12 / MATERN32 / MATERN52 / EXPONENTIAL
  int nd;              // active dims
  int ard;             // 0: scalar lengthscale (one gradient slot), 1: nd slots
  double variance;
  int dims[GR_MAXD];
  double inv_l[GR_MAXD];  // 1 / lengthscale_d
};

__device__ __forceinline__ void k_and_dkds(int type, double s, double var, double& k, double& dkds) {
  // s = scaled squared distance; k(s) and dk/ds as gpflow/kernels/stationaries.py:209-210,250-251,270-271,290-292,311-313
  // (the 1e-36 clip before the square root passes no gradient when active, like tf.maximum)
  if (type == GPK_K_RBF) {
    k = var * exp(-0.5 * s);
    dkds = -0.5 * k;
    return;
  }
  const bool clipped = !(s > 1e-36);
  const double r = sqrt(clipped ? 1e-36 : s);
  if (type == GPK_K_MATERN12) {
    k = var * exp(-r);
    dkds = clipped ? 0.0 : -k / (2.0 * r);
  } else if (type == GPK_K_EXPONENTIAL) {
    k = var * exp(-0.5 * r);
    dkds = clipped ? 0.0 : -k / (4.0 * r);
  } else if (type == GPK_K_MATERN32) {
    const double s3 = 1.7320508075688772935, e = exp(-s3 * r);
    k = var * (1.0 + s3 * r) * e;
    dkds = clipped ? 0.0 : -1.5 * var * e;
  } else {  // MATERN52
    const double s5 = 2.2360679774997896964, e = exp(-s5 * r);
    k = var * (1.0 + s5 * r + (5.0 / 3.0) * r * r) * e;
    dkds = clipped ? 0.0 : -(5.0 / 6.0) * var * (1.0 + s5 * r) * e;
  }
}

constexpr int GT = 64;  // tile edge

// gout: [0] d/dvariance, [1] d/dnoise_variance, [2 ...] d/dlengthscale (1 slot, or nd slots with ARD)
template <int ND>
__global__ void __launch_bounds__(256)
gpr_grad_kernel(GradKern gk, const double* __restrict__ X, int64_t N, int64_t ldx, const double* __restrict__ alpha,
                int P, const double* __restrict__ Kinv, int64_t ldk, double* __restrict__ gout) {
  __shared__ double xa[GT][ND + 1], xb[GT][ND + 1];
  __shared__ double red[8][ND + 2];
  // lower-triangular tile index -> (ti, tj), tj <= ti
  const int64_t t = blockIdx.x;
  int64_t ti = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (ti * (ti + 1) / 2 > t) --ti;
  while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
  const int64_t tj = t - ti * (ti + 1) / 2;
  const int tid = threadIdx.x, tr = tid >> 4, tc = tid & 15;
  const int nd = gk.nd;
  for (int e = tid; e < GT * ND; e += 256) {
    const int r = e / ND, d = e % ND;
    const int64_t ra = ti * GT + r, rb = tj * GT + r;
    const double sc = d < nd ? gk.inv_l[d] : 0.0;
    const int col = d < nd ? gk.dims[d] : 0;
    xa[r][d] = (ra < N && d < nd) ? X[ra * ldx + col] * sc : 0.0;
    xb[r][d] = (rb < N && d < nd) ? X[rb * ldx + col] * sc : 0.0;
  }
  __syncthreads();
  double gv = 0.0, gn = 0.0, gl[ND];
#pragma unroll
  for (int d = 0; d < ND; ++d) gl[d] = 0.0;
  double gls = 0.0;
#pragma unroll 1
  for (int a = 0; a < 4; ++a) {
    const int r = tr + 16 * a;
    const int64_t i = ti * GT + r;
#pragma unroll 1
    for (int b = 0; b < 4; ++b) {
      const int c = tc + 16 * b;
      const int64_t j = tj * GT + c;
      if (i >= N || j > i) continue;
      double s = 0.0;
#pragma unroll
      for (int d = 0; d < ND; ++d) {
        const double df = xa[r][d] - xb[c][d];
        s = fma(df, df, s);
      }
      double k, dkds;
      k_and_dkds(gk.type, s, gk.variance, k, dkds);
      double aa = 0.0;
      for (int p = 0; p < P; ++p) aa = fma(alpha[i * P + p], alpha[j * P + p], aa);
      const double G = 0.5 * (aa - (double)P * Kinv[i * ldk + j]);
      const double Ge = i == j ? G : 2.0 * G;  // the strict lower part stands for both (i,j) and (j,i)
      gv = fma(Ge, k, gv);
      if (i == j) gn += G;
      const double w = Ge * dkds * -2.0;
      if (gk.ard) {
#pragma unroll
        for (int d = 0; d < ND; ++d) {
          const double df = xa[r][d] - xb[c][d];
          gl[d] = fma(w, df * df, gl[d]);   // ds/dl_d = -2 diff_d^2 / l_d^3; the 1/l_d factor is applied at the end
        }
      } else {
        gls = fma(w, s, gls);               // ds/dl = -2 s / l
      }
    }
  }
  // CTA reduction: shuffles, then one atomicAdd per parameter
  const int lane = tid & 31, wp = tid >> 5;
  gv = warp_sum(gv);
  gn = warp_sum(gn);
  gls = warp_sum(gls);
#pragma unroll
  for (int d = 0; d < ND; ++d) gl[d] = warp_sum(gl[d]);
  if (lane == 0) {
    red[wp][0] = gv;
    red[wp][1] = gn;
#pragma unroll
    for (int d = 0; d < ND; ++d) red[wp][2 + d] = gk.ard ? gl[d] : (d == 0 ? gls : 0.0);
  }
  __syncthreads();
  if (tid < ND + 2) {
    double v = 0.0;
    for (int w2 = 0; w2 < 8; ++w2) v += red[w2][tid];
    if (tid == 0) atomicAdd(gout + 0, v / gk.variance);
    else if (tid == 1) atomicAdd(gout + 1, v);
    else {
      const int d = tid - 2;
      if (gk.ard) { if (d < nd) atomicAdd(gout + 2 + d, v * gk.inv_l[d]); }
      else if (d == 0) atomicAdd(gout + 2, v * gk.inv_l[0]);
    }
  }
}

// ---- L^-1 in place (lower), diagonal 128-blocks taken from the block inverses of the factorisation ------------
__global__ void put_dinv_kernel(double* __restrict__ L, int64_t ldl, int64_t n, const double* __restrict__ dinv) {
  const int64_t b0 = (int64_t)blockIdx.x * NB;
  const double* src = dinv + (size_t)blockIdx.x * NB * NB;
  for (int e = threadIdx.x; e < NB * NB; e += blockDim.x) {
    const int r = e / NB, c = e % NB;
    // the strict upper part of the block is zeroed: lauum reads the block as a dense operand, and the workspace above
    // the diagonal tiles of the K-build is uninitialised (0 x NaN)
    if (b0 + r < n && b0 + c < n) L[(b0 + r) * ldl + b0 + c] = c <= r ? src[r * NB + c] : 0.0;
  }
}

static inline int64_t split128(int64_t n) { return ((n / NB + 1) / 2) * NB; }

static int trtri_rec(double* L, int64_t n, int64_t ldl, double* tmp, cudaStream_t st) {
  if (n <= NB) return 0;  // diagonal blocks are already inverses
  const int64_t n1 = split128(n), n2 = n - n1;
  GPK_TRY(trtri_rec(L, n1, ldl, tmp, st));
  GPK_TRY(trtri_rec(L + n1 * ldl + n1, n2, ldl, tmp, st));
  double* L21 = L + n1 * ldl;
  double* A22 = L + n1 * ldl + n1;
  // Tt [n1, n2] = L11inv^T L21^T   (= (L21 L11inv)^T), the zero k-range of the triangular operand skipped
  GPK_TRY(gemm_t<double>(1, 1, n1, n2, n1, 1.0, L, ldl, L21, ldl, 0.0, tmp, n2, GPK_GEMM_A_LOWER, st));
  // L21 <- - L22inv (Tt)^T
  GPK_TRY(gemm_t<double>(0, 1, n2, n1, n2, -1.0, A22, ldl, tmp, n2, 0.0, L21, ldl, GPK_GEMM_A_LOWER, st));
  return 0;
}

// C (lower) = A^T A for lower-triangular A, out of place
static int lauum_rec(const double* A, int64_t n, int64_t lda, double* C, int64_t ldc, cudaStream_t st) {
  if (n <= NB)
    return gemm_t<double>(1, 0, n, n, n, 1.0, A, lda, A, lda, 0.0, C, ldc, GPK_GEMM_A_LOWER | GPK_GEMM_LOWER_ONLY, st);
  const int64_t n1 = split128(n), n2 = n - n1;
  const double* A21 = A + n1 * lda;
  const double* A22 = A + n1 * lda + n1;
  GPK_TRY(lauum_rec(A, n1, lda, C, ldc, st));
  GPK_TRY(lauum_rec(A22, n2, lda, C + n1 * ldc + n1, ldc, st));
  GPK_TRY(gemm_t<double>(1, 0, n1, n1, n2, 1.0, A21, lda, A21, lda, 1.0, C, ldc, GPK_GEMM_LOWER_ONLY, st));
  GPK_TRY(gemm_t<double>(1, 0, n2, n1, n2, 1.0, A22, lda, A21, lda, 0.0, C + n1 * ldc, ldc, GPK_GEMM_A_LOWER, st));
  return 0;
}

// K^-1 (lower triangle) from the factor L and its block inverses; L is overwritten by L^-1.
// tmp: (n/2 + 128)^2 doubles.
int potri_lower(double* L, int64_t n, int64_t ldl, const double* dinv, double* Kinv, int64_t ldk, double* tmp,
                cudaStream_t st) {
  const unsigned nblk = (unsigned)((n + NB - 1) / NB);
  put_dinv_kernel<<<nblk, 256, 0, st>>>(L, ldl, n, dinv);
  GPK_LAUNCH_OK();
  GPK_TRY(trtri_rec(L, n, ldl, tmp, st));
  return lauum_rec(L, n, ldl, Kinv, ldk, st);
}

// The kernel record of the backward passes: a single stationary leaf, its active dims and inverse lengthscales.
static int grad_kern(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, int64_t D,
                     const char* who, GradKern& gk) {
  GPK_CHECK_ARG(n_nodes == 1, "%s: the device backward covers a single stationary leaf kernel", who);
  const gpk_knode& nd = nodes[0];
  GPK_CHECK_ARG(nd.op == GPK_K_RBF || nd.op == GPK_K_MATERN12 || nd.op == GPK_K_MATERN32 || nd.op == GPK_K_MATERN52 ||
                    nd.op == GPK_K_EXPONENTIAL,
                "%s: kernel op %d has no device backward", who, nd.op);
  memset(&gk, 0, sizeof(gk));
  gk.type = nd.op;
  gk.variance = nd.variance;
  gk.nd = nd.n_dims > 0 ? nd.n_dims : (int)D;
  GPK_CHECK_ARG(gk.nd <= GR_MAXD, "%s: more than %d active dims", who, GR_MAXD);
  gk.ard = nd.n_ard > 0 ? 1 : 0;
  for (int d = 0; d < gk.nd; ++d) {
    gk.dims[d] = nd.n_dims > 0 ? dims[nd.dims_off + d] : d;
    gk.inv_l[d] = 1.0 / (nd.n_ard > 0 ? ard[nd.ard_off + d] : nd.lengthscale);
  }
  return 0;
}

int gpr_grad_launch(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const double* X,
                    int64_t N, int64_t ldx, int64_t D, const double* alpha, int P, const double* Kinv, int64_t ldk,
                    double* gout, cudaStream_t st) {
  GradKern gk;
  GPK_TRY(grad_kern(nodes, n_nodes, dims, ard, D, "gpr_lml_grad", gk));
  const int64_t nt = (N + GT - 1) / GT;
  const unsigned grid = (unsigned)(nt * (nt + 1) / 2);
  ProfScope ps(PROF_KBUILD, st);
  if (gk.nd <= 8) gpr_grad_kernel<8><<<grid, 256, 0, st>>>(gk, X, N, ldx, alpha, P, Kinv, ldk, gout);
  else if (gk.nd <= 16) gpr_grad_kernel<16><<<grid, 256, 0, st>>>(gk, X, N, ldx, alpha, P, Kinv, ldk, gout);
  else gpr_grad_kernel<32><<<grid, 256, 0, st>>>(gk, X, N, ldx, alpha, P, Kinv, ldk, gout);
  GPK_LAUNCH_OK();
  return 0;
}

// =====================================================================================================================
// SGPR ELBO backward (gpflow/models/sgpr.py:181-289; DESIGN.md section 4.9).  With E = Y - m(X), A' = L^-1 Kuf,
// B = A'A'^T / s2 + I = LB LB^T, c = LB^-1 A'E / s2, w~ = LB^-T c, v = L^-T w~:
//   dELBO/dKuf   = (L^-T C A' + v E^T) / s2,           C = P (I - B^-1) - w~ w~^T
//   dELBO/dKuu   = L^-T (P I - P/2 (B + B^-1) - 1/2 w~ w~^T) L^-1
//   dELBO/dKdiag = -P / (2 s2)
//   dELBO/ds2    = (1/s2) [-NP/2 + sum E^2/(2 s2) + P/2 (trace_k - trace_q) + P/2 (M - tr B^-1) - |c|^2/2 - |w~|^2/2]
// The M x M stage runs in fp64 for both dtypes; dKuf = G1 A' / s2 (G1 = L^-T C) is one M x M x N GEMM in the model
// dtype, and the rank-P term v E^T / s2 is added inside the reduction, which re-evaluates k and dk/ds from Z and X and
// sums dK (.) dK/dtheta into d/dvariance, d/dlengthscale and dZ.
// =====================================================================================================================

// dst [m, n] (ldd) = src (lds), converted; tril: entries above the diagonal are written as 0
template <typename TS, typename TD>
__global__ void convert_kernel(const TS* __restrict__ src, int64_t lds, TD* __restrict__ dst, int64_t ldd, int64_t m,
                               int64_t n, int tril) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < m * n; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / n, j = e % n;
    dst[i * ldd + j] = (tril && j > i) ? (TD)0 : (TD)src[i * lds + j];
  }
}

template <typename TS, typename TD>
static int convert(const TS* src, int64_t lds, TD* dst, int64_t ldd, int64_t m, int64_t n, int tril, cudaStream_t st) {
  const int64_t tot = m * n;
  const unsigned g = (unsigned)(tot < 148 * 64 * 256 ? (tot + 255) / 256 : 148 * 64);
  convert_kernel<TS, TD><<<g > 0 ? g : 1, 256, 0, st>>>(src, lds, dst, ldd, m, n, tril);
  GPK_LAUNCH_OK();
  return 0;
}

// C = P (I - Bi) - w~ w~^T and H = P I - P/2 (B + Bi) - 1/2 w~ w~^T, full [M, M]
__global__ void sgpr_inner_kernel(const double* __restrict__ B, const double* __restrict__ Bi, int64_t ld,
                                  const double* __restrict__ wt, int P, int64_t M, double* __restrict__ C,
                                  double* __restrict__ H) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < M * M; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / M, j = e % M;
    double ww = 0.0;
    for (int p = 0; p < P; ++p) ww = fma(wt[i * P + p], wt[j * P + p], ww);
    const double dg = i == j ? (double)P : 0.0, b = B[i * ld + j], bi = Bi[i * ld + j];
    C[i * ld + j] = dg - P * bi - ww;
    H[i * ld + j] = dg - 0.5 * P * (b + bi) - 0.5 * ww;
  }
}

// sc: [0] tr B^-1, [1] |w~|^2; scal: the forward's 0 trace_k, 1 trace_q, 3 sum E^2 / s2, 4 |c|^2
__global__ void sgpr_grad_finalize_kernel(double* out, const double* scal, const double* sc, double N, double P,
                                          double M, double noise) {
  const double inv = 1.0 / noise;
  out[8] -= 0.5 * P * N * inv;  // Kdiag = variance at every point (stationary)
  out[9] = inv * (-0.5 * N * P + 0.5 * scal[3] + 0.5 * P * (scal[0] - scal[1]) + 0.5 * P * (M - sc[0]) -
                  0.5 * scal[4] - 0.5 * sc[1]);
}

// 4 consecutive entries of a row from column j (zero past n); one 16-byte load where the row allows it
template <typename T>
__device__ __forceinline__ void load4(const T* row, int64_t j, int64_t n, double (&v)[4]) {
  if (j + 3 < n) {
    if (sizeof(T) == 4) {
      const float4 q = *reinterpret_cast<const float4*>(row + j);
      v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
      const double2 a = *reinterpret_cast<const double2*>(row + j), b = *reinterpret_cast<const double2*>(row + j + 2);
      v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = j + e < n ? (double)row[j + e] : 0.0;
  }
}

// One CTA: 64 rows of dK (inducing points z_m) x a strip of `tiles` 64-column tiles (points x_n).  Thread (row r, group
// g) owns columns q*16 + g*4 + e of every tile and keeps its row's dZ and lengthscale sums in registers across the whole
// strip: one shuffle reduction and one atomicAdd per (row, dim) per CTA.
//   dK_mn = dK[m, n] + inv_s2 sum_p v[m, p] E[n, p]   (P = 0: no rank-P term)
//   gout[0] += sum dK k / variance, gout[2 + d] += sum dK k' ds/dl_d, dZ[m, dims[d]] += zfac sum_n dK k' ds/dz_md
// The Kuu pass runs over the full symmetric dKuu with x = z and zfac = 2 (k(z_i, z_j) depends on z_m through i = m and
// j = m alike).
constexpr int SG_TILE = 64;
template <typename TK, typename TX, int ND, bool ARD>
__global__ void __launch_bounds__(256)
sgpr_grad_reduce_kernel(GradKern gk, const TX* __restrict__ Z, int64_t M, int64_t ldz, const TX* __restrict__ X,
                        int64_t N, int64_t ldx, const TK* __restrict__ dK, int64_t ldk, const double* __restrict__ v,
                        const TX* __restrict__ E, int P, double inv_s2, int tiles, double zfac, double* __restrict__ gout,
                        double* __restrict__ dZ, int64_t lddz) {
  __shared__ double zs[SG_TILE][ND + 1], xs[SG_TILE][ND + 1];
  __shared__ double red[8][ND + 2];
  const int tid = threadIdx.x, r = tid >> 2, g = tid & 3;
  const int nd = gk.nd;
  const int64_t m0 = (int64_t)blockIdx.x * SG_TILE, m = m0 + r;
  const bool row_ok = m < M;
  for (int e = tid; e < SG_TILE * ND; e += 256) {
    const int rr = e / ND, d = e % ND;
    zs[rr][d] = (m0 + rr < M && d < nd) ? (double)Z[(m0 + rr) * ldz + gk.dims[d]] * gk.inv_l[d] : 0.0;
  }
  double gv = 0.0, gls = 0.0, dz[ND], gl[ARD ? ND : 1];
#pragma unroll
  for (int d = 0; d < ND; ++d) dz[d] = 0.0;
#pragma unroll
  for (int d = 0; d < (ARD ? ND : 1); ++d) gl[d] = 0.0;
  const TK* dkrow = dK + (row_ok ? m : 0) * ldk;
  const int64_t t0 = (int64_t)blockIdx.y * tiles;
#pragma unroll 1
  for (int t = 0; t < tiles; ++t) {
    const int64_t n0 = (t0 + t) * SG_TILE;
    if (n0 >= N) break;
    __syncthreads();
    for (int e = tid; e < SG_TILE * ND; e += 256) {
      const int c = e / ND, d = e % ND;
      xs[c][d] = (n0 + c < N && d < nd) ? (double)X[(n0 + c) * ldx + gk.dims[d]] * gk.inv_l[d] : 0.0;
    }
    __syncthreads();
    if (!row_ok) continue;
#pragma unroll 1
    for (int q = 0; q < 4; ++q) {
      const int cb = q * 16 + g * 4;
      double dk4[4];
      load4(dkrow, n0 + cb, N, dk4);
#pragma unroll
      for (int e = 0; e < 4; ++e) {  // unrolled: dk4 stays in registers
        const int c = cb + e;
        const int64_t n = n0 + c;
        if (n >= N) continue;
        double dk = dk4[e];
        if (P > 0) {
          double ve = 0.0;
#pragma unroll 1
          for (int p = 0; p < P; ++p) ve = fma(v[m * P + p], (double)E[n * P + p], ve);
          dk = fma(inv_s2, ve, dk);
        }
        double s = 0.0;
#pragma unroll
        for (int d = 0; d < ND; ++d) {
          const double df = zs[r][d] - xs[c][d];
          s = fma(df, df, s);
        }
        double k, dkds;
        k_and_dkds(gk.type, s, gk.variance, k, dkds);
        gv = fma(dk, k, gv);
        const double w = dk * dkds;
        if (ARD) {
#pragma unroll
          for (int d = 0; d < ND; ++d) {
            const double df = zs[r][d] - xs[c][d];
            dz[d] = fma(w, df, dz[d]);
            gl[d] = fma(w * df, df, gl[d]);
          }
        } else {
#pragma unroll
          for (int d = 0; d < ND; ++d) dz[d] = fma(w, zs[r][d] - xs[c][d], dz[d]);
          gls = fma(w, s, gls);
        }
      }
    }
  }
  // dZ: the four threads of a row are adjacent lanes; ds/dz_md = 2 (z_md - x_nd) / l_d^2 = 2 df_d / l_d
#pragma unroll
  for (int d = 0; d < ND; ++d) {
    dz[d] += __shfl_xor_sync(0xffffffffu, dz[d], 1);
    dz[d] += __shfl_xor_sync(0xffffffffu, dz[d], 2);
  }
  if (row_ok && g == 0) {
#pragma unroll
    for (int d = 0; d < ND; ++d)
      if (d < nd) atomicAdd(dZ + m * lddz + gk.dims[d], zfac * 2.0 * dz[d] * gk.inv_l[d]);
  }
  // variance / lengthscale sums: shuffles, then one atomicAdd per parameter and CTA; ds/dl_d = -2 df_d^2 / l_d
  const int lane = tid & 31, wp = tid >> 5;
  gv = warp_sum(gv);
  if (ARD) {
#pragma unroll
    for (int d = 0; d < ND; ++d) gl[d] = warp_sum(gl[d]);
  } else {
    gls = warp_sum(gls);
  }
  if (lane == 0) {
    red[wp][0] = gv;
#pragma unroll
    for (int d = 0; d < ND; ++d) red[wp][2 + d] = ARD ? gl[ARD ? d : 0] : (d == 0 ? gls : 0.0);
  }
  __syncthreads();
  if (tid < ND + 2 && tid != 1) {
    double a = 0.0;
    for (int w2 = 0; w2 < 8; ++w2) a += red[w2][tid];
    if (tid == 0) atomicAdd(gout + 0, a / gk.variance);
    else {
      const int d = tid - 2;
      if (ARD) { if (d < nd) atomicAdd(gout + 2 + d, -2.0 * a * gk.inv_l[d]); }
      else if (d == 0) atomicAdd(gout + 2, -2.0 * a * gk.inv_l[0]);
    }
  }
}

template <typename TK, typename TX>
static int sgpr_reduce_launch(const GradKern& gk, const TX* Z, int64_t M, int64_t ldz, const TX* X, int64_t N,
                              int64_t ldx, const TK* dK, int64_t ldk, const double* v, const TX* E, int P, double inv_s2,
                              double zfac, double* gout, double* dZ, int64_t lddz, cudaStream_t st) {
  // strips of up to 16 column tiles per CTA, fewer while that leaves the grid short of ~8 CTAs per SM
  const int64_t mt = (M + SG_TILE - 1) / SG_TILE, nt = (N + SG_TILE - 1) / SG_TILE;
  int64_t tiles = (mt * nt) / (148 * 8);
  tiles = tiles < 1 ? 1 : (tiles > 16 ? 16 : tiles);
  const dim3 grid((unsigned)mt, (unsigned)((nt + tiles - 1) / tiles));
  GPK_CHECK_ARG(grid.y <= 65535, "sgpr_elbo_grad: too many column strips");
  ProfScope ps(PROF_KBUILD, st);
#define GO(ND_, ARD_)                                                                                              \
  sgpr_grad_reduce_kernel<TK, TX, ND_, ARD_><<<grid, 256, 0, st>>>(gk, Z, M, ldz, X, N, ldx, dK, ldk, v, E, P,     \
                                                                    inv_s2, (int)tiles, zfac, gout, dZ, lddz)
  if (gk.nd <= 8) { if (gk.ard) GO(8, true); else GO(8, false); }
  else if (gk.nd <= 16) { if (gk.ard) GO(16, true); else GO(16, false); }
  else { if (gk.ard) GO(32, true); else GO(32, false); }
#undef GO
  GPK_LAUNCH_OK();
  return 0;
}

int sgpr_grad_check(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, int64_t D) {
  GradKern gk;
  return grad_kern(nodes, n_nodes, dims, ard, D, "sgpr_elbo_grad", gk);
}

// inputs: the forward's L and LB (lower, model dtype, ld ldm), A' [M, ldn], c [M, P], scalars; out[0..7] written by the
// forward; writes out[8 ..] and dZ
int sgpr_grad_backward(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X,
                       int64_t N, int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M,
                       int64_t ldz, double noise, int dtype, const void* L, const void* LB, int64_t ldm, const void* Ap,
                       int64_t ldn, const void* c, const double* scal, const SgprBwdWs& b, double* out, int n_out,
                       double* dZ, int64_t lddz, cudaStream_t st) {
  GradKern gk;
  GPK_TRY(grad_kern(nodes, n_nodes, dims, ard, D, "sgpr_elbo_grad", gk));
  const double inv_s2 = 1.0 / noise;
  const bool f32 = dtype == GPK_F32;
  // fp64 copies of the two factors (upper parts zero) and of c
  if (f32) {
    GPK_TRY(convert((const float*)L, ldm, b.Li, ldm, M, M, 1, st));
    GPK_TRY(convert((const float*)LB, ldm, b.LBi, ldm, M, M, 1, st));
    GPK_TRY(convert((const float*)c, P, b.cw, P, M, P, 0, st));
  } else {
    GPK_TRY(convert((const double*)L, ldm, b.Li, ldm, M, M, 1, st));
    GPK_TRY(convert((const double*)LB, ldm, b.LBi, ldm, M, M, 1, st));
    GPK_TRY(convert((const double*)c, P, b.cw, P, M, P, 0, st));
  }
  // B = LB LB^T (full), then both factors inverted in place (128-block inverses + recursive blocking)
  GPK_TRY(gemm_t<double>(0, 1, M, M, M, 1.0, b.LBi, ldm, b.LBi, ldm, 0.0, b.B, ldm, GPK_GEMM_A_LOWER, st));
  const unsigned nblk = (unsigned)((M + NB - 1) / NB);
  GPK_TRY(trtri_diag_t<double>(b.Li, M, ldm, b.dinvL, st));
  put_dinv_kernel<<<nblk, 256, 0, st>>>(b.Li, ldm, M, b.dinvL);
  GPK_LAUNCH_OK();
  GPK_TRY(trtri_rec(b.Li, M, ldm, b.tmp, st));
  GPK_TRY(trtri_diag_t<double>(b.LBi, M, ldm, b.dinvB, st));
  put_dinv_kernel<<<nblk, 256, 0, st>>>(b.LBi, ldm, M, b.dinvB);
  GPK_LAUNCH_OK();
  GPK_TRY(trtri_rec(b.LBi, M, ldm, b.tmp, st));
  // B^-1 = LB^-T LB^-1 (full); w~ = LB^-T c; v = L^-T w~
  GPK_TRY(gemm_t<double>(1, 0, M, M, M, 1.0, b.LBi, ldm, b.LBi, ldm, 0.0, b.Bi, ldm, GPK_GEMM_A_LOWER, st));
  GPK_TRY(gemm_t<double>(1, 0, M, P, M, 1.0, b.LBi, ldm, b.cw, P, 0.0, b.wt, P, 0, st));
  GPK_TRY(gemm_t<double>(1, 0, M, P, M, 1.0, b.Li, ldm, b.wt, P, 0.0, b.v, P, 0, st));
  GPK_TRY(reduce_impl(0, b.Bi, M, ldm + 1, 1.0, 0, b.sc + 0, GPK_F64, st));
  GPK_TRY(reduce_impl(1, b.wt, M * P, 1, 1.0, 0, b.sc + 1, GPK_F64, st));
  {
    const int64_t tot = M * M;
    const unsigned g = (unsigned)(tot < 148 * 32 * 256 ? (tot + 255) / 256 : 148 * 32);
    sgpr_inner_kernel<<<g, 256, 0, st>>>(b.B, b.Bi, ldm, b.wt, (int)P, M, b.C, b.H);
    GPK_LAUNCH_OK();
  }
  // G1 = L^-T C ; dKuu = L^-T H L^-1 = L^-T (L^-T H)^T
  GPK_TRY(gemm_t<double>(1, 0, M, M, M, 1.0, b.Li, ldm, b.C, ldm, 0.0, b.G1, ldm, GPK_GEMM_A_LOWER, st));
  GPK_TRY(gemm_t<double>(1, 0, M, M, M, 1.0, b.Li, ldm, b.H, ldm, 0.0, b.T, ldm, GPK_GEMM_A_LOWER, st));
  GPK_TRY(gemm_t<double>(1, 1, M, M, M, 1.0, b.Li, ldm, b.T, ldm, 0.0, b.dKuu, ldm, GPK_GEMM_A_LOWER, st));
  // dKuf (without the rank-P term) = G1 A' / s2 in the model dtype: the one large contraction
  if (f32) {
    GPK_TRY(convert(b.G1, ldm, (float*)b.G1n, ldm, M, M, 0, st));
    GPK_TRY(gemm_t<float>(0, 0, M, N, M, (float)inv_s2, (const float*)b.G1n, ldm, (const float*)Ap, ldn, 0.0f,
                          (float*)b.dKuf, ldn, 0, st));
  } else {
    GPK_TRY(gemm_t<double>(0, 0, M, N, M, inv_s2, b.G1, ldm, (const double*)Ap, ldn, 0.0, (double*)b.dKuf, ldn, 0, st));
  }
  GPK_CUDA_OK(cudaMemsetAsync(out + 8, 0, (size_t)(n_out - 8) * sizeof(double), st));
  GPK_CUDA_OK(cudaMemsetAsync(dZ, 0, (size_t)M * lddz * sizeof(double), st));
  double* gout = out + 8;
  if (f32) {
    GPK_TRY((sgpr_reduce_launch<float, float>(gk, (const float*)Z, M, ldz, (const float*)X, N, ldx,
                                             (const float*)b.dKuf, ldn, b.v, (const float*)Yc, (int)P, inv_s2, 1.0,
                                             gout, dZ, lddz, st)));
    GPK_TRY((sgpr_reduce_launch<double, float>(gk, (const float*)Z, M, ldz, (const float*)Z, M, ldz, b.dKuu, ldm,
                                              nullptr, nullptr, 0, 0.0, 2.0, gout, dZ, lddz, st)));
  } else {
    GPK_TRY((sgpr_reduce_launch<double, double>(gk, (const double*)Z, M, ldz, (const double*)X, N, ldx,
                                               (const double*)b.dKuf, ldn, b.v, (const double*)Yc, (int)P, inv_s2, 1.0,
                                               gout, dZ, lddz, st)));
    GPK_TRY((sgpr_reduce_launch<double, double>(gk, (const double*)Z, M, ldz, (const double*)Z, M, ldz, b.dKuu, ldm,
                                               nullptr, nullptr, 0, 0.0, 2.0, gout, dZ, lddz, st)));
  }
  sgpr_grad_finalize_kernel<<<1, 1, 0, st>>>(out, scal, b.sc, (double)N, (double)P, (double)M, noise);
  GPK_LAUNCH_OK();
  return 0;
}

}  // namespace gpk
