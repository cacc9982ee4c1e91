// fused.cu — one-call objectives: GPR log marginal likelihood, SGPR ELBO, SVGP ELBO.
// Each function enqueues the whole evaluation on the caller's stream from a caller-provided
// workspace (no allocation, no host synchronisation) and leaves the scalars in device memory.
//   gpr_lml   : gpflow/models/gpr.py:91-107 + logdensities.py:139-156
//   sgpr_elbo : gpflow/models/sgpr.py:181-289 (+ the cache of posteriors.py:520-551)
//   svgp_elbo : gpflow/models/svgp.py:166-181 -> posteriors.py:827-841 -> conditionals/util.py:84-169
//               -> kullback_leiblers.py:59-165 -> likelihoods/scalar_continuous.py:139-148
#include <stdlib.h>

#include "internal.cuh"

namespace gpk {

static const double LOG2PI = 1.8378770664093454835606594728112;

struct Arena {
  char* base;
  size_t off;
  explicit Arena(void* p) : base((char*)p), off(0) {}
  void* take(size_t bytes) {
    void* r = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return r;
  }
};

static inline int64_t pad_ld(int64_t n) { return (n + 3) / 4 * 4; }

// ---------------------------------------------------------------------------------------------
// GPR
// ---------------------------------------------------------------------------------------------
// Upper bound of max_i K_ii for the expression tree when every leaf has a constant diagonal (stationary, White,
// Constant: the variance); <= 0 when a leaf's diagonal depends on x (Linear, Polynomial): unknown.
static double diag_bound(const gpk_knode* nodes, int idx) {
  const gpk_knode& nd = nodes[idx];
  if (nd.op == GPK_K_SUM || nd.op == GPK_K_PRODUCT) {
    double acc = nd.op == GPK_K_SUM ? 0.0 : 1.0;
    for (int c = 0; c < nd.n_children; ++c) {
      const double v = diag_bound(nodes, nd.child[c]);
      if (!(v > 0.0)) return 0.0;
      acc = nd.op == GPK_K_SUM ? acc + v : acc * v;
    }
    return acc;
  }
  if (nd.op == GPK_K_LINEAR || nd.op == GPK_K_POLYNOMIAL) return 0.0;
  return nd.variance;
}
static double gpr_cond_hint(const gpk_knode* nodes, int n_nodes, double noise_variance) {
  const double d = diag_bound(nodes, n_nodes - 1);
  return (d > 0.0 && noise_variance > 0.0) ? (d + noise_variance) / noise_variance : 0.0;
}

struct GprWs {
  void* A; int64_t lda; void* dinv; int32_t* info; size_t bytes;
};
static GprWs gpr_layout(void* ws, int64_t N, int64_t P, int dtype) {
  Arena a(ws);
  GprWs w;
  w.lda = pad_ld(N);
  w.A = a.take((size_t)(N + P) * w.lda * dtype_size(dtype));
  w.dinv = a.take(potrf_ws_bytes(N, N + P, dtype));
  w.info = (int32_t*)a.take(256);
  w.bytes = a.off;
  return w;
}

__global__ void gpr_finalize_kernel(double* out, const int32_t* info, double N, double P) {
  // logdensities.py:152-154 summed over the P columns (gpr.py:107)
  out[0] = -0.5 * out[1] - 0.5 * N * P * LOG2PI - P * out[2];
  out[3] = (double)info[0];
}

size_t gpr_lml_ws(int64_t N, int64_t P, int dtype) { return gpr_layout(nullptr, N, P, dtype).bytes; }

int gpr_lml(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
            int64_t ldx, int64_t D, const void* Yc, int64_t P, double noise_variance, const void* noise_vec,
            int dtype, double* out, void* ws, cudaStream_t st) {
  GPK_CHECK_ARG(N > 0 && P > 0 && ws && out && Yc, "gpr_lml: bad arguments");
  GprWs w = gpr_layout(ws, N, P, dtype);
  const size_t ts = dtype_size(dtype);
  // K(X,X) lower triangle + sigma^2 on the diagonal, no jitter (gpr.py:100-101, model_utils.py:33-50)
  GPK_TRY(kbuild_impl(nodes, n_nodes, dims, ard, X, N, ldx, nullptr, N, ldx, D, w.A, w.lda, dtype, GPK_LOWER,
                      noise_variance, noise_vec, st));
  // (Y - m)^T as P extra rows: the factorisation's panel solves turn them into alpha^T (logdensities.py:150)
  char* Yrows = (char*)w.A + (size_t)N * w.lda * ts;
  GPK_TRY(transpose_impl(Yc, N, P, P, Yrows, w.lda, dtype, st));
  // alpha comes out of the factorisation itself (extra rows): no trsm on this factor, block inverses not needed
  GPK_TRY(potrf_any(w.A, N, N + P, w.lda, dtype, w.info, w.dinv, st, /*need_dinv=*/false,
                    noise_vec ? 0.0 : gpr_cond_hint(nodes, n_nodes, noise_variance)));  // gpr.py:102
  GPK_CUDA_OK(cudaMemsetAsync(out, 0, 4 * sizeof(double), st));
  for (int64_t p = 0; p < P; ++p)
    GPK_TRY(reduce_impl(1, Yrows + (size_t)p * w.lda * ts, N, 1, 1.0, 1, out + 1, dtype, st));
  GPK_TRY(reduce_impl(2, w.A, N, w.lda + 1, 1.0, 1, out + 2, dtype, st));
  gpr_finalize_kernel<<<1, 1, 0, st>>>(out, w.info, (double)N, (double)P);
  GPK_LAUNCH_OK();
  return 0;
}

// ---- value + gradient (grad.cu) -----------------------------------------------------------------
int potri_lower(double* L, int64_t n, int64_t ldl, const double* dinv, double* Kinv, int64_t ldk, double* tmp,
                cudaStream_t st);
int gpr_grad_launch(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const double* X,
                    int64_t N, int64_t ldx, int64_t D, const double* alpha, int P, const double* Kinv, int64_t ldk,
                    double* gout, cudaStream_t st);

struct GprGradWs {
  GprWs f; void* Kinv; void* tmp; void* alpha; size_t bytes;
};
static GprGradWs gpr_grad_layout(void* ws, int64_t N, int64_t P, int dtype) {
  GprGradWs w;
  w.f = gpr_layout(ws, N, P, dtype);
  Arena a(ws);
  a.off = w.f.bytes;
  const size_t ts = dtype_size(dtype);
  const int64_t h = N / 2 + NB;
  w.Kinv = a.take((size_t)N * w.f.lda * ts);
  w.tmp = a.take((size_t)h * h * ts);
  w.alpha = a.take((size_t)N * P * ts);
  w.bytes = a.off;
  return w;
}

size_t gpr_lml_grad_ws(int64_t N, int64_t P, int dtype) { return gpr_grad_layout(nullptr, N, P, dtype).bytes; }

// out: [0..3] as gpr_lml; [4] d/dvariance, [5] d/dnoise_variance, [6 ...] d/dlengthscale (1 or n_ard entries)
int gpr_lml_grad(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
                 int64_t ldx, int64_t D, const void* Yc, int64_t P, double noise_variance, int dtype, double* out,
                 int n_out, void* ws, cudaStream_t st) {
  GPK_CHECK_ARG(dtype == GPK_F64, "gpr_lml_grad: the device backward computes in float64");
  GPK_CHECK_ARG(N > 0 && P > 0 && ws && out && Yc && n_out >= 7, "gpr_lml_grad: bad arguments");
  GprGradWs w = gpr_grad_layout(ws, N, P, dtype);
  const size_t ts = dtype_size(dtype);
  // forward pass (gpr.py:91-107) keeping the block inverses of the factor
  GPK_TRY(kbuild_impl(nodes, n_nodes, dims, ard, X, N, ldx, nullptr, N, ldx, D, w.f.A, w.f.lda, dtype, GPK_LOWER,
                      noise_variance, nullptr, st));
  char* Yrows = (char*)w.f.A + (size_t)N * w.f.lda * ts;
  GPK_TRY(transpose_impl(Yc, N, P, P, Yrows, w.f.lda, dtype, st));
  GPK_TRY(potrf_any(w.f.A, N, N + P, w.f.lda, dtype, w.f.info, w.f.dinv, st, /*need_dinv=*/true,
                    gpr_cond_hint(nodes, n_nodes, noise_variance)));
  GPK_CUDA_OK(cudaMemsetAsync(out, 0, (size_t)n_out * sizeof(double), st));
  for (int64_t p = 0; p < P; ++p)
    GPK_TRY(reduce_impl(1, Yrows + (size_t)p * w.f.lda * ts, N, 1, 1.0, 1, out + 1, dtype, st));
  GPK_TRY(reduce_impl(2, w.f.A, N, w.f.lda + 1, 1.0, 1, out + 2, dtype, st));
  gpr_finalize_kernel<<<1, 1, 0, st>>>(out, w.f.info, (double)N, (double)P);
  GPK_LAUNCH_OK();
  // alpha = L^-T beta  (beta^T = the extra rows)
  GPK_TRY(transpose_impl(Yrows, P, N, w.f.lda, w.alpha, P, dtype, st));
  GPK_TRY(trsm_any(1, w.f.A, N, w.f.lda, w.alpha, P, P, dtype, w.f.dinv, st));
  // K^-1 (lower) = L^-T L^-1; the factor is overwritten by its inverse
  GPK_TRY(potri_lower((double*)w.f.A, N, w.f.lda, (const double*)w.f.dinv, (double*)w.Kinv, w.f.lda, (double*)w.tmp, st));
  // sum G (.) dK/dtheta, G = 1/2 (alpha alpha^T - P K^-1)
  return gpr_grad_launch(nodes, n_nodes, dims, ard, (const double*)X, N, ldx, D, (const double*)w.alpha, (int)P,
                         (const double*)w.Kinv, w.f.lda, out + 4, st);
}

// ---------------------------------------------------------------------------------------------
// SGPR
// ---------------------------------------------------------------------------------------------
struct SgprWs {
  void *Kuu, *Kuf, *Bm, *dinvL, *dinvB, *kdiag, *c; int64_t ldm, ldn; int32_t* info; double* scal; size_t bytes;
};
static SgprWs sgpr_layout(void* ws, int64_t N, int64_t M, int64_t P, int dtype) {
  Arena a(ws);
  SgprWs w;
  const size_t ts = dtype_size(dtype);
  w.ldm = pad_ld(M);
  w.ldn = pad_ld(N);
  w.Kuu = a.take((size_t)M * w.ldm * ts);
  w.Kuf = a.take((size_t)M * w.ldn * ts);
  w.Bm = a.take((size_t)M * w.ldm * ts);
  w.dinvL = a.take(potrf_ws_bytes(M, M, dtype));
  w.dinvB = a.take(potrf_ws_bytes(M, M, dtype));
  w.kdiag = a.take((size_t)N * ts);
  w.c = a.take((size_t)M * P * ts);
  w.info = (int32_t*)a.take(256);
  w.scal = (double*)a.take(256);
  w.bytes = a.off;
  return w;
}

// scal: 0 trace_k, 1 trace_q, 2 half_logdet_b, 3 sum err^2, 4 sum c^2
__global__ void sgpr_finalize_kernel(double* out, const double* scal, const int32_t* info, double N, double P,
                                     double noise) {
  const double trace_k = scal[0], trace_q = scal[1], half_logdet_b = scal[2];
  const double log_sigma_sq = N * log(noise);
  const double logdet = -P * (half_logdet_b + 0.5 * log_sigma_sq + 0.5 * (trace_k - trace_q));  // sgpr.py:245
  const double quad = -0.5 * (scal[3] - scal[4]);                                              // sgpr.py:270
  const double cst = -0.5 * N * P * LOG2PI;                                                    // sgpr.py:286
  out[0] = cst + logdet + quad;
  out[1] = cst; out[2] = logdet; out[3] = quad; out[4] = trace_k; out[5] = trace_q; out[6] = half_logdet_b;
  out[7] = (double)(info[0] != 0 ? info[0] : info[1]);
}

size_t sgpr_elbo_ws(int64_t N, int64_t M, int64_t P, int dtype) { return sgpr_layout(nullptr, N, M, P, dtype).bytes; }

int sgpr_elbo(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
              int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M, int64_t ldz,
              double noise, double jitter, int dtype, double* out, void* cache_L, void* cache_LB, void* cache_c,
              void* ws, cudaStream_t st) {
  GPK_CHECK_ARG(N > 0 && M > 0 && P > 0 && ws && out, "sgpr_elbo: bad arguments");
  GPK_CHECK_ARG(noise > 0.0, "sgpr_elbo: noise variance must be positive");
  SgprWs w = sgpr_layout(ws, N, M, P, dtype);
  const size_t ts = dtype_size(dtype);
  const double inv_s2 = 1.0 / noise;
  GPK_CUDA_OK(cudaMemsetAsync(w.scal, 0, 8 * sizeof(double), st));
  GPK_CUDA_OK(cudaMemsetAsync(w.info, 0, 2 * sizeof(int32_t), st));
  // kuu = kernel(Z) + jitter I ; L = chol(kuu)   (sgpr.py:200-201)
  GPK_TRY(kbuild_impl(nodes, n_nodes, dims, ard, Z, M, ldz, nullptr, M, ldz, D, w.Kuu, w.ldm, dtype, GPK_LOWER, jitter,
                      nullptr, st));
  GPK_TRY(potrf_any(w.Kuu, M, M, w.ldm, dtype, w.info, w.dinvL, st));
  // kuf = kernel(Z, X) [M,N];  A' = L^-1 kuf  (the 1/sigma of sgpr.py:204 is folded into the scalars below)
  GPK_TRY(kbuild_impl(nodes, n_nodes, dims, ard, Z, M, ldz, X, N, ldx, D, w.Kuf, w.ldn, dtype, GPK_FULL, 0.0, nullptr,
                      st));
  GPK_TRY(trsm_any(0, w.Kuu, M, w.ldm, w.Kuf, N, w.ldn, dtype, w.dinvL, st));
  // AAT = A A^T = A'A'^T / sigma^2 (lower) ; trace_q = tr(AAT) ; B = AAT + I ; LB = chol(B)  (sgpr.py:205-207)
  GPK_TRY(gemm_any(0, 1, M, M, N, inv_s2, w.Kuf, w.ldn, w.Kuf, w.ldn, 0.0, w.Bm, w.ldm, dtype, GPK_GEMM_LOWER_ONLY, st));
  GPK_TRY(reduce_impl(0, w.Bm, M, w.ldm + 1, 1.0, 1, w.scal + 1, dtype, st));
  GPK_TRY(add_diag_impl(w.Bm, M, w.ldm, 1.0, nullptr, dtype, st));
  GPK_TRY(potrf_any(w.Bm, M, M, w.ldm, dtype, w.info + 1, w.dinvB, st));
  GPK_TRY(reduce_impl(2, w.Bm, M, w.ldm + 1, 1.0, 1, w.scal + 2, dtype, st));
  // trace_k = sum kdiag / sigma^2  (sgpr.py:231-233)
  GPK_TRY(kdiag_impl(nodes, n_nodes, dims, ard, X, N, ldx, D, w.kdiag, dtype, st));
  GPK_TRY(reduce_impl(0, w.kdiag, N, 1, inv_s2, 1, w.scal + 0, dtype, st));
  // quad: err = Yc/sigma ; Aerr = A err = A' Yc / sigma^2 ; c = LB^-1 Aerr  (sgpr.py:262-264)
  GPK_TRY(gemm_any(0, 0, M, P, N, inv_s2, w.Kuf, w.ldn, Yc, P, 0.0, w.c, P, dtype, 0, st));
  GPK_TRY(trsm_any(0, w.Bm, M, w.ldm, w.c, P, P, dtype, w.dinvB, st));
  GPK_TRY(reduce_impl(1, Yc, N * P, 1, inv_s2, 1, w.scal + 3, dtype, st));
  GPK_TRY(reduce_impl(1, w.c, M * P, 1, 1.0, 1, w.scal + 4, dtype, st));
  sgpr_finalize_kernel<<<1, 1, 0, st>>>(out, w.scal, w.info, (double)N, (double)P, noise);
  GPK_LAUNCH_OK();
  if (cache_L) {
    GPK_TRY(axpby_impl(M, M, 1.0, w.Kuu, w.ldm, 0.0, cache_L, M, dtype, st));
    GPK_TRY(tril_impl(cache_L, M, M, 0, 1, dtype, st));
  }
  if (cache_LB) {
    GPK_TRY(axpby_impl(M, M, 1.0, w.Bm, w.ldm, 0.0, cache_LB, M, dtype, st));
    GPK_TRY(tril_impl(cache_LB, M, M, 0, 1, dtype, st));
  }
  if (cache_c) GPK_CUDA_OK(cudaMemcpyAsync(cache_c, w.c, (size_t)M * P * ts, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// ---- value + gradient (grad.cu) -----------------------------------------------------------------
int sgpr_grad_check(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, int64_t D);
int sgpr_grad_backward(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X,
                       int64_t N, int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M,
                       int64_t ldz, double noise, int dtype, const void* L, const void* LB, int64_t ldm, const void* Ap,
                       int64_t ldn, const void* c, const double* scal, const SgprBwdWs& b, double* out, int n_out,
                       double* dZ, int64_t lddz, cudaStream_t st);

struct SgprGradWs {
  SgprWs f; SgprBwdWs b; size_t bytes;
};
static SgprGradWs sgpr_grad_layout(void* ws, int64_t N, int64_t M, int64_t P, int dtype) {
  SgprGradWs w;
  w.f = sgpr_layout(ws, N, M, P, dtype);
  Arena a(ws);
  a.off = w.f.bytes;
  const size_t ts = dtype_size(dtype), mm = (size_t)M * w.f.ldm * sizeof(double);
  const int64_t h = M / 2 + NB;
  SgprBwdWs& b = w.b;
  double** sq[] = {&b.Li, &b.LBi, &b.B, &b.Bi, &b.C, &b.H, &b.G1, &b.T, &b.dKuu};
  for (double** p : sq) *p = (double*)a.take(mm);
  b.dinvL = (double*)a.take(dinv_bytes(M, GPK_F64));
  b.dinvB = (double*)a.take(dinv_bytes(M, GPK_F64));
  b.tmp = (double*)a.take((size_t)h * h * sizeof(double));
  b.cw = (double*)a.take((size_t)M * P * sizeof(double));
  b.wt = (double*)a.take((size_t)M * P * sizeof(double));
  b.v = (double*)a.take((size_t)M * P * sizeof(double));
  b.sc = (double*)a.take(256);
  b.G1n = dtype == GPK_F32 ? a.take((size_t)M * w.f.ldm * ts) : nullptr;
  b.dKuf = a.take((size_t)M * w.f.ldn * ts);
  w.bytes = a.off;
  return w;
}

size_t sgpr_elbo_grad_ws(int64_t N, int64_t M, int64_t P, int dtype) {
  return sgpr_grad_layout(nullptr, N, M, P, dtype).bytes;
}

// out: [0..7] as sgpr_elbo; [8] d/dvariance, [9] d/dnoise_variance, [10 ...] d/dlengthscale (1 or n_ard entries);
// dZ [M, D] (lddz) fp64
int sgpr_elbo_grad(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
                   int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M, int64_t ldz,
                   double noise, double jitter, int dtype, double* out, int n_out, double* dZ, int64_t lddz, void* ws,
                   cudaStream_t st) {
  GPK_CHECK_ARG(N > 0 && M > 0 && P > 0 && D > 0 && ws && out && Yc && dZ && lddz >= D, "sgpr_elbo_grad: bad arguments");
  GPK_TRY(sgpr_grad_check(nodes, n_nodes, dims, ard, D));
  const int n_l = nodes[0].n_ard > 0 ? nodes[0].n_ard : 1;
  GPK_CHECK_ARG(n_out >= 10 + n_l, "sgpr_elbo_grad: n_out = %d < %d", n_out, 10 + n_l);
  SgprGradWs w = sgpr_grad_layout(ws, N, M, P, dtype);
  // forward pass (sgpr.py:181-289) into the head of the workspace: L, A' = L^-1 Kuf, LB, c and the scalars stay there
  GPK_TRY(sgpr_elbo(nodes, n_nodes, dims, ard, X, N, ldx, D, Yc, P, Z, M, ldz, noise, jitter, dtype, out, nullptr,
                    nullptr, nullptr, ws, st));
  return sgpr_grad_backward(nodes, n_nodes, dims, ard, X, N, ldx, D, Yc, P, Z, M, ldz, noise, dtype, w.f.Kuu, w.f.Bm,
                            w.f.ldm, w.f.Kuf, w.f.ldn, w.f.c, w.f.scal, w.b, out, n_out, dZ, lddz, st);
}

// ---------------------------------------------------------------------------------------------
// SVGP
// ---------------------------------------------------------------------------------------------
struct SvgpWs {
  void *Kuu, *A, *dinv, *v0, *fvar, *fmu, *tmpM, *tmpP, *kinv; int64_t ldm, ldb; int32_t* info; double* scal;
  size_t bytes;
};
static SvgpWs svgp_layout(void* ws, int64_t B, int64_t M, int64_t P, int dtype) {
  Arena a(ws);
  SvgpWs w;
  const size_t ts = dtype_size(dtype);
  w.ldm = pad_ld(M);
  w.ldb = pad_ld(B);
  w.Kuu = a.take((size_t)M * w.ldm * ts);
  w.A = a.take((size_t)M * w.ldb * ts);
  w.dinv = a.take(potrf_ws_bytes(M, M, dtype));
  w.v0 = a.take((size_t)B * ts);
  w.fvar = a.take((size_t)P * B * ts);   // [P][B]
  w.fmu = a.take((size_t)B * P * ts);    // [B][P]
  w.tmpM = a.take((size_t)M * w.ldm * ts);
  w.tmpP = a.take((size_t)M * P * ts);
  w.kinv = a.take((size_t)M * ts);
  w.info = (int32_t*)a.take(256);
  w.scal = (double*)a.take(256);
  w.bytes = a.off;
  return w;
}

// scal: 0 sum var_exp, 1 mahalanobis, 2 logdet_qcov, 3 trace, 4 sum log diag(Lp)^2
__global__ void svgp_finalize_kernel(double* out, const double* scal, const int32_t* info, double M, double Pl,
                                     double scale, int whiten) {
  double twoKL = scal[1] - M * Pl - scal[2] + scal[3];   // kullback_leiblers.py:124-155
  if (!whiten) twoKL += Pl * scal[4];                    // :158-163
  const double kl = 0.5 * twoKL;
  out[0] = scal[0] * scale - kl;                         // svgp.py:181
  out[1] = scal[0];
  out[2] = kl;
  out[3] = (double)info[0];
}

size_t svgp_elbo_ws(int64_t B, int64_t M, int64_t P, int dtype) { return svgp_layout(nullptr, B, M, P, dtype).bytes; }

// byte offset and leading dimension of A [M, ldb] inside the workspace (for the all-gather between stages 1 and 2)
size_t svgp_elbo_A(int64_t B, int64_t M, int64_t P, int dtype, int64_t* ld) {
  SvgpWs w = svgp_layout(nullptr, B, M, P, dtype);
  if (ld) *ld = w.ldb;
  return (size_t)((char*)w.A - (char*)nullptr);
}

int svgp_elbo(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* Xb, int64_t B,
              int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M, int64_t ldz,
              const void* q_mu, const void* q_sqrt, int q_diag, int whiten, double noise, double scale, double jitter,
              int p_begin, int p_end, int dtype, double* out, void* ws, cudaStream_t st, int stage, int64_t c0,
              int64_t c1) {
  // stage 0: the whole evaluation.  Latent sharding over GPUs with a column-sharded triangular solve (SURVEY 8(e)):
  //   stage 1: Kuu, chol, and ONLY the columns [c0, c1) of Kuf / A = Lm^-1 Kuf (written in place in the workspace's
  //            A [M, ldb]; gpk_svgp_elbo_A locates it) -- the caller then all-gathers the column blocks of A;
  //   stage 2: everything after the solve for the latents [p_begin, p_end), A taken complete from the workspace.
  GPK_CHECK_ARG(B > 0 && M > 0 && P > 0 && ws && out && q_mu && q_sqrt, "svgp_elbo: bad arguments");
  GPK_CHECK_ARG(stage >= 0 && stage <= 2, "svgp_elbo: bad stage %d", stage);
  GPK_CHECK_ARG(stage == 0 || whiten, "svgp_elbo: the staged (column-sharded) evaluation covers whiten=True");
  if (stage != 1) { c0 = 0; c1 = B; }
  GPK_CHECK_ARG(0 <= c0 && c0 <= c1 && c1 <= B, "svgp_elbo: bad column range [%lld,%lld) of %lld", (long long)c0,
                (long long)c1, (long long)B);
  GPK_CHECK_ARG(0 <= p_begin && p_begin < p_end && p_end <= P, "svgp_elbo: bad latent range [%d,%d) of %lld", p_begin,
                p_end, (long long)P);
  GPK_CHECK_ARG(noise > 0.0, "svgp_elbo: noise variance must be positive");
  SvgpWs w = svgp_layout(ws, B, M, P, dtype);
  const size_t ts = dtype_size(dtype);
  const int64_t Pl = p_end - p_begin;
  const char* qmu = (const char*)q_mu;
  const char* qs = (const char*)q_sqrt;
  GPK_CUDA_OK(cudaMemsetAsync(w.scal, 0, 8 * sizeof(double), st));
  if (stage != 2) {
    // Kmm = Kuu + jitter ; Lm = chol(Kmm)   (posteriors.py:835, util.py:67)
    GPK_TRY(kbuild_impl(nodes, n_nodes, dims, ard, Z, M, ldz, nullptr, M, ldz, D, w.Kuu, w.ldm, dtype, GPK_LOWER, jitter,
                        nullptr, st));
    GPK_TRY(potrf_any(w.Kuu, M, M, w.ldm, dtype, w.info, w.dinv, st));
    // Kmn = Kuf [M,B] ; A = Lm^-1 Kmn   (posteriors.py:836, util.py:125); columns [c0, c1) only in stage 1
    if (c1 > c0) {
      char* Ac = (char*)w.A + (size_t)c0 * ts;
      GPK_TRY(kbuild_impl(nodes, n_nodes, dims, ard, Z, M, ldz, (const char*)Xb + (size_t)c0 * ldx * ts, c1 - c0, ldx, D,
                          Ac, w.ldb, dtype, GPK_FULL, 0.0, nullptr, st));
      GPK_TRY(trsm_any(0, w.Kuu, M, w.ldm, Ac, c1 - c0, w.ldb, dtype, w.dinv, st));
    }
    if (stage == 1) return 0;
  } else {
    GPK_CUDA_OK(cudaMemsetAsync(w.info, 0, sizeof(int32_t), st));
  }
  // fvar0 = Knn - sum_m A^2   (util.py:133)
  GPK_TRY(kdiag_impl(nodes, n_nodes, dims, ard, Xb, B, ldx, D, w.v0, dtype, st));
  GPK_TRY(colsumsq_impl(w.A, M, B, w.ldb, -1.0, 1, w.v0, dtype, st));
  if (!whiten) GPK_TRY(trsm_any(1, w.Kuu, M, w.ldm, w.A, B, w.ldb, dtype, w.dinv, st));  // util.py:138-139
  // fmean = A^T q_mu[:, p_begin:p_end]   (util.py:144)
  GPK_TRY(gemm_any(1, 0, B, Pl, M, 1.0, w.A, w.ldb, qmu + (size_t)p_begin * ts, P, 0.0, w.fmu, Pl, dtype, 0, st));
  // fvar_p = fvar0 + sum_m (q_sqrt_p^T A)^2   (util.py:149-164) — LTA is never materialised
  // fp32, dense q_sqrt: ALL latents in one batched tcgen05 launch (A split into TF32 planes once, one persistent grid
  // over P x tiles instead of P launches with a 2-wave tail each)
  const bool batched = !q_diag && dtype == GPK_F32 && Pl > 1 && M % 256 == 0 &&
                       gemm_tf32_eligible(M, B, M, nullptr, nullptr, nullptr, 0);
  for (int64_t p = p_begin; p < p_end; ++p) {
    char* fv = (char*)w.fvar + (size_t)(p - p_begin) * B * ts;
    GPK_CUDA_OK(cudaMemcpyAsync(fv, w.v0, (size_t)B * ts, cudaMemcpyDeviceToDevice, st));
    if (batched) continue;
    if (q_diag) {
      GPK_TRY(colsumsq_impl(w.A, M, B, w.ldb, 1.0, 1, fv, dtype, st, qs + (size_t)p * ts, P));
    } else {
      GPK_TRY(gemm_any(1, 0, M, B, M, 1.0, qs + (size_t)p * M * M * ts, M, w.A, w.ldb, 0.0, fv, 0, dtype,
                       GPK_GEMM_A_LOWER | GPK_GEMM_COLSUMSQ, st));
    }
  }
  if (batched)
    GPK_TRY(gemm_tf32(1, 0, M, B, M, 1.0f, (const float*)(qs + (size_t)p_begin * M * M * ts), M, (const float*)w.A, w.ldb, 0.0f,
                      (float*)w.fvar, 0, GPK_GEMM_A_LOWER | GPK_GEMM_COLSUMSQ, st, (int)Pl, M * M, B));
  // sum of variational expectations (scalar_continuous.py:139-148); Yc column range [p_begin, p_end)
  GPK_TRY(varexp_impl(w.fmu, w.fvar, (const char*)Yc + (size_t)p_begin * ts, B, Pl, P, 1, B, noise, 1.0, 1,
                      w.scal + 0, dtype, st));
  // KL[q || p]   (kullback_leiblers.py:59-165)
  for (int64_t p = p_begin; p < p_end; ++p) {
    if (q_diag) {
      GPK_TRY(reduce_impl(3, qs + (size_t)p * ts, M, P, 1.0, 1, w.scal + 2, dtype, st));           // :130
    } else {
      GPK_TRY(reduce_impl(3, qs + (size_t)p * M * M * ts, M, M + 1, 1.0, 1, w.scal + 2, dtype, st));
    }
  }
  if (whiten) {
    for (int64_t p = p_begin; p < p_end; ++p)
      GPK_TRY(reduce_impl(1, qmu + (size_t)p * ts, M, P, 1.0, 1, w.scal + 1, dtype, st));           // :124
    if (q_diag) {
      for (int64_t p = p_begin; p < p_end; ++p)
        GPK_TRY(reduce_impl(1, qs + (size_t)p * ts, M, P, 1.0, 1, w.scal + 3, dtype, st));          // :134
    } else {
      GPK_TRY(tril_sumsq_impl(qs + (size_t)p_begin * M * M * ts, M, M, M * M, (int)Pl, 1.0, 1, w.scal + 3, dtype, st));
    }
  } else {
    // alpha = Lp^-1 q_mu  (:114)
    GPK_TRY(axpby_impl(M, Pl, 1.0, qmu + (size_t)p_begin * ts, P, 0.0, w.tmpP, Pl, dtype, st));
    GPK_TRY(trsm_any(0, w.Kuu, M, w.ldm, w.tmpP, Pl, Pl, dtype, w.dinv, st));
    GPK_TRY(reduce_impl(1, w.tmpP, M * Pl, 1, 1.0, 1, w.scal + 1, dtype, st));
    if (q_diag) {
      // K^-1 diagonal = column sums of squares of Lp^-1  (:136-145)
      GPK_TRY(fill_impl(w.tmpM, M, M, w.ldm, 0.0, dtype, st));
      GPK_TRY(add_diag_impl(w.tmpM, M, w.ldm, 1.0, nullptr, dtype, st));
      GPK_TRY(trsm_any(0, w.Kuu, M, w.ldm, w.tmpM, M, w.ldm, dtype, w.dinv, st));
      GPK_TRY(colsumsq_impl(w.tmpM, M, M, w.ldm, 1.0, 0, w.kinv, dtype, st));
      for (int64_t p = p_begin; p < p_end; ++p)
        GPK_TRY(reduce_wsq_impl(w.kinv, qs + (size_t)p * ts, M, P, 1.0, w.scal + 3, dtype, st));
    } else {
      for (int64_t p = p_begin; p < p_end; ++p) {  // trace = sum (Lp^-1 Lq)^2  (:152-153)
        GPK_TRY(axpby_impl(M, M, 1.0, qs + (size_t)p * M * M * ts, M, 0.0, w.tmpM, w.ldm, dtype, st));
        GPK_TRY(tril_impl(w.tmpM, M, w.ldm, 0, 1, dtype, st));
        GPK_TRY(trsm_any(0, w.Kuu, M, w.ldm, w.tmpM, M, w.ldm, dtype, w.dinv, st));
        GPK_TRY(colsumsq_impl(w.tmpM, M, M, w.ldm, 1.0, p == p_begin ? 0 : 1, w.kinv, dtype, st));
      }
      GPK_TRY(reduce_impl(0, w.kinv, M, 1, 1.0, 1, w.scal + 3, dtype, st));
    }
    GPK_TRY(reduce_impl(3, w.Kuu, M, w.ldm + 1, 1.0, 1, w.scal + 4, dtype, st));                   // :159-160
  }
  svgp_finalize_kernel<<<1, 1, 0, st>>>(out, w.scal, w.info, (double)M, (double)Pl, scale, whiten);
  GPK_LAUNCH_OK();
  return 0;
}

}  // namespace gpk
