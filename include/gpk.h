/*
 * gpk.h — C ABI of libgpk.so, the B200 (sm_100a) implementation of GPflow's GP-inference hot
 * path: covariance build -> Cholesky / triangular solves -> GPR LML, SGPR / SVGP ELBO, posterior.
 *
 * The reference (GPflow 2.9.2, /root/reference) has NO FFI boundary: it is pure Python on
 * TensorFlow ops.  Each entry point below therefore replaces a *TensorFlow-op call site* of the
 * reference; the site(s) are cited as `gpflow/...:line`.  The Python package `gpflow_b200`
 * mirrors the reference's Python plugin API (gpflow.kernels.Kernel, covariances.Kuu/Kuf,
 * conditionals, kullback_leiblers, posteriors, models.GPR/SGPR/SVGP) and reaches these symbols
 * through ctypes (gpflow_b200/_lib.py).  INTEGRATION.md shows the stub a GPflow maintainer adds.
 *
 * Conventions
 *  - All matrices are ROW-MAJOR (C order, like NumPy/TF); `ld*` = elements between rows.
 *  - All data pointers are DEVICE pointers (e.g. torch.Tensor.data_ptr()) unless named `host`.
 *    The caller owns all memory; workspaces come from the matching `*_ws` size query.  Two resources
 *    are library-owned, keyed by (device, stream), created on first use and never on the steady-state
 *    path: the side stream + 3 events of the Cholesky look-ahead, and the grow-only TF32 plane scratch
 *    of the fp32 tcgen05 GEMM (gpk_gemm has no workspace argument in the reference-shaped ABI).
 *    gpk_warm() creates / reserves them eagerly.
 *  - `dtype`: GPK_F32 or GPK_F64; every array of one call has that dtype (gpflow/base.py:299-311).
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it.
 *  - Return: 0 = OK; <0 = argument / launch error (text via gpk_last_error()); potrf reports a
 *    non-positive pivot through the device-side `info` word (LAPACK convention, 1-based column).
 */
#ifndef GPK_H_
#define GPK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPK_VERSION 1
#define GPK_API __attribute__((visibility("default")))

enum { GPK_F32 = 0, GPK_F64 = 1 };
enum { GPK_FULL = 0, GPK_LOWER = 1 };

/* Kernel-expression node ops.  Stationary ops follow gpflow/kernels/stationaries.py:209-313,
 * statics gpflow/kernels/statics.py:57-91, linear gpflow/kernels/linears.py:60-68,
 * combinations gpflow/kernels/base.py:305-314. */
enum {
  GPK_K_RBF = 0,      /* sigma^2 exp(-r2/2)                      stationaries.py:209-210 */
  GPK_K_MATERN12 = 1, /* sigma^2 exp(-r)                         stationaries.py:270-271 */
  GPK_K_MATERN32 = 2, /* sigma^2 (1+sqrt3 r) exp(-sqrt3 r)       stationaries.py:290-292 */
  GPK_K_MATERN52 = 3, /* sigma^2 (1+sqrt5 r+5/3 r^2) exp(-sqrt5 r) stationaries.py:311-313 */
  GPK_K_RQ = 4,       /* sigma^2 (1 + r2/(2 alpha))^-alpha       stationaries.py:237-238 */
  GPK_K_EXPONENTIAL = 5, /* sigma^2 exp(-r/2)                    stationaries.py:250-251 */
  GPK_K_LINEAR = 6,   /* (x*sigma^2) . x'                        linears.py:60-64 */
  GPK_K_WHITE = 7,    /* sigma^2 delta_ij iff X2 is NULL, else 0 statics.py:57-63 */
  GPK_K_CONSTANT = 8, /* sigma^2                                 statics.py:78-91 */
  GPK_K_SUM = 9,      /* add_n of children                       base.py:305-308 */
  GPK_K_PRODUCT = 10, /* product of children                     base.py:311-314 */
  GPK_K_POLYNOMIAL = 11 /* ((x*sigma^2) . x' + offset)^degree: offset in `lengthscale`, degree in `alpha`  linears.py:71-112 */
};

#define GPK_MAX_CHILDREN 8

/* One node of a flattened kernel expression tree, children before parents, root LAST.
 * Replaces the Python object graph walked by Kernel.__call__ / ReducingCombination.__call__
 * (gpflow/kernels/base.py:195-214, 281-291): every leaf applies its OWN active_dims to the
 * unsliced X.  `dims` / `ard` index into the side arrays handed to gpk_kbuild. */
typedef struct gpk_knode {
  int32_t op;
  int32_t n_children;
  int32_t child[GPK_MAX_CHILDREN];
  double variance;    /* scalar variance (ignored when LINEAR has ARD variances) */
  double lengthscale; /* scalar lengthscale (ignored when n_ard > 0) */
  double alpha;       /* RationalQuadratic only */
  int32_t n_dims;     /* #active dims; 0 = all D columns (slice(None)) base.py:90-109 */
  int32_t dims_off;   /* offset of this leaf's column indices in `dims` */
  int32_t n_ard;      /* 0 = scalar; else == #active dims: per-dim lengthscales (stationary)
                         or per-dim variances (LINEAR) stationaries.py:60-75, linears.py:38-49 */
  int32_t ard_off;    /* offset in `ard` */
} gpk_knode;

GPK_API int gpk_version(void);
GPK_API const char* gpk_last_error(void);

/* K = kernel(X, X2) [+ diag].  Replaces square_distance + K_r/K_r2 + Sum/Product temporaries
 * (gpflow/utilities/ops.py:105-122, kernels/stationaries.py:77-130, kernels/base.py:281-314) and
 * the diagonal shifts add_noise_cov (utilities/model_utils.py:33-38) / `+ jitter*eye`
 * (covariances/kuus.py:33).
 *   nodes/n_nodes, dims, ard : HOST arrays describing the expression (copied per call)
 *   X [N, D] (ldx), X2 [N2, D] (ldx2) or NULL => symmetric K(X, X) with White active
 *   K [N, N2] (ldk) output
 *   uplo: GPK_FULL, or GPK_LOWER (symmetric only: tiles strictly above the diagonal are skipped)
 *   diag_scalar / diag_vec[N] (device, may be NULL): added to K[i,i] (symmetric only) */
GPK_API int gpk_kbuild(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
               const void* X, int64_t N, int64_t ldx, const void* X2, int64_t N2, int64_t ldx2,
               int64_t D, void* K, int64_t ldk, int dtype, int uplo, double diag_scalar,
               const void* diag_vec, void* stream);

/* out[i] = K_diag(X)[i]  (kernel(X, full_cov=False); stationaries.py:82-83, statics.py:41-42,
 * linears.py:67-68, base.py:296-297). */
GPK_API int gpk_kdiag(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
              const void* X, int64_t N, int64_t ldx, int64_t D, void* out, int dtype, void* stream);

/* In-place lower Cholesky of the leading n x n block of the row-major [rows, n] matrix A; only the
 * lower triangle is read; the strict upper triangle is left untouched.  Rows n..rows-1 (if any)
 * are overwritten with A[n:, :] L^-T — i.e. appending B^T as extra rows yields (L^-1 B)^T for
 * free.  Replaces tf.linalg.cholesky (gpflow/models/gpr.py:102, posteriors.py:422,533,538,703,
 * models/sgpr.py:201,207, conditionals/util.py:67, kullback_leiblers.py:107) and the
 * triangular_solve of logdensities.py:150.
 *   ws: gpk_potrf_ws(n, rows, dtype) bytes; on return its head holds the inverses of the 128x128
 *       diagonal blocks of L (reused by gpk_trsm via `dinv`); the rest is scratch: the int8 digit planes of the
 *       tcgen05 trailing updates (fp64, n >= 256), or -- square fp32 matrices of n >= 512, which are widened,
 *       factored on the fp64 path and rounded back -- the fp64 copy with its own inverse slots and planes.
 *   info (device int32, may be NULL): 0, or 1-based index of the first non-positive pivot. */
GPK_API size_t gpk_potrf_ws(int64_t n, int64_t rows, int dtype);
GPK_API int gpk_potrf(void* A, int64_t n, int64_t rows, int64_t lda, int dtype, int32_t* info, void* ws,
              void* stream);

/* Batched variant: `batch` matrices `stride` elements apart (multi-output Kuu stacks [L, M, M],
 * gpflow/covariances/multioutput/kuus.py:62-122).  n <= 128: the whole batch is ONE launch (one CTA per matrix) and the
 * workspace receives one 128x128 inverse slot per matrix; larger n: the factorisations run back to back on the stream.
 * ws: gpk_potrf_batched_ws(n, batch, dtype) bytes.  info: `batch` device words. */
GPK_API size_t gpk_potrf_batched_ws(int64_t n, int batch, int dtype);
GPK_API int gpk_potrf_batched(void* A, int64_t n, int64_t lda, int64_t stride, int batch, int dtype,
                      int32_t* info, void* ws, void* stream);

/* B <- L^-1 B (trans=0) or L^-T B (trans=1); L [n,n] lower (ldl), B [n, nrhs] (ldb).
 * Replaces tf.linalg.triangular_solve (conditionals/util.py:125,139, models/sgpr.py:204,264,
 * posteriors.py:495-496,534,540,707,710, kullback_leiblers.py:114,152).
 *   dinv: inverses of L's 128x128 diagonal blocks as left by gpk_potrf in its ws, or NULL (then
 *         they are recomputed into ws).  ws: gpk_trsm_ws(n, dtype) bytes. */
GPK_API size_t gpk_trsm_ws(int64_t n, int dtype);
GPK_API int gpk_trsm(int trans, const void* L, int64_t n, int64_t ldl, void* B, int64_t nrhs, int64_t ldb,
             int dtype, const void* dinv, void* ws, void* stream);

/* C[m,n] = alpha * op(A) op(B) + beta * C.  transa=0: A stored [m,k]; 1: stored [k,m].
 * transb=0: B stored [k,n]; 1: stored [n,k].  flags: see below.
 * Replaces tf.linalg.matmul (models/sgpr.py:205,263, conditionals/util.py:144,157,
 * posteriors.py:497,535,539,728,734). */
enum {
  GPK_GEMM_LOWER_ONLY = 1,  /* only tiles touching the lower triangle of C (SYRK use) */
  GPK_GEMM_A_LOWER = 2,     /* stored A is lower triangular (band_part(-1,0), util.py:151):
                               entries above its diagonal are treated as zero and never read */
  GPK_GEMM_COLSUMSQ = 4     /* do not store C; instead colsum[j] += sum_i (alpha op(A)op(B))_ij^2
                               into `C` interpreted as a [n] vector (util.py:164 fused) */
};
GPK_API int gpk_gemm(int transa, int transb, int64_t m, int64_t n, int64_t k, double alpha, const void* A,
             int64_t lda, const void* B, int64_t ldb, double beta, void* C, int64_t ldc, int dtype,
             int flags, void* stream);

/* Reductions (device outputs, fp64 accumulators written as `dtype`):
 *   colsumsq: out[j] (+)= scale * sum_i A[i,j]^2      conditionals/util.py:133,164
 *   reduce  : out[0] (+)= scale * sum f(x)            logdensities.py:152-154, sgpr.py:233-243,
 *                                                     kullback_leiblers.py:124,130,134,159
 *             f: 0 sum, 1 sum of squares, 2 sum log, 3 sum log of squares
 *             x: strided vector (n elements, `inc` apart) — inc=ld+1 walks a diagonal.
 *   tril_sumsq: out[0] (+)= scale * sum_{b} sum_{i>=j} A[b,i,j]^2   kullback_leiblers.py:120,134 */
GPK_API int gpk_colsumsq(const void* A, int64_t m, int64_t n, int64_t lda, double scale, int accumulate,
                 void* out, int dtype, void* stream);
GPK_API int gpk_reduce(int f, const void* x, int64_t n, int64_t inc, double scale, int accumulate,
               double* out, int dtype, void* stream);
GPK_API int gpk_tril_sumsq(const void* A, int64_t n, int64_t lda, int64_t stride, int batch, double scale,
                   int accumulate, double* out, int dtype, void* stream);

/* Elementwise helpers used by the Python mirror where the reference has small TF ops:
 *   axpby:    Y[m,n] = a*X + b*Y                      (Y - m(X): gpr.py:103-105; + mean)
 *   scale_cols: A[i,j] *= s[j]  or  /= s[j]           (kuf / sigma: sgpr.py:204)
 *   scale_rows: A[i,j] *= s[i]  or  /= s[i]           (err / sigma[:,None]: sgpr.py:262)
 *   add_diag: A[i,i] += scalar + vec[i]               (add_noise_cov model_utils.py:33-38)
 *   fill / tril (zero strict upper, batched)          (band_part util.py:151) */
GPK_API int gpk_axpby(int64_t m, int64_t n, double a, const void* X, int64_t ldx, double b, void* Y,
              int64_t ldy, int dtype, void* stream);
GPK_API int gpk_scale_cols(void* A, int64_t m, int64_t n, int64_t lda, const void* s, int invert,
                   int dtype, void* stream);
GPK_API int gpk_scale_rows(void* A, int64_t m, int64_t n, int64_t lda, const void* s, int invert,
                   int dtype, void* stream);
GPK_API int gpk_add_diag(void* A, int64_t n, int64_t lda, double scalar, const void* vec, int dtype,
                 void* stream);
GPK_API int gpk_fill(void* A, int64_t m, int64_t n, int64_t lda, double value, int dtype, void* stream);
GPK_API int gpk_tril(void* A, int64_t n, int64_t lda, int64_t stride, int batch, int dtype, void* stream);
GPK_API int gpk_transpose(const void* A, int64_t m, int64_t n, int64_t lda, void* B, int64_t ldb, int dtype,
                  void* stream);

/* var_exp sum: out[0] (+)= scale * sum_{n,p} [-1/2 log 2pi - 1/2 log s2 - 1/2((y-mu)^2+v)/s2]
 * (gpflow/likelihoods/scalar_continuous.py:139-148 + models/svgp.py:174-181).
 * Fmu, Fvar, Y: [B, P] contiguous. */
GPK_API int gpk_gaussian_varexp_sum(const void* Fmu, const void* Fvar, const void* Y, int64_t B, int64_t P,
                            double noise_variance, double scale, int accumulate, double* out,
                            int dtype, void* stream);

/* predictive log density per row: out[n] = sum_p log N(Y[n,p] | Fmu[n,p], Fvar[n,p] + noise_variance), out [B] of the
 * same dtype (gpflow/likelihoods/scalar_continuous.py:133-136, logdensities.py:29-30; models/model.py:332-343). */
GPK_API int gpk_gaussian_log_density(const void* Fmu, const void* Fvar, const void* Y, int64_t B, int64_t P,
                             double noise_variance, void* out, int dtype, void* stream);

/* ---- Kernels that are not functions of a Gram term (materialised leaves; the Python layer composes them with
 * Sum / Product / ChangePoints through gpk_axpby / gpk_hadamard / gpk_scale_rows / gpk_scale_cols) ------------------ */
enum {
  GPK_KAUX_COSINE = 0,   /* sigma^2 cos(2 pi sum_d (x_d - x'_d) scale_d), scale = 1 / lengthscale   stationaries.py:316-332 */
  GPK_KAUX_PERIODIC = 1, /* base.K_r(sum_d |sin(pi (x_d - x'_d) / period_d)| scale_d) for bases with K_r (Matern12/32/52,
                            Exponential), base.K_r2(sum_d sin^2(...) scale_d^2) otherwise (RBF, RQ)    periodic.py:28-111 */
  GPK_KAUX_ARCCOS = 2,   /* sigma^2 / pi J_order(theta) |x|^order |x'|^order, |x|^2 = sum_d scale_d x_d^2 + bias
                            (scale = weight variances)                                               misc.py:27-200 */
  GPK_KAUX_COREGION = 3  /* table[int(x), int(x')], table = W W^T + diag(kappa) [table_dim^2 doubles]  misc.py:203-296 */
};
#define GPK_KAUX_MAXD 32
typedef struct gpk_kaux_desc {
  int32_t op;
  int32_t base;      /* PERIODIC: GPK_K_* op code of the base kernel */
  int32_t order;     /* ARCCOS: 0, 1 or 2 */
  int32_t n_dims;    /* active columns (explicit, 1..GPK_KAUX_MAXD) */
  int32_t table_dim; /* COREGION: output_dim */
  int32_t pad_;
  double variance, alpha, bias;
  const void* table; /* COREGION: DEVICE pointer to the [table_dim, table_dim] float64 matrix B */
  int32_t dims[GPK_KAUX_MAXD];
  double scale[GPK_KAUX_MAXD];
  double period[GPK_KAUX_MAXD];
} gpk_kaux_desc;

/* K [N, N2] = kernel(X, X2) (X2 NULL: K(X, X)) and its diagonal for the kernels above. */
GPK_API int gpk_kaux(const gpk_kaux_desc* desc, const void* X, int64_t N, int64_t ldx, const void* X2, int64_t N2,
             int64_t ldx2, void* K, int64_t ldk, int dtype, void* stream);
GPK_API int gpk_kaux_diag(const gpk_kaux_desc* desc, const void* X, int64_t N, int64_t ldx, void* out, int dtype,
                  void* stream);
/* ChangePoints sigmoid weights (gpflow/kernels/changepoints.py:118-137,189-193): out[n] =
 * (has_lo ? sig(steep_lo (x_n - loc_lo)) : 1) * (has_hi ? 1 - sig(steep_hi (x_n - loc_hi)) : 1), x_n = X[n, dim]. */
GPK_API int gpk_changepoint_weights(const void* X, int64_t N, int64_t ldx, int dim, int has_lo, double loc_lo,
                            double steep_lo, int has_hi, double loc_hi, double steep_hi, void* out,
                            int dtype, void* stream);
/* A[m, n] = max(A, lower), then squared (`square` = 1) or square-rooted (2): evaluation of a heteroskedastic
 * Gaussian(variance|scale=Function) (gpflow/likelihoods/scalar_continuous.py:92-102: tf.maximum(f(X), lower_bound) [** 2])
 * and tf.sqrt(cov) of sample_mvn (conditionals/util.py:199). */
GPK_API int gpk_clamp_min(void* A, int64_t m, int64_t n, int64_t lda, double lower, int square, int dtype,
                  void* stream);
/* Y[m, n] *= X elementwise (Product of materialised kernels, base.py:311-314). */
GPK_API int gpk_hadamard(int64_t m, int64_t n, const void* X, int64_t ldx, void* Y, int64_t ldy, int dtype,
                 void* stream);

/* ---- Fused objectives: one call per evaluation ------------------------------------------- */

/* GPR.log_marginal_likelihood (gpflow/models/gpr.py:91-107): K-build(lower)+noise, Cholesky with
 * (Y-m)^T appended as extra rows, log-density reduction.  Yc [N,P] = Y - mean_function(X)
 * (contiguous).  out: device double[4] = {lml, sum alpha^2, sum log diag L, info}.
 * ws: gpk_gpr_lml_ws(N, P, dtype) bytes. */
GPK_API size_t gpk_gpr_lml_ws(int64_t N, int64_t P, int dtype);
GPK_API int gpk_gpr_lml(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
                const void* X, int64_t N, int64_t ldx, int64_t D, const void* Yc, int64_t P,
                double noise_variance, const void* noise_vec, int dtype, double* out, void* ws,
                void* stream);

/* GPR log marginal likelihood AND its gradient w.r.t. the kernel variance, the likelihood variance and the
 * lengthscale(s): the backward pass that TensorFlow autodiff supplies to the reference's optimiser
 * (gpflow/optimizers/scipy.py:78-228 -> models/training_mixins.py:43-78 -> models/gpr.py:91-107), written out as
 * dLML/dK = 1/2 (alpha alpha^T - P K^-1), K^-1 = L^-T L^-1 from the factor of the forward pass, and one K-build-shaped
 * reduction sum_ij (dLML/dK)_ij dK_ij/dtheta.  Covers a single stationary leaf kernel (RBF, Matern12/32/52,
 * Exponential; scalar or ARD lengthscale), float64.
 *   out: device double[n_out]: [0..3] as gpk_gpr_lml, [4] d/dvariance, [5] d/dnoise_variance,
 *        [6 .. 6 + n_l) d/dlengthscale (n_l = 1, or the number of ARD lengthscales); n_out >= 6 + n_l.
 *   ws:  gpk_gpr_lml_grad_ws(N, P, dtype) bytes. */
GPK_API size_t gpk_gpr_lml_grad_ws(int64_t N, int64_t P, int dtype);
GPK_API int gpk_gpr_lml_grad(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
                     const void* X, int64_t N, int64_t ldx, int64_t D, const void* Yc, int64_t P,
                     double noise_variance, int dtype, double* out, int n_out, void* ws, void* stream);

/* SGPR.elbo (gpflow/models/sgpr.py:181-289).  Yc = Y - m(X) [N,P] contiguous, Z [M,D].
 * out: device double[8] = {elbo, const, logdet, quad, trace_k, trace_q, half_logdet_b, info}.
 * If `cache_L`, `cache_LB`, `cache_c` are non-NULL they receive L [M,M], LB [M,M], c [M,P]
 * (posteriors.py:520-551) for prediction. */
GPK_API size_t gpk_sgpr_elbo_ws(int64_t N, int64_t M, int64_t P, int dtype);
GPK_API int gpk_sgpr_elbo(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
                  const void* X, int64_t N, int64_t ldx, int64_t D, const void* Yc, int64_t P,
                  const void* Z, int64_t M, int64_t ldz, double noise_variance, double jitter,
                  int dtype, double* out, void* cache_L, void* cache_LB, void* cache_c, void* ws,
                  void* stream);

/* SGPR ELBO AND its gradient w.r.t. the kernel variance, the likelihood variance, the lengthscale(s) and the inducing
 * points: the backward pass that TensorFlow autodiff supplies to the reference's optimiser (gpflow/optimizers/scipy.py:78-228
 * -> models/training_mixins.py:43-78 -> models/sgpr.py:181-289), written out (DESIGN.md section 4.9).  The forward of
 * gpk_sgpr_elbo runs unchanged into the head of the workspace; the backward then forms, in fp64, L^-1, LB^-1, B^-1 and
 * dELBO/dKuu, computes dELBO/dKuf = (L^-T C A' + v E^T) / s2 with one M x M x N GEMM in the model dtype, and reduces
 * dK (.) dK/dtheta over the Kuf and Kuu tiles.  No host synchronisation.  Covers a single stationary leaf kernel (RBF,
 * Matern12/32/52, Exponential; scalar or ARD lengthscale; active_dims), float32 and float64.  Arguments as gpk_sgpr_elbo
 * without the cache pointers, plus:
 *   out: device double[n_out]: [0..7] as gpk_sgpr_elbo, [8] d/dvariance, [9] d/dnoise_variance,
 *        [10 .. 10 + n_l) d/dlengthscale (n_l = 1, or the number of ARD lengthscales); n_out >= 10 + n_l.
 *   dZ:  device double [M, D] (lddz >= D): d/dZ; zero in the columns outside the kernel's active dims.
 *   ws:  gpk_sgpr_elbo_grad_ws(N, M, P, dtype) bytes. */
GPK_API size_t gpk_sgpr_elbo_grad_ws(int64_t N, int64_t M, int64_t P, int dtype);
GPK_API int gpk_sgpr_elbo_grad(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
                       const void* X, int64_t N, int64_t ldx, int64_t D, const void* Yc, int64_t P,
                       const void* Z, int64_t M, int64_t ldz, double noise_variance, double jitter,
                       int dtype, double* out, int n_out, double* dZ, int64_t lddz, void* ws,
                       void* stream);

/* SVGP.elbo (gpflow/models/svgp.py:166-181) for a single-output kernel shared by P latent GPs
 * (posteriors.py:827-841 -> conditionals/util.py:84-169 -> kullback_leiblers.py:59-165 ->
 * likelihoods/scalar_continuous.py:139-148).  Xb [B,D], Yc = Yb - m(Xb) [B,P] contiguous,
 * Z [M,D], q_mu [M,P], q_sqrt [P,M,M] (q_diag=0) or [M,P] (q_diag=1).
 * Latent GPs p in [p_begin, p_end) are evaluated (latent sharding); KL is included for those p.
 * out: device double[4] = {elbo_partial, sum var_exp (unscaled), kl, info}. */
GPK_API size_t gpk_svgp_elbo_ws(int64_t B, int64_t M, int64_t P, int dtype);
GPK_API int gpk_svgp_elbo(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
                  const void* Xb, int64_t B, int64_t ldx, int64_t D, const void* Yc, int64_t P,
                  const void* Z, int64_t M, int64_t ldz, const void* q_mu, const void* q_sqrt,
                  int q_diag, int whiten, double noise_variance, double num_data_scale,
                  double jitter, int p_begin, int p_end, int dtype, double* out, void* ws,
                  void* stream);

/* The same evaluation in two stages, for latent-GP sharding over GPUs with a COLUMN-SHARDED triangular solve
 * (SURVEY.md 8(e); derived from conditionals/util.py:125-164: every column of A = Lm^-1 Kuf depends on its own x_n only):
 *   stage 1: Kuu, chol(Kuu), Kuf[:, col_begin:col_end] and A[:, col_begin:col_end] = Lm^-1 Kuf[:, ...], left in place in
 *            the workspace matrix A [M, ld] (gpk_svgp_elbo_A returns its byte offset in `ws` and `ld`); the caller
 *            all-gathers the column blocks of A between the ranks (NCCL);
 *   stage 2: everything after the solve (fmean, fvar, variational expectations, KL) for the latents [p_begin, p_end)
 *            with A complete in the workspace.  stage 0 = gpk_svgp_elbo.  whiten = 1 only. */
GPK_API size_t gpk_svgp_elbo_A(int64_t B, int64_t M, int64_t P, int dtype, int64_t* ld);
GPK_API int gpk_svgp_elbo_staged(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard,
                         const void* Xb, int64_t B, int64_t ldx, int64_t D, const void* Yc, int64_t P,
                         const void* Z, int64_t M, int64_t ldz, const void* q_mu, const void* q_sqrt,
                         int q_diag, int whiten, double noise_variance, double num_data_scale, double jitter,
                         int p_begin, int p_end, int stage, int64_t col_begin, int64_t col_end, int dtype,
                         double* out, void* ws, void* stream);

/* ---- Instrumentation (bench.py / tests; not on the numeric path) ---------------------------- */
/* Number of CUDA kernels launched by this library since the last reset. */
GPK_API int64_t gpk_launch_count(void);
GPK_API void gpk_launch_count_reset(void);
/* Per-kernel-class device timing with CUDA events recorded on the launch stream around every
 * launch (single-threaded diagnostic).  Classes: 0 kbuild, 1 tiled DMMA / SIMT GEMM (small-K trailing
 * updates, TRSM blocks), 2 potrf leaf (128x128 factor+invert; includes its look-ahead spin), 3 skinny
 * GEMM, 4 reductions/elementwise/slicing, 5 tcgen05 kernels (int8 digit SYRK, tf32 GEMM), 6 panel solve.
 * gpk_prof_read synchronises, writes summed milliseconds and launch counts for `n` classes and
 * clears the records; gpk_prof_read2 also returns the operations ISSUED per class (class 5: MACs on
 * the tensor pipe, padding tiles included). */
#define GPK_PROF_CLASSES 8
/* Tuning aid: runs ONE fp64 128x128 leaf (factor+invert) and stores clock64() at its phase
 * boundaries into dbg[0..11] (device int64, at least 12 entries; scripts/leaf_timing.py names them). */
GPK_API int gpk_debug_leaf(void* A, int64_t lda, int n, void* dinv, void* dbg, void* stream);
/* Tuning aid: device timeline of a factorisation.  While `buf` is set, thread 0 of selected CTAs of the leaf (id 1), fused
 * panel (2), plain panel (3) and tcgen05 update (4) kernels append (%globaltimer ns, id << 8 | phase) pairs to buf[2 * capacity]
 * (device uint64) through the counter *pos (device uint32).  phase 0 = first CTA started, 1 = inputs ready (leaf) / look-ahead
 * block published (panel, update), 2 = first CTA done, 3 = last CTA done.  buf = NULL switches it off.  scripts/trace_chain.py. */
GPK_API int gpk_debug_trace(void* buf, void* pos, unsigned int capacity);
GPK_API int gpk_prof_enable(int on);
GPK_API int gpk_prof_read(double* ms, int64_t* launches, int n);
GPK_API int gpk_prof_read2(double* ms, int64_t* launches, double* work, int n);
/* Pipe peaks measured in place (operands resident, every SM busy): out_host[0] = tcgen05 kind::i8 issue peak in
 * T(int8 op)/s (2 per MAC), out_host[1] = mma.sync.m8n8k4.f64 peak in TFLOP/s, out_host[2] = SM count.  Synchronises.
 * The roofline denominators bench.py reports for syrk_i8_kernel and the DMMA kernels. */
GPK_API int gpk_peak_probe(double* out_host, void* stream);
/* Digit planes S used by the tcgen05 trailing updates of the most recent fp64 factorisation on this process (chosen from
 * the conditioning hint of the caller: 6 or 7 base-256 planes; 0 = no update ran on tcgen05, e.g. n < 512 or fp32). */
GPK_API int gpk_potrf_last_slices(void);
/* Eager creation of the library-owned per-(device, stream) resources (see "Conventions"): the look-ahead side stream and
 * events, and `tf32_scratch_bytes` of TF32 plane scratch (0 = skip; 2 * 4 * (m + n) * k bytes cover an m x n x k product). */
GPK_API int gpk_warm(size_t tf32_scratch_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPK_H_ */
