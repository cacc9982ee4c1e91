// capi.cu — the extern "C" surface declared in include/gpk.h (argument checks + dtype dispatch).
#include <stdarg.h>

#include <atomic>
#include <vector>

#include "internal.cuh"

namespace gpk {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

struct ProfRec { cudaEvent_t a, b; int cls; double work; };
static std::vector<ProfRec> g_recs;
static bool g_prof = false;

ProfScope::ProfScope(int cls, cudaStream_t s, double work) : idx(-1), st(s) {
  if (!g_prof) return;
  ProfRec r;
  r.cls = cls;
  r.work = work;
  if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
  cudaEventRecord(r.a, s);
  g_recs.push_back(r);
  idx = (int)g_recs.size() - 1;
}
ProfScope::~ProfScope() {
  if (idx >= 0) cudaEventRecord(g_recs[idx].b, st);
}

int gemm_any(int ta, int tb, int64_t m, int64_t n, int64_t k, double alpha, const void* A, int64_t lda, const void* B,
             int64_t ldb, double beta, void* C, int64_t ldc, int dtype, int flags, cudaStream_t st) {
  if (dtype == GPK_F64)
    return gemm_t<double>(ta, tb, m, n, k, alpha, (const double*)A, lda, (const double*)B, ldb, beta, (double*)C, ldc,
                          flags, st);
  return gemm_t<float>(ta, tb, m, n, k, (float)alpha, (const float*)A, lda, (const float*)B, ldb, (float)beta,
                       (float*)C, ldc, flags, st);
}

int potrf_any(void* A, int64_t n, int64_t rows, int64_t lda, int dtype, int32_t* info, void* ws, cudaStream_t st,
              bool need_dinv, double cond_hint) {
  const size_t tcb = potrf_tc_ws_bytes(n, rows, dtype);
  void* tcws = tcb ? (char*)ws + align_up(dinv_bytes(n, dtype), 256) + 256 : nullptr;
  if (dtype == GPK_F64)
    return potrf_t<double>((double*)A, n, rows, lda, info, (double*)ws, tcws, tcb, st, need_dinv, cond_hint);
  return potrf_t<float>((float*)A, n, rows, lda, info, (float*)ws, tcws, tcb, st, need_dinv);
}

int trsm_any(int trans, const void* L, int64_t n, int64_t ldl, void* B, int64_t nrhs, int64_t ldb, int dtype,
             const void* dinv, cudaStream_t st) {
  if (dtype == GPK_F64)
    return trsm_t<double>(trans, (const double*)L, n, ldl, (double*)B, nrhs, ldb, (const double*)dinv, st);
  return trsm_t<float>(trans, (const float*)L, n, ldl, (float*)B, nrhs, ldb, (const float*)dinv, st);
}

int trtri_diag_any(const void* L, int64_t n, int64_t ldl, void* dinv, int dtype, cudaStream_t st) {
  if (dtype == GPK_F64) return trtri_diag_t<double>((const double*)L, n, ldl, (double*)dinv, st);
  return trtri_diag_t<float>((const float*)L, n, ldl, (float*)dinv, st);
}

int leaf_debug(double* A, int64_t lda, int n, double* dinv, long long* dbg, cudaStream_t st);
int peak_probe(double* out_host, cudaStream_t st);
int lookahead_warm(cudaStream_t st);
int tf32_reserve(size_t bytes, cudaStream_t st);
template <typename T>
int potrf_batched_small_t(T* A, int64_t n, int64_t lda, int64_t stride, int batch, int32_t* info, T* dinv, cudaStream_t st);
int kaux_impl(const gpk_kaux_desc* d, const void* X, int64_t N, int64_t ldx, const void* X2, int64_t N2, int64_t ldx2,
              void* K, int64_t ldk, int dtype, cudaStream_t st);
int kaux_diag_impl(const gpk_kaux_desc* d, const void* X, int64_t N, int64_t ldx, void* out, int dtype, cudaStream_t st);
int cp_weights_impl(const void* X, int64_t N, int64_t ldx, int dim, int has_lo, double loc_lo, double steep_lo,
                    int has_hi, double loc_hi, double steep_hi, void* out, int dtype, cudaStream_t st);
int hadamard_impl(int64_t m, int64_t n, const void* X, int64_t ldx, void* Y, int64_t ldy, int dtype, cudaStream_t st);
int clamp_min_impl(void* A, int64_t m, int64_t n, int64_t lda, double lower, int square, int dtype, cudaStream_t st);
int potrf_last_slices();
size_t gpr_lml_ws(int64_t N, int64_t P, int dtype);
int gpr_lml(const gpk_knode*, int, const int32_t*, const double*, const void*, int64_t, int64_t, int64_t, const void*,
            int64_t, double, const void*, int, double*, void*, cudaStream_t);
size_t gpr_lml_grad_ws(int64_t N, int64_t P, int dtype);
int gpr_lml_grad(const gpk_knode*, int, const int32_t*, const double*, const void*, int64_t, int64_t, int64_t,
                 const void*, int64_t, double, int, double*, int, void*, cudaStream_t);
size_t sgpr_elbo_ws(int64_t N, int64_t M, int64_t P, int dtype);
int sgpr_elbo(const gpk_knode*, int, const int32_t*, const double*, const void*, int64_t, int64_t, int64_t, const void*,
              int64_t, const void*, int64_t, int64_t, double, double, int, double*, void*, void*, void*, void*,
              cudaStream_t);
size_t sgpr_elbo_grad_ws(int64_t N, int64_t M, int64_t P, int dtype);
int sgpr_elbo_grad(const gpk_knode*, int, const int32_t*, const double*, const void*, int64_t, int64_t, int64_t,
                   const void*, int64_t, const void*, int64_t, int64_t, double, double, int, double*, int, double*,
                   int64_t, void*, cudaStream_t);
size_t svgp_elbo_ws(int64_t B, int64_t M, int64_t P, int dtype);
int svgp_elbo(const gpk_knode*, int, const int32_t*, const double*, const void*, int64_t, int64_t, int64_t, const void*,
              int64_t, const void*, int64_t, int64_t, const void*, const void*, int, int, double, double, double, int,
              int, int, double*, void*, cudaStream_t, int stage = 0, int64_t c0 = 0, int64_t c1 = 0);
size_t svgp_elbo_A(int64_t B, int64_t M, int64_t P, int dtype, int64_t* ld);

}  // namespace gpk

using namespace gpk;

#define GPK_DTYPE_OK(name) GPK_CHECK_ARG(dtype == GPK_F32 || dtype == GPK_F64, name ": bad dtype %d", dtype)

extern "C" {

int gpk_version(void) { return GPK_VERSION; }

int64_t gpk_launch_count(void) { return (int64_t)g_launches.load(); }
void gpk_launch_count_reset(void) { g_launches.store(0); }

int gpk_debug_leaf(void* A, int64_t lda, int n, void* dinv, void* dbg, void* stream) {
  return leaf_debug((double*)A, lda, n, (double*)dinv, (long long*)dbg, (cudaStream_t)stream);
}

int gpk_debug_trace(void* buf, void* pos, unsigned int capacity) {
  TraceBuf tb{(unsigned long long*)buf, (unsigned int*)pos, buf ? capacity : 0u};
  GPK_TRY(trace_set_potrf(tb));
  GPK_TRY(trace_set_tc(tb));
  return 0;
}

int gpk_prof_enable(int on) {
  for (auto& r : g_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_recs.clear();
  g_prof = on != 0;
  return 0;
}

int gpk_peak_probe(double* out_host, void* stream) {
  GPK_CHECK_ARG(out_host, "peak_probe: bad arguments");
  return peak_probe(out_host, (cudaStream_t)stream);
}

int gpk_prof_read(double* ms, int64_t* launches, int n) { return gpk_prof_read2(ms, launches, nullptr, n); }

int gpk_potrf_last_slices(void) { return potrf_last_slices(); }

int gpk_warm(size_t tf32_scratch_bytes, void* stream) {
  GPK_TRY(lookahead_warm((cudaStream_t)stream));
  if (tf32_scratch_bytes) GPK_TRY(tf32_reserve(tf32_scratch_bytes, (cudaStream_t)stream));
  return 0;
}

int gpk_kaux(const gpk_kaux_desc* desc, const void* X, int64_t N, int64_t ldx, const void* X2, int64_t N2, int64_t ldx2, void* K,
             int64_t ldk, int dtype, void* stream) {
  GPK_DTYPE_OK("kaux");
  return kaux_impl(desc, X, N, ldx, X2, N2, ldx2, K, ldk, dtype, (cudaStream_t)stream);
}
int gpk_kaux_diag(const gpk_kaux_desc* desc, const void* X, int64_t N, int64_t ldx, void* out, int dtype, void* stream) {
  GPK_DTYPE_OK("kaux_diag");
  return kaux_diag_impl(desc, X, N, ldx, out, dtype, (cudaStream_t)stream);
}
int gpk_changepoint_weights(const void* X, int64_t N, int64_t ldx, int dim, int has_lo, double loc_lo, double steep_lo,
                            int has_hi, double loc_hi, double steep_hi, void* out, int dtype, void* stream) {
  GPK_DTYPE_OK("changepoint_weights");
  return cp_weights_impl(X, N, ldx, dim, has_lo, loc_lo, steep_lo, has_hi, loc_hi, steep_hi, out, dtype,
                         (cudaStream_t)stream);
}
int gpk_clamp_min(void* A, int64_t m, int64_t n, int64_t lda, double lower, int square, int dtype, void* stream) {
  GPK_DTYPE_OK("clamp_min");
  return clamp_min_impl(A, m, n, lda, lower, square, dtype, (cudaStream_t)stream);
}
int gpk_hadamard(int64_t m, int64_t n, const void* X, int64_t ldx, void* Y, int64_t ldy, int dtype, void* stream) {
  GPK_DTYPE_OK("hadamard");
  return hadamard_impl(m, n, X, ldx, Y, ldy, dtype, (cudaStream_t)stream);
}

int gpk_prof_read2(double* ms, int64_t* launches, double* work, int n) {
  GPK_CHECK_ARG(ms && launches && n > 0, "prof_read: bad arguments");
  for (int i = 0; i < n; ++i) { ms[i] = 0.0; launches[i] = 0; if (work) work[i] = 0.0; }
  GPK_CUDA_OK(cudaDeviceSynchronize());
  for (auto& r : g_recs) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess && r.cls < n) {
      ms[r.cls] += t;
      launches[r.cls] += 1;
      if (work) work[r.cls] += r.work;
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_recs.clear();
  return 0;
}
const char* gpk_last_error(void) { return g_err; }

int gpk_kbuild(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
               int64_t ldx, const void* X2, int64_t N2, int64_t ldx2, int64_t D, void* K, int64_t ldk, int dtype,
               int uplo, double diag_scalar, const void* diag_vec, void* stream) {
  return kbuild_impl(nodes, n_nodes, dims, ard, X, N, ldx, X2, N2, ldx2, D, K, ldk, dtype, uplo, diag_scalar, diag_vec,
                     (cudaStream_t)stream);
}

int gpk_kdiag(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
              int64_t ldx, int64_t D, void* out, int dtype, void* stream) {
  return kdiag_impl(nodes, n_nodes, dims, ard, X, N, ldx, D, out, dtype, (cudaStream_t)stream);
}

size_t gpk_potrf_ws(int64_t n, int64_t rows, int dtype) { return potrf_ws_bytes(n, rows < n ? n : rows, dtype); }

int gpk_potrf(void* A, int64_t n, int64_t rows, int64_t lda, int dtype, int32_t* info, void* ws, void* stream) {
  GPK_DTYPE_OK("potrf");
  GPK_CHECK_ARG(A && ws && n >= 0 && rows >= n && lda >= n, "potrf: bad arguments (n=%lld rows=%lld lda=%lld)",
                (long long)n, (long long)rows, (long long)lda);
  return potrf_any(A, n, rows, lda, dtype, info, ws, (cudaStream_t)stream);
}

size_t gpk_potrf_batched_ws(int64_t n, int batch, int dtype) {
  if (n <= NB) return (size_t)(batch > 0 ? batch : 1) * NB * NB * dtype_size(dtype);  // one inverse slot per matrix
  return potrf_ws_bytes(n, n, dtype);
}

int gpk_potrf_batched(void* A, int64_t n, int64_t lda, int64_t stride, int batch, int dtype, int32_t* info, void* ws,
                      void* stream) {
  GPK_DTYPE_OK("potrf_batched");
  GPK_CHECK_ARG(A && ws && n >= 0 && lda >= n && batch >= 0, "potrf_batched: bad arguments");
  if (n <= NB) {  // the whole batch in ONE launch: grid over the matrices
    if (dtype == GPK_F64)
      return potrf_batched_small_t<double>((double*)A, n, lda, stride, batch, info, (double*)ws, (cudaStream_t)stream);
    return potrf_batched_small_t<float>((float*)A, n, lda, stride, batch, info, (float*)ws, (cudaStream_t)stream);
  }
  // larger matrices: each factorisation already fills the GPU; they run back to back on the stream and share the workspace
  for (int b = 0; b < batch; ++b)
    GPK_TRY(potrf_any((char*)A + (size_t)b * stride * dtype_size(dtype), n, n, lda, dtype, info ? info + b : nullptr,
                      ws, (cudaStream_t)stream));
  return 0;
}

size_t gpk_trsm_ws(int64_t n, int dtype) { return dinv_bytes(n, dtype); }

int gpk_trsm(int trans, const void* L, int64_t n, int64_t ldl, void* B, int64_t nrhs, int64_t ldb, int dtype,
             const void* dinv, void* ws, void* stream) {
  GPK_DTYPE_OK("trsm");
  GPK_CHECK_ARG(L && B && n >= 0 && nrhs >= 0 && ldl >= n && ldb >= nrhs, "trsm: bad arguments");
  GPK_CHECK_ARG(dinv || ws, "trsm: need either cached diagonal-block inverses or a workspace");
  if (!dinv) {
    GPK_TRY(trtri_diag_any(L, n, ldl, ws, dtype, (cudaStream_t)stream));
    dinv = ws;
  }
  return trsm_any(trans, L, n, ldl, B, nrhs, ldb, dtype, dinv, (cudaStream_t)stream);
}

int gpk_gemm(int transa, int transb, int64_t m, int64_t n, int64_t k, double alpha, const void* A, int64_t lda,
             const void* B, int64_t ldb, double beta, void* C, int64_t ldc, int dtype, int flags, void* stream) {
  GPK_DTYPE_OK("gemm");
  GPK_CHECK_ARG(A && B && C && m >= 0 && n >= 0 && k >= 0, "gemm: bad arguments");
  GPK_CHECK_ARG(lda >= (transa ? m : k) && ldb >= (transb ? k : n) && ((flags & GPK_GEMM_COLSUMSQ) || ldc >= n),
                "gemm: leading dimension too small");
  return gemm_any(transa, transb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, dtype, flags, (cudaStream_t)stream);
}

int gpk_colsumsq(const void* A, int64_t m, int64_t n, int64_t lda, double scale, int accumulate, void* out, int dtype,
                 void* stream) {
  GPK_DTYPE_OK("colsumsq");
  return colsumsq_impl(A, m, n, lda, scale, accumulate, out, dtype, (cudaStream_t)stream);
}

int gpk_reduce(int f, const void* x, int64_t n, int64_t inc, double scale, int accumulate, double* out, int dtype,
               void* stream) {
  GPK_DTYPE_OK("reduce");
  return reduce_impl(f, x, n, inc, scale, accumulate, out, dtype, (cudaStream_t)stream);
}

int gpk_tril_sumsq(const void* A, int64_t n, int64_t lda, int64_t stride, int batch, double scale, int accumulate,
                   double* out, int dtype, void* stream) {
  GPK_DTYPE_OK("tril_sumsq");
  return tril_sumsq_impl(A, n, lda, stride, batch, scale, accumulate, out, dtype, (cudaStream_t)stream);
}

int gpk_axpby(int64_t m, int64_t n, double a, const void* X, int64_t ldx, double b, void* Y, int64_t ldy, int dtype,
              void* stream) {
  GPK_DTYPE_OK("axpby");
  return axpby_impl(m, n, a, X, ldx, b, Y, ldy, dtype, (cudaStream_t)stream);
}

int gpk_scale_cols(void* A, int64_t m, int64_t n, int64_t lda, const void* s, int invert, int dtype, void* stream) {
  GPK_DTYPE_OK("scale_cols");
  return scale_impl(A, m, n, lda, s, 0, invert, dtype, (cudaStream_t)stream);
}

int gpk_scale_rows(void* A, int64_t m, int64_t n, int64_t lda, const void* s, int invert, int dtype, void* stream) {
  GPK_DTYPE_OK("scale_rows");
  return scale_impl(A, m, n, lda, s, 1, invert, dtype, (cudaStream_t)stream);
}

int gpk_add_diag(void* A, int64_t n, int64_t lda, double scalar, const void* vec, int dtype, void* stream) {
  GPK_DTYPE_OK("add_diag");
  return add_diag_impl(A, n, lda, scalar, vec, dtype, (cudaStream_t)stream);
}

int gpk_fill(void* A, int64_t m, int64_t n, int64_t lda, double value, int dtype, void* stream) {
  GPK_DTYPE_OK("fill");
  return fill_impl(A, m, n, lda, value, dtype, (cudaStream_t)stream);
}

int gpk_tril(void* A, int64_t n, int64_t lda, int64_t stride, int batch, int dtype, void* stream) {
  GPK_DTYPE_OK("tril");
  return tril_impl(A, n, lda, stride, batch, dtype, (cudaStream_t)stream);
}

int gpk_transpose(const void* A, int64_t m, int64_t n, int64_t lda, void* B, int64_t ldb, int dtype, void* stream) {
  GPK_DTYPE_OK("transpose");
  return transpose_impl(A, m, n, lda, B, ldb, dtype, (cudaStream_t)stream);
}

int gpk_gaussian_varexp_sum(const void* Fmu, const void* Fvar, const void* Y, int64_t B, int64_t P,
                            double noise_variance, double scale, int accumulate, double* out, int dtype,
                            void* stream) {
  GPK_DTYPE_OK("gaussian_varexp_sum");
  return varexp_impl(Fmu, Fvar, Y, B, P, P, P, 1, noise_variance, scale, accumulate, out, dtype, (cudaStream_t)stream);
}

int gpk_gaussian_log_density(const void* Fmu, const void* Fvar, const void* Y, int64_t B, int64_t P,
                             double noise_variance, void* out, int dtype, void* stream) {
  GPK_DTYPE_OK("gaussian_log_density");
  return logdensity_rows_impl(Fmu, Fvar, Y, B, P, noise_variance, out, dtype, (cudaStream_t)stream);
}

size_t gpk_gpr_lml_ws(int64_t N, int64_t P, int dtype) { return gpr_lml_ws(N, P, dtype); }

int gpk_gpr_lml(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
                int64_t ldx, int64_t D, const void* Yc, int64_t P, double noise_variance, const void* noise_vec,
                int dtype, double* out, void* ws, void* stream) {
  GPK_DTYPE_OK("gpr_lml");
  return gpr_lml(nodes, n_nodes, dims, ard, X, N, ldx, D, Yc, P, noise_variance, noise_vec, dtype, out, ws,
                 (cudaStream_t)stream);
}

size_t gpk_sgpr_elbo_ws(int64_t N, int64_t M, int64_t P, int dtype) { return sgpr_elbo_ws(N, M, P, dtype); }

int gpk_sgpr_elbo(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
                  int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M, int64_t ldz,
                  double noise_variance, double jitter, int dtype, double* out, void* cache_L, void* cache_LB,
                  void* cache_c, void* ws, void* stream) {
  GPK_DTYPE_OK("sgpr_elbo");
  return sgpr_elbo(nodes, n_nodes, dims, ard, X, N, ldx, D, Yc, P, Z, M, ldz, noise_variance, jitter, dtype, out,
                   cache_L, cache_LB, cache_c, ws, (cudaStream_t)stream);
}

size_t gpk_svgp_elbo_ws(int64_t B, int64_t M, int64_t P, int dtype) { return svgp_elbo_ws(B, M, P, dtype); }

int gpk_svgp_elbo(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* Xb, int64_t B,
                  int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M, int64_t ldz,
                  const void* q_mu, const void* q_sqrt, int q_diag, int whiten, double noise_variance,
                  double num_data_scale, double jitter, int p_begin, int p_end, int dtype, double* out, void* ws,
                  void* stream) {
  GPK_DTYPE_OK("svgp_elbo");
  return svgp_elbo(nodes, n_nodes, dims, ard, Xb, B, ldx, D, Yc, P, Z, M, ldz, q_mu, q_sqrt, q_diag, whiten,
                   noise_variance, num_data_scale, jitter, p_begin, p_end, dtype, out, ws, (cudaStream_t)stream);
}

size_t gpk_gpr_lml_grad_ws(int64_t N, int64_t P, int dtype) { return gpr_lml_grad_ws(N, P, dtype); }

int gpk_gpr_lml_grad(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X, int64_t N,
                     int64_t ldx, int64_t D, const void* Yc, int64_t P, double noise_variance, int dtype, double* out,
                     int n_out, void* ws, void* stream) {
  GPK_DTYPE_OK("gpr_lml_grad");
  return gpr_lml_grad(nodes, n_nodes, dims, ard, X, N, ldx, D, Yc, P, noise_variance, dtype, out, n_out, ws,
                      (cudaStream_t)stream);
}

size_t gpk_sgpr_elbo_grad_ws(int64_t N, int64_t M, int64_t P, int dtype) { return sgpr_elbo_grad_ws(N, M, P, dtype); }

int gpk_sgpr_elbo_grad(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X,
                       int64_t N, int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M,
                       int64_t ldz, double noise_variance, double jitter, int dtype, double* out, int n_out, double* dZ,
                       int64_t lddz, void* ws, void* stream) {
  GPK_DTYPE_OK("sgpr_elbo_grad");
  return sgpr_elbo_grad(nodes, n_nodes, dims, ard, X, N, ldx, D, Yc, P, Z, M, ldz, noise_variance, jitter, dtype, out,
                        n_out, dZ, lddz, ws, (cudaStream_t)stream);
}

size_t gpk_svgp_elbo_A(int64_t B, int64_t M, int64_t P, int dtype, int64_t* ld) { return svgp_elbo_A(B, M, P, dtype, ld); }

int gpk_svgp_elbo_staged(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* Xb,
                         int64_t B, int64_t ldx, int64_t D, const void* Yc, int64_t P, const void* Z, int64_t M,
                         int64_t ldz, const void* q_mu, const void* q_sqrt, int q_diag, int whiten,
                         double noise_variance, double num_data_scale, double jitter, int p_begin, int p_end, int stage,
                         int64_t col_begin, int64_t col_end, int dtype, double* out, void* ws, void* stream) {
  GPK_DTYPE_OK("svgp_elbo_staged");
  return svgp_elbo(nodes, n_nodes, dims, ard, Xb, B, ldx, D, Yc, P, Z, M, ldz, q_mu, q_sqrt, q_diag, whiten,
                   noise_variance, num_data_scale, jitter, p_begin, p_end, dtype, out, ws, (cudaStream_t)stream, stage,
                   col_begin, col_end);
}

}  // extern "C"
