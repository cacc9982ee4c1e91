// internal.cuh — untyped implementation entry points shared by capi.cu and fused.cu.
#pragma once
#include "common.cuh"

namespace gpk {

int kbuild_impl(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X,
                int64_t N, int64_t ldx, const void* X2, int64_t N2, int64_t ldx2, int64_t D, void* K, int64_t ldk,
                int dtype, int uplo, double diag_scalar, const void* diag_vec, cudaStream_t st);
int kdiag_impl(const gpk_knode* nodes, int n_nodes, const int32_t* dims, const double* ard, const void* X,
               int64_t N, int64_t ldx, int64_t D, void* out, int dtype, cudaStream_t st);

int colsumsq_impl(const void* A, int64_t m, int64_t n, int64_t lda, double scale, int accumulate, void* out, int dtype,
                  cudaStream_t st, const void* w = nullptr, int64_t winc = 0);
int reduce_impl(int f, const void* x, int64_t n, int64_t inc, double scale, int accumulate, double* out, int dtype,
                cudaStream_t st);
int reduce_wsq_impl(const void* w, const void* x, int64_t n, int64_t inc, double scale, double* out, int dtype,
                    cudaStream_t st);
int tril_sumsq_impl(const void* A, int64_t n, int64_t lda, int64_t stride, int batch, double scale, int accumulate,
                    double* out, int dtype, cudaStream_t st);
int logdensity_rows_impl(const void* Fmu, const void* Fvar, const void* Y, int64_t B, int64_t P, double noise, void* out,
                         int dtype, cudaStream_t st);
int varexp_impl(const void* Fmu, const void* Fvar, const void* Y, int64_t B, int64_t P, int64_t ldy, int64_t var_sb,
                int64_t var_sp, double noise, double scale, int accumulate, double* out, int dtype, cudaStream_t st);
int axpby_impl(int64_t m, int64_t n, double a, const void* X, int64_t ldx, double b, void* Y, int64_t ldy, int dtype,
               cudaStream_t st);
int scale_impl(void* A, int64_t m, int64_t n, int64_t lda, const void* s, int by_row, int invert, int dtype,
               cudaStream_t st);
int add_diag_impl(void* A, int64_t n, int64_t lda, double scalar, const void* vec, int dtype, cudaStream_t st);
int fill_impl(void* A, int64_t m, int64_t n, int64_t lda, double v, int dtype, cudaStream_t st);
int tril_impl(void* A, int64_t n, int64_t lda, int64_t stride, int batch, int dtype, cudaStream_t st);
int transpose_impl(const void* A, int64_t m, int64_t n, int64_t lda, void* B, int64_t ldb, int dtype, cudaStream_t st);

// dtype-erased wrappers over the typed templates
int gemm_any(int ta, int tb, int64_t m, int64_t n, int64_t k, double alpha, const void* A, int64_t lda, const void* B,
             int64_t ldb, double beta, void* C, int64_t ldc, int dtype, int flags, cudaStream_t st);
// ws = [dinv blocks | tcgen05 digit planes]; sized by potrf_ws_bytes(n, rows, dtype)
// need_dinv = false: the caller never runs trsm on this factor.  cond_hint: an upper bound of max_i A_ii / lambda_min(A)
// when the caller knows one (e.g. (kernel variance + noise) / noise), 0 = unknown; selects the number of digit planes /
// the engine of the fp64 trailing updates (potrf.cu::pick_slices).
int potrf_any(void* A, int64_t n, int64_t rows, int64_t lda, int dtype, int32_t* info, void* ws, cudaStream_t st,
              bool need_dinv = true, double cond_hint = 0.0);
inline size_t potrf_ws_bytes(int64_t n, int64_t rows, int dtype);
int trsm_any(int trans, const void* L, int64_t n, int64_t ldl, void* B, int64_t nrhs, int64_t ldb, int dtype,
             const void* dinv, cudaStream_t st);
int trtri_diag_any(const void* L, int64_t n, int64_t ldl, void* dinv, int dtype, cudaStream_t st);

// Scratch of the SGPR ELBO backward (grad.cu), laid out by fused.cu behind the forward's workspace.  fp64 [M, ldm]:
// Li, LBi (the factors, inverted in place), B, Bi, C, H, G1, T, dKuu; fp64 [M, P]: cw, wt, v; dinvL / dinvB: 128-block
// inverses; tmp: (M/2 + 128)^2 doubles; sc: 2 scalars; G1n: G1 in the model dtype; dKuf: [M, ldn] model dtype.
struct SgprBwdWs {
  double *Li, *LBi, *B, *Bi, *C, *H, *G1, *T, *dKuu, *dinvL, *dinvB, *tmp, *cw, *wt, *v, *sc;
  void *G1n, *dKuf;
};

inline size_t dinv_bytes(int64_t n, int dtype) { return (size_t)((n + NB - 1) / NB) * NB * NB * dtype_size(dtype); }
inline size_t potrf_ws_bytes(int64_t n, int64_t rows, int dtype) {
  return align_up(dinv_bytes(n, dtype), 256) + 256 /* look-ahead counter */ + potrf_tc_ws_bytes(n, rows, dtype);
}

}  // namespace gpk
