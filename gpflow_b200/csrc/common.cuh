// common.cuh — shared helpers for libgpk (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/gpk.h"

namespace gpk {

// ---- device timeline (tuning aid, gpk_debug_trace): %globaltimer stamps written by thread 0 of selected CTAs ------------------
// Every translation unit that marks has its own copy of g_trace (no relocatable device code); trace_set_* install the buffer.
struct TraceBuf {
  unsigned long long* buf;  // pairs (time in ns, id << 8 | phase)
  unsigned int* pos;
  unsigned int cap;
};
#ifdef __CUDACC__
static __device__ TraceBuf g_trace;
__device__ __forceinline__ void trace_mark(int id, int phase) {
  if (g_trace.buf) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const unsigned int i = atomicAdd(g_trace.pos, 1u);
    if (i < g_trace.cap) {
      g_trace.buf[2 * i] = t;
      g_trace.buf[2 * i + 1] = ((unsigned long long)id << 8) | (unsigned)phase;
    }
  }
}
#endif
int trace_set_potrf(TraceBuf tb);
int trace_set_tc(TraceBuf tb);


void set_error(const char* fmt, ...);
void count_launch();

// RAII event pair around one launch (active only while gpk_prof_enable(1))
struct ProfScope {
  int idx;
  cudaStream_t st;
  ProfScope(int cls, cudaStream_t s, double work = 0.0);  // work: operations ISSUED by the launch (class-specific unit)
  ~ProfScope();
};
// PROF_GEMM: DMMA / SIMT GEMMs, PROF_TC: tcgen05 kernels (work = int8 or tf32 MACs issued), PROF_PANEL: potrf_panel_kernel
enum { PROF_KBUILD = 0, PROF_GEMM = 1, PROF_LEAF = 2, PROF_SKINNY = 3, PROF_MISC = 4, PROF_TC = 5, PROF_PANEL = 6, PROF_NCLS = 8 };

#define GPK_CHECK_ARG(cond, ...)        \
  do {                                  \
    if (!(cond)) {                      \
      gpk::set_error(__VA_ARGS__);      \
      return -1;                        \
    }                                   \
  } while (0)

#define GPK_CUDA_OK(expr)                                                                  \
  do {                                                                                     \
    cudaError_t e__ = (expr);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      gpk::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__,    \
                     __LINE__);                                                            \
      return -2;                                                                           \
    }                                                                                      \
  } while (0)

#define GPK_LAUNCH_OK()                                                                    \
  do {                                                                                     \
    cudaError_t e__ = cudaGetLastError();                                                  \
    gpk::count_launch();                                                                   \
    if (e__ != cudaSuccess) {                                                              \
      gpk::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, \
                     __LINE__);                                                            \
      return -2;                                                                           \
    }                                                                                      \
  } while (0)

#define GPK_TRY(expr)         \
  do {                        \
    int r__ = (expr);         \
    if (r__ != 0) return r__; \
  } while (0)

// One-time setup that belongs to a DEVICE (constant-memory tables, cudaFuncSetAttribute, occupancy queries): runs
// `f` once per device under a lock, so a process that drives several GPUs initialises each of them.
class PerDeviceOnce {
  std::mutex mu_;
  std::vector<char> done_;

 public:
  template <class F>
  int run(F&& f) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -2;
    std::lock_guard<std::mutex> lk(mu_);
    if ((int)done_.size() <= dev) done_.resize(dev + 1, 0);
    if (done_[dev]) return 0;
    const int rc = f();
    if (rc == 0) done_[dev] = 1;
    return rc;
  }
};

inline size_t dtype_size(int dtype) { return dtype == GPK_F64 ? 8 : 4; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

constexpr int NB = 128;  // Cholesky / TRSM leaf block

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Head-first launch option for the Cholesky look-ahead: tiles of the first 128-column block of C are
// processed first and each one increments *head_flag (release) when its stores are done, so the
// next diagonal-block factorisation (spinning on the flag on a second stream) overlaps the rest.
struct GemmOpts {
  int* head_flag = nullptr;
};
// head_flag[1] counts the finished part of C's leading 128x128 block in 32x32 units, so kernels with
// different tile shapes publish comparable progress; the waiting leaf needs diag_units_total(m, n).
__host__ __device__ inline int diag_units_total(long long m, long long n) {
  const long long a = m < 128 ? m : 128, b = n < 128 ? n : 128;
  return (int)(((a + 31) / 32) * ((b + 31) / 32));
}
__device__ inline int diag_units_tile(long long m0, long long n0, int bm, int bn, long long m, long long n) {
  if (m0 >= 128 || n0 >= 128) return 0;
  const long long a = (m < 128 ? m : 128) - m0, b = (n < 128 ? n : 128) - n0;
  const long long ra = a < bm ? a : bm, rb = b < bn ? b : bn;
  if (ra <= 0 || rb <= 0) return 0;
  return (int)(((ra + 31) / 32) * ((rb + 31) / 32));
}

// Internal (typed, unchecked) entry points shared between translation units.
template <typename T>
int gemm_t(int transa, int transb, int64_t m, int64_t n, int64_t k, T alpha, const T* A, int64_t lda,
           const T* B, int64_t ldb, T beta, T* C, int64_t ldc, int flags, cudaStream_t st,
           const GemmOpts* opts = nullptr);

template <typename T>
int potrf_t(T* A, int64_t n, int64_t rows, int64_t lda, int32_t* info, T* dinv, void* tcws, size_t tcws_bytes,
            cudaStream_t st, bool need_dinv = true, double cond_hint = 0.0);

// workspace of the tcgen05 (int8-sliced fp64) trailing updates and of the fp64 detour of fp32 factorisations, potrf.cu
size_t potrf_tc_ws_bytes(int64_t n, int64_t rows, int dtype);

// tcgen05 kind::tf32 (3xTF32) fp32 GEMM, gemm_tf32.cu
bool gemm_tf32_eligible(int64_t m, int64_t n, int64_t k, const void* A, const void* B, const void* C, int flags);
int gemm_tf32(int transa, int transb, int64_t m, int64_t n, int64_t k, float alpha, const float* A, int64_t lda,
              const float* B, int64_t ldb, float beta, float* C, int64_t ldc, int flags, cudaStream_t st, int batch = 1,
              int64_t a_batch_stride = 0, int64_t c_batch_stride = 0);

template <typename T>
int trsm_t(int trans, const T* L, int64_t n, int64_t ldl, T* B, int64_t nrhs, int64_t ldb, const T* dinv,
           cudaStream_t st);

template <typename T>
int trtri_diag_t(const T* L, int64_t n, int64_t ldl, T* dinv, cudaStream_t st);

}  // namespace gpk
