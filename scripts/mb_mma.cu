// mb_mma.cu — issue-rate probe for tcgen05.mma kind::i8 (M = 128) on one SM: cycles per MMA as a function of N,
// operand source (A from shared memory / from TMEM) and with / without the tcgen05.cp of the A planes.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -I gpflow_b200/csrc -o scripts/mb_mma.bin scripts/mb_mma.cu
#include "tc_common.cuh"
#include <stdlib.h>

namespace gpk {
void set_error(const char*, ...) {}
void count_launch() {}
}  // namespace gpk
using namespace gpk;

// TS form: A operand read from TMEM (written there by tcgen05.cp), B from shared memory
__device__ __forceinline__ void tc_mma_i8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}
// shared memory (matrix descriptor) -> TMEM, 128 lanes x 256 bits (32 bytes per row = one K=32 int8 step)
__device__ __forceinline__ void tc_cp_128x256b(uint32_t d_tmem, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(d_tmem), "l"(sdesc) : "memory");
}

__host__ __device__ constexpr uint32_t idesc_n(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// mode 0: SS, `nm` MMAs of width N per round.   mode 1: TS (A in TMEM), same.   mode 2: TS + 7 tcgen05.cp per round.
template <int N, int MODE>
__global__ void __launch_bounds__(128, 1) k_mma(long long* out, int rounds, int nm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 96 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x01010101u;
  if (threadIdx.x == 0) { mbar_init(smem_u32(&bar), 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  if (warp == 0) tmem_alloc(smem_u32(&slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = slot;
  if (warp == 0) {
    const uint64_t hi = ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46);
    const uint32_t sa = smem_u32(smem);
    const uint64_t ad = hi | (uint64_t)((sa & 0x3FFFFu) >> 4);
    const uint64_t bd = ad + (32768 >> 4);
    long long t0 = clock64();
    for (int r = 0; r < rounds; ++r) {
      if (elect_one()) {
        if (MODE == 2)
          for (int s = 0; s < 7; ++s) tc_cp_128x256b(tm + 448 + s * 8, ad + (uint64_t)(s * 256));
        for (int i = 0; i < nm; ++i) {
          constexpr int slots = (MODE == 0 ? 512 : 448) / N;
          const uint32_t d = tm + (uint32_t)((i % slots) * N);
          if (MODE == 0) tc_mma_i8(d, ad + (uint64_t)((i % 7) * 256), bd + (uint64_t)((i % 4) * 128), idesc_n(N), 1u);
          else tc_mma_i8_ts(d, tm + 448 + (i % 7) * 8, bd + (uint64_t)((i % 4) * 128), idesc_n(N), 1u);
        }
      }
      __syncwarp();
    }
    if (elect_one()) tc_commit(smem_u32(&bar));
    __syncwarp();
    mbar_wait(smem_u32(&bar), 0, nullptr, 1);
    long long t1 = clock64();
    if (threadIdx.x == 0) out[blockIdx.x] = t1 - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, 512);
}

template <int N, int MODE>
static void run(const char* name, int nm, int grid) {
  long long* d;
  cudaMalloc(&d, 1024 * sizeof(long long));
  auto k = k_mma<N, MODE>;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  const int rounds = 2000;
  k<<<grid, 128, 96 * 1024>>>(d, 10, nm);
  k<<<grid, 128, 96 * 1024>>>(d, rounds, nm);
  cudaError_t e = cudaDeviceSynchronize();
  long long h[1024];
  cudaMemcpy(h, d, grid * sizeof(long long), cudaMemcpyDeviceToHost);
  long long mx = 0;
  for (int i = 0; i < grid; ++i) mx = h[i] > mx ? h[i] : mx;
  const double per_round = (double)mx / rounds;
  printf("%-28s grid %3d  N=%3d  %2d MMA/round: %8.1f cyc/round  %6.1f cyc/MMA  (floor %5.1f)  MAC-cols/cyc %.2f  %s\n", name,
         grid, N, nm, per_round, per_round / nm, 128.0 * N / 256.0, (double)nm * N / per_round, cudaGetErrorString(e));
  cudaFree(d);
}

int main() {
  for (int grid : {1, 148}) {
    run<64, 0>("SS N=64 x28", 28, grid);
    run<128, 0>("SS N=128 x14", 14, grid);
    run<256, 0>("SS N=256 x7", 7, grid);
    run<64, 1>("TS N=64 x28", 28, grid);
    run<128, 1>("TS N=128 x14", 14, grid);
    run<256, 1>("TS N=256 x7", 7, grid);
    run<64, 2>("TS+cp N=64 x28", 28, grid);
    run<256, 2>("TS+cp N=256 x7", 7, grid);
  }
  return 0;
}
