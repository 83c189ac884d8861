// b2s_trees3.cu -- the round-2 tree kernels (b2s_trees3.cuh) in their own translation unit, behind three launchers.
#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>

#include "b2s_rowthread.cuh"  // mbarrier / TMA helpers
#define B2S_T3_KERNELS
#include "b2s_trees3.cuh"

namespace b2s {

cudaError_t t3_launch_prep(const T3Prep& pr, const CUtensorMap& tmap, bool miss, int grid, int smem, int smem_optin, cudaStream_t st) {
  static std::atomic<bool> attr{false};
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(t3_prep_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(t3_prep_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  if (miss) t3_prep_kernel<true><<<grid, kT3PrepThreads, smem, st>>>(pr, tmap);
  else t3_prep_kernel<false><<<grid, kT3PrepThreads, smem, st>>>(pr, tmap);
  return cudaGetLastError();
}

template <int D, bool MISS>
static cudaError_t walk(const T3Params& t, int grid, int block, int smem, int smem_optin, cudaStream_t st) {
  static std::atomic<bool> attr{false};
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(trees3_kernel<D, MISS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  trees3_kernel<D, MISS><<<grid, block, smem, st>>>(t);
  return cudaGetLastError();
}

cudaError_t t3_launch_walk(const T3Params& t, int depth, bool miss, int grid, int block, int smem, int smem_optin, cudaStream_t st) {
#define B2S_T3_CASE(DD) \
  if (depth == DD) return miss ? walk<DD, true>(t, grid, block, smem, smem_optin, st) : walk<DD, false>(t, grid, block, smem, smem_optin, st);
  B2S_T3_CASE(2) B2S_T3_CASE(3) B2S_T3_CASE(4) B2S_T3_CASE(5) B2S_T3_CASE(6) B2S_T3_CASE(7) B2S_T3_CASE(8)
#undef B2S_T3_CASE
  return cudaErrorInvalidValue;
}

cudaError_t t3_launch_vote(const KParams& k, const double* partial, int64_t col_stride, const int32_t* col_score, int n_cols,
                           const int32_t* row_bad, int grid, cudaStream_t st) {
  t3_vote_kernel<<<grid, 256, 0, st>>>(k, partial, col_stride, col_score, n_cols, row_bad);
  return cudaGetLastError();
}

}  // namespace b2s
