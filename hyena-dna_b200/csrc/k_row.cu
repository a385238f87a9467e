#include <cstdint>

#include "launch.h"
namespace hy {

// batch-1 backward with cp.async-staged k / g spectrum rows (fft_passes.cuh row_bwd1_staged_body)
template <int LOGM2>
__global__ void __launch_bounds__(128, 2) row_pass_bwd1_staged_kernel(const PassArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  row_bwd1_staged_body<LOGM2>(a, blockIdx.x, blockIdx.y, smem_raw);
}

// forward row pass with the cp.async-staged filter spectrum row (fft_passes.cuh row_fwd_staged_body)
template <int LOGM2>
__global__ void __launch_bounds__(128, 3) row_pass_fwd_staged_kernel(const PassArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  row_fwd_staged_body<LOGM2>(a, blockIdx.x, blockIdx.y, smem_raw);
}

static cudaError_t go_fwd_staged(const PassArgs& a, int rows, cudaStream_t s) {
  using RG = RowGeo<10>;
  const int M1 = 1 << a.logM1;
  const int rows_cta = RG::ROWS >= 4 ? RG::ROWS / 2 : RG::ROWS;
  const int nslots = M1 < rows_cta ? M1 : rows_cta;
  const int ctas = M1 < rows_cta ? 1 : M1 / rows_cta;
  const size_t smem = row_fwd_staged_smem_elems<10>(nslots) * sizeof(float2);
  auto kern = row_pass_fwd_staged_kernel<10>;
  cudaError_t e = set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  prof_begin(K_ROW + (int)ROW_CONV_FWD, s);
  kern<<<dim3(ctas, rows), nslots * RG::TPR, smem, s>>>(a);
  prof_end(K_ROW + (int)ROW_CONV_FWD, s);
  return cudaGetLastError();
}

static cudaError_t go_bwd1_staged(const PassArgs& a, int rows, cudaStream_t s) {
  using RG = RowGeo<10>;
  const int M1 = 1 << a.logM1;
  const int rows_cta = RG::ROWS >= 4 ? RG::ROWS / 2 : RG::ROWS;
  const int nslots = M1 < rows_cta ? M1 : rows_cta;
  const int ctas = M1 < rows_cta ? 1 : M1 / rows_cta;
  const size_t smem = row_bwd1_staged_smem_elems<10>(nslots) * sizeof(float2);
  auto kern = row_pass_bwd1_staged_kernel<10>;
  cudaError_t e = set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  prof_begin(K_ROW + (int)ROW_CONV_BWD, s);
  kern<<<dim3(ctas, rows), nslots * RG::TPR, smem, s>>>(a);
  prof_end(K_ROW + (int)ROW_CONV_BWD, s);
  return cudaGetLastError();
}

template <int MODE, int LOGM2>
static cudaError_t go(const PassArgs& a, int rows, cudaStream_t s) {
  using RG = RowGeo<LOGM2>;
  const int M1 = 1 << a.logM1;
  const int nslots = M1 < RG::ROWS ? M1 : RG::ROWS;
  const int ctas = M1 < RG::ROWS ? 1 : M1 / RG::ROWS;
  const size_t smem = row_smem_elems<MODE, LOGM2>(nslots) * sizeof(float2);
  auto kern = row_pass_kernel<MODE, LOGM2>;
  cudaError_t e = set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  prof_begin(K_ROW + MODE, s);
  kern<<<dim3(ctas, rows), nslots * RG::TPR, smem, s>>>(a);
  prof_end(K_ROW + MODE, s);
  return cudaGetLastError();
}

template <int MODE>
static cudaError_t by_len(const PassArgs& a, int rows, cudaStream_t s) {
  if (a.logM2 == 10) return go<MODE, 10>(a, rows, s);
  return cudaErrorInvalidValue;
}

cudaError_t launch_row_pass(int mode, const PassArgs& a, int rows, cudaStream_t s) {
  switch (mode) {
    case ROW_FILTER: return by_len<ROW_FILTER>(a, rows, s);
    case ROW_CONV_FWD: {
      const bool al16 = (reinterpret_cast<uintptr_t>(a.kspec) & 15u) == 0;
      if (al16 && a.logM1 >= 2) return go_fwd_staged(a, rows, s);
      return by_len<ROW_CONV_FWD>(a, rows, s);
    }
    case ROW_CONV_BWD: {
      // batch 1 with the g spectrum saved by the forward pass: the staged kernel, no accumulator across the batch
      const bool al16 = ((reinterpret_cast<uintptr_t>(a.kspec) | reinterpret_cast<uintptr_t>(a.gspec)) & 15u) == 0;
      if (a.B == 1 && a.gspec && al16) return go_bwd1_staged(a, rows, s);
      return by_len<ROW_CONV_BWD>(a, rows, s);
    }
  }
  return cudaErrorInvalidValue;
}

}  // namespace hy
