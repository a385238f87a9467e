#include "launch.h"
#include "filter_tc.cuh"
namespace hy {

size_t filter_tc_wimg_bytes(int D) {
  const size_t a = tc::wimg_floats(D), b = tc::wimg_bwd_floats(D);
  return (a > b ? a : b) * sizeof(float);
}

cudaError_t launch_filter_bwd_tc(const FilterParams& P, float* wimg, const float* dk, float* dh, float* scratch,
                                 cudaStream_t s) {
  cudaError_t e = set_smem(tc::filter_tc_bwd_kernel, tc::kSmemBytes);
  if (e != cudaSuccess) return e;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  prof_begin(K_FILTER_TC_PREP, s);
  tc::filter_tc_prep_bwd_kernel<<<64, 256, 0, s>>>(P.W1, P.W2, P.W3, P.D, wimg);
  prof_end(K_FILTER_TC_PREP, s);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const int ntiles = (P.L + tc::kTileM - 1) / tc::kTileM;
  const int grid = ntiles < sms ? ntiles : sms;
  prof_begin(K_FILTER_TC_BWD, s);
  tc::filter_tc_bwd_kernel<<<grid, tc::kThreads, tc::kSmemBytes, s>>>(P, wimg, dk, dh, scratch, ntiles);
  prof_end(K_FILTER_TC_BWD, s);
  return cudaGetLastError();
}

cudaError_t launch_filter_fwd_tc(const FilterParams& P, float* wimg, float* kout, cudaStream_t s) {
  cudaError_t e = set_smem(tc::filter_tc_fwd_kernel, tc::kSmemBytes);
  if (e != cudaSuccess) return e;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  prof_begin(K_FILTER_TC_PREP, s);
  tc::filter_tc_prep_kernel<<<64, 256, 0, s>>>(P.W1, P.W2, P.W3, P.D, wimg);
  prof_end(K_FILTER_TC_PREP, s);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const int ntiles = (P.L + tc::kTileM - 1) / tc::kTileM;
  if (P.D <= 256) {   // TS form: activations in tensor memory, weights resident, two tiles in flight
    const size_t smem = tc::fwd2_smem_bytes(P.D);
    e = set_smem(tc::filter_tc_fwd2_kernel, smem);
    if (e != cudaSuccess) return e;
    const int pairs = (ntiles + 1) / 2;
    const int grid2 = pairs < sms ? pairs : sms;
    prof_begin(K_FILTER_TC_FWD, s);
    tc::filter_tc_fwd2_kernel<<<grid2, tc::kThreads, smem, s>>>(P, wimg, kout, ntiles);
    prof_end(K_FILTER_TC_FWD, s);
    return cudaGetLastError();
  }
  const int grid = ntiles < sms ? ntiles : sms;
  prof_begin(K_FILTER_TC_FWD, s);
  tc::filter_tc_fwd_kernel<<<grid, tc::kThreads, tc::kSmemBytes, s>>>(P, wimg, kout, ntiles);
  prof_end(K_FILTER_TC_FWD, s);
  return cudaGetLastError();
}

cudaError_t launch_filter_red_tc(const RedLaunch& r, cudaStream_t s) {
  cudaError_t e = set_smem(tc::filter_tc_red_kernel, tc::kRedSmemBytes);
  if (e != cudaSuccess) return e;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  tc::RedArgs R{r.dh, r.scratch, r.zT, r.dW0, r.db0, r.dW1, r.db1, r.dW2, r.db2, r.dW3, r.dfreq, r.L, r.D, r.E};
  const int nblocks = (r.L + tc::kRedKB - 1) / tc::kRedKB;
  const int grid = nblocks < sms ? nblocks : sms;
  prof_begin(K_FILTER_TC_RED, s);
  tc::filter_tc_red_kernel<<<grid, tc::kRedThreads, tc::kRedSmemBytes, s>>>(R, nblocks);
  prof_end(K_FILTER_TC_RED, s);
  return cudaGetLastError();
}

}  // namespace hy
