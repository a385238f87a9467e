#include "launch.h"
#include "filter_extra.cuh"
#include "short_conv.cuh"
namespace hy {

// fp64 sincospi -> fp32 twiddle tables (exact argument reduction, correctly rounded to ~0.5 ulp)
__global__ void twiddle_init_kernel(float2* tw1024, float2* twlo) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < 1024) {
    double s, c;
    sincospi(-2.0 * (double)j / 1024.0, &s, &c);
    tw1024[j] = make_float2((float)c, (float)s);
    sincospi(-2.0 * (double)j / 1048576.0, &s, &c);
    twlo[j] = make_float2((float)c, (float)s);
  }
}

cudaError_t launch_twiddle_init(float2* tw1024, float2* twlo, cudaStream_t s) {
  prof_begin(K_TWIDDLE, s);
  twiddle_init_kernel<<<4, 256, 0, s>>>(tw1024, twlo);
  prof_end(K_TWIDDLE, s);
  return cudaGetLastError();
}

cudaError_t launch_short_bwd(const ShortBwdArgs& a, int B, cudaStream_t s) {
  dim3 grid((a.L + kScSpan - 1) / kScSpan, a.C3, B);
  prof_begin(K_SHORT_BWD, s);
  short_conv_bwd_kernel<<<grid, 256, 0, s>>>(a);
  prof_end(K_SHORT_BWD, s);
  return cudaGetLastError();
}

// ---- filter_extra.cuh: deltas gradient (modulation_lr != 0) and the L1 normalisation over channels (normalized=True)
cudaError_t launch_filter_ddelta(const float* dk, const float* k, const float* t, const float* deltas, float shift, int D,
                                 int L, float* ddelta, cudaStream_t s) {
  prof_begin(K_FILTER_EXTRA, s);
  fx::filter_ddelta_kernel<<<D, 256, 0, s>>>(dk, k, t, deltas, shift, L, ddelta);
  prof_end(K_FILTER_EXTRA, s);
  return cudaGetLastError();
}
cudaError_t launch_l1norm_fwd(const float* k, float* out, float* norm, int D, int L, cudaStream_t s) {
  prof_begin(K_FILTER_EXTRA, s);
  fx::l1norm_fwd_kernel<<<(L + 255) / 256, 256, 0, s>>>(k, out, norm, D, L);
  prof_end(K_FILTER_EXTRA, s);
  return cudaGetLastError();
}
cudaError_t launch_l1norm_bwd(const float* dout, const float* out, const float* norm, float* dk, int D, int L, cudaStream_t s) {
  prof_begin(K_FILTER_EXTRA, s);
  fx::l1norm_bwd_kernel<<<(L + 255) / 256, 256, 0, s>>>(dout, out, norm, dk, D, L);
  prof_end(K_FILTER_EXTRA, s);
  return cudaGetLastError();
}

}  // namespace hy
