// Host-side launch entry points implemented in the k_*.cu translation units.
#pragma once
#include "fft_passes.cuh"
#include "filter_params.h"
#include "layernorm_args.h"

namespace hy {

// kernel classes for the launch counter / per-launch event timing (api.cu)
enum Kind {
  K_COL_FWD = 0,      // + ColMode  (0..3)
  K_COL_INV = 4,      // + InvMode  (4..8)
  K_ROW = 9,          // + RowMode  (9..11)
  K_SHORT_BWD = 12, K_TWIDDLE = 13, K_FILTER_TC_PREP = 14, K_FILTER_TC_FWD = 15, K_FILTER_TC_BWD = 16, K_FILTER_TC_RED = 17,
  K_CONVERT = 18, K_PROJ_PREP = 19, K_PROJ_GEMM = 20, K_PROJ_WGRAD = 21,
  K_ADD_LN = 22,            // residual add + LayerNorm (block glue, layernorm.cuh)
  K_FILTER_EXTRA = 23,      // deltas gradient / channel L1 normalisation (filter_extra.cuh; non-default filter options)
  K_DECODE_PREFILL = 24, K_DECODE_STEP_CONV = 25, K_DECODE_STEP_REDUCE = 26, K_DECODE_STEP_OUT = 27,   // k_decode.cu
  K_COUNT = 28
};
void prof_begin(int kind, cudaStream_t s);     // api.cu: records an event when profiling is on
void prof_end(int kind, cudaStream_t s);       // api.cu: records an event when profiling is on; counts the launch
cudaError_t launch_col_fwd(int mode, const PassArgs& a, int rows, cudaStream_t s);
cudaError_t launch_col_inv(int mode, const PassArgs& a, int rows, cudaStream_t s);
cudaError_t launch_row_pass(int mode, const PassArgs& a, int rows, cudaStream_t s);
template <int MODE> cudaError_t launch_col_fwd_mode(const PassArgs& a, int rows, cudaStream_t s);   // k_col_fwd_m*.cu
template <int MODE> cudaError_t launch_col_inv_mode(const PassArgs& a, int rows, cudaStream_t s);   // k_col_inv_m*.cu
cudaError_t launch_filter_fwd_tc(const FilterParams& P, float* wimg, float* kout, cudaStream_t s);   // k_filter_tc.cu
size_t filter_tc_wimg_bytes(int D);
cudaError_t launch_filter_bwd_tc(const FilterParams& P, float* wimg, const float* dk, float* dh, float* scratch, cudaStream_t s);
struct RedLaunch { const float* dh; const float* scratch; const float* zT; float* dW0; float* db0; float* dW1; float* db1;
                   float* dW2; float* db2; float* dW3; float* dfreq; int L, D, E; };
cudaError_t launch_filter_red_tc(const RedLaunch& r, cudaStream_t s);   // k_filter_tc.cu
// k_filter.cu: backward of the 3-tap short filter (short_conv.cuh)
struct ShortBwdArgs {
  const float* ds;      // (B,3D,L)
  const float* p;       // (B,3D,L), or null when dsw / dsb were already accumulated by pass 3
  const float* in_bias; // (3D) or null
  const float* sw;      // (3D,3)
  float* dp;            // (B,3D,L)
  float* dsw;           // (3D,3)  atomicAdd
  float* dsb;           // (3D)    atomicAdd
  float* dib;           // (3D)    atomicAdd (d in_proj.bias) or null
  int L, C3, vec;
};
cudaError_t launch_short_bwd(const ShortBwdArgs& a, int B, cudaStream_t s);
cudaError_t launch_twiddle_init(float2* tw1024, float2* twlo, cudaStream_t s);
// k_proj.cu: projection GEMMs on tcgen05 (3xTF32)
size_t proj_wimg_bytes(int N, int K);
cudaError_t launch_proj_gemm(const float* act, int act_layout, const float* W, int ldw, int w_transposed, const float* bias,
                             const float* fir, float* out, int out_layout, int B, int L, int K, int N, int l0, int ln,
                             float* wimg, cudaStream_t s);
size_t proj_wgrad_scratch_bytes(int M, int N);
cudaError_t launch_proj_wgrad(const float* X, const float* Y, const float* fir, float* dW, int transposed_out, float beta,
                              int B, int L, int M, int N, float* part, cudaStream_t s);
// k_filter.cu: filter_extra.cuh
cudaError_t launch_filter_ddelta(const float* dk, const float* k, const float* t, const float* deltas, float shift, int D,
                                 int L, float* ddelta, cudaStream_t s);
cudaError_t launch_l1norm_fwd(const float* k, float* out, float* norm, int D, int L, cudaStream_t s);
cudaError_t launch_l1norm_bwd(const float* dout, const float* out, const float* norm, float* dk, int D, int L, cudaStream_t s);
// k_layernorm.cu: residual add + LayerNorm (block glue)
int ln_partials(long long rows);                     // CTAs (= rows of the dw/db partial scratch) the kernels use for `rows`
cudaError_t launch_add_ln_fwd(const ln::FwdArgs& a, cudaStream_t s);
cudaError_t launch_add_ln_bwd(ln::BwdArgs a, float* dw, float* db, cudaStream_t s);
// k_convert.cu: reference filter-spectrum convention (rfft(k, fft_size), natural order) <-> packed spectrum
cudaError_t launch_rfft_to_packed(const float2* X, float2* Z, int H, int logM, int logM1, cudaStream_t s);
cudaError_t launch_packed_to_rfft(const float2* Z, float2* X, int H, int logM, int logM1, float scale, cudaStream_t s);
cudaError_t launch_rfft_to_time_small(const float2* X, float* k, int H, int L, int N, cudaStream_t s);
cudaError_t launch_time_to_rfft_small(const float* x, float2* X, int H, int L, int N, float scale, cudaStream_t s);
// k_decode.cu: incremental decoding (prompt prefill, per-token step)
struct DecodeStep {
  const float* u; const float* W_in; const float* in_bias; const float* sw; const float* sb; const float* k;
  const float* fbias; const float* W_out; const float* out_bias; float* g_hist; float* fir; float* y;
  int B, D, t, max_len;
};
size_t decode_workspace_bytes(int B, int D, int max_len);
int decode_max_batch();
cudaError_t launch_decode_prefill(const float* p, const float* in_bias, const float* sw, const float* sb, float* g_hist,
                                  float* fir, int B, int D, int Lp, int max_len, cudaStream_t s);
cudaError_t launch_decode_step(const DecodeStep& d, void* workspace, cudaStream_t s);

template <class K>
inline cudaError_t set_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return cudaSuccess;
}

}  // namespace hy
