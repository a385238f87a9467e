// Backward of the 3-tap depthwise short filter (src/models/sequence/hyena.py:363-369, :394).
//
// Forward (fused into the FFT column passes): s[t] = w0 P(t-2) + w1 P(t-1) + w2 P(t) + b for t in [0,L),
// P(t) = p[t] + in_bias inside [0,L) and 0 outside (p = in_proj output before its bias).
// Backward, given ds = d loss / d s  (B,3D,L):
//   dp[t]  = w2 ds[t] + w1 ds[t+1] + w0 ds[t+2]          (ds[t>=L] = 0)
//   dw_j   = sum_{b,t} ds[t] P(t-2+j),  db = sum ds,  d in_bias = sum dp
#pragma once
#include "launch.h"

namespace hy {

constexpr int kScSpan = 8192;     // positions per CTA

__global__ void __launch_bounds__(256) short_conv_bwd_kernel(const ShortBwdArgs a) {
  const int ch = blockIdx.y, b = blockIdx.z;
  const int L = a.L;
  const bool vec = a.vec;
  const float* ds = a.ds + row_off(b, ch, a.C3, L);
  const float* p = a.p ? a.p + row_off(b, ch, a.C3, L) : nullptr;
  float* dp = a.dp + row_off(b, ch, a.C3, L);
  const float w0 = __ldg(a.sw + 3 * ch), w1 = __ldg(a.sw + 3 * ch + 1), w2 = __ldg(a.sw + 3 * ch + 2);
  const float ib = a.in_bias ? __ldg(a.in_bias + ch) : 0.f;
  float r[5] = {0.f, 0.f, 0.f, 0.f, 0.f};      // dw0, dw1, dw2, db, dib
  const int tbeg = blockIdx.x * kScSpan;
  const int tend = min(L, tbeg + kScSpan);
  for (int t0 = tbeg + 2 * threadIdx.x; t0 < tend; t0 += 512) {
    float2 d0 = load_pair(ds, t0, L, vec);
    float2 d1 = (t0 + 2 < L) ? load_pair(ds, t0 + 2, L, vec) : make_float2(0.f, 0.f);
    float2 o;
    o.x = fmaf(w2, d0.x, fmaf(w1, d0.y, w0 * d1.x));
    o.y = fmaf(w2, d0.y, fmaf(w1, d1.x, w0 * d1.y));
    store_pair(dp, t0, L, vec, o);
    if (a.p) {
      float P[4];
      load_window(p, t0, L, vec, ib, P);
      r[0] = fmaf(d0.x, P[0], fmaf(d0.y, P[1], r[0]));
      r[1] = fmaf(d0.x, P[1], fmaf(d0.y, P[2], r[1]));
      r[2] = fmaf(d0.x, P[2], fmaf(d0.y, P[3], r[2]));
      r[3] += d0.x + d0.y;
    }
    r[4] += o.x + ((t0 + 1 < L) ? o.y : 0.f);
  }
  __shared__ float red[8][5];
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    float s = r[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][j] = s;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
    if (threadIdx.x < 3) { if (a.p) atomicAdd(a.dsw + 3 * ch + threadIdx.x, s); }
    else if (threadIdx.x == 3) { if (a.p) atomicAdd(a.dsb + ch, s); }
    else if (a.dib) atomicAdd(a.dib + ch, s);
  }
}

}  // namespace hy
