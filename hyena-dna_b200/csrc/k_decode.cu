// Incremental (token-by-token) decoding of the order-2 Hyena operator: prompt prefill and the per-token step.
//
// At position t, with P[t] = W_in u_t + in_bias (3D channels: x0, x1, v; hyena.py:391, :404):
//   s[t] = w0 P[t-2] + w1 P[t-1] + w2 P[t] + sb          depthwise Conv1d k=3, zero padding after the bias (:363-369)
//   g[t] = s_v[t] * s_x1[t]                                                                                  (:420)
//   c[t] = sum_{j=0..t} k[c][j] g[t-j] + fbias[c] g[t]     causal long convolution + skip term of fftconv_ref (:59-88)
//   y[t] = W_out (c[t] * s_x0[t]) + out_bias                                                            (:432-440)
//
// Decode state, per operator:
//   g_hist (B, D, max_len)  gated history g, channel-major (row stride max_len)
//   fir    (B, 3D, 2)       the biased in_proj outputs P[t-2], P[t-1] of every channel (zeros before the sequence)
//
// A step is three launches on the caller's stream, all fp32 FMAs on the CUDA cores (B rows are far too few for the tensor
// cores to pay off):
//   1. decode_step_conv   grid (history chunk, channel).  Every CTA streams its chunk of k[c] once and reuses each value
//                         for all batch rows of g_hist.  The CTA of chunk 0 also computes the new token: the three in_proj
//                         rows of its channel, the short filter, g_t (written to g_hist[t]) and x0_t, and shifts fir.  The
//                         other chunks read only g_hist[0, t), so nothing they read is written in the same launch.
//                         k is read forward and g backward, so their relative 16-byte alignment changes with t: both are
//                         read with coalesced scalar loads (a warp reads 32 consecutive floats of each), unrolled for
//                         enough loads in flight.  Partial sums go to the workspace; no atomics.
//   2. decode_step_reduce sums the partials of every (b, c) in chunk order, adds the skip term, applies the x0 gate.
//   3. decode_step_out    out_proj GEMV plus bias, one warp per output feature.
#include "launch.h"

namespace hy {

constexpr int kDecThreads = 256;
constexpr int kDecUnroll = 8;
constexpr int kDecChunk = 8192;            // history positions per CTA of decode_step_conv
constexpr int kDecMaxB = 64;               // batch rows a step handles (smem of the chunk-0 CTA)
static_assert(kDecChunk % (kDecThreads * kDecUnroll) == 0, "a chunk is whole unrolled sweeps");

static int dec_chunks(int n) { return (n + kDecChunk - 1) / kDecChunk; }

// ---------------------------------------------------------------- prefill
// g_hist[b][c][t] for t < Lp from the prompt's p (B, 3D, Lp) (without in_bias), and fir from its last two positions.
__global__ void __launch_bounds__(256) decode_prefill_kernel(const float* __restrict__ p, const float* __restrict__ in_bias,
                                                             const float* __restrict__ sw, const float* __restrict__ sb,
                                                             float* __restrict__ g_hist, float* __restrict__ fir, int D, int Lp,
                                                             int max_len) {
  const int c = blockIdx.y, b = blockIdx.z;
  const int C3 = 3 * D;
  const float* p1 = p + ((size_t)b * C3 + D + c) * Lp;
  const float* pv = p + ((size_t)b * C3 + 2 * D + c) * Lp;
  const float ib1 = in_bias ? __ldg(in_bias + D + c) : 0.f, ibv = in_bias ? __ldg(in_bias + 2 * D + c) : 0.f;
  const float a0 = __ldg(sw + 3 * (D + c)), a1 = __ldg(sw + 3 * (D + c) + 1), a2 = __ldg(sw + 3 * (D + c) + 2);
  const float v0 = __ldg(sw + 3 * (2 * D + c)), v1 = __ldg(sw + 3 * (2 * D + c) + 1), v2 = __ldg(sw + 3 * (2 * D + c) + 2);
  const float sb1 = __ldg(sb + D + c), sbv = __ldg(sb + 2 * D + c);
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < Lp) {
    auto P = [&](const float* row, float ib, int i) { return i >= 0 ? __ldg(row + i) + ib : 0.f; };
    const float s1 = fmaf(a0, P(p1, ib1, t - 2), fmaf(a1, P(p1, ib1, t - 1), fmaf(a2, P(p1, ib1, t), sb1)));
    const float sv = fmaf(v0, P(pv, ibv, t - 2), fmaf(v1, P(pv, ibv, t - 1), fmaf(v2, P(pv, ibv, t), sbv)));
    g_hist[((size_t)b * D + c) * max_len + t] = sv * s1;
  }
  if (blockIdx.x == 0 && threadIdx.x < 6) {      // fir[b][r*D + c][q] = P[Lp - 2 + q] of channel r*D + c
    const int r = threadIdx.x >> 1, q = threadIdx.x & 1, i = Lp - 2 + q;
    const int ch = r * D + c;
    const float ib = in_bias ? __ldg(in_bias + ch) : 0.f;
    fir[((size_t)b * C3 + ch) * 2 + q] = i >= 0 ? __ldg(p + ((size_t)b * C3 + ch) * Lp + i) + ib : 0.f;
  }
}

// ---------------------------------------------------------------- step 1: new token + chunked causal dot products
struct StepArgs {
  const float* u;        // (B, D)
  const float* W_in;     // (3D, D)
  const float* in_bias;  // (3D) or null
  const float* sw;       // (3D, 3)
  const float* sb;       // (3D)
  const float* k;        // (D, max_len)
  const float* fbias;    // (D)
  const float* W_out;    // (D, D)
  const float* out_bias; // (D) or null
  float* g_hist;         // (B, D, max_len)
  float* fir;            // (B, 3D, 2)
  float* y;              // (B, D)
  float* part;           // (chunks, B, D)
  float* x0;             // (B, D)
  float* ypre;           // (B, D)
  int B, D, t, max_len, chunks;
};

template <int NB>
__global__ void __launch_bounds__(kDecThreads) decode_step_conv_kernel(const StepArgs a) {
  const int chunk = blockIdx.x, c = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int B = a.B, D = a.D, t = a.t;
  __shared__ float Psm[3 * kDecMaxB];
  __shared__ float gsm[kDecMaxB];
  __shared__ float red[kDecThreads / 32][NB];

  if (chunk == 0) {
    // the new token: P = W_in[r*D + c] . u_b + in_bias, one warp per (r, b), fixed-order reduction
    for (int pr = warp; pr < 3 * B; pr += kDecThreads / 32) {
      const int r = pr / B, b = pr - r * B;
      const float* w = a.W_in + (size_t)(r * D + c) * D;
      const float* u = a.u + (size_t)b * D;
      float s = 0.f;
      for (int i = lane; i < D; i += 32) s = fmaf(__ldg(w + i), __ldg(u + i), s);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) Psm[pr] = s + (a.in_bias ? __ldg(a.in_bias + r * D + c) : 0.f);
    }
    __syncthreads();
    for (int b = tid; b < B; b += kDecThreads) {
      float s[3];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int ch = r * D + c;
        float* f = a.fir + ((size_t)b * 3 * D + ch) * 2;
        const float P = Psm[r * B + b], f0 = f[0], f1 = f[1];
        s[r] = fmaf(__ldg(a.sw + 3 * ch), f0, fmaf(__ldg(a.sw + 3 * ch + 1), f1, fmaf(__ldg(a.sw + 3 * ch + 2), P, __ldg(a.sb + ch))));
        f[0] = f1;
        f[1] = P;
      }
      const float g = s[2] * s[1];
      gsm[b] = g;
      a.g_hist[((size_t)b * D + c) * a.max_len + t] = g;
      a.x0[(size_t)b * D + c] = s[0];
    }
    __syncthreads();
  }

  // sum_{j in chunk, 1 <= j <= t} k[c][j] g[t - j]; the j = 0 term uses g_t from shared memory
  const float* kc = a.k + (size_t)c * a.max_len;
  const int j0 = chunk * kDecChunk;
  const int j1 = min(j0 + kDecChunk, t + 1);
  for (int b0 = 0; b0 < B; b0 += NB) {
    const int nb = min(NB, B - b0);
    float acc[NB];
#pragma unroll
    for (int i = 0; i < NB; ++i) acc[i] = 0.f;
    const float* grow = a.g_hist + ((size_t)b0 * D + c) * a.max_len + t;     // g[b0][c][t - j] = grow[-j]
    const size_t gstride = (size_t)D * a.max_len;
    for (int jb = j0; jb < j1; jb += kDecThreads * kDecUnroll) {
      float kv[kDecUnroll];
#pragma unroll
      for (int q = 0; q < kDecUnroll; ++q) {
        const int j = jb + q * kDecThreads + tid;
        kv[q] = (j >= 1 && j < j1) ? __ldg(kc + j) : 0.f;
      }
#pragma unroll
      for (int i = 0; i < NB; ++i) {
        if (i < nb) {
          float gv[kDecUnroll];
#pragma unroll
          for (int q = 0; q < kDecUnroll; ++q) {
            const int j = jb + q * kDecThreads + tid;
            gv[q] = (j >= 1 && j < j1) ? __ldg(grow + i * gstride - j) : 0.f;
          }
#pragma unroll
          for (int q = 0; q < kDecUnroll; ++q) acc[i] = fmaf(kv[q], gv[q], acc[i]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      float s = acc[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) red[warp][i] = s;
    }
    __syncthreads();
    if (tid < nb) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kDecThreads / 32; ++w) s += red[w][tid];
      if (chunk == 0) s = fmaf(__ldg(kc), gsm[b0 + tid], s);
      a.part[((size_t)chunk * B + b0 + tid) * D + c] = s;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- step 2: fixed-order chunk sum, skip term, x0 gate
__global__ void __launch_bounds__(256) decode_step_reduce_kernel(const StepArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;        // b * D + c
  if (i >= a.B * a.D) return;
  const int b = i / a.D, c = i - b * a.D;
  float s = 0.f;
  for (int ch = 0; ch < a.chunks; ++ch) s += a.part[(size_t)ch * a.B * a.D + i];
  const float g = a.g_hist[((size_t)b * a.D + c) * a.max_len + a.t];
  a.ypre[i] = fmaf(__ldg(a.fbias + c), g, s) * a.x0[i];
}

// ---------------------------------------------------------------- step 3: y = W_out y_pre + out_bias
__global__ void __launch_bounds__(256) decode_step_out_kernel(const StepArgs a) {
  constexpr int NB = 8;
  const int lane = threadIdx.x & 31;
  const int o = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (o >= a.D) return;
  const int D = a.D;
  const float* w = a.W_out + (size_t)o * D;
  const float ob = a.out_bias ? __ldg(a.out_bias + o) : 0.f;
  for (int b0 = 0; b0 < a.B; b0 += NB) {
    const int nb = min(NB, a.B - b0);
    float acc[NB];
#pragma unroll
    for (int i = 0; i < NB; ++i) acc[i] = 0.f;
    for (int c = lane; c < D; c += 32) {
      const float wv = __ldg(w + c);
#pragma unroll
      for (int i = 0; i < NB; ++i)
        if (i < nb) acc[i] = fmaf(wv, a.ypre[(size_t)(b0 + i) * D + c], acc[i]);
    }
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      float s = acc[i];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
      if (lane == 0 && i < nb) a.y[(size_t)(b0 + i) * D + o] = s + ob;
    }
  }
}

// ---------------------------------------------------------------- launchers
size_t decode_workspace_bytes(int B, int D, int max_len) {
  return ((size_t)dec_chunks(max_len) + 2) * (size_t)B * (size_t)D * sizeof(float);
}

int decode_max_batch() { return kDecMaxB; }

cudaError_t launch_decode_prefill(const float* p, const float* in_bias, const float* sw, const float* sb, float* g_hist,
                                  float* fir, int B, int D, int Lp, int max_len, cudaStream_t s) {
  prof_begin(K_DECODE_PREFILL, s);
  decode_prefill_kernel<<<dim3((Lp + 255) / 256, D, B), 256, 0, s>>>(p, in_bias, sw, sb, g_hist, fir, D, Lp, max_len);
  prof_end(K_DECODE_PREFILL, s);
  return cudaGetLastError();
}

cudaError_t launch_decode_step(const DecodeStep& d, void* workspace, cudaStream_t s) {
  StepArgs a;
  a.u = d.u; a.W_in = d.W_in; a.in_bias = d.in_bias; a.sw = d.sw; a.sb = d.sb; a.k = d.k; a.fbias = d.fbias;
  a.W_out = d.W_out; a.out_bias = d.out_bias; a.g_hist = d.g_hist; a.fir = d.fir; a.y = d.y;
  a.B = d.B; a.D = d.D; a.t = d.t; a.max_len = d.max_len;
  a.chunks = dec_chunks(d.t + 1);
  float* ws = reinterpret_cast<float*>(workspace);
  const size_t bd = (size_t)d.B * d.D;
  a.part = ws;
  a.x0 = ws + (size_t)dec_chunks(d.max_len) * bd;
  a.ypre = a.x0 + bd;
  const dim3 grid(a.chunks, d.D);
  prof_begin(K_DECODE_STEP_CONV, s);
  if (d.B <= 1) decode_step_conv_kernel<1><<<grid, kDecThreads, 0, s>>>(a);
  else if (d.B <= 2) decode_step_conv_kernel<2><<<grid, kDecThreads, 0, s>>>(a);
  else if (d.B <= 4) decode_step_conv_kernel<4><<<grid, kDecThreads, 0, s>>>(a);
  else decode_step_conv_kernel<8><<<grid, kDecThreads, 0, s>>>(a);
  prof_end(K_DECODE_STEP_CONV, s);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  prof_begin(K_DECODE_STEP_REDUCE, s);
  decode_step_reduce_kernel<<<(unsigned)((bd + 255) / 256), 256, 0, s>>>(a);
  prof_end(K_DECODE_STEP_REDUCE, s);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  prof_begin(K_DECODE_STEP_OUT, s);
  decode_step_out_kernel<<<(d.D + 7) / 8, 256, 0, s>>>(a);
  prof_end(K_DECODE_STEP_OUT, s);
  return cudaGetLastError();
}

}  // namespace hy
