// Implicit-filter forward on the 5th-generation tensor cores (tcgen05 / TMEM), sm_100a only.
//
// Reference semantics in filter_params.h (src/models/sequence/hyena.py:96-155,199-238).  The three GEMM-shaped layers
// run as tcgen05.mma.kind::tf32 with fp32 accumulators in tensor memory:
//
//   tile = 128 positions (UMMA M = 128, one TMEM lane per position, one thread per lane in the epilogues)
//   layer 1,2 : D[128 x 64]  = act[128 x 64] * W^T      (N = 64,  K = 64)
//   layer 3   : D[128 x 128] = act[128 x 64] * W3_h^T   (N = 128, K = 64) per half of 128 channels
//
// fp32 accuracy on tf32 tensor cores: every fp32 operand x is split x = hi + lo with hi = rna_tf32(x),
// lo = rna_tf32(x - hi), and each product is issued three times (hi*hi + lo*hi + hi*lo, the lo*lo term is
// below 2^-22 relative): "3xTF32".  Plain TF32 would put ~5e-4 relative error into k and hence into y.
//
// Operands are written to shared memory by the CUDA cores (the activations are produced in registers by the
// previous epilogue, so there is nothing for TMA to fetch) in the canonical no-swizzle K-major core-matrix
// layout: element (r, k) of an R x 64 fp32 operand sits at byte (r/8)*2048 + (k/4)*128 + (r%8)*16 + (k%4)*4,
// i.e. 8-row x 16-byte core matrices, LBO (K direction) = 128 B, SBO (M/N direction) = 2048 B.
// One elected thread issues the MMAs; completion is tracked with tcgen05.commit -> mbarrier.
#pragma once
#include "fft_passes.cuh"
#include "filter_params.h"
#include "tc_prims.cuh"

namespace hy {
namespace tc {

constexpr int kTileM = 128;
constexpr uint32_t kSBO = 2048, kLBO = 128;
constexpr int kImgW64 = 64 * 64;            // floats of a 64-row operand image
constexpr int kImgW128 = 128 * 64;          // floats of a 128-row operand image
constexpr int kTmemCols = 512;              // main accumulators: [0,64) hidden layer, [64,192) output half; correction ones at +256
constexpr uint32_t kCorr = 256;             // column offset of the correction accumulator of each main accumulator

__host__ __device__ constexpr uint32_t op_off(int r, int k) {   // byte offset inside an operand image
  return (uint32_t)((r >> 3) * 2048 + (k >> 2) * 128 + (r & 7) * 16 + (k & 3) * 4);
}

// shared memory map (bytes)
constexpr uint32_t kOffAhi = 0, kOffAlo = 32768, kOffW1hi = 65536, kOffW1lo = 81920, kOffW2hi = 98304,
                   kOffW2lo = 114688, kOffW3hi = 131072, kOffW3lo = 163840, kOffMisc = 196608;
// misc: W0[64][16] | b0[64] | b1[64] | b2[64] | freq[64] | mbar(8) | tmem_ptr(4)
constexpr uint32_t kMiscFloats = 64 * 16 + 4 * 64;
constexpr size_t kSmemBytes = kOffMisc + kMiscFloats * 4 + 16;

__host__ __device__ constexpr size_t wimg_floats(int D) { return 4 * (size_t)kImgW64 + (size_t)((D + 127) / 128) * 2 * kImgW128; }

// Accurate sinf / sincosf are ~100 instructions each with their large-argument paths; inlined 48x per tile they made
// the epilogue instruction-fetch bound (ncu: stall_no_instruction 5.1 per issue).  One out-of-line copy each.
__device__ __noinline__ float sin_ni(float x) { return sinf(x); }
__device__ __noinline__ float cos_ni(float x) { return cosf(x); }

// Inline sin / cos for the epilogues: three-term Cody-Waite reduction by pi/2 (FMA) + the classic degree-7 / degree-8 minimax
// polynomials on [-pi/4, pi/4], branch free.  <= 1.5 ulp for |x| <= 1e3 and <= 7e-8 absolute everywhere below the guard (checked
// against fp64 over 1e7 arguments; libm's fp32 sin has the same absolute error) -- the accuracy class of sinf / torch.sin, which the
// reference uses (hyena.py:105).  ~22 instructions with no call: the 16-32 evaluations of an epilogue are independent, so they
// overlap (the out-of-line sinf serialised them: one ~120-cycle dependent chain per call, 0.5 instructions per scheduler-cycle).
// Arguments here are freq * pre-activation (|x| <~ 1e2); beyond the guard the library function runs.
__device__ __forceinline__ void sincos_core(float x, float& sn, float& cs, int& q) {
  const float fq = rintf(x * 0.636619772367581343f);
  q = (int)fq;
  float r = fmaf(fq, -1.5707963705062866f, x);
  r = fmaf(fq, 4.371138828673793e-08f, r);
  r = fmaf(fq, 1.7763568394002505e-15f, r);
  const float s = r * r;
  float ps = fmaf(-1.95152959e-4f, s, 8.33216087e-3f);
  ps = fmaf(ps, s, -1.66666546e-1f);
  sn = fmaf(ps, s * r, r);
  float pc = fmaf(2.44331571e-5f, s, -1.38873163e-3f);
  pc = fmaf(pc, s, 4.16666457e-2f);
  pc = fmaf(pc, s, -0.5f);
  cs = fmaf(pc, s, 1.0f);
}
__device__ __forceinline__ float sin_acc(float x) {
  if (fabsf(x) > 30000.f) return sin_ni(x);
  float sn, cs; int q;
  sincos_core(x, sn, cs, q);
  const float v = (q & 1) ? cs : sn;
  return (q & 2) ? -v : v;
}
__device__ __forceinline__ float cos_acc(float x) {
  if (fabsf(x) > 30000.f) return cos_ni(x);
  float sn, cs; int q;
  sincos_core(x, sn, cs, q);
  const float v = (q & 1) ? sn : cs;
  return ((q + 1) & 2) ? -v : v;
}

// D[128 x N] = A * B^T as 3xTF32: 24 MMAs of K = 8, issued by the calling (single) thread.  The tensor core adds into
// its accumulator with truncation, so a chain of n MMAs biases the sum by ~n 2^-24 towards zero (measured: the filter came
// out 6x less accurate than the reference's fp32 path with all 24 products chained into one accumulator).  Hence two
// accumulators: the eight hi*hi products go to tmem_d, the sixteen lo*hi / hi*lo products (2^-11 times smaller, their
// bias is negligible) to tmem_d + kCorr; the epilogues add the two (ld_acc16 / ld_acc32).
__device__ __forceinline__ void issue_layer(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                            int N, uint32_t mbar) {
  const uint32_t idesc = make_idesc(N);
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t a = (pass == 1) ? a_lo : a_hi;
    const uint32_t b = (pass == 2) ? b_lo : b_hi;
    const uint32_t d = (pass == 0) ? tmem_d : tmem_d + kCorr;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks)
      mma_tf32(d, make_desc(a + ks * 2 * kLBO), make_desc(b + ks * 2 * kLBO), idesc, (ks > 0 || pass == 2) ? 1u : 0u);
  }
  mma_commit(mbar);
}

// main + correction accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void ld_acc16(uint32_t taddr, float (&v)[16]) {
  float c[16];
  tmem_ld16(taddr, v);
  tmem_ld16(taddr + kCorr, c);
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] += c[i];
}
__device__ __forceinline__ void ld_acc32(uint32_t taddr, float (&v)[32]) {
  float c[32];
  tmem_ld32(taddr, v);
  tmem_ld32(taddr + kCorr, c);
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] += c[i];
}

// write NV activations (features k0 .. k0+NV) of row `row` as hi/lo operand images
template <int NV>
__device__ __forceinline__ void store_row_split(unsigned char* smem, int row, int k0, const float (&a)[NV]) {
#pragma unroll
  for (int kc = 0; kc < NV / 4; ++kc) {
    float4 hi, lo;
    split_tf32(a[4 * kc + 0], hi.x, lo.x);
    split_tf32(a[4 * kc + 1], hi.y, lo.y);
    split_tf32(a[4 * kc + 2], hi.z, lo.z);
    split_tf32(a[4 * kc + 3], hi.w, lo.w);
    const uint32_t off = op_off(row, k0 + 4 * kc);
    *reinterpret_cast<float4*>(smem + kOffAhi + off) = hi;
    *reinterpret_cast<float4*>(smem + kOffAlo + off) = lo;
  }
}

// ---------------------------------------------------------------------------------------------- prep
// Split the weights into tf32 hi/lo operand images (global memory, in shared-memory image order):
// [W1 hi][W1 lo][W2 hi][W2 lo] then per 128-channel half h: [W3_h hi][W3_h lo] (rows >= D are zero).
__global__ void filter_tc_prep_kernel(const float* __restrict__ W1, const float* __restrict__ W2,
                                      const float* __restrict__ W3, int D, float* __restrict__ wimg) {
  const int nh = (D + 127) / 128;
  const int total = 2 * kImgW64 + nh * kImgW128;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    float x;
    float* hi_img;
    float* lo_img;
    int r, k;
    if (i < 2 * kImgW64) {
      const int w = i / kImgW64, e = i % kImgW64;
      r = e / 64; k = e % 64;
      x = (w == 0 ? W1 : W2)[r * 64 + k];
      hi_img = wimg + w * 2 * kImgW64;
      lo_img = hi_img + kImgW64;
    } else {
      const int j = i - 2 * kImgW64, h = j / kImgW128, e = j % kImgW128;
      r = e / 64; k = e % 64;
      const int c = h * 128 + r;
      x = (c < D) ? W3[(size_t)c * 64 + k] : 0.f;
      hi_img = wimg + 4 * kImgW64 + (size_t)h * 2 * kImgW128;
      lo_img = hi_img + kImgW128;
    }
    float hi, lo;
    split_tf32(x, hi, lo);
    hi_img[op_off(r, k) / 4] = hi;
    lo_img[op_off(r, k) / 4] = lo;
  }
}

// ---------------------------------------------------------------------------------------------- forward
// 512 threads: warp w works on TMEM lanes 32*(w%4).. (positions) and on column part w/4 of every accumulator,
// so four warps per scheduler hide the latency of the sin/exp epilogues.
constexpr int kThreads = 512;

__global__ void __launch_bounds__(kThreads, 1)
filter_tc_fwd_kernel(const FilterParams P, const float* __restrict__ wimg, float* __restrict__ kout, int ntiles) {
  extern __shared__ __align__(1024) unsigned char smem[];
  float* misc = reinterpret_cast<float*>(smem + kOffMisc);
  float* W0s = misc;                    // [64][16]
  float* b0s = misc + 64 * 16;
  float* b1s = b0s + 64;
  float* b2s = b1s + 64;
  float* frs = b2s + 64;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(frs + 64);
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(mbar_p + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int part = warp >> 2;                             // which quarter of the columns
  const int row = 32 * (warp & 3) + lane;                 // position inside the tile == TMEM lane
  const uint32_t sbase = smem_u32(smem);
  const uint32_t mbar = smem_u32(mbar_p);
  const int nh = (P.D + 127) / 128;

  // ---- one-time setup: TMEM allocation, mbarrier, resident weights
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_p)), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) mbar_init(mbar, 1);
  for (int i = tid; i < 4 * kImgW64 / 4; i += kThreads)   // W1/W2 hi/lo images: 64 KB, 16 bytes per cp.async
    cp_async16(smem + kOffW1hi + 16 * i, wimg + 4 * i, true);
  for (int i = tid; i < 64 * 16; i += kThreads) {
    const int r = i / 16, e = i % 16;
    W0s[i] = (e < P.E) ? __ldg(P.W0 + r * P.E + e) : 0.f;
  }
  if (tid < 64) {
    b0s[tid] = __ldg(P.b0 + tid); b1s[tid] = __ldg(P.b1 + tid); b2s[tid] = __ldg(P.b2 + tid);
    frs[tid] = __ldg(P.freq + tid);
  }
  cp_async_wait_all();
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_p;
  const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);   // this warp's 32 TMEM lanes
  uint32_t phase = 0;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int t = tile * kTileM + row;
    const bool tv = t < P.L;
    // prefetch output-layer half 0 (the buffer is free: the MMAs that read it completed last tile)
    {
      const float* src = wimg + 4 * kImgW64;
      for (int i = tid; i < 2 * kImgW128 / 4; i += kThreads) cp_async16(smem + kOffW3hi + 16 * i, src + 4 * i, true);
    }
    // ---- layer 0 on the CUDA cores: a1 = sin(f * (W0 z + b0)), 16 features per thread
    {
      float z[kMaxE];
#pragma unroll
      for (int e = 0; e < kMaxE; ++e) z[e] = (tv && e < P.E) ? __ldg(P.z + (size_t)t * P.z_stride + e) : 0.f;
      float a[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int i = part * 16 + j;
        float acc = b0s[i];
#pragma unroll
        for (int e = 0; e < kMaxE; ++e) acc = fmaf(W0s[i * 16 + e], z[e], acc);
        a[j] = sin_acc(frs[i] * acc);
      }
      store_row_split<16>(smem, row, part * 16, a);
    }
    fence_async_smem();
    __syncthreads();
    // ---- layers 1 and 2 on the tensor cores
#pragma unroll
    for (int layer = 0; layer < 2; ++layer) {
      if (tid == 0) {
        fence_after_sync();
        issue_layer(tmem, sbase + kOffAhi, sbase + kOffAlo, sbase + (layer ? kOffW2hi : kOffW1hi),
                    sbase + (layer ? kOffW2lo : kOffW1lo), 64, mbar);
      }
      mbar_wait(mbar, phase);
      phase ^= 1;
      fence_after_sync();
      const float* bs = layer ? b2s : b1s;
      float a[16];
      ld_acc16(lane_addr + part * 16, a);
#pragma unroll
      for (int j = 0; j < 16; ++j) a[j] = sin_acc(frs[part * 16 + j] * (a[j] + bs[part * 16 + j]));
      store_row_split<16>(smem, row, part * 16, a);        // the MMAs that read the A images have completed
      fence_before_sync();
      fence_async_smem();
      __syncthreads();
    }
    // ---- output layer, 128 channels at a time, modulation in the epilogue
    const float tpos = tv ? __ldg(P.t + t) : 0.f;
    for (int h = 0; h < nh; ++h) {
      cp_async_wait_all();                               // this thread's pieces of half h have landed
      fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        fence_after_sync();
        issue_layer(tmem + 64, sbase + kOffAhi, sbase + kOffAlo, sbase + kOffW3hi, sbase + kOffW3lo, 128, mbar);
      }
      mbar_wait(mbar, phase);
      phase ^= 1;
      fence_after_sync();
      if (h + 1 < nh) {                                  // stream the next half while this one is written out
        const float* src = wimg + 4 * kImgW64 + (size_t)(h + 1) * 2 * kImgW128;
        for (int i = tid; i < 2 * kImgW128 / 4; i += kThreads) cp_async16(smem + kOffW3hi + 16 * i, src + 4 * i, true);
      }
      float v[32];
      ld_acc32(lane_addr + 64 + part * 32, v);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int c = h * 128 + part * 32 + j;
        if (c < P.D && tv) {
          float x = v[j];
          if (P.modulate) x *= (expf(-tpos * fabsf(__ldg(P.deltas + c))) + P.shift);
          kout[(size_t)c * P.L + t] = x;
        }
      }
      fence_before_sync();
    }
    __syncthreads();                                     // A images and TMEM are free for the next tile
  }

  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- forward, TS form
// Round-2 form of the forward kernel (D <= 256; the kernel above stays for wider models):
//   * the activations of a layer are the A operand IN TENSOR MEMORY: the thread that owns a position writes its
//     (hi, lo) halves with tcgen05.st straight from the registers of the previous epilogue (TMEM lane = position,
//     column = feature is exactly the A layout of an M = 128 MMA) -- no operand images built by the CUDA cores in
//     shared memory, no bank conflicts, and 64 KB of shared memory back;
//   * with that space ALL weight images (W1, W2, both halves of W3: 192 KB) stay resident for the whole kernel;
//   * two tiles are in flight per CTA: warps 0-7 and 8-15 are two independent groups, each with its own half of
//     tensor memory (accumulator 128 columns + A operand 2 x 64 columns), its own issuing thread, mbarrier and named
//     barrier, working on alternate tiles -- one group's MMAs run under the other group's sin / exp epilogue (the
//     single-tile kernel issued 0.51 instructions per scheduler-cycle with the tensor pipe 12 % busy);
//   * one accumulator per layer, the 16 correction MMAs (lo*hi, hi*lo) first and the 8 hi*hi MMAs last, so that only
//     those eight truncate at full scale (same accuracy as a separate correction accumulator, half the columns).
constexpr uint32_t k2OffW3 = 65536;                               // after the W1 / W2 images (hi, lo each)
__host__ __device__ constexpr size_t fwd2_smem_bytes(int D) { return 65536 + (size_t)((D + 127) / 128) * 65536 + kMiscFloats * 4 + 32; }

__device__ __forceinline__ void issue_layer_ts(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                               int N, uint32_t mbar) {
  const uint32_t idesc = make_idesc(N);
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {                   // lo*hi, hi*lo, then hi*hi
    const uint32_t a = (pass == 0) ? a_lo : a_hi;
    const uint32_t b = (pass == 1) ? b_lo : b_hi;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks)
      mma_tf32_ts(tmem_d, a + 8 * ks, make_desc(b + ks * 2 * kLBO), idesc, (ks > 0 || pass > 0) ? 1u : 0u);
  }
  mma_commit(mbar);
}

__device__ __forceinline__ void split_store32(uint32_t taddr_hi, uint32_t taddr_lo, const float (&a)[32]) {
  uint32_t hi[32], lo[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    float h, l;
    split_tf32(a[j], h, l);
    hi[j] = __float_as_uint(h); lo[j] = __float_as_uint(l);
  }
  tmem_st32(taddr_hi, hi);
  tmem_st32(taddr_lo, lo);
  tmem_wait_st();
}

__global__ void __launch_bounds__(kThreads, 1)
filter_tc_fwd2_kernel(const FilterParams P, const float* __restrict__ wimg, float* __restrict__ kout, int ntiles) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int nh = (P.D + 127) / 128;                       // 1 or 2 (launcher)
  float* misc = reinterpret_cast<float*>(smem + k2OffW3 + (size_t)nh * 65536);
  float* W0s = misc;                    // [64][16]
  float* b0s = misc + 64 * 16;
  float* b1s = b0s + 64;
  float* b2s = b1s + 64;
  float* frs = b2s + 64;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(frs + 64);        // two barriers, one per group
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(mbar_p + 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int grp = warp >> 3;                              // tile group of this warp
  const int quad = warp & 3;                              // TMEM lane quadrant this warp may access
  const int half = (warp >> 2) & 1;                       // which half of the columns
  const int row = 32 * quad + lane;                       // position inside the tile == TMEM lane
  const bool issuer = (tid & 255) == 0;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t mbar = smem_u32(mbar_p + grp);

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_p)), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) { mbar_init(smem_u32(mbar_p), 1); mbar_init(smem_u32(mbar_p + 1), 1); }
  {
    const int pieces = (int)((65536 + (size_t)nh * 65536) / 16);   // all weight images, 16 bytes per cp.async
    for (int i = tid; i < pieces; i += kThreads) cp_async16(smem + 16 * (size_t)i, wimg + 4 * (size_t)i, true);
  }
  for (int i = tid; i < 64 * 16; i += kThreads) {
    const int r = i / 16, e = i % 16;
    W0s[i] = (e < P.E) ? __ldg(P.W0 + r * P.E + e) : 0.f;
  }
  if (tid < 64) {
    b0s[tid] = __ldg(P.b0 + tid); b1s[tid] = __ldg(P.b1 + tid); b2s[tid] = __ldg(P.b2 + tid);
    frs[tid] = __ldg(P.freq + tid);
  }
  cp_async_wait_all();
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t gbase = *tmem_p + (uint32_t)grp * 256u;           // this group's columns: acc [0,128) A hi [128,192) lo [192,256)
  const uint32_t lane_addr = gbase + ((uint32_t)(32 * quad) << 16);
  const uint32_t a_hi = gbase + 128, a_lo = gbase + 192;
  auto group_sync = [&]() { asm volatile("bar.sync %0, 256;" ::"r"(1 + grp) : "memory"); };
  uint32_t phase = 0;

  for (int tile = 2 * blockIdx.x + grp; tile < ntiles; tile += 2 * gridDim.x) {
    const int t = tile * kTileM + row;
    const bool tv = t < P.L;
    // ---- layer 0 on the CUDA cores: a1 = sin(f * (W0 z + b0)), 32 features per thread
    {
      float z[kMaxE];
#pragma unroll
      for (int e = 0; e < kMaxE; ++e) z[e] = (tv && e < P.E) ? __ldg(P.z + (size_t)t * P.z_stride + e) : 0.f;
      float a[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int i = half * 32 + j;
        float acc = b0s[i];
#pragma unroll
        for (int e = 0; e < kMaxE; ++e) acc = fmaf(W0s[i * 16 + e], z[e], acc);
        a[j] = sin_acc(frs[i] * acc);
      }
      split_store32(lane_addr + 128 + half * 32, lane_addr + 192 + half * 32, a);
    }
    fence_before_sync();
    group_sync();
    // ---- layers 1 and 2 on the tensor cores
#pragma unroll
    for (int layer = 0; layer < 2; ++layer) {
      if (issuer) {
        fence_after_sync();
        issue_layer_ts(gbase, a_hi, a_lo, sbase + (layer ? 32768u : 0u), sbase + (layer ? 49152u : 16384u), 64, mbar);
      }
      mbar_wait_u(mbar, phase);
      phase ^= 1;
      fence_after_sync();
      const float* bs = layer ? b2s : b1s;
      float a[32];
      tmem_ld32(lane_addr + half * 32, a);
#pragma unroll
      for (int j = 0; j < 32; ++j) a[j] = sin_acc(frs[half * 32 + j] * (a[j] + bs[half * 32 + j]));
      split_store32(lane_addr + 128 + half * 32, lane_addr + 192 + half * 32, a);   // the MMAs that read A have completed
      fence_before_sync();
      group_sync();
    }
    // ---- output layer, 128 channels at a time, modulation in the epilogue
    const float tpos = tv ? __ldg(P.t + t) : 0.f;
    for (int h = 0; h < nh; ++h) {
      if (issuer) {
        fence_after_sync();
        issue_layer_ts(gbase, a_hi, a_lo, sbase + k2OffW3 + h * 65536u, sbase + k2OffW3 + h * 65536u + 32768u, 128, mbar);
      }
      mbar_wait_u(mbar, phase);
      phase ^= 1;
      fence_after_sync();
#pragma unroll
      for (int c0 = 0; c0 < 64; c0 += 32) {
        float v[32];
        tmem_ld32(lane_addr + half * 64 + c0, v);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int c = h * 128 + half * 64 + c0 + j;
          if (c < P.D && tv) {
            float x = v[j];
            if (P.modulate) x *= (expf(-tpos * fabsf(__ldg(P.deltas + c))) + P.shift);
            kout[(size_t)c * P.L + t] = x;
          }
        }
      }
      fence_before_sync();
      group_sync();                                      // accumulator (and, after the last half, the A operand) is free
    }
  }

  fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_p), "r"(kTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- backward, stage 1
// Per 128-position tile, all GEMMs with M = positions (thread = position, same operand builders as forward):
//   recompute pre1..3 / a1..3;  da3 = dh W3 (dh = dk * modulation, K = channels in chunks of 64);
//   dp3 = da3 f cos(f pre3);  da2 = dp3 W2;  dp2 = ...;  da1 = dp2 W1;  dp1 = ...
// and writes, feature-major (64, L): a1, a2, a3, dp1, dp2, dp3, X = sum_l da_l cos(f pre_l) pre_l, plus dh (D, L).
// Stage 2 (host side, hyena-dna_b200/ops.py) turns those into the parameter gradients with GEMMs whose reduction
// dimension is the sequence: dW3 = dh a3, dW2 = dp3^T a2, dW1 = dp2^T a1, dW0 = dp1^T z, db_l = colsum(dp_l),
// dfreq = colsum(X), dz = dp1 W0.
//
// Streamed operand images (global, built by filter_tc_prep_bwd_kernel), item i lives in stream buffer i & 1:
//   items 0..nq-1: W3^T chunk q  [64 features x 64 channels of chunk q];  item nq: W2^T;  item nq+1: W1^T
constexpr int kScratchArrays = 7;

__host__ __device__ constexpr size_t wimg_bwd_floats(int D) {
  return 4 * (size_t)kImgW64 + (size_t)((D + 63) / 64 + 2) * 2 * kImgW64;
}

__global__ void filter_tc_prep_bwd_kernel(const float* __restrict__ W1, const float* __restrict__ W2,
                                          const float* __restrict__ W3, int D, float* __restrict__ wimg) {
  const int nq = (D + 63) / 64;
  const int total = (2 + nq + 2) * kImgW64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int item = i / kImgW64, e = i % kImgW64;
    const int r = e / 64, k = e % 64;
    float x;
    float* hi_img = wimg + (size_t)item * 2 * kImgW64;
    if (item == 0) x = W1[r * 64 + k];
    else if (item == 1) x = W2[r * 64 + k];
    else if (item < 2 + nq) {                  // W3^T chunk q: (feature r, channel k of the chunk)
      const int c = (item - 2) * 64 + k;
      x = (c < D) ? W3[(size_t)c * 64 + r] : 0.f;
    } else if (item == 2 + nq) x = W2[k * 64 + r];     // W2^T
    else x = W1[k * 64 + r];                           // W1^T
    float hi, lo;
    split_tf32(x, hi, lo);
    hi_img[op_off(r, k) / 4] = hi;
    hi_img[kImgW64 + op_off(r, k) / 4] = lo;
  }
}

__device__ __forceinline__ void stream_item(unsigned char* smem, const float* wimg, int item, int tid) {
  const float* src = wimg + (size_t)(2 + item) * 2 * kImgW64;
  unsigned char* dst = smem + kOffW3hi + (item & 1) * 32768;
  for (int i = tid; i < 2 * kImgW64 / 4; i += kThreads) cp_async16(dst + 16 * i, src + 4 * i, true);
}

// 16 features of one position into a feature-major (64, L) array: for a fixed feature the 32 lanes of a warp write
// 32 consecutive positions (128 bytes)
__device__ __forceinline__ void store16(float* dst, size_t L, const float (&a)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) dst[(size_t)i * L] = a[i];
}

__global__ void __launch_bounds__(kThreads, 1)
filter_tc_bwd_kernel(const FilterParams P, const float* __restrict__ wimg, const float* __restrict__ dk,
                     float* __restrict__ dh, float* __restrict__ scratch, int ntiles) {
  extern __shared__ __align__(1024) unsigned char smem[];
  float* misc = reinterpret_cast<float*>(smem + kOffMisc);
  float* W0s = misc;
  float* b0s = misc + 64 * 16;
  float* b1s = b0s + 64;
  float* b2s = b1s + 64;
  float* frs = b2s + 64;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(frs + 64);
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(mbar_p + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int part = warp >> 2;
  const int row = 32 * (warp & 3) + lane;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t mbar = smem_u32(mbar_p);
  const int nq = (P.D + 63) / 64;
  const size_t arr = (size_t)P.L * 64;                   // floats per scratch array

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_p)), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) mbar_init(mbar, 1);
  for (int i = tid; i < 4 * kImgW64 / 4; i += kThreads) cp_async16(smem + kOffW1hi + 16 * i, wimg + 4 * i, true);
  for (int i = tid; i < 64 * 16; i += kThreads) {
    const int r = i / 16, e = i % 16;
    W0s[i] = (e < P.E) ? __ldg(P.W0 + r * P.E + e) : 0.f;
  }
  if (tid < 64) {
    b0s[tid] = __ldg(P.b0 + tid); b1s[tid] = __ldg(P.b1 + tid); b2s[tid] = __ldg(P.b2 + tid);
    frs[tid] = __ldg(P.freq + tid);
  }
  cp_async_wait_all();
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_p;
  const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
  uint32_t phase = 0;
  const float* fr = frs + part * 16;                      // this thread's 16 frequencies (shared memory)

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int t = tile * kTileM + row;
    const bool tv = t < P.L;
    float* out = scratch + (size_t)(part * 16) * P.L + (tv ? t : 0);      // [array][feature][t]
    stream_item(smem, wimg, 0, tid);
    stream_item(smem, wimg, 1, tid);

    // ---- forward recompute
    float pre1[16], pre2[16], pre3[16], a[16];
    {
      float z[kMaxE];
#pragma unroll
      for (int e = 0; e < kMaxE; ++e) z[e] = (tv && e < P.E) ? __ldg(P.z + (size_t)t * P.z_stride + e) : 0.f;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int i = part * 16 + j;
        float acc = b0s[i];
#pragma unroll
        for (int e = 0; e < kMaxE; ++e) acc = fmaf(W0s[i * 16 + e], z[e], acc);
        pre1[j] = acc;
        a[j] = sin_acc(fr[j] * acc);
      }
      store_row_split<16>(smem, row, part * 16, a);
      if (tv) store16(out + 0 * arr, P.L, a);
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
      issue_layer(tmem, sbase + kOffAhi, sbase + kOffAlo, sbase + kOffW1hi, sbase + kOffW1lo, 64, mbar);
    }
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    ld_acc16(lane_addr + part * 16, pre2);
#pragma unroll
    for (int j = 0; j < 16; ++j) { pre2[j] += b1s[part * 16 + j]; a[j] = sin_acc(fr[j] * pre2[j]); }
    store_row_split<16>(smem, row, part * 16, a);
    if (tv) store16(out + 1 * arr, P.L, a);
    fence_before_sync();
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
      issue_layer(tmem, sbase + kOffAhi, sbase + kOffAlo, sbase + kOffW2hi, sbase + kOffW2lo, 64, mbar);
    }
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    ld_acc16(lane_addr + part * 16, pre3);
#pragma unroll
    for (int j = 0; j < 16; ++j) { pre3[j] += b2s[part * 16 + j]; a[j] = sin_acc(fr[j] * pre3[j]); }
    if (tv) store16(out + 2 * arr, P.L, a);
    fence_before_sync();

    // ---- da3 = dh W3, 64 channels per MMA group; dh = dk * (exp(-t|delta|) + shift) also goes to HBM (stage 2 needs it)
    const float tpos = tv ? __ldg(P.t + t) : 0.f;
    float nx[16];                                            // dk of the next chunk, loaded one MMA group ahead
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int c = part * 16 + j;
      nx[j] = (c < P.D && tv) ? __ldg(dk + (size_t)c * P.L + t) : 0.f;
    }
    for (int q = 0; q < nq; ++q) {
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int c = q * 64 + part * 16 + j;
        float x = nx[j];
        if (c < P.D && tv) {
          if (P.modulate) x *= (expf(-tpos * fabsf(__ldg(P.deltas + c))) + P.shift);
          dh[(size_t)c * P.L + t] = x;
        }
        a[j] = x;
      }
      store_row_split<16>(smem, row, part * 16, a);        // the previous MMA group has completed (waited below)
      cp_async_wait_all();
      fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        fence_after_sync();
        const uint32_t sb = sbase + kOffW3hi + (q & 1) * 32768;
        const uint32_t idesc = make_idesc(64);
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t aa = sbase + ((pass == 1) ? kOffAlo : kOffAhi);
          const uint32_t bb = sb + ((pass == 2) ? 16384u : 0u);
          const uint32_t dd = (pass == 0) ? tmem : tmem + kCorr;      // main / correction accumulator (see issue_layer)
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            mma_tf32(dd, make_desc(aa + ks * 2 * kLBO), make_desc(bb + ks * 2 * kLBO), idesc,
                     (q > 0 || ks > 0 || pass == 2) ? 1u : 0u);
        }
        mma_commit(mbar);
      }
      if (q + 1 < nq) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int c = (q + 1) * 64 + part * 16 + j;
          nx[j] = (c < P.D && tv) ? __ldg(dk + (size_t)c * P.L + t) : 0.f;
        }
      }
      mbar_wait(mbar, phase); phase ^= 1;
      fence_after_sync();
      stream_item(smem, wimg, q + 2, tid);                  // refill the buffer this group just released
    }

    // ---- layer 3 -> 2 -> 1 backward through the sine activations
    float X[16], da[16];
    ld_acc16(lane_addr + part * 16, da);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float cs = cos_acc(fr[j] * pre3[j]);
      const float g = da[j] * cs;
      X[j] = g * pre3[j];
      a[j] = g * fr[j];
    }
    if (tv) store16(out + 5 * arr, P.L, a);
    store_row_split<16>(smem, row, part * 16, a);
    cp_async_wait_all();
    fence_before_sync();
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {                                          // da2 = dp3 W2   (B = W2^T image, item nq)
      fence_after_sync();
      const uint32_t sb = sbase + kOffW3hi + (nq & 1) * 32768;
      issue_layer(tmem, sbase + kOffAhi, sbase + kOffAlo, sb, sb + 16384u, 64, mbar);
    }
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    ld_acc16(lane_addr + part * 16, da);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float cs = cos_acc(fr[j] * pre2[j]);
      const float g = da[j] * cs;
      X[j] = fmaf(g, pre2[j], X[j]);
      a[j] = g * fr[j];
    }
    if (tv) store16(out + 4 * arr, P.L, a);
    store_row_split<16>(smem, row, part * 16, a);
    fence_before_sync();
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {                                          // da1 = dp2 W1   (B = W1^T image, item nq+1)
      fence_after_sync();
      const uint32_t sb = sbase + kOffW3hi + ((nq + 1) & 1) * 32768;
      issue_layer(tmem, sbase + kOffAhi, sbase + kOffAlo, sb, sb + 16384u, 64, mbar);
    }
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    ld_acc16(lane_addr + part * 16, da);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float cs = cos_acc(fr[j] * pre1[j]);
      const float g = da[j] * cs;
      X[j] = fmaf(g, pre1[j], X[j]);
      a[j] = g * fr[j];
    }
    if (tv) { store16(out + 3 * arr, P.L, a); store16(out + 6 * arr, P.L, X); }
    fence_before_sync();
    __syncthreads();
  }

  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- backward, stage 2
// All parameter gradients of the filter are reductions over the sequence.  With the stage-1 arrays stored feature-
// major every operand is K-major with K = position, so they are three accumulating tcgen05 GEMM groups whose fp32
// accumulators stay in tensor memory for the whole kernel (persistent CTAs, split over the sequence, one atomic
// flush at the end):
//   G1  dW3[c][j]      = sum_t dh[c][t] a3[j][t]                       M = 128 channels per tile (<= 2 tiles), N = 64
//   G2  [dp3;dp2] x [a2;a1;1]^T : block(0,0) = dW2, block(1,1) = dW1, column 128 = (db2 ; db1)     M = 128, N = 144
//   G3  [dp1;X]  x [z;1]^T      : rows 0..63 -> (dW0 | db0), rows 64..127 col 8 -> dfreq             M = 128, N = 16
// K block = 32 positions (operand images: K-major, SBO 1024 B, LBO 128 B), 3xTF32 like everywhere else.
constexpr int kRedKB = 32;
constexpr int kRedThreads = 512;
constexpr int kRedItems = 12;                // ceil(8 * roundup8(256 + 7*64 + emb_dim) / 512)
constexpr uint32_t kRedSBO = 1024;
__host__ __device__ constexpr uint32_t red_off(int r, int k) {
  return (uint32_t)((r >> 3) * 1024 + (k >> 2) * 128 + (r & 7) * 16 + (k & 3) * 4);
}
constexpr uint32_t kRedImg128 = 128 * kRedKB * 4;      // bytes of a 128-row image (16 KB)
// shared memory map (bytes); every operand has a hi image followed by a lo image
constexpr uint32_t kRedOffDh = 0;                                  // 2 tiles x (hi 16K + lo 16K) = 64 KB
constexpr uint32_t kRedOffAs = 65536;                              // [dp3;dp2]   32 KB
constexpr uint32_t kRedOffAx = kRedOffAs + 32768;                  // [dp1;X]     32 KB
constexpr uint32_t kRedOffB3 = kRedOffAx + 32768;                  // a3 (64 rows): hi 8K + lo 8K
constexpr uint32_t kRedOffBs = kRedOffB3 + 16384;                  // [a2;a1;ones16] 144 rows: hi 18K + lo 18K
constexpr uint32_t kRedOffBz = kRedOffBs + 36864;                  // [z pad 8; ones 8] 16 rows: hi 2K + lo 2K
constexpr uint32_t kRedOffMisc = kRedOffBz + 4096;
constexpr size_t kRedSmemBytes = kRedOffMisc + 64;
constexpr int kRedTmemCols = 512;                                  // G1: [0,128)  G2: [128,272)  G3: [272,288)

__device__ __forceinline__ uint64_t make_desc_red(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(kLBO >> 4) << 16;
  d |= (uint64_t)(kRedSBO >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
__device__ __forceinline__ void issue_red(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                          int N, uint32_t first_acc) {
  const uint32_t idesc = make_idesc(N);
  uint32_t acc = first_acc;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t a = (pass == 1) ? a_lo : a_hi;
    const uint32_t b = (pass == 2) ? b_lo : b_hi;
#pragma unroll
    for (int ks = 0; ks < kRedKB / 8; ++ks) {
      mma_tf32(tmem_d, make_desc_red(a + ks * 2 * kLBO), make_desc_red(b + ks * 2 * kLBO), idesc, acc);
      acc = 1;
    }
  }
}

// four consecutive positions of a feature row (zero beyond L); vector load when rows are 16-byte aligned
__device__ __forceinline__ float4 load4_row(const float* __restrict__ src, size_t t, size_t L, bool v4) {
  float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
  if (v4 && t + 3 < L) return __ldg(reinterpret_cast<const float4*>(src + t));
  if (t < L) x.x = __ldg(src + t);
  if (t + 1 < L) x.y = __ldg(src + t + 1);
  if (t + 2 < L) x.z = __ldg(src + t + 2);
  if (t + 3 < L) x.w = __ldg(src + t + 3);
  return x;
}

struct RedArgs {
  const float* dh;        // (D, L)
  const float* scratch;   // (7, 64, L): a1 a2 a3 dp1 dp2 dp3 X
  const float* zT;        // (E, L)
  float* dW0; float* db0; float* dW1; float* db1; float* dW2; float* db2; float* dW3; float* dfreq;
  int L, D, E;
};

__global__ void __launch_bounds__(kRedThreads, 1) filter_tc_red_kernel(const RedArgs R, int nblocks) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(smem + kRedOffMisc);
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(mbar_p + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t mbar = smem_u32(mbar_p);
  const int nmt = (R.D + 127) / 128;                       // channel tiles (host guarantees <= 2)
  const size_t L = (size_t)R.L;
  const bool v4 = (R.L & 3) == 0;

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_p)), "r"(kRedTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) mbar_init(mbar, 1);
  // zero every image once (rows that are never loaded -- channel padding, z padding -- stay zero), then the ones rows
  for (uint32_t i = tid; i < kRedOffMisc / 16; i += kRedThreads) reinterpret_cast<float4*>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  for (int i = tid; i < 16 * kRedKB; i += kRedThreads) {   // [a2;a1;ones16]: rows 128..143 hi = 1
    const int r = 128 + i / kRedKB, k = i % kRedKB;
    *reinterpret_cast<float*>(smem + kRedOffBs + red_off(r, k)) = 1.f;
  }
  for (int i = tid; i < 8 * kRedKB; i += kRedThreads) {    // [z;ones8]: rows 8..15 hi = 1
    const int r = 8 + i / kRedKB, k = i % kRedKB;
    *reinterpret_cast<float*>(smem + kRedOffBz + red_off(r, k)) = 1.f;
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_p;

  // Work items: (row, 4-position piece) pairs, 8 pieces per row; item w = tid + kRedThreads*it, so every item of a
  // thread has the same piece index (tid >> 3) & 7.  The decode (source row pointer, destination offset, hi->lo distance
  // class) does not depend on the k-block: done once, kept in registers, so that all loads of a block can be issued
  // back to back (one DRAM latency per block instead of one per item).
  // Item -> (row, piece): inside every group of 64 items the ROW runs fastest (row = 8 (w >> 6) + (w & 7), piece =
  // (w >> 3) & 7), so the eight lanes of a quarter warp write the eight 16-byte rows of ONE core matrix = 128 contiguous
  // bytes (conflict free), and a warp reads 64 contiguous bytes of each of eight rows.  (Piece-fastest, as in round 1,
  // put the eight lanes 128 bytes apart: an 8-way bank conflict on every store, 87 % of all shared wavefronts.)
  const int nrow = R.D + 7 * 64 + R.E;                     // dh rows, six (64,L) arrays + X, z rows
  const int pc = (tid >> 3) & 7;
  const float* sp[kRedItems];
  uint32_t dof[kRedItems];                                 // bits [0,18): byte offset of the hi piece; [18,20): lo class
  static_for<0, kRedItems>([&](auto it_) {
    constexpr int it = decltype(it_)::value;
    const int row = (((tid + kRedThreads * it) >> 6) << 3) + (tid & 7);
    const float* src = nullptr;
    uint32_t img = 0, cls = 0;
    int r = 0;
    if (row < R.D) {
      src = R.dh + (size_t)row * L; img = kRedOffDh + (row >> 7) * 32768; cls = 0; r = row & 127;
    } else if (row < nrow) {
      const int q = row - R.D;
      if (q < 7 * 64) {
        const int arr = q >> 6, f = q & 63;                // scratch order: a1 a2 a3 dp1 dp2 dp3 X
        src = R.scratch + ((size_t)arr * 64 + f) * L;
        switch (arr) {
          case 0: img = kRedOffBs; cls = 1; r = 64 + f; break;      // a1  -> B_s rows 64..127
          case 1: img = kRedOffBs; cls = 1; r = f; break;           // a2  -> B_s rows 0..63
          case 2: img = kRedOffB3; cls = 2; r = f; break;           // a3
          case 3: img = kRedOffAx; cls = 0; r = f; break;           // dp1 -> A_x rows 0..63
          case 4: img = kRedOffAs; cls = 0; r = 64 + f; break;      // dp2 -> A_s rows 64..127
          case 5: img = kRedOffAs; cls = 0; r = f; break;           // dp3 -> A_s rows 0..63
          default: img = kRedOffAx; cls = 0; r = 64 + f; break;     // X   -> A_x rows 64..127
        }
      } else {
        const int e = q - 7 * 64;                          // z feature e -> B_z row e
        src = R.zT + (size_t)e * L; img = kRedOffBz; cls = 3; r = e;
      }
    }
    sp[it] = src;
    dof[it] = (img + red_off(r, 4 * pc)) | (cls << 18);
  });
  uint32_t phase = 0;
  bool first = true;
  for (int blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const size_t t = (size_t)blk * kRedKB + 4 * pc;
    float4 x[kRedItems];
    static_for<0, kRedItems>([&](auto it_) {               // all loads of this block in flight at once
      constexpr int it = decltype(it_)::value;
      x[it] = sp[it] ? load4_row(sp[it], t, L, v4) : make_float4(0.f, 0.f, 0.f, 0.f);
    });
    if (!first) { mbar_wait(mbar, phase); phase ^= 1; fence_after_sync(); }   // previous MMAs have read the images
    static_for<0, kRedItems>([&](auto it_) {
      constexpr int it = decltype(it_)::value;
      if (sp[it]) {
        float4 hi, lo;
        split_tf32(x[it].x, hi.x, lo.x); split_tf32(x[it].y, hi.y, lo.y);
        split_tf32(x[it].z, hi.z, lo.z); split_tf32(x[it].w, hi.w, lo.w);
        const uint32_t off = dof[it] & 0x3FFFFu, cls = dof[it] >> 18;
        const uint32_t lo_off = cls == 0 ? 16384u : cls == 1 ? 18432u : cls == 2 ? 8192u : 2048u;
        *reinterpret_cast<float4*>(smem + off) = hi;
        *reinterpret_cast<float4*>(smem + off + lo_off) = lo;
      }
    });
    fence_before_sync();
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
      const uint32_t acc0 = first ? 0u : 1u;
      for (int mt = 0; mt < nmt; ++mt)
        issue_red(tmem + mt * 64, sbase + kRedOffDh + mt * 32768, sbase + kRedOffDh + mt * 32768 + 16384,
                  sbase + kRedOffB3, sbase + kRedOffB3 + 8192, 64, acc0);
      issue_red(tmem + 128, sbase + kRedOffAs, sbase + kRedOffAs + 16384, sbase + kRedOffBs, sbase + kRedOffBs + 18432, 144, acc0);
      issue_red(tmem + 272, sbase + kRedOffAx, sbase + kRedOffAx + 16384, sbase + kRedOffBz, sbase + kRedOffBz + 2048, 16, acc0);
      mma_commit(mbar);
    }
    first = false;
  }
  if (!first) { mbar_wait(mbar, phase); phase ^= 1; fence_after_sync(); }

  // ---- flush: warps 0..3 own TMEM lanes 32*(w%4)..; warps 4..7 take the second half of the columns
  if (!first && warp < 8) {
    const int row = 32 * (warp & 3) + lane;                // accumulator row (TMEM lane)
    const int half = warp >> 2;
    const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
    float v[32];
    for (int mt = 0; mt < nmt; ++mt) {                     // G1: dW3 rows c = 128 mt + row, 64 columns (32 per half)
      tmem_ld32(lane_addr + mt * 64 + half * 32, v);
      const int c = mt * 128 + row;
      if (c < R.D)
#pragma unroll
        for (int j = 0; j < 32; ++j) atomicAdd(R.dW3 + (size_t)c * 64 + half * 32 + j, v[j]);
    }
    // G2: rows < 64: cols 0..63 -> dW2[row][j]; rows >= 64: cols 64..127 -> dW1[row-64][j]; col 128 -> db2 / db1
    {
      const int cbase = (row < 64) ? 0 : 64;
      tmem_ld32(lane_addr + 128 + cbase + half * 32, v);
      float* dst = (row < 64) ? (R.dW2 + row * 64) : (R.dW1 + (row - 64) * 64);
#pragma unroll
      for (int j = 0; j < 32; ++j) atomicAdd(dst + half * 32 + j, v[j]);
      if (half == 0) {
        float b16[16];
        tmem_ld16(lane_addr + 128 + 128, b16);
        atomicAdd(((row < 64) ? R.db2 : R.db1) + (row & 63), b16[0]);
      }
    }
    // G3: rows < 64: cols 0..E-1 -> dW0[row][e], col 8 -> db0[row]; rows >= 64: col 8 -> dfreq[row-64]
    if (half == 1) {
      float x16[16];
      tmem_ld16(lane_addr + 272, x16);
      if (row < 64) {
#pragma unroll
        for (int e = 0; e < 8; ++e)
          if (e < R.E) atomicAdd(R.dW0 + row * R.E + e, x16[e]);
        atomicAdd(R.db0 + row, x16[8]);
      } else {
        atomicAdd(R.dfreq + (row - 64), x16[8]);
      }
    }
    fence_before_sync();
  }
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kRedTmemCols) : "memory");
  }
}

}  // namespace tc
}  // namespace hy
