// The three passes of the long real-FFT convolution (see DESIGN.md "Kernels").
//
// A (batch, channel) row of L real samples is packed as z[m] = x[2m] + i x[2m+1] and zero padded
// to M = M1 * M2 complex points (n = 2M >= 2L).  M is split as m = M2*m1 + m2, k = k1 + M1*k2, with
// the row length M2 = 1024 for M <= 2^16 and M2 = 4096 above (so that a column tile of the large
// transforms spans 256 contiguous bytes of every row it touches):
//
//   pass 1  col_fwd : for every column m2, FFT over m1 (length M1) and twiddle W_M^{m2 k1}
//                     -> scratch A[row][k1][m2]                      (input side fused in)
//   pass 2  row_pass: for every k1, FFT over m2 (length 1024) -> spectrum Z[k1][k2];
//                     pointwise product with the filter spectrum (pairs bin k with bin M-k),
//                     inverse FFT over k2, conj twiddle -> scratch A[row][k1][m2] in place
//   pass 3  col_inv : for every column m2, inverse FFT over k1 -> z'[m1][m2] = y[2m] + i y[2m+1]
//                     (output side fused in)
//
// All spectra are kept in "[k1][k2]" order; nothing is ever transposed in HBM.
#pragma once
#include "fft_radix.cuh"

namespace hy {

// row FFT length M2 = 2^logM2: 1024 (one warp per row) or 4096 (four warps per row)
__host__ __device__ constexpr int log_m2_for(int logM) { return logM >= 17 ? 12 : 10; }

// ------------------------------------------------------------------------------------------------
// short depthwise filter + gates (reference: src/models/sequence/hyena.py:363-369, :394, :420, :432)
// ------------------------------------------------------------------------------------------------
struct Taps { float w0, w1, w2, b, ib; };

__device__ __forceinline__ Taps load_taps(const float* sw, const float* sb, const float* in_bias, int ch) {
  Taps k;
  k.w0 = __ldg(sw + 3 * ch + 0); k.w1 = __ldg(sw + 3 * ch + 1); k.w2 = __ldg(sw + 3 * ch + 2);
  k.b = __ldg(sb + ch);
  k.ib = in_bias ? __ldg(in_bias + ch) : 0.f;
  return k;
}

// P[0..3] = P(t0-2), P(t0-1), P(t0), P(t0+1) with P(t) = p[t] + ib inside [0,L) and 0 outside.
__device__ __forceinline__ void load_window(const float* __restrict__ row, int t0, int L, bool vec, float ib,
                                            float (&P)[4]) {
  if (vec) {   // L even, row base 8-byte aligned, t0 even, t0 < L  =>  t0+1 < L
    float2 a = make_float2(0.f, 0.f);
    if (t0 >= 2) { a = __ldg(reinterpret_cast<const float2*>(row + t0 - 2)); a.x += ib; a.y += ib; }
    float2 b = __ldg(reinterpret_cast<const float2*>(row + t0));
    P[0] = a.x; P[1] = a.y; P[2] = b.x + ib; P[3] = b.y + ib;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int t = t0 - 2 + j;
      P[j] = (t >= 0 && t < L) ? __ldg(row + t) + ib : 0.f;
    }
  }
}

// short filter output at t0 and t0+1 (zero for positions >= L)
__device__ __forceinline__ float2 conv_pair(const float* __restrict__ row, int t0, int L, bool vec, const Taps& k) {
  float P[4];
  load_window(row, t0, L, vec, k.ib, P);
  float2 r;
  r.x = fmaf(k.w0, P[0], fmaf(k.w1, P[1], fmaf(k.w2, P[2], k.b)));
  r.y = (t0 + 1 < L) ? fmaf(k.w0, P[1], fmaf(k.w1, P[2], fmaf(k.w2, P[3], k.b))) : 0.f;
  return r;
}

__device__ __forceinline__ float2 conv_window(const float (&P)[4], int t0, int L, const Taps& k) {
  float2 r;
  r.x = fmaf(k.w0, P[0], fmaf(k.w1, P[1], fmaf(k.w2, P[2], k.b)));
  r.y = (t0 + 1 < L) ? fmaf(k.w0, P[1], fmaf(k.w1, P[2], fmaf(k.w2, P[3], k.b))) : 0.f;
  return r;
}

__device__ __forceinline__ float2 load_pair(const float* __restrict__ row, int t0, int L, bool vec) {
  if (vec) return __ldg(reinterpret_cast<const float2*>(row + t0));
  return make_float2(__ldg(row + t0), (t0 + 1 < L) ? __ldg(row + t0 + 1) : 0.f);
}
__device__ __forceinline__ void store_pair(float* __restrict__ row, int t0, int L, bool vec, float2 v) {
  if (vec) { *reinterpret_cast<float2*>(row + t0) = v; return; }
  row[t0] = v.x;
  if (t0 + 1 < L) row[t0 + 1] = v.y;
}


// ------------------------------------------------------------------------------------------------
// cp.async staging of the HBM operands of a column tile.  A thread's 32-point transform needs 16 row
// chunks of up to five tensors; pulling them through registers serialises the loads into batches
// (register pressure), so they are copied global -> shared with cp.async (no registers, everything in
// flight at once, 272-byte contiguous pieces per row) and the math then reads shared memory.
// Requires L % 4 == 0 and 16-byte aligned rows (PassArgs.stage); otherwise the register path is used.
// ------------------------------------------------------------------------------------------------
// rows [row0, row0+nrows) x columns [colbase, colbase+C) of the packed row `prow` (L floats), with a 4-float
// halo on the left (the 3-tap filter reaches back two samples).  dst pitch: 2C+4 floats.
template <int C, int M2>
__device__ __forceinline__ void stage_windows(float* dst, const float* __restrict__ prow, int row0, int nrows,
                                              int colbase, int L) {
  constexpr int PIECES = C / 2 + 1, WP = 2 * C + 4;
  for (int i = threadIdx.x; i < nrows * PIECES; i += blockDim.x) {
    const int rr = i / PIECES, pc = i - rr * PIECES;
    const int t = 2 * ((row0 + rr) * M2 + colbase) - 4 + 4 * pc;
    const bool ok = (t >= 0) && (t + 4 <= L);
    cp_async16(dst + rr * WP + 4 * pc, prow + (ok ? t : 0), ok);
  }
}
// same without halo (pitch 2C floats)
template <int C, int M2>
__device__ __forceinline__ void stage_plain(float* dst, const float* __restrict__ prow, int row0, int nrows,
                                            int colbase, int L) {
  constexpr int PIECES = C / 2, XP = 2 * C;
  for (int i = threadIdx.x; i < nrows * PIECES; i += blockDim.x) {
    const int rr = i / PIECES, pc = i - rr * PIECES;
    const int t = 2 * ((row0 + rr) * M2 + colbase) + 4 * pc;
    const bool ok = (t + 4 <= L);
    cp_async16(dst + rr * XP + 4 * pc, prow + (ok ? t : 0), ok);
  }
}
// window of a staged row: P(t0-2..t0+1) with the in_proj bias added to in-range samples
template <int C>
__device__ __forceinline__ void staged_window(const float* st, int rr, int col, int t0, float ib, float (&P)[4]) {
  const float* w = st + rr * (2 * C + 4) + 2 + 2 * col;
  const float2 lo = *reinterpret_cast<const float2*>(w);
  const float2 hi = *reinterpret_cast<const float2*>(w + 2);
  const float lb = (t0 >= 2) ? ib : 0.f;             // samples before t = 0 are the conv padding: no bias
  P[0] = lo.x + lb; P[1] = lo.y + lb; P[2] = hi.x + ib; P[3] = hi.y + ib;
}
template <int C>
__device__ __forceinline__ float2 staged_pair(const float* st, int rr, int col) {
  return *reinterpret_cast<const float2*>(st + rr * (2 * C) + 2 * col);
}

// ------------------------------------------------------------------------------------------------
// argument blocks
// ------------------------------------------------------------------------------------------------
enum ColMode { COL_FILTER = 0, COL_GATE = 1, COL_DC = 2, COL_PLAIN = 3 };
enum InvMode { INV_CONV_FWD = 0, INV_BWD_DG = 1, INV_DK = 2, INV_PLAIN_FWD = 3, INV_PLAIN_BWD = 4 };
enum RowMode { ROW_FILTER = 0, ROW_CONV_FWD = 1, ROW_CONV_BWD = 2 };

// Rows of one launch are numbered r = ci*B + b (all batches of a channel adjacent), channel c = c0 + ci.
struct PassArgs {
  int L;            // samples per row
  int logM1;        // M = 2^logM1 * 2^logM2
  int logM2;        // 10 or 12
  int B;            // batch
  int D;            // channels (d_model, or H for the plain fftconv API)
  int c0;           // first channel of this launch
  float scale;      // 1/(4M), applied by col_inv
  int vec;          // 1: L even and every row base 8-byte aligned -> float2 accesses
  int stage;        // 1: L % 4 == 0 and every row base 16-byte aligned -> cp.async staging of column tiles
  Twiddles T;
  float2* A;        // scratch rows [r][k1][m2]
  float2* A2;       // second scratch (bwd: rows of g)
  float2* A3;       // third scratch (bwd: per-channel dK' rows [ci][k1][m2])
  const float2* kspec;   // filter spectrum [c][k1][k2]
  float2* kspec_out;     // ROW_FILTER output
  float2* gspec;         // ROW_CONV_FWD: optional output, spectrum of g per (b,c) row; ROW_CONV_BWD: optional input
  // tensors (see include/hyena_b200.h for layouts)
  const float* src;      // COL_FILTER: k (D,L); COL_PLAIN / INV_PLAIN_*: u (B,H,L); COL_DC & INV_BWD_DG: dy_pre (B,D,L)
  const float* src2;     // INV_PLAIN_BWD: dout (B,H,L); INV_BWD_DG: c_saved (B,D,L)
  const float* p;        // (B,3D,L) in_proj output (bias not yet added)
  const float* in_bias;  // (3D) or null
  const float* sw;       // (3D,3)
  const float* sb;       // (3D)
  const float* fbias;    // (D) filter bias / D vector of the plain API
  float* out;            // INV_CONV_FWD: y_pre (B,D,L); INV_DK: dk (D,L); INV_PLAIN_*: out/du (B,H,L)
  float* out2;           // INV_CONV_FWD: c_save (B,D,L) or null; INV_BWD_DG: dconv (B,3D,L)
  float* red;            // INV_BWD_DG: dfbias (D); INV_PLAIN_BWD: dD (H)   (atomicAdd)
  float* dsw;            // INV_BWD_DG: d short_filter.weight (3D,3) (atomicAdd)
  float* dsb;            // INV_BWD_DG: d short_filter.bias (3D)     (atomicAdd)
};

__device__ __forceinline__ size_t row_off(int b, int ch, int nch, int L) { return ((size_t)b * nch + ch) * (size_t)L; }

// ------------------------------------------------------------------------------------------------
// column-pass geometry
// ------------------------------------------------------------------------------------------------
template <int LOGM1, int LOGM2>
struct ColGeo {
  static constexpr int M1 = 1 << LOGM1;
  static constexpr int M2 = 1 << LOGM2;
  static constexpr bool TWO = LOGM1 >= 5;                       // thread-group FFT (>= 32 points)
  static constexpr int R2 = TWO ? M1 / 32 : 1;
  static constexpr int G = TWO ? 1 : 32 / M1;                   // columns per thread when M1 < 32
  static constexpr int THREADS = TWO ? 256 : (32 * M1 < 256 ? 32 * M1 : 256);
  static constexpr int C = TWO ? 256 / R2 : THREADS * G;        // columns per CTA
  static constexpr int CTAS = M2 / C;                           // CTAs per row
  static constexpr int PAD = C >= 16 ? 1 : 16 / C;
  static constexpr int PITCH = TWO ? Geo<TWO ? LOGM1 : 5>::ex_elems() + PAD : 0;   // exchange elems per column
  static constexpr size_t EXCH = (R2 > 1) ? (size_t)C * PITCH * sizeof(float2) : 0;
  // cp.async staging (TWO only): forward needs two tensors of the M1/2 data rows; the inverse epilogue is
  // staged four slots (4*R2 rows) at a time with up to five tensors
  static constexpr int DATA_ROWS = M1 >= 2 ? M1 / 2 : 1;
  static constexpr int WP = 2 * C + 4, XP = 2 * C;               // staged row pitches (floats): with / without halo
  // inverse epilogue: double-buffered batches of SB slots (SB*R2 consecutive rows): 4 slots for the forward
  // epilogue (three windowed tensors), 2 for the backward one (three windowed + two plain tensors)
  static constexpr int SB_FWD = 8, SB_BWD = 4;
  static constexpr size_t STAGE_FWD = TWO ? (size_t)DATA_ROWS * (WP + WP) * sizeof(float) : 0;
  static constexpr size_t BATCH_FWD_FLOATS = (size_t)SB_FWD * R2 * WP;       // x0 windows only
  static constexpr size_t BATCH_BWD_FLOATS = (size_t)SB_BWD * R2 * (3 * WP + 2 * XP);
  // both epilogues are double buffered: the cp.async group of batch k+1 is in flight while batch k is consumed.  (Round 1 kept the
  // larger backward batches single buffered: eight HALF-size double-buffered batches in the same shared memory had been 2x slower;
  // with two full-size buffers -- 94 KB per CTA, two CTAs per SM still fit -- col_inv<bwd_dg> went 2.56 -> 2.36 ms.)
  // Shared memory per mode: the forward kernel keeps its smaller footprint.
  template <int MODE>
  static constexpr size_t stage_inv() {
    return TWO ? 2 * (MODE == INV_BWD_DG ? BATCH_BWD_FLOATS : BATCH_FWD_FLOATS) * sizeof(float) : 0;
  }
  template <int MODE>
  static constexpr size_t smem_inv() {
    return (MODE == INV_BWD_DG || MODE == INV_CONV_FWD) && stage_inv<MODE>() > EXCH ? stage_inv<MODE>() : EXCH;
  }
  static constexpr size_t SMEM_FWD = EXCH > STAGE_FWD ? EXCH : STAGE_FWD;
  static constexpr size_t SMEM = EXCH;
  static_assert(C <= M2, "column tile wider than a row");
};

struct CtaSync { __device__ __forceinline__ void operator()() const { __syncthreads(); } };
struct WarpSync { __device__ __forceinline__ void operator()() const { __syncwarp(); } };

// input sample pair (x[t0], x[t0+1]) of row (b, c) for the forward column pass
template <int MODE>
__device__ __forceinline__ float2 col_input(const PassArgs& a, int b, int c, int t0, bool vec,
                                            const Taps& ka, const Taps& kb) {
  if constexpr (MODE == COL_FILTER) {
    return load_pair(a.src + (size_t)c * a.L, t0, a.L, vec);
  } else if constexpr (MODE == COL_PLAIN) {
    return load_pair(a.src + row_off(b, c, a.D, a.L), t0, a.L, vec);
  } else if constexpr (MODE == COL_GATE) {      // g = short(v) * short(x1)        hyena.py:420
    float2 x1 = conv_pair(a.p + row_off(b, a.D + c, 3 * a.D, a.L), t0, a.L, vec, ka);
    float2 v = conv_pair(a.p + row_off(b, 2 * a.D + c, 3 * a.D, a.L), t0, a.L, vec, kb);
    return make_float2(x1.x * v.x, x1.y * v.y);
  } else {                                       // COL_DC: dc = dy_pre * short(x0)
    float2 x0 = conv_pair(a.p + row_off(b, c, 3 * a.D, a.L), t0, a.L, vec, ka);
    float2 dy = load_pair(a.src + row_off(b, c, a.D, a.L), t0, a.L, vec);
    return make_float2(x0.x * dy.x, x0.y * dy.y);
  }
}

// ------------------------------------------------------------------------------------------------
// pass 1: forward column FFT with the input side fused in
// grid (CTAS, rows); block ColGeo::THREADS
// ------------------------------------------------------------------------------------------------
// body of pass 1 for the column tile `bx` of row `by` (the __global__ wrapper passes blockIdx; the fused
// cooperative kernel loops over tiles)
template <int LOGM1, int LOGM2, int MODE>
__device__ __forceinline__ void col_fwd_body(const PassArgs& a, const int bx, const int by, unsigned char* smem_raw) {
  using CG = ColGeo<LOGM1, LOGM2>;
  constexpr int M1 = CG::M1;
  constexpr int kM2 = CG::M2;
  float2* smem = reinterpret_cast<float2*>(smem_raw);

  const int r = by;
  const int ci = r / a.B, b = r - ci * a.B, c = a.c0 + ci;
  const int colbase = bx * CG::C;
  const int L = a.L;
  const bool vec = a.vec != 0;
  constexpr int logM = LOGM1 + LOGM2;
  float2* Arow = a.A + (size_t)r * ((size_t)M1 * kM2);

  Taps ka{}, kb{};
  if constexpr (MODE == COL_GATE) {
    ka = load_taps(a.sw, a.sb, a.in_bias, a.D + c);
    kb = load_taps(a.sw, a.sb, a.in_bias, 2 * a.D + c);
  } else if constexpr (MODE == COL_DC) {
    ka = load_taps(a.sw, a.sb, a.in_bias, c);
  }

  float2 v[32];
  if constexpr (CG::TWO) {
    const int col = threadIdx.x % CG::C, q = threadIdx.x / CG::C;
    const int m2 = colbase + col;
    // slots n1 >= 16 (m1 >= M1/2) are the zero padding: never loaded
    if ((MODE == COL_GATE || MODE == COL_DC) && a.stage) {
      float* st0 = reinterpret_cast<float*>(smem_raw);
      float* st1 = st0 + CG::DATA_ROWS * CG::WP;
      if constexpr (MODE == COL_GATE) {
        stage_windows<CG::C, kM2>(st0, a.p + row_off(b, a.D + c, 3 * a.D, L), 0, CG::DATA_ROWS, colbase, L);
        stage_windows<CG::C, kM2>(st1, a.p + row_off(b, 2 * a.D + c, 3 * a.D, L), 0, CG::DATA_ROWS, colbase, L);
      } else {
        stage_windows<CG::C, kM2>(st0, a.p + row_off(b, c, 3 * a.D, L), 0, CG::DATA_ROWS, colbase, L);
        stage_plain<CG::C, kM2>(st1, a.src + row_off(b, c, a.D, L), 0, CG::DATA_ROWS, colbase, L);
      }
      cp_async_wait_all();
      __syncthreads();
      static_for<0, 16>([&](auto n_) {
        constexpr int n1 = decltype(n_)::value;
        const int m1 = CG::R2 * n1 + q;
        const int t0 = 2 * (m1 * kM2 + m2);
        float2 g = make_float2(0.f, 0.f);
        if (t0 < L) {
          float P[4];
          staged_window<CG::C>(st0, m1, col, t0, ka.ib, P);
          const float2 x = conv_window(P, t0, L, ka);
          if constexpr (MODE == COL_GATE) {
            staged_window<CG::C>(st1, m1, col, t0, kb.ib, P);
            const float2 y = conv_window(P, t0, L, kb);
            g = make_float2(x.x * y.x, x.y * y.y);
          } else {
            const float2 dy = staged_pair<CG::C>(st1, m1, col);
            g = make_float2(x.x * dy.x, x.y * dy.y);
          }
        }
        v[n1] = g;
      });
      __syncthreads();                                  // the staging area becomes the FFT exchange area
    } else {
      static_for<0, 16>([&](auto n_) {
        constexpr int n1 = decltype(n_)::value;
        const int m1 = CG::R2 * n1 + q;
        const int t0 = 2 * (m1 * kM2 + m2);
        v[n1] = (t0 < L) ? col_input<MODE>(a, b, c, t0, vec, ka, kb) : make_float2(0.f, 0.f);
      });
    }
    static_for<16, 32>([&](auto n_) { v[decltype(n_)::value] = make_float2(0.f, 0.f); });
    block_fft<CG::TWO ? LOGM1 : 5, false, true>(v, smem + col * CG::PITCH, q, a.T.tw1024, CtaSync{});
    // 4-step twiddle W_M^{m2*k1}, k1 = R2*s + q : geometric in s
    const uint32_t Mmask = (1u << logM) - 1u;
    const uint32_t eb = ((uint32_t)m2 * (uint32_t)q) & Mmask;
    const uint32_t es = ((uint32_t)m2 * (uint32_t)CG::R2) & Mmask;
    {
      float2 lo[8], hi[4];
      twiddle_factors20(a.T, eb, es, logM, lo, hi);
      mul_twiddles<false>(v, lo, hi, SlotIdx<CG::TWO ? LOGM1 : 5>{});
    }
    static_for<0, 32>([&](auto s_) {
      constexpr int s = decltype(s_)::value;
      const int k1 = CG::R2 * s + q;
      Arow[(size_t)k1 * kM2 + m2] = v[Geo<CG::TWO ? LOGM1 : 5>::slot(s)];
    });
  } else {
    // M1 < 32: a thread owns G whole columns; column gi lives in v[gi*M1 .. gi*M1+M1)
    static_for<0, CG::G>([&](auto g_) {
      constexpr int gi = decltype(g_)::value;
      const int m2 = colbase + threadIdx.x + CG::THREADS * gi;
      static_for<0, M1>([&](auto m_) {
        constexpr int m1 = decltype(m_)::value;
        const int t0 = 2 * (m1 * kM2 + m2);
        v[gi * M1 + m1] = (t0 < L) ? col_input<MODE>(a, b, c, t0, vec, ka, kb) : make_float2(0.f, 0.f);
      });
      dif<M1, gi * M1, false, 32>(v);
      static_for<0, M1>([&](auto k_) {
        constexpr int k1 = decltype(k_)::value;
        float2 x = v[gi * M1 + brev(k1, LOGM1)];
        if constexpr (k1 > 0) {
          const uint32_t e = ((uint32_t)m2 * (uint32_t)k1) & ((1u << logM) - 1u);
          x = cmul(x, root20(a.T, e << (20 - logM)));
        }
        Arow[(size_t)k1 * kM2 + m2] = x;
      });
    });
  }
}

template <int LOGM1, int LOGM2, int MODE>
__global__ void __launch_bounds__(ColGeo<LOGM1, LOGM2>::THREADS, ColGeo<LOGM1, LOGM2>::TWO ? 2 : 1)
col_fwd_kernel(const PassArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  col_fwd_body<LOGM1, LOGM2, MODE>(a, blockIdx.x, blockIdx.y, smem_raw);
}

// ------------------------------------------------------------------------------------------------
// pass 3: inverse column FFT with the output side fused in
// ------------------------------------------------------------------------------------------------
struct InvCtx {
  Taps k0, k1, k2;     // taps of x0, x1, v channels
  float red;           // per-thread partial of the reduction this mode produces
  float rw[3][3];      // INV_BWD_DG: partials of d short_filter.weight for the x0 / x1 / v channels
  float rb[3];         //             and of d short_filter.bias
};

// dw_j += ds[t0] P(t0-2+j) + ds[t0+1] P(t0-1+j);  db += ds[t0] + ds[t0+1]     (P = window of the filter input)
__device__ __forceinline__ void tap_grads(float (&rw)[3], float& rb, const float2 ds, const float (&P)[4]) {
  rw[0] = fmaf(ds.x, P[0], fmaf(ds.y, P[1], rw[0]));
  rw[1] = fmaf(ds.x, P[1], fmaf(ds.y, P[2], rw[1]));
  rw[2] = fmaf(ds.x, P[2], fmaf(ds.y, P[3], rw[2]));
  rb += ds.x + ds.y;
}

// Everything pass 3 reads from HBM for one sample pair, loaded up front so that a batch of slots has all
// its loads in flight before the first use (the epilogue is latency-bound otherwise).
struct InvIn {
  float P0[4], P1[4], P2[4];   // raw windows of the x0 / x1 / v rows of p
  float2 a, b;                 // mode-specific extra operands
};

template <int MODE>
__device__ __forceinline__ void inv_load(const PassArgs& a, const InvCtx& cx, int b, int c, int t0, bool vec, InvIn& in) {
  const int L = a.L, D = a.D;
  if constexpr (MODE == INV_PLAIN_FWD) {
    // nothing: out = y (the u * D skip term went into the filter spectrum in pass 2)
  } else if constexpr (MODE == INV_PLAIN_BWD) {
    in.a = load_pair(a.src2 + row_off(b, c, D, L), t0, L, vec);
    in.b = load_pair(a.src + row_off(b, c, D, L), t0, L, vec);
  } else if constexpr (MODE == INV_CONV_FWD) {
    load_window(a.p + row_off(b, c, 3 * D, L), t0, L, vec, cx.k0.ib, in.P0);     // x0 only: c = y already holds bias * g
  } else if constexpr (MODE == INV_BWD_DG) {
    load_window(a.p + row_off(b, c, 3 * D, L), t0, L, vec, cx.k0.ib, in.P0);
    load_window(a.p + row_off(b, D + c, 3 * D, L), t0, L, vec, cx.k1.ib, in.P1);
    load_window(a.p + row_off(b, 2 * D + c, 3 * D, L), t0, L, vec, cx.k2.ib, in.P2);
    in.a = load_pair(a.src + row_off(b, c, D, L), t0, L, vec);
    in.b = load_pair(a.src2 + row_off(b, c, D, L), t0, L, vec);
  }
}

// y = (y[t0], y[t0+1]) already scaled
template <int MODE>
__device__ __forceinline__ void inv_finish(const PassArgs& a, InvCtx& cx, int b, int c, int t0, bool vec, float2 y,
                                           const InvIn& in) {
  const int L = a.L, D = a.D;
  if constexpr (MODE == INV_DK) {
    store_pair(a.out + (size_t)c * L, t0, L, vec, y);
  } else if constexpr (MODE == INV_PLAIN_FWD) {       // out = y (+ u * D inside the spectrum)      hyena.py:82
    store_pair(a.out + row_off(b, c, D, L), t0, L, vec, y);
  } else if constexpr (MODE == INV_PLAIN_BWD) {       // du = corr (+ dout * D inside the spectrum) ; dD += dout * u
    cx.red = fmaf(in.a.x, in.b.x, fmaf(in.a.y, in.b.y, cx.red));
    store_pair(a.out + row_off(b, c, D, L), t0, L, vec, y);
  } else if constexpr (MODE == INV_CONV_FWD) {        // c = y (bias*g inside the spectrum) ; y_pre = c * x0   hyena.py:82, :432
    const float2 x0 = conv_window(in.P0, t0, L, cx.k0);
    if (a.out2) store_pair(a.out2 + row_off(b, c, D, L), t0, L, vec, y);
    store_pair(a.out + row_off(b, c, D, L), t0, L, vec, pmul(y, x0));
  } else {                                            // INV_BWD_DG
    const float2 x0 = conv_window(in.P0, t0, L, cx.k0), x1 = conv_window(in.P1, t0, L, cx.k1),
                 vv = conv_window(in.P2, t0, L, cx.k2);
    const float2 dy = in.a, cs = in.b;
    const float2 dc = pmul(dy, x0);
    const float2 dg = y;                                         // corr(dc, k) + bias * dc (skip term inside the spectrum)
    cx.red = fmaf(dc.x, x1.x * vv.x, fmaf(dc.y, x1.y * vv.y, cx.red));           // dbias += dc * g
    const float2 d0 = pmul(dy, cs);                              // d short(x0)
    const float2 d1 = pmul(dg, vv);                              // d short(x1)
    const float2 d2 = pmul(dg, x1);                              // d short(v)
    store_pair(a.out2 + row_off(b, c, 3 * D, L), t0, L, vec, d0);
    store_pair(a.out2 + row_off(b, D + c, 3 * D, L), t0, L, vec, d1);
    store_pair(a.out2 + row_off(b, 2 * D + c, 3 * D, L), t0, L, vec, d2);
    tap_grads(cx.rw[0], cx.rb[0], d0, in.P0);                    // short-filter weight / bias grads, fused here so
    tap_grads(cx.rw[1], cx.rb[1], d1, in.P1);                    // that short_conv_bwd need not re-read p
    tap_grads(cx.rw[2], cx.rb[2], d2, in.P2);
  }
}

template <int MODE>
__device__ __forceinline__ void inv_output(const PassArgs& a, InvCtx& cx, int b, int c, int t0, bool vec, float2 y) {
  InvIn in;
  inv_load<MODE>(a, cx, b, c, t0, vec, in);
  inv_finish<MODE>(a, cx, b, c, t0, vec, y, in);
}

template <int LOGM1, int LOGM2, int MODE>
__device__ __forceinline__ void col_inv_body(const PassArgs& a, const int bx, const int by, unsigned char* smem_raw) {
  using CG = ColGeo<LOGM1, LOGM2>;
  constexpr int M1 = CG::M1;
  constexpr int kM2 = CG::M2;
  float2* smem = reinterpret_cast<float2*>(smem_raw);

  const int r = by;
  const int ci = r / a.B, b = r - ci * a.B, c = a.c0 + ci;
  const int colbase = bx * CG::C;
  const int L = a.L;
  const bool vec = a.vec != 0;
  const float2* Arow = (MODE == INV_DK ? a.A3 : a.A) + (size_t)r * ((size_t)M1 * kM2);

  InvCtx cx{};
  cx.red = 0.f;
  if constexpr (MODE == INV_CONV_FWD || MODE == INV_BWD_DG) cx.k0 = load_taps(a.sw, a.sb, a.in_bias, c);
  if constexpr (MODE == INV_BWD_DG) {
    cx.k1 = load_taps(a.sw, a.sb, a.in_bias, a.D + c);
    cx.k2 = load_taps(a.sw, a.sb, a.in_bias, 2 * a.D + c);
  }

  float2 v[32];
  if constexpr (CG::TWO) {
    const int col = threadIdx.x % CG::C, q = threadIdx.x / CG::C;
    const int m2 = colbase + col;
    static_for<0, 32>([&](auto n_) {
      constexpr int n1 = decltype(n_)::value;
      v[n1] = Arow[(size_t)(CG::R2 * n1 + q) * kM2 + m2];
    });
    block_fft<CG::TWO ? LOGM1 : 5, true, false>(v, smem + col * CG::PITCH, q, a.T.tw1024, CtaSync{});
    // only m1 < M1/2 (slots s < 16) can hold samples t < L
    if ((MODE == INV_CONV_FWD || MODE == INV_BWD_DG) && a.stage) {
      // epilogue operands staged through shared memory, SB slots (SB*R2 consecutive rows) per batch; forward:
      // double buffered, the cp.async group of batch k+1 is in flight while batch k is consumed
      constexpr bool DBL = true;
      constexpr int SB = (MODE == INV_BWD_DG) ? CG::SB_BWD : CG::SB_FWD;
      constexpr int NBATCH = 16 / SB;
      constexpr int BROWS = SB * CG::R2;
      constexpr size_t BFLOATS = (MODE == INV_BWD_DG) ? CG::BATCH_BWD_FLOATS : CG::BATCH_FWD_FLOATS;
      float* st = reinterpret_cast<float*>(smem_raw);
      const float* p0 = a.p + row_off(b, c, 3 * a.D, L);
      const float* p1 = a.p + row_off(b, a.D + c, 3 * a.D, L);
      const float* p2 = a.p + row_off(b, 2 * a.D + c, 3 * a.D, L);
      auto issue = [&](int k) {
        float* w0 = st + (size_t)(DBL ? (k & 1) : 0) * BFLOATS;
        float* w1 = w0 + BROWS * CG::WP;
        float* w2 = w1 + BROWS * CG::WP;
        const int row0 = BROWS * k;
        stage_windows<CG::C, kM2>(w0, p0, row0, BROWS, colbase, L);
        if constexpr (MODE == INV_BWD_DG) {
          stage_windows<CG::C, kM2>(w1, p1, row0, BROWS, colbase, L);
          stage_windows<CG::C, kM2>(w2, p2, row0, BROWS, colbase, L);
          float* x0 = w2 + BROWS * CG::WP;
          float* x1 = x0 + BROWS * CG::XP;
          stage_plain<CG::C, kM2>(x0, a.src + row_off(b, c, a.D, L), row0, BROWS, colbase, L);
          stage_plain<CG::C, kM2>(x1, a.src2 + row_off(b, c, a.D, L), row0, BROWS, colbase, L);
        }
        cp_async_commit();
      };
      __syncthreads();                                  // the FFT exchange area is free
      if constexpr (DBL) issue(0);
      static_for<0, NBATCH>([&](auto g_) {
        constexpr int k = decltype(g_)::value;
        if constexpr (DBL) {
          if constexpr (k + 1 < NBATCH) { issue(k + 1); cp_async_wait_group<1>(); } else { cp_async_wait_group<0>(); }
        } else {
          issue(k);
          cp_async_wait_group<0>();
        }
        __syncthreads();
        const float* w0 = st + (size_t)(DBL ? (k & 1) : 0) * BFLOATS;
        const float* w1 = w0 + BROWS * CG::WP;
        const float* w2 = w1 + BROWS * CG::WP;
        [[maybe_unused]] const float* x0 = w2 + BROWS * CG::WP;
        [[maybe_unused]] const float* x1 = x0 + BROWS * CG::XP;
        static_for<0, SB>([&](auto j_) {
          constexpr int j = decltype(j_)::value;
          constexpr int s = k * SB + j;
          const int m1 = CG::R2 * s + q;
          const int t0 = 2 * (m1 * kM2 + m2);
          if (t0 < L) {
            InvIn in;
            const int rr = m1 - BROWS * k;
            staged_window<CG::C>(w0, rr, col, t0, cx.k0.ib, in.P0);
            if constexpr (MODE == INV_BWD_DG) {
              staged_window<CG::C>(w1, rr, col, t0, cx.k1.ib, in.P1);
              staged_window<CG::C>(w2, rr, col, t0, cx.k2.ib, in.P2);
              in.a = staged_pair<CG::C>(x0, rr, col);
              in.b = staged_pair<CG::C>(x1, rr, col);
            }
            float2 y = v[Geo<CG::TWO ? LOGM1 : 5>::slot(s)];
            inv_finish<MODE>(a, cx, b, c, t0, vec, make_float2(y.x * a.scale, y.y * a.scale), in);
          }
        });
        if constexpr (DBL ? (k + 2 < NBATCH) : (k + 1 < NBATCH)) __syncthreads();   // the buffer is refilled next round
      });
    } else {
      // register path: slots are handled four at a time with all their loads issued before the first use
      constexpr int NB = (MODE == INV_DK) ? 1 : 4;
      static_for<0, 16 / NB>([&](auto g_) {
        constexpr int s0 = decltype(g_)::value * NB;
        InvIn in[NB];
        static_for<0, NB>([&](auto j_) {
          constexpr int j = decltype(j_)::value;
          const int t0 = 2 * ((CG::R2 * (s0 + j) + q) * kM2 + m2);
          if (t0 < L) inv_load<MODE>(a, cx, b, c, t0, vec, in[j]);
        });
        static_for<0, NB>([&](auto j_) {
          constexpr int j = decltype(j_)::value;
          const int t0 = 2 * ((CG::R2 * (s0 + j) + q) * kM2 + m2);
          if (t0 < L) {
            float2 y = v[Geo<CG::TWO ? LOGM1 : 5>::slot(s0 + j)];
            inv_finish<MODE>(a, cx, b, c, t0, vec, make_float2(y.x * a.scale, y.y * a.scale), in[j]);
          }
        });
      });
    }
  } else {
    static_for<0, CG::G>([&](auto g_) {
      constexpr int gi = decltype(g_)::value;
      const int m2 = colbase + threadIdx.x + CG::THREADS * gi;
      static_for<0, M1>([&](auto k_) {
        constexpr int k1 = decltype(k_)::value;
        v[gi * M1 + k1] = Arow[(size_t)k1 * kM2 + m2];
      });
      dif<M1, gi * M1, true, 32>(v);
      static_for<0, (M1 >= 2 ? M1 / 2 : 1)>([&](auto m_) {
        constexpr int m1 = decltype(m_)::value;
        const int t0 = 2 * (m1 * kM2 + m2);
        if (t0 < L) {
          float2 y = v[gi * M1 + brev(m1, LOGM1)];
          inv_output<MODE>(a, cx, b, c, t0, vec, make_float2(y.x * a.scale, y.y * a.scale));
        }
      });
    });
  }

  if constexpr (MODE == INV_BWD_DG || MODE == INV_PLAIN_BWD) {
    constexpr int NR = (MODE == INV_BWD_DG) ? 13 : 1;
    __shared__ float red_all[8][NR];
    float vals[NR];
    vals[0] = cx.red;
    if constexpr (MODE == INV_BWD_DG) {
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
#pragma unroll
        for (int j = 0; j < 3; ++j) vals[1 + 3 * ch + j] = cx.rw[ch][j];
        vals[10 + ch] = cx.rb[ch];
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NR; ++i) {
      float s = vals[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if ((threadIdx.x & 31) == 0) red_all[threadIdx.x >> 5][i] = s;
    }
    __syncthreads();
    if (threadIdx.x < NR) {
      float tot = 0.f;
      for (int w = 0; w < (CG::THREADS + 31) / 32; ++w) tot += red_all[w][threadIdx.x];
      const int i = threadIdx.x;
      if (i == 0) atomicAdd(a.red + c, tot);
      else if (i < 10) atomicAdd(a.dsw + 3 * (((i - 1) / 3) * a.D + c) + (i - 1) % 3, tot);
      else atomicAdd(a.dsb + (i - 10) * a.D + c, tot);
    }
  }
}

template <int LOGM1, int LOGM2, int MODE>
__global__ void __launch_bounds__(ColGeo<LOGM1, LOGM2>::THREADS, ColGeo<LOGM1, LOGM2>::TWO ? 2 : 1)
col_inv_kernel(const PassArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  col_inv_body<LOGM1, LOGM2, MODE>(a, blockIdx.x, blockIdx.y, smem_raw);
}

// ------------------------------------------------------------------------------------------------
// pass 2: row FFTs + pointwise spectrum product + inverse row FFTs
// A row of M2 = 2^LOGM2 points is owned by TPR = M2/32 threads (one warp for 1024, four for 4096);
// a CTA of 256 threads holds 256/TPR rows, arranged so that both rows of a (k, M-k) pair sit in the
// same CTA.  grid (pairs / pairs-per-CTA, channel-rows)
// ------------------------------------------------------------------------------------------------
template <int LOGM2>
struct RowGeo {
  static constexpr int M2 = 1 << LOGM2;
  static constexpr int TPR = M2 / 32;                         // threads per row
  static constexpr int ROWS = 256 / TPR;                      // rows per full CTA (8 or 2)
  static constexpr int EX = 32 * 33;                          // exchange elems per row (>= M2: also holds a spectrum)
  static_assert(EX >= M2, "the exchange area doubles as a natural-order row buffer");
};

struct RowIds {
  int k1;        // this row
  int pk1;       // row holding the partner bins
  int pslot;     // row slot of this CTA that holds row pk1
  int nz;        // 1 if k1 != 0 (partner column is M2-1-k2 instead of (M2-k2)%M2)
};

__device__ __forceinline__ RowIds row_ids(int M1, int rows_per_cta, int cta, int slot) {
  RowIds id;
  if (M1 == 1) { id.k1 = 0; id.pk1 = 0; id.pslot = 0; id.nz = 0; return id; }
  const int pair = cta * (rows_per_cta / 2) + (slot >> 1);      // pair 0 = rows (0, M1/2), both self-paired
  const int second = slot & 1;
  if (pair == 0) {
    id.k1 = second ? M1 / 2 : 0;
    id.pk1 = id.k1; id.pslot = slot;
  } else {
    id.k1 = second ? M1 - pair : pair;
    id.pk1 = M1 - id.k1; id.pslot = slot ^ 1;
  }
  id.nz = id.k1 != 0;
  return id;
}

// barrier over the TPR threads of one row
template <int LOGM2>
struct RowSync {
  int id;
  __device__ __forceinline__ void operator()() const {
    if constexpr (LOGM2 == 10) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(RowGeo<LOGM2>::TPR) : "memory");
  }
};

template <int LOGM2, bool INV>
__device__ __forceinline__ void row_fft(float2 (&v)[32], float2* ex, int q, const Twiddles& T, RowSync<LOGM2> sync) {
  static_assert(LOGM2 == 10, "1024-point rows");
  block_fft<10, INV, false>(v, ex, q, T.tw1024, sync);
}
template <int LOGM2>
struct RowSlot {
  __host__ __device__ static constexpr int at(int s) { return Geo<10>::slot(s); }
};

// forward FFT of one row; natural bin k2 = TPR*s + q left in dst[k2] (dst may be `ex` itself)
template <int LOGM2>
__device__ __forceinline__ void row_fft_to_smem(const float2* __restrict__ src, float2* ex, float2* dst, int q,
                                                const Twiddles& T, RowSync<LOGM2> sync) {
  constexpr int TPR = RowGeo<LOGM2>::TPR;
  float2 v[32];
  static_for<0, 32>([&](auto n_) {
    constexpr int n1 = decltype(n_)::value;
    v[n1] = src[TPR * n1 + q];
  });
  row_fft<LOGM2, false>(v, ex, q, T, sync);
  if (dst == ex) sync();                               // all reads of the exchange area are done
  static_for<0, 32>([&](auto s_) {
    constexpr int s = decltype(s_)::value;
    dst[TPR * s + q] = v[RowSlot<LOGM2>::at(s)];
  });
}

// inverse FFT of v (natural slots), conj 4-step twiddle W_M^{-k1 m2}, store to dst[m2 = TPR*s + q]
template <int LOGM2>
__device__ __forceinline__ void row_ifft_store(float2 (&v)[32], float2* ex, float2* __restrict__ dst, int q, int k1,
                                               int logM, const Twiddles& T, RowSync<LOGM2> sync) {
  constexpr int TPR = RowGeo<LOGM2>::TPR;
  row_fft<LOGM2, true>(v, ex, q, T, sync);
  const uint32_t Mmask = (1u << logM) - 1u;
  const uint32_t eb = ((uint32_t)k1 * (uint32_t)q) & Mmask;
  const uint32_t es = ((uint32_t)k1 * (uint32_t)TPR) & Mmask;
  {
    float2 lo[8], hi[4];
    twiddle_factors20(T, eb, es, logM, lo, hi);
    mul_twiddles<true>(v, lo, hi, RowSlot<LOGM2>{});
  }
  static_for<0, 32>([&](auto s_) {
    constexpr int s = decltype(s_)::value;
    dst[TPR * s + q] = v[RowSlot<LOGM2>::at(s)];
  });
}

// E2 = Z + conj(P), O2 = -i (Z - conj(P))    (P already conjugated by the caller)
__device__ __forceinline__ void even_odd(float2 z, float2 pc, float2& e, float2& o) {
  e = cadd(z, pc);
  o = cmul_negi(csub(z, pc));
}
// Same for the filter spectrum, with the skip term folded in: y = conv(k, g) + bias * g == conv(k + bias * delta, g), and
// adding `bias` to k[0] adds the real constant `bias` to every bin of the packed spectrum, i.e. 2 * bias to the (doubled)
// even part and nothing to the odd part.  The output pass then never re-reads g (hyena.py:82; fftconv_cuda.cu:470-476
// adds u * D in its epilogue instead).  fb2 = 2 * bias.
__device__ __forceinline__ void even_odd_filter(float2 z, float2 pc, float fb2, float2& e, float2& o) {
  e = cadd(z, pc);
  e.x += fb2;
  o = cmul_negi(csub(z, pc));
}

// shared memory per CTA (complex elements): FILTER: rows*EX; CONV_FWD: rows*EX (spectrum aliased onto the
// exchange area); CONV_BWD: rows*(EX + M2) (dc spectrum separate, g spectrum aliased onto the exchange area)
template <int MODE, int LOGM2>
__host__ __device__ constexpr size_t row_smem_elems(int rows) {
  return (size_t)rows * (RowGeo<LOGM2>::EX + (MODE == ROW_CONV_BWD ? RowGeo<LOGM2>::M2 : 0));
}

template <int MODE, int LOGM2>
__device__ __forceinline__ void row_pass_body(const PassArgs& a, const int bx, const int by, unsigned char* smem_raw) {
  using RG = RowGeo<LOGM2>;
  constexpr int M2 = RG::M2, TPR = RG::TPR;
  float2* smem = reinterpret_cast<float2*>(smem_raw);
  const int M1 = 1 << a.logM1;
  const int logM = a.logM1 + LOGM2;
  const int slot = threadIdx.x / TPR, q = threadIdx.x % TPR;
  const int nslots = blockDim.x / TPR;
  const RowIds id = row_ids(M1, nslots, bx, slot);
  const size_t rowElems = (size_t)M1 * M2;
  const RowSync<LOGM2> rsync{1 + slot};

  float2* ex = smem + slot * RG::EX;                    // exchange area, doubles as a spectrum buffer
  float2* exp_ = smem + id.pslot * RG::EX;              // the partner row's
  float2* zbuf = smem + nslots * RG::EX + slot * M2;    // ROW_CONV_BWD only: dc spectrum
  float2* zbufp = smem + nslots * RG::EX + id.pslot * M2;

  if constexpr (MODE == ROW_FILTER) {
    const int c = a.c0 + by;
    const float2* src = a.A + (size_t)by * rowElems + (size_t)id.k1 * M2;
    float2* dst = a.kspec_out + (size_t)c * rowElems + (size_t)id.k1 * M2;
    float2 v[32];
    static_for<0, 32>([&](auto n_) { constexpr int n1 = decltype(n_)::value; v[n1] = src[TPR * n1 + q]; });
    row_fft<LOGM2, false>(v, ex, q, a.T, rsync);
    static_for<0, 32>([&](auto s_) {
      constexpr int s = decltype(s_)::value;
      dst[TPR * s + q] = v[RowSlot<LOGM2>::at(s)];
    });
    return;
  } else {
    // W_M^k for k = k1 + M1*(TPR s + q) = base * W_32^s,  base = W_M^{k1} * W_{M2}^{q}
    const float2 wbase = root20(a.T, ((uint32_t)id.k1 + ((uint32_t)q << a.logM1)) << (20 - logM));
    // skip-term coefficient of this row's channel (filter bias / D vector), doubled: see even_odd_filter
    const int c_row = a.c0 + ((MODE == ROW_CONV_FWD) ? by / a.B : by);
    const float fb2 = a.fbias ? 2.f * __ldg(a.fbias + c_row) : 0.f;

    if constexpr (MODE == ROW_CONV_FWD) {
      const int r = by;
      const int ci = r / a.B, c = a.c0 + ci;
      float2* Arow = a.A + (size_t)r * rowElems + (size_t)id.k1 * M2;
      const float2* Krow = a.kspec + (size_t)c * rowElems + (size_t)id.k1 * M2;
      const float2* Kprow = a.kspec + (size_t)c * rowElems + (size_t)id.pk1 * M2;
      row_fft_to_smem<LOGM2>(Arow, ex, ex, q, a.T, rsync);
      if (a.gspec) {                                    // keep the spectrum of g for the backward pass
        float2* G = a.gspec + ((size_t)ci * a.B + (r - ci * a.B) + (size_t)a.c0 * a.B) * rowElems + (size_t)id.k1 * M2;
        static_for<0, 32>([&](auto s_) { constexpr int s = decltype(s_)::value; G[TPR * s + q] = ex[TPR * s + q]; });
      }
      __syncthreads();
      float2 v[32];
      static_for<0, 32>([&](auto s_) {
        constexpr int s = decltype(s_)::value;
        const int k2 = TPR * s + q;
        const int pc = (M2 - k2 - id.nz) & (M2 - 1);
        float2 E, O, He, Ho;
        even_odd(ex[k2], cconj(exp_[pc]), E, O);
        even_odd_filter(__ldg(Krow + k2), cconj(__ldg(Kprow + pc)), fb2, He, Ho);
        const float2 W = mul_w32<s, false>(wbase);
        float2 Ye = cadd(cmul(E, He), cmul(W, cmul(O, Ho)));
        float2 Yo = cadd(cmul(E, Ho), cmul(O, He));
        v[s] = cadd(Ye, cmul_i(Yo));
      });
      __syncthreads();                                  // partner rows are done reading this row's spectrum
      row_ifft_store<LOGM2>(v, ex, Arow, q, id.k1, logM, a.T, rsync);
    } else {   // ROW_CONV_BWD: loop over the batch, accumulate dK' in registers
      const int ci = by, c = a.c0 + ci;
      const float2* Krow = a.kspec + (size_t)c * rowElems + (size_t)id.k1 * M2;
      const float2* Kprow = a.kspec + (size_t)c * rowElems + (size_t)id.pk1 * M2;
      float2 acc[32];
      static_for<0, 32>([&](auto s_) { acc[decltype(s_)::value] = make_float2(0.f, 0.f); });
      for (int b = 0; b < a.B; ++b) {
        const size_t r = (size_t)ci * a.B + b;
        float2* Drow = a.A + r * rowElems + (size_t)id.k1 * M2;
        const float2* Grow = a.A2 + r * rowElems + (size_t)id.k1 * M2;
        row_fft_to_smem<LOGM2>(Drow, ex, zbuf, q, a.T, rsync);     // dc spectrum -> zbuf
        rsync();
        if (a.gspec) {                                             // saved by the forward pass: just load it
          const float2* G = a.gspec + ((size_t)(a.c0 + ci) * a.B + b) * rowElems + (size_t)id.k1 * M2;
          static_for<0, 32>([&](auto s_) { constexpr int s = decltype(s_)::value; ex[TPR * s + q] = __ldg(G + TPR * s + q); });
        } else {
          row_fft_to_smem<LOGM2>(Grow, ex, ex, q, a.T, rsync);     // g spectrum  -> the exchange area itself
        }
        __syncthreads();
        float2 v[32];
        static_for<0, 32>([&](auto s_) {
          constexpr int s = decltype(s_)::value;
          const int k2 = TPR * s + q;
          const int pc = (M2 - k2 - id.nz) & (M2 - 1);
          float2 E, O, He, Ho, Ge, Go;
          even_odd(zbuf[k2], cconj(zbufp[pc]), E, O);
          even_odd_filter(__ldg(Krow + k2), cconj(__ldg(Kprow + pc)), fb2, He, Ho);
          even_odd(ex[k2], cconj(exp_[pc]), Ge, Go);
          const float2 W = mul_w32<s, false>(wbase);
          const float2 WE = cmulc(E, W);                                  // conj(W) * E
          // dg spectrum: corr(dc, k)
          float2 Ye = cadd(cmulc(E, He), cmulc(O, Ho));
          float2 Yo = cadd(cmulc(WE, Ho), cmulc(O, He));
          v[s] = cadd(Ye, cmul_i(Yo));
          // dk spectrum: corr(dc, g), summed over the batch
          float2 Ke = cadd(cmulc(E, Ge), cmulc(O, Go));
          float2 Ko = cadd(cmulc(WE, Go), cmulc(O, Ge));
          acc[s] = cadd(acc[s], cadd(Ke, cmul_i(Ko)));
        });
        __syncthreads();                                // spectra consumed: the exchange area may be reused
        row_ifft_store<LOGM2>(v, ex, Drow, q, id.k1, logM, a.T, rsync);
        rsync();
      }
      float2* Krow_out = a.A3 + (size_t)ci * rowElems + (size_t)id.k1 * M2;
      row_ifft_store<LOGM2>(acc, ex, Krow_out, q, id.k1, logM, a.T, rsync);
    }
  }
}

// Batch-1 form of ROW_CONV_BWD with the spectrum of g saved by the forward pass: no register accumulator across the batch
// (the dc spectrum stays in shared memory between the two pointwise/inverse phases).  The filter spectrum row and then
// the saved g spectrum row are staged through shared memory by cp.async (issued before the forward row FFT / before the
// first inverse FFT, so the 2 x 64 dependent __ldg's per thread of the two pointwise phases -- `long_scoreboard`, the top
// stall of the register-load form -- become shared-memory reads).  One 8 KB buffer per row, reused for k then g; the
// partner row's buffer supplies the mirrored bins.  Shared memory per CTA: rows * (EX + 2 * M2) complex = 99 KB for four
// rows, two CTAs per SM.  2.75 vs 3.51 ms for the register-load form at large-1m (profiles/r2_ab.txt).
template <int LOGM2>
__host__ __device__ constexpr size_t row_bwd1_staged_smem_elems(int rows) {
  return (size_t)rows * (RowGeo<LOGM2>::EX + 2 * RowGeo<LOGM2>::M2);
}

template <int LOGM2>
__device__ __forceinline__ void row_bwd1_staged_body(const PassArgs& a, const int bx, const int by, unsigned char* smem_raw) {
  using RG = RowGeo<LOGM2>;
  constexpr int M2 = RG::M2, TPR = RG::TPR;
  static_assert(LOGM2 == 10, "one warp per row");
  float2* smem = reinterpret_cast<float2*>(smem_raw);
  const int M1 = 1 << a.logM1;
  const int logM = a.logM1 + LOGM2;
  const int slot = threadIdx.x / TPR, q = threadIdx.x % TPR;
  const int nslots = blockDim.x / TPR;
  const RowIds id = row_ids(M1, nslots, bx, slot);
  const size_t rowElems = (size_t)M1 * M2;
  const RowSync<LOGM2> rsync{1 + slot};

  float2* ex = smem + slot * RG::EX;
  float2* zbuf = smem + nslots * RG::EX + slot * M2;
  float2* zbufp = smem + nslots * RG::EX + id.pslot * M2;
  float2* kg = smem + nslots * (RG::EX + M2) + slot * M2;            // staged k row, later staged g row
  const float2* kgp = smem + nslots * (RG::EX + M2) + id.pslot * M2;

  const int ci = by, c = a.c0 + ci;                                  // B == 1
  const float2* Krow = a.kspec + (size_t)c * rowElems + (size_t)id.k1 * M2;
  const float2* Grow = a.gspec + (size_t)c * rowElems + (size_t)id.k1 * M2;
  float2* Drow = a.A + (size_t)ci * rowElems + (size_t)id.k1 * M2;
  auto stage_row = [&](const float2* src) {                          // 8 KB = 512 x 16 B, 16 per lane, coalesced
#pragma unroll
    for (int i = 0; i < M2 / 2 / TPR; ++i) {
      const int e = 2 * (TPR * i + q);
      cp_async16(kg + e, src + e, true);
    }
    cp_async_commit();
  };
  const float2 wbase = root20(a.T, ((uint32_t)id.k1 + ((uint32_t)q << a.logM1)) << (20 - logM));

  const float fb2 = a.fbias ? 2.f * __ldg(a.fbias + c) : 0.f;
  stage_row(Krow);                                                   // in flight under the forward FFT
  row_fft_to_smem<LOGM2>(Drow, ex, zbuf, q, a.T, rsync);             // dc spectrum -> zbuf (kept for both phases)
  cp_async_wait_group<0>();
  __syncthreads();                                                   // own + partner: dc spectrum and k row visible
  float2 v[32];
  static_for<0, 32>([&](auto s_) {                                   // phase 1: dg spectrum = corr(dc, k)
    constexpr int s = decltype(s_)::value;
    const int k2 = TPR * s + q;
    const int pc = (M2 - k2 - id.nz) & (M2 - 1);
    float2 E, O, He, Ho;
    even_odd(zbuf[k2], cconj(zbufp[pc]), E, O);
    even_odd_filter(kg[k2], cconj(kgp[pc]), fb2, He, Ho);
    const float2 WE = cmulc(E, mul_w32<s, false>(wbase));
    float2 Ye = cadd(cmulc(E, He), cmulc(O, Ho));
    float2 Yo = cadd(cmulc(WE, Ho), cmulc(O, He));
    v[s] = cadd(Ye, cmul_i(Yo));
  });
  __syncthreads();                                                   // the partner is done with this row's k
  stage_row(Grow);                                                   // in flight under the first inverse FFT
  row_ifft_store<LOGM2>(v, ex, Drow, q, id.k1, logM, a.T, rsync);
  cp_async_wait_group<0>();
  __syncthreads();                                                   // own + partner g rows visible
  static_for<0, 32>([&](auto s_) {                                   // phase 2: dk spectrum = corr(dc, g)
    constexpr int s = decltype(s_)::value;
    const int k2 = TPR * s + q;
    const int pc = (M2 - k2 - id.nz) & (M2 - 1);
    float2 E, O, Ge, Go;
    even_odd(zbuf[k2], cconj(zbufp[pc]), E, O);
    even_odd(kg[k2], cconj(kgp[pc]), Ge, Go);
    const float2 WE = cmulc(E, mul_w32<s, false>(wbase));
    float2 Ke = cadd(cmulc(E, Ge), cmulc(O, Go));
    float2 Ko = cadd(cmulc(WE, Go), cmulc(O, Ge));
    v[s] = cadd(Ke, cmul_i(Ko));
  });
  float2* Krow_out = a.A3 + (size_t)ci * rowElems + (size_t)id.k1 * M2;
  row_ifft_store<LOGM2>(v, ex, Krow_out, q, id.k1, logM, a.T, rsync);
}

// ------------------------------------------------------------------------------------------------
// Forward row pass with the filter spectrum row staged by cp.async under the forward row FFT (the register form issues 64
// __ldg per thread right in front of the pointwise product: long_scoreboard is its top stall).  128-thread CTAs of four
// rows, shared memory rows * (EX + M2) complex = 66.6 KB: three CTAs per SM.  2.13 -> 1.98 ms at large-1m
// (profiles/r2_ab.txt run E; a 256-thread staged form with 131 KB per CTA had lost in round 2's first sweep).  Needs a
// 16-byte aligned kspec and M1 >= 4; otherwise row_pass_kernel<ROW_CONV_FWD> runs.
// ------------------------------------------------------------------------------------------------
template <int LOGM2>
__host__ __device__ constexpr size_t row_fwd_staged_smem_elems(int rows) {
  return (size_t)rows * (RowGeo<LOGM2>::EX + RowGeo<LOGM2>::M2);
}

template <int LOGM2>
__device__ __forceinline__ void row_fwd_staged_body(const PassArgs& a, const int bx, const int by, unsigned char* smem_raw) {
  using RG = RowGeo<LOGM2>;
  constexpr int M2 = RG::M2, TPR = RG::TPR;
  float2* smem = reinterpret_cast<float2*>(smem_raw);
  const int M1 = 1 << a.logM1;
  const int logM = a.logM1 + LOGM2;
  const int slot = threadIdx.x / TPR, q = threadIdx.x % TPR;
  const int nslots = blockDim.x / TPR;
  const RowIds id = row_ids(M1, nslots, bx, slot);
  const size_t rowElems = (size_t)M1 * M2;
  const RowSync<LOGM2> rsync{1 + slot};
  float2* ex = smem + slot * RG::EX;
  const float2* exp_ = smem + id.pslot * RG::EX;
  float2* kg = smem + nslots * RG::EX + slot * M2;
  const float2* kgp = smem + nslots * RG::EX + id.pslot * M2;

  const int r = by;
  const int ci = r / a.B, c = a.c0 + ci;
  float2* Arow = a.A + (size_t)r * rowElems + (size_t)id.k1 * M2;
  const float2* Krow = a.kspec + (size_t)c * rowElems + (size_t)id.k1 * M2;
#pragma unroll
  for (int i = 0; i < M2 / 2 / TPR; ++i) {                           // 8 KB = 512 x 16 B, 16 per lane, coalesced
    const int e = 2 * (TPR * i + q);
    cp_async16(kg + e, Krow + e, true);
  }
  cp_async_commit();
  const float2 wbase = root20(a.T, ((uint32_t)id.k1 + ((uint32_t)q << a.logM1)) << (20 - logM));
  const float fb2 = a.fbias ? 2.f * __ldg(a.fbias + c) : 0.f;
  row_fft_to_smem<LOGM2>(Arow, ex, ex, q, a.T, rsync);
  if (a.gspec) {                                                     // keep the spectrum of g for the backward pass
    float2* G = a.gspec + ((size_t)ci * a.B + (r - ci * a.B) + (size_t)a.c0 * a.B) * rowElems + (size_t)id.k1 * M2;
    static_for<0, 32>([&](auto s_) { constexpr int s = decltype(s_)::value; G[TPR * s + q] = ex[TPR * s + q]; });
  }
  cp_async_wait_group<0>();
  __syncthreads();                                                   // own + partner: spectrum and k row visible
  float2 v[32];
  static_for<0, 32>([&](auto s_) {
    constexpr int s = decltype(s_)::value;
    const int k2 = TPR * s + q;
    const int pc = (M2 - k2 - id.nz) & (M2 - 1);
    float2 E, O, He, Ho;
    even_odd(ex[k2], cconj(exp_[pc]), E, O);
    even_odd_filter(kg[k2], cconj(kgp[pc]), fb2, He, Ho);
    const float2 W = mul_w32<s, false>(wbase);
    float2 Ye = cadd(cmul(E, He), cmul(W, cmul(O, Ho)));
    float2 Yo = cadd(cmul(E, Ho), cmul(O, He));
    v[s] = cadd(Ye, cmul_i(Yo));
  });
  __syncthreads();                                                   // partner rows are done reading this row's spectrum
  row_ifft_store<LOGM2>(v, ex, Arow, q, id.k1, logM, a.T, rsync);
}

template <int MODE, int LOGM2>
__global__ void __launch_bounds__(256, MODE == ROW_CONV_BWD ? 1 : 2)
row_pass_kernel(const PassArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  row_pass_body<MODE, LOGM2>(a, blockIdx.x, blockIdx.y, smem_raw);
}

}  // namespace hy
