// Arguments of the implicit Hyena filter kernels (filter_tc.cuh): positional features -> Sin-MLP -> exponential modulation.
//
// Reference semantics (src/models/sequence/hyena.py):
//   :109-131 PositionalEmbedding  z (L,E), t (L,)           -- read as tensors, never regenerated
//   :96-106  Sin                  sin(freq * x), ONE freq vector shared by the three activations
//   :199-215 implicit_filter      Linear(E,N) Sin Linear(N,N) Sin Linear(N,N) Sin Linear(N,D,no bias)
//   :134-155 ExponentialModulation h * (exp(-t * |deltas|) + shift)
//   :229-238 HyenaFilter.filter
// Output layout is channel-major k[c][t] (D, L) so the FFT column pass reads it coalesced.
#pragma once

namespace hy {

constexpr int kFN = 64;          // filter_order supported by these kernels
constexpr int kMaxE = 16;        // emb_dim limit (odd, >= 3)

struct FilterParams {
  const float* z;        // (L, E)   rows of pos_emb.z[0, :L]
  const float* t;        // (L,)     pos_emb.t[0, :L, 0]
  const float* W0; const float* b0;   // (N,E), (N)
  const float* W1; const float* b1;   // (N,N), (N)
  const float* W2; const float* b2;   // (N,N), (N)
  const float* W3;                    // (D,N)
  const float* freq;                  // (N)
  const float* deltas;                // (D)
  float shift;
  int modulate;
  int L, E, D;
  int z_stride;          // elements between consecutive positions of z (== E when contiguous)
};

}  // namespace hy
