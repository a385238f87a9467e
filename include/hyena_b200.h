/* hyena_b200 -- C ABI of the sm_100a Hyena long-convolution library (libhyena_b200.so).
 *
 * This is the drop-in boundary for the HyenaOperator hot path of HazyResearch/hyena-dna.  The
 * reference's own FFI for this path is the pybind11 module `fftconv`
 * (csrc/fftconv/fftconv.cpp:238-241: fftconv_fwd / fftconv_bwd) called from
 * src/ops/fftconv.py:58-108, plus the PyTorch graph of src/models/sequence/hyena.py:388-444.
 * Every entry point below names the reference interface it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers (fp32, contiguous, 8-byte aligned unless stated); sizes are
 *     element counts; `stream` is a cudaStream_t passed as void*.
 *   - inputs are borrowed and never written; outputs are fully overwritten unless marked (+=).
 *   - every function returns 0 on success and a non-zero code on failure; the message of the last
 *     failure on the calling thread is returned by hyena_b200_last_error().  Nothing here falls
 *     back to a CPU path: without a CUDA device the calls fail.
 *   - the functions are stateless and re-entrant apart from a per-device table of FFT twiddles that
 *     is built on first use; they enqueue work on `stream` and return without synchronising.
 *   - sequence length limit: L <= hyena_b200_max_seqlen() (= 2^20).  The reference extension stops at
 *     L <= 8192 (csrc/fftconv/fftconv.cpp:114-115).
 *
 * Layouts (B batch, D channels = d_model, L positions, N = filter_order = 64, E = emb_dim)
 *   p      (B, 3D, L)  in_proj output, channel-major, WITHOUT in_proj.bias (passed separately);
 *                      channels [0,D) = x0, [D,2D) = x1, [2D,3D) = v   (hyena.py:404)
 *   k      (D, L)      time-domain filter, channel-major
 *   kspec  (D, M) complex64 (interleaved re,im), M = hyena_b200_spectrum_elems(L): packed half-size
 *                      spectrum of k in the library's internal [k1][k2] order -- opaque to callers
 *   y_pre  (B, D, L)   operator output before out_proj, channel-major (hyena.py:432 before the rearrange)
 */
#ifndef HYENA_B200_H
#define HYENA_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HYENA_B200_ABI_VERSION 2
#if defined(__GNUC__)
#define HY_API __attribute__((visibility("default")))
#else
#define HY_API
#endif

HY_API int hyena_b200_abi_version(void);
HY_API const char* hyena_b200_last_error(void);
/* number of CUDA kernels this library has launched since it was loaded (all threads) */
HY_API unsigned long long hyena_b200_launch_count(void);
HY_API int hyena_b200_max_seqlen(void);

/* Optional per-launch timing with CUDA events on the launching stream (used by bench.py's roofline leg).
 * profile_begin() starts a window; profile_end() synchronises the device and returns, per kernel class
 * (index < hyena_b200_kind_count(), name from hyena_b200_kind_name), the summed device milliseconds and the launch count. */
HY_API int hyena_b200_profile_begin(void);
HY_API int hyena_b200_profile_end(double* ms_by_kind, unsigned long long* launches_by_kind, int n);
HY_API const char* hyena_b200_kind_name(int kind);
HY_API int hyena_b200_kind_count(void);

/* M: complex elements per channel of a filter spectrum for sequence length L (power of two >= L, >= 1024) */
HY_API size_t hyena_b200_spectrum_elems(int L);
/* scratch bytes the conv entry points want for (B, D, L); backward != 0 for the *_bwd calls.
 * Any size >= hyena_b200_workspace_min_bytes() works; more lets more rows be in flight per launch. */
HY_API size_t hyena_b200_workspace_bytes(int B, int D, int L, int backward);
HY_API size_t hyena_b200_workspace_min_bytes(int B, int D, int L, int backward);

/* ---- implicit filter -------------------------------------------------------------------------
 * replaces HyenaFilter.filter (src/models/sequence/hyena.py:229-238): PositionalEmbedding rows
 * z (L,E; row stride z_stride) and t (L), Sin-MLP (hyena.py:96-106, :199-215), ExponentialModulation
 * (hyena.py:152-155).  Output k (D, L) channel-major == filter(L)[0].transpose(0,1).
 * N (filter_order) must be 64; E odd in [3,15]. */
HY_API int hyena_b200_filter_fwd(const float* z, int z_stride, const float* t,
                          const float* W0, const float* b0, const float* W1, const float* b1,
                          const float* W2, const float* b2, const float* W3,
                          const float* freq, const float* deltas, float shift, int modulate,
                          int L, int E, int N, int D, float* k_out, void* stream);

/* Backward of the above (the reference relies on torch autograd; closed form restated in DESIGN.md), on the tensor
 * cores (tcgen05, 3xTF32) in two stages.  Stage 1: per position, recompute the activations and back-
 * propagate through the MLP, writing dh = dk * modulation (D,L) and seven feature-major (64,L) arrays into `scratch`
 * (7*64*L floats, 16-byte aligned): a1, a2, a3, dp1, dp2, dp3, X.  Stage 2: the parameter gradients are reductions
 * over the sequence, done as accumulating tcgen05 GEMMs with K = position (all outputs (+=); zT is z transposed,
 * (E,L)); D <= 256, E <= 8:
 *   dW3 = dh a3^T, dW2 = dp3 a2^T, dW1 = dp2 a1^T, dW0 = dp1 z, db_l = rowsum(dp_{l+1}), dfreq = rowsum(X) */
HY_API int hyena_b200_filter_bwd_stage1(const float* z, int z_stride, const float* t,
                                 const float* W0, const float* b0, const float* W1, const float* b1,
                                 const float* W2, const float* b2, const float* W3,
                                 const float* freq, const float* deltas, float shift, int modulate,
                                 int L, int E, int N, int D, const float* dk, float* dh, float* scratch, void* stream);

HY_API int hyena_b200_filter_bwd_stage2(const float* dh, const float* scratch, const float* zT,
                                 float* dW0, float* db0, float* dW1, float* db1, float* dW2, float* db2,
                                 float* dW3, float* dfreq, int L, int E, int D, void* stream);

/* ---- filter spectrum -------------------------------------------------------------------------
 * replaces `k_f = torch.fft.rfft(k, n=fft_size) / fft_size` (hyena.py:62, src/ops/fftconv.py:65). */
HY_API int hyena_b200_filter_spectrum(const float* k, float* kspec, int D, int L,
                               void* workspace, size_t workspace_bytes, void* stream);

/* ---- fused operator core ---------------------------------------------------------------------
 * replaces hyena.py:394-432 for order=2: short_filter (depthwise Conv1d k=3, :363-369,:394), split
 * (:404), gate v*x1 (:420), fftconv_ref with bias skip term (:59-88 via :261), gate *x0 (:432).
 *   sw (3D,3) = short_filter.weight[:,0,:], sb (3D) = short_filter.bias, in_bias (3D) = in_proj.bias
 *   or NULL, fbias (D) = filter_fn.bias.  c_save (B,D,L) receives the fftconv output (needed by
 *   core_bwd) when non-NULL.  gspec_save ((D*B) rows of M complex64, row = c*B + b; may be NULL) receives the
 *   packed spectrum of the gated input g = short(v)*short(x1); handing it back to core_bwd saves one column
 *   pass and one row FFT per (b,c) row there (the reference saves u_f the same way, hyena.py:41). */
HY_API int hyena_b200_core_fwd(const float* p, const float* in_bias, const float* sw, const float* sb,
                        const float* kspec, const float* fbias,
                        float* y_pre, float* c_save, float* gspec_save, int B, int D, int L,
                        void* workspace, size_t workspace_bytes, void* stream);

/* backward of core_fwd (closed form: hyena.py:43-56 FFTConvFuncv2.backward,
 * csrc/fftconv/fftconv_cuda.cu:1157-1179).  dy_pre (B,D,L).  Outputs: dp (B,3D,L), dk (D,L);
 * (+=): dsw (3D,3), dsb (3D), dfbias (D), d_in_bias (3D, may be NULL).
 * ds_scratch (B,3D,L) receives ds, the gradient w.r.t. the short-filter OUTPUTS.  With dp == NULL the transposed short
 * filter pass is skipped (d_in_bias is then not written): hand ds to hyena_b200_proj_gemm / hyena_b200_proj_wgrad with
 * fir = sw, which apply dp[t] = w2 ds[t] + w1 ds[t+1] + w0 ds[t+2] in registers. */
HY_API int hyena_b200_core_bwd(const float* dy_pre, const float* p, const float* in_bias, const float* sw,
                        const float* sb, const float* kspec, const float* fbias, const float* c_saved,
                        const float* gspec_saved /* from core_fwd, or NULL to recompute */,
                        float* dp, float* dk, float* dsw, float* dsb, float* dfbias, float* d_in_bias,
                        float* ds_scratch, int B, int D, int L,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- plain long convolution (the reference extension's own surface) ---------------------------
 * fftconv_fwd replaces csrc/fftconv/fftconv.cpp:53-132 for fp32, gelu=false, no dropout mask, no q/v,
 * head_dim=1:  out[b,h,:] = causal_conv(u[b,h,:], k[h,:]) + u[b,h,:] * Dvec[h]     (fftconv_ref,
 * src/ops/fftconv.py:15-34).  The filter is passed as the opaque kspec from hyena_b200_filter_spectrum.
 * fftconv_bwd replaces fftconv.cpp:134-236 + src/ops/fftconv.py:87-103: du (B,H,L), dk (H,L) time
 * domain (the reference returns dk_f and inverts it in Python), dD (H) (+=). */
HY_API int hyena_b200_fftconv_fwd(const float* u, const float* kspec, const float* Dvec, float* out,
                           int B, int H, int L, void* workspace, size_t workspace_bytes, void* stream);
HY_API int hyena_b200_fftconv_bwd(const float* dout, const float* u, const float* kspec, const float* Dvec,
                           float* du, float* dk, float* dD, int B, int H, int L,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ---- the reference extension's filter convention ---------------------------------------------
 * csrc/fftconv/fftconv.cpp:53-61 takes `filter = torch.fft.rfft(k, n=fft_size)`: (H, fft_size/2+1) complex64, natural
 * bin order, unnormalised (src/ops/fftconv.py:64-65); fftconv.cpp:134-143,235 returns `dfilter` in the same layout with
 * irfft(dfilter, n=fft_size, norm='forward')[:L] == dk (src/ops/fftconv.py:94-98).  These two entry points convert
 * between that convention and the packed kspec / the time-domain dk of fftconv_fwd / fftconv_bwd above, so that an
 * unmodified src/ops/fftconv.py:FFTConvFunc binds to this library (INTEGRATION.md).  fft_size: power of two >= 16 with
 * L <= fft_size/2 (fftconv.cpp:114-115).  k_scratch (H*L floats) is needed only when fft_size < 2*spectrum_elems(L);
 * kspec_scratch (H * spectrum_elems(L) complex64) only when fft_size == 2*spectrum_elems(L). */
HY_API int hyena_b200_spectrum_from_rfft(const float* filter, int fft_size, float* kspec, float* k_scratch, int H, int L,
                                  void* workspace, size_t workspace_bytes, void* stream);
HY_API int hyena_b200_spectrum_to_rfft(const float* dk, int fft_size, float* dfilter, float* kspec_scratch, int H, int L,
                                void* workspace, size_t workspace_bytes, void* stream);

/* ---- projections (library GEMM at the boundary of the custom-kernel span) ------------------------
 * in_proj / out_proj (hyena.py:350-351, :391, :440) are plain GEMMs and stay cuBLASLt calls.  These two
 * entry points run them on the CUDA 12.9 cuBLASLt with CUBLAS_COMPUTE_32F_EMULATED_16BFX9 (fp32 emulated
 * on bf16 tensor cores, fp32-level accuracy).  Column-major, strided-batched:
 * C[m,n] = alpha * op(A) op(B) + beta * C (+ bias[m]); op: 0 = N, 1 = T. */
HY_API int hyena_b200_gemm_available(void);

/* ---- projections on this library's own tensor-core kernel (csrc/proj_gemm.cuh) --------------------
 * The same GEMMs as above without the library call: tcgen05 / TMEM, fp32 accuracy through 3xTF32, weights streamed by
 * TMA bulk copies, the activation converted on the fly into tensor memory.  Computes, for every batch b,
 *     OUT[pos][n] = sum_k ACT[pos][k] * Wl[n][k] (+ bias[n]),    Wl[n][k] = w_transposed ? W[k*ldw + n] : W[n*ldw + k]
 *   act_layout 0: ACT is (B, L, K) row-major (u, dy: hyena.py:391, :440 backward)
 *              1: ACT is (B, K, L) channel-major (y_pre, ds: hyena.py:432-440)
 *   out_layout 0: OUT is (B, N, L) channel-major (p, dy_pre);   1: OUT is (B, L, N) row-major (y, du)
 *   fir (K,3) non-NULL (act_layout 1 only): ACT is ds, the gradient w.r.t. the short-filter OUTPUT, and the GEMM consumes
 *              dp[k][t] = fir[k][2] ds[k][t] + fir[k][1] ds[k][t+1] + fir[k][0] ds[k][t+2] (backward of the depthwise
 *              Conv1d, hyena.py:363-369) computed in registers -- dp never exists in HBM.
 *   l_begin, l_len: only positions [l_begin, l_begin + l_len) of every batch are computed (host-side pipelining of a
 *              long sequence against PCIe copies, hyena-dna_b200/host.py); l_len <= 0 means all L positions.
 *   wimg: scratch of hyena_b200_proj_wimg_bytes(N, K) bytes (tf32 hi/lo images of the weights, rebuilt every call). */
/* Weight gradients of the projections (hyena.py:391, :440 backward), reduction over the sequence positions:
 *     dW[m][n] (= or +=) sum_{b,pos} X[b][m][pos] * Y[b][pos][n]
 * X (B, M, L) channel-major (ds / y_pre), Y (B, L, N) row-major (u / dy); split-K over the SMs with the accumulators in
 * tensor memory, deterministic reduction of the partials.  transposed_out: dW is stored (N, M).  beta: 0 overwrite, else
 * dW = beta * dW + sum.  fir (M,3): X is ds and the transposed short filter is applied on the fly (see proj_gemm).
 * scratch: hyena_b200_proj_wgrad_scratch_bytes(M, N) bytes. */
HY_API size_t hyena_b200_proj_wgrad_scratch_bytes(int M, int N);
HY_API int hyena_b200_proj_wgrad(const float* X, const float* Y, const float* fir, float* dW, int transposed_out, float beta,
                          int B, int L, int M, int N, void* scratch, size_t scratch_bytes, void* stream);
HY_API size_t hyena_b200_proj_wimg_bytes(int N, int K);
/* debug aid (tools/dbg_proj_timing.py): device buffer of >= 16 int64 receiving per-role barrier-wait cycle counters */
HY_API int hyena_b200_proj_debug_buffer(void* buf);
HY_API int hyena_b200_proj_gemm(const float* act, int act_layout, const float* W, int ldw, int w_transposed,
                         const float* bias, const float* fir, float* out, int out_layout, int B, int L, int K, int N,
                         int l_begin, int l_len, void* wimg, size_t wimg_bytes, void* stream);
HY_API int hyena_b200_gemm(int transa, int transb, int m, int n, int k, float alpha, const float* A, int lda,
                           long long strideA, const float* B, int ldb, long long strideB, float beta, float* C,
                           int ldc, long long strideC, int batch, const float* bias, int emulate, void* workspace,
                           size_t workspace_bytes, void* stream);

/* ---- filter options outside the shipped configs -------------------------------------------------
 * modulation_lr != 0 (hyena.py:145-150: deltas is a Parameter): d deltas (D) from the filter k (D, L) the forward produced and
 * its gradient dk (D, L); t (L) = PositionalEmbedding.t.  Overwrites ddelta. */
HY_API int hyena_b200_filter_ddelta(const float* dk, const float* k, const float* t, const float* deltas, float shift, int D,
                             int L, float* ddelta, void* stream);
/* normalized=True (hyena.py:235-236, L1 norm over the channel dim of (1, L, D)): out[c][t] = k[c][t] / norm[t],
 * norm[t] = sum_c |k[c][t]| (L values, kept for the backward); bwd: dk = (dout - sign(out) * sum_c dout*out) / norm. */
HY_API int hyena_b200_filter_l1norm_fwd(const float* k, float* out, float* norm, int D, int L, void* stream);
HY_API int hyena_b200_filter_l1norm_bwd(const float* dout, const float* out, const float* norm, float* dk, int D, int L,
                                 void* stream);

/* ---- block glue: residual add + LayerNorm (SURVEY.md S8 f1) ---------------------------------------
 * replaces the dropout(p=0) -> add -> LayerNorm step of the pre-norm Block that wraps the mixer
 * (flash-attention/flash_attn/modules/block.py:111-148; with fused_dropout_add_ln it is
 * flash_attn.ops.layer_norm.dropout_add_layer_norm(..., prenorm=True, residual_in_fp32=True)):
 *   res_out = x + res (res may be NULL: first block, res_out may then be NULL too)
 *   y = (res_out - mean) * rstd * w + b      per row of D features, fp32; mean / rstd (rows) are saved for the backward
 * bwd: dy = grad of y, dres = grad arriving on res_out (may be NULL), r = res_out of the forward (x itself when no
 *   residual was added).  dx (rows, D) is the gradient of x AND of res; dw / db (D) are overwritten (db may be NULL).
 *   scratch: hyena_b200_add_layernorm_scratch_bytes(rows, D) bytes of per-CTA partial sums (deterministic reduction). */
HY_API size_t hyena_b200_add_layernorm_scratch_bytes(long long rows, int D);
HY_API int hyena_b200_add_layernorm_fwd(const float* x, const float* res, const float* w, const float* b, float eps,
                                 float* res_out, float* y, float* mean, float* rstd, long long rows, int D, void* stream);
HY_API int hyena_b200_add_layernorm_bwd(const float* dy, const float* dres, const float* r, const float* w, const float* mean,
                                 const float* rstd, float* dx, float* dw, float* db, long long rows, int D, void* scratch,
                                 size_t scratch_bytes, void* stream);

/* ---- incremental decoding (order 2, causal) --------------------------------------------------------
 * The reference has no recurrent mode (hyena.py:384-386 raises NotImplementedError).  After a prompt of Lp positions has
 * gone through the full-sequence path, every further token costs one causal dot product per channel over the history:
 *   P[t] = W_in u_t + in_bias (3D);  s = w0 P[t-2] + w1 P[t-1] + w2 P[t] + sb (P[<0] = 0);  x0, x1, v = split(s)
 *   g[t] = v * x1;  c[t] = sum_{j<=t} k[c][j] g[t-j] + fbias[c] g[t];  y_t = W_out (c[t] * x0) + out_bias
 * State (owned by the caller, fp32):
 *   g_hist (B, D, max_len)  gated history g, channel-major; positions >= the current one are never read
 *   fir    (B, 3D, 2)       P[t-2], P[t-1] of every in_proj channel (bias included; zeros before the sequence start)
 *   k      (D, max_len)     the filter for max_len positions (hyena_b200_filter_fwd); only k[:, :t+1] is read
 * max_len <= hyena_b200_max_seqlen(), 1 <= B <= 64.
 * prefill: p (B, 3D, Lp) = the prompt's in_proj output without in_proj.bias (the layout of core_fwd), 1 <= Lp <= max_len.
 *   Writes g_hist[:, :, :Lp] and all of fir.  A fresh state starting at t = 0 needs fir zeroed and no prefill.
 * step: position t (host int, 0 <= t < max_len), u_t (B, D) row-major, W_in (3D, D), W_out (D, D) nn.Linear layouts,
 *   in_bias (3D) / out_bias (D) may be NULL.  Writes y_t (B, D), g_hist[:, :, t] and fir.  workspace: at least
 *   hyena_b200_decode_workspace_bytes(B, D, max_len) bytes, 4-byte aligned.  Three kernels, deterministic (no atomics). */
HY_API size_t hyena_b200_decode_workspace_bytes(int B, int D, int max_len);
HY_API int hyena_b200_decode_prefill(const float* p, const float* in_bias, const float* sw, const float* sb, float* g_hist,
                                     float* fir, int B, int D, int Lp, int max_len, void* stream);
HY_API int hyena_b200_decode_step(const float* u_t, const float* W_in, const float* in_bias, const float* sw, const float* sb,
                                  const float* k, const float* fbias, const float* W_out, const float* out_bias,
                                  float* g_hist, float* fir, float* y_t, int B, int D, int t, int max_len,
                                  void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HYENA_B200_H */
