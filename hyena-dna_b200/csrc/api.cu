// C ABI of libhyena_b200.so (include/hyena_b200.h): argument checks, workspace carving, row-group
// scheduling of the three FFT passes.  No torch types; PyTorch hands in raw device pointers.
#include <atomic>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/hyena_b200.h"
#include "launch.h"

namespace hy {

extern long long* g_proj_dbg;          // k_proj.cu
static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

// ---- optional per-launch event timing (bench.py's roofline leg); off by default
struct ProfRec { int kind; cudaEvent_t e0, e1; };
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;            // records of the current profiling window
static std::vector<cudaEvent_t> g_ev_pool;     // recycled events
static thread_local cudaEvent_t g_cur_e0 = nullptr;

static cudaEvent_t get_event() {
  if (!g_ev_pool.empty()) { cudaEvent_t e = g_ev_pool.back(); g_ev_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
void prof_begin(int kind, cudaStream_t s) {
  (void)kind;
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_cur_e0 = get_event();
  cudaEventRecord(g_cur_e0, s);
}
void prof_end(int kind, cudaStream_t s) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (!g_prof_on || !g_cur_e0) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  cudaEvent_t e1 = get_event();
  cudaEventRecord(e1, s);
  g_prof.push_back({kind, g_cur_e0, e1});
  g_cur_e0 = nullptr;
}

int api_fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
static int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
#define HY_CUDA(expr)                                                                        \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) return fail("%s failed: %s", #expr, cudaGetErrorString(_e));      \
  } while (0)
#define HY_CHECK(cond, ...) \
  do { if (!(cond)) return fail(__VA_ARGS__); } while (0)

// ---------------------------------------------------------------- per-device twiddle tables
struct DevTables { float2* tw1024 = nullptr; float2* twlo = nullptr; };
static DevTables g_tables[64];
static std::mutex g_mu;

static int get_twiddles(cudaStream_t s, Twiddles* out) {
  int dev = -1;
  HY_CUDA(cudaGetDevice(&dev));
  HY_CHECK(dev >= 0 && dev < 64, "unsupported device ordinal %d", dev);
  std::lock_guard<std::mutex> lk(g_mu);
  DevTables& t = g_tables[dev];
  if (!t.tw1024) {
    float2* mem = nullptr;
    HY_CUDA(cudaMalloc(&mem, 2 * 1024 * sizeof(float2)));
    HY_CUDA(launch_twiddle_init(mem, mem + 1024, s));
    // later calls may come on other streams: make the table visible to all of them
    HY_CUDA(cudaStreamSynchronize(s));
    t.tw1024 = mem;
    t.twlo = mem + 1024;
  }
  out->tw1024 = t.tw1024;
  out->twlo = t.twlo;
  return 0;
}

// ---------------------------------------------------------------- geometry
static int log_m_for(int L) {         // M = 2^logM >= max(L, 1024)
  int lg = 10;
  while (((size_t)1 << lg) < (size_t)L) ++lg;
  return lg;
}
// Row length: 1024 points, one warp per row.  (A 4096-point variant existed in round 1 and lost: 43.85 vs 39.10 ms per
// step at L = 2^20, profiles/r1_config_sweep.txt; removed.)
static int pick_log_m2(int) { return 10; }
static size_t row_bytes(int L) { return ((size_t)1 << log_m_for(L)) * sizeof(float2); }

static size_t group_budget_bytes() {
  // scratch rows in flight per launch group.  Measured on B200 (profiles/r1_config_sweep.txt, two sweeps): with
  // separate kernels per pass the scratch does not survive in L2 anyway, and many waves per launch win, so the
  // default lets a whole (B=1, D=256, L=2^20) operator go in one launch per pass
  static size_t v = 0;
  if (!v) {
    const char* e = getenv("HYENA_B200_GROUP_MB");
    long mb = e ? atol(e) : 2048;
    if (mb < 1) mb = 1;
    v = (size_t)mb << 20;
  }
  return v;
}

// channels per group given the bytes available for ONE scratch array holding all batches of a channel
static int channels_per_group(size_t bytes_for_A, int B, int D, int L) {
  size_t per_ch = row_bytes(L) * (size_t)B;
  size_t n = bytes_for_A / per_ch;
  if (n > (size_t)D) n = D;
  size_t cap = 65535 / (size_t)B;
  if (n > cap) n = cap;
  return (int)n;
}

static bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct Carve { float2* A; float2* A2; float2* A3; int nch; };

// backward needs A and A2 (B rows per channel each) and A3 (1 row per channel)
static int carve(void* ws, size_t ws_bytes, int B, int D, int L, bool backward, Carve* c) {
  HY_CHECK(ws != nullptr && aligned8(ws), "workspace must be a non-null 8-byte aligned device pointer");
  const size_t rb = row_bytes(L);
  const size_t per_ch = backward ? rb * (2 * (size_t)B + 1) : rb * (size_t)B;
  HY_CHECK(ws_bytes >= per_ch, "workspace too small: %zu bytes given, %zu needed (hyena_b200_workspace_min_bytes)",
           ws_bytes, per_ch);
  size_t n = ws_bytes / per_ch;
  if (n > (size_t)D) n = D;
  size_t cap = 65535 / (size_t)B;
  if (n > cap) n = cap;
  c->nch = (int)n;
  c->A = reinterpret_cast<float2*>(ws);
  c->A2 = backward ? c->A + (rb / sizeof(float2)) * (size_t)B * n : nullptr;
  c->A3 = backward ? c->A2 + (rb / sizeof(float2)) * (size_t)B * n : nullptr;
  return 0;
}

static int check_shape(int B, int D, int L) {
  HY_CHECK(B >= 1 && D >= 1 && L >= 1, "bad shape B=%d D=%d L=%d", B, D, L);
  HY_CHECK(L <= (1 << 20), "sequence length %d exceeds the supported maximum %d", L, 1 << 20);
  HY_CHECK(B <= 65535, "batch %d too large", B);
  return 0;
}

static PassArgs base_args(int B, int D, int L, const Twiddles& T) {
  PassArgs a;
  memset(&a, 0, sizeof(a));
  const int logM = log_m_for(L);
  a.L = L; a.logM2 = pick_log_m2(logM); a.logM1 = logM - a.logM2; a.B = B; a.D = D; a.T = T;
  a.scale = 1.0f / (4.0f * (float)((size_t)1 << logM));
  return a;
}

}  // namespace hy

using namespace hy;

extern "C" {

HY_API int hyena_b200_abi_version(void) { return HYENA_B200_ABI_VERSION; }
HY_API const char* hyena_b200_last_error(void) { return g_err; }
HY_API unsigned long long hyena_b200_launch_count(void) { return g_launches.load(); }
HY_API int hyena_b200_max_seqlen(void) { return 1 << 20; }

HY_API int hyena_b200_profile_begin(void) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (auto& r : g_prof) { g_ev_pool.push_back(r.e0); g_ev_pool.push_back(r.e1); }
  g_prof.clear();
  g_prof_on = true;
  return 0;
}

HY_API int hyena_b200_profile_end(double* ms_by_kind, unsigned long long* launches_by_kind, int n) {
  HY_CHECK(ms_by_kind && launches_by_kind && n >= K_COUNT, "profile_end needs arrays of >= %d entries", K_COUNT);
  HY_CUDA(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = false;
  for (int i = 0; i < n; ++i) { ms_by_kind[i] = 0.0; launches_by_kind[i] = 0; }
  for (auto& r : g_prof) {
    float ms = 0.f;
    HY_CUDA(cudaEventElapsedTime(&ms, r.e0, r.e1));
    ms_by_kind[r.kind] += ms;
    launches_by_kind[r.kind] += 1;
    g_ev_pool.push_back(r.e0); g_ev_pool.push_back(r.e1);
  }
  g_prof.clear();
  return 0;
}

HY_API const char* hyena_b200_kind_name(int kind) {
  static const char* names[] = {
      "col_fwd<filter>", "col_fwd<gate>", "col_fwd<dc>", "col_fwd<plain>",
      "col_inv<conv_fwd>", "col_inv<bwd_dg>", "col_inv<dk>", "col_inv<plain_fwd>", "col_inv<plain_bwd>",
      "row_pass<filter>", "row_pass<conv_fwd>", "row_pass<conv_bwd>",
      "short_conv_bwd", "twiddle_init", "filter_tc_prep", "filter_tc_fwd", "filter_tc_bwd", "filter_tc_red",
      "spectrum_convert", "proj_prep", "proj_gemm", "proj_wgrad", "add_layer_norm", "filter_extra",
      "decode_prefill", "decode_step_conv", "decode_step_reduce", "decode_step_out"};
  static_assert(sizeof(names) / sizeof(names[0]) == K_COUNT, "one name per Kind");
  return (kind >= 0 && kind < K_COUNT) ? names[kind] : "?";
}

HY_API int hyena_b200_kind_count(void) { return K_COUNT; }

HY_API size_t hyena_b200_spectrum_elems(int L) { return L < 1 ? 0 : ((size_t)1 << log_m_for(L)); }

HY_API size_t hyena_b200_workspace_min_bytes(int B, int D, int L, int backward) {
  (void)D;
  if (B < 1 || L < 1) return 0;
  return backward ? row_bytes(L) * (2 * (size_t)B + 1) : row_bytes(L) * (size_t)B;
}

HY_API size_t hyena_b200_workspace_bytes(int B, int D, int L, int backward) {
  if (B < 1 || L < 1 || D < 1) return 0;
  int nch = channels_per_group(group_budget_bytes(), B, D, L);
  if (nch < 1) nch = 1;
  return hyena_b200_workspace_min_bytes(B, D, L, backward) * (size_t)nch;
}

// tensor-core filter path: scratch for the tf32 hi/lo weight images (~0.3 MB, grow-only), one per (device, stream): two
// operators driven from different streams never share it (the prep kernel of one would overwrite the images the other's
// tcgen05 kernel is still reading)
static int get_wimg(int D, cudaStream_t stream, float** out) {
  int dev = -1;
  HY_CUDA(cudaGetDevice(&dev));
  HY_CHECK(dev >= 0 && dev < 64, "unsupported device ordinal %d", dev);
  std::lock_guard<std::mutex> lk(g_mu);
  struct Buf { float* p = nullptr; size_t n = 0; };
  static std::map<std::pair<int, cudaStream_t>, Buf> bufs;
  Buf& b = bufs[std::make_pair(dev, stream)];
  const size_t need = filter_tc_wimg_bytes(D);
  if (b.n < need) {
    if (b.p) { HY_CUDA(cudaStreamSynchronize(stream)); HY_CUDA(cudaFree(b.p)); b.p = nullptr; b.n = 0; }
    HY_CUDA(cudaMalloc(&b.p, need));
    b.n = need;
  }
  *out = b.p;
  return 0;
}

static int fill_filter_params(FilterParams* P, const float* z, int z_stride, const float* t, const float* W0,
                              const float* b0, const float* W1, const float* b1, const float* W2, const float* b2,
                              const float* W3, const float* freq, const float* deltas, float shift, int modulate,
                              int L, int E, int N, int D) {
  HY_CHECK(N == kFN, "filter_order %d not supported (this build handles %d)", N, kFN);
  HY_CHECK(E >= 3 && E < kMaxE && (E & 1), "emb_dim %d not supported (odd, 3..%d)", E, kMaxE - 1);
  HY_CHECK(L >= 1 && D >= 1, "bad filter shape L=%d D=%d", L, D);
  HY_CHECK(z && t && W0 && b0 && W1 && b1 && W2 && b2 && W3 && freq && deltas, "null filter parameter");
  HY_CHECK((reinterpret_cast<uintptr_t>(W3) & 15u) == 0, "W3 must be 16-byte aligned");
  P->z = z; P->t = t; P->W0 = W0; P->b0 = b0; P->W1 = W1; P->b1 = b1; P->W2 = W2; P->b2 = b2; P->W3 = W3;
  P->freq = freq; P->deltas = deltas; P->shift = shift; P->modulate = modulate;
  P->L = L; P->E = E; P->D = D; P->z_stride = z_stride;
  return 0;
}

HY_API int hyena_b200_filter_fwd(const float* z, int z_stride, const float* t, const float* W0, const float* b0,
                          const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                          const float* freq, const float* deltas, float shift, int modulate, int L, int E, int N,
                          int D, float* k_out, void* stream) {
  FilterParams P;
  if (fill_filter_params(&P, z, z_stride, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L, E, N, D))
    return 1;
  HY_CHECK(k_out, "null output");
  float* wimg = nullptr;
  if (get_wimg(D, (cudaStream_t)stream, &wimg)) return 1;
  HY_CUDA(launch_filter_fwd_tc(P, wimg, k_out, (cudaStream_t)stream));
  return 0;
}

HY_API int hyena_b200_filter_bwd_stage1(const float* z, int z_stride, const float* t, const float* W0, const float* b0,
                                 const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                                 const float* freq, const float* deltas, float shift, int modulate, int L, int E,
                                 int N, int D, const float* dk, float* dh, float* scratch, void* stream) {
  FilterParams P;
  if (fill_filter_params(&P, z, z_stride, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L, E, N, D))
    return 1;
  HY_CHECK(dk && dh && scratch && ((reinterpret_cast<uintptr_t>(scratch) & 15u) == 0), "null or misaligned pointer");
  float* wimg = nullptr;
  if (get_wimg(D, (cudaStream_t)stream, &wimg)) return 1;
  HY_CUDA(launch_filter_bwd_tc(P, wimg, dk, dh, scratch, (cudaStream_t)stream));
  return 0;
}

HY_API int hyena_b200_filter_bwd_stage2(const float* dh, const float* scratch, const float* zT, float* dW0, float* db0,
                                 float* dW1, float* db1, float* dW2, float* db2, float* dW3, float* dfreq, int L,
                                 int E, int D, void* stream) {
  HY_CHECK(dh && scratch && zT && dW0 && db0 && dW1 && db1 && dW2 && db2 && dW3 && dfreq, "null pointer");
  HY_CHECK(D >= 1 && D <= 256 && E >= 1 && E <= 8 && L >= 1, "fused filter reduction handles D <= 256, E <= 8 (got D=%d E=%d)", D, E);
  HY_CHECK((reinterpret_cast<uintptr_t>(dh) & 15u) == 0 && (reinterpret_cast<uintptr_t>(scratch) & 15u) == 0 &&
               (reinterpret_cast<uintptr_t>(zT) & 15u) == 0, "misaligned pointer");
  RedLaunch r{dh, scratch, zT, dW0, db0, dW1, db1, dW2, db2, dW3, dfreq, L, D, E};
  HY_CUDA(launch_filter_red_tc(r, (cudaStream_t)stream));
  return 0;
}

HY_API int hyena_b200_filter_spectrum(const float* k, float* kspec, int D, int L, void* workspace, size_t workspace_bytes,
                               void* stream) {
  if (check_shape(1, D, L)) return 1;
  HY_CHECK(k && kspec && aligned8(kspec), "null or misaligned pointer");
  cudaStream_t s = (cudaStream_t)stream;
  Twiddles T;
  if (get_twiddles(s, &T)) return 1;
  Carve c;
  if (carve(workspace, workspace_bytes, 1, D, L, false, &c)) return 1;
  PassArgs a = base_args(1, D, L, T);
  a.A = c.A; a.src = k; a.kspec_out = reinterpret_cast<float2*>(kspec);
  a.vec = ((L & 1) == 0) && aligned8(k);
  for (int c0 = 0; c0 < D; c0 += c.nch) {
    const int n = (D - c0 < c.nch) ? D - c0 : c.nch;
    a.c0 = c0;
    HY_CUDA(launch_col_fwd(COL_FILTER, a, n, s));
    HY_CUDA(launch_row_pass(ROW_FILTER, a, n, s));
  }
  return 0;
}

/* filter = rfft(k, fft_size) (H, fft_size/2+1) complex64, natural order, unnormalised -> packed kspec (H, M).
 * k_scratch (H*L floats) is used only when fft_size < 2M (sequences shorter than the minimum transform). */
HY_API int hyena_b200_spectrum_from_rfft(const float* filter, int fft_size, float* kspec, float* k_scratch, int H, int L,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  if (check_shape(1, H, L)) return 1;
  HY_CHECK(filter && kspec && aligned8(filter) && aligned8(kspec), "null or misaligned pointer");
  HY_CHECK(fft_size >= 16 && (fft_size & (fft_size - 1)) == 0 && L <= fft_size / 2,
           "fft_size %d must be a power of two >= 16 with L = %d <= fft_size/2 (fftconv.cpp:114-115)", fft_size, L);
  cudaStream_t s = (cudaStream_t)stream;
  const int logM = log_m_for(L);
  const int logM2 = pick_log_m2(logM), logM1 = logM - logM2;
  if ((size_t)fft_size == ((size_t)2 << logM)) {
    HY_CUDA(launch_rfft_to_packed(reinterpret_cast<const float2*>(filter), reinterpret_cast<float2*>(kspec), H, logM, logM1, s));
    return 0;
  }
  HY_CHECK((size_t)fft_size < ((size_t)2 << logM), "fft_size %d larger than the transform of L = %d", fft_size, L);
  HY_CHECK(k_scratch, "k_scratch is required when fft_size < 2 * spectrum_elems(L)");
  HY_CUDA(launch_rfft_to_time_small(reinterpret_cast<const float2*>(filter), k_scratch, H, L, fft_size, s));
  return hyena_b200_filter_spectrum(k_scratch, kspec, H, L, workspace, workspace_bytes, stream);
}

/* dk (H, L) time domain -> dfilter (H, fft_size/2+1) complex64 with irfft(dfilter, n=fft_size, norm='forward')[:L] == dk
 * (the convention of csrc/fftconv/fftconv.cpp:235 consumed by src/ops/fftconv.py:98).  kspec_scratch: (H, M) complex. */
HY_API int hyena_b200_spectrum_to_rfft(const float* dk, int fft_size, float* dfilter, float* kspec_scratch, int H, int L,
                                void* workspace, size_t workspace_bytes, void* stream) {
  if (check_shape(1, H, L)) return 1;
  HY_CHECK(dk && dfilter && aligned8(dfilter), "null or misaligned pointer");
  HY_CHECK(fft_size >= 16 && (fft_size & (fft_size - 1)) == 0 && L <= fft_size / 2,
           "fft_size %d must be a power of two >= 16 with L = %d <= fft_size/2", fft_size, L);
  cudaStream_t s = (cudaStream_t)stream;
  const int logM = log_m_for(L);
  const int logM2 = pick_log_m2(logM), logM1 = logM - logM2;
  const float scale = 1.0f / (float)fft_size;
  if ((size_t)fft_size == ((size_t)2 << logM)) {
    HY_CHECK(kspec_scratch && aligned8(kspec_scratch), "kspec_scratch is required");
    if (hyena_b200_filter_spectrum(dk, kspec_scratch, H, L, workspace, workspace_bytes, stream)) return 1;
    HY_CUDA(launch_packed_to_rfft(reinterpret_cast<const float2*>(kspec_scratch), reinterpret_cast<float2*>(dfilter), H, logM,
                                  logM1, scale, s));
    return 0;
  }
  HY_CHECK((size_t)fft_size < ((size_t)2 << logM), "fft_size %d larger than the transform of L = %d", fft_size, L);
  HY_CUDA(launch_time_to_rfft_small(dk, reinterpret_cast<float2*>(dfilter), H, L, fft_size, scale, s));
  return 0;
}

HY_API int hyena_b200_core_fwd(const float* p, const float* in_bias, const float* sw, const float* sb, const float* kspec,
                        const float* fbias, float* y_pre, float* c_save, float* gspec_save, int B, int D, int L,
                        void* workspace, size_t workspace_bytes, void* stream) {
  if (check_shape(B, D, L)) return 1;
  HY_CHECK(p && sw && sb && kspec && fbias && y_pre, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  Twiddles T;
  if (get_twiddles(s, &T)) return 1;
  Carve c;
  if (carve(workspace, workspace_bytes, B, D, L, false, &c)) return 1;
  PassArgs a = base_args(B, D, L, T);
  a.A = c.A; a.kspec = reinterpret_cast<const float2*>(kspec);
  a.p = p; a.in_bias = in_bias; a.sw = sw; a.sb = sb; a.fbias = fbias; a.out = y_pre; a.out2 = c_save;
  a.gspec = reinterpret_cast<float2*>(gspec_save);
  a.vec = ((L & 1) == 0) && aligned8(p) && aligned8(y_pre) && (!c_save || aligned8(c_save));
  a.stage = ((L & 3) == 0) && aligned16(p);
  for (int c0 = 0; c0 < D; c0 += c.nch) {
    const int n = (D - c0 < c.nch) ? D - c0 : c.nch;
    a.c0 = c0;
    HY_CUDA(launch_col_fwd(COL_GATE, a, n * B, s));
    HY_CUDA(launch_row_pass(ROW_CONV_FWD, a, n * B, s));
    HY_CUDA(launch_col_inv(INV_CONV_FWD, a, n * B, s));
  }
  return 0;
}

HY_API int hyena_b200_core_bwd(const float* dy_pre, const float* p, const float* in_bias, const float* sw, const float* sb,
                        const float* kspec, const float* fbias, const float* c_saved, const float* gspec_saved,
                        float* dp, float* dk, float* dsw, float* dsb, float* dfbias, float* d_in_bias,
                        float* ds_scratch, int B, int D, int L, void* workspace, size_t workspace_bytes, void* stream) {
  if (check_shape(B, D, L)) return 1;
  HY_CHECK(dy_pre && p && sw && sb && kspec && fbias && c_saved && dk && dsw && dsb && dfbias && ds_scratch,
           "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  Twiddles T;
  if (get_twiddles(s, &T)) return 1;
  Carve c;
  if (carve(workspace, workspace_bytes, B, D, L, true, &c)) return 1;
  PassArgs a = base_args(B, D, L, T);
  a.kspec = reinterpret_cast<const float2*>(kspec);
  a.p = p; a.in_bias = in_bias; a.sw = sw; a.sb = sb; a.fbias = fbias;
  a.vec = ((L & 1) == 0) && aligned8(p) && aligned8(dy_pre) && aligned8(c_saved) && aligned8(dk) &&
          aligned8(ds_scratch);
  a.stage = ((L & 3) == 0) && aligned16(p) && aligned16(dy_pre) && aligned16(c_saved);
  for (int c0 = 0; c0 < D; c0 += c.nch) {
    const int n = (D - c0 < c.nch) ? D - c0 : c.nch;
    a.c0 = c0; a.B = B;
    a.A2 = c.A2; a.A3 = c.A3;
    a.A = c.A; a.src = dy_pre;
    HY_CUDA(launch_col_fwd(COL_DC, a, n * B, s));        // A  <- columns of dc = dy_pre * x0
    a.gspec = const_cast<float2*>(reinterpret_cast<const float2*>(gspec_saved));
    if (!gspec_saved) {
      a.A = c.A2;
      HY_CUDA(launch_col_fwd(COL_GATE, a, n * B, s));    // A2 <- columns of g = v * x1 (recomputed)
    }
    a.A = c.A;
    HY_CUDA(launch_row_pass(ROW_CONV_BWD, a, n, s));     // A <- rows of dg, A3 <- rows of dk
    a.src = dy_pre; a.src2 = c_saved; a.out2 = ds_scratch; a.red = dfbias; a.dsw = dsw; a.dsb = dsb;
    HY_CUDA(launch_col_inv(INV_BWD_DG, a, n * B, s));
    a.B = 1; a.out = dk;
    HY_CUDA(launch_col_inv(INV_DK, a, n, s));
  }
  // pass 3 already accumulated dsw / dsb from the operand windows it had staged: no second read of p here.
  // dp == NULL: the caller consumes ds directly (hyena_b200_proj_gemm / proj_wgrad apply the transposed short filter on
  // the fly and d in_proj.bias follows from dsb and two edge samples), so dp never exists in HBM.
  if (dp) {
    ShortBwdArgs sa{ds_scratch, nullptr, in_bias, sw, dp, dsw, dsb, d_in_bias, L, 3 * D, a.vec && aligned8(dp)};
    HY_CUDA(launch_short_bwd(sa, B, s));
  }
  return 0;
}

/* OUT[pos][n] = sum_k ACT[pos][k] W'[n][k] (+ bias[n]) on tcgen05, fp32 accuracy (3xTF32); see include/hyena_b200.h */
HY_API size_t hyena_b200_proj_wimg_bytes(int N, int K) { return (N < 1 || K < 1) ? 0 : proj_wimg_bytes(N, K); }

HY_API int hyena_b200_proj_gemm(const float* act, int act_layout, const float* W, int ldw, int w_transposed,
                         const float* bias, const float* fir, float* out, int out_layout, int B, int L, int K, int N,
                         int l_begin, int l_len, void* wimg, size_t wimg_bytes, void* stream) {
  HY_CHECK(act && W && out && wimg, "null pointer");
  if (l_len <= 0) { l_begin = 0; l_len = L; }
  HY_CHECK(l_begin >= 0 && l_begin + l_len <= L, "position range [%d, %d) outside [0, %d)", l_begin, l_begin + l_len, L);
  HY_CHECK(B >= 1 && L >= 1 && K >= 1 && N >= 1, "bad shape B=%d L=%d K=%d N=%d", B, L, K, N);
  HY_CHECK((act_layout == 0 || act_layout == 1) && (out_layout == 0 || out_layout == 1), "bad layout code");
  HY_CHECK(!fir || act_layout == 1, "the fused transposed short filter needs a channel-major activation");
  HY_CHECK(aligned16(act) && aligned16(out) && aligned16(wimg) && (!bias || aligned16(bias)), "pointers must be 16-byte aligned");
  HY_CHECK(wimg_bytes >= proj_wimg_bytes(N, K), "weight image scratch too small: %zu < %zu", wimg_bytes, proj_wimg_bytes(N, K));
  HY_CHECK(ldw >= (w_transposed ? N : K), "ldw %d too small", ldw);
  HY_CUDA(launch_proj_gemm(act, act_layout, W, ldw, w_transposed, bias, fir, out, out_layout, B, L, K, N, l_begin, l_len,
                           reinterpret_cast<float*>(wimg), (cudaStream_t)stream));
  return 0;
}

/* debug: device buffer of >= 16 long longs receiving the per-role barrier-wait cycle counters of CTA 0 (NULL: off) */
HY_API int hyena_b200_proj_debug_buffer(void* buf) { hy::g_proj_dbg = reinterpret_cast<long long*>(buf); return 0; }

HY_API size_t hyena_b200_proj_wgrad_scratch_bytes(int M, int N) { return (M < 1 || N < 1) ? 0 : proj_wgrad_scratch_bytes(M, N); }

HY_API int hyena_b200_proj_wgrad(const float* X, const float* Y, const float* fir, float* dW, int transposed_out, float beta,
                          int B, int L, int M, int N, void* scratch, size_t scratch_bytes, void* stream) {
  HY_CHECK(X && Y && dW && scratch, "null pointer");
  HY_CHECK(B >= 1 && L >= 1 && M >= 1 && N >= 1, "bad shape B=%d L=%d M=%d N=%d", B, L, M, N);
  HY_CHECK(aligned16(X) && aligned16(Y) && aligned16(scratch), "pointers must be 16-byte aligned");
  HY_CHECK(scratch_bytes >= proj_wgrad_scratch_bytes(M, N), "scratch too small: %zu < %zu", scratch_bytes,
           proj_wgrad_scratch_bytes(M, N));
  HY_CUDA(launch_proj_wgrad(X, Y, fir, dW, transposed_out, beta, B, L, M, N, reinterpret_cast<float*>(scratch),
                            (cudaStream_t)stream));
  return 0;
}

HY_API int hyena_b200_fftconv_fwd(const float* u, const float* kspec, const float* Dvec, float* out, int B, int H, int L,
                           void* workspace, size_t workspace_bytes, void* stream) {
  if (check_shape(B, H, L)) return 1;
  HY_CHECK(u && kspec && Dvec && out, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  Twiddles T;
  if (get_twiddles(s, &T)) return 1;
  Carve c;
  if (carve(workspace, workspace_bytes, B, H, L, false, &c)) return 1;
  PassArgs a = base_args(B, H, L, T);
  a.A = c.A; a.kspec = reinterpret_cast<const float2*>(kspec);
  a.src = u; a.fbias = Dvec; a.out = out;
  a.vec = ((L & 1) == 0) && aligned8(u) && aligned8(out);
  for (int c0 = 0; c0 < H; c0 += c.nch) {
    const int n = (H - c0 < c.nch) ? H - c0 : c.nch;
    a.c0 = c0;
    HY_CUDA(launch_col_fwd(COL_PLAIN, a, n * B, s));
    HY_CUDA(launch_row_pass(ROW_CONV_FWD, a, n * B, s));
    HY_CUDA(launch_col_inv(INV_PLAIN_FWD, a, n * B, s));
  }
  return 0;
}

HY_API int hyena_b200_fftconv_bwd(const float* dout, const float* u, const float* kspec, const float* Dvec, float* du,
                           float* dk, float* dD, int B, int H, int L, void* workspace, size_t workspace_bytes,
                           void* stream) {
  if (check_shape(B, H, L)) return 1;
  HY_CHECK(dout && u && kspec && Dvec && du && dk && dD, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  Twiddles T;
  if (get_twiddles(s, &T)) return 1;
  Carve c;
  if (carve(workspace, workspace_bytes, B, H, L, true, &c)) return 1;
  PassArgs a = base_args(B, H, L, T);
  a.kspec = reinterpret_cast<const float2*>(kspec);
  a.fbias = Dvec;
  a.vec = ((L & 1) == 0) && aligned8(u) && aligned8(dout) && aligned8(du) && aligned8(dk);
  for (int c0 = 0; c0 < H; c0 += c.nch) {
    const int n = (H - c0 < c.nch) ? H - c0 : c.nch;
    a.c0 = c0; a.B = B;
    a.A2 = c.A2; a.A3 = c.A3;
    a.A = c.A; a.src = dout;
    HY_CUDA(launch_col_fwd(COL_PLAIN, a, n * B, s));
    a.A = c.A2; a.src = u;
    HY_CUDA(launch_col_fwd(COL_PLAIN, a, n * B, s));
    a.A = c.A;
    HY_CUDA(launch_row_pass(ROW_CONV_BWD, a, n, s));
    a.src = u; a.src2 = dout; a.out = du; a.red = dD;
    HY_CUDA(launch_col_inv(INV_PLAIN_BWD, a, n * B, s));
    a.B = 1; a.out = dk;
    HY_CUDA(launch_col_inv(INV_DK, a, n, s));
  }
  return 0;
}

/* d deltas (D) = gradient of k = h * (exp(-t |deltas|) + shift) w.r.t. deltas (ExponentialModulation with modulation_lr != 0,
 * hyena.py:145-155); k is the filter the forward produced, dk its gradient, both (D, L); t (L). */
HY_API int hyena_b200_filter_ddelta(const float* dk, const float* k, const float* t, const float* deltas, float shift, int D,
                             int L, float* ddelta, void* stream) {
  HY_CHECK(D >= 1 && L >= 1 && dk && k && t && deltas && ddelta, "filter_ddelta: bad arguments");
  HY_CUDA(launch_filter_ddelta(dk, k, t, deltas, shift, D, L, ddelta, (cudaStream_t)stream));
  return 0;
}

/* normalized=True (hyena.py:235-236): out[c][t] = k[c][t] / norm[t], norm[t] = sum_c |k[c][t]|;  bwd: dk from dout, out, norm */
HY_API int hyena_b200_filter_l1norm_fwd(const float* k, float* out, float* norm, int D, int L, void* stream) {
  HY_CHECK(D >= 1 && L >= 1 && k && out && norm, "filter_l1norm_fwd: bad arguments");
  HY_CUDA(launch_l1norm_fwd(k, out, norm, D, L, (cudaStream_t)stream));
  return 0;
}
HY_API int hyena_b200_filter_l1norm_bwd(const float* dout, const float* out, const float* norm, float* dk, int D, int L,
                                 void* stream) {
  HY_CHECK(D >= 1 && L >= 1 && dout && out && norm && dk, "filter_l1norm_bwd: bad arguments");
  HY_CUDA(launch_l1norm_bwd(dout, out, norm, dk, D, L, (cudaStream_t)stream));
  return 0;
}

/* y = LayerNorm(x + res) * w + b, res_out = x + res (flash_attn/modules/block.py:111-148, pre-norm Block) */
HY_API size_t hyena_b200_add_layernorm_scratch_bytes(long long rows, int D) {
  return (rows < 1 || D < 1) ? 0 : (size_t)ln_partials(rows) * 2 * (size_t)D * sizeof(float);
}

HY_API int hyena_b200_add_layernorm_fwd(const float* x, const float* res, const float* w, const float* b, float eps,
                                 float* res_out, float* y, float* mean, float* rstd, long long rows, int D, void* stream) {
  HY_CHECK(rows >= 1 && D >= 1, "bad shape rows=%lld D=%d", rows, D);
  HY_CHECK(x && w && y && mean && rstd, "null pointer");
  HY_CHECK(res == nullptr || res_out != nullptr, "res_out is required when a residual is added");
  ln::FwdArgs a{x, res, w, b, res_out, y, mean, rstd, rows, D, eps};
  HY_CUDA(launch_add_ln_fwd(a, (cudaStream_t)stream));
  return 0;
}

HY_API int hyena_b200_add_layernorm_bwd(const float* dy, const float* dres, const float* r, const float* w, const float* mean,
                                 const float* rstd, float* dx, float* dw, float* db, long long rows, int D, void* scratch,
                                 size_t scratch_bytes, void* stream) {
  HY_CHECK(rows >= 1 && D >= 1, "bad shape rows=%lld D=%d", rows, D);
  HY_CHECK(dy && r && w && mean && rstd && dx && dw && scratch, "null pointer");
  HY_CHECK(scratch_bytes >= hyena_b200_add_layernorm_scratch_bytes(rows, D), "scratch too small (%zu bytes)", scratch_bytes);
  ln::BwdArgs a{dy, dres, r, w, mean, rstd, dx, reinterpret_cast<float*>(scratch), rows, D};
  HY_CUDA(launch_add_ln_bwd(a, dw, db, (cudaStream_t)stream));
  return 0;
}

/* incremental decoding of the order-2 operator (k_decode.cu): prompt prefill and the per-token step */
static int check_decode_shape(int B, int D, int max_len) {
  HY_CHECK(B >= 1 && D >= 1 && max_len >= 1, "bad decode shape B=%d D=%d max_len=%d", B, D, max_len);
  HY_CHECK(max_len <= hyena_b200_max_seqlen(), "max_len %d exceeds the supported maximum %d", max_len,
           hyena_b200_max_seqlen());
  HY_CHECK(B <= decode_max_batch(), "decode batch %d exceeds the supported maximum %d", B, decode_max_batch());
  return 0;
}

HY_API size_t hyena_b200_decode_workspace_bytes(int B, int D, int max_len) {
  return (B < 1 || D < 1 || max_len < 1) ? 0 : decode_workspace_bytes(B, D, max_len);
}

HY_API int hyena_b200_decode_prefill(const float* p, const float* in_bias, const float* sw, const float* sb, float* g_hist,
                                     float* fir, int B, int D, int Lp, int max_len, void* stream) {
  if (check_decode_shape(B, D, max_len)) return 1;
  HY_CHECK(Lp >= 1 && Lp <= max_len, "prompt length %d outside [1, max_len = %d]", Lp, max_len);
  HY_CHECK(p && sw && sb && g_hist && fir, "null pointer");
  HY_CUDA(launch_decode_prefill(p, in_bias, sw, sb, g_hist, fir, B, D, Lp, max_len, (cudaStream_t)stream));
  return 0;
}

HY_API int hyena_b200_decode_step(const float* u_t, const float* W_in, const float* in_bias, const float* sw, const float* sb,
                                  const float* k, const float* fbias, const float* W_out, const float* out_bias,
                                  float* g_hist, float* fir, float* y_t, int B, int D, int t, int max_len,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  if (check_decode_shape(B, D, max_len)) return 1;
  HY_CHECK(t >= 0 && t < max_len, "position t = %d outside [0, max_len = %d)", t, max_len);
  HY_CHECK(u_t && W_in && sw && sb && k && fbias && W_out && g_hist && fir && y_t && workspace, "null pointer");
  HY_CHECK(workspace_bytes >= decode_workspace_bytes(B, D, max_len),
           "decode workspace too small: %zu bytes given, %zu needed (hyena_b200_decode_workspace_bytes)", workspace_bytes,
           decode_workspace_bytes(B, D, max_len));
  DecodeStep d{u_t, W_in, in_bias, sw, sb, k, fbias, W_out, out_bias, g_hist, fir, y_t, B, D, t, max_len};
  HY_CUDA(launch_decode_step(d, workspace, (cudaStream_t)stream));
  return 0;
}

}  // extern "C"
