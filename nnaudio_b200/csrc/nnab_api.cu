// extern "C" entry points of libnnab.so — see include/nnab.h for the contract
// and the reference file:line each call replaces.
#include <cuda.h>
#include <cuda_bf16.h>
#include <atomic>
#include <mutex>
#include <stdlib.h>
#include <string.h>
#include <unordered_map>
#include <utility>
#include <vector>

#include "common.cuh"
#include "tc_host.cuh"

namespace nnab {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};
static std::atomic<uint64_t> g_balanced_launches{0};

void set_cuda_error(const char* where, cudaError_t e) {
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", where, cudaGetErrorName(e), cudaGetErrorString(e));
}
void set_error_text(const char* text) { snprintf(g_err, sizeof(g_err), "%s", text); }
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
void count_balanced_launch() { g_balanced_launches.fetch_add(1, std::memory_order_relaxed); }
static std::atomic<int> g_sm_reserve{0};
int sm_reserve() { return g_sm_reserve.load(std::memory_order_relaxed); }

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// T of a centred / un-centred framing: (L + 2*pad - K)/hop + 1
static inline int64_t frames_of(int64_t L, int K, int hop, int pad) {
  const int64_t span = L + 2 * (int64_t)pad - K;
  return span < 0 ? 0 : span / hop + 1;
}

static int check_common(const void* x, int64_t B, int64_t L, int64_t x_pitch, int K, int F,
                        int hop, int pad, int pad_mode, int64_t T) {
  if (x == nullptr || B < 0 || L <= 0 || x_pitch < L || K <= 0 || F <= 0 || hop <= 0)
    return NNAB_EINVAL;
  if (pad_mode != NNAB_PAD_REFLECT && pad_mode != NNAB_PAD_CONSTANT) return NNAB_EINVAL;
  // nn.ReflectionPad1d needs pad < L; callers raise the reference's exception first.
  if (pad > 0 && pad_mode == NNAB_PAD_REFLECT && pad >= L) return NNAB_EINVAL;
  if (T != frames_of(L, K, hop, pad) || T <= 0) return NNAB_EINVAL;
  return NNAB_OK;
}

static int check_arch() {
  int dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&dev));
  int major = 0;
  NNAB_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  return major == 10 ? NNAB_OK : NNAB_EARCH;
}

// ---- optional in-stream timing of the framed contraction (bench.py) --------
static std::atomic<int> g_prof_on{0};
static std::mutex g_prof_mu;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_pairs;  // recorded, unread
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_free;

static double g_exec_flops = 0.0;  // guarded by g_prof_mu
void add_exec_flops(double flops) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_exec_flops += flops;
}

static bool prof_begin(cudaStream_t s, std::pair<cudaEvent_t, cudaEvent_t>* pr) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return false;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_free.empty()) {
    *pr = g_prof_free.back();
    g_prof_free.pop_back();
  } else {
    if (cudaEventCreate(&pr->first) != cudaSuccess) return false;
    if (cudaEventCreate(&pr->second) != cudaSuccess) return false;
  }
  cudaEventRecord(pr->first, s);
  return true;
}
static void prof_end(cudaStream_t s, const std::pair<cudaEvent_t, cudaEvent_t>& pr) {
  cudaEventRecord(pr.second, s);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_pairs.push_back(pr);
}

static int run_framed_inner(const FramedProblem& p, const void* packed, void* ws, size_t ws_bytes,
                            int path, cudaStream_t stream);

// Run one framed contraction on the requested kernel family.
static int run_framed(const FramedProblem& p, const void* packed, void* ws, size_t ws_bytes,
                      int path, cudaStream_t stream) {
  std::pair<cudaEvent_t, cudaEvent_t> pr;
  const bool timed = prof_begin(stream, &pr);
  const int rc = run_framed_inner(p, packed, ws, ws_bytes, path, stream);
  if (timed) prof_end(stream, pr);
  return rc;
}

static int run_framed_inner(const FramedProblem& p, const void* packed, void* ws, size_t ws_bytes,
                      int path, cudaStream_t stream) {
  bool use_tc = false;
  if (path == NNAB_PATH_TCGEN05) {
    if (packed == nullptr || !tc_supported(p)) return NNAB_EALIGN;
    use_tc = true;
  } else if (path == NNAB_PATH_AUTO) {
    use_tc = (packed != nullptr) && tc_supported(p);
  } else if (path != NNAB_PATH_SIMT) {
    return NNAB_EINVAL;
  }
  if (use_tc) return launch_framed_tc(p, packed, ws, ws_bytes, stream);
  return launch_framed_simt(p, stream);
}

// The split-K scratch (long kernels only) sits behind the split-signal planes in the workspace.
static void attach_splitk_scratch(FramedProblem& p, void* workspace, size_t ws_bytes) {
  const size_t sk = tc_splitk_scratch_bytes(p.B, p.F, p.T, p.K);
  if (sk == 0 || workspace == nullptr) return;
  const size_t front = align_up(tc_workspace_bytes(p.B, p.L, p.K, p.hop, p.pad), 256);
  if (front + sk <= ws_bytes) p.raw = reinterpret_cast<float*>((char*)workspace + front);
}

static bool wants_tc(int path, int K, int hop) {
  if (path == NNAB_PATH_SIMT) return false;
  FramedProblem q{};
  q.K = K; q.hop = hop; q.F = 1; q.B = 1; q.L = K; q.T = 1;
  return tc_supported(q);
}

}  // namespace nnab

using namespace nnab;

extern "C" {

int nnab_abi_version(void) { return NNAB_ABI_VERSION; }

const char* nnab_strerror(int status) {
  switch (status) {
    case NNAB_OK: return "ok";
    case NNAB_EINVAL: return "invalid argument or shape mismatch";
    case NNAB_EALIGN: return "tcgen05 path forced but shape/alignment rules not met";
    case NNAB_EARCH: return "device is not sm_100 (B200)";
    case NNAB_ECUDA: return "CUDA error";
    case NNAB_EWORKSPACE: return "workspace missing or too small";
    case NNAB_EUNSUPPORTED: return "unsupported size";
    default: return "unknown status";
  }
}

const char* nnab_last_cuda_error(void) { return g_err; }

uint64_t nnab_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

uint64_t nnab_balanced_launch_count(void) { return g_balanced_launches.load(std::memory_order_relaxed); }

int nnab_set_sm_reserve(int n_sms) {
  if (n_sms < 0) n_sms = 0;
  if (n_sms > 64) n_sms = 64;
  return g_sm_reserve.exchange(n_sms);
}

void nnab_profile_enable(int on) { g_prof_on.store(on ? 1 : 0); }

int nnab_profile_read(double* framed_ms, uint64_t* framed_launches) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double total = 0.0;
  uint64_t n = 0;
  for (auto& pr : g_prof_pairs) {
    NNAB_CUDA_TRY(cudaEventSynchronize(pr.second));
    float ms = 0.f;
    NNAB_CUDA_TRY(cudaEventElapsedTime(&ms, pr.first, pr.second));
    total += ms;
    ++n;
    g_prof_free.push_back(pr);
  }
  g_prof_pairs.clear();
  if (framed_ms) *framed_ms = total;
  if (framed_launches) *framed_launches = n;
  return NNAB_OK;
}

int nnab_profile_read_exec_flops(double* exec_flops) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (exec_flops) *exec_flops = g_exec_flops;
  g_exec_flops = 0.0;
  return NNAB_OK;
}

int nnab_pack_tile_n(int F) { return tc_tile_n(F); }
size_t nnab_packed_basis_bytes(int F, int K) { return tc_packed_bytes(F, K); }
int nnab_pack_basis(const float* w_re, const float* w_im, int F, int K, void* packed,
                    void* stream) {
  if (w_re == nullptr || w_im == nullptr || packed == nullptr || F <= 0 || K <= 0)
    return NNAB_EINVAL;
  return tc_pack_basis(w_re, w_im, F, K, packed, (cudaStream_t)stream);
}

int nnab_pack_basis_ex(const float* w_re, const float* w_im, int F, int K, int layout, void* packed,
                       void* stream) {
  if (w_re == nullptr || w_im == nullptr || packed == nullptr || F <= 0 || K <= 0)
    return NNAB_EINVAL;
  return tc_pack_basis_layout(w_re, w_im, F, K, layout, packed, (cudaStream_t)stream);
}

// Stream memory operations (multi-GPU gather handshakes without kernels): thin wrappers over the driver
// entry points, resolved at run time like cuTensorMapEncodeTiled.
typedef CUresult (*StreamValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
static StreamValue32Fn memop_fn(const char* name) {
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint(name, &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  return reinterpret_cast<StreamValue32Fn>(ptr);
}
int nnab_stream_write_value32(void* stream, void* addr, uint32_t value) {
  static StreamValue32Fn fn = memop_fn("cuStreamWriteValue32");
  if (fn == nullptr || addr == nullptr) return NNAB_EUNSUPPORTED;
  const CUresult r = fn((CUstream)stream, (CUdeviceptr)(uintptr_t)addr, value, 0 /* default */);
  if (r != CUDA_SUCCESS) { set_error_text("cuStreamWriteValue32 failed"); return NNAB_ECUDA; }
  return NNAB_OK;
}
int nnab_stream_wait_value32_geq(void* stream, void* addr, uint32_t value) {
  static StreamValue32Fn fn = memop_fn("cuStreamWaitValue32");
  if (fn == nullptr || addr == nullptr) return NNAB_EUNSUPPORTED;
  const CUresult r = fn((CUstream)stream, (CUdeviceptr)(uintptr_t)addr, value, 0 /* GEQ */);
  if (r != CUDA_SUCCESS) { set_error_text("cuStreamWaitValue32 failed"); return NNAB_ECUDA; }
  return NNAB_OK;
}

int nnab_block_layout_ok(int n_fft, int hop) { return tc_block_shape_ok(n_fft, hop) ? 1 : 0; }

size_t nnab_packed_block_bytes(int n_fft, int hop) { return tc_packed_block_bytes(n_fft, hop); }

int nnab_pack_basis_block(int n_fft, int hop, void* packed, void* stream) {
  if (packed == nullptr) return NNAB_EINVAL;
  return tc_pack_basis_block(n_fft, hop, packed, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ STFT ----
size_t nnab_stft_workspace_bytes(int64_t B, int64_t L, int n_fft, int F, int hop, int center,
                                 int path) {
  if (!wants_tc(path, n_fft, hop)) return 0;
  const int pad = center ? n_fft / 2 : 0;
  return align_up(tc_workspace_bytes(B, L, n_fft, hop, pad), 256) +
         tc_splitk_scratch_bytes(B, F, frames_of(L, n_fft, hop, pad), n_fft);
}

int nnab_stft_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch, const float* wcos,
                      const float* wsin, const void* packed, int n_fft, int F, int hop,
                      int center, int pad_mode, int out_format, float sqrt_eps, float* out,
                      int64_t T, void* workspace, size_t ws_bytes, int path, void* stream) {
  return nnab_stft_forward_ex(x, B, L, x_pitch, wcos, wsin, packed, n_fft, F, hop, center, pad_mode,
                              out_format, sqrt_eps, out, T, workspace, ws_bytes, path, stream,
                              NNAB_DTYPE_F32);
}

int nnab_stft_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch, const float* wcos,
                         const float* wsin, const void* packed, int n_fft, int F, int hop,
                         int center, int pad_mode, int out_format, float sqrt_eps, float* out,
                         int64_t T, void* workspace, size_t ws_bytes, int path, void* stream,
                         int x_dtype) {
  if (!valid_x_dtype(x_dtype)) return NNAB_EINVAL;
  const int pad = center ? n_fft / 2 : 0;
  int rc = check_common(x, B, L, x_pitch, n_fft, F, hop, pad, pad_mode, T);
  if (rc) return rc;
  if (wcos == nullptr || wsin == nullptr || out == nullptr) return NNAB_EINVAL;
  if (out_format != NNAB_FMT_MAGNITUDE && out_format != NNAB_FMT_COMPLEX &&
      out_format != NNAB_FMT_PHASE_ANGLE)
    return NNAB_EINVAL;
  if ((rc = check_arch())) return rc;
  FramedProblem p{};
  p.x = x; p.B = B; p.L = L; p.x_pitch = x_pitch; p.x_dtype = x_dtype;
  p.w_re = wcos; p.w_im = wsin; p.F = F; p.K = n_fft; p.hop = hop;
  p.pad = pad; p.pad_mode = pad_mode; p.scale = nullptr; p.scale_all = 1.f;
  p.fmt = out_format; p.eps = sqrt_eps; p.power = 1.f; p.out = out; p.T = T;
  p.out_bins = F; p.bin_offset = 0;
  attach_splitk_scratch(p, workspace, ws_bytes);
  return run_framed(p, packed, workspace, ws_bytes, path, (cudaStream_t)stream);
}

// ------------------------------------------------- Mel / Gammatone / MFCC ----
// workspace layout: [P (B,F,T) fp32][tc scratch]  (+ [mel (B,n_mels,T)][B words] for MFCC)
static size_t power_bytes(int64_t B, int F, int64_t T) {
  return align_up((size_t)B * F * T * sizeof(float), 256);
}

// table buffer: [FbEntry x F][pad to 64][int max_nnz, widest, ok, -][pad to 256][FbStep x (F + FB_STEP_PAD)]
static size_t fb_meta_offset(int F) { return align_up((size_t)F * sizeof(FbEntry), 64); }
static size_t fb_steps_offset(int F) { return align_up(fb_meta_offset(F) + 64, 256); }
size_t nnab_filterbank_table_bytes(int F) {
  return fb_steps_offset(F) + (size_t)(F + FB_STEP_PAD) * sizeof(FbStep);
}

// deterministic-tile-width mask per table buffer (host copy of the device meta word; read at launch time)
static std::mutex g_fbw_mu;
static std::unordered_map<const void*, int> g_fb_width;
static int fb_width_of(const void* table) {
  std::lock_guard<std::mutex> lk(g_fbw_mu);
  auto it = g_fb_width.find(table);
  return it == g_fb_width.end() ? 0 : it->second;
}

int nnab_build_filterbank_table(const float* fb, int n_fb, int F, void* table, int* h_max_nnz,
                                void* stream) {
  if (fb == nullptr || table == nullptr || h_max_nnz == nullptr || n_fb <= 0 || F <= 0)
    return NNAB_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  char* base = reinterpret_cast<char*>(table);
  int* d_meta = reinterpret_cast<int*>(base + fb_meta_offset(F));
  int rc = launch_fb_table(fb, n_fb, F, reinterpret_cast<FbEntry*>(table), d_meta, s);
  if (rc) return rc;
  if (n_fb < 32768 &&
      (rc = launch_fb_steps(reinterpret_cast<const FbEntry*>(table), n_fb, F,
                            reinterpret_cast<FbStep*>(base + fb_steps_offset(F)), d_meta + 1, s)))
    return rc;
  int h_meta[3] = {0, 0, 0};
  NNAB_CUDA_TRY(cudaMemcpyAsync(h_meta, d_meta, sizeof(h_meta), cudaMemcpyDeviceToHost, s));
  NNAB_CUDA_TRY(cudaStreamSynchronize(s));
  *h_max_nnz = h_meta[0];
  {
    std::lock_guard<std::mutex> lk(g_fbw_mu);
    g_fb_width[table] = (n_fb < 32768) ? h_meta[2] : 0;
  }
  return NNAB_OK;
}

// ---- dense filterbank (Gammatonegram, dense mel banks) on the tensor cores -------------------------
// The block-partial STFT kernel writes |X| ** power straight into bf16 hi/lo operand planes (FMT_PLANES: one
// row per frame, 4 B per value, no fp32 (B, F, T) intermediate), a second tcgen05 launch contracts the rows
// with the re-indexed bank (real GEMM on the complex kernel, FMT_REALPAIR) and writes (B, n_fb, T).
// Workspace: [signal planes of the STFT][operand planes][bank fp32 re | im][packed bank].
static bool fb_planes_enabled() {
  if (const char* e = getenv("NNAB_FB_PLANES")) return atoi(e) != 0;
  // on by default: GPU-verified (profiles/r02c_*: oracle <= 8e-6, bit-repeatable; Gammatonegram at the cfg2
  // shape 0.330 -> 0.249 ms); 0 = fp32 (B, F, T) power spectrogram + CUDA-core filterbank GEMM (round 1)
  return true;
}

struct FbPlanes {
  int nb, n_tiles, kp, fh;
  int64_t rows;  // B * T frame rows
  size_t off_planes, off_w, off_packed, total;
};

static bool fb_planes_layout(int64_t B, int64_t L, int n_fft, int F, int hop, int pad, int64_t T, int n_fb,
                             FbPlanes* o) {
  if (!tc_block_shape_ok(n_fft, hop) || F != n_fft / 2 + 1 || n_fb < 1 || T <= 0 || B <= 0) return false;
  tc_block_tile_geometry(F, &o->nb, &o->n_tiles);
  o->kp = (o->nb * o->n_tiles + 63) / 64 * 64;
  o->fh = (n_fb + 1) / 2;
  o->rows = B * T;
  if (o->rows >= (1ll << 31) || o->kp > 32768) return false;
  size_t off = align_up(tc_workspace_bytes(B, L, n_fft, hop, pad), 256);
  o->off_planes = off; off += align_up((size_t)2 * o->rows * o->kp * 2, 256);
  o->off_w = off;      off += 2 * align_up((size_t)o->fh * o->kp * sizeof(float), 256);
  o->off_packed = off; off += align_up(tc_packed_bytes(o->fh, o->kp), 256);
  o->total = off + 256;
  return true;
}

static bool fused_fbank(int path, const void* packed, const void* fb_table, int n_fft, int hop) {
  return fb_table != nullptr && packed != nullptr && path != NNAB_PATH_SIMT &&
         wants_tc(path, n_fft, hop);
}

size_t nnab_filterbank_workspace_bytes(int64_t B, int64_t L, int n_fft, int F, int hop,
                                       int center, int n_fb, int path, int has_table) {
  const int pad = center ? n_fft / 2 : 0;
  const int64_t T = frames_of(L, n_fft, hop, pad);
  const bool tc = wants_tc(path, n_fft, hop);
  size_t n = 0;
  if (!(has_table && tc)) n += power_bytes(B, F, T);  // un-fused: (B,F,T) power spectrogram
  if (tc) n += tc_workspace_bytes(B, L, n_fft, hop, pad);
  if (!has_table && tc) {  // dense bank on the tensor cores: operand planes instead of the fp32 spectrogram
    FbPlanes fp;
    if (fb_planes_layout(B, L, n_fft, F, hop, pad, T, n_fb, &fp) && fp.total > n) n = fp.total;
  }
  return n;
}

static int power_spectrogram(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch,
                             const float* wcos, const float* wsin, const void* packed,
                             int n_fft, int F, int hop, int pad, int pad_mode, float sqrt_eps,
                             float power, float* P, int64_t T, void* tc_ws, size_t tc_ws_bytes,
                             int path, cudaStream_t stream) {
  FramedProblem p{};
  p.x = x; p.B = B; p.L = L; p.x_pitch = x_pitch; p.x_dtype = x_dtype;
  p.w_re = wcos; p.w_im = wsin; p.F = F; p.K = n_fft; p.hop = hop;
  p.pad = pad; p.pad_mode = pad_mode; p.scale = nullptr; p.scale_all = 1.f;
  p.fmt = FMT_POWER; p.eps = sqrt_eps; p.power = power; p.out = P; p.T = T;
  p.out_bins = F; p.bin_offset = 0;
  return run_framed(p, packed, tc_ws, tc_ws_bytes, path, stream);
}

int nnab_stft_filterbank_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch,
                                 const float* wcos, const float* wsin, const void* packed,
                                 int n_fft, int F, int hop, int center, int pad_mode,
                                 float sqrt_eps, float power, const float* fb, int n_fb,
                                 const void* fb_table, float* out, int64_t T, void* workspace,
                                 size_t ws_bytes, int path, void* stream) {
  return nnab_stft_filterbank_forward_ex(x, B, L, x_pitch, wcos, wsin, packed, n_fft, F, hop, center,
                                         pad_mode, sqrt_eps, power, fb, n_fb, fb_table, out, T,
                                         workspace, ws_bytes, path, stream, NNAB_DTYPE_F32);
}

int nnab_stft_filterbank_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch,
                                    const float* wcos, const float* wsin, const void* packed,
                                    int n_fft, int F, int hop, int center, int pad_mode,
                                    float sqrt_eps, float power, const float* fb, int n_fb,
                                    const void* fb_table, float* out, int64_t T, void* workspace,
                                    size_t ws_bytes, int path, void* stream, int x_dtype) {
  if (!valid_x_dtype(x_dtype)) return NNAB_EINVAL;
  const int pad = center ? n_fft / 2 : 0;
  int rc = check_common(x, B, L, x_pitch, n_fft, F, hop, pad, pad_mode, T);
  if (rc) return rc;
  if (wcos == nullptr || wsin == nullptr || fb == nullptr || out == nullptr || n_fb <= 0)
    return NNAB_EINVAL;
  if ((rc = check_arch())) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  bool fused = fused_fbank(path, packed, fb_table, n_fft, hop);
  if (fused) {
    FramedProblem p{};
    p.x = x; p.B = B; p.L = L; p.x_pitch = x_pitch; p.x_dtype = x_dtype;
    p.w_re = wcos; p.w_im = wsin; p.F = F; p.K = n_fft; p.hop = hop;
    p.pad = pad; p.pad_mode = pad_mode; p.scale = nullptr; p.scale_all = 1.f;
    p.fmt = FMT_FBANK; p.eps = sqrt_eps; p.power = power; p.out = out; p.T = T;
    p.out_bins = n_fb; p.bin_offset = 0;
    p.fb_table = reinterpret_cast<const FbEntry*>(fb_table); p.n_fb = n_fb;
    p.fb_steps = reinterpret_cast<const FbStep*>(reinterpret_cast<const char*>(fb_table) + fb_steps_offset(F));
    p.fb_nb_mask = fb_width_of(fb_table);
    if (tc_supported(p)) {
      const size_t need = tc_workspace_bytes(B, L, n_fft, hop, pad);
      if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
      // the epilogue accumulates filter sums with fp32 atomics: start from zero
      NNAB_CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)B * n_fb * T * sizeof(float), s));
      return run_framed(p, packed, workspace, ws_bytes, NNAB_PATH_TCGEN05, s);
    }
    fused = false;
  }
  const size_t need = nnab_filterbank_workspace_bytes(B, L, n_fft, F, hop, center, n_fb, path, 0);
  if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  {
    FbPlanes fp;
    if (fb_planes_enabled() && path != NNAB_PATH_SIMT && packed != nullptr && packed_kind(packed) == PACK_BLOCK &&
        wants_tc(path, n_fft, hop) && B <= 65535 &&
        fb_planes_layout(B, L, n_fft, F, hop, pad, T, n_fb, &fp) && ws_bytes >= fp.total) {
      char* ws = reinterpret_cast<char*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
      __nv_bfloat16* planes = reinterpret_cast<__nv_bfloat16*>(ws + fp.off_planes);
      float* w_re = reinterpret_cast<float*>(ws + fp.off_w);
      float* w_im = reinterpret_cast<float*>(ws + fp.off_w + align_up((size_t)fp.fh * fp.kp * sizeof(float), 256));
      void* bank = ws + fp.off_packed;
      const int64_t plane_stride = fp.rows * fp.kp;
      // the re-indexed bank (tiny: fh x kp) and its bf16 hi/lo packing
      if ((rc = launch_fb_tile_bank(fb, n_fb, F, fp.nb, fp.n_tiles, fp.kp, fp.fh, w_re, w_im, s))) return rc;
      if ((rc = tc_pack_basis(w_re, w_im, fp.fh, fp.kp, bank, s))) return rc;
      // columns no tile writes (kp is the 64-multiple above n_tiles * nb): finite zeros in both planes
      if (fp.kp > fp.nb * fp.n_tiles)
        NNAB_CUDA_TRY(cudaMemset2DAsync(planes + fp.nb * fp.n_tiles, (size_t)fp.kp * 2, 0,
                                        (size_t)(fp.kp - fp.nb * fp.n_tiles) * 2, (size_t)(2 * fp.rows), s));
      // 1. STFT -> |X| ** power as operand planes (block-partial kernel, FMT_PLANES)
      FramedProblem p{};
      p.x = x; p.B = B; p.L = L; p.x_pitch = x_pitch; p.x_dtype = x_dtype;
      p.w_re = wcos; p.w_im = wsin; p.F = F; p.K = n_fft; p.hop = hop;
      p.pad = pad; p.pad_mode = pad_mode; p.scale = nullptr; p.scale_all = 1.f;
      p.fmt = FMT_PLANES; p.eps = sqrt_eps; p.power = power; p.out = reinterpret_cast<float*>(planes); p.T = T;
      p.out_bins = F; p.bin_offset = 0;
      p.planes_stride = plane_stride; p.planes_pitch = fp.kp;
      if ((rc = run_framed(p, packed, ws, fp.off_planes, NNAB_PATH_TCGEN05, s))) return rc;
      // 2. rows x bank on the dense kernel: every frame is one "hop" of kp samples
      FramedProblem g{};
      g.x = nullptr; g.B = B; g.L = T * fp.kp; g.x_pitch = T * fp.kp;
      g.w_re = w_re; g.w_im = w_im; g.F = fp.fh; g.K = fp.kp; g.hop = fp.kp;
      g.pad = 0; g.pad_mode = NNAB_PAD_CONSTANT; g.scale = nullptr; g.scale_all = 1.f;
      g.fmt = FMT_REALPAIR; g.eps = 0.f; g.power = 1.f; g.out = out; g.T = T;
      g.out_bins = n_fb; g.bin_offset = 0;
      g.presplit = planes; g.presplit_t_slots = T; g.presplit_plane_stride = plane_stride;
      return run_framed(g, bank, nullptr, 0, NNAB_PATH_TCGEN05, s);
    }
  }
  float* P = (float*)workspace;
  const size_t pb = power_bytes(B, F, T);
  rc = power_spectrogram(x, x_dtype, B, L, x_pitch, wcos, wsin, packed, n_fft, F, hop, pad, pad_mode,
                         sqrt_eps, power, P, T, (char*)workspace + pb, ws_bytes - pb, path, s);
  if (rc) return rc;
  return launch_filterbank(P, fb, B, F, T, n_fb, out, s);
}

static size_t mel_bytes(int64_t B, int n_mels, int64_t T) {
  return align_up((size_t)B * n_mels * T * sizeof(float), 256);
}

size_t nnab_mfcc_workspace_bytes(int64_t B, int64_t L, int n_fft, int F, int hop, int center,
                                 int n_mels, int path, int has_table) {
  const int pad = center ? n_fft / 2 : 0;
  const int64_t T = frames_of(L, n_fft, hop, pad);
  // the un-fused size is the upper bound (a huge batch can still fall back to it)
  const size_t fbw = nnab_filterbank_workspace_bytes(B, L, n_fft, F, hop, center, n_mels, path, 0);
  (void)has_table;
  return align_up(fbw, 256) + mel_bytes(B, n_mels, T) + align_up((size_t)B * sizeof(unsigned int), 256);
}

int nnab_mfcc_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch, const float* wcos,
                      const float* wsin, const void* packed, int n_fft, int F, int hop,
                      int center, int pad_mode, float sqrt_eps, float power,
                      const float* mel_basis, int n_mels, const void* fb_table, float amin,
                      float ref, float top_db, const float* dct, int n_mfcc, float* out,
                      int64_t T, void* workspace, size_t ws_bytes, int path, void* stream) {
  return nnab_mfcc_forward_ex(x, B, L, x_pitch, wcos, wsin, packed, n_fft, F, hop, center, pad_mode,
                              sqrt_eps, power, mel_basis, n_mels, fb_table, amin, ref, top_db, dct,
                              n_mfcc, out, T, workspace, ws_bytes, path, stream, NNAB_DTYPE_F32);
}

int nnab_mfcc_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch, const float* wcos,
                         const float* wsin, const void* packed, int n_fft, int F, int hop,
                         int center, int pad_mode, float sqrt_eps, float power,
                         const float* mel_basis, int n_mels, const void* fb_table, float amin,
                         float ref, float top_db, const float* dct, int n_mfcc, float* out,
                         int64_t T, void* workspace, size_t ws_bytes, int path, void* stream,
                         int x_dtype) {
  if (!valid_x_dtype(x_dtype)) return NNAB_EINVAL;
  const int pad = center ? n_fft / 2 : 0;
  int rc = check_common(x, B, L, x_pitch, n_fft, F, hop, pad, pad_mode, T);
  if (rc) return rc;
  if (wcos == nullptr || wsin == nullptr || mel_basis == nullptr || dct == nullptr ||
      out == nullptr || n_mels <= 0 || n_mfcc <= 0 || !(amin > 0.f))
    return NNAB_EINVAL;
  if ((rc = check_arch())) return rc;
  const size_t need = nnab_mfcc_workspace_bytes(B, L, n_fft, F, hop, center, n_mels, path, 0);
  if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  const size_t fbw =
      align_up(nnab_filterbank_workspace_bytes(B, L, n_fft, F, hop, center, n_mels, path, 0), 256);
  float* mel = (float*)((char*)workspace + fbw);
  unsigned int* scratch = (unsigned int*)((char*)workspace + fbw + mel_bytes(B, n_mels, T));
  rc = nnab_stft_filterbank_forward_ex(x, B, L, x_pitch, wcos, wsin, packed, n_fft, F, hop, center,
                                       pad_mode, sqrt_eps, power, mel_basis, n_mels, fb_table, mel,
                                       T, workspace, fbw, path, stream, x_dtype);
  if (rc) return rc;
  return launch_mfcc_tail(mel, B, n_mels, T, amin, ref, top_db, dct, n_mfcc, out, scratch,
                          (cudaStream_t)stream);
}

// ------------------------------------------------------------- CQT1992v2 ----
size_t nnab_cqt1992v2_workspace_bytes(int64_t B, int64_t L, int width, int n_bins, int hop,
                                      int center, int path) {
  if (!wants_tc(path, width, hop)) return 0;
  const int pad = center ? width / 2 : 0;
  return align_up(tc_workspace_bytes(B, L, width, hop, pad), 256) +
         tc_splitk_scratch_bytes(B, n_bins, frames_of(L, width, hop, pad), width);
}

int nnab_cqt1992v2_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch,
                           const float* k_real, const float* k_imag, const void* packed,
                           const int32_t* h_k_begin, const int32_t* h_k_end, int n_bins,
                           int width, int hop, int center, int pad_mode, const float* scale,
                           float scale_all, int out_format, float sqrt_eps, float* out,
                           int64_t T, void* workspace, size_t ws_bytes, int path,
                           void* stream) {
  return nnab_cqt1992v2_forward_ex(x, B, L, x_pitch, k_real, k_imag, packed, h_k_begin, h_k_end, n_bins,
                                   width, hop, center, pad_mode, scale, scale_all, out_format, sqrt_eps,
                                   out, T, workspace, ws_bytes, path, stream, NNAB_DTYPE_F32);
}

int nnab_cqt1992v2_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch,
                              const float* k_real, const float* k_imag, const void* packed,
                              const int32_t* h_k_begin, const int32_t* h_k_end, int n_bins,
                              int width, int hop, int center, int pad_mode, const float* scale,
                              float scale_all, int out_format, float sqrt_eps, float* out,
                              int64_t T, void* workspace, size_t ws_bytes, int path, void* stream,
                              int x_dtype) {
  if (!valid_x_dtype(x_dtype)) return NNAB_EINVAL;
  const int pad = center ? width / 2 : 0;
  int rc = check_common(x, B, L, x_pitch, width, n_bins, hop, pad, pad_mode, T);
  if (rc) return rc;
  if (k_real == nullptr || k_imag == nullptr || out == nullptr) return NNAB_EINVAL;
  if (out_format != NNAB_FMT_MAGNITUDE && out_format != NNAB_FMT_COMPLEX &&
      out_format != NNAB_FMT_PHASE_UNIT)
    return NNAB_EINVAL;
  if ((rc = check_arch())) return rc;
  FramedProblem p{};
  p.x = x; p.B = B; p.L = L; p.x_pitch = x_pitch; p.x_dtype = x_dtype;
  p.w_re = k_real; p.w_im = k_imag; p.F = n_bins; p.K = width; p.hop = hop;
  p.pad = pad; p.pad_mode = pad_mode; p.scale = scale; p.scale_all = scale_all;
  p.fmt = out_format; p.eps = sqrt_eps; p.power = 1.f; p.out = out; p.T = T;
  p.out_bins = n_bins; p.bin_offset = 0;
  p.h_k_begin = h_k_begin; p.h_k_end = h_k_end;
  attach_splitk_scratch(p, workspace, ws_bytes);
  return run_framed(p, packed, workspace, ws_bytes, path, (cudaStream_t)stream);
}

// ------------------------------------------------ CQT2010v2 / VQT pyramid ----
// Level lengths follow conv1d(stride=n, padding=127, kernel=256): (len - 2)/n + 1.
static inline int64_t decimated_len(int64_t len, int factor) {
  return len < 2 ? 0 : (len - 2) / factor + 1;
}

static size_t pyramid_level_bytes(int64_t B, int64_t L, int early_factor) {
  // [early (B, L0)] + ping/pong level buffers (B, <= L0/2 + 1)
  const int64_t L0 = early_factor > 1 ? decimated_len(L, early_factor) : L;
  size_t n = 0;
  if (early_factor > 1) n += align_up((size_t)B * align_up((size_t)L0, 4) * sizeof(float), 256);
  const size_t half = align_up((size_t)(L0 / 2 + 1), 4);
  n += 2 * align_up((size_t)B * half * sizeof(float), 256);
  return n;
}

// ---- plan of the all-tensor-core pyramid -----------------------------------------
constexpr int FIR_TAPS = 256;
constexpr int FIR_OFF = 128;  // sample m of a level sits at plane offset 128 + m in FIR inputs

struct PyrLevel {
  int64_t len;
  int hop, width, pad, mode;
  bool presplit;          // octave reads pre-split planes (single frame phase)
  size_t pc, pf, y32;     // workspace offsets (SIZE_MAX = not needed)
  int64_t pc_pitch, pc_plane, pf_pitch, pf_plane, y32_pitch;
};

static size_t planes_bytes(int64_t B, int64_t L, int K, int hop, int pad, int64_t* pitch,
                           int64_t* plane) {
  int64_t t_slots = 0, ps = 0;
  int he = 0;
  tc_split_geometry(B, L, K, hop, pad, &t_slots, &ps, &he);
  if (pitch) *pitch = t_slots * he;
  if (plane) *plane = ps;
  return align_up((size_t)(2 * ps) * 2, 256);
}

// Fills lv[0..n_octaves) and returns the workspace size; `pf_early` receives the offset of
// the raw-signal FIR input when early downsampling is active.
static size_t plan_pyramid(int64_t B, int64_t L, int n_octaves, int early_factor, int hop,
                           const int32_t* widths, int fixed_width, int pad_mode, PyrLevel* lv,
                           size_t* pf_early) {
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off += n; return o; };
  int64_t len = L;
  if (early_factor > 1) {
    const size_t o = take(planes_bytes(B, L, tc_fir_k(FIR_TAPS, early_factor), 128 * early_factor,
                                       FIR_OFF, nullptr, nullptr));
    if (pf_early) *pf_early = o;
    len = decimated_len(L, early_factor);
  }
  int cur_hop = hop;
  for (int i = 0; i < n_octaves; ++i) {
    if (i > 0) { len = decimated_len(len, 2); cur_hop /= 2; }
    PyrLevel& l = lv[i];
    l.len = len; l.hop = cur_hop;
    l.width = widths ? widths[i] : fixed_width;
    l.pad = l.width / 2;
    l.mode = (pad_mode == NNAB_PAD_REFLECT && l.pad >= len) ? NNAB_PAD_CONSTANT : pad_mode;
    l.presplit = cur_hop > 0 && (cur_hop % 8) == 0;
    l.pc = l.pf = l.y32 = SIZE_MAX;
    l.pc_pitch = l.pc_plane = l.pf_pitch = l.pf_plane = l.y32_pitch = 0;
    if (len <= 0 || cur_hop <= 0) continue;
    const bool from_x = (i == 0 && early_factor <= 1);  // level 0 is the caller's fp32 input
    if (l.presplit)
      l.pc = take(planes_bytes(B, len, l.width, cur_hop, l.pad, &l.pc_pitch, &l.pc_plane));
    else if (!from_x) {
      l.y32_pitch = (int64_t)align_up((size_t)len, 8);
      l.y32 = take(align_up((size_t)B * l.y32_pitch * sizeof(float), 256));
    }
    if (i < n_octaves - 1)
      l.pf = take(planes_bytes(B, len, tc_fir_k(FIR_TAPS, 2), 256, FIR_OFF, &l.pf_pitch,
                               &l.pf_plane));
  }
  // scratch for octaves that run from fp32 (several frame phases): sized for the first such level
  for (int i = 0; i < n_octaves; ++i)
    if (!lv[i].presplit && lv[i].len > 0 && lv[i].hop > 0) {
      off += tc_workspace_bytes(B, lv[i].len, lv[i].width, lv[i].hop, lv[i].pad);
      break;
    }
  return off;
}

// ---------------------------------------------------------------------------------------------
// Pyramid, second generation (round 2): ONE plane set per level, shared by the level's octave CQT
// (reflect margins of `pad` samples, frames every `hop`) and by the FIR stage that produces the next
// level (256-sample rows, resident taps, clip edges recomputed: launch_fir_stage_tc).  Per level and
// sample: one 4-byte write and one read by each consumer, instead of two differently padded copies.
// ---------------------------------------------------------------------------------------------
struct Lvl2 {
  int64_t len;
  int hop, width, pad, mode;
  bool presplit;        // the octave CQT reads the planes directly (single frame phase)
  bool planes;          // the level has planes (CQT and / or FIR source)
  size_t pc, y32;       // workspace offsets (SIZE_MAX = none)
  int64_t pitch, plane, t_slots, y32_pitch;
};

static int64_t gcd64(int64_t a, int64_t b) { return b == 0 ? a : gcd64(b, a % b); }

// false: the shape does not fit this plan (caller uses the first-generation pyramid)
static bool plan_pyramid2(int64_t B, int64_t L, int n_octaves, int hop, const int32_t* widths,
                          int fixed_width, int pad_mode, Lvl2* lv, size_t* total) {
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off += align_up(n, 256); return o; };
  int64_t len = L;
  int cur_hop = hop;
  for (int i = 0; i < n_octaves; ++i) {
    if (i > 0) { len = decimated_len(len, 2); cur_hop /= 2; }
    Lvl2& l = lv[i];
    l.len = len; l.hop = cur_hop;
    l.width = widths ? widths[i] : fixed_width;
    l.pad = l.width / 2;
    if (len <= 0 || cur_hop <= 0) return false;
    l.mode = (pad_mode == NNAB_PAD_REFLECT && l.pad >= len) ? NNAB_PAD_CONSTANT : pad_mode;
    l.presplit = (cur_hop % 8) == 0;
    const bool fir_src = i < n_octaves - 1;
    l.planes = l.presplit || fir_src;
    l.pc = l.y32 = SIZE_MAX;
    l.pitch = l.plane = l.t_slots = l.y32_pitch = 0;
    if (fir_src && l.pad != 128) return false;  // FIR frame origin = CQT padding origin (256-tap banks)
    if (l.planes) {
      const int he = l.presplit ? cur_hop : 8;  // planes of multi-phase levels only feed the FIR
      const int kpad = (l.width + 63) / 64 * 64;
      int64_t need = len + 2 * (int64_t)l.pad + kpad;
      if (fir_src) {
        const int64_t FT = (decimated_len(len, 2) + 127) / 128;
        const int64_t rows = FT + 2;
        if (256 * rows > need) need = 256 * rows;
      }
      const int64_t gran = (int64_t)he / gcd64(he, 256) * 256;  // lcm(he, 256)
      l.pitch = (need + gran - 1) / gran * gran;
      l.t_slots = l.pitch / he;
      const int64_t rows = B * l.t_slots + (kpad + he - 1) / he + 1;
      l.plane = (rows * he + 255) / 256 * 256;
      l.pc = take((size_t)2 * l.plane * 2);
    }
    if (!l.presplit && i > 0) {
      l.y32_pitch = (int64_t)align_up((size_t)len, 8);
      l.y32 = take((size_t)B * l.y32_pitch * sizeof(float));
    }
  }
  // scratch for octaves that run from fp32 (several frame phases): sized for the first such level
  for (int i = 0; i < n_octaves; ++i)
    if (!lv[i].presplit) {
      off += tc_workspace_bytes(B, lv[i].len, lv[i].width, lv[i].hop, lv[i].pad) + 256;
      break;
    }
  *total = off;
  return true;
}

size_t nnab_packed_fir_bytes(int taps, int dec) { return tc_packed_fir_bytes(taps, dec); }
int nnab_pack_fir(const float* fir, int taps, int dec, void* packed, void* stream) {
  if (fir == nullptr || packed == nullptr || taps <= 0 || dec < 1) return NNAB_EINVAL;
  return tc_pack_fir(fir, taps, dec, packed, (cudaStream_t)stream);
}

int nnab_debug_varn_plan(const int32_t* h_k_begin, const int32_t* h_k_end, int n_bins, int width,
                         int want_chunks, int32_t* order, int32_t* groups, int32_t* chunk_begin,
                         int32_t* n_blocks, int32_t* n_chunks) {
  if (order == nullptr || groups == nullptr || chunk_begin == nullptr || n_blocks == nullptr ||
      n_chunks == nullptr || n_bins <= 0 || width <= 0)
    return NNAB_EINVAL;
  return tc_varn_plan_export(h_k_begin, h_k_end, n_bins, width, want_chunks, order, groups,
                             chunk_begin, n_blocks, n_chunks);
}

int nnab_fir_decimate(const float* x, int64_t B, int64_t L, int64_t x_pitch, const float* fir,
                      int taps, int factor, float* y, int64_t Ly, void* stream) {
  if (x == nullptr || fir == nullptr || y == nullptr || B < 0 || L <= 0 || x_pitch < L || taps <= 0 ||
      factor < 1)
    return NNAB_EINVAL;
  const int half = (taps - 1) / 2;
  if (L + 2 * (int64_t)half < taps || Ly != (L + 2 * (int64_t)half - taps) / factor + 1)
    return NNAB_EINVAL;
  int rc = check_arch();
  if (rc) return rc;
  return launch_fir_decimate(x, NNAB_DTYPE_F32, B, L, x_pitch, fir, taps, factor, y, Ly, Ly,
                             (cudaStream_t)stream);
}

int nnab_fir_decimate_adjoint(const float* g, int64_t B, int64_t Ly, int64_t g_pitch,
                              const float* fir, int taps, int factor, float* dx, int64_t L,
                              void* stream) {
  if (g == nullptr || fir == nullptr || dx == nullptr || B < 0 || L <= 0 || Ly <= 0 || g_pitch < Ly ||
      taps <= 0 || factor < 1)
    return NNAB_EINVAL;
  const int half = (taps - 1) / 2;
  if (L + 2 * (int64_t)half < taps || Ly != (L + 2 * (int64_t)half - taps) / factor + 1)
    return NNAB_EINVAL;
  int rc = check_arch();
  if (rc) return rc;
  return launch_fir_decimate_adjoint(g, B, Ly, g_pitch, fir, taps, factor, dx, L, L,
                                     (cudaStream_t)stream);
}

size_t nnab_cqt_pyramid_workspace_bytes(int64_t B, int64_t L, int n_octaves, int early_factor,
                                        int max_width, int hop, int path) {
  size_t n = pyramid_level_bytes(B, L, early_factor);
  if (path != NNAB_PATH_SIMT) {
    // (a) per-octave tensor-core path: split-signal scratch of the largest level
    const int64_t L0 = early_factor > 1 ? decimated_len(L, early_factor) : L;
    n += tc_workspace_bytes(B, L0, max_width, hop, max_width / 2);
    // (b) all-tensor-core pyramid: every level's planes (upper bound with max_width)
    if (n_octaves <= 32) {
      PyrLevel lv[32];
      const size_t full = plan_pyramid(B, L, n_octaves, early_factor, hop, nullptr, max_width,
                                       NNAB_PAD_REFLECT, lv, nullptr) + 1024;
      if (full > n) n = full;
      Lvl2 lv2[32];
      size_t full2 = 0;
      if (early_factor <= 1 &&
          plan_pyramid2(B, L, n_octaves, hop, nullptr, max_width, NNAB_PAD_REFLECT, lv2, &full2)) {
        full2 += 2048;
        if (full2 > n) n = full2;
      }
    }
  }
  return n;
}

static int pyramid_fused2(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch, int n_octaves,
                          const float* const* h_k_real, const float* const* h_k_imag,
                          const void* const* h_packed, const int32_t* h_widths, int n_filters,
                          const float* lowpass, const void* lowpass_packed, int hop, int pad_mode,
                          int n_bins, const float* scale, float scale_all, int out_format,
                          float sqrt_eps, float* out, int64_t T, void* workspace, size_t ws_bytes,
                          cudaStream_t s) {
  if (n_octaves > 32 || B > 65535) return NNAB_EUNSUPPORTED;
  Lvl2 lv[32];
  size_t need = 0;
  if (!plan_pyramid2(B, L, n_octaves, hop, h_widths, 0, pad_mode, lv, &need)) return NNAB_EUNSUPPORTED;
  char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  if (need + 512 > ws_bytes) return NNAB_EUNSUPPORTED;
  for (int i = 0; i < n_octaves; ++i)
    if (frames_of(lv[i].len, lv[i].width, lv[i].hop, lv[i].pad) != T) return NNAB_EINVAL;
  size_t scratch_off = need;
  for (int i = 0; i < n_octaves; ++i)
    if (!lv[i].presplit) {
      scratch_off -= tc_workspace_bytes(B, lv[i].len, lv[i].width, lv[i].hop, lv[i].pad) + 256;
      break;
    }
  char* scratch = ws + scratch_off;
  int rc;
  const size_t scratch_bytes = ws_bytes - 256 - scratch_off;

  // level 0: the caller's waveform -> planes (one pass; writes the whole clip slot, both planes: the
  // octave and FIR kernels run the three-term split whatever the input type)
  if (lv[0].planes) {
    rc = tc_pad_split_ex(x, x_dtype, B, L, x_pitch, lv[0].pad, lv[0].mode, lv[0].pitch, lv[0].plane,
                         ws + lv[0].pc, s);
    if (rc) return rc;
  }
  for (int i = 0; i < n_octaves; ++i) {
    Lvl2& l = lv[i];
    FramedProblem p{};
    p.B = B; p.L = l.len;
    p.w_re = h_k_real[i]; p.w_im = h_k_imag[i]; p.F = n_filters; p.K = l.width; p.hop = l.hop;
    p.pad = l.pad; p.pad_mode = l.mode; p.scale_all = scale_all;
    p.fmt = out_format; p.eps = sqrt_eps; p.power = 1.f; p.out = out; p.T = T;
    p.out_bins = n_bins;
    p.bin_offset = n_bins - n_filters * (i + 1);
    p.scale = scale ? scale + p.bin_offset : nullptr;
    if (l.presplit) {
      p.presplit = ws + l.pc;
      p.presplit_t_slots = l.t_slots;
      p.presplit_plane_stride = l.plane;
      bool done = false;
      if (!done) {
        // resident bank + tall A blocks + frame phases: one fetch per sample and tile
        std::pair<cudaEvent_t, cudaEvent_t> pr;
        const bool timed = prof_begin(s, &pr);
        rc = launch_octave_tc(p, h_packed[i], s);
        if (timed) prof_end(s, pr);
        if (rc == NNAB_OK) done = true;
        else if (rc != NNAB_EUNSUPPORTED) return rc;
      }
      if (!done && (rc = run_framed(p, h_packed[i], nullptr, 0, NNAB_PATH_TCGEN05, s))) return rc;
    } else {
      p.x = (i == 0) ? x : (const void*)(ws + l.y32);
      p.x_pitch = (i == 0) ? x_pitch : l.y32_pitch;
      p.x_dtype = (i == 0) ? x_dtype : NNAB_DTYPE_F32;
      if ((rc = run_framed(p, h_packed[i], scratch, scratch_bytes, NNAB_PATH_TCGEN05, s))) return rc;
    }
    if (i == n_octaves - 1) break;
    // ---- FIR stage: level i -> level i + 1
    Lvl2& d = lv[i + 1];
    DecimParams dec{};
    dec.len_out = d.len;
    if (d.planes) {
      const bool refl = d.mode == NNAB_PAD_REFLECT;
      // what the stage's epilogue never writes: everything outside the samples (+ reflect margins)
      rc = tc_zero_slots(ws + d.pc, B, d.pitch, d.plane, refl ? 0 : d.pad,
                         refl ? d.len + 2 * (int64_t)d.pad : d.pad + d.len, s);
      if (rc) return rc;
      dec.pc = ws + d.pc; dec.pc_plane = d.plane; dec.pc_pitch = d.pitch; dec.pc_off = d.pad;
      dec.pc_reflect = refl ? 1 : 0;
    }
    if (d.y32 != SIZE_MAX) { dec.y32 = (float*)(ws + d.y32); dec.y32_pitch = d.y32_pitch; }
    rc = launch_fir_stage_tc(ws + l.pc, B, l.len, l.pitch, l.plane, l.pad, lowpass_packed, lowpass,
                             FIR_TAPS, dec, s);
    if (rc) return rc;  // (EUNSUPPORTED cannot happen after plan_pyramid2 accepted the shape)
  }
  return NNAB_OK;
}

// All-tensor-core pyramid; returns NNAB_EUNSUPPORTED when the plan cannot be used (the caller
// then takes the per-octave path).
static int pyramid_fused(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch, int n_octaves,
                         const float* const* h_k_real, const float* const* h_k_imag,
                         const void* const* h_packed, const int32_t* h_widths, int n_filters,
                         const void* lowpass_packed, const void* early_packed, int early_factor,
                         int hop, int pad_mode, int n_bins, const float* scale, float scale_all,
                         int out_format, float sqrt_eps, float* out, int64_t T, void* workspace,
                         size_t ws_bytes, cudaStream_t s) {
  if (n_octaves > 32 || B > 65535) return NNAB_EUNSUPPORTED;
  PyrLevel lv[32];
  size_t pf_early = SIZE_MAX;
  const size_t need = plan_pyramid(B, L, n_octaves, early_factor, hop, h_widths, 0, pad_mode, lv,
                                   &pf_early);
  char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  if (need + 256 > ws_bytes) return NNAB_EUNSUPPORTED;
  for (int i = 0; i < n_octaves; ++i) {
    if (lv[i].len <= 0 || lv[i].hop <= 0) return NNAB_EINVAL;
    if (frames_of(lv[i].len, lv[i].width, lv[i].hop, lv[i].pad) != T) return NNAB_EINVAL;
  }
  // scratch region for fp32-driven octaves lives after the planned buffers
  size_t planned = 0;
  {
    PyrLevel tmp[32];
    planned = plan_pyramid(B, L, n_octaves, early_factor, hop, h_widths, 0, pad_mode, tmp, nullptr);
    for (int i = 0; i < n_octaves; ++i)
      if (!tmp[i].presplit) {
        planned -= tc_workspace_bytes(B, tmp[i].len, tmp[i].width, tmp[i].hop, tmp[i].pad);
        break;
      }
  }
  char* scratch = ws + planned;
  const size_t scratch_bytes = ws_bytes - 256 - planned;
  int rc;

  // One FIR stage: planes `src` (level signal, zero margins) -> level `dst`
  auto fir_stage = [&](const void* src, int64_t src_len, int dec, const void* fir_packed,
                       PyrLevel& dst) -> int {
    const int kf = tc_fir_k(FIR_TAPS, dec);
    // parts of the destination buffers the epilogue never writes
    if (dst.pc != SIZE_MAX) {
      const bool refl = dst.mode == NNAB_PAD_REFLECT;
      rc = tc_zero_margins(ws + dst.pc, B, dst.len, dst.width, dst.hop, dst.pad,
                           refl ? 0 : dst.pad, refl ? dst.len + 2 * dst.pad : dst.pad + dst.len, s);
      if (rc) return rc;
    }
    if (dst.pf != SIZE_MAX) {
      rc = tc_zero_margins(ws + dst.pf, B, dst.len, tc_fir_k(FIR_TAPS, 2), 256, FIR_OFF, FIR_OFF,
                           FIR_OFF + dst.len, s);
      if (rc) return rc;
    }
    FramedProblem p{};
    p.x = nullptr; p.B = B; p.L = src_len; p.x_pitch = 0;
    p.w_re = nullptr; p.w_im = nullptr; p.F = 64; p.K = kf; p.hop = 128 * dec;
    p.pad = FIR_OFF; p.pad_mode = NNAB_PAD_CONSTANT; p.scale = nullptr; p.scale_all = 1.f;
    p.fmt = FMT_DECIM; p.eps = 0.f; p.power = 1.f; p.out = nullptr;
    p.T = (dst.len + 127) / 128;
    p.out_bins = 64; p.bin_offset = 0;
    p.presplit = src;
    p.dec.pc = dst.pc != SIZE_MAX ? ws + dst.pc : nullptr;
    p.dec.pc_plane = dst.pc_plane; p.dec.pc_pitch = dst.pc_pitch; p.dec.pc_off = dst.pad;
    p.dec.pc_reflect = dst.mode == NNAB_PAD_REFLECT ? 1 : 0;
    p.dec.pf = dst.pf != SIZE_MAX ? ws + dst.pf : nullptr;
    p.dec.pf_plane = dst.pf_plane; p.dec.pf_pitch = dst.pf_pitch;
    p.dec.y32 = dst.y32 != SIZE_MAX ? (float*)(ws + dst.y32) : nullptr;
    p.dec.y32_pitch = dst.y32_pitch;
    p.dec.len_out = dst.len;
    return run_framed(p, fir_packed, nullptr, 0, NNAB_PATH_TCGEN05, s);
  };

  // ---- level 0 ------------------------------------------------------------------------
  const void* x0 = x;          // level-0 signal when available (x0_dtype)
  int64_t x0_pitch = x_pitch;
  int x0_dtype = x_dtype;
  if (early_factor > 1) {
    rc = tc_pad_split(x, x_dtype, B, L, x_pitch, tc_fir_k(FIR_TAPS, early_factor), 128 * early_factor,
                      FIR_OFF, NNAB_PAD_CONSTANT, ws + pf_early, s);
    if (rc) return rc;
    if ((rc = fir_stage(ws + pf_early, L, early_factor, early_packed, lv[0]))) return rc;
    x0 = lv[0].y32 != SIZE_MAX ? (const void*)(ws + lv[0].y32) : nullptr;
    x0_pitch = lv[0].y32_pitch;
    x0_dtype = NNAB_DTYPE_F32;
  } else {
    if (lv[0].pc != SIZE_MAX && lv[0].pf != SIZE_MAX) {
      // one pass over x: reflect-padded copy for the octave CQT + zero-margin copy for the FIR
      rc = tc_pad_split2(x, x_dtype, B, L, x_pitch, lv[0].width, lv[0].hop, lv[0].pad, lv[0].mode,
                         ws + lv[0].pc, tc_fir_k(FIR_TAPS, 2), 256, FIR_OFF, NNAB_PAD_CONSTANT,
                         ws + lv[0].pf, s);
      if (rc) return rc;
    } else if (lv[0].pc != SIZE_MAX) {
      rc = tc_pad_split(x, x_dtype, B, L, x_pitch, lv[0].width, lv[0].hop, lv[0].pad, lv[0].mode,
                        ws + lv[0].pc, s);
      if (rc) return rc;
    } else if (lv[0].pf != SIZE_MAX) {
      rc = tc_pad_split(x, x_dtype, B, L, x_pitch, tc_fir_k(FIR_TAPS, 2), 256, FIR_OFF, NNAB_PAD_CONSTANT,
                        ws + lv[0].pf, s);
      if (rc) return rc;
    }
  }

  // ---- octaves --------------------------------------------------------------------------
  for (int i = 0; i < n_octaves; ++i) {
    PyrLevel& l = lv[i];
    FramedProblem p{};
    p.B = B; p.L = l.len;
    p.w_re = h_k_real[i]; p.w_im = h_k_imag[i]; p.F = n_filters; p.K = l.width; p.hop = l.hop;
    p.pad = l.pad; p.pad_mode = l.mode; p.scale_all = scale_all;
    p.fmt = out_format; p.eps = sqrt_eps; p.power = 1.f; p.out = out; p.T = T;
    p.out_bins = n_bins;
    p.bin_offset = n_bins - n_filters * (i + 1);
    p.scale = scale ? scale + p.bin_offset : nullptr;
    if (l.presplit) {
      p.x = nullptr; p.x_pitch = 0; p.presplit = ws + l.pc;
      if ((rc = run_framed(p, h_packed[i], nullptr, 0, NNAB_PATH_TCGEN05, s))) return rc;
    } else {
      const void* src = (i == 0) ? x0 : (const void*)(ws + l.y32);
      const int64_t pitch = (i == 0) ? x0_pitch : l.y32_pitch;
      if (src == nullptr) return NNAB_EINVAL;
      p.x = src; p.x_pitch = pitch; p.presplit = nullptr;
      p.x_dtype = (i == 0) ? x0_dtype : NNAB_DTYPE_F32;
      if ((rc = run_framed(p, h_packed[i], scratch, scratch_bytes, NNAB_PATH_TCGEN05, s))) return rc;
    }
    if (i < n_octaves - 1)
      if ((rc = fir_stage(ws + l.pf, l.len, 2, lowpass_packed, lv[i + 1]))) return rc;
  }
  return NNAB_OK;
}

int nnab_cqt_pyramid_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch, int n_octaves,
                             const float* const* h_k_real, const float* const* h_k_imag,
                             const void* const* h_packed, const int32_t* h_widths, int n_filters,
                             const float* lowpass, const void* lowpass_packed,
                             const float* early_filter, const void* early_packed,
                             int early_factor, int hop, int pad_mode, int n_bins,
                             const float* scale, float scale_all, int out_format, float sqrt_eps,
                             float* out, int64_t T, void* workspace, size_t ws_bytes, int path,
                             void* stream) {
  return nnab_cqt_pyramid_forward_ex(x, B, L, x_pitch, n_octaves, h_k_real, h_k_imag, h_packed, h_widths,
                                     n_filters, lowpass, lowpass_packed, early_filter, early_packed,
                                     early_factor, hop, pad_mode, n_bins, scale, scale_all, out_format,
                                     sqrt_eps, out, T, workspace, ws_bytes, path, stream, NNAB_DTYPE_F32);
}

int nnab_cqt_pyramid_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch, int n_octaves,
                                const float* const* h_k_real, const float* const* h_k_imag,
                                const void* const* h_packed, const int32_t* h_widths, int n_filters,
                                const float* lowpass, const void* lowpass_packed,
                                const float* early_filter, const void* early_packed,
                                int early_factor, int hop, int pad_mode, int n_bins,
                                const float* scale, float scale_all, int out_format, float sqrt_eps,
                                float* out, int64_t T, void* workspace, size_t ws_bytes, int path,
                                void* stream, int x_dtype) {
  if (!valid_x_dtype(x_dtype)) return NNAB_EINVAL;
  if (x == nullptr || out == nullptr || h_k_real == nullptr || h_k_imag == nullptr ||
      h_widths == nullptr || lowpass == nullptr || B < 0 || L <= 0 || x_pitch < L ||
      n_octaves <= 0 || n_filters <= 0 || hop <= 0 || n_bins <= 0 || early_factor < 1)
    return NNAB_EINVAL;
  if (early_factor > 1 && early_filter == nullptr) return NNAB_EINVAL;
  if (out_format != NNAB_FMT_MAGNITUDE && out_format != NNAB_FMT_COMPLEX &&
      out_format != NNAB_FMT_PHASE_UNIT)
    return NNAB_EINVAL;
  if (pad_mode != NNAB_PAD_REFLECT && pad_mode != NNAB_PAD_CONSTANT) return NNAB_EINVAL;
  int rc = check_arch();
  if (rc) return rc;
  int max_width = 0;
  for (int i = 0; i < n_octaves; ++i) max_width = h_widths[i] > max_width ? h_widths[i] : max_width;
  const size_t need =
      nnab_cqt_pyramid_workspace_bytes(B, L, n_octaves, early_factor, max_width, hop, path);
  if (need > 0 && (workspace == nullptr || ws_bytes < need)) return NNAB_EWORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;

  // ---- all-tensor-core pyramid when every packed operand is available -------------------
  bool all_packed = (path != NNAB_PATH_SIMT) && h_packed != nullptr && lowpass_packed != nullptr &&
                    (early_factor <= 1 || early_packed != nullptr);
  for (int i = 0; all_packed && i < n_octaves; ++i) all_packed = h_packed[i] != nullptr;
  if (all_packed && getenv("NNAB_PYRAMID_UNFUSED") == nullptr && early_factor <= 1 &&
      !(getenv("NNAB_PYRAMID2") != nullptr && atoi(getenv("NNAB_PYRAMID2")) == 0)) {
    rc = pyramid_fused2(x, x_dtype, B, L, x_pitch, n_octaves, h_k_real, h_k_imag, h_packed, h_widths, n_filters,
                        lowpass, lowpass_packed, hop, pad_mode, n_bins, scale, scale_all, out_format,
                        sqrt_eps, out, T, workspace, ws_bytes, s);
    if (rc != NNAB_EUNSUPPORTED) return rc;
  }
  if (all_packed && getenv("NNAB_PYRAMID_UNFUSED") == nullptr) {
    rc = pyramid_fused(x, x_dtype, B, L, x_pitch, n_octaves, h_k_real, h_k_imag, h_packed, h_widths,
                       n_filters, lowpass_packed, early_packed, early_factor, hop, pad_mode, n_bins,
                       scale, scale_all, out_format, sqrt_eps, out, T, workspace, ws_bytes, s);
    if (rc != NNAB_EUNSUPPORTED) return rc;
  }

  // ---- per-octave path: CUDA-core FIR stages, octaves on either kernel family -----------
  const size_t level_bytes = pyramid_level_bytes(B, L, early_factor);
  char* tc_ws = (char*)workspace + level_bytes;
  const size_t tc_ws_bytes = ws_bytes - level_bytes;
  char* wsp = (char*)workspace;
  const void* cur = x;  // level signal: x (x_dtype) at level 0, fp32 below
  int cur_dtype = x_dtype;
  int64_t cur_len = L, cur_pitch = x_pitch;
  if (early_factor > 1) {
    const int64_t L0 = decimated_len(L, early_factor);
    const int64_t pitch0 = (int64_t)align_up((size_t)L0, 4);
    float* e = (float*)wsp;
    wsp += align_up((size_t)B * pitch0 * sizeof(float), 256);
    if ((rc = launch_fir_decimate(x, x_dtype, B, L, x_pitch, early_filter, 256, early_factor, e, L0,
                                  pitch0, s)))
      return rc;
    cur = e; cur_dtype = NNAB_DTYPE_F32; cur_len = L0; cur_pitch = pitch0;
  }
  const int64_t half_pitch = (int64_t)align_up((size_t)(cur_len / 2 + 1), 4);
  float* pingpong[2];
  pingpong[0] = (float*)wsp;
  pingpong[1] = (float*)(wsp + align_up((size_t)B * half_pitch * sizeof(float), 256));

  int cur_hop = hop;
  for (int i = 0; i < n_octaves; ++i) {
    if (i > 0) {
      const int64_t nl = decimated_len(cur_len, 2);
      float* dst = pingpong[i & 1];
      if ((rc = launch_fir_decimate(cur, cur_dtype, B, cur_len, cur_pitch, lowpass, 256, 2, dst, nl,
                                    half_pitch, s)))
        return rc;
      cur = dst; cur_dtype = NNAB_DTYPE_F32; cur_len = nl; cur_pitch = half_pitch;
      cur_hop /= 2;
    }
    if (cur_hop <= 0 || cur_len <= 0) return NNAB_EINVAL;
    const int width = h_widths[i];
    const int pad = width / 2;
    // get_cqt_complex: reflect padding that torch would reject falls back to zero padding.
    int mode = pad_mode;
    if (mode == NNAB_PAD_REFLECT && pad >= cur_len) mode = NNAB_PAD_CONSTANT;
    if (frames_of(cur_len, width, cur_hop, pad) != T) return NNAB_EINVAL;
    FramedProblem p{};
    p.x = cur; p.B = B; p.L = cur_len; p.x_pitch = cur_pitch; p.x_dtype = cur_dtype;
    p.w_re = h_k_real[i]; p.w_im = h_k_imag[i]; p.F = n_filters; p.K = width; p.hop = cur_hop;
    p.pad = pad; p.pad_mode = mode; p.scale = nullptr; p.scale_all = scale_all;
    p.fmt = out_format; p.eps = sqrt_eps; p.power = 1.f; p.out = out; p.T = T;
    p.out_bins = n_bins;
    // octave i (0 = top) lands n_filters*(i+1) rows below the top of the output
    p.bin_offset = n_bins - n_filters * (i + 1);
    // per-bin scale is indexed by OUTPUT row: shift the pointer by the same offset
    p.scale = scale ? scale + p.bin_offset : nullptr;
    const void* pk = (h_packed != nullptr) ? h_packed[i] : nullptr;
    if (pk != nullptr && path != NNAB_PATH_SIMT && tc_supported(p) &&
        tc_ws_bytes >= tc_workspace_bytes(B, cur_len, width, cur_hop, pad)) {
      if ((rc = run_framed(p, pk, tc_ws, tc_ws_bytes, NNAB_PATH_TCGEN05, s))) return rc;
    } else {
      if (path == NNAB_PATH_TCGEN05) return NNAB_EALIGN;
      if ((rc = run_framed(p, nullptr, nullptr, 0, NNAB_PATH_SIMT, s))) return rc;
    }
  }
  return NNAB_OK;
}

// ----------------------------------------------------------------- inverse STFT ----
static __global__ void istft_scale_kernel(const float* __restrict__ window, float inv_n, int n,
                                          float* __restrict__ scale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) scale[i] = window[i] * inv_n;
}

size_t nnab_packed_istft_bytes(int n_fft, int f_in) { return tc_packed_istft_bytes(n_fft, f_in); }

int nnab_pack_istft_basis(const float* kernel_cos, const float* kernel_sin, int n_fft, int f_in,
                          int onesided, void* packed, void* stream) {
  if (kernel_cos == nullptr || kernel_sin == nullptr || packed == nullptr || n_fft <= 0 ||
      f_in <= 0 || f_in > n_fft)
    return NNAB_EINVAL;
  return tc_pack_istft(kernel_cos, kernel_sin, n_fft, f_in, onesided, packed, (cudaStream_t)stream);
}

static size_t istft_ola_bytes(int64_t B, int64_t T, int n_fft, int hop, int64_t* pitch) {
  const int64_t len = n_fft + (int64_t)hop * (T - 1);
  const int64_t p = (int64_t)align_up((size_t)len, 8);
  if (pitch) *pitch = p;
  return align_up((size_t)B * p * sizeof(float), 256);
}

size_t nnab_istft_workspace_bytes(int64_t B, int f_in, int64_t T, int n_fft, int hop) {
  return align_up(tc_istft_planes_bytes(B, T, f_in), 256) + istft_ola_bytes(B, T, n_fft, hop, nullptr) +
         align_up((size_t)n_fft * sizeof(float), 256) + 256;
}

int nnab_istft_forward(const float* X, int64_t B, int f_in, int64_t T, const void* packed,
                       const float* window, int n_fft, int hop, int center, int64_t length,
                       float* out, int64_t out_len, void* workspace, size_t ws_bytes,
                       void* stream) {
  if (X == nullptr || packed == nullptr || window == nullptr || out == nullptr || B < 0 ||
      f_in <= 0 || T <= 0 || n_fft <= 0 || hop <= 0)
    return NNAB_EINVAL;
  int rc = check_arch();
  if (rc) return rc;
  const size_t need = nnab_istft_workspace_bytes(B, f_in, T, n_fft, hop);
  if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  const int64_t ola_len = n_fft + (int64_t)hop * (T - 1);
  const int pad = n_fft / 2;
  const int64_t offset = center ? pad : 0;
  int64_t want = length >= 0 ? length : (center ? ola_len - 2 * pad : ola_len);
  if (offset + want > ola_len) want = ola_len - offset;  // slicing past the end just truncates
  if (want < 0) want = 0;
  if (out_len != want) return NNAB_EINVAL;
  if (B == 0 || want == 0) return NNAB_OK;
  cudaStream_t s = (cudaStream_t)stream;

  char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  void* planes = ws;
  int64_t ola_pitch = 0;
  const size_t planes_b = align_up(tc_istft_planes_bytes(B, T, f_in), 256);
  const size_t ola_b = istft_ola_bytes(B, T, n_fft, hop, &ola_pitch);
  float* ola = (float*)(ws + planes_b);
  float* scale = (float*)(ws + planes_b + ola_b);

  if ((rc = tc_istft_prep(X, B, f_in, T, planes, s))) return rc;
  NNAB_CUDA_TRY(cudaMemsetAsync(ola, 0, (size_t)B * ola_pitch * sizeof(float), s));
  istft_scale_kernel<<<(n_fft + 255) / 256, 256, 0, s>>>(window, 1.0f / (float)n_fft, n_fft, scale);
  NNAB_LAUNCH_CHECK();

  const int kpad = tc_istft_k(f_in);
  FramedProblem p{};
  p.x = nullptr; p.B = B; p.L = T * (int64_t)kpad; p.x_pitch = 0;
  p.F = n_fft; p.K = kpad; p.hop = kpad; p.pad = 0; p.pad_mode = NNAB_PAD_CONSTANT;
  p.scale = scale; p.scale_all = 1.f; p.fmt = FMT_OLA; p.eps = 0.f; p.power = 1.f;
  p.out = ola; p.T = T; p.out_bins = n_fft; p.bin_offset = 0;
  p.presplit = planes;
  p.ola_pitch = ola_pitch; p.ola_hop = hop;
  if ((rc = run_framed(p, packed, nullptr, 0, NNAB_PATH_TCGEN05, s))) return rc;
  return tc_istft_finalize(ola, ola_pitch, B, window, n_fft, hop, T, offset, out, want, s);
}

// ------------------------------------------------------------- input gradient ----
size_t nnab_packed_adjoint_bytes(int K, int F) { return tc_packed_istft_bytes(K, F); }

int nnab_pack_adjoint_basis(const float* w_re, const float* w_im, int F, int K, void* packed,
                            void* stream) {
  if (w_re == nullptr || w_im == nullptr || packed == nullptr || F <= 0 || K <= 0) return NNAB_EINVAL;
  return tc_pack_istft(w_re, w_im, K, F, 0, packed, (cudaStream_t)stream, /*transposed=*/1);
}

size_t nnab_framed_backward_input_workspace_bytes(int64_t B, int64_t L, int K, int F, int hop,
                                                  int center) {
  const int pad = center ? K / 2 : 0;
  const int64_t T = frames_of(L, K, hop, pad);
  const int64_t pitch = (int64_t)align_up((size_t)(L + 2 * (int64_t)pad + K), 8);
  return align_up(tc_istft_planes_bytes(B, T, F), 256) +
         align_up((size_t)B * pitch * sizeof(float), 256) + 256;
}

int nnab_framed_backward_input(const float* g, int64_t B, int F, int64_t T, const void* packed_adj,
                               int K, int hop, int center, int pad_mode, float* dx, int64_t L,
                               void* workspace, size_t ws_bytes, void* stream) {
  if (g == nullptr || packed_adj == nullptr || dx == nullptr || B < 0 || F <= 0 || K <= 0 ||
      hop <= 0 || L <= 0)
    return NNAB_EINVAL;
  const int pad = center ? K / 2 : 0;
  if (T != frames_of(L, K, hop, pad) || T <= 0) return NNAB_EINVAL;
  int rc = check_arch();
  if (rc) return rc;
  const size_t need = nnab_framed_backward_input_workspace_bytes(B, L, K, F, hop, center);
  if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  if (B == 0) return NNAB_OK;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  void* planes = ws;
  const size_t planes_b = align_up(tc_istft_planes_bytes(B, T, F), 256);
  const int64_t gp_len = L + 2 * (int64_t)pad;
  const int64_t pitch = (int64_t)align_up((size_t)(gp_len + K), 8);
  float* gp = (float*)(ws + planes_b);

  if ((rc = tc_istft_prep(g, B, F, T, planes, s))) return rc;
  NNAB_CUDA_TRY(cudaMemsetAsync(gp, 0, (size_t)B * pitch * sizeof(float), s));
  const int kpad = tc_istft_k(F);
  FramedProblem p{};
  p.x = nullptr; p.B = B; p.L = T * (int64_t)kpad; p.x_pitch = 0;
  p.F = K; p.K = kpad; p.hop = kpad; p.pad = 0; p.pad_mode = NNAB_PAD_CONSTANT;
  p.scale = nullptr; p.scale_all = 1.f; p.fmt = FMT_OLA; p.eps = 0.f; p.power = 1.f;
  p.out = gp; p.T = T; p.out_bins = K; p.bin_offset = 0;
  p.presplit = planes;
  p.ola_pitch = pitch; p.ola_hop = hop;
  if ((rc = run_framed(p, packed_adj, nullptr, 0, NNAB_PATH_TCGEN05, s))) return rc;
  return tc_unpad_adjoint(gp, pitch, gp_len, B, pad, pad_mode, L, dx, s);
}

size_t nnab_framed_backward_weight_workspace_bytes(int64_t B, int64_t L, int K, int F, int hop,
                                                   int center) {
  const int pad = center ? K / 2 : 0;
  const int64_t T = frames_of(L, K, hop, pad);
  return align_up(tc_dw_grad_planes_bytes(B, T, F), 256) + align_up(tc_dw_frames_bytes(B, T, K), 256) +
         512;
}

int nnab_framed_backward_weight(const float* g, const float* x, int64_t B, int64_t L,
                                int64_t x_pitch, int F, int64_t T, int K, int hop, int center,
                                int pad_mode, float* dw, void* workspace, size_t ws_bytes,
                                void* stream) {
  if (g == nullptr || x == nullptr || dw == nullptr || B <= 0 || L <= 0 || x_pitch < L || F <= 0 ||
      K <= 0 || hop <= 0)
    return NNAB_EINVAL;
  const int pad = center ? K / 2 : 0;
  if (T != frames_of(L, K, hop, pad) || T <= 0) return NNAB_EINVAL;
  int rc = check_arch();
  if (rc) return rc;
  const size_t need = nnab_framed_backward_weight_workspace_bytes(B, L, K, F, hop, center);
  if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  void* gplanes = ws;
  void* frames = ws + align_up(tc_dw_grad_planes_bytes(B, T, F), 256);
  const int64_t gpad = tc_dw_gpad(B, T);
  if (gpad >= (1ll << 31)) return NNAB_EUNSUPPORTED;

  if ((rc = tc_dw_prep_grad(g, B, F, T, gplanes, s))) return rc;
  if ((rc = tc_dw_prep_frames(x, B, L, x_pitch, K, hop, pad, pad_mode, T, frames, s))) return rc;
  NNAB_CUDA_TRY(cudaMemsetAsync(dw, 0, (size_t)2 * F * K * sizeof(float), s));

  FramedProblem p{};
  p.x = nullptr; p.B = 1; p.L = (int64_t)2 * F * gpad; p.x_pitch = 0;
  p.F = K; p.K = (int)gpad; p.hop = (int)gpad; p.pad = 0; p.pad_mode = NNAB_PAD_CONSTANT;
  p.scale = nullptr; p.scale_all = 1.f; p.fmt = FMT_OLA; p.eps = 0.f; p.power = 1.f;
  p.out = dw; p.T = 2 * F; p.out_bins = K; p.bin_offset = 0;
  p.presplit = gplanes;
  p.ola_pitch = 0; p.ola_hop = K;        // row m of dW starts at m * K
  p.k_splits_hint = (int)((gpad / 64 + 63) / 64);  // <= 64 k-blocks per accumulator chunk
  if (p.k_splits_hint > 64) p.k_splits_hint = 64;
  return run_framed(p, frames, nullptr, 0, NNAB_PATH_TCGEN05, s);
}

}  // extern "C"
