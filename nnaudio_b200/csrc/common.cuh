// Shared declarations for libnnab.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "nnab.h"

namespace nnab {

// ---- error plumbing -------------------------------------------------------
void set_cuda_error(const char* where, cudaError_t e);
void set_error_text(const char* text);
void count_launch();
void count_balanced_launch();
int sm_reserve();
// tensor-pipe accounting for bench.py: MMA flops a tensor-core launch EXECUTES (all split terms,
// tile padding and structural zeros included); summed while nnab_profile_enable(1)
void add_exec_flops(double flops);

#define NNAB_CUDA_TRY(expr)                         \
  do {                                              \
    cudaError_t _e = (expr);                        \
    if (_e != cudaSuccess) {                        \
      ::nnab::set_cuda_error(#expr, _e);            \
      return NNAB_ECUDA;                            \
    }                                               \
  } while (0)

#define NNAB_LAUNCH_CHECK()                         \
  do {                                              \
    ::nnab::count_launch();                         \
    cudaError_t _e = cudaGetLastError();            \
    if (_e != cudaSuccess) {                        \
      ::nnab::set_cuda_error("kernel launch", _e);  \
      return NNAB_ECUDA;                            \
    }                                               \
  } while (0)

// ---- waveform element types (nnab_dtype) ----------------------------------
// Every bf16 / fp16 value is exactly representable in fp32, so a kernel that reads 16-bit samples and
// converts them computes what it computes on the fp32 copy of the same tensor.
inline bool valid_x_dtype(int x_dtype) {
  return x_dtype == NNAB_DTYPE_F32 || x_dtype == NNAB_DTYPE_BF16 || x_dtype == NNAB_DTYPE_F16;
}

__device__ __forceinline__ float ldg_sample(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg_sample(const __nv_bfloat16* p) {
  return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}
__device__ __forceinline__ float ldg_sample(const __half* p) {
  return __half2float(__ushort_as_half(__ldg(reinterpret_cast<const unsigned short*>(p))));
}
// eight consecutive 16-bit samples of one 16-byte word, converted to fp32
__device__ __forceinline__ void unpack8(uint4 w, const __nv_bfloat16*, float* v) {
  const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    v[2 * e] = __uint_as_float(u[e] << 16);
    v[2 * e + 1] = __uint_as_float(u[e] & 0xFFFF0000u);
  }
}
__device__ __forceinline__ void unpack8(uint4 w, const __half*, float* v) {
  const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    v[2 * e] = __half2float(__ushort_as_half((unsigned short)(u[e] & 0xFFFFu)));
    v[2 * e + 1] = __half2float(__ushort_as_half((unsigned short)(u[e] >> 16)));
  }
}

// ---- problem description shared by the SIMT and tcgen05 framed kernels ----
// One "framed complex contraction":
//   re[b,f,t] = sum_k xpad[b, t*hop + k] * w_re[f,k]
//   im[b,f,t] = -sum_k xpad[b, t*hop + k] * w_im[f,k]
// followed by a per-bin scale and one of the output formats of nnab.h (or the
// internal POWER format used by the filterbank ops).
constexpr int FMT_POWER = 100;  // internal: (sqrt(re^2+im^2+eps)) ** power -> (B,F,T)
constexpr int FMT_FBANK = 101;  // internal (tcgen05 only): power -> banded filterbank -> (B,n_fb,T)
constexpr int FMT_DECIM = 102;  // internal (tcgen05 only): FIR decimator stage of the CQT pyramid
constexpr int FMT_RAW = 103;    // internal (tcgen05 only): split-K partial sums -> raw (re, im) scratch
constexpr int FMT_OLA = 104;    // internal (tcgen05 only): inverse STFT frames -> overlap-add buffer
constexpr int FMT_PLANES = 105;   // internal (block-partial kernel only): power spectrum -> bf16 hi/lo operand
                                  //   planes of the dense-filterbank GEMM (`out` = plane base, see planes_*)
constexpr int FMT_REALPAIR = 106; // internal (dense tcgen05 kernel only): two real outputs per complex column
                                  //   pair: re -> row f, im -> row f + F of a real (B, out_bins, T) tensor

// FMT_DECIM epilogue target: the NEXT pyramid level, written as bf16 hi/lo planes in
// the layout the tensor-core kernels read (sample m of clip b at b*pitch + off + m).
//   pc: input of the level's octave CQT — reflect (or zero) margins of `pc_off` samples
//   pf: input of the level's own FIR stage — zero margins, samples at offset 128
//   y32: optional fp32 copy (levels whose hop needs several frame phases)
struct DecimParams {
  void* pc; int64_t pc_plane, pc_pitch; int pc_off, pc_reflect;
  void* pf; int64_t pf_plane, pf_pitch;
  float* y32; int64_t y32_pitch;
  int64_t len_out;  // valid samples per clip of the next level
};

// Banded filterbank table: the (at most two) non-zero weights of every FFT bin.
struct FbEntry {
  int j0, j1;    // filter rows (-1 = none)
  float w0, w1;
};

// Static action list of the banded-filterbank epilogue (block-partial kernel): what the two running
// filter sums of a row do at FFT bin k -- the control flow depends on k only, so it is resolved once
// per filterbank instead of per (row, bin).  Before accumulating bin k: a slot whose flush id is
// >= 0 adds its sum to that filter's output and restarts from zero; then slot a += wa * P[k],
// slot b += wb * P[k].  cur_a / cur_b = filters the slots hold after bin k (flushed at a range end).
struct FbStep {
  float wa, wb;
  short flush_a, flush_b;
  short cur_a, cur_b;
};
static_assert(sizeof(FbStep) == 16, "one 128-bit load per bin");
constexpr int FB_STEP_PAD = 160;  // entries past F (a tile's last chunk may overrun the last bin)
// epilogue warps per TMEM lane quarter of the fused-filterbank block kernel: each covers a contiguous
// range of a tile's 8-column chunks, [n_chunks * part / PARTS, n_chunks * (part + 1) / PARTS)
// (3 measured 7 % faster at cfg2 -- 0.197 vs 0.211 ms -- but then a 53-bin mel filter spans three
// ranges, its three atomic partial sums no longer commute and results differ run to run: 2 it is.)
constexpr int FB_EPI_PARTS = 2;

struct FramedProblem {
  const void* x;       // (B, L) rows, pitch x_pitch (elements of x_dtype)
  int64_t B, L, x_pitch;
  int x_dtype;         // NNAB_DTYPE_* of x (0 = fp32 in a zero-initialised problem)
  const float* w_re;   // (F, K)
  const float* w_im;   // (F, K)
  int F, K, hop;
  int pad;             // samples of centre padding on each side (0 if !center)
  int pad_mode;        // NNAB_PAD_*
  const float* scale;  // per-bin or nullptr
  float scale_all;
  int fmt;
  float eps;
  float power;         // FMT_POWER only
  float* out;
  int64_t T;
  int out_bins;        // rows of the output tensor (>= bins written)
  int bin_offset;      // output row of bin 0 (may be negative: rows < 0 dropped)
  const int32_t* h_k_begin;  // host, per-bin support or nullptr
  const int32_t* h_k_end;
  const FbEntry* fb_table;   // FMT_FBANK: device table [F]; out is (B, n_fb, T), pre-zeroed
  const FbStep* fb_steps;    // FMT_FBANK, block-partial kernel: [F + FB_STEP_PAD] (nullptr: MelRun path)
  int fb_nb_mask;            // bit i: tile width nb = 32 + 8 i gives <= 2 partial sums per filter
  int n_fb;
  float* raw;                // tcgen05 split-K scratch: 2 planes (re, im) of B*F*T floats, or nullptr
  const void* presplit;      // tcgen05: already padded + split signal planes (skip pad_split)
  int64_t presplit_t_slots;  // > 0: frames per clip slot of the pre-split planes (else derived)
  int64_t presplit_plane_stride;  // elements per plane when presplit_t_slots > 0
  DecimParams dec;           // FMT_DECIM
  int64_t ola_pitch;         // FMT_OLA: out = overlap-add buffer (B, ola_pitch); scale = window/n_fft
  int ola_hop;
  int k_splits_hint;         // FMT_OLA only (its atomics already accumulate): cut K into chunks
  int64_t planes_stride;     // FMT_PLANES: elements between the hi and the lo plane
  int planes_pitch;          // FMT_PLANES: elements per frame row (multiple of 64)
};

// bf16 input has a zero lo plane: the tensor-core kernels skip its TMA loads and the x_lo * w_hi
// MMA (two bf16 terms instead of three).  Only for a signal the launcher splits itself from x.
inline bool two_term(const FramedProblem& p) {
  return p.x_dtype == NNAB_DTYPE_BF16 && p.presplit == nullptr && p.x != nullptr;
}

int launch_framed_simt(const FramedProblem& p, cudaStream_t stream);

// tcgen05 path (tc_kernels.cu)
bool tc_supported(const FramedProblem& p);
size_t tc_workspace_bytes(int64_t B, int64_t L, int K, int hop, int pad);
int launch_framed_tc(const FramedProblem& p, const void* packed, void* workspace,
                     size_t ws_bytes, cudaStream_t stream);
size_t tc_packed_bytes(int F, int K);
int tc_pack_basis(const float* w_re, const float* w_im, int F, int K, void* packed,
                  cudaStream_t stream);
int tc_tile_n(int F);
int tc_pack_basis_layout(const float* w_re, const float* w_im, int F, int K, int layout, void* packed,
                         cudaStream_t stream);
// split-signal geometry / helpers for callers that manage the planes themselves (pyramid)
void tc_split_geometry(int64_t B, int64_t L, int K, int hop, int pad, int64_t* t_slots,
                       int64_t* plane_stride, int* hop_eff);
// x_dtype: NNAB_DTYPE_* of x.  hi_only (bf16 input only): write the hi plane alone -- for the
// two-term kernels, which never read the lo plane.
int tc_pad_split(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch, int K, int hop,
                 int pad, int pad_mode, void* planes, cudaStream_t stream, bool hi_only = false);
int tc_pad_split_ex(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch, int pad,
                    int pad_mode, int64_t clip_pitch, int64_t plane_stride, void* planes,
                    cudaStream_t stream);
int tc_zero_slots(void* planes, int64_t B, int64_t clip_pitch, int64_t plane_stride, int64_t keep_lo,
                  int64_t keep_hi, cudaStream_t stream);
int tc_pad_split2(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch,
                  int K_a, int hop_a, int pad_a, int mode_a, void* planes_a,
                  int K_b, int hop_b, int pad_b, int mode_b, void* planes_b, cudaStream_t stream);
int tc_zero_margins(void* planes, int64_t B, int64_t L, int K, int hop, int pad, int64_t keep_lo,
                    int64_t keep_hi, cudaStream_t stream);
// inverse STFT pieces (tc_kernels.cu)
int tc_istft_k(int f_in);
int tc_istft_bn(int n_fft);
size_t tc_packed_istft_bytes(int n_fft, int f_in);
int tc_pack_istft(const float* kc, const float* ks, int n_fft, int f_in, int onesided, void* packed,
                  cudaStream_t stream, int transposed = 0);
// weight-gradient operands (tc_kernels.cu)
int64_t tc_dw_gpad(int64_t B, int64_t T);
size_t tc_dw_grad_planes_bytes(int64_t B, int64_t T, int F);
size_t tc_dw_frames_bytes(int64_t B, int64_t T, int K);
int tc_dw_prep_grad(const float* g, int64_t B, int F, int64_t T, void* planes, cudaStream_t stream);
int tc_dw_prep_frames(const float* x, int64_t B, int64_t L, int64_t x_pitch, int K, int hop, int pad,
                      int pad_mode, int64_t T, void* packed, cudaStream_t stream);
int tc_unpad_adjoint(const float* gp, int64_t gp_pitch, int64_t gp_len, int64_t B, int pad,
                     int pad_mode, int64_t L, float* dx, cudaStream_t stream);
size_t tc_istft_planes_bytes(int64_t B, int64_t T, int f_in);
int tc_istft_prep(const float* X, int64_t B, int f_in, int64_t T, void* planes, cudaStream_t stream);
int tc_istft_finalize(const float* ola, int64_t ola_pitch, int64_t B, const float* window,
                      int n_fft, int hop, int64_t T, int64_t offset, float* out, int64_t out_len,
                      cudaStream_t stream);
size_t tc_splitk_scratch_bytes(int64_t B, int F, int64_t T, int K);
// block-partial kernel (tcb_kernels.cu): default N-tile geometry for F bins (nb packed columns per tile,
// nb - 2 new bins each) -- the column layout of the FMT_PLANES operand planes
void tc_block_tile_geometry(int F, int* nb, int* n_tiles);
bool tc_block_shape_ok(int n_fft, int hop);
size_t tc_packed_fir_bytes(int taps, int dec);
int tc_fir_k(int taps, int dec);
int tc_pack_fir(const float* fir, int taps, int dec, void* packed, cudaStream_t stream);
int launch_fb_table(const float* fb, int n_fb, int F, FbEntry* table, int* d_max_nnz,
                    cudaStream_t stream);
// FbEntry[F] -> FbStep[F + FB_STEP_PAD]; d_meta[0] = widest filter support (bins), d_meta[1] = bit mask
// of the tile widths nb = 32 + 8 i under which every filter gets <= 2 partial sums
int launch_fb_steps(const FbEntry* table, int n_fb, int F, FbStep* steps, int* d_meta,
                    cudaStream_t stream);

// filterbank / MFCC tail / FIR decimation (simt_kernels.cu)
int launch_filterbank(const float* P, const float* fb, int64_t B, int F, int64_t T, int n_fb,
                      float* out, cudaStream_t stream);
int launch_fb_tile_bank(const float* fb, int n_fb, int F, int nb, int n_tiles, int kp, int fh, float* w_re,
                        float* w_im, cudaStream_t stream);
int launch_mfcc_tail(const float* mel, int64_t B, int n_mels, int64_t T, float amin, float ref,
                     float top_db, const float* dct, int n_mfcc, float* out,
                     unsigned int* scratch /* B words */, cudaStream_t stream);
int tc_varn_plan_export(const int32_t* k_begin, const int32_t* k_end, int F, int K, int want_chunks,
                        int32_t* order, int32_t* groups, int32_t* chunk_begin, int32_t* n_blocks,
                        int32_t* n_chunks);
int launch_fir_decimate_adjoint(const float* g, int64_t B, int64_t T, int64_t g_pitch,
                                const float* fir, int taps, int factor, float* dx, int64_t L,
                                int64_t dx_pitch, cudaStream_t stream);
int launch_fir_decimate(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch,
                        const float* fir, int taps, int factor, float* y, int64_t Ly, int64_t y_pitch,
                        cudaStream_t stream);

inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace nnab
