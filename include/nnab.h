/*
 * nnab.h — C ABI of the nnaudio-b200 hot path (libnnab.so).
 *
 * The reference (KinWaiCheuk/nnAudio v0.3.3) is pure Python/PyTorch and has no
 * FFI of its own; its hot path is the body of each module's forward():
 * reflect/constant centre padding, conv1d(x, basis, stride=hop) framing +
 * contraction, and the element-wise / filterbank / dB / DCT tail.  Each entry
 * point below replaces exactly one such forward body (file:line cited per
 * function, paths relative to Installation/nnAudio/) and is what a ctypes /
 * cffi binding inside the reference would call (see INTEGRATION.md).
 *
 * Conventions (all entry points):
 *   - plain C types only; every data pointer is a DEVICE pointer owned by the
 *     caller unless the name starts with h_ (host memory);
 *   - inputs are the reference's own fp32 buffers, in the reference's own
 *     layouts (row-major, last dim contiguous); outputs are freshly written
 *     contiguous fp32 tensors in the reference's output layout;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); the call
 *     never synchronises, never allocates device memory and never throws;
 *   - return 0 on success or a negative nnab_status; nnab_strerror() names it;
 *   - `workspace` is caller-provided scratch of at least the number of bytes
 *     the matching nnab_*_workspace_bytes() query returns (may be NULL iff
 *     that query returns 0);
 *   - `path` selects the kernel family: NNAB_PATH_AUTO picks the tcgen05/TMA
 *     kernel when shape/alignment allow and the packed basis is supplied,
 *     otherwise the generic SIMT kernel.  Both are sm_100a CUDA; there is no
 *     CPU fallback.
 */
#ifndef NNAB_H_
#define NNAB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* every entry point below is exported; everything else in the library is hidden */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define NNAB_ABI_VERSION 1

typedef enum nnab_status {
  NNAB_OK = 0,
  NNAB_EINVAL = -1,     /* bad argument / shape mismatch                      */
  NNAB_EALIGN = -2,     /* forced tcgen05 path but alignment rules not met    */
  NNAB_EARCH = -3,      /* device is not sm_100                               */
  NNAB_ECUDA = -4,      /* a CUDA runtime / driver call failed                */
  NNAB_EWORKSPACE = -5, /* workspace NULL or too small                        */
  NNAB_EUNSUPPORTED = -6
} nnab_status;

/* centre padding mode (stft.py:278-289, cqt.py:740-746) */
#define NNAB_PAD_REFLECT 0
#define NNAB_PAD_CONSTANT 1

/* output formats */
#define NNAB_FMT_MAGNITUDE 0   /* (B, F, T)     sqrt(re^2 + im^2 [+ eps])            */
#define NNAB_FMT_COMPLEX 1     /* (B, F, T, 2)  (re, im)                             */
#define NNAB_FMT_PHASE_ANGLE 2 /* (B, F, T)     atan2(im + 0.0, re)   STFT 'Phase'   */
#define NNAB_FMT_PHASE_UNIT 3  /* (B, F, T, 2)  (cos, sin)(atan2(im, re)) CQT 'Phase'*/

/* element type of a waveform input `x` (the *_ex entry points).  Outputs stay fp32.  A 16-bit
 * input gives the same result as its fp32 copy on the same kernel path (every bf16 / fp16 value
 * is exact in fp32 and in a bf16 hi + lo split); bf16 input lets the tensor-core kernels drop the
 * x_lo term of the split (two MMAs per K16 slice instead of three). */
typedef enum nnab_dtype {
  NNAB_DTYPE_F32 = 0,
  NNAB_DTYPE_BF16 = 1,
  NNAB_DTYPE_F16 = 2
} nnab_dtype;

/* kernel family */
#define NNAB_PATH_AUTO 0
#define NNAB_PATH_SIMT 1
#define NNAB_PATH_TCGEN05 2

int nnab_abi_version(void);
const char* nnab_strerror(int status);
/* Last CUDA error string recorded by a call that returned NNAB_ECUDA (thread local). */
const char* nnab_last_cuda_error(void);

/* ------------------------------------------------------------------------- *
 * Basis packing for the tcgen05 path.
 *
 * Splits the fp32 basis pair (re rows, im rows), each (F, K) row-major, into
 * bf16 hi/lo planes (x = hi + lo to ~2^-17) laid out for TMA/UMMA:
 *   packed[plane][tile*BN + part*BN/2 + j][k]   plane 0 = hi, 1 = lo
 *   part 0 = re rows, part 1 = NEGATED im rows, j < BN/2 bins per tile
 * with K padded to a multiple of 64 and bins zero-padded to a multiple of BN/2.
 * BN = nnab_pack_tile_n(F) is chosen per basis to minimise padded columns (208
 * for F = 1025; <= 256).  Negation folds the reference's minus signs
 * (stft.py:308-311 `-spec_imag`, cqt.py:750 `-conv1d(...)`) into the basis.
 * ------------------------------------------------------------------------- */
int nnab_pack_tile_n(int F);
size_t nnab_packed_basis_bytes(int F, int K);
int nnab_pack_basis(const float* w_re, const float* w_im, int F, int K,
                    void* packed, void* stream);
/* Same buffer size, explicit layout request:
 *   NNAB_LAYOUT_DENSE (0)   the layout above
 *   NNAB_LAYOUT_GROUPS (3)  8-bin (re | im) row groups for long nested banks (F <= 128, CQT1992v2): the
 *                           per-K-block-width and tall-A kernels skip the zeros of the shorter wavelets.
 * The forward entry points recognise the layout of the buffer they are given. */
#define NNAB_LAYOUT_DENSE 0
#define NNAB_LAYOUT_GROUPS 3
int nnab_pack_basis_ex(const float* w_re, const float* w_im, int F, int K, int layout,
                       void* packed, void* stream);

/* Block-partial ("sliding") layout for the STFT family: periodic Hann window of length n_fft,
 * integer bins (freq_scale='no', F = n_fft/2 + 1) and hop = n_fft/R with R = 2 or 4, hop % 64 == 0
 * -- the reference's defaults (stft.py:177-178, utils.py:379-384).  The contraction then runs once
 * per hop-sized block against the UN-windowed basis (K = hop instead of n_fft: R x fewer MMA flops);
 * the window is a 3-tap filter along the bin axis and the frame sum a combination of R consecutive
 * block rows, both in the kernel's epilogue.  The packed rows are generated analytically (float64),
 * so the CALLER vouches that its wcos/wsin buffers are exactly that transform
 * (nnaudio_b200/features/_common.py:is_hann_dft checks the tensors).  `packed` needs
 * nnab_packed_block_bytes(n_fft, hop) bytes; the forward entry points recognise the layout.
 * nnab_block_layout_ok() is host-only: 1 when (n_fft, hop) is eligible. */
int nnab_block_layout_ok(int n_fft, int hop);

/* Stream-ordered 32-bit store / cyclic >= wait on a device address (may be peer-mapped): front-end
 * memory operations (cuStreamWriteValue32 / cuStreamWaitValue32), no kernel, no SM.  The multi-GPU
 * gather uses them for its slot handshakes (nnaudio_b200/parallel.py). */
int nnab_stream_write_value32(void* stream, void* addr, uint32_t value);
int nnab_stream_wait_value32_geq(void* stream, void* addr, uint32_t value);
size_t nnab_packed_block_bytes(int n_fft, int hop);
int nnab_pack_basis_block(int n_fft, int hop, void* packed, void* stream);

/* ------------------------------------------------------------------------- *
 * STFT.forward — features/stft.py:256-316.
 *   x        (B, L) rows with pitch x_pitch floats
 *   wcos/wsin (F, n_fft) = the module's `wcos` / `wsin` buffers (window applied)
 *   out      Magnitude/Phase: (B, F, T); Complex: (B, F, T, 2) = (real, -imag)
 *   T must equal (L + 2*pad - n_fft)/hop + 1, pad = center ? n_fft/2 : 0
 *   sqrt_eps = 1e-8 iff the module is trainable (stft.py:301-304), else 0
 * ------------------------------------------------------------------------- */
size_t nnab_stft_workspace_bytes(int64_t B, int64_t L, int n_fft, int F, int hop,
                                 int center, int path);
int nnab_stft_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch,
                      const float* wcos, const float* wsin, const void* packed,
                      int n_fft, int F, int hop, int center, int pad_mode,
                      int out_format, float sqrt_eps, float* out, int64_t T,
                      void* workspace, size_t ws_bytes, int path, void* stream);
/* Same, for x of element type x_dtype (nnab_dtype); x_pitch in elements.  Every waveform entry
 * point has such an _ex form; the plain one is the _ex call with NNAB_DTYPE_F32.  The workspace
 * queries do not depend on the dtype.  An unknown dtype returns NNAB_EINVAL before any device work. */
int nnab_stft_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch, const float* wcos,
                         const float* wsin, const void* packed, int n_fft, int F, int hop,
                         int center, int pad_mode, int out_format, float sqrt_eps, float* out,
                         int64_t T, void* workspace, size_t ws_bytes, int path, void* stream,
                         int x_dtype);

/* ------------------------------------------------------------------------- *
 * Banded filterbank table (tcgen05 path): for every FFT bin the (at most two)
 * non-zero weights of the (n_fb, F) filterbank.  Mel banks are banded like that;
 * for denser banks (gammatone) *h_max_nnz > 2 and the forward calls must be
 * given fb_table = NULL (they then run the un-fused filterbank GEMM).
 * Init-time helper: this call synchronises `stream` to return *h_max_nnz.
 * ------------------------------------------------------------------------- */
size_t nnab_filterbank_table_bytes(int F);
int nnab_build_filterbank_table(const float* fb, int n_fb, int F, void* table,
                                int* h_max_nnz, void* stream);

/* ------------------------------------------------------------------------- *
 * MelSpectrogram.forward / Gammatonegram.forward — features/mel.py:171-189,
 * features/gammatone.py:171-189:  out = fb @ (|STFT(x)| ** power).
 *   fb (n_fb, F) = `mel_basis` or `gammatone_basis`;  out (B, n_fb, T)
 *   fb_table: table from nnab_build_filterbank_table (max_nnz <= 2) or NULL.
 *     With a table and the tcgen05 path the filterbank is applied in the
 *     contraction kernel's epilogue (no (B,F,T) intermediate in HBM).
 * ------------------------------------------------------------------------- */
size_t nnab_filterbank_workspace_bytes(int64_t B, int64_t L, int n_fft, int F, int hop,
                                       int center, int n_fb, int path, int has_table);
int nnab_stft_filterbank_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch,
                                 const float* wcos, const float* wsin, const void* packed,
                                 int n_fft, int F, int hop, int center, int pad_mode,
                                 float sqrt_eps, float power, const float* fb, int n_fb,
                                 const void* fb_table, float* out, int64_t T,
                                 void* workspace, size_t ws_bytes, int path, void* stream);
int nnab_stft_filterbank_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch,
                                    const float* wcos, const float* wsin, const void* packed,
                                    int n_fft, int F, int hop, int center, int pad_mode,
                                    float sqrt_eps, float power, const float* fb, int n_fb,
                                    const void* fb_table, float* out, int64_t T, void* workspace,
                                    size_t ws_bytes, int path, void* stream, int x_dtype);

/* ------------------------------------------------------------------------- *
 * MFCC.forward — features/mel.py:309-326 (= mel -> _power_to_db :263-279 ->
 * _dct(norm='ortho') :281-307 -> [:, :n_mfcc]).
 *   top_db < 0 means None;  dct (n_mfcc, n_mels) fp32 orthonormal DCT-II rows;
 *   out (B, n_mfcc, T)
 * ------------------------------------------------------------------------- */
size_t nnab_mfcc_workspace_bytes(int64_t B, int64_t L, int n_fft, int F, int hop,
                                 int center, int n_mels, int path, int has_table);
int nnab_mfcc_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch,
                      const float* wcos, const float* wsin, const void* packed,
                      int n_fft, int F, int hop, int center, int pad_mode,
                      float sqrt_eps, float power, const float* mel_basis, int n_mels,
                      const void* fb_table, float amin, float ref, float top_db,
                      const float* dct, int n_mfcc, float* out, int64_t T,
                      void* workspace, size_t ws_bytes, int path, void* stream);
int nnab_mfcc_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch, const float* wcos,
                         const float* wsin, const void* packed, int n_fft, int F, int hop,
                         int center, int pad_mode, float sqrt_eps, float power,
                         const float* mel_basis, int n_mels, const void* fb_table, float amin,
                         float ref, float top_db, const float* dct, int n_mfcc, float* out,
                         int64_t T, void* workspace, size_t ws_bytes, int path, void* stream,
                         int x_dtype);

/* ------------------------------------------------------------------------- *
 * CQT1992v2.forward — features/cqt.py:712-780.
 *   k_real/k_imag (n_bins, width) = `cqt_kernels_real/imag` buffers
 *   h_k_begin/h_k_end: HOST int32[n_bins], the non-zero tap support
 *     [begin, end) of every bin (NULL = treat the bank as dense)
 *   scale: DEVICE fp32[n_bins] per-bin factor (sqrt(lenghts) for 'librosa') or
 *     NULL; scale_all: scalar factor (2 for 'wrap', else 1)
 *   out_format: MAGNITUDE, COMPLEX (real, imag) or PHASE_UNIT (cos, sin)
 * ------------------------------------------------------------------------- */
size_t nnab_cqt1992v2_workspace_bytes(int64_t B, int64_t L, int width, int n_bins, int hop,
                                      int center, int path);
int nnab_cqt1992v2_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch,
                           const float* k_real, const float* k_imag, const void* packed,
                           const int32_t* h_k_begin, const int32_t* h_k_end,
                           int n_bins, int width, int hop, int center, int pad_mode,
                           const float* scale, float scale_all, int out_format,
                           float sqrt_eps, float* out, int64_t T,
                           void* workspace, size_t ws_bytes, int path, void* stream);
int nnab_cqt1992v2_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch,
                              const float* k_real, const float* k_imag, const void* packed,
                              const int32_t* h_k_begin, const int32_t* h_k_end, int n_bins,
                              int width, int hop, int center, int pad_mode, const float* scale,
                              float scale_all, int out_format, float sqrt_eps, float* out,
                              int64_t T, void* workspace, size_t ws_bytes, int path, void* stream,
                              int x_dtype);

/* ------------------------------------------------------------------------- *
 * CQT2010v2.forward / VQT.forward — features/cqt.py:1070-1139,
 * features/vqt.py:143-215 (+ utils.py:73-124 downsampling, :498-521
 * get_cqt_complex with its reflect -> zero-padding fallback).
 *   h_k_real/h_k_imag: HOST arrays of n_octaves DEVICE pointers, octave 0 = top;
 *     bank i is (n_filters, h_widths[i]) fp32 (CQT2010v2 passes the same bank
 *     n_octaves times)
 *   lowpass (256) = `lowpass_filter`; early_filter (256) or NULL with
 *     early_factor (1 = inactive) = `early_downsample_filter`
 *   hop = the module's hop_length AFTER early downsampling
 *   scale: DEVICE fp32[n_bins] = downsample_factor * sqrt(lenghts) etc.
 *   out (B, n_bins, T[, 2]);  T = floor(L_early / hop) + 1 for every octave,
 *     otherwise NNAB_EINVAL (the reference's torch.cat would fail)
 * ------------------------------------------------------------------------- */
/* Packed (bf16 hi/lo, banded-Toeplitz) form of a 256-tap decimation FIR for the
 * tensor-core pyramid: lowpass_filter with dec = 2, early_downsample_filter with
 * dec = early_factor.  Init-time, cached by the caller. */
size_t nnab_packed_fir_bytes(int taps, int dec);
int nnab_pack_fir(const float* fir, int taps, int dec, void* packed, void* stream);

/* Host only (tests / tooling): the K-block plan of the per-block-width kernel
 * (order[i] = 64-sample K block, groups[i] = 8-bin groups it reaches, widest first;
 * chunk_begin[0..n_chunks] = split-K chunks of equal modelled cost).  Arrays: 512 / 512 / 17 ints. */
int nnab_debug_varn_plan(const int32_t* h_k_begin, const int32_t* h_k_end, int n_bins, int width,
                         int want_chunks, int32_t* order, int32_t* groups, int32_t* chunk_begin,
                         int32_t* n_blocks, int32_t* n_chunks);

/* One decimating-FIR stage and its adjoint, for the training path
 * of the pyramid.  Replace `downsampling_by_n` / `downsampling_by_2` (utils.py:73-124) and what
 * autograd derives from them.
 *   y  (B, Ly) = conv1d(x (B, L), fir (taps), stride=factor, padding=(taps-1)/2),
 *     Ly = (L + 2*((taps-1)/2) - taps) / factor + 1
 *   dx (B, L)  = the gradient of that w.r.t. x for an upstream gradient g (B, Ly)
 * All tensors fp32, contiguous rows with the given pitches. */
int nnab_fir_decimate(const float* x, int64_t B, int64_t L, int64_t x_pitch, const float* fir,
                      int taps, int factor, float* y, int64_t Ly, void* stream);
int nnab_fir_decimate_adjoint(const float* g, int64_t B, int64_t Ly, int64_t g_pitch,
                              const float* fir, int taps, int factor, float* dx, int64_t L,
                              void* stream);

size_t nnab_cqt_pyramid_workspace_bytes(int64_t B, int64_t L, int n_octaves, int early_factor,
                                        int max_width, int hop, int path);
/*   h_packed: HOST array of n_octaves DEVICE pointers to the nnab_pack_basis() copy of
 *     each bank (octave i's real/imag pair), or NULL / NULL entries = CUDA-core kernel
 *     for that octave.
 *   lowpass_packed / early_packed: nnab_pack_fir() copies or NULL.  With all packed
 *     inputs present the whole pyramid runs on the tensor cores: every anti-alias stage
 *     is a framed contraction whose epilogue writes the next level's padded bf16 planes. */
int nnab_cqt_pyramid_forward(const float* x, int64_t B, int64_t L, int64_t x_pitch,
                             int n_octaves, const float* const* h_k_real,
                             const float* const* h_k_imag, const void* const* h_packed,
                             const int32_t* h_widths,
                             int n_filters, const float* lowpass, const void* lowpass_packed,
                             const float* early_filter, const void* early_packed,
                             int early_factor, int hop, int pad_mode, int n_bins,
                             const float* scale, float scale_all, int out_format,
                             float sqrt_eps, float* out, int64_t T,
                             void* workspace, size_t ws_bytes, int path, void* stream);
/* With a 16-bit x only the first pyramid level reads it (and only level 0's octave runs the
 * two-term contraction for bf16); the decimated levels are fp32 signals as before. */
int nnab_cqt_pyramid_forward_ex(const void* x, int64_t B, int64_t L, int64_t x_pitch,
                                int n_octaves, const float* const* h_k_real,
                                const float* const* h_k_imag, const void* const* h_packed,
                                const int32_t* h_widths, int n_filters, const float* lowpass,
                                const void* lowpass_packed, const float* early_filter,
                                const void* early_packed, int early_factor, int hop, int pad_mode,
                                int n_bins, const float* scale, float scale_all, int out_format,
                                float sqrt_eps, float* out, int64_t T, void* workspace,
                                size_t ws_bytes, int path, void* stream, int x_dtype);

/* ------------------------------------------------------------------------- *
 * STFT.inverse / iSTFT.forward — features/stft.py:15-63 (inverse_stft), :318-356,
 * :526-546; helpers utils.py:43-70 (SURVEY §8f "next" #2).
 *   X (B, f_in, T, 2) complex spectrogram; f_in = n_fft/2+1 with onesided, else n_fft
 *   kernel_cos / kernel_sin (n_fft, n_fft) = `kernel_cos_inv`/`kernel_sin_inv` of
 *     STFT(iSTFT=True) or `kernel_cos`/`kernel_sin` of the iSTFT module; packed once with
 *     nnab_pack_istft_basis (the one-sided mirroring of utils.py:63-70 is folded in)
 *   window (n_fft) = `window_mask`;  length < 0 means None
 *   out (B, out_len): out_len = n_fft + hop*(T-1) - 2*pad (length None, center) etc.
 * Runs on the tensor-core kernel only (inverse-DFT GEMM + overlap-add epilogue +
 * window-sumsquare normalisation).
 * ------------------------------------------------------------------------- */
size_t nnab_packed_istft_bytes(int n_fft, int f_in);
int nnab_pack_istft_basis(const float* kernel_cos, const float* kernel_sin, int n_fft, int f_in,
                          int onesided, void* packed, void* stream);
size_t nnab_istft_workspace_bytes(int64_t B, int f_in, int64_t T, int n_fft, int hop);
int nnab_istft_forward(const float* X, int64_t B, int f_in, int64_t T, const void* packed,
                       const float* window, int n_fft, int hop, int center, int64_t length,
                       float* out, int64_t out_len, void* workspace, size_t ws_bytes,
                       void* stream);

/* ------------------------------------------------------------------------- *
 * Input gradient of the framed complex contraction (SURVEY §8f "next" #1, the dX half;
 * the reference gets it from autograd through conv1d, stft.py:290-293 / cqt.py:749-750):
 *   g   (B, F, T, 2)  gradient w.r.t. (real, imag) = (conv(x, w_re), -conv(x, w_im))
 *   dx  (B, L)        = pad^T ( overlap_add_t ( g_re[., t] @ w_re - g_im[., t] @ w_im ) )
 * `packed_adj` = nnab_pack_adjoint_basis(w_re, w_im) (W^T rows, bf16 hi/lo).  One GEMM on
 * the tensor-core kernel with the overlap-add epilogue, then the padding adjoint.
 * ------------------------------------------------------------------------- */
size_t nnab_packed_adjoint_bytes(int K, int F);
int nnab_pack_adjoint_basis(const float* w_re, const float* w_im, int F, int K, void* packed,
                            void* stream);
size_t nnab_framed_backward_input_workspace_bytes(int64_t B, int64_t L, int K, int F, int hop,
                                                  int center);
int nnab_framed_backward_input(const float* g, int64_t B, int F, int64_t T, const void* packed_adj,
                               int K, int hop, int center, int pad_mode, float* dx, int64_t L,
                               void* workspace, size_t ws_bytes, void* stream);

/* Weight gradient of the framed complex contraction (the dW half of SURVEY §8f #1):
 *   dw (2F, K) fp32:  rows [0, F)  = sum_{b,t} g_re[b,f,t] * frame_{b,t}   (= d loss / d w_re)
 *                     rows [F, 2F) = sum_{b,t} g_im[b,f,t] * frame_{b,t}   (= -d loss / d w_im)
 * One split-K GEMM on the tensor-core kernel: gradient rows x transposed frame matrix. */
size_t nnab_framed_backward_weight_workspace_bytes(int64_t B, int64_t L, int K, int F, int hop,
                                                   int center);
int nnab_framed_backward_weight(const float* g, const float* x, int64_t B, int64_t L,
                                int64_t x_pitch, int F, int64_t T, int K, int hop, int center,
                                int pad_mode, float* dw, void* workspace, size_t ws_bytes,
                                void* stream);

/* Kernel launches issued by this library since load (process wide; used by
 * bench.py for its `gpu_launches` claim). */
uint64_t nnab_launch_count(void);

/* Leave `n_sms` SMs out of the persistent tensor-core grids (process wide, default 0) so
 * that a concurrently running collective (the NCCL output gather of the multi-GPU path)
 * has SMs to run on; returns the previous value. */
int nnab_set_sm_reserve(int n_sms);

/* Live timing of the dominant kernel (the framed contraction) for bench.py's
 * roofline: while enabled, every framed-contraction launch is bracketed by a
 * cudaEvent pair recorded on the launching stream.  nnab_profile_read()
 * synchronises those events, returns the summed duration in ms and the number
 * of launches timed since the last read, and resets the accumulator. */
void nnab_profile_enable(int on);
int nnab_profile_read(double* framed_ms, uint64_t* framed_launches);
/* MMA flops the tensor-core launches EXECUTED since the last read (all bf16 split terms, tile
 * padding and structural zeros included) -> bench.py's roofline.tensor_pipe. */
int nnab_profile_read_exec_flops(double* exec_flops);
/* Launches of the tall-A CQT kernel that ran the balanced schedule (tiles shared between two CTA
 * pairs, framed_tc2t_kernel<., true>) since load -- lets a test tell which schedule it exercised. */
uint64_t nnab_balanced_launch_count(void);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* NNAB_H_ */
