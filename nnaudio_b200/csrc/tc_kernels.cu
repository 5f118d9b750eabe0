// tcgen05 / TMA framed contraction for sm_100a.
//
//   D[g, n] = sum_k A[g, k] * W[n, k]        g = virtual frame, n = basis row
//
// * A is never materialised: the padded waveform is written once as bf16 hi/lo
//   planes (pad_split_kernel) with a per-clip pitch that is a multiple of hop, so
//   the frames of the WHOLE batch form one Toeplitz matrix whose row g starts at
//   element g*hop.  TMA reads 128-frame x BK tiles of it straight into
//   128B/64B-swizzled shared memory (either as a plain (rows x hop) matrix when
//   BK | hop, or through an overlapping-stride tensor map otherwise).
// * W (basis) is pre-split into bf16 hi/lo planes, re rows and NEGATED im rows
//   grouped per N tile (pack_basis_kernel).
// * fp32 parity on bf16 tensor cores: x*w ~= xhi*whi + xlo*whi + xhi*wlo
//   (3 tcgen05.mma passes into one fp32 TMEM accumulator; error ~2^-16).
// * Warp roles (256 threads, 1 CTA/SM, persistent over output tiles):
//     warp 0  TMA producer      warp 1  MMA issuer      warp 2  TMEM alloc
//     warps 4-7  epilogue: tcgen05.ld -> magnitude/complex/phase/power ->
//                coalesced stores in the reference's (B, F, T[,2]) layout
//   smem full/empty mbarrier ring + double-buffered TMEM accumulators.
#include <cuda.h>
#include <atomic>
#include <mutex>
#include <unordered_map>
#include <algorithm>
#include <vector>
#include <cuda_bf16.h>
#include <stdlib.h>

#include "common.cuh"
#include "epilogue.cuh"
#include "tc_ptx.cuh"
#include "tc_host.cuh"
#include "tc_decim.cuh"

namespace nnab {

constexpr int TC_MAX_N_TILES = 128;
constexpr int TC_ACC_STRIDE = 256;  // TMEM columns per accumulator buffer


// N tile (columns = re + im rows of bn/2 bins): minimise padded columns.
static int choose_bn(int F) {
  const int cols = 2 * F;
  if (cols <= 256) return round_up_i(cols, 16) < 32 ? 32 : round_up_i(cols, 16);
  int best = 256, best_total = round_up_i(cols, 256);
  for (int bn = 240; bn >= 128; bn -= 16) {
    const int total = (cols + bn - 1) / bn * bn;
    if (total < best_total) { best_total = total; best = bn; }
  }
  return best;
}

int tc_tile_n(int F) { return choose_bn(F > 0 ? F : 1); }

size_t tc_packed_bytes(int F, int K) {
  const int bn = choose_bn(F);
  const int n_tiles = (2 * F + bn - 1) / bn;
  const size_t rows = (size_t)n_tiles * bn;
  const size_t kpad = (size_t)round_up_i(K, 64);
  return 2 * rows * kpad * sizeof(__nv_bfloat16);
}

// ---------------------------------------------------------------------------
// geometry of the split / padded signal workspace
// ---------------------------------------------------------------------------

// Frames t = p, p + np, p + 2 np, ... (phase p of np = 8 / gcd(hop, 8)) start at
// multiples of hop * np, which is always a multiple of 8 samples = 16 bytes in
// bf16: every hop is served by TMA, one pass per phase over a signal shifted by
// p * hop samples.
static int gcd_i(int a, int b) { return b == 0 ? a : gcd_i(b, a % b); }
int num_phases(int hop) { return 8 / gcd_i(hop, 8); }

SplitGeom split_geom(int64_t B, int64_t L, int K, int hop, int pad) {
  const int hop_eff = hop * num_phases(hop);
  SplitGeom g;
  g.t_slots = (L + 2 * (int64_t)pad + hop_eff - 1) / hop_eff;
  g.nv = B * g.t_slots;
  const int kpad = round_up_i(K, 64);
  g.rows = g.nv + (kpad + hop_eff - 1) / hop_eff + 1;
  g.plane_stride = (g.rows * hop_eff + 63) / 64 * 64;
  return g;
}

size_t tc_workspace_bytes(int64_t B, int64_t L, int K, int hop, int pad) {
  const SplitGeom g = split_geom(B, L, K, hop, pad);
  return (size_t)(2 * g.plane_stride) * sizeof(__nv_bfloat16) + 256;
}

bool tc_supported(const FramedProblem& p) {
  if (p.hop <= 0 || p.K < 16) return false;
  // (pre-split planes are laid out by the caller, which guarantees >= 1 valid frame)
  if (p.presplit == nullptr && p.L + 2 * (int64_t)p.pad < p.K) return false;
  const SplitGeom g = split_geom(p.B > 0 ? p.B : 1, p.L, p.K, p.hop, p.pad);
  if (g.rows >= (1ll << 31) || g.plane_stride >= (1ll << 38)) return false;
  const int bn = choose_bn(p.F);
  if ((2 * p.F + bn - 1) / bn > TC_MAX_N_TILES) return false;
  return true;
}

// ---------------------------------------------------------------------------
// pre-pass kernels
// ---------------------------------------------------------------------------

// Eight consecutive samples i0 .. i0 + 7 of a centre-padded clip (reflect / zero padding folded
// into the index).  16-bit input: one 16-byte load when the eight are interior and aligned.
template <typename T>
__device__ __forceinline__ void fetch8_padded(const T* __restrict__ xb, int64_t L, int64_t i0,
                                              int pad, int pad_mode, float* v) {
  const int64_t padded_len = L + 2 * (int64_t)pad;
  if constexpr (sizeof(T) == 2) {
    const int64_t j0 = i0 - pad;
    if (j0 >= 0 && j0 + 8 <= L && ((reinterpret_cast<uintptr_t>(xb + j0) & 15u) == 0)) {
      unpack8(__ldg(reinterpret_cast<const uint4*>(xb + j0)), xb, v);
      return;
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int64_t i = i0 + e;  // index into the centre-padded clip
    v[e] = 0.f;
    if (i < padded_len) {
      int64_t j = i - pad;
      if (j < 0) j = (pad_mode == NNAB_PAD_REFLECT) ? -j : -1;
      else if (j >= L) j = (pad_mode == NNAB_PAD_REFLECT) ? 2 * (L - 1) - j : -1;
      if (j >= 0 && j < L) v[e] = ldg_sample(xb + j);
    }
  }
}

// One thread = 8 consecutive samples of one clip's slot region (16-byte stores).  hi_only: the lo
// plane is left alone (bf16 input: it would be all zeros, and the two-term kernels never read it).
template <typename T>
__global__ void __launch_bounds__(256) pad_split_kernel(
    const T* __restrict__ x, int64_t L, int64_t x_pitch, int pad, int pad_mode, int shift,
    int64_t clip_pitch, int64_t plane_stride, __nv_bfloat16* __restrict__ planes, int hi_only) {
  const int64_t b = blockIdx.y;
  const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i0 >= clip_pitch) return;
  const T* __restrict__ xb = x + b * x_pitch;
  float v[8];
  fetch8_padded(xb, L, i0 + shift, pad, pad_mode, v);
  __align__(16) __nv_bfloat16 hi[8];
  __align__(16) __nv_bfloat16 lo[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) split_bf16(v[e], hi[e], lo[e]);
  const int64_t o = b * clip_pitch + i0;
  *reinterpret_cast<uint4*>(planes + o) = *reinterpret_cast<const uint4*>(hi);
  if (!hi_only)
    *reinterpret_cast<uint4*>(planes + plane_stride + o) = *reinterpret_cast<const uint4*>(lo);
}

// Two differently padded split copies of the same batch in one pass over x (level 0 of
// the CQT pyramid: reflect-padded copy for the octave CQT + zero-margin copy for the FIR).
template <typename T>
__global__ void __launch_bounds__(256) pad_split2_kernel(
    const T* __restrict__ x, int64_t L, int64_t x_pitch,
    int pad_a, int mode_a, int64_t pitch_a, int64_t plane_a, __nv_bfloat16* __restrict__ pa,
    int pad_b, int mode_b, int64_t pitch_b, int64_t plane_b, __nv_bfloat16* __restrict__ pb) {
  const int64_t b = blockIdx.y;
  const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  const T* __restrict__ xb = x + b * x_pitch;
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    const int pad = which ? pad_b : pad_a;
    const int mode = which ? mode_b : mode_a;
    const int64_t pitch = which ? pitch_b : pitch_a;
    const int64_t plane = which ? plane_b : plane_a;
    __nv_bfloat16* __restrict__ dst = which ? pb : pa;
    if (i0 >= pitch) continue;
    float v[8];
    fetch8_padded(xb, L, i0, pad, mode, v);
    __align__(16) __nv_bfloat16 hi[8];
    __align__(16) __nv_bfloat16 lo[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) split_bf16(v[e], hi[e], lo[e]);
    const int64_t o = b * pitch + i0;
    *reinterpret_cast<uint4*>(dst + o) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(dst + plane + o) = *reinterpret_cast<const uint4*>(lo);
  }
}

// pad_split_kernel launch for the element type of x
static int launch_pad_split(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch, int pad,
                            int pad_mode, int shift, int64_t clip_pitch, int64_t plane_stride,
                            __nv_bfloat16* planes, bool hi_only, cudaStream_t stream) {
  if (hi_only && x_dtype != NNAB_DTYPE_BF16) return NNAB_EINVAL;
  dim3 grid((unsigned)ceil_div64(clip_pitch, 256 * 8), (unsigned)B);
  switch (x_dtype) {
    case NNAB_DTYPE_F32:
      pad_split_kernel<<<grid, 256, 0, stream>>>((const float*)x, L, x_pitch, pad, pad_mode, shift,
                                                 clip_pitch, plane_stride, planes, 0);
      break;
    case NNAB_DTYPE_BF16:
      pad_split_kernel<<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, L, x_pitch, pad, pad_mode,
                                                 shift, clip_pitch, plane_stride, planes, hi_only ? 1 : 0);
      break;
    case NNAB_DTYPE_F16:
      pad_split_kernel<<<grid, 256, 0, stream>>>((const __half*)x, L, x_pitch, pad, pad_mode, shift,
                                                 clip_pitch, plane_stride, planes, 0);
      break;
    default: return NNAB_EINVAL;
  }
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// packed[plane][tile*bn + part*bn/2 + j][k]; part 1 rows are NEGATED im rows.
__global__ void __launch_bounds__(256) pack_basis_kernel(
    const float* __restrict__ w_re, const float* __restrict__ w_im, int F, int K, int bn,
    int rows, int kpad, __nv_bfloat16* __restrict__ packed) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int k8 = kpad / 8;
  if (idx >= (int64_t)rows * k8) return;
  const int r = (int)(idx / k8);
  const int k0 = (int)(idx % k8) * 8;
  const int half = bn / 2;
  const int tile = r / bn, within = r % bn;
  const int part = within / half, j = within % half;
  const int f = tile * half + j;
  __align__(16) __nv_bfloat16 hi[8];
  __align__(16) __nv_bfloat16 lo[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = k0 + e;
    float v = 0.f;
    if (f < F && k < K)
      v = part == 0 ? __ldg(w_re + (int64_t)f * K + k) : -__ldg(w_im + (int64_t)f * K + k);
    split_bf16(v, hi[e], lo[e]);
  }
  const int64_t o = (int64_t)r * kpad + k0;
  *reinterpret_cast<uint4*>(packed + o) = *reinterpret_cast<const uint4*>(hi);
  *reinterpret_cast<uint4*>(packed + (int64_t)rows * kpad + o) = *reinterpret_cast<const uint4*>(lo);
}

void tc_forget_packed(const void* packed);
bool tc_varn_enabled();
bool tc_varn_basis_ok(int F, int K);
int tc_pack_basis_varn(const float* w_re, const float* w_im, int F, int K, void* packed,
                       cudaStream_t stream);

// layout: 0 = dense (always valid); 3 = 8-bin-group layout for the per-K-block-width / tall-A kernels
// (any basis with F <= 128).  NNAB_VARN=0 forces dense.
int tc_pack_basis_layout(const float* w_re, const float* w_im, int F, int K, int layout, void* packed,
                         cudaStream_t stream) {
  const char* ev = getenv("NNAB_VARN");
  if (layout == 3 && !(ev != nullptr && atoi(ev) == 0) && tc_varn_basis_ok(F, K))
    return tc_pack_basis_varn(w_re, w_im, F, K, packed, stream);
  if (layout != 0 && layout != 3) return NNAB_EINVAL;
  return tc_pack_basis(w_re, w_im, F, K, packed, stream);
}

int tc_pack_basis(const float* w_re, const float* w_im, int F, int K, void* packed,
                  cudaStream_t stream) {
  // (NNAB_VARN=1: debugging switch -- the 8-bin-group layout for every long bank)
  if (tc_varn_enabled() && tc_varn_basis_ok(F, K) && K >= 4096)
    return tc_pack_basis_varn(w_re, w_im, F, K, packed, stream);
  tc_forget_packed(packed);
  const int bn = choose_bn(F);
  const int n_tiles = (2 * F + bn - 1) / bn;
  const int rows = n_tiles * bn;
  const int kpad = round_up_i(K, 64);
  const int64_t threads = (int64_t)rows * (kpad / 8);
  pack_basis_kernel<<<(unsigned)ceil_div64(threads, 256), 256, 0, stream>>>(
      w_re, w_im, F, K, bn, rows, kpad, (__nv_bfloat16*)packed);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// Decimating FIR as a framed contraction: frame t of the zero-padded level signal
// (sample m at plane offset 128 + m, hop 128*dec) against the banded Toeplitz rows
//   H[j][k] = fir[k - 1 - dec*j]        j = 0..127 outputs per frame
// gives y[128 t + j] = sum_m fir[m] x[dec*(128 t + j) + m - 127]
// (utils.py:73-100: conv1d(stride=dec, padding=127)).  Rows 0..63 sit in the "re" half
// of the single N tile and rows 64..127 in the "im" half (not negated).
int tc_fir_k(int taps, int dec) { return round_up_i(dec * 127 + taps + 1, 64); }
size_t tc_packed_fir_bytes(int taps, int dec) {
  return (size_t)2 * 128 * tc_fir_k(taps, dec) * sizeof(__nv_bfloat16);
}

__global__ void __launch_bounds__(256) pack_fir_kernel(const float* __restrict__ fir, int taps,
                                                       int dec, int kpad,
                                                       __nv_bfloat16* __restrict__ packed) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 128 * kpad) return;
  const int r = idx / kpad, k = idx % kpad;
  const int m = k - 1 - dec * r;
  const float v = (m >= 0 && m < taps) ? __ldg(fir + m) : 0.f;
  __nv_bfloat16 hi, lo;
  split_bf16(v, hi, lo);
  packed[idx] = hi;
  packed[(int64_t)128 * kpad + idx] = lo;
}

int tc_pack_fir(const float* fir, int taps, int dec, void* packed, cudaStream_t stream) {
  tc_forget_packed(packed);  // dense rows: drop any stale layout tag of a recycled address
  const int kpad = tc_fir_k(taps, dec);
  pack_fir_kernel<<<(128 * kpad + 255) / 256, 256, 0, stream>>>(fir, taps, dec, kpad,
                                                               (__nv_bfloat16*)packed);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

void tc_split_geometry(int64_t B, int64_t L, int K, int hop, int pad, int64_t* t_slots,
                       int64_t* plane_stride, int* hop_eff) {
  const SplitGeom g = split_geom(B, L, K, hop, pad);
  if (t_slots) *t_slots = g.t_slots;
  if (plane_stride) *plane_stride = g.plane_stride;
  if (hop_eff) *hop_eff = hop * num_phases(hop);
}

static int zero_tail(__nv_bfloat16* planes, const SplitGeom& g, int hop_eff, cudaStream_t stream,
                     bool hi_only = false) {
  const int64_t tail = g.plane_stride - g.nv * hop_eff;
  for (int pl = 0; pl < (hi_only ? 1 : 2); ++pl)
    NNAB_CUDA_TRY(cudaMemsetAsync(planes + pl * g.plane_stride + g.nv * hop_eff, 0,
                                  (size_t)tail * sizeof(__nv_bfloat16), stream));
  return NNAB_OK;
}

// phase-0 pad + split of a batch into caller-managed planes
int tc_pad_split(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch, int K, int hop,
                 int pad, int pad_mode, void* planes_v, cudaStream_t stream, bool hi_only) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  const SplitGeom g = split_geom(B, L, K, hop, pad);
  const int hop_eff = hop * num_phases(hop);
  __nv_bfloat16* planes = (__nv_bfloat16*)planes_v;
  int rc = zero_tail(planes, g, hop_eff, stream, hi_only);
  if (rc) return rc;
  const int64_t clip_pitch = g.t_slots * hop_eff;
  return launch_pad_split(x, x_dtype, B, L, x_pitch, pad, pad_mode, 0, clip_pitch, g.plane_stride,
                          planes, hi_only, stream);
}

__global__ void zero_margins_kernel(__nv_bfloat16* __restrict__ planes, int64_t plane_stride,
                                    int64_t pitch, int64_t keep_lo, int64_t keep_hi);

// pad + split into caller-defined geometry (clip pitch / plane stride in elements).  pad_split_kernel
// writes the whole [0, clip_pitch) slot of every clip (zeros past the padded signal); the tail
// [B * clip_pitch, plane_stride) is zeroed here.
int tc_pad_split_ex(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch, int pad,
                    int pad_mode, int64_t clip_pitch, int64_t plane_stride, void* planes_v,
                    cudaStream_t stream) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  if (clip_pitch % 8 != 0 || plane_stride < B * clip_pitch) return NNAB_EINVAL;
  __nv_bfloat16* planes = (__nv_bfloat16*)planes_v;
  const int64_t tail = plane_stride - B * clip_pitch;
  for (int pl = 0; pl < 2 && tail > 0; ++pl)
    NNAB_CUDA_TRY(cudaMemsetAsync(planes + pl * plane_stride + B * clip_pitch, 0,
                                  (size_t)tail * sizeof(__nv_bfloat16), stream));
  return launch_pad_split(x, x_dtype, B, L, x_pitch, pad, pad_mode, 0, clip_pitch, plane_stride, planes,
                          false, stream);
}

// zero [keep_hi, clip_pitch) and [0, keep_lo) of every clip slot (both planes) + the tail of the planes
int tc_zero_slots(void* planes_v, int64_t B, int64_t clip_pitch, int64_t plane_stride, int64_t keep_lo,
                  int64_t keep_hi, cudaStream_t stream) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  __nv_bfloat16* planes = (__nv_bfloat16*)planes_v;
  const int64_t tail = plane_stride - B * clip_pitch;
  for (int pl = 0; pl < 2 && tail > 0; ++pl)
    NNAB_CUDA_TRY(cudaMemsetAsync(planes + pl * plane_stride + B * clip_pitch, 0,
                                  (size_t)tail * sizeof(__nv_bfloat16), stream));
  if (keep_hi > clip_pitch) keep_hi = clip_pitch;
  if (keep_lo < 0) keep_lo = 0;
  const int64_t n = keep_lo + (clip_pitch - keep_hi);
  if (n <= 0) return NNAB_OK;
  int gx = (int)ceil_div64(n, 256);
  if (gx > 64) gx = 64;
  zero_margins_kernel<<<dim3(gx, (unsigned)B), 256, 0, stream>>>(planes, plane_stride, clip_pitch,
                                                                keep_lo, keep_hi);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

int tc_pad_split2(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch,
                  int K_a, int hop_a, int pad_a, int mode_a, void* planes_a,
                  int K_b, int hop_b, int pad_b, int mode_b, void* planes_b, cudaStream_t stream) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  const SplitGeom ga = split_geom(B, L, K_a, hop_a, pad_a);
  const SplitGeom gb = split_geom(B, L, K_b, hop_b, pad_b);
  const int he_a = hop_a * num_phases(hop_a), he_b = hop_b * num_phases(hop_b);
  int rc = zero_tail((__nv_bfloat16*)planes_a, ga, he_a, stream);
  if (rc) return rc;
  if ((rc = zero_tail((__nv_bfloat16*)planes_b, gb, he_b, stream))) return rc;
  const int64_t pitch_a = ga.t_slots * he_a, pitch_b = gb.t_slots * he_b;
  const int64_t pmax = pitch_a > pitch_b ? pitch_a : pitch_b;
  dim3 grid((unsigned)ceil_div64(pmax, 256 * 8), (unsigned)B);
  __nv_bfloat16* pa = (__nv_bfloat16*)planes_a;
  __nv_bfloat16* pb = (__nv_bfloat16*)planes_b;
  switch (x_dtype) {
    case NNAB_DTYPE_F32:
      pad_split2_kernel<<<grid, 256, 0, stream>>>((const float*)x, L, x_pitch, pad_a, mode_a, pitch_a,
                                                  ga.plane_stride, pa, pad_b, mode_b, pitch_b,
                                                  gb.plane_stride, pb);
      break;
    case NNAB_DTYPE_BF16:
      pad_split2_kernel<<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, L, x_pitch, pad_a, mode_a,
                                                  pitch_a, ga.plane_stride, pa, pad_b, mode_b, pitch_b,
                                                  gb.plane_stride, pb);
      break;
    case NNAB_DTYPE_F16:
      pad_split2_kernel<<<grid, 256, 0, stream>>>((const __half*)x, L, x_pitch, pad_a, mode_a, pitch_a,
                                                  ga.plane_stride, pa, pad_b, mode_b, pitch_b,
                                                  gb.plane_stride, pb);
      break;
    default: return NNAB_EINVAL;
  }
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// Zero every element of each clip's slot region outside [keep_lo, keep_hi) (both planes)
// plus the K-overhang tail: the parts of a level buffer the FIR epilogue never writes.
__global__ void __launch_bounds__(256) zero_margins_kernel(__nv_bfloat16* __restrict__ planes,
                                                           int64_t plane_stride, int64_t pitch,
                                                           int64_t keep_lo, int64_t keep_hi) {
  const int64_t b = blockIdx.y;
  const int64_t lo_n = keep_lo, hi_n = pitch - keep_hi;
  const int64_t n = lo_n + hi_n;
  const __nv_bfloat16 z = __float2bfloat16_rn(0.f);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pos = i < lo_n ? i : keep_hi + (i - lo_n);
    planes[b * pitch + pos] = z;
    planes[plane_stride + b * pitch + pos] = z;
  }
}

int tc_zero_margins(void* planes_v, int64_t B, int64_t L, int K, int hop, int pad, int64_t keep_lo,
                    int64_t keep_hi, cudaStream_t stream) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  const SplitGeom g = split_geom(B, L, K, hop, pad);
  const int hop_eff = hop * num_phases(hop);
  __nv_bfloat16* planes = (__nv_bfloat16*)planes_v;
  int rc = zero_tail(planes, g, hop_eff, stream);
  if (rc) return rc;
  const int64_t pitch = g.t_slots * hop_eff;
  if (keep_hi > pitch) keep_hi = pitch;
  if (keep_lo < 0) keep_lo = 0;
  const int64_t n = keep_lo + (pitch - keep_hi);
  if (n <= 0) return NNAB_OK;
  int gx = (int)ceil_div64(n, 256);
  if (gx > 64) gx = 64;
  zero_margins_kernel<<<dim3(gx, (unsigned)B), 256, 0, stream>>>(planes, g.plane_stride, pitch,
                                                                keep_lo, keep_hi);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// ---------------------------------------------------------------------------
// inverse STFT (stft.py:15-63) as a plain GEMM on the framed kernel:
//   frame[g, n] = sum_k A[g, k] * Winv[n, k],  g = b*T + t,  k = (re | im) x frequency
// "hop = Kpad" rows: every frame is its own row, so the Toeplitz machinery degenerates to a
// row-major matrix.  The FMT_OLA epilogue windows the frame and overlap-adds it.
// ---------------------------------------------------------------------------
int tc_istft_k(int f_in) { return round_up_i(2 * f_in, 64); }
int tc_istft_bn(int n_fft) { return n_fft >= 256 ? 256 : (round_up_i(n_fft, 16) < 32 ? 32 : round_up_i(n_fft, 16)); }
size_t tc_packed_istft_bytes(int n_fft, int f_in) {
  const int bn = tc_istft_bn(n_fft);
  const size_t rows = (size_t)((n_fft + bn - 1) / bn) * bn;
  return 2 * rows * tc_istft_k(f_in) * sizeof(__nv_bfloat16);
}

// Winv[n][f]        = KC[n][f] (+ KC[n][N-f] for a mirrored one-sided bin)          re part
// Winv[n][F_in + f] = -(KS[n][f] (- KS[n][N-f]))                                    im part
// i.e. the reference's extend_fbins (utils.py:63-70) folded into the kernels.
// With `transposed` the inputs are the FORWARD bases (f_in, n_fft) = wcos / wsin and the rows
// become W^T (the adjoint used by the input gradient): Winv[n][f] = wcos[f][n], -wsin[f][n].
__global__ void __launch_bounds__(256) pack_istft_kernel(const float* __restrict__ kc,
                                                         const float* __restrict__ ks, int n_fft,
                                                         int f_in, int onesided, int transposed,
                                                         int rows, int kpad,
                                                         __nv_bfloat16* __restrict__ packed) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * kpad) return;
  const int n = (int)(idx / kpad), k = (int)(idx % kpad);
  float v = 0.f;
  if (n < n_fft && k < 2 * f_in) {
    const int part = k / f_in, f = k % f_in;
    const bool mirror = onesided && !transposed && f > 0 && f < n_fft - f && (n_fft - f) < n_fft;
    if (transposed) {
      v = part == 0 ? __ldg(kc + (int64_t)f * n_fft + n) : -__ldg(ks + (int64_t)f * n_fft + n);
    } else if (part == 0) {
      v = __ldg(kc + (int64_t)n * n_fft + f);
      if (mirror) v += __ldg(kc + (int64_t)n * n_fft + (n_fft - f));
    } else {
      v = __ldg(ks + (int64_t)n * n_fft + f);
      if (mirror) v -= __ldg(ks + (int64_t)n * n_fft + (n_fft - f));
      v = -v;
    }
  }
  __nv_bfloat16 hi, lo;
  split_bf16(v, hi, lo);
  packed[idx] = hi;
  packed[(int64_t)rows * kpad + idx] = lo;
}

int tc_pack_istft(const float* kc, const float* ks, int n_fft, int f_in, int onesided, void* packed,
                  cudaStream_t stream, int transposed) {
  tc_forget_packed(packed);
  const int bn = tc_istft_bn(n_fft);
  const int rows = (n_fft + bn - 1) / bn * bn;
  const int kpad = tc_istft_k(f_in);
  const int64_t n = (int64_t)rows * kpad;
  pack_istft_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, stream>>>(
      kc, ks, n_fft, f_in, onesided, transposed, rows, kpad, (__nv_bfloat16*)packed);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

size_t tc_istft_planes_bytes(int64_t B, int64_t T, int f_in) {
  const int kpad = tc_istft_k(f_in);
  return tc_workspace_bytes(B, T * kpad, kpad, kpad, 0);
}

// X (B, F, T, 2) fp32 -> A planes: row g = b*T + t, column part*F + f (K-major), bf16 hi/lo.
__global__ void __launch_bounds__(256) istft_prep_kernel(const float* __restrict__ X, int f_in,
                                                         int64_t T, int kpad, int64_t plane_stride,
                                                         __nv_bfloat16* __restrict__ planes) {
  __shared__ float tile[2][32][33];
  const int64_t b = blockIdx.z;
  const int64_t t0 = (int64_t)blockIdx.x * 32;
  const int f0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const float* __restrict__ Xb = X + b * (int64_t)f_in * T * 2;
  for (int r = ty; r < 32; r += 8) {
    const int f = f0 + r;
    const int64_t t = t0 + tx;
    float2 v = make_float2(0.f, 0.f);
    if (f < f_in && t < T) v = *reinterpret_cast<const float2*>(Xb + ((int64_t)f * T + t) * 2);
    tile[0][r][tx] = v.x;
    tile[1][r][tx] = v.y;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int64_t t = t0 + r;
    const int f = f0 + tx;
    if (t < T && f < f_in) {
      const int64_t row = (b * T + t) * kpad;
#pragma unroll
      for (int part = 0; part < 2; ++part) {
        __nv_bfloat16 hi, lo;
        split_bf16(tile[part][tx][r], hi, lo);
        planes[row + part * f_in + f] = hi;
        planes[plane_stride + row + part * f_in + f] = lo;
      }
    }
  }
}

int tc_istft_prep(const float* X, int64_t B, int f_in, int64_t T, void* planes_v,
                  cudaStream_t stream) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  const int kpad = tc_istft_k(f_in);
  const SplitGeom g = split_geom(B, T * kpad, kpad, kpad, 0);
  __nv_bfloat16* planes = (__nv_bfloat16*)planes_v;
  // zero everything once when K has padding columns, else just the overhang rows
  if (kpad != 2 * f_in) {
    NNAB_CUDA_TRY(cudaMemsetAsync(planes, 0, (size_t)2 * g.plane_stride * sizeof(__nv_bfloat16), stream));
  } else {
    const int rc = zero_tail(planes, g, kpad, stream);
    if (rc) return rc;
  }
  dim3 grid((unsigned)ceil_div64(T, 32), (unsigned)((f_in + 31) / 32), (unsigned)B);
  istft_prep_kernel<<<grid, 256, 0, stream>>>(X, f_in, T, kpad, g.plane_stride, planes);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// ---------------------------------------------------------------------------
// Weight gradient dW[m, k] = sum_{b,t} G[m, (b,t)] * frame_{b,t}[k]   (m = re rows then im rows)
// as a GEMM on the same kernel: the gradient rows are the "signal" (plain-matrix rows of
// length G = B*T), the transposed frame matrix FT[k][(b,t)] takes the packed-basis slot.
// ---------------------------------------------------------------------------
int64_t tc_dw_gpad(int64_t B, int64_t T) { return (B * T + 63) / 64 * 64; }

size_t tc_dw_grad_planes_bytes(int64_t B, int64_t T, int F) {
  const int64_t gpad = tc_dw_gpad(B, T);
  return tc_workspace_bytes(1, (int64_t)2 * F * gpad, (int)gpad, (int)gpad, 0);
}
size_t tc_dw_frames_bytes(int64_t B, int64_t T, int K) {
  const int bn = tc_istft_bn(K);
  const size_t rows = (size_t)((K + bn - 1) / bn) * bn;
  return 2 * rows * (size_t)tc_dw_gpad(B, T) * sizeof(__nv_bfloat16) + 256;
}

// g (B, F, T, 2) -> rows part*F + f, columns b*T + t (bf16 hi/lo planes)
__global__ void __launch_bounds__(256) dw_prep_grad_kernel(const float* __restrict__ g, int F,
                                                           int64_t T, int64_t gpad,
                                                           int64_t plane_stride,
                                                           __nv_bfloat16* __restrict__ planes) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int f = blockIdx.y;
  const int64_t b = blockIdx.z;
  if (t >= T) return;
  const float2 v = *reinterpret_cast<const float2*>(g + (((int64_t)b * F + f) * T + t) * 2);
  const int64_t col = b * T + t;
  __nv_bfloat16 hi, lo;
  split_bf16(v.x, hi, lo);
  planes[(int64_t)f * gpad + col] = hi;
  planes[plane_stride + (int64_t)f * gpad + col] = lo;
  split_bf16(v.y, hi, lo);
  planes[(int64_t)(F + f) * gpad + col] = hi;
  planes[plane_stride + (int64_t)(F + f) * gpad + col] = lo;
}

int tc_dw_prep_grad(const float* g, int64_t B, int F, int64_t T, void* planes_v, cudaStream_t stream) {
  if (B > 65535 || F > 65535) return NNAB_EUNSUPPORTED;
  const int64_t gpad = tc_dw_gpad(B, T);
  const SplitGeom geo = split_geom(1, (int64_t)2 * F * gpad, (int)gpad, (int)gpad, 0);
  __nv_bfloat16* planes = (__nv_bfloat16*)planes_v;
  NNAB_CUDA_TRY(cudaMemsetAsync(planes, 0, (size_t)2 * geo.plane_stride * sizeof(__nv_bfloat16), stream));
  dim3 grid((unsigned)ceil_div64(T, 256), (unsigned)F, (unsigned)B);
  dw_prep_grad_kernel<<<grid, 256, 0, stream>>>(g, F, T, gpad, geo.plane_stride, planes);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// FT[k][b*T + t] = xpad[b, t*hop + k]   (packed-basis layout: [plane][rows][gpad])
__global__ void __launch_bounds__(256) dw_prep_frames_kernel(
    const float* __restrict__ x, int64_t L, int64_t x_pitch, int K, int hop, int pad, int pad_mode,
    int64_t T, int64_t G, int64_t gpad, int64_t rows, __nv_bfloat16* __restrict__ packed) {
  __shared__ float tile[32][33];
  const int64_t c0 = (int64_t)blockIdx.x * 32;
  const int k0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {  // r: column (frame) index in the tile, tx: k
    const int64_t c = c0 + r;
    const int k = k0 + tx;
    float v = 0.f;
    if (c < G && k < K) {
      const int64_t b = c / T, t = c - b * T;
      int64_t j = t * hop + k - pad;
      if (j < 0) j = (pad_mode == NNAB_PAD_REFLECT) ? -j : -1;
      else if (j >= L) j = (pad_mode == NNAB_PAD_REFLECT) ? 2 * (L - 1) - j : -1;
      if (j >= 0 && j < L) v = __ldg(x + b * x_pitch + j);
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {  // r: k index in the tile, tx: frame
    const int k = k0 + r;
    const int64_t c = c0 + tx;
    if (k < K && c < G) {
      __nv_bfloat16 hi, lo;
      split_bf16(tile[tx][r], hi, lo);
      packed[(int64_t)k * gpad + c] = hi;
      packed[rows * gpad + (int64_t)k * gpad + c] = lo;
    }
  }
}

int tc_dw_prep_frames(const float* x, int64_t B, int64_t L, int64_t x_pitch, int K, int hop, int pad,
                      int pad_mode, int64_t T, void* packed_v, cudaStream_t stream) {
  const int64_t G = B * T, gpad = tc_dw_gpad(B, T);
  const int bn = tc_istft_bn(K);
  const int64_t rows = (int64_t)((K + bn - 1) / bn) * bn;
  __nv_bfloat16* packed = (__nv_bfloat16*)packed_v;
  tc_forget_packed(packed_v);
  NNAB_CUDA_TRY(cudaMemsetAsync(packed, 0, (size_t)2 * rows * gpad * sizeof(__nv_bfloat16), stream));
  if ((K + 31) / 32 > 65535) return NNAB_EUNSUPPORTED;
  dim3 grid((unsigned)ceil_div64(G, 32), (unsigned)((K + 31) / 32));
  dw_prep_frames_kernel<<<grid, 256, 0, stream>>>(x, L, x_pitch, K, hop, pad, pad_mode, T, G, gpad,
                                                  rows, packed);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// Adjoint of nn.ReflectionPad1d / ConstantPad1d(pad): fold the gradient of the padded signal
// back onto the clip (mirror margins add onto samples 1..pad and L-1-pad..L-2).
__global__ void __launch_bounds__(256) unpad_adjoint_kernel(const float* __restrict__ gp,
                                                            int64_t gp_pitch, int64_t gp_len,
                                                            int pad, int pad_mode, int64_t L,
                                                            float* __restrict__ dx) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t b = blockIdx.y;
  if (j >= L) return;
  const float* __restrict__ g = gp + b * gp_pitch;
  auto at = [&](int64_t i) { return (i >= 0 && i < gp_len) ? g[i] : 0.f; };
  float v = at(pad + j);
  if (pad > 0 && pad_mode == NNAB_PAD_REFLECT) {
    if (j >= 1 && j <= pad) v += at(pad - j);
    if (j >= L - 1 - pad && j <= L - 2) v += at(pad + 2 * (L - 1) - j);
  }
  dx[b * L + j] = v;
}

int tc_unpad_adjoint(const float* gp, int64_t gp_pitch, int64_t gp_len, int64_t B, int pad,
                     int pad_mode, int64_t L, float* dx, cudaStream_t stream) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  if (B <= 0 || L <= 0) return NNAB_OK;
  dim3 grid((unsigned)ceil_div64(L, 256), (unsigned)B);
  unpad_adjoint_kernel<<<grid, 256, 0, stream>>>(gp, gp_pitch, gp_len, pad, pad_mode, L, dx);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// Divide the overlap-added frames by the window sum-square (utils.py:43-49; only where it
// exceeds 1e-10) and strip the centre padding: out[b, i] = ola[b, i + offset] / wss(i + offset).
__global__ void __launch_bounds__(256) istft_finalize_kernel(const float* __restrict__ ola,
                                                             int64_t ola_pitch,
                                                             const float* __restrict__ window,
                                                             int n_fft, int hop, int64_t T,
                                                             int64_t offset, float* __restrict__ out,
                                                             int64_t out_len) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t b = blockIdx.y;
  if (i >= out_len) return;
  const int64_t s = i + offset;
  int64_t t_hi = s / hop;
  if (t_hi > T - 1) t_hi = T - 1;
  float wss = 0.f;
  for (int64_t t = t_hi; t >= 0; --t) {
    const int64_t n = s - t * hop;
    if (n >= n_fft) break;
    const float w = __ldg(window + n);
    wss = fmaf(w, w, wss);
  }
  float v = ola[b * ola_pitch + s];
  if (wss > 1e-10f) v = v / wss;
  out[b * out_len + i] = v;
}

int tc_istft_finalize(const float* ola, int64_t ola_pitch, int64_t B, const float* window,
                      int n_fft, int hop, int64_t T, int64_t offset, float* out, int64_t out_len,
                      cudaStream_t stream) {
  if (B > 65535) return NNAB_EUNSUPPORTED;
  if (out_len <= 0 || B <= 0) return NNAB_OK;
  dim3 grid((unsigned)ceil_div64(out_len, 256), (unsigned)B);
  istft_finalize_kernel<<<grid, 256, 0, stream>>>(ola, ola_pitch, window, n_fft, hop, T, offset,
                                                  out, out_len);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// PTX wrappers: tc_ptx.cuh

// ---------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------
struct TcParams {
  int num_m_tiles, num_n_tiles, bn;
  int rows_mode;   // 1: A viewed as (rows x hop) matrix (BK | hop); 0: overlapping-stride map
  int hop;          // effective hop (hop * phases)
  int t_mul, t_add;  // output frame index = t * t_mul + t_add (frame phases)
  int k_splits;      // >1: every (m, n) tile is cut into k_splits K-chunks (FMT_RAW epilogue)
  int split4;        // EXPERIMENTAL (NNAB_SPLIT4=1): add the x_lo * w_lo term (4 MMAs per K16 step)
  int two_term;      // bf16 input: the A lo plane is zero -- neither loaded nor multiplied
  int64_t nv, t_slots, T;  // T = valid frames of this phase
  int kb_begin[TC_MAX_N_TILES];
  int kb_end[TC_MAX_N_TILES];
  EpiParams epi;
};

// Work order of a persistent worker: its u-th unit (unit = tile * ks + K-chunk), or -1 when done.
// Split-K partial sums are combined by ORDERED read-modify-writes (run-to-run identical; no atomics,
// no zero-fill of the scratch): all chunks of a tile go to the same worker, consecutively, so chunk c
// of a tile adds after chunk c-1 has stored, in program order of one thread.  (A balanced round-robin
// of the units with flag-ordered adds measured 2.04 ms vs 1.27 ms at cfg3: the chunks of a tile
// finish their MMAs together and their epilogues then serialise while holding TMEM buffers.)
__device__ __forceinline__ int sched_tile(int u, int worker, int n_workers, int num_mn, int ks) {
  const int mn = worker + (u / ks) * n_workers;
  return mn < num_mn ? mn * ks + (u % ks) : -1;
}

// tile index -> (m tile, n tile, k-block range); K-chunks of one (m, n) tile are adjacent
__device__ __forceinline__ void decode_tile(const TcParams& p, int tile, int& m_tile, int& n_tile,
                                            int& kb0, int& kb1) {
  const int ks = tile % p.k_splits;
  const int mn = tile / p.k_splits;
  m_tile = mn / p.num_n_tiles;
  n_tile = mn - m_tile * p.num_n_tiles;
  const int lo = p.kb_begin[n_tile], n = p.kb_end[n_tile] - lo;
  kb0 = lo + (int)(((int64_t)n * ks) / p.k_splits);
  kb1 = lo + (int)(((int64_t)n * (ks + 1)) / p.k_splits);
}

// Read one 128-frame x bn accumulator tile out of TMEM (this warp's 32 lanes =
// 32 consecutive frames) and emit it in the requested output format.
template <int FMT>
__device__ __forceinline__ void epilogue_tile(const TcParams& p, uint32_t trow, int64_t g,
                                              int n_tile, int half, int k_chunk, int mn_tile) {
      const int64_t b = g / p.t_slots;
      const int64_t tl = g - b * p.t_slots;
      const bool valid = (g < p.nv) && (tl < p.T);
      const int64_t t = tl * p.t_mul + p.t_add;  // frame index in the output
      const int f_base = n_tile * half;
      if constexpr (FMT == 8) {
        // ---- inverse STFT: window the frame's samples and overlap-add them ----
        float* dst = p.epi.out + b * p.epi.ola_pitch + t * p.epi.ola_hop;
        const int n_base = n_tile * (2 * half);
#pragma unroll 1
        for (int c0 = 0; c0 < 2 * half; c0 += 8) {
          uint32_t v[8];
          tmem_ld8(trow + (uint32_t)c0, v);
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int n = n_base + c0 + j;
              if (n < p.epi.F)  // F = n_fft samples per frame
                atomicAdd(dst + n, p.epi.scale != nullptr
                                       ? __uint_as_float(v[j]) * __ldg(p.epi.scale + n)
                                       : __uint_as_float(v[j]));
            }
          }
        }
      } else if constexpr (FMT == 7) {
        // ---- split-K partial sums: ordered read-modify-write of the raw planes (this thread owns
        // the element for every chunk of the tile; chunk 0 stores, later chunks add) ----
        float* rre = p.epi.raw + ((int64_t)b * p.epi.F) * p.epi.T + t;
#pragma unroll 1
        for (int c0 = 0; c0 < half; c0 += 8) {
          uint32_t re[8], im[8];
          tmem_ld8(trow + (uint32_t)c0, re);
          tmem_ld8(trow + (uint32_t)(half + c0), im);
          tmem_ld_wait();
          if (valid) {
            const int jmax = min(8, min(half - c0, p.epi.F - f_base - c0));
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (j < jmax) {
                float* q = rre + (int64_t)(f_base + c0 + j) * p.epi.T;
                float vr = __uint_as_float(re[j]), vi = __uint_as_float(im[j]);
                if (k_chunk > 0) { vr += __ldcg(q); vi += __ldcg(q + p.epi.raw_plane); }
                __stcg(q, vr);
                __stcg(q + p.epi.raw_plane, vi);
              }
          }
        }

      } else if constexpr (FMT == 6) {
        // ---- FIR decimator stage: this thread holds outputs n0 .. n0 + 2*half - 1 of clip b ----
        epilogue_decim(p.epi.dec, trow, b, tl, valid, half);
      } else if constexpr (FMT == 5) {
        // ---- fused banded filterbank: two running filter sums per frame ----
        float* mel = p.epi.out + ((int64_t)b * p.epi.n_fb) * p.epi.T + t;
        int cj0 = -1, cj1 = -1;
        float a0 = 0.f, a1 = 0.f;
        // rolled loop over 8-column TMEM loads: the body must stay I-cache resident
        // (a 32x unrolled version was ~80 KB of code per tile and fetch-stalled)
#pragma unroll 1
        for (int c0 = 0; c0 < half; c0 += 8) {
          uint32_t re[8], im[8];
          tmem_ld8(trow + (uint32_t)c0, re);
          tmem_ld8(trow + (uint32_t)(half + c0), im);
          tmem_ld_wait();
          const int jmax = min(8, min(half - c0, p.epi.F - f_base - c0));
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (j < jmax) {  // warp-uniform
              const int4 raw = __ldg(reinterpret_cast<const int4*>(p.epi.fb_table) + f_base + c0 + j);
              const float pw = epi_power(p.epi, __uint_as_float(re[j]), __uint_as_float(im[j]));
              if (raw.x != cj0) {
                if (raw.x == cj1) {
                  const int tj = cj0; cj0 = cj1; cj1 = tj;
                  const float ta = a0; a0 = a1; a1 = ta;
                } else {
                  if (cj0 >= 0 && valid) atomicAdd(mel + (int64_t)cj0 * p.epi.T, a0);
                  cj0 = raw.x; a0 = 0.f;
                }
              }
              if (raw.y != cj1) {
                if (cj1 >= 0 && valid) atomicAdd(mel + (int64_t)cj1 * p.epi.T, a1);
                cj1 = raw.y; a1 = 0.f;
              }
              a0 = fmaf(__int_as_float(raw.z), pw, a0);
              a1 = fmaf(__int_as_float(raw.w), pw, a1);
            }
          }
        }
        if (cj0 >= 0 && valid) atomicAdd(mel + (int64_t)cj0 * p.epi.T, a0);
        if (cj1 >= 0 && valid) atomicAdd(mel + (int64_t)cj1 * p.epi.T, a1);
      } else {
      constexpr int CH = (FMT == NNAB_FMT_COMPLEX || FMT == NNAB_FMT_PHASE_UNIT) ? 2 : 1;
      float* dst = p.epi.out + (((int64_t)b * p.epi.out_bins + p.epi.bin_offset) * p.epi.T + t) * CH;
      if constexpr (FMT == NNAB_FMT_MAGNITUDE || FMT == NNAB_FMT_COMPLEX) {
        // light per-bin code: 32 columns per TMEM load, fully unrolled
        for (int c0 = 0; c0 < half; c0 += 32) {
          uint32_t re[32], im[32];
          tmem_ld32(trow + (uint32_t)c0, re);
          tmem_ld32(trow + (uint32_t)(half + c0), im);
          tmem_ld_wait();
          if (valid) {
            const int jmax = min(32, min(half - c0, p.epi.F - f_base - c0));
            if (jmax == 32) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                epi_store_fmt<FMT>(p.epi, dst, f_base + c0 + j, __uint_as_float(re[j]),
                                   __uint_as_float(im[j]));
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < jmax)
                  epi_store_fmt<FMT>(p.epi, dst, f_base + c0 + j, __uint_as_float(re[j]),
                                     __uint_as_float(im[j]));
            }
          }
        }
      } else {
        // atan2f / sincosf / powf bodies: rolled loop over 8 columns keeps the code I-cache sized
#pragma unroll 1
        for (int c0 = 0; c0 < half; c0 += 8) {
          uint32_t re[8], im[8];
          tmem_ld8(trow + (uint32_t)c0, re);
          tmem_ld8(trow + (uint32_t)(half + c0), im);
          tmem_ld_wait();
          if (valid) {
            const int jmax = min(8, min(half - c0, p.epi.F - f_base - c0));
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (j < jmax)
                epi_store_fmt<FMT>(p.epi, dst, f_base + c0 + j, __uint_as_float(re[j]),
                                   __uint_as_float(im[j]));
          }
        }
      }
      }
}

template <int BK, int STAGES>
struct TcSmem {
  static constexpr uint32_t A_BYTES = TC_BM * BK * 2;
  static constexpr uint32_t B_BYTES = 256 * BK * 2;
  static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr uint32_t BAR_OFFSET = STAGES * STAGE_BYTES;
  static constexpr uint32_t TOTAL = BAR_OFFSET + 256 + 1024;  // + barriers + align slack
};

template <int BK, int STAGES, int FMT>
__global__ void __launch_bounds__(TC_THREADS, 1)
framed_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const TcParams p) {
  using S = TcSmem<BK, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + S::BAR_OFFSET;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 4);  // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int num_mn = p.num_m_tiles * p.num_n_tiles;
  const uint32_t b_tile_bytes = (uint32_t)p.bn * BK * 2;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = 0, tile; (tile = sched_tile(u, blockIdx.x, gridDim.x, num_mn, p.k_splits)) >= 0; ++u) {
        int m_tile, n_tile, kb0, kb1;
        decode_tile(p, tile, m_tile, n_tile, kb0, kb1);
        const int m0 = m_tile * TC_BM;
        const int n0 = n_tile * p.bn;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sb = base + stage * S::STAGE_BYTES;
          mbar_expect_tx(full_bar(stage), (p.two_term ? 1 : 2) * S::A_BYTES + 2 * b_tile_bytes);
          const int k0 = kb * BK;
          int c0 = k0, c1 = m0;
          if (p.rows_mode) {
            c1 = m0 + k0 / p.hop;
            c0 = k0 - (k0 / p.hop) * p.hop;
          }
          tma_load_3d(sb, &tm_a, full_bar(stage), c0, c1, 0);
          if (!p.two_term) tma_load_3d(sb + S::A_BYTES, &tm_a, full_bar(stage), c0, c1, 1);
          tma_load_3d(sb + 2 * S::A_BYTES, &tm_b, full_bar(stage), k0, n0, 0);
          tma_load_3d(sb + 2 * S::A_BYTES + S::B_BYTES, &tm_b, full_bar(stage), k0, n0, 1);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      // instruction descriptor: D=f32 (bit4), A=B=bf16 (bits 7,10), K-major, N>>3 @17, M>>4 @24
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.bn >> 3) << 17) |
                             ((uint32_t)(TC_BM >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int u = 0, tile; (tile = sched_tile(u, blockIdx.x, gridDim.x, num_mn, p.k_splits)) >= 0; ++u) {
        int m_tile, n_tile, kb0, kb1;
        decode_tile(p, tile, m_tile, n_tile, kb0, kb1);
        (void)m_tile;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * TC_ACC_STRIDE;
        uint32_t accumulate = 0;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t sb = base + stage * S::STAGE_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint32_t koff = (uint32_t)k * 32u;  // 16 bf16 along K inside the swizzle atom
            const uint64_t a_hi = make_smem_desc<BK>(sb + koff);
            const uint64_t a_lo = make_smem_desc<BK>(sb + S::A_BYTES + koff);
            const uint64_t b_hi = make_smem_desc<BK>(sb + 2 * S::A_BYTES + koff);
            const uint64_t b_lo = make_smem_desc<BK>(sb + 2 * S::A_BYTES + S::B_BYTES + koff);
            if (!p.two_term) {
              umma_bf16(d_tmem, a_lo, b_hi, idesc, accumulate);
              accumulate = 1u;
            }
            umma_bf16(d_tmem, a_hi, b_lo, idesc, accumulate);
            umma_bf16(d_tmem, a_hi, b_hi, idesc, 1u);
            accumulate = 1u;
          }
          umma_commit(empty_bar(stage));  // frees the smem slot when these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        umma_commit(tfull_bar(acc));  // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (warps 4..7 <-> TMEM lane quarters) =====================
    const int quarter = warp & 3;
    const int half = p.bn >> 1;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int u = 0, tile; (tile = sched_tile(u, blockIdx.x, gridDim.x, num_mn, p.k_splits)) >= 0; ++u) {
      int m_tile, n_tile, kb0, kb1;
      decode_tile(p, tile, m_tile, n_tile, kb0, kb1);
      (void)kb0; (void)kb1;
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const int64_t g = (int64_t)m_tile * TC_BM + quarter * 32 + lane;
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                            (uint32_t)acc * TC_ACC_STRIDE;
      epilogue_tile<FMT>(p, trow, g, n_tile, half, tile % p.k_splits, tile / p.k_splits);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}


// ---------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2): a cluster of two CTAs computes a
// 256-frame x bn tile.  Each CTA stages its own 128 A rows and HALF of the B
// tile (CTA 0: the re rows, CTA 1: the negated im rows), the leader issues
// M=256 MMAs that read B from both SMs, and every CTA keeps its 128 x bn
// accumulators in its own TMEM.  Per SM this halves the B operand reads and TMA
// fills — the shared-memory bandwidth that bounds the 1-CTA kernel at ~76 %.
// ---------------------------------------------------------------------------
template <int BK, int STAGES>
struct Tc2Smem {
  static constexpr uint32_t A_BYTES = TC_BM * BK * 2;
  static constexpr uint32_t B_BYTES = 128 * BK * 2;  // half of a bn <= 256 tile
  static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr uint32_t BAR_OFFSET = STAGES * STAGE_BYTES;
  static constexpr uint32_t TOTAL = BAR_OFFSET + 256 + 1024;
};

template <int BK, int STAGES, int FMT>
__global__ void __launch_bounds__(TC_THREADS, 1)
framed_tc2_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                  const TcParams p) {
  using S = Tc2Smem<BK, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + S::BAR_OFFSET;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };            // used in the leader
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };  // per CTA
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };       // per CTA
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };  // leader
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta = cluster_ctarank();  // 0 = leader
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 2);   // one arrive.expect_tx per CTA's producer
      mbar_init(empty_bar(s), 1);  // multicast commit from the leader
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 8);  // 4 epilogue warps x 2 CTAs
    }
    fence_barrier_init();
  }
  cluster_sync_all();  // peer barriers are initialised before any remote arrive / TMA credit
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, 512);
    tmem_relinquish_2sm();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int num_mn = p.num_m_tiles * p.num_n_tiles;  // num_m_tiles: 256-frame pairs
  const int halfn = p.bn >> 1;
  const uint32_t b_half_bytes = (uint32_t)halfn * BK * 2;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = 0, tile; (tile = sched_tile(u, pair, num_pairs, num_mn, p.k_splits)) >= 0; ++u) {
        int m_tile, n_tile, kb0, kb1;
        decode_tile(p, tile, m_tile, n_tile, kb0, kb1);
        const int m0 = m_tile * (2 * TC_BM) + (int)cta * TC_BM;
        const int n0 = n_tile * p.bn + (int)cta * halfn;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sb = base + stage * S::STAGE_BYTES;
          mbar_expect_tx_remote(full_bar(stage), 0, (p.two_term ? 1 : 2) * S::A_BYTES + 2 * b_half_bytes);
          const int k0 = kb * BK;
          int c0 = k0, c1 = m0;
          if (p.rows_mode) {
            c1 = m0 + k0 / p.hop;
            c0 = k0 - (k0 / p.hop) * p.hop;
          }
          tma_load_3d_2sm(sb, &tm_a, full_bar(stage), c0, c1, 0);
          if (!p.two_term) tma_load_3d_2sm(sb + S::A_BYTES, &tm_a, full_bar(stage), c0, c1, 1);
          tma_load_3d_2sm(sb + 2 * S::A_BYTES, &tm_b, full_bar(stage), k0, n0, 0);
          tma_load_3d_2sm(sb + 2 * S::A_BYTES + S::B_BYTES, &tm_b, full_bar(stage), k0, n0, 1);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (cta == 0 && elect_one()) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.bn >> 3) << 17) |
                             ((uint32_t)((2 * TC_BM) >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int u = 0, tile; (tile = sched_tile(u, pair, num_pairs, num_mn, p.k_splits)) >= 0; ++u) {
        int m_tile, n_tile, kb0, kb1;
        decode_tile(p, tile, m_tile, n_tile, kb0, kb1);
        (void)m_tile;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * TC_ACC_STRIDE;
        uint32_t accumulate = 0;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t sb = base + stage * S::STAGE_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint32_t koff = (uint32_t)k * 32u;
            const uint64_t a_hi = make_smem_desc<BK>(sb + koff);
            const uint64_t a_lo = make_smem_desc<BK>(sb + S::A_BYTES + koff);
            const uint64_t b_hi = make_smem_desc<BK>(sb + 2 * S::A_BYTES + koff);
            const uint64_t b_lo = make_smem_desc<BK>(sb + 2 * S::A_BYTES + S::B_BYTES + koff);
            if (!p.two_term) {
              if (p.split4) {  // smallest term first: fp32-like accuracy for the training forward
                umma_bf16_2sm(d_tmem, a_lo, b_lo, idesc, accumulate);
                accumulate = 1u;
              }
              umma_bf16_2sm(d_tmem, a_lo, b_hi, idesc, accumulate);
              accumulate = 1u;
            }
            umma_bf16_2sm(d_tmem, a_hi, b_lo, idesc, accumulate);
            umma_bf16_2sm(d_tmem, a_hi, b_hi, idesc, 1u);
            accumulate = 1u;
          }
          umma_commit_2sm(empty_bar(stage));
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        umma_commit_2sm(tfull_bar(acc));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (both CTAs, own 128 rows) =====================
    const int quarter = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int u = 0, tile; (tile = sched_tile(u, pair, num_pairs, num_mn, p.k_splits)) >= 0; ++u) {
      int m_tile, n_tile, kb0, kb1;
      decode_tile(p, tile, m_tile, n_tile, kb0, kb1);
      (void)kb0; (void)kb1;
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const int64_t g = (int64_t)m_tile * (2 * TC_BM) + (int64_t)cta * TC_BM + quarter * 32 + lane;
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                            (uint32_t)acc * TC_ACC_STRIDE;
      epilogue_tile<FMT>(p, trow, g, n_tile, halfn, tile % p.k_splits, tile / p.k_splits);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(tempty_bar(acc), 0);
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA leaves (or frees TMEM) while its peer may still touch it
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}


// ===========================================================================
// Per-K-block MMA width for banks
// whose rows have nested, centred supports (CQT1992v2).
//
// Packed rows are ordered in 8-bin groups, [re bins 8g..8g+7 | negated im of the same bins], so
// basis row r is accumulator column r and a K block that only the G longest groups reach needs
// an MMA of width N = 16 G: TMA fetches 8 G rows per CTA of the pair, the instruction descriptor
// carries N, the accumulation still lands in TMEM columns [0, N).  K blocks are visited in order
// of decreasing width, so the first MMA of a tile (accumulate = 0) initialises every column the
// tile will touch, and the epilogue of a split-K chunk reads only those.
// ===========================================================================
constexpr int VN_MAX_BLOCKS = 512;
struct VarNPlan {
  int n_blocks;              // active K blocks
  int n_chunks;              // split-K chunks (1 = none)
  int chunk_begin[17];       // chunk c = ordered blocks [chunk_begin[c], chunk_begin[c+1])
  uint16_t order[VN_MAX_BLOCKS];  // K block index (64 samples each), widest first
  uint8_t groups[VN_MAX_BLOCKS];  // 8-bin groups the block reaches (N = 16 * groups)
};

// packed[plane][row][k]: row = 16 g + 8 part + j  <->  bin 8 g + j, part 0 = re, 1 = negated im
__global__ void __launch_bounds__(256) pack_basis_varn_kernel(
    const float* __restrict__ w_re, const float* __restrict__ w_im, int F, int K, int rows, int kpad,
    __nv_bfloat16* __restrict__ packed) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int k8 = kpad / 8;
  if (idx >= (int64_t)rows * k8) return;
  const int r = (int)(idx / k8);
  const int k0 = (int)(idx % k8) * 8;
  const int f = (r >> 4) * 8 + (r & 7);
  const int part = (r >> 3) & 1;
  __align__(16) __nv_bfloat16 hi[8];
  __align__(16) __nv_bfloat16 lo[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = k0 + e;
    float v = 0.f;
    if (f < F && k < K)
      v = part == 0 ? __ldg(w_re + (int64_t)f * K + k) : -__ldg(w_im + (int64_t)f * K + k);
    split_bf16(v, hi[e], lo[e]);
  }
  const int64_t o = (int64_t)r * kpad + k0;
  *reinterpret_cast<uint4*>(packed + o) = *reinterpret_cast<const uint4*>(hi);
  *reinterpret_cast<uint4*>(packed + (int64_t)rows * kpad + o) = *reinterpret_cast<const uint4*>(lo);
}

// FMT: 0 Magnitude, 1 Complex, 3 PhaseUnit (direct), 7 split-K partial sums.
template <int FMT>
__device__ __forceinline__ void epilogue_tile_varn(const TcParams& p, uint32_t trow, int64_t g,
                                                   int n_groups, int k_chunk, int mn_tile) {
  const int64_t b = g / p.t_slots;
  const int64_t tl = g - b * p.t_slots;
  const bool valid = (g < p.nv) && (tl < p.T);
  const int64_t t = tl * p.t_mul + p.t_add;
  constexpr int CH = (FMT == NNAB_FMT_COMPLEX || FMT == NNAB_FMT_PHASE_UNIT) ? 2 : 1;
  float* dst = p.epi.out + (((int64_t)b * p.epi.out_bins + p.epi.bin_offset) * p.epi.T + t) * CH;
  float* rre = (FMT == 7) ? p.epi.raw + ((int64_t)b * p.epi.F) * p.epi.T + t : nullptr;
#pragma unroll 1
  for (int gi = 0; gi < n_groups; ++gi) {
    uint32_t re[8], im[8];
    tmem_ld8(trow + (uint32_t)(16 * gi), re);
    tmem_ld8(trow + (uint32_t)(16 * gi + 8), im);
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int f = 8 * gi + j;
        if (f < p.epi.F) {
          if constexpr (FMT == 7) {
            float* q = rre + (int64_t)f * p.epi.T;
            float vr = __uint_as_float(re[j]), vi = __uint_as_float(im[j]);
            if (k_chunk > 0) { vr += __ldcg(q); vi += __ldcg(q + p.epi.raw_plane); }  // ordered by chunk
            __stcg(q, vr);
            __stcg(q + p.epi.raw_plane, vi);
          } else {
            epi_store_fmt<FMT>(p.epi, dst, f, __uint_as_float(re[j]), __uint_as_float(im[j]));
          }
        }
      }
    }
  }
}

template <int FMT>
__global__ void __launch_bounds__(TC_THREADS, 1)
framed_tc2v_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b8,
                   const __grid_constant__ CUtensorMap tm_b32, const TcParams p,
                   const __grid_constant__ VarNPlan plan) {
  constexpr int BK = 64, STAGES = 3;
  using S = Tc2Smem<BK, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + S::BAR_OFFSET;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta = cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_b8);
    prefetch_tmap(&tm_b32);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 2);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 8);
    }
    fence_barrier_init();
  }
  cluster_sync_all();
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, 512);
    tmem_relinquish_2sm();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;


  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = 0, tile; (tile = sched_tile(u, pair, num_pairs, p.num_m_tiles, plan.n_chunks)) >= 0; ++u) {
        const int chunk = tile % plan.n_chunks;
        const int m_tile = tile / plan.n_chunks;
        const int m0 = m_tile * (2 * TC_BM) + (int)cta * TC_BM;
        for (int i = plan.chunk_begin[chunk]; i < plan.chunk_begin[chunk + 1]; ++i) {
          const int k0 = (int)plan.order[i] * BK;
          const int rows = 8 * (int)plan.groups[i];  // basis rows this CTA stages
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sb = base + stage * S::STAGE_BYTES;
          mbar_expect_tx_remote(full_bar(stage), 0,
                                (p.two_term ? 1 : 2) * S::A_BYTES + 2 * (uint32_t)rows * BK * 2);
          int c0 = k0, c1 = m0;
          if (p.rows_mode) {
            c1 = m0 + k0 / p.hop;
            c0 = k0 - (k0 / p.hop) * p.hop;
          }
          tma_load_3d_2sm(sb, &tm_a, full_bar(stage), c0, c1, 0);
          if (!p.two_term) tma_load_3d_2sm(sb + S::A_BYTES, &tm_a, full_bar(stage), c0, c1, 1);
          const int row0 = (int)cta * rows;
          const uint32_t bh = sb + 2 * S::A_BYTES, bl = bh + S::B_BYTES;
          int r = 0;
          for (; rows - r >= 32; r += 32) {
            tma_load_3d_2sm(bh + (uint32_t)r * BK * 2, &tm_b32, full_bar(stage), k0, row0 + r, 0);
            tma_load_3d_2sm(bl + (uint32_t)r * BK * 2, &tm_b32, full_bar(stage), k0, row0 + r, 1);
          }
          for (; r < rows; r += 8) {
            tma_load_3d_2sm(bh + (uint32_t)r * BK * 2, &tm_b8, full_bar(stage), k0, row0 + r, 0);
            tma_load_3d_2sm(bl + (uint32_t)r * BK * 2, &tm_b8, full_bar(stage), k0, row0 + r, 1);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (cta == 0 && elect_one()) {
      const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((2 * TC_BM) >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int u = 0, tile; (tile = sched_tile(u, pair, num_pairs, p.num_m_tiles, plan.n_chunks)) >= 0; ++u) {
        const int chunk = tile % plan.n_chunks;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * TC_ACC_STRIDE;
        uint32_t accumulate = 0;
        for (int i = plan.chunk_begin[chunk]; i < plan.chunk_begin[chunk + 1]; ++i) {
          const uint32_t idesc = idesc0 | ((uint32_t)(2 * (int)plan.groups[i]) << 17);  // N = 16 G
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t sb = base + stage * S::STAGE_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint32_t koff = (uint32_t)k * 32u;
            const uint64_t a_hi = make_smem_desc<BK>(sb + koff);
            const uint64_t a_lo = make_smem_desc<BK>(sb + S::A_BYTES + koff);
            const uint64_t b_hi = make_smem_desc<BK>(sb + 2 * S::A_BYTES + koff);
            const uint64_t b_lo = make_smem_desc<BK>(sb + 2 * S::A_BYTES + S::B_BYTES + koff);
            if (!p.two_term) {
              umma_bf16_2sm(d_tmem, a_lo, b_hi, idesc, accumulate);
              accumulate = 1u;
            }
            umma_bf16_2sm(d_tmem, a_hi, b_lo, idesc, accumulate);
            umma_bf16_2sm(d_tmem, a_hi, b_hi, idesc, 1u);
            accumulate = 1u;
          }
          umma_commit_2sm(empty_bar(stage));
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        umma_commit_2sm(tfull_bar(acc));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int u = 0, tile; (tile = sched_tile(u, pair, num_pairs, p.num_m_tiles, plan.n_chunks)) >= 0; ++u) {
      const int chunk = tile % plan.n_chunks;
      const int m_tile = tile / plan.n_chunks;
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const int64_t g = (int64_t)m_tile * (2 * TC_BM) + (int64_t)cta * TC_BM + quarter * 32 + lane;
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                            (uint32_t)acc * TC_ACC_STRIDE;
      // widest block of the chunk = its first: the columns this tile initialised
      epilogue_tile_varn<FMT>(p, trow, g, (int)plan.groups[plan.chunk_begin[chunk]], chunk, m_tile);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(tempty_bar(acc), 0);
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// Split-K finalize: raw (re, im) sums -> per-bin scale + output format (generic epilogue).
__global__ void __launch_bounds__(256) splitk_finalize_kernel(const EpiParams e, int64_t B) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int f = blockIdx.y;
  if (t >= e.T) return;
  for (int64_t b = blockIdx.z; b < B; b += gridDim.z) {
    const int64_t i = ((int64_t)b * e.F + f) * e.T + t;
    epi_store(e, b, f, t, e.raw[i], e.raw[e.raw_plane + i]);
  }
}

// Long kernels only: the scratch exists to bound the tensor-core accumulation length
// (its error grows with the number of accumulated MMAs) and to even out the tile count.
size_t tc_splitk_scratch_bytes(int64_t B, int F, int64_t T, int K) {
  if (K < 8192) return 0;
  return (size_t)2 * B * F * T * sizeof(float) + 256;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) ==
            cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

int encode_3d(CUtensorMap* map, void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                     uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1,
                     int bk) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_error_text("cuTensorMapEncodeTiled entry point not available");
    return NNAB_ECUDA;
  }
  cuuint64_t gdim[3] = {d0, d1, d2};
  cuuint64_t gstr[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {box0, box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapSwizzle sw = (bk == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char msg[200];
    snprintf(msg, sizeof(msg),
             "cuTensorMapEncodeTiled failed (%d): dims {%llu,%llu,%llu} strides {%llu,%llu} box {%u,%u}",
             (int)r, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
             (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, box0, box1);
    set_error_text(msg);
    return NNAB_ECUDA;
  }
  return NNAB_OK;
}

// 4-D bf16 map, SWIZZLE_128B, box {box0, box1, box2, 1}; strides in bytes for dims 1..3 (any order of
// magnitude: a dimension may step by less than the extent of the one below it -- overlapping views)
int encode_4d(CUtensorMap* map, void* base, const uint64_t dims[4], const uint64_t strides[3],
              const uint32_t box[3]) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_error_text("cuTensorMapEncodeTiled entry point not available");
    return NNAB_ECUDA;
  }
  cuuint64_t gdim[4] = {dims[0], dims[1], dims[2], dims[3]};
  cuuint64_t gstr[3] = {strides[0], strides[1], strides[2]};
  cuuint32_t bx[4] = {box[0], box[1], box[2], 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, gdim, gstr, bx, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char msg[240];
    snprintf(msg, sizeof(msg),
             "cuTensorMapEncodeTiled(4d) failed (%d): dims {%llu,%llu,%llu,%llu} strides {%llu,%llu,%llu}",
             (int)r, (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2],
             (unsigned long long)dims[3], (unsigned long long)strides[0], (unsigned long long)strides[1],
             (unsigned long long)strides[2]);
    set_error_text(msg);
    return NNAB_ECUDA;
  }
  return NNAB_OK;
}

template <int BK, int STAGES, int FMT>
static int launch_tc_kernel_fmt(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& prm,
                                int grid, cudaStream_t stream) {
  using S = TcSmem<BK, STAGES>;
  // the attribute is per device: one process may drive several GPUs (torch.nn.DataParallel)
  static std::atomic<uint64_t> configured_devs{0};
  int cfg_dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&cfg_dev));
  const bool configured = (configured_devs.load(std::memory_order_relaxed) >> (cfg_dev & 63)) & 1u;
  if (!configured) {
    NNAB_CUDA_TRY(cudaFuncSetAttribute(framed_tc_kernel<BK, STAGES, FMT>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
    configured_devs.fetch_or(1ull << (cfg_dev & 63), std::memory_order_relaxed);
  }
  framed_tc_kernel<BK, STAGES, FMT><<<grid, TC_THREADS, S::TOTAL, stream>>>(ma, mb, prm);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

template <int BK, int STAGES, int FMT>
static int launch_tc2_kernel_fmt(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& prm,
                                 int n_pairs, cudaStream_t stream) {
  using S = Tc2Smem<BK, STAGES>;
  // the attribute is per device: one process may drive several GPUs (torch.nn.DataParallel)
  static std::atomic<uint64_t> configured_devs{0};
  int cfg_dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&cfg_dev));
  const bool configured = (configured_devs.load(std::memory_order_relaxed) >> (cfg_dev & 63)) & 1u;
  if (!configured) {
    NNAB_CUDA_TRY(cudaFuncSetAttribute(framed_tc2_kernel<BK, STAGES, FMT>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
    configured_devs.fetch_or(1ull << (cfg_dev & 63), std::memory_order_relaxed);
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * n_pairs));
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  NNAB_CUDA_TRY(cudaLaunchKernelEx(&cfg, framed_tc2_kernel<BK, STAGES, FMT>, ma, mb, prm));
  count_launch();
  return NNAB_OK;
}

template <int BK, int STAGES>
static int launch_tc2_kernel(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& prm,
                             int n_pairs, cudaStream_t stream) {
  switch (prm.epi.fmt) {
    case NNAB_FMT_MAGNITUDE: return launch_tc2_kernel_fmt<BK, STAGES, 0>(ma, mb, prm, n_pairs, stream);
    case NNAB_FMT_COMPLEX: return launch_tc2_kernel_fmt<BK, STAGES, 1>(ma, mb, prm, n_pairs, stream);
    case NNAB_FMT_PHASE_ANGLE: return launch_tc2_kernel_fmt<BK, STAGES, 2>(ma, mb, prm, n_pairs, stream);
    case NNAB_FMT_PHASE_UNIT: return launch_tc2_kernel_fmt<BK, STAGES, 3>(ma, mb, prm, n_pairs, stream);
    case FMT_POWER: return launch_tc2_kernel_fmt<BK, STAGES, 4>(ma, mb, prm, n_pairs, stream);
    case FMT_FBANK: return launch_tc2_kernel_fmt<BK, STAGES, 5>(ma, mb, prm, n_pairs, stream);
    case FMT_DECIM: return launch_tc2_kernel_fmt<BK, STAGES, 6>(ma, mb, prm, n_pairs, stream);
    case FMT_RAW: return launch_tc2_kernel_fmt<BK, STAGES, 7>(ma, mb, prm, n_pairs, stream);
    case FMT_OLA: return launch_tc2_kernel_fmt<BK, STAGES, 8>(ma, mb, prm, n_pairs, stream);
    case FMT_REALPAIR: return launch_tc2_kernel_fmt<BK, STAGES, 9>(ma, mb, prm, n_pairs, stream);
    default: return NNAB_EINVAL;
  }
}

template <int BK, int STAGES>
static int launch_tc_kernel(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& prm,
                            int grid, cudaStream_t stream) {
  switch (prm.epi.fmt) {
    case NNAB_FMT_MAGNITUDE: return launch_tc_kernel_fmt<BK, STAGES, 0>(ma, mb, prm, grid, stream);
    case NNAB_FMT_COMPLEX: return launch_tc_kernel_fmt<BK, STAGES, 1>(ma, mb, prm, grid, stream);
    case NNAB_FMT_PHASE_ANGLE: return launch_tc_kernel_fmt<BK, STAGES, 2>(ma, mb, prm, grid, stream);
    case NNAB_FMT_PHASE_UNIT: return launch_tc_kernel_fmt<BK, STAGES, 3>(ma, mb, prm, grid, stream);
    case FMT_POWER: return launch_tc_kernel_fmt<BK, STAGES, 4>(ma, mb, prm, grid, stream);
    case FMT_FBANK: return launch_tc_kernel_fmt<BK, STAGES, 5>(ma, mb, prm, grid, stream);
    case FMT_DECIM: return launch_tc_kernel_fmt<BK, STAGES, 6>(ma, mb, prm, grid, stream);
    case FMT_RAW: return launch_tc_kernel_fmt<BK, STAGES, 7>(ma, mb, prm, grid, stream);
    case FMT_OLA: return launch_tc_kernel_fmt<BK, STAGES, 8>(ma, mb, prm, grid, stream);
    case FMT_REALPAIR: return launch_tc_kernel_fmt<BK, STAGES, 9>(ma, mb, prm, grid, stream);
    default: return NNAB_EINVAL;
  }
}


// ---------------------------------------------------------------------------
// layout of a packed basis, keyed by its device pointer.  Every function that produces a buffer for the
// `packed` argument of launch_framed_tc sets (or clears) the tag, so a recycled address cannot carry a
// stale layout.
// ---------------------------------------------------------------------------
static std::mutex g_pack_mu;
static std::unordered_map<const void*, int> g_pack_kind;

int packed_kind(const void* packed) {
  std::lock_guard<std::mutex> lk(g_pack_mu);
  auto it = g_pack_kind.find(packed);
  return it == g_pack_kind.end() ? PACK_DENSE : it->second;
}

void mark_packed(const void* packed, int kind) {
  std::lock_guard<std::mutex> lk(g_pack_mu);
  if (kind == PACK_DENSE) g_pack_kind.erase(packed);
  else g_pack_kind[packed] = kind;
}

void tc_forget_packed(const void* packed) { mark_packed(packed, PACK_DENSE); }


// ---------------------------------------------------------------------------
// per-K-block MMA width, host side (layout NNAB_LAYOUT_GROUPS; NNAB_VARN=0 forces dense)
// ---------------------------------------------------------------------------
bool tc_varn_enabled() {
  const char* e = getenv("NNAB_VARN");
  return e != nullptr && atoi(e) == 1;
}

bool tc_varn_basis_ok(int F, int K) { return F >= 1 && F <= 128 && K >= 64 && K <= 64 * VN_MAX_BLOCKS; }

int tc_pack_basis_varn(const float* w_re, const float* w_im, int F, int K, void* packed,
                       cudaStream_t stream) {
  if (!tc_varn_basis_ok(F, K)) return NNAB_EINVAL;
  const int rows = 16 * ((F + 7) / 8);
  const int kpad = round_up_i(K, 64);
  const int64_t threads = (int64_t)rows * (kpad / 8);
  pack_basis_varn_kernel<<<(unsigned)ceil_div64(threads, 256), 256, 0, stream>>>(
      w_re, w_im, F, K, rows, kpad, (__nv_bfloat16*)packed);
  NNAB_LAUNCH_CHECK();
  mark_packed(packed, PACK_VARN);
  return NNAB_OK;
}

// Pure host: which K blocks are touched, by how many 8-bin groups, in which order, and how the
// ordered list is cut into split-K chunks of equal modelled cost (max(N, 64) per block: below
// N = 64 the A-operand reads, not the MMA, set the pace).  Returns NNAB_OK or NNAB_EUNSUPPORTED.
int tc_varn_plan(const int32_t* k_begin, const int32_t* k_end, int F, int K, int want_chunks,
                 VarNPlan* plan) {
  const int nkb = (K + 63) / 64;
  if (nkb > VN_MAX_BLOCKS || F > 128 || F < 1) return NNAB_EUNSUPPORTED;
  std::vector<std::pair<int, int>> blocks;  // (groups, kb)
  for (int kb = 0; kb < nkb; ++kb) {
    int gmax = 0;
    for (int f = 0; f < F; ++f) {
      const int lo = k_begin ? k_begin[f] : 0, hi = k_end ? k_end[f] : K;
      if (hi > lo && hi > kb * 64 && lo < kb * 64 + 64) gmax = std::max(gmax, f / 8 + 1);
    }
    if (gmax > 0) blocks.push_back({gmax, kb});
  }
  if (blocks.empty()) blocks.push_back({(F + 7) / 8, 0});
  std::stable_sort(blocks.begin(), blocks.end(),
                   [](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.first > b.first; });
  plan->n_blocks = (int)blocks.size();
  int64_t total = 0;
  for (int i = 0; i < plan->n_blocks; ++i) {
    plan->groups[i] = (uint8_t)blocks[i].first;
    plan->order[i] = (uint16_t)blocks[i].second;
    total += std::max(16 * blocks[i].first, 64);
  }
  int chunks = want_chunks < 1 ? 1 : (want_chunks > 16 ? 16 : want_chunks);
  if (chunks > plan->n_blocks) chunks = plan->n_blocks;
  plan->n_chunks = chunks;
  plan->chunk_begin[0] = 0;
  int64_t acc = 0;
  int c = 1;
  for (int i = 0; i < plan->n_blocks && c < chunks; ++i) {
    acc += std::max(16 * (int)plan->groups[i], 64);
    // close chunk c-1 once its share of the cost is reached, leaving >= 1 block per later chunk
    if (acc * chunks >= total * c && plan->n_blocks - (i + 1) >= chunks - c) plan->chunk_begin[c++] = i + 1;
  }
  while (c < chunks) { plan->chunk_begin[c] = plan->n_blocks - (chunks - c); ++c; }
  plan->chunk_begin[chunks] = plan->n_blocks;
  for (int k = chunks + 1; k < 17; ++k) plan->chunk_begin[k] = plan->n_blocks;
  return NNAB_OK;
}

// host-only view of the plan for tests / tooling
int tc_varn_plan_export(const int32_t* k_begin, const int32_t* k_end, int F, int K, int want_chunks,
                        int32_t* order, int32_t* groups, int32_t* chunk_begin, int32_t* n_blocks,
                        int32_t* n_chunks) {
  VarNPlan plan;
  const int rc = tc_varn_plan(k_begin, k_end, F, K, want_chunks, &plan);
  if (rc) return rc;
  *n_blocks = plan.n_blocks;
  *n_chunks = plan.n_chunks;
  for (int i = 0; i < plan.n_blocks; ++i) { order[i] = plan.order[i]; groups[i] = plan.groups[i]; }
  for (int c = 0; c <= plan.n_chunks; ++c) chunk_begin[c] = plan.chunk_begin[c];
  return NNAB_OK;
}

static bool varn_problem_ok(const FramedProblem& q) {
  if (!tc_varn_basis_ok(q.F, q.K)) return false;
  if (num_phases(q.hop) != 1 || q.presplit != nullptr) return false;
  if (q.bin_offset != 0 || q.out_bins != q.F) return false;
  return q.fmt == NNAB_FMT_MAGNITUDE || q.fmt == NNAB_FMT_COMPLEX || q.fmt == NNAB_FMT_PHASE_UNIT;
}

template <int FMT>
static int launch_tc2v_fmt(const CUtensorMap& ma, const CUtensorMap& mb8, const CUtensorMap& mb32,
                           const TcParams& prm, const VarNPlan& plan, int n_pairs,
                           cudaStream_t stream) {
  using S = Tc2Smem<64, 3>;
  // the attribute is per device: one process may drive several GPUs (torch.nn.DataParallel)
  static std::atomic<uint64_t> configured_devs{0};
  int cfg_dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&cfg_dev));
  const bool configured = (configured_devs.load(std::memory_order_relaxed) >> (cfg_dev & 63)) & 1u;
  if (!configured) {
    NNAB_CUDA_TRY(cudaFuncSetAttribute(framed_tc2v_kernel<FMT>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
    configured_devs.fetch_or(1ull << (cfg_dev & 63), std::memory_order_relaxed);
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * n_pairs));
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  NNAB_CUDA_TRY(cudaLaunchKernelEx(&cfg, framed_tc2v_kernel<FMT>, ma, mb8, mb32, prm, plan));
  count_launch();
  return NNAB_OK;
}

static int launch_framed_tc_varn(const FramedProblem& q, const void* packed, void* workspace,
                                 size_t ws_bytes, cudaStream_t stream) {
  if (!varn_problem_ok(q)) return NNAB_EINVAL;  // the basis was packed for this kernel only
  {
    // same packed layout, A operand read in place from one tall block per column (tct_kernels.cu)
    const int trc = launch_framed_tc_tall(q, packed, workspace, ws_bytes, stream);
    if (trc != NNAB_EUNSUPPORTED) return trc;
  }
  const size_t need = tc_workspace_bytes(q.B, q.L, q.K, q.hop, q.pad);
  if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  if (q.B > 65535) return NNAB_EUNSUPPORTED;
  const SplitGeom g = split_geom(q.B, q.L, q.K, q.hop, q.pad);
  const int kpad = round_up_i(q.K, 64);
  const int rows_w = 16 * ((q.F + 7) / 8);
  __nv_bfloat16* planes =
      reinterpret_cast<__nv_bfloat16*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  const bool two = two_term(q);
  int rc = zero_tail(planes, g, q.hop, stream, two);
  if (rc) return rc;
  const int64_t clip_pitch = g.t_slots * q.hop;
  if ((rc = launch_pad_split(q.x, q.x_dtype, q.B, q.L, q.x_pitch, q.pad, q.pad_mode, 0, clip_pitch,
                             g.plane_stride, planes, two, stream)))
    return rc;

  // split-K only with the caller's raw scratch (long kernels): <= 64 K blocks per accumulator
  VarNPlan plan;
  {
    VarNPlan probe;
    if ((rc = tc_varn_plan(q.h_k_begin, q.h_k_end, q.F, q.K, 1, &probe))) return rc;
    int ks = 1;
    if (q.raw != nullptr) {
      ks = (probe.n_blocks + 63) / 64;
      if (ks > 16) ks = 16;
    }
    if ((rc = tc_varn_plan(q.h_k_begin, q.h_k_end, q.F, q.K, ks, &plan))) return rc;
  }

  int dev = 0, sms = 148;
  NNAB_CUDA_TRY(cudaGetDevice(&dev));
  NNAB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  sms -= sm_reserve();
  if (sms < 2) sms = 2;

  CUtensorMap ma, mb8, mb32;
  const int rows_mode = (q.hop % 64 == 0) ? 1 : 0;
  if (rows_mode)
    rc = encode_3d(&ma, planes, (uint64_t)q.hop, (uint64_t)g.rows, 2, (uint64_t)q.hop * 2,
                   (uint64_t)g.plane_stride * 2, 64, TC_BM, 64);
  else
    rc = encode_3d(&ma, planes, (uint64_t)kpad, (uint64_t)g.nv, 2, (uint64_t)q.hop * 2,
                   (uint64_t)g.plane_stride * 2, 64, TC_BM, 64);
  if (rc) return rc;
  if ((rc = encode_3d(&mb8, const_cast<void*>(packed), (uint64_t)kpad, (uint64_t)rows_w, 2,
                      (uint64_t)kpad * 2, (uint64_t)rows_w * kpad * 2, 64, 8, 64)))
    return rc;
  if ((rc = encode_3d(&mb32, const_cast<void*>(packed), (uint64_t)kpad, (uint64_t)rows_w, 2,
                      (uint64_t)kpad * 2, (uint64_t)rows_w * kpad * 2, 64, 32, 64)))
    return rc;

  TcParams prm{};
  prm.num_n_tiles = 1;
  prm.bn = rows_w;
  prm.rows_mode = rows_mode;
  prm.hop = q.hop;
  prm.nv = g.nv;
  prm.t_slots = g.t_slots;
  prm.t_mul = 1;
  prm.t_add = 0;
  prm.T = q.T;
  prm.k_splits = plan.n_chunks;
  prm.two_term = two ? 1 : 0;
  prm.epi.scale = q.scale; prm.epi.scale_all = q.scale_all; prm.epi.fmt = q.fmt;
  prm.epi.eps = q.eps; prm.epi.power = q.power; prm.epi.out = q.out; prm.epi.T = q.T;
  prm.epi.out_bins = q.out_bins; prm.epi.bin_offset = q.bin_offset; prm.epi.F = q.F;
  prm.epi.fb_table = nullptr; prm.epi.n_fb = 0;
  prm.epi.dec = q.dec;
  prm.epi.raw = nullptr; prm.epi.raw_plane = 0;
  prm.epi.ola_pitch = 0; prm.epi.ola_hop = 0;
  EpiParams final_epi = prm.epi;
  const bool split = plan.n_chunks > 1;
  if (split) {
    float* raw = reinterpret_cast<float*>(((uintptr_t)q.raw + 255) & ~(uintptr_t)255);
    const int64_t plane = (int64_t)q.B * q.F * q.T;
    prm.epi.fmt = FMT_RAW;
    prm.epi.raw = raw;
    prm.epi.raw_plane = plane;
    final_epi.raw = raw;
    final_epi.raw_plane = plane;
  }
  prm.num_m_tiles = (int)ceil_div64(g.nv, 2 * TC_BM);
  const int64_t ptiles = (int64_t)prm.num_m_tiles * plan.n_chunks;
  const int n_pairs = (int)(ptiles < sms / 2 ? ptiles : sms / 2);
  {
    double cols = 0.0;
    for (int i = 0; i < plan.n_blocks; ++i) cols += 16.0 * plan.groups[i] * 64.0;
    add_exec_flops((two ? 2.0 : 3.0) * 2.0 * (double)prm.num_m_tiles * (2 * TC_BM) * cols);
  }
  switch (prm.epi.fmt) {
    case NNAB_FMT_MAGNITUDE: rc = launch_tc2v_fmt<0>(ma, mb8, mb32, prm, plan, n_pairs, stream); break;
    case NNAB_FMT_COMPLEX: rc = launch_tc2v_fmt<1>(ma, mb8, mb32, prm, plan, n_pairs, stream); break;
    case NNAB_FMT_PHASE_UNIT: rc = launch_tc2v_fmt<3>(ma, mb8, mb32, prm, plan, n_pairs, stream); break;
    case FMT_RAW: rc = launch_tc2v_fmt<7>(ma, mb8, mb32, prm, plan, n_pairs, stream); break;
    default: rc = NNAB_EINVAL;
  }
  if (rc) return rc;
  if (split) {
    dim3 grid((unsigned)ceil_div64(q.T, 256), (unsigned)q.F, (unsigned)(q.B < 64 ? q.B : 64));
    splitk_finalize_kernel<<<grid, 256, 0, stream>>>(final_epi, q.B);
    NNAB_LAUNCH_CHECK();
  }
  return NNAB_OK;
}

int launch_framed_tc(const FramedProblem& q, const void* packed, void* workspace, size_t ws_bytes,
                     cudaStream_t stream) {
  if (q.B <= 0 || q.T <= 0 || q.F <= 0) return NNAB_OK;
  if (packed == nullptr) return NNAB_EINVAL;
  if (packed_kind(packed) == PACK_BLOCK)
    return launch_framed_tc_block(q, packed, workspace, ws_bytes, stream);
  if (packed_kind(packed) == PACK_VARN)
    return launch_framed_tc_varn(q, packed, workspace, ws_bytes, stream);
  if (q.presplit == nullptr) {
    const size_t need = tc_workspace_bytes(q.B, q.L, q.K, q.hop, q.pad);
    if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  } else if (num_phases(q.hop) != 1) {
    return NNAB_EALIGN;  // pre-split planes exist for one frame phase only
  }
  if (q.B > 65535) return NNAB_EUNSUPPORTED;

  int bk = 64;
  if (const char* e = getenv("NNAB_TC_BK")) bk = atoi(e) == 32 ? 32 : 64;

  const int n_ph = num_phases(q.hop);
  const int hop_eff = q.hop * n_ph;
  SplitGeom g = split_geom(q.B, q.L, q.K, q.hop, q.pad);
  if (q.presplit != nullptr && q.presplit_t_slots > 0) {
    // caller-defined plane geometry (pyramid levels shared with the FIR stage): frame g of the batch
    // still starts at element g * hop, with presplit_t_slots frames per clip slot
    g.t_slots = q.presplit_t_slots;
    g.nv = q.B * g.t_slots;
    g.plane_stride = q.presplit_plane_stride;
    g.rows = g.plane_stride / hop_eff;
    if (g.rows < g.nv) return NNAB_EINVAL;
  }
  const int kpad = round_up_i(q.K, 64);
  // FMT_OLA: the N axis is the frame's n_fft output samples (q.F), not (re | im) bin pairs
  const int bn = (q.fmt == FMT_OLA) ? tc_istft_bn(q.F) : choose_bn(q.F);
  const int n_tiles = (q.fmt == FMT_OLA) ? (q.F + bn - 1) / bn : (2 * q.F + bn - 1) / bn;
  const int rows_w = n_tiles * bn;
  __nv_bfloat16* planes =
      q.presplit != nullptr
          ? reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(q.presplit))
          : reinterpret_cast<__nv_bfloat16*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);

  // K overhang rows past the last clip must be finite zeros (the basis is zero-padded there)
  const int64_t clip_pitch = g.t_slots * hop_eff;
  const bool two = two_term(q);
  if (q.presplit == nullptr) {
    const int zrc = zero_tail(planes, g, hop_eff, stream, two);
    if (zrc) return zrc;
  }

  // ---- tensor maps (shared by all phases) -------------------------------------------
  // CTA pairs (cta_group::2) by default when there are enough 256-frame tiles to fill the
  // 74 SM pairs; NNAB_TC_CTA=1|2 overrides (debugging / A-B measurements).
  int dev = 0, sms = 148;
  NNAB_CUDA_TRY(cudaGetDevice(&dev));
  NNAB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  sms -= sm_reserve();  // SMs left to a concurrent collective (nnab_set_sm_reserve)
  if (sms < 2) sms = 2;
  int cta_group = (ceil_div64(g.nv, 2 * TC_BM) * n_tiles >= sms / 2) ? 2 : 1;
  if (const char* e = getenv("NNAB_TC_CTA")) cta_group = atoi(e) == 2 ? 2 : 1;
  if (cta_group == 2) bk = 64;
  CUtensorMap ma, mb;
  const int rows_mode = (hop_eff % bk == 0) ? 1 : 0;
  int rc;
  if (rows_mode) {
    rc = encode_3d(&ma, planes, (uint64_t)hop_eff, (uint64_t)g.rows, 2, (uint64_t)hop_eff * 2,
                   (uint64_t)g.plane_stride * 2, bk, TC_BM, bk);
  } else {
    // overlapping rows: row g starts at element g*hop_eff and is kpad long
    rc = encode_3d(&ma, planes, (uint64_t)kpad, (uint64_t)g.nv, 2, (uint64_t)hop_eff * 2,
                   (uint64_t)g.plane_stride * 2, bk, TC_BM, bk);
  }
  if (rc) return rc;
  rc = encode_3d(&mb, const_cast<void*>(packed), (uint64_t)kpad, (uint64_t)rows_w, 2,
                 (uint64_t)kpad * 2, (uint64_t)rows_w * kpad * 2, bk,
                 cta_group == 2 ? bn / 2 : bn, bk);
  if (rc) return rc;

  // ---- parameters -------------------------------------------------------------------
  TcParams prm;
  prm.num_n_tiles = n_tiles;
  prm.bn = bn;
  prm.rows_mode = rows_mode;
  prm.hop = hop_eff;
  prm.nv = g.nv;
  prm.t_slots = g.t_slots;
  prm.t_mul = n_ph;
  {
    const char* e4 = getenv("NNAB_SPLIT4");
    prm.split4 = (e4 != nullptr && atoi(e4) == 1) ? 1 : 0;  // CTA-pair kernel only
  }
  prm.two_term = two ? 1 : 0;
  const int nkb = kpad / bk;
  const int half = bn / 2;
  for (int tl = 0; tl < n_tiles; ++tl) {
    int lo = 0, hi = (q.K + bk - 1) / bk;
    if (q.h_k_begin != nullptr && q.h_k_end != nullptr) {
      int klo = q.K, khi = 0;
      for (int f = tl * half; f < q.F && f < (tl + 1) * half; ++f)
        if (q.h_k_end[f] > q.h_k_begin[f]) {
          klo = q.h_k_begin[f] < klo ? q.h_k_begin[f] : klo;
          khi = q.h_k_end[f] > khi ? q.h_k_end[f] : khi;
        }
      if (khi > klo) {
        lo = klo / bk;
        hi = (khi + bk - 1) / bk;
      } else {
        lo = 0;
        hi = 1;
      }
    }
    if (hi > nkb) hi = nkb;
    if (lo >= hi) lo = hi - 1;
    prm.kb_begin[tl] = lo;
    prm.kb_end[tl] = hi;
  }
  prm.epi.scale = q.scale; prm.epi.scale_all = q.scale_all; prm.epi.fmt = q.fmt;
  prm.epi.eps = q.eps; prm.epi.power = q.power; prm.epi.out = q.out; prm.epi.T = q.T;
  prm.epi.out_bins = q.out_bins; prm.epi.bin_offset = q.bin_offset; prm.epi.F = q.F;
  prm.epi.fb_table = q.fb_table; prm.epi.n_fb = q.n_fb;
  prm.epi.dec = q.dec;
  prm.epi.raw = nullptr; prm.epi.raw_plane = 0;
  prm.epi.ola_pitch = q.ola_pitch; prm.epi.ola_hop = q.ola_hop;
  prm.k_splits = 1;
  if (q.fmt == FMT_FBANK && (q.fb_table == nullptr || q.n_fb <= 0)) return NNAB_EINVAL;
  if (q.fmt == FMT_DECIM && (bn != 128 || n_tiles != 1)) return NNAB_EINVAL;

  if (q.fmt == FMT_OLA && q.k_splits_hint > 1) {  // the OLA atomics accumulate K chunks as is
    int min_range = nkb;
    for (int tl = 0; tl < n_tiles; ++tl) {
      const int r = prm.kb_end[tl] - prm.kb_begin[tl];
      min_range = r < min_range ? r : min_range;
    }
    prm.k_splits = q.k_splits_hint < min_range ? q.k_splits_hint : min_range;
    if (prm.k_splits < 1) prm.k_splits = 1;
  }

  // ---- split-K (long kernels, caller supplied the raw scratch) ---------------------------
  EpiParams final_epi = prm.epi;
  bool split = false;
  if (q.raw != nullptr && q.fmt != FMT_FBANK && q.fmt != FMT_DECIM && q.fmt != FMT_OLA &&
      q.bin_offset == 0 &&
      q.out_bins == q.F) {
    int min_range = nkb;
    for (int tl = 0; tl < n_tiles; ++tl) {
      const int r = prm.kb_end[tl] - prm.kb_begin[tl];
      min_range = r < min_range ? r : min_range;
    }
    int ks = (min_range + 63) / 64;  // <= 64 k-blocks (4096 taps) per accumulator
    if (ks > 16) ks = 16;
    if (ks > min_range) ks = min_range;
    if (ks > 1) {
      split = true;
      prm.k_splits = ks;
      float* raw = reinterpret_cast<float*>(((uintptr_t)q.raw + 255) & ~(uintptr_t)255);
      const int64_t plane = (int64_t)q.B * q.F * q.T;
        prm.epi.fmt = FMT_RAW;
      prm.epi.raw = raw;
      prm.epi.raw_plane = plane;
      final_epi.raw = raw;
      final_epi.raw_plane = plane;
    }
  }

  // ---- one pad/split + GEMM pass per frame phase ----------------------------------------
  for (int ph = 0; ph < n_ph; ++ph) {
    if (ph >= q.T) break;
    prm.t_add = ph;
    prm.T = (q.T - ph + n_ph - 1) / n_ph;  // frames t = ph, ph + n_ph, ... < T
    if (q.presplit == nullptr &&
        (rc = launch_pad_split(q.x, q.x_dtype, q.B, q.L, q.x_pitch, q.pad, q.pad_mode, ph * q.hop,
                               clip_pitch, g.plane_stride, planes, two, stream)))
      return rc;
    {
      const int mrows = (cta_group == 2 ? 2 : 1) * TC_BM;
      double kcols = 0.0;  // sum over N tiles of (k-blocks executed) x bk x bn
      for (int tl = 0; tl < n_tiles; ++tl) kcols += (double)(prm.kb_end[tl] - prm.kb_begin[tl]) * bk * bn;
      const double terms = two ? 2.0 : (prm.split4 && cta_group == 2 ? 4.0 : 3.0);
      add_exec_flops(terms * 2.0 *
                     (double)ceil_div64(g.nv, mrows) * mrows * kcols);
    }
    if (cta_group == 2) {
      prm.num_m_tiles = (int)ceil_div64(g.nv, 2 * TC_BM);  // 256-frame pair tiles
      const int64_t ptiles = (int64_t)prm.num_m_tiles * prm.num_n_tiles * prm.k_splits;
      const int n_pairs = (int)(ptiles < sms / 2 ? ptiles : sms / 2);
      rc = launch_tc2_kernel<64, 3>(ma, mb, prm, n_pairs, stream);
    } else {
      prm.num_m_tiles = (int)ceil_div64(g.nv, TC_BM);
      const int64_t tiles = (int64_t)prm.num_m_tiles * prm.num_n_tiles * prm.k_splits;
      const int grid = (int)(tiles < sms ? tiles : sms);
      rc = (bk == 64) ? launch_tc_kernel<64, 2>(ma, mb, prm, grid, stream)
                      : launch_tc_kernel<32, 4>(ma, mb, prm, grid, stream);
    }
    if (rc) return rc;
  }
  if (split) {
    dim3 grid((unsigned)ceil_div64(q.T, 256), (unsigned)q.F, (unsigned)(q.B < 64 ? q.B : 64));
    splitk_finalize_kernel<<<grid, 256, 0, stream>>>(final_epi, q.B);
    NNAB_LAUNCH_CHECK();
  }
  return NNAB_OK;
}

}  // namespace nnab
