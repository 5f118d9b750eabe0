// Generic fp32 CUDA-core kernels of libnnab.so (sm_100a):
//   * framed complex contraction (any hop / K / F, sparse-support aware)
//   * filterbank GEMM  out = fb @ P      (mel.py:188, gammatone.py:188)
//   * MFCC tail        dB -> top_db clamp -> DCT   (mel.py:263-307, 325)
//   * FIR decimation   conv1d(x, fir, stride=n, padding=127)  (utils.py:73-124)
// They are the first-correct path and the fallback for shapes the tcgen05/TMA
// kernel does not take (hop % 8 != 0, tiny banks, ...).  No CPU fallback exists.
#include "common.cuh"
#include "epilogue.cuh"

namespace nnab {

// --------------------------------------------------------------------------
// sample fetch with the centre padding folded into the index
// (nn.ReflectionPad1d / nn.ConstantPad1d semantics, stft.py:278-289)
// --------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float fetch_padded(const T* __restrict__ xb, int64_t L, int64_t j,
                                              int pad_mode) {
  if (j < 0) {
    if (pad_mode == NNAB_PAD_CONSTANT) return 0.f;
    j = -j;
  } else if (j >= L) {
    if (pad_mode == NNAB_PAD_CONSTANT) return 0.f;
    j = 2 * (L - 1) - j;
  }
  return (j >= 0 && j < L) ? ldg_sample(xb + j) : 0.f;
}

// --------------------------------------------------------------------------
// framed complex contraction, SIMT
//   CTA tile: 128 frames x (16*TN) bins, 256 threads, thread tile 8 x TN x {re,im}
// --------------------------------------------------------------------------
constexpr int SIMT_MAX_BIN_TILES = 128;

struct SimtParams {
  const void* x;  // element type: the kernel's T
  int64_t L, x_pitch;
  const float* w_re;
  const float* w_im;
  int F, K, hop, pad, pad_mode;
  int n_ranges;  // 0 => dense [0, K) for every bin tile
  int kb[SIMT_MAX_BIN_TILES];
  int ke[SIMT_MAX_BIN_TILES];
  EpiParams epi;
};

template <int TN, typename T>
__global__ void __launch_bounds__(256) framed_cplx_simt_kernel(const SimtParams p) {
  constexpr int TM = 8, BM = 128, BNB = 16 * TN, BK = 16;
  __shared__ float As[BM][BK + 1];
  __shared__ __align__(16) float Wr[BK][BNB + 4];
  __shared__ __align__(16) float Wi[BK][BNB + 4];

  const int tid = threadIdx.x;
  const int tx = tid & 15;  // frame lane
  const int ty = tid >> 4;  // bin group
  const int64_t b = blockIdx.z;
  const int64_t t0 = (int64_t)blockIdx.x * BM;
  const int f0 = blockIdx.y * BNB;
  const T* __restrict__ xb = static_cast<const T*>(p.x) + b * p.x_pitch;

  int kbeg = 0, kend = p.K;
  if (p.n_ranges > 0) {
    kbeg = p.kb[blockIdx.y];
    kend = p.ke[blockIdx.y];
  }

  float acc_re[TM][TN], acc_im[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc_re[i][j] = acc_im[i][j] = 0.f;

  const int lk = tid & 15;
  const int lr = tid >> 4;
  for (int k0 = kbeg; k0 < kend; k0 += BK) {
    const int k = k0 + lk;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int m = lr + 16 * i;
      const int64_t t = t0 + m;
      float v = 0.f;
      if (t < p.epi.T && k < kend)
        v = fetch_padded(xb, p.L, t * (int64_t)p.hop + k - p.pad, p.pad_mode);
      As[m][lk] = v;
    }
#pragma unroll
    for (int i = 0; i < TN; ++i) {
      const int j = lr + 16 * i;
      const int f = f0 + j;
      float vr = 0.f, vi = 0.f;
      if (f < p.F && k < kend) {
        vr = __ldg(p.w_re + (int64_t)f * p.K + k);
        vi = __ldg(p.w_im + (int64_t)f * p.K + k);
      }
      Wr[lk][j] = vr;
      Wi[lk][j] = vi;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[TM], wr[TN], wi[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = As[tx + 16 * i][kk];
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        wr[j] = Wr[kk][ty * TN + j];
        wi[j] = Wi[kk][ty * TN + j];
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) {
          acc_re[i][j] = fmaf(a[i], wr[j], acc_re[i][j]);
          acc_im[i][j] = fmaf(a[i], wi[j], acc_im[i][j]);
        }
    }
    __syncthreads();
  }

#pragma unroll
  for (int j = 0; j < TN; ++j) {
    const int f = f0 + ty * TN + j;
    if (f >= p.F) continue;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int64_t t = t0 + tx + 16 * i;
      if (t < p.epi.T) epi_store(p.epi, b, f, t, acc_re[i][j], -acc_im[i][j]);
    }
  }
}

int launch_framed_simt(const FramedProblem& q, cudaStream_t stream) {
  if (q.B <= 0 || q.T <= 0 || q.F <= 0) return NNAB_OK;
  if (q.B > 65535) return NNAB_EUNSUPPORTED;
  SimtParams p;
  p.x = q.x; p.L = q.L; p.x_pitch = q.x_pitch;
  p.w_re = q.w_re; p.w_im = q.w_im;
  p.F = q.F; p.K = q.K; p.hop = q.hop; p.pad = q.pad; p.pad_mode = q.pad_mode;
  p.epi.scale = q.scale; p.epi.scale_all = q.scale_all; p.epi.fmt = q.fmt;
  p.epi.eps = q.eps; p.epi.power = q.power; p.epi.out = q.out; p.epi.T = q.T;
  p.epi.out_bins = q.out_bins; p.epi.bin_offset = q.bin_offset; p.epi.F = q.F;
  p.epi.fb_table = nullptr; p.epi.n_fb = 0;
  p.epi.dec = DecimParams{};
  p.epi.raw = nullptr; p.epi.raw_plane = 0;
  p.epi.ola_pitch = 0; p.epi.ola_hop = 0;
  if (q.fmt == FMT_FBANK || q.fmt == FMT_DECIM || q.fmt == FMT_RAW || q.fmt == FMT_OLA)
    return NNAB_EINVAL;  // fused filterbank exists on the tcgen05 path only

  const int TN = (q.F > 32) ? 4 : 2;
  const int BNB = 16 * TN;
  const int n_tiles = (q.F + BNB - 1) / BNB;
  p.n_ranges = 0;
  if (q.h_k_begin != nullptr && q.h_k_end != nullptr && n_tiles <= SIMT_MAX_BIN_TILES) {
    p.n_ranges = n_tiles;
    for (int tl = 0; tl < n_tiles; ++tl) {
      int lo = q.K, hi = 0;
      for (int f = tl * BNB; f < q.F && f < (tl + 1) * BNB; ++f) {
        if (q.h_k_end[f] > q.h_k_begin[f]) {
          lo = q.h_k_begin[f] < lo ? q.h_k_begin[f] : lo;
          hi = q.h_k_end[f] > hi ? q.h_k_end[f] : hi;
        }
      }
      if (hi < lo) { lo = 0; hi = 0; }
      if (lo < 0) lo = 0;
      if (hi > q.K) hi = q.K;
      p.kb[tl] = lo;
      p.ke[tl] = hi;
    }
  }
  dim3 grid((unsigned)ceil_div64(q.T, 128), (unsigned)n_tiles, (unsigned)q.B);
  switch (q.x_dtype) {
    case NNAB_DTYPE_F32:
      if (TN == 4) framed_cplx_simt_kernel<4, float><<<grid, 256, 0, stream>>>(p);
      else framed_cplx_simt_kernel<2, float><<<grid, 256, 0, stream>>>(p);
      break;
    case NNAB_DTYPE_BF16:
      if (TN == 4) framed_cplx_simt_kernel<4, __nv_bfloat16><<<grid, 256, 0, stream>>>(p);
      else framed_cplx_simt_kernel<2, __nv_bfloat16><<<grid, 256, 0, stream>>>(p);
      break;
    case NNAB_DTYPE_F16:
      if (TN == 4) framed_cplx_simt_kernel<4, __half><<<grid, 256, 0, stream>>>(p);
      else framed_cplx_simt_kernel<2, __half><<<grid, 256, 0, stream>>>(p);
      break;
    default: return NNAB_EINVAL;
  }
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// --------------------------------------------------------------------------
// filterbank GEMM: out[b, j, t] = sum_f fb[j, f] * P[b, f, t]
//   CTA tile 64 filters x 128 frames, BK = 16 bins; all-zero fb blocks (the
//   mel matrix is ~98.5 % zeros) skip their P tile entirely.
// --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) filterbank_kernel(const float* __restrict__ P,
                                                         const float* __restrict__ fb, int F,
                                                         int64_t T, int n_fb,
                                                         float* __restrict__ out) {
  constexpr int BJ = 64, BT = 128, BK = 16;
  __shared__ float Ps[BK][BT];
  __shared__ __align__(16) float Fs[BK][BJ + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 31, ty = tid >> 5;
  const int64_t b = blockIdx.z;
  const int64_t t0 = (int64_t)blockIdx.x * BT;
  const int j0 = blockIdx.y * BJ;
  const float* __restrict__ Pb = P + b * (int64_t)F * T;

  float acc[8][4];
#pragma unroll
  for (int jj = 0; jj < 8; ++jj)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[jj][i] = 0.f;

  const int lk = tid & 15, lr = tid >> 4;
  for (int fk = 0; fk < F; fk += BK) {
    int nz = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int j = lr + 16 * i;
      float v = 0.f;
      if (j0 + j < n_fb && fk + lk < F) v = __ldg(fb + (int64_t)(j0 + j) * F + fk + lk);
      Fs[lk][j] = v;
      nz |= (v != 0.f);
    }
    nz = __syncthreads_or(nz);
    if (!nz) continue;  // uniform: nothing of this filter tile lives in these bins
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int idx = tid + 256 * i;
      const int r = idx >> 7, c = idx & 127;
      float v = 0.f;
      if (fk + r < F && t0 + c < T) v = __ldg(Pb + (int64_t)(fk + r) * T + t0 + c);
      Ps[r][c] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float pv[4], w[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) pv[i] = Ps[kk][tx + 32 * i];
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) w[jj] = Fs[kk][ty * 8 + jj];
#pragma unroll
      for (int jj = 0; jj < 8; ++jj)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[jj][i] = fmaf(w[jj], pv[i], acc[jj][i]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int j = j0 + ty * 8 + jj;
    if (j >= n_fb) continue;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t t = t0 + tx + 32 * i;
      if (t < T) out[((int64_t)b * n_fb + j) * T + t] = acc[jj][i];
    }
  }
}

// One thread per FFT bin: record its (<= 2) non-zero filter weights and the
// largest per-bin count (a dense bank such as the gammatone one reports > 2 and
// is then served by the un-fused filterbank GEMM).
__global__ void fb_table_kernel(const float* __restrict__ fb, int n_fb, int F,
                                FbEntry* __restrict__ table, int* __restrict__ max_nnz) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  FbEntry e{-1, -1, 0.f, 0.f};
  int nnz = 0;
  for (int j = 0; j < n_fb; ++j) {
    const float w = __ldg(fb + (int64_t)j * F + f);
    if (w != 0.f) {
      if (nnz == 0) { e.j0 = j; e.w0 = w; }
      else if (nnz == 1) { e.j1 = j; e.w1 = w; }
      ++nnz;
    }
  }
  table[f] = e;
  atomicMax(max_nnz, nnz);
}

int launch_fb_table(const float* fb, int n_fb, int F, FbEntry* table, int* d_max_nnz,
                    cudaStream_t stream) {
  NNAB_CUDA_TRY(cudaMemsetAsync(d_max_nnz, 0, sizeof(int), stream));
  fb_table_kernel<<<(F + 127) / 128, 128, 0, stream>>>(fb, n_fb, F, table, d_max_nnz);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// Sequential (one thread; F ~ 1e3, init time) replay of the two-slot running-sum logic over the bin
// axis, recording the actions per bin (see FbStep).
__global__ void fb_steps_kernel(const FbEntry* __restrict__ table, int n_fb, int F,
                                FbStep* __restrict__ steps, int* __restrict__ meta) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  int cur_a = -1, cur_b = -1;
  for (int k = 0; k < F + FB_STEP_PAD; ++k) {
    FbStep st{0.f, 0.f, (short)-1, (short)-1, (short)cur_a, (short)cur_b};
    if (k < F) {
      const FbEntry e = table[k];
      const int js[2] = {e.j0, e.j1};
      const float ws[2] = {e.w0, e.w1};
      bool used_a = false;
      for (int i = 0; i < 2; ++i) {  // filters already held keep their slot
        if (js[i] < 0) continue;
        if (js[i] == cur_a) { st.wa = ws[i]; used_a = true; }
        else if (js[i] == cur_b) { st.wb = ws[i]; }
      }
      for (int i = 0; i < 2; ++i) {  // new filters take a free slot (its old sum is flushed first)
        if (js[i] < 0 || js[i] == cur_a || js[i] == cur_b) continue;
        if (!used_a) {
          if (cur_a >= 0) st.flush_a = (short)cur_a;
          cur_a = js[i]; st.wa = ws[i]; used_a = true;
        } else {
          if (cur_b >= 0) st.flush_b = (short)cur_b;
          cur_b = js[i]; st.wb = ws[i];
        }
      }
    }
    st.cur_a = (short)cur_a;
    st.cur_b = (short)cur_b;
    steps[k] = st;
  }
  // For which tile widths nb = 32 + 8 i (i = 0..12) does every filter receive at most two partial
  // sums?  A partial sum comes from each bin range (tile x warp part, cut exactly as
  // framed_tcb_kernel cuts them) that intersects the filter's support; with <= 2 of them the
  // atomic adds commute and the fused filterbank is run-to-run identical.
  int widest = 0;
  unsigned mask = 0x1FFFu;
  for (int j = 0; j < n_fb; ++j) {
    int lo = -1, hi = -1;
    for (int k = 0; k < F; ++k) {
      const FbEntry e = table[k];
      if (e.j0 == j || e.j1 == j) { if (lo < 0) lo = k; hi = k; }
    }
    if (lo < 0) continue;
    if (hi - lo + 1 > widest) widest = hi - lo + 1;
    for (int i = 0; i < 13; ++i) {
      const int nb = 32 + 8 * i, outs = nb - 2, n_chunks = nb / 8;
      // range index of bin k: tile k / outs, then the warp part that owns chunk (o + 2) / 8 of output o
      auto range_of = [&](int k) {
        const int c = (k % outs + 2) / 8;
        int part = 0;
        while (part + 1 < FB_EPI_PARTS && c >= (n_chunks * (part + 1)) / FB_EPI_PARTS) ++part;
        return FB_EPI_PARTS * (k / outs) + part;
      };
      if (range_of(hi) - range_of(lo) + 1 > 2) mask &= ~(1u << i);
    }
  }
  meta[0] = widest;
  meta[1] = (int)mask;
}

int launch_fb_steps(const FbEntry* table, int n_fb, int F, FbStep* steps, int* d_meta,
                    cudaStream_t stream) {
  fb_steps_kernel<<<1, 32, 0, stream>>>(table, n_fb, F, steps, d_meta);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

int launch_filterbank(const float* P, const float* fb, int64_t B, int F, int64_t T, int n_fb,
                      float* out, cudaStream_t stream) {
  if (B <= 0 || T <= 0 || n_fb <= 0) return NNAB_OK;
  if (B > 65535) return NNAB_EUNSUPPORTED;
  dim3 grid((unsigned)ceil_div64(T, 128), (unsigned)((n_fb + 63) / 64), (unsigned)B);
  filterbank_kernel<<<grid, 256, 0, stream>>>(P, fb, F, T, n_fb, out);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// Dense filterbank as the B operand of a real GEMM on the complex tcgen05 kernel: the (n_fb, F) weights
// re-indexed to the column layout of the block-partial kernel's FMT_PLANES output (tile n, packed column
// i  <->  FFT bin n (nb - 2) + i - 2; columns 0, 1 of a tile and bins >= F carry zeros), filters
// [0, fh) in the real bank and filters [fh, 2 fh) NEGATED in the imaginary bank (the contraction returns
// -sum x w_im, FMT_REALPAIR then writes re -> row f, im -> row f + fh).
__global__ void __launch_bounds__(256) fb_tile_bank_kernel(const float* __restrict__ fb, int n_fb, int F,
                                                           int nb, int n_tiles, int kp, int fh,
                                                           float* __restrict__ w_re, float* __restrict__ w_im) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)fh * kp) return;
  const int j = (int)(idx / kp), col = (int)(idx % kp);
  const int n = col / nb, i = col - n * nb;
  float a = 0.f, b = 0.f;
  if (n < n_tiles && i >= 2) {
    const int k = n * (nb - 2) + i - 2;
    if (k < F) {
      a = __ldg(fb + (int64_t)j * F + k);
      if (j + fh < n_fb) b = -__ldg(fb + (int64_t)(j + fh) * F + k);
    }
  }
  w_re[idx] = a;
  w_im[idx] = b;
}

int launch_fb_tile_bank(const float* fb, int n_fb, int F, int nb, int n_tiles, int kp, int fh, float* w_re,
                        float* w_im, cudaStream_t stream) {
  const int64_t n = (int64_t)fh * kp;
  fb_tile_bank_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, stream>>>(fb, n_fb, F, nb, n_tiles, kp, fh,
                                                                        w_re, w_im);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

// --------------------------------------------------------------------------
// MFCC tail
//   pass 1: per-clip max of max(S, amin)  (float bits are monotone for > 0)
//   pass 2: dB, clamp to (clip max dB - top_db), orthonormal DCT-II rows
// --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) clip_max_kernel(const float* __restrict__ S,
                                                       int64_t per_clip, float amin,
                                                       unsigned int* __restrict__ clip_max) {
  const int64_t b = blockIdx.y;
  const float* __restrict__ Sb = S + b * per_clip;
  float m = amin;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_clip;
       i += (int64_t)gridDim.x * blockDim.x)
    m = fmaxf(m, __ldg(Sb + i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float wm[8];
  if ((threadIdx.x & 31) == 0) wm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) m = fmaxf(m, wm[w]);
    atomicMax(clip_max + b, __float_as_uint(m));  // m >= amin > 0
  }
}

constexpr int MFCC_CHUNK = 32;

// One thread per (clip, frame), flattened over the batch so every block is full (T = 157 at cfg5
// would leave 38 % of a per-clip grid idle).  dB through MUFU.LG2 (10 log10 x = 3.0103 log2 x; abs
// error ~1e-6 dB on a +-100 dB range), DCT rows transposed in shared memory ([mel][coef], float4
// broadcast reads: 1 LDS.128 per 4 FMAs).  HBM-bound target: read (B, n_mels, T) once, coalesced in t.
__global__ void __launch_bounds__(128) mfcc_tail_kernel(const float* __restrict__ S, int n_mels,
                                                        int64_t T, int64_t BT, float amin, float ref_db,
                                                        float top_db,
                                                        const unsigned int* __restrict__ clip_max,
                                                        const float* __restrict__ dct, int n_mfcc,
                                                        int c0, float* __restrict__ out) {
  extern __shared__ __align__(16) float dsm[];  // [n_mels][MFCC_CHUNK]
  const int nc = min(MFCC_CHUNK, n_mfcc - c0);
  for (int i = threadIdx.x; i < n_mels * MFCC_CHUNK; i += blockDim.x) {
    const int m = i / MFCC_CHUNK, c = i % MFCC_CHUNK;
    dsm[i] = (c < nc) ? __ldg(dct + (int64_t)(c0 + c) * n_mels + m) : 0.f;
  }
  __syncthreads();
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= BT) return;
  const int64_t b = g / T, t = g - b * T;
  const float* __restrict__ Sb = S + b * (int64_t)n_mels * T + t;
  float floor_db = -INFINITY;
  if (top_db >= 0.f) {
    const float peak = 3.0102999566f * __log2f(__uint_as_float(clip_max[b])) - ref_db;
    floor_db = peak - top_db;
  }
  float acc[MFCC_CHUNK];
#pragma unroll
  for (int c = 0; c < MFCC_CHUNK; ++c) acc[c] = 0.f;
#pragma unroll 4
  for (int m = 0; m < n_mels; ++m) {
    float v = 3.0102999566f * __log2f(fmaxf(__ldg(Sb + (int64_t)m * T), amin)) - ref_db;
    v = fmaxf(v, floor_db);
    const float4* w = reinterpret_cast<const float4*>(dsm + m * MFCC_CHUNK);
#pragma unroll
    for (int c4 = 0; c4 < MFCC_CHUNK / 4; ++c4) {
      if (4 * c4 < nc) {  // block-uniform
        const float4 d = w[c4];
        acc[4 * c4 + 0] = fmaf(d.x, v, acc[4 * c4 + 0]);
        acc[4 * c4 + 1] = fmaf(d.y, v, acc[4 * c4 + 1]);
        acc[4 * c4 + 2] = fmaf(d.z, v, acc[4 * c4 + 2]);
        acc[4 * c4 + 3] = fmaf(d.w, v, acc[4 * c4 + 3]);
      }
    }
  }
  float* __restrict__ ob = out + ((int64_t)b * n_mfcc + c0) * T + t;
#pragma unroll
  for (int c = 0; c < MFCC_CHUNK; ++c)
    if (c < nc) ob[(int64_t)c * T] = acc[c];
}

// `scratch` holds B uint32 (per-clip max bits), provided by the caller's workspace.
int launch_mfcc_tail(const float* mel, int64_t B, int n_mels, int64_t T, float amin,
                          float ref, float top_db, const float* dct, int n_mfcc, float* out,
                          unsigned int* scratch, cudaStream_t stream) {
  if (B <= 0 || T <= 0) return NNAB_OK;
  if (B > 65535) return NNAB_EUNSUPPORTED;
  const size_t smem = (size_t)MFCC_CHUNK * n_mels * sizeof(float);
  if (smem > 200 * 1024) return NNAB_EUNSUPPORTED;
  const float ref_db = 10.0f * log10f(fmaxf(amin, fabsf(ref)));
  if (top_db >= 0.f) {
    NNAB_CUDA_TRY(cudaMemsetAsync(scratch, 0, (size_t)B * sizeof(unsigned int), stream));
    const int64_t per_clip = (int64_t)n_mels * T;
    int gx = (int)ceil_div64(per_clip, 256 * 8);
    if (gx < 1) gx = 1;
    if (gx > 64) gx = 64;
    clip_max_kernel<<<dim3(gx, (unsigned)B), 256, 0, stream>>>(mel, per_clip, amin, scratch);
    NNAB_LAUNCH_CHECK();
  }
  if (smem > 48 * 1024)
    NNAB_CUDA_TRY(cudaFuncSetAttribute(mfcc_tail_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t BT = B * T;
  for (int c0 = 0; c0 < n_mfcc; c0 += MFCC_CHUNK) {
    mfcc_tail_kernel<<<(unsigned)ceil_div64(BT, 128), 128, smem, stream>>>(
        mel, n_mels, T, BT, amin, ref_db, top_db, scratch, dct, n_mfcc, c0, out);
    NNAB_LAUNCH_CHECK();
  }
  return NNAB_OK;
}

// --------------------------------------------------------------------------
// FIR decimation: y[n] = sum_j fir[j] * x[n*factor + j - (taps-1)/2], zero outside
//   Polyphase in shared memory so a thread's 4 consecutive outputs slide over
//   unit-stride data: 2 LDS.128 per 16 FMAs.
// --------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) fir_decimate_kernel(
    const T* __restrict__ x, int64_t L, int64_t x_pitch, const float* __restrict__ fir,
    int taps, int factor, int qtaps, int ph_len, float* __restrict__ y, int64_t Ly,
    int64_t y_pitch) {
  extern __shared__ __align__(16) float fsm[];
  float* xs = fsm;                    // [factor][ph_len]
  float* fs = fsm + factor * ph_len;  // [factor][qtaps]
  const int tid = threadIdx.x;
  const int64_t b = blockIdx.y;
  const int64_t n0 = (int64_t)blockIdx.x * 1024;
  const int64_t base = n0 * factor - (taps - 1) / 2;
  const T* __restrict__ xb = x + b * x_pitch;

  for (int idx = tid; idx < ph_len * factor; idx += 256) {
    const int64_t g = base + idx;
    const float v = (g >= 0 && g < L) ? ldg_sample(xb + g) : 0.f;
    xs[(idx % factor) * ph_len + idx / factor] = v;
  }
  for (int j = tid; j < qtaps * factor; j += 256)
    fs[(j % factor) * qtaps + j / factor] = (j < taps) ? __ldg(fir + j) : 0.f;
  __syncthreads();

  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int ph = 0; ph < factor; ++ph) {
    const float* xp = xs + ph * ph_len + 4 * tid;
    const float* fp = fs + ph * qtaps;
    float4 v0 = *reinterpret_cast<const float4*>(xp);
    for (int qb = 0; qb < qtaps; qb += 4) {
      const float4 v1 = *reinterpret_cast<const float4*>(xp + qb + 4);
      const float4 f = *reinterpret_cast<const float4*>(fp + qb);
      const float w[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        acc[o] = fmaf(f.x, w[o], acc[o]);
        acc[o] = fmaf(f.y, w[o + 1], acc[o]);
        acc[o] = fmaf(f.z, w[o + 2], acc[o]);
        acc[o] = fmaf(f.w, w[o + 3], acc[o]);
      }
      v0 = v1;
    }
  }
  float* __restrict__ yb = y + b * y_pitch;
#pragma unroll
  for (int o = 0; o < 4; ++o) {
    const int64_t n = n0 + 4 * tid + o;
    if (n < Ly) yb[n] = acc[o];
  }
}

template <typename T>
static int launch_fir_decimate_t(const T* x, int64_t B, int64_t L, int64_t x_pitch, const float* fir,
                                 int taps, int factor, float* y, int64_t Ly, int64_t y_pitch,
                                 cudaStream_t stream) {
  if (B <= 0 || Ly <= 0) return NNAB_OK;
  if (B > 65535 || factor < 1 || taps < 1) return NNAB_EUNSUPPORTED;
  int qtaps = (taps + factor - 1) / factor;
  qtaps = (qtaps + 3) & ~3;
  const int ph_len = 1024 + qtaps + 4;  // +4: the rolling float4 window reads one vector ahead
  const size_t smem = (size_t)factor * (ph_len + qtaps) * sizeof(float);
  if (smem > 200 * 1024) return NNAB_EUNSUPPORTED;
  if (smem > 48 * 1024)
    NNAB_CUDA_TRY(cudaFuncSetAttribute(fir_decimate_kernel<T>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)ceil_div64(Ly, 1024), (unsigned)B);
  fir_decimate_kernel<T><<<grid, 256, smem, stream>>>(x, L, x_pitch, fir, taps, factor, qtaps,
                                                      ph_len, y, Ly, y_pitch);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

int launch_fir_decimate(const void* x, int x_dtype, int64_t B, int64_t L, int64_t x_pitch,
                        const float* fir, int taps, int factor, float* y, int64_t Ly, int64_t y_pitch,
                        cudaStream_t stream) {
  switch (x_dtype) {
    case NNAB_DTYPE_F32:
      return launch_fir_decimate_t((const float*)x, B, L, x_pitch, fir, taps, factor, y, Ly, y_pitch, stream);
    case NNAB_DTYPE_BF16:
      return launch_fir_decimate_t((const __nv_bfloat16*)x, B, L, x_pitch, fir, taps, factor, y, Ly, y_pitch,
                                   stream);
    case NNAB_DTYPE_F16:
      return launch_fir_decimate_t((const __half*)x, B, L, x_pitch, fir, taps, factor, y, Ly, y_pitch, stream);
    default: return NNAB_EINVAL;
  }
}

// --------------------------------------------------------------------------
// Adjoint of the decimating FIR (GPU-verified round 2, default of the pyramid training path),
//   dx[i] = sum_j g[j] * fir[i + half - factor*j],   half = (taps-1)/2,  0 <= i < L
// (the gradient of y = conv1d(x, fir, stride=factor, padding=half), utils.py:73-100).
// One CTA = 1024 consecutive inputs of one clip; the g samples and the filter they touch are
// staged in shared memory; every input is written exactly once (no atomics).
// --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fir_decimate_adjoint_kernel(
    const float* __restrict__ g, int64_t T, int64_t g_pitch, const float* __restrict__ fir, int taps,
    int factor, int g_len, float* __restrict__ dx, int64_t L, int64_t dx_pitch) {
  extern __shared__ float asm_[];
  float* fs = asm_;         // [taps]
  float* gs = asm_ + taps;  // [g_len]
  const int tid = threadIdx.x;
  const int64_t b = blockIdx.y;
  const int64_t i0 = (int64_t)blockIdx.x * 1024;
  const int half = (taps - 1) / 2;
  // smallest j any output of this block can touch: factor*j >= i0 + half - (taps-1)
  int64_t lo = i0 + half - (taps - 1);
  const int64_t j_lo = lo <= 0 ? 0 : (lo + factor - 1) / factor;
  const float* __restrict__ gb = g + b * g_pitch;
  for (int idx = tid; idx < taps; idx += 256) fs[idx] = __ldg(fir + idx);
  for (int idx = tid; idx < g_len; idx += 256) {
    const int64_t j = j_lo + idx;
    gs[idx] = (j < T) ? __ldg(gb + j) : 0.f;
  }
  __syncthreads();
  float* __restrict__ db = dx + b * dx_pitch;
#pragma unroll
  for (int o = 0; o < 4; ++o) {
    const int64_t i = i0 + tid + 256 * o;
    if (i >= L) continue;
    const int64_t top = i + half;               // tap index at j = 0
    int64_t ja = top - (taps - 1);
    ja = ja <= 0 ? 0 : (ja + factor - 1) / factor;
    int64_t jb = top / factor;                  // last j with a non-negative tap index
    if (jb > T - 1) jb = T - 1;
    float acc = 0.f;
    for (int64_t j = ja; j <= jb; ++j)
      acc = fmaf(gs[(int)(j - j_lo)], fs[(int)(top - factor * j)], acc);
    db[i] = acc;
  }
}

int launch_fir_decimate_adjoint(const float* g, int64_t B, int64_t T, int64_t g_pitch,
                                const float* fir, int taps, int factor, float* dx, int64_t L,
                                int64_t dx_pitch, cudaStream_t stream) {
  if (B <= 0 || L <= 0) return NNAB_OK;
  if (B > 65535 || factor < 1 || taps < 1) return NNAB_EUNSUPPORTED;
  // j range of one block: (1023 + taps - 1) / factor + 2 values at most
  const int g_len = (1023 + taps - 1) / factor + 3;
  const size_t smem = (size_t)(taps + g_len) * sizeof(float);
  if (smem > 200 * 1024) return NNAB_EUNSUPPORTED;
  if (smem > 48 * 1024)
    NNAB_CUDA_TRY(cudaFuncSetAttribute(fir_decimate_adjoint_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)ceil_div64(L, 1024), (unsigned)B);
  fir_decimate_adjoint_kernel<<<grid, 256, smem, stream>>>(g, T, g_pitch, fir, taps, factor, g_len,
                                                           dx, L, dx_pitch);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}

}  // namespace nnab
