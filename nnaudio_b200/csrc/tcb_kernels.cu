// Block-partial ("sliding") STFT on tcgen05 for sm_100a — the default kernel of the STFT family
// (STFT / MelSpectrogram / MFCC / Gammatonegram with a periodic Hann window and hop = n_fft / R,
// R = 2 or 4: the reference's defaults, stft.py:177-178).
//
// The dense path contracts every frame with the windowed n_fft-point basis (features/stft.py:290-293:
// conv1d(x, wsin/wcos, stride=hop)).  Consecutive frames share R-1 of their R hop-sized blocks, so
// here the contraction runs ONCE per block against the UN-windowed basis:
//
//   Z_g[k]  = sum_{n < hop} xpad[g*hop + n] exp(-2 pi i k n / N)                    K = hop, not N
//   hann[m] = 1/2 - 1/4 e^{+i theta m} - 1/4 e^{-i theta m}    (theta = 2 pi / N)   3 taps along k
//   X_t[k]  = sum_{j<R} c_k^j V_j(Z_{t+j})[k],   c_k = exp(-2 pi i k / R)
//   V_j(Z)[k] = 1/2 Z[k] - 1/4 w^j Z[k-1] - 1/4 w^-j Z[k+1],   w = exp(2 pi i / R)
//
// (tools/block_dft_emulation.py is the executable spec; exact in exact arithmetic.)  R times fewer
// MMA flops than the dense form, the A operand is a plain (blocks x hop) matrix, and the epilogue
// does the 3-tap bin filter in registers and the R-block frame sum with warp shuffles.
//
// GEMM view: M = block rows g of the whole batch (the split-signal planes of tc_kernels.cu viewed
// as a (rows x hop) matrix), K = hop, N = 2 * (F + 2) columns (re | im of bins -1 .. F: the two
// extra bins are the k-1 / k+1 neighbours of the edge bins).
//
// Tiling (CTA pairs, cta_group::2, same pipeline roles as framed_tc2_kernel):
//   * N tile = nb packed bins (re half staged by CTA 0, im half by CTA 1); consecutive tiles
//     overlap by 2 bins, a tile emits nb - 2 output bins.
//   * M: each epilogue warp owns one 32-lane TMEM quarter = 32 consecutive block rows and emits
//     33 - R frames; the 4 quarters of a CTA are loaded as four 32-row TMA boxes whose row origins
//     are 33 - R apart, so no frame needs a row of another warp (no smem exchange, no barrier).
//     4 * (33 - R) frames per CTA tile (116 of 128 rows for R = 4).
//   * fp32 parity: x*w = xhi*whi + xlo*whi + xhi*wlo on bf16 tensor cores, fp32 accumulation.
#include <cuda.h>
#include <cuda_bf16.h>
#include <atomic>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "epilogue.cuh"
#include "tc_ptx.cuh"
#include "tc_host.cuh"
#include "tc_decim.cuh"

namespace nnab {

constexpr int TCB_BK = 64;
constexpr int TCB_STAGES = 3;
constexpr int TCB_ACC_STRIDE = 256;

struct TcbParams {
  int num_m_pairs;   // pair tiles along M
  int num_n_tiles;
  int nb;            // packed bins per N tile (MMA N = 2 nb)
  int kb_n;          // hop / 64
  int two_term;      // bf16 input: the A lo plane is zero -- neither loaded nor multiplied
  int64_t nv, t_slots, T;
  EpiParams epi;
};

struct TcbSmem {
  static constexpr uint32_t A_BYTES = TC_BM * TCB_BK * 2;   // one plane, 128 rows
  static constexpr uint32_t B_BYTES = 128 * TCB_BK * 2;     // one plane, <= 128 rows (this CTA's half)
  static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr uint32_t BAR_OFFSET = TCB_STAGES * STAGE_BYTES;
  static constexpr uint32_t TOTAL = BAR_OFFSET + 256 + 1024;
};

// rows of one (plane, part) slab of the packed block basis
static int block_choose_nb(int F) {
  int best = 32, best_cost = 1 << 30;
  for (int nb = 128; nb >= 32; nb -= 8) {
    const int tiles = (F + nb - 3) / (nb - 2);
    const int cost = tiles * (nb + 6);  // + a little per-tile overhead: prefer fewer, wider tiles on ties
    if (cost < best_cost) { best_cost = cost; best = nb; }
  }
  return best;
}
static int block_n_tiles(int F, int nb) { return (F + nb - 3) / (nb - 2); }
void tc_block_tile_geometry(int F, int* nb, int* n_tiles) {
  *nb = block_choose_nb(F);
  *n_tiles = block_n_tiles(F, *nb);
}
// rows of one (plane, part) slab: bins -1 .. F plus zero rows so that the last tile of ANY nb <= 128
// stays inside the slab (the launch picks nb, e.g. wider tiles for the fused filterbank)
static int block_p_rows(int F) { return round_up_i(F + 2 + 128, 8); }

size_t tc_packed_block_bytes(int n_fft, int hop) {
  if (!tc_block_shape_ok(n_fft, hop)) return 0;
  return (size_t)4 * block_p_rows(n_fft / 2 + 1) * hop * sizeof(__nv_bfloat16) + 256;
}

bool tc_block_shape_ok(int n_fft, int hop) {
  if (hop <= 0 || n_fft % hop != 0) return false;
  const int R = n_fft / hop;
  return (R == 2 || R == 4) && hop % 64 == 0 && n_fft >= 128 && n_fft <= 32768;
}

// packed[plane hi|lo][part re|im][p][n]: bin k = p - 1, sample n < hop:
//   re row:  cos(2 pi k n / N)      im row: -sin(2 pi k n / N)     (so re + i im = e^{-i theta k n})
__global__ void __launch_bounds__(256) pack_block_basis_kernel(int n_fft, int hop, int F, int p_rows,
                                                               __nv_bfloat16* __restrict__ packed) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int k8 = hop / 8;
  if (idx >= (int64_t)p_rows * k8) return;
  const int p = (int)(idx / k8);
  const int n0 = (int)(idx % k8) * 8;
  const int k = p - 1;
  __align__(16) __nv_bfloat16 rh[8], rl[8], ih[8], il[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    float c = 0.f, s = 0.f;
    if (p < F + 2) {
      const int n = n0 + e;
      long long m = ((long long)k * n) % n_fft;
      if (m < 0) m += n_fft;
      double sd, cd;
      sincospi(2.0 * (double)m / (double)n_fft, &sd, &cd);
      c = (float)cd;
      s = (float)(-sd);
    }
    rh[e] = __float2bfloat16_rn(c);
    rl[e] = __float2bfloat16_rn(c - __bfloat162float(rh[e]));
    ih[e] = __float2bfloat16_rn(s);
    il[e] = __float2bfloat16_rn(s - __bfloat162float(ih[e]));
  }
  const int64_t slab = (int64_t)p_rows * hop;
  const int64_t o = (int64_t)p * hop + n0;
  *reinterpret_cast<uint4*>(packed + 0 * slab + o) = *reinterpret_cast<const uint4*>(rh);
  *reinterpret_cast<uint4*>(packed + 1 * slab + o) = *reinterpret_cast<const uint4*>(ih);
  *reinterpret_cast<uint4*>(packed + 2 * slab + o) = *reinterpret_cast<const uint4*>(rl);
  *reinterpret_cast<uint4*>(packed + 3 * slab + o) = *reinterpret_cast<const uint4*>(il);
}

struct BlockPack { int n_fft, hop; };
static std::mutex g_blk_mu;
static std::unordered_map<const void*, BlockPack> g_blk;

int tc_pack_basis_block(int n_fft, int hop, void* packed, cudaStream_t stream) {
  if (!tc_block_shape_ok(n_fft, hop) || packed == nullptr) return NNAB_EINVAL;
  const int F = n_fft / 2 + 1;
  const int p_rows = block_p_rows(F);
  const int64_t threads = (int64_t)p_rows * (hop / 8);
  pack_block_basis_kernel<<<(unsigned)ceil_div64(threads, 256), 256, 0, stream>>>(
      n_fft, hop, F, p_rows, (__nv_bfloat16*)packed);
  NNAB_LAUNCH_CHECK();
  {
    std::lock_guard<std::mutex> lk(g_blk_mu);
    g_blk[packed] = BlockPack{n_fft, hop};
  }
  mark_packed(packed, PACK_BLOCK);
  return NNAB_OK;
}

// ---------------------------------------------------------------------------
// epilogue: one warp = one TMEM lane quarter (32 consecutive block rows) x a range of 8-column chunks.
// The body of a chunk is straight-line code (no branches between the TMEM load and the stores), so
// the 8 bins' dependency chains (3-tap filter -> shuffles -> twiddles -> magnitude) interleave: with
// one or two warps per scheduler the epilogue is latency-bound, not issue-bound.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));  // <= 1 ulp-ish: far below the 1e-4 bar
  return r;
}

// fire-and-forget fp32 add, predicated (no branch: the chunk body stays one basic block)
__device__ __forceinline__ void red_add_if(float* addr, float v, bool on) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %2, 0;\n\t"
      "@p red.global.add.f32 [%0], %1;\n\t}"
      ::"l"(addr), "f"(v), "r"((int)on)
      : "memory");
}

template <int FMT, int R>
__device__ __forceinline__ void epilogue_tile_block(const TcbParams& p, uint32_t trow, int64_t g,
                                                    int lane, int n_tile, int c_begin, int c_end) {
  const int nb = p.nb;
  const int64_t b = g / p.t_slots;
  const int64_t t = g - b * p.t_slots;  // frame index inside the clip = index of its first block
  const bool valid = (lane < 33 - R) && (g < p.nv) && (t < p.T);
  const int k_tile0 = n_tile * (nb - 2);  // first output bin of this tile
  constexpr int CH = (FMT == NNAB_FMT_COMPLEX) ? 2 : 1;
  float* dst = nullptr;
  float* mel = nullptr;
  if constexpr (FMT == 5) mel = p.epi.out + ((int64_t)b * p.epi.n_fb) * p.epi.T + t;
  else if constexpr (FMT != 9) dst = p.epi.out + (((int64_t)b * p.epi.out_bins + p.epi.bin_offset) * p.epi.T + t) * CH;
  MelRun run;
  // FMT 5 fast path: static action list and the default power 2 without eps; anything else (other
  // powers, trainable eps, no action list) takes the rolled MelRun path below
  const bool fast_fb = (FMT == 5) && p.epi.fb_steps != nullptr && p.epi.power == 2.0f && p.epi.eps == 0.f;
  float ma = 0.f, mb = 0.f;  // FMT 5, static action list: the two running filter sums
  int mca = -1, mcb = -1;    //   and the filters they currently belong to

  // twiddles c_k^j of the 4 residues the unrolled loop meets: output o = 8c - 2 + e is bin
  // k = k_tile0 + o, so k mod 4 = (k_tile0 + 2 + e) mod 4 (8c drops out).
  float cr[4], ci[4], c2[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = (k_tile0 + 2 + i) & 3;
    if constexpr (R == 4) {  // c = (-i)^k
      cr[i] = (m == 0) ? 1.f : ((m == 2) ? -1.f : 0.f);
      ci[i] = (m == 3) ? 1.f : ((m == 1) ? -1.f : 0.f);
    } else {
      cr[i] = 0.f; ci[i] = 0.f;
    }
    c2[i] = (m & 1) ? -1.f : 1.f;  // R = 4: c^2 = (-1)^k;  R = 2: c = (-1)^k
  }

  float wr[10], wi[10];  // packed columns 8c-2 .. 8c+7 of this row (re, im)
  wr[8] = wr[9] = wi[8] = wi[9] = 0.f;
  if (c_begin > 0) {  // a column range that starts inside the tile: seed the two carried columns
    uint32_t re[8], im[8];
    tmem_ld8(trow + (uint32_t)(8 * (c_begin - 1)), re);
    tmem_ld8(trow + (uint32_t)(nb + 8 * (c_begin - 1)), im);
    tmem_ld_wait();
    wr[8] = __uint_as_float(re[6]); wr[9] = __uint_as_float(re[7]);
    wi[8] = __uint_as_float(im[6]); wi[9] = __uint_as_float(im[7]);
  }
#pragma unroll 1
  for (int c = c_begin; c < c_end; ++c) {
    wr[0] = wr[8]; wr[1] = wr[9]; wi[0] = wi[8]; wi[1] = wi[9];
    int4 st[8];  // FMT 5: this chunk's filterbank actions, requested before the TMEM round trip
    if constexpr (FMT == 5) {
      if (fast_fb) {
        const int kq = k_tile0 + 8 * c - 2;
#pragma unroll
        for (int e = 0; e < 8; ++e)
          st[e] = __ldg(reinterpret_cast<const int4*>(p.epi.fb_steps) + (kq + e < 0 ? 0 : kq + e));
      }
    }
    {
      uint32_t re[8], im[8];
      tmem_ld8(trow + (uint32_t)(8 * c), re);
      tmem_ld8(trow + (uint32_t)(nb + 8 * c), im);
      tmem_ld_wait();
#pragma unroll
      for (int e = 0; e < 8; ++e) { wr[e + 2] = __uint_as_float(re[e]); wi[e + 2] = __uint_as_float(im[e]); }
    }
    float xr[8], xi[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float zmr = wr[e], zmi = wi[e], z0r = wr[e + 1], z0i = wi[e + 1], zpr = wr[e + 2],
                  zpi = wi[e + 2];
      const float sr = zmr + zpr, si = zmi + zpi;
      const float ar = 0.5f * z0r, ai = 0.5f * z0i;
      if constexpr (R == 4) {
        const float dr = zmr - zpr, di = zmi - zpi;
        const float v0r = fmaf(-0.25f, sr, ar), v0i = fmaf(-0.25f, si, ai);
        float v2r = fmaf(0.25f, sr, ar), v2i = fmaf(0.25f, si, ai);
        float v1r = fmaf(0.25f, di, ar), v1i = fmaf(-0.25f, dr, ai);   // a - (i/4) D
        float v3r = fmaf(-0.25f, di, ar), v3i = fmaf(0.25f, dr, ai);   // a + (i/4) D
        v1r = __shfl_down_sync(0xffffffffu, v1r, 1); v1i = __shfl_down_sync(0xffffffffu, v1i, 1);
        v2r = __shfl_down_sync(0xffffffffu, v2r, 2); v2i = __shfl_down_sync(0xffffffffu, v2i, 2);
        v3r = __shfl_down_sync(0xffffffffu, v3r, 3); v3i = __shfl_down_sync(0xffffffffu, v3i, 3);
        const float qr = cr[e & 3], qi = ci[e & 3], q2 = c2[e & 3];
        // X = V0 + c V1 + c^2 V2 + conj(c) V3
        xr[e] = v0r + (qr * v1r - qi * v1i) + q2 * v2r + (qr * v3r + qi * v3i);
        xi[e] = v0i + (qr * v1i + qi * v1r) + q2 * v2i + (qr * v3i - qi * v3r);
      } else {
        const float v0r = fmaf(-0.25f, sr, ar), v0i = fmaf(-0.25f, si, ai);
        float v1r = fmaf(0.25f, sr, ar), v1i = fmaf(0.25f, si, ai);
        v1r = __shfl_down_sync(0xffffffffu, v1r, 1); v1i = __shfl_down_sync(0xffffffffu, v1i, 1);
        const float q2 = c2[e & 3];
        xr[e] = fmaf(q2, v1r, v0r);
        xi[e] = fmaf(q2, v1i, v0i);
      }
    }
    const int k0 = k_tile0 + 8 * c - 2;          // bin of e = 0 (outputs -2, -1 of chunk 0 do not exist)
    const int e_lo = (c == 0) ? 2 : 0;
    if constexpr (FMT == NNAB_FMT_MAGNITUDE || FMT == NNAB_FMT_COMPLEX || FMT == 4) {
      float* q = dst + (int64_t)k0 * p.epi.T * CH;
      const int64_t step = p.epi.T * CH;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const bool ok = valid && e >= e_lo && (k0 + e) < p.epi.F;
        if constexpr (FMT == NNAB_FMT_COMPLEX) {
          if (ok) *reinterpret_cast<float2*>(q) = make_float2(xr[e], xi[e]);
        } else {
          float pw = __fadd_rn(__fmul_rn(xr[e], xr[e]), __fmul_rn(xi[e], xi[e]));
          if (p.epi.eps != 0.f) pw = __fadd_rn(pw, p.epi.eps);
          float v;
          if constexpr (FMT == NNAB_FMT_MAGNITUDE) {
            v = sqrt_approx(pw);
          } else {  // |X| ** power (mel.py:186); ** 2 is the power spectrum itself to 1 ulp
            v = (p.epi.power == 2.0f) ? pw
                : ((p.epi.power == 1.0f) ? sqrt_approx(pw) : powf(sqrt_approx(pw), p.epi.power));
          }
          if (ok) *q = v;
        }
        q += step;
      }
    } else if constexpr (FMT == 9) {
      // operand planes of the dense-filterbank GEMM (FMT_PLANES): frame (b, t) is row b * T + t, the 8
      // packed columns of chunk c of tile n sit at nb * n + 8 c (16-byte aligned: nb is a multiple of 8),
      // |X| ** power as bf16 hi / lo.  The two columns a tile repeats from its left neighbour and the bins
      // past F are written as zeros (the re-indexed bank has zero rows there).
      __align__(16) __nv_bfloat16 hi[8];
      __align__(16) __nv_bfloat16 lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float pw = __fadd_rn(__fmul_rn(xr[e], xr[e]), __fmul_rn(xi[e], xi[e]));
        if (p.epi.eps != 0.f) pw = __fadd_rn(pw, p.epi.eps);
        float v = (p.epi.power == 2.0f) ? pw
                  : ((p.epi.power == 1.0f) ? sqrt_approx(pw) : powf(sqrt_approx(pw), p.epi.power));
        if (e < e_lo || (k0 + e) >= p.epi.F) v = 0.f;
        split_bf16(v, hi[e], lo[e]);
      }
      if (valid) {
        __nv_bfloat16* q = reinterpret_cast<__nv_bfloat16*>(p.epi.out) +
                           (b * p.epi.T + t) * (int64_t)p.epi.planes_pitch + (int64_t)nb * n_tile + 8 * c;
        *reinterpret_cast<uint4*>(q) = *reinterpret_cast<const uint4*>(hi);
        *reinterpret_cast<uint4*>(q + p.epi.planes_stride) = *reinterpret_cast<const uint4*>(lo);
      }
    } else if constexpr (FMT == 5) {
      if (fast_fb) {
        // banded filterbank, static action list: branch-free, two running sums per row.
        // Bins past F have neutral table entries (and zero basis rows); the two columns of chunk 0
        // that belong to the previous tile contribute with power 0.
        if (c == 0) { xr[0] = xi[0] = xr[1] = xi[1] = 0.f; }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int4 raw = st[e];
          // power == 2 (the default, mel.py:186: |X| ** 2): the power spectrum itself, to 1 ulp
          const float pw = __fadd_rn(__fmul_rn(xr[e], xr[e]), __fmul_rn(xi[e], xi[e]));
          // a filter ends at ~1 bin in 6 (and at the same bins for every row): one warp-uniform test
          // on the packed flush word keeps the address / predicate / RED code off the common path
          if (__any_sync(0xffffffffu, raw.z != -1)) {
            const int fa = (int)(short)(raw.z & 0xffff), fb = (int)(short)((unsigned)raw.z >> 16);
            red_add_if(mel + (int64_t)fa * p.epi.T, ma, fa >= 0 && valid);
            red_add_if(mel + (int64_t)fb * p.epi.T, mb, fb >= 0 && valid);
            ma = fa >= 0 ? 0.f : ma;
            mb = fb >= 0 ? 0.f : mb;
          }
          ma = fmaf(__int_as_float(raw.x), pw, ma);
          mb = fmaf(__int_as_float(raw.y), pw, mb);
        }
        mca = (int)(short)(st[7].w & 0xffff);  // filters the two sums belong to after this chunk
        mcb = (int)(short)((unsigned)st[7].w >> 16);
      } else {
#pragma unroll 1
        for (int e = e_lo; e < 8; ++e) {
          const int k = k0 + e;
          if (k >= p.epi.F) break;  // warp-uniform
          float re = xr[0], im = xi[0];
#pragma unroll
          for (int j = 1; j < 8; ++j) { re = (e == j) ? xr[j] : re; im = (e == j) ? xi[j] : im; }
          run.add(p.epi, mel, valid, k, epi_power(p.epi, re, im));
        }
      }
    } else {
      // atan2f tail: rolled per bin (code size), after the straight-line part
#pragma unroll 1
      for (int e = e_lo; e < 8; ++e) {
        const int k = k0 + e;
        if (k >= p.epi.F) break;  // warp-uniform
        // dynamic index into xr/xi would spill: select with a short unrolled scan
        float re = xr[0], im = xi[0];
#pragma unroll
        for (int j = 1; j < 8; ++j) { re = (e == j) ? xr[j] : re; im = (e == j) ? xi[j] : im; }
        if (valid) epi_store_fmt<FMT>(p.epi, dst, k, re, im);
      }
    }
  }
  if constexpr (FMT == 5) {
    red_add_if(mel + (int64_t)mca * p.epi.T, ma, mca >= 0 && valid);
    red_add_if(mel + (int64_t)mcb * p.epi.T, mb, mcb >= 0 && valid);
  }
  if constexpr (FMT == 5) run.flush(p.epi, mel, valid);
}

// epilogue warps: 2 per TMEM lane quarter (column halves); 3 for the fused filterbank, whose longer
// per-bin chain needs the extra warp per scheduler to stay under the MMA time of a tile
template <int FMT> struct TcbCfg {
  static constexpr int PARTS = (FMT == 5) ? FB_EPI_PARTS : 2;
  static constexpr int EPI_WARPS = 4 * PARTS;
  static constexpr int THREADS = 128 + 32 * EPI_WARPS;  // warps 0-3: TMA, MMA, TMEM alloc, idle
};

template <int FMT, int R>
__global__ void __launch_bounds__(TcbCfg<FMT>::THREADS, 1)
framed_tcb_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                  const TcbParams p) {
  constexpr int BK = TCB_BK, STAGES = TCB_STAGES;
  constexpr int FW = 33 - R;  // frames per warp quarter
  using S = TcbSmem;
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
      mbar_init(tempty_bar(a), 2 * TcbCfg<FMT>::EPI_WARPS);  // epilogue warps x 2 CTAs
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

  const int num_tiles = p.num_m_pairs * p.num_n_tiles;
  const int nb = p.nb;
  const uint32_t b_bytes = (uint32_t)nb * BK * 2;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        const int m_pair = tile / p.num_n_tiles;
        const int n_tile = tile - m_pair * p.num_n_tiles;
        const int m0 = (2 * m_pair + (int)cta) * (4 * FW);
        const int n0 = n_tile * (nb - 2);
        for (int kb = 0; kb < p.kb_n; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sb = base + stage * S::STAGE_BYTES;
          mbar_expect_tx_remote(full_bar(stage), 0, (p.two_term ? 1 : 2) * S::A_BYTES + 2 * b_bytes);
          const int k0 = kb * BK;
#pragma unroll
          for (int q = 0; q < 4; ++q) {  // 32-row boxes, row origins FW apart
            tma_load_3d_2sm(sb + (uint32_t)q * 32u * BK * 2u, &tm_a, full_bar(stage), k0,
                            m0 + q * FW, 0);
            if (!p.two_term)
              tma_load_3d_2sm(sb + S::A_BYTES + (uint32_t)q * 32u * BK * 2u, &tm_a, full_bar(stage), k0,
                              m0 + q * FW, 1);
          }
          tma_load_3d_2sm(sb + 2 * S::A_BYTES, &tm_b, full_bar(stage), k0, n0, (int)cta);
          tma_load_3d_2sm(sb + 2 * S::A_BYTES + S::B_BYTES, &tm_b, full_bar(stage), k0, n0,
                          2 + (int)cta);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (cta == 0 && elect_one()) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((2 * nb) >> 3) << 17) |
                             ((uint32_t)((2 * TC_BM) >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * TCB_ACC_STRIDE;
        uint32_t accumulate = 0;
        for (int kb = 0; kb < p.kb_n; ++kb) {
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
    // ===================== epilogue (both CTAs, own rows) =====================
    const int quarter = warp & 3;             // TMEM lanes 32 * (warp % 4) .. + 31
    constexpr int PARTS = TcbCfg<FMT>::PARTS;  // warps per quarter, each a contiguous chunk range
    const int part = (warp - 4) >> 2;
    const int n_chunks = nb / 8;
    const int c_begin = (n_chunks * part) / PARTS, c_end = (n_chunks * (part + 1)) / PARTS;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs) {
      const int m_pair = tile / p.num_n_tiles;
      const int n_tile = tile - m_pair * p.num_n_tiles;
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const int64_t g = (int64_t)(2 * m_pair + (int)cta) * (4 * FW) + quarter * FW + lane;
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                            (uint32_t)acc * TCB_ACC_STRIDE;
      epilogue_tile_block<FMT, R>(p, trow, g, lane, n_tile, c_begin, c_end);
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

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
template <int FMT, int R>
static int launch_tcb_fmt(const CUtensorMap& ma, const CUtensorMap& mb, const TcbParams& prm,
                          int n_pairs, cudaStream_t stream) {
  using S = TcbSmem;
  static std::atomic<uint64_t> configured_devs{0};  // the attribute is per device
  int cfg_dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&cfg_dev));
  if (!((configured_devs.load(std::memory_order_relaxed) >> (cfg_dev & 63)) & 1u)) {
    NNAB_CUDA_TRY(cudaFuncSetAttribute(framed_tcb_kernel<FMT, R>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
    configured_devs.fetch_or(1ull << (cfg_dev & 63), std::memory_order_relaxed);
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * n_pairs));
  cfg.blockDim = dim3(TcbCfg<FMT>::THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  NNAB_CUDA_TRY(cudaLaunchKernelEx(&cfg, framed_tcb_kernel<FMT, R>, ma, mb, prm));
  count_launch();
  return NNAB_OK;
}

template <int R>
static int launch_tcb(int fmt, const CUtensorMap& ma, const CUtensorMap& mb, const TcbParams& prm,
                      int n_pairs, cudaStream_t stream) {
  switch (fmt) {
    case NNAB_FMT_MAGNITUDE: return launch_tcb_fmt<0, R>(ma, mb, prm, n_pairs, stream);
    case NNAB_FMT_COMPLEX: return launch_tcb_fmt<1, R>(ma, mb, prm, n_pairs, stream);
    case NNAB_FMT_PHASE_ANGLE: return launch_tcb_fmt<2, R>(ma, mb, prm, n_pairs, stream);
    case FMT_POWER: return launch_tcb_fmt<4, R>(ma, mb, prm, n_pairs, stream);
    case FMT_FBANK: return launch_tcb_fmt<5, R>(ma, mb, prm, n_pairs, stream);
    case FMT_PLANES: return launch_tcb_fmt<9, R>(ma, mb, prm, n_pairs, stream);
    default: return NNAB_EINVAL;
  }
}

int launch_framed_tc_block(const FramedProblem& q, const void* packed, void* workspace,
                           size_t ws_bytes, cudaStream_t stream) {
  BlockPack bp{};
  {
    std::lock_guard<std::mutex> lk(g_blk_mu);
    auto it = g_blk.find(packed);
    if (it == g_blk.end()) return NNAB_EINVAL;
    bp = it->second;
  }
  // the basis was packed for exactly this transform: anything else is a caller bug
  if (bp.n_fft != q.K || bp.hop != q.hop || q.F != q.K / 2 + 1) return NNAB_EINVAL;
  if (q.presplit != nullptr || q.h_k_begin != nullptr || q.scale != nullptr || q.scale_all != 1.f)
    return NNAB_EINVAL;
  switch (q.fmt) {
    case NNAB_FMT_MAGNITUDE: case NNAB_FMT_COMPLEX: case NNAB_FMT_PHASE_ANGLE: case FMT_POWER:
      if (q.bin_offset != 0 || q.out_bins < q.F) return NNAB_EINVAL;
      break;
    case FMT_FBANK:
      if (q.fb_table == nullptr || q.n_fb <= 0) return NNAB_EINVAL;
      break;
    case FMT_PLANES:
      if (q.out == nullptr || q.planes_pitch <= 0 || q.planes_pitch % 8 != 0 || q.planes_stride <= 0 ||
          q.planes_stride % 8 != 0 || ((uintptr_t)q.out & 15u) != 0)
        return NNAB_EINVAL;
      break;
    default: return NNAB_EINVAL;
  }
  const size_t need = tc_workspace_bytes(q.B, q.L, q.K, q.hop, q.pad);
  if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
  if (q.B > 65535) return NNAB_EUNSUPPORTED;

  const int R = q.K / q.hop;
  const SplitGeom g = split_geom(q.B, q.L, q.K, q.hop, q.pad);
  __nv_bfloat16* planes =
      reinterpret_cast<__nv_bfloat16*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  const bool two = two_term(q);
  int rc = tc_pad_split(q.x, q.x_dtype, q.B, q.L, q.x_pitch, q.K, q.hop, q.pad, q.pad_mode, planes, stream,
                        two);
  if (rc) return rc;

  int dev = 0, sms = 148;
  NNAB_CUDA_TRY(cudaGetDevice(&dev));
  NNAB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  sms -= sm_reserve();
  if (sms < 2) sms = 2;

  int nb = block_choose_nb(q.F);
  if (q.fmt == FMT_FBANK && q.fb_steps != nullptr && q.fb_nb_mask != 0) {
    // run-to-run identical filterbank sums: with at most two partial sums per filter the atomic
    // adds commute.  The table builder replayed the range cuts for every tile width; take the
    // cheapest width that qualifies (fewest padded columns), else keep the default.
    int best = -1, best_cost = 1 << 30;
    for (int i = 0; i < 13; ++i) {
      if (!((q.fb_nb_mask >> i) & 1)) continue;
      const int c = 32 + 8 * i;
      const int cost = block_n_tiles(q.F, c) * (c + 6);
      if (cost < best_cost) { best_cost = cost; best = c; }
    }
    if (best > 0) nb = best;
  }
  const int n_tiles = block_n_tiles(q.F, nb);
  const int p_rows = block_p_rows(q.F);
  CUtensorMap ma, mb;
  rc = encode_3d(&ma, planes, (uint64_t)q.hop, (uint64_t)g.rows, 2, (uint64_t)q.hop * 2,
                 (uint64_t)g.plane_stride * 2, 64, 32, 64);
  if (rc) return rc;
  rc = encode_3d(&mb, const_cast<void*>(packed), (uint64_t)q.hop, (uint64_t)p_rows, 4,
                 (uint64_t)q.hop * 2, (uint64_t)p_rows * q.hop * 2, 64, (uint32_t)nb, 64);
  if (rc) return rc;

  TcbParams prm{};
  const int frames_per_cta = 4 * (33 - R);
  const int64_t cta_tiles = ceil_div64(g.nv, frames_per_cta);
  prm.num_m_pairs = (int)((cta_tiles + 1) / 2);
  prm.num_n_tiles = n_tiles;
  prm.nb = nb;
  prm.kb_n = q.hop / 64;
  prm.two_term = two ? 1 : 0;
  prm.nv = g.nv;
  prm.t_slots = g.t_slots;
  prm.T = q.T;
  prm.epi.scale = nullptr; prm.epi.scale_all = 1.f; prm.epi.fmt = q.fmt;
  prm.epi.eps = q.eps; prm.epi.power = q.power; prm.epi.out = q.out; prm.epi.T = q.T;
  prm.epi.out_bins = q.out_bins; prm.epi.bin_offset = q.bin_offset; prm.epi.F = q.F;
  prm.epi.fb_table = q.fb_table; prm.epi.n_fb = q.n_fb; prm.epi.fb_steps = q.fb_steps;
  prm.epi.raw = nullptr; prm.epi.raw_plane = 0;
  prm.epi.ola_pitch = 0; prm.epi.ola_hop = 0;
  prm.epi.planes_stride = q.planes_stride; prm.epi.planes_pitch = q.planes_pitch;
  if (q.fmt == FMT_PLANES && (int64_t)n_tiles * nb > q.planes_pitch) return NNAB_EINVAL;
  const int64_t ptiles = (int64_t)prm.num_m_pairs * n_tiles;
  const int n_pairs = (int)(ptiles < sms / 2 ? ptiles : sms / 2);
  add_exec_flops((two ? 2.0 : 3.0) * 2.0 * (double)ptiles * (2 * TC_BM) * (2 * nb) * q.hop);
  return R == 4 ? launch_tcb<4>(q.fmt, ma, mb, prm, n_pairs, stream)
                : launch_tcb<2>(q.fmt, ma, mb, prm, n_pairs, stream);
}

}  // namespace nnab
