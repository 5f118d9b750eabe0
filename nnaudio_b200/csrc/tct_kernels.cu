// "Tall-A" framed contraction for long, nested banks (CQT1992v2: features/cqt.py:749-750) on tcgen05.
//
// The A operand of the framed GEMM is a Toeplitz matrix: K block kb of frame m holds the samples
// [m*hop + 64 kb, +64).  With 64 | hop and HB = hop / 64, block kb = HB*r + c of frame m is column
// block c of plane row m + r -- so ONE shared-memory block of (128 + r_span) rows x 64 columns serves
// every K block of column c: the MMA of shift r reads the same bytes through a descriptor that
// starts r rows further down.  (Hardware probe csrc/tc_probe.cu, profiles/r02_probe_rowoffset.json:
// a K-major SWIZZLE_128B descriptor may start at ANY 128-byte row of a TMA-written block, descriptor
// base-offset field 0.)  Per tile the A bytes fetched from L2 drop from n_blocks * 32 KB to
// HB * ~44 KB (cfg3: 11.4 MB -> 0.35 MB per 256-frame tile); what remains on the shared-memory port
// is the MMA's own operand read.
//
// Everything else follows the per-K-block-width kernel (framed_tc2v_kernel, tc_kernels.cu): packed
// rows in 8-bin (re | im) groups, each K block issues MMAs of width N = 16 * groups(kb), B rows by
// 32- / 8-row TMA boxes, CTA pairs (cta_group::2), bf16 hi/lo split (3 MMAs per K16 step).
//
// Accuracy / determinism: the K range is cut per column block (<= 64 K blocks per TMEM accumulation
// chain, as the split-K path of the other kernels), but the partial sums never leave the SM: the
// epilogue warps keep the running (re, im) sums of their bins in registers across the column blocks
// of a tile and write the final format once.  No scratch, no atomics, no finalize kernel.
#include <cuda.h>
#include <cuda_bf16.h>
#include <atomic>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "epilogue.cuh"
#include "tc_ptx.cuh"
#include "tc_host.cuh"
#include "tc_decim.cuh"

namespace nnab {

constexpr int TCT_BK = 64;
constexpr int TCT_B_STAGES = 4;
constexpr int TCT_A_ROWS = 192;      // 128 frames + up to 64 row shifts
constexpr int TCT_B_ROWS = 96;       // rows one CTA stages per K block (8 * groups, groups <= 12)
constexpr int TCT_MAX_COLS = 16;     // hop / 64
constexpr int TCT_MAX_KB = 512;
constexpr int TCT_EPI_WARPS = 8;
constexpr int TCT_THREADS = 128 + 32 * TCT_EPI_WARPS;
constexpr int TCT_GROUPS_PER_PART = 6;  // 2 epilogue warps per TMEM lane quarter x 6 groups = 96 bins

struct TallPlan {
  int n_cols;                     // column blocks with work = accumulation chunks of a tile
  int col[TCT_MAX_COLS];          // column block index c
  int r_min[TCT_MAX_COLS];        // first active row shift of the column
  int r_cnt[TCT_MAX_COLS];        // number of active shifts (contiguous)
  int r_first[TCT_MAX_COLS];      // shift visited first: the column's widest block
  int g_max[TCT_MAX_COLS];        // its width in 8-bin groups = columns the chunk initialises
  int hb;                         // hop_eff / 64
  int a_rows;                     // rows of a tall A block (128 + widest shift span, multiple of 8)
  int col_off[TCT_MAX_COLS];      // first entry of the column in `order`
  uint16_t order[TCT_MAX_KB];     // K blocks in visiting order, column after column (widest block first)
  uint8_t shift[TCT_MAX_KB];      // row shift (kb - c) / hb of the same entries, relative to r_min
  uint8_t groups[TCT_MAX_KB];     // 8-bin groups K block kb reaches (0 = inactive)
};

struct TctParams {
  int num_m_tiles;                // 256-frame pair tiles (per frame phase)
  int n_phases;                   // frames t = s * n_phases + p: phase p reads the planes shifted by p * hop
  int two_term;                   // bf16 input: the A lo plane is zero -- neither loaded nor multiplied
  int64_t nv, t_slots, T;         // per phase: virtual frames, frames per clip slot; T = frames of the output
  EpiParams epi;
  float* sk_scratch;              // balanced schedule only: partial sums of the tiles two pairs share
  uint32_t* sk_flags;             //   one word per (slot, CTA, epilogue warp), zeroed before the launch
};

// Work of one CTA pair.  Static schedule (SK = false): tiles pair, pair + num_pairs, ... -- whole tiles,
// so a launch lasts ceil(tiles / pairs) tiles (cfg3: 463 tiles on 74 pairs = 7 rounds for 6.26 of work).
// Balanced schedule (SK = true): the (tile, column chunk) units are cut into num_pairs equal contiguous
// ranges.  A range is at least one tile long (pairs <= tiles), so a tile is shared by at most two pairs:
// the pair that owns its LAST chunks meets it first, parks its register sums in `sk_scratch` and raises
// the flags; the pair that owns its FIRST chunks meets it at the end of its range, adds the parked sums in
// a fixed order (own + other: bit-repeatable) and writes the output.
constexpr int TCT_SK_WARP_VALUES = 2 * 8 * TCT_GROUPS_PER_PART;                      // (re, im) x 8 x 6
constexpr size_t TCT_SK_SLOT_BYTES = (size_t)2 * TCT_EPI_WARPS * TCT_SK_WARP_VALUES * 32 * sizeof(float);
constexpr size_t TCT_SK_FLAG_BYTES_PER_SLOT = (size_t)2 * TCT_EPI_WARPS * sizeof(uint32_t);

template <bool SK>
struct TallSched {
  int tile, ci_lo, ci_hi;  // the current piece: column chunks [ci_lo, ci_hi) of `tile`
  int64_t u, u_end;
  int n_cols, stride;
  __device__ TallSched(int pair, int num_pairs, int total_tiles, int n_cols_) : n_cols(n_cols_) {
    if (SK) {
      const int64_t U = (int64_t)total_tiles * n_cols;
      u = U * pair / num_pairs;
      u_end = U * (pair + 1) / num_pairs;
      stride = 0;
    } else {
      u = pair;
      u_end = total_tiles;
      stride = num_pairs;
    }
  }
  __device__ bool next() {
    if (u >= u_end) return false;
    if (SK) {
      tile = (int)(u / n_cols);
      ci_lo = (int)(u - (int64_t)tile * n_cols);
      const int64_t rem = u_end - (int64_t)tile * n_cols;
      ci_hi = rem < n_cols ? (int)rem : n_cols;
      u = (int64_t)tile * n_cols + ci_hi;
    } else {
      tile = (int)u;
      ci_lo = 0;
      ci_hi = n_cols;
      u += stride;
    }
    return true;
  }
};

// Bounded spin on a flag word another CTA pair raises (release / acquire at GPU scope).
__device__ __forceinline__ void sk_wait_flag(const uint32_t* flag) {
  unsigned long long t0 = 0;
  uint32_t spins = 0, v;
  for (;;) {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if (v != 0u) return;
    if ((++spins & 0x3FFu) == 0) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) {  // 4 s
        printf("nnab: stream-K flag wait timeout (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void sk_raise_flag(uint32_t* flag) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(1u) : "memory");
}

struct TctSmem {
  static constexpr uint32_t A_PLANE = TCT_A_ROWS * TCT_BK * 2;   // 24 KB
  static constexpr uint32_t A_BUF = 2 * A_PLANE;                 // hi + lo
  static constexpr uint32_t B_PLANE = TCT_B_ROWS * TCT_BK * 2;   // 12 KB
  static constexpr uint32_t B_STAGE = 2 * B_PLANE;
  static constexpr uint32_t B_OFFSET = 2 * A_BUF;                // two A buffers
  static constexpr uint32_t BAR_OFFSET = B_OFFSET + TCT_B_STAGES * B_STAGE;
  static constexpr uint32_t TOTAL = BAR_OFFSET + 256 + 1024;
};

template <int FMT, bool SK>
__global__ void __launch_bounds__(TCT_THREADS, 1)
framed_tc2t_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b8,
                   const __grid_constant__ CUtensorMap tm_b32, const TctParams p,
                   const __grid_constant__ TallPlan plan) {
  constexpr int BK = TCT_BK, BS = TCT_B_STAGES;
  using S = TctSmem;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + S::BAR_OFFSET;
  auto b_full = [&](int s) { return bar_base + 8u * s; };                // leader
  auto b_empty = [&](int s) { return bar_base + 8u * (BS + s); };         // per CTA
  auto a_full = [&](int a) { return bar_base + 8u * (2 * BS + a); };      // leader
  auto a_empty = [&](int a) { return bar_base + 8u * (2 * BS + 2 + a); };  // per CTA
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * BS + 4 + a); };   // per CTA
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * BS + 6 + a); };  // leader
  const uint32_t tmem_slot = bar_base + 8u * (2 * BS + 8);
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
    for (int s = 0; s < BS; ++s) {
      mbar_init(b_full(s), 2);
      mbar_init(b_empty(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(a_full(a), 2);
      mbar_init(a_empty(a), 1);
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 2 * TCT_EPI_WARPS);
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
    // ===================== TMA producer (both CTAs) =====================
    if (elect_one()) {
      int stage = 0, abuf = 0;
      uint32_t phase = 0, aphase = 0;
      TallSched<SK> it(pair, num_pairs, p.num_m_tiles * p.n_phases, plan.n_cols);
      while (it.next()) {
        const int ph = it.tile / p.num_m_tiles, m_tile = it.tile - ph * p.num_m_tiles;
        const int m0 = m_tile * (2 * TC_BM) + (int)cta * TC_BM;
        for (int ci = it.ci_lo; ci < it.ci_hi; ++ci) {
          const int c = plan.col[ci], r_min = plan.r_min[ci], r_cnt = plan.r_cnt[ci];
          // ---- the column's tall A block: rows m0 + r_min .. + a_rows, columns [64 c, 64 c + 64)
          mbar_wait(a_empty(abuf), aphase ^ 1u);
          const uint32_t ab = base + (uint32_t)abuf * S::A_BUF;
          mbar_expect_tx_remote(a_full(abuf), 0, (p.two_term ? 1u : 2u) * (uint32_t)plan.a_rows * BK * 2u);
          tma_load_4d_2sm(ab, &tm_a, a_full(abuf), c * BK, ph, m0 + r_min, 0);
          if (!p.two_term) tma_load_4d_2sm(ab + S::A_PLANE, &tm_a, a_full(abuf), c * BK, ph, m0 + r_min, 1);
          if (++abuf == 2) { abuf = 0; aphase ^= 1u; }
          // ---- the basis rows of every K block of this column
          for (int i = 0; i < r_cnt; ++i) {
            const int kb = plan.order[plan.col_off[ci] + i];
            const int rows = 8 * (int)plan.groups[kb];  // basis rows this CTA stages
            mbar_wait(b_empty(stage), phase ^ 1u);
            const uint32_t bh = base + S::B_OFFSET + (uint32_t)stage * S::B_STAGE, bl = bh + S::B_PLANE;
            mbar_expect_tx_remote(b_full(stage), 0, 2 * (uint32_t)rows * BK * 2);
            const int k0 = kb * BK, row0 = (int)cta * rows;
            int q = 0;
            for (; rows - q >= 32; q += 32) {
              tma_load_3d_2sm(bh + (uint32_t)q * BK * 2, &tm_b32, b_full(stage), k0, row0 + q, 0);
              tma_load_3d_2sm(bl + (uint32_t)q * BK * 2, &tm_b32, b_full(stage), k0, row0 + q, 1);
            }
            for (; q < rows; q += 8) {
              tma_load_3d_2sm(bh + (uint32_t)q * BK * 2, &tm_b8, b_full(stage), k0, row0 + q, 0);
              tma_load_3d_2sm(bl + (uint32_t)q * BK * 2, &tm_b8, b_full(stage), k0, row0 + q, 1);
            }
            if (++stage == BS) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (cta == 0 && elect_one()) {
      const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((2 * TC_BM) >> 4) << 24);
      int stage = 0, abuf = 0, acc = 0;
      uint32_t phase = 0, aphase = 0, acc_phase = 0;
      TallSched<SK> it(pair, num_pairs, p.num_m_tiles * p.n_phases, plan.n_cols);
      while (it.next()) {
        for (int ci = it.ci_lo; ci < it.ci_hi; ++ci) {
          const int r_cnt = plan.r_cnt[ci];
          mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
          mbar_wait(a_full(abuf), aphase);
          tcgen05_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
          const uint32_t ab = base + (uint32_t)abuf * S::A_BUF;
          uint32_t accumulate = 0;
          for (int i = 0; i < r_cnt; ++i) {
            const int kb = plan.order[plan.col_off[ci] + i];
            const uint32_t idesc = idesc0 | ((uint32_t)(2 * (int)plan.groups[kb]) << 17);  // N = 16 G
            mbar_wait(b_full(stage), phase);
            tcgen05_fence_after();
            const uint32_t bh = base + S::B_OFFSET + (uint32_t)stage * S::B_STAGE;
            const uint32_t a_row = (uint32_t)plan.shift[plan.col_off[ci] + i] * (BK * 2);  // r rows down
            if (p.two_term)
              umma_kblock_split2(d_tmem, smem_desc_lo<BK>(ab + a_row), smem_desc_lo<BK>(bh),
                                 smem_desc_lo<BK>(bh + S::B_PLANE), smem_desc_hi<BK>(), idesc, accumulate != 0);
            else
              umma_kblock_split3(d_tmem, smem_desc_lo<BK>(ab + a_row), smem_desc_lo<BK>(ab + S::A_PLANE + a_row),
                                 smem_desc_lo<BK>(bh), smem_desc_lo<BK>(bh + S::B_PLANE), smem_desc_hi<BK>(),
                                 idesc, accumulate != 0);
            accumulate = 1u;
            umma_commit_2sm(b_empty(stage));
            if (++stage == BS) { stage = 0; phase ^= 1u; }
          }
          umma_commit_2sm(a_empty(abuf));   // the column's A block is free once its MMAs retire
          umma_commit_2sm(tfull_bar(acc));  // chunk complete -> epilogue
          if (++abuf == 2) { abuf = 0; aphase ^= 1u; }
          if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: register-resident sums over the column blocks ==========
    const int quarter = warp & 3;
    const int part = (warp - 4) >> 2;  // which 6 groups of the tile's <= 12
    int acc = 0;
    uint32_t acc_phase = 0;
    float sre[TCT_GROUPS_PER_PART][8], sim[TCT_GROUPS_PER_PART][8];
    TallSched<SK> it(pair, num_pairs, p.num_m_tiles * p.n_phases, plan.n_cols);
    while (it.next()) {
      const int ph = it.tile / p.num_m_tiles, m_tile = it.tile - ph * p.num_m_tiles;
#pragma unroll
      for (int gi = 0; gi < TCT_GROUPS_PER_PART; ++gi)
#pragma unroll
        for (int j = 0; j < 8; ++j) { sre[gi][j] = 0.f; sim[gi][j] = 0.f; }
      for (int ci = it.ci_lo; ci < it.ci_hi; ++ci) {
        mbar_wait(tfull_bar(acc), acc_phase);
        tcgen05_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * 256u;
        const int g_lim = plan.g_max[ci];  // columns this chunk initialised
#pragma unroll
        for (int gi = 0; gi < TCT_GROUPS_PER_PART; ++gi) {
          const int g = part * TCT_GROUPS_PER_PART + gi;
          if (g < g_lim) {  // warp-uniform
            uint32_t re[8], im[8];
            tmem_ld8(trow + (uint32_t)(16 * g), re);
            tmem_ld8(trow + (uint32_t)(16 * g + 8), im);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              sre[gi][j] += __uint_as_float(re[j]);
              sim[gi][j] += __uint_as_float(im[j]);
            }
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(tempty_bar(acc), 0);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
      if (SK) {
        // a tile shared with a neighbour pair: its last chunks (met first, by pair + 1) are parked in
        // scratch slot `pair`, its first chunks (met last, by this pair) pick them up
        const int ew = warp - 4;
        if (it.ci_lo > 0) {
          float* dst = p.sk_scratch +
                       (((size_t)pair * 2 + cta) * TCT_EPI_WARPS + ew) * (TCT_SK_WARP_VALUES * 32) + lane;
#pragma unroll
          for (int gi = 0; gi < TCT_GROUPS_PER_PART; ++gi)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              __stcg(dst + (size_t)((gi * 8 + j) * 2) * 32, sre[gi][j]);
              __stcg(dst + (size_t)((gi * 8 + j) * 2 + 1) * 32, sim[gi][j]);
            }
          __threadfence();
          __syncwarp();
          if (lane == 0) sk_raise_flag(p.sk_flags + ((size_t)pair * 2 + cta) * TCT_EPI_WARPS + ew);
          continue;  // the neighbour writes this tile's output
        }
        if (it.ci_hi < plan.n_cols) {
          const int other = pair + 1;
          if (lane == 0) sk_wait_flag(p.sk_flags + ((size_t)other * 2 + cta) * TCT_EPI_WARPS + ew);
          __syncwarp();
          __threadfence();
          const float* src = p.sk_scratch +
                             (((size_t)other * 2 + cta) * TCT_EPI_WARPS + ew) * (TCT_SK_WARP_VALUES * 32) + lane;
#pragma unroll
          for (int gi = 0; gi < TCT_GROUPS_PER_PART; ++gi)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              sre[gi][j] += __ldcg(src + (size_t)((gi * 8 + j) * 2) * 32);
              sim[gi][j] += __ldcg(src + (size_t)((gi * 8 + j) * 2 + 1) * 32);
            }
        }
      }
      // ---- final format, once per tile
      const int64_t g_row = (int64_t)m_tile * (2 * TC_BM) + (int64_t)cta * TC_BM + quarter * 32 + lane;
      const int64_t b = g_row / p.t_slots;
      const int64_t t = (g_row - b * p.t_slots) * p.n_phases + ph;  // frame index in the output
      if (g_row < p.nv && t < p.T) {
        constexpr int CH = (FMT == NNAB_FMT_COMPLEX || FMT == NNAB_FMT_PHASE_UNIT) ? 2 : 1;
        float* dst = p.epi.out + (((int64_t)b * p.epi.out_bins + p.epi.bin_offset) * p.epi.T + t) * CH;
#pragma unroll
        for (int gi = 0; gi < TCT_GROUPS_PER_PART; ++gi) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int f = 8 * (part * TCT_GROUPS_PER_PART + gi) + j;
            if (f < p.epi.F) epi_store_fmt<FMT>(p.epi, dst, f, sre[gi][j], sim[gi][j]);
          }
        }
      }
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
// frame phases: hop < 64 runs as P = 64 / hop interleaved problems with 64-sample rows, phase p
// reading the planes p * hop samples further on (16-byte aligned for hop >= 8)
static int tall_phases(int hop) { return hop >= 64 ? 1 : 64 / hop; }

bool tc_tall_problem_ok(const FramedProblem& q) {
  if (q.hop >= 64) {
    if (q.hop % 64 != 0 || q.hop / 64 > TCT_MAX_COLS) return false;
  } else if (q.hop < 8 || 64 % q.hop != 0) {
    return false;
  }
  if (q.F > 8 * 2 * TCT_GROUPS_PER_PART || q.K > 64 * TCT_MAX_KB) return false;
  if (q.presplit != nullptr && q.presplit_t_slots <= 0) return false;  // needs the explicit geometry
  if (q.presplit == nullptr && q.hop < 64) return false;               // phases only on shared planes
  return q.fmt == NNAB_FMT_MAGNITUDE || q.fmt == NNAB_FMT_COMPLEX || q.fmt == NNAB_FMT_PHASE_UNIT;
}

// NNAB_TALL_BALANCE=1|0: balanced (shared-tile) schedule of framed_tc2t_kernel on / off.
static bool tall_balance_enabled() {
  if (const char* e = getenv("NNAB_TALL_BALANCE")) return atoi(e) != 0;
  // on by default: GPU-verified (profiles/r02b_*: bit-repeatable, 2e-6 of the static schedule, 1e-4 of the
  // oracle; cfg3 0.889 -> 0.822 ms per step)
  return true;
}

// Returns NNAB_EUNSUPPORTED when the bank does not fit the tall layout (caller falls back).
static int build_tall_plan(const FramedProblem& q, TallPlan* plan) {
  const int hop_eff = q.hop >= 64 ? q.hop : 64;
  const int hb = hop_eff / 64;
  const int nkb = (q.K + 63) / 64;
  memset(plan, 0, sizeof(*plan));
  plan->hb = hb;
  int kb_lo = nkb, kb_hi = -1;
  for (int kb = 0; kb < nkb; ++kb) {
    int gmax = 0;
    if (q.h_k_begin == nullptr || q.h_k_end == nullptr) {
      gmax = (q.F + 7) / 8;  // no support information: every block reaches every bin
    } else {
      for (int f = 0; f < q.F; ++f) {
        const int lo = q.h_k_begin[f], hi = q.h_k_end[f];
        if (hi > lo && hi > kb * 64 && lo < kb * 64 + 64) gmax = gmax > f / 8 + 1 ? gmax : f / 8 + 1;
      }
    }
    plan->groups[kb] = (uint8_t)gmax;
    if (gmax > 0) { kb_lo = kb < kb_lo ? kb : kb_lo; kb_hi = kb; }
  }
  if (kb_hi < 0) return NNAB_EUNSUPPORTED;
  // inactive blocks inside the active interval (a gap in every wavelet) still get the narrowest MMA
  for (int kb = kb_lo; kb <= kb_hi; ++kb)
    if (plan->groups[kb] == 0) plan->groups[kb] = 1;
  int n = 0, span = 1, n_order = 0;
  for (int c = 0; c < hb; ++c) {
    const int r_lo = (kb_lo - c + hb - 1) / hb > 0 ? (kb_lo - c + hb - 1) / hb : 0;
    const int r_hi = (kb_hi - c) >= 0 ? (kb_hi - c) / hb : -1;
    if (r_hi < r_lo) continue;
    if (r_hi - r_lo + 1 > 64) return NNAB_EUNSUPPORTED;  // A block rows: 128 + 63
    span = r_hi - r_lo + 1 > span ? r_hi - r_lo + 1 : span;
    int best = r_lo;
    for (int r = r_lo; r <= r_hi; ++r)
      if (plan->groups[r * hb + c] > plan->groups[best * hb + c]) best = r;
    plan->col[n] = c;
    plan->r_min[n] = r_lo;
    plan->r_cnt[n] = r_hi - r_lo + 1;
    plan->r_first[n] = best;
    plan->g_max[n] = plan->groups[best * hb + c];
    plan->col_off[n] = n_order;
    {
      // visiting order: the widest block first (it initialises every TMEM column the chunk touches),
      // then alternately above / below it
      const int cnt = r_hi - r_lo + 1, below = best - r_lo, above = r_hi - best;
      const int pairs = below < above ? below : above;
      for (int i = 0; i < cnt; ++i) {
        int r;
        if (i == 0) r = best;
        else if (i <= 2 * pairs) r = (i & 1) ? best + (i + 1) / 2 : best - i / 2;
        else r = above > below ? best + pairs + (i - 2 * pairs) : best - pairs - (i - 2 * pairs);
        plan->shift[n_order] = (uint8_t)(r - r_lo);
        plan->order[n_order++] = (uint16_t)(r * hb + c);
      }
    }
    ++n;
  }
  plan->n_cols = n;
  plan->a_rows = round_up_i(128 + span - 1, 8);
  return n > 0 ? NNAB_OK : NNAB_EUNSUPPORTED;
}

template <int FMT, bool SK>
static int launch_tc2t_fmt(const CUtensorMap& ma, const CUtensorMap& mb8, const CUtensorMap& mb32,
                           const TctParams& prm, const TallPlan& plan, int n_pairs,
                           cudaStream_t stream) {
  using S = TctSmem;
  static std::atomic<uint64_t> configured_devs{0};  // the attribute is per device
  int cfg_dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&cfg_dev));
  if (!((configured_devs.load(std::memory_order_relaxed) >> (cfg_dev & 63)) & 1u)) {
    NNAB_CUDA_TRY(cudaFuncSetAttribute(framed_tc2t_kernel<FMT, SK>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
    configured_devs.fetch_or(1ull << (cfg_dev & 63), std::memory_order_relaxed);
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * n_pairs));
  cfg.blockDim = dim3(TCT_THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  NNAB_CUDA_TRY(cudaLaunchKernelEx(&cfg, framed_tc2t_kernel<FMT, SK>, ma, mb8, mb32, prm, plan));
  count_launch();
  return NNAB_OK;
}

// `packed`: the 8-bin-group layout of tc_pack_basis_varn.  Returns NNAB_EUNSUPPORTED (nothing
// enqueued) when the bank does not fit; the caller then runs framed_tc2v_kernel.
int launch_framed_tc_tall(const FramedProblem& q, const void* packed, void* workspace, size_t ws_bytes,
                          cudaStream_t stream) {
  if (!tc_tall_problem_ok(q)) return NNAB_EUNSUPPORTED;
  if (const char* e = getenv("NNAB_TALL")) {
    if (atoi(e) == 0) return NNAB_EUNSUPPORTED;  // A/B switch: per-K-block-width kernel without A reuse
  }
  TallPlan plan;
  int rc = build_tall_plan(q, &plan);
  if (rc) return rc;
  if (q.B > 65535) return NNAB_EUNSUPPORTED;
  const int P = tall_phases(q.hop);
  const int hop_eff = q.hop >= 64 ? q.hop : 64;
  const int kpad = round_up_i(q.K, 64);
  const int rows_w = 16 * ((q.F + 7) / 8);
  __nv_bfloat16* planes;
  int64_t t_slots, nv, plane_stride;
  if (q.presplit != nullptr) {
    // caller-managed planes (pyramid levels): clip slot = presplit_t_slots frames of `hop` samples
    planes = reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(q.presplit));
    const int64_t pitch = q.presplit_t_slots * q.hop;
    if (pitch % hop_eff != 0) return NNAB_EUNSUPPORTED;
    t_slots = pitch / hop_eff;  // frames of ONE phase per clip slot
    plane_stride = q.presplit_plane_stride;
  } else {
    const size_t need = tc_workspace_bytes(q.B, q.L, q.K, q.hop, q.pad);
    if (workspace == nullptr || ws_bytes < need) return NNAB_EWORKSPACE;
    const SplitGeom g = split_geom(q.B, q.L, q.K, q.hop, q.pad);
    planes = reinterpret_cast<__nv_bfloat16*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    rc = tc_pad_split(q.x, q.x_dtype, q.B, q.L, q.x_pitch, q.K, q.hop, q.pad, q.pad_mode, planes, stream,
                      two_term(q));
    if (rc) return rc;
    t_slots = g.t_slots;
    plane_stride = g.plane_stride;
  }
  nv = q.B * t_slots;
  // frames of a phase that exist: ceil((T - p) / P) <= t_slots by construction of the planes
  int dev = 0, sms = 148;
  NNAB_CUDA_TRY(cudaGetDevice(&dev));
  NNAB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  sms -= sm_reserve();
  if (sms < 2) sms = 2;

  CUtensorMap ma, mb8, mb32;
  {
    // A: {column within a row, frame phase, row, plane}; rows past the end: zero fill
    const int64_t rows = (plane_stride - (int64_t)(P - 1) * q.hop) / hop_eff;
    const uint64_t dims[4] = {(uint64_t)hop_eff, (uint64_t)P, (uint64_t)rows, 2};
    const uint64_t strides[3] = {(uint64_t)(P > 1 ? q.hop : hop_eff) * 2, (uint64_t)hop_eff * 2,
                                 (uint64_t)plane_stride * 2};
    const uint32_t box[3] = {64, 1, (uint32_t)plan.a_rows};
    rc = encode_4d(&ma, planes, dims, strides, box);
    if (rc) return NNAB_EUNSUPPORTED;  // (e.g. a driver that rejects the overlapping phase stride)
  }
  if ((rc = encode_3d(&mb8, const_cast<void*>(packed), (uint64_t)kpad, (uint64_t)rows_w, 2,
                      (uint64_t)kpad * 2, (uint64_t)rows_w * kpad * 2, 64, 8, 64)))
    return rc;
  if ((rc = encode_3d(&mb32, const_cast<void*>(packed), (uint64_t)kpad, (uint64_t)rows_w, 2,
                      (uint64_t)kpad * 2, (uint64_t)rows_w * kpad * 2, 64, 32, 64)))
    return rc;

  TctParams prm{};
  prm.sk_scratch = nullptr;
  prm.sk_flags = nullptr;
  prm.num_m_tiles = (int)ceil_div64(nv, 2 * TC_BM);
  prm.n_phases = P;
  prm.two_term = two_term(q) ? 1 : 0;
  prm.nv = nv;
  prm.t_slots = t_slots;
  prm.T = q.T;
  prm.epi.scale = q.scale; prm.epi.scale_all = q.scale_all; prm.epi.fmt = q.fmt;
  prm.epi.eps = q.eps; prm.epi.power = q.power; prm.epi.out = q.out; prm.epi.T = q.T;
  prm.epi.out_bins = q.out_bins; prm.epi.bin_offset = q.bin_offset; prm.epi.F = q.F;
  const int64_t tiles = (int64_t)prm.num_m_tiles * P;
  int n_pairs = (int)(tiles < sms / 2 ? tiles : sms / 2);
  if (const char* e = getenv("NNAB_TALL_PAIRS")) {  // tests: force shared tiles on small problems
    const int v = atoi(e);
    if (v >= 1 && v < n_pairs) n_pairs = v;
  }
  {
    double cols = 0.0;
    for (int kb = 0; kb < TCT_MAX_KB; ++kb) cols += 16.0 * plan.groups[kb] * 64.0;
    add_exec_flops((prm.two_term ? 2.0 : 3.0) * 2.0 * (double)tiles * (2 * TC_BM) * cols);
  }
  // Balanced schedule (TallSched<true>): only when the static one leaves a ragged last round, and the
  // split-K scratch of this problem (long kernels: attach_splitk_scratch) can hold one slot per pair.
  // The pairs of a launch wait on each other, so the whole grid must be resident: n_pairs <= SMs / 2.
  bool balanced = false;
  if (tall_balance_enabled() && q.raw != nullptr && tiles > n_pairs && tiles % n_pairs != 0) {
    const size_t flag_bytes = ((size_t)n_pairs * TCT_SK_FLAG_BYTES_PER_SLOT + 255) / 256 * 256;
    const size_t have = tc_splitk_scratch_bytes(q.B, q.F, q.T, q.K);
    if (have >= flag_bytes + (size_t)n_pairs * TCT_SK_SLOT_BYTES + 256) {
      char* base = reinterpret_cast<char*>(((uintptr_t)q.raw + 255) & ~(uintptr_t)255);
      prm.sk_flags = reinterpret_cast<uint32_t*>(base);
      prm.sk_scratch = reinterpret_cast<float*>(base + flag_bytes);
      NNAB_CUDA_TRY(cudaMemsetAsync(prm.sk_flags, 0, flag_bytes, stream));
      balanced = true;
    }
  }
  if (balanced) {
    count_balanced_launch();
    switch (q.fmt) {
      case NNAB_FMT_MAGNITUDE: return launch_tc2t_fmt<0, true>(ma, mb8, mb32, prm, plan, n_pairs, stream);
      case NNAB_FMT_COMPLEX: return launch_tc2t_fmt<1, true>(ma, mb8, mb32, prm, plan, n_pairs, stream);
      case NNAB_FMT_PHASE_UNIT: return launch_tc2t_fmt<3, true>(ma, mb8, mb32, prm, plan, n_pairs, stream);
      default: return NNAB_EINVAL;
    }
  }
  switch (q.fmt) {
    case NNAB_FMT_MAGNITUDE: return launch_tc2t_fmt<0, false>(ma, mb8, mb32, prm, plan, n_pairs, stream);
    case NNAB_FMT_COMPLEX: return launch_tc2t_fmt<1, false>(ma, mb8, mb32, prm, plan, n_pairs, stream);
    case NNAB_FMT_PHASE_UNIT: return launch_tc2t_fmt<3, false>(ma, mb8, mb32, prm, plan, n_pairs, stream);
    default: return NNAB_EINVAL;
  }
}

// ===========================================================================
// FIR decimator stage of the CQT pyramid (utils.py:73-124: conv1d(x, lowpass(256), stride=2,
// padding=127)) with RESIDENT taps and tall A blocks.
//
// As in tc_kernels.cu the stage is a framed contraction: frame t of a level covers its samples
// [256 t - 128, 256 t + 384) and yields the 128 outputs y[128 t + j] through the banded Toeplitz rows
// H[j][k] = fir[k - 1 - 2 j] (K = 512, N = 128).  New here:
//   * the level lives in ONE plane set (hi / lo bf16) shared with the level's octave CQT: sample m of
//     clip b at b * pitch + pad + m with the CQT's reflect margins.  The FIR wants ZERO margins; only
//     the first / last 64 outputs of a clip see the margins, and fir_edge_fix_kernel recomputes
//     those (plus their mirror copies) afterwards.  One write + one read of 4 B per sample and level
//     instead of two differently padded copies.
//   * the signal is read through tall A blocks (see framed_tc2t_kernel): with 256-sample rows, K block
//     kb is column kb % 4 of row t + kb / 4, so 4 blocks of 129 rows x 64 columns feed all 8 K blocks
//     (pad = 128, i.e. 256-tap octave banks: the CQT's padding origin is the FIR frame origin).
//   * a 3-stage ring of (column block + its two tap blocks); the taps (256 KB) stream from L2.
// ===========================================================================
constexpr int FIR_KBLOCKS = 8;
constexpr int FIR_A_ROWS = 136;   // 128 frames + row shifts 0 / 1 (multiple of 8)
constexpr int FIR_THREADS = 128 + 32 * 8;
constexpr int FIR_STAGES = 3;

// The tap matrix H[j][k] = fir[k - 1 - 2 j] is banded: K block kb (64 samples) meets only the outputs
// j in [32 kb - 128, 32 kb + 32), i.e. the column ranges below (multiples of 32, 640 of 1024 column
// blocks).  Each K block issues MMAs of exactly that width into TMEM columns [lo, lo + n): 37.5 % fewer
// MMA flops, and each CTA of the pair keeps only its half of every range resident: 320 rows = 80 KB.
__device__ __host__ __forceinline__ int fir_col_lo(int kb) { return kb <= 4 ? 0 : 32 * (kb - 4); }
__device__ __host__ __forceinline__ int fir_col_n(int kb) { return kb < 4 ? 32 * (kb + 1) : 32 * (8 - kb); }
// first row (of this CTA's 320) of K block kb: prefix sums of n / 2 = {16,32,48,64,64,48,32,16}
__device__ __host__ __forceinline__ int fir_row0(int kb) {
  const int pre[9] = {0, 16, 48, 96, 160, 224, 272, 304, 320};
  return pre[kb];
}

// Shared memory: resident banded taps (hi 40 KB + lo 40 KB) + a 3-deep ring of tall A blocks (one
// column block of the 256-sample rows: 136 rows x 64, hi + lo = 34 KB).  Two column loads stay in
// flight while the MMAs of a third run; the first version kept the full tap matrix (128 KB), had room
// for two A buffers only -- one load in flight -- and sat at 50 % tensor / 46 % DRAM
// (profiles/r02_ncu_cfg4_fir.txt); streaming the taps per stage instead doubled the L2->SM bytes.
struct FirSmem {
  static constexpr uint32_t B_PLANE = 320 * TCT_BK * 2;          // 40 KB
  static constexpr uint32_t A_PLANE = FIR_A_ROWS * TCT_BK * 2;   // 17 KB
  static constexpr uint32_t A_BUF = 2 * A_PLANE;
  static constexpr uint32_t A_OFFSET = 2 * B_PLANE;
  static constexpr uint32_t BAR_OFFSET = A_OFFSET + FIR_STAGES * A_BUF;
  static constexpr uint32_t TOTAL = BAR_OFFSET + 256 + 1024;
};

struct FirParams {
  int num_m_tiles;       // 256-frame pair tiles over the virtual frames b * t_slots + t
  int64_t nv, t_slots, FT;  // frames: virtual total, per clip slot, valid per clip
  DecimParams dec;
};

__global__ void __launch_bounds__(FIR_THREADS, 1)
fir_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
              const FirParams p) {
  constexpr int BK = TCT_BK, ST = FIR_STAGES;
  using S = FirSmem;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + S::BAR_OFFSET;
  const uint32_t b_full = bar_base;                                           // leader
  auto full_bar = [&](int s) { return bar_base + 8u * (1 + s); };              // leader
  auto empty_bar = [&](int s) { return bar_base + 8u * (1 + ST + s); };        // per CTA
  auto tfull_bar = [&](int a) { return bar_base + 8u * (1 + 2 * ST + a); };    // per CTA
  auto tempty_bar = [&](int a) { return bar_base + 8u * (3 + 2 * ST + a); };   // leader
  const uint32_t tmem_slot = bar_base + 8u * (5 + 2 * ST);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta = cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_b);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(b_full, 2);
    for (int s = 0; s < ST; ++s) {
      mbar_init(full_bar(s), 2);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 2 * 8);
    }
    fence_barrier_init();
  }
  cluster_sync_all();
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, 256);
    tmem_relinquish_2sm();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (elect_one()) {
      // resident taps: for every K block this CTA's half of the block's column range, 16-row boxes
      mbar_expect_tx_remote(b_full, 0, 2 * S::B_PLANE);
      for (int kb = 0; kb < FIR_KBLOCKS; ++kb) {
        const int half = fir_col_n(kb) / 2;
        const int j0 = fir_col_lo(kb) + (int)cta * half;  // first tap row (= output j) this CTA stages
        for (int q = 0; q < half; q += 16) {
          const uint32_t dst = base + (uint32_t)(fir_row0(kb) + q) * (BK * 2);
          tma_load_3d_2sm(dst, &tm_b, b_full, kb * BK, j0 + q, 0);
          tma_load_3d_2sm(dst + S::B_PLANE, &tm_b, b_full, kb * BK, j0 + q, 1);
        }
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int m_tile = pair; m_tile < p.num_m_tiles; m_tile += num_pairs) {
        const int m0 = m_tile * (2 * TC_BM) + (int)cta * TC_BM;
        for (int ci = 0; ci < 4; ++ci) {
          const int c = (ci + 3) & 3;  // 3, 0, 1, 2: the tile's first MMA (kb = 3) is full width
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t ab = base + S::A_OFFSET + (uint32_t)stage * S::A_BUF;
          mbar_expect_tx_remote(full_bar(stage), 0, S::A_BUF);
          tma_load_3d_2sm(ab, &tm_a, full_bar(stage), c * BK, m0, 0);
          tma_load_3d_2sm(ab + S::A_PLANE, &tm_a, full_bar(stage), c * BK, m0, 1);
          if (++stage == ST) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (cta == 0 && elect_one()) {
      const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((2 * TC_BM) >> 4) << 24);
      mbar_wait(b_full, 0);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int m_tile = pair; m_tile < p.num_m_tiles; m_tile += num_pairs) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        uint32_t accumulate = 0;
        for (int ci = 0; ci < 4; ++ci) {
          const int c = (ci + 3) & 3;
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t ab = base + S::A_OFFSET + (uint32_t)stage * S::A_BUF;
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const int kb = 4 * r + c;  // frame t reads row t + r, column block c
            const uint32_t idesc = idesc0 | ((uint32_t)(fir_col_n(kb) >> 3) << 17);
            const uint32_t d_tmem = tmem_base + (uint32_t)acc * 128u + (uint32_t)fir_col_lo(kb);
            const uint32_t a_row = (uint32_t)r * (BK * 2);
            const uint32_t bh = base + (uint32_t)fir_row0(kb) * (BK * 2), bl = bh + S::B_PLANE;
            // kb = 3 (first of a tile) covers all 128 columns and starts the accumulation
            umma_kblock_split3(d_tmem, smem_desc_lo<BK>(ab + a_row), smem_desc_lo<BK>(ab + S::A_PLANE + a_row),
                               smem_desc_lo<BK>(bh), smem_desc_lo<BK>(bl), smem_desc_hi<BK>(), idesc,
                               accumulate != 0);
            accumulate = 1u;
          }
          umma_commit_2sm(empty_bar(stage));
          if (++stage == ST) { stage = 0; phase ^= 1u; }
        }
        umma_commit_2sm(tfull_bar(acc));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3;
    const int part = (warp - 4) >> 2;  // column half of the 128 outputs
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int m_tile = pair; m_tile < p.num_m_tiles; m_tile += num_pairs) {
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const int64_t g = (int64_t)m_tile * (2 * TC_BM) + (int64_t)cta * TC_BM + quarter * 32 + lane;
      const int64_t b = g / p.t_slots;
      const int64_t tl = g - b * p.t_slots;
      const bool valid = (g < p.nv) && (tl < p.FT);
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * 128u;
      epilogue_decim(p.dec, trow, b, tl, valid, 64, 64 * part, 64 * part + 64);
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
    tmem_dealloc_2sm(tmem_base, 256);
  }
}

// Outputs whose taps reach past a clip edge: y[n] = sum_m fir[m] x[2 n + m - 127] with x = 0 outside
// [0, len_src) -- n < 64 and n >= len_out - 64 -- recomputed from the source planes (hi + lo) and
// written over what fir_tc_kernel produced from the reflect margins: the sample itself, its mirror
// copies in the destination's reflect margins, and the fp32 copy when the level keeps one.
__global__ void __launch_bounds__(128) fir_edge_fix_kernel(
    const __nv_bfloat16* __restrict__ src, int64_t src_pitch, int64_t src_plane, int src_off,
    int64_t len_src, const float* __restrict__ fir, int taps, DecimParams d) {
  // one warp per output (taps strided over the lanes, shuffle reduction): grid (32, B), 4 warps each
  const int64_t b = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);  // 0..63: head outputs, 64..127: tail outputs
  const int64_t n = (i < 64) ? i : d.len_out - 128 + i;
  if (i >= 64 && n < 64) return;  // short clip: the head half already covers it
  if (n < 0 || n >= d.len_out) return;
  const __nv_bfloat16* sb = src + b * src_pitch + src_off;
  float acc = 0.f;
#pragma unroll 8
  for (int m = lane; m < taps; m += 32) {  // taps / 32 independent loads in flight per lane
    const int64_t j = 2 * n + m - (taps - 1) / 2;
    const bool in = j >= 0 && j < len_src;
    const float hi = in ? __bfloat162float(sb[j]) : 0.f;
    const float lo = in ? __bfloat162float(sb[src_plane + j]) : 0.f;
    acc = fmaf(__ldg(fir + m), hi + lo, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane != 0) return;
  __nv_bfloat16 hi, lo;
  split_bf16(acc, hi, lo);
  if (d.pc != nullptr) {
    __nv_bfloat16* base = reinterpret_cast<__nv_bfloat16*>(d.pc) + b * d.pc_pitch + d.pc_off;
    base[n] = hi; base[d.pc_plane + n] = lo;
    if (d.pc_reflect) {
      if (n >= 1 && n <= d.pc_off) { base[-n] = hi; base[d.pc_plane - n] = lo; }
      if (n >= d.len_out - 1 - d.pc_off && n <= d.len_out - 2) {
        const int64_t r = 2 * (d.len_out - 1) - n;
        base[r] = hi; base[d.pc_plane + r] = lo;
      }
    }
  }
  if (d.y32 != nullptr) d.y32[b * d.y32_pitch + n] = acc;
}

// One FIR stage: source level planes (single set, samples at offset src_pad, clip pitch a multiple of
// 256) -> destination level through `dec` (pc planes with their own pad, optional fp32 copy).
int launch_fir_stage_tc(const void* src_planes, int64_t B, int64_t src_len, int64_t src_pitch,
                        int64_t src_plane_stride, int src_pad, const void* fir_packed,
                        const float* fir, int taps, const DecimParams& dec, cudaStream_t stream) {
  if (taps != 256 || src_pad != 128) return NNAB_EUNSUPPORTED;  // frame origin = row origin
  if (src_pitch % 256 != 0 || B > 65535 || dec.pf != nullptr) return NNAB_EUNSUPPORTED;
  const int64_t FT = (dec.len_out + 127) / 128;
  const int64_t t_slots = src_pitch / 256;
  if (256 * (FT + 2) > src_pitch + 256) return NNAB_EUNSUPPORTED;  // last frame's rows
  int dev = 0, sms = 148;
  NNAB_CUDA_TRY(cudaGetDevice(&dev));
  NNAB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  sms -= sm_reserve();
  if (sms < 2) sms = 2;
  CUtensorMap ma, mb;
  const int64_t rows = src_plane_stride / 256;
  int rc = encode_3d(&ma, const_cast<void*>(src_planes), 256, (uint64_t)rows, 2, 512,
                     (uint64_t)src_plane_stride * 2, 64, FIR_A_ROWS, 64);
  if (rc) return rc;
  const int kf = tc_fir_k(taps, 2);  // 512
  if (kf != 64 * FIR_KBLOCKS) return NNAB_EUNSUPPORTED;
  rc = encode_3d(&mb, const_cast<void*>(fir_packed), (uint64_t)kf, 128, 2, (uint64_t)kf * 2,
                 (uint64_t)128 * kf * 2, 64, 16, 64);
  if (rc) return rc;
  FirParams prm{};
  prm.nv = B * t_slots;
  prm.t_slots = t_slots;
  prm.FT = FT;
  prm.num_m_tiles = (int)ceil_div64(prm.nv, 2 * TC_BM);
  prm.dec = dec;
  const int n_pairs = prm.num_m_tiles < sms / 2 ? prm.num_m_tiles : sms / 2;
  static std::atomic<uint64_t> configured_devs{0};
  int cfg_dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&cfg_dev));
  if (!((configured_devs.load(std::memory_order_relaxed) >> (cfg_dev & 63)) & 1u)) {
    NNAB_CUDA_TRY(cudaFuncSetAttribute(fir_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)FirSmem::TOTAL));
    configured_devs.fetch_or(1ull << (cfg_dev & 63), std::memory_order_relaxed);
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * n_pairs));
  cfg.blockDim = dim3(FIR_THREADS);
  cfg.dynamicSmemBytes = FirSmem::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  NNAB_CUDA_TRY(cudaLaunchKernelEx(&cfg, fir_tc_kernel, ma, mb, prm));
  count_launch();
  add_exec_flops(3.0 * 2.0 * (double)prm.num_m_tiles * (2 * TC_BM) * 640.0 * 64.0);  // banded: 640 columns x 64
  // clip edges
  fir_edge_fix_kernel<<<dim3(32, (unsigned)B), 128, 0, stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(src_planes), src_pitch, src_plane_stride, src_pad, src_len,
      fir, taps, dec);
  NNAB_LAUNCH_CHECK();
  return NNAB_OK;
}


// ===========================================================================
// Octave CQT of the pyramid (utils.py:498-521 get_cqt_complex: conv1d(x, bank(<=16 bins, 256 taps), hop))
// on the level planes it shares with fir_tc_kernel.  With N = 32 columns the contraction is not an MMA
// problem but an operand-delivery problem: the dense kernel fetched 1 KB of A per frame from L2 (338 MB
// per octave whatever the level, ~80 us each) and re-fetched the bank per tile.  Here
//   * the bank (this CTA's 16 rows of every K block, hi + lo: <= 32 KB) is resident,
//   * the signal comes through tall A blocks (framed_tc2t_kernel): rows of hop_eff = max(hop, 64)
//     samples, K block kb = column kb % HB at row shift kb / HB, so a sample is fetched once per tile
//     however much the frames overlap (HB = hop_eff / 64),
//   * hop < 64 runs as P = 64 / hop interleaved frame phases through a 4-D tensor map (phase p reads
//     the planes p * hop samples further on),
//   * a 5-deep ring of column blocks keeps four loads in flight.
// Packed bank = the DENSE layout of tc_kernels.cu with bn = 32: rows [0,16) re, [16,32) negated im.
// ===========================================================================
constexpr int OCT_STAGES = 5;
constexpr int OCT_A_ROWS = 136;
constexpr int OCT_MAX_KB = 8;
constexpr int OCT_THREADS = 256;

struct OctSmem {
  static constexpr uint32_t B_KB = 16 * TCT_BK * 2;               // one K block, one plane, 16 rows: 2 KB
  static constexpr uint32_t B_PLANE = OCT_MAX_KB * B_KB;          // 16 KB
  static constexpr uint32_t A_PLANE = OCT_A_ROWS * TCT_BK * 2;    // 17 KB
  static constexpr uint32_t A_BUF = 2 * A_PLANE;
  static constexpr uint32_t A_OFFSET = 2 * B_PLANE;
  static constexpr uint32_t BAR_OFFSET = A_OFFSET + OCT_STAGES * A_BUF;
  static constexpr uint32_t TOTAL = BAR_OFFSET + 256 + 1024;
};

struct OctParams {
  int num_m_tiles;        // 256-frame pair tiles per frame phase
  int n_phases, hb, n_kb; // frame phases, column blocks per row (power of two), K blocks (K / 64)
  int hb_log2;
  int64_t nv, t_slots, T; // per phase: virtual frames, frames per clip slot; T = frames of the output
  EpiParams epi;
};

template <int FMT>
__global__ void __launch_bounds__(OCT_THREADS, 1)
octave_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const OctParams p) {
  constexpr int BK = TCT_BK, ST = OCT_STAGES;
  using S = OctSmem;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + S::BAR_OFFSET;
  const uint32_t b_full = bar_base;
  auto full_bar = [&](int s) { return bar_base + 8u * (1 + s); };
  auto empty_bar = [&](int s) { return bar_base + 8u * (1 + ST + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (1 + 2 * ST + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (3 + 2 * ST + a); };
  const uint32_t tmem_slot = bar_base + 8u * (5 + 2 * ST);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta = cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const int total_tiles = p.num_m_tiles * p.n_phases;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_b);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(b_full, 2);
    for (int s = 0; s < ST; ++s) {
      mbar_init(full_bar(s), 2);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 2 * 4);
    }
    fence_barrier_init();
  }
  cluster_sync_all();
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, 64);
    tmem_relinquish_2sm();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx_remote(b_full, 0, 2u * (uint32_t)p.n_kb * S::B_KB);
      for (int kb = 0; kb < p.n_kb; ++kb) {  // resident bank: rows [16 cta, +16) of every K block
        tma_load_3d_2sm(base + (uint32_t)kb * S::B_KB, &tm_b, b_full, kb * BK, (int)cta * 16, 0);
        tma_load_3d_2sm(base + S::B_PLANE + (uint32_t)kb * S::B_KB, &tm_b, b_full, kb * BK, (int)cta * 16, 1);
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < total_tiles; tile += num_pairs) {
        const int ph = tile / p.num_m_tiles, m_tile = tile - ph * p.num_m_tiles;
        const int m0 = m_tile * (2 * TC_BM) + (int)cta * TC_BM;
        for (int c = 0; c < p.hb && c < p.n_kb; ++c) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t ab = base + S::A_OFFSET + (uint32_t)stage * S::A_BUF;
          mbar_expect_tx_remote(full_bar(stage), 0, S::A_BUF);
          tma_load_4d_2sm(ab, &tm_a, full_bar(stage), c * BK, ph, m0, 0);
          tma_load_4d_2sm(ab + S::A_PLANE, &tm_a, full_bar(stage), c * BK, ph, m0, 1);
          if (++stage == ST) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (cta == 0 && elect_one()) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(32 >> 3) << 17) |
                             ((uint32_t)((2 * TC_BM) >> 4) << 24);
      mbar_wait(b_full, 0);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int tile = pair; tile < total_tiles; tile += num_pairs) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * 32u;
        uint32_t accumulate = 0;
        for (int c = 0; c < p.hb && c < p.n_kb; ++c) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t ab = base + S::A_OFFSET + (uint32_t)stage * S::A_BUF;
          for (int kb = c; kb < p.n_kb; kb += p.hb) {  // K blocks of this column: row shift kb / hb
            const uint32_t a_row = (uint32_t)(kb >> p.hb_log2) * (BK * 2);  // row shift kb / hb
            const uint32_t bh = base + (uint32_t)kb * S::B_KB, bl = bh + S::B_PLANE;
            umma_kblock_split3(d_tmem, smem_desc_lo<BK>(ab + a_row), smem_desc_lo<BK>(ab + S::A_PLANE + a_row),
                               smem_desc_lo<BK>(bh), smem_desc_lo<BK>(bl), smem_desc_hi<BK>(), idesc,
                               accumulate != 0);
            accumulate = 1u;
          }
          umma_commit_2sm(empty_bar(stage));
          if (++stage == ST) { stage = 0; phase ^= 1u; }
        }
        umma_commit_2sm(tfull_bar(acc));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    constexpr int CH = (FMT == NNAB_FMT_COMPLEX || FMT == NNAB_FMT_PHASE_UNIT) ? 2 : 1;
    for (int tile = pair; tile < total_tiles; tile += num_pairs) {
      const int ph = tile / p.num_m_tiles, m_tile = tile - ph * p.num_m_tiles;
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const int64_t g = (int64_t)m_tile * (2 * TC_BM) + (int64_t)cta * TC_BM + quarter * 32 + lane;
      const int64_t b = g / p.t_slots;
      const int64_t t = (g - b * p.t_slots) * p.n_phases + ph;
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * 32u;
      uint32_t re[16], im[16];
      tmem_ld8(trow, *reinterpret_cast<uint32_t(*)[8]>(&re[0]));
      tmem_ld8(trow + 8u, *reinterpret_cast<uint32_t(*)[8]>(&re[8]));
      tmem_ld8(trow + 16u, *reinterpret_cast<uint32_t(*)[8]>(&im[0]));
      tmem_ld8(trow + 24u, *reinterpret_cast<uint32_t(*)[8]>(&im[8]));
      tmem_ld_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(tempty_bar(acc), 0);  // the accumulator is in registers now
      if (g < p.nv && t < p.T) {
        float* dst = p.epi.out + (((int64_t)b * p.epi.out_bins + p.epi.bin_offset) * p.epi.T + t) * CH;
#pragma unroll
        for (int f = 0; f < 16; ++f)
          if (f < p.epi.F) epi_store_fmt<FMT>(p.epi, dst, f, __uint_as_float(re[f]), __uint_as_float(im[f]));
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc_2sm(tmem_base, 64);
  }
}

template <int FMT>
static int launch_octave_fmt(const CUtensorMap& ma, const CUtensorMap& mb, const OctParams& prm, int n_pairs,
                             cudaStream_t stream) {
  static std::atomic<uint64_t> configured_devs{0};
  int cfg_dev = 0;
  NNAB_CUDA_TRY(cudaGetDevice(&cfg_dev));
  if (!((configured_devs.load(std::memory_order_relaxed) >> (cfg_dev & 63)) & 1u)) {
    NNAB_CUDA_TRY(cudaFuncSetAttribute(octave_tc_kernel<FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)OctSmem::TOTAL));
    configured_devs.fetch_or(1ull << (cfg_dev & 63), std::memory_order_relaxed);
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * n_pairs));
  cfg.blockDim = dim3(OCT_THREADS);
  cfg.dynamicSmemBytes = OctSmem::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  NNAB_CUDA_TRY(cudaLaunchKernelEx(&cfg, octave_tc_kernel<FMT>, ma, mb, prm));
  count_launch();
  return NNAB_OK;
}

// q: an octave problem on caller-managed planes (presplit + presplit_t_slots); packed: the DENSE
// packed bank (tc_pack_basis) with bn = 32.  NNAB_EUNSUPPORTED = not applicable, nothing enqueued.
int launch_octave_tc(const FramedProblem& q, const void* packed, cudaStream_t stream) {
  if (const char* e = getenv("NNAB_OCTAVE_TC")) {
    if (atoi(e) == 0) return NNAB_EUNSUPPORTED;
  }
  if (q.presplit == nullptr || q.presplit_t_slots <= 0 || packed == nullptr) return NNAB_EUNSUPPORTED;
  if (q.F > 16 || tc_tile_n(q.F) != 32 || q.K % 64 != 0 || q.K / 64 > OCT_MAX_KB || q.B > 65535)
    return NNAB_EUNSUPPORTED;
  if (q.h_k_begin != nullptr) return NNAB_EUNSUPPORTED;
  if (q.fmt != NNAB_FMT_MAGNITUDE && q.fmt != NNAB_FMT_COMPLEX && q.fmt != NNAB_FMT_PHASE_UNIT)
    return NNAB_EUNSUPPORTED;
  int P = 1, hop_eff = q.hop;
  if (q.hop >= 64) {
    if (q.hop % 64 != 0) return NNAB_EUNSUPPORTED;
  } else {
    if (q.hop < 8 || 64 % q.hop != 0) return NNAB_EUNSUPPORTED;
    P = 64 / q.hop;
    hop_eff = 64;
  }
  const int hb = hop_eff / 64;
  const int n_kb = q.K / 64;
  if ((n_kb - 1) / hb > 8) return NNAB_EUNSUPPORTED;  // row shifts must fit the 136-row block
  const int64_t pitch = q.presplit_t_slots * q.hop;
  if (pitch % hop_eff != 0) return NNAB_EUNSUPPORTED;
  const int64_t t_slots = pitch / hop_eff;
  const int64_t plane_stride = q.presplit_plane_stride;
  __nv_bfloat16* planes = reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(q.presplit));

  int dev = 0, sms = 148;
  NNAB_CUDA_TRY(cudaGetDevice(&dev));
  NNAB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  sms -= sm_reserve();
  if (sms < 2) sms = 2;
  CUtensorMap ma, mb;
  {
    const int64_t rows = (plane_stride - (int64_t)(P - 1) * q.hop) / hop_eff;
    const uint64_t dims[4] = {(uint64_t)hop_eff, (uint64_t)P, (uint64_t)rows, 2};
    const uint64_t strides[3] = {(uint64_t)(P > 1 ? q.hop : hop_eff) * 2, (uint64_t)hop_eff * 2,
                                 (uint64_t)plane_stride * 2};
    const uint32_t box[3] = {64, 1, OCT_A_ROWS};
    if (encode_4d(&ma, planes, dims, strides, box)) return NNAB_EUNSUPPORTED;
  }
  const int kpad = round_up_i(q.K, 64);
  int rc = encode_3d(&mb, const_cast<void*>(packed), (uint64_t)kpad, 32, 2, (uint64_t)kpad * 2,
                     (uint64_t)32 * kpad * 2, 64, 16, 64);
  if (rc) return rc;
  OctParams prm{};
  prm.n_phases = P;
  prm.hb = hb;
  prm.hb_log2 = 0;
  while ((1 << prm.hb_log2) < hb) ++prm.hb_log2;
  if ((1 << prm.hb_log2) != hb) return NNAB_EUNSUPPORTED;
  prm.n_kb = n_kb;
  prm.nv = q.B * t_slots;
  prm.t_slots = t_slots;
  prm.T = q.T;
  prm.num_m_tiles = (int)ceil_div64(prm.nv, 2 * TC_BM);
  prm.epi.scale = q.scale; prm.epi.scale_all = q.scale_all; prm.epi.fmt = q.fmt;
  prm.epi.eps = q.eps; prm.epi.power = q.power; prm.epi.out = q.out; prm.epi.T = q.T;
  prm.epi.out_bins = q.out_bins; prm.epi.bin_offset = q.bin_offset; prm.epi.F = q.F;
  const int64_t tiles = (int64_t)prm.num_m_tiles * P;
  const int n_pairs = (int)(tiles < sms / 2 ? tiles : sms / 2);
  add_exec_flops(3.0 * 2.0 * (double)tiles * (2 * TC_BM) * 32.0 * q.K);
  switch (q.fmt) {
    case NNAB_FMT_MAGNITUDE: return launch_octave_fmt<0>(ma, mb, prm, n_pairs, stream);
    case NNAB_FMT_COMPLEX: return launch_octave_fmt<1>(ma, mb, prm, n_pairs, stream);
    case NNAB_FMT_PHASE_UNIT: return launch_octave_fmt<3>(ma, mb, prm, n_pairs, stream);
    default: return NNAB_EINVAL;
  }
}

}  // namespace nnab
